// crane_oracle.cpp — CPU oracle of CraneCtld's scheduling hot path.
//
// TEST INFRASTRUCTURE ONLY. Nothing under cranesched_b200/ may include, link
// or call this file; it exists so tests/ and bench.py can check the CUDA path
// against a line-by-line restatement of the reference algorithm and time a
// representative CPU baseline.
//
// PARITY STATUS: UNPINNED. The reference (PKUHPC/CraneSched @ e2992182) has no
// test of SchedulerAlgo / NodeSelect / priority / backfill and cannot be built
// in this image (needs GCC >= 14, ~20 network-fetched deps, protoc). The only
// known-answer vectors it holds for this path are the 14 DedicatedResourceInNode
// cases in test/Utilities/dedicated_resource_test.cpp:27-171, ported in
// crane_oracle_selftest() below. Third-party arithmetic restated from its
// published semantics: fpm::fixed<int64_t,__int128,8> (MikeLankamp/fpm @
// b46537fe, dependencies/cmake/fpm/CMakeLists.txt:6-8): raw = value * 2^8,
// to-double = raw / 256.0, to-int64 = raw / 256 truncating, *= uint multiplies
// raw.
//
// To be a representative CPU baseline the restatement keeps the reference's
// container choices: std::map timelines, std::set<pair<double,NodeState*>>
// cost order, std::set core-id and slot-id sets, string-keyed maps, per-job
// std::priority_queue of resource copies.
//
// Documented deviations (SURVEY.md §8c), all replacing nondeterministic order
// in the reference by a fixed rule that the GPU path also implements:
//   D1 equal-cost nodes are ordered by node index (ref: heap pointer order,
//      JobScheduler.h:588). NodeStates live in one vector in node-index order,
//      so pointer order IS index order here.
//   D2 equal-priority jobs keep input order (ref: unstable std::ranges::sort,
//      JobScheduler.cpp:6541) -> std::stable_sort.
//   D3 craned_ids are reported in node-index order (ref: unordered_map order,
//      JobScheduler.cpp:5365; satisfaction order, JobScheduler.h:836-841).
//   D4 gres names/types iterate in dictionary-index order (ref: unordered_map
//      order, PublicHeader.cpp:549,564,583) -> ordered std::map keyed by
//      zero-padded strings whose lexicographic order is the index order.
//   D5 built with -ffp-contract=off (ref: GCC default may fuse a*b+c).
//   D6 running jobs are visited in input order (ref: flat_hash_map order,
//      JobScheduler.cpp:1124).
//   D7 RnJobInScheduler::node_num is an explicit input (ref reads it
//      uninitialised, JobScheduler.h:69 vs JobScheduler.cpp:6614).
// Out of scope here (SURVEY.md §8f): reservations (R15), preemption (R14),
// licenses.

#include "crane_oracle.h"

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <functional>
#include <limits>
#include <list>
#include <map>
#include <memory>
#include <queue>
#include <set>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

namespace {

constexpr int64_t kInfFuture = std::numeric_limits<int64_t>::max();

// ---------------------------------------------------------------------------
// cpu_t: the subset of fpm::fixed<int64_t,__int128,8> the path uses
// (PublicHeader.h:44; call sites listed in SURVEY.md §8c).
// ---------------------------------------------------------------------------
struct CpuT {
  int64_t raw{0};
  static CpuT FromRaw(int64_t r) { CpuT c; c.raw = r; return c; }
  static CpuT FromInt(int64_t v) { return FromRaw(v * 256); }
  int64_t ToInt() const { return raw / 256; }          // truncates toward zero
  double ToDouble() const { return static_cast<double>(raw) / 256.0; }
  CpuT& operator+=(CpuT o) { raw += o.raw; return *this; }
  CpuT& operator-=(CpuT o) { raw -= o.raw; return *this; }
  CpuT& operator*=(uint32_t k) { raw *= static_cast<int64_t>(k); return *this; }
};
inline bool operator==(CpuT a, CpuT b) { return a.raw == b.raw; }
inline bool operator<(CpuT a, CpuT b) { return a.raw < b.raw; }
inline bool operator>(CpuT a, CpuT b) { return a.raw > b.raw; }
inline bool operator<=(CpuT a, CpuT b) { return a.raw <= b.raw; }

using SlotId = std::string;

// ---------------------------------------------------------------------------
// TypeSlotsMap / DedicatedResourceInNode  (PublicHeader.h:412-479,
// PublicHeader.cpp:159-359). Ordered maps instead of unordered (deviation D4).
// ---------------------------------------------------------------------------
struct TypeSlots {
  std::map<std::string, std::set<SlotId>> by_type;

  bool Empty() const { return by_type.empty(); }

  // PublicHeader.cpp:309-314
  void Add(const TypeSlots& o) {
    for (const auto& [t, s] : o.by_type) by_type[t].insert(s.begin(), s.end());
  }
  // PublicHeader.cpp:316-328 : set difference, drop types that become empty.
  void Sub(const TypeSlots& o) {
    for (const auto& [t, s] : o.by_type) {
      std::set<SlotId> rest;
      const std::set<SlotId>& mine = by_type.at(t);
      std::set_difference(mine.begin(), mine.end(), s.begin(), s.end(),
                          std::inserter(rest, rest.begin()));
      if (rest.empty())
        by_type.erase(t);
      else
        by_type[t] = std::move(rest);
    }
  }
};
// PublicHeader.cpp:334-343 : every lhs type present in rhs and a subset.
bool SlotsLe(const TypeSlots& a, const TypeSlots& b) {
  for (const auto& [t, s] : a.by_type) {
    auto it = b.by_type.find(t);
    if (it == b.by_type.end()) return false;
    if (!std::includes(it->second.begin(), it->second.end(), s.begin(), s.end()))
      return false;
  }
  return true;
}
// PublicHeader.cpp:345-359
TypeSlots SlotsIntersect(const TypeSlots& a, const TypeSlots& b) {
  TypeSlots r;
  for (const auto& [t, s] : a.by_type) {
    auto it = b.by_type.find(t);
    if (it == b.by_type.end()) continue;
    std::set<SlotId> both;
    std::set_intersection(s.begin(), s.end(), it->second.begin(),
                          it->second.end(), std::inserter(both, both.begin()));
    if (!both.empty()) r.by_type[t] = std::move(both);
  }
  return r;
}

struct DedicatedRes {
  std::map<std::string, TypeSlots> by_name;

  bool IsZero() const { return by_name.empty(); }   // PublicHeader.cpp:192
  TypeSlots& operator[](const std::string& n) { return by_name[n]; }

  // PublicHeader.cpp:196-202
  void Add(const DedicatedRes& o) {
    for (const auto& [n, ts] : o.by_name) by_name[n].Add(ts);
  }
  // PublicHeader.cpp:204-217 : names that become empty are erased.
  void Sub(const DedicatedRes& o) {
    for (const auto& [n, ts] : o.by_name) {
      auto it = by_name.find(n);
      if (it == by_name.end()) continue;  // reference asserts presence
      it->second.Sub(ts);
      if (it->second.Empty()) by_name.erase(it);
    }
  }
};
// PublicHeader.cpp:159-169
bool DedicatedLe(const DedicatedRes& a, const DedicatedRes& b) {
  for (const auto& [n, ts] : a.by_name) {
    auto it = b.by_name.find(n);
    if (it == b.by_name.end()) return false;
    if (!SlotsLe(ts, it->second)) return false;
  }
  return true;
}
bool DedicatedEq(const DedicatedRes& a, const DedicatedRes& b) {  // :171-174
  if (a.by_name.size() != b.by_name.size()) return false;
  auto ia = a.by_name.begin();
  auto ib = b.by_name.begin();
  for (; ia != a.by_name.end(); ++ia, ++ib) {
    if (ia->first != ib->first) return false;
    if (ia->second.by_type != ib->second.by_type) return false;
  }
  return true;
}
// PublicHeader.cpp:176-190
DedicatedRes DedicatedIntersect(const DedicatedRes& a, const DedicatedRes& b) {
  DedicatedRes r;
  for (const auto& [n, ts] : a.by_name) {
    auto it = b.by_name.find(n);
    if (it == b.by_name.end()) continue;
    TypeSlots both = SlotsIntersect(ts, it->second);
    if (!both.Empty()) r.by_name[n] = std::move(both);
  }
  return r;
}

// ---------------------------------------------------------------------------
// GresCount / GresMap (PublicHeader.h:490-523, PublicHeader.cpp:23-51)
// ---------------------------------------------------------------------------
struct GresCount {
  uint64_t total{0};
  std::map<std::string, uint64_t> specified;
  void Add(const GresCount& o) {
    total += o.total;
    for (const auto& [t, c] : o.specified) specified[t] += c;
  }
  void Mul(uint32_t k) {
    total *= k;
    for (auto& [t, c] : specified) c *= k;
  }
};
using GresMap = std::map<std::string, GresCount>;

// ---------------------------------------------------------------------------
// CpuSet / ResourceInNodeV3 (PublicHeader.h:540-615, PublicHeader.cpp:744-890)
// ---------------------------------------------------------------------------
struct ResInNode {
  std::set<uint32_t> core_ids;
  CpuT cpu_count;
  uint64_t mem{0};
  uint64_t mem_sw{0};
  DedicatedRes gres;

  // PublicHeader.cpp:781-787, 752-756
  void Add(const ResInNode& o) {
    core_ids.insert(o.core_ids.begin(), o.core_ids.end());
    cpu_count += o.cpu_count;
    mem += o.mem;
    mem_sw += o.mem_sw;
    gres.Add(o.gres);
  }
  // PublicHeader.cpp:789-796, 758-766 (tolerant core erase)
  void Sub(const ResInNode& o) {
    for (uint32_t id : o.core_ids) core_ids.erase(id);
    cpu_count -= o.cpu_count;
    mem -= o.mem;
    mem_sw -= o.mem_sw;
    gres.Sub(o.gres);
  }
  void SetToZero() {  // PublicHeader.cpp:808-813
    core_ids.clear();
    cpu_count = CpuT{};
    mem = mem_sw = 0;
    gres.by_name.clear();
  }
  // PublicHeader.cpp:815-827
  void Ckmin(const ResInNode& o) {
    cpu_count = std::min(cpu_count, o.cpu_count);
    if (!core_ids.empty() && !o.core_ids.empty()) {
      std::set<uint32_t> both;
      std::set_intersection(core_ids.begin(), core_ids.end(),
                            o.core_ids.begin(), o.core_ids.end(),
                            std::inserter(both, both.begin()));
      core_ids = std::move(both);
    }
    mem = std::min(mem, o.mem);
    mem_sw = std::min(mem_sw, o.mem_sw);
    gres = DedicatedIntersect(gres, o.gres);
  }
};
// PublicHeader.cpp:886-890 : core ids and mem_sw are NOT compared.
bool ResLe(const ResInNode& a, const ResInNode& b) {
  if (a.cpu_count > b.cpu_count) return false;
  if (a.mem > b.mem) return false;
  return DedicatedLe(a.gres, b.gres);
}

// ---------------------------------------------------------------------------
// ResourceView (PublicHeader.h:671-737, PublicHeader.cpp:448-481, 519-611)
// ---------------------------------------------------------------------------
struct ResView {
  CpuT cpu;
  uint64_t mem{0};
  uint64_t mem_sw{0};
  GresMap gres;

  void Add(const ResView& o) {  // PublicHeader.cpp:448-456
    cpu += o.cpu;
    mem += o.mem;
    mem_sw += o.mem_sw;
    for (const auto& [n, gc] : o.gres) gres[n].Add(gc);
  }
  void Mul(uint32_t k) {  // PublicHeader.cpp:473-481
    cpu *= k;
    mem *= k;
    mem_sw *= k;
    for (auto& [n, gc] : gres) gc.Mul(k);
  }
  double CpuDouble() const { return cpu.ToDouble(); }  // :509-511

  // PublicHeader.cpp:519-599. Picks concrete cores/slots out of `avail`.
  bool Feasible(const ResInNode& avail, ResInNode* out) const {
    if (cpu > avail.cpu_count) return false;
    if (mem > avail.mem) return false;

    ResInNode cand;
    int64_t whole = cpu.ToInt();
    bool integer_req =
        (CpuT::FromInt(whole) == cpu) && !avail.core_ids.empty();
    if (integer_req) {
      uint32_t n = static_cast<uint32_t>(whole);
      if (avail.core_ids.size() < n) return false;
      auto it = avail.core_ids.begin();
      for (uint32_t i = 0; i < n; ++i, ++it) cand.core_ids.insert(*it);
    }
    cand.cpu_count = cpu;
    cand.mem = mem;
    cand.mem_sw = mem_sw;

    for (const auto& [name, want] : gres) {
      auto have_it = avail.gres.by_name.find(name);
      if (have_it == avail.gres.by_name.end()) return false;
      const TypeSlots& have = have_it->second;

      uint64_t typed_sum = 0;
      for (const auto& [t, c] : want.specified) typed_sum += c;
      uint64_t untyped = want.total > typed_sum ? want.total - typed_sum : 0;

      TypeSlots& picked = cand.gres[name];
      // typed requests first; leftover slots of the same type then serve the
      // untyped part (PublicHeader.cpp:563-579)
      for (const auto& [t, c] : want.specified) {
        auto slots_it = have.by_type.find(t);
        if (slots_it == have.by_type.end()) return false;
        const std::set<SlotId>& slots = slots_it->second;
        if (slots.size() < c) return false;
        std::set<SlotId>& dst = picked.by_type[t];
        auto it = slots.begin();
        for (uint64_t i = 0; i < c; ++i, ++it) dst.insert(*it);
        for (; untyped > 0 && it != slots.end(); ++it, --untyped)
          dst.insert(*it);
      }
      // remaining untyped from the other types (PublicHeader.cpp:581-592)
      if (untyped > 0) {
        for (const auto& [t, slots] : have.by_type) {
          if (want.specified.count(t)) continue;
          auto it = slots.begin();
          for (; untyped > 0 && it != slots.end(); ++it, --untyped)
            picked.by_type[t].insert(*it);
          if (untyped == 0) break;
        }
      }
      if (untyped != 0) return false;
    }
    *out = std::move(cand);
    return true;
  }
};

// ---------------------------------------------------------------------------
// ABI <-> container conversions. Name/type/slot strings are zero-padded so
// lexicographic order == dictionary index order (deviation D4).
// ---------------------------------------------------------------------------
struct Dict {
  uint32_t n_entries{0};
  uint8_t entry_name[CRANE_GRES_ENTRIES]{};
  std::string name_str[CRANE_GRES_NAMES];
  std::string type_str[CRANE_GRES_ENTRIES];
  std::string slot_str[CRANE_MAX_SLOTS];
  explicit Dict(const crane_cluster_t* c) {
    if (c) {
      n_entries = std::min<uint32_t>(c->n_gres_entries, CRANE_GRES_ENTRIES);
      for (uint32_t e = 0; e < n_entries; ++e)
        entry_name[e] = c->gres_entry_name[e];
    }
    char buf[32];
    for (int g = 0; g < CRANE_GRES_NAMES; ++g) {
      snprintf(buf, sizeof buf, "gres%02d", g);
      name_str[g] = buf;
    }
    for (int e = 0; e < CRANE_GRES_ENTRIES; ++e) {
      snprintf(buf, sizeof buf, "type%02d", e);
      type_str[e] = buf;
    }
    for (int s = 0; s < CRANE_MAX_SLOTS; ++s) {
      snprintf(buf, sizeof buf, "/dev/slot%02d", s);
      slot_str[s] = buf;
    }
  }
};

ResInNode FromAbi(const Dict& d, const crane_res_in_node_t& r) {
  ResInNode x;
  x.cpu_count = CpuT::FromRaw(r.cpu_raw);
  x.mem = r.mem;
  x.mem_sw = r.mem_sw;
  for (int w = 0; w < CRANE_CORE_WORDS; ++w)
    for (int b = 0; b < 64; ++b)
      if (r.core[w] >> b & 1) x.core_ids.insert(w * 64 + b);
  for (uint32_t e = 0; e < d.n_entries; ++e) {
    if (!r.gres[e]) continue;
    std::set<SlotId>& s =
        x.gres[d.name_str[d.entry_name[e]]].by_type[d.type_str[e]];
    for (int b = 0; b < CRANE_MAX_SLOTS; ++b)
      if (r.gres[e] >> b & 1) s.insert(d.slot_str[b]);
  }
  return x;
}

void ToAbi(const Dict& d, const ResInNode& x, crane_res_in_node_t* r) {
  memset(r, 0, sizeof *r);
  r->cpu_raw = x.cpu_count.raw;
  r->mem = x.mem;
  r->mem_sw = x.mem_sw;
  for (uint32_t id : x.core_ids)
    if (id < 64 * CRANE_CORE_WORDS) r->core[id / 64] |= 1ull << (id % 64);
  for (uint32_t e = 0; e < d.n_entries; ++e) {
    auto nit = x.gres.by_name.find(d.name_str[d.entry_name[e]]);
    if (nit == x.gres.by_name.end()) continue;
    auto tit = nit->second.by_type.find(d.type_str[e]);
    if (tit == nit->second.by_type.end()) continue;
    for (int b = 0; b < CRANE_MAX_SLOTS; ++b)
      if (tit->second.count(d.slot_str[b])) r->gres[e] |= uint16_t(1u << b);
  }
}

ResView ViewFromAbi(const Dict& d, const crane_res_view_t& v) {
  ResView x;
  x.cpu = CpuT::FromRaw(v.cpu_raw);
  x.mem = v.mem;
  x.mem_sw = v.mem_sw;
  for (int g = 0; g < CRANE_GRES_NAMES; ++g) {
    bool any = v.gres_total[g] != 0;
    for (uint32_t e = 0; e < d.n_entries; ++e)
      if (d.entry_name[e] == g && v.gres_spec[e]) any = true;
    if (!any) continue;
    GresCount& gc = x.gres[d.name_str[g]];
    gc.total = v.gres_total[g];
    for (uint32_t e = 0; e < d.n_entries; ++e)
      if (d.entry_name[e] == g && v.gres_spec[e])
        gc.specified[d.type_str[e]] = v.gres_spec[e];
  }
  return x;
}

// ---------------------------------------------------------------------------
// Job records (JobScheduler.h:56-164), times in int64 seconds.
// ---------------------------------------------------------------------------
struct RnJob {
  int64_t start_time, end_time;
  uint32_t node_num;
  uint32_t partition_priority, qos_priority;
  std::string account;
  CpuT view_cpu;
  uint64_t view_mem;
  std::map<std::string, ResInNode> allocated_res;  // ResourceV3
  uint32_t reservation{0xffffffffu};               // index, 0xffffffff = none
};

struct PdJob {
  uint32_t index;  // input position == job-id order
  uint32_t reservation{0xffffffffu};
  int64_t time_limit;
  uint32_t partition;
  ResView req_node, req_task, req_total;
  uint32_t node_num, ntasks_min, ntasks_max, ntasks;
  bool exclusive;
  std::unordered_set<std::string> included, excluded;
  int64_t submit_time;
  uint32_t partition_priority, qos_priority;
  std::string account;
  double priority;
  std::map<std::string, uint32_t> node_task_num;   // craned_id_to_task_num
  int64_t start_time{0}, end_time{0};
  std::map<std::string, ResInNode> allocated_res;  // ResourceV3
  std::vector<std::string> craned_ids;
  int reason{CRANE_REASON_NONE};
};

// ---------------------------------------------------------------------------
// MinCpuTimeRatioFirst (JobScheduler.h:40-54)
// ---------------------------------------------------------------------------
inline void UpdateCostMinCpuTimeRatio(double& cost, int64_t start, int64_t end,
                                      const ResInNode& res,
                                      const ResInNode& total) {
  double delta = static_cast<double>(end - start) *
                 (res.cpu_count.ToDouble() / total.cpu_count.ToDouble());
  cost += delta;
}

// BestFit — NOT in the reference: BASELINE.json config 4 asks for "best-fit
// selection", defined here (SURVEY.md §8d) through the reference's own hook
// IUpdateNodeCostPolicy::UpdateCost (JobScheduler.h:30-38): a node's cost is
// its free cpu count over ALL allocations on it (running jobs and everything
// placed this tick, whenever it starts), so the fullest node comes first;
// NodeRater seeds the cost with the node's cpu count. Raw cpu_t values as
// doubles: integers, exact.
inline void UpdateCostBestFit(double& cost, const ResInNode& res) {
  cost -= static_cast<double>(res.cpu_count.raw);
}
inline void UpdateCostPolicy(uint32_t policy, double& cost, int64_t start, int64_t end,
                             const ResInNode& res, const ResInNode& total) {
  if (policy == 1) UpdateCostBestFit(cost, res);
  else UpdateCostMinCpuTimeRatio(cost, start, end, res, total);
}

// ---------------------------------------------------------------------------
// NodeState (JobScheduler.h:266-454)
// ---------------------------------------------------------------------------
using Timeline = std::map<int64_t, ResInNode>;

struct NodeState {
  std::string craned_id;
  uint32_t index;
  ResInNode res_total;
  ResInNode res_avail;
  struct Alloc { int64_t end_time; ResInNode res; };
  std::vector<Alloc> allocated;
  struct Resv { int64_t start_time, end_time; ResInNode res; };
  std::vector<Resv> reserved;  // reservations that start later (JobScheduler.cpp:5704-5711)
  Timeline timeline;

  // JobScheduler.h:295-332: change events = (-res at start, +res at end) of
  // every later reservation and +res at the end of every allocation; sorted by
  // time, a release before an allocation at the same time; `end` is the key of
  // the zero sentinel (+inf, or the end of the reservation this node belongs to).
  void InitTimeline(int64_t now, int64_t end = kInfFuture) {
    struct Change { int64_t t; bool alloc; const ResInNode* res; };
    std::vector<Change> changes;
    for (const auto& r : reserved) {
      changes.push_back({r.start_time, true, &r.res});
      changes.push_back({r.end_time, false, &r.res});
    }
    for (const auto& a : allocated) {
      changes.push_back({a.end_time, false, &a.res});
      res_avail.Sub(a.res);
    }
    std::stable_sort(changes.begin(), changes.end(), [](const Change& l, const Change& r) {
      return l.t < r.t || (l.t == r.t && l.alloc < r.alloc);
    });
    auto cur = timeline.emplace(now, res_avail).first;
    for (const auto& ch : changes) {
      if (ch.t != cur->first) cur = timeline.emplace(ch.t, cur->second).first;
      if (ch.alloc) cur->second.Sub(*ch.res); else cur->second.Add(*ch.res);
    }
    timeline[end].SetToZero();
  }

  // JobScheduler.h:334-453, allocation direction only (is_release=false).
  void Update(int64_t start, int64_t end, const ResInNode& res) {
    auto begin_it = timeline.upper_bound(start);
    if (begin_it == timeline.end()) {
      // cases #1/#2: start at or after the last key (unreachable while the
      // +inf sentinel exists; kept for fidelity)
      --begin_it;
      timeline.emplace(end, begin_it->second);
      if (begin_it->first == start) {
        begin_it->second.Sub(res);
      } else {
        auto ins = timeline.emplace(start, begin_it->second).first;
        ins->second.Sub(res);
      }
      return;
    }
    --begin_it;  // key <= start
    if (begin_it->first != start)  // case #3: split the covering segment
      begin_it = timeline.emplace(start, begin_it->second).first;
    auto end_it = std::prev(timeline.upper_bound(end));  // key <= end
    for (auto it = begin_it; it != end_it; ++it) it->second.Sub(res);
    if (end_it->first != end) {
      timeline.emplace(end, end_it->second);
      end_it->second.Sub(res);
    }
  }
};

// ---------------------------------------------------------------------------
// NodeSelector (JobScheduler.h:486-589) with the MinCpuTimeRatioFirst policy
// ---------------------------------------------------------------------------
struct NodeSelector {
  struct Rater {
    NodeState* node;
    double cost;
    std::set<std::pair<double, NodeState*>>::iterator pos;
  };
  std::unordered_map<std::string, Rater> info;
  std::set<std::pair<double, NodeState*>> order;  // (cost, pointer==index) D1
  uint32_t policy{0};                             // crane_sched_config_t::cost_policy

  void AddNode(int64_t now, NodeState* ns) {  // JobScheduler.h:492-505,534-544
    double cost = policy == 1 ? static_cast<double>(ns->res_total.cpu_count.raw) : 0.0;
    for (const auto& r : ns->reserved)  // JobScheduler.h:496-500
      UpdateCostPolicy(policy, cost, r.start_time, r.end_time, r.res, ns->res_total);
    for (const auto& a : ns->allocated)
      UpdateCostPolicy(policy, cost, now, a.end_time, a.res, ns->res_total);
    Rater& r = info.emplace(ns->craned_id, Rater{ns, cost, {}}).first->second;
    r.pos = order.emplace(r.cost, ns).first;
  }
  void UpdateCost(const std::string& id, int64_t s, int64_t e,
                  const ResInNode& res) {  // JobScheduler.h:520-532
    Rater& r = info.at(id);
    order.erase(r.pos);
    UpdateCostPolicy(policy, r.cost, s, e, res, r.node->res_total);
    r.pos = order.emplace(r.cost, r.node).first;
  }
  void Allocate(int64_t s, int64_t e,
                const std::map<std::string, ResInNode>& res) {  // :561-569
    for (const auto& [id, r] : res) {
      info.at(id).node->Update(s, e, r);
      UpdateCost(id, s, e, r);
    }
  }
};

// ---------------------------------------------------------------------------
// Earliest-start selector (JobScheduler.h:672-859)
// ---------------------------------------------------------------------------
struct TrackList;
struct Cursor {  // TimeAvailResMapIter
  const std::string* craned_id;
  Timeline::const_iterator it, end;
  const ResInNode* job_res;
  bool satisfied;
  std::list<struct TrackNode>::iterator where;
  bool Sat() const { return ResLe(*job_res, it->second); }
  bool AtEnd() const { return it == end; }
  void Advance() {  // JobScheduler.h:764-773
    satisfied = !satisfied;
    if (satisfied) {
      while (++it != end && !Sat()) {}
    } else {
      while (++it != end && Sat()) {}
    }
  }
};
struct TrackNode { Cursor* cur; int64_t time; bool first_k; };
struct TrackList {  // ResMapIterList, JobScheduler.h:672-729
  std::list<TrackNode> items;
  size_t k;
  std::list<TrackNode>::iterator kth;
  explicit TrackList(size_t k_) : k(k_), kth(items.end()) {}
  void PushBack(Cursor* c, int64_t t) {
    if (c->where != items.end()) return;
    items.push_back(TrackNode{c, t, items.size() < k});
    if (items.size() == k) kth = std::prev(items.end());
    c->where = std::prev(items.end());
  }
  void Erase(Cursor* c) {
    if (c->where == items.end()) return;
    if (kth != items.end() && c->where->first_k) {
      kth = std::next(kth);
      if (kth != items.end()) kth->first_k = true;
    }
    items.erase(c->where);
    c->where = items.end();
  }
  int64_t KthTime() const { return kth == items.end() ? kInfFuture : kth->time; }
};

bool EarliestStart(int64_t now, int64_t max_window, PdJob* job,
                   const std::vector<NodeState*>& nodes) {
  TrackList sat(job->node_num);
  std::vector<Cursor> cursors;
  cursors.reserve(nodes.size());
  auto later = [](const Cursor* a, const Cursor* b) {
    return a->it->first > b->it->first;
  };
  std::priority_queue<Cursor*, std::vector<Cursor*>,
                      std::function<bool(const Cursor*, const Cursor*)>>
      pq(later);
  for (NodeState* n : nodes) {
    Cursor c;
    c.craned_id = &n->craned_id;
    c.it = n->timeline.begin();
    c.end = n->timeline.end();
    c.job_res = &job->allocated_res.at(n->craned_id);
    c.where = sat.items.end();
    c.satisfied = c.Sat();
    cursors.push_back(c);
    pq.push(&cursors.back());
  }
  // JobScheduler.h:806-849
  while (!pq.empty()) {
    int64_t t = pq.top()->it->first;
    // `current_time - now > kAlgoMaxTimeWindow`; the +inf sentinel is always
    // beyond the window (absl::InfiniteFuture() - now is infinite).
    if (t == kInfFuture || t - now > max_window) return false;
    while (!pq.empty()) {
      Cursor* c = pq.top();
      if (c->it->first != t) break;
      pq.pop();
      if (c->satisfied)
        sat.PushBack(c, t);
      else
        sat.Erase(c);
      c->Advance();
      if (!c->AtEnd()) pq.push(c);
    }
    int64_t kth = sat.KthTime();
    if (kth == kInfFuture) continue;
    bool fits = pq.empty();
    if (!fits) {
      int64_t next = pq.top()->it->first;
      fits = (next == kInfFuture) || (kth + job->time_limit <= next);
    }
    if (fits) {
      job->start_time = kth;
      job->craned_ids.clear();
      for (auto it = sat.items.begin();; ++it) {
        job->craned_ids.push_back(*it->cur->craned_id);
        if (it == sat.kth) break;
      }
      return true;
    }
  }
  return false;
}

// ---------------------------------------------------------------------------
// LocalScheduler (JobScheduler.cpp:5165-5412)
// ---------------------------------------------------------------------------
struct LocalScheduler {
  NodeSelector sel;
  uint32_t max_jobs_per_node;
  int64_t max_window;

  // JobScheduler.cpp:5185-5405
  bool GetNodesAndTry(int64_t now, PdJob* job, std::vector<NodeState*>* to_sched) {
    int64_t earliest_end = now + job->time_limit;
    ResView min_view = job->req_task;
    min_view.Mul(job->ntasks_min);
    {
      ResView t = job->req_node;
      t.Add(min_view);
      min_view = std::move(t);
    }
    struct Info {
      int ntasks;
      ResInNode res;
      NodeState* node;
      bool operator<(const Info& o) const { return ntasks > o.ntasks; }
    };
    std::priority_queue<Info> top_total, top_avail;
    int sum_total = 0, sum_avail = 0;

    auto max_tasks = [&](const ResInNode& on_node) {  // :5207-5222
      ResInNode got;
      if (!min_view.Feasible(on_node, &got)) return 0;
      ResInNode rest = on_node;
      rest.Sub(got);
      int n = static_cast<int>(job->ntasks_min);
      while (n < static_cast<int>(job->ntasks_max) &&
             job->req_task.Feasible(rest, &got)) {
        ++n;
        rest.Sub(got);
      }
      return n;
    };

    for (const auto& entry : sel.order) {
      NodeState* ns = entry.second;
      if (ns->timeline.size() >= max_jobs_per_node) continue;          // :5230
      if (!job->included.empty() && !job->included.count(ns->craned_id))
        continue;                                                      // :5238
      if (!job->excluded.empty() && job->excluded.count(ns->craned_id))
        continue;                                                      // :5249
      int n_total = max_tasks(ns->res_total);                          // :5258
      if (n_total == 0) continue;

      if (top_total.size() < job->node_num ||
          sum_total < static_cast<int>(job->ntasks)) {                 // :5269
        sum_total += n_total;
        top_total.push(Info{n_total, ns->res_total, ns});
        if (top_total.size() > job->node_num) {
          sum_total -= top_total.top().ntasks;
          top_total.pop();
        }
      }

      if (job->exclusive) {                                            // :5285
        bool ok = true;
        for (const auto& [t, res] : ns->timeline) {
          if (t >= earliest_end) break;
          if (!ResLe(ns->res_total, res)) { ok = false; break; }
        }
        if (!ok) continue;
        sum_avail += n_total;
        top_avail.push(Info{n_total, ns->res_total, ns});
        if (top_avail.size() > job->node_num) {
          sum_avail -= top_avail.top().ntasks;
          top_avail.pop();
        }
        if (top_avail.size() == job->node_num &&
            sum_avail >= static_cast<int>(job->ntasks))
          break;
      } else {                                                         // :5308
        ResInNode got;
        if (!min_view.Feasible(ns->res_avail, &got)) continue;
        ResInNode window_min = ns->res_avail;
        for (const auto& [t, res] : ns->timeline) {
          if (t >= earliest_end) break;
          window_min.Ckmin(res);
        }
        int n_avail = max_tasks(window_min);
        if (n_avail) {
          sum_avail += n_avail;
          top_avail.push(Info{n_avail, window_min, ns});
          if (top_avail.size() > job->node_num) {
            sum_avail -= top_avail.top().ntasks;
            top_avail.pop();
          }
          if (top_avail.size() == job->node_num &&
              sum_avail >= static_cast<int>(job->ntasks))
            break;
        }
      }
    }

    auto hand_out = [&](std::priority_queue<Info>& q,
                        std::vector<NodeState*>* collect) {  // :5340-5361,5381-5403
      int rest = static_cast<int>(job->ntasks) - static_cast<int>(job->node_num);
      while (!q.empty()) {
        const Info& info = q.top();
        int n = std::min(rest, info.ntasks - 1) + 1;
        if (job->exclusive) {
          job->allocated_res[info.node->craned_id].Add(info.res);
        } else {
          ResView want = job->req_task;
          want.Mul(static_cast<uint32_t>(n));
          ResView full = job->req_node;
          full.Add(want);
          ResInNode got;
          bool ok = full.Feasible(info.res, &got);
          (void)ok;  // reference asserts
          job->allocated_res[info.node->craned_id].Add(got);
        }
        job->node_task_num[info.node->craned_id] = static_cast<uint32_t>(n);
        if (collect) collect->push_back(info.node);
        rest -= n - 1;
        q.pop();
      }
    };

    if (top_avail.size() == job->node_num &&
        sum_avail >= static_cast<int>(job->ntasks)) {                  // :5338
      hand_out(top_avail, nullptr);
      job->start_time = now;
      job->craned_ids.clear();
      for (const auto& [id, n] : job->node_task_num) job->craned_ids.push_back(id);
      return true;
    }
    if (top_total.size() < job->node_num ||
        sum_total < static_cast<int>(job->ntasks))                     // :5371
      return false;
    hand_out(top_total, to_sched);
    return false;
  }

  // JobScheduler.cpp:5165-5183 with PreemptType == PREEMPT_NONE
  bool Schedule(int64_t now, PdJob* job) {
    std::vector<NodeState*> to_sched;
    if (GetNodesAndTry(now, job, &to_sched)) return true;
    if (to_sched.size() < job->node_num) return false;
    return EarliestStart(now, max_window, job, to_sched);              // :5407
  }
};

// ---------------------------------------------------------------------------
// Priority sorters (JobScheduler.h:177-195, JobScheduler.cpp:6526-6739)
// ---------------------------------------------------------------------------
struct FactorBound {
  uint64_t age_max, age_min;
  uint32_t qos_max, qos_min, part_max, part_min, nodes_max, nodes_min;
  uint64_t mem_max, mem_min;
  double cpus_max, cpus_min, svc_max, svc_min;
  std::unordered_map<std::string, double> acc_service;
};

void FactorBounds(const crane_sched_config_t& cfg, int64_t now,
                  const std::vector<std::unique_ptr<PdJob>>& pd,
                  const std::vector<std::unique_ptr<RnJob>>& rn,
                  FactorBound& b) {  // JobScheduler.cpp:6553-6672
  b.age_max = 0; b.age_min = std::numeric_limits<uint64_t>::max();
  b.qos_max = 0; b.qos_min = std::numeric_limits<uint32_t>::max();
  b.part_max = 0; b.part_min = std::numeric_limits<uint32_t>::max();
  b.nodes_max = 0; b.nodes_min = std::numeric_limits<uint32_t>::max();
  b.mem_max = 0; b.mem_min = std::numeric_limits<uint64_t>::max();
  b.cpus_max = 0; b.cpus_min = std::numeric_limits<double>::max();
  b.svc_max = 0; b.svc_min = std::numeric_limits<uint32_t>::max();
  b.acc_service.clear();

  for (const auto& j : pd) {
    uint64_t age = static_cast<uint64_t>(now - j->submit_time);
    age = std::min<uint64_t>(age, cfg.max_age_s);
    b.acc_service[j->account] = 0.0;
    b.age_min = std::min(age, b.age_min);
    b.age_max = std::max(age, b.age_max);
    b.nodes_min = std::min(j->node_num, b.nodes_min);
    b.nodes_max = std::max(j->node_num, b.nodes_max);
    b.mem_min = std::min(j->req_total.mem, b.mem_min);
    b.mem_max = std::max(j->req_total.mem, b.mem_max);
    double c = j->req_total.CpuDouble();
    b.cpus_min = std::min(c, b.cpus_min);
    b.cpus_max = std::max(c, b.cpus_max);
    b.qos_min = std::min(j->qos_priority, b.qos_min);
    b.qos_max = std::max(j->qos_priority, b.qos_max);
    b.part_min = std::min(j->partition_priority, b.part_min);
    b.part_max = std::max(j->partition_priority, b.part_max);
  }
  for (const auto& j : rn) {
    b.nodes_min = std::min(j->node_num, b.nodes_min);
    b.nodes_max = std::max(j->node_num, b.nodes_max);
    b.mem_min = std::min(j->view_mem, b.mem_min);
    b.mem_max = std::max(j->view_mem, b.mem_max);
    double c = j->view_cpu.ToDouble();
    b.cpus_min = std::min(c, b.cpus_min);
    b.cpus_max = std::max(c, b.cpus_max);
    b.qos_min = std::min(j->qos_priority, b.qos_min);
    b.qos_max = std::max(j->qos_priority, b.qos_max);
    b.part_min = std::min(j->partition_priority, b.part_min);
    b.part_max = std::max(j->partition_priority, b.part_max);
  }
  for (const auto& j : rn) {  // deviation D6: input order
    double sv = 0;
    if (b.cpus_max > b.cpus_min)
      sv += 1.0 * (j->view_cpu.ToDouble() - b.cpus_min) / (b.cpus_max - b.cpus_min);
    else
      sv += 1.0;
    if (b.nodes_max > b.nodes_min)
      sv += 1.0 * (j->node_num - b.nodes_min) / (b.nodes_max - b.nodes_min);
    else
      sv += 1.0;
    if (b.mem_max > b.mem_min)
      sv += 1.0 * static_cast<double>(j->view_mem - b.mem_min) /
            static_cast<double>(b.mem_max - b.mem_min);
    else
      sv += 1.0;
    uint64_t run_time = static_cast<uint64_t>(now - j->start_time);
    b.acc_service[j->account] += sv * static_cast<double>(run_time);
  }
  for (const auto& [acc, v] : b.acc_service) {
    b.svc_min = std::min(v, b.svc_min);
    b.svc_max = std::max(v, b.svc_max);
  }
}

double JobPriority(const crane_sched_config_t& cfg, int64_t now,
                   const FactorBound& b, const PdJob* j) {  // :6674-6739
  uint64_t age = static_cast<uint64_t>(now - j->submit_time);
  age = std::min<uint64_t>(age, cfg.max_age_s);
  uint32_t qos = j->qos_priority, part = j->partition_priority;
  uint32_t nodes = j->node_num;
  uint64_t mem = j->req_total.mem;
  double cpus = j->req_total.CpuDouble();
  double svc = b.acc_service.at(j->account);

  double f_qos = 0, f_age = 0, f_part = 0, f_size = 0, f_fs = 0;
  if (b.age_max > b.age_min)
    f_age = 1.0 * static_cast<double>(age - b.age_min) /
            static_cast<double>(b.age_max - b.age_min);
  if (b.qos_max > b.qos_min)
    f_qos = 1.0 * (qos - b.qos_min) / (b.qos_max - b.qos_min);
  if (b.part_max > b.part_min)
    f_part = 1.0 * (part - b.part_min) / (b.part_max - b.part_min);
  if (b.cpus_max > b.cpus_min)
    f_size += 1.0 * (cpus - b.cpus_min) / (b.cpus_max - b.cpus_min);
  if (b.nodes_max > b.nodes_min)
    f_size += 1.0 * (nodes - b.nodes_min) / (b.nodes_max - b.nodes_min);
  if (b.mem_max > b.mem_min)
    f_size += 1.0 * static_cast<double>(mem - b.mem_min) /
              static_cast<double>(b.mem_max - b.mem_min);
  if (cfg.favor_small)
    f_size = 1.0 - f_size / 3;
  else
    f_size /= 3.0;
  if (b.svc_max > b.svc_min)
    f_fs = 1.0 - (svc - b.svc_min) / (b.svc_max - b.svc_min);

  double p = cfg.weight_age * f_age + cfg.weight_partition * f_part +
             cfg.weight_job_size * f_size + cfg.weight_fair_share * f_fs +
             cfg.weight_qos * f_qos;
  return p;
}

void OrderJobs(const crane_sched_config_t& cfg, int64_t now,
               const std::vector<std::unique_ptr<PdJob>>& pd,
               const std::vector<std::unique_ptr<RnJob>>& rn,
               std::vector<PdJob*>& order) {
  size_t limit = cfg.scheduled_batch_size;
  if (cfg.priority_type == 0) {  // BasicPriority, JobScheduler.h:179-194
    size_t len = std::min(pd.size(), limit);
    order.reserve(len);
    for (size_t i = 0; i < len; ++i) order.push_back(pd[i].get());
    for (size_t i = len; i < pd.size(); ++i) pd[i]->reason = CRANE_REASON_PRIORITY;
    return;
  }
  FactorBound b;  // MultiFactorPriority, JobScheduler.cpp:6526-6551
  FactorBounds(cfg, now, pd, rn, b);
  order.reserve(pd.size());
  for (const auto& j : pd) {
    if (j->priority == 0.0) j->priority = JobPriority(cfg, now, b, j.get());
    order.push_back(j.get());
  }
  std::stable_sort(order.begin(), order.end(),  // deviation D2
                   [](const PdJob* a, const PdJob* c) { return a->priority > c->priority; });
  if (order.size() > limit) {
    for (size_t i = limit; i < order.size(); ++i)
      order[i]->reason = CRANE_REASON_PRIORITY;
    order.resize(limit);
  }
}

std::string NodeName(uint32_t idx) {
  char buf[24];
  snprintf(buf, sizeof buf, "cn%08u", idx);  // lexicographic == index order
  return buf;
}

}  // namespace

// ===========================================================================
// C interface
// ===========================================================================
namespace { const crane_reservations_t* g_resv = nullptr; }
extern "C" void crane_oracle_set_reservations(const crane_reservations_t* resv) { g_resv = resv; }

extern "C" int crane_oracle_node_select(
    const crane_sched_config_t* cfg, const crane_cluster_t* cl, int64_t now,
    const crane_running_t* running, const crane_pending_t* pending,
    crane_placements_t* out, double* elapsed_ms, uint32_t max_jobs,
    uint32_t* jobs_done) {
  if (!cfg || !cl || !pending || !out) return CRANE_EINVAL;
  Dict dict(cl);
  const uint32_t M = cl->n_nodes;
  const uint32_t N = pending->n;
  const uint32_t R = running ? running->n : 0;

  std::vector<std::string> node_names(M);
  for (uint32_t i = 0; i < M; ++i) node_names[i] = NodeName(i);

  // --- what JobScheduler.cpp:1090-1127 builds before the timed region ------
  std::vector<std::unique_ptr<PdJob>> pd;
  pd.reserve(N);
  for (uint32_t i = 0; i < N; ++i) {
    auto j = std::make_unique<PdJob>();
    j->index = i;
    j->time_limit = pending->time_limit[i];
    j->partition = pending->partition[i];
    j->req_node = ViewFromAbi(dict, pending->req_node[i]);
    j->req_task = ViewFromAbi(dict, pending->req_task[i]);
    j->req_total = ViewFromAbi(dict, pending->req_total[i]);
    j->node_num = pending->node_num[i];
    j->ntasks_min = pending->ntasks_per_node_min[i];
    j->ntasks_max = pending->ntasks_per_node_max[i];
    j->ntasks = pending->ntasks[i];
    j->exclusive = pending->exclusive[i] != 0;
    if (pending->incl_off)
      for (uint32_t k = pending->incl_off[i]; k < pending->incl_off[i + 1]; ++k)
        j->included.insert(NodeName(pending->incl_nodes[k]));
    if (pending->excl_off)
      for (uint32_t k = pending->excl_off[i]; k < pending->excl_off[i + 1]; ++k)
        j->excluded.insert(NodeName(pending->excl_nodes[k]));
    j->submit_time = pending->submit_time[i];
    j->partition_priority = pending->partition_priority[i];
    j->qos_priority = pending->qos_priority[i];
    j->account = "acct" + std::to_string(pending->account[i]);
    j->priority = pending->mandated_priority ? pending->mandated_priority[i] : 0.0;
    if (pending->reservation) j->reservation = pending->reservation[i];
    pd.push_back(std::move(j));
  }
  std::vector<std::unique_ptr<RnJob>> rn;
  rn.reserve(R);
  for (uint32_t i = 0; i < R; ++i) {
    auto j = std::make_unique<RnJob>();
    j->start_time = running->start_time[i];
    j->end_time = running->end_time[i];
    j->node_num = running->node_num[i];
    j->partition_priority = running->partition_priority[i];
    j->qos_priority = running->qos_priority[i];
    j->account = "acct" + std::to_string(running->account[i]);
    j->view_cpu = CpuT::FromRaw(running->view_cpu_raw[i]);
    j->view_mem = running->view_mem[i];
    if (running->reservation) j->reservation = running->reservation[i];
    for (uint32_t k = running->alloc_off[i]; k < running->alloc_off[i + 1]; ++k)
      j->allocated_res[node_names[running->alloc_node[k]]].Add(
          FromAbi(dict, running->alloc_res[k]));
    rn.push_back(std::move(j));
  }
  // g_meta_container's view: res_total per node (CranedMeta, NodeDefs.h:57-79)
  std::vector<ResInNode> totals(M);
  for (uint32_t i = 0; i < M; ++i) totals[i] = FromAbi(dict, cl->res_total[i]);

  auto t0 = std::chrono::steady_clock::now();

  // ======================= NodeSelect (JobScheduler.cpp:5543) ==============
  for (auto& j : rn) j->end_time = std::max(j->end_time, now + 1);      // :5547

  std::vector<char> part_has_jobs(cl->n_partitions, 0);                 // :5551
  const uint32_t n_resv = g_resv ? g_resv->n : 0;
  std::vector<char> resv_has_jobs(n_resv, 0);
  for (const auto& j : pd) {  // :5557-5562: a job sits in its reservation's list or in its partition's
    if (j->reservation != 0xffffffffu) {
      if (j->reservation < n_resv) resv_has_jobs[j->reservation] = 1;
    } else if (j->partition < cl->n_partitions) {
      part_has_jobs[j->partition] = 1;
    }
  }

  // node_state_map (:5597-5651). One vector in node-index order => pointer
  // order == index order (deviation D1).
  std::vector<NodeState> states(M);
  std::vector<char> in_map(M, 0);
  std::unordered_map<std::string, NodeState*> state_by_name;
  std::vector<std::vector<NodeState*>> part_nodes(cl->n_partitions);
  for (uint32_t p = 0; p < cl->n_partitions; ++p) {
    if (!part_has_jobs[p]) continue;
    for (uint32_t k = cl->part_off[p]; k < cl->part_off[p + 1]; ++k) {
      uint32_t n = cl->part_nodes[k];
      if (!in_map[n]) {
        if (!cl->alive[n] || cl->drain[n]) continue;                    // :5629
        in_map[n] = 1;
        states[n].craned_id = node_names[n];
        states[n].index = n;
        states[n].res_total = totals[n];
        states[n].res_avail = totals[n];
        state_by_name.emplace(node_names[n], &states[n]);
      }
      part_nodes[p].push_back(&states[n]);
    }
  }
  // reservations (:5655-5713)
  struct ResvSched {
    int64_t end_time{0};
    // node states holding the reserved resources, ONE vector in node-index order: the cost
    // set orders equal costs by NodeState address (JobScheduler.h:588), deviation D1
    std::vector<NodeState> states;
    std::map<std::string, NodeState*> nodes;
    std::unique_ptr<LocalScheduler> sched;
  };
  std::vector<std::unique_ptr<ResvSched>> resv_scheds(n_resv);
  std::unordered_map<std::string, int64_t> first_resv;  // craned_id_first_resv_map
  for (uint32_t r = 0; r < n_resv; ++r) {
    const int64_t rs = g_resv->start_time[r], re = g_resv->end_time[r];
    if (now >= re) continue;  // expired but not cleaned up
    for (uint32_t k = g_resv->node_off[r]; k < g_resv->node_off[r + 1]; ++k) {
      const std::string& id = node_names[g_resv->node[k]];
      auto it = first_resv.find(id);
      if (it == first_resv.end()) first_resv[id] = rs;
      else if (rs < it->second) it->second = rs;
    }
    if (now >= rs) {
      for (uint32_t k = g_resv->node_off[r]; k < g_resv->node_off[r + 1]; ++k) {
        auto it = state_by_name.find(node_names[g_resv->node[k]]);
        if (it != state_by_name.end()) it->second->allocated.push_back({re, FromAbi(dict, g_resv->res[k])});
      }
      if (!resv_has_jobs[r]) continue;
      auto rsd = std::make_unique<ResvSched>();
      rsd->end_time = re;
      std::vector<uint32_t> ks;
      for (uint32_t k = g_resv->node_off[r]; k < g_resv->node_off[r + 1]; ++k) ks.push_back(k);
      std::sort(ks.begin(), ks.end(), [&](uint32_t x, uint32_t y) { return g_resv->node[x] < g_resv->node[y]; });
      rsd->states.resize(ks.size());
      for (size_t i = 0; i < ks.size(); ++i) {
        NodeState& ns = rsd->states[i];
        ns.craned_id = node_names[g_resv->node[ks[i]]];
        ns.index = g_resv->node[ks[i]];
        ns.res_total = FromAbi(dict, g_resv->res[ks[i]]);
        ns.res_avail = ns.res_total;
        rsd->nodes[ns.craned_id] = &ns;
      }
      resv_scheds[r] = std::move(rsd);
    } else {
      for (uint32_t k = g_resv->node_off[r]; k < g_resv->node_off[r + 1]; ++k) {
        auto it = state_by_name.find(node_names[g_resv->node[k]]);
        if (it != state_by_name.end()) it->second->reserved.push_back({rs, re, FromAbi(dict, g_resv->res[k])});
      }
    }
  }
  for (const auto& j : rn) {                                            // :5715
    if (j->reservation == 0xffffffffu) {
      for (const auto& [id, res] : j->allocated_res) {
        auto it = state_by_name.find(id);
        if (it != state_by_name.end())
          it->second->allocated.push_back({j->end_time, res});
      }
    } else {
      if (j->reservation >= n_resv || !resv_scheds[j->reservation]) continue;  // :5727 (error logged, job skipped)
      for (const auto& [id, res] : j->allocated_res) {
        auto it = resv_scheds[j->reservation]->nodes.find(id);
        if (it != resv_scheds[j->reservation]->nodes.end()) it->second->allocated.push_back({j->end_time, res});
      }
    }
  }
  for (uint32_t n = 0; n < M; ++n)                                      // :5746
    if (in_map[n]) states[n].InitTimeline(now);
  for (auto& rsd : resv_scheds)
    if (rsd)
      for (auto& ns : rsd->states) ns.InitTimeline(now, rsd->end_time);

  std::vector<std::unique_ptr<LocalScheduler>> scheds(cl->n_partitions);
  for (uint32_t p = 0; p < cl->n_partitions; ++p) {                     // :5757
    if (!part_has_jobs[p]) continue;
    scheds[p] = std::make_unique<LocalScheduler>();
    scheds[p]->max_jobs_per_node = cfg->max_jobs_per_node;
    scheds[p]->max_window = cfg->max_time_window_s;
    scheds[p]->sel.policy = cfg->cost_policy;
    for (NodeState* ns : part_nodes[p]) scheds[p]->sel.AddNode(now, ns);
  }
  for (auto& rsd : resv_scheds) {                                       // :5763
    if (!rsd) continue;
    rsd->sched = std::make_unique<LocalScheduler>();
    rsd->sched->max_jobs_per_node = cfg->max_jobs_per_node;
    rsd->sched->max_window = cfg->max_time_window_s;
    rsd->sched->sel.policy = cfg->cost_policy;
    // node states in node-index order: pointer order == index order (deviation D1)
    for (NodeState& ns : rsd->states) rsd->sched->sel.AddNode(now, &ns);
  }

  std::vector<PdJob*> order;
  OrderJobs(*cfg, now, pd, rn, order);                                  // :5769

  uint32_t done = 0;
  for (PdJob* job : order) {                                            // :5777
    if (max_jobs && done >= max_jobs) break;
    ++done;
    if (job->reason != CRANE_REASON_NONE) continue;
    LocalScheduler* s = nullptr;
    ResvSched* rsd = nullptr;
    if (job->reservation == 0xffffffffu) {
      if (job->partition >= cl->n_partitions || !scheds[job->partition]) {
        job->reason = CRANE_REASON_PART_NOT_FOUND;                      // :5784
        continue;
      }
      s = scheds[job->partition].get();
    } else {
      if (job->reservation >= n_resv || !resv_scheds[job->reservation]) {
        job->reason = CRANE_REASON_RESV_NOT_FOUND;                      // :5793
        continue;
      }
      rsd = resv_scheds[job->reservation].get();
      s = rsd->sched.get();
    }
    bool ok = s->Schedule(now, job);
    if (!ok) {
      job->reason = CRANE_REASON_RESOURCE;                              // :5802
      continue;
    }
    job->end_time = job->start_time + job->time_limit;
    s->sel.Allocate(job->start_time, job->end_time, job->allocated_res);  // :5827
    if (job->start_time != now) {                                       // :5829
      if (!rsd) {
        for (const std::string& id : job->craned_ids) {
          auto it = first_resv.find(id);
          if (it != first_resv.end() && it->second < now + job->time_limit) {
            job->reason = CRANE_REASON_RESERVED;
            break;
          }
        }
        if (job->reason != CRANE_REASON_NONE) continue;
        for (const std::string& id : job->craned_ids) {
          const ResInNode& avail = state_by_name.at(id)->res_avail;
          if (!ResLe(job->allocated_res.at(id), avail)) {
            job->reason = CRANE_REASON_RESOURCE;
            break;
          }
        }
      } else {
        for (const std::string& id : job->craned_ids) {
          const ResInNode& avail = rsd->nodes.at(id)->res_avail;
          if (!ResLe(job->allocated_res.at(id), avail)) {
            job->reason = CRANE_REASON_RESOURCE;
            break;
          }
        }
      }
      if (job->reason == CRANE_REASON_NONE) job->reason = CRANE_REASON_PRIORITY;
    }
  }
  // =========================================================================
  auto t1 = std::chrono::steady_clock::now();
  if (elapsed_ms)
    *elapsed_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
  if (jobs_done) *jobs_done = done;

  // --- write-back in the C-ABI layout --------------------------------------
  std::unordered_map<std::string, uint32_t> index_by_name;
  for (uint32_t i = 0; i < M; ++i) index_by_name.emplace(node_names[i], i);
  uint32_t off = 0;
  for (uint32_t i = 0; i < N; ++i) {
    const PdJob* j = pd[i].get();
    out->alloc_off[i] = off;
    out->reason[i] = static_cast<uint8_t>(j->reason);
    out->priority[i] = j->priority;
    bool placed = j->start_time != 0 && j->end_time != 0;
    out->start_time[i] = placed ? j->start_time : 0;
    out->end_time[i] = placed ? j->end_time : 0;
    out->n_alloc[i] = placed ? j->node_num : 0;
    for (uint32_t k = 0; k < j->node_num; ++k) {
      out->alloc_node[off + k] = 0;
      out->alloc_ntasks[off + k] = 0;
      memset(&out->alloc_res[off + k], 0, sizeof(crane_res_in_node_t));
    }
    if (placed) {
      uint32_t k = 0;  // std::map iterates node names == node index ascending
      for (const auto& [id, res] : j->allocated_res) {
        if (k >= j->node_num) break;
        out->alloc_node[off + k] = index_by_name.at(id);
        out->alloc_ntasks[off + k] = j->node_task_num.at(id);
        ToAbi(dict, res, &out->alloc_res[off + k]);
        ++k;
      }
    }
    off += j->node_num;
  }
  out->alloc_off[N] = off;
  return CRANE_OK;
}

extern "C" int crane_oracle_feasible(const crane_cluster_t* cl,
                                     const crane_res_view_t* req,
                                     const crane_res_in_node_t* avail,
                                     crane_res_in_node_t* alloc) {
  Dict d(cl);
  ResView v = ViewFromAbi(d, *req);
  ResInNode a = FromAbi(d, *avail);
  ResInNode got;
  if (!v.Feasible(a, &got)) return 0;
  if (alloc) ToAbi(d, got, alloc);
  return 1;
}

extern "C" void crane_oracle_ckmin(const crane_cluster_t* cl,
                                   crane_res_in_node_t* a,
                                   const crane_res_in_node_t* b) {
  Dict d(cl);
  ResInNode x = FromAbi(d, *a);
  x.Ckmin(FromAbi(d, *b));
  ToAbi(d, x, a);
}

extern "C" int crane_oracle_res_le(const crane_cluster_t* cl,
                                   const crane_res_in_node_t* a,
                                   const crane_res_in_node_t* b) {
  Dict d(cl);
  return ResLe(FromAbi(d, *a), FromAbi(d, *b)) ? 1 : 0;
}

extern "C" int crane_oracle_timeline_update(
    const crane_cluster_t* cl, int64_t* times, crane_res_in_node_t* rows,
    uint32_t* n_seg, uint32_t cap, int64_t start, int64_t end,
    const crane_res_in_node_t* res) {
  Dict d(cl);
  NodeState ns;
  for (uint32_t i = 0; i < *n_seg; ++i)
    ns.timeline.emplace(times[i], FromAbi(d, rows[i]));
  ns.Update(start, end, FromAbi(d, *res));
  if (ns.timeline.size() > cap) return -1;
  uint32_t i = 0;
  for (const auto& [t, r] : ns.timeline) {
    times[i] = t;
    ToAbi(d, r, &rows[i]);
    ++i;
  }
  *n_seg = i;
  return 0;
}

extern "C" int crane_oracle_earliest_start(
    const crane_cluster_t* cl, uint32_t n_nodes, uint32_t node_num,
    const uint32_t* off, const int64_t* times, const crane_res_in_node_t* rows,
    const crane_res_in_node_t* alloc, int64_t now, int64_t time_limit,
    int64_t max_window, int64_t* start) {
  Dict d(cl);
  std::vector<NodeState> states(n_nodes);
  std::vector<NodeState*> ptrs;
  PdJob job{};
  job.node_num = node_num;
  job.time_limit = time_limit;
  for (uint32_t k = 0; k < n_nodes; ++k) {
    states[k].craned_id = NodeName(k);
    states[k].index = k;
    for (uint32_t i = off[k]; i < off[k + 1]; ++i)
      states[k].timeline.emplace(times[i], FromAbi(d, rows[i]));
    job.allocated_res.emplace(states[k].craned_id, FromAbi(d, alloc[k]));
    ptrs.push_back(&states[k]);
  }
  if (!EarliestStart(now, max_window, &job, ptrs)) return 0;
  *start = job.start_time;
  return 1;
}

// ---------------------------------------------------------------------------
// Known-answer tests. Cases 1-14 port
// /root/reference/test/Utilities/dedicated_resource_test.cpp:27-171.
// ---------------------------------------------------------------------------
// ---------------------------------------------------------------------------
// QoS post-filter (R12): Accounting/AccountMetaContainer.cpp
// ---------------------------------------------------------------------------
namespace {

// GresMap (PublicHeader.h:490-508) keyed by dictionary ids. A key exists iff
// its count is non-zero (deviation D8: the reference iterates an unordered_map
// whose zero-count keys and order are unspecified; here names and types are
// walked in dictionary order).
struct QGresCount {
  uint64_t total = 0;
  std::map<uint32_t, uint64_t> specified;
};
using QGresMap = std::map<uint32_t, QGresCount>;
struct QView {
  int64_t cpu_raw = 0;
  uint64_t mem = 0, mem_sw = 0;
  QGresMap gres;
};

QView qview_of_usage(const crane_cluster_t* cl, const crane_meta_resource_t& u) {
  QView v;
  v.cpu_raw = u.cpu_raw; v.mem = u.mem; v.mem_sw = u.mem_sw;
  for (uint32_t e = 0; e < cl->n_gres_entries; ++e) {
    uint32_t g = cl->gres_entry_name[e];
    if (u.gres_total[g]) v.gres[g].total = u.gres_total[g];
    if (u.gres_spec[e]) v.gres[g].specified[e] = u.gres_spec[e];
  }
  return v;
}
QView qview_of_limit(const crane_cluster_t* cl, const crane_tres_limit_t& l) {
  QView v;
  v.cpu_raw = l.view.cpu_raw; v.mem = l.view.mem; v.mem_sw = l.view.mem_sw;
  for (uint32_t e = 0; e < cl->n_gres_entries; ++e) {
    uint32_t g = cl->gres_entry_name[e];
    if (!((l.gres_name_present >> g) & 1)) continue;
    v.gres[g].total = l.view.gres_total[g];
    if ((l.gres_spec_present >> e) & 1) v.gres[g].specified[e] = l.view.gres_spec[e];
  }
  return v;
}
// ResourceV3::View (PublicHeader.cpp:946-952, 399-427)
QView qview_of_alloc(const crane_cluster_t* cl, const crane_res_in_node_t* rows, uint32_t n) {
  QView v;
  for (uint32_t k = 0; k < n; ++k) {
    v.cpu_raw += rows[k].cpu_raw;
    v.mem += rows[k].mem;
    v.mem_sw += rows[k].mem_sw;
    for (uint32_t e = 0; e < cl->n_gres_entries; ++e) {
      uint64_t cnt = (uint64_t)__builtin_popcount(rows[k].gres[e]);
      if (!cnt) continue;
      QGresCount& gc = v.gres[cl->gres_entry_name[e]];
      gc.total += cnt;
      gc.specified[e] += cnt;
    }
  }
  return v;
}
// ResourceView::operator+=(ResourceView) (PublicHeader.cpp:448-456)
void qview_add(QView& a, const QView& b) {
  a.cpu_raw += b.cpu_raw; a.mem += b.mem; a.mem_sw += b.mem_sw;
  for (const auto& [g, gc] : b.gres) {
    QGresCount& d = a.gres[g];
    d.total += gc.total;
    for (const auto& [e, c] : gc.specified) d.specified[e] += c;
  }
}
// AccountMetaContainer::CheckGres_ (AccountMetaContainer.cpp:509-531)
bool q_check_gres(const QGresMap& req, const QGresMap& total) {
  for (const auto& [name, lhs] : req) {
    auto rhs_it = total.find(name);
    if (rhs_it == total.end()) return true;
    const QGresCount& rhs = rhs_it->second;
    if (lhs.total > rhs.total) return false;
    for (const auto& [type, lhs_cnt] : lhs.specified) {
      auto t_it = rhs.specified.find(type);
      if (t_it == rhs.specified.end()) return true;
      if (lhs_cnt > t_it->second) return false;
    }
  }
  return true;
}
// AccountMetaContainer::CheckTres_ (AccountMetaContainer.cpp:493-507)
uint8_t q_check_tres(const QView& req, const QView& total) {
  if (req.cpu_raw > total.cpu_raw) return CRANE_REASON_QOS_CPU;
  if (req.mem > total.mem) return CRANE_REASON_QOS_MEM;
  if (!q_check_gres(req.gres, total.gres)) return CRANE_REASON_QOS_GRES;
  return CRANE_REASON_NONE;
}
// MetaResource::operator+= (AccountMetaContainer.cpp:33-39)
void q_malloc(const crane_cluster_t* cl, crane_meta_resource_t& u, const QView& a, int64_t wall) {
  u.cpu_raw += a.cpu_raw; u.mem += a.mem; u.mem_sw += a.mem_sw;
  for (const auto& [g, gc] : a.gres) {
    u.gres_total[g] += (uint32_t)gc.total;
    for (const auto& [e, c] : gc.specified) u.gres_spec[e] += (uint32_t)c;
  }
  (void)cl;
  u.jobs_count += 1;
  u.wall_time += wall;
}

}  // namespace

extern "C" int crane_oracle_qos_filter(const crane_cluster_t* cl, const crane_pending_t* pd,
                                       crane_placements_t* out, const crane_qos_table_t* qt) {
  if (!cl || !pd || !out || !qt) return CRANE_EINVAL;
  for (uint32_t i = 0; i < pd->n; ++i) {  // commit loop order = job-id order (JS.cpp:1192)
    if (out->reason[i] != CRANE_REASON_NONE || out->n_alloc[i] == 0) continue;
    const uint32_t q = pd->qos[i], user = pd->user[i];
    // CheckAndMallocQosResource (AccountMetaContainer.cpp:164-191)
    if (q >= qt->n_qos || !qt->valid[q]) { out->reason[i] = CRANE_REASON_QOS_INVALID; continue; }
    if (user >= qt->n_users) return CRANE_EINVAL;
    const QView alloc = qview_of_alloc(cl, out->alloc_res + out->alloc_off[i], out->n_alloc[i]);
    const int64_t tl = pd->time_limit[i];
    const int64_t max_wall = qt->max_wall[q];
    uint8_t result = CRANE_REASON_NONE;
    // CheckQosResource_ (AccountMetaContainer.cpp:382-491): user
    {
      crane_meta_resource_t& val = qt->user_usage[(size_t)user * qt->n_qos + q];
      QView use = alloc;
      qview_add(use, qview_of_usage(cl, val));
      if (use.cpu_raw > qt->max_cpus_per_user_raw[q]) result = CRANE_REASON_QOS_CPU;
      else if ((uint64_t)val.jobs_count + 1 > qt->max_jobs_per_user[q]) result = CRANE_REASON_QOS_JOBS;
      else if (max_wall > 0 && val.wall_time + tl > max_wall) result = CRANE_REASON_QOS_WALL;
      else result = q_check_tres(use, qview_of_limit(cl, qt->max_tres_per_user[q]));
    }
    // account chain
    if (result == CRANE_REASON_NONE) {
      for (uint32_t c = qt->chain_off[i]; c < qt->chain_off[i + 1]; ++c) {
        uint32_t a = qt->chain_acct[c];
        if (a >= qt->n_accounts) return CRANE_EINVAL;
        crane_meta_resource_t& val = qt->account_usage[(size_t)a * qt->n_qos + q];
        QView use = alloc;
        qview_add(use, qview_of_usage(cl, val));
        if ((uint64_t)val.jobs_count + 1 > qt->max_jobs_per_account[q]) result = CRANE_REASON_QOS_JOBS;
        else if (max_wall > 0 && val.wall_time + tl > max_wall) result = CRANE_REASON_QOS_WALL;
        else result = q_check_tres(use, qview_of_limit(cl, qt->max_tres_per_account[q]));
        if (result != CRANE_REASON_NONE) break;
      }
    }
    // qos
    if (result == CRANE_REASON_NONE) {
      crane_meta_resource_t& val = qt->qos_usage[q];
      QView use = alloc;
      qview_add(use, qview_of_usage(cl, val));
      if ((uint64_t)val.jobs_count + 1 > qt->max_jobs[q]) result = CRANE_REASON_QOS_JOBS;
      else if (max_wall > 0 && val.wall_time + tl > max_wall) result = CRANE_REASON_QOS_WALL;
      else result = q_check_tres(use, qview_of_limit(cl, qt->max_tres[q]));
    }
    if (result != CRANE_REASON_NONE) { out->reason[i] = result; continue; }
    // DoMallocResource_ (AccountMetaContainer.cpp:546-587)
    q_malloc(cl, qt->user_usage[(size_t)user * qt->n_qos + q], alloc, tl);
    for (uint32_t c = qt->chain_off[i]; c < qt->chain_off[i + 1]; ++c)
      q_malloc(cl, qt->account_usage[(size_t)qt->chain_acct[c] * qt->n_qos + q], alloc, tl);
    q_malloc(cl, qt->qos_usage[q], alloc, tl);
  }
  return CRANE_OK;
}

extern "C" int crane_oracle_selftest(char* log, size_t log_cap) {
  int failed = 0;
  size_t used = 0;
  auto fail = [&](const char* name) {
    ++failed;
    if (log && used < log_cap)
      used += snprintf(log + used, log_cap - used, "FAIL %s\n", name);
  };
  const char* s[8] = {"/dev/nvidia0", "/dev/nvidia1", "/dev/nvidia2",
                      "/dev/nvidia3", "/dev/nvidia4", "/dev/nvidia5",
                      "/dev/nvidia6", "/dev/nvidia7"};
  auto mk = [&](std::initializer_list<int> idx) {
    std::set<SlotId> r;
    for (int i : idx) r.insert(s[i]);
    return r;
  };
  {  // le_gt :27
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1, 3, 2});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    if (DedicatedLe(a, b)) fail("le_gt");
  }
  for (int rep = 0; rep < 2; ++rep) {  // le_lt1 :37, le_lt2 :45
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    if (!DedicatedLe(a, b)) fail(rep ? "le_lt2" : "le_lt1");
  }
  {  // le_lt3 :53
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["GPU"].by_type["A200"] = mk({0, 1, 3});
    if (!DedicatedLe(a, b)) fail("le_lt3");
  }
  {  // le_nle :63
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 2});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    if (DedicatedLe(a, b)) fail("le_nle");
  }
  {  // le_equ :72
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1});
    b["GPU"].by_type["A100"] = mk({0, 1});
    if (!DedicatedLe(a, b)) fail("le_equ");
  }
  {  // le_equ2 :80
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1});
    a["XPU"].by_type["A100"] = mk({0, 1});
    b["GPU"].by_type["A100"] = mk({0, 1});
    b["XPU"].by_type["A100"] = mk({0, 1});
    if (!DedicatedLe(a, b)) fail("le_equ2");
  }
  {  // equ_equ :90
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1});
    b["GPU"].by_type["A100"] = mk({0, 1});
    if (!DedicatedEq(a, b)) fail("equ_equ");
  }
  {  // equ_lt :98
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0});
    a["XPU"].by_type["X100"];
    b["GPU"].by_type["A100"] = mk({0, 1});
    b["TPU"].by_type["T100"];
    if (DedicatedEq(a, b)) fail("equ_lt");
  }
  {  // equ_gt :109
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1, 3});
    a["XPU"].by_type["X100"];
    b["GPU"].by_type["A100"] = mk({0, 1});
    b["TPU"].by_type["T100"];
    if (DedicatedEq(a, b)) fail("equ_gt");
  }
  {  // plus1 :120
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1, 3});
    b.Add(a);
    if (!DedicatedEq(a, b)) fail("plus1");
  }
  {  // plus2 :128
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["XPU"].by_type["X100"] = mk({1, 6, 5});
    DedicatedRes t = b;
    t.Add(a);
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    if (!DedicatedEq(t, b)) fail("plus2");
  }
  {  // plus3 :139
    DedicatedRes a, b;
    a["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["XPU"].by_type["X100"] = mk({1, 6, 5});
    DedicatedRes t = b;
    t.Add(a);
    if (!DedicatedEq(t, b)) fail("plus3");
  }
  {  // minus1 :150
    DedicatedRes a, b, r;
    a["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["GPU"].by_type["A100"] = mk({0, 1, 3});
    b["XPU"].by_type["X100"] = mk({1, 6, 5});
    b.Sub(a);
    r["XPU"].by_type["X100"] = mk({1, 6, 5});
    if (!DedicatedEq(r, b)) fail("minus1");
  }
  {  // minus2 :162
    DedicatedRes a, b, r;
    a["GPU"].by_type["A100"] = mk({0});
    b["GPU"].by_type["A100"] = mk({0});
    b.Sub(a);
    if (!DedicatedEq(r, b)) fail("minus2");
  }

  // ---- hand-derived micro-cases (SURVEY.md §8c) ---------------------------
  {  // integer-cpu core rule, PublicHeader.cpp:528-538
    ResInNode avail;
    avail.cpu_count = CpuT::FromInt(4);
    avail.core_ids = {1, 3, 5, 7};
    avail.mem = 100;
    ResView v;
    v.cpu = CpuT::FromInt(2);
    v.mem = 10;
    ResInNode got;
    if (!v.Feasible(avail, &got) || got.core_ids != std::set<uint32_t>{1, 3})
      fail("int_cpu_lowest_cores");
    avail.core_ids = {5};  // count suffices, cores do not
    if (v.Feasible(avail, &got)) fail("int_cpu_core_shortage");
    v.cpu = CpuT::FromRaw(384);  // 1.5 cpus: fractional -> no cores bound
    if (!v.Feasible(avail, &got) || !got.core_ids.empty() || got.cpu_count.raw != 384)
      fail("frac_cpu_no_cores");
  }
  {  // untyped gres spill order, PublicHeader.cpp:555-594
    ResInNode avail;
    avail.cpu_count = CpuT::FromInt(1);
    avail.gres["gpu"].by_type["a100"] = mk({0, 1, 2});
    avail.gres["gpu"].by_type["h100"] = mk({4, 5});
    ResView v;
    GresCount gc;
    gc.total = 4;
    gc.specified["a100"] = 1;
    v.gres["gpu"] = gc;  // 1 typed a100 + 3 untyped
    ResInNode got;
    bool ok = v.Feasible(avail, &got);
    if (!ok || got.gres.by_name["gpu"].by_type["a100"] != mk({0, 1, 2}) ||
        got.gres.by_name["gpu"].by_type["h100"] != mk({4}))
      fail("untyped_spill");
    gc.total = 6;
    v.gres["gpu"] = gc;
    if (v.Feasible(avail, &got)) fail("untyped_overflow");
  }
  {  // Ckmin core rule, PublicHeader.cpp:815-827
    ResInNode a, b;
    a.core_ids = {0, 1, 2};
    a.cpu_count = CpuT::FromInt(3);
    b.cpu_count = CpuT::FromInt(5);  // b has no core ids -> a's cores kept
    a.Ckmin(b);
    if (a.core_ids != std::set<uint32_t>{0, 1, 2} || a.cpu_count.raw != 768)
      fail("ckmin_empty_rhs_cores");
    b.core_ids = {2, 3};
    a.Ckmin(b);
    if (a.core_ids != std::set<uint32_t>{2}) fail("ckmin_intersect");
  }
  {  // the 4 timeline-update diagrams, JobScheduler.h:343-412 (cases 3/4 are
     // the reachable ones with a +inf sentinel)
    ResInNode full, one;
    full.cpu_count = CpuT::FromInt(8);
    full.mem = 80;
    one.cpu_count = CpuT::FromInt(2);
    one.mem = 10;
    NodeState ns;
    ns.timeline.emplace(100, full);
    ns.timeline[kInfFuture].SetToZero();
    ns.Update(100, 200, one);  // case 4 at the left edge, insert at 200
    bool ok = ns.timeline.size() == 3 && ns.timeline.at(100).cpu_count.raw == 6 * 256 &&
              ns.timeline.at(200).cpu_count.raw == 8 * 256;
    ns.Update(150, 250, one);  // case 3: inserts 150 and 250
    ok = ok && ns.timeline.size() == 5 &&
         ns.timeline.at(100).cpu_count.raw == 6 * 256 &&
         ns.timeline.at(150).cpu_count.raw == 4 * 256 &&
         ns.timeline.at(200).cpu_count.raw == 6 * 256 &&
         ns.timeline.at(250).cpu_count.raw == 8 * 256 &&
         ns.timeline.at(kInfFuture).cpu_count.raw == 0;
    ns.Update(150, 200, one);  // exact segment, no insert
    ok = ok && ns.timeline.size() == 5 && ns.timeline.at(150).cpu_count.raw == 2 * 256 &&
         ns.timeline.at(200).cpu_count.raw == 6 * 256;
    if (!ok) fail("timeline_update");
  }
  return failed;
}
