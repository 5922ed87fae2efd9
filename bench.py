#!/usr/bin/env python
"""bench.py — placement decisions / second of the NodeSelect hot path.

A "step" is one full scheduling tick (SchedulerAlgo::NodeSelect,
JobScheduler.cpp:5543-5868) over one synthetic pending queue: BASELINE.json
configs[1], 100k pending jobs x 10k nodes, cpu+mem+gres(GPU), 4 partitions,
multifactor priority + backfill.

  N = 1   value = decisions/s with the tables resident in HBM when the timed
          region starts (device time of crane_sched_run, CUDA events on the
          launching stream); e2e = the same metric through
          crane_sched_node_select with HOST buffers (H2D of the pending table
          + D2H of the placements inside the region).
  N > 1   ONE queue — the same 100k x 10k queue — over N GPUs (strong scaling):
          partitions are dealt to the ranks (cranesched_b200/sharding.py), every
          rank commits its own partitions and the placement columns are
          all-reduced over NCCL; the gathered result is compared with the
          unsplit single-GPU answer inside the bench ("sharded_equals_unsplit").
          The job loop of a partition is a dependency chain that one GPU already
          runs concurrently with the other partitions, so more GPUs shorten the
          tick only as far as the largest partition allows — the line reports
          that honestly. "weak" in the same line: N independent clusters, one
          per rank, each its own draw (seed 1000*rank + 2).
  --impl reference   the reference's CPU NodeSelect on a bounded sample of the
          same queue: oracle/_ref (the reference's own source compiled against
          shim headers, kind "reference") when it was built, else the oracle
          port (kind "port"); single thread, as the reference is.
  --dump-outputs DIR   after the timed steps, the placements of the last one
          as DIR/<name>.npy (float32/float64, at most 64 MB; see dump_outputs),
          so two builds can be compared output for output on the same queue.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "placement decisions/sec (jobs through the NodeSelect job loop)"
UNIT = "decisions/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.samples, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in o.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of k_commit from the committed
    `ncu --set full` capture (profiles/r02_ncu_k_commit2_summary.csv: captured on the shipped build), per launch."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_k_commit2_summary.csv")
    if not os.path.exists(p):
        return None
    tot = 0.0
    for line in open(p):
        f = line.strip().split(",")
        if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(f[2], 1.0)
            tot += float(f[1]) * mult
    return tot or None


def algorithmic_bytes(cluster, pending, n_decided):
    """SURVEY.md §8d: B_dec(j) = job_row + M_part(j) * node_row + out_row(j),
    job_row 64 B, node_row 48 B (24 B when the cluster has no gres), out_row
    16 B + 32 B * node_num."""
    part_size = np.diff(cluster.part_off.astype(np.int64))
    node_row = 48 if cluster.n_gres_entries else 24
    p = pending.partition
    ok = p < cluster.n_partitions
    mp = np.where(ok, part_size[np.minimum(p, cluster.n_partitions - 1)], 0)
    b = 64 + mp * node_row + 16 + 32 * pending.node_num.astype(np.int64)
    return int(b.sum()), node_row


def workload(args, rank=0):
    """The bench queue. rank > 0: that rank's own draw of the same shape (weak line)."""
    from cranesched_b200 import sharding
    if args.config not in (1, 2, 5):
        raise SystemExit("bench.py --config must be 1, 2 or 5")
    return sharding.shard_workload(args.config, rank, 1, args.jobs, args.nodes)


def cpu_reference(cfg, cl, rn, pd, now, sample):
    """The reference's CPU NodeSelect on the first `sample` jobs of the priority
    order (ScheduledBatchSize = sample: the rest of the queue only gets its
    priority computed and the reason "Priority"). Returns (ms, jobs, kind)."""
    import copy
    from oracle import pyoracle, pyref
    if pyref.available():
        c2 = copy.copy(cfg)
        c2.scheduled_batch_size = min(sample, pd.n)
        _, ms = pyref.node_select(c2, cl, rn, pd, now)
        return ms, int(min(sample, pd.n)), "reference"
    pyoracle.build()
    _, ms, done = pyoracle.node_select(cfg, cl, rn, pd, now, max_jobs=sample)
    return ms, done, "port"


def workload_name(args):
    return {1: "config1: 1k jobs x 128 nodes, cpu+mem, FIFO",
            2: "config2: %dk pending jobs x %dk nodes, cpu+mem+gres(GPU), 4 partitions, multifactor priority + backfill"
               % ((args.jobs or 100_000) // 1000, (args.nodes or 10_000) // 1000),
            5: "config5: backfill stress, %dk jobs x %dk nodes, 1 partition"
               % ((args.jobs or 200_000) // 1000, (args.nodes or 5_000) // 1000)}[args.config]


def run_reference(args, rank, world):
    """CPU arm: the reference's NodeSelect, single thread as upstream ("TODO: do it
    in parallel", JobScheduler.cpp:5756,5776), on a bounded sample of the queue."""
    if rank != 0:
        return
    cfg, cl, rn, pd, now = workload(args, 0)
    times, done, kind = [], 0, "port"
    for i in range(args.warmup + args.steps):
        ms, done, kind = cpu_reference(cfg, cl, rn, pd, now, args.ref_sample)
        if i >= args.warmup:
            times.append(ms)
    ms = float(np.mean(times))
    v = done / (ms / 1e3)
    what = ("oracle/_ref: the reference's own JobScheduler/PublicHeader source compiled against shim headers"
            if kind == "reference" else "oracle/: CPU restatement of NodeSelect")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "int64+u64 masks, f64 cost/priority",
            "data": "synthetic", "config": {"workload": workload_name(args)},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": kind,
                             "sample": "%s, 1 thread, first %d jobs of the priority order of the same queue (cost per job "
                                       "grows as the cluster fills, so this flatters the CPU)" % (what, done)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


DUMP_BYTES = 64 << 20


def snapshot(out):
    """Host copy of a Placements (the pinned buffers are reused by later ticks)."""
    from cranesched_b200 import abi
    return abi.Placements(**{f: np.array(getattr(out, f), copy=True) for f in abi.Placements.__dataclass_fields__})


def dump_outputs(out, node_num, directory):
    """Writes the placements of one tick as DIR/<name>.npy so that two builds can be
    compared output for output. Per job: reason, priority, start_time, end_time,
    n_alloc; per allocated node, in job order: alloc_node, alloc_ntasks and the
    allocated resources (alloc_cpu_raw, alloc_mem, alloc_mem_sw; the core bit masks
    as alloc_core_lo / alloc_core_hi, 32 bits each; the gres slot masks as
    alloc_gres). job_index names the jobs written and alloc_off their rows. Counts,
    times and 32-bit halves are float64, the 16-bit gres masks float32: exact
    below 2**53. When the queue could exceed DUMP_BYTES, the jobs written are a
    fixed sample drawn from the requested node counts alone (seed 0), so every
    build writes the same jobs."""
    n = out.reason.shape[0]
    per_row = (5 + 2 * out.alloc_res["core"].shape[1]) * 8 + out.alloc_res["gres"].shape[1] * 4
    bound = 7 * 8 + per_row * node_num.astype(np.int64)  # bytes a job can take at most
    room = DUMP_BYTES - 4096  # npy headers
    if int(bound.sum()) <= room:
        jobs = np.arange(n)
    else:
        perm = np.random.default_rng(0).permutation(n)
        jobs = np.sort(perm[:int(np.searchsorted(np.cumsum(bound[perm]), room, side="right"))])
    cnt = out.n_alloc.astype(np.int64)[jobs]
    first = out.alloc_off[:-1].astype(np.int64)[jobs]
    rows = np.repeat(first - (np.cumsum(cnt) - cnt), cnt) + np.arange(int(cnt.sum()))
    res = out.alloc_res[rows]
    core = res["core"]
    arrays = {
        "job_index": jobs.astype(np.float64),
        "reason": out.reason[jobs].astype(np.float64),
        "priority": out.priority[jobs].astype(np.float64),
        "start_time": out.start_time[jobs].astype(np.float64),
        "end_time": out.end_time[jobs].astype(np.float64),
        "n_alloc": cnt.astype(np.float64),
        "alloc_off": np.concatenate([[0], np.cumsum(cnt)]).astype(np.float64),
        "alloc_node": out.alloc_node[rows].astype(np.float64),
        "alloc_ntasks": out.alloc_ntasks[rows].astype(np.float64),
        "alloc_cpu_raw": res["cpu_raw"].astype(np.float64),
        "alloc_mem": res["mem"].astype(np.float64),
        "alloc_mem_sw": res["mem_sw"].astype(np.float64),
        "alloc_core_lo": (core & np.uint64(0xFFFFFFFF)).astype(np.float64),
        "alloc_core_hi": (core >> np.uint64(32)).astype(np.float64),
        "alloc_gres": res["gres"].astype(np.float32),
    }
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def digest(out):
    import hashlib
    h = hashlib.sha256()
    for f in ("reason", "priority", "start_time", "end_time", "n_alloc", "alloc_node", "alloc_ntasks", "alloc_res"):
        h.update(np.ascontiguousarray(getattr(out, f)).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--jobs", type=int, default=0)
    ap.add_argument("--nodes", type=int, default=0)
    ap.add_argument("--ref-sample", type=int, default=1500, help="jobs per step of the CPU arm")
    ap.add_argument("--cpu-sample", type=int, default=1500, help="jobs of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the placements of the last one as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from cranesched_b200 import abi, sharding
    from cranesched_b200.scheduler import GpuScheduler

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def one_gpu_line(case):
        """K ticks of one whole queue on this rank's GPU: (device ms total, e2e ms total,
        wall ms, timing of the last tick, placements, clocks)."""
        cfg, cl, rn, pd, now = case
        sched = GpuScheduler(cfg, local_rank)
        sched.set_cluster(cl)
        out = abi.Placements.for_pending(pd, pinned=True)
        sched.upload(rn, pd)
        sched.sync()
        dev_ms = []

        def step(record):
            flush.fill_(1)  # L2 flush between timed iterations
            torch.cuda.synchronize()
            sched.run(now)
            ms = sched.sync()
            if record:
                dev_ms.append(ms)

        for _ in range(args.warmup):
            step(False)
        barrier()
        with ClockSampler(local_rank) as clocks:
            t0 = time.perf_counter()
            for _ in range(args.steps):
                step(True)
            barrier()
            wall = time.perf_counter() - t0
        timing_last = sched.timing()
        sched.fetch(out)
        timed_out = snapshot(out)
        # e2e: host buffers through crane_sched_node_select
        e2e_ms = []
        for i in range(2 + args.steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            sched.node_select(now, rn, pd, out)
            dt = (time.perf_counter() - t1) * 1e3
            if i >= 2:
                e2e_ms.append(dt)
        barrier()
        sched.close()
        return float(np.sum(dev_ms)), float(np.sum(e2e_ms)), wall * 1e3, timing_last, timed_out, clocks.summary()

    case0 = workload(args, 0)
    cfg, cl, rn, pd, now = case0
    n_decided = int(min(pd.n, cfg.scheduled_batch_size))
    h2d = sum(getattr(pd, f).nbytes for f in pd.__dataclass_fields__ if getattr(pd, f) is not None)
    line = {"metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "vs_baseline": None,
            "dtype": "int64 cpu / u64 mem + bit masks; f64 cost and priority", "data": "synthetic"}

    if world == 1:
        dev_total_ms, e2e_total_ms, wall_ms, timing_last, out, clk = one_gpu_line(case0)
        value = n_decided * args.steps / (dev_total_ms / 1e3)
        e2e_value = n_decided * args.steps / (e2e_total_ms / 1e3)
        line.update({"value": value, "ms_per_step": dev_total_ms / args.steps, "scaling": "weak",
                     "config": {"workload": workload_name(args), "jobs": pd.n, "nodes": cl.n_nodes,
                                "partitions": cl.n_partitions, "l2": "256 MiB flush write between timed iterations",
                                "started_now": int((out.reason == 0).sum()),
                                "backfill_reserved": int(((out.reason != 0) & (out.n_alloc > 0)).sum())},
                     "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                             "d2h_bytes_per_step": int(out.nbytes()), "ms_per_step": e2e_total_ms / args.steps},
                     "gpu_launches": int(timing_last["kernel_launches"]) * args.steps,
                     "wall_ms_per_step_incl_flush": wall_ms / args.steps, "clocks": clk})
    else:
        # ---- ONE queue over `world` GPUs: partitions dealt to the ranks ------------
        owner = sharding.deal_partitions(pd, cl.n_partitions, world, cl)
        sched = GpuScheduler(cfg, local_rank)
        sched.set_cluster(cl)
        out = abi.Placements.for_pending(pd, pinned=True)
        sched.upload(rn, pd)
        sched.sync()
        step_ms, e2e_ms = [], []
        for i in range(args.warmup + args.steps):
            flush.fill_(1)
            barrier()
            t1 = time.perf_counter()
            sharding.sharded_tick(sched, now, rn, pd, owner, dist, out=out, upload=False)  # run + all-reduce + fetch
            torch.cuda.synchronize()
            if i >= args.warmup:
                step_ms.append((time.perf_counter() - t1) * 1e3)
        timed_out = snapshot(out)
        own_commit_ms = float(sched.timing()["commit_ms"])
        launches = int(sched.timing()["kernel_launches"])
        barrier()
        with ClockSampler(local_rank) as clocks:
            for i in range(2 + args.steps):
                flush.fill_(1)
                barrier()
                t1 = time.perf_counter()
                sharding.sharded_tick(sched, now, rn, pd, owner, dist, out=out, upload=True)  # + H2D of the whole table
                torch.cuda.synchronize()
                if i >= 2:
                    e2e_ms.append((time.perf_counter() - t1) * 1e3)
            barrier()
        sched.close()
        got = digest(out)
        # the unsplit answer, on rank 0's GPU, outside the timed region
        same = True
        if rank == 0:
            s1 = GpuScheduler(cfg, local_rank)
            s1.set_cluster(cl)
            ref_out = s1.node_select(now, rn, pd)
            s1.close()
            same = digest(ref_out) == got
        tot_ms, e2e_total_ms, commit_max = reduce_max([float(np.sum(step_ms)), float(np.sum(e2e_ms)), own_commit_ms])
        value = n_decided * args.steps / (tot_ms / 1e3)
        jobs_per_rank = np.bincount(owner[pd.partition[pd.partition < cl.n_partitions]], minlength=world).tolist()
        # ---- weak line: `world` independent clusters, one per rank, each its own draw --
        wcase = workload(args, rank)
        w_dev, w_e2e, _, w_timing, w_out, _ = one_gpu_line(wcase)
        w_dev, w_e2e = reduce_max([w_dev, w_e2e])
        w_dec = int(min(wcase[3].n, wcase[0].scheduled_batch_size)) * world
        timing_last = w_timing
        d2h = out.nbytes()
        line.update({"value": value, "ms_per_step": tot_ms / args.steps, "scaling": "strong",
                     "config": {"workload": workload_name(args) + " — ONE queue split over %d GPUs by partition" % world,
                                "jobs": pd.n, "nodes": cl.n_nodes, "partitions": cl.n_partitions,
                                "partition_owner": owner.tolist(), "jobs_per_rank": jobs_per_rank,
                                "timed": "run of the own partitions + NCCL all-reduce(sum) of the 7 placement columns "
                                         "+ D2H on every rank; wall clock between barriers, max over ranks",
                                "collective_bytes_per_step": int(d2h - out.priority.nbytes - out.alloc_off.nbytes),
                                "l2": "256 MiB flush write between timed iterations"},
                     "sharded_equals_unsplit": bool(same),
                     "slowest_rank_commit_ms": commit_max,
                     "e2e": {"value": n_decided * args.steps / (e2e_total_ms / 1e3), "unit": UNIT,
                             "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                             "ms_per_step": e2e_total_ms / args.steps},
                     "gpu_launches": launches * args.steps,
                     "weak": {"value": w_dec * args.steps / (w_dev / 1e3), "unit": UNIT, "scaling": "weak",
                              "workload": "%d independent clusters of the config's shape, one per GPU, each its own draw "
                                          "(seed 1000*rank + config)" % world,
                              "e2e_value": w_dec * args.steps / (w_e2e / 1e3), "ms_per_step": w_dev / args.steps},
                     "clocks": clocks.summary()})
        out = w_out if False else out

    if rank == 0:
        peak, peak_src = load_peaks()
        alg_bytes, node_row = algorithmic_bytes(cl, pd, n_decided)
        if world == 1:
            commit_ms = timing_last["commit_ms"]
            line["phases_ms"] = {k: round(float(v), 4) for k, v in timing_last.items() if k.endswith("_ms")}
        else:
            commit_ms = line["slowest_rank_commit_ms"]
        achieved = alg_bytes / (commit_ms / 1e3) / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": "k_commit2", "achieved": achieved, "peak": peak, "unit": "GB/s",
                            "frac": achieved / peak,
                            "traffic": measured_traffic() if args.config == 2 and not args.jobs and world == 1 else None,
                            "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                            "kernel_ms": commit_ms,
                            "note": "per decision 64 B job row + M_part x %d B node row + 16 B + 32 B x node_num "
                                    "(SURVEY.md 8d); the job loop is a dependency chain, so the binding limit is "
                                    "per-batch latency, not DRAM" % node_row}
        if not args.no_cpu_baseline and world == 1:
            ms, done, kind = cpu_reference(cfg, cl, rn, pd, now, args.cpu_sample)
            line["cpu_baseline"] = {
                "value": done / (ms / 1e3), "unit": UNIT, "cores": 1, "kind": kind,
                "sample": "%s, 1 thread like the reference, on the first %d jobs of the priority order of the same queue, %.1f s"
                          % ("oracle/_ref (the reference's own NodeSelect source compiled against shim headers)"
                             if kind == "reference" else "oracle (CPU restatement of NodeSelect)", done, ms / 1e3)}
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(out if world == 1 else timed_out, pd.node_num, args.dump_outputs)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
