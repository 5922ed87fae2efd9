"""Pins the oracle (oracle/crane_oracle.cpp, our restatement) to the REFERENCE'S OWN
CODE: oracle/_ref/libcrane_ref.so is compiled from the unmodified text of
JobScheduler.{h,cpp} / PublicHeader.{h,cpp} (oracle/ref_build.py + oracle/ref_shim/).
Its answers on every case here are stored under tests/golden/ (ref_pin.json: one
SHA-256 digest per output column; ref_algebra.npz), written by
tests/golden/make_ref_golden.py, so the pin holds on any checkout.

What the pin covers: priority (fp64 bits), reasons, start/end times, node sets,
task counts, concrete cores and gres slots of every job, on feature-mix cases
(running jobs, backfill, exclusive, include/exclude lists, fractional cpus,
typed + untyped gres, dead/drained nodes, unknown partitions, mandated
priorities, batch limit) and on the BASELINE configs at small size.

What it cannot cover (run-to-run nondeterminism of the reference itself, fixed by
a documented rule in the oracle and the CUDA path, SURVEY.md §8c):
  * a node holding several types of ONE gres name together with a request that has
    an untyped remainder: which type serves it follows std::unordered_map hash
    order in the reference (PublicHeader.cpp:564,583) — generator option
    one_type_per_name=True keeps such nodes out;
  * equal computed priorities (std::ranges::sort is unstable, JobScheduler.cpp:6541)
    — a draw with ties is skipped only if the results differ (none does today).
"""
import ctypes as C

import numpy as np
import pytest

from cranesched_b200 import abi, synth
from tests.golden import make_ref_golden as G
from tests.golden.make_full_golden import COLUMNS, digest_of

REF = G.load()


def _same(oracle, group, name, ties_may_differ=False):
    """The oracle's NodeSelect of a stored case against the reference's, column by column."""
    cfg, cl, rn, pd, now, resv = G.NODE_SELECT[group][name]()
    a, _, _ = oracle.node_select(cfg, cl, rn, pd, now, resv=resv)
    have, want = digest_of(a), REF[group][name]
    bad = [c for c in COLUMNS if have[c] != want[c]]
    if bad and ties_may_differ and cfg.priority_type != 0 and len(np.unique(a.priority)) != pd.n:
        pytest.skip("equal priorities in this draw and the unstable sort ordered them differently: outside the pin")
    assert not bad, "oracle differs from the reference's own NodeSelect in %s (reason counts %s, reference %s)" % (
        bad, have["reason_hist"], want["reason_hist"])
    return a


@pytest.mark.parametrize("seed", range(24))
def test_feature_mix_matches_reference(oracle, seed):
    out = _same(oracle, "feature_mix", "s%d" % seed, ties_may_differ=True)
    if seed == 1:
        assert (out.n_alloc == 0).sum() >= 70  # 250 jobs, batch limit 180


def test_config1_full_matches_reference(oracle):
    _same(oracle, "configs", "config1", ties_may_differ=True)


@pytest.mark.parametrize("seed_id,n_jobs", [(2, 3500), (3002, 3000)])
def test_config2_small_matches_reference(oracle, seed_id, n_jobs):
    out = _same(oracle, "configs", "config2_s%d" % seed_id, ties_may_differ=True)
    assert out.reason.shape == (n_jobs,)
    assert (out.reason == abi.REASON_NONE).any() and ((out.reason != 0) & (out.n_alloc > 0)).any()


def test_config3_and_5_small_match_reference(oracle):
    _same(oracle, "configs", "config3", ties_may_differ=True)
    _same(oracle, "configs", "config5", ties_may_differ=True)


def test_general_task_distribution_matches_reference(oracle):
    """ntasks_per_node_max > min and ntasks != node_num * ntpn (JobScheduler.cpp:5193-5222,
    5269-5278, 5340-5361): the top-K heaps behave the same (both are libstdc++'s)."""
    for seed in range(8):
        _same(oracle, "general_task", "s%d" % seed, ties_may_differ=True)


def test_resource_algebra_matches_reference(oracle):
    """GetFeasibleResourceInNode / Ckmin / operator<= of the reference itself on random rows
    (single type per name, see module docstring)."""
    cl = G.algebra_cluster()
    with np.load(G.ALGEBRA) as z:
        ref = {k: z[k] for k in z.files}
    for i, (req, avail, other) in enumerate(G.algebra_inputs()):
        ok_o, al_o = oracle.feasible(cl, req, avail)
        assert ok_o == bool(ref["ok"][i]), i
        if ok_o:
            assert al_o.tobytes() == ref["alloc"][i].tobytes(), i
        assert oracle.ckmin(cl, avail, other).tobytes() == ref["ckmin"][i].tobytes(), i
        assert oracle.res_le(cl, avail, other) == bool(ref["res_le"][i]), i


def test_earliest_start_known_answers(oracle):
    """EarliestStartSubsetSelector (JobScheduler.h:786-859) on hand-made timelines: the
    answers the reference's own selector gives, which the oracle and the CUDA path's
    per-node fixed point must reproduce."""
    cl = synth.make_cluster([(2, synth.node_row(4, 16))])
    inf = np.iinfo(np.int64).max
    window = abi.Config().max_time_window_s  # kAlgoMaxTimeWindow, 7 days

    def row(cpus):
        r = np.zeros((), abi.RES_IN_NODE)
        r["cpu_raw"] = cpus * 256
        r["mem"] = 16
        return r

    def ask(timelines, K, limit, now=1000):
        times, rows, off = [], [], [0]
        for tl in timelines:
            for t, c in tl:
                times.append(t)
                rows.append(row(c))
            off.append(len(times))
        times = np.array(times, np.int64)
        rows = np.array(rows, abi.RES_IN_NODE)
        off = np.array(off, np.uint32)
        alloc = np.array([row(2)] * len(timelines), abi.RES_IN_NODE)
        st = C.c_int64(0)
        c = cl.as_c()
        rc = oracle.lib().crane_oracle_earliest_start(
            C.byref(c), len(timelines), K, C.c_void_p(off.ctypes.data), C.c_void_p(times.ctypes.data),
            C.c_void_p(rows.ctypes.data), C.c_void_p(alloc.ctypes.data), now, limit, window, C.byref(st))
        return st.value if rc else None

    a = [(1000, 0), (1100, 4), (1500, 1), (1600, 4), (inf, 0)]
    b = [(1000, 0), (1300, 4), (inf, 0)]
    assert ask([a], 1, 50) == 1100
    assert ask([a], 1, 400) == 1100
    assert ask([a], 1, 401) == 1600      # the hole at 1500 is too close
    assert ask([a, b], 2, 100) == 1300   # both free from 1300, a is taken again at 1500
    assert ask([a, b], 2, 201) == 1600
    assert ask([a, b], 2, 10**9) == 1600  # last segment before the sentinel: no end in sight, accepted
    assert ask([[(1000, 0), (inf, 0)]], 1, 10) is None
    assert ask([[(1000, 0), (1000 + 8 * 86400, 4), (inf, 0)]], 1, 10) is None  # beyond the 7-day window


@pytest.mark.parametrize("seed", range(400, 416))
def test_reservations(oracle, seed):
    """Reservations (JobScheduler.cpp:5655-5753, 5788-5795, 5829-5861): expired, started
    and later ones; jobs submitted into them (also into unknown ones: "Reservation Not
    Found"), running jobs inside them, "Resource Reserved" for backfills that run into
    a reservation. One node per reservation: inside a reservation the reference orders
    equal-cost nodes by the addresses of node states created in unordered_map order."""
    a = _same(oracle, "reservations", "s%d" % seed)
    assert (a.reason == abi.REASON_RESERVED).any() or (a.reason == 5).any() or seed % 4


@pytest.mark.parametrize("seed", range(700, 712))
def test_overlapping_partitions(oracle, seed):
    """Partitions that share nodes: one NodeState per node, referenced by every
    LocalScheduler whose partition lists it (JobScheduler.cpp:5597-5651), so a placement
    in one partition changes what the others can start on the node (their own costs stay)."""
    _same(oracle, "overlapping", "s%d" % seed)


@pytest.mark.parametrize("seed", range(720, 728))
def test_overlapping_partitions_with_reservations(oracle, seed):
    """Both at once: reservations cut out of nodes that two partitions share."""
    _same(oracle, "overlapping_resv", "s%d" % seed)


@pytest.mark.parametrize("seed,tight,invalid", G.QOS_PARAMS)
def test_qos_filter_matches_reference(oracle, seed, tight, invalid):
    """R12: the oracle's QoS pass against the reference's own CheckAndMallocQosResource / CheckQosResource_ /
    CheckTres_ / CheckGres_ / DoMallocResource_ (Accounting/AccountMetaContainer.cpp:164-191, 382-587),
    compiled from its text: reasons of every job and the three usage tables, byte for byte. (CheckGres_ walks
    an unordered_map and stops at the first name the limit does not list; the oracle walks names in dictionary
    order, deviation D8 — the two can only differ for a job holding two gres names of which the limit lists
    one, which these draws do not produce.)"""
    cl, pd, out, table = G.qos_case(seed, tight, invalid)
    oracle.qos_filter(cl, pd, out, table)
    have, want = G.qos_digest(out.reason, table), REF["qos"]["s%d" % seed]
    for f in G.QOS_COLUMNS:
        assert have[f] == want[f], "%s (reason counts %s, reference %s)" % (f, have["reason_hist"], want["reason_hist"])
    assert (out.reason >= 16).any() or tight >= 8.0
