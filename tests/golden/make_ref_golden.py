"""The reference's own answers for tests/test_ref_pin.py, stored as golden data.

    python -m tests.golden.make_ref_golden      (from the repo root; needs oracle/_ref, oracle/ref_build.py)

oracle/_ref/libcrane_ref.so is the reference's NodeSelect and QoS check compiled
from its source text; it can only be built where that source is at hand. Its
results on every case below are stored so that tests/test_ref_pin.py compares
the oracle with the reference on any checkout: NodeSelect and QoS results as
one SHA-256 digest per output column (tests/golden/ref_pin.json, the digests of
make_full_golden.digest_of), the resource-algebra rows in full
(tests/golden/ref_algebra.npz).
"""
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from cranesched_b200 import abi, synth  # noqa: E402
from tests.golden.make_full_golden import digest_of  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
DIGESTS = os.path.join(HERE, "ref_pin.json")
ALGEBRA = os.path.join(HERE, "ref_algebra.npz")
QOS_COLUMNS = ("reason", "user_usage", "account_usage", "qos_usage")


def _plain(case):
    cfg, cl, rn, pd, now = case
    return cfg, cl, rn, pd, now, None


def _with_resv(seed, case, n_resv):
    resv, pd2, rn2 = synth.random_reservations(seed, case, n_resv=n_resv, single_node=True)
    cfg, cl, rn, pd, now = case
    return cfg, cl, rn2, pd2, now, resv


def feature_mix(seed):
    return _plain(synth.random_case(seed, n_jobs=250, n_nodes=40, n_parts=3 + seed % 3, n_running=30,
                                    fifo=(seed % 4 == 0), one_type_per_name=True, short=(seed % 5 == 0),
                                    limit=(180 if seed % 6 == 1 else None)))


def general_task(seed):
    return _plain(synth.random_case(100 + seed, n_jobs=200, n_nodes=36, n_running=20,
                                    one_type_per_name=True, ntpn_range=True))


def reservations(seed):
    case = synth.random_case(seed, n_jobs=200, n_nodes=30, n_parts=1 + seed % 3, n_running=12,
                             one_type_per_name=True, lists=bool(seed % 2))
    return _with_resv(seed, case, 6)


def overlapping(seed):
    base = synth.random_case(seed, n_jobs=220, n_nodes=36, n_parts=2 + seed % 3, n_running=14,
                             one_type_per_name=True, lists=bool(seed % 2), short=bool(seed % 3 == 0))
    return _plain(synth.overlap_partitions(base, seed, frac=0.25 + 0.15 * (seed % 4),
                                           which=None if seed % 3 else {1}))


def overlapping_resv(seed):
    base = synth.random_case(seed, n_jobs=200, n_nodes=34, n_parts=2 + seed % 2, n_running=12,
                             one_type_per_name=True, lists=bool(seed % 2))
    return _with_resv(seed, synth.overlap_partitions(base, seed, frac=0.3 + 0.1 * (seed % 3)), 5)


# group -> {case name -> builder of (cfg, cluster, running, pending, now, reservations or None)}
NODE_SELECT = {
    "feature_mix": {"s%d" % s: (lambda s=s: feature_mix(s)) for s in range(24)},
    "configs": {
        "config1": lambda: _plain(synth.config1()),
        "config2_s2": lambda: _plain(synth.config2(n_jobs=3500, n_nodes=300, seed_id=2)),
        "config2_s3002": lambda: _plain(synth.config2(n_jobs=3000, n_nodes=300, seed_id=3002)),
        "config3": lambda: _plain(synth.config3(n_jobs=3000, n_nodes=400, n_parts=8)),
        "config5": lambda: _plain(synth.config5(n_jobs=1500, n_nodes=60)),
    },
    "general_task": {"s%d" % s: (lambda s=s: general_task(s)) for s in range(8)},
    "reservations": {"s%d" % s: (lambda s=s: reservations(s)) for s in range(400, 416)},
    "overlapping": {"s%d" % s: (lambda s=s: overlapping(s)) for s in range(700, 712)},
    "overlapping_resv": {"s%d" % s: (lambda s=s: overlapping_resv(s)) for s in range(720, 728)},
}

QOS_PARAMS = [(801, 1.0, 0.0), (802, 3.0, 0.1), (803, 0.5, 0.4), (804, 8.0, 0.0),
              (805, 1.5, 0.2), (806, 0.8, 0.0), (807, 2.0, 0.05), (808, 20.0, 0.3)]


def qos_case(seed, tight, invalid):
    """(cluster, pending, placements of the oracle's NodeSelect, QoS table)."""
    from oracle import pyoracle
    case = synth.random_case(seed, n_jobs=600, n_nodes=60, n_parts=3, n_running=20, one_type_per_name=True)
    cfg, cl, rn, pd, now = case
    table = synth.random_qos(seed, cl, pd, tight=tight, invalid_frac=invalid)
    out, _, _ = pyoracle.node_select(cfg, cl, rn, pd, now)
    return cl, pd, out, table


def algebra_cluster():
    return synth.make_cluster([(1, synth.node_row(8, 1 << 30))], gres_entry_name=(0, 1, 2))


def algebra_inputs(n=400):
    """Seeded random (request, available, other) rows for GetFeasibleResourceInNode /
    Ckmin / operator<= (a single gres type per name)."""
    rng = np.random.default_rng(5)
    for _ in range(n):
        avail = np.zeros((), abi.RES_IN_NODE)
        avail["cpu_raw"] = int(rng.integers(0, 20)) * 128
        avail["mem"] = int(rng.integers(0, 64))
        avail["core"][0] = int(rng.integers(0, 1 << 16))
        for e in range(3):
            avail["gres"][e] = int(rng.integers(0, 1 << 6)) if rng.random() < 0.7 else 0
        req = np.zeros((), abi.RES_VIEW)
        req["cpu_raw"] = int(rng.integers(0, 12)) * 128
        req["mem"] = int(rng.integers(0, 48))
        for e in range(3):
            if rng.random() < 0.5:
                sp = int(rng.integers(0, 4)) if rng.random() < 0.5 else 0
                req["gres_spec"][e] = sp
                req["gres_total"][e] = sp + (int(rng.integers(0, 3)) if rng.random() < 0.5 else 0)
        other = avail.copy()
        other["cpu_raw"] = int(rng.integers(0, 20)) * 128
        other["core"][0] = int(rng.integers(0, 1 << 16)) if rng.random() < 0.8 else 0
        other["gres"][:3] = rng.integers(0, 1 << 6, 3)
        yield req, avail, other


def qos_digest(reason, table) -> dict:
    d = {"reason": hashlib.sha256(np.ascontiguousarray(reason).tobytes()).hexdigest()}
    for f in QOS_COLUMNS[1:]:
        d[f] = hashlib.sha256(np.ascontiguousarray(getattr(table, f)).tobytes()).hexdigest()
    d["reason_hist"] = np.bincount(reason, minlength=24).tolist()
    return d


def load() -> dict:
    with open(DIGESTS) as f:
        return json.load(f)


def main():
    from oracle import pyref
    if not pyref.available():
        raise SystemExit("make_ref_golden: oracle/_ref/libcrane_ref.so cannot be built here")
    digests = {}
    for group, cases in NODE_SELECT.items():
        digests[group] = {}
        for name, mk in cases.items():
            cfg, cl, rn, pd, now, resv = mk()
            extra = None
            if resv is not None:
                extra = pyref.RefExtra(resv_start=resv.start_time, resv_end=resv.end_time, resv_off=resv.node_off,
                                       resv_node=resv.node, resv_res=resv.res, pd_resv=pd.reservation,
                                       rn_resv=rn.reservation)
            out, _ = pyref.node_select(cfg, cl, rn, pd, now, extra)
            digests[group][name] = digest_of(out)
        print(group, len(cases), "cases", flush=True)

    digests["qos"] = {}
    for seed, tight, invalid in QOS_PARAMS:
        cl, pd, out, table = qos_case(seed, tight, invalid)
        pyref.qos_filter(cl, pd, out, table)
        digests["qos"]["s%d" % seed] = qos_digest(out.reason, table)
    with open(DIGESTS, "w") as f:
        json.dump(digests, f, indent=1, sort_keys=True)
        f.write("\n")

    cl = algebra_cluster()
    ok, alloc, ckmin, le = [], [], [], []
    for req, avail, other in algebra_inputs():
        o, a = pyref.feasible(cl, req, avail)
        ok.append(o)
        alloc.append(a)
        ckmin.append(pyref.ckmin(cl, avail, other))
        le.append(pyref.res_le(cl, avail, other))
    np.savez_compressed(ALGEBRA, ok=np.array(ok), alloc=np.array(alloc, abi.RES_IN_NODE),
                        ckmin=np.array(ckmin, abi.RES_IN_NODE), res_le=np.array(le))
    print("written:", DIGESTS, ALGEBRA, flush=True)


if __name__ == "__main__":
    main()
