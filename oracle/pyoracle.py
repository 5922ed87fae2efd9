"""ctypes front-end of oracle/libcrane_oracle.so (TEST INFRASTRUCTURE ONLY)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from cranesched_b200 import abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libcrane_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile the C++ restatement (g++ only; no reference sources needed)."""
    src = os.path.join(_HERE, "crane_oracle.cpp")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        _lib = C.CDLL(_SO)
        _lib.crane_oracle_node_select.restype = C.c_int
        _lib.crane_oracle_node_select.argtypes = [
            C.POINTER(abi.SchedConfig), C.POINTER(abi.ClusterC), C.c_int64,
            C.POINTER(abi.RunningC), C.POINTER(abi.PendingC), C.POINTER(abi.PlacementsC),
            C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_uint32)]
        _lib.crane_oracle_feasible.restype = C.c_int
        _lib.crane_oracle_feasible.argtypes = [C.POINTER(abi.ClusterC), C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.crane_oracle_ckmin.restype = None
        _lib.crane_oracle_ckmin.argtypes = [C.POINTER(abi.ClusterC), C.c_void_p, C.c_void_p]
        _lib.crane_oracle_res_le.restype = C.c_int
        _lib.crane_oracle_res_le.argtypes = [C.POINTER(abi.ClusterC), C.c_void_p, C.c_void_p]
        _lib.crane_oracle_timeline_update.restype = C.c_int
        _lib.crane_oracle_timeline_update.argtypes = [
            C.POINTER(abi.ClusterC), C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32), C.c_uint32,
            C.c_int64, C.c_int64, C.c_void_p]
        _lib.crane_oracle_earliest_start.restype = C.c_int
        _lib.crane_oracle_earliest_start.argtypes = [
            C.POINTER(abi.ClusterC), C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
            C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_int64)]
        _lib.crane_oracle_qos_filter.restype = C.c_int
        _lib.crane_oracle_qos_filter.argtypes = [
            C.POINTER(abi.ClusterC), C.POINTER(abi.PendingC), C.POINTER(abi.PlacementsC),
            C.POINTER(abi.QosTableC)]
        _lib.crane_oracle_selftest.restype = C.c_int
        _lib.crane_oracle_selftest.argtypes = [C.c_char_p, C.c_size_t]
    return _lib


def node_select(cfg: abi.Config, cluster: abi.Cluster, running: abi.Running,
                pending: abi.Pending, now: int, max_jobs: int = 0, resv: "abi.Reservations | None" = None):
    """Returns (Placements, elapsed_ms, jobs_done)."""
    out = abi.Placements.for_pending(pending)
    c_resv = resv.as_c() if resv is not None else None
    lib().crane_oracle_set_reservations.restype = None
    lib().crane_oracle_set_reservations.argtypes = [C.c_void_p]
    lib().crane_oracle_set_reservations(C.byref(c_resv) if c_resv is not None else None)
    c_cfg, c_cl, c_rn, c_pd, c_out = cfg.as_c(), cluster.as_c(), running.as_c(), pending.as_c(), out.as_c()
    ms = C.c_double(0.0)
    done = C.c_uint32(0)
    rc = lib().crane_oracle_node_select(C.byref(c_cfg), C.byref(c_cl), now, C.byref(c_rn),
                                         C.byref(c_pd), C.byref(c_out), C.byref(ms),
                                         max_jobs, C.byref(done))
    lib().crane_oracle_set_reservations(None)
    if rc != 0:
        raise RuntimeError(f"crane_oracle_node_select rc={rc}")
    return out, ms.value, done.value


def feasible(cluster: abi.Cluster, req: np.ndarray, avail: np.ndarray):
    alloc = np.zeros((), abi.RES_IN_NODE)
    req = np.ascontiguousarray(req, abi.RES_VIEW)
    avail = np.ascontiguousarray(avail, abi.RES_IN_NODE)
    c = cluster.as_c()
    ok = lib().crane_oracle_feasible(C.byref(c), req.ctypes.data, avail.ctypes.data, alloc.ctypes.data)
    return bool(ok), alloc


def ckmin(cluster: abi.Cluster, a: np.ndarray, b: np.ndarray) -> np.ndarray:
    a = np.array(a, abi.RES_IN_NODE, copy=True)
    b = np.ascontiguousarray(b, abi.RES_IN_NODE)
    c = cluster.as_c()
    lib().crane_oracle_ckmin(C.byref(c), a.ctypes.data, b.ctypes.data)
    return a


def res_le(cluster: abi.Cluster, a: np.ndarray, b: np.ndarray) -> bool:
    a = np.ascontiguousarray(a, abi.RES_IN_NODE)
    b = np.ascontiguousarray(b, abi.RES_IN_NODE)
    c = cluster.as_c()
    return bool(lib().crane_oracle_res_le(C.byref(c), a.ctypes.data, b.ctypes.data))


def qos_filter(cluster: abi.Cluster, pending: abi.Pending, out: abi.Placements, qos: abi.QosTable):
    """In place on out.reason and qos.*_usage."""
    c_cl, c_pd, c_out, c_q = cluster.as_c(), pending.as_c(), out.as_c(), qos.as_c()
    rc = lib().crane_oracle_qos_filter(C.byref(c_cl), C.byref(c_pd), C.byref(c_out), C.byref(c_q))
    if rc != 0:
        raise RuntimeError(f"crane_oracle_qos_filter rc={rc}")
    return out


def selftest():
    buf = C.create_string_buffer(4096)
    n = lib().crane_oracle_selftest(buf, 4096)
    return n, buf.value.decode()
