"""ctypes binding of the CPU oracle (oracle/libpdmpc_oracle.so), of the
reference's own priority queue compiled against stub MEX headers
(oracle/_ref/libpq_ref.so) and of the same queue on libstdc++'s
std::priority_queue (oracle/libpq_std.so).

TEST INFRASTRUCTURE: import only from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  Never from p-dmpc_b200/.
"""
from __future__ import annotations

import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
if _ROOT not in sys.path:
    sys.path.insert(0, _ROOT)

from pdmpc_b200 import capi  # noqa: E402  (boundary structs only)
from pdmpc_b200.records import BatchResult, SearchBatch  # noqa: E402

ORACLE_LIB = os.path.join(_HERE, "libpdmpc_oracle.so")
PQ_REF_LIB = os.path.join(_HERE, "_ref", "libpq_ref.so")
PQ_STD_LIB = os.path.join(_HERE, "libpq_std.so")

_p_f64 = C.POINTER(C.c_double)
_p_i64 = C.POINTER(C.c_int64)


def build(force: bool = False) -> None:
    """make -C oracle: the oracle .so, the std::priority_queue .so and, when the reference checkout is given
    (oracle/Makefile REFERENCE=...), the reference's own PQ .so."""
    if force or not os.path.exists(ORACLE_LIB) or \
            os.path.getmtime(ORACLE_LIB) < os.path.getmtime(os.path.join(_HERE, "pdmpc_oracle.c")):
        subprocess.run(["make", "-C", _HERE, "libpdmpc_oracle.so"], check=True, capture_output=True)
    if force or not os.path.exists(PQ_STD_LIB) or \
            os.path.getmtime(PQ_STD_LIB) < os.path.getmtime(os.path.join(_HERE, "pq_std_driver.cpp")):
        subprocess.run(["make", "-C", _HERE, "libpq_std.so"], check=True, capture_output=True)
    if not os.path.exists(PQ_REF_LIB) or force:
        subprocess.run(["make", "-C", _HERE, "ref"], check=True, capture_output=True)


@functools.lru_cache(maxsize=None)
def have_reference_pq() -> bool:
    """True when the reference's priority-queue MEX is built (oracle/_ref/libpq_ref.so).  It is built from the
    reference checkout (oracle/Makefile, REFERENCE=...), which is not part of this repository; without it the
    tests drive the matrix-form restatement with StdPQ instead."""
    build()
    return os.path.exists(PQ_REF_LIB)


_LIB = None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        build()
        L = C.CDLL(ORACLE_LIB)
        L.oracle_sincos.argtypes = [C.c_double, _p_f64, _p_f64]
        L.oracle_sincos.restype = None
        L.oracle_intersect_sat.argtypes = [_p_f64, _p_f64, C.c_int, _p_f64, _p_f64, C.c_int]
        L.oracle_intersect_sat.restype = C.c_int
        L.oracle_intersect_lanelets.argtypes = [_p_f64, _p_f64, C.c_int, _p_f64, _p_f64, _p_f64, _p_f64, C.c_int]
        L.oracle_intersect_lanelets.restype = C.c_int
        L.oracle_intersect_lanelet_boundary.argtypes = [_p_f64, _p_f64, C.c_int, _p_f64, _p_f64, C.c_int,
                                                        _p_f64, _p_f64, C.c_int]
        L.oracle_intersect_lanelet_boundary.restype = C.c_int
        L.oracle_interx.argtypes = [_p_f64, _p_f64, C.c_int, _p_f64, _p_f64, C.c_int]
        L.oracle_interx.restype = C.c_int
        L.oracle_pq_new.argtypes = []
        L.oracle_pq_new.restype = C.c_void_p
        L.oracle_pq_free.argtypes = [C.c_void_p]
        L.oracle_pq_free.restype = None
        L.oracle_pq_push.argtypes = [C.c_void_p, C.c_int64, C.c_double]
        L.oracle_pq_push.restype = None
        L.oracle_pq_pop.argtypes = [C.c_void_p, _p_f64]
        L.oracle_pq_pop.restype = C.c_int64
        L.oracle_pq_size.argtypes = [C.c_void_p]
        L.oracle_pq_size.restype = C.c_int64
        L.oracle_plan_batch.argtypes = [C.POINTER(capi.MpaDesc), C.POINTER(capi.BatchIn),
                                        C.POINTER(capi.BatchOut), C.c_int]
        L.oracle_plan_batch.restype = C.c_int
        L.oracle_joint_plan_batch.argtypes = [C.POINTER(capi.MpaDesc), C.POINTER(capi.BatchIn), C.c_int,
                                              C.POINTER(capi.BatchOut), C.c_int64]
        L.oracle_joint_plan_batch.restype = C.c_int
        L.oracle_plan_trace.argtypes = [C.POINTER(capi.MpaDesc), C.POINTER(capi.BatchIn), C.c_int,
                                        _p_i64, C.c_int64, _p_i64]
        L.oracle_plan_trace.restype = C.c_int
        L.oracle_mcts_plan_batch.argtypes = [C.POINTER(capi.MpaDesc), C.POINTER(capi.BatchIn),
                                             C.POINTER(capi.MctsParams), C.POINTER(capi.BatchOut), C.c_int]
        L.oracle_mcts_plan_batch.restype = C.c_int
        L.oracle_mt19937_rand.argtypes = [C.c_uint32, _p_f64, C.c_int]
        L.oracle_mt19937_rand.restype = None
        L.oracle_set_hash_valid_pops_only.argtypes = [C.c_int]
        L.oracle_set_hash_valid_pops_only.restype = None
        _LIB = L
    return _LIB


def _xy(p):
    p = np.asarray(p, dtype=np.float64)
    x = np.ascontiguousarray(p[0])
    y = np.ascontiguousarray(p[1])
    return x, y, x.ctypes.data_as(_p_f64), y.ctypes.data_as(_p_f64), int(x.size)


def sincos(x: float):
    s, c = C.c_double(), C.c_double()
    lib().oracle_sincos(float(x), C.byref(s), C.byref(c))
    return s.value, c.value


def intersect_sat(shape1, shape2) -> bool:
    a = _xy(shape1)
    b = _xy(shape2)
    return bool(lib().oracle_intersect_sat(a[2], a[3], a[4], b[2], b[3], b[4]))


def intersect_lanelets(shape, lanelet) -> bool:
    """lanelet: [n, 6] with LaneletInfo columns rx, ry, lx, ly, cx, cy."""
    s = _xy(shape)
    lan = np.asarray(lanelet, dtype=np.float64)
    cols = [np.ascontiguousarray(lan[:, i]) for i in range(4)]
    ptrs = [c.ctypes.data_as(_p_f64) for c in cols]
    return bool(lib().oracle_intersect_lanelets(s[2], s[3], s[4], ptrs[0], ptrs[1], ptrs[2], ptrs[3],
                                                int(lan.shape[0])))


def intersect_lanelet_boundary(shape, left, right) -> bool:
    s, l, r = _xy(shape), _xy(left), _xy(right)
    return bool(lib().oracle_intersect_lanelet_boundary(s[2], s[3], s[4], l[2], l[3], l[4], r[2], r[3], r[4]))


def interx(l1, l2) -> bool:
    a, b = _xy(l1), _xy(l2)
    return bool(lib().oracle_interx(a[2], a[3], a[4], b[2], b[3], b[4]))


class OraclePQ:
    """The oracle's restated libstdc++ heap."""

    def __init__(self):
        self.q = lib().oracle_pq_new()

    def push(self, ident: int, value: float):
        lib().oracle_pq_push(self.q, int(ident), float(value))

    def pop(self):
        v = C.c_double()
        i = lib().oracle_pq_pop(self.q, C.byref(v))
        return int(i), v.value

    def size(self) -> int:
        return int(lib().oracle_pq_size(self.q))

    def __del__(self):
        try:
            lib().oracle_pq_free(self.q)
        except Exception:
            pass


class ReferencePQ:
    """The reference's unmodified priority_queue_interface_mex.cpp (stub MEX API)."""

    _lib = None

    def __init__(self):
        if ReferencePQ._lib is None:
            build()
            if not os.path.exists(PQ_REF_LIB):
                raise FileNotFoundError(PQ_REF_LIB)
            L = C.CDLL(PQ_REF_LIB)
            L.pq_ref_new.restype = C.c_int64
            L.pq_ref_push.argtypes = [C.c_int64, _p_f64, _p_f64, C.c_int64]
            L.pq_ref_push.restype = None
            L.pq_ref_pop.argtypes = [C.c_int64, _p_f64]
            L.pq_ref_pop.restype = C.c_int64
            L.pq_ref_size.argtypes = [C.c_int64]
            L.pq_ref_size.restype = C.c_int64
            ReferencePQ._lib = L
        self.obj = ReferencePQ._lib.pq_ref_new()

    def push(self, ids, vals):
        ids = np.ascontiguousarray(np.atleast_1d(ids), dtype=np.float64)
        vals = np.ascontiguousarray(np.atleast_1d(vals), dtype=np.float64)
        ReferencePQ._lib.pq_ref_push(self.obj, ids.ctypes.data_as(_p_f64), vals.ctypes.data_as(_p_f64),
                                     int(ids.size))

    def pop(self):
        # The reference answers -1 for an empty queue (mex.cpp:87-94) but then still calls
        # std::priority_queue::pop() on it (:96-99), which is undefined behaviour in libstdc++
        # (the vector's size underflows).  The search never touches the queue again after that
        # (GraphSearch.m:57-61), a test harness does: answer -1 without executing the UB.
        if self.size() == 0:
            return -1, -1.0
        v = C.c_double()
        i = ReferencePQ._lib.pq_ref_pop(self.obj, C.byref(v))
        return int(i), v.value

    def size(self) -> int:
        return int(ReferencePQ._lib.pq_ref_size(self.obj))


class StdPQ:
    """The reference's queue on libstdc++'s std::priority_queue (oracle/pq_std_driver.cpp): shares no code with
    OraclePQ.  Same interface as ReferencePQ."""

    _lib = None

    def __init__(self):
        if StdPQ._lib is None:
            build()
            L = C.CDLL(PQ_STD_LIB)
            L.pq_std_new.restype = C.c_void_p
            L.pq_std_free.argtypes = [C.c_void_p]
            L.pq_std_free.restype = None
            L.pq_std_push.argtypes = [C.c_void_p, _p_f64, _p_f64, C.c_int64]
            L.pq_std_push.restype = None
            L.pq_std_pop.argtypes = [C.c_void_p, _p_f64]
            L.pq_std_pop.restype = C.c_int64
            L.pq_std_size.argtypes = [C.c_void_p]
            L.pq_std_size.restype = C.c_int64
            StdPQ._lib = L
        self.obj = StdPQ._lib.pq_std_new()

    def push(self, ids, vals):
        ids = np.ascontiguousarray(np.atleast_1d(ids), dtype=np.float64)
        vals = np.ascontiguousarray(np.atleast_1d(vals), dtype=np.float64)
        StdPQ._lib.pq_std_push(self.obj, ids.ctypes.data_as(_p_f64), vals.ctypes.data_as(_p_f64), int(ids.size))

    def pop(self):
        v = C.c_double()
        i = StdPQ._lib.pq_std_pop(self.obj, C.byref(v))
        return int(i), v.value

    def size(self) -> int:
        return int(StdPQ._lib.pq_std_size(self.obj))

    def __del__(self):
        try:
            StdPQ._lib.pq_std_free(self.obj)
        except Exception:
            pass


def plan_batch(mpa, batch: SearchBatch, n_threads: int = 1, hash_valid_pops_only: bool = False) -> BatchResult:
    """GraphSearch.do_graph_search for every search of the batch on the CPU.
    hash_valid_pops_only: pop_hash as CUDA launch shape 5 reports it (include/pdmpc_b200.h)."""
    d, keep = capi.mpa_desc(mpa)
    r = BatchResult.empty(batch.n, batch.Hp)
    bi, bo = capi.batch_in(batch), capi.batch_out(r)
    lib().oracle_set_hash_valid_pops_only(1 if hash_valid_pops_only else 0)
    try:
        rc = lib().oracle_plan_batch(C.byref(d), C.byref(bi), C.byref(bo), int(n_threads))
    finally:
        lib().oracle_set_hash_valid_pops_only(0)
    if rc != 0:
        raise RuntimeError(f"oracle_plan_batch failed: {rc}")
    del keep
    return r


def joint_plan_batch(mpa, batch: SearchBatch, n_vehicles: int, max_nodes: int = 1 << 21,
                     hash_valid_pops_only: bool = False) -> BatchResult:
    """Centralized (joint) search: rows of the batch = searches x n_vehicles (oracle_joint_plan_batch)."""
    d, keep = capi.mpa_desc(mpa)
    r = BatchResult.empty(batch.n, batch.Hp)
    bi, bo = capi.batch_in(batch), capi.batch_out(r)
    lib().oracle_set_hash_valid_pops_only(1 if hash_valid_pops_only else 0)
    try:
        rc = lib().oracle_joint_plan_batch(C.byref(d), C.byref(bi), int(n_vehicles), C.byref(bo), int(max_nodes))
    finally:
        lib().oracle_set_hash_valid_pops_only(0)
    if rc != 0:
        raise RuntimeError(f"oracle_joint_plan_batch failed: {rc}")
    del keep
    return r


def plan_trace(mpa, batch: SearchBatch, search: int, cap: int = 1 << 20) -> np.ndarray:
    d, keep = capi.mpa_desc(mpa)
    bi = capi.batch_in(batch)
    tr = np.zeros(cap, dtype=np.int64)
    n = C.c_int64()
    rc = lib().oracle_plan_trace(C.byref(d), C.byref(bi), int(search), tr.ctypes.data_as(_p_i64), cap,
                                 C.byref(n))
    if rc != 0:
        raise RuntimeError(f"oracle_plan_trace failed: {rc}")
    del keep
    return tr[: n.value].copy()


def mcts_plan_batch(mpa, batch: SearchBatch, seeds, n_expansions_max: int = 250, n_threads: int = 1) -> BatchResult:
    """MonteCarloTreeSearch.do_graph_search for every search of the batch on the CPU."""
    d, keep = capi.mpa_desc(mpa)
    r = BatchResult.empty(batch.n, batch.Hp)
    bi, bo = capi.batch_in(batch), capi.batch_out(r)
    prm, keep2 = capi.mcts_params(seeds, n_expansions_max, batch.n)
    rc = lib().oracle_mcts_plan_batch(C.byref(d), C.byref(bi), C.byref(prm), C.byref(bo), int(n_threads))
    if rc != 0:
        raise RuntimeError(f"oracle_mcts_plan_batch failed: {rc}")
    del keep, keep2
    return r


def mt19937_rand(seed: int, n: int) -> np.ndarray:
    """rand(RandStream('mt19937ar', Seed = seed), 1, n) as the oracle restates it."""
    out = np.zeros(n)
    lib().oracle_mt19937_rand(int(seed), out.ctypes.data_as(_p_f64), int(n))
    return out
