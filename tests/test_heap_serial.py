"""The single-thread heap of the lane-per-search kernel (p-dmpc_b200/csrc/pdmpc_heap_serial.h,
compiled here as host code) against the reference's unmodified priority-queue MEX source
(oracle/_ref/libpq_ref.so, when built), the same queue on libstdc++'s std::priority_queue and
the oracle's literal libstdc++ restatement: identical pop
sequences on tie-dense push/pop mixes, including the early-stop pop."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "heap_serial_host.cpp")
LIB = os.path.join(HERE, "native", "libheap_serial_host.so")
HDR = os.path.join(os.path.dirname(HERE), "p-dmpc_b200", "csrc", "pdmpc_heap_serial.h")


@pytest.fixture(scope="module")
def hs():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(SRC), os.path.getmtime(HDR)):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", LIB, SRC], check=True)
    L = C.CDLL(LIB)
    L.hs_new.restype = C.c_void_p
    L.hs_free.argtypes = [C.c_void_p]
    L.hs_push.argtypes = [C.c_void_p, C.c_longlong, C.c_double]
    L.hs_pop.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
    L.hs_pop.restype = C.c_longlong
    L.hs_size.argtypes = [C.c_void_p]
    L.hs_size.restype = C.c_int
    return L


@pytest.mark.parametrize("seed", range(12))
def test_serial_heap_matches_reference_and_oracle(hs, seed):
    rng = np.random.default_rng(1000 + seed)
    refs = [oracle_py.OraclePQ(), oracle_py.StdPQ()]
    if oracle_py.have_reference_pq():
        refs.append(oracle_py.ReferencePQ())
    q = hs.hs_new()
    next_id = 1
    f = C.c_double()

    def pop_all_equal():
        got = hs.hs_pop(q, C.byref(f))
        for r in refs:
            a = r.pop()
            assert a[0] == got
            if got != -1:
                assert a[1] == f.value
        return got

    try:
        for _ in range(600):
            if rng.random() < 0.55 or hs.hs_size(q) == 0:
                m = int(rng.integers(1, 13))
                if seed % 3 == 0:
                    vals = rng.random(m)
                elif seed % 3 == 1:   # few distinct values: ties everywhere
                    vals = rng.integers(0, 5, size=m).astype(np.float64) * 0.25
                else:                 # all equal: order is pure heap mechanics
                    vals = np.full(m, 1.5)
                ids = np.arange(next_id, next_id + m)
                next_id += m
                for r in refs:
                    if isinstance(r, (oracle_py.ReferencePQ, oracle_py.StdPQ)):
                        r.push(ids, vals)
                    else:
                        for i, v in zip(ids, vals):
                            r.push(int(i), float(v))
                for i, v in zip(ids, vals):
                    hs.hs_push(q, int(i), float(v))
            else:
                for _ in range(int(rng.integers(1, 8))):
                    pop_all_equal()
            for r in refs:
                assert r.size() == hs.hs_size(q)
        while pop_all_equal() != -1:
            pass
    finally:
        hs.hs_free(q)
