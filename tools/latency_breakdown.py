#!/usr/bin/env python3
"""Where the wall time of one pdmpc_plan_timestep call goes: the bench's 560 time steps (block 0), per call the wall
time, the device time of the search kernel (CUDA events) and the copies."""
import ctypes as C
import os
import pickle
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
from bench import RECORD_CACHE  # noqa: E402
from pdmpc_b200 import capi  # noqa: E402
from pdmpc_b200.mpa import get_mpa  # noqa: E402
from pdmpc_b200.records import BatchResult  # noqa: E402

mpa = get_mpa("triple_speed", non_convex=True)
ts = pickle.load(open(os.path.join(RECORD_CACHE, "triple_speed_20v_35t_block0000.npz.ts.pkl"), "rb"))
p = capi.Planner(0)
p.upload_mpa(mpa)
p.set_cta_queue(True)
calls = []
for step, tb, td in ts:
    ro = BatchResult.empty(tb.n, mpa.Hp)
    pidx = td.pred_idx if td.pred_idx.size else np.zeros(1, dtype=np.int32)
    dc = capi.TimestepDepsC(pred_ptr=capi._ptr(td.pred_ptr, capi._p_i32), pred_idx=capi._ptr(pidx, capi._p_i32),
                            fb_npts=capi._ptr(td.fb_npts, capi._p_i32), fb_x=capi._ptr(td.fb_x, capi._p_f64),
                            fb_y=capi._ptr(td.fb_y, capi._p_f64))
    calls.append((tb, td, pidx, ro, capi.batch_in(tb), dc, capi.batch_out(ro)))
rows = []
for rep in range(3):
    for tb, td, pidx, ro, bi, dc, bo in calls:
        t0 = time.perf_counter()
        p._check(p.lib.pdmpc_plan_timestep(p.h, C.byref(bi), C.byref(dc), C.byref(bo)))
        wall = (time.perf_counter() - t0) * 1e3
        if rep:
            st = p.stats()
            rows.append((wall, st.kernel_ms, st.h2d_ms, st.d2h_ms, int(ro.n_pops.max()), int(ro.n_pops.sum())))
a = np.array(rows)
for name, col in (("wall", a[:, 0]), ("kernel", a[:, 1]), ("wall - kernel", a[:, 0] - a[:, 1])):
    print(f"{name:14s} p50 {np.percentile(col, 50):.3f}  p90 {np.percentile(col, 90):.3f}  p99 {np.percentile(col, 99):.3f}  max {col.max():.3f} ms")
worst = np.argsort(-a[:, 0])[:8]
for i in worst:
    print("slow step: wall %.3f kernel %.3f h2d %.3f d2h %.3f  longest search %d pops, all %d pops" % tuple(a[i]))
