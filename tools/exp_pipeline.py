#!/usr/bin/env python3
"""e2e time of pdmpc_plan_batch on the bench's records (pinned host buffers) for different chunk counts of the
copy/search pipeline and escalation thresholds."""
import ctypes as C
import dataclasses
import glob
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from bench import RECORD_CACHE  # noqa: E402
from pdmpc_b200 import capi  # noqa: E402
if os.environ.get('PDMPC_LIB'):
    capi.LIB_PATH = os.environ['PDMPC_LIB']
    capi.load_library.__defaults__ = (capi.LIB_PATH,)
from pdmpc_b200.mpa import get_mpa  # noqa: E402
from pdmpc_b200.records import BatchResult, SearchBatch  # noqa: E402

files = sorted(glob.glob(sys.argv[1] if len(sys.argv) > 1 else os.path.join(RECORD_CACHE, "triple_speed_20v_35t_block00*.npz")))[:64]
mpa = get_mpa("triple_speed", non_convex=True)
batch = SearchBatch.concat([SearchBatch.load(f) for f in files])
p = capi.Planner(0)
p.upload_mpa(mpa)
p.set_cta_queue(True)
keep = []


def pinned_like(a):
    t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
    keep.append(t)
    return t.numpy()[: a.nbytes].view(a.dtype).reshape(a.shape)


host_in = {}
for f in dataclasses.fields(batch):
    a = getattr(batch, f.name)
    if isinstance(a, np.ndarray):
        host_in[f.name] = pinned_like(a)
        host_in[f.name][...] = a
hb = dataclasses.replace(batch, **host_in)
out = BatchResult.empty(batch.n, mpa.Hp)
for f in dataclasses.fields(out):
    a = getattr(out, f.name)
    if isinstance(a, np.ndarray):
        setattr(out, f.name, pinned_like(a))
bi, bo = capi.batch_in(hb), capi.batch_out(out)
print(batch.n, "searches")
for chunks in [int(c) for c in os.environ.get('PDMPC_CHUNKS', '1,2,3,4,5,6,8,12').split(',')]:
    p.set_pipeline_chunks(chunks)
    for esc in [int(v) for v in os.environ.get('PDMPC_ESC_SWEEP', '-1').split(',')]:
        p.set_escalation(esc)
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            p._check(p.lib.pdmpc_plan_batch(p.h, C.byref(bi), C.byref(bo)))
            ts.append((time.perf_counter() - t0) * 1e3)
        st = p.stats()
        print(f"chunks {chunks:2d} escalation {esc}: {min(ts[2:]):.1f} ms -> {batch.n / min(ts[2:]) / 1e3:.3f} M plans/s  "
              f"(h2d {st.h2d_ms:.1f} kernel {st.kernel_ms:.1f} d2h {st.d2h_ms:.1f} ms, escalated {st.escalated})")
        if chunks != 1 and hasattr(p, "pipeline_timeline"):
            hm, im, dm = p.pipeline_timeline()
            print("   chunk: enqueued by the host at / inputs landed at / searches done at [ms]:",
                  "  ".join(f"{a:.1f}/{b:.1f}/{c:.1f}" for a, b, c in zip(hm, im, dm)))
