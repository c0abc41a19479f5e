#!/usr/bin/env python3
"""Where the end of the throughput launch goes: one pdmpc_run_staged over the bench's own records (bench.py's record
cache and generator), timed from %globaltimer stamps of a library built with -DPDMPC_TAIL_STAMPS.

Prints per escalation schedule: the launch (kernel time of the call), the time until the work list ran dry, the tile tail
(list dry -> last tile CTA exit) with percentiles of the tile CTAs' exit times after the list ran dry, the escalation
(CTA) phase (last tile CTA exit -> last escalated search done) and the escalated searches at the full and at a reduced
budget.

  python tools/tail_anatomy.py [--scenarios 512] [--schedules default,0:0,1024:32] [--runs 3] [--lib PATH]

A schedule "P_MIN:S" sets the experiment variables PDMPC_ESC_MIN / PDMPC_ESC_SLOPE (S = 0: the uniform threshold of the
batch size); "default" leaves them unset.  Without --lib the stamped library is compiled into a temporary directory.
"""
import argparse
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402


def build_stamped(out_dir: str) -> str:
    from __graft_entry__ import NVCC_FLAGS
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    lib = os.path.join(out_dir, "libpdmpc_b200_stamps.so")
    subprocess.run([nvcc] + NVCC_FLAGS + ["-DPDMPC_TAIL_STAMPS", "-o", lib,
                                          os.path.join(ROOT, "p-dmpc_b200", "csrc", "pdmpc_capi.cu")], check=True)
    return lib


def set_schedule(spec: str) -> None:
    for k in ("PDMPC_ESC_MIN", "PDMPC_ESC_SLOPE"):
        os.environ.pop(k, None)
    if spec != "default":
        p_min, slope = spec.split(":")
        os.environ["PDMPC_ESC_MIN"], os.environ["PDMPC_ESC_SLOPE"] = p_min, slope


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenarios", type=int, default=512, help="bench scenarios (512 = the bench's 358 400 records)")
    ap.add_argument("--schedules", default="0:0,default")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--lib", default="")
    a = ap.parse_args()

    import bench
    from pdmpc_b200 import capi
    from pdmpc_b200.mpa import get_mpa
    args = argparse.Namespace(no_cache=False, mpa="triple_speed", vehicles=20, sim_steps=35, scenarios=a.scenarios,
                              scenarios_total=0)
    tmp = tempfile.mkdtemp(prefix="pdmpc_tail_")
    capi._LIB = None   # the stamped library serves this process (records rolled out here too: same results)
    lib = capi.load_library(a.lib or build_stamped(tmp))
    batch, _, _ = bench.get_records(args, bench.rank_blocks(args, 0, 1), "gpu", 0, os.cpu_count() or 1)
    lib.pdmpc_get_tail_stamps.argtypes = [capi.C.c_void_p, capi.C.c_int32, capi.C.POINTER(capi.C.c_uint64)]
    lib.pdmpc_get_tail_stamps.restype = capi.C.c_int

    p = capi.Planner(0)
    p.upload_mpa(get_mpa("triple_speed", non_convex=True))
    p.set_cta_queue(True)   # as the bench
    p.stage(batch)
    n = batch.n
    print(f"{n} searches ({a.scenarios} bench scenarios), one pdmpc_run_staged per row, times in ms: list dry = from the "
          f"first tile CTA's start; exits = tile CTA exit times after the list ran dry")
    buf = np.zeros(8 + 148 * 64, dtype=np.uint64)
    for spec in a.schedules.split(","):
        set_schedule(spec)
        budgets = capi.escalation_budgets(n, [0, n // 2, (2 * n) // 3, n - 7104, n - 1], lib=lib)
        rows = []
        for _ in range(a.runs + 1):   # the first run warms up
            p.run_staged()
            p.sync()
            st = p.stats()
            rc = lib.pdmpc_get_tail_stamps(p.h, buf.size, buf.ctypes.data_as(capi.C.POINTER(capi.C.c_uint64)))
            assert rc == 0, rc
            t0 = int(buf[0])
            ctas = int(buf[4])
            ex = (buf[8:8 + ctas].astype(np.int64) - t0) / 1e6
            dry = (int(buf[1]) - t0) / 1e6
            last = ex.max()
            cta_end = (int(buf[3]) - t0) / 1e6 if buf[3] else last
            rows.append(dict(ms=st.kernel_ms, dry=dry, tail=last - dry, cta=cta_end - last,
                             pct=np.percentile(ex - dry, [50, 90, 99]), full=int(buf[5]), red=int(buf[6]),
                             esc=st.escalated, ctas=ctas))
        rows = rows[1:]
        print(f"\nschedule {spec}: budget at positions 0, n/2, 2n/3, n-7104, n-1 = {budgets.tolist()}")
        for r in rows:
            print(f"  launch {r['ms']:7.2f} ms | list dry {r['dry']:6.2f} | tile tail {r['tail']:6.2f} "
                  f"(exits p50/p90/p99 {r['pct'][0]:5.2f} / {r['pct'][1]:5.2f} / {r['pct'][2]:5.2f}, {r['ctas']} CTAs) | "
                  f"CTA phase {r['cta']:5.2f} | escalated {r['full']} full + {r['red']} reduced")
        best = min(rows, key=lambda r: r["ms"])
        print(f"  best launch {best['ms']:.2f} ms -> {n / best['ms'] / 1e3:.3f} M plans/s")
    p.close()


if __name__ == "__main__":
    main()
