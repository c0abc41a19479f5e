#!/usr/bin/env python3
"""Simultaneous prioritizations in one call (pdmpc_plan_timestep_explorative, DESIGN.md §4.13), measured:

  latency     live 20-vehicle closed loops (seeds 1.., road network, triple_speed MPA, all n_CL permutations), wall time
              per time step of (a) the host path: ExplorativeRunner with pdmpc_plan_timestep over host-built batches and
              the host exchange, and (b) ExplorativeRunner(explorative_fn=Planner.plan_timestep_explorative); the two
              loops run alternately per seed in the same session and must end in the same poses (asserted);
  throughput  one time step (the first) of 64 and of 512 scenarios x 20 vehicles x all their permutations as ONE call:
              CUDA events on the planner's stream recorded before and after the call (device time of the whole call,
              including the gaps while the host expands and validates the rows), pdmpc_stats.kernel_ms (the searches,
              the choice and the commit), wall time of the call, searches/s.
              The slots are reset before every call (outside the timed region), so every call plans the same step.

usage: timestep_explorative.py [OUT.json] [STEPS] [SEEDS]   (prints a summary; writes every number to OUT.json)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from pdmpc_b200 import capi, scenario  # noqa: E402
from pdmpc_b200.mpa import get_mpa  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else ""
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 35
SEEDS = [int(s) for s in sys.argv[3].split(",")] if len(sys.argv) > 3 else [1, 2, 3, 4]
WARM = 5   # first time steps of every loop: module loading, buffer growth


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (v.strip() for v in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def pct(t) -> dict:
    t = np.asarray(t)
    return {"p50_ms": float(np.percentile(t, 50)), "p99_ms": float(np.percentile(t, 99)), "max_ms": float(t.max()),
            "n": int(t.size)}


mpa = get_mpa("triple_speed", non_convex=True)
p = capi.Planner(0)
p.upload_mpa(mpa)
hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
explorative = lambda *a, **k: p.plan_timestep_explorative(*a, **k, raise_on_search_error=False)
step_a, step_b, perms = [], [], []

for seed in SEEDS:
    sc = scenario.commonroad_scenario(mpa, 20, seed=seed)
    p.upload_road(scenario.road_tables([sc]))
    p.closed_loop_reset(20, hl, hw)
    a = scenario.ExplorativeRunner(scenario.commonroad_scenario(mpa, 20, seed=seed), lambda b, d: p.plan_timestep(b, d, False))
    b = scenario.ExplorativeRunner(sc, None, explorative_fn=explorative)
    for k in range(STEPS):
        for r, bucket in ((a, step_a), (b, step_b)):
            t0 = time.perf_counter()
            r.step()
            if k >= WARM:
                bucket.append((time.perf_counter() - t0) * 1e3)
        perms.append(b.explorative_records[-1]["n_permutations"])
    assert np.array_equal(a.pose, b.pose) and np.array_equal(a.trim, b.trim), seed

stream = torch.cuda.ExternalStream(p.stream())
throughput = {}
for n_sc in (64, 512):
    scs = [scenario.commonroad_scenario(mpa, 20, seed=s) for s in range(1, n_sc + 1)]
    p.upload_road(scenario.road_tables(scs))
    p.closed_loop_reset(20 * n_sc, hl, hw)
    runners = []
    for k, sc in enumerate(scs):
        r = scenario.ExplorativeRunner(sc, None)
        r.path_id0 = 20 * k
        runners.append(r)
    captured = {}

    def capture(*a, **kw):
        captured["args"], captured["kw"] = a, kw
        return explorative(*a, **kw)

    first = scenario.explorative_lockstep_step(runners, capture)
    dev, wall, kern = [], [], []
    for i in range(25):
        p.closed_loop_reset(20 * n_sc, hl, hw)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        res, _ = explorative(*captured["args"], **captured["kw"])
        w = (time.perf_counter() - t0) * 1e3
        e1.record(stream)
        e1.synchronize()
        if i >= 5:
            dev.append(e0.elapsed_time(e1))
            wall.append(w)
            kern.append(p.stats().kernel_ms)
        assert np.array_equal(res.pop_hash, first.pop_hash)
    rows = int(first.status.size)
    throughput[f"{n_sc}x20"] = {"rows": rows, "exhausted_rows": int(first.is_exhausted.sum()), "shape": int(p.stats().shape),
                                "device_events": pct(dev), "searches_choice_commit_kernel": pct(kern),
                                "call_wall": pct(wall),
                                "searches_per_s_device": rows / (np.median(dev) * 1e-3),
                                "searches_per_s_wall": rows / (np.median(wall) * 1e-3)}

res = {**gpu_info(), "closed_loops": {"vehicles": 20, "seeds": SEEDS, "steps": STEPS, "warm_steps_dropped": WARM,
                                      "permutations_per_step": {"mean": float(np.mean(perms)), "max": int(np.max(perms))},
                                      "a_host_path_step": pct(step_a), "b_explorative_call_step": pct(step_b)},
       "throughput_first_step": throughput}
print(json.dumps(res, indent=1))
if OUT:
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
p.close()
