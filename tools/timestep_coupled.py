#!/usr/bin/env python3
"""Coupling on the device (pdmpc_couple, DESIGN.md §4.12), measured:

  latency     live 20-vehicle closed loops (seeds 1.., road network, triple_speed MPA), wall time per time step of
              (a) the host's reachable-set coupling + decide_relations + pdmpc_plan_timestep_from_states and
              (b) pdmpc_plan_timestep_from_states_coupled; both loops must end in the same poses (asserted);
  throughput  device time of pdmpc_couple alone (CUDA events around its memsets and two kernels) for 512 scenarios x 20
              vehicles at random poses along the reference paths, after a warm-up.

usage: timestep_coupled.py [OUT.json] [STEPS] [SEEDS]   (prints a summary; writes every number to OUT.json)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
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
p.set_cta_queue(True)
p.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
step_a, call_a, step_b, call_b = [], [], [], []


def timed(bucket, fn):
    def wrapped(*a):
        t0 = time.perf_counter()
        r = fn(*a)
        bucket[-1] += (time.perf_counter() - t0) * 1e3
        return r
    return wrapped


for seed in SEEDS:
    sc = scenario.commonroad_scenario(mpa, 20, seed=seed)
    p.upload_road(scenario.road_tables([sc]))
    loops = {}
    for name, steps, calls in (("a", step_a, call_a), ("b", step_b, call_b)):
        p.closed_loop_reset(20, hl, hw)
        if name == "a":
            r = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=seed), None, coupler="reachable_set",
                                        states_fn=timed(calls, lambda *a: p.plan_timestep_from_states(*a, raise_on_search_error=False)))
        else:
            r = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=seed), None,
                                        coupled_fn=timed(calls, lambda *a: p.plan_timestep_from_states_coupled(*a, raise_on_search_error=False)))
        for k in range(STEPS):
            calls.append(0.0)
            t0 = time.perf_counter()
            r.step_timestep()
            dt = (time.perf_counter() - t0) * 1e3
            if k < WARM:
                calls.pop()
            else:
                steps.append(dt)
        loops[name] = r
    assert np.array_equal(loops["a"].pose, loops["b"].pose) and np.array_equal(loops["a"].trim, loops["b"].trim)

# throughput: 512 scenarios x 20 vehicles in one pdmpc_couple call
rng = np.random.default_rng(0)
pool = [v.reference_path for v in scenario.commonroad_scenario(mpa, 33, seed=1).vehicles]
N = 512 * 20
pose = np.zeros((N, 3))
for i in range(N):
    path = pool[rng.integers(len(pool))]
    j = int(rng.integers(0, path.shape[0] - 1))
    d = path[j + 1] - path[j]
    pose[i] = [*(path[j] + rng.normal(scale=0.05, size=2)), np.arctan2(d[1], d[0]) + rng.normal(scale=0.2)]
trim = rng.integers(1, mpa.n_trims + 1, size=N).astype(np.int32)
sp = np.arange(0, N + 1, 20)
for _ in range(5):
    rel = p.couple(pose[:, 0], pose[:, 1], pose[:, 2], trim, sp, "coloring", 99)
dev, wall = [], []
for _ in range(50):
    t0 = time.perf_counter()
    p.couple(pose[:, 0], pose[:, 1], pose[:, 2], trim, sp, "coloring", 99)
    wall.append((time.perf_counter() - t0) * 1e3)
    dev.append(p.stats().kernel_ms)
coupled_pairs = int(sum((a > 1e-3).sum() for a in rel["overlap_area"]) // 2)

res = {**gpu_info(), "closed_loops": {"vehicles": 20, "seeds": SEEDS, "steps": STEPS, "warm_steps_dropped": WARM,
                                      "a_host_coupling_step": pct(step_a), "a_plan_timestep_from_states_call": pct(call_a),
                                      "a_host_coupling_share_ms": float(np.median(np.array(step_a) - np.array(call_a))),
                                      "b_coupled_step": pct(step_b), "b_plan_timestep_from_states_coupled_call": pct(call_b)},
       "couple_512x20": {"pairs": 512 * 190, "coupled_pairs": coupled_pairs, "max_level": int(rel["level"].max()),
                         "device": pct(dev), "call_wall": pct(wall)}}
print(json.dumps(res, indent=1))
if OUT:
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
p.close()
