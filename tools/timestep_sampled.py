#!/usr/bin/env python3
"""Time steps with the sampled optimizer (pdmpc_mcts_plan_timestep*, DESIGN.md §4.14), measured:

  latency     live 20-vehicle closed loops (seeds 1.., road network, triple_speed MPA, n_expansions_max = 250), wall time
              per time step of (a) ScenarioRunner level by level with pdmpc_mcts_plan_batch and host-side obstacle
              assembly, (b) one pdmpc_mcts_plan_timestep call per step over host-built batches, (c) one
              pdmpc_mcts_plan_timestep_from_states call per step; the three loops advance alternately step by step in the
              same session and must end in the same poses (asserted);
  throughput  the first time step of 512 scenarios x 20 vehicles as ONE pdmpc_mcts_plan_timestep call: CUDA events on the
              planner's stream around the call, pdmpc_stats.kernel_ms and the call's wall time.

usage: timestep_sampled.py [OUT.json] [STEPS] [SEEDS]   (prints a summary; writes every number to OUT.json)"""
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
from pdmpc_b200.records import SearchBatch, TimestepDeps  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else ""
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 35
SEEDS = [int(s) for s in sys.argv[3].split(",")] if len(sys.argv) > 3 else [1, 2, 3, 4]
WARM = 5      # first time steps of every loop: module loading, buffer growth
NMAX = 250    # MonteCarloTreeSearch.m:8


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
p.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
times = {"a": [], "b": [], "c": []}
fallbacks = 0

for seed in SEEDS:
    sc = scenario.commonroad_scenario(mpa, 20, seed=seed)
    p.upload_road(scenario.road_tables([sc]))
    p.closed_loop_reset(20, hl, hw)
    mk = lambda: scenario.commonroad_scenario(mpa, 20, seed=seed)
    loops = {
        "a": scenario.ScenarioRunner(mk(), lambda b, s: p.mcts_plan_batch(b, s, NMAX, False), n_expansions_max=NMAX),
        "b": scenario.ScenarioRunner(mk(), None, n_expansions_max=NMAX,
                                     timestep_fn=lambda b, d, s: p.mcts_plan_timestep(b, d, s, NMAX, False)),
        "c": scenario.ScenarioRunner(sc, None, n_expansions_max=NMAX,
                                     states_fn=lambda *a: p.mcts_plan_timestep_from_states(
                                         *a[:-1], seeds=a[-1], n_expansions_max=NMAX, raise_on_search_error=False)),
    }
    for k in range(STEPS):
        for key, r in loops.items():
            t0 = time.perf_counter()
            r.step()
            if k >= WARM:
                times[key].append((time.perf_counter() - t0) * 1e3)
    for key in "bc":
        assert np.array_equal(loops["a"].pose, loops[key].pose) and np.array_equal(loops["a"].trim, loops[key].trim), seed
    fallbacks += loops["a"].n_fallbacks

# throughput: the first time step of 512 scenarios x 20 vehicles as one call
parts = []
for s in range(1, 513):
    r = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=s), None)
    r.k = 1   # the first time step: the seeds below are mcts_seeds(1, 20)
    iters, preds, fb = r.timestep_inputs()
    parts.append((SearchBatch.from_iters(iters, mpa.Hp, r.sc.checker, mpa.dt_seconds),
                  TimestepDeps.build(preds, [f[0] for f in fb], mpa.Hp)))
batch = SearchBatch.concat([b for b, _d in parts])
deps = TimestepDeps.concat([d for _b, d in parts], [b.n for b, _d in parts])
seeds = np.tile(scenario.mcts_seeds(1, 20), 512)
stream = torch.cuda.ExternalStream(p.stream())
first = p.mcts_plan_timestep(batch, deps, seeds, NMAX, False)
dev, wall, kern = [], [], []
for i in range(25):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    t0 = time.perf_counter()
    res = p.mcts_plan_timestep(batch, deps, seeds, NMAX, False)
    w = (time.perf_counter() - t0) * 1e3
    e1.record(stream)
    e1.synchronize()
    if i >= 5:
        dev.append(e0.elapsed_time(e1))
        wall.append(w)
        kern.append(p.stats().kernel_ms)
    assert np.array_equal(res.pop_hash, first.pop_hash)

res = {**gpu_info(), "n_expansions_max": NMAX,
       "closed_loops": {"vehicles": 20, "seeds": SEEDS, "steps": STEPS, "warm_steps_dropped": WARM,
                        "fallbacks": fallbacks,
                        "a_levels_mcts_plan_batch_step": pct(times["a"]),
                        "b_mcts_plan_timestep_step": pct(times["b"]),
                        "c_mcts_plan_timestep_from_states_step": pct(times["c"])},
       "throughput_first_step_512x20": {"rows": int(batch.n), "exhausted_rows": int(first.is_exhausted.sum()),
                                        "predecessor_edges": int(deps.pred_idx.size),
                                        "device_events": pct(dev), "kernel": pct(kern), "call_wall": pct(wall),
                                        "searches_per_s_device": batch.n / (np.median(dev) * 1e-3),
                                        "searches_per_s_wall": batch.n / (np.median(wall) * 1e-3)}}
print(json.dumps(res, indent=1))
if OUT:
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1)
p.close()
