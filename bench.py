#!/usr/bin/env python3
"""bench.py — vehicle-plans/sec of the MPA graph-search optimizer on B200.

Workload at N=1 (BASELINE.json configs[1]): CPM Lab road network, 20 vehicles,
coloring-based prioritisation, triple_speed MPA, Hp 6, InterX checker, 35 time
steps per scenario, R = 512 scenarios per GPU planned concurrently ("parallel_threads
equivalent on 1 B200"; 8 GPUs x 512 = the 4096 scenarios of configs[4]).  Scenarios are rolled out closed loop once (untimed) so
that every (scenario, step, vehicle) search record is fixed; one bench "step" =
one pass of the hot path over all records of the rank.  Both arms plan the SAME
records: they come from the same seeds, are rolled out by bit-identical planners
(GPU library / C oracle) and are shared through a per-user cache in the temporary
directory (never in the source tree, which may be read-only).

  value     : records already resident in HBM, search kernel timed with CUDA
              events on the library's stream, L2 flushed between steps.
  e2e       : same records through the C-ABI call pdmpc_plan_batch with HOST
              (pinned) buffers: H2D staging + kernels + D2H results inside the
              timed region.
  roofline  : algorithmic bytes of the search kernel (SURVEY.md §8d formula from
              the kernel's own counters) / its CUDA-event time vs measured HBM peak;
              plus the FP64-pipe and the warp-instruction-issue figures — the issue
              rate is the bound that actually bites.
  cpu_baseline : the C oracle (a port of the reference; MATLAB is not available)
              timed on this box's host cores on a bounded sample of the same records,
              plus the per-time-step latency of the CPU path (level by level).

`--impl reference` times that CPU implementation alone (all host threads).
`--scenarios-total T` fixes the total batch (BASELINE configs[4]: 4096) and splits it
over the ranks (strong scaling).  `--optimizer sampled` times the sampled optimizer
(MonteCarloTreeSearch) on the same records.  `--config explorative` runs BASELINE
configs[2] (8 priority permutations per time step, sharded over the GPUs) closed loop.
`--dump-outputs DIR` writes what the timed search returned in its last step as DIR/<field>.npy
(float64; a fixed sample of searches when all of them exceed 60 MB; with several GPUs DIR/rank<r>/
per rank, 60 MB over all ranks), so that two builds can be compared output for output on the same
records.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

BLOCK = 8            # scenarios per record-cache file (the unit of generation and of sharding)
LAT_SCENARIOS = 8    # scenarios whose time steps are replayed for the per-time-step latency (= block 0)
L2_NOTE = "GPU arm: flushed between timed steps (256 MiB write); CPU arm: not applicable"
DUMP_LIMIT = 60_000_000   # array bytes --dump-outputs writes over all ranks: under 64 MB with the .npy headers


def records_version() -> str:
    """Digest of what the rolled-out records depend on: the scenario generator, the record layout, both rollout
    planners (CUDA library, C oracle), the map and this file's rollout.  The cache is keyed on it, so a cached block
    is only read by the version of the project that wrote it."""
    import glob
    import hashlib
    files = [os.path.join(ROOT, "bench.py")]
    for pat in ("p-dmpc_b200/*.py", "p-dmpc_b200/data/*", "p-dmpc_b200/csrc/*.cu", "p-dmpc_b200/csrc/*.cuh",
                "p-dmpc_b200/csrc/*.h", "include/*.h", "oracle/pdmpc_oracle.[ch]"):
        files += sorted(glob.glob(os.path.join(ROOT, pat)))
    h = hashlib.sha256()
    for f in files:
        h.update(os.path.relpath(f, ROOT).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


# per user (the owner is checked before use) and per version, outside the source tree, which may be read-only
RECORD_CACHE_ROOT = os.path.join(tempfile.gettempdir(), f"pdmpc_bench_records_{os.getuid()}")
RECORD_CACHE = os.path.join(RECORD_CACHE_ROOT, records_version())


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="road", choices=["road", "explorative"],
                    help="road = BASELINE configs[1]/[4] (default); explorative = configs[2]")
    ap.add_argument("--optimizer", default="graph", choices=["graph", "sampled"],
                    help="graph = GraphSearch (default); sampled = MonteCarloTreeSearch")
    ap.add_argument("--scenarios", type=int, default=int(os.environ.get("PDMPC_BENCH_SCENARIOS", "512")),
                    help="scenarios per GPU (weak scaling; 512 = what BASELINE configs[4], 4096 scenarios, gives each of 8 GPUs)")
    ap.add_argument("--scenarios-total", type=int, default=0,
                    help="total scenarios, split block-cyclically over the ranks (strong scaling; BASELINE configs[4]: 4096)")
    ap.add_argument("--gen-workers", type=int, default=0,
                    help="processes that roll the scenarios out (0 = auto)")
    ap.add_argument("--sim-steps", type=int, default=35)
    ap.add_argument("--vehicles", type=int, default=20)
    ap.add_argument("--mpa", default="triple_speed")
    ap.add_argument("--no-cache", action="store_true", help=f"do not read/write the record cache ({RECORD_CACHE})")
    ap.add_argument("--cpu-sample", type=int, default=0, help="searches in the CPU sample (0 = auto)")
    ap.add_argument("--pipeline-chunks", type=int, default=0,
                    help="chunks of the e2e call's copy/search pipeline (0 = library default, 1 = off)")
    ap.add_argument("--permutations", type=int, default=8, help="--config explorative: priority permutations per time step")
    ap.add_argument("--mcts-expansions", type=int, default=250, help="--optimizer sampled: n_expansions_max")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<field>.npy (float64, under 64 MB)")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "ours" or a.config != "road"):
        ap.error("--dump-outputs covers the timed search of the GPU arm (--impl ours, --config road)")
    for v in (a.scenarios, a.scenarios_total):
        if v % BLOCK:
            ap.error(f"scenario counts must be multiples of {BLOCK}")
    return a


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), \
        int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------- records
def block_path(args, block: int) -> str:
    return os.path.join(RECORD_CACHE, f"{args.mpa}_{args.vehicles}v_{args.sim_steps}t_block{block:04d}.npz")


def _roll_block(job):
    """Worker process: roll one block of BLOCK scenarios (seeds 1 + BLOCK*block ...) out closed loop.
    planner 'gpu': its own GPU planner; 'oracle': the C oracle (one thread) — bit-identical plans, hence
    identical records.  Block 0 also keeps the level structure and the one-call inputs of its time steps."""
    kind, dev, mpa_type, vehicles, sim_steps, block, out_path = job
    import pickle
    from pdmpc_b200 import scenario
    from pdmpc_b200.mpa import get_mpa
    from pdmpc_b200.records import SearchBatch, TimestepDeps
    mpa = get_mpa(mpa_type, non_convex=True)
    planner = None
    if kind == "gpu":
        from pdmpc_b200 import capi
        planner = capi.Planner(dev)
        planner.upload_mpa(mpa)
        plan = planner.plan_batch
    else:
        from oracle import oracle_py
        plan = lambda b: oracle_py.plan_batch(mpa, b, 1)   # noqa: E731
    batches, levels, timesteps = [], [], []
    for si in range(BLOCK):
        sc = scenario.commonroad_scenario(mpa, vehicles, seed=1 + BLOCK * block + si)
        runner = scenario.ScenarioRunner(sc, plan)
        if block == 0 and si < LAT_SCENARIOS:
            for _ in range(sim_steps):
                iters, preds, fbs = runner.timestep_inputs()
                timesteps.append((si * 100000 + runner.k + 1,
                                  SearchBatch.from_iters(iters, mpa.Hp, sc.checker, mpa.dt_seconds),
                                  TimestepDeps.build(preds, [f[0] for f in fbs], mpa.Hp)))
                runner.step()
            recs = runner.records
            levels.extend((si * 100000 + r.step, r.level, r.batch.n) for r in recs)
        else:
            recs = runner.run(sim_steps)
        batches.extend(r.batch for r in recs)
    if planner is not None:
        planner.close()
    os.makedirs(os.path.dirname(out_path), exist_ok=True)
    tmp = out_path + f".tmp{os.getpid()}.npz"
    SearchBatch.concat(batches).save(tmp)
    if block == 0:
        np.save(out_path + ".levels.npy", np.array(levels, dtype=np.int64))
        with open(out_path + ".ts.pkl", "wb") as f:
            pickle.dump(timesteps, f)
    os.replace(tmp, out_path)
    return out_path


def rank_blocks(args, rank: int, world: int):
    """Blocks of BLOCK scenarios this rank owns.  Weak scaling: `--scenarios` per rank, consecutive;
    strong scaling (`--scenarios-total`): all blocks dealt block-cyclically."""
    if args.scenarios_total:
        return [b for b in range(args.scenarios_total // BLOCK) if b % world == rank]
    per = args.scenarios // BLOCK
    return list(range(rank * per, (rank + 1) * per))


def get_records(args, blocks, kind: str, dev: int, workers: int):
    """Flat batch of every search record of `blocks` (+ level structure and one-call inputs of block 0 when
    it is among them).  Missing blocks are rolled out by `workers` processes and cached in RECORD_CACHE."""
    import pickle
    import multiprocessing as mp
    from pdmpc_b200.records import SearchBatch
    if not args.no_cache:
        os.makedirs(RECORD_CACHE_ROOT, mode=0o700, exist_ok=True)
        if os.stat(RECORD_CACHE_ROOT).st_uid != os.getuid():   # the cache holds pickles: read only our own
            raise SystemExit(f"{RECORD_CACHE_ROOT} belongs to another user; run with --no-cache")
        os.makedirs(RECORD_CACHE, mode=0o700, exist_ok=True)
    tmpdir = tempfile.mkdtemp(prefix="pdmpc_gen_") if args.no_cache else None
    path = (lambda b: os.path.join(tmpdir, f"block{b:04d}.npz")) if tmpdir else (lambda b: block_path(args, b))
    todo = [b for b in blocks if not os.path.exists(path(b)) or
            (b == 0 and not os.path.exists(path(b) + ".ts.pkl"))]
    if todo:
        jobs = [(kind, dev, args.mpa, args.vehicles, args.sim_steps, b, path(b)) for b in todo]
        w = max(1, min(workers, len(jobs)))
        if w == 1:
            for j in jobs:
                _roll_block(j)
        else:
            with mp.get_context("spawn").Pool(w) as pool:
                pool.map(_roll_block, jobs, chunksize=1)
    batch = SearchBatch.concat([SearchBatch.load(path(b)) for b in blocks])
    levels, timesteps = np.zeros((0, 3), dtype=np.int64), []
    if 0 in blocks:
        levels = np.load(path(0) + ".levels.npy")
        timesteps = pickle.load(open(path(0) + ".ts.pkl", "rb"))
    if tmpdir:
        import shutil
        shutil.rmtree(tmpdir, ignore_errors=True)
    return batch, levels, timesteps


def dump_outputs(res, out_dir: str, limit: int) -> None:
    """The BatchResult of the timed path (what pdmpc_fetch_staged hands a caller), one DIR/<field>.npy per field, in
    float64: every integer field is exact in it, the 64-bit pop-order hash is split into two 32-bit halves.  When all
    searches do not fit in `limit` bytes, a fixed sample of them (seed 0, ascending; DIR/rows.npy lists it) is written.
    An exhausted search has no plan: its poses and costs are NaN and are written as 0 (is_exhausted marks those rows).
    Any other value that is not finite is a wrong result and raises."""
    import dataclasses
    exhausted = res.is_exhausted.astype(bool)
    fields = {}
    for f in dataclasses.fields(res):
        a = getattr(res, f.name)
        if not isinstance(a, np.ndarray):
            continue
        if a.dtype == np.uint64:
            fields[f.name + "_hi"] = (a >> np.uint64(32)).astype(np.float64)
            fields[f.name + "_lo"] = (a & np.uint64(0xFFFFFFFF)).astype(np.float64)
        else:
            a = a.astype(np.float64)          # a copy: the caller's result stays as the library returned it
            a[exhausted] = np.nan_to_num(a[exhausted], nan=0.0, posinf=np.inf, neginf=-np.inf)
            if not np.isfinite(a).all():
                bad = np.argwhere(~np.isfinite(a))[0]
                raise RuntimeError(f"--dump-outputs: {f.name} is not finite at {tuple(bad)}")
            fields[f.name] = a
    n = res.status.size
    row_bytes = 8 * (1 + sum(a[:1].size for a in fields.values()))    # + the row index itself
    m = min(n, limit // row_bytes)
    rows = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    for name, a in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows])


def workload_config(args, world: int, n: int, Hp: int) -> dict:
    """`config` of the JSON line — identical in both arms (same records)."""
    if args.scenarios_total:
        size = (f"{args.scenarios_total} scenarios in total (BASELINE configs[4]) split block-cyclically over "
                f"{world} GPU(s) x {args.sim_steps} steps")
    else:
        size = f"{args.scenarios} scenarios/GPU x {args.sim_steps} steps"
    opt = "" if args.optimizer == "graph" else f", sampled optimizer (MonteCarloTreeSearch, n_expansions_max {args.mcts_expansions})"
    return {"workload": f"CPM Lab road network (BASELINE configs[1]), {args.vehicles} vehicles, coloring priorities, "
                        f"{args.mpa} MPA, Hp {Hp}, InterX checker{opt}, {size}, pre-rolled closed loop "
                        f"(seeds 1.., same records in both arms)",
            "searches_per_step_per_gpu": n, "l2": L2_NOTE}


def algorithmic_bytes(batch, stats, Hp: int) -> float:
    """SURVEY.md §8(d): B_in + 80*M + 80*P + B_out per search, summed over the batch.
    The per-pop obstacle re-read term is counted separately (obstacle columns are
    L1/L2 resident, not HBM traffic)."""
    b_in = batch.input_bytes()
    b_out = batch.n * (8 * (Hp * (4 + 2 * 7)) + 16)
    return float(b_in + 80 * stats.total_nodes + 80 * stats.total_pops + b_out)


def fp64_ops(batch, stats, Hp: int) -> float:
    """FP64 instructions (mul/add/sqrt, no FMA) the algorithm needs: per pop the
    sin/cos (2 x ~45) and shape placement (~6 pts x 2 shapes x 6), per obstacle
    column tested ~6 edges x 5 ops (C1 pass of InterX), per created node pose+g+h
    (~12 + 8 + 9*(Hp-1)/2)."""
    return float(stats.total_pops * (90 + 72) + stats.total_obstacle_cols * 30 +
                 stats.total_nodes * (20 + 9 * (Hp - 1) / 2))


def states_latency(planner, mpa, args, n_scenarios: int = 4, steps: int = 35):
    """Wall time of pdmpc_plan_timestep_from_states per 20-vehicle time step over live closed loops (seeds 1..)."""
    from pdmpc_b200 import scenario
    hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
    planner.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
    ts, fallbacks = [], 0
    for seed in range(1, 1 + n_scenarios):
        sc = scenario.commonroad_scenario(mpa, args.vehicles, seed=seed)
        planner.upload_road(scenario.road_tables([sc]))
        planner.closed_loop_reset(args.vehicles, hl, hw)

        def call(*a):
            t0 = time.perf_counter()
            r = planner.plan_timestep_from_states(*a, raise_on_search_error=False)
            ts.append((time.perf_counter() - t0) * 1e3)
            return r

        runner = scenario.ScenarioRunner(sc, None, states_fn=call)
        for _ in range(steps):
            runner.step_timestep()
        fallbacks += runner.n_fallbacks
    t = np.array(ts)
    return {"p50": float(np.percentile(t, 50)), "p99": float(np.percentile(t, 99)), "max": float(t.max()), "n": int(t.size),
            "fallback_plans": int(fallbacks),
            "what": "wall time of ONE pdmpc_plan_timestep_from_states call per 20-vehicle time step: inputs, obstacle "
                    "assembly, dependency-ordered searches and fallback plans on the device, measured states in, plans out; "
                    f"live closed loops of {n_scenarios} scenarios"}


def cpu_timestep_latency(mpa, batch, step_recs, cores: int, reps: int = 2):
    """BASELINE.md §2 "CPU-step": wall time of one 20-vehicle time step on the CPU path the way the
    reference's parallel_threads mode runs it — computation levels one after the other, the vehicles of
    a level on parallel threads (PrioritizedSequentialController.m:74-92) — over the time steps of the
    first LAT_SCENARIOS scenarios (the same steps the GPU latency replays)."""
    from oracle import oracle_py
    by_step, off = {}, 0
    for step, _level, cnt in step_recs:
        by_step.setdefault(int(step), []).append(batch.select(np.arange(off, off + int(cnt))))
        off += int(cnt)
    lat = []
    for rep in range(reps + 1):
        for _k, levels in sorted(by_step.items()):
            t0 = time.perf_counter()
            for lb in levels:
                oracle_py.plan_batch(mpa, lb, min(cores, lb.n))
            if rep:
                lat.append((time.perf_counter() - t0) * 1e3)
    if not lat:
        return None
    return {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)), "max": float(np.max(lat)),
            "n": len(lat), "levels_per_step": float(np.mean([len(v) for v in by_step.values()])),
            "what": f"wall time of one {int(sum(b.n for b in next(iter(by_step.values()))))}-vehicle time step on the CPU "
                    f"path: computation levels one after the other, the vehicles of a level on up to {cores} threads"}


# ---------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path (C oracle port; the MATLAB reference cannot
    run here) on all host threads, over the records of rank 0 of the GPU arm — the same seeds, hence
    byte-identical search records; each step plans all of them (or a stated prefix on a slow host)."""
    if rank != 0:
        return
    import __graft_entry__ as entry
    from oracle import oracle_py
    from pdmpc_b200.mpa import get_mpa
    entry.build_oracle()
    mpa = get_mpa(args.mpa, non_convex=True)
    cores = os.cpu_count() or 1
    t_gen = time.perf_counter()
    batch, step_recs, _ts = get_records(args, rank_blocks(args, 0, world), "oracle", 0, args.gen_workers or cores)
    t_gen = time.perf_counter() - t_gen
    n = batch.n
    if args.optimizer == "sampled":
        seeds = (np.arange(n) % 35 + 2).astype(np.uint32)
        plan = lambda b, s=None: oracle_py.mcts_plan_batch(mpa, b, seeds[: b.n], args.mcts_expansions, cores)   # noqa: E731
    else:
        plan = lambda b: oracle_py.plan_batch(mpa, b, cores)   # noqa: E731
    # bounded: the whole run (warmup + steps passes) within ~3 minutes
    probe = batch.select(np.arange(min(n, 8000)))
    t0 = time.perf_counter()
    plan(probe)
    rate = probe.n / max(time.perf_counter() - t0, 1e-6)
    passes = args.steps + args.warmup
    m = int(min(n, max(2000, rate * 180.0 / max(passes, 1))))
    sample = batch if m == n else batch.select(np.arange(m))
    for _ in range(args.warmup):
        plan(sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        plan(sample)
    el = time.perf_counter() - t0
    val = sample.n * args.steps / el
    desc = (f"all {n} search records of GPU rank 0 per step" if m == n else
            f"first {m} of the {n} search records of GPU rank 0 per step (slow host: bounded to ~3 min)")
    lat = cpu_timestep_latency(mpa, batch, step_recs, cores) if args.optimizer == "graph" else None
    print(json.dumps({
        "impl": "reference", "metric": "vehicle-plans/sec", "value": val, "unit": "plans/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": el / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.scenarios_total else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world, n, mpa.Hp),
        "cpu_baseline": {"value": val, "unit": "plans/s", "cores": cores, "kind": "port", "sample": desc,
                         "latency_ms_per_timestep": lat,
                         "note": "C oracle (gcc -O2, no FMA contraction) restating the MATLAB reference, one pthread per "
                                 "host core pulling searches from a shared counter (parallel_threads equivalent); "
                                 "MATLAB R2023a itself is unavailable in this image"},
        "e2e": {"value": val, "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "record_generation_s": round(t_gen, 1),
    }))


# ---------------------------------------------------------------------------- GPU arm
def captured_kernel_figures(n: int, mpa: str, shape: int):
    """DRAM traffic and warp instructions of ONE launch of the dominant kernel, from the committed
    `ncu --set full` capture of this same launch (tools/gpu_round.sh writes profiles/search_kernel_traffic.json
    from the capture of the bench's own records); None when the workload or the launch shape differs."""
    try:
        cap = json.load(open(os.path.join(ROOT, "profiles", "search_kernel_traffic.json")))
        if int(cap.get("searches", -1)) == n and cap.get("mpa") == mpa and int(cap.get("shape", shape)) == shape:
            return cap
    except Exception:
        pass
    return None


def main():
    args = parse_args()
    rank, local_rank, world = dist_env()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry
    if rank == 0:
        entry.build()
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    if args.config == "explorative":
        from pdmpc_b200 import bench_explorative
        bench_explorative.run(args, rank, local_rank, world, ClockSampler)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    from pdmpc_b200 import capi
    from pdmpc_b200.mpa import get_mpa
    from pdmpc_b200.records import BatchResult

    dev = local_rank if world > 1 else 0
    torch.cuda.set_device(dev)
    planner = capi.Planner(dev)        # raises if the CUDA library / device is missing
    mpa = get_mpa(args.mpa, non_convex=True)
    planner.upload_mpa(mpa)
    planner.set_cta_queue(True)   # what the MATLAB drop-in selects: valid-only queue wherever the CTA shape runs
    Hp = mpa.Hp

    t_gen = time.perf_counter()
    workers = args.gen_workers or max(1, (os.cpu_count() or 1) // max(world, 1))
    batch, step_recs, ts_recs = get_records(args, rank_blocks(args, rank, world), "gpu", dev, workers)
    t_gen = time.perf_counter() - t_gen
    n = batch.n
    sampled = args.optimizer == "sampled"
    seeds = (np.arange(n) % 35 + 2).astype(np.uint32)

    stream = torch.cuda.ExternalStream(planner.stream(), device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{dev}")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_staged():
        if sampled:
            planner.mcts_run_staged(seeds, args.mcts_expansions)
        else:
            planner.run_staged()

    # ---- device-resident throughput ("value") ------------------------------------
    planner.stage(batch)
    for _ in range(max(args.warmup, 3)):
        run_staged()
    planner.sync()
    launches_per_step = int(planner.stats().kernel_launches)
    sampler = ClockSampler(dev)
    barrier()
    sampler.start()
    kernel_ms = []
    for _ in range(args.steps):
        with torch.cuda.stream(stream):
            flush.zero_()                     # L2 flush, outside the per-step events
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run_staged()
            e1.record(stream)
        e1.synchronize()
        kernel_ms.append(e0.elapsed_time(e1))
    barrier()
    clocks = sampler.stop()
    res = planner.fetch()
    if args.dump_outputs:
        # each rank holds its own records: with several GPUs, DIR/rank<r>/ per rank, the byte budget split evenly
        dump_outputs(res, args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"),
                     DUMP_LIMIT // world)
    stats = planner.stats()
    shape = int(stats.shape)
    ms_step = float(np.mean(kernel_ms))
    t_local = torch.tensor([sum(kernel_ms)], dtype=torch.float64, device=f"cuda:{dev}")
    n_all = torch.tensor([n], dtype=torch.int64, device=f"cuda:{dev}")
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_all, op=dist.ReduceOp.SUM)
    total_ms = float(t_local.item())
    n_total = int(n_all.item())
    value = n_total * args.steps / (total_ms * 1e-3)

    # ---- end to end through the C ABI with host buffers ("e2e") ------------------
    import dataclasses
    import ctypes as C
    pinned = []   # keep the pinned torch storages alive

    def pinned_like(a: np.ndarray) -> np.ndarray:
        t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
        pinned.append(t)
        return t.numpy()[: a.nbytes].view(a.dtype).reshape(a.shape)

    host_in = {}
    for f in dataclasses.fields(batch):
        a = getattr(batch, f.name)
        if isinstance(a, np.ndarray):
            host_in[f.name] = pinned_like(a)
            host_in[f.name][...] = a
    hb = dataclasses.replace(batch, **host_in)
    out = BatchResult.empty(n, Hp)
    for f in dataclasses.fields(out):
        a = getattr(out, f.name)
        if isinstance(a, np.ndarray):
            setattr(out, f.name, pinned_like(a))
    bi, bo = capi.batch_in(hb), capi.batch_out(out)
    prm, prm_keep = capi.mcts_params(seeds, args.mcts_expansions, n)
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_call():
        if sampled:
            planner._check(planner.lib.pdmpc_mcts_plan_batch(planner.h, C.byref(bi), C.byref(prm), C.byref(bo)))
        else:
            planner._check(planner.lib.pdmpc_plan_batch(planner.h, C.byref(bi), C.byref(bo)))

    def time_e2e(chunks: int, steps: int) -> float:
        planner.set_pipeline_chunks(chunks)
        for _ in range(2):
            e2e_call()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_call()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=f"cuda:{dev}")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert np.array_equal(out.pop_hash, res.pop_hash), "e2e path and staged path disagree"
        assert np.array_equal(out.trims, res.trims), "e2e path and staged path disagree"
        return n_total * steps / float(t.item())

    e2e_serial = None if sampled else time_e2e(1, 3)   # copy in, search, copy out, one after the other
    e2e_val = time_e2e(args.pipeline_chunks, e2e_steps)   # the library's default: chunked pipeline
    st2 = planner.stats()
    planner.set_pipeline_chunks(0)

    # ---- per-time-step latency (levels sequential, host buffers) -----------------
    # What the drop-in does for one 20-vehicle time step: one pdmpc_plan_batch call per
    # computation level (host buffers in, host buffers out), levels one after the other.
    # Replayed for the first LAT_SCENARIOS scenarios of rank 0, whose records come first.
    lat, lat1 = [], []
    lat_levels = 0
    if rank == 0 and not sampled and len(step_recs):
        by_step, off = {}, 0
        for step, _level, cnt in step_recs:
            lb = batch.select(np.arange(off, off + int(cnt)))
            ro = BatchResult.empty(lb.n, Hp)
            by_step.setdefault(int(step), []).append((lb, ro, capi.batch_in(lb), capi.batch_out(ro)))
            off += int(cnt)
        lat_levels = float(np.mean([len(v) for v in by_step.values()]))
        for rep in range(3):
            for k, levels in sorted(by_step.items()):
                t0 = time.perf_counter()
                for _lb, _ro, lbi, lbo in levels:
                    planner._check(planner.lib.pdmpc_plan_batch(planner.h, C.byref(lbi), C.byref(lbo)))
                if rep:
                    lat.append((time.perf_counter() - t0) * 1e3)

        # ---- the same time steps, ONE call each (pdmpc_plan_timestep) ------------------------------
        # Base iter_v of all 20 vehicles + predecessor lists + fallback areas in, all plans out: one
        # H2D, one dependency-ordered launch (searches wait for their own predecessors' flags), one D2H.
        calls = []
        for step, tb, td in ts_recs:
            ro = BatchResult.empty(tb.n, Hp)
            pidx = td.pred_idx if td.pred_idx.size else np.zeros(1, dtype=np.int32)
            dc = capi.TimestepDepsC(pred_ptr=capi._ptr(td.pred_ptr, capi._p_i32), pred_idx=capi._ptr(pidx, capi._p_i32),
                                    fb_npts=capi._ptr(td.fb_npts, capi._p_i32), fb_x=capi._ptr(td.fb_x, capi._p_f64),
                                    fb_y=capi._ptr(td.fb_y, capi._p_f64))
            calls.append((int(step), tb, td, pidx, ro, capi.batch_in(tb), dc, capi.batch_out(ro)))
        for rep in range(3):
            for _step, _tb, _td, _pidx, _ro, tbi, tdc, tbo in calls:
                t0 = time.perf_counter()
                planner._check(planner.lib.pdmpc_plan_timestep(planner.h, C.byref(tbi), C.byref(tdc), C.byref(tbo)))
                if rep:
                    lat1.append((time.perf_counter() - t0) * 1e3)
        # same searches, same answers as the level-by-level replay above (pop-order hashes per time step)
        for step, _tb, _td, _pidx, ro, *_ in calls:
            a = np.sort(np.concatenate([r.pop_hash for _lb, r, _i, _o in by_step[step]]))
            assert np.array_equal(a, np.sort(ro.pop_hash)), f"time step {step}: one-call path != level-by-level path"

    # ---- the whole time step from the measured states, ONE call (pdmpc_plan_timestep_from_states) -----------------
    # Inputs (reference trajectories, lanelet boundaries), obstacle assembly, dependency-ordered searches and fallback
    # plans chained on the device; the host only decides coupling and priorities.  A live closed loop over the first
    # scenarios of rank 0 (the latency legs above replay recorded time steps); only the device call is timed.
    lat_states = None
    if rank == 0 and not sampled and len(step_recs):
        try:
            lat_states = states_latency(planner, mpa, args)
        except Exception as e:   # a diagnostic leg: it must never take the bench line down
            lat_states = {"error": f"{type(e).__name__}: {e}"}
        planner.upload_mpa(mpa)

    # ---- CPU baseline beside it (rank 0, N=1 only) -------------------------------
    cpu = None
    if rank == 0 and world == 1:
        from oracle import oracle_py, parity
        cores = os.cpu_count() or 1
        m = args.cpu_sample or min(n, 4000 if sampled else 14000)
        sample = batch.select(np.arange(m))
        t0 = time.perf_counter()
        if sampled:
            ref = oracle_py.mcts_plan_batch(mpa, sample, seeds[:m], args.mcts_expansions, cores)
        else:
            ref = oracle_py.plan_batch(mpa, sample, cores, hash_valid_pops_only=True)
        t_cpu = time.perf_counter() - t0
        m1 = min(m, 500 if sampled else 2000)
        t0 = time.perf_counter()
        if sampled:
            oracle_py.mcts_plan_batch(mpa, batch.select(np.arange(m1)), seeds[:m1], args.mcts_expansions, 1)
        else:
            oracle_py.plan_batch(mpa, batch.select(np.arange(m1)), 1)
        t_cpu1 = time.perf_counter() - t0
        # parity of the timed outputs against the checker, on the sample
        sub = dataclasses.replace(res, **{f.name: getattr(res, f.name)[:m] for f in dataclasses.fields(res)
                                          if isinstance(getattr(res, f.name), np.ndarray)})
        parity.compare(sub, ref)
        cpu = {"value": m / t_cpu, "unit": "plans/s", "cores": cores, "kind": "port",
               "sample": f"first {m} of the {n} timed search records, one pass, {cores} threads",
               "single_thread_plans_per_s": m1 / t_cpu1,
               "parity_checked": True,
               "latency_ms_per_timestep": (cpu_timestep_latency(mpa, batch, step_recs, cores)
                                           if not sampled and len(step_recs) else None),
               "note": "C oracle restating the MATLAB reference (MATLAB R2023a unavailable here)"}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        kname = ("pdmpc::mcts_kernel" if sampled else
                 {1: "pdmpc::search_kernel", 2: "pdmpc::search_tile_kernel<16,...>", 3: "pdmpc::search_tile_kernel<8,...>",
                  4: "pdmpc::search_cta_kernel", 5: "pdmpc::search_cta_kernel"}.get(shape, "pdmpc::search_kernel"))
        cap = None if sampled else captured_kernel_figures(n, args.mpa, shape)
        traffic = float(cap["dram_bytes_read"]) + float(cap["dram_bytes_write"]) if cap else None
        fp64_peak = planner.measure_fp64_peak()
        alg_bytes = algorithmic_bytes(batch, stats, Hp)
        achieved = alg_bytes / (ms_step * 1e-3) / 1e9
        f64 = fp64_ops(batch, stats, Hp)
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic,
                "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)",
                "kernel": kname, "launch_shape": shape, "algorithmic_bytes_per_launch": alg_bytes,
                "note": "neither HBM nor the FP64 pipe binds; the search is a chain of dependent instructions per "
                        "search, see `issue` and DESIGN.md §4.1"}
        if not sampled:
            roof["fp64"] = {"ops_per_launch": f64, "achieved_tops": f64 / (ms_step * 1e-3) / 1e12,
                            "peak_tops_mul_add": fp64_peak[0], "peak_tflops_fma": fp64_peak[1],
                            "frac": f64 / (ms_step * 1e-3) / 1e12 / fp64_peak[0],
                            "peak_source": "measured in this run (pdmpc_measure_fp64_peak, register-only kernel)",
                            "note": "mul/add/sqrt without FMA"}
            if cap and cap.get("warp_instructions") and cap.get("pops"):
                # warp instructions per pop from the ncu capture of this launch x this run's pops / this run's time,
                # against 4 warp instructions per clock per SM (one per scheduler)
                sm_clk = (clocks.get("sm_mhz") or 1965.0) * 1e6
                n_sm = int(cap.get("sms", 148))
                inst = float(cap["warp_instructions"]) / float(cap["pops"]) * stats.total_pops
                roof["issue"] = {"warp_inst_per_pop": float(cap["warp_instructions"]) / float(cap["pops"]),
                                 "warp_inst_per_launch": inst,
                                 "achieved_ginst_s": inst / (ms_step * 1e-3) / 1e9,
                                 "peak_ginst_s": 4.0 * n_sm * sm_clk / 1e9,
                                 "frac": inst / (ms_step * 1e-3) / (4.0 * n_sm * sm_clk),
                                 "source": f"smsp__inst_executed.sum of the {cap.get('round', '?')} ncu capture "
                                           "(profiles/search_kernel_traffic.json), 4 issue slots/clk/SM"}
        line = {
            "metric": "vehicle-plans/sec", "value": value, "unit": "plans/s", "n_gpus": world,
            "steps": len(kernel_ms), "warmup": max(args.warmup, 3), "ms_per_step": total_ms / len(kernel_ms),
            "higher_is_better": True, "scaling": "strong" if args.scenarios_total else "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world, n, Hp),
            "e2e": {"value": e2e_val, "unit": "plans/s", "h2d_bytes_per_step": int(st2.h2d_bytes),
                    "d2h_bytes_per_step": int(st2.d2h_bytes), "steps": e2e_steps,
                    "pipeline": "chunked copy/search overlap inside pdmpc_plan_batch (pdmpc_set_pipeline_chunks "
                                f"{args.pipeline_chunks}: 0 = library default)",
                    "value_without_pipeline": e2e_serial,
                    "h2d_ms": st2.h2d_ms, "kernel_ms": st2.kernel_ms, "d2h_ms": st2.d2h_ms},
            "gpu_launches": int(args.steps * launches_per_step),   # persistent search kernel(s) per timed step (staged path)
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "search_stats": {"pops_per_plan": stats.total_pops / max(n, 1),
                             "nodes_per_plan": stats.total_nodes / max(n, 1),
                             "exhausted_frac": float(res.is_exhausted.mean()),
                             "obstacle_cols_per_pop": stats.total_obstacle_cols / max(stats.total_pops, 1),
                             "max_pops": int(res.n_pops.max()), "searches_total": n_total,
                             "escalated_to_cta_shape": int(stats.escalated)},
            "latency_ms_per_timestep": ({"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)),
                                         "max": float(np.max(lat)), "n": len(lat), "levels_per_step": lat_levels,
                                         "what": "wall time of all computation levels of one 20-vehicle time step, one "
                                                 "pdmpc_plan_batch call per level, host buffers in and out"}
                                        if lat else None),
            "latency_ms_per_timestep_one_call": ({"p50": float(np.percentile(lat1, 50)), "p99": float(np.percentile(lat1, 99)),
                                                  "max": float(np.max(lat1)), "n": len(lat1),
                                                  "what": "wall time of ONE pdmpc_plan_timestep call per 20-vehicle time "
                                                          "step (predecessor hand-over on the device), host buffers in "
                                                          "and out; same time steps and answers as above"}
                                                 if lat1 else None),
            "latency_ms_per_timestep_from_states": lat_states,
            "record_generation_s": round(t_gen, 1),
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    planner.close()


if __name__ == "__main__":
    main()
