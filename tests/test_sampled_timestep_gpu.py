"""Time steps with the sampled optimizer (pdmpc_mcts_plan_timestep, _closed_loop, _from_states) against their
specification: the level-by-level loop with host-side obstacle assembly, every level planned by the CPU oracle's
MonteCarloTreeSearch with Seed = time_step + vehicle_index (scenario.plan_timestep_by_levels with seeds;
PrioritizedController.m:297-352, :449-506, MonteCarloTreeSearch.m:31).  Bit-exact on every output field."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import mexfake
from oracle import oracle_py, parity
from pdmpc_b200 import capi, scenario
from pdmpc_b200.mpa import get_mpa
from pdmpc_b200.records import CHECKER_INTERX, CHECKER_SAT, BatchResult, SearchBatch, TimestepDeps

from helpers import rect, straight_iter
from test_mex_shim import _timestep_args
from test_timestep_gpu import concat_timesteps

pytestmark = pytest.mark.gpu

PLAN_TIMESTEP_SAMPLED = 13
NMAX = 250


def oracle_fn(mpa, nmax=NMAX):
    return lambda b, s: oracle_py.mcts_plan_batch(mpa, b, s, nmax, 4)


def spec(mpa, batch, deps, seeds, nmax=NMAX):
    return scenario.plan_timestep_by_levels(oracle_fn(mpa, nmax), batch, deps, seeds=seeds)


def closed_loop(planner, mpa, sc, steps):
    """Closed loop driven by pdmpc_mcts_plan_timestep; every step checked against the specification."""
    planner.upload_mpa(mpa)
    runner = scenario.ScenarioRunner(sc, None, n_expansions_max=NMAX,
                                     timestep_fn=lambda b, d, s: planner.mcts_plan_timestep(b, d, s, NMAX, False))
    tot = {"preds": 0, "exhausted": 0}
    for _ in range(steps):
        dev = runner.step_timestep()
        k, batch, deps, _ = runner.timestep_records[-1]
        ref = spec(mpa, batch, deps, scenario.mcts_seeds(k, batch.n))
        parity.compare(dev, ref)
        assert planner.stats().shape == 1
        tot["preds"] += int(deps.pred_idx.size)
        tot["exhausted"] += int(ref.is_exhausted.sum())
    return tot


def collect_timesteps(mpa, sc, steps):
    """(batch, deps, seeds, spec result) of every time step of an oracle-driven closed loop."""
    plan = oracle_fn(mpa)
    runner = scenario.ScenarioRunner(sc, None, n_expansions_max=NMAX,
                                     timestep_fn=lambda b, d, s: scenario.plan_timestep_by_levels(plan, b, d, seeds=s))
    runner.run(steps)
    return [(b, d, scenario.mcts_seeds(k, b.n), r) for k, b, d, r in runner.timestep_records]


def test_closed_loops_circle_sat_and_road_interx(planner):
    tot = []
    mpa = get_mpa("single_speed", non_convex=False)
    tot.append(closed_loop(planner, mpa, scenario.circle_scenario(mpa, 4), 30))
    for mpa_type, steps in (("single_speed", 12), ("triple_speed", 10)):
        mpa = get_mpa(mpa_type, non_convex=True)
        tot.append(closed_loop(planner, mpa, scenario.commonroad_scenario(mpa, 20, seed=2), steps))
    assert all(t["preds"] > 0 for t in tot)
    assert sum(t["exhausted"] for t in tot) > 0


@pytest.mark.parametrize("checker", [CHECKER_SAT, CHECKER_INTERX])
def test_chain_and_fallback_areas_of_exhausted_predecessor(planner, checker):
    """A chain 0 <- 1 <- 2 ... on parallel lines; vehicle 0 is blocked (exhausted) and publishes fallback areas that
    lie across vehicle 1's line; vehicle 5 has several unordered predecessors."""
    mpa = get_mpa("single_speed", non_convex=checker == CHECKER_INTERX)
    Hp, n = mpa.Hp, 24
    iters = [straight_iter(mpa, x=0.0, y=1.0 * i) for i in range(n)]
    iters[0].obstacles.append(rect(0.05, 0.0, 0.02, 0.3))      # crosses every first maneuver of vehicle 0
    batch = SearchBatch.from_iters(iters, Hp, checker, mpa.dt_seconds)
    preds = [[]] + [[i - 1] for i in range(1, n)]
    preds[5] = [4, 2, 0]
    fb = [None] * n
    fb[0] = [rect(0.5, 1.0, 0.05, 0.3)] * Hp
    deps = TimestepDeps.build(preds, fb, Hp)
    seeds = scenario.mcts_seeds(3, n)
    planner.upload_mpa(mpa)
    ref = spec(mpa, batch, deps, seeds)
    parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), ref)
    assert ref.is_exhausted[0] == 1
    free = oracle_py.mcts_plan_batch(mpa, SearchBatch.from_iters([iters[1]], Hp, checker, mpa.dt_seconds), seeds[1:2], NMAX)
    assert ref.pop_hash[1] != free.pop_hash[0]


def test_many_timesteps_in_one_call_forward_and_reversed(planner):
    """12 time steps x 20 vehicles of one closed loop in one call against the oracle, then the same searches in reversed
    index order (predecessors with higher indices than their successors).  The 512-scenario test below repeats the
    reversed order with more searches than can be resident."""
    mpa = get_mpa("triple_speed", non_convex=True)
    items = collect_timesteps(mpa, scenario.commonroad_scenario(mpa, 20, seed=3), 12)
    batch, deps, ref = concat_timesteps([(b, d, r) for b, d, _s, r in items])
    seeds = np.concatenate([s for _b, _d, s, _r in items])
    planner.upload_mpa(mpa)
    parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), ref)
    perm = np.arange(batch.n)[::-1].copy()
    inv = np.empty_like(perm)
    inv[perm] = np.arange(batch.n)
    rdeps = TimestepDeps.build([inv[deps.preds(int(i))] for i in perm], [deps.fallback_shapes(int(i)) for i in perm],
                               batch.Hp)
    rref = dataclasses.replace(ref, **{f.name: getattr(ref, f.name)[perm] for f in dataclasses.fields(ref)
                                       if isinstance(getattr(ref, f.name), np.ndarray)})
    parity.compare(planner.mcts_plan_timestep(batch.select(perm), rdeps, seeds[perm], NMAX, False), rref)


def test_equals_level_by_level_device_calls(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    for batch, deps, seeds, _ref in collect_timesteps(mpa, scenario.commonroad_scenario(mpa, 20, seed=5), 6):
        levels = scenario.plan_timestep_by_levels(lambda b, s: planner.mcts_plan_batch(b, s, NMAX, False), batch, deps,
                                                  seeds=seeds)
        parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), levels)


def _closed_loop_runner(planner, sc, path_id0=0):
    return scenario.ScenarioRunner(
        sc, None, inputs_fn=planner.sample_inputs, path_id0=path_id0, n_expansions_max=NMAX,
        closed_loop_fn=lambda b, d, sl, st, s: planner.mcts_plan_timestep_closed_loop(b, d, sl, st, s, NMAX, False))


def test_closed_loop_equals_the_host_fallback_loop(planner):
    """Fallback plans built and kept on the device == the host fallback logic with the oracle level by level; a call
    rejected for its parameters leaves the slots as they were."""
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    sc = scenario.commonroad_scenario(mpa, 20, seed=7)
    planner.upload_road(scenario.road_tables([sc]))
    planner.closed_loop_reset(20, scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01)
    dev = _closed_loop_runner(planner, sc)
    ref = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=7), oracle_fn(mpa), n_expansions_max=NMAX)
    for step in range(12):
        dev.step()
        ref.step()
        assert np.array_equal(dev.pose.view(np.uint64), ref.pose.view(np.uint64)), step
        assert np.array_equal(dev.trim, ref.trim)
        for i in range(20):
            for a, b in zip(dev.prev_shapes[i], ref.prev_shapes[i]):
                assert np.array_equal(a, b)
        if step == 5:   # rejected before anything runs: the next step still equals the reference
            _k, b, d, _r = dev.timestep_records[-1]
            with pytest.raises(capi.PdmpcError) as e:
                planner.mcts_plan_timestep_closed_loop(b, d, np.arange(20), np.zeros(20, np.uint8),
                                                       scenario.mcts_seeds(1, 20), 0)
            assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
    assert dev.n_fallbacks == ref.n_fallbacks


@pytest.mark.parametrize("amount,max_cls,seed", [(20, 99, 7), (40, 2, 3)])
def test_from_states_equals_the_closed_loop_path(planner, amount, max_cls, seed):
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    mk = lambda: scenario.commonroad_scenario(mpa, amount, seed=seed, allow_shared_paths=amount > 33)
    sc = mk()
    planner.upload_road(scenario.road_tables([sc]))
    planner.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
    hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
    planner.closed_loop_reset(amount, hl, hw)
    one = scenario.ScenarioRunner(sc, None, max_num_CLs=max_cls, n_expansions_max=NMAX,
                                  states_fn=lambda *a: planner.mcts_plan_timestep_from_states(
                                      *a[:-1], seeds=a[-1], n_expansions_max=NMAX, raise_on_search_error=False))
    res_one = [one.step_timestep() for _ in range(7)]
    planner.closed_loop_reset(amount, hl, hw)
    sep = scenario.ScenarioRunner(mk(), None, max_num_CLs=max_cls, inputs_fn=planner.sample_inputs,
                                  obstacles_fn=planner.assemble_obstacles, n_expansions_max=NMAX,
                                  closed_loop_fn=lambda b, d, sl, st, s: planner.mcts_plan_timestep_closed_loop(
                                      b, d, sl, st, s, NMAX, False))
    for k in range(7):
        parity.compare(res_one[k], sep.step_timestep())
    assert np.array_equal(one.pose.view(np.uint64), sep.pose.view(np.uint64)) and np.array_equal(one.trim, sep.trim)
    assert one.n_fallbacks == sep.n_fallbacks
    if max_cls >= amount:   # the host functions + oracle, level by level
        ref = scenario.ScenarioRunner(mk(), oracle_fn(mpa), n_expansions_max=NMAX)
        ref.run(7)
        assert np.array_equal(one.pose.view(np.uint64), ref.pose.view(np.uint64)) and np.array_equal(one.trim, ref.trim)


def test_512_scenarios_in_one_call_equal_their_separate_calls_forward_and_reversed(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    items = []
    for s in range(1, 513):
        r = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=s), None)
        r.k = 1
        iters, preds, fallbacks = r.timestep_inputs()
        b = SearchBatch.from_iters(iters, mpa.Hp, r.sc.checker, mpa.dt_seconds)
        d = TimestepDeps.build(preds, [f[0] for f in fallbacks], mpa.Hp)
        items.append((b, d, planner.mcts_plan_timestep(b, d, scenario.mcts_seeds(1, 20), NMAX, False)))
    batch, deps, ref = concat_timesteps(items)
    seeds = np.tile(scenario.mcts_seeds(1, 20), 512)
    # more searches than can ever be resident (an SM holds at most 32 CTAs), so warps take searches one after another
    import torch
    assert batch.n == 10240 > 32 * torch.cuda.get_device_properties(0).multi_processor_count
    parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), ref)
    # reversed index order: every predecessor now has a higher index than its successors, so only the topological
    # work order keeps a warp from waiting for a search that no resident warp has taken
    perm = np.arange(batch.n)[::-1].copy()
    inv = np.empty_like(perm)
    inv[perm] = np.arange(batch.n)
    rdeps = TimestepDeps.build([inv[deps.preds(int(i))] for i in perm], [deps.fallback_shapes(int(i)) for i in perm],
                               batch.Hp)
    rref = dataclasses.replace(ref, **{f.name: getattr(ref, f.name)[perm] for f in dataclasses.fields(ref)
                                       if isinstance(getattr(ref, f.name), np.ndarray)})
    parity.compare(planner.mcts_plan_timestep(batch.select(perm), rdeps, seeds[perm], NMAX, False), rref)


def test_input_errors(planner):
    mpa = get_mpa("single_speed", non_convex=True)
    planner.upload_mpa(mpa)
    Hp = mpa.Hp
    batch = SearchBatch.from_iters([straight_iter(mpa, y=float(i)) for i in range(3)], Hp, CHECKER_INTERX, mpa.dt_seconds)
    ok = TimestepDeps.build([[], [0], [1]], [None] * 3, Hp)
    seeds = scenario.mcts_seeds(1, 3)
    bad = [(TimestepDeps.build(p, [None] * 3, Hp), seeds, NMAX) for p in ([[1], [2], [0]], [[], [7], []], [[], [-1], []])]
    bad += [(ok, seeds, 0), (ok, seeds, 1024)]
    for d, s, nmax in bad:
        with pytest.raises(capi.PdmpcError) as e:
            planner.mcts_plan_timestep(batch, d, s, nmax)
        assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
    # NULL seeds with n > 0
    r = BatchResult.empty(batch.n, Hp)
    bi, bo = capi.batch_in(batch), capi.batch_out(r)
    dc = capi.TimestepDepsC(pred_ptr=capi._ptr(ok.pred_ptr, capi._p_i32), pred_idx=capi._ptr(ok.pred_idx, capi._p_i32))
    prm = capi.MctsParams(n_expansions_max=NMAX, seed=None)
    assert planner.lib.pdmpc_mcts_plan_timestep(planner.h, C.byref(bi), C.byref(dc), C.byref(prm), C.byref(bo)) == \
        capi.PDMPC_ERR_BAD_INPUT
    assert planner.lib.pdmpc_mcts_plan_timestep(planner.h, C.byref(bi), C.byref(dc), None, C.byref(bo)) == \
        capi.PDMPC_ERR_BAD_INPUT
    planner.upload_mpa(mpa)
    parity.compare(planner.mcts_plan_timestep(batch, ok, seeds, NMAX, False), spec(mpa, batch, ok, seeds))


def test_graph_search_time_step_after_a_sampled_one(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    batch, deps, seeds, ref = collect_timesteps(mpa, scenario.commonroad_scenario(mpa, 20, seed=4), 2)[-1]
    parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), ref)
    parity.compare(planner.plan_timestep(batch, deps, False),
                   scenario.plan_timestep_by_levels(lambda b: oracle_py.plan_batch(mpa, b), batch, deps))
    parity.compare(planner.mcts_plan_timestep(batch, deps, seeds, NMAX, False), ref)


def test_mex_command_matches_the_spec(built):
    matlab = mexfake.FakeMatlab()
    mpa = get_mpa("triple_speed", non_convex=True)
    steps = collect_timesteps(mpa, scenario.commonroad_scenario(mpa, 20, seed=6), 4)
    (h,) = matlab.call(1, mexfake.CREATE, 0.0)
    try:
        trans, man = mexfake.matlab_mpa(mpa)
        matlab.call(0, mexfake.UPLOAD_MPA, float(h), trans, man)
        for batch, deps, seeds, exp in steps:
            exh, n_exp, trims, y, shapes, g, hh = matlab.call(7, PLAN_TIMESTEP_SAMPLED, float(h), *_timestep_args(batch, deps),
                                                              seeds.astype(np.float64), float(NMAX))
            n, Hp = batch.n, batch.Hp
            assert exh.reshape(-1).astype(int).tolist() == exp.is_exhausted.tolist()
            assert n_exp.reshape(-1).astype(int).tolist() == exp.n_expanded.tolist()
            y = y.reshape(3, Hp, n, order="F")
            for i in range(n):
                if exp.is_exhausted[i]:
                    continue
                assert trims[i].astype(int).tolist() == exp.trims[i].tolist()
                assert np.array_equal(y[:, :, i].T.view(np.uint64), exp.y_predicted[i].view(np.uint64))
                assert np.array_equal(np.ascontiguousarray(g[i]).view(np.uint64), exp.g_path[i].view(np.uint64))
                assert np.array_equal(np.ascontiguousarray(hh[i]).view(np.uint64), exp.h_path[i].view(np.uint64))
                for k in range(Hp):
                    m = int(exp.shape_npts[i, k])
                    assert shapes[i + n * k].shape == (2, m)
                    assert np.array_equal(shapes[i + n * k][0].view(np.uint64), exp.shape_x[i, k, :m].view(np.uint64))
    finally:
        matlab.call(0, mexfake.DESTROY, float(h))
        matlab.clear_mex()
