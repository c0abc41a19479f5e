"""pdmpc_plan_timestep_explorative (DESIGN.md §4.13): all permutations of all scenarios planned from the measured states,
chosen per weakly connected sub-graph and committed to the closed-loop slots in one call, equal bit for bit to
ExplorativeRunner's host path (pdmpc_plan_timestep per time step + the host exchange, sharding.solution_costs) and to
the oracle; every input error is loud and leaves the slots as they were."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

from oracle import oracle_py, parity
from pdmpc_b200 import capi, scenario
from pdmpc_b200.mpa import get_mpa

pytestmark = pytest.mark.gpu

HL, HW = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
ROAD_SEED = 3   # 20 vehicles: a step with >= 3 permutations and exhausted rows within the first 7 steps


def bits(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64)).view(np.uint64)


def rows(res, idx):
    return dataclasses.replace(res, **{f.name: getattr(res, f.name)[idx] for f in dataclasses.fields(res)
                                       if isinstance(getattr(res, f.name), np.ndarray)})


def explorative_fn(planner):
    return lambda *a, **k: planner.plan_timestep_explorative(*a, **k, raise_on_search_error=False)


def setup(planner, scs, n_slots=None):
    mpa = scs[0].mpa
    planner.upload_mpa(mpa)
    planner.upload_road(scenario.road_tables(scs))
    planner.closed_loop_reset(n_slots or sum(s.amount for s in scs), HL, HW)


def compare_step(dev, host, fallbacks):
    """One time step of the device call against the host path: the choice, every planned row, the exhausted rows'
    fallback plans and the closed-loop state."""
    a, b = dev.explorative_records[-1], host.explorative_records[-1]
    assert a["n_permutations"] == b["n_permutations"] and a["n_levels"] == b["n_levels"]
    assert np.array_equal(a["chosen"], b["chosen"])
    assert a["solution_cost"].shape == b["solution_cost"].shape and np.array_equal(bits(a["solution_cost"]), bits(b["solution_cost"]))
    ra, rb = a["result_local"], b["result_local"]
    assert np.array_equal(ra.is_exhausted, rb.is_exhausted)
    planned = np.flatnonzero(ra.is_exhausted == 0)
    parity.compare(rows(ra, planned), rows(rb, planned))
    n = dev.sc.amount
    for r in np.flatnonzero(ra.is_exhausted):
        shapes, traj, trims = fallbacks[r % n]
        assert np.array_equal(ra.trims[r, 1:], trims)
        assert np.array_equal(bits(ra.y_predicted[r]), bits(traj))
        for got, want in zip(ra.shapes(r), shapes):
            assert np.array_equal(bits(got), bits(want))
    assert np.array_equal(bits(dev.pose), bits(host.pose)) and np.array_equal(dev.trim, host.trim)
    return int(ra.is_exhausted.sum())


def closed_loop_against_host(planner, make, steps, **kw):
    sc = make()
    setup(planner, [sc])
    dev = scenario.ExplorativeRunner(sc, None, explorative_fn=explorative_fn(planner), **kw)
    host = scenario.ExplorativeRunner(make(), lambda b, d: planner.plan_timestep(b, d, False), **kw)
    exhausted = 0
    for _ in range(steps):
        fallbacks = [host._fallback_plan(i) for i in range(sc.amount)]
        dev.step()
        host.step()
        exhausted += compare_step(dev, host, fallbacks)
    assert dev.n_fallbacks == host.n_fallbacks
    return dev, exhausted


def test_road_closed_loop_equals_the_host_path_and_the_oracle(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    make = lambda: scenario.commonroad_scenario(mpa, 20, seed=ROAD_SEED)
    dev, exhausted = closed_loop_against_host(planner, make, 7)
    assert max(e["n_permutations"] for e in dev.explorative_records) >= 3
    assert exhausted > 0
    plan = lambda b: oracle_py.plan_batch(mpa, b, 4)
    ref = scenario.ExplorativeRunner(make(), lambda b, d: scenario.plan_timestep_by_levels(plan, b, d))
    ref.run(7)
    assert np.array_equal(bits(dev.pose), bits(ref.pose)) and np.array_equal(dev.trim, ref.trim)
    for a, b in zip(dev.explorative_records, ref.explorative_records):
        assert np.array_equal(a["chosen"], b["chosen"]) and np.array_equal(bits(a["solution_cost"]), bits(b["solution_cost"]))


def test_fixed_permutations_padded_and_repeated_rows(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    dev, _ = closed_loop_against_host(planner, lambda: scenario.commonroad_scenario(mpa, 20, seed=1), 6, fixed_permutations=8)
    assert all(e["n_permutations"] == 8 for e in dev.explorative_records)
    assert any(e["n_levels"] <= 3 for e in dev.explorative_records)   # identity rows repeated: the first minimum wins


def test_sat_checker_with_constant_priorities(planner):
    """The SAT checker and constant priorities on the road map (the from-states family needs lanelets, so the circle
    scenario has no path through it)."""
    mpa = get_mpa("triple_speed", non_convex=True)

    def make():
        sc = scenario.commonroad_scenario(mpa, 12, seed=2)
        sc.checker, sc.priority = scenario.CHECKER_SAT, "constant"
        return sc

    dev, _ = closed_loop_against_host(planner, make, 6)
    assert max(e["n_permutations"] for e in dev.explorative_records) >= 2


def _runners(mpa, seeds, path_id0, **kw):
    out = []
    for k, s in enumerate(seeds):
        r = scenario.ExplorativeRunner(scenario.commonroad_scenario(mpa, 20, seed=s), None, **kw)
        r.path_id0 = path_id0 + 20 * k
        out.append(r)
    return out


def test_many_scenarios_in_one_call_equal_their_separate_calls(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    seeds = list(range(1, 9))
    scs = [scenario.commonroad_scenario(mpa, 20, seed=s) for s in seeds]
    setup(planner, scs + scs)                                   # slots / paths 0..159 together, 160..319 alone
    fn = explorative_fn(planner)
    together = _runners(mpa, seeds, 0)
    alone = _runners(mpa, seeds, 160, explorative_fn=fn)
    for _ in range(5):
        res = scenario.explorative_lockstep_step(together, fn)
        assert res.status.size == sum(e.explorative_records[-1]["searches_local"] for e in together)
        for t, a in zip(together, alone):
            a.step()
            x, y = t.explorative_records[-1], a.explorative_records[-1]
            assert np.array_equal(x["chosen"], y["chosen"]) and np.array_equal(bits(x["solution_cost"]), bits(y["solution_cost"]))
            assert np.array_equal(bits(t.pose), bits(a.pose)) and np.array_equal(t.trim, a.trim)


def test_512_scenarios_take_the_warp_shape_and_equal_the_per_scenario_calls(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    seeds = list(range(1, 513))
    scs = [scenario.commonroad_scenario(mpa, 20, seed=s) for s in seeds]
    setup(planner, scs)
    fn = explorative_fn(planner)
    together = _runners(mpa, seeds, 0)
    res = scenario.explorative_lockstep_step(together, fn)
    assert res.status.size > 7104 and planner.stats().shape == 1
    planner.closed_loop_reset(20 * 512, HL, HW)
    off = 0
    for t, s in zip(together, seeds):
        a = _runners(mpa, [s], t.path_id0, explorative_fn=fn)[0]
        a.step()
        x, y = t.explorative_records[-1], a.explorative_records[-1]
        assert np.array_equal(x["chosen"], y["chosen"]) and np.array_equal(bits(x["solution_cost"]), bits(y["solution_cost"]))
        m = y["searches_local"]
        parity.compare(rows(res, np.arange(off, off + m)), y["result_local"])
        off += m
        assert np.array_equal(bits(t.pose), bits(a.pose)) and np.array_equal(t.trim, a.trim)
    assert off == res.status.size


@pytest.mark.parametrize("variant", [1, 4])
def test_forced_launch_shapes(planner, variant):
    mpa = get_mpa("triple_speed", non_convex=True)
    try:
        planner.set_variant(variant)
        closed_loop_against_host(planner, lambda: scenario.commonroad_scenario(mpa, 20, seed=ROAD_SEED), 3)
    finally:
        planner.set_variant(0)


def test_reachable_set_coupling_drives_it(planner):
    """pdmpc_couple (max_num_CLs = 64) gives the relation and levels the runner hands to the call; the loop equals the
    host path with the same coupler."""
    mpa = get_mpa("triple_speed", non_convex=True)
    make = lambda: scenario.commonroad_scenario(mpa, 20, seed=ROAD_SEED)
    sc = make()
    setup(planner, [sc])
    planner.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
    dev = scenario.ExplorativeRunner(sc, None, explorative_fn=explorative_fn(planner), coupler="reachable_set")
    host = scenario.ExplorativeRunner(make(), lambda b, d: planner.plan_timestep(b, d, False), coupler="reachable_set")
    for _ in range(6):
        rel = planner.couple(dev.pose[:, 0], dev.pose[:, 1], dev.pose[:, 2], dev.trim, priority=sc.priority, max_num_CLs=64)
        dev.k += 1
        D, levels, _perms = dev.decide()
        dev.k -= 1
        assert np.array_equal(rel["level"], levels)
        assert rel["succ_idx"].tolist() == [j for i in range(20) for j in np.flatnonzero(D[i])]
        fallbacks = [host._fallback_plan(i) for i in range(20)]
        dev.step()
        host.step()
        compare_step(dev, host, fallbacks)


def _base(sc):
    r = scenario.ExplorativeRunner(sc, None)
    r.k = 1
    (D, levels, perms), args = r.explorative_args()
    return list(args), [perms], D


def _call(planner, args, perms, mpa, **kw):
    return planner.plan_timestep_explorative(*args, perms, HL, HW, mpa.dt_seconds, scenario.CHECKER_INTERX,
                                             raise_on_search_error=False, **kw)


def test_errors_are_loud_and_leave_the_slots_untouched(planner):
    mpa = get_mpa("triple_speed", non_convex=True)
    sc44 = scenario.commonroad_scenario(mpa, 44, seed=1, allow_shared_paths=True)
    setup(planner, [sc44])
    args, perms, D = _base(sc44)
    n = sc44.amount
    assert int(args[8].max()) >= 2 and D.sum() > 0

    def code(args=args, perms=perms, **kw):
        with pytest.raises(capi.PdmpcError) as e:
            _call(planner, args, perms, mpa, **kw)
        return e.value.code

    first, _ = _call(planner, args, perms, mpa)                  # commits step 1
    bad = [p.copy() for p in perms]
    bad[0][0, 0] = bad[0][0, 1]
    assert code(perms=bad) == capi.PDMPC_ERR_BAD_INPUT          # not a permutation
    lv = args[8].copy()
    i = int(np.flatnonzero(D.any(axis=1))[0])
    lv[i] = lv[np.flatnonzero(D[i])[0]]
    assert code(args=args[:8] + [lv]) == capi.PDMPC_ERR_BAD_INPUT              # level not increasing along D
    lv2 = np.ones(n, dtype=np.int64)
    lv2[30] = 2
    succ2 = [[] for _ in range(n)]
    succ2[0] = [30]                                                             # an edge across scenarios
    sp, p2 = [0, 22, n], [np.array([[1]]), np.array([[1, 2]])]
    assert code(args=args[:7] + [succ2, lv2], perms=p2, scenario_ptr=sp) == capi.PDMPC_ERR_BAD_INPUT
    slot = args[6].copy()
    slot[1] = slot[0]
    assert code(args=args[:6] + [slot] + args[7:]) == capi.PDMPC_ERR_BAD_INPUT   # repeated base slots
    assert code(perms=[np.zeros((0, perms[0].shape[1]), dtype=np.int32)]) == capi.PDMPC_ERR_BAD_INPUT   # P_s = 0
    # too many predecessors after reversal: one vehicle coupled to 43 of lower priority, levels swapped
    star = [list(range(1, n))] + [[] for _ in range(n - 1)]
    lv3 = np.array([1] + [2] * (n - 1))
    _call(planner, args[:7] + [star, lv3], [np.array([[1, 2]])], mpa)   # 43 successors, one predecessor each: fine
    planner.closed_loop_reset(n, HL, HW)
    first, _ = _call(planner, args, perms, mpa)
    assert code(args=args[:7] + [star, lv3], perms=[np.array([[1, 2], [2, 1]])]) == capi.PDMPC_ERR_BAD_INPUT
    # relations passed in
    i32 = lambda v: np.ascontiguousarray(v, dtype=np.int32)
    f64 = lambda v: np.ascontiguousarray(v, dtype=np.float64)
    keep = [i32(args[0]), f64(args[1]), f64(args[2]), f64(args[3]), f64(args[4]), i32(args[5]), i32(args[6]),
            i32(np.zeros(n + 1)), i32([0]), i32([0, n]), i32(args[8]), i32([0, perms[0].shape[0]]), i32([0, perms[0].size]),
            i32(perms[0].reshape(-1))]
    st = capi.TimestepStatesC(n=n, path_id=capi._ptr(keep[0], capi._p_i32), x=capi._ptr(keep[1], capi._p_f64),
                              y=capi._ptr(keep[2], capi._p_f64), yaw=capi._ptr(keep[3], capi._p_f64),
                              speed=capi._ptr(keep[4], capi._p_f64), trim=capi._ptr(keep[5], capi._p_i32),
                              slot=capi._ptr(keep[6], capi._p_i32), succ_ptr=capi._ptr(keep[7], capi._p_i32),
                              succ_idx=capi._ptr(keep[8], capi._p_i32), pred_ptr=capi._ptr(keep[7], capi._p_i32),
                              pred_idx=capi._ptr(keep[8], capi._p_i32), half_length=HL, half_width=HW,
                              dt_seconds=mpa.dt_seconds, checker=scenario.CHECKER_INTERX)
    ex = capi.ExplorativeInC(n_scenarios=1, scenario_ptr=capi._ptr(keep[9], capi._p_i32), level=capi._ptr(keep[10], capi._p_i32),
                             perm_ptr=capi._ptr(keep[11], capi._p_i32), perm_val_ptr=capi._ptr(keep[12], capi._p_i32),
                             perm=capi._ptr(keep[13], capi._p_i32))
    res = scenario.BatchResult.empty(n * perms[0].shape[0], mpa.Hp)
    assert planner.lib.pdmpc_plan_timestep_explorative(planner.h, C.byref(st), C.byref(ex), C.byref(capi.batch_out(res)),
                                                       None) == capi.PDMPC_ERR_BAD_INPUT
    # after the failed calls the slots hold what the first call committed: the next call equals a run without them
    after, choice = _call(planner, args, perms, mpa)
    planner.closed_loop_reset(44, HL, HW)
    again, _ = _call(planner, args, perms, mpa)
    parity.compare(again, first)
    want, want_choice = _call(planner, args, perms, mpa)
    parity.compare(after, want)
    assert np.array_equal(choice["chosen"], want_choice["chosen"])
    # no closed_loop_reset
    fresh = capi.Planner(0)
    try:
        fresh.upload_mpa(mpa)
        fresh.upload_road(scenario.road_tables([sc44]))
        with pytest.raises(capi.PdmpcError) as e:
            _call(fresh, args, perms, mpa)
        assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
    finally:
        fresh.close()
