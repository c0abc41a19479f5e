"""pdmpc_couple and pdmpc_plan_timestep_from_states_coupled (DESIGN.md §4.12): the reachable-set coupling, priorities,
level cut and computation levels decided on the device equal the host specification (scenario.reachable_set_overlaps,
decide_relations) bit for bit, on random poses along the reference paths and along closed loops; every input error is
loud."""
import ctypes as C

import numpy as np
import pytest

import mexfake
from oracle import oracle_py, parity
from pdmpc_b200 import capi, scenario
from pdmpc_b200.mpa import get_mpa

pytestmark = pytest.mark.gpu

COUPLE = 12   # pdmpc_b200_mex.cpp: enum Command


def host_relations(mpa, pose, trim, scenario_ptr, priority, max_cls) -> dict:
    """What Planner.couple returns, from the host specification, scenario by scenario."""
    rel = {k: [0] for k in ("succ_ptr", "par_ptr", "pred_ptr")}
    rel.update({k: [] for k in ("succ_idx", "par_idx", "pred_idx", "level", "overlap_area")})
    for a, b in zip(scenario_ptr[:-1], scenario_ptr[1:]):
        area = scenario.reachable_set_overlaps(mpa, pose[a:b], trim[a:b])
        rel["overlap_area"].append(area)
        if b == a:
            continue
        D, seq, levels = scenario.decide_relations((area > scenario.COUPLING_AREA_THRESHOLD).astype(np.int64), priority, max_cls)
        for i in range(b - a):
            for k, rows in (("succ", D[i, :]), ("par", D[:, i] & ~seq[:, i]), ("pred", seq[:, i])):
                rel[f"{k}_idx"].extend(a + np.flatnonzero(rows))
                rel[f"{k}_ptr"].append(len(rel[f"{k}_idx"]))
        rel["level"].extend(levels.tolist())
    return rel


def assert_relations_equal(got, want):
    for k in ("succ_ptr", "succ_idx", "par_ptr", "par_idx", "pred_ptr", "pred_idx", "level"):
        assert np.asarray(got[k]).tolist() == [int(v) for v in want[k]], k
    assert len(got["overlap_area"]) == len(want["overlap_area"])
    for g, w in zip(got["overlap_area"], want["overlap_area"]):
        assert g.shape == w.shape and np.array_equal(g.view(np.uint64), w.view(np.uint64))


def random_poses(mpa, n, rng):
    """n vehicles anywhere along the map's reference paths, off the centre line, any heading offset and trim."""
    pool = [v.reference_path for v in scenario.commonroad_scenario(mpa, 33, seed=1).vehicles]
    pose = np.zeros((n, 3))
    for r in range(n):
        path = pool[rng.integers(len(pool))]
        j = int(rng.integers(0, path.shape[0] - 1))
        d = path[j + 1] - path[j]
        pose[r, :2] = path[j] + rng.normal(scale=0.05, size=2)
        pose[r, 2] = np.arctan2(d[1], d[0]) + rng.normal(scale=0.2)
    return pose, rng.integers(1, mpa.n_trims + 1, size=n).astype(np.int32)


def setup(planner, mpa_type):
    mpa = get_mpa(mpa_type, non_convex=True)
    planner.upload_mpa(mpa)
    planner.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
    return mpa


def test_512_scenarios_of_20_vehicles_in_one_call(planner):
    mpa = setup(planner, "triple_speed")
    rng = np.random.default_rng(2024)
    sp = np.arange(0, 512 * 20 + 1, 20)
    pose, trim = random_poses(mpa, 512 * 20, rng)
    got = planner.couple(pose[:, 0], pose[:, 1], pose[:, 2], trim, sp, "coloring", 99)
    want = host_relations(mpa, pose, trim, sp, "coloring", 99)
    assert_relations_equal(got, want)
    areas = np.concatenate([a.reshape(-1) for a in want["overlap_area"]])
    assert (areas > 1e-3).sum() > 512 * 20 and ((areas > 0) & (areas <= 1e-3)).sum() > 0   # the threshold decides cases
    assert int(got["level"].max()) > 2


@pytest.mark.parametrize("mpa_type", ["triple_speed", "single_speed"])
def test_both_prioritizers_level_cuts_and_scenario_sizes(planner, mpa_type):
    """Scenarios of 40, 40, 1, 0, 64 and 20 rows in one call; both prioritizers; max_num_CLs 1, 2 and 99."""
    mpa = setup(planner, mpa_type)
    rng = np.random.default_rng(7)
    sizes = [40, 40, 1, 0, 64, 20]
    sp = np.concatenate([[0], np.cumsum(sizes)])
    pose, trim = random_poses(mpa, int(sp[-1]), rng)
    for priority in ("coloring", "constant"):
        for max_cls in (1, 2, 99):
            got = planner.couple(pose[:, 0], pose[:, 1], pose[:, 2], trim, sp, priority, max_cls)
            assert_relations_equal(got, host_relations(mpa, pose, trim, sp, priority, max_cls))
            assert int(got["level"].max()) <= max_cls


def test_errors_are_loud(planner):
    mpa = setup(planner, "triple_speed")
    rng = np.random.default_rng(3)
    pose, trim = random_poses(mpa, 65, rng)
    x, y, yaw = pose[:, 0], pose[:, 1], pose[:, 2]

    def code(**kw):
        args = dict(x=x, y=y, yaw=yaw, trim=trim, scenario_ptr=[0, 65])
        args.update(kw)
        with pytest.raises(capi.PdmpcError) as e:
            planner.couple(**args)
        return e.value.code

    assert code() == capi.PDMPC_ERR_BAD_INPUT                                     # 65 rows in one scenario
    assert code(scenario_ptr=[0, 30, 64]) == capi.PDMPC_ERR_BAD_INPUT             # does not end at n
    assert code(scenario_ptr=[0, 40, 30, 65]) == capi.PDMPC_ERR_BAD_INPUT         # not monotone
    assert code(scenario_ptr=[1, 33, 65]) == capi.PDMPC_ERR_BAD_INPUT             # does not start at 0
    ok = [0, 33, 65]
    for bad in (0, mpa.n_trims + 1):
        t = trim.copy()
        t[5] = bad
        assert code(trim=t, scenario_ptr=ok) == capi.PDMPC_ERR_BAD_INPUT
    assert code(scenario_ptr=ok, priority=2) == capi.PDMPC_ERR_BAD_INPUT
    assert code(scenario_ptr=ok, max_num_CLs=0) == capi.PDMPC_ERR_BAD_INPUT
    assert code(scenario_ptr=ok, idx_capacity=1) == capi.PDMPC_ERR_CAPACITY
    planner.couple(x, y, yaw, trim, ok)                                          # the handle is still usable
    # relation pointers passed to the coupled time step
    n = 2
    arr = lambda v, t: np.ascontiguousarray(v, dtype=t)
    i32, f64 = (lambda v: arr(v, np.int32)), (lambda v: arr(v, np.float64))
    keep = [i32([0, 1]), f64([1.0, 2.0]), f64([1.0, 2.0]), f64([0.0, 0.0]), f64([0.0, 0.0]), i32([1, 1]), i32([0, 0, 0]), i32([0])]
    st = capi.TimestepStatesC(n=n, path_id=capi._ptr(keep[0], capi._p_i32), x=capi._ptr(keep[1], capi._p_f64),
                              y=capi._ptr(keep[2], capi._p_f64), yaw=capi._ptr(keep[3], capi._p_f64),
                              speed=capi._ptr(keep[4], capi._p_f64), trim=capi._ptr(keep[5], capi._p_i32),
                              succ_ptr=capi._ptr(keep[6], capi._p_i32), slot=capi._ptr(keep[7], capi._p_i32),
                              half_length=0.12, half_width=0.0625, dt_seconds=mpa.dt_seconds, checker=1)
    sp = i32([0, n])
    prm = capi.CoupleParamsC(n_scenarios=1, scenario_ptr=capi._ptr(sp, capi._p_i32), prioritizer=1, max_num_CLs=99)
    res = scenario.BatchResult.empty(n, mpa.Hp)
    assert planner.lib.pdmpc_plan_timestep_from_states_coupled(planner.h, C.byref(st), C.byref(prm), None,
                                                                C.byref(capi.batch_out(res))) == capi.PDMPC_ERR_BAD_INPUT
    # no reachable sets uploaded / sets of another automaton
    fresh = capi.Planner(0)
    try:
        fresh.upload_mpa(mpa)
        with pytest.raises(capi.PdmpcError) as e:
            fresh.couple(x[:4], y[:4], yaw[:4], trim[:4])
        assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
        fresh.upload_reachable_sets(scenario.local_reachable_sets_conv(get_mpa("single_speed", non_convex=True)))
        with pytest.raises(capi.PdmpcError) as e:
            fresh.couple(x[:4], y[:4], yaw[:4], trim[:4])
        assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
    finally:
        fresh.close()


@pytest.mark.parametrize("amount,max_cls,seed", [(20, 99, 7), (40, 2, 3)])
def test_coupled_time_step_closed_loop(planner, amount, max_cls, seed):
    """pdmpc_plan_timestep_from_states_coupled drives the same closed loop as the host's reachable-set coupling with
    pdmpc_plan_timestep_from_states: the relations of every step equal the host specification, every step's result
    equals, and so do the final poses and trims; for 20 vehicles also the host functions + oracle level by level."""
    mpa = get_mpa("triple_speed", non_convex=True)
    planner.upload_mpa(mpa)
    mk = lambda: scenario.commonroad_scenario(mpa, amount, seed=seed, allow_shared_paths=amount > 33)
    sc = mk()
    planner.upload_road(scenario.road_tables([sc]))
    planner.upload_reachable_sets(scenario.local_reachable_sets_conv(mpa))
    hl, hw = scenario.VEH_LENGTH / 2 + 0.01, scenario.VEH_WIDTH / 2 + 0.01
    planner.closed_loop_reset(amount, hl, hw)
    one = scenario.ScenarioRunner(sc, None, max_num_CLs=max_cls,
                                  coupled_fn=lambda *a: planner.plan_timestep_from_states_coupled(*a, raise_on_search_error=False))
    res_one, preds = [], 0
    for _ in range(7):
        want = host_relations(mpa, one.pose, one.trim, [0, amount], sc.priority, max_cls)
        res_one.append(one.step_timestep())
        got = one.timestep_records[-1][2]
        assert_relations_equal(got, want)
        preds += len(want["pred_idx"]) + len(want["par_idx"])
    assert preds > 0
    planner.closed_loop_reset(amount, hl, hw)
    host = scenario.ScenarioRunner(mk(), None, max_num_CLs=max_cls, coupler="reachable_set",
                                   states_fn=lambda *a: planner.plan_timestep_from_states(*a, raise_on_search_error=False))
    for k in range(7):
        parity.compare(res_one[k], host.step_timestep())
    assert np.array_equal(one.pose.view(np.uint64), host.pose.view(np.uint64)) and np.array_equal(one.trim, host.trim)
    assert one.n_fallbacks == host.n_fallbacks
    if max_cls >= amount:
        ref = scenario.ScenarioRunner(mk(), lambda b: oracle_py.plan_batch(mpa, b, 4), coupler="reachable_set")
        for _ in range(7):
            ref.step()
        assert np.array_equal(one.pose.view(np.uint64), ref.pose.view(np.uint64)) and np.array_equal(one.trim, ref.trim)


def test_mex_couple_matches_the_host_specification(built):
    mpa = get_mpa("triple_speed", non_convex=True)
    matlab = mexfake.FakeMatlab()
    (h,) = matlab.call(1, mexfake.CREATE, 0.0)
    try:
        trans, man = mexfake.matlab_mpa(mpa)
        matlab.call(0, mexfake.UPLOAD_MPA, float(h), trans, man)
        sets = scenario.local_reachable_sets_conv(mpa)
        matlab.call(0, mexfake.UPLOAD_REACHABLE_SETS, float(h), [[np.ascontiguousarray(a) for a in row] for row in sets])
        pose, trim = random_poses(mpa, 24, np.random.default_rng(11))
        adj, area = matlab.call(2, COUPLE, float(h), pose, trim.astype(np.float64))
        want = scenario.reachable_set_overlaps(mpa, pose, trim)
        assert np.array_equal(area.view(np.uint64), want.view(np.uint64))
        assert np.array_equal(adj, scenario.couple_reachable_sets(mpa, pose, trim).astype(np.float64)) and adj.sum() > 0
        with pytest.raises(mexfake.MexError, match="pdmpc:status"):
            matlab.call(2, COUPLE, float(h), np.zeros((65, 3)), np.ones(65))
    finally:
        matlab.call(0, mexfake.DESTROY, float(h))
        matlab.clear_mex()
