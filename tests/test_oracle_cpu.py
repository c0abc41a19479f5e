"""CPU suite, part 1: the oracle is pinned before anything trusts it.

  * the reference's own known-answer tests (tests/unittests/hlc/intersect_unittest.m:8-54)
  * the heap restatement against the reference's UNMODIFIED priority-queue source
    compiled here (oracle/_ref/libpq_ref.so) + this container's libstdc++, and against
    the same queue on libstdc++'s std::priority_queue (oracle/libpq_std.so)
  * the C oracle against the second, matrix-form restatement (oracle/matlab_literal.py)
  * both against the committed golden fixtures (tests/golden, tools/make_golden.py)
"""
import os

import numpy as np
import pytest

from oracle import matlab_literal as ml
from oracle import oracle_py, parity

from helpers import GOLDEN_CASES, GOLDEN_DIR, load_golden, rect

HEX = np.array([[-7.0749, -2.8728, 9.8889, 21.3024, 15.3469, 7.9387],
                [-6.4707, -12.1152, -24.4428, -3.0950, 19.3838, 18.7030]])


@pytest.fixture(scope="module")
def lanelet1():
    return np.load(os.path.join(GOLDEN_DIR, "kat_lanelet1.npz"))["lanelet"]


# ---- reference KATs: intersect_unittest.m ----------------------------------------
@pytest.mark.parametrize("impl", [oracle_py, ml], ids=["c_oracle", "matrix_form"])
def test_kat_polygon_pos_neg(impl):
    assert impl.intersect_sat(HEX, HEX - 5.0) is True       # testPolygonPos :38-45
    assert impl.intersect_sat(HEX, HEX - 40.0) is False     # testPolygonNeg :47-54


@pytest.mark.parametrize("impl", [oracle_py, ml], ids=["c_oracle", "matrix_form"])
def test_kat_intersect_lanelets(impl, lanelet1):
    assert lanelet1.shape == (12, 6)
    assert np.allclose(lanelet1[0, 2:4], [2.25, 3.82]) and np.allclose(lanelet1[0, 0:2], [2.25, 3.67])
    inside = np.array([[0, 5, 5, 0], [0, 0, 5, 5]], dtype=float)                  # :8-16 -> true
    within = np.array([[2.4, 2.5, 2.5, 2.4], [3.7, 3.7, 3.8, 3.8]])               # :18-26 -> false
    on_left = np.array([[2.2, 2.4, 2.4, 2.2], [3.7, 3.7, 3.9, 3.9]])              # :28-36 -> true
    assert impl.intersect_lanelets(inside, lanelet1) is True
    assert impl.intersect_lanelets(within, lanelet1) is False
    assert impl.intersect_lanelets(on_left, lanelet1) is True


# ---- priority queue: oracle heap == reference MEX + libstdc++ ----------------------
@pytest.mark.parametrize("seed", range(6))
def test_pq_matches_reference_mex(seed):
    if not oracle_py.have_reference_pq():
        pytest.skip("needs the reference's priority-queue source (oracle/Makefile REFERENCE=<reference checkout>)")
    _pq_script_matches(seed, oracle_py.ReferencePQ())


@pytest.mark.parametrize("seed", range(6))
def test_pq_matches_std_priority_queue(seed):
    """The same scripts against the queue on libstdc++'s std::priority_queue, which shares no code with the
    oracle's heap and is the matrix-form restatement's queue where the reference's source is not built."""
    _pq_script_matches(seed, oracle_py.StdPQ())


def _pq_script_matches(seed, ref):
    rng = np.random.default_rng(seed)
    mine = oracle_py.OraclePQ()
    assert ref.pop()[0] == -1 and mine.pop()[0] == -1        # empty -> -1 (mex.cpp:87-94)
    next_id = 1
    for _ in range(400):
        if rng.random() < 0.6 or mine.size() == 0:
            m = int(rng.integers(1, 13))
            # few distinct values -> many exact ties, the case only heap mechanics decide
            vals = rng.integers(0, 6, size=m).astype(np.float64) * 0.25 if seed % 2 else rng.random(m)
            ids = np.arange(next_id, next_id + m)
            next_id += m
            ref.push(ids, vals)
            for i, v in zip(ids, vals):
                mine.push(int(i), float(v))
        else:
            for _ in range(int(rng.integers(1, 6))):
                a, b = ref.pop(), mine.pop()
                assert a[0] == b[0]
                if a[0] != -1:
                    assert a[1] == b[1]
        assert ref.size() == mine.size()
    while True:
        a, b = ref.pop(), mine.pop()
        assert a[0] == b[0]
        if a[0] == -1:
            break


# ---- sin/cos spec --------------------------------------------------------------------
def test_sincos_spec_accuracy():
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.uniform(-50, 50, 4000), [0.0, np.pi / 2, -np.pi, 1e-9, 3 * np.pi / 4]])
    for x in xs:
        s, c = oracle_py.sincos(float(x))
        assert abs(s - np.sin(x)) <= 4 * np.spacing(1.0) and abs(c - np.cos(x)) <= 4 * np.spacing(1.0)
        assert abs(s * s + c * c - 1.0) < 1e-15


# ---- checkers: C oracle == matrix form on random inputs ------------------------------
def _random_polyline(rng, n_polys, closed=True):
    cols = []
    for _ in range(n_polys):
        m = int(rng.integers(3, 9))
        p = rng.uniform(-1, 1, (2, 1)) + rng.uniform(-0.6, 0.6, (2, m))
        if closed:
            p = np.hstack([p, p[:, :1]])
        cols += [p, ml.NAN_COL]
    return np.hstack(cols)


def test_interx_c_equals_matrix_form():
    rng = np.random.default_rng(1)
    hits = 0
    for _ in range(300):
        shape = rect(rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(0.05, 0.4), rng.uniform(0.05, 0.4))
        obs = _random_polyline(rng, int(rng.integers(1, 5)))
        a, b = oracle_py.interx(shape, obs), ml.interx(shape, obs)
        assert a == b
        hits += a
    assert 20 < hits < 280
    assert oracle_py.interx(rect(0, 0, 1, 1), np.zeros((2, 0))) is False          # InterX.m:48-52
    # containment is NOT detected (Config.m:75-84) and touching does not count (strict <)
    assert oracle_py.interx(rect(0, 0, 0.1, 0.1), rect(0, 0, 1, 1)) is False
    assert oracle_py.interx(rect(0, 0, 1, 1), rect(2, 0, 1, 1)) is False


def test_sat_and_lanelet_boundary_c_equals_matrix_form():
    rng = np.random.default_rng(2)
    for _ in range(300):
        a = rect(rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(0.05, 0.5), rng.uniform(0.05, 0.5))
        ang = rng.uniform(0, np.pi)
        R = np.array([[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]])
        b = R @ rect(0, 0, rng.uniform(0.05, 0.5), rng.uniform(0.05, 0.5)) + rng.uniform(-1, 1, (2, 1))
        assert oracle_py.intersect_sat(a, b) == ml.intersect_sat(a, b)
        left = np.cumsum(rng.uniform(0, 0.3, (2, 8)), axis=1) - 1
        right = left + np.array([[0.0], [0.3]])
        assert oracle_py.intersect_lanelet_boundary(a, left, right) == ml.intersect_lanelet_boundary(a, left, right)
    # closed polygon (repeated first vertex): zero edge -> NaN axis -> ignored (intersect_sat.m:23)
    assert oracle_py.intersect_sat(rect(0, 0, 1, 1), rect(0.5, 0.5, 1, 1)) is True
    assert oracle_py.intersect_sat(rect(0, 0, 1, 1), rect(3, 0, 1, 1)) is False


# ---- golden fixtures ---------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_reproduces_golden(name):
    mpa, batch, exp = load_golden(name)
    for threads in (1, 4):
        got = oracle_py.plan_batch(mpa, batch, threads)
        info = parity.compare(got, exp)
    assert info["n"] == batch.n and info["exhausted"] >= 3


def _iters_from_batch(batch, i):
    """Rebuild the IterationData of search i from the flat record (inverse of from_iters)."""
    from pdmpc_b200.records import IterationData
    Hp, S = batch.Hp, batch.Hp + 1

    def polys(slot):
        out = []
        for p in range(batch.slot_ptr[i * S + slot], batch.slot_ptr[i * S + slot + 1]):
            v0, v1 = batch.poly_ptr[p], batch.poly_ptr[p + 1]
            out.append(np.vstack([batch.vert_x[v0:v1], batch.vert_y[v0:v1]]))
        return out

    dyn = [polys(k) for k in range(1, S)]
    n_rows = max(len(d) for d in dyn)
    assert all(len(d) == n_rows for d in dyn)
    rows = [[dyn[k][r] for k in range(Hp)] for r in range(n_rows)]
    l0, l1, l2 = batch.lane_ptr[2 * i: 2 * i + 3]
    return IterationData(
        x0=np.array([batch.x0[i], batch.y0[i], batch.yaw0[i], 0.0]), trim_indices=int(batch.trim0[i]),
        reference_trajectory_points=np.column_stack([batch.ref_x[i * Hp:(i + 1) * Hp], batch.ref_y[i * Hp:(i + 1) * Hp]]),
        v_ref=batch.v_ref[i * Hp:(i + 1) * Hp].copy(), obstacles=polys(0), dynamic_obstacle_area=rows,
        predicted_lanelet_boundary=(np.vstack([batch.lane_x[l0:l1], batch.lane_y[l0:l1]]),
                                    np.vstack([batch.lane_x[l1:l2], batch.lane_y[l1:l2]])))


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_matrix_form_reproduces_golden_subset(name):
    """Second restatement (driving the reference's own PQ source when built) on a subset:
    the cheapest, the most expensive and every exhausted search of the fixture."""
    mpa, batch, exp = load_golden(name)
    order = np.argsort(exp.n_pops)
    pick = set(order[:3].tolist() + order[-2:].tolist() + np.flatnonzero(exp.is_exhausted)[:2].tolist())
    for i in sorted(pick):
        info = ml.do_graph_search(_iters_from_batch(batch, i), mpa, batch.checker, use_reference_pq=oracle_py.have_reference_pq())
        assert info.is_exhausted == bool(exp.is_exhausted[i])
        assert info.n_expanded == exp.n_expanded[i] and len(info.pops) == exp.n_pops[i]
        h = 0xcbf29ce484222325
        for p in info.pops:
            h = ((h ^ p) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
        assert h == int(exp.pop_hash[i])
        if not info.is_exhausted:
            assert info.predicted_trims == exp.trims[i, 1:].tolist()
            assert info.tree_path == exp.tree_path[i].tolist()
            assert np.array_equal(info.y_predicted.view(np.uint64), exp.y_predicted[i].view(np.uint64))


def test_libm_trig_changes_no_discrete_result():
    """MATLAB's sin/cos are unpinned (SURVEY.md §8c).  Re-running the matrix-form search with
    numpy's libm trig instead of the shared spec leaves trims / flags / node counts unchanged and
    poses within the 1e-9 relative tolerance north_star states, on the sampled searches."""
    mpa, batch, exp = load_golden("road_interx_single_speed")
    order = np.argsort(exp.n_pops)
    for i in order[:4].tolist() + order[-1:].tolist():
        info = ml.do_graph_search(_iters_from_batch(batch, i), mpa, batch.checker, trig="libm",
                                  use_reference_pq=oracle_py.have_reference_pq())
        assert info.is_exhausted == bool(exp.is_exhausted[i])
        if not info.is_exhausted:
            assert info.predicted_trims == exp.trims[i, 1:].tolist()
            err = np.abs(info.y_predicted - exp.y_predicted[i]) / np.maximum(np.abs(exp.y_predicted[i]), 1e-300)
            assert err.max() <= 1e-9


# ---- hand-countable micro scenarios (SURVEY.md §7 step 1) ------------------------------
def test_free_space_and_blocked_world_counts():
    from pdmpc_b200.mpa import get_mpa
    from pdmpc_b200.records import CHECKER_INTERX, CHECKER_SAT, SearchBatch
    from helpers import straight_iter
    for checker in (CHECKER_SAT, CHECKER_INTERX):
        mpa = get_mpa("single_speed", non_convex=(checker == CHECKER_INTERX))
        b = SearchBatch.from_iters([straight_iter(mpa)], mpa.Hp, checker, mpa.dt_seconds)
        r = oracle_py.plan_batch(mpa, b)
        assert not r.is_exhausted[0] and r.trims[0, -1] == 1 and r.n_pops[0] >= mpa.Hp + 1
        obs = rect(0.0, 0.0, 5.0, 5.0) if checker == CHECKER_SAT else rect(0.05, 0.0, 0.001, 3.0)
        it = straight_iter(mpa, obstacles=[obs])
        b = SearchBatch.from_iters([it], mpa.Hp, checker, mpa.dt_seconds)
        r = oracle_py.plan_batch(mpa, b)
        n_children = int(mpa.transition[0, it.trim_indices - 1].sum())
        assert r.is_exhausted[0] == 1 and r.n_expanded[0] == 1 + n_children == r.n_pops[0]
        assert np.isnan(r.y_predicted[0]).all()


@pytest.mark.parametrize("name", ["timestep_road_triple_speed", "timestep_circle_single_speed"])
def test_oracle_reproduces_golden_timesteps(name):
    """The time-step fixtures (one-call inputs + expected outputs) against the C oracle driven level by
    level with host-side obstacle assembly — the specification of pdmpc_plan_timestep."""
    from helpers import load_golden_timesteps
    from oracle import parity
    from pdmpc_b200 import scenario
    mpa, steps = load_golden_timesteps(name)
    assert len(steps) >= 8
    edges = 0
    for batch, deps, exp in steps:
        got = scenario.plan_timestep_by_levels(lambda b: oracle_py.plan_batch(mpa, b), batch, deps)
        parity.compare(got, exp)
        edges += deps.pred_idx.size
    assert edges > 50
