"""MonteCarloTreeSearch (SURVEY.md §8 a10) on the CPU: the C oracle against the
matrix-form restatement that uses numpy's independent MT19937, the reference's
own priority-queue source (when built) and MATLAB-style `children` bookkeeping;
hand-countable cases; the random stream against numpy's RandomState."""
import numpy as np
import pytest

from oracle import matlab_literal as ml
from oracle import oracle_py

from helpers import load_golden, rect, straight_iter
from test_oracle_cpu import _iters_from_batch
from pdmpc_b200.mpa import get_mpa
from pdmpc_b200.records import CHECKER_INTERX, CHECKER_SAT, SearchBatch


@pytest.mark.parametrize("seed", [1, 2, 42, 5489, 2**31 + 7])
def test_mt19937_rand_equals_numpy_randomstate(seed):
    """rand(RandStream('mt19937ar', Seed = s)) is MT19937 + genrand_res53 — numpy's legacy
    RandomState implements the same published algorithm independently."""
    got = oracle_py.mt19937_rand(seed, 1500)
    exp = np.random.RandomState(seed).random_sample(1500)
    assert np.array_equal(got.view(np.uint64), exp.view(np.uint64))
    assert got.min() > 0.0 and got.max() < 1.0


def _fnv(words):
    h = 0xcbf29ce484222325
    for p in words:
        h = ((h ^ p) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
    return h


def _compare_with_literal(mpa, batch, picks, seeds, nmax):
    got = oracle_py.mcts_plan_batch(mpa, batch, seeds, nmax, 2)
    assert (got.status == 0).all()
    for i in picks:
        info = ml.do_mcts(_iters_from_batch(batch, i), mpa, batch.checker, int(seeds[i]), nmax,
                          use_reference_pq=oracle_py.have_reference_pq())
        assert info.is_exhausted == bool(got.is_exhausted[i]), i
        assert info.n_expanded == got.n_expanded[i] and info.n_traversals == got.n_pops[i], i
        assert _fnv(info.pops) == int(got.pop_hash[i]), i
        if not info.is_exhausted:
            assert info.predicted_trims == got.trims[i, 1:].tolist()
            assert info.tree_path == got.tree_path[i].tolist()
            assert np.array_equal(info.y_predicted.view(np.uint64), got.y_predicted[i].view(np.uint64))
            assert got.g_path[i, -1] == info.cost and (got.g_path[i, :-1] == -1).all() and (got.h_path[i] == -1).all()
            for k, shp in enumerate(info.shapes):
                n = int(got.shape_npts[i, k])
                assert n == shp.shape[1]
                assert np.array_equal(got.shape_x[i, k, :n].view(np.uint64), shp[0].view(np.uint64))
                assert np.array_equal(got.shape_y[i, k, :n].view(np.uint64), shp[1].view(np.uint64))
        else:
            assert np.isnan(got.y_predicted[i]).all() and (got.trims[i, 1:] == 0).all()
    return got


@pytest.mark.parametrize("name,nmax", [("road_interx_triple_speed", 250), ("road_interx_single_speed", 60),
                                       ("circle_sat_single_speed", 40)])
def test_c_oracle_equals_matrix_form(name, nmax):
    mpa, batch, exp = load_golden(name)
    rng = np.random.default_rng(7)
    seeds = rng.integers(2, 60, size=batch.n).astype(np.uint32)      # time_step + vehicle_index
    order = np.argsort(exp.n_pops)
    picks = sorted(set(order[:2].tolist() + order[-2:].tolist() + np.flatnonzero(exp.is_exhausted)[:2].tolist()
                       + [batch.n // 2]))
    got = _compare_with_literal(mpa, batch, picks, seeds, nmax)
    # the sampled optimizer finds plans in the searches the optimal one solves easily
    easy = order[: batch.n // 2]
    assert got.is_exhausted[easy].mean() < 0.5
    # the budget is tested between roll-outs only (MonteCarloTreeSearch.m:86): overshoot < Hp
    assert (got.n_expanded < nmax + mpa.Hp).all()


def test_free_space_and_walled_in():
    """Hand-countable: in free space every roll-out is valid, so the first Hp expansions reach
    depth Hp and n_expansions hits the budget; boxed in by a static obstacle covering the
    vehicle, every first-step edge is invalid: one expansion per root successor, then finished."""
    mpa = get_mpa("single_speed", non_convex=False)
    Hp = mpa.Hp
    it = straight_iter(mpa)
    b = SearchBatch.from_iters([it], Hp, CHECKER_SAT, mpa.dt_seconds)
    # budget 1: the test at :86 admits exactly one roll-out, which expands Hp fresh nodes 2..Hp+1
    r = oracle_py.mcts_plan_batch(mpa, b, [3], 1)
    assert r.status[0] == 0 and not r.is_exhausted[0]
    assert r.n_expanded[0] == Hp and r.n_pops[0] == Hp
    assert r.tree_path[0].tolist() == list(range(1, Hp + 2))
    r = oracle_py.mcts_plan_batch(mpa, b, [3], 30)
    assert 30 <= r.n_expanded[0] < 30 + Hp and not r.is_exhausted[0]
    assert (np.diff(r.tree_path[0]) > 0).all()                   # ids grow along any root-to-leaf path
    blocked = straight_iter(mpa, obstacles=[rect(0.1, 0.0, 2.0, 2.0)])
    b2 = SearchBatch.from_iters([blocked], Hp, CHECKER_SAT, mpa.dt_seconds)
    r2 = oracle_py.mcts_plan_batch(mpa, b2, [3], 30)
    n_root_succ = int(mpa.transition[0, it.trim_indices - 1].sum())
    assert r2.is_exhausted[0] and r2.n_expanded[0] == n_root_succ
    # every roll-out consumed exactly one random number, plus the final visit that finds the root childless
    assert r2.n_pops[0] == n_root_succ + 1


def test_same_seed_same_plan_and_seed_matters():
    mpa, batch, _ = load_golden("road_interx_triple_speed")
    sub = batch.select(np.arange(12))
    a = oracle_py.mcts_plan_batch(mpa, sub, np.full(12, 9), 100, 1)
    b = oracle_py.mcts_plan_batch(mpa, sub, np.full(12, 9), 100, 3)
    c = oracle_py.mcts_plan_batch(mpa, sub, np.full(12, 10), 100, 1)
    assert np.array_equal(a.pop_hash, b.pop_hash) and np.array_equal(a.trims, b.trims)
    assert not np.array_equal(a.pop_hash, c.pop_hash)
