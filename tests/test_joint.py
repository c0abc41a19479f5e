"""Centralized (joint) search, iter.amount = nV > 1 (CentralizedController.m:33-59, expand_node.m:15-75,
are_constraints_satisfied_sat.m:15-53): the C oracle's properties on the CPU, the CUDA path
(pdmpc_joint_plan_batch) against it on the GPU."""
import dataclasses

import numpy as np
import pytest

from oracle import oracle_py, parity
from pdmpc_b200 import capi, scenario
from pdmpc_b200.mpa import get_mpa
from pdmpc_b200.records import CHECKER_INTERX, CHECKER_SAT, SearchBatch

from helpers import rect, straight_iter


def crossing_pair(mpa, gap=0.3):
    """Two vehicles whose straight plans cross: independent searches collide, the joint one must not."""
    return [straight_iter(mpa, x=0.0, y=0.0, yaw=0.0), straight_iter(mpa, x=0.6, y=-gap, yaw=np.pi / 2)]


def joint_cases(mpa):
    Hp = mpa.Hp
    cases = []
    # (name, rows, nV)
    cases.append(("crossing pair", crossing_pair(mpa), 2))
    three = crossing_pair(mpa) + [straight_iter(mpa, x=1.2, y=0.25, yaw=np.pi)]
    cases.append(("three vehicles", three, 3))
    blocked = crossing_pair(mpa, 0.35)
    blocked[0].obstacles.append(rect(0.9, 0.0, 0.05, 0.5))                  # static obstacle of the search
    blocked[0].dynamic_obstacle_area.append([rect(0.6, 0.6, 0.3, 0.05)] * Hp)  # and a dynamic one
    cases.append(("with obstacles", blocked, 2))
    caged = [straight_iter(mpa, x=0.0, y=0.0), straight_iter(mpa, x=0.0, y=0.14)]   # start overlapping: every child collides
    cases.append(("exhausted", caged, 2))
    two_searches = crossing_pair(mpa) + crossing_pair(mpa, 0.5)
    cases.append(("two searches in one batch", two_searches, 2))
    return [(name, SearchBatch.from_iters(rows, Hp, CHECKER_SAT, mpa.dt_seconds), nV) for name, rows, nV in cases]


def test_oracle_joint_search_properties():
    mpa = get_mpa("single_speed", non_convex=False)
    Hp = mpa.Hp
    # nV = 1 is the plain search
    its = [straight_iter(mpa, y=float(i), obstacles=[rect(0.5, float(i) + 0.02, 0.05, 0.05)]) for i in range(3)]
    b = SearchBatch.from_iters(its, Hp, CHECKER_SAT, mpa.dt_seconds)
    parity.compare(oracle_py.joint_plan_batch(mpa, b, 1), oracle_py.plan_batch(mpa, b))
    # crossing pair: the independent plans collide at some step, the joint plan never does and costs more
    b2 = SearchBatch.from_iters(crossing_pair(mpa), Hp, CHECKER_SAT, mpa.dt_seconds)
    joint, alone = oracle_py.joint_plan_batch(mpa, b2, 2), oracle_py.plan_batch(mpa, b2)
    assert not joint.is_exhausted.any()
    hit = lambda r: [oracle_py.intersect_sat(r.shapes(0)[k], r.shapes(1)[k]) for k in range(Hp)]
    assert any(hit(alone)) and not any(hit(joint))
    assert joint.g_path[0, Hp] > alone.g_path[:, Hp].sum() and joint.g_path[0, Hp] == joint.g_path[1, Hp]
    assert joint.n_expanded[0] == joint.n_expanded[1] and joint.pop_hash[0] == joint.pop_hash[1]
    # far apart: the joint optimum is the pair of independent optima
    far = SearchBatch.from_iters([straight_iter(mpa), straight_iter(mpa, y=5.0)], Hp, CHECKER_SAT, mpa.dt_seconds)
    jf, af = oracle_py.joint_plan_batch(mpa, far, 2), oracle_py.plan_batch(mpa, far)
    assert np.array_equal(jf.trims, af.trims) and np.array_equal(jf.y_predicted, af.y_predicted)
    # capacity is reported, never truncated silently
    small = oracle_py.joint_plan_batch(mpa, b2, 2, max_nodes=500)
    assert (small.status == capi.PDMPC_ERR_CAPACITY).all() and small.is_exhausted.all()


def test_centralized_closed_loop_on_the_oracle():
    mpa = get_mpa("single_speed", non_convex=False)
    r = scenario.CentralizedRunner(scenario.circle_scenario(mpa, 2), lambda b, n: oracle_py.joint_plan_batch(mpa, b, n))
    start = r.pose.copy()
    r.run(6)
    assert (np.hypot(*(r.pose[:, :2] - start[:, :2]).T) > 0.3).all() and r.n_fallbacks == 0


# pop_hash over every pop (default) or, after pdmpc_set_cta_queue(1), over the popped nodes that passed their check
JOINT_MODES = ("full_hash", "valid_hash")


class joint_mode:
    def __init__(self, planner, mode):
        self.planner, self.mode = planner, mode

    def __enter__(self):
        self.planner.set_cta_queue(self.mode == "valid_hash")
        return self.mode == "valid_hash"      # -> hash_valid_pops_only of the oracle

    def __exit__(self, *a):
        self.planner.set_cta_queue(False)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", JOINT_MODES)
def test_joint_search_matches_oracle(planner, mode):
    mpa = get_mpa("single_speed", non_convex=False)
    planner.upload_mpa(mpa)
    CAP = 1 << 23
    planner.set_node_capacity(CAP)
    try:
        with joint_mode(planner, mode) as hv:
            solved = 0
            for name, batch, nV in joint_cases(mpa):
                ref = oracle_py.joint_plan_batch(mpa, batch, nV, max_nodes=CAP, hash_valid_pops_only=hv)
                dev = planner.joint_plan_batch(batch, nV, raise_on_search_error=False)
                try:
                    parity.compare(dev, ref)
                except AssertionError as e:
                    raise AssertionError(f"{name}: {e}")
                solved += int((ref.status == 0).sum())
            assert solved >= 10 and ref.n_expanded[0] > 1000
    finally:
        planner.set_node_capacity(0)


@pytest.mark.gpu
def test_joint_nv1_equals_plain_search_and_triple_speed(planner):
    mpa = get_mpa("triple_speed", non_convex=False)
    planner.upload_mpa(mpa)
    Hp = mpa.Hp
    its = [straight_iter(mpa, y=float(i), obstacles=[rect(0.5, float(i) + 0.02, 0.05, 0.05)]) for i in range(5)]
    b = SearchBatch.from_iters(its, Hp, CHECKER_SAT, mpa.dt_seconds)
    parity.compare(planner.joint_plan_batch(b, 1), planner.plan_batch(b))
    b2 = SearchBatch.from_iters(crossing_pair(mpa), Hp, CHECKER_SAT, mpa.dt_seconds)
    planner.set_node_capacity(1 << 20)
    try:
        parity.compare(planner.joint_plan_batch(b2, 2, False), oracle_py.joint_plan_batch(mpa, b2, 2, max_nodes=1 << 20))
    finally:
        planner.set_node_capacity(0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", JOINT_MODES)
def test_centralized_closed_loop_circle(planner, mode):
    """Circle scenario, 2 and 3 vehicles, centralized (the reference's system tests run these sizes,
    tests/systemtests/systemtests.m:16-34): closed loop on the device equals the oracle-driven one."""
    mpa = get_mpa("single_speed", non_convex=False)
    planner.upload_mpa(mpa)
    CAP = 1 << 23
    planner.set_node_capacity(CAP)
    try:
        with joint_mode(planner, mode) as hv:
            for amount, steps in ((2, 12), (3, 2 if mode == "full_hash" else 1)):
                dev = scenario.CentralizedRunner(scenario.circle_scenario(mpa, amount), lambda b, n: planner.joint_plan_batch(b, n, False))
                ref = scenario.CentralizedRunner(scenario.circle_scenario(mpa, amount),
                                                 lambda b, n: oracle_py.joint_plan_batch(mpa, b, n, max_nodes=CAP,
                                                                                         hash_valid_pops_only=hv))
                dev.run(steps)
                ref.run(steps)
                assert np.array_equal(dev.pose, ref.pose) and np.array_equal(dev.trim, ref.trim)
                for (_k, _b, a), (_k2, _b2, e) in zip(dev.joint_records, ref.joint_records):
                    parity.compare(a, e)
                assert sum(int(e.status[0] == 0) for _k, _b, e in ref.joint_records) >= steps - 1
    finally:
        planner.set_node_capacity(0)


@pytest.mark.gpu
def test_joint_errors_are_loud(planner):
    mpa = get_mpa("single_speed", non_convex=False)
    planner.upload_mpa(mpa)
    Hp = mpa.Hp
    b2 = SearchBatch.from_iters(crossing_pair(mpa), Hp, CHECKER_SAT, mpa.dt_seconds)
    planner.set_node_capacity(512)
    try:
        for mode in JOINT_MODES:
            with joint_mode(planner, mode) as hv:
                r = planner.joint_plan_batch(b2, 2, raise_on_search_error=False)
                assert (r.status == capi.PDMPC_ERR_CAPACITY).all()
                parity.compare(r, oracle_py.joint_plan_batch(mpa, b2, 2, max_nodes=512, hash_valid_pops_only=hv))
    finally:
        planner.set_node_capacity(0)
    for bad_nv in (0, 5, 3):
        with pytest.raises(capi.PdmpcError) as e:
            planner.joint_plan_batch(b2, bad_nv)
        assert e.value.code == capi.PDMPC_ERR_BAD_INPUT
    with pytest.raises(capi.PdmpcError):
        planner.joint_plan_batch(dataclasses.replace(b2, checker=CHECKER_INTERX), 2)
    rows = crossing_pair(mpa)
    rows[1].obstacles.append(rect(3.0, 3.0, 0.1, 0.1))            # obstacle in a non-first row
    with pytest.raises(capi.PdmpcError):
        planner.joint_plan_batch(SearchBatch.from_iters(rows, Hp, CHECKER_SAT, mpa.dt_seconds), 2)


def test_joint_oracle_against_matrix_form_restatement():
    """Second, independent restatement of the joint search (oracle/matlab_literal.py: nV x nNodes arrays,
    successor ids through trim_tuple / cartprod with the radix offsets, the reference's own priority-queue
    source when built): same pop sequence length, node count, trims, poses and joint costs as the C oracle."""
    from oracle import matlab_literal as ml
    use_reference_pq = oracle_py.have_reference_pq()
    mpa6 = get_mpa("single_speed", non_convex=False)
    mpa3 = get_mpa("single_speed", Hp=3, non_convex=False)     # three vehicles: 12^3 children per expansion
    blocked = crossing_pair(mpa6, 0.35)
    blocked[0].obstacles.append(rect(0.9, 0.0, 0.05, 0.5))
    three = [straight_iter(mpa3, x=0.0, y=0.0), straight_iter(mpa3, x=0.45, y=-0.2, yaw=np.pi / 2),
             straight_iter(mpa3, x=0.9, y=0.1, yaw=np.pi)]
    for mpa, rows in ((mpa6, crossing_pair(mpa6)), (mpa6, blocked), (mpa3, three)):
        Hp = mpa.Hp
        nV = len(rows)
        batch = SearchBatch.from_iters(rows, Hp, CHECKER_SAT, mpa.dt_seconds)
        ref = oracle_py.joint_plan_batch(mpa, batch, nV)
        info = ml.do_joint_graph_search(rows, mpa, use_reference_pq=use_reference_pq)
        assert info.is_exhausted == bool(ref.is_exhausted[0])
        assert info.n_expanded == int(ref.n_expanded[0]) and len(info.pops) == int(ref.n_pops[0])
        h = 0xcbf29ce484222325
        for p in info.pops:
            h = ((h ^ p) * 0x100000001b3) & 0xFFFFFFFFFFFFFFFF
        assert h == int(ref.pop_hash[0])                          # identical pop ORDER
        assert info.tree_path == ref.tree_path[0].tolist()
        for v in range(nV):
            assert info.predicted_trims[v].tolist() == ref.trims[v, 1:].tolist()
            assert np.array_equal(info.y_predicted[v].view(np.uint64), ref.y_predicted[v].view(np.uint64))
        assert np.array_equal(np.array(info.g_path).view(np.uint64), ref.g_path[0].view(np.uint64))
