"""Coupling, priorities and computation levels of a time step (DESIGN.md §4.12), CPU part: the host specification of the
reachable-set overlap (scenario.convex_overlap_area) against an exact rational run of the same clipping, literal cases,
the relations decide_relations derives, the C layout of the new ABI structs and the MEX shim's COUPLE command."""
import ctypes as C
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import mexfake
from pdmpc_b200 import scenario
from pdmpc_b200.mpa import get_mpa

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def exact_overlap_area(P, Q) -> Fraction:
    """convex_overlap_area's clipping in exact rational arithmetic."""
    p = [(Fraction(float(x)), Fraction(float(y))) for x, y in zip(P[0][:-1], P[1][:-1])]
    q = [(Fraction(float(x)), Fraction(float(y))) for x, y in zip(Q[0][:-1], Q[1][:-1])]
    sq = sum(q[k][0] * q[(k + 1) % len(q)][1] - q[(k + 1) % len(q)][0] * q[k][1] for k in range(len(q)))
    if sq == 0:
        return Fraction(0)
    if sq < 0:
        q = q[::-1]
    cur = p
    for k in range(len(q)):
        a, b = q[k], q[(k + 1) % len(q)]
        side = lambda v: (b[0] - a[0]) * (v[1] - a[1]) - (b[1] - a[1]) * (v[0] - a[0])
        out, s = [], cur[-1]
        for e in cur:
            ds, de = side(s), side(e)
            if (de >= 0) != (ds >= 0):
                t = ds / (ds - de)
                out.append((s[0] + t * (e[0] - s[0]), s[1] + t * (e[1] - s[1])))
            if de >= 0:
                out.append(e)
            s = e
        if not out:
            return Fraction(0)
        cur = out
    acc = sum(cur[k][0] * cur[(k + 1) % len(cur)][1] - cur[(k + 1) % len(cur)][0] * cur[k][1] for k in range(len(cur)))
    return abs(acc) / 2


def random_hull(rng, cx, cy, r):
    pts = np.column_stack([cx + rng.uniform(-r, r, 12), cy + rng.uniform(-r, r, 12)])
    return scenario._convex_hull_closed(pts)


def square(x0, y0, s):
    return np.array([[x0, x0 + s, x0 + s, x0, x0], [y0, y0, y0 + s, y0 + s, y0]], dtype=np.float64)


def test_overlap_area_equals_the_exact_clipping():
    rng = np.random.default_rng(3)
    checked = 0
    for _ in range(300):
        P = random_hull(rng, 0.0, 0.0, 1.0)
        Q = random_hull(rng, rng.uniform(-1.2, 1.2), rng.uniform(-1.2, 1.2), rng.uniform(0.3, 1.5))
        if rng.random() < 0.5:
            Q = Q[:, ::-1].copy()                   # clockwise clip polygon
        got, want = scenario.convex_overlap_area(P, Q), exact_overlap_area(P, Q)
        if want == 0:
            assert got == 0.0
            continue
        # relative 1e-12 from the decision threshold up; below it the shoelace's cancellation error scales with the
        # coordinates, not with the sliver's area, so the bound is 1e-15 absolute there
        assert abs(Fraction(got) - want) <= Fraction(1, 10 ** 12) * max(want, Fraction(1, 1000)), (got, float(want))
        checked += 1
    assert checked > 150


def test_overlap_area_literal_cases():
    sq = square(0.0, 0.0, 2.0)
    assert scenario.convex_overlap_area(sq, sq) == 4.0
    assert scenario.convex_overlap_area(sq, square(0.5, 0.5, 1.0)) == 1.0          # containment: the inner area
    assert scenario.convex_overlap_area(square(0.5, 0.5, 1.0), sq) == 1.0
    assert scenario.convex_overlap_area(sq, square(1.0, 1.0, 2.0)) == 1.0
    far = square(2.5, 0.0, 1.0)
    assert scenario.convex_overlap_area(sq, far) == 0.0                           # disjoint boxes: exactly 0.0
    assert scenario.convex_overlap_area(sq, square(2.0, 2.0, 1.0)) == 0.0         # touching corner
    assert scenario.convex_overlap_area(sq, sq[:, :3]) == 0.0                     # fewer than 3 vertices
    flat = np.array([[0.0, 1.0, 2.0, 0.0], [0.0, 1.0, 2.0, 0.0]])
    assert scenario.convex_overlap_area(sq, flat) == 0.0                          # degenerate clip polygon
    rng = np.random.default_rng(5)
    for _ in range(100):                          # orientation of either polygon changes no decision
        P, Q = random_hull(rng, 0.0, 0.0, 0.5), random_hull(rng, rng.uniform(-0.6, 0.6), rng.uniform(-0.6, 0.6), 0.4)
        Pr, Qr = P[:, ::-1].copy(), Q[:, ::-1].copy()
        areas = [scenario.convex_overlap_area(a, b) for a in (P, Pr) for b in (Q, Qr)]
        assert len({a > scenario.COUPLING_AREA_THRESHOLD for a in areas}) == 1
        assert max(areas) - min(areas) <= 1e-12 * max(1.0, max(areas))


@pytest.mark.parametrize("mpa_type", ["triple_speed", "single_speed"])
def test_reachable_set_adjacency_and_relations(mpa_type):
    mpa = get_mpa(mpa_type, non_convex=True)
    sc = scenario.commonroad_scenario(mpa, 40, seed=2, allow_shared_paths=True)
    rng = np.random.default_rng(1)
    pose = np.array([[v.x_start, v.y_start, v.yaw_start] for v in sc.vehicles])
    trim = rng.integers(1, mpa.n_trims + 1, size=40)
    area = scenario.reachable_set_overlaps(mpa, pose, trim)
    A = scenario.couple_reachable_sets(mpa, pose, trim)
    assert np.array_equal(area, area.T) and np.array_equal(A, A.T) and not A.diagonal().any()
    assert np.array_equal(A, (area > 1e-3).astype(np.int64)) and A.sum() > 0
    for priority in ("coloring", "constant"):
        D_full = None
        for max_cls in (1, 2, 3, 99):
            D, seq, levels = scenario.decide_relations(A, priority, max_cls)
            assert np.array_equal(D | D.T, A.astype(bool)) and not (D & D.T).any()
            assert not (seq & ~D).any() and levels.max() <= max_cls
            assert np.array_equal(levels, scenario.kahn(seq.astype(np.int64)))   # a DAG: kahn raises on a cycle
            for i, j in zip(*np.nonzero(seq)):
                assert levels[i] < levels[j]
            D_full = D if D_full is None else D_full
            assert np.array_equal(D, D_full)
        assert np.array_equal(seq, D)                                         # max_num_CLs >= depth: no cut


def test_runner_coupler_option():
    mpa = get_mpa("triple_speed", non_convex=True)
    sc = scenario.commonroad_scenario(mpa, 20, seed=1)
    with pytest.raises(ValueError):
        scenario.ScenarioRunner(sc, None, coupler="polyshape")
    r = scenario.ScenarioRunner(sc, None, coupler="reachable_set")
    assert np.array_equal(r._adjacency(), scenario.couple_reachable_sets(mpa, r.pose, r.trim))
    assert np.array_equal(scenario.ScenarioRunner(sc, None)._adjacency(), scenario.couple(sc, r.pose))


def test_couple_structs_match_the_c_layout(tmp_path, built):
    from pdmpc_b200 import capi
    header = os.path.join(ROOT, "include", "pdmpc_b200.h")
    structs = {"pdmpc_couple_params": capi.CoupleParamsC, "pdmpc_couple_out": capi.CoupleOutC}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{header}"', "int main(void){"]
    for cname, cls in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines.append("return 0;}")
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == C.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(out[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"


COUPLE = 12   # pdmpc_b200_mex.cpp: enum Command


def test_mex_couple_command_dispatch(built):
    import torch
    matlab = mexfake.FakeMatlab()
    with pytest.raises(mexfake.MexError, match="pdmpc:handle"):
        matlab.call(2, COUPLE, 99.0, np.zeros((2, 3)), np.ones(2))
    if not torch.cuda.is_available():
        with pytest.raises(mexfake.MexError, match="no CPU fallback"):
            matlab.call(1, mexfake.CREATE, 0.0)
        return
    (h,) = matlab.call(1, mexfake.CREATE, 0.0)
    try:
        with pytest.raises(mexfake.MexError, match="COUPLE needs 4 arguments"):
            matlab.call(2, COUPLE, float(h), np.zeros((2, 3)))
    finally:
        matlab.call(0, mexfake.DESTROY, float(h))
        matlab.clear_mex()


def test_couple_matlab_helper_present():
    src = open(os.path.join(ROOT, "p-dmpc_b200", "matlab", "couple_cuda.m")).read()
    assert "COUPLE = 12" in src and "UPLOAD_REACHABLE_SETS = 10" in src and "local_reachable_sets_conv" in src
    shim = open(os.path.join(ROOT, "p-dmpc_b200", "matlab", "pdmpc_b200_mex.cpp")).read()
    assert "COUPLE = 12" in shim and "case COUPLE:" in shim
