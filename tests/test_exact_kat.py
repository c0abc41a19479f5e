"""Known-answer vectors computed in EXACT rational arithmetic (Python fractions), independent of both CPU
restatements: the sign decisions of InterX on literal polylines, and the cost arithmetic of expand_node
(operation order and every rounding) on a literal motion-primitive automaton.

InterX.m:63-85: coordinates are multiples of 1/64 below 8 in magnitude, so every difference, product and sum
of the reference's expressions is exact in double precision — the floating-point boolean must equal the
rational one, including the strict inequalities on touching / collinear configurations and the NaN separators.

expand_node.m:50-75: IEEE double arithmetic is emulated operation by operation (every +, -, *, / and sqrt is the
exact rational result rounded to nearest), in the reference's order; g and h along the path the oracle returns
must equal the emulated values bit for bit (a fused multiply-add, a reordered sum or pow() instead of x*x
anywhere in the chain would show)."""
from decimal import Decimal, getcontext
from fractions import Fraction

import numpy as np

from oracle import matlab_literal as ml
from oracle import oracle_py
from pdmpc_b200.mpa import MotionPrimitiveAutomaton
from pdmpc_b200.records import CHECKER_SAT, IterationData, SearchBatch


# ---------------------------------------------------------------------------------------------- InterX
def interx_exact(L1, L2) -> bool:
    """InterX.m:63-85 over the rationals; a NaN coordinate makes every comparison it enters false."""
    def seg(L):
        out = []
        for i in range(L.shape[1] - 1):
            c = L[:, i:i + 2]
            out.append(None if np.isnan(c).any() else tuple(Fraction(float(v)) for v in (c[0, 0], c[1, 0], c[0, 1], c[1, 1])))
        return out
    for s1 in seg(L1):
        for s2 in seg(L2):
            if s1 is None or s2 is None:
                continue
            x1, y1, x1b, y1b = s1
            x2, y2, x2b, y2b = s2
            dx1, dy1, dx2, dy2 = x1b - x1, y1b - y1, x2b - x2, y2b - y2
            S1, S2 = dx1 * y1 - dy1 * x1, dx2 * y2 - dy2 * x2
            c1 = (dx1 * y2 - dy1 * x2 - S1) * (dx1 * y2b - dy1 * x2b - S1) < 0
            c2 = (y1 * dx2 - x1 * dy2 - S2) * (y1b * dx2 - x1b * dy2 - S2) < 0
            if c1 and c2:
                return True
    return False


def q64(a):
    return np.round(np.asarray(a, dtype=np.float64) * 64) / 64


def closed(p):
    return np.column_stack([p, p[:, :1]])


NANCOL = np.array([[np.nan], [np.nan]])


def test_interx_literal_cases():
    sq = closed(np.array([[0.0, 1.0, 1.0, 0.0], [0.0, 0.0, 1.0, 1.0]]))
    cases = [
        (sq, closed(np.array([[0.5, 1.5, 1.5, 0.5], [0.5, 0.5, 1.5, 1.5]])), True),     # proper crossing
        (sq, closed(np.array([[1.0, 2.0, 2.0, 1.0], [0.0, 0.0, 1.0, 1.0]])), False),    # shared edge: collinear, no hit
        (sq, closed(np.array([[1.0, 2.0, 2.0, 1.0], [1.0, 1.0, 2.0, 2.0]])), False),    # touching in one vertex
        (sq, closed(np.array([[0.25, 0.75, 0.75, 0.25], [0.25, 0.25, 0.75, 0.75]])), False),   # containment is not detected
        (sq, np.array([[0.5, 0.5], [-1.0, 0.5]]), True),                                # segment ends inside
        (sq, np.array([[0.5, 0.5], [-1.0, 0.0]]), False),                               # ... ends ON the edge: strict
        (sq, np.array([[-1.0, 2.0], [0.0, 0.0]]), False),                               # runs along an edge
        (sq, np.column_stack([np.array([[2.0, 3.0], [2.0, 3.0]]), NANCOL, np.array([[0.5, 0.5], [-1.0, 2.0]]), NANCOL]), True),
        (sq, np.column_stack([np.array([[-1.0, -0.5], [0.5, 0.5]]), NANCOL, np.array([[1.5, 2.0], [0.5, 0.5]])]), False),  # pseudo-segment across the NaN would cross
        (sq, np.zeros((2, 0)), False),
        (sq, np.array([[0.5], [0.5]]), False),
    ]
    for k, (a, b, want) in enumerate(cases):
        assert interx_exact(a, b) == want, k
        assert oracle_py.interx(a, b) == want, k
        assert ml.interx(a, b) == want, k


def test_interx_random_dyadic_polylines_against_exact_arithmetic():
    rng = np.random.default_rng(7)
    hits = 0
    for _ in range(400):
        n1 = rng.integers(4, 8)
        ang = np.sort(rng.uniform(0, 2 * np.pi, n1))
        c = rng.uniform(-2, 2, 2)
        shape = closed(q64(np.vstack([c[0] + 0.4 * np.cos(ang), c[1] + 0.4 * np.sin(ang)])))
        parts = []
        for _p in range(rng.integers(1, 5)):
            m = rng.integers(2, 7)
            cc = c + rng.normal(scale=0.6, size=2)
            poly = q64(np.vstack([cc[0] + rng.uniform(-0.5, 0.5, m), cc[1] + rng.uniform(-0.5, 0.5, m)]))
            if rng.random() < 0.3:                      # vertices snapped onto shape vertices: exact zeros
                poly[:, 0] = shape[:, rng.integers(0, n1)]
            parts += [closed(poly), NANCOL]
        obst = np.column_stack(parts)
        want = interx_exact(shape, obst)
        hits += want
        assert oracle_py.interx(shape, obst) == want
        assert ml.interx(shape, obst) == want
        assert oracle_py.interx(obst, shape) == interx_exact(obst, shape)
    assert 50 < hits < 350


# ---------------------------------------------------------------------------------------- expand_node costs
getcontext().prec = 80


def rn(x: Fraction) -> float:
    return x.numerator / x.denominator                 # int / int: correctly rounded


def F(x: float) -> Fraction:
    return Fraction(float(x))


def rn_sqrt(x: Fraction) -> float:
    d = (Decimal(x.numerator) / Decimal(x.denominator)).sqrt()
    return float(d)                                    # 80 digits, then one correctly rounded conversion


def add(a, b): return rn(F(a) + F(b))
def sub(a, b): return rn(F(a) - F(b))
def mul(a, b): return rn(F(a) * F(b))


def literal_mpa(Hp=3, dt=0.2):
    """Two trims (1 standstill, 2 moving), every transition allowed, yaw-preserving maneuvers with dyadic offsets."""
    nT = 2
    ef, et = np.array([1, 1, 2, 2], dtype=np.int32), np.array([1, 2, 1, 2], dtype=np.int32)
    dx = np.array([0.0, 0.109375, 0.078125, 0.21875])
    dy = np.array([0.0, 0.015625, -0.03125, 0.046875])
    area = np.array([[-0.12, 0.12, 0.12, -0.12, -0.12], [-0.06, -0.06, 0.06, 0.06, -0.06]])
    ax = np.zeros((4, 3, 8)); ay = np.zeros((4, 3, 8))
    for e in range(4):
        for k in range(3):
            ax[e, k, :5] = area[0] + dx[e] / 2
            ay[e, k, :5] = area[1] + dy[e] / 2
    edge_index = np.array([[0, 1], [2, 3]], dtype=np.int32)
    return MotionPrimitiveAutomaton(
        mpa_type="literal", Hp=Hp, dt_seconds=dt, non_convex=False, recursive_feasibility=False,
        trim_steering=np.zeros(nT), trim_speed=np.array([0.0, 0.75]), transition=np.ones((Hp, nT, nT), dtype=np.uint8),
        adjacency=np.ones((nT, nT), dtype=np.uint8), edge_from=ef, edge_to=et, edge_dx=dx, edge_dy=dy,
        edge_dyaw=np.zeros(4), area_npts=np.full((4, 3), 5, dtype=np.int32), area_x=ax, area_y=ay,
        distance_to_equilibrium=np.zeros(nT), edge_index=edge_index)


def emulate_costs(mpa, x0, y0, trims, ref, v_ref, dt):
    """g, h of the nodes along a trim sequence, expand_node.m:50-75 with yaw = 0 (cos = 1, sin = 0), every operation
    rounded as IEEE double rounds it."""
    Hp = mpa.Hp
    x, y, g = x0, y0, 0.0
    gs, hs = [0.0], [0.0]
    for k in range(1, Hp + 1):
        e = int(mpa.edge_index[trims[k - 1] - 1, trims[k] - 1])
        mdx, mdy = float(mpa.edge_dx[e]), float(mpa.edge_dy[e])
        c, s = 1.0, 0.0
        x_new = add(sub(mul(c, mdx), mul(s, mdy)), x)            # :53  c*dx - s*dy + x
        y_new = add(add(mul(s, mdx), mul(c, mdy)), y)            # :54
        ddx, ddy = sub(x_new, ref[k - 1][0]), sub(y_new, ref[k - 1][1])
        nrm = rn_sqrt(F(add(mul(ddx, ddx), mul(ddy, ddy))))      # norm([ddx; ddy])
        g = add(g, mul(nrm, nrm))                                # :61  g + norm(...)^2
        h, d_max = 0.0, 0.0
        for it in range(1, Hp - k + 1):                          # :66-73
            d_max = add(d_max, mul(dt, v_ref[k + it - 1]))
            hx, hy = sub(x_new, ref[k + it - 1][0]), sub(y_new, ref[k + it - 1][1])
            m = max(0.0, sub(rn_sqrt(F(add(mul(hx, hx), mul(hy, hy)))), d_max))
            h = add(h, mul(m, m))
        gs.append(g); hs.append(h)
        x, y = x_new, y_new
    return np.array(gs), np.array(hs), (x, y)


def test_expand_node_costs_against_emulated_ieee_arithmetic():
    rng = np.random.default_rng(3)
    use_reference_pq = oracle_py.have_reference_pq()
    for Hp, dt in ((3, 0.2), (4, 0.2), (3, 0.25)):
        mpa = literal_mpa(Hp, dt)
        iters = []
        for _ in range(24):
            x0, y0 = (float(v) for v in rng.uniform(-1, 1, 2))
            ref = np.cumsum(rng.uniform(0.02, 0.2, (Hp, 2)), axis=0) + [x0, y0]
            v_ref = rng.uniform(0.1, 0.9, Hp)
            iters.append(IterationData(x0=np.array([x0, y0, 0.0, 0.0]), trim_indices=1, reference_trajectory_points=ref, v_ref=v_ref))
        batch = SearchBatch.from_iters(iters, Hp, CHECKER_SAT, dt)
        res = oracle_py.plan_batch(mpa, batch)
        assert not res.is_exhausted.any()
        for i, it in enumerate(iters):
            g, h, (x, y) = emulate_costs(mpa, float(it.x0[0]), float(it.x0[1]), res.trims[i].tolist(),
                                         it.reference_trajectory_points.tolist(), it.v_ref.tolist(), dt)
            assert np.array_equal(g.view(np.uint64), res.g_path[i].view(np.uint64)), (Hp, dt, i)
            assert np.array_equal(h.view(np.uint64), res.h_path[i].view(np.uint64)), (Hp, dt, i)
            assert (x, y) == (res.y_predicted[i, -1, 0], res.y_predicted[i, -1, 1])
            # the matrix-form restatement follows the same arithmetic
            info = ml.do_graph_search(it, mpa, CHECKER_SAT, use_reference_pq=use_reference_pq)
            g2 = np.array([info.tree.g[j - 1] for j in info.tree_path])      # node ids are 1-based
            h2 = np.array([info.tree.h[j - 1] for j in info.tree_path])
            assert np.array_equal(g2.view(np.uint64), g.view(np.uint64)) and np.array_equal(h2.view(np.uint64), h.view(np.uint64))


import pytest  # noqa: E402


@pytest.mark.gpu
def test_cuda_costs_against_emulated_ieee_arithmetic(planner):
    """The same literal automaton through the C ABI: the CUDA path's g, h and end poses equal the operation-by-operation
    emulation in exact rational arithmetic (no oracle involved)."""
    rng = np.random.default_rng(11)
    for Hp, dt in ((3, 0.2), (4, 0.2)):
        mpa = literal_mpa(Hp, dt)
        planner.upload_mpa(mpa)
        iters = []
        for _ in range(40):
            x0, y0 = (float(v) for v in rng.uniform(-1, 1, 2))
            ref = np.cumsum(rng.uniform(0.02, 0.2, (Hp, 2)), axis=0) + [x0, y0]
            iters.append(IterationData(x0=np.array([x0, y0, 0.0, 0.0]), trim_indices=1, reference_trajectory_points=ref,
                                       v_ref=rng.uniform(0.1, 0.9, Hp)))
        batch = SearchBatch.from_iters(iters, Hp, CHECKER_SAT, dt)
        for variant in (1, 4):
            planner.set_variant(variant)
            res = planner.plan_batch(batch)
            for i, it in enumerate(iters):
                g, h, (x, y) = emulate_costs(mpa, float(it.x0[0]), float(it.x0[1]), res.trims[i].tolist(),
                                             it.reference_trajectory_points.tolist(), it.v_ref.tolist(), dt)
                assert np.array_equal(g.view(np.uint64), res.g_path[i].view(np.uint64)), (variant, i)
                assert np.array_equal(h.view(np.uint64), res.h_path[i].view(np.uint64)), (variant, i)
                assert (x, y) == (res.y_predicted[i, -1, 0], res.y_predicted[i, -1, 1])
        planner.set_variant(0)
