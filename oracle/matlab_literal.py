"""Second, independent CPU restatement of the reference's graph search (TEST INFRASTRUCTURE).

Where ``pdmpc_oracle.c`` restates the reference as scalar C loops over the flat
boundary structs, this module follows the MATLAB sources in their own MATRIX
form (outer products, ``diff``, ``min``/``max`` that skip NaN, cell arrays of
2xN polygons) on ``IterationData`` objects, and drives the reference's own
UNMODIFIED priority queue (``oracle/_ref/libpq_ref.so``, compiled from
hlc/optimizer/graph_search/priority_queue/priority_queue_interface_mex.cpp) when
it is available.  Two restatements written against the same sources in
different styles, agreeing on every field, is what pins the C oracle where the
reference ships no golden vectors (SURVEY.md §8c).

Pure Python + numpy: small cases only.  Import from tests/ only.

sin/cos: MATLAB's are closed source.  ``trig="spec"`` uses the algorithm the
oracle and the device share (DESIGN.md §sincos) so results are bit-comparable;
``trig="libm"`` uses numpy's, which tests use to show that discrete results do
not depend on last-bit differences of the trig functions.
"""
from __future__ import annotations

import dataclasses
from typing import List, Optional

import numpy as np

from . import oracle_py

NAN_COL = np.array([[np.nan], [np.nan]])


def _trig(yaw: float, trig: str):
    if trig == "spec":
        s, c = oracle_py.sincos(yaw)
        return c, s
    return float(np.cos(yaw)), float(np.sin(yaw))


# ---------------------------------------------------------------- InterX.m:48-85,108-110
def _D(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """InterX.m:108-110"""
    return (x[:, :-1] - y) * (x[:, 1:] - y)


def interx(L1: np.ndarray, L2: np.ndarray) -> bool:
    if L1.size == 0 or L2.size == 0:                    # :48-52
        return False
    x1 = L1[0, :][:, None]                              # column
    y1 = L1[1, :][:, None]
    x2 = L2[0, :][None, :]                              # row
    y2 = L2[1, :][None, :]
    dx1, dy1 = np.diff(x1, axis=0), np.diff(y1, axis=0)
    dx2, dy2 = np.diff(x2, axis=1), np.diff(y2, axis=1)
    S1 = dx1 * y1[:-1] - dy1 * x1[:-1]                  # :67
    S2 = dx2 * y2[:, :-1] - dy2 * x2[:, :-1]            # :68
    with np.errstate(invalid="ignore"):
        C1 = _D(dx1 * y2 - dy1 * x2, S1) < 0            # :70  (outer products)
        C2 = (_D((y1 * dx2 - x1 * dy2).T, S2.T) < 0).T  # :71
        return bool(np.any(C1 & C2))                    # :74-85


# ---------------------------------------------------------------- intersect_sat.m
def _intersect_a_b(shape1: np.ndarray, shape2: np.ndarray) -> bool:
    edge = np.diff(np.hstack([shape1, shape1[:, :1]]), axis=1)          # :19
    axis = np.vstack([-edge[1], edge[0]])                                # :21
    with np.errstate(invalid="ignore", divide="ignore"):
        normed = axis / np.sqrt(axis[0] * axis[0] + axis[1] * axis[1])   # :23 vecnorm
        # :26-32: explicit a*x + b*y (a 2-term product-sum, evaluated left to right)
        d1 = normed[0][:, None] * shape1[0][None, :] + normed[1][:, None] * shape1[1][None, :]
        d2 = normed[0][:, None] * shape2[0][None, :] + normed[1][:, None] * shape2[1][None, :]
        # MATLAB min/max ignore NaN unless all are NaN
        all_nan = np.isnan(d1).all(axis=1)
        mn1 = np.where(all_nan, np.nan, np.nanmin(np.where(np.isnan(d1), np.inf, d1), axis=1))
        mx1 = np.where(all_nan, np.nan, np.nanmax(np.where(np.isnan(d1), -np.inf, d1), axis=1))
        all_nan2 = np.isnan(d2).all(axis=1)
        mn2 = np.where(all_nan2, np.nan, np.nanmin(np.where(np.isnan(d2), np.inf, d2), axis=1))
        mx2 = np.where(all_nan2, np.nan, np.nanmax(np.where(np.isnan(d2), -np.inf, d2), axis=1))
        return not (np.any(mn1 - mx2 > 0) or np.any(mn2 - mx1 > 0))       # :33-40


def intersect_sat(shape1: np.ndarray, shape2: np.ndarray) -> bool:
    """intersect_sat.m:1-15"""
    if not _intersect_a_b(shape1, shape2):
        return False
    if not _intersect_a_b(shape2, shape1):
        return False
    return True


def intersect_lanelets(shape: np.ndarray, lanelet: np.ndarray) -> bool:
    """intersect_lanelets.m:1-22; lanelet [n, 6] with LaneletInfo columns rx ry lx ly cx cy."""
    for i in range(lanelet.shape[0] - 1):
        if intersect_sat(shape, lanelet[i:i + 2, [0, 1]].T):
            return True
        if intersect_sat(shape, lanelet[i:i + 2, [2, 3]].T):
            return True
    return False


def intersect_lanelet_boundary(shape: np.ndarray, left: np.ndarray, right: np.ndarray) -> bool:
    """intersect_lanelet_boundary.m:1-56"""
    max_x, min_x = shape[0].max(), shape[0].min()
    max_y, min_y = shape[1].max(), shape[1].min()
    for pts in (left, right):
        for n in range(pts.shape[1] - 1):
            seg = pts[:, n:n + 2]
            if (np.all(max_x < seg[0]) or np.all(min_x > seg[0]) or np.all(max_y < seg[1])
                    or np.all(min_y > seg[1])):
                continue
            if intersect_sat(shape, seg):
                return True
    return False


# ---------------------------------------------------------------- vectorize_all_obstacles.m:27-63
def vectorize_all_obstacles(it, Hp: int):
    left, right = it.predicted_lanelet_boundary[:2]
    lanelet = np.hstack([np.asarray(left, float).reshape(2, -1), NAN_COL,
                         np.asarray(right, float).reshape(2, -1), NAN_COL])
    veh = []
    for k in range(Hp):
        polys = list(it.obstacles) + [row[k] for row in it.dynamic_obstacle_area]
        for p in polys:
            assert np.all(p[:, 0] == p[:, -1]), "check_closeness"   # :71-76
        cols = [np.hstack([np.asarray(p, float), NAN_COL]) for p in polys]
        veh.append(np.hstack(cols) if cols else np.zeros((2, 0)))
    return veh, lanelet


# ---------------------------------------------------------------- Tree.m
@dataclasses.dataclass
class Tree:
    x: List[float]
    y: List[float]
    yaw: List[float]
    trim: List[int]
    k: List[int]
    g: List[float]
    h: List[float]
    parent: List[int]

    def size(self) -> int:
        return len(self.x)


@dataclasses.dataclass
class Info:
    """ControlResultsInfo.m:5-17 (nV == 1)"""

    is_exhausted: bool = False
    n_expanded: int = 0
    tree_path: Optional[List[int]] = None
    predicted_trims: Optional[List[int]] = None
    y_predicted: Optional[np.ndarray] = None          # [Hp, 3]
    shapes: Optional[List[np.ndarray]] = None
    pops: Optional[List[int]] = None
    tree: Optional[Tree] = None


def _new_pq(use_reference_pq: bool):
    """The reference's own queue source, or (where it is not built) its restatement on libstdc++'s
    std::priority_queue (StdPQ); neither shares code with the C oracle's heap."""
    if use_reference_pq:
        return oracle_py.ReferencePQ()
    return oracle_py.StdPQ()


def do_graph_search(it, mpa, checker: int, trig: str = "spec", use_reference_pq: bool = True) -> Info:
    """GraphSearch.m:23-109 for one vehicle (iter.amount == 1)."""
    Hp, dt = mpa.Hp, mpa.dt_seconds
    tree = Tree([float(it.x0[0])], [float(it.x0[1])], [float(it.x0[2])], [int(it.trim_indices)], [0], [0.0],
                [0.0], [0])
    pq = _new_pq(use_reference_pq)
    pq.push([1], [0.0])
    if checker == 1:                                    # OptimizerInterface.m:36-46
        veh_obs, lanelet = vectorize_all_obstacles(it, Hp)
    shapes_tmp = {}
    pops = []
    ref = np.asarray(it.reference_trajectory_points, float)
    v_ref = np.asarray(it.v_ref, float)
    info = Info(tree=tree, pops=pops)

    def area(edge, kind, c, s, px, py):
        n = int(mpa.area_npts[edge, kind])
        ax, ay = mpa.area_x[edge, kind, :n], mpa.area_y[edge, kind, :n]
        return np.vstack([c * ax - s * ay + px, s * ax + c * ay + py])   # GraphSearch.m:158-159

    while True:
        nid, _ = pq.pop()                               # :55
        if nid == -1:                                   # :57-61
            info.n_expanded = tree.size()
            info.is_exhausted = True
            return info
        pops.append(nid)
        i = nid - 1
        par = tree.parent[i]
        valid = True
        shape = None
        if par:                                         # eval_edge_exact :111-196
            p = par - 1
            edge = int(mpa.edge_index[tree.trim[p] - 1, tree.trim[i] - 1])
            c, s = _trig(tree.yaw[p], trig)
            shape = area(edge, 0, c, s, tree.x[p], tree.y[p])
            kind = 2 if tree.k[i] == Hp else 1          # :166-174
            bshape = area(edge, kind, c, s, tree.x[p], tree.y[p])
            k = tree.k[i]
            if checker == 1:                            # are_constraints_satisfied_interx.m:17-37
                if interx(shape, veh_obs[k - 1]):
                    valid = False
                elif interx(bshape, lanelet):
                    valid = False
            else:                                       # are_constraints_satisfied_sat.m:15-53
                for o in it.obstacles:
                    if intersect_sat(shape, np.asarray(o, float)):
                        valid = False
                        break
                if valid:
                    for row in it.dynamic_obstacle_area:
                        if intersect_sat(shape, np.asarray(row[k - 1], float)):
                            valid = False
                            break
                if valid:
                    left, right = it.predicted_lanelet_boundary[:2]
                    if intersect_lanelet_boundary(bshape, np.asarray(left, float).reshape(2, -1),
                                                  np.asarray(right, float).reshape(2, -1)):
                        valid = False
        if not valid:
            continue                                    # :75-77
        shapes_tmp[nid] = shape                         # :79
        if tree.k[i] == Hp:                             # :81-90
            path = []
            n = nid
            while n:
                path.append(n)
                n = tree.parent[n - 1]
            path = path[::-1]
            info.tree_path = path
            info.predicted_trims = [tree.trim[q - 1] for q in path[1:]]
            info.y_predicted = np.array([[tree.x[q - 1], tree.y[q - 1], tree.yaw[q - 1]] for q in path[1:]])
            info.shapes = [shapes_tmp[q] for q in path[1:]]
            info.n_expanded = tree.size()
            return info
        # expand_node.m:1-91
        k_exp = tree.k[i] + 1
        succ = np.flatnonzero(mpa.transition[k_exp - 1, tree.trim[i] - 1]) + 1   # :18 find(...)
        c, s = _trig(tree.yaw[i], trig)
        new_ids, new_vals = [], []
        for t2 in succ:
            edge = int(mpa.edge_index[tree.trim[i] - 1, t2 - 1])
            dx, dy, dyaw = mpa.edge_dx[edge], mpa.edge_dy[edge], mpa.edge_dyaw[edge]
            ex = c * dx - s * dy + tree.x[i]
            ey = s * dx + c * dy + tree.y[i]
            eyaw = tree.yaw[i] + dyaw
            v = np.array([ex - ref[k_exp - 1, 0], ey - ref[k_exp - 1, 1]])
            nrm = float(np.sqrt(v[0] * v[0] + v[1] * v[1]))
            eg = tree.g[i] + nrm * nrm                                            # :61  norm(.)^2
            eh = 0.0
            d_max = 0.0
            for i_t in range(1, Hp - k_exp + 1):                                  # :66-73
                d_max = d_max + dt * v_ref[k_exp + i_t - 1]
                w = np.array([ex - ref[k_exp + i_t - 1, 0], ey - ref[k_exp + i_t - 1, 1]])
                m = max(0.0, float(np.sqrt(w[0] * w[0] + w[1] * w[1])) - d_max)
                eh = eh + m * m
            tree.x.append(float(ex)); tree.y.append(float(ey)); tree.yaw.append(float(eyaw))
            tree.trim.append(int(t2)); tree.k.append(k_exp); tree.g.append(float(eg)); tree.h.append(float(eh))
            tree.parent.append(nid)
            new_ids.append(tree.size())
            new_vals.append(float(eg) * 1 + float(eh) * 1)                        # GraphSearch.m:100-102
        if new_ids:
            pq.push(new_ids, new_vals)                                            # :104


# ---------------------------------------------------------------- joint search (iter.amount > 1)
def cartprod(*sets):
    """hlc/optimizer/common/cartprod.m:30-61: rows = ind2sub over the sets' sizes, FIRST set fastest."""
    sizes = [len(x) for x in sets]
    sets = [np.sort(np.asarray(x)) for x in sets]
    out = np.zeros((int(np.prod(sizes)), len(sets)), dtype=np.int64)
    for i in range(out.shape[0]):
        ix = np.unravel_index(i, sizes, order="F")
        for j in range(len(sets)):
            out[i, j] = sets[j][ix[j]]
    return out


@dataclasses.dataclass
class JointInfo:
    is_exhausted: bool = False
    n_expanded: int = 0
    pops: Optional[List[int]] = None
    tree_path: Optional[List[int]] = None
    predicted_trims: Optional[np.ndarray] = None      # [nV, Hp]
    y_predicted: Optional[np.ndarray] = None          # [nV, Hp, 3]
    g_path: Optional[List[float]] = None


def do_joint_graph_search(iters, mpa, trig: str = "spec", use_reference_pq: bool = True) -> JointInfo:
    """GraphSearch.m:23-109 with iter.amount = nV > 1, matrix form as the MATLAB code has it: nV x nNodes tree
    arrays (Tree.m), successor ids through mpa.trim_tuple and cartprod with the per-vehicle radix offsets
    (expand_node.m:15-31), the vehicles' checks in order with the shapes of the vehicles before them
    (GraphSearch.m:150-192, are_constraints_satisfied_sat.m:15-53).  iters[0] carries the search's obstacles."""
    Hp, dt, nV, nT = mpa.Hp, mpa.dt_seconds, len(iters), mpa.n_trims
    trim_tuple = cartprod(*[np.arange(1, nT + 1)] * nV)                       # MotionPrimitiveAutomaton.m:141
    X = [np.array([float(it.x0[0]) for it in iters])]
    Y = [np.array([float(it.x0[1]) for it in iters])]
    YAW = [np.array([float(it.x0[2]) for it in iters])]
    TRIM = [np.array([int(it.trim_indices) for it in iters])]
    K, G, H, PARENT = [0], [0.0], [0.0], [0]
    ref = np.stack([np.asarray(it.reference_trajectory_points, float) for it in iters])   # [nV, Hp, 2]
    v_ref = np.stack([np.asarray(it.v_ref, float) for it in iters])
    pq = _new_pq(use_reference_pq)
    pq.push([1], [0.0])
    info = JointInfo(pops=[])

    def area(edge, kind, c, s, px, py):
        n = int(mpa.area_npts[edge, kind])
        ax, ay = mpa.area_x[edge, kind, :n], mpa.area_y[edge, kind, :n]
        return np.vstack([c * ax - s * ay + px, s * ax + c * ay + py])

    while True:
        nid, _ = pq.pop()
        if nid == -1:
            info.n_expanded, info.is_exhausted = len(K), True
            return info
        info.pops.append(nid)
        i = nid - 1
        par = PARENT[i]
        valid = True
        if par:
            p = par - 1
            shapes = [None] * nV
            for v in range(nV):
                edge = int(mpa.edge_index[TRIM[p][v] - 1, TRIM[i][v] - 1])
                c, s = _trig(YAW[p][v], trig)
                shapes[v] = area(edge, 0, c, s, X[p][v], Y[p][v])
                bshape = area(edge, 2 if K[i] == Hp else 1, c, s, X[p][v], Y[p][v])
                for o in iters[0].obstacles:
                    if valid and intersect_sat(shapes[v], np.asarray(o, float)):
                        valid = False
                for row in iters[0].dynamic_obstacle_area:
                    if valid and intersect_sat(shapes[v], np.asarray(row[K[i] - 1], float)):
                        valid = False
                for u in range(v - 1, -1, -1):                               # are_constraints_satisfied_sat.m:37-44
                    if valid and intersect_sat(shapes[u], shapes[v]):
                        valid = False
                if valid:
                    left, right = iters[v].predicted_lanelet_boundary[:2]
                    if intersect_lanelet_boundary(bshape, np.asarray(left, float).reshape(2, -1),
                                                  np.asarray(right, float).reshape(2, -1)):
                        valid = False
                if not valid:
                    break                                                     # GraphSearch.m:189-191
        if not valid:
            continue
        if K[i] == Hp:
            path = []
            n = nid
            while n:
                path.append(n)
                n = PARENT[n - 1]
            path = path[::-1]
            info.tree_path = path
            info.predicted_trims = np.array([[TRIM[q - 1][v] for q in path[1:]] for v in range(nV)])
            info.y_predicted = np.array([[[X[q - 1][v], Y[q - 1][v], YAW[q - 1][v]] for q in path[1:]] for v in range(nV)])
            info.g_path = [G[q - 1] for q in path]
            info.n_expanded = len(K)
            return info
        k_exp = K[i] + 1
        per_vehicle = []
        for v in range(nV):                                                   # expand_node.m:17-26
            tr = np.flatnonzero(mpa.transition[k_exp - 1, TRIM[i][v] - 1]) + 1
            per_vehicle.append(tr if v == 0 else (tr - 1) * nT ** v)
        ids = cartprod(*per_vehicle).sum(axis=1)                              # :28
        new_ids, new_vals = [], []
        for sid in ids:
            trims = trim_tuple[sid - 1]                                       # :41
            ex, ey, eyaw = np.zeros(nV), np.zeros(nV), np.zeros(nV)
            eg, eh = G[i], 0.0
            for v in range(nV):
                edge = int(mpa.edge_index[TRIM[i][v] - 1, trims[v] - 1])
                c, s = _trig(YAW[i][v], trig)
                ex[v] = c * mpa.edge_dx[edge] - s * mpa.edge_dy[edge] + X[i][v]
                ey[v] = s * mpa.edge_dx[edge] + c * mpa.edge_dy[edge] + Y[i][v]
                eyaw[v] = YAW[i][v] + mpa.edge_dyaw[edge]
                d0, d1 = ex[v] - ref[v, k_exp - 1, 0], ey[v] - ref[v, k_exp - 1, 1]
                nrm = float(np.sqrt(d0 * d0 + d1 * d1))
                eg = eg + nrm * nrm                                           # :61
                d_max = 0.0
                for i_t in range(1, Hp - k_exp + 1):                          # :66-73
                    d_max = d_max + dt * v_ref[v, k_exp + i_t - 1]
                    w0, w1 = ex[v] - ref[v, k_exp + i_t - 1, 0], ey[v] - ref[v, k_exp + i_t - 1, 1]
                    m = max(0.0, float(np.sqrt(w0 * w0 + w1 * w1)) - d_max)
                    eh = eh + m * m
            X.append(ex); Y.append(ey); YAW.append(eyaw); TRIM.append(np.array(trims))
            K.append(k_exp); G.append(float(eg)); H.append(float(eh)); PARENT.append(nid)
            new_ids.append(len(K))
            new_vals.append(float(eg) * 1 + float(eh) * 1)
        if new_ids:
            pq.push(new_ids, new_vals)


# ---------------------------------------------------------------- MonteCarloTreeSearch.m:29-251
def do_mcts(it, mpa, checker: int, seed: int, n_expansions_max: int = 250, trig: str = "spec",
            use_reference_pq: bool = True) -> Info:
    """MonteCarloTreeSearch.run_optimizer + do_graph_search for one vehicle, in the
    reference's own array form: `children` is the (max branching x nodes) uint32 matrix of
    :64, poses are 3-vectors updated with the 3x3 `transform` of :127-132, and the random
    stream is numpy's RandomState (MT19937 + 53-bit doubles == MATLAB's 'mt19937ar' rand,
    an implementation independent of the oracle's)."""
    Hp = mpa.Hp
    rs = np.random.RandomState(int(seed) if int(seed) != 0 else 5489)
    random_numbers = rs.random_sample(Hp * n_expansions_max)                 # :52
    B = int(mpa.transition.sum(axis=2).max())                                 # :53 maximum_branching_factor
    succ_of = lambda trim, step: np.flatnonzero(mpa.transition[step - 1, trim - 1]) + 1   # successor_trims{trim, step}
    info = Info()
    trims = np.zeros(n_expansions_max + Hp + 2, dtype=np.int64)                    # MATLAB grows on assignment
    parents = np.zeros(n_expansions_max + Hp + 2, dtype=np.int64)
    children = np.zeros((B, n_expansions_max + Hp + 2), dtype=np.int64)            # column j <-> node j+1
    root_pose = np.array([float(it.x0[0]), float(it.x0[1]), float(it.x0[2])])
    trims[0] = int(it.trim_indices)
    children[:succ_of(trims[0], 1).size, 0] = 1                               # :69
    n_nodes = 1
    pq = _new_pq(use_reference_pq)
    shapes_tmp = {}
    if checker == 1:
        veh_obs, lanelet = vectorize_all_obstacles(it, Hp)
    ref = np.asarray(it.reference_trajectory_points, float).T                 # 2 x Hp  (:83)
    n_expansions = 0
    n_traversals = 0
    is_finished = False
    steps = []

    def check(shape, bshape, k):
        if checker == 1:
            if interx(shape, veh_obs[k - 1]):
                return False
            return not interx(bshape, lanelet)
        for o in it.obstacles:
            if intersect_sat(shape, np.asarray(o, float)):
                return False
        for row in it.dynamic_obstacle_area:
            if intersect_sat(shape, np.asarray(row[k - 1], float)):
                return False
        left, right = it.predicted_lanelet_boundary[:2]
        return not intersect_lanelet_boundary(bshape, np.asarray(left, float).reshape(2, -1),
                                              np.asarray(right, float).reshape(2, -1))

    def area(edge, kind):
        n = int(mpa.area_npts[edge, kind])
        return np.vstack([mpa.area_x[edge, kind, :n], mpa.area_y[edge, kind, :n]])

    def rot_apply(c, s, pts, start):
        # transform(1:2,1:2) * area + start_pose(1:2): row i = c*ax + (-s)*ay + px (2-term product sums)
        return np.vstack([c * pts[0] + (-s) * pts[1] + start[0], s * pts[0] + c * pts[1] + start[1]])

    while n_expansions < n_expansions_max and not is_finished:                # :86
        node_id = 1
        solution_cost = 0.0
        node_pose = root_pose.copy()
        is_valid = False
        child_position = node_parent = None
        for i_step in range(1, Hp + 1):                                       # :92
            is_valid = False
            n_traversals += 1
            trim_positions = np.flatnonzero(children[:, node_id - 1]) + 1     # :97
            n_trims = trim_positions.size
            if n_trims != 0:
                child_position = int(trim_positions[int(np.ceil(random_numbers[n_traversals - 1] * n_trims)) - 1])
            else:
                if node_id != 1:                                              # :106-109
                    parent_id = int(parents[node_id - 1])
                    children[children[:, parent_id - 1] == node_id, parent_id - 1] = 0
                    break
                is_finished = True                                            # :110-113
                break
            steps.append((node_id << 8) | child_position)
            parent_trim = int(trims[node_id - 1])
            goal_trim = int(succ_of(parent_trim, i_step)[child_position - 1])
            edge = int(mpa.edge_index[parent_trim - 1, goal_trim - 1])
            c, s = _trig(float(node_pose[2]), trig)
            dpose = np.array([mpa.edge_dx[edge], mpa.edge_dy[edge], mpa.edge_dyaw[edge]])
            start_pose = node_pose.copy()
            # :132 node_pose + transform * dpose, rows of the 3x3 product written out left to right
            tp = np.array([c * dpose[0] + (-s) * dpose[1] + 0.0 * dpose[2],
                           s * dpose[0] + c * dpose[1] + 0.0 * dpose[2],
                           0.0 * dpose[0] + 0.0 * dpose[1] + 1.0 * dpose[2]])
            node_pose = node_pose + tp
            v = node_pose[:2] - ref[:, i_step - 1]
            nrm = float(np.sqrt(v[0] * v[0] + v[1] * v[1]))
            solution_cost = solution_cost + nrm * nrm                         # :137
            if children[child_position - 1, node_id - 1] != 1:                # :139-144
                node_id = int(children[child_position - 1, node_id - 1])
                continue
            n_expansions += 1
            node_parent = node_id
            shape = rot_apply(c, s, area(edge, 0), start_pose)                # :151
            if i_step != Hp:                                                  # :153-159
                bshape = rot_apply(c, s, area(edge, 1), start_pose)
                child_succ = succ_of(goal_trim, i_step + 1)
            else:
                bshape = rot_apply(c, s, area(edge, 2), start_pose)
                child_succ = np.zeros(0, dtype=np.int64)
            is_valid = check(shape, bshape, i_step)                           # :161-170
            if not is_valid:
                children[child_position - 1, node_parent - 1] = 0             # :174
                break
            n_nodes += 1                                                      # :177-184
            parents[n_nodes - 1] = node_parent
            trims[n_nodes - 1] = goal_trim
            children[:child_succ.size, n_nodes - 1] = 1
            children[child_position - 1, node_parent - 1] = n_nodes
            shapes_tmp[n_nodes] = shape
            node_id = n_nodes
        if is_valid:                                                          # :189-193
            pq.push([node_id], [solution_cost])
            children[child_position - 1, node_parent - 1] = 0
    best, cost = pq.pop()                                                     # :197
    info.n_expanded = n_expansions
    info.pops = steps
    info.n_traversals = n_traversals
    if best == -1:
        info.is_exhausted = True
        return info
    path = []
    n = int(best)
    while n:
        path.append(n)
        n = int(parents[n - 1])
    path = path[::-1]
    pose = np.zeros((3, len(path)))
    pose[:, 0] = root_pose
    for i in range(1, len(path)):                                             # :220-232
        edge = int(mpa.edge_index[trims[path[i - 1] - 1] - 1, trims[path[i] - 1] - 1])
        c, s = _trig(float(pose[2, i - 1]), trig)
        d = np.array([mpa.edge_dx[edge], mpa.edge_dy[edge], mpa.edge_dyaw[edge]])
        pose[:, i] = pose[:, i - 1] + np.array([c * d[0] + (-s) * d[1] + 0.0 * d[2],
                                                s * d[0] + c * d[1] + 0.0 * d[2],
                                                0.0 * d[0] + 0.0 * d[1] + 1.0 * d[2]])
    info.tree_path = path
    info.predicted_trims = [int(trims[q - 1]) for q in path[1:]]
    info.y_predicted = pose[:, 1:].T.copy()
    info.shapes = [shapes_tmp[q] for q in path[1:]]
    info.cost = float(cost)
    return info
