"""Synthetic scenario harness: produces the search records of the BASELINE configs.

Host-side Python (numpy) stand-in for the parts of the reference that FEED the
hot path and stay MATLAB in the drop-in (SURVEY.md §2 "caller" rows): scenario
set-up, reference-trajectory sampling, predicted lanelet boundary, coupling,
prioritisation, computation levels, obstacle assembly, closed loop with the
perfect `Simulation` plant.  It exists so that tests and bench.py have inputs of
the named shapes without MATLAB; it is NOT part of the accelerated path.

Follows (reference file:line), with documented simplifications marked [dev]:
  * circle scenario ............... scenarios/free_space/Circle.m:16-42
  * road network ................... scenarios/road_network/Commonroad.m:5-48,
                                     get_reference_lanelets_loop.m:24-154,
                                     generate_reference_path_loop.m:1-46
  * lanelet boundary per lanelet ... RoadDataCommonRoad.get_lanelet_boundary :262-290
                                     [dev] merging/forking extensions (:292-388) omitted
  * reference trajectory ........... hlc/controller/common/get_reference_trajectory.m:1-48,
                                     sample_reference_trajectory.m:1-103,
                                     get_arc_distance_to_endpoint.m
  * predicted lanelets / boundary .. get_predicted_lanelets.m:1-63, get_lanelets_boundary.m:1-75
  * coupling ....................... [dev] corridor-distance proxy for ReachableSetCoupler.m:5-54 (couple, the default),
                                     or ReachableSetCoupler.m:5-54 with the overlap area by a convex clipping instead
                                     of polyshape intersect (couple_reachable_sets, DESIGN.md §4.12)
  * priorities ..................... ConstantPrioritizer.m:6-18, ColoringPrioritizer.m:11-153,
                                     Prioritizer.directed_coupling_from_priorities :62-74
  * computation levels ............. utility/kahn.m:1-24
  * obstacle assembly .............. PrioritizedController.m:297-324,449-566
                                     (sequential predecessors -> predicted areas;
                                      successors at standstill -> static obstacle)
  * plant .......................... plant/Simulation.m:86-117
  * exhaustion fallback ............ [dev] local only: PrioritizedController.m:568-621,678-718
                                     (standstill plan / previous plan shifted); graph-wide
                                     fallback propagation (:623-676) omitted
"""
from __future__ import annotations

import dataclasses
import os
from typing import Callable, List, Optional, Sequence

import math

import numpy as np

from .mpa import VEH_LENGTH, VEH_WIDTH, MotionPrimitiveAutomaton
from .records import CHECKER_INTERX, CHECKER_SAT, BatchResult, IterationData, SearchBatch, TimestepDeps

_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "lab_map.npz")

# get_reference_lanelets_loop.m:24-37 (lanelet ids, 1-based)
_LOOPS = {
    1: [4, 6, 8, 60, 58, 56, 54, 80, 82, 84, 86, 34, 32, 30, 28, 2],
    2: [1, 3, 23, 10, 12, 17, 43, 38, 36, 49, 29, 27],
    3: [64, 62, 75, 55, 53, 79, 81, 101, 88, 90, 95, 69],
    4: [40, 45, 97, 92, 94, 100, 83, 85, 33, 31, 48, 42],
    5: [5, 7, 59, 57, 74, 68, 66, 71, 19, 14, 16, 22],
    6: [41, 39, 20, 63, 61, 57, 55, 67, 65, 98, 37, 35, 31, 29],
    7: [3, 5, 9, 11, 72, 91, 93, 81, 83, 87, 89, 46, 13, 15],
}
# path id -> (loop, starting lanelet): get_reference_lanelets_loop.m:39-127 (ids 1..41)
_PATH_START = {}
for _loop, _starts, _first in (
        (1, [4, 8, 58, 54, 82, 86, 32, 28], 1), (2, [1, 10, 17, 38, 49], 9),
        (3, [64, 75, 79, 88, 95], 14), (4, [42, 45, 92, 100, 33], 19),
        (5, [22, 59, 68, 19, 14], 24), (6, [39, 61, 55, 65, 35, 29], 29),
        (7, [15, 5, 11, 93, 83, 89], 35)):
    for _i, _s in enumerate(_starts):
        _PATH_START[_first + _i] = (_loop, _s)
_PATH_START[41] = (5, 71)


class RoadMap:
    """Lanelet geometry + the per-lanelet boundaries the planner is constrained by."""

    def __init__(self, path: str = _DATA):
        z = np.load(path)
        ptr = z["ptr"]
        self.n = ptr.size - 1
        self.lanelets = []   # [n_pts, 6]: rx ry lx ly cx cy  (LaneletInfo.m)
        for i in range(self.n):
            a, b = ptr[i], ptr[i + 1]
            rx, ry, lx, ly = z["rx"][a:b], z["ry"][a:b], z["lx"][a:b], z["ly"][a:b]
            self.lanelets.append(np.column_stack([rx, ry, lx, ly, 0.5 * (lx + rx), 0.5 * (ly + ry)]))
        self.pred, self.succ = z["pred"], z["succ"]
        adj_left, adj_right = z["adj_left"], z["adj_right"]
        left_same, right_same = z["adj_left_same"], z["adj_right_same"]
        # RoadDataCommonRoad.m:262-290: widen to the same-direction neighbour's outer bound
        self.boundary = []
        for i in range(self.n):
            L = self.lanelets[i]
            left = L[:, 2:4]
            right = L[:, 0:2]
            if adj_left[i] and left_same[i]:
                left = self.lanelets[adj_left[i] - 1][:, 2:4]
            elif adj_right[i] and right_same[i]:
                right = self.lanelets[adj_right[i] - 1][:, 0:2]
            self.boundary.append((np.ascontiguousarray(left), np.ascontiguousarray(right)))

    def is_longitudinal(self, a: int, b: int) -> bool:
        """a, b 1-based: one is the other's predecessor (loop closure test, Commonroad.m:28-35)."""
        return bool(self.pred[a - 1, b - 1] or self.pred[b - 1, a - 1])


_MAP: Optional[RoadMap] = None


def road_map() -> RoadMap:
    global _MAP
    if _MAP is None:
        _MAP = RoadMap()
    return _MAP


@dataclasses.dataclass
class Vehicle:
    """scenarios/Vehicle.m:5-18"""

    x_start: float
    y_start: float
    yaw_start: float
    reference_path: np.ndarray
    reference_speed: float
    lanelets_index: Optional[np.ndarray] = None
    points_index: Optional[np.ndarray] = None
    is_loop: bool = True


@dataclasses.dataclass
class Scenario:
    kind: str                      # "circle" | "commonroad"
    vehicles: List[Vehicle]
    mpa: MotionPrimitiveAutomaton
    checker: int
    priority: str                  # "constant" | "coloring"
    road: Optional[RoadMap] = None

    @property
    def amount(self) -> int:
        return len(self.vehicles)


def circle_scenario(mpa: MotionPrimitiveAutomaton, amount: int = 4) -> Scenario:
    """Circle.m:16-42; SAT checker, constant priorities (Config.m:71-79, :24)."""
    radius = 2.0
    vehicles = []
    ref_speed = float(mpa.get_straight_speeds_of_mpa().max())
    for i in range(amount):
        yaw = np.pi * 2 / amount * i
        s, c = np.sin(yaw), np.cos(yaw)
        xs = -c * radius + 2.25
        ys = -s * radius + 2.0
        path = np.array([[xs, ys], [xs + c * 2 * radius, ys + s * 2 * radius]])
        vehicles.append(Vehicle(xs, ys, yaw, path, ref_speed, is_loop=False))
    return Scenario("circle", vehicles, mpa, CHECKER_SAT, "constant")


def reference_path_loop(path_id: int, road: RoadMap):
    """get_reference_lanelets_loop.m:146-154 + generate_reference_path_loop.m:15-46."""
    loop, start = _PATH_START[path_id]
    seq = _LOOPS[loop]
    k = seq.index(start)
    lanelets_index = np.array(seq[k:] + seq[:k])
    parts = [road.lanelets[i - 1][:, 4:6] for i in lanelets_index]
    path = np.vstack(parts)
    d = np.diff(path, axis=0).sum(axis=1)
    redundant = np.concatenate([[False], np.abs(d) <= 1e-4])   # ismembertol(..., 0, 1e-4) [dev: abs tol]
    reduced = path[~redundant]
    n_cum = np.cumsum([p.shape[0] for p in parts])
    red_cum = np.cumsum(redundant)
    points_index = n_cum - red_cum[n_cum - 1]
    return lanelets_index, reduced, points_index


def calculate_yaw_first(path: np.ndarray) -> float:
    """utility/calculate_yaw.m: yaw(1)"""
    return float(np.arctan2(path[1, 1] - path[0, 1], path[1, 0] - path[0, 0]))


def commonroad_scenario(mpa: MotionPrimitiveAutomaton, amount: int = 20, seed: int = 1,
                        allow_shared_paths: bool = False) -> Scenario:
    """Commonroad.m:5-48 with path ids drawn from 9..41 (Config.m:135-150).

    [dev] MATLAB's randsample / mt19937ar streams are replaced by numpy PCG64(seed).
    With ``allow_shared_paths`` (config 4, 40 vehicles) ids repeat and the second
    vehicle of an id starts half a loop further along the same path.
    """
    road = road_map()
    rng = np.random.Generator(np.random.PCG64(seed))
    pool = np.arange(9, 42)
    if amount <= pool.size and not allow_shared_paths:
        ids = rng.choice(pool, size=amount, replace=False)
        offs = np.zeros(amount)
    else:
        ids = np.concatenate([rng.permutation(pool) for _ in range((amount + pool.size - 1) // pool.size)])[:amount]
        offs = (np.arange(amount) // pool.size) * 0.5
    speeds = mpa.get_straight_speeds_of_mpa()
    vehicles = []
    for pid, off in zip(ids, offs):
        lan_idx, path, pts_idx = reference_path_loop(int(pid), road)
        is_loop = road.is_longitudinal(int(lan_idx[0]), int(lan_idx[-1]))
        if off > 0:
            seglen = np.hypot(*np.diff(path, axis=0).T)
            cum = np.concatenate([[0], np.cumsum(seglen)])
            j = int(np.searchsorted(cum, off * cum[-1]))
            j = min(max(j, 1), path.shape[0] - 2)
            x, y = path[j]
            yaw = float(np.arctan2(path[j + 1, 1] - path[j - 1, 1], path[j + 1, 0] - path[j - 1, 0]))
        else:
            x, y = path[0]
            yaw = calculate_yaw_first(path)
        vehicles.append(Vehicle(float(x), float(y), yaw, path, float(speeds[rng.integers(speeds.size)]),
                                lanelets_index=lan_idx, points_index=pts_idx, is_loop=is_loop))
    return Scenario("commonroad", vehicles, mpa, CHECKER_INTERX, "coloring", road=road)


# --------------------------------------------------------------------------- reference trajectory
def _norm2(dx: float, dy: float) -> float:
    """norm([dx dy], 2) as the arithmetic specification of this path states it: sqrt(dx*dx + dy*dy), no FMA
    (the device kernel prepare_inputs_kernel and this restatement share it; MATLAB's own norm is closed source)."""
    return math.sqrt(dx * dx + dy * dy)


def _projection_2d(x1, y1, x2, y2, x3, y3):
    """projection_2d.m:1-27, operation by operation -> (xp, yp, lambda)."""
    b = _norm2(x2 - x1, y2 - y1)
    if b != 0:
        xn, yn = (x2 - x1) / b, (y2 - y1) / b
        x31, y31 = x3 - x1, y3 - y1
        dot = xn * x31 + yn * y31
        return x1 + dot * xn, y1 + dot * yn, dot / b
    return x1, y1, 0.0


def _closest_point(path: np.ndarray, x: float, y: float):
    """get_arc_distance_to_endpoint.m:41-113: projected point and idx_next (1-based)."""
    n = path.shape[0]
    dxs, dys = path[:, 0] - x, path[:, 1] - y
    d2 = dxs * dxs + dys * dys
    ic = int(np.argmin(d2)) + 1                     # first minimum, like min()
    if ic == 1:
        a, b = 1, 2
    elif ic == n:
        a, b = n - 1, n
    else:
        if d2[ic - 2] <= d2[ic]:                    # min([left, right]): the left one on a tie
            a, b = ic - 1, ic
        else:
            a, b = ic, ic + 1
    xp, yp, lam = _projection_2d(float(path[a - 1, 0]), float(path[a - 1, 1]), float(path[b - 1, 0]), float(path[b - 1, 1]),
                                 float(x), float(y))
    idx_next = ic
    if (0 <= lam <= 0.5) or lam >= 1:
        idx_next = ic + 1 if ic < n else 1
    return xp, yp, max(2, idx_next)


def sample_reference_trajectory(n_samples: int, path: np.ndarray, x: float, y: float, step_distances):
    """sample_reference_trajectory.m:24-97 -> (points [n,2], points_index [n], current_point_index).
    Scalar arithmetic in the reference's order (the device kernel pdmpc_sample_inputs is compared bit for bit)."""
    out = np.zeros((n_samples, 2))
    out_idx = np.zeros(n_samples, dtype=np.int64)
    cx, cy, point_index = _closest_point(path, x, y)
    current_point_index = point_index
    n_pts = path.shape[0]
    px = [float(v) for v in path[:, 0]]
    py = [float(v) for v in path[:, 1]]
    is_loop = _norm2(px[0] - px[-1], py[0] - py[-1]) < 1e-8
    point_index_last = point_index - 1
    if is_loop and point_index == n_pts:
        point_index = 1
    for i in range(n_samples):
        step = float(step_distances[i])
        remaining = _norm2(cx - px[point_index - 1], cy - py[point_index - 1])
        if remaining > step or point_index == n_pts:
            while (px[point_index - 1] == px[point_index_last - 1] and py[point_index - 1] == py[point_index_last - 1]
                   and point_index_last > 1):
                point_index_last -= 1
            ux, uy = px[point_index - 1] - px[point_index_last - 1], py[point_index - 1] - py[point_index_last - 1]
            nrm = _norm2(ux, uy)
            cx, cy = cx + step * (ux / nrm), cy + step * (uy / nrm)
        else:
            reflength = remaining
            while remaining < step:
                reflength = remaining
                cx, cy = px[point_index - 1], py[point_index - 1]
                point_index_last = point_index
                point_index = min(point_index + 1, n_pts)
                if is_loop and point_index == n_pts:
                    point_index = 1
                remaining = remaining + _norm2(cx - px[point_index - 1], cy - py[point_index - 1])
            ux, uy = px[point_index - 1] - px[point_index_last - 1], py[point_index - 1] - py[point_index_last - 1]
            nrm = _norm2(ux, uy)
            cx, cy = cx + (step - reflength) * (ux / nrm), cy + (step - reflength) * (uy / nrm)
        out[i, 0], out[i, 1] = cx, cy
        out_idx[i] = point_index
    return out, out_idx, current_point_index


def get_reference_trajectory(mpa, veh: Vehicle, x, y, trim_current, dt):
    """get_reference_trajectory.m:28-46"""
    Hp = mpa.Hp
    v_ref = np.ones(Hp) * veh.reference_speed
    v_cur = mpa.trim_speed[trim_current - 1]
    v_mid = (np.concatenate([[v_cur], v_ref[:-1]]) + v_ref) / 2
    pts, idx, cur_idx = sample_reference_trajectory(Hp, veh.reference_path, x, y, v_mid * dt)
    return pts, v_ref, idx, cur_idx


def get_predicted_lanelets(veh: Vehicle, ref_idx: np.ndarray) -> np.ndarray:
    """get_predicted_lanelets.m:34-62"""
    n_total = veh.reference_path.shape[0]
    add = ref_idx[-1] + 4
    if add > n_total:
        add -= n_total
    idxs = np.concatenate([ref_idx, [add]])
    lan = np.array([int((i > veh.points_index).sum()) + 1 for i in idxs])
    _, first = np.unique(lan, return_index=True)
    lan = lan[np.sort(first)]
    if lan.size == 1:
        nxt = lan[0] + 1
        if nxt > veh.lanelets_index.size:
            nxt = 1
        lan = np.array([lan[0], nxt])
    return veh.lanelets_index[lan - 1]


def get_lanelets_boundary(predicted: np.ndarray, road: RoadMap, veh: Vehicle):
    """get_lanelets_boundary.m:19-68 -> (left [2,nL], right [2,nR])"""
    lefts = [road.boundary[i - 1][0][:-1] for i in predicted] + [road.boundary[predicted[-1] - 1][0][-1:]]
    rights = [road.boundary[i - 1][1][:-1] for i in predicted] + [road.boundary[predicted[-1] - 1][1][-1:]]
    pos = int(np.flatnonzero(veh.lanelets_index == predicted[0])[0])
    if pos != 0:
        pre = int(veh.lanelets_index[pos - 1])
    elif veh.is_loop:
        pre = int(veh.lanelets_index[-1])
    else:
        pre = 0
    if pre:
        pl, pr = road.boundary[pre - 1]
        k = min(4, min(pr.shape[0] - 1, pl.shape[0] - 1))
        lefts.insert(0, pl[-1 - k:-1])
        rights.insert(0, pr[-1 - k:-1])
    return np.ascontiguousarray(np.vstack(lefts).T), np.ascontiguousarray(np.vstack(rights).T)


def road_tables(scenarios: Sequence["Scenario"]) -> dict:
    """Flat tables of pdmpc_upload_road for the vehicles of `scenarios` (path id = running vehicle index): the map's
    lanelet boundaries (RoadMap.boundary, lanelet_boundaries{l}{1:2}) and every vehicle's reference path with its
    lanelets_index / points_index (reference_path_struct)."""
    road = scenarios[0].road
    bptr, bx, by = [0], [], []
    for left, right in road.boundary:
        for side in (left, right):
            bx.append(side[:, 0]); by.append(side[:, 1])
            bptr.append(bptr[-1] + side.shape[0])
    pptr, px, py, lptr, lidx, pidx, loop, speed = [0], [], [], [0], [], [], [], []
    for sc in scenarios:
        for v in sc.vehicles:
            px.append(v.reference_path[:, 0]); py.append(v.reference_path[:, 1])
            pptr.append(pptr[-1] + v.reference_path.shape[0])
            lidx.append(np.asarray(v.lanelets_index)); pidx.append(np.asarray(v.points_index))
            lptr.append(lptr[-1] + len(v.lanelets_index))
            loop.append(1 if v.is_loop else 0)
            speed.append(v.reference_speed)
    return {"bound_ptr": np.array(bptr, dtype=np.int32), "bound_x": np.concatenate(bx).astype(np.float64),
            "bound_y": np.concatenate(by).astype(np.float64), "path_ptr": np.array(pptr, dtype=np.int32),
            "path_x": np.concatenate(px).astype(np.float64), "path_y": np.concatenate(py).astype(np.float64),
            "lan_ptr": np.array(lptr, dtype=np.int32), "lanelets_index": np.concatenate(lidx).astype(np.int32),
            "points_index": np.concatenate(pidx).astype(np.int32), "is_loop": np.array(loop, dtype=np.uint8),
            "reference_speed": np.array(speed, dtype=np.float64)}


# --------------------------------------------------------------------------- coupling / priorities
_SC_TWO_OVER_PI = float.fromhex("0x1.45f306dc9c883p-1")
_SC_P = tuple(float.fromhex(v) for v in ("0x1.921fb54400000p+0", "0x1.0b4611a600000p-34", "0x1.3198a2e037073p-69"))
_SC_S = tuple(float.fromhex(v) for v in (
    "-0x1.5555555555555p-3", "0x1.1111111111111p-7", "-0x1.a01a01a01a01ap-13", "0x1.71de3a556c734p-19",
    "-0x1.ae64567f544e4p-26", "0x1.6124613a86d09p-33", "-0x1.ae7f3e733b81fp-41", "0x1.952c77030ad4ap-49",
    "-0x1.2f49b46814157p-57", "0x1.71b8ef6dcf572p-66"))
_SC_C = tuple(float.fromhex(v) for v in (
    "-0x1.0000000000000p-1", "0x1.5555555555555p-5", "-0x1.6c16c16c16c17p-10", "0x1.a01a01a01a01ap-16",
    "-0x1.27e4fb7789f5cp-22", "0x1.1eed8eff8d898p-29", "-0x1.93974a8c07c9dp-37", "0x1.ae7f3e733b81fp-45",
    "-0x1.6827863b97d97p-53", "0x1.e542ba4020225p-62"))


def sincos_spec(x: float):
    """(sin x, cos x) by the arithmetic specification of DESIGN.md §2 (three-term Cody-Waite reduction, degree-10
    polynomials, no FMA) — the algorithm of sincos_ref in pdmpc_kernels.cuh, operation by operation, so that areas
    placed on the host and on the device agree bit for bit."""
    x = float(x)
    n = float(round(x * _SC_TWO_OVER_PI))                       # rint: ties to even
    r = ((x - n * _SC_P[0]) - n * _SC_P[1]) - n * _SC_P[2]
    z = r * r
    ps, pc = _SC_S[9], _SC_C[9]
    for i in range(8, -1, -1):
        ps = ps * z + _SC_S[i]
        pc = pc * z + _SC_C[i]
    sr = r + (r * z) * ps
    cr = 1.0 + z * pc
    q = int(n) & 3
    return ((sr, cr), (cr, -sr), (-sr, -cr), (-cr, sr))[q]


def occupied_area(x, y, yaw, offset=0.01) -> np.ndarray:
    """get_occupied_areas.m:21-25 (normal_offset, closed 5-point rectangle)"""
    xl = np.array([-1.0, -1.0, 1.0, 1.0, -1.0]) * (VEH_LENGTH / 2 + offset)
    yl = np.array([-1.0, 1.0, 1.0, -1.0, -1.0]) * (VEH_WIDTH / 2 + offset)
    s, c = sincos_spec(yaw)
    return np.vstack([c * xl - s * yl + x, s * xl + c * yl + y])


def kahn(A: np.ndarray) -> np.ndarray:
    """utility/kahn.m:1-24: computation level (1-based) of each vertex of a DAG."""
    A = A.copy().astype(np.int64)
    n = A.shape[0]
    L = np.zeros(n, dtype=np.int64)
    done = np.zeros(n, dtype=bool)
    in_d = A.sum(axis=0)
    level = 1
    while not done.all():
        src = (in_d == 0)
        if not src.any():
            raise ValueError("coupling graph is not a DAG")
        L[src] = level
        A[src, :] = 0
        done |= src
        in_d = A.sum(axis=0)
        in_d[done] = 1
        level += 1
    return L


def coloring_priorities(adjacency: np.ndarray) -> np.ndarray:
    """ColoringPrioritizer.m:11-153 -> directed coupling (row = higher priority)."""
    A = adjacency.astype(np.int64)
    n = A.shape[0]
    degree = A.sum(axis=0)
    color = np.zeros(n, dtype=np.int64)
    color[degree == 0] = 1
    while (color == 0).any():
        best, idx = -1, -1
        for i in np.flatnonzero(color == 0):
            d = np.unique(color[A[i] == 1])
            d = int((d != 0).sum())
            if d > best:
                best, idx = d, i
            if d == best and degree[i] > degree[idx]:
                idx = i
        used = set(np.unique(color[A[idx] == 1]).tolist())
        c = 1
        while c in used:
            c += 1
        color[idx] = c
    used_col = np.unique(color)
    levels = [np.flatnonzero(color == c) for c in used_col]
    # order_topo :96-131: repeatedly take the level holding the highest-degree vertex
    deg = A.sum(axis=0).astype(np.int64)
    if deg.sum() == 0:
        order = [0]
    else:
        order = []
        while deg.sum() != 0:
            max_idx = int(np.argmax(deg))   # first maximum, as the reference's strict '>' scan
            lvl = next(j for j, m in enumerate(levels) if max_idx in m)
            order.append(lvl)
            deg[levels[lvl]] = 0
    ordered = [levels[j] for j in order] + [levels[j] for j in range(len(levels)) if j not in order]
    prio = np.zeros(n, dtype=np.int64)
    for lvl, members in enumerate(ordered):
        prio[members] = lvl + 1
    # directed: edge i -> j iff adjacent and level(i) < level(j)
    return (A > 0) & (prio[:, None] < prio[None, :])


def constant_priorities(adjacency: np.ndarray) -> np.ndarray:
    """ConstantPrioritizer.m:6-18: priority = vehicle index; lower index first."""
    n = adjacency.shape[0]
    idx = np.arange(n)
    return (adjacency > 0) & (idx[:, None] < idx[None, :])


def _corridor(veh: Vehicle, x, y, reach: float) -> np.ndarray:
    """Sample points of the reference path from the projection of (x, y) forward by `reach`."""
    path = veh.reference_path
    xp, yp, nxt = _closest_point(path, x, y)
    pts = [np.array([xp, yp])]
    left = reach
    i = nxt - 1
    n = path.shape[0]
    guard = 0
    while left > 0 and guard < 4 * n:
        guard += 1
        seg = path[i] - pts[-1]
        L = np.hypot(*seg)
        if L > 1e-12:
            step = min(L, left)
            m = max(1, int(np.ceil(step / 0.05)))
            base = pts[-1]
            for t in range(1, m + 1):
                pts.append(base + seg / L * (step * t / m))
            left -= step
            if step < L:
                break
        i += 1
        if i >= n:
            if not veh.is_loop:
                break
            i = 1
    return np.array(pts)


def couple(sc: Scenario, poses: np.ndarray, all_coupled: bool = False) -> np.ndarray:
    """[dev] stand-in for ReachableSetCoupler.m:5-54: vehicles are coupled when the
    corridors they can reach within Hp steps come closer than one lane width.  In
    the circle scenario every pair is coupled (SURVEY.md §8d config 1)."""
    n = sc.amount
    if sc.kind == "circle" or all_coupled:
        return np.ones((n, n), dtype=np.int64) - np.eye(n, dtype=np.int64)
    reach = sc.mpa.get_max_speed_of_mpa() * sc.mpa.dt_seconds * sc.mpa.Hp + VEH_LENGTH
    cors = [_corridor(v, poses[i, 0], poses[i, 1], reach) for i, v in enumerate(sc.vehicles)]
    A = np.zeros((n, n), dtype=np.int64)
    for i in range(n):
        for j in range(i + 1, n):
            if np.hypot(*(poses[i, :2] - poses[j, :2])) > 2 * reach + 0.5:
                continue
            d = cors[i][:, None, :] - cors[j][None, :, :]
            if (d[..., 0] ** 2 + d[..., 1] ** 2).min() < 0.25 ** 2:
                A[i, j] = A[j, i] = 1
    return A


# --------------------------------------------------------------------------- BASELINE config 4
_REACH_CACHE: dict = {}


def _convex_hull_closed(pts: np.ndarray) -> np.ndarray:
    """Andrew's monotone chain: counter-clockwise hull of [m, 2] points as a closed [2, h + 1] polygon."""
    p = np.unique(pts, axis=0)                     # sorted by x, then y
    if p.shape[0] < 3:
        return np.vstack([p, p[:1]]).T

    def half(seq):
        out = []
        for q in seq:
            while len(out) >= 2 and ((out[-1][0] - out[-2][0]) * (q[1] - out[-2][1]) -
                                     (out[-1][1] - out[-2][1]) * (q[0] - out[-2][0])) <= 0:
                out.pop()
            out.append(q)
        return out

    lower, upper = half(p), half(p[::-1])
    hull = np.array(lower[:-1] + upper[:-1])
    return np.vstack([hull, hull[:1]]).T


def local_reachable_sets_conv(mpa: MotionPrimitiveAutomaton) -> List[List[np.ndarray]]:
    """reachability_analysis_offline (MotionPrimitiveAutomaton.m:252-392): for every start trim i and step t
    the convexified union of the offset areas of all maneuvers a vehicle can execute in step t after any trim
    sequence from i, in the vehicle frame of step 0 (local_reachable_sets_conv{i, t}).  [dev] convhull(union(.))
    is computed as the hull of the areas' vertices (the same set; polyshape's vertex order is not reproduced)."""
    key = id(mpa)
    if key in _REACH_CACHE:
        return _REACH_CACHE[key]
    nT, Hp = mpa.n_trims, mpa.Hp
    out: List[List[np.ndarray]] = []
    for i in range(nT):
        st = np.array([[0.0, 0.0, 0.0]])
        tr = np.array([i])
        per_step = []
        for t in range(Hp):
            pts, nst, ntr = [], [], []
            for f in np.unique(tr):
                sel = st[tr == f]
                c, sn = np.cos(sel[:, 2]), np.sin(sel[:, 2])
                for to in np.flatnonzero(mpa.transition[t, f]):
                    e = int(mpa.edge_index[f, to])
                    m = int(mpa.area_npts[e, 0])
                    ax, ay = mpa.area_x[e, 0, :m], mpa.area_y[e, 0, :m]
                    px = c[:, None] * ax[None] - sn[:, None] * ay[None] + sel[:, 0:1]     # translate_global
                    py = sn[:, None] * ax[None] + c[:, None] * ay[None] + sel[:, 1:2]
                    pts.append(np.stack([px.reshape(-1), py.reshape(-1)], axis=1))
                    nst.append(np.stack([c * mpa.edge_dx[e] - sn * mpa.edge_dy[e] + sel[:, 0],
                                         sn * mpa.edge_dx[e] + c * mpa.edge_dy[e] + sel[:, 1],
                                         sel[:, 2] + mpa.edge_dyaw[e]], axis=1))
                    ntr.append(np.full(sel.shape[0], to))
            per_step.append(_convex_hull_closed(np.round(np.concatenate(pts), 12)))
            st, tr = np.concatenate(nst), np.concatenate(ntr)
            # states that coincide (same trim, same pose) need to be expanded once only
            keyed = np.round(np.column_stack([tr, st]), 9)
            _, first = np.unique(keyed, axis=0, return_index=True)
            st, tr = st[np.sort(first)], tr[np.sort(first)]
        out.append(per_step)
    _REACH_CACHE[key] = out
    return out


def reachable_sets_at(mpa: MotionPrimitiveAutomaton, x: float, y: float, yaw: float, trim: int) -> List[np.ndarray]:
    """get_reachable_sets (MotionPrimitiveAutomaton.m:649-687): the local sets of the current trim placed at the pose."""
    s_, c = sincos_spec(yaw)   # the arithmetic specification (DESIGN.md §2): the device places them with the same bits
    return [np.vstack([c * a[0] - s_ * a[1] + x, s_ * a[0] + c * a[1] + y]) for a in local_reachable_sets_conv(mpa)[trim - 1]]


def assemble_obstacles_host(mpa: MotionPrimitiveAutomaton, x, y, yaw, speed, trim, successors, parallel,
                            half_length: float, half_width: float) -> dict:
    """Host restatement of pdmpc_assemble_obstacles (same arguments and result as capi.Planner.assemble_obstacles):
    slot i*(Hp+1) = the offset rectangles of row i's standing successors (PrioritizedController.m:508-540,
    get_occupied_areas.m:19-25), slot i*(Hp+1)+k = the step-k reachable set of each parallel predecessor
    (:391-407, MotionPrimitiveAutomaton.m:649-687), as the obstacle CSR of a SearchBatch."""
    n, Hp = len(x), mpa.Hp
    xl = np.array([-1.0, -1.0, 1.0, 1.0, -1.0]) * half_length
    yl = np.array([-1.0, 1.0, 1.0, -1.0, -1.0]) * half_width
    slot_ptr, poly_ptr, vx, vy = [0], [0], [], []

    def put(px, py):
        vx.append(px); vy.append(py)
        poly_ptr.append(poly_ptr[-1] + len(px))

    for i in range(n):
        cnt = 0
        for j in successors[i]:
            if abs(speed[j]) < 0.01:
                s_, c = sincos_spec(yaw[j])
                put(c * xl - s_ * yl + x[j], s_ * xl + c * yl + y[j])
                cnt += 1
        slot_ptr.append(slot_ptr[-1] + cnt)
        sets = [reachable_sets_at(mpa, x[j], y[j], yaw[j], int(trim[j])) for j in parallel[i]]
        for k in range(Hp):
            for rs in sets:
                put(rs[k][0], rs[k][1])
            slot_ptr.append(slot_ptr[-1] + len(sets))
    cat = lambda parts: np.ascontiguousarray(np.concatenate(parts)) if parts else np.zeros(0)
    return {"slot_ptr": np.array(slot_ptr, dtype=np.int32), "poly_ptr": np.array(poly_ptr, dtype=np.int32),
            "vert_x": cat(vx), "vert_y": cat(vy)}


COUPLING_AREA_THRESHOLD = 1e-3   # ReachableSetCoupler.m:39-42: coupled iff area(intersect(...)) > 1e-3


def convex_overlap_area(P, Q) -> float:
    """Area of the intersection of two convex polygons by the arithmetic specification of DESIGN.md §4.12, operation by
    operation (pdmpc_coupling.cuh computes the same bits): P, Q = closed [2, m + 1] polygons (first vertex repeated last);
    P is clipped by Q with Sutherland-Hodgman in FP64 without FMA.  [dev] stand-in for polyshape intersect + area
    (ReachableSetCoupler.m:39-42), whose vertex arithmetic is closed source."""
    px, py = [float(v) for v in P[0][:-1]], [float(v) for v in P[1][:-1]]
    qx, qy = [float(v) for v in Q[0][:-1]], [float(v) for v in Q[1][:-1]]
    mp, mq = len(px), len(qx)
    if mp < 3 or mq < 3:
        return 0.0
    if max(px) < min(qx) or max(qx) < min(px) or max(py) < min(qy) or max(qy) < min(py):
        return 0.0
    sq = 0.0
    for k in range(mq):
        k1 = (k + 1) % mq
        sq = sq + (qx[k] * qy[k1] - qx[k1] * qy[k])
    if sq == 0.0:
        return 0.0
    if sq < 0.0:
        qx.reverse()
        qy.reverse()
    cx, cy = px, py
    for k in range(mq):
        ax, ay, bx, by = qx[k], qy[k], qx[(k + 1) % mq], qy[(k + 1) % mq]
        ex_, ey_ = bx - ax, by - ay
        nx, ny = [], []
        sx, sy = cx[-1], cy[-1]
        ds = ex_ * (sy - ay) - ey_ * (sx - ax)
        for x, y in zip(cx, cy):
            de = ex_ * (y - ay) - ey_ * (x - ax)
            if de >= 0.0:
                if ds < 0.0:
                    t = ds / (ds - de)
                    nx.append(sx + t * (x - sx)); ny.append(sy + t * (y - sy))
                nx.append(x); ny.append(y)
            elif ds >= 0.0:
                t = ds / (ds - de)
                nx.append(sx + t * (x - sx)); ny.append(sy + t * (y - sy))
            sx, sy, ds = x, y, de
        if not nx:
            return 0.0
        cx, cy = nx, ny
    m = len(cx)
    if m < 3:
        return 0.0
    acc = 0.0
    for k in range(m):
        k1 = (k + 1) % m
        acc = acc + (cx[k] * cy[k1] - cx[k1] * cy[k])
    return 0.5 * abs(acc)


def reachable_set_overlaps(mpa: MotionPrimitiveAutomaton, pose: np.ndarray, trim) -> np.ndarray:
    """[n, n] overlap areas of the step-Hp reachable sets (reachable_sets{i, end}) of n vehicles at pose [n, 3] with their
    current trims (1-based); 0.0 on the diagonal.  Set i is clipped by set j for i < j; the matrix is symmetric."""
    n = pose.shape[0]
    sets = [reachable_sets_at(mpa, *pose[i], int(trim[i]))[-1] for i in range(n)]
    area = np.zeros((n, n))
    for i in range(n):
        for j in range(i + 1, n):
            area[i, j] = area[j, i] = convex_overlap_area(sets[i], sets[j])
    return area


def couple_reachable_sets(mpa: MotionPrimitiveAutomaton, pose: np.ndarray, trim) -> np.ndarray:
    """ReachableSetCoupler.couple (ReachableSetCoupler.m:5-54): vehicles i, j are coupled iff their step-Hp reachable sets
    overlap by more than 1e-3 m^2.  [dev] the sets are not clipped by the predicted lanelets first
    (HighLevelController.m:241-246).  Symmetric int64 adjacency with a zero diagonal."""
    return (reachable_set_overlaps(mpa, pose, trim) > COUPLING_AREA_THRESHOLD).astype(np.int64)


def decide_relations(A: np.ndarray, priority: str, max_num_CLs: int):
    """Priorities, the level cut and the computation levels of one scenario from its adjacency:
    D = directed coupling (row = higher priority; coloring_priorities or constant_priorities), seq = the sequential part
    of D (limit_computation_levels, equal to D when max_num_CLs >= the depth), levels = kahn(seq) (1-based)."""
    D = (constant_priorities(A) if priority == "constant" else coloring_priorities(A)).astype(bool)
    seq = limit_computation_levels(D, max_num_CLs)
    return D, seq, kahn(seq.astype(np.int64))


def limit_computation_levels(D: np.ndarray, max_num_CLs: int) -> np.ndarray:
    """[dev] stand-in for the weigh + cut step (PrioritizedController.group :381-397, GreedyCut): the edges kept as
    SEQUENTIAL are chosen greedily in topological order so that no vehicle sits deeper than max_num_CLs
    computation levels; the other predecessors plan in PARALLEL and are considered through their reachable
    sets (parallel_coupling_reachability :399-415)."""
    n = D.shape[0]
    seq = np.zeros_like(D, dtype=bool)
    level = np.zeros(n, dtype=np.int64)
    for j in np.argsort(kahn(D.astype(np.int64)), kind="stable"):
        lv = 1
        for i in np.flatnonzero(D[:, j]):
            if level[i] < max_num_CLs:
                seq[i, j] = True
                lv = max(lv, level[i] + 1)
        level[j] = lv
    return seq


# --------------------------------------------------------------------------- closed loop
PlanFn = Callable[[SearchBatch], BatchResult]


@dataclasses.dataclass
class StepRecord:
    step: int
    level: int
    vehicles: np.ndarray       # vehicle indices planned in this (step, level)
    batch: SearchBatch
    result: BatchResult


class ScenarioRunner:
    """HighLevelController.main_control_loop (HighLevelController.m:334-373) for the
    sequential prioritized controller, with the optimizer call batched per
    computation level (vehicles of one level are independent,
    PrioritizedSequentialController.m:83-92)."""

    def __init__(self, sc: Scenario, plan_fn: PlanFn, max_num_CLs: int = 99, timestep_fn=None, inputs_fn=None,
                 path_id0: int = 0, closed_loop_fn=None, obstacles_fn=None, states_fn=None, coupler: str = "corridor",
                 coupled_fn=None, n_expansions_max: Optional[int] = None):
        """plan_fn(batch) plans one computation level; with timestep_fn(batch, deps) the whole time
        step is ONE call and the predecessors' areas are handed over behind it (pdmpc_plan_timestep).
        inputs_fn(path_id, x, y, speed, dt) -> dict (capi.Planner.sample_inputs): reference trajectories and lanelet
        boundaries of all vehicles come from the device in one call per time step instead of the host functions
        above; path_id0 = path id of vehicle 0 in the uploaded road tables (road_tables of several scenarios)."""
        self.sc = sc
        self.plan_fn = plan_fn
        self.timestep_fn = timestep_fn
        self.inputs_fn = inputs_fn
        self.path_id0 = path_id0
        # obstacles_fn(x, y, yaw, speed, trim, successors, parallel, half_length, half_width) -> obstacle CSR dict
        # (capi.Planner.assemble_obstacles): the standstill areas of successors and the reachable sets of parallel
        # predecessors of all vehicles are placed on the device in one call per time step (one-call path)
        self.obstacles_fn = obstacles_fn
        # states_fn(path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot, half_length, half_width, dt,
        # checker) -> BatchResult with the FINAL plan of every vehicle (capi.Planner.plan_timestep_from_states): inputs,
        # obstacle assembly, planning and fallback plans of a time step in ONE call; the host only decides coupling and
        # priorities
        self.states_fn = states_fn
        # coupler: "corridor" (couple, the [dev] proxy) or "reachable_set" (couple_reachable_sets, ReachableSetCoupler)
        if coupler not in ("corridor", "reachable_set"):
            raise ValueError(f"unknown coupler {coupler!r}")
        self.coupler = coupler
        # coupled_fn(path_id, x, y, yaw, speed, trim, slot, half_length, half_width, dt, checker, priority, max_num_CLs)
        # -> (BatchResult, relations) (capi.Planner.plan_timestep_from_states_coupled): states_fn with the reachable-set
        # coupling, the priorities and the level cut decided on the device too; the relations the device returned are
        # recorded in timestep_records as (step, None, relations, result)
        self.coupled_fn = coupled_fn
        # closed_loop_fn(batch, deps, slot, standstill) -> BatchResult with the FINAL plan of every vehicle
        # (capi.Planner.plan_timestep_closed_loop): fallback plans are built and kept on the device, slot = path_id0 + i
        self.closed_loop_fn = closed_loop_fn
        # n_expansions_max: the optimizer is MonteCarloTreeSearch with this budget (the callbacks pass it on); plan_fn,
        # timestep_fn, closed_loop_fn and states_fn then also receive the RandStream seeds of the rows they plan as their
        # last argument: time_step + vehicle_index, both 1-based (MonteCarloTreeSearch.m:31, PrioritizedController.m:335-341)
        self.n_expansions_max = n_expansions_max
        self.max_num_CLs = max_num_CLs              # honoured by the one-call path (timestep_inputs)
        self.timestep_records: List[tuple] = []     # (step, batch, deps, result) of the one-call path
        self.mpa = sc.mpa
        n = sc.amount
        self.pose = np.array([[v.x_start, v.y_start, v.yaw_start] for v in sc.vehicles])
        self.trim = np.array([sc.mpa.trim_from_values(0.0, 0.0)] * n)   # start at standstill
        self.prev_shapes: List[Optional[List[np.ndarray]]] = [None] * n
        self.prev_traj: List[Optional[np.ndarray]] = [None] * n
        self.prev_trims: List[Optional[np.ndarray]] = [None] * n
        self.k = 0
        self.records: List[StepRecord] = []
        self.n_fallbacks = 0

    def _seeded(self, fn, *args, rows=None):
        """fn(*args), or fn(*args, seeds of `rows` (default: all vehicles)) for the sampled optimizer."""
        if self.n_expansions_max is None:
            return fn(*args)
        seeds = mcts_seeds(self.k, self.sc.amount)
        return fn(*args, seeds if rows is None else seeds[rows])

    def _adjacency(self) -> np.ndarray:
        if self.coupler == "reachable_set":
            return couple_reachable_sets(self.mpa, self.pose, self.trim)
        return couple(self.sc, self.pose)

    def _iter_for(self, i: int) -> IterationData:
        sc, mpa = self.sc, self.mpa
        v = sc.vehicles[i]
        x, y, yaw = self.pose[i]
        pts, v_ref, ref_idx, _ = get_reference_trajectory(mpa, v, x, y, int(self.trim[i]), mpa.dt_seconds)
        if sc.kind == "commonroad":
            pred_lan = get_predicted_lanelets(v, ref_idx)
            boundary = get_lanelets_boundary(pred_lan, sc.road, v)
        else:
            boundary = (np.zeros((2, 0)), np.zeros((2, 0)))
        return IterationData(x0=np.array([x, y, yaw, mpa.trim_speed[self.trim[i] - 1]]),
                             trim_indices=int(self.trim[i]), reference_trajectory_points=pts, v_ref=v_ref,
                             predicted_lanelet_boundary=boundary)

    def _iters(self) -> List[IterationData]:
        """iter_v of every vehicle for this time step (HighLevelController.m:167-270), host or device side."""
        n = self.sc.amount
        if self.inputs_fn is None or self.sc.kind != "commonroad":
            return [self._iter_for(i) for i in range(n)]
        mpa = self.mpa
        speed = np.array([mpa.trim_speed[self.trim[i] - 1] for i in range(n)], dtype=np.float64)
        o = self.inputs_fn(self.path_id0 + np.arange(n), self.pose[:, 0], self.pose[:, 1], speed, mpa.dt_seconds)
        out = []
        for i in range(n):
            x, y, yaw = self.pose[i]
            l0, l1, l2 = (int(v) for v in o["lane_ptr"][2 * i:2 * i + 3])
            boundary = (np.ascontiguousarray(np.vstack([o["lane_x"][l0:l1], o["lane_y"][l0:l1]])),
                        np.ascontiguousarray(np.vstack([o["lane_x"][l1:l2], o["lane_y"][l1:l2]])))
            out.append(IterationData(x0=np.array([x, y, yaw, speed[i]]), trim_indices=int(self.trim[i]),
                                     reference_trajectory_points=np.column_stack([o["ref_x"][i], o["ref_y"][i]]),
                                     v_ref=o["v_ref"][i].copy(), predicted_lanelet_boundary=boundary))
        return out

    def _fallback_plan(self, i: int):
        """What vehicle i does (and publishes) when its search is exhausted — known before the time
        step starts.  [dev] local fallback: PrioritizedController.m:568-621 (standstill), :678-718
        (previous plan shifted, del_first_rpt_last)."""
        mpa, Hp = self.mpa, self.mpa.Hp
        if self.prev_shapes[i] is None or abs(mpa.trim_speed[self.trim[i] - 1]) < 0.01:
            stand = occupied_area(*self.pose[i])
            return [stand] * Hp, np.tile(self.pose[i], (Hp, 1)), np.full(Hp, self.trim[i])
        ps = self.prev_shapes[i]
        return (ps[1:] + [ps[-1]], np.vstack([self.prev_traj[i][1:], self.prev_traj[i][-1:]]),
                np.concatenate([self.prev_trims[i][1:], self.prev_trims[i][-1:]]))

    def timestep_inputs(self):
        """The inputs of ONE call for the whole time step: every vehicle's iter_v without its
        sequential predecessors' areas, the predecessor lists and the fallback plans."""
        sc, mpa = self.sc, self.mpa
        n = sc.amount
        iters = self._iters()
        A = self._adjacency()
        D = constant_priorities(A) if sc.priority == "constant" else coloring_priorities(A)
        Db = D.astype(bool)
        seq = limit_computation_levels(Db, self.max_num_CLs) if self.max_num_CLs < n else Db
        if self.obstacles_fn is not None:
            # the same two rules on the device (pdmpc_assemble_obstacles), all vehicles in one call
            speed = np.array([mpa.trim_speed[self.trim[j] - 1] for j in range(n)], dtype=np.float64)
            o = self.obstacles_fn(self.pose[:, 0], self.pose[:, 1], self.pose[:, 2], speed, self.trim,
                                  [np.flatnonzero(D[i, :]) for i in range(n)],
                                  [np.flatnonzero(Db[:, i] & ~seq[:, i]) for i in range(n)],
                                  VEH_LENGTH / 2 + 0.01, VEH_WIDTH / 2 + 0.01)
            sp, pp = o["slot_ptr"], o["poly_ptr"]
            poly = lambda p: np.ascontiguousarray(np.vstack([o["vert_x"][pp[p]:pp[p + 1]], o["vert_y"][pp[p]:pp[p + 1]]]))
            Hp = mpa.Hp
            for i in range(n):
                s0 = i * (Hp + 1)
                iters[i].obstacles.extend(poly(p) for p in range(sp[s0], sp[s0 + 1]))
                for q in range(sp[s0 + 2] - sp[s0 + 1]):     # one row per parallel predecessor, a column per step
                    iters[i].dynamic_obstacle_area.append([poly(sp[s0 + k] + q) for k in range(1, Hp + 1)])
        else:
            for i in range(n):   # consider_successors, area_of_standstill: PrioritizedController.m:508-540
                for j in np.flatnonzero(D[i, :]):
                    if abs(mpa.trim_speed[self.trim[j] - 1]) < 0.01:
                        iters[i].obstacles.append(occupied_area(*self.pose[j]))
            for i in range(n):   # parallel predecessors: reachable sets as dynamic obstacles, PrioritizedController.m:399-415,493-501
                for j in np.flatnonzero(Db[:, i] & ~seq[:, i]):
                    iters[i].dynamic_obstacle_area.append(reachable_sets_at(mpa, *self.pose[j], int(self.trim[j])))
        D = Db
        preds = [np.flatnonzero(seq[:, i]) for i in range(n)]
        fallbacks = [self._fallback_plan(i) for i in range(n)]
        return iters, preds, fallbacks

    def step_timestep(self) -> BatchResult:
        """One time step through timestep_fn: same closed loop as step(), one optimizer call."""
        sc, mpa = self.sc, self.mpa
        n, Hp = sc.amount, mpa.Hp
        self.k += 1
        if self.coupled_fn is not None:
            speed = np.array([mpa.trim_speed[self.trim[i] - 1] for i in range(n)], dtype=np.float64)
            ids = self.path_id0 + np.arange(n)
            res, rel = self.coupled_fn(ids, self.pose[:, 0], self.pose[:, 1], self.pose[:, 2], speed, self.trim, ids,
                                       VEH_LENGTH / 2 + 0.01, VEH_WIDTH / 2 + 0.01, mpa.dt_seconds, sc.checker, sc.priority,
                                       self.max_num_CLs)
            self.apply_final(res)
            self.timestep_records.append((self.k, None, rel, res))
            return res
        if self.states_fn is not None:
            A = self._adjacency()
            D = (constant_priorities(A) if sc.priority == "constant" else coloring_priorities(A)).astype(bool)
            seq = limit_computation_levels(D, self.max_num_CLs) if self.max_num_CLs < n else D
            speed = np.array([mpa.trim_speed[self.trim[i] - 1] for i in range(n)], dtype=np.float64)
            ids = self.path_id0 + np.arange(n)
            res = self._seeded(self.states_fn, ids, self.pose[:, 0], self.pose[:, 1], self.pose[:, 2], speed, self.trim,
                               [np.flatnonzero(D[i, :]) for i in range(n)],
                               [np.flatnonzero(D[:, i] & ~seq[:, i]) for i in range(n)],
                               [np.flatnonzero(seq[:, i]) for i in range(n)], ids,
                               VEH_LENGTH / 2 + 0.01, VEH_WIDTH / 2 + 0.01, mpa.dt_seconds, sc.checker)
            self.apply_final(res)
            self.timestep_records.append((self.k, None, None, res))
            return res
        iters, preds, fallbacks = self.timestep_inputs()
        batch = SearchBatch.from_iters(iters, Hp, sc.checker, mpa.dt_seconds)
        if self.closed_loop_fn is not None:
            deps = TimestepDeps.build(preds, [None] * n, Hp)
            still = np.array([abs(mpa.trim_speed[self.trim[i] - 1]) < 0.01 for i in range(n)], dtype=np.uint8)
            res = self._seeded(self.closed_loop_fn, batch, deps, self.path_id0 + np.arange(n), still)
            self.apply_final(res)
        else:
            deps = TimestepDeps.build(preds, [f[0] for f in fallbacks], Hp)
            res = self._seeded(self.timestep_fn, batch, deps)
            self.apply_timestep(res, fallbacks)
        self.timestep_records.append((self.k, batch, deps, res))
        return res

    def apply_final(self, res: BatchResult) -> None:
        """Plans of one time step whose exhausted rows already hold the fallback plan (device-side closed loop)."""
        n = self.sc.amount
        shapes_now: List[Optional[List[np.ndarray]]] = [None] * n
        for i in range(n):
            self.n_fallbacks += int(res.is_exhausted[i])
            shapes_now[i] = res.shapes(i)
            self.prev_traj[i] = res.y_predicted[i].copy()
            self.prev_trims[i] = res.trims[i, 1:].copy()
            self.pose[i] = self.prev_traj[i][0]
            self.trim[i] = self.prev_trims[i][0]
        self.prev_shapes = shapes_now

    def apply_timestep(self, res: BatchResult, fallbacks) -> None:
        """Take the plans of one time step (row i = vehicle i): exhausted vehicles execute their fallback
        plan, the plant applies the first step (plant/Simulation.m:93-98)."""
        n = self.sc.amount
        shapes_now: List[Optional[List[np.ndarray]]] = [None] * n
        new_pose, new_trim = self.pose.copy(), self.trim.copy()
        for i in range(n):
            if not res.is_exhausted[i]:
                shapes_now[i] = res.shapes(i)
                self.prev_traj[i] = res.y_predicted[i].copy()
                self.prev_trims[i] = res.trims[i, 1:].copy()
            else:
                self.n_fallbacks += 1
                shapes_now[i], self.prev_traj[i], self.prev_trims[i] = fallbacks[i]
            new_pose[i] = self.prev_traj[i][0]      # Simulation.apply: plant/Simulation.m:93-98
            new_trim[i] = self.prev_trims[i][0]
        self.prev_shapes = shapes_now
        self.pose, self.trim = new_pose, new_trim

    def step(self) -> List[StepRecord]:
        if (self.timestep_fn is not None or self.closed_loop_fn is not None or self.states_fn is not None
                or self.coupled_fn is not None):
            self.step_timestep()
            return []
        sc, mpa = self.sc, self.mpa
        n, Hp = sc.amount, mpa.Hp
        self.k += 1
        iters = self._iters()
        A = self._adjacency()
        D = constant_priorities(A) if sc.priority == "constant" else coloring_priorities(A)
        levels = kahn(D.astype(np.int64))
        shapes_now: List[Optional[List[np.ndarray]]] = [None] * n
        new_pose = self.pose.copy()
        new_trim = self.trim.copy()
        out: List[StepRecord] = []
        for lvl in range(1, int(levels.max()) + 1):
            members = np.flatnonzero(levels == lvl)
            its = []
            for i in members:
                it = iters[i]
                # consider_predecessors (sequential): PrioritizedController.m:449-506
                for j in np.flatnonzero(D[:, i]):
                    it.dynamic_obstacle_area.append(shapes_now[j])
                # consider_successors, area_of_standstill: :508-540
                for j in np.flatnonzero(D[i, :]):
                    if abs(mpa.trim_speed[self.trim[j] - 1]) < 0.01:
                        it.obstacles.append(occupied_area(*self.pose[j]))
                its.append(it)
            batch = SearchBatch.from_iters(its, Hp, sc.checker, mpa.dt_seconds)
            res = self._seeded(self.plan_fn, batch, rows=members)
            for b, i in enumerate(members):
                if not res.is_exhausted[b]:
                    shapes_now[i] = res.shapes(b)
                    self.prev_traj[i] = res.y_predicted[b].copy()
                    self.prev_trims[i] = res.trims[b, 1:].copy()
                else:
                    # [dev] local fallback: PrioritizedController.m:568-621,678-718
                    self.n_fallbacks += 1
                    if self.prev_shapes[i] is None or abs(mpa.trim_speed[self.trim[i] - 1]) < 0.01:
                        stand = occupied_area(*self.pose[i])
                        shapes_now[i] = [stand] * Hp
                        self.prev_traj[i] = np.tile(self.pose[i], (Hp, 1))
                        self.prev_trims[i] = np.full(Hp, self.trim[i])
                    else:
                        ps = self.prev_shapes[i]
                        shapes_now[i] = ps[1:] + [ps[-1]]
                        self.prev_traj[i] = np.vstack([self.prev_traj[i][1:], self.prev_traj[i][-1:]])
                        self.prev_trims[i] = np.concatenate([self.prev_trims[i][1:], self.prev_trims[i][-1:]])
                # Simulation.apply: plant/Simulation.m:93-98
                new_pose[i] = self.prev_traj[i][0]
                new_trim[i] = self.prev_trims[i][0]
            out.append(StepRecord(self.k, lvl, members, batch, res))
        self.prev_shapes = shapes_now
        self.pose, self.trim = new_pose, new_trim
        self.records.extend(out)
        return out

    def run(self, n_steps: int) -> List[StepRecord]:
        for _ in range(n_steps):
            self.step()
        return self.records


# --------------------------------------------------------------------------- BASELINE config 3
def computation_level_permutations(n_levels: int, seed: int) -> np.ndarray:
    """PrioritizedExplorativeController.computation_level_permutations :241-309: n_levels permutations of
    the computation levels forming a Latin square (every level class is tried at every position once);
    row 1 is the identity, the others are filled cell by cell — always the cell with the fewest
    possibilities, one of them at random — and re-drawn on a dead end.  Stream: RandStream('mt19937ar',
    Seed = time step), which numpy's RandomState reproduces; [dev] randi(stream, n) is taken as
    floor(n * rand) + 1 (MATLAB's exact rule is not published: parity unpinned)."""
    n = int(n_levels)
    result = np.zeros((n, n), dtype=np.int64)
    result[0] = np.arange(1, n + 1)
    rs = np.random.RandomState(int(seed) if int(seed) != 0 else 5489)
    nth = 1
    while nth < n:
        perm = np.zeros(n, dtype=np.int64)
        allowed = np.ones((n, n), dtype=bool)            # [level, class]
        for col in range(n):
            picked = result[:, col][result[:, col] != 0]
            allowed[picked - 1, col] = False
        filled, valid = 0, True
        while filled < n:
            sums = allowed.sum(axis=0)
            cell = int(np.argmin(sums))                  # first minimum, like min()
            n_pos = int(sums[cell])
            if n_pos == 0:
                valid = False
                break
            poss = np.flatnonzero(allowed[:, cell])
            level = int(poss[int(np.floor(rs.random_sample() * n_pos))])
            perm[cell] = level + 1
            allowed[level, :] = False
            allowed[:, cell] = True                      # never the minimum again
            filled += 1
        if not valid:
            continue
        result[nth] = perm
        nth += 1
    return result


def fixed_permutation_set(n_levels: int, seed: int, count: int) -> np.ndarray:
    """BASELINE configs[2] asks for a FIXED number of priority permutations per time step (8, one per GPU), the
    reference generates n_CL of them (one Latin square).  [dev] pad / truncate (SURVEY.md §8(d)):
      n_CL >= count  the first `count` rows of the reference's Latin square;
      n_CL <  count  the reference's n_CL rows first, then uniformly drawn permutations of the levels (MT19937 stream
                     seeded seed + 7919) that are not in the set yet; if the n_CL! distinct permutations run out
                     (n_CL <= 3), the identity is repeated.
    The reference's own rows always come first and the choice takes the FIRST minimum, so a padded row only wins
    when it is strictly cheaper than every reference row."""
    perms = computation_level_permutations(n_levels, seed)
    if perms.shape[0] >= count:
        return perms[:count]
    rows = [tuple(int(x) for x in r) for r in perms]
    seen = set(rows)
    import math
    limit = min(count, math.factorial(n_levels))
    rs = np.random.RandomState(int(seed) + 7919)
    while len(rows) < limit:
        r = tuple(int(x) + 1 for x in rs.permutation(n_levels))
        if r not in seen:
            seen.add(r)
            rows.append(r)
    while len(rows) < count:
        rows.append(rows[0])
    return np.array(rows, dtype=np.int64)


def weak_components(D: np.ndarray) -> np.ndarray:
    """conncomp(digraph(D), 'Type', 'weak'): 1-based component label per vertex, components numbered in
    the order of their lowest vertex (PrioritizedExplorativeController.m:207)."""
    n = D.shape[0]
    und = (D | D.T).astype(bool)
    label = np.zeros(n, dtype=np.int64)
    nxt = 0
    for s0 in range(n):
        if label[s0]:
            continue
        nxt += 1
        stack = [s0]
        label[s0] = nxt
        while stack:
            u = stack.pop()
            for v in np.flatnonzero(und[u]):
                if not label[v]:
                    label[v] = nxt
                    stack.append(int(v))
    return label


def permuted_coupling(D: np.ndarray, levels: np.ndarray, perm: np.ndarray) -> np.ndarray:
    """The directed coupling of one permutation of the computation levels (PrioritizedExplorativeController.m:55-78):
    lev_p = perm[levels - 1] (i11changem), and every edge i -> j of D with lev_p(i) > lev_p(j) is reversed."""
    lev_p = np.asarray(perm)[np.asarray(levels) - 1]
    Dp = D.copy()
    for i, j in zip(*np.nonzero(D)):
        if lev_p[i] > lev_p[j]:
            Dp[i, j], Dp[j, i] = False, True
    return Dp


class ExplorativeRunner(ScenarioRunner):
    """BASELINE configs[2]: simultaneous multiple prioritizations.  Every time step the n_CL computation
    levels of the base prioritisation are permuted n_CL times (Latin square), every permutation is solved
    as a complete time step, the cheapest one per weakly connected sub-graph is applied
    (PrioritizedExplorativeController.m:21-176, PrioritizedExplorativeSequentialController.m:29-38).

    All permutations a rank owns (sharding.shard_block_cyclic over `world` ranks = GPUs) go into ONE
    timestep_fn call (len(my permutations) x n searches, predecessor relations block by block); the only
    exchange between ranks is the cost matrix and the winners' plans (sharding.choose_permutation /
    gather_winner_plans: one all_gather each, NCCL on GPUs).  The host logic is replicated on every rank.
    [dev] the cost of an exhausted vehicle is the re-computed cost of its fallback trajectory
    (plan_fallback :696-711); the winner does not re-seed the prioritizer (:169-173)."""

    def __init__(self, sc: Scenario, timestep_fn, rank: int = 0, world: int = 1, device=None, max_permutations: int = 0,
                 fixed_permutations: int = 0, exchange=None, explorative_fn=None, coupler: str = "corridor"):
        """fixed_permutations: exactly that many permutations per time step (fixed_permutation_set: BASELINE's 8).
        exchange(n_rows_local, n, fallback_rows, mine, P, belonging) -> (chosen, solution_cost, plans): replaces the
        host-side exchange below by one that starts from the plans in DEVICE memory (bench: pdmpc_pack_plan_rows +
        one NCCL all_gather); fallback_rows [n, 2 + 21*Hp] = cost and plan a vehicle takes when its search is exhausted.
        explorative_fn(path_id, x, y, yaw, speed, trim, slot, successors, level, permutations, half_length, half_width, dt,
        checker) -> (BatchResult, choice) (capi.Planner.plan_timestep_explorative): the whole time step — inputs,
        obstacles, every permutation's searches, fallback plans, the choice and the closed-loop state — in ONE call;
        D, the levels and the permutations are still decided here; slot = path id = path_id0 + vehicle.
        coupler: as ScenarioRunner's."""
        super().__init__(sc, None, timestep_fn=timestep_fn, coupler=coupler)
        self.explorative_fn = explorative_fn
        self.rank, self.world, self.device = rank, world, device
        self.max_permutations = max_permutations      # 0 = all n_CL
        self.fixed_permutations = fixed_permutations
        self.exchange = exchange
        self.explorative_records: List[dict] = []

    def decide(self):
        """Directed coupling D, computation levels and the permutations of this time step (self.k)."""
        A = self._adjacency()
        D = (constant_priorities(A) if self.sc.priority == "constant" else coloring_priorities(A)).astype(bool)
        levels = kahn(D.astype(np.int64))
        n_cl = int(levels.max())
        if self.fixed_permutations:
            perms = fixed_permutation_set(n_cl, self.k, self.fixed_permutations)
        else:
            perms = computation_level_permutations(n_cl, self.k)
        if self.max_permutations:
            perms = perms[: self.max_permutations]
        return D, levels, perms

    def explorative_args(self):
        """(D, levels, perms) and the per-vehicle arguments of explorative_fn up to the permutations."""
        D, levels, perms = self.decide()
        mpa, n = self.mpa, self.sc.amount
        speed = np.array([mpa.trim_speed[self.trim[i] - 1] for i in range(n)], dtype=np.float64)
        ids = self.path_id0 + np.arange(n)
        return (D, levels, perms), (ids, self.pose[:, 0], self.pose[:, 1], self.pose[:, 2], speed, self.trim, ids,
                                    [np.flatnonzero(D[i, :]) for i in range(n)], levels)

    def apply_explorative(self, res: BatchResult, choice: dict, decision) -> None:
        """Take the winners of one explorative call (rows of res, choice of this scenario) and record the step."""
        _D, levels, perms = decision
        bel, chosen = np.asarray(choice["belonging"]), np.asarray(choice["chosen"])
        rows = np.asarray(choice["applied_row"])
        self.apply_final(dataclasses.replace(res, **{f.name: getattr(res, f.name)[rows] for f in dataclasses.fields(res)
                                                     if isinstance(getattr(res, f.name), np.ndarray)}))
        first = [int(np.flatnonzero(bel == g)[0]) for g in range(1, int(bel.max()) + 1)]
        self.explorative_records.append({"step": self.k, "n_permutations": perms.shape[0], "n_levels": int(levels.max()),
                                         "chosen": chosen[first].astype(np.int64), "solution_cost": choice["solution_cost"],
                                         "searches_local": perms.shape[0] * self.sc.amount, "result_local": res})

    def step(self):
        from . import sharding
        sc, mpa = self.sc, self.mpa
        n, Hp = sc.amount, mpa.Hp
        self.k += 1
        if self.explorative_fn is not None:
            decision, args = self.explorative_args()
            res, choice = self.explorative_fn(*args, [decision[2]], VEH_LENGTH / 2 + 0.01, VEH_WIDTH / 2 + 0.01,
                                              mpa.dt_seconds, sc.checker)
            choice = dict(choice, solution_cost=choice["solution_cost"][0])
            self.apply_explorative(res, choice, decision)
            return []
        base = self._iters()
        D, levels, perms = self.decide()
        n_cl = int(levels.max())
        P = perms.shape[0]
        belonging = weak_components(D)
        fallbacks = [self._fallback_plan(i) for i in range(n)]
        fb_cost = np.array([float(np.sum((base[i].reference_trajectory_points - fallbacks[i][1][:, :2]) ** 2))
                            for i in range(n)])
        mine = sharding.shard_block_cyclic(P, self.rank, self.world)
        batches, deps = [], []
        for p in mine:
            Dp = permuted_coupling(D, levels, perms[p])
            its = []
            for i in range(n):
                it = dataclasses.replace(base[i], obstacles=list(base[i].obstacles),
                                         dynamic_obstacle_area=list(base[i].dynamic_obstacle_area))
                for j in np.flatnonzero(Dp[i, :]):         # consider_successors, area_of_standstill
                    if abs(mpa.trim_speed[self.trim[j] - 1]) < 0.01:
                        it.obstacles.append(occupied_area(*self.pose[j]))
                its.append(it)
            batches.append(SearchBatch.from_iters(its, Hp, sc.checker, mpa.dt_seconds))
            deps.append(TimestepDeps.build([np.flatnonzero(Dp[:, i]) for i in range(n)], [f[0] for f in fallbacks], Hp))
        plan_len = 1 + Hp + 3 * Hp + Hp + 2 * Hp * 8

        def fallback_row(v):
            shapes, traj, trims = fallbacks[v]
            npts = np.array([s.shape[1] for s in shapes])
            sx = np.zeros((Hp, 8)); sy = np.zeros((Hp, 8))
            for k2, s2 in enumerate(shapes):
                sx[k2, :s2.shape[1]], sy[k2, :s2.shape[1]] = s2[0], s2[1]
            return np.concatenate([[1.0], trims, traj.reshape(-1), npts, sx.reshape(-1), sy.reshape(-1)])

        res = None
        batch = dep_all = None
        if len(mine):
            batch = SearchBatch.concat(batches)
            dep_all = TimestepDeps.concat(deps, [n] * len(mine))
            res = self.timestep_fn(batch, dep_all)
        if self.exchange is not None:
            fb_rows = np.stack([np.concatenate([[fb_cost[v]], fallback_row(v)]) for v in range(n)])
            chosen, solution_cost, plans = self.exchange(len(mine) * n, n, fb_rows, mine, P, belonging)
        else:
            cost_local = np.zeros((len(mine), n))
            plans_local = np.zeros((len(mine), n, plan_len))
            for pl in range(len(mine)):
                for v in range(n):
                    r = pl * n + v
                    if res.is_exhausted[r]:
                        cost_local[pl, v] = fb_cost[v]
                        plans_local[pl, v] = fallback_row(v)
                    else:
                        cost_local[pl, v] = res.g_path[r, Hp]   # tree.get_cost(tree_path(end)), :100-104
                        plans_local[pl, v] = np.concatenate([[0.0], res.trims[r, 1:], res.y_predicted[r].reshape(-1),
                                                             res.shape_npts[r], res.shape_x[r].reshape(-1),
                                                             res.shape_y[r].reshape(-1)])
            coll = self.world > 1
            chosen, solution_cost = sharding.choose_permutation(cost_local, mine, P, belonging, self.device, coll)
            plans = sharding.gather_winner_plans(plans_local, mine, P, chosen, belonging, self.device, coll)
        shapes_now: List[Optional[List[np.ndarray]]] = [None] * n
        new_pose, new_trim = self.pose.copy(), self.trim.copy()
        for v in range(n):
            row = plans[v]
            self.n_fallbacks += int(row[0])
            o = 1
            self.prev_trims[v] = row[o:o + Hp].astype(np.int64); o += Hp
            self.prev_traj[v] = row[o:o + 3 * Hp].reshape(Hp, 3).copy(); o += 3 * Hp
            npts = row[o:o + Hp].astype(np.int64); o += Hp
            sx = row[o:o + Hp * 8].reshape(Hp, 8); o += Hp * 8
            sy = row[o:o + Hp * 8].reshape(Hp, 8)
            shapes_now[v] = [np.vstack([sx[k2, :npts[k2]], sy[k2, :npts[k2]]]) for k2 in range(Hp)]
            new_pose[v] = self.prev_traj[v][0]
            new_trim[v] = self.prev_trims[v][0]
        self.prev_shapes = shapes_now
        self.pose, self.trim = new_pose, new_trim
        self.explorative_records.append({"step": self.k, "n_permutations": P, "n_levels": n_cl, "chosen": chosen,
                                         "solution_cost": solution_cost, "searches_local": len(mine) * n,
                                         "result_local": res})
        return []


def lockstep_step(runners: Sequence[ScenarioRunner], timestep_fn) -> BatchResult:
    """One time step of MANY independent scenarios as ONE optimizer call (BASELINE configs[4] in closed
    loop): the scenarios' searches and predecessor DAGs are concatenated block by block."""
    parts, sizes, fbs = [], [], []
    for r in runners:
        r.k += 1
        iters, preds, fallbacks = r.timestep_inputs()
        parts.append((SearchBatch.from_iters(iters, r.mpa.Hp, r.sc.checker, r.mpa.dt_seconds),
                      TimestepDeps.build(preds, [f[0] for f in fallbacks], r.mpa.Hp)))
        sizes.append(r.sc.amount)
        fbs.append(fallbacks)
    batch = SearchBatch.concat([b for b, _d in parts])
    res = timestep_fn(batch, TimestepDeps.concat([d for _b, d in parts], sizes))
    off = 0
    for r, n, fallbacks in zip(runners, sizes, fbs):
        rows = dataclasses.replace(res, **{f.name: getattr(res, f.name)[off:off + n] for f in dataclasses.fields(res)
                                           if isinstance(getattr(res, f.name), np.ndarray)})
        r.apply_timestep(rows, fallbacks)
        off += n
    return res


def explorative_lockstep_step(runners: Sequence[ExplorativeRunner], explorative_fn) -> BatchResult:
    """One time step of MANY explorative scenarios as ONE explorative_fn call (capi.Planner.plan_timestep_explorative with
    scenario_ptr): every runner decides its coupling, levels and permutations on the host, then all permutations of all
    scenarios are planned, chosen and committed together; each runner applies its winners."""
    decisions, cols = [], None
    for r in runners:
        r.k += 1
        d, args = r.explorative_args()
        decisions.append(d)
        cols = [list(a) for a in args] if cols is None else [c + list(a) for c, a in zip(cols, args)]
    sizes = [r.sc.amount for r in runners]
    sp = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    path_id, x, y, yaw, speed, trim, slot, succ, level = cols
    succ = [np.asarray(sv) + sp[s] for s in range(len(runners)) for sv in succ[sp[s]:sp[s + 1]]]
    r0 = runners[0]
    res, choice = explorative_fn(np.array(path_id), np.array(x), np.array(y), np.array(yaw), np.array(speed), np.array(trim),
                                 np.array(slot), succ, np.array(level), [d[2] for d in decisions], VEH_LENGTH / 2 + 0.01,
                                 VEH_WIDTH / 2 + 0.01, r0.mpa.dt_seconds, r0.sc.checker, scenario_ptr=sp)
    for s, (r, d) in enumerate(zip(runners, decisions)):
        a, b = sp[s], sp[s + 1]
        r.apply_explorative(res, {"belonging": choice["belonging"][a:b], "chosen": choice["chosen"][a:b],
                                  "applied_row": choice["applied_row"][a:b], "solution_cost": choice["solution_cost"][s]}, d)
    return res


class CentralizedRunner(ScenarioRunner):
    """CentralizedController (hlc/controller/centralized/CentralizedController.m:33-59): ONE joint search over all
    vehicles per time step (rows of the batch = vehicles), SAT checker, no priorities.  joint_fn(batch, n_vehicles)
    plans it; an exhausted search makes every vehicle take its fallback plan (:46-54)."""

    def __init__(self, sc: Scenario, joint_fn):
        super().__init__(sc, None)
        self.joint_fn = joint_fn
        self.joint_records: List[tuple] = []

    def step(self):
        sc, mpa = self.sc, self.mpa
        n = sc.amount
        self.k += 1
        iters = [self._iter_for(i) for i in range(n)]
        fallbacks = [self._fallback_plan(i) for i in range(n)]
        batch = SearchBatch.from_iters(iters, mpa.Hp, CHECKER_SAT, mpa.dt_seconds)
        res = self.joint_fn(batch, n)
        self.apply_timestep(res, fallbacks)
        self.joint_records.append((self.k, batch, res))
        return []


def _assign_rows(dst: BatchResult, rows, src: BatchResult) -> None:
    for f in dataclasses.fields(dst):
        a = getattr(dst, f.name)
        if isinstance(a, np.ndarray):
            a[rows] = getattr(src, f.name)


def mcts_seeds(time_step: int, n: int) -> np.ndarray:
    """RandStream seeds of vehicles 1..n at time step `time_step` (1-based): time_step + vehicle_index
    (MonteCarloTreeSearch.m:31 with the arguments PrioritizedController.plan passes, :335-341)."""
    return (int(time_step) + np.arange(1, n + 1)).astype(np.uint32)


def plan_timestep_by_levels(plan_fn: PlanFn, batch: SearchBatch, deps: TimestepDeps, seeds=None) -> BatchResult:
    """The reference's way through one time step, as the specification of pdmpc_plan_timestep:
    computation levels one after the other (utility/kahn.m, PrioritizedSequentialController.m:83-92),
    each vehicle's iter_v extended on the HOST by the areas its sequential predecessors published
    (PrioritizedController.m:297-324, consider_predecessors :449-506), an exhausted predecessor
    publishing its fallback areas (:568-621, :678-718).  With `seeds` (the sampled optimizer, the specification of
    pdmpc_mcts_plan_timestep) a level is planned as plan_fn(sub_batch, seeds[members])."""
    iters, Hp, checker, dt_seconds = batch.to_iters(), batch.Hp, batch.checker, batch.dt_seconds
    n = len(iters)
    level = np.zeros(n, dtype=np.int64)
    remaining = set(range(n))
    lvl = 0
    while remaining:
        lvl += 1
        ready = [i for i in sorted(remaining) if all(level[j] != 0 and level[j] < lvl for j in deps.preds(i))]
        if not ready:
            raise ValueError("predecessor relation has a cycle")
        for i in ready:
            level[i] = lvl
        remaining -= set(ready)
    out = BatchResult.empty(n, Hp)
    published: List[Optional[List[np.ndarray]]] = [None] * n
    for l in range(1, lvl + 1):
        members = np.flatnonzero(level == l)
        its = []
        for i in members:
            it = dataclasses.replace(iters[i], obstacles=list(iters[i].obstacles),
                                     dynamic_obstacle_area=list(iters[i].dynamic_obstacle_area))
            for j in deps.preds(i):
                if all(a.shape[1] == 0 for a in published[j]):
                    continue   # nothing published (no fallback areas given)
                it.dynamic_obstacle_area.append(published[j])
            its.append(it)
        sub = SearchBatch.from_iters(its, Hp, checker, dt_seconds)
        res = plan_fn(sub) if seeds is None else plan_fn(sub, np.asarray(seeds)[members])
        _assign_rows(out, members, res)
        for b, i in enumerate(members):
            published[i] = deps.fallback_shapes(i) if res.is_exhausted[b] else res.shapes(b)
    return out


def roll_out(sc: Scenario, plan_fn: PlanFn, n_steps: int) -> SearchBatch:
    """Closed-loop roll-out; returns every search record of the run as one flat batch."""
    recs = ScenarioRunner(sc, plan_fn).run(n_steps)
    return SearchBatch.concat([r.batch for r in recs])
