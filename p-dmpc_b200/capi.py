"""ctypes binding of the C ABI in include/pdmpc_b200.h.

This is the Python stand-in for the MEX shim (MATLAB/mex are absent from this
image, SURVEY.md §8c): tests, bench.py and the host harness go through exactly
the entry points a MATLAB maintainer would bind (INTEGRATION.md).

There is no CPU fallback: if ``libpdmpc_b200.so`` is missing or no CUDA device is
visible, ``load_library`` / ``Planner`` raise.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

from .mpa import MotionPrimitiveAutomaton
from .records import BatchResult, SearchBatch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "csrc", "libpdmpc_b200.so")

PDMPC_OK = 0
PDMPC_ERR_BAD_INPUT = 1
PDMPC_ERR_CUDA = 2
PDMPC_ERR_CAPACITY = 3
PDMPC_ERR_NO_MPA = 4
PDMPC_ERR_ALLOC = 5

EXPORTED_SYMBOLS = (
    "pdmpc_create", "pdmpc_destroy", "pdmpc_last_error", "pdmpc_abi_version",
    "pdmpc_set_node_capacity", "pdmpc_set_variant", "pdmpc_set_tile_points", "pdmpc_set_cta_queue", "pdmpc_set_escalation", "pdmpc_get_hp", "pdmpc_pack_plan_rows", "pdmpc_upload_road", "pdmpc_sample_inputs", "pdmpc_upload_reachable_sets", "pdmpc_assemble_obstacles", "pdmpc_get_pipeline_timeline", "pdmpc_pipeline_bounds", "pdmpc_escalation_budgets", "pdmpc_plan_timestep_from_states", "pdmpc_closed_loop_reset", "pdmpc_plan_timestep_closed_loop", "pdmpc_host_alloc", "pdmpc_host_free",
    "pdmpc_trace_staged", "pdmpc_upload_mpa", "pdmpc_plan_batch", "pdmpc_stage_batch",
    "pdmpc_run_staged", "pdmpc_sync", "pdmpc_fetch_staged", "pdmpc_get_stats", "pdmpc_stream",
    "pdmpc_mcts_plan_batch", "pdmpc_mcts_run_staged", "pdmpc_set_cta_heap_smem", "pdmpc_plan_timestep",
    "pdmpc_set_pipeline_chunks", "pdmpc_measure_fp64_peak", "pdmpc_joint_plan_batch",
    "pdmpc_couple", "pdmpc_plan_timestep_from_states_coupled", "pdmpc_plan_timestep_explorative",
    "pdmpc_mcts_plan_timestep", "pdmpc_mcts_plan_timestep_closed_loop", "pdmpc_mcts_plan_timestep_from_states",
)

_p_u8 = C.POINTER(C.c_uint8)
_p_i32 = C.POINTER(C.c_int32)
_p_u64 = C.POINTER(C.c_uint64)
_p_f64 = C.POINTER(C.c_double)


class MpaDesc(C.Structure):
    _fields_ = [
        ("n_trims", C.c_int32), ("Hp", C.c_int32), ("n_edges", C.c_int32),
        ("transition", _p_u8), ("edge_from", _p_i32), ("edge_to", _p_i32),
        ("edge_dx", _p_f64), ("edge_dy", _p_f64), ("edge_dyaw", _p_f64),
        ("area_npts", _p_i32), ("area_x", _p_f64), ("area_y", _p_f64),
    ]


class BatchIn(C.Structure):
    _fields_ = [
        ("n_searches", C.c_int32), ("checker", C.c_int32), ("dt_seconds", C.c_double),
        ("x0", _p_f64), ("y0", _p_f64), ("yaw0", _p_f64), ("trim0", _p_i32),
        ("ref_x", _p_f64), ("ref_y", _p_f64), ("v_ref", _p_f64),
        ("slot_ptr", _p_i32), ("poly_ptr", _p_i32), ("vert_x", _p_f64), ("vert_y", _p_f64),
        ("lane_ptr", _p_i32), ("lane_x", _p_f64), ("lane_y", _p_f64),
    ]


class MctsParams(C.Structure):
    _fields_ = [("n_expansions_max", C.c_int32), ("seed", C.POINTER(C.c_uint32))]


class TimestepDepsC(C.Structure):
    _fields_ = [("pred_ptr", _p_i32), ("pred_idx", _p_i32), ("fb_npts", _p_i32), ("fb_x", _p_f64), ("fb_y", _p_f64)]


class BatchOut(C.Structure):
    _fields_ = [
        ("status", _p_i32), ("is_exhausted", _p_u8), ("n_expanded", _p_i32), ("n_pops", _p_i32),
        ("pop_hash", _p_u64), ("trims", _p_i32), ("tree_path", _p_i32), ("y_predicted", _p_f64),
        ("g_path", _p_f64), ("h_path", _p_f64), ("shape_npts", _p_i32),
        ("shape_x", _p_f64), ("shape_y", _p_f64),
    ]


class RoadDescC(C.Structure):
    _fields_ = [("n_lanelets", C.c_int32), ("bound_ptr", _p_i32), ("bound_x", _p_f64), ("bound_y", _p_f64),
                ("n_paths", C.c_int32), ("path_ptr", _p_i32), ("path_x", _p_f64), ("path_y", _p_f64),
                ("lan_ptr", _p_i32), ("lanelets_index", _p_i32), ("points_index", _p_i32),
                ("is_loop", C.POINTER(C.c_uint8)), ("reference_speed", _p_f64)]


class InputsOutC(C.Structure):
    _fields_ = [("ref_x", _p_f64), ("ref_y", _p_f64), ("v_ref", _p_f64), ("ref_index", _p_i32), ("current_index", _p_i32),
                ("predicted_lanelets", _p_i32), ("lane_ptr", _p_i32), ("lane_x", _p_f64), ("lane_y", _p_f64),
                ("lane_capacity", C.c_int32)]


class ReachDescC(C.Structure):
    _fields_ = [("n_trims", C.c_int32), ("Hp", C.c_int32), ("ptr", _p_i32), ("x", _p_f64), ("y", _p_f64)]


class CouplingInC(C.Structure):
    _fields_ = [("n", C.c_int32), ("x", _p_f64), ("y", _p_f64), ("yaw", _p_f64), ("speed", _p_f64), ("trim", _p_i32),
                ("succ_ptr", _p_i32), ("succ_idx", _p_i32), ("par_ptr", _p_i32), ("par_idx", _p_i32),
                ("half_length", C.c_double), ("half_width", C.c_double)]


class ObstaclesOutC(C.Structure):
    _fields_ = [("slot_ptr", _p_i32), ("poly_ptr", _p_i32), ("vert_x", _p_f64), ("vert_y", _p_f64),
                ("poly_capacity", C.c_int32), ("vert_capacity", C.c_int32), ("n_polys", C.c_int32), ("n_verts", C.c_int32)]


class TimestepStatesC(C.Structure):
    _fields_ = [("n", C.c_int32), ("path_id", _p_i32), ("x", _p_f64), ("y", _p_f64), ("yaw", _p_f64), ("speed", _p_f64),
                ("trim", _p_i32), ("succ_ptr", _p_i32), ("succ_idx", _p_i32), ("par_ptr", _p_i32), ("par_idx", _p_i32),
                ("pred_ptr", _p_i32), ("pred_idx", _p_i32), ("slot", _p_i32),
                ("half_length", C.c_double), ("half_width", C.c_double), ("dt_seconds", C.c_double), ("checker", C.c_int32)]


class CoupleParamsC(C.Structure):
    _fields_ = [("n_scenarios", C.c_int32), ("scenario_ptr", _p_i32), ("prioritizer", C.c_int32), ("max_num_CLs", C.c_int32)]


class CoupleOutC(C.Structure):
    _fields_ = [("succ_ptr", _p_i32), ("succ_idx", _p_i32), ("par_ptr", _p_i32), ("par_idx", _p_i32),
                ("pred_ptr", _p_i32), ("pred_idx", _p_i32), ("idx_capacity", C.c_int32), ("level", _p_i32),
                ("overlap_area", _p_f64)]


class ExplorativeInC(C.Structure):
    _fields_ = [("n_scenarios", C.c_int32), ("scenario_ptr", _p_i32), ("level", _p_i32), ("perm_ptr", _p_i32),
                ("perm_val_ptr", _p_i32), ("perm", _p_i32)]


class ExplorativeOutC(C.Structure):
    _fields_ = [("belonging", _p_i32), ("chosen", _p_i32), ("applied_row", _p_i32), ("row_cost", _p_f64),
                ("solution_cost", _p_f64)]


MAX_PRED_LANELETS = 8
PRIORITY_CONSTANT, PRIORITY_COLORING = 0, 1
COUPLE_MAX_VEHICLES = 64


class Stats(C.Structure):
    _fields_ = [
        ("kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("total_pops", C.c_int64),
        ("total_nodes", C.c_int64), ("total_obstacle_cols", C.c_int64),
        ("kernel_launches", C.c_int32), ("handed_over", C.c_int32), ("shape", C.c_int32), ("escalated", C.c_int32),
    ]


def _ptr(a: np.ndarray, ty):
    assert a.flags["C_CONTIGUOUS"], "array must be contiguous"
    return a.ctypes.data_as(ty)


def mpa_desc(mpa: MotionPrimitiveAutomaton):
    """Returns (MpaDesc, keepalive) for an MPA table set."""
    keep = dict(
        transition=np.ascontiguousarray(mpa.transition, dtype=np.uint8),
        edge_from=np.ascontiguousarray(mpa.edge_from, dtype=np.int32),
        edge_to=np.ascontiguousarray(mpa.edge_to, dtype=np.int32),
        edge_dx=np.ascontiguousarray(mpa.edge_dx, dtype=np.float64),
        edge_dy=np.ascontiguousarray(mpa.edge_dy, dtype=np.float64),
        edge_dyaw=np.ascontiguousarray(mpa.edge_dyaw, dtype=np.float64),
        area_npts=np.ascontiguousarray(mpa.area_npts, dtype=np.int32),
        area_x=np.ascontiguousarray(mpa.area_x, dtype=np.float64),
        area_y=np.ascontiguousarray(mpa.area_y, dtype=np.float64),
    )
    d = MpaDesc(
        n_trims=mpa.n_trims, Hp=mpa.Hp, n_edges=mpa.n_edges,
        transition=_ptr(keep["transition"], _p_u8), edge_from=_ptr(keep["edge_from"], _p_i32),
        edge_to=_ptr(keep["edge_to"], _p_i32), edge_dx=_ptr(keep["edge_dx"], _p_f64),
        edge_dy=_ptr(keep["edge_dy"], _p_f64), edge_dyaw=_ptr(keep["edge_dyaw"], _p_f64),
        area_npts=_ptr(keep["area_npts"], _p_i32), area_x=_ptr(keep["area_x"], _p_f64),
        area_y=_ptr(keep["area_y"], _p_f64))
    return d, keep


def batch_in(b: SearchBatch) -> BatchIn:
    return BatchIn(
        n_searches=b.n, checker=b.checker, dt_seconds=b.dt_seconds,
        x0=_ptr(b.x0, _p_f64), y0=_ptr(b.y0, _p_f64), yaw0=_ptr(b.yaw0, _p_f64),
        trim0=_ptr(b.trim0, _p_i32), ref_x=_ptr(b.ref_x, _p_f64), ref_y=_ptr(b.ref_y, _p_f64),
        v_ref=_ptr(b.v_ref, _p_f64), slot_ptr=_ptr(b.slot_ptr, _p_i32),
        poly_ptr=_ptr(b.poly_ptr, _p_i32), vert_x=_ptr(b.vert_x, _p_f64),
        vert_y=_ptr(b.vert_y, _p_f64), lane_ptr=_ptr(b.lane_ptr, _p_i32),
        lane_x=_ptr(b.lane_x, _p_f64), lane_y=_ptr(b.lane_y, _p_f64))


def mcts_params(seeds, n_expansions_max: int, n: int):
    """Returns (MctsParams, keepalive): seed[i] = time_step + vehicle_index (MonteCarloTreeSearch.m:31)."""
    seeds = np.ascontiguousarray(np.broadcast_to(np.asarray(seeds, dtype=np.uint32), (n,)))
    return MctsParams(n_expansions_max=int(n_expansions_max),
                      seed=seeds.ctypes.data_as(C.POINTER(C.c_uint32))), seeds


def batch_out(r: BatchResult) -> BatchOut:
    return BatchOut(
        status=_ptr(r.status, _p_i32), is_exhausted=_ptr(r.is_exhausted, _p_u8),
        n_expanded=_ptr(r.n_expanded, _p_i32), n_pops=_ptr(r.n_pops, _p_i32),
        pop_hash=_ptr(r.pop_hash, _p_u64), trims=_ptr(r.trims, _p_i32),
        tree_path=_ptr(r.tree_path, _p_i32), y_predicted=_ptr(r.y_predicted, _p_f64),
        g_path=_ptr(r.g_path, _p_f64), h_path=_ptr(r.h_path, _p_f64),
        shape_npts=_ptr(r.shape_npts, _p_i32), shape_x=_ptr(r.shape_x, _p_f64),
        shape_y=_ptr(r.shape_y, _p_f64))


_LIB: Optional[C.CDLL] = None


def load_library(path: str = LIB_PATH) -> C.CDLL:
    """dlopen the C-ABI library and declare every prototype.  Raises if absent."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "There is no CPU fallback for the optimizer.")
    lib = C.CDLL(path)
    H = C.c_void_p
    lib.pdmpc_create.argtypes = [C.c_int, C.POINTER(H)]
    lib.pdmpc_create.restype = C.c_int
    lib.pdmpc_destroy.argtypes = [H]
    lib.pdmpc_destroy.restype = C.c_int
    lib.pdmpc_last_error.argtypes = [H]
    lib.pdmpc_last_error.restype = C.c_char_p
    lib.pdmpc_abi_version.argtypes = []
    lib.pdmpc_abi_version.restype = C.c_int
    lib.pdmpc_set_node_capacity.argtypes = [H, C.c_int32]
    lib.pdmpc_set_node_capacity.restype = C.c_int
    lib.pdmpc_set_variant.argtypes = [H, C.c_int32]
    lib.pdmpc_set_variant.restype = C.c_int
    lib.pdmpc_set_cta_heap_smem.argtypes = [H, C.c_int32]
    lib.pdmpc_set_cta_heap_smem.restype = C.c_int
    lib.pdmpc_joint_plan_batch.argtypes = [H, C.POINTER(BatchIn), C.c_int32, C.POINTER(BatchOut)]
    lib.pdmpc_joint_plan_batch.restype = C.c_int
    lib.pdmpc_measure_fp64_peak.argtypes = [H, _p_f64, _p_f64]
    lib.pdmpc_measure_fp64_peak.restype = C.c_int
    lib.pdmpc_set_pipeline_chunks.argtypes = [H, C.c_int32]
    lib.pdmpc_set_pipeline_chunks.restype = C.c_int
    lib.pdmpc_set_cta_queue.argtypes = [H, C.c_int32]
    lib.pdmpc_set_cta_queue.restype = C.c_int
    lib.pdmpc_pack_plan_rows.argtypes = [H, C.c_int32, C.c_int32, _p_f64, C.c_void_p]
    lib.pdmpc_pack_plan_rows.restype = C.c_int
    lib.pdmpc_upload_road.argtypes = [H, C.POINTER(RoadDescC)]
    lib.pdmpc_upload_road.restype = C.c_int
    lib.pdmpc_sample_inputs.argtypes = [H, C.c_int32, _p_i32, _p_f64, _p_f64, _p_f64, C.c_double, C.POINTER(InputsOutC)]
    lib.pdmpc_sample_inputs.restype = C.c_int
    lib.pdmpc_upload_reachable_sets.argtypes = [H, C.POINTER(ReachDescC)]
    lib.pdmpc_upload_reachable_sets.restype = C.c_int
    lib.pdmpc_assemble_obstacles.argtypes = [H, C.POINTER(CouplingInC), C.POINTER(ObstaclesOutC)]
    lib.pdmpc_assemble_obstacles.restype = C.c_int
    lib.pdmpc_get_pipeline_timeline.argtypes = [H, C.c_int32, _p_f64, _p_f64, _p_f64, C.POINTER(C.c_int32)]
    lib.pdmpc_get_pipeline_timeline.restype = C.c_int
    lib.pdmpc_pipeline_bounds.argtypes = [C.c_int32, C.c_int32, C.c_int32, _p_i32, C.POINTER(C.c_int32)]
    lib.pdmpc_pipeline_bounds.restype = C.c_int
    lib.pdmpc_escalation_budgets.argtypes = [C.c_int32, C.c_int32, _p_i32, _p_i32]
    lib.pdmpc_escalation_budgets.restype = C.c_int
    lib.pdmpc_plan_timestep_from_states.argtypes = [H, C.POINTER(TimestepStatesC), C.POINTER(BatchOut)]
    lib.pdmpc_plan_timestep_from_states.restype = C.c_int
    lib.pdmpc_couple.argtypes = [H, C.c_int32, _p_f64, _p_f64, _p_f64, _p_i32, C.POINTER(CoupleParamsC), C.POINTER(CoupleOutC)]
    lib.pdmpc_couple.restype = C.c_int
    lib.pdmpc_plan_timestep_from_states_coupled.argtypes = [H, C.POINTER(TimestepStatesC), C.POINTER(CoupleParamsC),
                                                            C.POINTER(CoupleOutC), C.POINTER(BatchOut)]
    lib.pdmpc_plan_timestep_from_states_coupled.restype = C.c_int
    lib.pdmpc_plan_timestep_explorative.argtypes = [H, C.POINTER(TimestepStatesC), C.POINTER(ExplorativeInC),
                                                    C.POINTER(BatchOut), C.POINTER(ExplorativeOutC)]
    lib.pdmpc_plan_timestep_explorative.restype = C.c_int
    lib.pdmpc_closed_loop_reset.argtypes = [H, C.c_int32, C.c_double, C.c_double]
    lib.pdmpc_closed_loop_reset.restype = C.c_int
    lib.pdmpc_plan_timestep_closed_loop.argtypes = [H, C.POINTER(BatchIn), C.POINTER(TimestepDepsC), _p_i32,
                                                    C.POINTER(C.c_uint8), C.POINTER(BatchOut)]
    lib.pdmpc_plan_timestep_closed_loop.restype = C.c_int
    lib.pdmpc_get_hp.argtypes = [H]
    lib.pdmpc_get_hp.restype = C.c_int
    lib.pdmpc_set_escalation.argtypes = [H, C.c_int32, C.c_int32]
    lib.pdmpc_set_escalation.restype = C.c_int
    lib.pdmpc_set_tile_points.argtypes = [H, C.c_int32]
    lib.pdmpc_set_tile_points.restype = C.c_int
    lib.pdmpc_trace_staged.argtypes = [H, C.c_int32, C.POINTER(C.c_int64), C.c_int64, C.POINTER(C.c_int64)]
    lib.pdmpc_trace_staged.restype = C.c_int
    lib.pdmpc_host_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    lib.pdmpc_host_alloc.restype = C.c_int
    lib.pdmpc_host_free.argtypes = [C.c_void_p]
    lib.pdmpc_host_free.restype = C.c_int
    lib.pdmpc_upload_mpa.argtypes = [H, C.POINTER(MpaDesc)]
    lib.pdmpc_upload_mpa.restype = C.c_int
    lib.pdmpc_plan_batch.argtypes = [H, C.POINTER(BatchIn), C.POINTER(BatchOut)]
    lib.pdmpc_plan_batch.restype = C.c_int
    lib.pdmpc_stage_batch.argtypes = [H, C.POINTER(BatchIn)]
    lib.pdmpc_stage_batch.restype = C.c_int
    lib.pdmpc_run_staged.argtypes = [H]
    lib.pdmpc_run_staged.restype = C.c_int
    lib.pdmpc_sync.argtypes = [H]
    lib.pdmpc_sync.restype = C.c_int
    lib.pdmpc_fetch_staged.argtypes = [H, C.POINTER(BatchOut)]
    lib.pdmpc_fetch_staged.restype = C.c_int
    lib.pdmpc_get_stats.argtypes = [H, C.POINTER(Stats)]
    lib.pdmpc_get_stats.restype = C.c_int
    lib.pdmpc_mcts_plan_batch.argtypes = [H, C.POINTER(BatchIn), C.POINTER(MctsParams), C.POINTER(BatchOut)]
    lib.pdmpc_mcts_plan_batch.restype = C.c_int
    lib.pdmpc_mcts_run_staged.argtypes = [H, C.POINTER(MctsParams)]
    lib.pdmpc_mcts_run_staged.restype = C.c_int
    lib.pdmpc_plan_timestep.argtypes = [H, C.POINTER(BatchIn), C.POINTER(TimestepDepsC), C.POINTER(BatchOut)]
    lib.pdmpc_plan_timestep.restype = C.c_int
    lib.pdmpc_mcts_plan_timestep.argtypes = [H, C.POINTER(BatchIn), C.POINTER(TimestepDepsC), C.POINTER(MctsParams),
                                             C.POINTER(BatchOut)]
    lib.pdmpc_mcts_plan_timestep.restype = C.c_int
    lib.pdmpc_mcts_plan_timestep_closed_loop.argtypes = [H, C.POINTER(BatchIn), C.POINTER(TimestepDepsC), _p_i32,
                                                         C.POINTER(C.c_uint8), C.POINTER(MctsParams), C.POINTER(BatchOut)]
    lib.pdmpc_mcts_plan_timestep_closed_loop.restype = C.c_int
    lib.pdmpc_mcts_plan_timestep_from_states.argtypes = [H, C.POINTER(TimestepStatesC), C.POINTER(MctsParams),
                                                         C.POINTER(BatchOut)]
    lib.pdmpc_mcts_plan_timestep_from_states.restype = C.c_int
    lib.pdmpc_stream.argtypes = [H]
    lib.pdmpc_stream.restype = C.c_void_p
    _LIB = lib
    return lib


def pipeline_bounds(n_searches: int, chunks: int = 0, lib=None) -> np.ndarray:
    """Chunk boundaries of the copy/search pipeline for a batch of n_searches (pdmpc_pipeline_bounds; host-only)."""
    lib = lib or load_library()
    out = np.zeros(64, dtype=np.int32)
    n = C.c_int32()
    rc = lib.pdmpc_pipeline_bounds(int(n_searches), int(chunks), out.size, _ptr(out, _p_i32), C.byref(n))
    if rc != PDMPC_OK:
        raise PdmpcError(rc, "pdmpc_pipeline_bounds")
    return out[: n.value + 1].copy()


def escalation_budgets(n_searches: int, positions, lib=None) -> np.ndarray:
    """Pop budgets of the throughput shapes under the default escalation threshold for the searches at work positions
    `positions` of a batch of n_searches (pdmpc_escalation_budgets; host-only)."""
    lib = lib or load_library()
    pos = np.ascontiguousarray(positions, dtype=np.int32)
    out = np.zeros(pos.size, dtype=np.int32)
    rc = lib.pdmpc_escalation_budgets(int(n_searches), pos.size, _ptr(pos, _p_i32), _ptr(out, _p_i32))
    if rc != PDMPC_OK:
        raise PdmpcError(rc, "pdmpc_escalation_budgets")
    return out


class PdmpcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"pdmpc status {code}: {msg}")
        self.code = code


class Planner:
    """Owns one pdmpc_handle (one CUDA device, one stream)."""

    def __init__(self, device_id: int = 0):
        self.lib = load_library()
        self.h = C.c_void_p()
        rc = self.lib.pdmpc_create(device_id, C.byref(self.h))
        if rc != PDMPC_OK:
            msg = self.lib.pdmpc_last_error(None)
            raise PdmpcError(rc, (msg or b"pdmpc_create failed").decode())
        self._mpa_keep = None
        self._mpa = None
        self._staged_n = 0
        self._staged_Hp = 0

    def _check(self, rc: int):
        if rc != PDMPC_OK:
            raise PdmpcError(rc, (self.lib.pdmpc_last_error(self.h) or b"").decode())

    def close(self):
        if self.h:
            self.lib.pdmpc_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_node_capacity(self, n: int):
        self._check(self.lib.pdmpc_set_node_capacity(self.h, int(n)))

    def set_variant(self, variant: int):
        """0 = auto, 1 = one search per warp, 2 / 3 = tiles (2 / 4 searches per warp), 4 / 5 = one CTA per search (pdmpc_set_variant)."""
        self._check(self.lib.pdmpc_set_variant(self.h, int(variant)))

    def set_cta_heap_smem(self, entries: int = 0):
        """Shape 4 knob (pdmpc_set_cta_heap_smem); results do not depend on it."""
        self._check(self.lib.pdmpc_set_cta_heap_smem(self.h, int(entries)))

    def measure_fp64_peak(self):
        """(separate mul+add Tops/s, FMA TFLOP/s) of the device's FP64 pipe (pdmpc_measure_fp64_peak)."""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.pdmpc_measure_fp64_peak(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_pipeline_chunks(self, chunks: int = 0):
        """Chunked copy/search pipeline of plan_batch (pdmpc_set_pipeline_chunks); results do not depend on it."""
        self._check(self.lib.pdmpc_set_pipeline_chunks(self.h, int(chunks)))

    def set_cta_queue(self, valid_only: bool):
        """Valid-only queue whenever the CTA shape runs (pdmpc_set_cta_queue)."""
        self._check(self.lib.pdmpc_set_cta_queue(self.h, 1 if valid_only else 0))

    def pack_plan_rows(self, n_rows: int, n_vehicles: int, fallback_rows, device_ptr: int):
        """Plans of the last plan call as [n_rows, 2 + 21*Hp] doubles in device memory (pdmpc_pack_plan_rows)."""
        fb = None
        if fallback_rows is not None:
            fb = np.ascontiguousarray(fallback_rows, dtype=np.float64)
        self._check(self.lib.pdmpc_pack_plan_rows(self.h, int(n_rows), int(n_vehicles),
                                                  _ptr(fb, _p_f64) if fb is not None else None, C.c_void_p(int(device_ptr))))

    def upload_road(self, tables: dict):
        """Road boundaries + reference paths (scenario.road_tables) for pdmpc_sample_inputs (pdmpc_upload_road)."""
        t = {k: np.ascontiguousarray(v) for k, v in tables.items()}
        d = RoadDescC(n_lanelets=int(t["bound_ptr"].size // 2), bound_ptr=_ptr(t["bound_ptr"], _p_i32),
                      bound_x=_ptr(t["bound_x"], _p_f64), bound_y=_ptr(t["bound_y"], _p_f64),
                      n_paths=int(t["path_ptr"].size - 1), path_ptr=_ptr(t["path_ptr"], _p_i32),
                      path_x=_ptr(t["path_x"], _p_f64), path_y=_ptr(t["path_y"], _p_f64),
                      lan_ptr=_ptr(t["lan_ptr"], _p_i32), lanelets_index=_ptr(t["lanelets_index"], _p_i32),
                      points_index=_ptr(t["points_index"], _p_i32), is_loop=_ptr(t["is_loop"], C.POINTER(C.c_uint8)),
                      reference_speed=_ptr(t["reference_speed"], _p_f64))
        self._check(self.lib.pdmpc_upload_road(self.h, C.byref(d)))

    def sample_inputs(self, path_id, x, y, speed, dt_seconds: float, lane_capacity: int = 0) -> dict:
        """Reference trajectories and lanelet boundaries of n vehicles on the device (pdmpc_sample_inputs):
        ref_x, ref_y, v_ref [n, Hp], ref_index [n, Hp], current_index [n], predicted_lanelets [n, 8],
        lane_ptr [2n + 1], lane_x, lane_y."""
        path_id = np.ascontiguousarray(path_id, dtype=np.int32)
        x, y, speed = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, speed))
        n, Hp = int(path_id.size), int(self.lib.pdmpc_get_hp(self.h))
        cap = int(lane_capacity) or 512 * max(n, 1)
        o = {"ref_x": np.zeros((n, Hp)), "ref_y": np.zeros((n, Hp)), "v_ref": np.zeros((n, Hp)),
             "ref_index": np.zeros((n, Hp), dtype=np.int32), "current_index": np.zeros(n, dtype=np.int32),
             "predicted_lanelets": np.zeros((n, MAX_PRED_LANELETS), dtype=np.int32),
             "lane_ptr": np.zeros(2 * n + 1, dtype=np.int32), "lane_x": np.zeros(cap), "lane_y": np.zeros(cap)}
        oc = InputsOutC(ref_x=_ptr(o["ref_x"], _p_f64), ref_y=_ptr(o["ref_y"], _p_f64), v_ref=_ptr(o["v_ref"], _p_f64),
                        ref_index=_ptr(o["ref_index"], _p_i32), current_index=_ptr(o["current_index"], _p_i32),
                        predicted_lanelets=_ptr(o["predicted_lanelets"], _p_i32), lane_ptr=_ptr(o["lane_ptr"], _p_i32),
                        lane_x=_ptr(o["lane_x"], _p_f64), lane_y=_ptr(o["lane_y"], _p_f64), lane_capacity=cap)
        self._check(self.lib.pdmpc_sample_inputs(self.h, n, _ptr(path_id, _p_i32), _ptr(x, _p_f64), _ptr(y, _p_f64),
                                                 _ptr(speed, _p_f64), float(dt_seconds), C.byref(oc)))
        tot = int(o["lane_ptr"][-1])
        o["lane_x"], o["lane_y"] = o["lane_x"][:tot], o["lane_y"][:tot]
        return o

    def pipeline_timeline(self):
        """Per chunk of the last pipelined plan_batch call: (host_ms, in_ms, done_ms) arrays (pdmpc_get_pipeline_timeline)."""
        cap = 32
        a, b, c = np.zeros(cap), np.zeros(cap), np.zeros(cap)
        n = C.c_int32()
        self._check(self.lib.pdmpc_get_pipeline_timeline(self.h, cap, _ptr(a, _p_f64), _ptr(b, _p_f64), _ptr(c, _p_f64), C.byref(n)))
        return a[: n.value], b[: n.value], c[: n.value]

    def upload_reachable_sets(self, sets):
        """mpa.local_reachable_sets_conv as sets[trim][step] = closed (2, m) polygon (scenario.local_reachable_sets_conv)
        for pdmpc_assemble_obstacles (pdmpc_upload_reachable_sets)."""
        nT, Hp = len(sets), len(sets[0])
        ptr = np.zeros(nT * Hp + 1, dtype=np.int32)
        xs, ys = [], []
        for i in range(nT):
            for t in range(Hp):
                a = np.asarray(sets[i][t], dtype=np.float64)
                ptr[i * Hp + t + 1] = ptr[i * Hp + t] + a.shape[1]
                xs.append(a[0]); ys.append(a[1])
        x, y = np.ascontiguousarray(np.concatenate(xs)), np.ascontiguousarray(np.concatenate(ys))
        d = ReachDescC(n_trims=nT, Hp=Hp, ptr=_ptr(ptr, _p_i32), x=_ptr(x, _p_f64), y=_ptr(y, _p_f64))
        self._check(self.lib.pdmpc_upload_reachable_sets(self.h, C.byref(d)))

    def assemble_obstacles(self, x, y, yaw, speed, trim, successors, parallel, half_length: float, half_width: float,
                           poly_capacity: int = 0, vert_capacity: int = 0) -> dict:
        """Static obstacles (standing successors) and dynamic obstacles (reachable sets of parallel predecessors) of every
        row as the obstacle CSR of a SearchBatch (pdmpc_assemble_obstacles): slot_ptr [n(Hp+1)+1], poly_ptr, vert_x,
        vert_y.  successors / parallel: per row a sequence of row indices."""
        x, y, yaw, speed = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, yaw, speed))
        trim = np.ascontiguousarray(trim, dtype=np.int32)
        n, Hp = int(x.size), int(self.lib.pdmpc_get_hp(self.h))

        def csr(rows):
            ptr = np.zeros(n + 1, dtype=np.int32)
            for i in range(n):
                ptr[i + 1] = ptr[i] + len(rows[i])
            idx = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.int32) for r in rows] + [np.zeros(0, np.int32)]),
                                       dtype=np.int32)
            return ptr, idx

        sp, si = csr(successors)
        pp, pi = csr(parallel)
        pc = int(poly_capacity) or max(1, si.size + Hp * pi.size)
        vc = int(vert_capacity) or max(1, 5 * si.size + 256 * Hp * pi.size)
        o = {"slot_ptr": np.zeros(n * (Hp + 1) + 1, dtype=np.int32), "poly_ptr": np.zeros(pc + 1, dtype=np.int32),
             "vert_x": np.zeros(vc), "vert_y": np.zeros(vc)}
        ci = CouplingInC(n=n, x=_ptr(x, _p_f64), y=_ptr(y, _p_f64), yaw=_ptr(yaw, _p_f64), speed=_ptr(speed, _p_f64),
                         trim=_ptr(trim, _p_i32), succ_ptr=_ptr(sp, _p_i32), succ_idx=_ptr(si, _p_i32),
                         par_ptr=_ptr(pp, _p_i32), par_idx=_ptr(pi, _p_i32),
                         half_length=float(half_length), half_width=float(half_width))
        oc = ObstaclesOutC(slot_ptr=_ptr(o["slot_ptr"], _p_i32), poly_ptr=_ptr(o["poly_ptr"], _p_i32),
                           vert_x=_ptr(o["vert_x"], _p_f64), vert_y=_ptr(o["vert_y"], _p_f64), poly_capacity=pc, vert_capacity=vc)
        self._check(self.lib.pdmpc_assemble_obstacles(self.h, C.byref(ci), C.byref(oc)))
        o["poly_ptr"] = o["poly_ptr"][: oc.n_polys + 1]
        o["vert_x"], o["vert_y"] = o["vert_x"][: oc.n_verts], o["vert_y"][: oc.n_verts]
        return o

    def set_escalation(self, pops: int, short_list_max: int = -1):
        """Shapes 2, 3: searches beyond `pops` pops go to the CTA shape (pdmpc_set_escalation; 0 = never)."""
        self._check(self.lib.pdmpc_set_escalation(self.h, int(pops), int(short_list_max)))

    def set_tile_points(self, points: int = 0):
        """Shapes 2, 3 test knob (pdmpc_set_tile_points); results do not depend on it."""
        self._check(self.lib.pdmpc_set_tile_points(self.h, int(points)))

    def trace(self, search: int, cap: int = 1 << 20) -> np.ndarray:
        """Node ids popped by staged search `search`, in order (pdmpc_trace_staged)."""
        ids = np.zeros(cap, dtype=np.int64)
        n = C.c_int64()
        self._check(self.lib.pdmpc_trace_staged(self.h, int(search), ids.ctypes.data_as(C.POINTER(C.c_int64)),
                                                cap, C.byref(n)))
        return ids[: min(n.value, cap)].copy()

    def upload_mpa(self, mpa: MotionPrimitiveAutomaton):
        d, keep = mpa_desc(mpa)
        self._check(self.lib.pdmpc_upload_mpa(self.h, C.byref(d)))
        self._mpa_keep = keep
        self._mpa = mpa

    def _check_hp(self, b: SearchBatch):
        """pdmpc_batch_in carries no Hp: the library indexes the per-step arrays with the MPA's (pdmpc_get_hp)."""
        hp = int(self.lib.pdmpc_get_hp(self.h))
        if hp and b.Hp != hp:
            raise PdmpcError(PDMPC_ERR_BAD_INPUT, f"batch has Hp {b.Hp}, the uploaded MPA has Hp {hp}")

    def plan_batch(self, b: SearchBatch, raise_on_search_error: bool = True) -> BatchResult:
        self._check_hp(b)
        r = BatchResult.empty(b.n, b.Hp)
        bi, bo = batch_in(b), batch_out(r)
        self._check(self.lib.pdmpc_plan_batch(self.h, C.byref(bi), C.byref(bo)))
        if raise_on_search_error and b.n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r

    def plan_timestep(self, b: SearchBatch, deps, raise_on_search_error: bool = True) -> BatchResult:
        """All searches of one (or many) time steps in one dependency-ordered launch
        (pdmpc_plan_timestep): PrioritizedController.plan's hand-over of predecessors' areas on the device."""
        return self._timestep(b, deps, None, raise_on_search_error)

    def mcts_plan_timestep(self, b: SearchBatch, deps, seeds, n_expansions_max: int = 250,
                           raise_on_search_error: bool = True) -> BatchResult:
        """plan_timestep with MonteCarloTreeSearch as the optimizer (pdmpc_mcts_plan_timestep); seeds[i] = time_step +
        vehicle_index of row i."""
        return self._timestep(b, deps, (seeds, n_expansions_max), raise_on_search_error)

    def _timestep(self, b: SearchBatch, deps, mcts, raise_on_search_error: bool) -> BatchResult:
        self._check_hp(b)
        r = BatchResult.empty(b.n, b.Hp)
        bi, bo = batch_in(b), batch_out(r)
        pidx = deps.pred_idx if deps.pred_idx.size else np.zeros(1, dtype=np.int32)
        d = TimestepDepsC(pred_ptr=_ptr(deps.pred_ptr, _p_i32), pred_idx=_ptr(pidx, _p_i32),
                          fb_npts=_ptr(deps.fb_npts, _p_i32), fb_x=_ptr(deps.fb_x, _p_f64), fb_y=_ptr(deps.fb_y, _p_f64))
        if mcts is None:
            self._check(self.lib.pdmpc_plan_timestep(self.h, C.byref(bi), C.byref(d), C.byref(bo)))
        else:
            prm, keep = mcts_params(mcts[0], mcts[1], b.n)
            self._check(self.lib.pdmpc_mcts_plan_timestep(self.h, C.byref(bi), C.byref(d), C.byref(prm), C.byref(bo)))
            del keep
        if raise_on_search_error and b.n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r

    def closed_loop_reset(self, n_slots: int, half_length: float, half_width: float):
        """Forget the previous plans of all vehicle slots (pdmpc_closed_loop_reset)."""
        self._check(self.lib.pdmpc_closed_loop_reset(self.h, int(n_slots), float(half_length), float(half_width)))

    def plan_timestep_closed_loop(self, b: SearchBatch, deps, slot, standstill, raise_on_search_error: bool = True) -> BatchResult:
        """pdmpc_plan_timestep_closed_loop: like plan_timestep, but the fallback plans of exhausted vehicles are built on
        the device from the previous time step's plans kept there; exhausted rows return their fallback plan."""
        return self._closed_loop(b, deps, slot, standstill, None, raise_on_search_error)

    def mcts_plan_timestep_closed_loop(self, b: SearchBatch, deps, slot, standstill, seeds, n_expansions_max: int = 250,
                                       raise_on_search_error: bool = True) -> BatchResult:
        """plan_timestep_closed_loop with MonteCarloTreeSearch as the optimizer (pdmpc_mcts_plan_timestep_closed_loop)."""
        return self._closed_loop(b, deps, slot, standstill, (seeds, n_expansions_max), raise_on_search_error)

    def _closed_loop(self, b: SearchBatch, deps, slot, standstill, mcts, raise_on_search_error: bool) -> BatchResult:
        self._check_hp(b)
        r = BatchResult.empty(b.n, b.Hp)
        bi, bo = batch_in(b), batch_out(r)
        pidx = deps.pred_idx if deps.pred_idx.size else np.zeros(1, dtype=np.int32)
        d = TimestepDepsC(pred_ptr=_ptr(deps.pred_ptr, _p_i32), pred_idx=_ptr(pidx, _p_i32), fb_npts=None, fb_x=None, fb_y=None)
        slot = np.ascontiguousarray(slot, dtype=np.int32)
        still = np.ascontiguousarray(standstill, dtype=np.uint8)
        if mcts is None:
            self._check(self.lib.pdmpc_plan_timestep_closed_loop(self.h, C.byref(bi), C.byref(d), _ptr(slot, _p_i32),
                                                                 _ptr(still, C.POINTER(C.c_uint8)), C.byref(bo)))
        else:
            prm, keep = mcts_params(mcts[0], mcts[1], b.n)
            self._check(self.lib.pdmpc_mcts_plan_timestep_closed_loop(self.h, C.byref(bi), C.byref(d), _ptr(slot, _p_i32),
                                                                      _ptr(still, C.POINTER(C.c_uint8)), C.byref(prm),
                                                                      C.byref(bo)))
            del keep
        if raise_on_search_error and b.n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r

    def plan_timestep_from_states(self, path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot,
                                  half_length: float, half_width: float, dt_seconds: float, checker: int,
                                  raise_on_search_error: bool = True) -> BatchResult:
        """One whole time step from the measured states (pdmpc_plan_timestep_from_states): inputs, obstacle assembly,
        dependency-ordered searches and fallback plans chained on the device.  successors / parallel / predecessors:
        per row a sequence of row indices.  Exhausted rows return their fallback plan."""
        return self._from_states(path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot, half_length,
                                 half_width, dt_seconds, checker, None, raise_on_search_error)

    def mcts_plan_timestep_from_states(self, path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot,
                                       half_length: float, half_width: float, dt_seconds: float, checker: int, seeds,
                                       n_expansions_max: int = 250, raise_on_search_error: bool = True) -> BatchResult:
        """plan_timestep_from_states with MonteCarloTreeSearch as the optimizer (pdmpc_mcts_plan_timestep_from_states)."""
        return self._from_states(path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot, half_length,
                                 half_width, dt_seconds, checker, (seeds, n_expansions_max), raise_on_search_error)

    def _from_states(self, path_id, x, y, yaw, speed, trim, successors, parallel, predecessors, slot, half_length,
                     half_width, dt_seconds, checker, mcts, raise_on_search_error: bool) -> BatchResult:
        path_id, trim, slot = (np.ascontiguousarray(a, dtype=np.int32) for a in (path_id, trim, slot))
        x, y, yaw, speed = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, yaw, speed))
        n, Hp = int(x.size), int(self.lib.pdmpc_get_hp(self.h))

        def csr(rows):
            ptr = np.zeros(n + 1, dtype=np.int32)
            for i in range(n):
                ptr[i + 1] = ptr[i] + len(rows[i])
            idx = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.int32) for r in rows] + [np.zeros(1, np.int32)]),
                                       dtype=np.int32)
            return ptr, idx

        (sp, si), (pp, pi), (dp, di) = csr(successors), csr(parallel), csr(predecessors)
        r = BatchResult.empty(n, Hp)
        bo = batch_out(r)
        st = TimestepStatesC(n=n, path_id=_ptr(path_id, _p_i32), x=_ptr(x, _p_f64), y=_ptr(y, _p_f64), yaw=_ptr(yaw, _p_f64),
                             speed=_ptr(speed, _p_f64), trim=_ptr(trim, _p_i32), succ_ptr=_ptr(sp, _p_i32),
                             succ_idx=_ptr(si, _p_i32), par_ptr=_ptr(pp, _p_i32), par_idx=_ptr(pi, _p_i32),
                             pred_ptr=_ptr(dp, _p_i32), pred_idx=_ptr(di, _p_i32), slot=_ptr(slot, _p_i32),
                             half_length=float(half_length), half_width=float(half_width), dt_seconds=float(dt_seconds),
                             checker=int(checker))
        if mcts is None:
            self._check(self.lib.pdmpc_plan_timestep_from_states(self.h, C.byref(st), C.byref(bo)))
        else:
            prm, keep = mcts_params(mcts[0], mcts[1], n)
            self._check(self.lib.pdmpc_mcts_plan_timestep_from_states(self.h, C.byref(st), C.byref(prm), C.byref(bo)))
            del keep
        if raise_on_search_error and n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r

    def _couple_args(self, n: int, priority, max_num_CLs: int, scenario_ptr, idx_capacity: int):
        """(params, out struct, relations dict, keepalive) of pdmpc_couple / pdmpc_plan_timestep_from_states_coupled."""
        sp = np.ascontiguousarray([0, n] if scenario_ptr is None else scenario_ptr, dtype=np.int32)
        if isinstance(priority, str):
            priority = {"constant": PRIORITY_CONSTANT, "coloring": PRIORITY_COLORING}[priority]
        sizes = np.diff(sp).astype(np.int64)
        cap = int(idx_capacity) or max(1, int((sizes * (sizes - 1) // 2).sum()))
        rel = {k: np.zeros(n + 1, dtype=np.int32) for k in ("succ_ptr", "par_ptr", "pred_ptr")}
        rel.update({k: np.zeros(cap, dtype=np.int32) for k in ("succ_idx", "par_idx", "pred_idx")})
        rel["level"] = np.zeros(max(n, 1), dtype=np.int32)
        area = np.zeros(max(1, int((sizes * sizes).sum())))
        prm = CoupleParamsC(n_scenarios=int(sp.size - 1), scenario_ptr=_ptr(sp, _p_i32), prioritizer=int(priority),
                            max_num_CLs=int(max_num_CLs))
        oc = CoupleOutC(idx_capacity=cap, overlap_area=_ptr(area, _p_f64), **{k: _ptr(v, _p_i32) for k, v in rel.items()})
        return prm, oc, rel, (sp, sizes, area)

    @staticmethod
    def _relations(n: int, rel: dict, keep) -> dict:
        _sp, sizes, area = keep
        for k in ("succ", "par", "pred"):
            rel[f"{k}_idx"] = rel[f"{k}_idx"][: int(rel[f"{k}_ptr"][-1])]
        rel["level"] = rel["level"][:n]
        ends = np.cumsum(sizes * sizes)
        rel["overlap_area"] = [area[e - s * s:e].reshape(s, s) for s, e in zip(sizes, ends)]
        return rel

    def couple(self, x, y, yaw, trim, scenario_ptr=None, priority="coloring", max_num_CLs: int = 99,
               idx_capacity: int = 0) -> dict:
        """Coupling (reachable-set overlap > 1e-3), priorities, the level cut and computation levels of every scenario
        (pdmpc_couple).  scenario_ptr: rows of scenario s are [ptr[s], ptr[s+1]) (default: one scenario).  Returns
        succ_ptr / succ_idx, par_ptr / par_idx, pred_ptr / pred_idx (the relations of plan_timestep_from_states, global
        rows), level [n] (1-based) and overlap_area (one [n_s, n_s] matrix per scenario)."""
        x, y, yaw = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, yaw))
        trim = np.ascontiguousarray(trim, dtype=np.int32)
        n = int(x.size)
        prm, oc, rel, keep = self._couple_args(n, priority, max_num_CLs, scenario_ptr, idx_capacity)
        self._check(self.lib.pdmpc_couple(self.h, n, _ptr(x, _p_f64), _ptr(y, _p_f64), _ptr(yaw, _p_f64), _ptr(trim, _p_i32),
                                          C.byref(prm), C.byref(oc)))
        return self._relations(n, rel, keep)

    def plan_timestep_from_states_coupled(self, path_id, x, y, yaw, speed, trim, slot, half_length: float,
                                          half_width: float, dt_seconds: float, checker: int, priority="coloring",
                                          max_num_CLs: int = 99, scenario_ptr=None, idx_capacity: int = 0,
                                          raise_on_search_error: bool = True):
        """plan_timestep_from_states with the relations decided on the device (pdmpc_plan_timestep_from_states_coupled):
        returns (BatchResult, relations as Planner.couple returns them)."""
        path_id, trim, slot = (np.ascontiguousarray(a, dtype=np.int32) for a in (path_id, trim, slot))
        x, y, yaw, speed = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, yaw, speed))
        n, Hp = int(x.size), int(self.lib.pdmpc_get_hp(self.h))
        prm, oc, rel, keep = self._couple_args(n, priority, max_num_CLs, scenario_ptr, idx_capacity)
        r = BatchResult.empty(n, Hp)
        bo = batch_out(r)
        st = TimestepStatesC(n=n, path_id=_ptr(path_id, _p_i32), x=_ptr(x, _p_f64), y=_ptr(y, _p_f64), yaw=_ptr(yaw, _p_f64),
                             speed=_ptr(speed, _p_f64), trim=_ptr(trim, _p_i32), slot=_ptr(slot, _p_i32),
                             half_length=float(half_length), half_width=float(half_width), dt_seconds=float(dt_seconds),
                             checker=int(checker))
        self._check(self.lib.pdmpc_plan_timestep_from_states_coupled(self.h, C.byref(st), C.byref(prm), C.byref(oc), C.byref(bo)))
        if raise_on_search_error and n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r, self._relations(n, rel, keep)

    def plan_timestep_explorative(self, path_id, x, y, yaw, speed, trim, slot, successors, level, permutations,
                                  half_length: float, half_width: float, dt_seconds: float, checker: int, scenario_ptr=None,
                                  raise_on_search_error: bool = True):
        """Simultaneous prioritizations of every scenario in one call (pdmpc_plan_timestep_explorative): every permutation
        planned from the measured states, the cheapest per weakly connected sub-graph chosen and committed to the slots.
        successors: per base row the coupled rows of lower priority (global rows); level [n] 1-based; permutations: one
        [P_s, L_s] array per scenario.  Returns (BatchResult of all P_s * n_s rows per scenario, dict with belonging [n],
        chosen [n], applied_row [n], row_cost [rows] and solution_cost = one [P_s, G_s] array per scenario)."""
        path_id, trim, slot, level = (np.ascontiguousarray(a, dtype=np.int32) for a in (path_id, trim, slot, level))
        x, y, yaw, speed = (np.ascontiguousarray(a, dtype=np.float64) for a in (x, y, yaw, speed))
        n, Hp = int(x.size), int(self.lib.pdmpc_get_hp(self.h))
        sp = np.ascontiguousarray([0, n] if scenario_ptr is None else scenario_ptr, dtype=np.int32)
        perms = [np.atleast_2d(np.asarray(p, dtype=np.int32)) for p in permutations]
        S = int(sp.size - 1)
        if len(perms) != S:
            raise PdmpcError(PDMPC_ERR_BAD_INPUT, f"{len(perms)} permutation arrays for {S} scenarios")
        pp = np.concatenate([[0], np.cumsum([p.shape[0] for p in perms])]).astype(np.int32)
        pv = np.concatenate([[0], np.cumsum([p.size for p in perms])]).astype(np.int32)
        pflat = np.ascontiguousarray(np.concatenate([p.reshape(-1) for p in perms] + [np.zeros(1, np.int32)]), dtype=np.int32)
        sizes = np.diff(sp).astype(np.int64)
        rows = int((np.diff(pp).astype(np.int64) * sizes).sum())
        succ_ptr = np.zeros(n + 1, dtype=np.int32)
        for i in range(n):
            succ_ptr[i + 1] = succ_ptr[i] + len(successors[i])
        succ_idx = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.int32) for r in successors] + [np.zeros(1, np.int32)]),
                                        dtype=np.int32)
        r = BatchResult.empty(rows, Hp)
        bo = batch_out(r)
        eo = {"belonging": np.zeros(max(n, 1), dtype=np.int32), "chosen": np.zeros(max(n, 1), dtype=np.int32),
              "applied_row": np.zeros(max(n, 1), dtype=np.int32), "row_cost": np.zeros(max(rows, 1)),
              "solution_cost": np.zeros(max(rows, 1))}
        oc = ExplorativeOutC(**{k: _ptr(v, _p_i32 if v.dtype == np.int32 else _p_f64) for k, v in eo.items()})
        ex = ExplorativeInC(n_scenarios=S, scenario_ptr=_ptr(sp, _p_i32), level=_ptr(level, _p_i32), perm_ptr=_ptr(pp, _p_i32),
                            perm_val_ptr=_ptr(pv, _p_i32), perm=_ptr(pflat, _p_i32))
        st = TimestepStatesC(n=n, path_id=_ptr(path_id, _p_i32), x=_ptr(x, _p_f64), y=_ptr(y, _p_f64), yaw=_ptr(yaw, _p_f64),
                             speed=_ptr(speed, _p_f64), trim=_ptr(trim, _p_i32), succ_ptr=_ptr(succ_ptr, _p_i32),
                             succ_idx=_ptr(succ_idx, _p_i32), slot=_ptr(slot, _p_i32),
                             half_length=float(half_length), half_width=float(half_width), dt_seconds=float(dt_seconds),
                             checker=int(checker))
        self._check(self.lib.pdmpc_plan_timestep_explorative(self.h, C.byref(st), C.byref(ex), C.byref(bo), C.byref(oc)))
        if raise_on_search_error and rows and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"row {bad} failed")
        for k in ("belonging", "chosen", "applied_row"):
            eo[k] = eo[k][:n]
        eo["row_cost"] = eo["row_cost"][:rows]
        sol, blocks, r0 = eo["solution_cost"], [], 0
        for s in range(S):
            ns, P = int(sizes[s]), int(pp[s + 1] - pp[s])
            G = int(eo["belonging"][sp[s]:sp[s + 1]].max()) if ns else 0
            blocks.append(sol[r0:r0 + P * ns].reshape(P, ns)[:, :G].copy())
            r0 += P * ns
        eo["solution_cost"] = blocks
        return r, eo

    def joint_plan_batch(self, b: SearchBatch, n_vehicles: int, raise_on_search_error: bool = True) -> BatchResult:
        """Centralized (joint) searches: rows of `b` are searches x n_vehicles (pdmpc_joint_plan_batch)."""
        self._check_hp(b)
        r = BatchResult.empty(b.n, b.Hp)
        bi, bo = batch_in(b), batch_out(r)
        self._check(self.lib.pdmpc_joint_plan_batch(self.h, C.byref(bi), int(n_vehicles), C.byref(bo)))
        if raise_on_search_error and b.n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"row {bad} failed")
        return r

    def mcts_plan_batch(self, b: SearchBatch, seeds, n_expansions_max: int = 250,
                        raise_on_search_error: bool = True) -> BatchResult:
        """MonteCarloTreeSearch.run_optimizer for every search (pdmpc_mcts_plan_batch)."""
        self._check_hp(b)
        r = BatchResult.empty(b.n, b.Hp)
        bi, bo = batch_in(b), batch_out(r)
        prm, keep = mcts_params(seeds, n_expansions_max, b.n)
        self._check(self.lib.pdmpc_mcts_plan_batch(self.h, C.byref(bi), C.byref(prm), C.byref(bo)))
        del keep
        if raise_on_search_error and b.n and int(r.status.max()) != PDMPC_OK:
            bad = int(np.flatnonzero(r.status != PDMPC_OK)[0])
            raise PdmpcError(int(r.status[bad]), f"search {bad} failed")
        return r

    def mcts_run_staged(self, seeds, n_expansions_max: int = 250):
        prm, keep = mcts_params(seeds, n_expansions_max, self._staged_n)
        self._check(self.lib.pdmpc_mcts_run_staged(self.h, C.byref(prm)))
        del keep

    def stage(self, b: SearchBatch):
        self._check_hp(b)
        bi = batch_in(b)
        self._check(self.lib.pdmpc_stage_batch(self.h, C.byref(bi)))
        self._staged_n, self._staged_Hp = b.n, b.Hp

    def run_staged(self):
        self._check(self.lib.pdmpc_run_staged(self.h))

    def sync(self):
        self._check(self.lib.pdmpc_sync(self.h))

    def fetch(self) -> BatchResult:
        r = BatchResult.empty(self._staged_n, self._staged_Hp)
        bo = batch_out(r)
        self._check(self.lib.pdmpc_fetch_staged(self.h, C.byref(bo)))
        return r

    def stats(self) -> Stats:
        s = Stats()
        self._check(self.lib.pdmpc_get_stats(self.h, C.byref(s)))
        return s

    def stream(self) -> int:
        return int(self.lib.pdmpc_stream(self.h) or 0)
