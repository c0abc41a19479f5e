"""CPU side of the sampled optimizer's time steps: the level-by-level specification driven by the C oracle against
the same procedure driven by the matrix-form restatement (matlab_literal.do_mcts, numpy's own MT19937); the new C
entry points and their ctypes prototypes; the kernel instances' resources; the MEX command and the MATLAB helper."""
import ctypes as C
import os

import numpy as np

from oracle import matlab_literal as ml
from oracle import oracle_py
from pdmpc_b200 import capi, scenario
from pdmpc_b200.mpa import get_mpa
from pdmpc_b200.records import BatchResult

from test_kernel_resources import resource_usage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NMAX = 250


def literal_plan(mpa, n_expansions_max):
    """plan_fn(batch, seeds) of the matrix-form restatement: one do_mcts per row."""
    def plan(batch, seeds):
        r = BatchResult.empty(batch.n, batch.Hp)
        for i, it in enumerate(batch.to_iters()):
            info = ml.do_mcts(it, mpa, batch.checker, int(seeds[i]), n_expansions_max,
                              use_reference_pq=oracle_py.have_reference_pq())
            r.status[i] = 0
            r.is_exhausted[i] = int(info.is_exhausted)
            r.n_expanded[i] = info.n_expanded
            r.n_pops[i] = info.n_traversals
            if not info.is_exhausted:
                r.trims[i, 1:] = info.predicted_trims
                r.y_predicted[i] = info.y_predicted
                for k, shp in enumerate(info.shapes):
                    r.shape_npts[i, k] = shp.shape[1]
                    r.shape_x[i, k, :shp.shape[1]] = shp[0]
                    r.shape_y[i, k, :shp.shape[1]] = shp[1]
        return r
    return plan


def test_level_by_level_spec_oracle_equals_matrix_form():
    mpa = get_mpa("triple_speed", non_convex=True)
    plan = lambda b, s: oracle_py.mcts_plan_batch(mpa, b, s, NMAX, 4)
    runner = scenario.ScenarioRunner(scenario.commonroad_scenario(mpa, 20, seed=2), None, n_expansions_max=NMAX,
                                     timestep_fn=lambda b, d, s: scenario.plan_timestep_by_levels(plan, b, d, seeds=s))
    runner.run(3)
    preds = 0
    for k, batch, deps, got in runner.timestep_records:
        seeds = scenario.mcts_seeds(k, batch.n)
        lit = scenario.plan_timestep_by_levels(literal_plan(mpa, NMAX), batch, deps, seeds=seeds)
        ok = got.is_exhausted == 0
        assert np.array_equal(lit.is_exhausted, got.is_exhausted) and (got.status == 0).all()
        assert np.array_equal(lit.n_expanded, got.n_expanded) and np.array_equal(lit.n_pops, got.n_pops)
        assert np.array_equal(lit.trims[ok, 1:], got.trims[ok, 1:])
        assert np.array_equal(lit.y_predicted[ok].view(np.uint64), got.y_predicted[ok].view(np.uint64))
        assert np.array_equal(lit.shape_npts[ok], got.shape_npts[ok])
        assert np.array_equal(lit.shape_x[ok].view(np.uint64), got.shape_x[ok].view(np.uint64))
        preds += int(deps.pred_idx.size)
    assert preds > 0


def test_seeds_follow_time_step_and_vehicle_index():
    assert scenario.mcts_seeds(1, 3).tolist() == [2, 3, 4]
    assert scenario.mcts_seeds(7, 20)[-1] == 27 and scenario.mcts_seeds(7, 20).dtype == np.uint32


def test_new_symbols_are_exported_with_their_prototypes(built):
    lib = capi.load_library()
    H = C.c_void_p
    want = {
        "pdmpc_mcts_plan_timestep": [H, C.POINTER(capi.BatchIn), C.POINTER(capi.TimestepDepsC), C.POINTER(capi.MctsParams),
                                     C.POINTER(capi.BatchOut)],
        "pdmpc_mcts_plan_timestep_closed_loop": [H, C.POINTER(capi.BatchIn), C.POINTER(capi.TimestepDepsC), capi._p_i32,
                                                 C.POINTER(C.c_uint8), C.POINTER(capi.MctsParams), C.POINTER(capi.BatchOut)],
        "pdmpc_mcts_plan_timestep_from_states": [H, C.POINTER(capi.TimestepStatesC), C.POINTER(capi.MctsParams),
                                                 C.POINTER(capi.BatchOut)],
    }
    for name, args in want.items():
        assert name in capi.EXPORTED_SYMBOLS
        f = getattr(lib, name)
        assert f.restype is C.c_int and f.argtypes == args, name
        assert f(None, None, None, None, *([None] * (len(args) - 4))) == capi.PDMPC_ERR_BAD_INPUT
    hdr = open(os.path.join(ROOT, "include", "pdmpc_b200.h")).read()
    assert "#define PDMPC_ABI_VERSION 2" in hdr and all(n + "(" in hdr for n in want)


def ptxas_report(tmp_path):
    """-Xptxas -v of both mcts_kernel instances, compiled with the library's flags: {instance: {stack, spill_st,
    spill_ld, regs}}."""
    import re
    import subprocess

    import __graft_entry__ as entry
    src = tmp_path / "mcts_instances.cu"
    src.write_text('#include "pdmpc_mcts.cuh"\n'
                   "template __global__ void pdmpc::mcts_kernel<false>(pdmpc::MpaDev, pdmpc::BatchDev, pdmpc::OutDev, "
                   "pdmpc::MctsDev, unsigned *, pdmpc::DepsDev);\n"
                   "template __global__ void pdmpc::mcts_kernel<true>(pdmpc::MpaDev, pdmpc::BatchDev, pdmpc::OutDev, "
                   "pdmpc::MctsDev, unsigned *, pdmpc::DepsDev);\n")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = [f for f in entry.NVCC_FLAGS if f not in ("-Xcompiler", "-fPIC", "-shared")]
    out = subprocess.run([nvcc] + flags + ["-I", entry.CSRC, "-cubin", "-Xptxas", "-v", "-o", str(tmp_path / "m.cubin"),
                          str(src)], check=True, capture_output=True, text=True).stderr
    rep, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function properties for _ZN5pdmpc11mcts_kernelILb([01])E", line)
        if m:
            name = "true" if m.group(1) == "1" else "false"
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if name and m:
            rep[name] = dict(zip(("stack", "spill_st", "spill_ld"), map(int, m.groups())))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if name and m:
            rep[name]["regs"] = int(m.group(1))
            name = None
    return rep


def test_sampled_kernel_instances_resources(built, tmp_path):
    """ptxas on both instances (DESIGN.md §4.14).  mcts_kernel<false> is the parent's kernel unchanged: 128 registers, an
    80-byte frame, 104 / 84 bytes of spill stores / loads.  mcts_kernel<true> stays within what it was measured at: 168
    registers, a 48-byte frame (32 bytes of it lanelet_side_sat's indexed two-point arrays) and 20 / 68 bytes of spill
    stores / loads of per-search values; it has no local memory beyond that frame."""
    rep = ptxas_report(tmp_path)
    assert rep["false"] == {"stack": 80, "spill_st": 104, "spill_ld": 84, "regs": 128}, rep
    t = rep["true"]
    assert t["stack"] <= 48 and t["spill_st"] <= 20 and t["spill_ld"] <= 68 and t["regs"] <= 168, rep
    u = resource_usage()
    dep = [r for n, r in u.items() if n.startswith("_ZN5pdmpc11mcts_kernelILb1E")]
    assert len(dep) == 1 and dep[0]["LOCAL"] == 0 and dep[0]["STACK"] == t["stack"], dep


def test_mex_source_and_matlab_helper_carry_the_command():
    mex = open(os.path.join(ROOT, "p-dmpc_b200", "matlab", "pdmpc_b200_mex.cpp")).read()
    assert "PLAN_TIMESTEP_SAMPLED = 13" in mex and "pdmpc_mcts_plan_timestep(h, &in, &deps, &prm, &out)" in mex
    m = open(os.path.join(ROOT, "p-dmpc_b200", "matlab", "plan_timestep_cuda.m")).read()
    assert "PLAN_TIMESTEP_SAMPLED = 13" in m and "isa(hlcs(1).optimizer, 'MonteCarloTreeSearchCuda')" in m
    assert "time_step + (1:N)" in m and "tree.h = -1 * ones(1, Hp + 1)" in m
