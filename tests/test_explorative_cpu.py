"""CPU suite for the simultaneous prioritizations on the device (DESIGN.md §4.13): the summation order the choice kernel
states equals numpy's, an explicit-loop restatement of the choice equals sharding.solution_costs, permuted_coupling is
the host's swap loop and gives acyclic relations, the ctypes mirrors have the C layout, and the choice kernels use no
stack or local memory."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from pdmpc_b200 import scenario, sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pdmpc_b200.h")


def spec_sum(e):
    """The order of explorative_row_cost_kernel: left to right from 0.0 below 8 values; else 8 accumulators over the
    complete blocks of 8, ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)), then the rest left to right."""
    if len(e) < 8:
        s = 0.0
        for v in e:
            s += v
        return s
    r = [float(v) for v in e[:8]]
    m = 8
    while m + 8 <= len(e):
        for j in range(8):
            r[j] += e[m + j]
        m += 8
    s = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
    for v in e[m:]:
        s += v
    return s


@pytest.mark.parametrize("Hp", [3, 6, 10])
def test_fallback_cost_summation_order_equals_numpy(Hp):
    rng = np.random.default_rng(Hp)
    for _ in range(4000):
        ref = rng.normal(size=(Hp, 2)) * 10.0 ** rng.uniform(-6, 6, size=(Hp, 2))
        traj = rng.normal(size=(Hp, 3)) * 10.0 ** rng.uniform(-6, 6, size=(Hp, 3))
        want = float(np.sum((ref - traj[:, :2]) ** 2))
        d = ref - traj[:, :2]
        e = [float(v) * float(v) for v in d.reshape(-1)]
        assert np.float64(spec_sum(e)).view(np.uint64) == np.float64(want).view(np.uint64)


def choice_restated(cost, belonging):
    """explorative_choose_kernel as plain loops: per (p, g) a sum from 0.0 in vehicle order, sign(y) * floor(|y| + 0.5)
    / 1e8 with y = x * 1e8, first minimum over p."""
    P, n = cost.shape
    G = int(belonging.max())
    sol = np.zeros((P, G))
    for p in range(P):
        for g in range(1, G + 1):
            s = 0.0
            for v in range(n):
                if belonging[v] == g:
                    s = s + float(cost[p, v])
            y = s * 1e8
            sg = 1.0 if y > 0 else (-1.0 if y < 0 else 0.0)
            sol[p, g - 1] = sg * np.floor(abs(y) + 0.5) / 1e8
    chosen = np.zeros(G, dtype=np.int64)
    for g in range(G):
        best = 0
        for p in range(1, P):
            if sol[p, g] < sol[best, g]:
                best = p
        chosen[g] = best
    return chosen, sol


def test_choice_restatement_equals_solution_costs():
    rng = np.random.default_rng(5)
    ties = 0
    for t in range(400):
        n, P = int(rng.integers(1, 25)), int(rng.integers(1, 9))
        belonging = scenario.weak_components(rng.random((n, n)) < 0.08)
        cost = rng.random((P, n)) * 10.0 ** rng.uniform(-3, 3)
        if t % 3 == 0 and P > 1:   # permutations equal after rounding: the first one must win
            cost[P - 1] = cost[0] + rng.random(n) * 1e-12
            ties += 1
        want_c, want_s = sharding.solution_costs(cost, belonging)
        got_c, got_s = choice_restated(cost, belonging)
        assert np.array_equal(got_s.view(np.uint64), want_s.view(np.uint64))
        assert np.array_equal(got_c, want_c)
    assert ties > 50


def test_permuted_coupling_is_the_host_loop_and_acyclic():
    rng = np.random.default_rng(11)
    for _ in range(200):
        n = int(rng.integers(2, 20))
        A = np.triu(rng.random((n, n)) < 0.3, 1)
        A = (A | A.T).astype(np.int64)
        D = scenario.coloring_priorities(A).astype(bool)
        levels = scenario.kahn(D.astype(np.int64))
        for perm in scenario.computation_level_permutations(int(levels.max()), int(rng.integers(1, 100))):
            lev_p = perm[levels - 1]
            want = D.copy()
            for i, j in zip(*np.nonzero(D)):
                if lev_p[i] > lev_p[j]:
                    want[i, j], want[j, i] = False, True
            got = scenario.permuted_coupling(D, levels, perm)
            assert np.array_equal(got, want)
            assert np.array_equal(got | got.T, D | D.T) and not (got & got.T).any()
            scenario.kahn(got.astype(np.int64))            # raises / loops on a cycle: every edge climbs lev_p
            assert all(lev_p[i] < lev_p[j] for i, j in zip(*np.nonzero(got)))


def test_explorative_structs_match_the_c_layout(tmp_path, built):
    from pdmpc_b200 import capi
    structs = {"pdmpc_explorative_in": capi.ExplorativeInC, "pdmpc_explorative_out": capi.ExplorativeOutC}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
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
    assert "pdmpc_plan_timestep_explorative" in capi.EXPORTED_SYMBOLS


def test_choice_kernels_use_no_stack_or_local_memory(built):
    from test_kernel_resources import resource_usage
    usage = resource_usage()
    names = [k for k in usage if "explorative_row_cost_kernel" in k or "explorative_choose_kernel" in k]
    assert len(names) == 2, names
    for k in names:
        assert usage[k]["STACK"] == 0 and usage[k]["LOCAL"] == 0, (k, usage[k])
