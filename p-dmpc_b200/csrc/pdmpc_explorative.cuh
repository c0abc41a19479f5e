// pdmpc_explorative.cuh — the choice between simultaneously planned prioritizations on the device (DESIGN.md §4.13):
//
//   compute_solution_cost   hlc/controller/prioritized/PrioritizedExplorativeController.m:94-109  (cost of every
//                           (permutation, vehicle) row: tree.get_cost of the goal node, or the re-computed cost of the
//                           fallback trajectory of an exhausted search)
//   receive_solution_cost   :124-144  (summed per weakly connected sub-graph, in vehicle order)
//   choose_solution         :146-176  (round(., 8), first minimum)
//
// pdmpc_plan_timestep_explorative runs every permutation of every scenario as rows of ONE dependency-ordered launch;
// these two kernels run behind it on the same stream, before finalize_closed_loop_kernel, which commits to the
// vehicles' slots only the rows whose commit flag they set.  The arithmetic is the host's (ExplorativeRunner with
// sharding.solution_costs) operation by operation, in FP64 without FMA (the build passes --fmad=false).
#pragma once

#include "pdmpc_fallback.cuh"

namespace pdmpc {

struct ExplorativeDev {
    int n_scenarios;
    const int *base_ptr;        // [S+1] base rows (vehicles) of scenario s
    const int *row_ptr;         // [S+1] first row of scenario s in the call: rows (s, p, v) = row_ptr[s] + p * n_s + v
    const int *belonging;       // [n] 1-based weakly connected sub-graph of the base row within its scenario
    double *row_cost;           // [rows]
    double *solution_cost;      // [rows] per scenario a P_s x n_s block; (p, g - 1) = rounded sum of sub-graph g
    int *chosen, *applied_row;  // [n]
    unsigned char *commit;      // [rows] 1: the row's plan becomes its slot's state (FallbackDev.commit)
};

// MATLAB round(x, 8) as sharding.matlab_round states it: y = x * 1e8, sign(y) * floor(|y| + 0.5) / 1e8
__device__ __forceinline__ double matlab_round8(double x) {
    const double y = x * 1e8;
    const double sg = y > 0.0 ? 1.0 : (y < 0.0 ? -1.0 : (y == 0.0 ? 0.0 : y));
    return sg * floor(fabs(y) + 0.5) / 1e8;
}

// One thread per row.  A planned row costs g_path[Hp]; an exhausted row the squared distance of its fallback trajectory
// to the reference, np.sum((ref_points - fb_traj[:, :2]) ** 2) in numpy's order over e = [dx0^2, dy0^2, dx1^2, ...]:
// left to right from 0.0 below 8 values, else 8 accumulators over the complete blocks of 8, combined
// ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)), then the rest left to right.
__global__ void explorative_row_cost_kernel(int rows, int Hp, OutDev o, BatchDev b, FallbackDev fb, double *row_cost) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    if (!o.is_exhausted[row]) {
        row_cost[row] = o.g_path[(size_t)row * (Hp + 1) + Hp];
        return;
    }
    const double *rx = b.ref_x + (size_t)row * Hp, *ry = b.ref_y + (size_t)row * Hp;
    const double *tr = fb.fb_traj + (size_t)row * Hp * 3;
    auto e = [&](int j) {
        const int k = j >> 1;
        const double d = (j & 1) ? ry[k] - tr[k * 3 + 1] : rx[k] - tr[k * 3];
        return d * d;
    };
    const int m = 2 * Hp;
    double s;
    if (m < 8) {
        s = 0.0;
        for (int j = 0; j < m; ++j) s += e(j);
    } else {
        double r0 = e(0), r1 = e(1), r2 = e(2), r3 = e(3), r4 = e(4), r5 = e(5), r6 = e(6), r7 = e(7);
        int j = 8;
        for (; j + 8 <= m; j += 8) {
            r0 += e(j); r1 += e(j + 1); r2 += e(j + 2); r3 += e(j + 3);
            r4 += e(j + 4); r5 += e(j + 5); r6 += e(j + 6); r7 += e(j + 7);
        }
        s = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
        for (; j < m; ++j) s += e(j);
    }
    row_cost[row] = s;
}

// One warp per scenario: the sums per (permutation, sub-graph), their rounding, the first minimum per sub-graph, and per
// vehicle the chosen permutation, the row holding its plan and the commit flags of all the scenario's rows.
__global__ void explorative_choose_kernel(ExplorativeDev e) {
    const int w = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= e.n_scenarios) return;
    const int v0 = e.base_ptr[w], ns = e.base_ptr[w + 1] - v0, r0 = e.row_ptr[w];
    if (ns == 0) return;
    const int P = (e.row_ptr[w + 1] - r0) / ns;
    const int *bel = e.belonging + v0;
    int G = 0;
    for (int v = lane; v < ns; v += 32) G = max(G, bel[v]);
    G = __reduce_max_sync(0xffffffffu, G);
    for (int q = lane; q < P * ns; q += 32) {
        const int p = q / ns, g = q % ns + 1;
        double s = 0.0;
        if (g <= G) {
            for (int v = 0; v < ns; ++v)
                if (bel[v] == g) s = s + e.row_cost[r0 + p * ns + v];
            s = matlab_round8(s);
        }
        e.solution_cost[r0 + q] = s;
    }
    __syncwarp();
    for (int v = lane; v < ns; v += 32) {
        const double *col = e.solution_cost + r0 + bel[v] - 1;
        int best = 0;
        double bc = col[0];
        for (int p = 1; p < P; ++p)
            if (col[(size_t)p * ns] < bc) {
                bc = col[(size_t)p * ns];
                best = p;
            }
        e.chosen[v0 + v] = best;
        e.applied_row[v0 + v] = r0 + best * ns + v;
    }
    __syncwarp();
    for (int q = lane; q < P * ns; q += 32) e.commit[r0 + q] = e.chosen[v0 + q % ns] == q / ns ? 1 : 0;
}

}  // namespace pdmpc
