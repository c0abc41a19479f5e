// pdmpc_coupling.cuh — coupling, priorities and computation levels of a time step on the device (pdmpc_couple): what
// HighLevelController / PrioritizedController decide before the optimizer runs, for every scenario of the time step in
// two launches.
//
//   ReachableSetCoupler.couple       hlc/controller/coupling/ReachableSetCoupler.m:5-54: vehicles i, j are coupled when
//                                    area(intersect(reachable_sets{i, end}, reachable_sets{j, end})) > 1e-3 (:39-42);
//                                    the sets are the step-Hp local reachable sets of the current trim placed at the
//                                    pose (MotionPrimitiveAutomaton.m:649-687), placed exactly as fill_obstacles_kernel
//                                    places them.  [dev] polyshape intersect is replaced by the Sutherland-Hodgman
//                                    clipping of DESIGN.md §4.12 (the sets are convex hulls), the lanelet clipping of
//                                    HighLevelController.m:241-246 is not reproduced.
//   ColoringPrioritizer / ConstantPrioritizer, the level cut and kahn.m: as scenario.decide_relations states them.
//
// couple_pairs_kernel: one warp per (scenario, pair i < j).  Both sets are placed into shared memory, a bounding-box test
// rejects most pairs, the clipping runs with the lanes over the vertices of the current list: each lane emits 0, 1 or 2
// points and a warp prefix sum places them, order-preserving, into the other buffer.  One lane takes the final shoelace
// sum in list order, so every bit equals the sequential specification (scenario.convex_overlap_area).
// couple_decide_kernel: one warp per scenario (at most 64 rows: a relation row is one uint64), the coloring greedy,
// order_topo, the directed relation, Kahn levels and the level cut on masks.
#pragma once

#include "pdmpc_obstacles.cuh"

namespace pdmpc {

constexpr int kCoupleMaxRows = PDMPC_COUPLE_MAX_VEHICLES;
constexpr int kCoupleMaxVerts = 128;                   // vertices of one reachable set (closing vertex dropped)
constexpr int kCoupleListCap = 2 * kCoupleMaxVerts;    // a clipped list has at most m_P + m_Q points in exact arithmetic
constexpr int kCoupleWarps = 4;
constexpr double kCoupleArea = 1e-3;                   // ReachableSetCoupler.m:42

struct CoupleDev {
    int n_scen;
    const int *scen_ptr;                // [n_scen + 1] rows of scenario s: [scen_ptr[s], scen_ptr[s + 1])
    const int *pair_ptr;                // [n_scen + 1] prefix sums of n_s (n_s - 1) / 2
    const int *area_ptr;                // [n_scen + 1] prefix sums of n_s^2
    const double *x, *y, *yaw;
    const int *trim;                    // 1-based
    double *area;                       // n_s x n_s row-major per scenario, zeroed before the launch
    unsigned long long *adj;            // [n] coupled rows of the same scenario as a bit mask, zeroed before the launch
    int *overflow;                      // set when a clipped list outgrows kCoupleListCap
};

struct RelRow {                         // one row's relations as masks over the rows of its scenario
    unsigned long long succ, par, pred; // D(i, :), D(:, i) & ~seq(:, i), seq(:, i)
    int level, pad;                     // kahn(seq), 1-based
};

struct CoupleSm {
    double2 q[kCoupleMaxVerts];         // the clip polygon
    double2 buf[2][kCoupleListCap];     // the current list and the next one
};

// the step-Hp reachable set of `row`, closing vertex dropped, placed at its pose (translate_global)
__device__ __forceinline__ int place_last_set(const ReachDev &r, const CoupleDev &c, int row, double2 *dst, int lane) {
    const int t = c.trim[row] - 1;
    const int a0 = r.ptr[t * r.Hp + r.Hp - 1], m = r.ptr[t * r.Hp + r.Hp] - a0 - 1;
    double sn, cs;
    sincos_ref(c.yaw[row], sn, cs);
    const double x0 = c.x[row], y0 = c.y[row];
    for (int u = lane; u < m; u += kWarp) {
        const double xl = r.x[a0 + u], yl = r.y[a0 + u];
        dst[u] = make_double2(cs * xl - sn * yl + x0, sn * xl + cs * yl + y0);
    }
    return m;
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int d = kWarp / 2; d; d >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int d = kWarp / 2; d; d >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, d));
    return v;
}

// true iff the bounding boxes of the two placed sets are disjoint (any strict max < min)
__device__ __forceinline__ bool boxes_disjoint(const double2 *P, int mp, const double2 *Q, int mq, int lane) {
    double b[8] = {INFINITY, -INFINITY, INFINITY, -INFINITY, INFINITY, -INFINITY, INFINITY, -INFINITY};
    for (int u = lane; u < mp; u += kWarp) {
        b[0] = fmin(b[0], P[u].x); b[1] = fmax(b[1], P[u].x); b[2] = fmin(b[2], P[u].y); b[3] = fmax(b[3], P[u].y);
    }
    for (int u = lane; u < mq; u += kWarp) {
        b[4] = fmin(b[4], Q[u].x); b[5] = fmax(b[5], Q[u].x); b[6] = fmin(b[6], Q[u].y); b[7] = fmax(b[7], Q[u].y);
    }
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
        b[k] = warp_min(b[k]);
        b[k + 1] = warp_max(b[k + 1]);
    }
    return b[1] < b[4] || b[5] < b[0] || b[3] < b[6] || b[7] < b[2];
}

__global__ void __launch_bounds__(kCoupleWarps * kWarp) couple_pairs_kernel(ReachDev r, CoupleDev c, int n_pairs) {
    __shared__ CoupleSm sm_all[kCoupleWarps];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x % kWarp, w = threadIdx.x / kWarp;
    const int p = blockIdx.x * kCoupleWarps + w;
    if (p >= n_pairs) return;
    CoupleSm &sm = sm_all[w];
    int lo = 0, hi = c.n_scen - 1;      // the last scenario whose pairs start at or before p
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (c.pair_ptr[mid] <= p) lo = mid;
        else hi = mid - 1;
    }
    const int s = lo, r0 = c.scen_ptr[s], ns = c.scen_ptr[s + 1] - r0;
    int q = p - c.pair_ptr[s], i = 0;
    while (q >= ns - 1 - i) {
        q -= ns - 1 - i;
        ++i;
    }
    const int j = i + 1 + q;
    const int mp = place_last_set(r, c, r0 + i, sm.buf[0], lane);
    const int mq = place_last_set(r, c, r0 + j, sm.q, lane);
    __syncwarp();
    if (mp < 3 || mq < 3 || boxes_disjoint(sm.buf[0], mp, sm.q, mq, lane)) return;   // area 0.0 (zeroed)
    double sq = 0.0;                    // orientation of Q, summed in index order
    if (lane == 0)
        for (int k = 0; k < mq; ++k) {
            const double2 a = sm.q[k], b = sm.q[k + 1 < mq ? k + 1 : 0];
            sq = sq + (a.x * b.y - b.x * a.y);
        }
    sq = __shfl_sync(FULL, sq, 0);
    if (sq == 0.0) return;
    if (sq < 0.0) {                     // counter-clockwise: inside = left of every edge
        for (int u = lane; u < mq / 2; u += kWarp) {
            const double2 t = sm.q[u];
            sm.q[u] = sm.q[mq - 1 - u];
            sm.q[mq - 1 - u] = t;
        }
        __syncwarp();
    }
    int cur = 0, nc = mp;
    bool overflow = false;
    for (int k = 0; k < mq && nc > 0; ++k) {    // Sutherland-Hodgman: clip by the half-plane left of Q[k] -> Q[k+1]
        const double2 a = sm.q[k], b = sm.q[k + 1 < mq ? k + 1 : 0];
        const double ex = b.x - a.x, ey = b.y - a.y;
        const double2 *in = sm.buf[cur];
        double2 *out = sm.buf[cur ^ 1];
        int total = 0;
        for (int base = 0; base < nc; base += kWarp) {
            const int u = base + lane;
            int cnt = 0;
            bool e_in = false, s_in = false;
            double2 e = make_double2(0.0, 0.0), ip = e;
            if (u < nc) {               // e = this vertex, s = the one before it (the last one for u = 0)
                e = in[u];
                const double2 sv = in[u > 0 ? u - 1 : nc - 1];
                const double de = ex * (e.y - a.y) - ey * (e.x - a.x);
                const double ds = ex * (sv.y - a.y) - ey * (sv.x - a.x);
                e_in = de >= 0.0;
                s_in = ds >= 0.0;
                if (e_in != s_in) {
                    const double t = ds / (ds - de);
                    ip = make_double2(sv.x + t * (e.x - sv.x), sv.y + t * (e.y - sv.y));
                }
                cnt = (e_in ? 1 : 0) + (e_in != s_in ? 1 : 0);
            }
            int incl = cnt;
#pragma unroll
            for (int d = 1; d < kWarp; d <<= 1) {
                const int v = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += v;
            }
            int off = total + incl - cnt;
            if (off + cnt <= kCoupleListCap) {
                if (e_in != s_in) out[off++] = ip;
                if (e_in) out[off] = e;
            }
            total += __shfl_sync(FULL, incl, kWarp - 1);
        }
        __syncwarp();
        if (total > kCoupleListCap) {
            overflow = true;
            break;
        }
        nc = total;
        cur ^= 1;
    }
    if (lane != 0) return;
    if (overflow) {
        atomicExch(c.overflow, 1);
        return;
    }
    if (nc < 3) return;
    const double2 *L = sm.buf[cur];
    double acc = 0.0;                   // shoelace in list order
    for (int k = 0; k < nc; ++k) {
        const double2 a = L[k], b = L[k + 1 < nc ? k + 1 : 0];
        acc = acc + (a.x * b.y - b.x * a.y);
    }
    const double area = 0.5 * fabs(acc);
    double *A = c.area + c.area_ptr[s];
    A[i * ns + j] = area;
    A[j * ns + i] = area;
    if (area > kCoupleArea) {
        atomicOr(&c.adj[r0 + i], 1ull << j);
        atomicOr(&c.adj[r0 + j], 1ull << i);
    }
}

__device__ __forceinline__ unsigned long long warp_or64(unsigned long long v) {
    const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v), hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
    return ((unsigned long long)hi << 32) | lo;
}

// One warp per scenario; lane l holds rows l and l + 32 (h = 0, 1).
__global__ void __launch_bounds__(kWarp) couple_decide_kernel(CoupleDev c, int prioritizer, int max_cls, RelRow *rel) {
    __shared__ unsigned long long Ds[kCoupleMaxRows];
    __shared__ int prio[kCoupleMaxRows], lvl[kCoupleMaxRows], prio_of_color[kCoupleMaxRows + 1];
    const unsigned FULL = 0xffffffffu;
    const int s = blockIdx.x, lane = threadIdx.x;
    const int r0 = c.scen_ptr[s], n = c.scen_ptr[s + 1] - r0;
    unsigned long long A[2];
    int deg[2], color[2] = {0, 0};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int r = lane + kWarp * h;
        A[h] = r < n ? c.adj[r0 + r] : 0ull;
        deg[h] = __popcll(A[h]);
    }
    if (prioritizer == PDMPC_PRIORITY_COLORING) {
        // ColoringPrioritizer.m:11-95: isolated rows get colour 1; then, repeatedly, the uncoloured row with the most
        // distinct colours among its neighbours (ties: the higher degree, then the lower index) gets the smallest colour
        // none of its neighbours has.  nc = colours of a row's coloured neighbours as a mask (bit c - 1).
        unsigned long long nc[2] = {0ull, 0ull};
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (lane + kWarp * h < n && deg[h] == 0) color[h] = 1;
        for (;;) {
            unsigned best = 0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = lane + kWarp * h;
                if (r < n && color[h] == 0)
                    best = max(best, (1u << 24) | ((unsigned)__popcll(nc[h]) << 16) | ((unsigned)deg[h] << 8) | (unsigned)(63 - r));
            }
            best = __reduce_max_sync(FULL, best);
            if (!best) break;
            const int idx = 63 - (int)(best & 0xffu), hi = idx >= kWarp;
            int col = __ffsll((long long)~(hi ? nc[1] : nc[0]));
            col = __shfl_sync(FULL, col, idx % kWarp);
            if (lane == idx % kWarp) {
                if (hi) color[1] = col;
                else color[0] = col;
            }
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if ((A[h] >> idx) & 1ull) nc[h] |= 1ull << (col - 1);
        }
        // order_topo :96-131: the colour class holding the row of highest remaining degree (first such row) comes next,
        // its rows' degrees drop to 0; classes never picked follow in colour order.  Priority = position (1-based).
        unsigned long long used = 0ull;
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (lane + kWarp * h < n) used |= 1ull << (color[h] - 1);
        used = warp_or64(used);
        int dg[2] = {deg[0], deg[1]}, norder = 0;
        unsigned long long placed = 0ull;
        for (;;) {
            unsigned best = 0;
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (dg[h] > 0) best = max(best, ((unsigned)dg[h] << 8) | (unsigned)(63 - (lane + kWarp * h)));
            best = __reduce_max_sync(FULL, best);
            if (!best) break;
            const int m = 63 - (int)(best & 0xffu);
            const int col = __shfl_sync(FULL, m >= kWarp ? color[1] : color[0], m % kWarp);
            ++norder;
            if (lane == 0) prio_of_color[col] = norder;
            placed |= 1ull << (col - 1);
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (color[h] == col) dg[h] = 0;
        }
        for (unsigned long long rest = used & ~placed; rest; rest &= rest - 1) {
            ++norder;
            if (lane == 0) prio_of_color[__ffsll((long long)rest)] = norder;
        }
        __syncwarp();
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (lane + kWarp * h < n) prio[lane + kWarp * h] = prio_of_color[color[h]];
    } else {                            // ConstantPrioritizer.m:6-18: the lower index first
#pragma unroll
        for (int h = 0; h < 2; ++h)
            if (lane + kWarp * h < n) prio[lane + kWarp * h] = lane + kWarp * h;
    }
    __syncwarp();
    // directed coupling: i -> j iff coupled and prio(i) < prio(j) (Prioritizer.directed_coupling_from_priorities)
    unsigned long long D[2], P[2] = {0ull, 0ull}, seqP[2] = {0ull, 0ull};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int r = lane + kWarp * h;
        D[h] = 0ull;
        if (r >= n) continue;
        for (unsigned long long m = A[h]; m; m &= m - 1) {
            const int jj = __ffsll((long long)m) - 1;
            if (prio[jj] > prio[r]) D[h] |= 1ull << jj;
        }
        Ds[r] = D[h];
    }
    __syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int r = lane + kWarp * h;
        if (r >= n) continue;
        for (int ii = 0; ii < n; ++ii)
            if ((Ds[ii] >> r) & 1ull) P[h] |= 1ull << ii;
    }
    // kahn.m levels of D
    const unsigned long long all = n >= 64 ? ~0ull : (1ull << n) - 1;
    unsigned long long done = 0ull;
    int kl[2] = {0, 0}, L = 0;
    while (done != all) {
        ++L;
        const bool src0 = lane < n && !((done >> lane) & 1ull) && !(P[0] & ~done);
        const bool src1 = lane + kWarp < n && !((done >> (lane + kWarp)) & 1ull) && !(P[1] & ~done);
        const unsigned long long src = __ballot_sync(FULL, src0) | ((unsigned long long)__ballot_sync(FULL, src1) << 32);
        if (!src) break;                // cannot happen: the priorities are a strict order
        if (src0) kl[0] = L;
        if (src1) kl[1] = L;
        done |= src;
    }
    // limit_computation_levels: rows in order of their Kahn level (rows of one level are independent); a predecessor
    // stays sequential while its own level is below max_cls, the others plan in parallel
    for (int l = 1; l <= L; ++l) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = lane + kWarp * h;
            if (r >= n || kl[h] != l) continue;
            int lv = 1;
            for (unsigned long long m = P[h]; m; m &= m - 1) {
                const int ii = __ffsll((long long)m) - 1;
                if (lvl[ii] < max_cls) {
                    seqP[h] |= 1ull << ii;
                    lv = max(lv, lvl[ii] + 1);
                }
            }
            lvl[r] = lv;
        }
        __syncwarp();
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int r = lane + kWarp * h;
        if (r >= n) continue;
        RelRow o;
        o.succ = D[h];
        o.par = P[h] & ~seqP[h];
        o.pred = seqP[h];
        o.level = lvl[r];               // = kahn(seq): the longest chain of kept predecessors
        o.pad = 0;
        rel[r0 + r] = o;
    }
}

}  // namespace pdmpc
