// pdmpc_kernels.cuh — device code of the B200-native MPA graph search: shared device types, the
// checkers, and the one-search-per-warp kernel (lowest-latency warp shape; also the carrier of pop
// traces, the SAT checker and the time-step dependencies).  The throughput shape — several searches per
// warp — is pdmpc_tiles.cuh, the one-CTA-per-search shape pdmpc_cta.cuh.
//
// Every shape reproduces the reference's best-first loop exactly:
//   GraphSearch.do_graph_search      hlc/optimizer/graph_search/GraphSearch.m:23-109
//   eval_edge_exact                  GraphSearch.m:111-196
//   expand_node                      hlc/optimizer/graph_search/expand_node.m:1-91
//   priority queue                   .../priority_queue/priority_queue_interface_mex.cpp:19-108
//                                    == libstdc++ __push_heap / __adjust_heap on (id, f)
//   SAT / lanelet / InterX checkers  intersect_sat.m, intersect_lanelet_boundary.m, InterX.m
//
// Bit-exactness rules: IEEE double everywhere, compiled with --fmad=false (no
// contraction), the same operation order as the reference's expressions, and
// the sin/cos algorithm of DESIGN.md §sincos.
//
// Design notes (the search is a serial pop -> check -> expand -> push chain; ncu
// shows it is bound by the number of warp instructions per pop, so everything
// here minimises uniform/scalar work per pop):
//   * the binary heap (pdmpc_heap_split.cuh): the pop's hole walk is a minimal uniform
//     loop (one aligned pair load + one compare per level), the moves along the path are
//     done by the lanes in parallel.  Pushes of all children go through a one-round fast
//     path when no child has to sift up.  The resulting array is identical to what
//     libstdc++'s sequential routines produce.
//   * heap entries carry (f, id, parent id): everything a pop needs is fetched in
//     ONE round of independent loads (own record + parent record).
//   * sin/cos of a node's yaw is computed once, when the node is expanded, and
//     cached for the edge checks of its children.
//   * the per-search obstacle polylines (lanelet bounds + all steps' obstacle
//     polygons) are staged once into shared memory; InterX then runs out of smem.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstddef>
#include <type_traits>

#include "../../include/pdmpc_b200.h"

// Optional per-phase cycle accounting (build with -DPDMPC_PROFILE; profiling builds only)
#ifdef PDMPC_PROFILE
#define PROF_DECL long long prof_t0 = clock64(), prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#define PROF_MARK(i)                      \
    do {                                  \
        long long _t = clock64();         \
        prof_acc[i] += _t - prof_t0;      \
        prof_t0 = _t;                     \
    } while (0)
#define PROF_FLUSH(o, lane0)                                                              \
    do {                                                                                  \
        if (lane0)                                                                        \
            for (int _i = 0; _i < 8; ++_i) atomicAdd((o).counters + 8 + _i, (unsigned long long)prof_acc[_i]); \
        for (int _i = 0; _i < 8; ++_i) prof_acc[_i] = 0;                                  \
    } while (0)
#else
#define PROF_DECL
#define PROF_MARK(i)
#define PROF_FLUSH(o, lane0)
#endif

// Optional launch anatomy of the throughput launch (build with -DPDMPC_TAIL_STAMPS; tools/tail_anatomy.py):
// %globaltimer stamps in ns, read back with pdmpc_get_tail_stamps.  Slots: [0] first tile CTA start (min),
// [1] first fetch that found the work list empty (min), [2] first escalation CTA start (min), [3] last escalation
// master done (max), [4] tile CTAs exited, [8 + i] exit of tile CTA i.  The default build has none of it.
#ifdef PDMPC_TAIL_STAMPS
constexpr int kTailStampSlots = 8 + 148 * 64;
__device__ unsigned long long g_tail_stamps[kTailStampSlots];
__device__ __forceinline__ unsigned long long tail_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TAIL_MIN(i) atomicMin(g_tail_stamps + (i), tail_now())
#define TAIL_MAX(i) atomicMax(g_tail_stamps + (i), tail_now())
#define TAIL_EXIT(cta)                                                                     \
    do {                                                                                   \
        atomicAdd(g_tail_stamps + 4, 1ull);                                                \
        if ((cta) < (unsigned)kTailStampSlots - 8u) g_tail_stamps[8 + (cta)] = tail_now(); \
    } while (0)
#else
#define TAIL_MIN(i)
#define TAIL_MAX(i)
#define TAIL_EXIT(cta)
#endif

namespace pdmpc {

constexpr int kWarp = 32;
constexpr int kAreaStride = PDMPC_AREA_STRIDE;
constexpr int kMaxHp = PDMPC_MAX_HP;
constexpr int kParentCache = 32;   // entries, power of two

// ---- device views -----------------------------------------------------------
// MPA tables as the kernels read them (through L1/L2: 10-73 KB, hot in every SM's L1).  All arrays
// are 16-byte aligned.
struct MpaDev {
    int nT, Hp, nE;
    const int *succ_ptr;        // [Hp*nT + 1] successors of (step k, trim t) at (k-1)*nT + (t-1)
    const int *succ_te;         // per successor: (edge << 8) | (end trim - 1), ascending end trim (expand_node.m:18)
    const double *edge_d;       // [nE*4] maneuver dx, dy, dyaw, 0
    const int *area_npts;       // [nE*3 (+pad)]
    const double *area_x, *area_y;  // [nE*3*8], zero padded
    unsigned bytes_succ_ptr, bytes_succ_te, bytes_edge_d, bytes_area_npts, bytes_area;   // multiples of 16
    unsigned table_bytes;       // sum of the above (area counted twice)
    int areas_closed;           // every maneuver area repeats its first point as its last (the reference's are)
};

struct BatchDev {
    int n, checker;
    double dt;
    const int *order;           // work item -> search index (heaviest-looking searches first), or null
    // pop_hash covers the popped nodes that passed their edge check only (pdmpc_set_cta_queue(1)); else every pop
    int hash_valid_only = 0;
    // ESCALATION (throughput shapes -> CTA shape).  A tile kernel gives a search up after its pop budget
    // (esc_budget) and appends its index to the list esc_list[0, esc_cap) (entries start as -1): a search given up
    // at the full budget `pop_limit` at esc_list[atomicAdd(esc_count)], one given up at a reduced budget at
    // esc_list[esc_cap - 1 - atomicAdd(esc_count + 2)].  Every tile CTA counts itself in esc_done when it exits.
    // The CTA kernel launched behind it takes its work items from that list (esc_producers = CTAs of the tile
    // kernel(s) > 0 selects this mode) once all producers are done: the full-budget ones first (esc_item).
    int pop_limit = 0;
    // position schedule (pop_slope > 0): the search at work position p (of pos_n in the whole batch; a chunk's item
    // 0 is at pos0) gets min(pop_limit, pop_min + (pos_n - p) / pop_slope) pops
    int pop_min = 0, pop_slope = 0;
    unsigned pos0 = 0, pos_n = 0;
    int *esc_list = nullptr;
    unsigned *esc_count = nullptr, *esc_done = nullptr;
    unsigned esc_cap = 0;
    unsigned esc_producers = 0;
    unsigned esc_gate_lo = 0, esc_gate_hi = 0xffffffffu;   // the CTA kernel instance runs iff lo < count <= hi
    const double *x0, *y0, *yaw0;
    const int *trim0;
    const double *ref_x, *ref_y, *v_ref;
    // raw CSR (SAT checker)
    const int *slot_ptr, *poly_ptr;
    const double *vert_x, *vert_y;
    // NaN-separated polylines (InterX checker), vectorize_all_obstacles.m:36-63:
    // vertex v of polygon p sits at v + p, a NaN column at poly_ptr[p+1] + p.
    const double *pl_x, *pl_y;
    // the same columns as (x, y) pairs: what the tile shape reads (one 16-byte load per point); may be null
    const double2 *pl_xy = nullptr, *ll_xy = nullptr;
    // lanelet bounds: raw (SAT) and [left, NaN, right, NaN] per search (InterX),
    // side s of search i at lane_ptr[2i+s] + 2i + s.
    const int *lane_ptr;
    const double *lane_x, *lane_y;
    const double *ll_x, *ll_y;
};

struct OutDev {
    int *status;
    uint8_t *is_exhausted;
    int *n_expanded, *n_pops;
    unsigned long long *pop_hash;
    int *trims, *tree_path;
    double *y_predicted, *g_path, *h_path;
    int *shape_npts;
    double *shape_x, *shape_y;
    unsigned long long *counters;  // [0] pops, [1] nodes, [2] obstacle columns tested
};

// Dependencies between the searches of one batch (pdmpc_plan_timestep): search i waits for
// done[j] != 0 of each predecessor j and takes j's planned areas (or its fallback areas when j
// is exhausted) as dynamic obstacles: PrioritizedController.m:449-506 consider_predecessors.
struct DepsDev {
    const int *pred_ptr, *pred_idx;   // CSR over the searches of the batch
    const int *fb_npts;               // [n*Hp] fallback areas (may be null)
    const double *fb_x, *fb_y;        // [n*Hp*kAreaStride]
    int *done;                        // [n] 0 pending, 1 planned, 2 exhausted (release/acquire at gpu scope)
    // warp-per-search kernel only: per-slot scratch in HBM for the predecessors' areas (the CTA kernel keeps
    // them in shared memory): kDepCols columns / kDepCols / 8 point counts per slot
    double *dep_x, *dep_y;
    int *dep_n;
};
constexpr int kDepCols = PDMPC_TIMESTEP_COLS;
__device__ __forceinline__ int ld_acquire_gpu(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int *p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Pop budget of the search at work position p < n (BatchDev::pop_min / pop_slope): the searches that start late get
// fewer pops before they are escalated, so none of them runs on long after the work list is empty.  Host and device.
__host__ __device__ inline int esc_budget(int p_max, int p_min, int slope, unsigned n, unsigned p) {
    if (slope <= 0) return p_max;
    const unsigned b = (unsigned)p_min + (n - p) / (unsigned)slope;
    return b < (unsigned)p_max ? (int)b : p_max;
}
// Item i of a complete escalation list with n_full full-budget entries (BatchDev::esc_list).
__device__ __forceinline__ const int *esc_item(const int *list, unsigned cap, unsigned n_full, unsigned i) {
    return i < n_full ? list + i : list + (cap - 1u - (i - n_full));
}

// Node arena + heap overflow of one resident tile ("slot"), all in HBM.
struct __align__(16) NodeA {  // 32 B: pose + cost to come, written when the node is created
    double x, y, yaw, g;
};
struct __align__(16) NodeB {  // 16 B, written when the node is created
    double h;
    unsigned parent;          // 1-based, 0 for the root (Tree.m:18)
    unsigned short edge;      // maneuver (parent trim -> trim) that leads to this node
    unsigned char trim;       // 1-based
    unsigned char k;
};
struct __align__(16) NodeCS {  // 16 B, written when the node is created
    double c, s;               // cos / sin of the node's yaw
};
struct __align__(16) HEnt {    // heap entry
    double f;
    // id:21 | parent id:21 | edge:10 | k:5 | trim-1:7 — everything the edge check and the
    // expansion of a popped node need, so that no table lookup depends on a node record
    unsigned long long w;
    __device__ __forceinline__ static unsigned long long pack(unsigned id, unsigned pid, unsigned edge, unsigned k,
                                                              unsigned trim) {
        return (unsigned long long)id | ((unsigned long long)pid << 21) | ((unsigned long long)edge << 42) |
               ((unsigned long long)k << 52) | ((unsigned long long)(trim - 1u) << 57);
    }
    __device__ __forceinline__ unsigned id() const { return (unsigned)(w & 0x1fffffu); }
    __device__ __forceinline__ unsigned pid() const { return (unsigned)((w >> 21) & 0x1fffffu); }
    __device__ __forceinline__ unsigned edge() const { return (unsigned)((w >> 42) & 0x3ffu); }
    __device__ __forceinline__ unsigned k() const { return (unsigned)((w >> 52) & 0x1fu); }
    __device__ __forceinline__ unsigned trim() const { return (unsigned)(w >> 57) + 1u; }
};
constexpr int kMaxNodeCap = 1 << 21;   // ids must fit 21 bits
constexpr int kMaxEdges = 1 << 10;
struct ArenaDev {
    NodeA *a;                 // [slots * cap]; index 0 of each slot unused (ids are 1-based)
    NodeB *b;
    NodeCS *cs;
    HEnt *heap;               // [slots * cap] overflow of the shared-memory heap top
    int cap;                  // nodes per slot
};

struct TraceDev {
    int search;               // -1: off
    long long *ids;
    long long cap;
    long long *n;
};

// ---- tile helpers -------------------------------------------------------------
template <int TILE>
struct Tile {
    unsigned mask;   // lanes of this tile within the warp
    int shift;       // first lane of the tile
    int lane;        // lane within the tile
    static constexpr unsigned kBits = TILE == 32 ? 0xffffffffu : ((1u << TILE) - 1u);

    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
    __device__ __forceinline__ unsigned ballot(bool p) const {
        return (__ballot_sync(mask, p) >> shift) & kBits;
    }
    __device__ __forceinline__ bool any(bool p) const { return __any_sync(mask, p) != 0; }
    template <class T> __device__ __forceinline__ T shfl(T v, int src) const {
        return __shfl_sync(mask, v, src, TILE);
    }
    template <class T> __device__ __forceinline__ T shfl_xor(T v, int m) const {
        return __shfl_xor_sync(mask, v, m, TILE);
    }
};

// ---- sin / cos (DESIGN.md §sincos; oracle/pdmpc_oracle.c holds the CPU twin) --
__device__ __forceinline__ void sincos_ref(double x, double &s, double &c) {
    const double TWO_OVER_PI = 0x1.45f306dc9c883p-1;
    const double P1 = 0x1.921fb54400000p+0, P2 = 0x1.0b4611a600000p-34, P3 = 0x1.3198a2e037073p-69;
    const double S[10] = {-0x1.5555555555555p-3, 0x1.1111111111111p-7, -0x1.a01a01a01a01ap-13,
                          0x1.71de3a556c734p-19, -0x1.ae64567f544e4p-26, 0x1.6124613a86d09p-33,
                          -0x1.ae7f3e733b81fp-41, 0x1.952c77030ad4ap-49, -0x1.2f49b46814157p-57,
                          0x1.71b8ef6dcf572p-66};
    const double C[10] = {-0x1.0000000000000p-1, 0x1.5555555555555p-5, -0x1.6c16c16c16c17p-10,
                          0x1.a01a01a01a01ap-16, -0x1.27e4fb7789f5cp-22, 0x1.1eed8eff8d898p-29,
                          -0x1.93974a8c07c9dp-37, 0x1.ae7f3e733b81fp-45, -0x1.6827863b97d97p-53,
                          0x1.e542ba4020225p-62};
    double n = rint(x * TWO_OVER_PI);
    double r = ((x - n * P1) - n * P2) - n * P3;
    double z = r * r;
    double ps = S[9], pc = C[9];
#pragma unroll
    for (int i = 8; i >= 0; --i) {
        ps = ps * z + S[i];
        pc = pc * z + C[i];
    }
    double sr = r + (r * z) * ps;
    double cr = 1.0 + z * pc;
    long long q = (long long)n & 3LL;
    if (q == 0) { s = sr; c = cr; }
    else if (q == 1) { s = cr; c = -sr; }
    else if (q == 2) { s = -sr; c = -cr; }
    else { s = -cr; c = sr; }
}

}  // namespace pdmpc
#include "pdmpc_heap_split.cuh"   // HeapSplit: the priority queue (libstdc++ heap order, exact array states)
namespace pdmpc {

// ---- InterX (InterX.m:63-85,108-110) ---------------------------------------
// Shape (NE segments, points in shared memory) against the NaN-separated polyline
// points [lo, hi) of (px, py) (shared or global memory).  Every lane keeps the
// constants of all NE shape edges in registers and owns a short contiguous run of
// obstacle segments, so a range takes ceil(nseg / TILE) iterations with NE
// independent dependency chains each (the search is latency bound, not FP64
// bound).  C1(i,j): obstacle points j, j+1 on opposite sides of edge i's line;
// C2(i,j): edge i's end points on opposite sides of segment j's line; both are
// evaluated branch-free.  any(C1 & C2) is the reference's boolean.
template <int NE, int TILE>
__device__ __forceinline__ bool interx_ranges(const double *px, const double *py, int lo0, int hi0, int lo1,
                                              int hi1, const double *shx, const double *shy,
                                              const Tile<TILE> &t) {
    double vx[NE + 1], vy[NE + 1], dx1[NE], dy1[NE], S1[NE];
#pragma unroll
    for (int i = 0; i <= NE; ++i) {
        vx[i] = shx[i];
        vy[i] = shy[i];
    }
#pragma unroll
    for (int i = 0; i < NE; ++i) {
        dx1[i] = vx[i + 1] - vx[i];
        dy1[i] = vy[i + 1] - vy[i];
        S1[i] = dx1[i] * vy[i] - dy1[i] * vx[i];
    }
    bool hit = false;
#pragma unroll 1
    for (int r = 0; r < 2; ++r) {
        const int lo = r ? lo1 : lo0, hi = r ? hi1 : hi0;
        const int nseg = hi - lo - 1;
        if (nseg < 1) continue;                  // InterX.m:48-52 and single-column inputs
        const int per = (nseg + TILE - 1) / TILE;
        const int j0 = lo + t.lane * per;
        const int j1 = min(j0 + per, lo + nseg);
        if (j0 < j1) {
            double x = px[j0], y = py[j0];
            double a[NE];
#pragma unroll
            for (int i = 0; i < NE; ++i) a[i] = (dx1[i] * y - dy1[i] * x) - S1[i];
#pragma unroll 1
            for (int j = j0; j < j1; ++j) {
                const double xn = px[j + 1], yn = py[j + 1];
                const double dx2 = xn - x, dy2 = yn - y;
                const double S2 = dx2 * y - dy2 * x;
                double bprev = (vy[0] * dx2 - vx[0] * dy2) - S2;
#pragma unroll
                for (int i = 0; i < NE; ++i) {
                    const double an = (dx1[i] * yn - dy1[i] * xn) - S1[i];
                    const double bn = (vy[i + 1] * dx2 - vx[i + 1] * dy2) - S2;
                    hit = hit || ((a[i] * an < 0) && (bprev * bn < 0));
                    a[i] = an;
                    bprev = bn;
                }
                x = xn;
                y = yn;
            }
        }
    }
    return t.any(hit);
}

template <int TILE>
__device__ __forceinline__ bool interx_dispatch(int ns, const double *px, const double *py, int lo0, int hi0,
                                                int lo1, int hi1, const double *shx, const double *shy,
                                                const Tile<TILE> &t) {
    switch (ns) {   // ns points -> ns-1 segments; maneuver areas have 5, 6 or 7 points
    case 5: return interx_ranges<4, TILE>(px, py, lo0, hi0, lo1, hi1, shx, shy, t);
    case 6: return interx_ranges<5, TILE>(px, py, lo0, hi0, lo1, hi1, shx, shy, t);
    case 7: return interx_ranges<6, TILE>(px, py, lo0, hi0, lo1, hi1, shx, shy, t);
    default: {
        bool hit = false;   // generic (never taken with MPA areas): one shape segment at a time
        for (int i = 0; i + 1 < ns && !hit; ++i)
            hit = interx_ranges<1, TILE>(px, py, lo0, hi0, lo1, hi1, shx + i, shy + i, t);
        return hit;
    }
    }
}

// ---- SAT (intersect_sat.m:1-42): polygon 1 in shared memory, polygon 2 in
// global memory.  Lanes own axes (edges of both polygons incl. the closing one).
// NC = false: polygon 2 is read with plain loads (it may live in shared memory).
// STRIDE: distance between consecutive points of polygon 2 in doubles (2: interleaved (x, y) pairs).
template <int TILE, bool NC = true, int STRIDE = 1>
__device__ __forceinline__ bool sat_collide(const double *x1, const double *y1, int n1,
                                            const double *__restrict__ x2, const double *__restrict__ y2,
                                            int n2, const Tile<TILE> &t) {
    bool sep = false;
    for (int e = t.lane; e < n1 + n2; e += TILE) {
        double ex, ey;
        if (e < n1) {
            int e1 = (e + 1 == n1) ? 0 : e + 1;
            ex = x1[e1] - x1[e];
            ey = y1[e1] - y1[e];
        } else {
            int f = e - n1, f1 = (f + 1 == n2) ? 0 : f + 1;
            ex = NC ? __ldg(x2 + f1 * STRIDE) - __ldg(x2 + f * STRIDE) : x2[f1 * STRIDE] - x2[f * STRIDE];
            ey = NC ? __ldg(y2 + f1 * STRIDE) - __ldg(y2 + f * STRIDE) : y2[f1 * STRIDE] - y2[f * STRIDE];
        }
        double ax = -ey, ay = ex;
        double nrm = sqrt(ax * ax + ay * ay);
        double nx = ax / nrm, ny = ay / nrm;   // zero edge -> NaN axis -> never separates
        double mn1 = nan(""), mx1 = nan(""), mn2 = nan(""), mx2 = nan("");
        for (int v = 0; v < n1; ++v) {
            double d = nx * x1[v] + ny * y1[v];
            mn1 = fmin(mn1, d);
            mx1 = fmax(mx1, d);
        }
        for (int v = 0; v < n2; ++v) {
            double d = NC ? nx * __ldg(x2 + v * STRIDE) + ny * __ldg(y2 + v * STRIDE) : nx * x2[v * STRIDE] + ny * y2[v * STRIDE];
            mn2 = fmin(mn2, d);
            mx2 = fmax(mx2, d);
        }
        // d1/d2 of intersect_a_b; which polygon owns the axis only swaps them
        if ((mn1 - mx2 > 0) || (mn2 - mx1 > 0)) sep = true;
    }
    return !t.any(sep);
}

// ---- intersect_lanelet_boundary.m:1-56 for one side; lanes own boundary segments.
template <int TILE>
__device__ __forceinline__ bool lanelet_side_sat(const double *sx, const double *sy, int ns,
                                                 const double *__restrict__ bx, const double *__restrict__ by,
                                                 int nb, const Tile<TILE> &t) {
    if (nb < 2) return false;
    double max_x = sx[0], min_x = sx[0], max_y = sy[0], min_y = sy[0];
    for (int i = 1; i < ns; ++i) {
        max_x = fmax(max_x, sx[i]);
        min_x = fmin(min_x, sx[i]);
        max_y = fmax(max_y, sy[i]);
        min_y = fmin(min_y, sy[i]);
    }
    bool hit = false;
    for (int n = t.lane; n + 1 < nb; n += TILE) {
        double ax = __ldg(bx + n), bx2 = __ldg(bx + n + 1), ay = __ldg(by + n), by2 = __ldg(by + n + 1);
        if ((max_x < ax && max_x < bx2) || (min_x > ax && min_x > bx2) || (max_y < ay && max_y < by2) ||
            (min_y > ay && min_y > by2))
            continue;
        // intersect_sat(shape, segment): ns shape axes + the segment's two (opposite) axes
        double qx[2] = {ax, bx2}, qy[2] = {ay, by2};
        bool sep = false;
        for (int e = 0; e < ns + 2 && !sep; ++e) {
            double ex, ey;
            if (e < ns) {
                int e1 = (e + 1 == ns) ? 0 : e + 1;
                ex = sx[e1] - sx[e];
                ey = sy[e1] - sy[e];
            } else {
                int f = e - ns;
                ex = qx[1 - f] - qx[f];
                ey = qy[1 - f] - qy[f];
            }
            double nxx = -ey, nyy = ex;
            double nrm = sqrt(nxx * nxx + nyy * nyy);
            double nx = nxx / nrm, ny = nyy / nrm;
            double mn1 = nan(""), mx1 = nan("");
            for (int v = 0; v < ns; ++v) {
                double d = nx * sx[v] + ny * sy[v];
                mn1 = fmin(mn1, d);
                mx1 = fmax(mx1, d);
            }
            double d0 = nx * qx[0] + ny * qy[0], d1 = nx * qx[1] + ny * qy[1];
            double mn2 = fmin(d0, d1), mx2 = fmax(d0, d1);
            if ((mn1 - mx2 > 0) || (mn2 - mx1 > 0)) sep = true;
        }
        if (!sep) hit = true;
    }
    return t.any(hit);
}

// FNV-1a over the popped ids taken as 32-bit words (parity trace of the pop order)
constexpr unsigned long long kHashSeed = 0xcbf29ce484222325ULL;
__device__ __forceinline__ unsigned long long hash_step(unsigned long long h, unsigned v) {
    return (h ^ (unsigned long long)v) * 0x100000001b3ULL;
}

// Rotate/translate one maneuver area point: GraphSearch.m:158-159.
__device__ __forceinline__ void place_point(const MpaDev &m, int edge, int kind, int i, double c, double s,
                                            double px, double py, double &ox, double &oy) {
    const int base = (edge * 3 + kind) * kAreaStride + i;
    const double ax = m.area_x[base], ay = m.area_y[base];
    ox = c * ax - s * ay + px;
    oy = s * ax + c * ay + py;
}

// ---- per-search pieces every launch shape shares ------------------------------------------------------------
// Each is called by the TILE lanes that own the search, outside the pop loop.

// Root of search si (GraphSearch.m:34-46): writes node 1 and returns the first heap entry for the caller to store.
__device__ __forceinline__ HEnt init_root(const BatchDev &b, int si, int trim0, NodeA *na, NodeB *nb, NodeCS *ncs) {
    NodeA ra;
    ra.x = __ldg(b.x0 + si); ra.y = __ldg(b.y0 + si); ra.yaw = __ldg(b.yaw0 + si); ra.g = 0.0;
    NodeCS rcs;
    sincos_ref(ra.yaw, rcs.s, rcs.c);
    NodeB rb;
    rb.h = 0.0; rb.parent = 0; rb.edge = 0xffff; rb.trim = (unsigned char)trim0; rb.k = 0;
    na[1] = ra; nb[1] = rb; ncs[1] = rcs;
    HEnt re;
    re.f = 0.0; re.w = HEnt::pack(1u, 0u, 0u, 0u, (unsigned)trim0);
    return re;
}

// Reference trajectory of search si into shared memory, and its speeds unless vref is nullptr (a shape that
// keeps running sums of them instead).
template <int TILE, class VRef>
__device__ __forceinline__ void stage_reference(const BatchDev &b, int si, int Hp, double *refx, double *refy,
                                                VRef vref, const Tile<TILE> &t) {
    for (int k = t.lane; k < Hp; k += TILE) {
        refx[k] = __ldg(b.ref_x + (size_t)si * Hp + k);
        refy[k] = __ldg(b.ref_y + (size_t)si * Hp + k);
        if constexpr (!std::is_same<VRef, std::nullptr_t>::value) vref[k] = __ldg(b.v_ref + (size_t)si * Hp + k);
    }
}

// Polyline layout of search si (vectorize_all_obstacles.m:27-63): obstacle slot s covers
// [ob_lo + rng[s], ob_lo + rng[s+1]), the lanelet bounds [left, NaN, right, NaN] cover [ll_lo, ll_hi).
// Fills rng[0..Hp+1]; staging the points is the caller's (each shape has its own layout).
struct SearchPolylines {
    int ob_lo, ob_hi, ll_lo, ll_hi;
};
template <int TILE>
__device__ __forceinline__ SearchPolylines search_polylines(const BatchDev &b, int si, int Hp, int *rng,
                                                            const Tile<TILE> &t) {
    const int *slot = b.slot_ptr + (size_t)si * (Hp + 1);
    const int sp0 = __ldg(slot + 0), spE = __ldg(slot + Hp + 1);
    const int lp0 = __ldg(b.lane_ptr + 2 * si), lp2 = __ldg(b.lane_ptr + 2 * si + 2);
    SearchPolylines p;
    p.ob_lo = __ldg(b.poly_ptr + sp0) + sp0; p.ob_hi = __ldg(b.poly_ptr + spE) + spE;
    p.ll_lo = lp0 + 2 * si; p.ll_hi = lp2 + 2 * si + 2;
    for (int k = t.lane; k <= Hp + 1; k += TILE) {
        const int q = __ldg(slot + k);
        rng[k] = __ldg(b.poly_ptr + q) + q - p.ob_lo;
    }
    return p;
}

// consider_predecessors (PrioritizedController.m:449-506) on the device.  Waits until every predecessor of search
// si is done, then hands each column of their areas to put_pt(idx, x, y) and each area's point count to
// put_n(pk, k0, np): predecessor r at step k0 + 1 is area pk = k0 * n_pred + r, its columns are
// [pk * kAreaStride, (pk + 1) * kAreaStride), points first, then NaN.  A planned predecessor's areas were written
// during this launch and are read through L2; an exhausted one's are its fallback areas.  Returns n_pred.
template <int TILE, class PutPt, class PutN>
__device__ __forceinline__ int gather_predecessor_areas(const DepsDev &dp, const OutDev &o, int si, int Hp,
                                                        unsigned nap_ns, const Tile<TILE> &t, PutPt put_pt,
                                                        PutN put_n) {
    const int q0 = __ldg(dp.pred_ptr + si);
    const int n_pred = __ldg(dp.pred_ptr + si + 1) - q0;
    for (int r = t.lane; r < n_pred; r += TILE) {
        const int *flag = dp.done + __ldg(dp.pred_idx + q0 + r);
        while (ld_acquire_gpu(flag) == 0) __nanosleep(nap_ns);
    }
    t.sync();
    const double qn = nan("");
    for (int idx = t.lane; idx < n_pred * Hp * kAreaStride; idx += TILE) {
        const int v = idx % kAreaStride, pk = idx / kAreaStride;
        const int r = pk % n_pred, k0 = pk / n_pred;
        const int j = __ldg(dp.pred_idx + q0 + r);
        const bool planned = ld_acquire_gpu(dp.done + j) == 1;
        const size_t os = (size_t)j * Hp + k0;
        int np = 0;
        double vx = qn, vy = qn;
        if (planned) {
            np = __ldcg(o.shape_npts + os);
            if (v < np) { vx = __ldcg(o.shape_x + os * kAreaStride + v); vy = __ldcg(o.shape_y + os * kAreaStride + v); }
        } else if (dp.fb_npts) {
            np = __ldg(dp.fb_npts + os);
            if (v < np) { vx = __ldg(dp.fb_x + os * kAreaStride + v); vy = __ldg(dp.fb_y + os * kAreaStride + v); }
        }
        put_pt(idx, vx, vy);
        if (v == 0) put_n(pk, k0, np);
    }
    return n_pred;
}

// Results of one search: GraphSearch.m:58-60 / :82-89.  A search that failed takes the "no plan" defaults of an
// exhausted one.  path is the caller's shared scratch of Hp + 1 ids.  cols is added to the obstacle-column
// counter when non-zero (a shape whose checkers count them passes 0).  cs_l2 reads the nodes' cos/sin through L2:
// the CTA shape needs it (its checker warps write them).  A warp that wrote them itself may use either; the choice
// is the one that keeps its pop loop as compiled before (with an L2 read in the one-search-per-warp kernel ptxas can
// no longer prove the warp converged at the pop loop's collectives, and its DEPS instance needs the L2 read to stay
// at 166 registers).  With `done` set (time-step dependencies), done[si] is released once the areas are written:
// publish_predictions, PrioritizedController.m:355-364.
template <int TILE>
__device__ __forceinline__ void write_search_result(const MpaDev &m, const OutDev &o, const NodeA *na, const NodeB *nb,
                                                    const NodeCS *ncs, unsigned *path, int si, int trim0,
                                                    unsigned goal, int status, bool exhausted, int n_nodes,
                                                    int n_pops, unsigned long long hash, unsigned long long cols,
                                                    bool cs_l2, int *done, const Tile<TILE> &t) {
    const int Hp = m.Hp;
    if (status != PDMPC_OK) exhausted = true;
    t.sync();
    if (t.lane == 0) {
        unsigned cur = goal;
        for (int d = Hp; d >= 0; --d) {           // Tree.m:44-52 path_to_root, flipped
            path[d] = exhausted ? 0u : cur;
            if (!exhausted && d > 0) cur = nb[cur].parent;
        }
        o.status[si] = status;
        if (o.is_exhausted) o.is_exhausted[si] = exhausted ? 1 : 0;
        if (o.n_expanded) o.n_expanded[si] = n_nodes;
        if (o.n_pops) o.n_pops[si] = n_pops;
        if (o.pop_hash) o.pop_hash[si] = hash;
        atomicAdd(o.counters + 0, (unsigned long long)n_pops);
        atomicAdd(o.counters + 1, (unsigned long long)n_nodes);
        if (cols) atomicAdd(o.counters + 2, cols);
    }
    t.sync();
    const double qnan = nan("");
    for (int d = t.lane; d <= Hp; d += TILE) {
        const unsigned pid = path[d];
        NodeA pa = {qnan, qnan, qnan, qnan};
        NodeB pb;
        pb.h = qnan; pb.parent = 0; pb.edge = 0; pb.trim = 0; pb.k = 0;
        if (!exhausted) { pa = na[pid]; pb = nb[pid]; }
        const size_t oo = (size_t)si * (Hp + 1) + d;
        if (o.trims) o.trims[oo] = exhausted ? (d == 0 ? trim0 : 0) : (int)pb.trim;
        if (o.tree_path) o.tree_path[oo] = (int)pid;
        if (o.g_path) o.g_path[oo] = pa.g;
        if (o.h_path) o.h_path[oo] = pb.h;
        if (d >= 1) {
            const size_t os = (size_t)si * Hp + (d - 1);
            if (o.y_predicted) {                   // return_path_to.m:11-25
                o.y_predicted[os * 3 + 0] = pa.x;
                o.y_predicted[os * 3 + 1] = pa.y;
                o.y_predicted[os * 3 + 2] = pa.yaw;
            }
            if (o.shape_npts) {                    // return_path_area.m:5-7
                int edge = 0, ns = 0;
                NodeA qa = {0.0, 0.0, 0.0, 0.0};
                NodeCS qcs = {0.0, 0.0};
                if (!exhausted) {
                    const unsigned qid = path[d - 1];   // parent on the path (was expanded)
                    qa = na[qid];
                    if (cs_l2) {
                        const double2 v = __ldcg(reinterpret_cast<const double2 *>(ncs + qid));
                        qcs.c = v.x; qcs.s = v.y;
                    } else {
                        qcs = ncs[qid];
                    }
                    edge = pb.edge;
                    ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                }
                o.shape_npts[os] = ns;
                if (o.shape_x && o.shape_y) {
                    for (int i = 0; i < kAreaStride; ++i) {
                        double ox = 0.0, oy = 0.0;
                        if (i < ns) place_point(m, edge, PDMPC_AREA_NORMAL, i, qcs.c, qcs.s, qa.x, qa.y, ox, oy);
                        o.shape_x[os * kAreaStride + i] = ox;
                        o.shape_y[os * kAreaStride + i] = oy;
                    }
                }
            }
        }
    }
    if (done) {   // the areas above are final
        __threadfence();
        t.sync();
        if (t.lane == 0) st_release_gpu(done + si, exhausted ? 2 : 1);
    }
}

template <int HS, int SP>
struct __align__(16) TileSmem {
    double hf[HS + 2];                           // heap costs, entry i at hf[i + 1] (pdmpc_heap_split.cuh)
    unsigned long long hw[HS];                   // heap payloads
    double pts_x[SP], pts_y[SP];                 // staged polylines: [lanelet bounds][obstacle slots 0..Hp]
    double refx[kMaxHp], refy[kMaxHp], vref[kMaxHp];
    double shx[kAreaStride], shy[kAreaStride];   // shape (normal offset)
    double bhx[kAreaStride], bhy[kAreaStride];   // boundary-check shape
    int rng[kMaxHp + 2];                         // polyline offset of obstacle slot s (static, steps 1..Hp)
    unsigned path[kMaxHp + 1];
    // direct-mapped cache of expanded nodes' (x, y, cos, sin): the parent record a popped
    // child needs for its edge check (children are usually popped soon after the expansion)
    unsigned pc_id[kParentCache];
    double pc_x[kParentCache], pc_y[kParentCache], pc_c[kParentCache], pc_s[kParentCache];
};

// ============================================================================
// The one-search-per-warp kernel.  Persistent: every one-warp CTA owns one arena slot and pulls
// work items from a global counter until the batch is drained.  The body is ONE loop (a small
// state machine): an iteration is "finish / fetch a search if needed, then one pop".
#ifndef PDMPC_MIN_CTAS_LAT
#define PDMPC_MIN_CTAS_LAT 12  // resident one-warp CTAs per SM the kernel is compiled for (register cap)
#endif
// DEPS (pdmpc_plan_timestep for batches beyond one CTA per search): a search waits for its predecessors'
// done flags, copies their planned (or fallback) areas into its slot's scratch and checks against them;
// work items are handed out in a topological order, so a warp only ever waits for searches taken earlier.
template <int HS, int SP, bool DEPS = false>
__global__ void __launch_bounds__(kWarp, PDMPC_MIN_CTAS_LAT) search_kernel(MpaDev m, BatchDev b, OutDev o, ArenaDev ar,
                                                              unsigned *work_counter, TraceDev tr,
                                                              DepsDev dp = DepsDev{}) {
    constexpr int TILE = kWarp;
    constexpr int WARPS = 1;
    const unsigned n_work = (unsigned)b.n;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp_id = threadIdx.x / kWarp;
    TileSmem<HS, SP> &sm = reinterpret_cast<TileSmem<HS, SP> *>(smem_raw)[warp_id];

    Tile<TILE> t;
    t.shift = 0;
    t.lane = threadIdx.x % kWarp;
    t.mask = 0xffffffffu;

    const int Hp = m.Hp, nT = m.nT;
    const size_t slot_base = ((size_t)blockIdx.x * WARPS + warp_id) * (size_t)ar.cap;
    NodeA *__restrict__ na = ar.a + slot_base;
    NodeB *__restrict__ nb = ar.b + slot_base;
    NodeCS *__restrict__ ncs = ar.cs + slot_base;
    HeapSplit heap;
    heap.sf = shared_base_once(sm.hf);
    heap.sw = shared_base_once(sm.hw);
    heap.gl = ar.heap + slot_base;
    heap.hs = HS;
    heap.len = 0;

    enum { IDLE = 0, RUN = 1, DONE = 2 };
    int phase = IDLE;
    PROF_DECL
    int si = 0, trim0 = 0;
    const int *slot = nullptr;
    int sp0 = 0, sp1 = 0, lp0 = 0, lp1 = 0, lp2 = 0;
    // InterX polylines of the current search: obstacles (slot ranges via sm.rng) and lanelet bounds
    const double *opx = nullptr, *opy = nullptr, *lpx = nullptr, *lpy = nullptr;
    int obase = 0, llo = 0, lhi = 0;
    int n_nodes = 0, n_pops = 0, status = PDMPC_OK;
    unsigned long long hash = 0, cols = 0;
    bool exhausted = false;
    unsigned goal = 0;
    // the parent record of the last pop (siblings are usually popped back to back)
    unsigned last_par = 0;
    double ppx = 0.0, ppy = 0.0, pc = 0.0, ps = 0.0;
    // DEPS: this slot's scratch for the predecessors' areas; lane k - 1 keeps the real column count of step k
    int n_pred = 0, my_dep_cols = 0;
    double *dpx = nullptr, *dpy = nullptr;
    int *dpn = nullptr;
    if (DEPS) {
        const size_t sl = (size_t)blockIdx.x * WARPS + warp_id;
        dpx = dp.dep_x + sl * kDepCols; dpy = dp.dep_y + sl * kDepCols; dpn = dp.dep_n + sl * (kDepCols / kAreaStride);
    }

    for (;;) {
        PROF_MARK(7);
        if (phase == DONE) {
            PROF_FLUSH(o, t.lane == 0);
            write_search_result(m, o, na, nb, ncs, sm.path, si, trim0, goal, status, exhausted, n_nodes, n_pops, hash,
                                cols, DEPS, DEPS ? dp.done : nullptr, t);
            phase = IDLE;
        }
        if (phase == IDLE) {
            unsigned si_u = 0;
            if (t.lane == 0) si_u = atomicAdd(work_counter, 1u);
            si_u = t.shfl(si_u, 0);
            if (si_u >= n_work) break;
            si = b.order ? __ldg(b.order + si_u) : (int)si_u;
            // ---- per-search set-up ------------------------------------------------
            t.sync();
            if (DEPS) {
                n_pred = gather_predecessor_areas(
                    dp, o, si, Hp, 200, t, [=](int idx, double x, double y) { dpx[idx] = x; dpy[idx] = y; },
                    [=](int pk, int, int np) { dpn[pk] = np; });
                __threadfence_block();
                t.sync();
                my_dep_cols = 0;
                if (t.lane < Hp)
                    for (int r = 0; r < n_pred; ++r) {
                        const int np = dpn[t.lane * n_pred + r];
                        if (np) my_dep_cols += np + 1;
                    }
            }
            stage_reference(b, si, Hp, sm.refx, sm.refy, sm.vref, t);
            slot = b.slot_ptr + (size_t)si * (Hp + 1);
            trim0 = __ldg(b.trim0 + si);
            for (int k = t.lane; k < kParentCache; k += TILE) sm.pc_id[k] = 0u;
            if (t.lane == 0) heap.st(0, init_root(b, si, trim0, na, nb, ncs));
            heap.len = 1;
            sp0 = __ldg(slot + 0); sp1 = __ldg(slot + 1);
            lp0 = __ldg(b.lane_ptr + 2 * si); lp1 = __ldg(b.lane_ptr + 2 * si + 1);
            lp2 = __ldg(b.lane_ptr + 2 * si + 2);
            if (b.checker == PDMPC_CHECKER_INTERX) {
                const SearchPolylines pl = search_polylines(b, si, Hp, sm.rng, t);
                const int nl = pl.ll_hi - pl.ll_lo, no = pl.ob_hi - pl.ob_lo;
                int used = 0;
                if (nl <= SP) {      // stage the lanelet polyline
                    for (int j = t.lane; j < nl; j += TILE) {
                        sm.pts_x[j] = __ldg(b.ll_x + pl.ll_lo + j);
                        sm.pts_y[j] = __ldg(b.ll_y + pl.ll_lo + j);
                    }
                    lpx = sm.pts_x; lpy = sm.pts_y; llo = 0; lhi = nl;
                    used = nl;
                } else {
                    lpx = b.ll_x; lpy = b.ll_y; llo = pl.ll_lo; lhi = pl.ll_hi;
                }
                if (used + no <= SP) {   // stage the obstacle polylines of all steps
                    for (int j = t.lane; j < no; j += TILE) {
                        sm.pts_x[used + j] = __ldg(b.pl_x + pl.ob_lo + j);
                        sm.pts_y[used + j] = __ldg(b.pl_y + pl.ob_lo + j);
                    }
                    opx = sm.pts_x; opy = sm.pts_y; obase = used;
                } else {
                    opx = b.pl_x; opy = b.pl_y; obase = pl.ob_lo;
                }
            }
            n_nodes = 1; n_pops = 0;
            hash = kHashSeed; cols = 0;
            status = PDMPC_OK;
            exhausted = false;
            goal = 0;
            last_par = 0;
            phase = RUN;
            t.sync();
        }
        PROF_MARK(0);   // finalize + fetch + set-up

        // ---- one iteration of the best-first loop: GraphSearch.m:53-107 ----------
        if (heap.len == 0) { exhausted = true; phase = DONE; continue; }   // :57-61
        const HEnt top = heap.pop(t.lane);
        PROF_MARK(1);   // heap pop
        const unsigned id = top.id(), par = top.pid();
        const int cK = (int)top.k();
        ++n_pops;
        if (!b.hash_valid_only) hash = hash_step(hash, id);
        if (tr.search == si && t.lane == 0) {
            if (n_pops <= tr.cap) tr.ids[n_pops - 1] = (long long)id;
            *tr.n = n_pops;
        }

        // one round of independent loads: own record (needed by the expansion only, its
        // latency hides behind the edge check), the parent's record (unless cached) and the
        // maneuver areas / successor list (edge, depth and trim ride in the heap entry)
        const NodeA ca = na[id];
        const NodeCS ccs = ncs[id];
        const int ctrim = (int)top.trim();
        const int k_exp = cK + 1;
        int sbase = 0, nchild = 0;
        if (cK < Hp) {
            sbase = m.succ_ptr[(k_exp - 1) * nT + (ctrim - 1)];
            nchild = m.succ_ptr[(k_exp - 1) * nT + (ctrim - 1) + 1] - sbase;
        }
        bool valid = true;
        if (par != 0) {   // eval_edge_exact :137-192 (root is valid unchecked)
            if (par != last_par) {
                const int cslot = par & (kParentCache - 1);
                if (sm.pc_id[cslot] == par) {
                    ppx = sm.pc_x[cslot]; ppy = sm.pc_y[cslot]; pc = sm.pc_c[cslot]; ps = sm.pc_s[cslot];
                } else {
                    const NodeA pa = na[par];
                    const NodeCS pcs = ncs[par];              // cos/sin(parent yaw), :155-156
                    ppx = pa.x; ppy = pa.y; pc = pcs.c; ps = pcs.s;
                }
                last_par = par;
            }
            const int edge = (int)top.edge();
            const int bkind = (cK == Hp) ? PDMPC_AREA_LARGE_OFFSET : PDMPC_AREA_WITHOUT_OFFSET;  // :166-174
            const int ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
            const int nbs = m.area_npts[edge * 3 + bkind];
            // (no barrier needed before the writes: the vote that ended the previous edge check
            // ordered all lanes' reads of the shape arrays)
            // all 8 (zero padded) points of both areas are placed; only the first ns / nbs are used
            if (t.lane < 8)
                place_point(m, edge, PDMPC_AREA_NORMAL, t.lane, pc, ps, ppx, ppy, sm.shx[t.lane], sm.shy[t.lane]);
            else if (t.lane < 16)
                place_point(m, edge, bkind, t.lane - 8, pc, ps, ppx, ppy, sm.bhx[t.lane - 8], sm.bhy[t.lane - 8]);
            t.sync();
            PROF_MARK(2);   // record loads + shape placement

            if (b.checker == PDMPC_CHECKER_INTERX) {
                // are_constraints_satisfied_interx.m:17,34 (no HDVs)
                const int st_lo = obase + sm.rng[0], st_hi = obase + sm.rng[1];
                const int dy_lo = obase + sm.rng[cK], dy_hi = obase + sm.rng[cK + 1];
                cols += (unsigned long long)((st_hi - st_lo) + (dy_hi - dy_lo) + (lhi - llo));
                if (DEPS) cols += (unsigned long long)t.shfl(my_dep_cols, cK - 1);
                if (interx_dispatch<TILE>(ns, opx, opy, st_lo, st_hi, dy_lo, dy_hi, sm.shx, sm.shy, t))
                    valid = false;
                else if (DEPS && n_pred > 0 &&
                         interx_dispatch<TILE>(ns, dpx, dpy, (cK - 1) * n_pred * kAreaStride, cK * n_pred * kAreaStride,
                                               0, 0, sm.shx, sm.shy, t))
                    valid = false;
                else if (interx_dispatch<TILE>(nbs, lpx, lpy, llo, lhi, 0, 0, sm.bhx, sm.bhy, t))
                    valid = false;
            } else {
                // are_constraints_satisfied_sat.m:15-53 (nV == 1; HDV block unreachable)
                const int dp0 = __ldg(slot + cK), dp1 = __ldg(slot + cK + 1);
                for (int pass = 0; pass < 2 && valid; ++pass) {
                    const int q0 = pass == 0 ? sp0 : dp0, q1 = pass == 0 ? sp1 : dp1;
                    for (int p = q0; p < q1 && valid; ++p) {
                        const int v0 = __ldg(b.poly_ptr + p), v1 = __ldg(b.poly_ptr + p + 1);
                        cols += (unsigned long long)(v1 - v0);
                        if (sat_collide<TILE>(sm.shx, sm.shy, ns, b.vert_x + v0, b.vert_y + v0, v1 - v0, t))
                            valid = false;
                    }
                }
                if (DEPS) {
                    for (int r = 0; r < n_pred && valid; ++r) {
                        const int pk = (cK - 1) * n_pred + r, nv = dpn[pk];
                        if (nv < 2) continue;
                        cols += (unsigned long long)nv;
                        if (sat_collide<TILE, false>(sm.shx, sm.shy, ns, dpx + pk * kAreaStride, dpy + pk * kAreaStride, nv, t))
                            valid = false;
                    }
                }
                if (valid) {
                    cols += (unsigned long long)(lp2 - lp0);
                    if (lanelet_side_sat<TILE>(sm.bhx, sm.bhy, nbs, b.lane_x + lp0, b.lane_y + lp0, lp1 - lp0, t))
                        valid = false;
                    else if (lanelet_side_sat<TILE>(sm.bhx, sm.bhy, nbs, b.lane_x + lp1, b.lane_y + lp1, lp2 - lp1, t))
                        valid = false;
                }
            }
        }
        PROF_MARK(3);   // constraint check
        if (!valid) continue;                                   // :75-77
        if (b.hash_valid_only) hash = hash_step(hash, id);
        if (cK == Hp) { goal = id; phase = DONE; continue; }    // :81-90

        // ---- expand_node.m:1-91 (nV == 1) --------------------------------------
        if (n_nodes + nchild >= ar.cap) { status = PDMPC_ERR_CAPACITY; phase = DONE; continue; }
        // :50-51 cos/sin of this node's yaw were computed when the node was created
        const double s = ccs.s, c = ccs.c;
        if (t.lane == 0) {
            const int cslot = id & (kParentCache - 1);
            sm.pc_id[cslot] = id;
            sm.pc_x[cslot] = ca.x; sm.pc_y[cslot] = ca.y; sm.pc_c[cslot] = c; sm.pc_s[cslot] = s;
        }
        const int to_go = Hp - k_exp;               // :37
        for (int c0 = 0; c0 < nchild; c0 += TILE) {
            const int ci = c0 + t.lane;
            const int cnt = min(TILE, nchild - c0);
            HEnt he;
            he.f = 0.0; he.w = 0;
            const unsigned nid = (unsigned)(n_nodes + 1 + ci);
            if (ci < nchild) {
                const int te = m.succ_te[sbase + ci];
                const int cedge = te >> 8, t2 = (te & 0xff) + 1;
                const double mdx = m.edge_d[cedge * 4 + 0], mdy = m.edge_d[cedge * 4 + 1],
                             mdyaw = m.edge_d[cedge * 4 + 2];
                NodeA ea;
                ea.x = c * mdx - s * mdy + ca.x;          // :53
                ea.y = s * mdx + c * mdy + ca.y;          // :54
                ea.yaw = ca.yaw + mdyaw;                  // :55
                const double ddx = ea.x - sm.refx[k_exp - 1], ddy = ea.y - sm.refy[k_exp - 1];
                const double nrm = sqrt(ddx * ddx + ddy * ddy);
                ea.g = ca.g + nrm * nrm;            // :61
                double eh = 0.0, d_max = 0.0;       // :66-73
                for (int it0 = 1; it0 <= to_go; it0 += 4) {
                    // the square roots of four steps are independent: issue them together
                    double hn[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int kk = min(k_exp + it0 + u - 1, Hp - 1);
                        const double hx = ea.x - sm.refx[kk], hy = ea.y - sm.refy[kk];
                        hn[u] = sqrt(hx * hx + hy * hy);
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (it0 + u <= to_go) {
                            d_max = d_max + b.dt * sm.vref[k_exp + it0 + u - 1];
                            const double mm = fmax(0.0, hn[u] - d_max);
                            eh = eh + mm * mm;
                        }
                    }
                }
                NodeB eb;
                eb.h = eh; eb.parent = id; eb.edge = (unsigned short)cedge;
                eb.trim = (unsigned char)t2; eb.k = (unsigned char)k_exp;
                NodeCS ecs;                         // for the child's own expansion (off the critical path)
                sincos_ref(ea.yaw, ecs.s, ecs.c);
                na[nid] = ea;                       // Tree.m:54-70 add_nodes
                nb[nid] = eb;
                ncs[nid] = ecs;
                he.f = ea.g + eh;                   // GraphSearch.m:102 (weights 1)
                he.w = HEnt::pack(nid, id, (unsigned)cedge, (unsigned)k_exp, (unsigned)t2);
            }
            PROF_MARK(4);   // successor generation
            heap.push_many(he, cnt, t.lane);        // :104, one push per child, in order
            PROF_MARK(5);   // heap pushes
        }
        n_nodes += nchild;
    }
}

// ---- staging kernels --------------------------------------------------------
// vectorize_all_obstacles.m:36-63: copy polygon p to [poly_ptr[p] + p, ...) and
// append the [NaN; NaN] column.  One thread per polygon.
__global__ void build_polyline_kernel(int n_polys, const int *__restrict__ poly_ptr,
                                      const double *__restrict__ vx, const double *__restrict__ vy,
                                      double *__restrict__ px, double *__restrict__ py, int p_base = 0,
                                      double2 *__restrict__ pxy = nullptr) {
    const int p = p_base + blockIdx.x * blockDim.x + threadIdx.x;   // polygons [p_base, p_base + n_polys)
    if (p >= p_base + n_polys) return;
    const int v0 = poly_ptr[p], v1 = poly_ptr[p + 1];
    for (int v = v0; v < v1; ++v) {
        const double x = vx[v], y = vy[v];
        px[v + p] = x;
        py[v + p] = y;
        if (pxy) pxy[v + p] = make_double2(x, y);
    }
    px[v1 + p] = nan("");
    py[v1 + p] = nan("");
    if (pxy) pxy[v1 + p] = make_double2(nan(""), nan(""));
}

}  // namespace pdmpc
