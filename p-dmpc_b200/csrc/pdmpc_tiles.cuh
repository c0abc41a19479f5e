// pdmpc_tiles.cuh — throughput launch shape of the graph search: T = 32 / TILE searches share
// one warp's instruction stream ("tiles" of TILE lanes), one warp per CTA.
//
// Same algorithm and bit-identical results as search_kernel (pdmpc_kernels.cuh):
//   GraphSearch.do_graph_search / eval_edge_exact   hlc/optimizer/graph_search/GraphSearch.m:23-196
//   expand_node                                      hlc/optimizer/graph_search/expand_node.m:1-91
//   priority queue                                   .../priority_queue/priority_queue_interface_mex.cpp:19-108
//                                                    == libstdc++ __push_heap / __adjust_heap (exact array states)
//   InterX + vectorize_all_obstacles                 hlc/optimizer/graph_search/InterX.m:63-85, vectorize_all_obstacles.m:27-63
//
// Why tiles.  ncu of the one-search-per-warp kernel (profiles/r01f_search_ncu.md): 1149 warp instructions
// per pop, of which ~60 % is work that is uniform over the warp (heap walk, record loads, table lookups,
// state machine) — it costs the same whether 32 lanes serve one search or several.  Here every iteration of
// the main loop performs ONE pop for EACH of the warp's T searches: the uniform part is issued once for all
// of them, the lane-parallel parts (edge check, successor generation) use lanes that idled before (22.8 of
// 32 active lanes per instruction in the old kernel).
//
// Control flow is kept warp-uniform: every phase of an iteration is executed by all 32 lanes with per-tile
// predicates, collectives are full-mask with the tile's bits extracted; loops whose trip count depends on
// the tile (heap walk, deferred C1 tests) are plain divergent loops without collectives inside.  Only the
// rare per-search prologue / epilogue runs under tile-masked divergence.
//
// InterX per pop (are_constraints_satisfied_interx.m:17,34): ONE item list per search — the segments of
// [static obstacles | dynamic obstacles of the node's step] against the normal-offset shape and the segments
// of [left, NaN, right, NaN] against the boundary-check shape — one segment per lane per round:
//   C2 row   b_i = (y1_i*dx2 - x1_i*dy2) - S2 at every shape vertex, C2(i,j) = b_i*b_{i+1} < 0 (InterX.m:71)
//   C1       only for the (i,j) with C2 true (22 % of the segments on road records, two edges each):
//            a = (dx1*y2 - dy1*x2) - S1 at both segment ends, C1 = a_j*a_{j+1} < 0 (:70); the edge
//            constants dx1, dy1, S1 (:63,67) are computed once per pop by the lanes that place the shape.
// Every product / difference is the reference's own expression (no FMA), so any(C1 & C2) is its boolean.
// Shapes are padded to the widest shape of the warp by repeating their last vertex (= the first one,
// closed polygon): b_i = b_0 there, b_0*b_0 >= 0 never satisfies the strict inequality.
//
// A point of a polyline is an (x, y) pair read with one 16-byte load through a GENERIC pointer: the copy staged in the
// tile's shared memory or — for the searches whose polylines exceed the SP staged points (48 % of the road records at
// SP = 128; lanelet bounds are staged first, they are tested at every pop) — the batch's interleaved polyline arrays
// (BatchDev::pl_xy / ll_xy, L1 / L2).  One item loop serves both; it is instantiated once per edge count of the widest
// shape of the warp (4..7), so a round pays no dispatch.
// Limits (fail over, never silently): SAT batches and pop traces are served by search_kernel.
#pragma once

#include <type_traits>

#include "pdmpc_kernels.cuh"

namespace pdmpc {

__device__ __forceinline__ unsigned keep_u32(unsigned a) {
    unsigned b;
    asm volatile("mov.u32 %0, %1;" : "=r"(b) : "r"(a));   // not rematerialisable
    return b;
}
__device__ __forceinline__ void sts_f64x2(unsigned a, double x, double y) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(x), "d"(y) : "memory");
}

// C2 row of InterX.m:71 for ONE obstacle segment against the NE edges of a placed shape (vertices at `vb`, 16 bytes
// each, padded behind the shape's last point by copies of it): bit i = b_i * b_{i+1} < 0 with
// b_i = (y1_i*dx2 - x1_i*dy2) - S2.  All vertex loads first, then NE independent chains — no branch between
// them, so their latencies overlap (the loop with `if (i < ne)` compiled to one serial load->5 FP64 ops->compare
// block per vertex).  CLOSED: vertex NE is a copy of vertex 0 (closed polygon with at most NE edges, padded by
// its last = first point), so b_NE is b_0, bit for bit, without being computed.
template <int NE, bool CLOSED>
__device__ __forceinline__ unsigned interx_c2_row(unsigned vb, double dx2, double dy2, double S2) {
    double b[NE + 1];
#pragma unroll
    for (int i = 0; i < NE + (CLOSED ? 0 : 1); ++i) {
        const double2 vv = lds_f64x2(vb + 16u * (unsigned)i);
        b[i] = (vv.y * dx2 - vv.x * dy2) - S2;
    }
    if (CLOSED) b[NE] = b[0];
    unsigned c2 = 0;
#pragma unroll
    for (int i = 0; i < NE; ++i)
        if (b[i] * b[i + 1] < 0) c2 |= 1u << i;
    return c2;
}
// ne edges, 1 <= ne <= kAreaStride - 1 (warp-uniform): the instance with the next even edge count is exact as
// well (padded vertices repeat the last one: b_i = b_{i+1} there, b*b >= 0 never sets a bit)
template <bool CLOSED>
__device__ __forceinline__ unsigned interx_c2_dispatch(int ne, unsigned vb, double dx2, double dy2, double S2) {
    static_assert(kAreaStride == 8, "edge-count dispatch");
    switch (ne) {
    case 7: return interx_c2_row<7, CLOSED>(vb, dx2, dy2, S2);
    case 6: return interx_c2_row<6, CLOSED>(vb, dx2, dy2, S2);
    case 5: return interx_c2_row<5, CLOSED>(vb, dx2, dy2, S2);
    default: return interx_c2_row<4, CLOSED>(vb, dx2, dy2, S2) & ((1u << ne) - 1u);
    }
}

template <int HS, int SP>
struct __align__(16) TileSm {
    double hf[HS + 2];                      // heap costs, entry i at hf[i + 1] (pdmpc_heap_split.cuh layout)
    unsigned long long hw[HS];              // heap payloads
    double2 pts[SP];                        // staged polylines (x, y): [lanelet bounds][obstacle slots 0..Hp]
    double2 shp[2][kAreaStride];            // placed areas: [0] normal offset, [1] boundary check; tail = last vertex
    double ec[2][kAreaStride][4];           // per shape edge: dx1, dy1, S1, -
    double refx[kMaxHp], refy[kMaxHp], vref[kMaxHp];
    int rng[kMaxHp + 2];                    // polyline offset of obstacle slot s
    unsigned path[kMaxHp + 1];
};


template <int TILE, int HS, int SP, int MINB>
__global__ void __launch_bounds__(kWarp, MINB)
search_tile_kernel(MpaDev m, BatchDev b, OutDev o, ArenaDev ar, unsigned *work_counter, TraceDev tr, int pts_limit) {
    // pts_limit: 0 = SP, else a smaller staging limit (test knob: exercises the unstaged path)
    constexpr int T = kWarp / TILE;
    constexpr unsigned FULL = 0xffffffffu;
    constexpr unsigned TB = TILE == 32 ? FULL : ((1u << TILE) - 1u);
    static_assert(TILE == 8 || TILE == 16 || TILE == 32, "tile width");
    static_assert(HS % 2 == 0, "aligned child pairs");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const int tile = lane / TILE;
    // read once: nvcc otherwise re-derives them from SR_TID.X (a slow special-register read) all over the pop loop
    const int tl = (int)keep_u32((unsigned)(lane % TILE)), shift = (int)keep_u32((unsigned)(tile * TILE));
    const unsigned tmask = TB << shift;
    Tile<TILE> t;
    t.mask = tmask; t.shift = shift; t.lane = tl;
    TileSm<HS, SP> &sm = reinterpret_cast<TileSm<HS, SP> *>(smem_raw)[tile];
    const unsigned sf = shared_base_once(sm.hf), sw = shared_base_once(sm.hw);
    const unsigned spts = shared_base_once(sm.pts), sshp = shared_base_once(sm.shp), sec = shared_base_once(sm.ec);

    const int Hp = m.Hp, nT = m.nT;
    const size_t slot_base = ((size_t)blockIdx.x * T + tile) * (size_t)ar.cap;
    NodeA *__restrict__ na = ar.a + slot_base;
    NodeB *__restrict__ nb = ar.b + slot_base;
    NodeCS *__restrict__ ncs = ar.cs + slot_base;
    HEnt *__restrict__ hgl = ar.heap + slot_base;

    // ---- heap access: entries [0, HS) in shared memory, the rest in the slot's arena ----------------
    auto h_f = [&](int i) -> double { return i < HS ? lds_f64(sf + 8u * (unsigned)(i + 1)) : hgl[i].f; };
    auto h_ld = [&](int i) -> HEnt {
        HEnt e;
        if (i < HS) { e.f = lds_f64(sf + 8u * (unsigned)(i + 1)); e.w = lds_u64(sw + 8u * (unsigned)i); }
        else e = hgl[i];
        return e;
    };
    auto h_st = [&](int i, const HEnt &e) {
        if (i < HS) { sts_f64(sf + 8u * (unsigned)(i + 1), e.f); sts_u64(sw + 8u * (unsigned)i, e.w); }
        else hgl[i] = e;
    };
    // __push_heap(first, p, 0, v) for the tiles with `su` (stl_heap.h:135-147): lanes <-> ancestors of p
    auto sift_up_at = [&](bool su, int p, const HEnt &v) {
        const int D = 31 - __clz(p + 1);               // number of ancestors of position p
        int base = 0, Tt = 0;
        bool fin = !su;
        for (;;) {
            const int a = base + tl + 1;               // this lane's ancestor, `a` levels up
            const bool anc = !fin && a <= D;
            HEnt e;
            e.f = 0.0; e.w = 0;
            if (anc) e = h_ld(((p + 1) >> a) - 1);
            const unsigned gt = (__ballot_sync(FULL, anc && e.f > v.f) >> shift) & TB;
            const int run = (gt == TB) ? TILE : (__ffs(~gt) - 1);   // leading run of greater ancestors
            if (!fin && tl < run) h_st(((p + 1) >> (a - 1)) - 1, e);
            if (!fin) {
                Tt = base + run;
                if (run < TILE || base + TILE >= D) fin = true;
            }
            if (__all_sync(FULL, fin)) break;
            base += TILE;
        }
        if (su && tl == 0) h_st(((p + 1) >> Tt) - 1, v);
        __syncwarp();
    };

    enum { IDLE = 0, RUN = 1, DONE = 2, EXIT = 3 };
    int phase = IDLE;
    int si = 0, trim0 = 0, len = 0;
    // polylines of the current search as (x, y) pairs, read through GENERIC pointers: the staged copy in shared
    // memory or, when a polyline does not fit, the batch's interleaved arrays (L1 / L2) — one code path for both
    const double2 *Op = nullptr, *Lp = nullptr;   // obstacle slot s at Op + rng[s]; lanelet bounds [Lp, Lp + nlan)
    int nlan = 0;
    int n_nodes = 0, n_pops = 0, status = PDMPC_OK;
    unsigned long long hash = 0, cols = 0;
    bool exhausted = false;
    unsigned goal = 0;

    for (;;) {
        if (phase == RUN && b.pop_limit > 0 && n_pops >= b.pop_limit) {
            // ---- escalation: a search this long is the tail of the launch; the CTA shape behind this kernel
            //      runs it from scratch at a fraction of the per-pop latency.  Nothing of it is written here.
            if (tl == 0) {
                const unsigned q = atomicAdd(b.esc_count, 1u);
                st_release_gpu(b.esc_list + q, si);
            }
            phase = IDLE;
        }
        if (phase == DONE) {
            // ---- results (tile-masked: other tiles wait) ----------------------------------------------
            write_search_result(m, o, na, nb, ncs, sm.path, si, trim0, goal, status, exhausted, n_nodes, n_pops, hash,
                                cols, false, nullptr, t);
            phase = IDLE;
        }
        while (phase == IDLE) {
            // ---- fetch the next search; per-search set-up (tile-masked) -------------------------
            unsigned si_u = 0;
            if (tl == 0) si_u = atomicAdd(work_counter, 1u);
            si_u = __shfl_sync(tmask, si_u, shift);
            if (si_u >= (unsigned)b.n) { phase = EXIT; break; }
            si = b.order ? __ldg(b.order + si_u) : (int)si_u;
            __syncwarp(tmask);
            stage_reference(b, si, Hp, sm.refx, sm.refy, sm.vref, t);
            const SearchPolylines pl = search_polylines(b, si, Hp, sm.rng, t);
            const int nl = pl.ll_hi - pl.ll_lo, no = pl.ob_hi - pl.ob_lo;
            const int sp_lim = pts_limit > 0 ? min(pts_limit, SP) : SP;
            const bool lst = nl <= sp_lim, ost = (lst ? nl : 0) + no <= sp_lim;
            // lanelet bounds first (they are tested at every pop), then the obstacle slots
            if (lst)
                for (int j = tl; j < nl; j += TILE) sm.pts[j] = __ldg(b.ll_xy + pl.ll_lo + j);
            if (ost)
                for (int j = tl; j < no; j += TILE) sm.pts[(lst ? nl : 0) + j] = __ldg(b.pl_xy + pl.ob_lo + j);
            Lp = lst ? sm.pts : b.ll_xy + pl.ll_lo;
            Op = ost ? sm.pts + (lst ? nl : 0) : b.pl_xy + pl.ob_lo;
            nlan = nl;
            trim0 = __ldg(b.trim0 + si);
            if (tl == 0) h_st(0, init_root(b, si, trim0, na, nb, ncs));
            len = 1;
            n_nodes = 1; n_pops = 0;
            hash = kHashSeed; cols = 0;
            status = PDMPC_OK;
            exhausted = false;
            goal = 0;
            phase = RUN;
            __threadfence_block();
            __syncwarp(tmask);
        }
        if (__all_sync(FULL, phase == EXIT)) break;
        __syncwarp();

        // =========== one pop for every running tile: GraphSearch.m:53-107 ==========================
        const bool run = phase == RUN;
        const bool has = run && len > 0;
        if (run && !has) { exhausted = true; phase = DONE; }                // :57-61
        HEnt top;
        top.f = 0.0; top.w = 0;
        if (has) { top.f = lds_f64(sf + 8u); top.w = lds_u64(sw); }
        const unsigned id = top.id(), par = top.pid();
        const int cK = (int)top.k(), ctrim = (int)top.trim(), edge = (int)top.edge();
        const bool chk = has && par != 0;       // eval_edge_exact :137-139: the root is valid unchecked
        // ---- early loads (their latency hides behind the heap walk): own record, parent pose,
        //      successor list, point counts of the maneuver's areas
        NodeA ca = {0.0, 0.0, 0.0, 0.0};
        NodeCS ccs = {0.0, 0.0}, pcs = {0.0, 0.0};
        double2 pxy = make_double2(0.0, 0.0);
        int sbase = 0, send = 0, ns = 0, nbs = 0;   // consumed after the heap walk (their loads overlap it)
        const int bkind = (cK == Hp) ? PDMPC_AREA_LARGE_OFFSET : PDMPC_AREA_WITHOUT_OFFSET;   // :166-174
        // the maneuver's area points this lane places (tables are padded by the last point: no count needed first)
        double ax0 = 0.0, ay0 = 0.0, ax1 = 0.0, ay1 = 0.0;
        if (chk) {
            if (TILE >= 16) {
                if (tl < 16) {
                    const int ab = (edge * 3 + ((tl >> 3) ? bkind : PDMPC_AREA_NORMAL)) * kAreaStride + (tl & 7);
                    ax0 = __ldg(m.area_x + ab); ay0 = __ldg(m.area_y + ab);
                }
            } else {
                const int a0 = (edge * 3 + PDMPC_AREA_NORMAL) * kAreaStride + tl, a1 = (edge * 3 + bkind) * kAreaStride + tl;
                ax0 = __ldg(m.area_x + a0); ay0 = __ldg(m.area_y + a0);
                ax1 = __ldg(m.area_x + a1); ay1 = __ldg(m.area_y + a1);
            }
        }
        if (has) {
            if (cK < Hp) {                                // own record and successor list: only an expansion reads them
                ca = na[id];
                ccs = ncs[id];
                const int q = cK * nT + (ctrim - 1);      // step k_exp = cK + 1
                sbase = __ldg(m.succ_ptr + q);
                send = __ldg(m.succ_ptr + q + 1);
            }
            if (par != 0) {
                pxy = *reinterpret_cast<const double2 *>(na + par);
                pcs = ncs[par];                            // cos/sin(parent yaw), :155-156
                ns = __ldg(m.area_npts + edge * 3 + PDMPC_AREA_NORMAL);
                nbs = __ldg(m.area_npts + edge * 3 + bkind);
            }
            ++n_pops;
            if (!b.hash_valid_only) hash = hash_step(hash, id);
            if (tr.search == si && tl == 0) {
                if (n_pops <= tr.cap) tr.ids[n_pops - 1] = (long long)id;
                *tr.n = n_pops;
            }
        }
        // ---- pq.pop(): __adjust_heap's walk + __push_heap of the last entry (stl_heap.h:224-249) ---
        {
            const int n = len - 1;          // heap size after the pop; entry[n] is re-inserted
            const bool act = has && n > 0;
            HEnt v;
            v.f = 0.0; v.w = 0;
            int hole = 0, D = 0;
            if (act) {
                v = h_ld(n);
                const int lim = (n - 1) >> 1;       // hole < lim: both children exist
                if (n <= HS) {
                    while (hole < lim) {            // the hole follows the smaller child (right unless right.f > left.f)
                        const double2 p = lds_f64x2(sf + 16u * (unsigned)hole + 16u);
                        hole = 2 * hole + 2 - (p.y > p.x ? 1 : 0);
                        ++D;
                    }
                } else {
                    while (hole < lim) {
                        if (2 * hole + 2 < HS) {
                            const double2 p = lds_f64x2(sf + 16u * (unsigned)hole + 16u);
                            hole = 2 * hole + 2 - (p.y > p.x ? 1 : 0);
                            ++D;
                            continue;
                        }
                        const double fl = h_f(2 * hole + 1), fr = h_f(2 * hole + 2);
                        hole = 2 * hole + 2 - (fr > fl ? 1 : 0);
                        ++D;
                    }
                }
                if ((n & 1) == 0 && hole == ((n - 2) >> 1)) {   // single (left) child at n - 1
                    hole = n - 1;
                    ++D;
                }
            }
            if (has) len = n;
            // the path is determined by its last entry: level L (1..D) is the ancestor D - L levels above
            // the final hole.  Path costs are non-decreasing, so __push_heap stops at the deepest path
            // entry with f <= v.f: the entries down to it move up one level, v lands in its place.
            bool todo = act;
            for (int base = 0;; base += TILE) {
                const int L = base + tl + 1;
                const bool on = todo && L <= D;
                const int myc = on ? (((hole + 1) >> (D - L)) - 1) : 0;
                HEnt e;
                e.f = 0.0; e.w = 0;
                if (on) e = h_ld(myc);
                const unsigned le = (__ballot_sync(FULL, on && !(e.f > v.f)) >> shift) & TB;
                const int Mr = 32 - __clz(le);             // entries of this round that stay above v
                if (on && tl < Mr) h_st((myc - 1) >> 1, e);
                const bool more = todo && Mr == TILE && base + TILE < D;
                if (todo && !more) {
                    const int Lv = base + Mr;              // v lands where path level Lv was (0: the root)
                    if (tl == 0) h_st(Lv ? (((hole + 1) >> (D - Lv)) - 1) : 0, v);
                    todo = false;
                }
                if (!__any_sync(FULL, more)) break;
            }
            __syncwarp();
        }

        // ---- eval_edge_exact :141-192: place the maneuver's areas by the PARENT pose ---------------
        const int nchild = send - sbase;
        bool valid = has;
        if (TILE >= 16) {
            if (chk && tl < 16)
                sts_f64x2(sshp + 16u * (unsigned)tl, pcs.c * ax0 - pcs.s * ay0 + pxy.x, pcs.s * ax0 + pcs.c * ay0 + pxy.y);
        } else if (chk) {
            sts_f64x2(sshp + 16u * (unsigned)tl, pcs.c * ax0 - pcs.s * ay0 + pxy.x, pcs.s * ax0 + pcs.c * ay0 + pxy.y);
            sts_f64x2(sshp + 16u * (unsigned)(8 + tl), pcs.c * ax1 - pcs.s * ay1 + pxy.x, pcs.s * ax1 + pcs.c * ay1 + pxy.y);
        }
        __syncwarp();
        // edge constants of InterX.m:63,67 — dx1, dy1, S1 = dx1*y1 - dy1*x1 — one edge per lane
        if (TILE >= 16) {
            if (chk && tl < 16) {
                const int i = tl & 7;
                const double2 v0 = lds_f64x2(sshp + 16u * (unsigned)tl);
                const double2 v1 = lds_f64x2(sshp + 16u * (unsigned)((tl & 8) + min(i + 1, 7)));
                const double dx1 = v1.x - v0.x, dy1 = v1.y - v0.y;
                sts_f64x2(sec + 32u * (unsigned)tl, dx1, dy1);
                sts_f64(sec + 32u * (unsigned)tl + 16u, dx1 * v0.y - dy1 * v0.x);
            }
        } else {
#pragma unroll
            for (int sel = 0; sel < 2; ++sel) {
                if (chk) {
                    const double2 v0 = lds_f64x2(sshp + 16u * (unsigned)(sel * 8 + tl));
                    const double2 v1 = lds_f64x2(sshp + 16u * (unsigned)(sel * 8 + min(tl + 1, 7)));
                    const double dx1 = v1.x - v0.x, dy1 = v1.y - v0.y;
                    sts_f64x2(sec + 32u * (unsigned)(sel * 8 + tl), dx1, dy1);
                    sts_f64(sec + 32u * (unsigned)(sel * 8 + tl) + 16u, dx1 * v0.y - dy1 * v0.x);
                }
            }
        }
        // ---- InterX item list of this pop: item e < n0 is segment e of the static obstacles, n0 <= e < n01 a
        //      segment of the dynamic obstacles of step cK, e >= n01 a segment of [left, NaN, right, NaN] -----------
        int n0 = 0, n01 = 0, ntot = 0;
        const double2 *P0 = nullptr, *P1 = nullptr, *P2 = nullptr;   // first point of item e: P[range of e] + e
        if (chk) {
            const int st_lo = sm.rng[0], st_hi = sm.rng[1];
            const int dy_lo = sm.rng[cK], dy_hi = sm.rng[cK + 1];
            cols += (unsigned long long)((st_hi - st_lo) + (dy_hi - dy_lo) + nlan);
            n0 = max(st_hi - st_lo - 1, 0);                       // InterX.m:48-52 and single-column inputs
            n01 = n0 + max(dy_hi - dy_lo - 1, 0);
            ntot = n01 + max(nlan - 1, 0);
            P0 = Op + st_lo; P1 = Op + (dy_lo - n0); P2 = Lp - n01;
        }
        // widest shape of the warp: edges evaluated per item (others see their padded last vertex)
        const int ne_max = __reduce_max_sync(FULL, chk ? max(ns, nbs) - 1 : 0);
        __syncwarp();
        // one instance of the loop per edge count (warp-uniform), so the C2 row needs no dispatch per round
        auto interx_items = [&](auto ne_c, auto closed_c) {
            constexpr int NE = decltype(ne_c)::value;
            constexpr bool CLOSED = decltype(closed_c)::value;
            bool hit = false;
            for (int e = tl;; e += TILE) {
                const bool act = e < ntot;
                if (!__any_sync(FULL, act)) break;
                if (act) {
                    const bool lb = e >= n01;                                   // lanelet boundary item
                    const double2 *pp = (lb ? P2 : (e < n0 ? P0 : P1)) + e;
                    const double2 p0 = pp[0], p1 = pp[1];
                    const double dx2 = p1.x - p0.x, dy2 = p1.y - p0.y;          // InterX.m:64
                    const double S2 = dx2 * p0.y - dy2 * p0.x;                  // :68
                    unsigned c2 = interx_c2_row<NE, CLOSED>(lb ? sshp + 128u : sshp, dx2, dy2, S2);   // :71
                    if (NE == 4) c2 &= (1u << ne_max) - 1u;                     // ne_max < 4: the instance is wider
                    const unsigned ebase = lb ? sec + 256u : sec;
                    for (unsigned cc = c2; cc; cc &= cc - 1u) {                 // C1 of the edges with C2, :70
                        const unsigned eb = ebase + 32u * (unsigned)(__ffs(cc) - 1);
                        const double2 d1 = lds_f64x2(eb);
                        const double S1 = lds_f64(eb + 16u);
                        const double a0 = (d1.x * p0.y - d1.y * p0.x) - S1;
                        const double a1 = (d1.x * p1.y - d1.y * p1.x) - S1;
                        if (a0 * a1 < 0) hit = true;
                    }
                }
                const unsigned hm = (__ballot_sync(FULL, hit) >> shift) & TB;
                if (hm) { valid = false; ntot = 0; }                            // :17/:34 -> is_valid = false
            }
        };
        static_assert(kAreaStride == 8, "edge-count dispatch");
        if (m.areas_closed) {
            switch (ne_max) {
            case 7: interx_items(std::integral_constant<int, 7>{}, std::true_type{}); break;
            case 6: interx_items(std::integral_constant<int, 6>{}, std::true_type{}); break;
            case 5: interx_items(std::integral_constant<int, 5>{}, std::true_type{}); break;
            default: interx_items(std::integral_constant<int, 4>{}, std::true_type{}); break;
            }
        } else {
            switch (ne_max) {
            case 7: interx_items(std::integral_constant<int, 7>{}, std::false_type{}); break;
            case 6: interx_items(std::integral_constant<int, 6>{}, std::false_type{}); break;
            case 5: interx_items(std::integral_constant<int, 5>{}, std::false_type{}); break;
            default: interx_items(std::integral_constant<int, 4>{}, std::false_type{}); break;
            }
        }
        __syncwarp();

        // ---- :75-90 ------------------------------------------------------------------------------
        if (has && valid && b.hash_valid_only) hash = hash_step(hash, id);
        if (has && valid && cK == Hp) { goal = id; phase = DONE; }
        bool doexp = has && valid && cK < Hp;
        if (doexp && n_nodes + nchild >= ar.cap) { status = PDMPC_ERR_CAPACITY; phase = DONE; doexp = false; }
        if (!__any_sync(FULL, doexp)) continue;

        // ---- expand_node.m:1-91 (nV == 1): lane q creates child q ---------------------------------
        const int k_exp = cK + 1;
        const int to_go = Hp - k_exp;               // :37
        const double s = ccs.s, c = ccs.c;          // :50-51, computed when the node was created
        for (int c0 = 0;; c0 += TILE) {
            const bool again = doexp && c0 < nchild;
            if (!__any_sync(FULL, again)) break;
            const int ci = c0 + tl;
            HEnt he;
            he.f = 0.0; he.w = 0;
            if (again && ci < nchild) {
                const unsigned nid = (unsigned)(n_nodes + 1 + ci);
                const int te = __ldg(m.succ_te + sbase + ci);
                const int cedge = te >> 8, t2 = (te & 0xff) + 1;
                const double2 md = *reinterpret_cast<const double2 *>(m.edge_d + cedge * 4);
                const double mdyaw = __ldg(m.edge_d + cedge * 4 + 2);
                NodeA ea;
                ea.x = c * md.x - s * md.y + ca.x;          // :53
                ea.y = s * md.x + c * md.y + ca.y;          // :54
                ea.yaw = ca.yaw + mdyaw;                    // :55
                const double ddx = ea.x - sm.refx[k_exp - 1], ddy = ea.y - sm.refy[k_exp - 1];
                const double nrm = sqrt(ddx * ddx + ddy * ddy);
                ea.g = ca.g + nrm * nrm;                    // :61
                double eh = 0.0, d_max = 0.0;               // :66-73
                for (int it0 = 1; it0 <= to_go; it0 += 4) {
                    double hn[4];                           // independent square roots issued together
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
                na[nid] = ea;                               // Tree.m:54-70 add_nodes
                nb[nid] = eb;
                if (k_exp < Hp) {                           // cos/sin of the child's yaw: for ITS expansion and for placing
                    NodeCS ecs;                             // its children's areas — a node of depth Hp has neither
                    sincos_ref(ea.yaw, ecs.s, ecs.c);
                    ncs[nid] = ecs;
                }
                he.f = ea.g + eh;                           // GraphSearch.m:102 (weights 1)
                he.w = HEnt::pack(nid, id, (unsigned)cedge, (unsigned)k_exp, (unsigned)t2);
            }
            // ---- :104 one pq.push per child, in order (lane q holds child q of this round) ---------
            const int mcnt = again ? min(TILE, nchild - c0) : 0;
            int done = 0;
            for (;;) {
                if (!__any_sync(FULL, done < mcnt)) break;
                const bool act = tl >= done && tl < mcnt;
                const int p = len + (tl - done);
                const int hpar = (p - 1) >> 1;
                const int src = done + max(hpar - len, 0);
                const double nf = __shfl_sync(FULL, he.f, src & (TILE - 1), TILE);
                bool need = false;
                if (act && p > 0) {
                    const double pf = (hpar < len) ? h_f(hpar) : nf;
                    need = pf > he.f;
                }
                const unsigned nm = (__ballot_sync(FULL, need) >> shift) & TB;
                const int nfast = max(nm ? (__ffs(nm) - 1 - done) : (mcnt - done), 0);
                if (act && tl < done + nfast) h_st(p, he);
                len += nfast;
                done += nfast;
                __syncwarp();
                const bool su = done < mcnt;
                HEnt v;
                v.f = __shfl_sync(FULL, he.f, done & (TILE - 1), TILE);
                v.w = __shfl_sync(FULL, he.w, done & (TILE - 1), TILE);
                if (__any_sync(FULL, su)) sift_up_at(su, len, v);
                if (su) { ++len; ++done; }
            }
        }
        if (doexp) n_nodes += nchild;
        __syncwarp();
    }
    if (b.esc_done) {   // this producer is done: everything it appended to the escalation list is visible
        __syncwarp();
        __threadfence();
        if (lane == 0) atomicAdd(b.esc_done, 1u);
    }
}

}  // namespace pdmpc
