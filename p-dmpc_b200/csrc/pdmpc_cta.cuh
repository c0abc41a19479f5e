// pdmpc_cta.cuh — the CTA launch shape of the graph search: NM searches per CTA, each owned by a MASTER
// warp (queue + tree), their edge checks done ahead of time by a pool of NC CHECKER warps the masters share.
// One CTA per SM.  Lowest single-search latency (a 20-vehicle time step puts one search on an SM and all
// checkers serve it) and, with several masters per SM, a throughput shape whose per-search latency stays low
// enough that the batch has no tail.
//
// Same algorithm and bit-identical results as search_kernel (pdmpc_kernels.cuh):
//   GraphSearch.do_graph_search / eval_edge_exact   hlc/optimizer/graph_search/GraphSearch.m:23-196
//   expand_node                                      hlc/optimizer/graph_search/expand_node.m:1-91
//   priority queue                                   .../priority_queue/priority_queue_interface_mex.cpp:19-108
//   InterX / SAT checkers                            InterX.m:63-85, intersect_sat.m, intersect_lanelet_boundary.m
//
// The reference validates an edge lazily, when its end node is popped (GraphSearch.m:64-77).  Whether an
// edge is valid is a pure function of the node (parent pose, maneuver, depth), so the answer can be computed
// EARLY without changing any result:
//   * a master owns the priority queue and the tree of its search: pop -> expand -> push.  Node ids and
//     n_expanded are exactly the reference's.
//   * the checkers validate the children of every expansion as soon as they are created, one child per warp
//     (placement of the maneuver areas, InterX / SAT against the staged obstacle polylines), compute cos/sin
//     of a valid child's yaw for its own later expansion, and publish a 2-bit flag per node in shared memory.
//
// Two queue disciplines (`fast` launch argument):
//   0  EXACT (launch shape 4): the reference's lazy queue — every child is pushed, an invalid node is popped,
//      found invalid (its flag) and skipped, exactly as GraphSearch.m:75-77 does.  pop_hash covers every pop.
//   1  VALID-ONLY QUEUE WITH DEFERRED INSERTION (launch shape 5).  With the answers known early, an invalid
//      child need not enter the queue at all, provided no pop ever has to break a tie:
//      * the reference's next VALID pop is a minimum of the whole queue, hence a minimum of the valid entries;
//        if that minimum is unique among the valid entries it is the same node whatever invalid entries
//        surround it, so the sequence of valid pops — and with it every expansion, node id, n_expanded, the
//        goal and the path — equals the reference's;
//      * new children wait in a PENDING buffer (one entry per lane of the master) until their flag arrives:
//        valid ones are then pushed, invalid ones dropped.  The master only blocks on a pending child whose
//        cost is not above the queue's current minimum — only such a child could be the next pop (6.5 % of
//        the pops of road-network records are children of the expansion before them);
//      * before every pop the minimum must be strictly below both children of the root.  On the first
//        non-unique minimum the search is RE-RUN from scratch with the exact queue (never observed on
//        road-network records: 0 of 4 M pops; 14 of 80 searches of the symmetric circle scenario);
//      * n_pops is recovered exactly: an invalid node was popped by the reference iff its f is below the
//        goal's (an equal f re-runs the search); all nodes are popped when the search exhausts.  pop_hash
//        covers the valid pops only in this discipline (documented in include/pdmpc_b200.h).
//      A search then costs one heap pop per EXPANSION instead of one per created node cheaper than the goal
//      (66 % of the pops of the longest road-network search are invalid nodes), on a queue a third the size.
//
// Hand-over: ONE ring of kRing job descriptors per CTA, shared by the masters.  A master takes a ticket
// (shared-memory atomic), waits until every checker is done with the job that used the ring slot before,
// fills the slot and arrives on the slot's named barrier; the checkers take the tickets in order and wait for
// each in bar.sync (no issue slots are spent spinning).  A job names its search slot; everything a checker
// needs to know about a running search sits in that slot of shared memory.
#pragma once

#include "pdmpc_kernels.cuh"
#include "pdmpc_tiles.cuh"   // sts_f64x2

namespace pdmpc {

constexpr int kRing = 8;            // job descriptors in flight (named barriers 1..kRing)
constexpr int kCtaFlags = 32768;    // node ids with a validity flag (2 bits each) — searches need cap <= this
constexpr int kCtaDepCols = kDepCols;   // columns of predecessors' areas (pdmpc_plan_timestep)
constexpr int kCtaDepPolys = kCtaDepCols / kAreaStride;

struct __align__(16) CtaJob {       // one expansion: children nid0 .. nid0 + nchild - 1 of search slot `slot`
    double px, py, pyaw, c, s;      // pose and cos/sin(yaw) of the expanded node
    unsigned nid0;
    int nchild, sbase, k;           // successor list base, depth of the children
    int terminate;
    int rot;                        // checker that takes child 0; child ci goes to checker (rot + ci) % NC
    int slot;
};

// Everything about ONE running search that lives in shared memory: the master's queue top, the staged
// polylines, the validity flags, and the constants the checkers read.
template <int HS, int SP, bool DEPS>
struct __align__(16) CtaSearch {
    double hf[HS + 2];               // heap costs, entry i at hf[i + 1] (pdmpc_heap_split.cuh)
    unsigned long long hw[HS];       // heap payloads
    double2 pts[SP];                 // staged polylines (x, y): [lanelet bounds][obstacle slots 0..Hp]
    double refx[kMaxHp], refy[kMaxHp];
    double dmax[kMaxHp * kMaxHp];    // [k' * kMaxHp + t] = sum_{tau <= t} dt * v_ref(k' + tau), summed in order (expand_node.m:68)
    unsigned flag2[kCtaFlags / 16];  // 2 bits per node id: 0 pending, 1 valid, 2 invalid
    // pdmpc_plan_timestep: the areas the predecessors of this search have planned, kAreaStride columns each
    // (points, then NaN: the separator column of vectorize_all_obstacles.m:36-63 and padding that no InterX
    // inequality can satisfy); predecessor r at step k sits at ((k - 1) * n_pred + r) * kAreaStride
    double2 dep[DEPS ? kCtaDepCols : 1];
    int dep_n[DEPS ? kCtaDepPolys : 1];   // points of each of them (SAT needs the exact count)
    int dep_cols[kMaxHp + 1];             // real columns per step (statistics only)
    // constants of the running search (written by its master during set-up, read by the checkers)
    const double *gx0, *gy0, *gx1, *gy1;  // polylines that are NOT staged (0: obstacles, 1: lanelet bounds), else null
    const int *slot;                      // SAT: obstacle CSR of the search
    int rng[kMaxHp + 2];
    int nl, sadj, sp0, sp1, lp0, lp1, lp2, n_pred;
    int abort_flag;
    unsigned path[kMaxHp + 1];
};

template <int HS, int SP, int NC, int NM, bool DEPS>
struct __align__(16) CtaSmem {
    CtaSearch<HS, SP, DEPS> S[NM];
    double2 shp[NC][2][kAreaStride];     // a checker's placed areas: [0] normal offset, [1] boundary check
    double ec[NC][2][kAreaStride][4];    // per shape edge: dx1, dy1, S1, -  (InterX.m:63,67)
    CtaJob ring[kRing];
    unsigned done[NC];                   // tickets checker w has completed
    unsigned n_jobs;                     // ticket counter
    unsigned rot;                        // running child count: spreads consecutive jobs over the checkers
    unsigned masters_done;
};

// Ordering between masters and checkers (flags, descriptors live in shared memory; the global data handed
// over is cos/sin of a node, same SM).  An acquire-release fence at CTA scope is enough; __threadfence_block()
// compiles to the sequentially consistent MEMBAR.SC.CTA, which drains the outstanding arena stores.
__device__ __forceinline__ void fence_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int count) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int count) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ unsigned flag_get(const volatile unsigned *f, unsigned id) {
    return (f[id >> 4] >> (2u * (id & 15u))) & 3u;
}
__device__ __forceinline__ void flag_set(unsigned *f, unsigned id, unsigned v) {
    atomicOr(f + (id >> 4), v << (2u * (id & 15u)));
}

// NM masters + NC checkers (+ with a single master: the warps that would share the master's scheduler —
// 4, 8, 12, ... — are left idle, so that its dependent instruction chain never waits for an issue slot behind
// a checker's FP64 stream, profiles/r01e_cta_latency.txt).
template <int NM, int NC>
struct CtaShape {
    static constexpr int kParked = NM == 1 ? NC / 3 - 1 : 0;   // NC = 12: warps 4, 8, 12 of 16
    static constexpr int kWarps = NM + NC + kParked;
    static constexpr int kThreads = kWarps * kWarp;
    static constexpr int kBarThreads = (NC + 1) * kWarp;   // a ticket's named barrier: all checkers + its master
};

template <int HS, int SP, int NC, int NM, bool DEPS = false>
__global__ void __launch_bounds__(CtaShape<NM, NC>::kThreads, 1)
search_cta_kernel(MpaDev m, BatchDev b, OutDev o, ArenaDev ar, unsigned *work_counter, int heap_smem, int fast,
                  DepsDev dp) {
    using Shape = CtaShape<NM, NC>;
    static_assert(NM >= 1 && NC >= 1 && NC <= kWarp, "pool sizes");
    static_assert(NM > 1 || NC % 3 == 0, "single master: three checker warps per scheduler group");
    static_assert(kRing * PDMPC_MAX_TRIMS <= kCtaFlags, "ids in flight");
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int kBarThreads = Shape::kBarThreads;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    CtaSmem<HS, SP, NC, NM, DEPS> &sm = *reinterpret_cast<CtaSmem<HS, SP, NC, NM, DEPS> *>(smem_raw);

    const int warp_id = threadIdx.x / kWarp;
    const int lane = threadIdx.x % kWarp;
    Tile<kWarp> t;
    t.shift = 0; t.lane = lane; t.mask = FULL;
    const int Hp = m.Hp, nT = m.nT;
    volatile unsigned *vdone = sm.done;
    // work items: the batch — or, with b.esc_producers > 0, the escalation list of the tile kernel(s) (BatchDev;
    // they may still be appending to it): master slot s = blockIdx.x + gridDim.x * master takes item s first
    // (a short list puts one search on every SM before any SM gets two), then whatever item is next on the
    // shared ticket counter (S, S + 1, ...; S = gridDim.x * NM).  This instance runs only if the list ends up
    // with esc_gate_lo < count <= esc_gate_hi items (two instances with different NM share one list; the gate
    // is evaluated when the producers are done — until then the instance only waits).
    const bool polling = b.esc_producers > 0u;
    if (polling && threadIdx.x == 0) TAIL_MIN(2);
    if (threadIdx.x < NC) sm.done[threadIdx.x] = 0u;
    if (threadIdx.x == 0) { sm.n_jobs = 0u; sm.rot = 0u; sm.masters_done = 0u; }
    for (int s = 0; s < NM; ++s)
        for (int i = threadIdx.x; i < kCtaFlags / 16; i += Shape::kThreads) sm.S[s].flag2[i] = 0u;
    __syncthreads();

    // ---- roles -----------------------------------------------------------------------------------------
    int role_master = -1, role_checker = -1;
    if (NM == 1) {
        if (warp_id == 0) role_master = 0;
        else if ((warp_id & 3) != 0) role_checker = warp_id - 1 - (warp_id >> 2);
    } else {
        if (warp_id < NM) role_master = warp_id;
        else role_checker = warp_id - NM;
    }
    if (role_master < 0 && role_checker < 0) return;   // parked warp

    if (role_checker >= 0) {
        // =================== checker warps: eval_edge_exact, eagerly ======================================
        const int w = role_checker;
        const unsigned sshp = shared_base_once(sm.shp[w]), sec = shared_base_once(sm.ec[w]);
        unsigned long long cols = 0;
        for (unsigned j = 0;; ++j) {
            named_bar_sync(1 + (int)(j % kRing), kBarThreads);          // ticket j is published
            const CtaJob &jb = sm.ring[j % kRing];
            if (jb.terminate) break;
            CtaSearch<HS, SP, DEPS> &S = sm.S[jb.slot];
            const int nchild = jb.nchild, cK = jb.k;
            if (!*reinterpret_cast<volatile int *>(&S.abort_flag)) {
                const double ppx = jb.px, ppy = jb.py, pc = jb.c, ps = jb.s, pyaw = jb.pyaw;
                const unsigned nid0 = jb.nid0;
                const int sbase = jb.sbase;
                NodeCS *__restrict__ ncs = ar.cs + ((size_t)blockIdx.x * NM + jb.slot) * (size_t)ar.cap;
                const unsigned spts = shared_base_once(S.pts);
                // consecutive expansions start at different checkers: with 3-4 children per expansion a fixed
                // child -> checker map would serialise every job on checkers 0..3
                for (int ci = (w - jb.rot + NC) % NC; ci < nchild; ci += NC) {
                    const int te = m.succ_te[sbase + ci];
                    const int edge = te >> 8;
                    const unsigned nid = nid0 + (unsigned)ci;
                    const int bkind = (cK == Hp) ? PDMPC_AREA_LARGE_OFFSET : PDMPC_AREA_WITHOUT_OFFSET;  // GraphSearch.m:166-174
                    const int ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                    const int nbs = m.area_npts[edge * 3 + bkind];
                    // place both areas by the PARENT pose (GraphSearch.m:155-160); the tail repeats the last vertex
                    if (lane < 16) {
                        const int sel = lane >> 3, i = lane & 7;
                        const int ab = (edge * 3 + (sel ? bkind : PDMPC_AREA_NORMAL)) * kAreaStride + i;   // (padded by the last point)
                        const double ax = m.area_x[ab], ay = m.area_y[ab];
                        sts_f64x2(sshp + 16u * (unsigned)lane, pc * ax - ps * ay + ppx, ps * ax + pc * ay + ppy);
                    }
                    __syncwarp();
                    bool valid = true;
                    if (b.checker == PDMPC_CHECKER_INTERX) {
                        // edge constants of InterX.m:63,67, one edge per lane
                        if (lane < 16) {
                            const int i = lane & 7;
                            const double2 v0 = lds_f64x2(sshp + 16u * (unsigned)lane);
                            const double2 v1 = lds_f64x2(sshp + 16u * (unsigned)((lane & 8) + min(i + 1, 7)));
                            const double dx1 = v1.x - v0.x, dy1 = v1.y - v0.y;
                            sts_f64x2(sec + 32u * (unsigned)lane, dx1, dy1);
                            sts_f64(sec + 32u * (unsigned)lane + 16u, dx1 * v0.y - dy1 * v0.x);
                        }
                        // ONE item list: segments of [static | dynamic of step cK | predecessors' areas of step cK]
                        // against the normal-offset shape, segments of [left, NaN, right, NaN] against the boundary shape
                        const int obase = S.nl;
                        const int st_lo = obase + S.rng[0], st_hi = obase + S.rng[1];
                        const int dy_lo = obase + S.rng[cK], dy_hi = obase + S.rng[cK + 1];
                        const int npred = DEPS ? S.n_pred : 0;
                        const int dp_lo = (cK - 1) * npred * kAreaStride, dp_hi = cK * npred * kAreaStride;
                        cols += (unsigned long long)((st_hi - st_lo) + (dy_hi - dy_lo) + S.nl);
                        if (DEPS) cols += (unsigned long long)S.dep_cols[cK];
                        const int n0 = max(st_hi - st_lo - 1, 0);                 // InterX.m:48-52 and single-column inputs
                        const int n01 = n0 + max(dy_hi - dy_lo - 1, 0);
                        const int n012 = n01 + max(dp_hi - dp_lo - 1, 0);
                        const int ntot = n012 + max(S.nl - 1, 0);
                        const int ne = max(ns, nbs) - 1;
                        const unsigned sdep = DEPS ? shared_base_once(S.dep) : 0u;
                        const double *gx0 = S.gx0, *gy0 = S.gy0, *gx1 = S.gx1, *gy1 = S.gy1;
                        const int sadj = S.sadj;
                        __syncwarp();
                        bool hit = false;
                        for (int e0 = 0; e0 < ntot; e0 += kWarp) {
                            const int e = e0 + lane;
                            if (e < ntot) {
                                const int sel = e >= n012 ? 1 : 0;
                                const bool isdep = DEPS && e >= n01 && e < n012;
                                const int j2 = e < n0 ? st_lo + e
                                                      : (e < n01 ? dy_lo + (e - n0) : (e < n012 ? dp_lo + (e - n01) : e - n012));
                                double2 p0, p1;
                                const double *gxs = sel ? gx1 : gx0;
                                if (isdep) {
                                    p0 = lds_f64x2(sdep + 16u * (unsigned)j2);
                                    p1 = lds_f64x2(sdep + 16u * (unsigned)j2 + 16u);
                                } else if (gxs == nullptr) {
                                    const unsigned pa = spts + 16u * (unsigned)(j2 + (sel ? 0 : sadj));
                                    p0 = lds_f64x2(pa);
                                    p1 = lds_f64x2(pa + 16u);
                                } else {
                                    const double *gys = sel ? gy1 : gy0;
                                    p0 = make_double2(__ldg(gxs + j2), __ldg(gys + j2));
                                    p1 = make_double2(__ldg(gxs + j2 + 1), __ldg(gys + j2 + 1));
                                }
                                const double dx2 = p1.x - p0.x, dy2 = p1.y - p0.y;          // InterX.m:64
                                const double S2 = dx2 * p0.y - dy2 * p0.x;                  // :68
                                const unsigned vb = sshp + 128u * (unsigned)sel;
                                unsigned c2 = m.areas_closed ? interx_c2_dispatch<true>(ne, vb, dx2, dy2, S2)
                                                             : interx_c2_dispatch<false>(ne, vb, dx2, dy2, S2);   // :71
                                while (c2) {                                                // C1 of the edges with C2, :70
                                    const int i = __ffs(c2) - 1;
                                    c2 &= c2 - 1u;
                                    const unsigned eb = sec + 32u * (unsigned)(sel * 8 + i);
                                    const double2 d1 = lds_f64x2(eb);
                                    const double S1 = lds_f64(eb + 16u);
                                    const double a0 = (d1.x * p0.y - d1.y * p0.x) - S1;
                                    const double a1 = (d1.x * p1.y - d1.y * p1.x) - S1;
                                    if (a0 * a1 < 0) hit = true;
                                }
                            }
                            if (__any_sync(FULL, hit)) { valid = false; break; }
                        }
                    } else {
                        // are_constraints_satisfied_sat.m:15-53 on the raw CSR (polygons in HBM/L2); SoA copies of the
                        // placed areas for the SAT routines sit in the (unused) edge-constant block: 4 x 8 doubles
                        double *sx = reinterpret_cast<double *>(sm.ec[w]);
                        double *sy = sx + kAreaStride, *bx = sx + 2 * kAreaStride, *by = sx + 3 * kAreaStride;
                        if (lane < 16) {
                            const double2 v = sm.shp[w][lane >> 3][lane & 7];
                            (lane < 8 ? sx : bx)[lane & 7] = v.x;
                            (lane < 8 ? sy : by)[lane & 7] = v.y;
                        }
                        __syncwarp();
                        const int *slot = S.slot;
                        const int dp0 = __ldg(slot + cK), dp1 = __ldg(slot + cK + 1);
                        for (int pass = 0; pass < 2 && valid; ++pass) {
                            const int q0 = pass == 0 ? S.sp0 : dp0, q1 = pass == 0 ? S.sp1 : dp1;
                            for (int p = q0; p < q1 && valid; ++p) {
                                const int v0 = __ldg(b.poly_ptr + p), v1 = __ldg(b.poly_ptr + p + 1);
                                cols += (unsigned long long)(v1 - v0);
                                if (sat_collide<kWarp>(sx, sy, ns, b.vert_x + v0, b.vert_y + v0, v1 - v0, t))
                                    valid = false;
                            }
                        }
                        if (DEPS) {
                            const int np_ = S.n_pred;
                            for (int r = 0; r < np_ && valid; ++r) {
                                const int pk = (cK - 1) * np_ + r, nv = S.dep_n[pk];
                                if (nv < 2) continue;
                                cols += (unsigned long long)nv;
                                const double *dxy = reinterpret_cast<const double *>(S.dep + pk * kAreaStride);
                                if (sat_collide<kWarp, false, 2>(sx, sy, ns, dxy, dxy + 1, nv, t))
                                    valid = false;
                            }
                        }
                        if (valid) {
                            cols += (unsigned long long)(S.lp2 - S.lp0);
                            if (lanelet_side_sat<kWarp>(bx, by, nbs, b.lane_x + S.lp0, b.lane_y + S.lp0, S.lp1 - S.lp0, t))
                                valid = false;
                            else if (lanelet_side_sat<kWarp>(bx, by, nbs, b.lane_x + S.lp1, b.lane_y + S.lp1, S.lp2 - S.lp1, t))
                                valid = false;
                        }
                    }
                    if (lane == 0) {
                        if (valid && cK < Hp) {
                            // cos/sin of the child's yaw for ITS expansion (expand_node.m:50-51);
                            // yaw' = yaw + dyaw exactly as the master computes it (:55)
                            NodeCS ecs;
                            sincos_ref(pyaw + m.edge_d[edge * 4 + 2], ecs.s, ecs.c);
                            ncs[nid] = ecs;
                        }
                        fence_cta();
                        flag_set(S.flag2, nid, valid ? 1u : 2u);
                    }
                    __syncwarp();   // the shapes are rewritten by the next child
                }
            }
            __syncwarp();   // every lane is done with the descriptor
            if (lane == 0) { fence_cta(); vdone[w] = j + 1u; }
        }
        if (lane == 0 && cols) atomicAdd(o.counters + 2, cols);
        return;
    }

    // =================== master warp: queue + tree of ONE search at a time ==================================
    const int ms = role_master;
    CtaSearch<HS, SP, DEPS> &S = sm.S[ms];
    const size_t slot_base = ((size_t)blockIdx.x * NM + ms) * (size_t)ar.cap;
    NodeA *__restrict__ na = ar.a + slot_base;
    NodeB *__restrict__ nb = ar.b + slot_base;
    NodeCS *__restrict__ ncs = ar.cs + slot_base;
    volatile unsigned *vflag = S.flag2;
    const unsigned hf_addr = shared_base_once(S.hf), hw_addr = shared_base_once(S.hw);
    int clear_upto = 0;            // highest node id of the previous search (flags to clear)
    bool redo_exact = false;
    PROF_DECL
    unsigned si_u = 0;
    unsigned next_item = blockIdx.x + gridDim.x * (unsigned)role_master;   // escalation list: this master's first item
    bool first_item = true;

    unsigned my_jobs = 0, my_rot = 0;   // NM == 1: ticket and child counters of the only master
    // publish one job (an expansion, or the terminate order) on the shared ring; returns its ticket
    auto publish = [&](const NodeA &ca, double c, double s, unsigned nid0, int nchild, int sbase, int k,
                       int terminate) -> unsigned {
        unsigned tk = 0, rt = 0;
        if (NM == 1) {   // the only producer: its tickets need no atomics
            tk = my_jobs++;
            rt = my_rot;
            my_rot += (unsigned)max(nchild, 0);
        } else {
            if (lane == 0) {
                tk = atomicAdd(&sm.n_jobs, 1u);
                rt = atomicAdd(&sm.rot, (unsigned)max(nchild, 0));
            }
            tk = __shfl_sync(FULL, tk, 0);
            rt = __shfl_sync(FULL, rt, 0);
        }
        while (true) {   // ring slot free: every checker is done with ticket tk - kRing
            const unsigned d = lane < NC ? vdone[lane] : tk;
            if (__all_sync(FULL, d + kRing > tk)) break;
        }
        fence_cta();
        if (lane == 0) {
            CtaJob &jb = sm.ring[tk % kRing];
            jb.px = ca.x; jb.py = ca.y; jb.pyaw = ca.yaw; jb.c = c; jb.s = s;
            jb.nid0 = nid0; jb.nchild = nchild; jb.sbase = sbase; jb.k = k;
            jb.terminate = terminate; jb.rot = (int)(rt % NC); jb.slot = ms;
        }
        // (no fence: the barrier orders the descriptor against the checkers that wait in bar.sync on it)
        __syncwarp();
        named_bar_arrive(1 + (int)(tk % kRing), kBarThreads);
        return tk;
    };

    for (;;) {
        // ---- fetch a search (or run the same one again with the exact queue); set-up by this warp -----------
        bool exact;
        const bool exact_again = redo_exact;
        if (redo_exact) { redo_exact = false; exact = true; }
        else {
            if (!polling) {
                if (lane == 0) si_u = atomicAdd(work_counter, 1u);
                si_u = __shfl_sync(FULL, si_u, 0);
            }
            exact = fast == 0;
        }
        int si;
        if (polling) {
            if (!exact_again) {
                int got = -1;
                if (lane == 0) {
                    const int *cnt = reinterpret_cast<const int *>(b.esc_count);
                    // the gate needs the final count: wait for the producers (same stream: they are done)
                    while (ld_acquire_gpu(reinterpret_cast<const int *>(b.esc_done)) < (int)b.esc_producers) __nanosleep(2000);
                    const int n_full = ld_acquire_gpu(cnt), total = n_full + ld_acquire_gpu(cnt + 2);
                    if ((unsigned)total > b.esc_gate_lo && (unsigned)total <= b.esc_gate_hi) {
                        if (!first_item) next_item = atomicAdd(work_counter, 1u) + gridDim.x * NM;
                        if ((int)next_item < total) {
                            const int *e = esc_item(b.esc_list, b.esc_cap, (unsigned)n_full, next_item);
                            while ((got = ld_acquire_gpu(e)) < 0) __nanosleep(200);
                        }
                    }
                }
                first_item = false;
                got = __shfl_sync(FULL, got, 0);
                if (got < 0) break;
                si_u = (unsigned)got;
                if (lane == 0 && o.counters) atomicAdd(o.counters + 6, 1ULL);
            }
            si = (int)si_u;
        } else {
            if (si_u >= (unsigned)b.n) break;
            si = b.order ? __ldg(b.order + si_u) : (int)si_u;
        }
        for (int i = lane; i <= clear_upto / 16; i += kWarp) S.flag2[i] = 0u;
        stage_reference(b, si, Hp, S.refx, S.refy, nullptr, t);
        if (lane >= 1 && lane < Hp) {   // d_traveled_max of expand_node.m:68 for children of step k'
            double d = 0.0;
            for (int it = 1; it <= Hp - lane; ++it) {
                d = d + b.dt * __ldg(b.v_ref + (size_t)si * Hp + lane + it - 1);
                S.dmax[lane * kMaxHp + it] = d;
            }
        }
        const int *slot = b.slot_ptr + (size_t)si * (Hp + 1);
        const int trim0 = __ldg(b.trim0 + si);
        if (lane == 0) {
            S.slot = slot;
            S.sp0 = __ldg(slot + 0); S.sp1 = __ldg(slot + 1);
            S.lp0 = __ldg(b.lane_ptr + 2 * si); S.lp1 = __ldg(b.lane_ptr + 2 * si + 1); S.lp2 = __ldg(b.lane_ptr + 2 * si + 2);
            S.abort_flag = 0;
            S.n_pred = 0;
            S.gx0 = S.gy0 = S.gx1 = S.gy1 = nullptr;
            S.nl = 0; S.sadj = 0;
        }
        if (lane <= Hp) S.dep_cols[lane] = 0;
        __syncwarp();
        if (b.checker == PDMPC_CHECKER_INTERX) {
            // polyline layout (vectorize_all_obstacles.m:27-63) as if everything were staged: lanelets
            // [left, NaN, right, NaN] at [0, nl), obstacle slot s at nl + rng[s]
            const SearchPolylines pl = search_polylines(b, si, Hp, S.rng, t);
            const int ll_lo = pl.ll_lo, ob_lo = pl.ob_lo;
            const int nl = pl.ll_hi - ll_lo, no = pl.ob_hi - ob_lo;
            const bool lst = nl <= SP, ost = (lst ? nl : 0) + no <= SP;
            if (lst)
                for (int j = lane; j < nl; j += kWarp)
                    S.pts[j] = make_double2(__ldg(b.ll_x + ll_lo + j), __ldg(b.ll_y + ll_lo + j));
            if (ost)
                for (int j = lane; j < no; j += kWarp)
                    S.pts[(lst ? nl : 0) + j] = make_double2(__ldg(b.pl_x + ob_lo + j), __ldg(b.pl_y + ob_lo + j));
            if (lane == 0) {
                S.nl = nl;
                S.sadj = lst ? 0 : -nl;
                S.gx1 = lst ? nullptr : b.ll_x + ll_lo; S.gy1 = lst ? nullptr : b.ll_y + ll_lo;
                S.gx0 = ost ? nullptr : b.pl_x + (ob_lo - nl); S.gy0 = ost ? nullptr : b.pl_y + (ob_lo - nl);
            }
        }
        // (everything above is independent of the predecessors: it overlaps their searches)
        if (DEPS) {
            // Work items are handed out in a topological order of the DAG (the host sorts them), so every
            // predecessor's ticket is below this one's: it is finished or running on another master, never
            // waiting behind this one.
            const int npred = gather_predecessor_areas(
                dp, o, si, Hp, 100, t, [&](int idx, double x, double y) { S.dep[idx] = make_double2(x, y); },
                [&](int pk, int k0, int np) {
                    S.dep_n[pk] = np;
                    if (np) atomicAdd(&S.dep_cols[k0 + 1], np + 1);
                });
            if (lane == 0) S.n_pred = npred;
        }

        HeapSplit heap;
        heap.sf = hf_addr; heap.sw = hw_addr;
        heap.gl = ar.heap + slot_base;
        heap.hs = min(heap_smem, HS);   // smaller values only exercise the arena overflow (tests)
        heap.len = 1;
        int n_nodes = 1, n_pops = 0, status = PDMPC_OK;
        unsigned long long hash = kHashSeed;
        bool exhausted = false, tie = false;
        unsigned goal = 0, last_ticket = 0;
        bool any_job = false;
        double f_last = 0.0;
        // valid-only queue: children whose flag is not known yet, one per lane
        bool pocc = false;
        double pf = 0.0;
        unsigned long long pw = 0;
        // flags of the pending children: valid -> pushed, invalid -> dropped (cost parked in the unused cos/sin
        // record for the n_pops accounting).  Blocks while a child that could be the next pop has no answer.
        auto resolve_pending = [&](bool wait_all) {
            for (;;) {
                const unsigned pid_ = (unsigned)(pw & 0x1fffffu);
                const unsigned fl = pocc ? flag_get(vflag, pid_) : 0u;
                fence_cta();
                if (pocc && fl == 2u) { NodeCS park; park.c = pf; park.s = 0.0; ncs[pid_] = park; pocc = false; }
                const bool okv = pocc && fl == 1u;
                const unsigned vm = __ballot_sync(FULL, okv);
                if (vm) {
                    const int mv = __popc(vm);
                    unsigned mm = vm;
                    for (int i = 0; i < lane && i < mv; ++i) mm &= mm - 1u;
                    const int src = lane < mv ? __ffs(mm) - 1 : 0;
                    HEnt hv;
                    hv.f = __shfl_sync(FULL, pf, src);
                    hv.w = __shfl_sync(FULL, pw, src);
                    heap.push_many(hv, mv, lane);
                    if (okv) pocc = false;
                }
                // only a pending child whose cost is not above the queue's minimum can be the next pop
                const bool some = heap.len > 0;
                const double thr = some ? heap.f_at(0) : 0.0;
                const bool must = pocc && (wait_all || !some || !(pf > thr));
                if (!__any_sync(FULL, must)) break;
                __nanosleep(20);
            }
        };
        if (lane == 0) heap.st(0, init_root(b, si, trim0, na, nb, ncs));
        __threadfence_block();
        __syncwarp();

        PROF_MARK(0);   // fetch + set-up
        for (;;) {   // GraphSearch.m:53-107
            if (!exact) resolve_pending(false);
            PROF_MARK(1);   // pending children: flags, pushes of the valid ones, waits
            if (heap.len == 0) { exhausted = true; break; }               // :57-61 (no pending child is left either)
            if (!exact && !heap.min_is_unique()) { tie = true; break; }   // tie mechanics would matter: re-run exact
            // the node about to be popped: fetch its records now, their latency hides behind the heap walk
            // (valid-only queue: it is valid and its records are complete; exact queue: cos/sin may not be
            // there yet and is fetched again after the flag)
            const unsigned long long w0 = lds_u64(heap.sw);
            const unsigned id0 = (unsigned)(w0 & 0x1fffffu);
            const int k0 = (int)((w0 >> 52) & 0x1fu), tr0 = (int)(w0 >> 57) + 1;
            // (L2 loads: the checkers' cos/sin stores come from other warps of this SM, never rely on L1)
            const double2 a0 = __ldcg(reinterpret_cast<const double2 *>(na + id0));
            const double2 a1 = __ldcg(reinterpret_cast<const double2 *>(na + id0) + 1);
            double2 cs0 = __ldcg(reinterpret_cast<const double2 *>(ncs + id0));
            int sbase = 0, nchild = 0;
            if (k0 < Hp) {
                sbase = m.succ_ptr[k0 * nT + (tr0 - 1)];
                nchild = m.succ_ptr[k0 * nT + (tr0 - 1) + 1] - sbase;
            }
            const HEnt top = heap.pop<true>(lane);
            PROF_MARK(2);   // early loads + heap pop
            const unsigned id = top.id(), par = top.pid();
            const int cK = (int)top.k();
            ++n_pops;
            if (!fast) hash = hash_step(hash, id);   // shape 4: every pop; shape 5: valid pops only (below)
            f_last = top.f;
            if (exact && par != 0) {   // eval_edge_exact's answer, computed by a checker warp
                unsigned f;
                do { f = flag_get(vflag, id); } while (f == 0u);
                fence_cta();
                if (f != 1u) continue;                                    // :75-77
                cs0 = __ldcg(reinterpret_cast<const double2 *>(ncs + id));
            }
            if (fast) hash = hash_step(hash, id);
            if (cK == Hp) { goal = id; break; }                           // :81-90

            // ---- expand_node.m:1-91 (nV == 1) ----------------------------------------------
            const int k_exp = cK + 1;
            if (n_nodes + nchild >= ar.cap || n_nodes + nchild >= kCtaFlags) { status = PDMPC_ERR_CAPACITY; break; }
            NodeA ca;
            ca.x = a0.x; ca.y = a0.y; ca.yaw = a1.x; ca.g = a1.y;
            const double c = cs0.x, s = cs0.y;
            // publish the job first: the checkers work while the master computes costs and pushes
            PROF_MARK(3);   // flag wait (exact queue), record use
            last_ticket = publish(ca, c, s, (unsigned)(n_nodes + 1), nchild, sbase, k_exp, 0);
            any_job = true;
            PROF_MARK(4);   // job hand-over
            const int to_go = Hp - k_exp;               // :37
            for (int c0 = 0; c0 < nchild; c0 += kWarp) {
                const int ci = c0 + lane;
                const int cnt = min(kWarp, nchild - c0);
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
                    const double ddx = ea.x - S.refx[k_exp - 1], ddy = ea.y - S.refy[k_exp - 1];
                    const double nrm = sqrt(ddx * ddx + ddy * ddy);
                    ea.g = ca.g + nrm * nrm;            // :61
                    double eh = 0.0;                    // :66-73
                    for (int it0 = 1; it0 <= to_go; it0 += 6) {
                        double hn[6];                   // independent square roots, issued together
#pragma unroll
                        for (int u = 0; u < 6; ++u) {
                            const int kk = min(k_exp + it0 + u - 1, Hp - 1);
                            const double hx = ea.x - S.refx[kk], hy = ea.y - S.refy[kk];
                            hn[u] = sqrt(hx * hx + hy * hy);
                        }
#pragma unroll
                        for (int u = 0; u < 6; ++u) {
                            if (it0 + u <= to_go) {
                                const double mm = fmax(0.0, hn[u] - S.dmax[k_exp * kMaxHp + it0 + u]);
                                eh = eh + mm * mm;
                            }
                        }
                    }
                    NodeB eb;
                    eb.h = eh; eb.parent = id; eb.edge = (unsigned short)cedge;
                    eb.trim = (unsigned char)t2; eb.k = (unsigned char)k_exp;
                    na[nid] = ea;                       // Tree.m:54-70 add_nodes
                    nb[nid] = eb;
                    he.f = ea.g + eh;                   // GraphSearch.m:102 (weights 1)
                    he.w = HEnt::pack(nid, id, (unsigned)cedge, (unsigned)k_exp, (unsigned)t2);
                }
                PROF_MARK(5);   // children: poses, costs, records
                if (exact) {
                    heap.push_many(he, cnt, lane);      // :104, one push per child, in order
                } else {
                    // valid-only queue: the children wait in the pending buffer for their flags
                    while (__popc(__ballot_sync(FULL, !pocc)) < cnt) resolve_pending(true);
                    const unsigned freem = __ballot_sync(FULL, !pocc);
                    const int r = __popc(freem & ((1u << lane) - 1u));   // this lane's rank among the free lanes
                    const double nf = __shfl_sync(FULL, he.f, r & 31);
                    const unsigned long long nw = __shfl_sync(FULL, he.w, r & 31);
                    if (!pocc && r < cnt) { pocc = true; pf = nf; pw = nw; }
                }
                PROF_MARK(6);   // pushes / pending insertion
            }
            n_nodes += nchild;
        }
        PROF_MARK(7);

        // ---- let the checkers finish this search's jobs, then write the results (GraphSearch.m:58-60 / :82-89)
        const bool account = !exact && !tie && status == PDMPC_OK;
        if (!account && lane == 0) *reinterpret_cast<volatile int *>(&S.abort_flag) = 1;   // nobody needs the rest
        if (any_job) {
            // (valid-only queue: the n_pops accounting needs the flag of every node cheaper than the goal; in
            // every case no checker may touch this slot once the next search is set up in it)
            while (true) {
                const unsigned d = lane < NC ? vdone[lane] : last_ticket + 1u;
                if (__all_sync(FULL, d > last_ticket)) break;
                __nanosleep(32);
            }
            fence_cta();
        }
        if (status != PDMPC_OK) exhausted = true;
        if (account) {
            resolve_pending(true);
            // pops of the reference's queue = valid pops + the invalid nodes it met on the way:
            // all of them if the search exhausted, those cheaper than the goal otherwise
            int extra = 0;
            bool amb = false;
            for (int i0 = 2; i0 <= n_nodes; i0 += kWarp) {
                const int i = i0 + lane;
                if (i <= n_nodes && flag_get(vflag, (unsigned)i) == 2u) {
                    if (exhausted) ++extra;
                    else {
                        const double fi = __ldcg(reinterpret_cast<const double *>(ncs + i));
                        if (fi < f_last) ++extra;
                        else if (fi == f_last) amb = true;
                    }
                }
            }
            for (int d = 16; d > 0; d >>= 1) extra += __shfl_xor_sync(FULL, extra, d);
            if (__any_sync(FULL, amb)) tie = true;
            n_pops += extra;
        }
        PROF_MARK(7);   // wait for the checkers, accounting
        PROF_FLUSH(o, lane == 0);
        clear_upto = n_nodes;
        if (tie) {   // undecidable without the reference's tie mechanics: same search again, exact queue
            if (lane == 0) atomicAdd(o.counters + 3, 1ULL);
            redo_exact = true;
            continue;
        }
        // (the checkers count the obstacle columns)
        write_search_result(m, o, na, nb, ncs, S.path, si, trim0, goal, status, exhausted, n_nodes, n_pops, hash, 0ull,
                            true, DEPS ? dp.done : nullptr, t);
    }
    // ---- the last master to run out of work releases the checkers -----------------------------------------
    unsigned fin = 0;
    if (polling && lane == 0) TAIL_MAX(3);
    if (lane == 0) fin = atomicAdd(&sm.masters_done, 1u);
    fin = __shfl_sync(FULL, fin, 0);
    if (fin == NM - 1) {
        NodeA z = {0.0, 0.0, 0.0, 0.0};
        publish(z, 0.0, 0.0, 0u, 0, 0, 0, 1);
    }
}

}  // namespace pdmpc
