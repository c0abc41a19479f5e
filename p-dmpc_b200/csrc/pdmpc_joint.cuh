// pdmpc_joint.cuh — centralized (joint) graph search: GraphSearch.do_graph_search with iter.amount = nV > 1.
//
//   CentralizedController.controller                 hlc/controller/centralized/CentralizedController.m:33-59
//   expand_node (Cartesian product of successors)    hlc/optimizer/graph_search/expand_node.m:15-26 (cartprod: first
//                                                    vehicle fastest), costs summed over the vehicles in order :43-75
//   eval_edge_exact (vehicles in order)              hlc/optimizer/graph_search/GraphSearch.m:150-192
//   are_constraints_satisfied_sat                    .../are_constraints_satisfied_sat.m:15-53 (static obstacles, dynamic
//                                                    obstacles of the step, vehicles i < iVeh of the same node, own lanelets)
//   priority queue, goal test, path extraction       as in pdmpc_kernels.cuh
//
// Rows of the batch are (search, vehicle): r = search * nV + v; the obstacle slots of a search are those of its
// vehicle-0 row.  One warp per search.  A node is nV vehicle records (pose, cos/sin of the yaw, trim, the maneuver that
// led to it) plus one shared record (g, h, parent, k) in an HBM arena; branching is the product of the vehicles'
// successor counts (up to 12^nV), so the children of an expansion are generated 32 at a time, one per lane, and pushed
// in order.  The edge check of a popped node runs the vehicles one after the other, each vehicle's SAT tests spread over
// the lanes (axes), and stops at the first failure, as the reference does.
#pragma once

#include "pdmpc_kernels.cuh"

namespace pdmpc {

constexpr int kMaxJoint = PDMPC_MAX_JOINT;
constexpr int kJointHeap = 6144;  // heap entries in shared memory per search (100 KB: two searches per SM); joint
                                  // queues hold 10^4..10^6 entries, every level kept out of HBM shortens the pop chain
// Joint trees are large (up to 12^nV children per expansion): heap payload = node id in 28 bits | depth << 52; the
// parent is read from the node record.
constexpr int kJointMaxCap = (1 << 28) - 1;
__device__ __forceinline__ unsigned long long jpack(unsigned id, unsigned k) {
    return (unsigned long long)id | ((unsigned long long)k << 52);
}

struct __align__(16) JVeh {       // 48 B per (node, vehicle)
    double x, y, yaw, c, s;
    unsigned short edge;          // maneuver that led to this node (0xffff: root)
    unsigned char trim, pad;
    unsigned pad2;
};
struct __align__(16) JNode {      // 32 B per node
    double g, h;
    unsigned parent;
    int k;
    unsigned long long pad;
};
struct JointArena {
    JVeh *veh;                    // [slots * cap * nV]
    JNode *node;                  // [slots * cap]
    HEnt *heap;                   // [slots * cap] overflow of the shared-memory heap
    int cap, nV;
};

struct __align__(16) JointSmem {
    double hf[kJointHeap + 2];
    unsigned long long hw[kJointHeap];
    double refx[kMaxJoint][kMaxHp], refy[kMaxJoint][kMaxHp], vref[kMaxJoint][kMaxHp];
    double shx[kMaxJoint][kAreaStride], shy[kMaxJoint][kAreaStride];
    double bhx[kMaxJoint][kAreaStride], bhy[kMaxJoint][kAreaStride];
    int edge_of[kMaxJoint];
    unsigned path[kMaxHp + 1];
};

__global__ void __launch_bounds__(kWarp) joint_search_kernel(MpaDev m, BatchDev b, OutDev o, JointArena ar, unsigned *work_counter) {
    constexpr int TILE = kWarp;
    extern __shared__ __align__(16) unsigned char joint_smem_raw[];
    JointSmem &sm = *reinterpret_cast<JointSmem *>(joint_smem_raw);
    Tile<TILE> t;
    t.shift = 0; t.lane = threadIdx.x; t.mask = 0xffffffffu;
    const int Hp = m.Hp, nT = m.nT, nV = ar.nV;
    const int n_joint = b.n / nV;
    JVeh *__restrict__ nv = ar.veh + (size_t)blockIdx.x * ar.cap * nV;
    JNode *__restrict__ nn = ar.node + (size_t)blockIdx.x * ar.cap;
    HeapSplit heap;
    heap.sf = shared_base_once(sm.hf);
    heap.sw = shared_base_once(sm.hw);
    heap.gl = ar.heap + (size_t)blockIdx.x * ar.cap;
    heap.hs = kJointHeap;

    for (;;) {
        unsigned su = 0;
        if (t.lane == 0) su = atomicAdd(work_counter, 1u);
        su = t.shfl(su, 0);
        if (su >= (unsigned)n_joint) break;
        const int r0 = (int)su * nV;
        t.sync();
        for (int i = t.lane; i < nV * Hp; i += TILE) {
            const int v = i / Hp, k = i % Hp;
            sm.refx[v][k] = __ldg(b.ref_x + (size_t)(r0 + v) * Hp + k);
            sm.refy[v][k] = __ldg(b.ref_y + (size_t)(r0 + v) * Hp + k);
            sm.vref[v][k] = __ldg(b.v_ref + (size_t)(r0 + v) * Hp + k);
        }
        if (t.lane < nV) {   // root: GraphSearch.m:34-46
            JVeh rv;
            rv.x = __ldg(b.x0 + r0 + t.lane); rv.y = __ldg(b.y0 + r0 + t.lane); rv.yaw = __ldg(b.yaw0 + r0 + t.lane);
            sincos_ref(rv.yaw, rv.s, rv.c);
            rv.edge = 0xffff; rv.trim = (unsigned char)__ldg(b.trim0 + r0 + t.lane); rv.pad = 0; rv.pad2 = 0;
            nv[(size_t)1 * nV + t.lane] = rv;
        }
        if (t.lane == 0) {
            JNode rn;
            rn.g = 0.0; rn.h = 0.0; rn.parent = 0; rn.k = 0; rn.pad = 0;
            nn[1] = rn;
            HEnt re;
            re.f = 0.0; re.w = jpack(1u, 0u);
            heap.st(0, re);
        }
        heap.len = 1;
        const int *slot = b.slot_ptr + (size_t)r0 * (Hp + 1);
        int n_nodes = 1, n_pops = 0, status = PDMPC_OK;
        unsigned long long hash = kHashSeed, cols = 0;
        bool exhausted = false;
        unsigned goal = 0;
        __threadfence_block();
        t.sync();

        for (;;) {   // GraphSearch.m:53-107
            if (heap.len == 0) { exhausted = true; break; }
            const HEnt top = heap.pop(t.lane);
            const unsigned id = (unsigned)(top.w & 0xfffffffULL);
            const int cK = (int)((top.w >> 52) & 0x1fULL);
            const JNode cn = nn[id];
            const unsigned par = cn.parent;
            ++n_pops;
            if (!b.hash_valid_only) hash = hash_step(hash, id);
            bool valid = true;
            if (par != 0) {   // eval_edge_exact, GraphSearch.m:150-192
                const int sp0 = __ldg(slot + 0), sp1 = __ldg(slot + 1), dp0 = __ldg(slot + cK), dp1 = __ldg(slot + cK + 1);
                const int bkind = (cK == Hp) ? PDMPC_AREA_LARGE_OFFSET : PDMPC_AREA_WITHOUT_OFFSET;
                {   // all vehicles' records in ONE round of loads, all areas placed together (8 lanes per vehicle);
                    // whether an edge is valid does not depend on the order in which its shapes are computed
                    const int pv_i = t.lane / kAreaStride, pt_i = t.lane % kAreaStride;
                    if (pv_i < nV) {
                        const JVeh pv = nv[(size_t)par * nV + pv_i];
                        const int edge = (int)nv[(size_t)id * nV + pv_i].edge;
                        place_point(m, edge, PDMPC_AREA_NORMAL, pt_i, pv.c, pv.s, pv.x, pv.y, sm.shx[pv_i][pt_i], sm.shy[pv_i][pt_i]);
                        place_point(m, edge, bkind, pt_i, pv.c, pv.s, pv.x, pv.y, sm.bhx[pv_i][pt_i], sm.bhy[pv_i][pt_i]);
                        if (pt_i == 0) sm.edge_of[pv_i] = edge;
                    }
                    t.sync();
                }
                for (int v = 0; v < nV && valid; ++v) {
                    const int edge = sm.edge_of[v];
                    const int ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                    const int nbs = m.area_npts[edge * 3 + bkind];
                    // are_constraints_satisfied_sat.m:15-35: static obstacles, dynamic obstacles of this step
                    for (int pass = 0; pass < 2 && valid; ++pass) {
                        const int q0 = pass == 0 ? sp0 : dp0, q1 = pass == 0 ? sp1 : dp1;
                        for (int p = q0; p < q1 && valid; ++p) {
                            const int v0 = __ldg(b.poly_ptr + p), v1 = __ldg(b.poly_ptr + p + 1);
                            cols += (unsigned long long)(v1 - v0);
                            if (sat_collide<TILE>(sm.shx[v], sm.shy[v], ns, b.vert_x + v0, b.vert_y + v0, v1 - v0, t)) valid = false;
                        }
                    }
                    // :37-44 vehicles of the same node with a lower index
                    for (int u = v - 1; u >= 0 && valid; --u) {
                        const int eu = sm.edge_of[u];
                        const int nsu = m.area_npts[eu * 3 + PDMPC_AREA_NORMAL];
                        cols += (unsigned long long)nsu;
                        if (sat_collide<TILE, false>(sm.shx[u], sm.shy[u], nsu, sm.shx[v], sm.shy[v], ns, t)) valid = false;
                    }
                    if (valid) {   // :46-53 own lanelet boundary
                        const int r = r0 + v;
                        const int lp0 = __ldg(b.lane_ptr + 2 * r), lp1 = __ldg(b.lane_ptr + 2 * r + 1), lp2 = __ldg(b.lane_ptr + 2 * r + 2);
                        cols += (unsigned long long)(lp2 - lp0);
                        if (lanelet_side_sat<TILE>(sm.bhx[v], sm.bhy[v], nbs, b.lane_x + lp0, b.lane_y + lp0, lp1 - lp0, t)) valid = false;
                        else if (lanelet_side_sat<TILE>(sm.bhx[v], sm.bhy[v], nbs, b.lane_x + lp1, b.lane_y + lp1, lp2 - lp1, t)) valid = false;
                    }
                }
            }
            if (!valid) continue;                         // :75-77
            if (b.hash_valid_only) hash = hash_step(hash, id);
            if (cK == Hp) { goal = id; break; }           // :81-90

            // ---- expand_node.m -----------------------------------------------------------------
            const int k_exp = cK + 1;
            JVeh cv[kMaxJoint];
            int sbase[kMaxJoint], nsucc[kMaxJoint];
            long long total = 1;
#pragma unroll
            for (int v = 0; v < kMaxJoint; ++v) {
                if (v < nV) {
                    cv[v] = nv[(size_t)id * nV + v];
                    sbase[v] = m.succ_ptr[(k_exp - 1) * nT + ((int)cv[v].trim - 1)];
                    nsucc[v] = m.succ_ptr[(k_exp - 1) * nT + ((int)cv[v].trim - 1) + 1] - sbase[v];
                    total *= nsucc[v];
                }
            }
            if ((long long)n_nodes + total >= (long long)ar.cap) { status = PDMPC_ERR_CAPACITY; break; }
            const int to_go = Hp - k_exp;
            for (long long c0 = 0; c0 < total; c0 += TILE) {
                const long long ci = c0 + t.lane;
                const int cnt = (int)min((long long)TILE, total - c0);
                HEnt he;
                he.f = 0.0; he.w = 0;
                if (ci < total) {
                    const unsigned nid = (unsigned)(n_nodes + 1 + ci);
                    long long rem = ci;
                    double eg = cn.g, eh = 0.0;
#pragma unroll
                    for (int v = 0; v < kMaxJoint; ++v) {
                        if (v < nV) {
                            const int iv = (int)(rem % nsucc[v]);   // cartprod: first vehicle fastest
                            rem /= nsucc[v];
                            const int te = m.succ_te[sbase[v] + iv];
                            const int cedge = te >> 8, t2 = (te & 0xff) + 1;
                            const double mdx = m.edge_d[cedge * 4 + 0], mdy = m.edge_d[cedge * 4 + 1], mdyaw = m.edge_d[cedge * 4 + 2];
                            JVeh ev;
                            ev.x = cv[v].c * mdx - cv[v].s * mdy + cv[v].x;      // :53
                            ev.y = cv[v].s * mdx + cv[v].c * mdy + cv[v].y;      // :54
                            ev.yaw = cv[v].yaw + mdyaw;                          // :55
                            const double ddx = ev.x - sm.refx[v][k_exp - 1], ddy = ev.y - sm.refy[v][k_exp - 1];
                            const double nrm = sqrt(ddx * ddx + ddy * ddy);
                            eg = eg + nrm * nrm;                                 // :61
                            double d_max = 0.0;
                            for (int it = 1; it <= to_go; ++it) {                // :66-73
                                d_max = d_max + b.dt * sm.vref[v][k_exp + it - 1];
                                const double hx = ev.x - sm.refx[v][k_exp + it - 1], hy = ev.y - sm.refy[v][k_exp + it - 1];
                                const double mm = fmax(0.0, sqrt(hx * hx + hy * hy) - d_max);
                                eh = eh + mm * mm;
                            }
                            sincos_ref(ev.yaw, ev.s, ev.c);
                            ev.edge = (unsigned short)cedge; ev.trim = (unsigned char)t2; ev.pad = 0; ev.pad2 = 0;
                            nv[(size_t)nid * nV + v] = ev;
                        }
                    }
                    JNode en;
                    en.g = eg; en.h = eh; en.parent = id; en.k = k_exp; en.pad = 0;
                    nn[nid] = en;
                    he.f = eg + eh;                                             // GraphSearch.m:102
                    he.w = jpack(nid, (unsigned)k_exp);
                }
                __threadfence_block();
                heap.push_many(he, cnt, t.lane);                                // :104, in order
            }
            n_nodes += (int)total;
            t.sync();
        }

        // ---- results, row-wise (every vehicle of the search carries the shared fields) -------------
        if (status != PDMPC_OK) exhausted = true;
        if (t.lane == 0) {
            unsigned cur = goal;
            for (int d = Hp; d >= 0; --d) {
                sm.path[d] = exhausted ? 0u : cur;
                if (!exhausted && d > 0) cur = nn[cur].parent;
            }
            atomicAdd(o.counters + 0, (unsigned long long)n_pops);
            atomicAdd(o.counters + 1, (unsigned long long)n_nodes);
            atomicAdd(o.counters + 2, cols);
        }
        t.sync();
        const double qnan = nan("");
        for (int v = 0; v < nV; ++v) {
            const int r = r0 + v;
            if (t.lane == 0) {
                o.status[r] = status;
                o.is_exhausted[r] = exhausted ? 1 : 0;
                o.n_expanded[r] = n_nodes;
                o.n_pops[r] = n_pops;
                o.pop_hash[r] = hash;
            }
            for (int d = t.lane; d <= Hp; d += TILE) {
                const unsigned pid = sm.path[d];
                const size_t oo = (size_t)r * (Hp + 1) + d;
                JVeh pv;
                JNode pn;
                pv.x = pv.y = pv.yaw = qnan; pv.trim = 0; pv.edge = 0;
                pn.g = pn.h = qnan;
                if (!exhausted) { pv = nv[(size_t)pid * nV + v]; pn = nn[pid]; }
                o.trims[oo] = exhausted ? (d == 0 ? __ldg(b.trim0 + r) : 0) : (int)pv.trim;
                o.tree_path[oo] = (int)pid;
                o.g_path[oo] = pn.g;
                o.h_path[oo] = pn.h;
                if (d >= 1) {
                    const size_t os = (size_t)r * Hp + (d - 1);
                    o.y_predicted[os * 3 + 0] = pv.x;
                    o.y_predicted[os * 3 + 1] = pv.y;
                    o.y_predicted[os * 3 + 2] = pv.yaw;
                    int ns = 0, edge = 0;
                    JVeh qv;
                    qv.x = qv.y = qv.c = qv.s = 0.0;
                    if (!exhausted) {
                        qv = nv[(size_t)sm.path[d - 1] * nV + v];
                        edge = (int)pv.edge;
                        ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                    }
                    o.shape_npts[os] = ns;
                    for (int i = 0; i < kAreaStride; ++i) {
                        double ox = 0.0, oy = 0.0;
                        if (i < ns) place_point(m, edge, PDMPC_AREA_NORMAL, i, qv.c, qv.s, qv.x, qv.y, ox, oy);
                        o.shape_x[os * kAreaStride + i] = ox;
                        o.shape_y[os * kAreaStride + i] = oy;
                    }
                }
            }
        }
        t.sync();
    }
}

}  // namespace pdmpc
