// pdmpc_mcts.cuh — device code of the sampled optimizer (OptimizerType.MatlabSampled).
//
//   MonteCarloTreeSearch.run_optimizer / do_graph_search
//       hlc/optimizer/graph_search/MonteCarloTreeSearch.m:29-251
//   random stream: rand(RandStream('mt19937ar', Seed = time_step + vehicle_index), 1, Hp * n_max)
//       (:31,52) = MT19937 (init_genrand / genrand_int32) + genrand_res53
//
// One warp per search, everything of the search in shared memory (the sampled tree has at
// most n_expansions_max + Hp nodes).  The roll-out is a serial walk, executed uniformly by
// the warp: lanes 0..15 hold one column of the reference's `children` matrix, a ballot is
// `find(children(:, node))`, the ceil(r * n)-th set bit is the chosen position (:97-102).  The edge
// check of an expansion is the warp-parallel InterX / SAT code of the graph search
// (pdmpc_kernels.cuh), on the same staged polylines.
//
// What is cached instead of recomputed (bit-identical, every value is a pure function of
// the node): the pose, cos/sin of the yaw and the cost to come of a tree node are stored
// when the node is created — the reference recomputes them on every pass from the root
// with the same operations in the same order (:124-137).  The path shapes are re-placed at
// the end from the parent pose instead of being kept per node (shapes_tmp, :183).
//
// valid_nodes_at_hp (:72,190,197) is pushed to many times but popped ONCE: with the
// reference's comparator (parent.f > v.f, strict) a pushed entry reaches the root of the
// libstdc++ heap iff root.f > v.f, so the single pop returns the earliest-pushed entry
// among those of minimal cost.  The kernel keeps that running minimum (strict <).
#pragma once

#include "pdmpc_kernels.cuh"

namespace pdmpc {

constexpr int kMctsBranch = PDMPC_MCTS_MAX_BRANCH;   // rows of `children`
constexpr int kMctsPts = 256;                        // staged polyline points per search
constexpr int kMtN = 624, kMtM = 397;
constexpr int kRndBlock = kMtN / 2;                  // doubles per MT state regeneration

struct MctsDev {
    int n_max;                 // n_expansions_max
    int node_cap;              // n_max + Hp + 1 (ids are 1-based)
    const unsigned *seed;      // [n]
};

__host__ __device__ inline size_t mcts_smem_bytes(int node_cap) {
    const size_t nc = (size_t)node_cap + 1;
    size_t b = 6 * nc * sizeof(double);                        // x, y, yaw, cos, sin, cost
    b += kRndBlock * sizeof(double);                           // current block of random numbers
    b += 2 * kMctsPts * sizeof(double);                        // staged polylines
    b += (3 * kMaxHp + 4 * kAreaStride) * sizeof(double);      // reference points, v_ref (unused), shapes
    b += kMtN * sizeof(unsigned);                              // MT19937 state
    b += (kMaxHp + 2 + kMaxHp + 1) * sizeof(int);              // polyline ranges, path
    b += nc * kMctsBranch * sizeof(unsigned short);            // children
    b += 2 * nc * sizeof(unsigned short);                      // parent, edge
    b += nc;                                                   // trim
    return (b + 15) / 16 * 16;
}

__device__ __forceinline__ unsigned mt_temper(unsigned y) {
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
}

// One state regeneration (the 624-step twist of genrand_int32) by the warp, 32 entries at a
// time.  Entry kk needs the OLD mt[kk], mt[kk+1] and, for kk < 227, the OLD mt[kk+397]; for
// kk >= 227 the NEW mt[kk-227] and for kk = 623 the NEW mt[0] — all written by earlier
// chunks because a chunk (32) is shorter than 227.  Reads of a chunk complete before its writes.
__device__ __forceinline__ void mt_twist(unsigned *mt, int lane) {
    for (int k0 = 0; k0 < kMtN; k0 += kWarp) {
        const int kk = k0 + lane;
        unsigned v = 0;
        if (kk < kMtN) {
            const int k1 = kk + 1 == kMtN ? 0 : kk + 1;
            const int km = kk + kMtM >= kMtN ? kk + kMtM - kMtN : kk + kMtM;
            const unsigned y = (mt[kk] & 0x80000000u) | (mt[k1] & 0x7fffffffu);
            v = mt[km] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
        }
        __syncwarp();
        if (kk < kMtN) mt[kk] = v;
        __syncwarp();
    }
}

// The sampled search.  Persistent one-warp CTAs pulling searches from a global counter.
__global__ void __launch_bounds__(kWarp) mcts_kernel(MpaDev m, BatchDev b, OutDev o, MctsDev mc,
                                                     unsigned *work_counter) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    const int nc = mc.node_cap + 1;
    unsigned char *q = smem_raw;
    auto take = [&](size_t bytes) { unsigned char *p = q; q += bytes; return p; };
    double *nx = (double *)take(nc * sizeof(double));
    double *ny = (double *)take(nc * sizeof(double));
    double *nyaw = (double *)take(nc * sizeof(double));
    double *ncos = (double *)take(nc * sizeof(double));
    double *nsin = (double *)take(nc * sizeof(double));
    double *ncost = (double *)take(nc * sizeof(double));
    double *rnd = (double *)take(kRndBlock * sizeof(double));
    double *pts_x = (double *)take(kMctsPts * sizeof(double));
    double *pts_y = (double *)take(kMctsPts * sizeof(double));
    double *refx = (double *)take(kMaxHp * sizeof(double));
    double *refy = (double *)take(kMaxHp * sizeof(double));
    take(kMaxHp * sizeof(double));
    double *shx = (double *)take(kAreaStride * sizeof(double));
    double *shy = (double *)take(kAreaStride * sizeof(double));
    double *bhx = (double *)take(kAreaStride * sizeof(double));
    double *bhy = (double *)take(kAreaStride * sizeof(double));
    unsigned *mt = (unsigned *)take(kMtN * sizeof(unsigned));
    int *rng = (int *)take((kMaxHp + 2) * sizeof(int));
    int *path = (int *)take((kMaxHp + 1) * sizeof(int));
    unsigned short *children = (unsigned short *)take((size_t)nc * kMctsBranch * sizeof(unsigned short));
    unsigned short *npar = (unsigned short *)take(nc * sizeof(unsigned short));
    unsigned short *nedge = (unsigned short *)take(nc * sizeof(unsigned short));
    unsigned char *ntrim = (unsigned char *)take(nc);

    Tile<kWarp> t;
    t.shift = 0; t.lane = lane; t.mask = 0xffffffffu;
    const int Hp = m.Hp, nT = m.nT;
    const int n_rand = Hp * mc.n_max;

    for (;;) {
        unsigned si_u = 0;
        if (lane == 0) si_u = atomicAdd(work_counter, 1u);
        si_u = __shfl_sync(0xffffffffu, si_u, 0);
        if (si_u >= (unsigned)b.n) break;
        const int si = b.order ? __ldg(b.order + si_u) : (int)si_u;
        __syncwarp();

        // ---- per-search set-up (as in search_kernel) -------------------------------
        for (int k = lane; k < Hp; k += kWarp) {
            refx[k] = __ldg(b.ref_x + (size_t)si * Hp + k);
            refy[k] = __ldg(b.ref_y + (size_t)si * Hp + k);
        }
        const int *slot = b.slot_ptr + (size_t)si * (Hp + 1);
        const int trim0 = __ldg(b.trim0 + si);
        const int sp0 = __ldg(slot + 0), sp1 = __ldg(slot + 1);
        const int lp0 = __ldg(b.lane_ptr + 2 * si), lp1 = __ldg(b.lane_ptr + 2 * si + 1),
                  lp2 = __ldg(b.lane_ptr + 2 * si + 2);
        const double *opx = nullptr, *opy = nullptr, *lpx = nullptr, *lpy = nullptr;
        int obase = 0, llo = 0, lhi = 0;
        if (b.checker == PDMPC_CHECKER_INTERX) {
            const int spE = __ldg(slot + Hp + 1);
            const int ob_lo = __ldg(b.poly_ptr + sp0) + sp0, ob_hi = __ldg(b.poly_ptr + spE) + spE;
            const int ll_lo = lp0 + 2 * si, ll_hi = lp2 + 2 * si + 2;
            for (int k = lane; k <= Hp + 1; k += kWarp) {
                const int qq = __ldg(slot + k);
                rng[k] = __ldg(b.poly_ptr + qq) + qq - ob_lo;
            }
            const int nl = ll_hi - ll_lo, no = ob_hi - ob_lo;
            int used = 0;
            if (nl <= kMctsPts) {
                for (int j = lane; j < nl; j += kWarp) {
                    pts_x[j] = __ldg(b.ll_x + ll_lo + j);
                    pts_y[j] = __ldg(b.ll_y + ll_lo + j);
                }
                lpx = pts_x; lpy = pts_y; llo = 0; lhi = nl;
                used = nl;
            } else {
                lpx = b.ll_x; lpy = b.ll_y; llo = ll_lo; lhi = ll_hi;
            }
            if (used + no <= kMctsPts) {
                for (int j = lane; j < no; j += kWarp) {
                    pts_x[used + j] = __ldg(b.pl_x + ob_lo + j);
                    pts_y[used + j] = __ldg(b.pl_y + ob_lo + j);
                }
                opx = pts_x; opy = pts_y; obase = used;
            } else {
                opx = b.pl_x; opy = b.pl_y; obase = ob_lo;
            }
        }
        // :31 RandStream('mt19937ar', Seed = s): init_genrand (serial recurrence; Seed 0 -> 5489)
        if (lane == 0) {
            unsigned s = __ldg(mc.seed + si);
            if (s == 0u) s = 5489u;
            mt[0] = s;
            for (int i = 1; i < kMtN; ++i) {
                s = 1812433253u * (s ^ (s >> 30)) + (unsigned)i;
                mt[i] = s;
            }
        }
        int rnd_block = -1;
        // :59-70 root
        if (lane == 0) {
            const double yaw = __ldg(b.yaw0 + si);
            nx[1] = __ldg(b.x0 + si); ny[1] = __ldg(b.y0 + si); nyaw[1] = yaw;
            double s, c;
            sincos_ref(yaw, s, c);
            ncos[1] = c; nsin[1] = s; ncost[1] = 0.0;
            npar[1] = 0; nedge[1] = 0xffff; ntrim[1] = (unsigned char)trim0;
        }
        if (lane < kMctsBranch) {
            const int nroot = m.succ_ptr[(trim0 - 1) + 1] - m.succ_ptr[trim0 - 1];   // successor_trims{trim, 1}
            children[1 * kMctsBranch + lane] = lane < nroot ? 1 : 0;
        }
        __syncwarp();

        int n_nodes = 1, n_exp = 0, n_trav = 0, status = PDMPC_OK;
        bool finished = false;
        unsigned long long hash = kHashSeed, cols = 0;
        double best_f = 0.0;
        int best_id = 0;

        while (n_exp < mc.n_max && !finished && status == PDMPC_OK) {   // :86
            int node = 1;
            bool valid = false;
            int node_parent = 0, pos = 0;
            for (int step = 1; step <= Hp; ++step) {                    // :92
                valid = false;
                ++n_trav;
                const unsigned ch = lane < kMctsBranch ? children[node * kMctsBranch + lane] : 0;
                const unsigned mask = __ballot_sync(0xffffffffu, ch != 0);    // :97 find(children(:, node))
                const int n_trims = __popc(mask);
                if (n_trims == 0) {
                    if (node != 1) {                                    // :106-109
                        const int parent = npar[node];
                        __syncwarp();
                        if (lane < kMctsBranch && children[parent * kMctsBranch + lane] == node)
                            children[parent * kMctsBranch + lane] = 0;
                        __syncwarp();
                    } else {
                        finished = true;                                // :110-113
                    }
                    break;
                }
                if (n_trav > n_rand) { status = PDMPC_ERR_CAPACITY; break; }   // MATLAB: index out of bounds
                const int blk = (n_trav - 1) / kRndBlock;
                while (rnd_block < blk) {                               // next 312 numbers of the stream
                    mt_twist(mt, lane);
                    for (int j = lane; j < kRndBlock; j += kWarp) {
                        const unsigned a = mt_temper(mt[2 * j]) >> 5, bb = mt_temper(mt[2 * j + 1]) >> 6;
                        rnd[j] = ((double)a * 67108864.0 + (double)bb) * (1.0 / 9007199254740992.0);
                    }
                    ++rnd_block;
                    __syncwarp();
                }
                const double r = rnd[(n_trav - 1) - blk * kRndBlock];
                const int pick = (int)ceil(r * (double)n_trims);        // :102
                unsigned mm = mask;                                     // pick-th set bit = 0-based child_position
                for (int i = 1; i < pick; ++i) mm &= mm - 1u;
                pos = __ffs(mm) - 1;
                hash = hash_step(hash, ((unsigned)node << 8) | (unsigned)(pos + 1));
                const unsigned chv = __shfl_sync(0xffffffffu, ch, pos);
                if (chv != 1u) { node = (int)chv; continue; }           // :139-144 already expanded

                ++n_exp;                                                // :146
                node_parent = node;
                const int ptrim = ntrim[node];
                const int sbase = m.succ_ptr[(step - 1) * nT + (ptrim - 1)];
                const int te = m.succ_te[sbase + pos];
                const int edge = te >> 8, gtrim = (te & 0xff) + 1;
                const double px = nx[node], py = ny[node], pyaw = nyaw[node], c = ncos[node], s = nsin[node];
                const int bkind = (step == Hp) ? PDMPC_AREA_LARGE_OFFSET : PDMPC_AREA_WITHOUT_OFFSET;   // :153-159
                const int ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                const int nbs = m.area_npts[edge * 3 + bkind];
                if (lane < 8)
                    place_point(m, edge, PDMPC_AREA_NORMAL, lane, c, s, px, py, shx[lane], shy[lane]);
                else if (lane < 16)
                    place_point(m, edge, bkind, lane - 8, c, s, px, py, bhx[lane - 8], bhy[lane - 8]);
                __syncwarp();
                valid = true;
                if (b.checker == PDMPC_CHECKER_INTERX) {
                    const int st_lo = obase + rng[0], st_hi = obase + rng[1];
                    const int dy_lo = obase + rng[step], dy_hi = obase + rng[step + 1];
                    cols += (unsigned long long)((st_hi - st_lo) + (dy_hi - dy_lo) + (lhi - llo));
                    if (interx_dispatch<kWarp>(ns, opx, opy, st_lo, st_hi, dy_lo, dy_hi, shx, shy, t))
                        valid = false;
                    else if (interx_dispatch<kWarp>(nbs, lpx, lpy, llo, lhi, 0, 0, bhx, bhy, t))
                        valid = false;
                } else {
                    const int dp0 = __ldg(slot + step), dp1 = __ldg(slot + step + 1);
                    for (int pass = 0; pass < 2 && valid; ++pass) {
                        const int q0 = pass == 0 ? sp0 : dp0, q1 = pass == 0 ? sp1 : dp1;
                        for (int p = q0; p < q1 && valid; ++p) {
                            const int v0 = __ldg(b.poly_ptr + p), v1 = __ldg(b.poly_ptr + p + 1);
                            cols += (unsigned long long)(v1 - v0);
                            if (sat_collide<kWarp>(shx, shy, ns, b.vert_x + v0, b.vert_y + v0, v1 - v0, t))
                                valid = false;
                        }
                    }
                    if (valid) {
                        cols += (unsigned long long)(lp2 - lp0);
                        if (lanelet_side_sat<kWarp>(bhx, bhy, nbs, b.lane_x + lp0, b.lane_y + lp0, lp1 - lp0, t))
                            valid = false;
                        else if (lanelet_side_sat<kWarp>(bhx, bhy, nbs, b.lane_x + lp1, b.lane_y + lp1, lp2 - lp1, t))
                            valid = false;
                    }
                }
                if (!valid) {                                           // :172-175 remove edge
                    if (lane == 0) children[node_parent * kMctsBranch + pos] = 0;
                    __syncwarp();
                    break;
                }
                // :176-185 add node
                if (n_nodes + 1 > mc.node_cap) { status = PDMPC_ERR_CAPACITY; valid = false; break; }
                ++n_nodes;
                const int id = n_nodes;
                int nsucc = 0;
                if (step < Hp) {
                    const int sb2 = m.succ_ptr[step * nT + (gtrim - 1)];
                    nsucc = m.succ_ptr[step * nT + (gtrim - 1) + 1] - sb2;
                }
                if (lane < kMctsBranch) children[id * kMctsBranch + lane] = lane < nsucc ? 1 : 0;
                if (lane == 0) {
                    const double mdx = m.edge_d[edge * 4 + 0], mdy = m.edge_d[edge * 4 + 1],
                                 mdyaw = m.edge_d[edge * 4 + 2];
                    const double ex = px + (c * mdx - s * mdy);         // :127-132
                    const double ey = py + (s * mdx + c * mdy);
                    const double eyaw = pyaw + mdyaw;
                    const double ddx = ex - refx[step - 1], ddy = ey - refy[step - 1];
                    const double nrm = sqrt(ddx * ddx + ddy * ddy);
                    nx[id] = ex; ny[id] = ey; nyaw[id] = eyaw;
                    ncost[id] = ncost[node_parent] + nrm * nrm;         // :137
                    double es, ec;
                    sincos_ref(eyaw, es, ec);
                    ncos[id] = ec; nsin[id] = es;
                    npar[id] = (unsigned short)node_parent;
                    nedge[id] = (unsigned short)edge;
                    ntrim[id] = (unsigned char)gtrim;
                    children[node_parent * kMctsBranch + pos] = (unsigned short)id;
                }
                __syncwarp();
                node = id;
            }
            if (valid) {                                                // :189-193
                const double cst = ncost[node];
                if (best_id == 0 || cst < best_f) { best_f = cst; best_id = node; }
                if (lane == 0) children[node_parent * kMctsBranch + pos] = 0;
                __syncwarp();
            }
        }

        // ---- results (:197-249) ---------------------------------------------------------
        const bool exhausted = best_id == 0 || status != PDMPC_OK;
        if (lane == 0) {
            int cur = best_id;
            for (int d = Hp; d >= 0; --d) {
                path[d] = exhausted ? 0 : cur;
                if (!exhausted && d > 0) cur = npar[cur];
            }
            o.status[si] = status;
            if (o.is_exhausted) o.is_exhausted[si] = exhausted ? 1 : 0;
            if (o.n_expanded) o.n_expanded[si] = n_exp;                 // :199
            if (o.n_pops) o.n_pops[si] = n_trav;
            if (o.pop_hash) o.pop_hash[si] = hash;
            atomicAdd(o.counters + 0, (unsigned long long)n_trav);
            atomicAdd(o.counters + 1, (unsigned long long)n_nodes);
            atomicAdd(o.counters + 2, cols);
        }
        __syncwarp();
        const double qnan = nan("");
        for (int d = lane; d <= Hp; d += kWarp) {
            const int pid = path[d];
            const size_t oo = (size_t)si * (Hp + 1) + d;
            if (o.trims) o.trims[oo] = exhausted ? (d == 0 ? trim0 : 0) : (int)ntrim[pid];
            if (o.tree_path) o.tree_path[oo] = pid;
            if (o.g_path) o.g_path[oo] = exhausted ? qnan : (d == Hp ? best_f : -1.0);   // :211,239
            if (o.h_path) o.h_path[oo] = exhausted ? qnan : -1.0;                        // :213
            if (d >= 1) {
                const size_t os = (size_t)si * Hp + (d - 1);
                if (o.y_predicted) {
                    o.y_predicted[os * 3 + 0] = exhausted ? qnan : nx[pid];
                    o.y_predicted[os * 3 + 1] = exhausted ? qnan : ny[pid];
                    o.y_predicted[os * 3 + 2] = exhausted ? qnan : nyaw[pid];
                }
                if (o.shape_npts) {
                    int edge = 0, ns = 0, qid = 0;
                    if (!exhausted) {
                        qid = path[d - 1];
                        edge = nedge[pid];
                        ns = m.area_npts[edge * 3 + PDMPC_AREA_NORMAL];
                    }
                    o.shape_npts[os] = ns;
                    if (o.shape_x && o.shape_y) {
                        for (int i = 0; i < kAreaStride; ++i) {
                            double ox = 0.0, oy = 0.0;
                            if (i < ns)
                                place_point(m, edge, PDMPC_AREA_NORMAL, i, ncos[qid], nsin[qid], nx[qid], ny[qid], ox, oy);
                            o.shape_x[os * kAreaStride + i] = ox;
                            o.shape_y[os * kAreaStride + i] = oy;
                        }
                    }
                }
            }
        }
        __syncwarp();
    }
}

}  // namespace pdmpc
