// pdmpc_capi.cu — host side of the C ABI declared in include/pdmpc_b200.h.
//
// Stages the MPA tables and one batch of searches in HBM as SoA/CSR arrays,
// launches the persistent search kernel (pdmpc_kernels.cuh) on the handle's
// stream and copies the results back.  No CPU fallback exists: every entry
// point fails with PDMPC_ERR_CUDA when the device is unusable.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <new>
#include <string>
#include <vector>

#include "pdmpc_kernels.cuh"
#include "pdmpc_tiles.cuh"
#include "pdmpc_mcts.cuh"
#include "pdmpc_cta.cuh"
#include "pdmpc_joint.cuh"
#include "pdmpc_inputs.cuh"
#include "pdmpc_fallback.cuh"
#include "pdmpc_obstacles.cuh"

using namespace pdmpc;

namespace {

// Launch shapes of the warp-level search kernels: "latency" = one search per one-warp CTA
// (pdmpc_kernels.cuh); "tiles" = 2 or 4 searches per warp (pdmpc_tiles.cuh), the throughput shape.
#ifndef PDMPC_HEAP_SMEM
#define PDMPC_HEAP_SMEM 256
#endif
#ifndef PDMPC_PTS_SMEM
#define PDMPC_PTS_SMEM 256
#endif
constexpr int kHeapSmem = PDMPC_HEAP_SMEM;   // heap entries kept in shared memory per search
constexpr int kPts = PDMPC_PTS_SMEM;         // polyline points (lanelet bounds + obstacles of all steps) staged per search
#define KERNEL_LAT search_kernel<kHeapSmem, kPts, false>
#define KERNEL_LAT_DEPS search_kernel<kHeapSmem, kPts, true>
using WarpSmem = TileSmem<kHeapSmem, kPts>;
constexpr size_t kSmemLimit = 227 * 1024;
// tiles: TILE lanes per search; heap entries / staged polyline points per search in shared memory;
// one-warp CTAs per SM the shape is compiled for (register cap) — sized so that the CTAs fill 228 KB
#ifndef PDMPC_TILE2_CTAS
#define PDMPC_TILE2_CTAS 20
#endif
#ifndef PDMPC_TILE4_CTAS
#define PDMPC_TILE4_CTAS 8
#endif
#ifndef PDMPC_TILE2_HEAP
#define PDMPC_TILE2_HEAP 64
#endif
#ifndef PDMPC_TILE2_PTS
#define PDMPC_TILE2_PTS 128
#endif
#ifndef PDMPC_TILE4_HEAP
#define PDMPC_TILE4_HEAP 96
#endif
#ifndef PDMPC_TILE4_PTS
#define PDMPC_TILE4_PTS 256
#endif
constexpr int kTile2Heap = PDMPC_TILE2_HEAP, kTile2Pts = PDMPC_TILE2_PTS, kTile2Ctas = PDMPC_TILE2_CTAS;
constexpr int kTile4Heap = PDMPC_TILE4_HEAP, kTile4Pts = PDMPC_TILE4_PTS, kTile4Ctas = PDMPC_TILE4_CTAS;
#define KERNEL_TILE2 search_tile_kernel<16, kTile2Heap, kTile2Pts, kTile2Ctas>
#define KERNEL_TILE4 search_tile_kernel<8, kTile4Heap, kTile4Pts, kTile4Ctas>
constexpr size_t kTile2Smem = 2 * sizeof(TileSm<kTile2Heap, kTile2Pts>);
constexpr size_t kTile4Smem = 4 * sizeof(TileSm<kTile4Heap, kTile4Pts>);
// "cta" = masters + shared checker warps, one CTA per SM (pdmpc_cta.cuh).  Two configurations:
//   1 master, 12 checkers (+ 3 parked warps): a batch of at most one search per SM — lowest latency
//   NM masters, 12 checkers: larger batches — every SM runs NM searches at (almost) the same latency
#ifndef PDMPC_CTA_MASTERS
#define PDMPC_CTA_MASTERS 4
#endif
#ifndef PDMPC_ESCALATE_POPS
#define PDMPC_ESCALATE_POPS 2560
#endif
constexpr int kCtaCheckers = 12;
constexpr int kCtaHeap = 4096, kCtaPts = 512;          // single master: heap entries / polyline points in shared memory
constexpr int kCtaMHeap = 1024, kCtaMPts = 256;        // several masters: per search
constexpr int kCtaMasters = PDMPC_CTA_MASTERS, kCtaMastersDeps = 2;
#define KERNEL_CTA search_cta_kernel<kCtaHeap, kCtaPts, kCtaCheckers, 1, false>
#define KERNEL_CTA_DEPS search_cta_kernel<kCtaHeap, kCtaPts, kCtaCheckers, 1, true>
#define KERNEL_CTAM search_cta_kernel<kCtaMHeap, kCtaMPts, kCtaCheckers, kCtaMasters, false>
#define KERNEL_CTAM_DEPS search_cta_kernel<kCtaMHeap, kCtaMPts, kCtaCheckers, kCtaMastersDeps, true>
using CtaSmemT = CtaSmem<kCtaHeap, kCtaPts, kCtaCheckers, 1, false>;
using CtaDepsSmemT = CtaSmem<kCtaHeap, kCtaPts, kCtaCheckers, 1, true>;
using CtaMSmemT = CtaSmem<kCtaMHeap, kCtaMPts, kCtaCheckers, kCtaMasters, false>;
using CtaMDepsSmemT = CtaSmem<kCtaMHeap, kCtaMPts, kCtaCheckers, kCtaMastersDeps, true>;
static_assert(sizeof(CtaSmemT) <= kSmemLimit && sizeof(CtaDepsSmemT) <= kSmemLimit && sizeof(CtaMSmemT) <= kSmemLimit &&
              sizeof(CtaMDepsSmemT) <= kSmemLimit, "CTA shapes must fit one SM");

// Buffer that grows on demand and frees its memory with the handle: device memory, or pinned host memory for staging.
template <bool kPinned>
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    ~Buf() { drop(); }
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        drop();
        const size_t want = kPinned ? bytes + bytes / 4 + 4096 : bytes + bytes / 8 + 256;
        cudaError_t e = kPinned ? cudaHostAlloc(&p, want, cudaHostAllocDefault) : cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        else p = nullptr;
        return e;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }

  private:
    void drop() {
        if (p) kPinned ? cudaFreeHost(p) : cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};
using DBuf = Buf<false>;
using PinnedBuf = Buf<true>;

// Launch shapes of the search.  The values are those of pdmpc_set_variant and pdmpc_stats.shape.
enum Shape {
    kShapeAuto = 0,
    kShapeLatency = 1,   // one search per one-warp CTA (search_kernel): every checker, pop traces, dependencies
    kShapeTile2 = 2,     // two searches per warp (search_tile_kernel<16>): InterX batches, the throughput shape
    kShapeTile4 = 3,     // four searches per warp (search_tile_kernel<8>)
    kShapeCta = 4,       // one CTA per search, or several masters per CTA (pdmpc_cta.cuh)
    kShapeCtaValid = 5,  // the same with the valid-only queue
};

// The input arrays of a batch, in the order of their device buffers (pdmpc_handle::b_in) and of the packed staging block.
enum InArray {
    kInX0, kInY0, kInYaw0, kInTrim0, kInRefX, kInRefY, kInVRef, kInSlotPtr, kInPolyPtr, kInVertX, kInVertY,
    kInLanePtr, kInLaneX, kInLaneY, kInOrder, kNumIn
};
constexpr size_t kInElem[kNumIn] = {sizeof(double), sizeof(double), sizeof(double), sizeof(int),
                                    sizeof(double), sizeof(double), sizeof(double), sizeof(int),
                                    sizeof(int),    sizeof(double), sizeof(double), sizeof(int),
                                    sizeof(double), sizeof(double), sizeof(int)};

// Element ranges [lo, hi) of the input arrays that belong to searches [s0, s1).  p, v and l are the obstacle polygons,
// vertices and lanelet points before s0 and s1 (the CSR offsets there); the offset arrays take one entry more.
// The whole batch is the range [0, n) with p, v, l = 0 and the totals.
struct InRange {
    size_t lo[kNumIn], hi[kNumIn];
};
static InRange in_range(int Hp, int s0, int s1, int p0, int p1, int v0, int v1, int l0, int l1) {
    const size_t H = (size_t)Hp;
    return {{(size_t)s0, (size_t)s0, (size_t)s0, (size_t)s0, s0 * H, s0 * H, s0 * H, s0 * (H + 1), (size_t)p0,
             (size_t)v0, (size_t)v0, (size_t)2 * s0, (size_t)l0, (size_t)l0, (size_t)s0},
            {(size_t)s1, (size_t)s1, (size_t)s1, (size_t)s1, s1 * H, s1 * H, s1 * H, s1 * (H + 1) + 1, (size_t)p1 + 1,
             (size_t)v1, (size_t)v1, (size_t)2 * s1 + 1, (size_t)l1, (size_t)l1, (size_t)s1}};
}

// The caller's input arrays; the work order comes from the host library.
static void in_sources(const pdmpc_batch_in *in, const int *order, const void *src[kNumIn]) {
    const void *s[kNumIn] = {in->x0,       in->y0,     in->yaw0,   in->trim0,    in->ref_x,  in->ref_y,  in->v_ref, in->slot_ptr,
                             in->poly_ptr, in->vert_x, in->vert_y, in->lane_ptr, in->lane_x, in->lane_y, order};
    std::copy(s, s + kNumIn, src);
}

// Names the staged input arrays `d` in b; a single search runs without a work order.
static void set_batch(BatchDev &b, int n, int checker, double dt, const void *const d[kNumIn]) {
    b.n = n; b.checker = checker; b.dt = dt;
    b.x0 = (const double *)d[kInX0]; b.y0 = (const double *)d[kInY0]; b.yaw0 = (const double *)d[kInYaw0];
    b.trim0 = (const int *)d[kInTrim0];
    b.ref_x = (const double *)d[kInRefX]; b.ref_y = (const double *)d[kInRefY]; b.v_ref = (const double *)d[kInVRef];
    b.slot_ptr = (const int *)d[kInSlotPtr]; b.poly_ptr = (const int *)d[kInPolyPtr];
    b.vert_x = (const double *)d[kInVertX]; b.vert_y = (const double *)d[kInVertY];
    b.lane_ptr = (const int *)d[kInLanePtr]; b.lane_x = (const double *)d[kInLaneX]; b.lane_y = (const double *)d[kInLaneY];
    b.order = n > 1 ? (const int *)d[kInOrder] : nullptr;
}

// Work order of searches [s0, s1) into order[0, s1 - s0): the searches with the most obstacle polygons first (they are
// the ones most likely to run long / exhaust, so the tail of a launch is made of short searches).  A stable counting
// sort; false if slot_ptr decreases.
static bool heavy_first_order(const int *slot_ptr, int Hp, int s0, int s1, int *order) {
    auto key = [&](int i) { return slot_ptr[(size_t)(i + 1) * (Hp + 1)] - slot_ptr[(size_t)i * (Hp + 1)]; };
    int kmax = 0;
    for (int i = s0; i < s1; ++i) {
        if (key(i) < 0) return false;
        kmax = std::max(kmax, key(i));
    }
    std::vector<int> cnt(kmax + 2, 0);
    for (int i = s0; i < s1; ++i) cnt[kmax - key(i) + 1]++;
    for (int k = 0; k <= kmax; ++k) cnt[k + 1] += cnt[k];
    for (int i = s0; i < s1; ++i) order[cnt[kmax - key(i)]++] = i;
    return true;
}

// The result fields in the order of pdmpc_batch_out and of the output block (d_out_pack); the counter block follows them.
constexpr int kNumOut = 13;
constexpr size_t kCounterBytes = 16 * sizeof(unsigned long long);
struct OutFields {
    size_t bytes[kNumOut];   // per search
    void *dst[kNumOut];      // the caller's arrays (null: not wanted)
};
static OutFields out_fields(int Hp, const pdmpc_batch_out *o = nullptr) {
    const size_t H = (size_t)Hp, S = PDMPC_AREA_STRIDE;
    OutFields f = {{sizeof(int), 1, sizeof(int), sizeof(int), sizeof(uint64_t), (H + 1) * sizeof(int),
                    (H + 1) * sizeof(int), H * 3 * sizeof(double), (H + 1) * sizeof(double), (H + 1) * sizeof(double),
                    H * sizeof(int), H * S * sizeof(double), H * S * sizeof(double)},
                   {}};
    if (o) {
        void *d[kNumOut] = {o->status, o->is_exhausted, o->n_expanded, o->n_pops,     o->pop_hash, o->trims, o->tree_path,
                            o->y_predicted, o->g_path,  o->h_path,     o->shape_npts, o->shape_x,  o->shape_y};
        std::copy(d, d + kNumOut, f.dst);
    }
    return f;
}

// The arena slots from `slot` on: a launch that runs beside others gets slots of its own.
static ArenaDev arena_from(const ArenaDev &a, size_t slot) {
    ArenaDev x = a;
    const size_t off = slot * (size_t)a.cap;
    x.a += off; x.b += off; x.cs += off; x.heap += off;
    return x;
}

}  // namespace

struct pdmpc_handle {
    int device = 0;
    int num_sms = 0;
    int lat_ctas_per_sm = 0;          // occupancy of the latency shape
    int tile_ctas_per_sm[2] = {0, 0}; // occupancy of the tile shapes (2 / 4 searches per warp); 0 = not launchable
    int tile_pts_limit = 0;           // staged-points limit of the tile shapes (0 = what the kernel holds; test knob)
    int variant_mode = 0;             // 0 = auto, 1 = latency, 2 / 3 = tiles (2 / 4 searches per warp), 4 / 5 = cta
    int cta_heap_smem = kCtaHeap;     // heap entries the CTA shape keeps in shared memory (tuning/test knob)
    int escalate_pops = -1;           // tile shapes give a search up after this many pops (0 = never, -1 = by batch size), pdmpc_set_escalation
    int esc_short_list = -1;          // lists up to this long run with one master per CTA (-1: 3 per SM)
    DBuf esc;                         // [0] count, [1] producers done, [4..] escalated search indices
    DBuf esc_rows;                    // pipeline: packed output rows of the escalated searches
    PinnedBuf pin_esc;

    bool cta_valid_only = false;      // pdmpc_set_cta_queue: the CTA shape runs its valid-only queue (shape 5) whenever it is chosen
    bool cta_ok = false;              // the CTA-per-search kernel is launchable (shared memory opt-in granted)
    bool cta_deps_ok = false;         // ... and its pdmpc_plan_timestep instance
    // pdmpc_plan_timestep: dependency CSR, fallback areas, done flags (one packed upload)
    DBuf j_veh, j_node, j_heap;       // centralized (joint) search arena
    DBuf d_deps, d_done, d_depx, d_depy, d_depn;
    bool lat_deps_ok = false;
    PinnedBuf pin_deps;
    DepsDev deps{};
    bool deps_staged = false;
    std::vector<int> topo_order;      // work order override for the next pdmpc_stage_batch (time-step calls)
    // pipelined pdmpc_plan_batch (large host batches): copy-in, two compute and copy-out streams
    cudaStream_t s_in = nullptr, s_out = nullptr, s_comp[7] = {};   // + the handle's stream
    std::vector<cudaEvent_t> ev_chunk;   // 2 per chunk: inputs landed, searches done
    std::vector<double> chunk_host_ms;   // host time at which chunk c's launch was enqueued (pdmpc_get_pipeline_timeline)
    int chunks_last = 0;
    cudaEvent_t ev_fork = nullptr;
    PinnedBuf pin_order;
    DBuf wc_chunks;
    int pipeline_chunks = 0;          // 0 = auto, 1 = off (tuning/test knob, pdmpc_set_pipeline_chunks)
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[7] = {};   // 0/1 h2d, 2/3 kernel, 4/5 d2h
    std::string err;

    // MPA
    bool has_mpa = false;
    MpaDev mpa{};
    DBuf m_succ_ptr, m_succ_te, m_edge_d, m_npts, m_ax, m_ay;
    int full_tree_nodes = 0;
    int user_node_cap = 0;
    int max_branch = 0;               // mpa.maximum_branching_factor()
    int max_area_npts = 0;            // most points of any maneuver's normal-offset area

    // staged batch
    bool staged = false;
    BatchDev batch{};
    DBuf b_in[kNumIn];                // input arrays of a batch staged one by one (large batches, the pipeline)
    DBuf b_plx, b_ply, b_plxy, b_llx, b_lly, b_llxy, b_seed;

    // small batches (one computation level of a time step): every input array in ONE pinned
    // staging buffer -> one H2D copy; every output array in one device block -> one D2H copy
    DBuf d_in_pack, d_out_pack;
    PinnedBuf pin_in, pin_out;
    cudaEvent_t ev_pack = nullptr;    // completion of the last packed H2D (the pinned buffer is reused)
    bool pack_in_flight = false;
    size_t out_off[kNumOut + 1] = {}; // byte offsets of the output arrays (+ counters) inside d_out_pack
    size_t out_bytes = 0;

    // outputs
    OutDev out{};
    DBuf work_counter;

    // arena
    ArenaDev arena{};
    DBuf a_a, a_b, a_cs, a_heap;
    int arena_slots = 0;

    // road + reference paths (pdmpc_upload_road) and the buffers of pdmpc_sample_inputs
    bool has_road = false;
    RoadDev road{};
    bool has_reach = false;           // pdmpc_upload_reachable_sets
    int reach_max_pts = 0;            // points of the largest uploaded reachable set
    ReachDev reach{};
    DBuf q_rptr, q_rx, q_ry, q_x, q_y, q_yaw, q_speed, q_trim, q_sptr, q_sidx, q_pptr, q_pidx, q_cs, q_cntp, q_cntv,
        q_slot, q_vbase, q_poly, q_vx, q_vy;
    std::vector<int> road_bound_ptr;   // host copy (capacity checks)
    DBuf r_bptr, r_bx, r_by, r_pptr, r_px, r_py, r_lptr, r_lidx, r_pidx, r_loop, r_speed;
    DBuf i_pid, i_x, i_y, i_speed, i_refx, i_refy, i_vref, i_ridx, i_cur, i_pred, i_pre, i_cnt, i_lptr, i_lx, i_ly;

    // closed loop on the device (pdmpc_closed_loop_reset / pdmpc_plan_timestep_closed_loop)
    ClosedLoopDev cl{};
    DBuf cl_valid, cl_trims, cl_traj, cl_npts, cl_sx, cl_sy;
    DBuf cf_slot, cf_still, cf_npts, cf_x, cf_y, cf_traj, cf_trims;

    // trace (debug / parity tests)
    DBuf t_ids, t_n;

    pdmpc_stats stats{};
    bool timing_pending_h2d = false, timing_pending_kernel = false, timing_pending_d2h = false;
};

static thread_local std::string g_create_error;

static int fail(pdmpc_handle *h, int code, const std::string &msg) {
    if (h) h->err = msg;
    else g_create_error = msg;
    return code;
}

#define CU_TRY(h, expr)                                                                          \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess)                                                                   \
            return fail(h, PDMPC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
    } while (0)

// FP64 pipe peak of this device, measured (SURVEY.md §8(d) asks for it next to the HBM roofline):
// 8 independent accumulator chains per thread, no memory traffic; once as separate DMUL + DADD (what
// the search executes: FMA contraction is off for bit-exactness) and once as DFMA.
namespace {
template <bool FMA>
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *sink, int iters, double a, double b2) {
    double v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (FMA) v[i] = __fma_rn(v[i], a, b2);
            else v[i] = __dadd_rn(__dmul_rn(v[i], a), b2);
        }
    }
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) acc += v[i];
    if (acc == 123.456) sink[0] = acc;   // never true: keeps the chains alive
}
}  // namespace


extern "C" {

int pdmpc_abi_version(void) { return PDMPC_ABI_VERSION; }

int pdmpc_get_hp(const pdmpc_handle *h) { return h && h->has_mpa ? h->mpa.Hp : 0; }

const char *pdmpc_last_error(const pdmpc_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int pdmpc_create(int device_id, pdmpc_handle **out) {
    if (!out) return fail(nullptr, PDMPC_ERR_BAD_INPUT, "pdmpc_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(nullptr, PDMPC_ERR_CUDA,
                    std::string("pdmpc_create: no CUDA device (") + cudaGetErrorString(e) +
                        "); the optimizer has no CPU fallback");
    if (device_id < 0 || device_id >= count)
        return fail(nullptr, PDMPC_ERR_CUDA, "pdmpc_create: device id out of range");
    pdmpc_handle *h = new (std::nothrow) pdmpc_handle();
    if (!h) return fail(nullptr, PDMPC_ERR_ALLOC, "pdmpc_create: out of host memory");
    h->device = device_id;
    if ((e = cudaSetDevice(device_id)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        std::string msg = std::string("pdmpc_create: ") + cudaGetErrorString(e);
        delete h;
        return fail(nullptr, PDMPC_ERR_CUDA, msg);
    }
    for (auto &ev : h->ev) cudaEventCreate(&ev);
    cudaEventCreateWithFlags(&h->ev_pack, cudaEventDisableTiming);
    cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device_id);
    int occ = 0;
    e = cudaFuncSetAttribute(KERNEL_LAT, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WarpSmem));
    if (e == cudaSuccess)
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERNEL_LAT, kWarp, sizeof(WarpSmem));
    if (e != cudaSuccess || occ < 1) {
        std::string msg = std::string("pdmpc_create: search kernel is not launchable on this device (") +
                          cudaGetErrorString(e) + "); built for sm_100a";
        cudaStreamDestroy(h->stream);
        delete h;
        return fail(nullptr, PDMPC_ERR_CUDA, msg);
    }
    h->lat_ctas_per_sm = occ;
    if (cudaFuncSetAttribute(KERNEL_TILE2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTile2Smem) == cudaSuccess &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERNEL_TILE2, kWarp, kTile2Smem) == cudaSuccess)
        h->tile_ctas_per_sm[0] = occ;
    if (cudaFuncSetAttribute(KERNEL_TILE4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTile4Smem) == cudaSuccess &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, KERNEL_TILE4, kWarp, kTile4Smem) == cudaSuccess)
        h->tile_ctas_per_sm[1] = occ;
    h->cta_ok = cudaFuncSetAttribute(KERNEL_CTA, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)sizeof(CtaSmemT)) == cudaSuccess &&
                cudaFuncSetAttribute(KERNEL_CTAM, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)sizeof(CtaMSmemT)) == cudaSuccess;
    h->lat_deps_ok = cudaFuncSetAttribute(KERNEL_LAT_DEPS, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(WarpSmem)) == cudaSuccess;
    h->cta_deps_ok = cudaFuncSetAttribute(KERNEL_CTA_DEPS, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(CtaDepsSmemT)) == cudaSuccess &&
                     cudaFuncSetAttribute(KERNEL_CTAM_DEPS, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)sizeof(CtaMDepsSmemT)) == cudaSuccess;
    cudaGetLastError();
    *out = h;
    return PDMPC_OK;
}

int pdmpc_destroy(pdmpc_handle *h) {
    if (!h) return PDMPC_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (cudaEvent_t e : h->ev_chunk) cudaEventDestroy(e);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (cudaStream_t st : h->s_comp)
        if (st) cudaStreamDestroy(st);
    for (cudaStream_t st : {h->s_in, h->s_out})
        if (st) cudaStreamDestroy(st);
    if (h->ev_pack) cudaEventDestroy(h->ev_pack);
    for (auto &ev : h->ev)
        if (ev) cudaEventDestroy(ev);
    cudaStreamDestroy(h->stream);
    delete h;   // the device and pinned buffers free themselves
    return PDMPC_OK;
}

void *pdmpc_stream(pdmpc_handle *h) { return h ? (void *)h->stream : nullptr; }

int pdmpc_host_alloc(void **p, size_t bytes) {
    if (!p) return PDMPC_ERR_BAD_INPUT;
    return cudaHostAlloc(p, bytes ? bytes : 1, cudaHostAllocDefault) == cudaSuccess ? PDMPC_OK : PDMPC_ERR_ALLOC;
}
int pdmpc_host_free(void *p) {
    if (p) cudaFreeHost(p);
    return PDMPC_OK;
}

int pdmpc_set_variant(pdmpc_handle *h, int32_t variant) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (variant < kShapeAuto || variant > kShapeCtaValid)
        return fail(h, PDMPC_ERR_BAD_INPUT,
                    "variant must be 0 (auto), 1 (one search per warp), 2 / 3 (tiles: 2 / 4 searches per warp), 4 (cta) or 5 (cta, valid-only queue)");
    h->variant_mode = variant;
    return PDMPC_OK;
}

int pdmpc_set_cta_heap_smem(pdmpc_handle *h, int32_t entries) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (entries < 0 || entries > kCtaHeap || (entries & 1))
        return fail(h, PDMPC_ERR_BAD_INPUT, "cta heap: entries must be 0 (default) or an even number <= 4096");
    h->cta_heap_smem = entries ? entries : kCtaHeap;
    return PDMPC_OK;
}

int pdmpc_set_cta_queue(pdmpc_handle *h, int32_t valid_only) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    h->cta_valid_only = valid_only != 0;
    return PDMPC_OK;
}

int pdmpc_set_tile_points(pdmpc_handle *h, int32_t points) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (points < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "tile points: must be 0 (default) or > 0");
    h->tile_pts_limit = points;
    return PDMPC_OK;
}

int pdmpc_set_node_capacity(pdmpc_handle *h, int32_t cap) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (cap != 0 && cap < 64) return fail(h, PDMPC_ERR_BAD_INPUT, "node capacity must be 0 (default) or >= 64");
    h->user_node_cap = cap;
    return PDMPC_OK;
}

}  // extern "C"

template <class T>
static int upload(pdmpc_handle *h, DBuf &buf, const T *src, size_t count) {
    CU_TRY(h, buf.reserve(std::max<size_t>(count, 1) * sizeof(T)));
    if (count) CU_TRY(h, cudaMemcpyAsync(buf.p, src, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (int64_t)(count * sizeof(T));
    return PDMPC_OK;
}
#define UP(h, buf, src, count)                         \
    do {                                               \
        int _rc = upload(h, buf, src, (size_t)(count)); \
        if (_rc != PDMPC_OK) return _rc;               \
    } while (0)

template <class T>
static int download(pdmpc_handle *h, T *dst, const DBuf &buf, size_t count) {
    if (!dst || !count) return PDMPC_OK;
    CU_TRY(h, cudaMemcpyAsync(dst, buf.p, count * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
    h->stats.d2h_bytes += (int64_t)(count * sizeof(T));
    return PDMPC_OK;
}

extern "C" {

int pdmpc_upload_mpa(pdmpc_handle *h, const pdmpc_mpa_desc *d) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!d || !d->transition || !d->edge_from || !d->edge_to || !d->edge_dx || !d->edge_dy || !d->edge_dyaw ||
        !d->area_npts || !d->area_x || !d->area_y)
        return fail(h, PDMPC_ERR_BAD_INPUT, "upload_mpa: NULL table pointer");
    const int nT = d->n_trims, Hp = d->Hp, nE = d->n_edges;
    if (nT < 1 || nT > PDMPC_MAX_TRIMS || nT > 255 || Hp < 1 || Hp > PDMPC_MAX_HP || nE < 1 || nE >= kMaxEdges)
        return fail(h, PDMPC_ERR_BAD_INPUT, "upload_mpa: n_trims/Hp/n_edges out of range");
    CU_TRY(h, cudaSetDevice(h->device));
    std::vector<int16_t> edge_of((size_t)nT * nT, -1);
    int max_npts = 0;
    for (int e = 0; e < nE; ++e) {
        int f = d->edge_from[e], t = d->edge_to[e];
        if (f < 1 || f > nT || t < 1 || t > nT) return fail(h, PDMPC_ERR_BAD_INPUT, "upload_mpa: edge trim out of range");
        edge_of[(size_t)(f - 1) * nT + (t - 1)] = (int16_t)e;
        for (int k = 0; k < 3; ++k) {
            int np = d->area_npts[e * 3 + k];
            if (np < 2 || np > PDMPC_AREA_STRIDE) return fail(h, PDMPC_ERR_BAD_INPUT, "upload_mpa: area_npts out of range");
            if (k == PDMPC_AREA_NORMAL) max_npts = std::max(max_npts, np);
        }
    }
    // successor lists: find(transition_matrix_single(t,:,k)) ascending (expand_node.m:18)
    std::vector<int> succ_ptr((size_t)Hp * nT + 1, 0);
    std::vector<int> succ_te;
    h->max_branch = 0;
    for (int k = 0; k < Hp; ++k)
        for (int t = 0; t < nT; ++t) {
            const uint8_t *row = d->transition + ((size_t)k * nT + t) * nT;
            for (int j = 0; j < nT; ++j)
                if (row[j]) {
                    int e = edge_of[(size_t)t * nT + j];
                    if (e < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "upload_mpa: transition without maneuver");
                    succ_te.push_back((e << 8) | j);
                }
            succ_ptr[(size_t)k * nT + t + 1] = (int)succ_te.size();
            h->max_branch = std::max(h->max_branch, succ_ptr[(size_t)k * nT + t + 1] - succ_ptr[(size_t)k * nT + t]);
        }
    // capacity bound: nodes of the full tree from the worst start trim
    double worst = 1;
    for (int t0 = 0; t0 < nT; ++t0) {
        std::vector<double> cnt(nT, 0.0), nxt(nT);
        cnt[t0] = 1;
        double total = 1;
        for (int k = 0; k < Hp; ++k) {
            std::fill(nxt.begin(), nxt.end(), 0.0);
            for (int t = 0; t < nT; ++t)
                if (cnt[t] > 0) {
                    const uint8_t *row = d->transition + ((size_t)k * nT + t) * nT;
                    for (int j = 0; j < nT; ++j)
                        if (row[j]) nxt[j] += cnt[t];
                }
            cnt.swap(nxt);
            for (double c : cnt) total += c;
        }
        worst = std::max(worst, total);
    }
    h->full_tree_nodes = (int)std::min(worst, (double)(1 << 30));

    int64_t keep = h->stats.h2d_bytes;
    auto pad16 = [](size_t bytes) { return (bytes + 15) / 16 * 16; };
    auto padded = [&](auto &v, size_t elem) { v.resize(pad16(v.size() * elem) / elem); };
    padded(succ_ptr, sizeof(int));
    padded(succ_te, sizeof(int));
    std::vector<double> edge_d((size_t)nE * 4, 0.0);
    for (int e = 0; e < nE; ++e) {
        edge_d[(size_t)e * 4 + 0] = d->edge_dx[e];
        edge_d[(size_t)e * 4 + 1] = d->edge_dy[e];
        edge_d[(size_t)e * 4 + 2] = d->edge_dyaw[e];
    }
    std::vector<int> npts(d->area_npts, d->area_npts + (size_t)nE * 3);
    padded(npts, sizeof(int));
    // area points padded to the fixed stride by REPEATING THE LAST POINT: the kernels place all 8 columns without
    // looking at the point count first (one dependent table load less per pop), and the InterX row of a padded column
    // equals that of the last = first vertex
    std::vector<double> ax((size_t)nE * 3 * PDMPC_AREA_STRIDE, 0.0), ay(ax.size(), 0.0);
    bool closed = true;   // first point == last point, bit for bit (InterX shortcut b_last = b_first)
    for (int e = 0; e < nE * 3; ++e) {
        for (int i = 0; i < PDMPC_AREA_STRIDE; ++i) {
            const int src = std::min(i, d->area_npts[e] - 1);
            ax[(size_t)e * PDMPC_AREA_STRIDE + i] = d->area_x[(size_t)e * PDMPC_AREA_STRIDE + src];
            ay[(size_t)e * PDMPC_AREA_STRIDE + i] = d->area_y[(size_t)e * PDMPC_AREA_STRIDE + src];
        }
        const size_t f = (size_t)e * PDMPC_AREA_STRIDE, l = f + d->area_npts[e] - 1;
        if (memcmp(&ax[f], &ax[l], sizeof(double)) != 0 || memcmp(&ay[f], &ay[l], sizeof(double)) != 0) closed = false;
    }
    UP(h, h->m_succ_ptr, succ_ptr.data(), succ_ptr.size());
    UP(h, h->m_succ_te, succ_te.data(), succ_te.size());
    UP(h, h->m_edge_d, edge_d.data(), edge_d.size());
    UP(h, h->m_npts, npts.data(), npts.size());
    UP(h, h->m_ax, ax.data(), ax.size());
    UP(h, h->m_ay, ay.data(), ay.size());
    CU_TRY(h, cudaStreamSynchronize(h->stream));   // host vectors go out of scope
    h->stats.h2d_bytes = keep;
    MpaDev &m = h->mpa;
    m.nT = nT; m.Hp = Hp; m.nE = nE;
    m.succ_ptr = h->m_succ_ptr.as<int>();
    m.succ_te = h->m_succ_te.as<int>();
    m.edge_d = h->m_edge_d.as<double>();
    m.area_npts = h->m_npts.as<int>();
    m.areas_closed = closed ? 1 : 0;
    m.area_x = h->m_ax.as<double>(); m.area_y = h->m_ay.as<double>();
    m.bytes_succ_ptr = (unsigned)(succ_ptr.size() * sizeof(int));
    m.bytes_succ_te = (unsigned)(succ_te.size() * sizeof(int));
    m.bytes_edge_d = (unsigned)(edge_d.size() * sizeof(double));
    m.bytes_area_npts = (unsigned)(npts.size() * sizeof(int));
    m.bytes_area = (unsigned)(ax.size() * sizeof(double));
    m.table_bytes = m.bytes_succ_ptr + m.bytes_succ_te + m.bytes_edge_d + m.bytes_area_npts + 2 * m.bytes_area;
    h->has_mpa = true;
    h->max_area_npts = max_npts;
    h->staged = false;
    return PDMPC_OK;
}

static int validate_header(pdmpc_handle *h, const pdmpc_batch_in *in) {
    const int n = in->n_searches;
    if (n < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: n_searches < 0");
    if (in->checker != PDMPC_CHECKER_SAT && in->checker != PDMPC_CHECKER_INTERX)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan: unknown checker");
    if (!(in->dt_seconds > 0)) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: dt_seconds must be > 0");
    if (n == 0) return PDMPC_OK;
    if (!in->x0 || !in->y0 || !in->yaw0 || !in->trim0 || !in->ref_x || !in->ref_y || !in->v_ref ||
        !in->slot_ptr || !in->poly_ptr || !in->lane_ptr)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan: NULL input pointer");
    if (in->slot_ptr[0] != 0 || in->poly_ptr[0] != 0 || in->lane_ptr[0] != 0)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan: CSR offsets must start at 0");
    return PDMPC_OK;
}

// searches [s0, s1) of the batch (validate_header has passed)
static int validate_range(pdmpc_handle *h, const pdmpc_batch_in *in, int s0, int s1) {
    const int Hp = h->mpa.Hp, nT = h->mpa.nT;
    for (int i = s0; i < s1; ++i)
        if (in->trim0[i] < 1 || in->trim0[i] > nT) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: trim0 out of range");
    for (size_t s = (size_t)s0 * (Hp + 1); s < (size_t)s1 * (Hp + 1); ++s)
        if (in->slot_ptr[s + 1] < in->slot_ptr[s]) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: slot_ptr not monotone");
    const int np0 = in->slot_ptr[(size_t)s0 * (Hp + 1)], np = in->slot_ptr[(size_t)s1 * (Hp + 1)];
    for (int p = np0; p < np; ++p) {
        const int v0 = in->poly_ptr[p], v1 = in->poly_ptr[p + 1];
        if (v1 - v0 < 2) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: obstacle polygon with fewer than 2 vertices");
        if (!in->vert_x || !in->vert_y) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: NULL vertex arrays");
        // vectorize_all_obstacles.m:71-76 check_closeness (asserted by the reference for InterX)
        if (in->checker == PDMPC_CHECKER_INTERX &&
            !(in->vert_x[v0] == in->vert_x[v1 - 1] && in->vert_y[v0] == in->vert_y[v1 - 1]))
            return fail(h, PDMPC_ERR_BAD_INPUT, "plan: obstacle polygon is not closed");
    }
    for (int i = 2 * s0; i < 2 * s1; ++i)
        if (in->lane_ptr[i + 1] < in->lane_ptr[i]) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: lane_ptr not monotone");
    if (in->lane_ptr[2 * s1] > in->lane_ptr[2 * s0] && (!in->lane_x || !in->lane_y))
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan: NULL lanelet arrays");
    return PDMPC_OK;
}

static int validate_batch(pdmpc_handle *h, const pdmpc_batch_in *in) {
    int rc = validate_header(h, in);
    if (rc != PDMPC_OK || in->n_searches == 0) return rc;
    return validate_range(h, in, 0, in->n_searches);
}

constexpr size_t kPackLimit = 1u << 20;   // batches whose arrays total at most 1 MiB take the packed path

static int ensure_pinned(pdmpc_handle *h, PinnedBuf &buf, size_t bytes) {
    return buf.reserve(bytes) == cudaSuccess ? PDMPC_OK : fail(h, PDMPC_ERR_ALLOC, "pinned staging buffer allocation failed");
}

// All output arrays live in one device block (d_out_pack) so that a small batch needs a single
// device->host copy; the order is the one of pdmpc_batch_out, the counters come last.
static int ensure_outputs(pdmpc_handle *h, int n) {
    const OutFields f = out_fields(h->mpa.Hp);
    const size_t n1 = std::max(n, 1);
    size_t off = 0;
    for (int i = 0; i <= kNumOut; ++i) {
        h->out_off[i] = off;
        off = (off + (i < kNumOut ? n1 * f.bytes[i] : kCounterBytes) + 15) / 16 * 16;
    }
    h->out_bytes = off;
    CU_TRY(h, h->d_out_pack.reserve(off));
    CU_TRY(h, h->work_counter.reserve(4 * sizeof(unsigned)));   // [0] the search kernel, [1], [2] the escalation kernels
    unsigned char *base = h->d_out_pack.as<unsigned char>();
    OutDev &o = h->out;
    o.status = reinterpret_cast<int *>(base + h->out_off[0]);
    o.is_exhausted = reinterpret_cast<uint8_t *>(base + h->out_off[1]);
    o.n_expanded = reinterpret_cast<int *>(base + h->out_off[2]);
    o.n_pops = reinterpret_cast<int *>(base + h->out_off[3]);
    o.pop_hash = reinterpret_cast<unsigned long long *>(base + h->out_off[4]);
    o.trims = reinterpret_cast<int *>(base + h->out_off[5]);
    o.tree_path = reinterpret_cast<int *>(base + h->out_off[6]);
    o.y_predicted = reinterpret_cast<double *>(base + h->out_off[7]);
    o.g_path = reinterpret_cast<double *>(base + h->out_off[8]);
    o.h_path = reinterpret_cast<double *>(base + h->out_off[9]);
    o.shape_npts = reinterpret_cast<int *>(base + h->out_off[10]);
    o.shape_x = reinterpret_cast<double *>(base + h->out_off[11]);
    o.shape_y = reinterpret_cast<double *>(base + h->out_off[12]);
    o.counters = reinterpret_cast<unsigned long long *>(base + h->out_off[kNumOut]);
    return PDMPC_OK;
}

// The statistics in the counter block of a finished launch.
static void read_counters(pdmpc_handle *h, const unsigned long long counters[16]) {
    h->stats.total_pops = (int64_t)counters[0];
    h->stats.total_nodes = (int64_t)counters[1];
    h->stats.total_obstacle_cols = (int64_t)counters[2];
    if (counters[3]) h->stats.handed_over = (int32_t)counters[3];   // shape 5: searches re-run with the exact queue
    h->stats.escalated = (int32_t)counters[6];
#ifdef PDMPC_PROFILE
    {
#ifdef PDMPC_PROFILE_CHECKER
        static const char *names[8] = {"c:wait_job", "c:tables+place", "c:interx_obstacles", "c:interx_rest", "c:sincos+publish", "-", "-", "c:other"};
#else
        static const char *names[8] = {"setup", "heap_pop", "loads+place", "check", "expand", "heap_push", "wait_children", "loop"};
        // (CTA kernel master: set-up, pending children, loads + heap pop, flag wait, job hand-over, children, pushes, end)
#endif
        double tot = 0;
        for (int i = 0; i < 8; ++i) tot += (double)counters[8 + i];
        fprintf(stderr, "[pdmpc profile] cycles per pop:");
        for (int i = 0; i < 8; ++i)
            fprintf(stderr, " %s=%.0f", names[i], (double)counters[8 + i] / (double)std::max<unsigned long long>(counters[0], 1));
        fprintf(stderr, " total=%.0f\n", tot / (double)std::max<unsigned long long>(counters[0], 1));
        if (counters[5])
            fprintf(stderr, "[pdmpc profile] checker 0: %.0f cycles per job over %llu jobs\n",
                    (double)counters[4] / (double)counters[5], counters[5]);
    }
#endif
}

// InterX checker: NaN-separated polylines (vectorize_all_obstacles.m) of the obstacles and lanelet bounds, built on the
// device.  reserve_polylines sizes them for the staged batch with np polygons, nv vertices and nl lanelet points and
// names them in it (the SAT checker has none); build_polylines builds those of polygons [p0, p1) and of the lanelet
// bounds of searches [s0, s1) on stream S.
static int reserve_polylines(pdmpc_handle *h, int np, int nv, int nl) {
    BatchDev &b = h->batch;
    b.pl_x = b.pl_y = b.ll_x = b.ll_y = nullptr;
    b.pl_xy = b.ll_xy = nullptr;
    if (b.checker != PDMPC_CHECKER_INTERX) return PDMPC_OK;
    CU_TRY(h, h->b_plx.reserve(((size_t)nv + np + 1) * sizeof(double)));
    CU_TRY(h, h->b_ply.reserve(((size_t)nv + np + 1) * sizeof(double)));
    CU_TRY(h, h->b_llx.reserve(((size_t)nl + 2 * b.n + 1) * sizeof(double)));
    CU_TRY(h, h->b_lly.reserve(((size_t)nl + 2 * b.n + 1) * sizeof(double)));
    CU_TRY(h, h->b_plxy.reserve(((size_t)nv + np + 1) * sizeof(double2)));
    CU_TRY(h, h->b_llxy.reserve(((size_t)nl + 2 * b.n + 1) * sizeof(double2)));
    b.pl_x = h->b_plx.as<double>(); b.pl_y = h->b_ply.as<double>();
    b.ll_x = h->b_llx.as<double>(); b.ll_y = h->b_lly.as<double>();
    b.pl_xy = h->b_plxy.as<double2>(); b.ll_xy = h->b_llxy.as<double2>();
    return PDMPC_OK;
}
static void build_polylines(pdmpc_handle *h, int p0, int p1, int s0, int s1, cudaStream_t S) {
    const BatchDev &b = h->batch;
    if (p1 > p0) {
        build_polyline_kernel<<<(p1 - p0 + 127) / 128, 128, 0, S>>>(p1 - p0, b.poly_ptr, b.vert_x, b.vert_y, h->b_plx.as<double>(),
                                                                  h->b_ply.as<double>(), p0, h->b_plxy.as<double2>());
        h->stats.kernel_launches++;
    }
    if (s1 > s0) {
        build_polyline_kernel<<<(2 * (s1 - s0) + 127) / 128, 128, 0, S>>>(2 * (s1 - s0), b.lane_ptr, b.lane_x, b.lane_y,
                                                                        h->b_llx.as<double>(), h->b_lly.as<double>(), 2 * s0,
                                                                        h->b_llxy.as<double2>());
        h->stats.kernel_launches++;
    }
}

// The device side of staging: `dptr` = the batch's input arrays in device memory, np / nv / nl = its polygons, vertices
// and lanelet points; polylines of the InterX checker, output block.  Shared by the host-buffer path and
// pdmpc_plan_timestep_from_states.
static int stage_finish(pdmpc_handle *h, int n, int checker, double dt, const void *const dptr[kNumIn], int np, int nv, int nl) {
    set_batch(h->batch, n, checker, dt, dptr);
    h->stats.kernel_launches = 0;
    int rc = reserve_polylines(h, np, nv, nl);
    if (rc != PDMPC_OK) return rc;
    if (checker == PDMPC_CHECKER_INTERX) {
        build_polylines(h, 0, np, 0, n, h->stream);
        CU_TRY(h, cudaGetLastError());
    }
    rc = ensure_outputs(h, n);
    if (rc != PDMPC_OK) return rc;
    // (caller-owned source buffers were either copied into the pinned block or their copies
    // have completed above: the caller may reuse them)
    h->staged = true;
    return PDMPC_OK;
}


int pdmpc_stage_batch(pdmpc_handle *h, const pdmpc_batch_in *in) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "plan: call pdmpc_upload_mpa first");
    if (!in) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: batch is NULL");
    int rc = validate_batch(h, in);
    if (rc != PDMPC_OK) return rc;
    CU_TRY(h, cudaSetDevice(h->device));
    const int n = in->n_searches, Hp = h->mpa.Hp;
    const int np = n ? in->slot_ptr[(size_t)n * (Hp + 1)] : 0;
    const int nv = np ? in->poly_ptr[np] : 0;
    const int nl = n ? in->lane_ptr[2 * n] : 0;
    h->staged = false;
    h->stats.h2d_bytes = 0;
    CU_TRY(h, cudaEventRecord(h->ev[0], h->stream));
    static const int zero1[1] = {0};
    std::vector<int> order;
    h->deps_staged = false;
    if (n > 1 && (int)h->topo_order.size() == n) {
        order.swap(h->topo_order);   // pdmpc_plan_timestep: a topological order of the dependency DAG
    } else if (n > 1 && getenv("PDMPC_NO_REORDER")) {   // experiments: work order = batch order
        order.resize(n);
        for (int i = 0; i < n; ++i) order[i] = i;
    } else if (n > 1) {
        order.resize(n);
        heavy_first_order(in->slot_ptr, Hp, 0, n, order.data());
    }
    const void *srcs[kNumIn];
    in_sources(in, order.data(), srcs);
    if (n == 0) srcs[kInSlotPtr] = srcs[kInPolyPtr] = srcs[kInLanePtr] = zero1;
    const InRange all = in_range(Hp, 0, n, 0, np, 0, nv, 0, nl);
    size_t nbytes[kNumIn], in_off[kNumIn], in_total = 0;
    for (int i = 0; i < kNumIn; ++i) nbytes[i] = all.hi[i] * kInElem[i];
    nbytes[kInOrder] = order.size() * sizeof(int);   // a single search has none
    for (int i = 0; i < kNumIn; ++i) {
        in_off[i] = in_total;
        in_total = (in_total + nbytes[i] + 15) / 16 * 16;
    }
    const void *dptr[kNumIn];
    if (in_total <= kPackLimit) {
        // one pinned staging block, one host->device copy (a level of a time step is a few KB:
        // fifteen separate pageable copies cost more than the search itself)
        if (h->pack_in_flight) {
            CU_TRY(h, cudaEventSynchronize(h->ev_pack));
            h->pack_in_flight = false;
        }
        int rc2 = ensure_pinned(h, h->pin_in, std::max<size_t>(in_total, 16));
        if (rc2 != PDMPC_OK) return rc2;
        CU_TRY(h, h->d_in_pack.reserve(std::max<size_t>(in_total, 16)));
        unsigned char *pin = h->pin_in.as<unsigned char>();
        for (int i = 0; i < kNumIn; ++i) {
            if (nbytes[i]) memcpy(pin + in_off[i], srcs[i], nbytes[i]);
            dptr[i] = h->d_in_pack.as<unsigned char>() + in_off[i];
        }
        if (in_total) CU_TRY(h, cudaMemcpyAsync(h->d_in_pack.p, pin, in_total, cudaMemcpyHostToDevice, h->stream));
        CU_TRY(h, cudaEventRecord(h->ev_pack, h->stream));
        h->pack_in_flight = true;
        h->stats.h2d_bytes += (int64_t)in_total;
    } else {
        for (int i = 0; i < kNumIn; ++i) {
            int rc2 = upload(h, h->b_in[i], static_cast<const unsigned char *>(srcs[i]), nbytes[i]);
            if (rc2 != PDMPC_OK) return rc2;
            dptr[i] = h->b_in[i].p;
        }
        CU_TRY(h, cudaStreamSynchronize(h->stream));   // `order` goes out of scope; callers may reuse their buffers
    }
    CU_TRY(h, cudaEventRecord(h->ev[1], h->stream));
    h->timing_pending_h2d = true;

    return stage_finish(h, n, in->checker, in->dt_seconds, dptr, np, nv, nl);
}

// Node capacity of one search's arena: pdmpc_set_node_capacity, or the full tree from the worst start trim (at most
// 2^20 nodes), within what the node ids address.
static int node_cap(const pdmpc_handle *h) {
    const int cap = h->user_node_cap ? h->user_node_cap : std::min(h->full_tree_nodes + 8, 1 << 20);
    return std::max(std::min(cap, kMaxNodeCap - 1), 64);
}

// The CTA kernels (`deps`: their pdmpc_plan_timestep instances) can run: shared memory granted, and the validity flags
// of a whole search tree fit in shared memory.
static bool cta_launchable(const pdmpc_handle *h, bool deps) {
    return (deps ? h->cta_deps_ok : h->cta_ok) && node_cap(h) <= kCtaFlags;
}

static int ensure_arena(pdmpc_handle *h, int slots) {
    const int cap = node_cap(h);
    if (slots <= h->arena_slots && cap == h->arena.cap) return PDMPC_OK;
    slots = std::max(slots, h->arena_slots);
    const size_t tot = (size_t)slots * cap;
    // (DBuf::reserve frees before it allocates: until all four succeed the handle must not keep pointers
    // into buffers that may be gone — a failed call leaves NO arena, the next one allocates afresh)
    h->arena = ArenaDev{};
    h->arena_slots = 0;
    CU_TRY(h, h->a_a.reserve(tot * sizeof(NodeA)));
    CU_TRY(h, h->a_b.reserve(tot * sizeof(NodeB)));
    CU_TRY(h, h->a_cs.reserve(tot * sizeof(NodeCS)));
    CU_TRY(h, h->a_heap.reserve(tot * sizeof(HEnt)));
    h->arena.a = h->a_a.as<NodeA>();
    h->arena.b = h->a_b.as<NodeB>();
    h->arena.cs = h->a_cs.as<NodeCS>();
    h->arena.heap = h->a_heap.as<HEnt>();
    h->arena.cap = cap;
    h->arena_slots = slots;
    return PDMPC_OK;
}

// ---- warp-level launch shapes -------------------------------------------------------------------------
// Grid and arena slots (concurrently running searches, if `slots`) of shape `shape` for n searches.
static int warp_shape_grid(const pdmpc_handle *h, int shape, int n, int *slots = nullptr) {
    const bool tiles = shape == kShapeTile2 || shape == kShapeTile4;
    const int T = shape == kShapeTile2 ? 2 : shape == kShapeTile4 ? 4 : 1;
    const int per_sm = tiles ? h->tile_ctas_per_sm[shape - kShapeTile2] : h->lat_ctas_per_sm;
    const int grid = std::max(1, std::min((n + T - 1) / T, h->num_sms * per_sm));
    if (slots) *slots = grid * T;
    return grid;
}

// The shape a batch of n searches runs in when the caller asked for `variant` (kShapeAuto = choose).
static int resolve_warp_shape(const pdmpc_handle *h, int variant, int n, int checker, bool tracing) {
    if (tracing) return kShapeLatency;   // pop traces come from the one-search-per-warp kernel
    if (variant == kShapeAuto) {
        // more searches than the latency shape keeps in flight: share the warps (profiles/r02a_*)
        variant = n > h->num_sms * h->lat_ctas_per_sm ? kShapeTile2 : kShapeLatency;
    }
    if ((variant == kShapeTile2 || variant == kShapeTile4) &&
        (checker != PDMPC_CHECKER_INTERX || h->tile_ctas_per_sm[variant - kShapeTile2] < 1))
        variant = kShapeLatency;         // the tile shapes hold the InterX checker only
    return variant;
}

// One persistent launch of a warp-level shape over batch `bc` on stream S with arena `ar` (sized by warp_shape_grid).
static int launch_warp_shape(pdmpc_handle *h, int shape, const BatchDev &bc, const ArenaDev &ar, unsigned *wc,
                             const TraceDev &tr, cudaStream_t S) {
    const int grid = warp_shape_grid(h, shape, bc.n);
    if (shape == kShapeTile2) KERNEL_TILE2<<<grid, kWarp, kTile2Smem, S>>>(h->mpa, bc, h->out, ar, wc, tr, h->tile_pts_limit);
    else if (shape == kShapeTile4) KERNEL_TILE4<<<grid, kWarp, kTile4Smem, S>>>(h->mpa, bc, h->out, ar, wc, tr, h->tile_pts_limit);
    else KERNEL_LAT<<<grid, kWarp, sizeof(WarpSmem), S>>>(h->mpa, bc, h->out, ar, wc, tr);
    if (cudaGetLastError() != cudaSuccess) return fail(h, PDMPC_ERR_CUDA, "search kernel launch failed");
    h->stats.kernel_launches++;
    return PDMPC_OK;
}

// ---- escalation: the longest searches of a throughput launch go to the CTA shape ------------------------
// A tile warp runs a pop in ~5 us, so ONE search of 8000 pops (1 in 10^5 of the road-network records; nothing
// in its inputs tells it apart beforehand) holds the whole launch open for 40 ms.  The tile kernels therefore
// give a search up after `escalate_pops` pops and append its index to a list; two gated instances of the CTA
// kernel (one master per CTA for a short list, several masters for a long one) launched behind the tile kernel
// on the same stream run the list from scratch at 0.65-1.0 us per pop.  Results are those of any other shape.
// The threshold for a launch over n searches.  Measured after the tile kernel's InterX loop was rewritten
// (profiles/r02j_escalation_threshold.txt): the larger the batch, the smaller the launch's tail is against its
// body and the later giving up pays — 2560 pops is best at 56 k searches, 2560-3072 at 168 k, 4096 at 358 k.
static int escalation_pops(const pdmpc_handle *h, int n) {
    if (h->escalate_pops >= 0) return h->escalate_pops;
    return n >= 300000 ? 4096 : n >= 120000 ? 3072 : PDMPC_ESCALATE_POPS;
}
static bool escalation_on(const pdmpc_handle *h, int shape, int n) {
    return (shape == kShapeTile2 || shape == kShapeTile4) && escalation_pops(h, n) > 0 && cta_launchable(h, false) &&
           n > h->num_sms && h->batch.checker == PDMPC_CHECKER_INTERX;
}

// Resets the list (count, producers-done counter, entries = -1) on stream S and names it in the batch the tile
// kernels get.
static int escalation_prepare(pdmpc_handle *h, int n, BatchDev *bt, cudaStream_t S) {
    CU_TRY(h, h->esc.reserve(((size_t)n + 4) * sizeof(int)));
    CU_TRY(h, cudaMemsetAsync(h->esc.p, 0, 4 * sizeof(int), S));
    CU_TRY(h, cudaMemsetAsync(h->esc.as<int>() + 4, 0xff, (size_t)n * sizeof(int), S));
    bt->pop_limit = escalation_pops(h, n);
    bt->esc_count = h->esc.as<unsigned>();
    bt->esc_done = h->esc.as<unsigned>() + 1;
    bt->esc_list = h->esc.as<int>() + 4;
    return PDMPC_OK;
}

// The CTA kernel over the escalation list, on stream S behind the `producers` tile CTAs (all of them joined S).
// Measured (profiles/r02_escalation.txt): launched on a stream of its own BESIDE the tile kernel — the kernel
// polls the list and ends when every producer has exited — it is no faster: its 16-warp CTAs only fit an SM
// once most of the SM's tile CTAs have left, i.e. at the end anyway.  The kernel keeps the polling protocol
// (a list that is complete when it starts is its trivial case); `ar` = arena slots of its own.
static int launch_escalated(pdmpc_handle *h, const ArenaDev &ar, int producers, cudaStream_t S) {
    BatchDev be = h->batch;
    be.order = nullptr;
    be.esc_count = h->esc.as<unsigned>();
    be.esc_done = h->esc.as<unsigned>() + 1;
    be.esc_list = h->esc.as<int>() + 4;
    be.esc_producers = (unsigned)producers;
    const int fast = h->cta_valid_only ? 1 : 0;
    unsigned *wc = h->work_counter.as<unsigned>();
    // a short list: one master per CTA, all twelve checkers serve it (0.65 us per pop: the launch then ends with
    // its longest search, ~5 ms for 8000 pops); a long list: several masters per CTA
    be.esc_gate_lo = 0u; be.esc_gate_hi = (unsigned)(h->esc_short_list >= 0 ? h->esc_short_list : 3 * h->num_sms);
    KERNEL_CTA<<<h->num_sms, CtaShape<1, kCtaCheckers>::kThreads, sizeof(CtaSmemT), S>>>(
        h->mpa, be, h->out, ar, wc + 1, h->cta_heap_smem, fast, DepsDev{});
    be.esc_gate_lo = be.esc_gate_hi; be.esc_gate_hi = 0xffffffffu;
    KERNEL_CTAM<<<h->num_sms, CtaShape<kCtaMasters, kCtaCheckers>::kThreads, sizeof(CtaMSmemT), S>>>(
        h->mpa, be, h->out, ar, wc + 2, h->cta_heap_smem, fast, DepsDev{});
    if (cudaGetLastError() != cudaSuccess) return fail(h, PDMPC_ERR_CUDA, "escalation kernel launch failed");
    h->stats.kernel_launches += 2;
    return PDMPC_OK;
}

// Launches the search of the staged batch (results are identical for all shapes):
//   the warp-level shapes see above;  kShapeCta / kShapeCtaValid are chosen for at most one search per SM
static int launch_search(pdmpc_handle *h, const TraceDev &tr) {
    const int n = h->batch.n;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaMemsetAsync(h->out.counters, 0, kCounterBytes, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->work_counter.p, 0, 4 * sizeof(unsigned), h->stream));
    h->stats.handed_over = 0;
    h->stats.escalated = 0;
    h->stats.shape = 0;
    h->batch.hash_valid_only = h->cta_valid_only ? 1 : 0;
    if (n == 0) return PDMPC_OK;
    int shape = h->variant_mode;
    if (shape == kShapeAuto && n <= h->num_sms && tr.search < 0) shape = kShapeCta;   // one computation level of a time step
    const bool cta = shape == kShapeCta || shape == kShapeCtaValid;
    if (cta && (!cta_launchable(h, false) || tr.search >= 0)) shape = kShapeLatency;
    if (shape == kShapeCta && h->cta_valid_only) shape = kShapeCtaValid;
    if (shape < kShapeCta) shape = resolve_warp_shape(h, shape, n, h->batch.checker, tr.search >= 0);
    unsigned *wc = h->work_counter.as<unsigned>();
    h->stats.shape = shape;
    if (shape == kShapeCta || shape == kShapeCtaValid) {
        // at most one search per SM: one master per CTA, every checker serves it; else several masters per CTA
        const bool single = n <= h->num_sms;
        const int nm = single ? 1 : kCtaMasters;
        const int grid = std::min((n + nm - 1) / nm, h->num_sms);
        int rc = ensure_arena(h, grid * nm);
        if (rc != PDMPC_OK) return rc;
        CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
        if (single)
            KERNEL_CTA<<<grid, CtaShape<1, kCtaCheckers>::kThreads, sizeof(CtaSmemT), h->stream>>>(
                h->mpa, h->batch, h->out, h->arena, wc, h->cta_heap_smem, shape == kShapeCtaValid ? 1 : 0, DepsDev{});
        else
            KERNEL_CTAM<<<grid, CtaShape<kCtaMasters, kCtaCheckers>::kThreads, sizeof(CtaMSmemT), h->stream>>>(
                h->mpa, h->batch, h->out, h->arena, wc, h->cta_heap_smem, shape == kShapeCtaValid ? 1 : 0, DepsDev{});
        CU_TRY(h, cudaGetLastError());
        h->stats.kernel_launches++;
    } else {
        int slots = 0;
        warp_shape_grid(h, shape, n, &slots);
        const bool esc = escalation_on(h, shape, n) && tr.search < 0;
        int rc = ensure_arena(h, esc ? slots + h->num_sms * kCtaMasters : slots);
        if (rc != PDMPC_OK) return rc;
        BatchDev bt = h->batch;
        if (esc) {
            rc = escalation_prepare(h, n, &bt, h->stream);
            if (rc != PDMPC_OK) return rc;
        }
        CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
        rc = launch_warp_shape(h, shape, bt, h->arena, wc, tr, h->stream);
        if (rc != PDMPC_OK) return rc;
        if (esc) {   // its own slots behind the tile kernel's
            rc = launch_escalated(h, arena_from(h->arena, slots), warp_shape_grid(h, shape, n), h->stream);
            if (rc != PDMPC_OK) return rc;
        }
    }
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    h->timing_pending_kernel = true;
    return PDMPC_OK;
}

int pdmpc_run_staged(pdmpc_handle *h) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->staged) return fail(h, PDMPC_ERR_BAD_INPUT, "run_staged: no staged batch");
    TraceDev tr{-1, nullptr, 0, nullptr};
    return launch_search(h, tr);
}

int pdmpc_sync(pdmpc_handle *h) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return PDMPC_OK;
}

#define DOWN(h, dst, buf, count)                         \
    do {                                                 \
        int _rc = download(h, dst, buf, (size_t)(count)); \
        if (_rc != PDMPC_OK) return _rc;                 \
    } while (0)

int pdmpc_fetch_staged(pdmpc_handle *h, pdmpc_batch_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->staged) return fail(h, PDMPC_ERR_BAD_INPUT, "fetch: no staged batch");
    if (!out || !out->status) return fail(h, PDMPC_ERR_BAD_INPUT, "fetch: out/status is NULL");
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t n = (size_t)h->batch.n;
    const OutFields f = out_fields(h->mpa.Hp, out);
    h->stats.d2h_bytes = 0;
    unsigned long long counters[16] = {0};
    const unsigned char *dbase = h->d_out_pack.as<unsigned char>();
    CU_TRY(h, cudaEventRecord(h->ev[4], h->stream));
    if (h->out_bytes <= kPackLimit) {
        // one copy of the whole output block into pinned memory, then scatter on the host
        int rc = ensure_pinned(h, h->pin_out, h->out_bytes);
        if (rc != PDMPC_OK) return rc;
        CU_TRY(h, cudaMemcpyAsync(h->pin_out.p, dbase, h->out_bytes, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaEventRecord(h->ev[5], h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        const unsigned char *src = h->pin_out.as<const unsigned char>();
        for (int i = 0; i < kNumOut; ++i)
            if (f.dst[i] && n) memcpy(f.dst[i], src + h->out_off[i], n * f.bytes[i]);
        memcpy(counters, src + h->out_off[kNumOut], sizeof(counters));
        h->stats.d2h_bytes = (int64_t)h->out_bytes;
    } else {
        for (int i = 0; i < kNumOut; ++i)
            if (f.dst[i] && n) {
                CU_TRY(h, cudaMemcpyAsync(f.dst[i], dbase + h->out_off[i], n * f.bytes[i], cudaMemcpyDeviceToHost, h->stream));
                h->stats.d2h_bytes += (int64_t)(n * f.bytes[i]);
            }
        CU_TRY(h, cudaMemcpyAsync(counters, dbase + h->out_off[kNumOut], sizeof(counters), cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaEventRecord(h->ev[5], h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
    }
    h->timing_pending_d2h = true;
    read_counters(h, counters);
    return PDMPC_OK;
}

// Output rows of the escalated searches, packed (pipeline: their slices went to the host before the CTA
// kernels wrote them).  One warp per item; row = the 13 output fields of one search, each padded to 8 bytes.
struct PackDesc {
    const unsigned char *src[kNumOut];
    int bytes[kNumOut], off[kNumOut];
    int row_bytes;
};
__global__ void pack_rows_kernel(PackDesc d, const unsigned *count, const int *list, unsigned char *rows) {
    const unsigned n = *count;
    const int lane = threadIdx.x % 32;
    for (unsigned j = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32; j < n; j += gridDim.x * (blockDim.x / 32)) {
        const size_t si = (size_t)list[j];
        unsigned char *row = rows + (size_t)j * d.row_bytes;
        for (int f = 0; f < kNumOut; ++f) {
            if (!d.src[f]) continue;
            const unsigned char *s = d.src[f] + si * (size_t)d.bytes[f];
            for (int q = lane; q < d.bytes[f]; q += 32) row[d.off[f] + q] = s[q];
        }
    }
}

// pdmpc_pack_plan_rows: one thread per (row, column).  Row layout (doubles), L = 2 + 21 * Hp:
//   [0] cost  [1] fallback flag  [2, 2+Hp) trims 1..Hp  [.., +3Hp) y_predicted  [.., +Hp) shape_npts
//   [.., +8Hp) shape_x  [.., +8Hp) shape_y
__global__ void pack_plan_rows_kernel(OutDev o, int Hp, int n_rows, int n_veh, const double *fb, double *dst) {
    const int L = 2 + 21 * Hp;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < (long long)n_rows * L;
         idx += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(idx / L), c = (int)(idx % L);
        double v;
        if (o.is_exhausted[r]) {
            v = fb ? fb[(size_t)(r % n_veh) * L + c] : 0.0;
            if (c == 1) v = 1.0;
        } else if (c == 0) v = o.g_path[(size_t)r * (Hp + 1) + Hp];     // tree.get_cost(tree_path(end))
        else if (c == 1) v = 0.0;
        else if (c < 2 + Hp) v = (double)o.trims[(size_t)r * (Hp + 1) + (c - 2) + 1];
        else if (c < 2 + 4 * Hp) v = o.y_predicted[(size_t)r * Hp * 3 + (c - 2 - Hp)];
        else if (c < 2 + 5 * Hp) v = (double)o.shape_npts[(size_t)r * Hp + (c - 2 - 4 * Hp)];
        else if (c < 2 + 13 * Hp) v = o.shape_x[(size_t)r * Hp * kAreaStride + (c - 2 - 5 * Hp)];
        else v = o.shape_y[(size_t)r * Hp * kAreaStride + (c - 2 - 13 * Hp)];
        dst[idx] = v;
    }
}

int pdmpc_set_escalation(pdmpc_handle *h, int32_t pops, int32_t short_list_max) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (pops < -1) return fail(h, PDMPC_ERR_BAD_INPUT, "escalation threshold must be -1 (by batch size), 0 (off) or a pop count");
    h->escalate_pops = pops;
    h->esc_short_list = short_list_max;
    return PDMPC_OK;
}

// ---- large host batches: chunked pipeline ---------------------------------------------------------
// The searches are cut into C contiguous chunks.  Chunk c's input slices go host->device on a copy
// stream while earlier chunks are searched; the chunks' persistent search kernels rotate over up to
// eight compute streams (each with its own node arena): a chunk's kernel is pending as soon as its
// inputs have landed, so its long searches start early and its one-warp CTAs take over the SMs as the
// searches of the other chunks drain; results come back on another copy stream.  CSR offsets stay global (every array is allocated for
// the whole batch), so the device ends up holding exactly what pdmpc_stage_batch would have staged.
constexpr int kPipelineMinSearches = 16384;
constexpr int kPipelineMaxChunks = 16;

static int pipeline_sync_all(pdmpc_handle *h) {
    cudaError_t e = cudaSuccess, e2;
    for (cudaStream_t st : h->s_comp)
        if (st && (e2 = cudaStreamSynchronize(st)) != cudaSuccess) e = e2;
    for (cudaStream_t st : {h->s_in, h->s_out, h->stream})
        if (st && (e2 = cudaStreamSynchronize(st)) != cudaSuccess) e = e2;
    return e == cudaSuccess ? PDMPC_OK : fail(h, PDMPC_ERR_CUDA, std::string("pipeline sync: ") + cudaGetErrorString(e));
}

// Chunk boundaries of the pipeline: bnd[c] .. bnd[c + 1] are the searches of chunk c.  C chunks of equal size, the first
// one half of that (nothing overlaps the first chunk's validation and copy); C = C_req (pdmpc_set_pipeline_chunks) or, by
// default, ~60 k searches per chunk (at most 12 chunks).
// Measured and NOT the default (profiles/r02k_pipeline_timeline.txt): sizes doubling from 24 k searches (24 k / 48 k / 96 k /
// 190 k at 358 400 records) are 4 % faster on ONE GPU (83.1 against 86.8 ms per call) and 17 % SLOWER when eight processes
// share one host (25.4 M against 30.7 M plans/s end to end on 8 GPUs): the copies of the large last chunk run at a
// fraction of the bandwidth then, its results come back exposed behind the last searches.
static std::vector<int> pipeline_bounds(int n, int C_req) {
    const int C = C_req > 1 ? C_req : std::min(12, std::max(2, n / 60000));
    constexpr double first_frac = 0.5;
    std::vector<int> bnd(1, 0);
    for (int c = 1; c < C; ++c)
        bnd.push_back(C < 3 ? (int)((long long)n * c / C)
                            : (int)((double)n * ((double)(c - 1) + first_frac) / ((double)(C - 1) + first_frac)));
    bnd.push_back(n);
    return bnd;
}

static int plan_batch_pipelined(pdmpc_handle *h, const pdmpc_batch_in *in, pdmpc_batch_out *out, int C_req) {
    int rc = validate_header(h, in);
    if (rc != PDMPC_OK) return rc;
    if (!out || !out->status) return fail(h, PDMPC_ERR_BAD_INPUT, "fetch: out/status is NULL");
    CU_TRY(h, cudaSetDevice(h->device));
    const int n = in->n_searches, Hp = h->mpa.Hp;
    const std::vector<int> bnd = pipeline_bounds(n, C_req);   // chunk c covers the searches [bnd[c], bnd[c + 1])
    const int C = (int)bnd.size() - 1;
    const int np = in->slot_ptr[(size_t)n * (Hp + 1)];
    if (np < 0 || (np > 0 && (!in->vert_x || !in->vert_y)))
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan: malformed obstacle CSR");
    const int nv = np ? in->poly_ptr[np] : 0, nl = in->lane_ptr[2 * n];
    if (nv < 0 || nl < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "plan: malformed CSR totals");
    const bool interx = in->checker == PDMPC_CHECKER_INTERX;
    h->staged = false;
    h->deps_staged = false;
    if (!h->s_in) {
        CU_TRY(h, cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
        for (auto &st : h->s_comp) CU_TRY(h, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        CU_TRY(h, cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
        CU_TRY(h, cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    }
    while ((int)h->ev_chunk.size() < 2 * C) {
        cudaEvent_t e;
        CU_TRY(h, cudaEventCreate(&e));
        h->ev_chunk.push_back(e);
    }
    // ---- device arrays for the whole batch ----------------------------------------------------
    const InRange all = in_range(Hp, 0, n, 0, np, 0, nv, 0, nl);
    const void *dptr[kNumIn];
    for (int i = 0; i < kNumIn; ++i) {
        CU_TRY(h, h->b_in[i].reserve(std::max<size_t>(all.hi[i], 1) * kInElem[i]));
        dptr[i] = h->b_in[i].p;
    }
    BatchDev &b = h->batch;
    set_batch(b, n, in->checker, in->dt_seconds, dptr);
    rc = reserve_polylines(h, np, nv, nl);
    if (rc != PDMPC_OK) return rc;
    rc = ensure_outputs(h, n);
    if (rc != PDMPC_OK) return rc;
    rc = ensure_pinned(h, h->pin_order, (size_t)n * sizeof(int));
    if (rc != PDMPC_OK) return rc;
    CU_TRY(h, h->wc_chunks.reserve(kPipelineMaxChunks * sizeof(unsigned)));
    // one-warp CTAs leave an SM one by one as their searches end, so the next chunk's CTAs move in early
    constexpr int kLanes = 8;   // most concurrent chunk kernels (streams, arenas)
    int per_chunk = 1;
    for (int c = 0; c < C; ++c) per_chunk = std::max(per_chunk, bnd[c + 1] - bnd[c]);
    const int shape = resolve_warp_shape(h, h->variant_mode, per_chunk, in->checker, false);
    int slots = 0;
    warp_shape_grid(h, shape, per_chunk, &slots);
    int lanes = std::min(C, kLanes);
    {   // node arenas of all lanes within 32 GiB
        const double per_lane = (double)slots * node_cap(h) * (sizeof(NodeA) + sizeof(NodeB) + sizeof(NodeCS) + sizeof(HEnt));
        lanes = std::max(2, std::min(lanes, (int)(32.0 * 1024 * 1024 * 1024 / per_lane)));
    }
    const bool esc = escalation_on(h, shape, n);
    rc = ensure_arena(h, esc ? lanes * slots + h->num_sms * kCtaMasters : lanes * slots);
    if (rc != PDMPC_OK) return rc;
    cudaStream_t comp[kLanes] = {h->stream, h->s_comp[0], h->s_comp[1], h->s_comp[2],
                                 h->s_comp[3], h->s_comp[4], h->s_comp[5], h->s_comp[6]};
    h->stats.h2d_bytes = 0;
    h->stats.d2h_bytes = 0;
    h->stats.kernel_launches = 0;
    h->stats.handed_over = 0;
    h->stats.escalated = 0;
    h->stats.shape = shape;
    b.hash_valid_only = h->cta_valid_only ? 1 : 0;
    b.pop_limit = 0; b.esc_list = nullptr; b.esc_count = nullptr; b.esc_done = nullptr; b.esc_producers = 0;
    BatchDev bproto = b;     // what the chunk kernels see: + the escalation list

    CU_TRY(h, cudaMemsetAsync(h->out.counters, 0, kCounterBytes, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->wc_chunks.p, 0, kPipelineMaxChunks * sizeof(unsigned), h->stream));
    CU_TRY(h, cudaMemsetAsync(h->work_counter.p, 0, 4 * sizeof(unsigned), h->stream));
    if (esc) {
        rc = escalation_prepare(h, n, &bproto, h->stream);
        if (rc != PDMPC_OK) return rc;
        rc = ensure_pinned(h, h->pin_esc, 4096);
        if (rc != PDMPC_OK) return rc;
    }
    CU_TRY(h, cudaEventRecord(h->ev_fork, h->stream));
    for (auto &st : h->s_comp) CU_TRY(h, cudaStreamWaitEvent(st, h->ev_fork, 0));
    CU_TRY(h, cudaStreamWaitEvent(h->s_in, h->ev_fork, 0));
    CU_TRY(h, cudaEventRecord(h->ev[0], h->s_in));
    CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
    bool d2h_started = false;
    int esc_producers = 0;   // tile CTAs launched: the escalation kernel ends when all of them have
    int *pin_order = h->pin_order.as<int>();
    const void *srcs[kNumIn];
    in_sources(in, pin_order, srcs);
    const OutFields f = out_fields(Hp, out);
    const TraceDev tr{-1, nullptr, 0, nullptr};
    const unsigned char *dbase = h->d_out_pack.as<unsigned char>();
    auto bail = [&](int code) {
        pipeline_sync_all(h);
        return code;
    };
    const auto t_call = std::chrono::steady_clock::now();
    h->chunk_host_ms.assign(C, 0.0);
    h->chunks_last = C;
    for (int c = 0; c < C; ++c) {
        const int s0 = bnd[c], s1 = bnd[c + 1];
        if (s1 == s0) continue;
        const int p0 = in->slot_ptr[(size_t)s0 * (Hp + 1)], p1 = in->slot_ptr[(size_t)s1 * (Hp + 1)];
        const int v0 = in->poly_ptr[p0], v1 = in->poly_ptr[p1];
        const int l0 = in->lane_ptr[2 * s0], l1 = in->lane_ptr[2 * s1];
        if (p0 < 0 || p1 > np || p1 < p0 || v0 < 0 || v1 > nv || v1 < v0 || l0 < 0 || l1 > nl || l1 < l0)   // the arrays were sized from the totals
            return bail(fail(h, PDMPC_ERR_BAD_INPUT, "plan: CSR offsets exceed their totals"));
        if (!heavy_first_order(in->slot_ptr, Hp, s0, s1, pin_order + s0))
            return bail(fail(h, PDMPC_ERR_BAD_INPUT, "plan: slot_ptr not monotone"));   // (validated in full below)
        const InRange r = in_range(Hp, s0, s1, p0, p1, v0, v1, l0, l1);
        for (int i = 0; i < kNumIn; ++i) {
            if (r.hi[i] <= r.lo[i]) continue;
            const size_t e = kInElem[i], bytes = (r.hi[i] - r.lo[i]) * e;
            if (cudaMemcpyAsync(h->b_in[i].as<unsigned char>() + r.lo[i] * e,
                                static_cast<const unsigned char *>(srcs[i]) + r.lo[i] * e, bytes, cudaMemcpyHostToDevice,
                                h->s_in) != cudaSuccess)
                return bail(fail(h, PDMPC_ERR_CUDA, std::string("pipeline H2D: ") + cudaGetErrorString(cudaGetLastError())));
            h->stats.h2d_bytes += (int64_t)bytes;
        }
        // the slice is validated while it is on its way (its copies only needed the offsets checked above); nothing of
        // the chunk runs before that
        rc = validate_range(h, in, s0, s1);
        if (rc != PDMPC_OK) return bail(rc);
        cudaEvent_t ev_in = h->ev_chunk[2 * c], ev_done = h->ev_chunk[2 * c + 1];
        cudaStream_t S = comp[c % lanes];
        if (cudaEventRecord(ev_in, h->s_in) != cudaSuccess || cudaStreamWaitEvent(S, ev_in, 0) != cudaSuccess)
            return bail(fail(h, PDMPC_ERR_CUDA, "pipeline: event"));
        if (interx) build_polylines(h, p0, p1, s0, s1, S);
        BatchDev bc = bproto;
        bc.n = s1 - s0;
        bc.order = b.order + s0;
        unsigned *wc = h->wc_chunks.as<unsigned>() + c;
        if (launch_warp_shape(h, shape, bc, arena_from(h->arena, (size_t)(c % lanes) * slots), wc, tr, S) != PDMPC_OK)
            return bail(PDMPC_ERR_CUDA);
        esc_producers += warp_shape_grid(h, shape, bc.n);
        if (cudaGetLastError() != cudaSuccess || cudaEventRecord(ev_done, S) != cudaSuccess ||
            cudaStreamWaitEvent(h->s_out, ev_done, 0) != cudaSuccess)
            return bail(fail(h, PDMPC_ERR_CUDA, "pipeline: search kernel launch failed"));
        h->chunk_host_ms[c] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count();
        if (!d2h_started) {
            cudaEventRecord(h->ev[4], h->s_out);
            d2h_started = true;
        }
        for (int i = 0; i < kNumOut; ++i) {
            if (!f.dst[i]) continue;
            const size_t o0 = (size_t)s0 * f.bytes[i], bytes = (size_t)(s1 - s0) * f.bytes[i];
            if (cudaMemcpyAsync(static_cast<unsigned char *>(f.dst[i]) + o0, dbase + h->out_off[i] + o0, bytes,
                                cudaMemcpyDeviceToHost, h->s_out) != cudaSuccess)
                return bail(fail(h, PDMPC_ERR_CUDA, "pipeline D2H failed"));
            h->stats.d2h_bytes += (int64_t)bytes;
        }
    }
    for (int c = 0; c < C; ++c)   // every chunk joins the handle's stream
        if (c % lanes != 0 && bnd[c + 1] > bnd[c])
            CU_TRY(h, cudaStreamWaitEvent(h->stream, h->ev_chunk[2 * c + 1], 0));
    if (esc) {   // the searches the chunk kernels give up: CTA shape, all chunks' leftovers in one launch
        rc = launch_escalated(h, arena_from(h->arena, (size_t)lanes * slots), esc_producers, h->stream);
        if (rc != PDMPC_OK) return bail(rc);
        CU_TRY(h, cudaMemcpyAsync(h->pin_esc.p, h->esc.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    }
    CU_TRY(h, cudaEventRecord(h->ev[1], h->s_in));
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    if (esc) {   // the counters are complete after the escalated searches
        CU_TRY(h, cudaEventRecord(h->ev_fork, h->stream));
        CU_TRY(h, cudaStreamWaitEvent(h->s_out, h->ev_fork, 0));
    }
    unsigned long long counters[16] = {0};
    CU_TRY(h, cudaMemcpyAsync(counters, dbase + h->out_off[kNumOut], sizeof(counters), cudaMemcpyDeviceToHost, h->s_out));
    CU_TRY(h, cudaEventRecord(h->ev[5], h->s_out));
    rc = pipeline_sync_all(h);
    if (rc != PDMPC_OK) return rc;
    if (esc && *h->pin_esc.as<const unsigned>() > 0) {
        // their output rows: packed on the device, one copy, scattered into the caller's arrays
        const unsigned cnt = *h->pin_esc.as<const unsigned>();
        PackDesc pd;
        int off = 0;
        for (int i = 0; i < kNumOut; ++i) {
            pd.src[i] = f.dst[i] ? dbase + h->out_off[i] : nullptr;
            pd.bytes[i] = (int)f.bytes[i];
            pd.off[i] = off;
            off += ((int)f.bytes[i] + 7) / 8 * 8;
        }
        pd.row_bytes = off;
        const size_t list_bytes = ((size_t)cnt * sizeof(int) + 15) / 16 * 16;
        CU_TRY(h, h->esc_rows.reserve((size_t)cnt * off));
        rc = ensure_pinned(h, h->pin_esc, list_bytes + (size_t)cnt * off);
        if (rc != PDMPC_OK) return rc;
        pack_rows_kernel<<<std::min<unsigned>((cnt + 3) / 4, 256u), 128, 0, h->stream>>>(
            pd, h->esc.as<unsigned>(), h->esc.as<int>() + 4, h->esc_rows.as<unsigned char>());
        CU_TRY(h, cudaGetLastError());
        h->stats.kernel_launches++;
        unsigned char *pin = h->pin_esc.as<unsigned char>();
        CU_TRY(h, cudaMemcpyAsync(pin, h->esc.as<int>() + 4, (size_t)cnt * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaMemcpyAsync(pin + list_bytes, h->esc_rows.p, (size_t)cnt * off, cudaMemcpyDeviceToHost, h->stream));
        CU_TRY(h, cudaStreamSynchronize(h->stream));
        const int *list = reinterpret_cast<const int *>(pin);
        for (unsigned j = 0; j < cnt; ++j) {
            const unsigned char *row = pin + list_bytes + (size_t)j * off;
            for (int i = 0; i < kNumOut; ++i)
                if (f.dst[i]) memcpy(static_cast<unsigned char *>(f.dst[i]) + (size_t)list[j] * f.bytes[i], row + pd.off[i], f.bytes[i]);
        }
        h->stats.d2h_bytes += (int64_t)(list_bytes + (size_t)cnt * off);
    }
    h->timing_pending_h2d = h->timing_pending_kernel = h->timing_pending_d2h = true;
    read_counters(h, counters);
    h->staged = true;   // the device holds the whole batch: pdmpc_run_staged / pdmpc_fetch_staged work on it
    return PDMPC_OK;
}

int pdmpc_pipeline_bounds(int32_t n_searches, int32_t chunks, int32_t cap, int32_t *bounds, int32_t *n_chunks) {
    if (n_searches < 2 || chunks < 0 || chunks == 1 || chunks > kPipelineMaxChunks || !bounds || !n_chunks) return PDMPC_ERR_BAD_INPUT;
    const std::vector<int> bnd = pipeline_bounds(n_searches, chunks);
    *n_chunks = (int32_t)bnd.size() - 1;
    if ((int)bnd.size() > cap) return PDMPC_ERR_CAPACITY;
    for (size_t i = 0; i < bnd.size(); ++i) bounds[i] = bnd[i];
    return PDMPC_OK;
}

int pdmpc_get_pipeline_timeline(pdmpc_handle *h, int32_t cap, double *host_ms, double *in_ms, double *done_ms, int32_t *n_chunks) {
    if (!h || !n_chunks) return PDMPC_ERR_BAD_INPUT;
    CU_TRY(h, cudaSetDevice(h->device));
    if (pipeline_sync_all(h) != PDMPC_OK) return PDMPC_ERR_CUDA;
    *n_chunks = h->chunks_last;
    for (int c = 0; c < h->chunks_last && c < cap; ++c) {
        float a = 0.f, b = 0.f;
        if ((int)h->ev_chunk.size() < 2 * c + 2 || cudaEventElapsedTime(&a, h->ev[0], h->ev_chunk[2 * c]) != cudaSuccess ||
            cudaEventElapsedTime(&b, h->ev[0], h->ev_chunk[2 * c + 1]) != cudaSuccess) {
            cudaGetLastError();
            a = b = -1.f;
        }
        if (host_ms) host_ms[c] = h->chunk_host_ms[c];
        if (in_ms) in_ms[c] = a;
        if (done_ms) done_ms[c] = b;
    }
    return PDMPC_OK;
}

int pdmpc_set_pipeline_chunks(pdmpc_handle *h, int32_t chunks) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (chunks < 0 || chunks > kPipelineMaxChunks)
        return fail(h, PDMPC_ERR_BAD_INPUT, "pipeline chunks must be 0 (auto), 1 (off) or 2..16");
    h->pipeline_chunks = chunks;
    return PDMPC_OK;
}

int pdmpc_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, pdmpc_batch_out *out) {
    if (h && in && h->has_mpa && h->pipeline_chunks != 1 && h->variant_mode < kShapeCta &&
        (h->pipeline_chunks > 1 ? in->n_searches >= 2 * h->pipeline_chunks : in->n_searches >= kPipelineMinSearches)) {
        return plan_batch_pipelined(h, in, out, h->pipeline_chunks > 1 ? h->pipeline_chunks : 0);
    }
    int rc = pdmpc_stage_batch(h, in);
    if (rc != PDMPC_OK) return rc;
    rc = pdmpc_run_staged(h);
    if (rc != PDMPC_OK) return rc;
    return pdmpc_fetch_staged(h, out);
}

// One whole time step (or many) as ONE dependency-ordered launch: see include/pdmpc_b200.h.
// slot / standstill != NULL: the closed-loop variant — fallback plans come from (and final plans go to) the state on
// the device (pdmpc_fallback.cuh); deps->fb_* are then ignored.
// `dev` != NULL: the batch is in device memory already (pdmpc_plan_timestep_from_states: its input arrays but the work
// order, dev_totals = polygons, vertices, lanelet points); `in` then only carries n_searches, checker and dt_seconds.
static int plan_timestep_impl(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                              pdmpc_batch_out *out, const int32_t *slot, const uint8_t *standstill,
                              const void **dev = nullptr, const int *dev_totals = nullptr) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "plan_timestep: call pdmpc_upload_mpa first");
    if (!in || !deps || !deps->pred_ptr) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: NULL argument");
    const int n = in->n_searches, Hp = h->mpa.Hp;
    if (n < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: n_searches < 0");
    // launch shape: one CTA per search (lowest latency) for up to 48 searches per SM, else — and for search
    // trees beyond what that kernel holds — one warp per search; pdmpc_set_variant 1..3 / 4..5 force either
    bool use_cta;
    {
        const bool cta_possible = cta_launchable(h, true);
        if (h->variant_mode >= kShapeCta) use_cta = cta_possible;
        else if (h->variant_mode >= kShapeLatency) use_cta = false;
        // measured (profiles/r01h_closed_loop_sweep.txt): a time step is bound by its chains of dependent
        // searches, so the 2.5x lower per-pop latency of the CTA shape beats the 12x higher concurrency of the
        // warp shape up to several thousand searches per call
        else use_cta = cta_possible && n <= 48 * h->num_sms;
        if (!use_cta && !h->lat_deps_ok)
            return fail(h, PDMPC_ERR_CUDA, "plan_timestep: search kernel is not launchable on this device");
    }
    // ---- validate the relation, order the searches topologically (utility/kahn.m:1-24) ----------
    if (deps->pred_ptr[0] != 0) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: pred_ptr must start at 0");
    for (int i = 0; i < n; ++i) {
        const int np = deps->pred_ptr[i + 1] - deps->pred_ptr[i];
        if (np < 0) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: pred_ptr not monotone");
        if ((long long)np * Hp * PDMPC_AREA_STRIDE > PDMPC_TIMESTEP_COLS)
            return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: too many predecessors for one search (PDMPC_TIMESTEP_COLS)");
    }
    const int total = n ? deps->pred_ptr[n] : 0;
    if (total > 0 && !deps->pred_idx) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: pred_idx is NULL");
    if (deps->fb_npts && (!deps->fb_x || !deps->fb_y))
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: fallback areas without coordinates");
    if (deps->fb_npts)
        for (size_t i = 0; i < (size_t)n * Hp; ++i) {
            const int np = deps->fb_npts[i];
            if (np != 0 && (np < 2 || np > PDMPC_AREA_STRIDE - 1))
                return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: fb_npts must be 0 or 2..PDMPC_AREA_STRIDE-1");
        }
    std::vector<int> indeg(n, 0), succ_ptr(n + 1, 0), succ(total), order;
    for (int i = 0; i < n; ++i)
        for (int q = deps->pred_ptr[i]; q < deps->pred_ptr[i + 1]; ++q) {
            const int j = deps->pred_idx[q];
            if (j < 0 || j >= n || j == i) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: pred_idx out of range");
            succ_ptr[j + 1]++;
            indeg[i]++;
        }
    for (int i = 0; i < n; ++i) succ_ptr[i + 1] += succ_ptr[i];
    {
        std::vector<int> fill(succ_ptr.begin(), succ_ptr.end() - 1);
        for (int i = 0; i < n; ++i)
            for (int q = deps->pred_ptr[i]; q < deps->pred_ptr[i + 1]; ++q) succ[fill[deps->pred_idx[q]]++] = i;
    }
    order.reserve(n);
    for (int i = 0; i < n; ++i)
        if (indeg[i] == 0) order.push_back(i);
    for (size_t head = 0; head < order.size(); ++head) {   // FIFO: level-major
        const int j = order[head];
        for (int q = succ_ptr[j]; q < succ_ptr[j + 1]; ++q)
            if (--indeg[succ[q]] == 0) order.push_back(succ[q]);
    }
    if ((int)order.size() != n) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: the predecessor relation has a cycle");

    if (in->checker == PDMPC_CHECKER_INTERX && h->max_area_npts >= PDMPC_AREA_STRIDE)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep: the InterX hand-over keeps one NaN column after each planned area: "
                                            "maneuver areas must have at most PDMPC_AREA_STRIDE - 1 points");
    int rc;
    if (dev) {
        CU_TRY(h, cudaSetDevice(h->device));
        h->staged = false;
        h->deps_staged = false;
        CU_TRY(h, cudaEventRecord(h->ev[0], h->stream));
        UP(h, h->b_in[kInOrder], order.data(), n);      // the only array that still comes from the host
        CU_TRY(h, cudaStreamSynchronize(h->stream));   // `order` is pageable
        CU_TRY(h, cudaEventRecord(h->ev[1], h->stream));
        h->timing_pending_h2d = true;
        dev[kInOrder] = h->b_in[kInOrder].p;
        rc = stage_finish(h, n, in->checker, in->dt_seconds, dev, dev_totals[0], dev_totals[1], dev_totals[2]);
    } else {
        h->topo_order.swap(order);
        rc = pdmpc_stage_batch(h, in);
        h->topo_order.clear();
    }
    if (rc != PDMPC_OK) return rc;
    if (n == 0) {
        rc = pdmpc_run_staged(h);
        return rc != PDMPC_OK ? rc : pdmpc_fetch_staged(h, out);
    }
    // ---- dependency CSR + fallback areas: one pinned block, one copy ------------------------------
    const size_t nhp = (size_t)n * Hp;
    const bool closed_loop = slot != nullptr;
    const bool has_fb = !closed_loop && deps->fb_npts != nullptr;
    const size_t sz[5] = {((size_t)n + 1) * sizeof(int), (size_t)std::max(total, 1) * sizeof(int),
                          has_fb ? nhp * sizeof(int) : 0, has_fb ? nhp * PDMPC_AREA_STRIDE * sizeof(double) : 0,
                          has_fb ? nhp * PDMPC_AREA_STRIDE * sizeof(double) : 0};
    const void *src[5] = {deps->pred_ptr, deps->pred_idx, deps->fb_npts, deps->fb_x, deps->fb_y};
    size_t off[5], tot = 0;
    for (int i = 0; i < 5; ++i) {
        off[i] = tot;
        tot = (tot + sz[i] + 15) / 16 * 16;
    }
    rc = ensure_pinned(h, h->pin_deps, tot);
    if (rc != PDMPC_OK) return rc;
    CU_TRY(h, h->d_deps.reserve(tot));
    CU_TRY(h, h->d_done.reserve((size_t)n * sizeof(int)));
    unsigned char *pin = h->pin_deps.as<unsigned char>();
    for (int i = 0; i < 5; ++i)
        if (sz[i] && src[i]) memcpy(pin + off[i], src[i], i == 1 ? (size_t)total * sizeof(int) : sz[i]);
    CU_TRY(h, cudaMemcpyAsync(h->d_deps.p, pin, tot, cudaMemcpyHostToDevice, h->stream));
    h->stats.h2d_bytes += (int64_t)tot;
    CU_TRY(h, cudaMemsetAsync(h->d_done.p, 0, (size_t)n * sizeof(int), h->stream));
    const unsigned char *db = h->d_deps.as<unsigned char>();
    DepsDev dp;
    dp.pred_ptr = reinterpret_cast<const int *>(db + off[0]);
    dp.pred_idx = reinterpret_cast<const int *>(db + off[1]);
    dp.fb_npts = has_fb ? reinterpret_cast<const int *>(db + off[2]) : nullptr;
    dp.fb_x = has_fb ? reinterpret_cast<const double *>(db + off[3]) : nullptr;
    dp.fb_y = has_fb ? reinterpret_cast<const double *>(db + off[4]) : nullptr;
    dp.done = h->d_done.as<int>();
    dp.dep_x = dp.dep_y = nullptr;
    dp.dep_n = nullptr;
    FallbackDev fbd{};
    if (closed_loop) {
        // fallback plans of all rows from the previous time step's plans on the device (known before the searches start)
        UP(h, h->cf_slot, slot, n);
        UP(h, h->cf_still, standstill, n);
        CU_TRY(h, h->cf_npts.reserve(nhp * sizeof(int)));
        CU_TRY(h, h->cf_x.reserve(nhp * PDMPC_AREA_STRIDE * sizeof(double)));
        CU_TRY(h, h->cf_y.reserve(nhp * PDMPC_AREA_STRIDE * sizeof(double)));
        CU_TRY(h, h->cf_traj.reserve(nhp * 3 * sizeof(double)));
        CU_TRY(h, h->cf_trims.reserve(nhp * sizeof(int)));
        fbd.slot = h->cf_slot.as<int>(); fbd.still = h->cf_still.as<unsigned char>();
        fbd.fb_npts = h->cf_npts.as<int>(); fbd.fb_x = h->cf_x.as<double>(); fbd.fb_y = h->cf_y.as<double>();
        fbd.fb_traj = h->cf_traj.as<double>(); fbd.fb_trims = h->cf_trims.as<int>();
        make_fallback_kernel<<<(unsigned)((nhp + 127) / 128), 128, 0, h->stream>>>(h->batch, h->cl, fbd);
        CU_TRY(h, cudaGetLastError());
        h->stats.kernel_launches++;
        dp.fb_npts = fbd.fb_npts; dp.fb_x = fbd.fb_x; dp.fb_y = fbd.fb_y;
    }
    // ---- one persistent launch: CTAs / warps take the searches in topological order ----------------
    CU_TRY(h, cudaMemsetAsync(h->out.counters, 0, kCounterBytes, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->work_counter.p, 0, sizeof(unsigned), h->stream));
    const bool cta_single = n <= h->num_sms;
    const int cta_nm = cta_single ? 1 : kCtaMastersDeps;
    const int grid = use_cta ? std::min((n + cta_nm - 1) / cta_nm, h->num_sms) : std::min(n, h->num_sms * h->lat_ctas_per_sm);
    rc = ensure_arena(h, use_cta ? grid * cta_nm : grid);
    if (rc != PDMPC_OK) return rc;
    if (!use_cta) {   // per-slot scratch for the predecessors' areas
        CU_TRY(h, h->d_depx.reserve((size_t)grid * kDepCols * sizeof(double)));
        CU_TRY(h, h->d_depy.reserve((size_t)grid * kDepCols * sizeof(double)));
        CU_TRY(h, h->d_depn.reserve((size_t)grid * (kDepCols / kAreaStride) * sizeof(int)));
        dp.dep_x = h->d_depx.as<double>(); dp.dep_y = h->d_depy.as<double>(); dp.dep_n = h->d_depn.as<int>();
    }
    const bool cta_fast = h->variant_mode == kShapeCtaValid || h->cta_valid_only;
    h->batch.hash_valid_only = h->cta_valid_only ? 1 : 0;   // one kind of pop_hash whatever shape runs
    h->stats.shape = use_cta ? (cta_fast ? kShapeCtaValid : kShapeCta) : kShapeLatency;
    CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
    if (use_cta && cta_single)
        KERNEL_CTA_DEPS<<<grid, CtaShape<1, kCtaCheckers>::kThreads, sizeof(CtaDepsSmemT), h->stream>>>(
            h->mpa, h->batch, h->out, h->arena, h->work_counter.as<unsigned>(), h->cta_heap_smem, cta_fast ? 1 : 0, dp);
    else if (use_cta)
        KERNEL_CTAM_DEPS<<<grid, CtaShape<kCtaMastersDeps, kCtaCheckers>::kThreads, sizeof(CtaMDepsSmemT), h->stream>>>(
            h->mpa, h->batch, h->out, h->arena, h->work_counter.as<unsigned>(), h->cta_heap_smem, cta_fast ? 1 : 0, dp);
    else
        KERNEL_LAT_DEPS<<<grid, kWarp, sizeof(WarpSmem), h->stream>>>(h->mpa, h->batch, h->out, h->arena,
                                                                      h->work_counter.as<unsigned>(),
                                                                      TraceDev{-1, nullptr, 0, nullptr}, dp);
    CU_TRY(h, cudaGetLastError());
    h->stats.kernel_launches++;
    if (closed_loop) {
        finalize_closed_loop_kernel<<<(unsigned)((nhp + 127) / 128), 128, 0, h->stream>>>(n, h->out, h->cl, fbd);
        CU_TRY(h, cudaGetLastError());
        h->stats.kernel_launches++;
    }
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    h->timing_pending_kernel = true;
    h->stats.handed_over = 0;
    return pdmpc_fetch_staged(h, out);
}

int pdmpc_plan_timestep(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                        pdmpc_batch_out *out) {
    return plan_timestep_impl(h, in, deps, out, nullptr, nullptr);
}

int pdmpc_closed_loop_reset(pdmpc_handle *h, int32_t n_slots, double half_length, double half_width) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "closed_loop_reset: call pdmpc_upload_mpa first (Hp)");
    if (n_slots < 1 || !(half_length > 0) || !(half_width > 0))
        return fail(h, PDMPC_ERR_BAD_INPUT, "closed_loop_reset: n_slots >= 1, half_length > 0, half_width > 0");
    CU_TRY(h, cudaSetDevice(h->device));
    const size_t sh = (size_t)n_slots * h->mpa.Hp;
    CU_TRY(h, h->cl_valid.reserve((size_t)n_slots * sizeof(int)));
    CU_TRY(h, h->cl_trims.reserve(sh * sizeof(int)));
    CU_TRY(h, h->cl_traj.reserve(sh * 3 * sizeof(double)));
    CU_TRY(h, h->cl_npts.reserve(sh * sizeof(int)));
    CU_TRY(h, h->cl_sx.reserve(sh * PDMPC_AREA_STRIDE * sizeof(double)));
    CU_TRY(h, h->cl_sy.reserve(sh * PDMPC_AREA_STRIDE * sizeof(double)));
    CU_TRY(h, cudaMemsetAsync(h->cl_valid.p, 0, (size_t)n_slots * sizeof(int), h->stream));
    ClosedLoopDev &c = h->cl;
    c.n_slots = n_slots; c.Hp = h->mpa.Hp; c.half_len = half_length; c.half_wid = half_width;
    c.valid = h->cl_valid.as<int>(); c.trims = h->cl_trims.as<int>(); c.traj = h->cl_traj.as<double>();
    c.npts = h->cl_npts.as<int>(); c.sx = h->cl_sx.as<double>(); c.sy = h->cl_sy.as<double>();
    return PDMPC_OK;
}

int pdmpc_plan_timestep_closed_loop(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                                    const int32_t *slot, const uint8_t *standstill, pdmpc_batch_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (h->cl.n_slots < 1 || h->cl.Hp != h->mpa.Hp)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_closed_loop: call pdmpc_closed_loop_reset first (after pdmpc_upload_mpa)");
    if (!in || !slot || !standstill || !out || !out->is_exhausted || !out->trims || !out->y_predicted || !out->shape_npts ||
        !out->shape_x || !out->shape_y)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_closed_loop: slot, standstill and the plan outputs are required");
    {
        std::vector<char> seen((size_t)h->cl.n_slots, 0);
        for (int i = 0; i < in->n_searches; ++i) {
            if (slot[i] < 0 || slot[i] >= h->cl.n_slots || seen[slot[i]])
                return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_closed_loop: slots must be distinct and below n_slots");
            seen[slot[i]] = 1;
        }
    }
    return plan_timestep_impl(h, in, deps, out, slot, standstill);
}

static int run_sample_inputs(pdmpc_handle *h, int n, const int32_t *path_id, const double *x, const double *y,
                             const double *speed, double dt_seconds, int lane_capacity);
static int run_assemble_obstacles(pdmpc_handle *h, const pdmpc_coupling_in *in, int poly_capacity, int vert_capacity, int totals[2]);

// One whole time step from the vehicles' measured states: inputs (pdmpc_inputs.cuh), obstacles that do not depend on this
// step's plans (pdmpc_obstacles.cuh), dependency-ordered searches, fallback plans (pdmpc_fallback.cuh) — nothing of the
// batch passes through the host.
int pdmpc_plan_timestep_from_states(pdmpc_handle *h, const pdmpc_timestep_states *st, pdmpc_batch_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "plan_timestep_from_states: call pdmpc_upload_mpa first");
    if (!h->has_road) return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: call pdmpc_upload_road first");
    if (h->cl.n_slots < 1 || h->cl.Hp != h->mpa.Hp)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: call pdmpc_closed_loop_reset first (after pdmpc_upload_mpa)");
    if (!st || !out || st->n < 0 || !out->status || !out->is_exhausted || !out->trims || !out->y_predicted || !out->shape_npts ||
        !out->shape_x || !out->shape_y)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: states and the plan outputs are required");
    const int n = st->n, Hp = h->mpa.Hp;
    if (n == 0) return PDMPC_OK;
    if (!st->path_id || !st->x || !st->y || !st->yaw || !st->speed || !st->trim || !st->succ_ptr || !st->par_ptr || !st->pred_ptr ||
        !st->slot)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: NULL argument");
    if (st->checker != PDMPC_CHECKER_INTERX && st->checker != PDMPC_CHECKER_SAT)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: unknown checker");
    std::vector<uint8_t> still((size_t)n);
    {
        std::vector<char> seen((size_t)h->cl.n_slots, 0);
        for (int i = 0; i < n; ++i) {
            if (st->path_id[i] < 0 || st->path_id[i] >= h->road.n_paths)
                return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: path_id out of range");
            if (st->slot[i] < 0 || st->slot[i] >= h->cl.n_slots || seen[st->slot[i]])
                return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: slots must be distinct and below n_slots");
            seen[st->slot[i]] = 1;
            still[i] = fabs(st->speed[i]) < kStandstillSpeed ? 1 : 0;   // PrioritizedController.m:580 / :527
        }
    }
    // ---- inputs and obstacles on the device; capacities from the relations -----------------------------------------
    const int lane_cap = 512 * n;
    int rc = run_sample_inputs(h, n, st->path_id, st->x, st->y, st->speed, st->dt_seconds, lane_cap);
    if (rc != PDMPC_OK) return rc;
    pdmpc_coupling_in ci;
    memset(&ci, 0, sizeof(ci));
    ci.n = n; ci.x = st->x; ci.y = st->y; ci.yaw = st->yaw; ci.speed = st->speed; ci.trim = st->trim;
    ci.succ_ptr = st->succ_ptr; ci.succ_idx = st->succ_idx; ci.par_ptr = st->par_ptr; ci.par_idx = st->par_idx;
    ci.half_length = st->half_length; ci.half_width = st->half_width;
    if (st->succ_ptr[0] != 0 || st->par_ptr[0] != 0 || st->succ_ptr[n] < 0 || st->par_ptr[n] < 0)
        return fail(h, PDMPC_ERR_BAD_INPUT, "plan_timestep_from_states: malformed relation");
    const long long poly_cap = (long long)st->succ_ptr[n] + (long long)Hp * st->par_ptr[n];
    const long long vert_cap = 5LL * st->succ_ptr[n] + (long long)Hp * st->par_ptr[n] * std::max(h->reach_max_pts, 1);
    if (poly_cap > 0x3fffffff || vert_cap > 0x3fffffff) return fail(h, PDMPC_ERR_CAPACITY, "plan_timestep_from_states: too many obstacles");
    int totals[3] = {0, 0, 0};   // polygons, vertices, lanelet points
    rc = run_assemble_obstacles(h, &ci, (int)poly_cap, (int)vert_cap, totals);
    if (rc != PDMPC_OK) return rc;
    CU_TRY(h, cudaMemcpyAsync(&totals[2], h->i_lptr.as<int>() + 2 * n, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (totals[2] > lane_cap) return fail(h, PDMPC_ERR_CAPACITY, "plan_timestep_from_states: the lanelet bounds need more than 512 points per vehicle");
    if (totals[0] > poly_cap || totals[1] > vert_cap) return fail(h, PDMPC_ERR_CAPACITY, "plan_timestep_from_states: obstacle capacity");
    const void *dev[kNumIn] = {h->q_x.p,    h->q_y.p,  h->q_yaw.p, h->q_trim.p, h->i_refx.p, h->i_refy.p, h->i_vref.p, h->q_slot.p,
                               h->q_poly.p, h->q_vx.p, h->q_vy.p,  h->i_lptr.p, h->i_lx.p,   h->i_ly.p,   nullptr};   // + the work order
    pdmpc_batch_in stub;
    memset(&stub, 0, sizeof(stub));
    stub.n_searches = n; stub.checker = st->checker; stub.dt_seconds = st->dt_seconds;
    pdmpc_timestep_deps deps;
    memset(&deps, 0, sizeof(deps));
    deps.pred_ptr = st->pred_ptr; deps.pred_idx = st->pred_idx;
    return plan_timestep_impl(h, &stub, &deps, out, st->slot, still.data(), dev, totals);
}

// Centralized (joint) search: rows = searches x n_vehicles (pdmpc_joint.cuh).
int pdmpc_joint_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, int32_t n_vehicles, pdmpc_batch_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "joint: call pdmpc_upload_mpa first");
    if (!in) return fail(h, PDMPC_ERR_BAD_INPUT, "joint: batch is NULL");
    if (n_vehicles < 1 || n_vehicles > PDMPC_MAX_JOINT)
        return fail(h, PDMPC_ERR_BAD_INPUT, "joint: n_vehicles must be 1..PDMPC_MAX_JOINT");
    if (in->n_searches < 0 || in->n_searches % n_vehicles)
        return fail(h, PDMPC_ERR_BAD_INPUT, "joint: the number of rows must be a multiple of n_vehicles");
    if (in->checker != PDMPC_CHECKER_SAT)   // are_constraints_satisfied_interx.m:12 asserts iter.amount == 1
        return fail(h, PDMPC_ERR_BAD_INPUT, "joint: the InterX checker is defined for single-vehicle searches only");
    const int Hp = h->mpa.Hp, n = in->n_searches, nj = n / n_vehicles;
    int rc = pdmpc_stage_batch(h, in);
    if (rc != PDMPC_OK) return rc;
    for (int r = 0; r < n; ++r)   // obstacles belong to the search: they sit in the slots of its first row
        if (r % n_vehicles && in->slot_ptr[(size_t)(r + 1) * (Hp + 1)] != in->slot_ptr[(size_t)r * (Hp + 1)]) {
            h->staged = false;
            return fail(h, PDMPC_ERR_BAD_INPUT, "joint: obstacle slots of rows other than a search's first row must be empty");
        }
    CU_TRY(h, cudaMemsetAsync(h->out.counters, 0, kCounterBytes, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->work_counter.p, 0, sizeof(unsigned), h->stream));
    h->stats.kernel_launches = 0;
    h->batch.hash_valid_only = h->cta_valid_only ? 1 : 0;
    if (nj > 0) {
        // one warp per search, the reference's loop statement by statement (pdmpc_joint.cuh; a CTA-per-search kernel
        // with factorized expansion was measured no faster: profiles/r02_joint_factorized_experiment.txt)
        const int grid = std::min(nj, h->num_sms * 2);   // two searches per SM (shared-memory heap tops)
        // default capacity: what 2 GiB of arena give every resident search, at least 2^17 nodes
        const double per_node = (double)n_vehicles * sizeof(JVeh) + sizeof(JNode) + sizeof(HEnt);
        int cap = h->user_node_cap ? h->user_node_cap
                                   : (int)std::min<double>(kJointMaxCap, std::max<double>(1 << 17, 2.0 * (1 << 30) / (grid * per_node)));
        cap = std::min(cap, kJointMaxCap);
        const size_t tot = (size_t)grid * cap;
        CU_TRY(h, h->j_veh.reserve(tot * n_vehicles * sizeof(JVeh)));
        CU_TRY(h, h->j_node.reserve(tot * sizeof(JNode)));
        CU_TRY(h, h->j_heap.reserve(tot * sizeof(HEnt)));
        JointArena ar;
        ar.veh = h->j_veh.as<JVeh>(); ar.node = h->j_node.as<JNode>(); ar.heap = h->j_heap.as<HEnt>();
        ar.cap = cap; ar.nV = n_vehicles;
        CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
        CU_TRY(h, cudaFuncSetAttribute(joint_search_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(JointSmem)));
        joint_search_kernel<<<grid, kWarp, sizeof(JointSmem), h->stream>>>(h->mpa, h->batch, h->out, ar,
                                                                           h->work_counter.as<unsigned>());
        CU_TRY(h, cudaGetLastError());
        CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
        h->timing_pending_kernel = true;
        h->stats.kernel_launches = 1;
        h->stats.shape = kShapeLatency;
    }
    return pdmpc_fetch_staged(h, out);
}

// MonteCarloTreeSearch over the staged batch: one warp per search (pdmpc_mcts.cuh).
int pdmpc_mcts_run_staged(pdmpc_handle *h, const pdmpc_mcts_params *prm) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->staged) return fail(h, PDMPC_ERR_BAD_INPUT, "mcts: no staged batch");
    if (!prm || prm->n_expansions_max < 1 || prm->n_expansions_max > PDMPC_MCTS_MAX_EXPANSIONS)
        return fail(h, PDMPC_ERR_BAD_INPUT, "mcts: n_expansions_max out of range");
    const int n = h->batch.n;
    if (n && !prm->seed) return fail(h, PDMPC_ERR_BAD_INPUT, "mcts: seed is NULL");
    if (h->max_branch > PDMPC_MCTS_MAX_BRANCH)
        return fail(h, PDMPC_ERR_BAD_INPUT, "mcts: branching factor of the MPA exceeds PDMPC_MCTS_MAX_BRANCH");
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaMemsetAsync(h->out.counters, 0, kCounterBytes, h->stream));
    CU_TRY(h, cudaMemsetAsync(h->work_counter.p, 0, sizeof(unsigned), h->stream));
    h->stats.kernel_launches = 0;
    if (n == 0) return PDMPC_OK;
    {
        int rc = upload(h, h->b_seed, prm->seed, (size_t)n);
        if (rc != PDMPC_OK) return rc;
        CU_TRY(h, cudaStreamSynchronize(h->stream));   // the seeds are caller-owned
    }
    MctsDev mc;
    mc.n_max = prm->n_expansions_max;
    mc.node_cap = prm->n_expansions_max + h->mpa.Hp + 1;
    mc.seed = h->b_seed.as<unsigned>();
    const size_t smem = mcts_smem_bytes(mc.node_cap);
    if (smem > kSmemLimit) return fail(h, PDMPC_ERR_CAPACITY, "mcts: sampled tree does not fit in shared memory");
    CU_TRY(h, cudaFuncSetAttribute(mcts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CU_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, mcts_kernel, kWarp, smem));
    if (occ < 1) return fail(h, PDMPC_ERR_CUDA, "mcts: kernel is not launchable on this device");
    const int grid = std::min(n, h->num_sms * occ);
    CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
    mcts_kernel<<<grid, kWarp, smem, h->stream>>>(h->mpa, h->batch, h->out, mc, h->work_counter.as<unsigned>());
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    h->timing_pending_kernel = true;
    h->stats.kernel_launches++;
    return PDMPC_OK;
}

int pdmpc_mcts_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_mcts_params *prm,
                          pdmpc_batch_out *out) {
    int rc = pdmpc_stage_batch(h, in);
    if (rc != PDMPC_OK) return rc;
    rc = pdmpc_mcts_run_staged(h, prm);
    if (rc != PDMPC_OK) return rc;
    return pdmpc_fetch_staged(h, out);
}

int pdmpc_trace_staged(pdmpc_handle *h, int32_t search, int64_t *ids, int64_t cap, int64_t *n_out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->staged) return fail(h, PDMPC_ERR_BAD_INPUT, "trace: no staged batch");
    if (search < 0 || search >= h->batch.n || !ids || cap < 1 || !n_out)
        return fail(h, PDMPC_ERR_BAD_INPUT, "trace: bad arguments");
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, h->t_ids.reserve((size_t)cap * sizeof(long long)));
    CU_TRY(h, h->t_n.reserve(sizeof(long long)));
    CU_TRY(h, cudaMemsetAsync(h->t_n.p, 0, sizeof(long long), h->stream));
    TraceDev tr{search, h->t_ids.as<long long>(), (long long)cap, h->t_n.as<long long>()};
    int rc = launch_search(h, tr);
    if (rc != PDMPC_OK) return rc;
    long long n = 0;
    CU_TRY(h, cudaMemcpyAsync(&n, h->t_n.p, sizeof(n), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    const long long m = std::min<long long>(n, cap);
    if (m > 0) CU_TRY(h, cudaMemcpy(ids, h->t_ids.p, (size_t)m * sizeof(long long), cudaMemcpyDeviceToHost));
    *n_out = n;
    return PDMPC_OK;
}

int pdmpc_measure_fp64_peak(pdmpc_handle *h, double *mul_add_tops, double *fma_tflops) {
    if (!h || !mul_add_tops || !fma_tflops) return PDMPC_ERR_BAD_INPUT;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, h->t_n.reserve(sizeof(double)));
    const int iters = 4096, grid = h->num_sms * 8, block = 256;
    float ms[2] = {0.f, 0.f};
    for (int pass = 0; pass < 2; ++pass)       // pass 0 warms up
        for (int k = 0; k < 2; ++k) {
            CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
            if (k == 0) fp64_peak_kernel<false><<<grid, block, 0, h->stream>>>(h->t_n.as<double>(), iters, 1.0000001, 1e-7);
            else fp64_peak_kernel<true><<<grid, block, 0, h->stream>>>(h->t_n.as<double>(), iters, 1.0000001, 1e-7);
            CU_TRY(h, cudaGetLastError());
            CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
            CU_TRY(h, cudaStreamSynchronize(h->stream));
            CU_TRY(h, cudaEventElapsedTime(&ms[k], h->ev[2], h->ev[3]));
        }
    const double ops = (double)grid * block * iters * 8.0 * 2.0;   // a multiply and an add per chain step
    *mul_add_tops = ops / (ms[0] * 1e-3) / 1e12;
    *fma_tflops = ops / (ms[1] * 1e-3) / 1e12;
    h->timing_pending_kernel = false;
    return PDMPC_OK;
}

int pdmpc_pack_plan_rows(pdmpc_handle *h, int32_t n_rows, int32_t n_vehicles, const double *fallback_rows,
                         void *device_dst) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->staged || n_rows < 0 || n_rows > h->batch.n || n_vehicles < 1 || !device_dst)
        return fail(h, PDMPC_ERR_BAD_INPUT, "pack_plan_rows: needs the results of a plan call, 0 <= n_rows <= its searches, "
                                            "n_vehicles >= 1 and a device destination");
    if (n_rows == 0) return PDMPC_OK;
    CU_TRY(h, cudaSetDevice(h->device));
    const int Hp = h->mpa.Hp, L = 2 + 21 * Hp;
    const double *fb = nullptr;
    if (fallback_rows) {
        const size_t bytes = (size_t)n_vehicles * L * sizeof(double);
        CU_TRY(h, h->esc_rows.reserve(bytes));   // (scratch: no escalation rows are pending between calls)
        CU_TRY(h, cudaMemcpyAsync(h->esc_rows.p, fallback_rows, bytes, cudaMemcpyHostToDevice, h->stream));
        fb = h->esc_rows.as<double>();
    }
    const long long tot = (long long)n_rows * L;
    pack_plan_rows_kernel<<<(unsigned)std::min<long long>((tot + 255) / 256, 1184), 256, 0, h->stream>>>(
        h->out, Hp, n_rows, n_vehicles, fb, static_cast<double *>(device_dst));
    CU_TRY(h, cudaGetLastError());
    h->stats.kernel_launches++;
    CU_TRY(h, cudaStreamSynchronize(h->stream));   // the caller hands device_dst to its collective next
    return PDMPC_OK;
}

int pdmpc_upload_road(pdmpc_handle *h, const pdmpc_road_desc *r) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!r || r->n_lanelets < 1 || r->n_paths < 1 || !r->bound_ptr || !r->bound_x || !r->bound_y || !r->path_ptr ||
        !r->path_x || !r->path_y || !r->lan_ptr || !r->lanelets_index || !r->points_index || !r->is_loop || !r->reference_speed)
        return fail(h, PDMPC_ERR_BAD_INPUT, "upload_road: NULL table or empty road");
    h->has_road = false;
    const int nb = 2 * r->n_lanelets, np = r->n_paths;
    for (int i = 0; i < nb; ++i)
        if (r->bound_ptr[i + 1] - r->bound_ptr[i] < 2 || r->bound_ptr[0] != 0)
            return fail(h, PDMPC_ERR_BAD_INPUT, "upload_road: every lanelet bound needs at least two points");
    for (int p = 0; p < np; ++p) {
        if (r->path_ptr[p + 1] - r->path_ptr[p] < 2 || r->lan_ptr[p + 1] - r->lan_ptr[p] < 1)
            return fail(h, PDMPC_ERR_BAD_INPUT, "upload_road: a reference path needs two points and one lanelet");
        for (int j = r->lan_ptr[p]; j < r->lan_ptr[p + 1]; ++j)
            if (r->lanelets_index[j] < 1 || r->lanelets_index[j] > r->n_lanelets)
                return fail(h, PDMPC_ERR_BAD_INPUT, "upload_road: lanelet id out of range");
    }
    CU_TRY(h, cudaSetDevice(h->device));
    UP(h, h->r_bptr, r->bound_ptr, nb + 1);
    UP(h, h->r_bx, r->bound_x, r->bound_ptr[nb]);
    UP(h, h->r_by, r->bound_y, r->bound_ptr[nb]);
    UP(h, h->r_pptr, r->path_ptr, np + 1);
    UP(h, h->r_px, r->path_x, r->path_ptr[np]);
    UP(h, h->r_py, r->path_y, r->path_ptr[np]);
    UP(h, h->r_lptr, r->lan_ptr, np + 1);
    UP(h, h->r_lidx, r->lanelets_index, r->lan_ptr[np]);
    UP(h, h->r_pidx, r->points_index, r->lan_ptr[np]);
    UP(h, h->r_loop, r->is_loop, np);
    UP(h, h->r_speed, r->reference_speed, np);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    RoadDev &d = h->road;
    d.n_lanelets = r->n_lanelets; d.n_paths = np;
    d.bound_ptr = h->r_bptr.as<int>(); d.bound_x = h->r_bx.as<double>(); d.bound_y = h->r_by.as<double>();
    d.path_ptr = h->r_pptr.as<int>(); d.path_x = h->r_px.as<double>(); d.path_y = h->r_py.as<double>();
    d.lan_ptr = h->r_lptr.as<int>(); d.lanelets_index = h->r_lidx.as<int>(); d.points_index = h->r_pidx.as<int>();
    d.is_loop = h->r_loop.as<unsigned char>(); d.reference_speed = h->r_speed.as<double>();
    h->has_road = true;
    return PDMPC_OK;
}

// The device side of pdmpc_sample_inputs: uploads the rows, runs the three kernels; results stay in the handle's i_* buffers.
static int run_sample_inputs(pdmpc_handle *h, int n, const int32_t *path_id, const double *x, const double *y,
                             const double *speed, double dt_seconds, int lane_capacity) {
    CU_TRY(h, cudaSetDevice(h->device));
    const int Hp = h->mpa.Hp;
    const size_t nh = (size_t)n * Hp;
    h->stats.h2d_bytes = 0;
    h->stats.d2h_bytes = 0;
    h->stats.kernel_launches = 0;
    UP(h, h->i_pid, path_id, n);
    UP(h, h->i_x, x, n);
    UP(h, h->i_y, y, n);
    UP(h, h->i_speed, speed, n);
    CU_TRY(h, h->i_refx.reserve(nh * sizeof(double)));
    CU_TRY(h, h->i_refy.reserve(nh * sizeof(double)));
    CU_TRY(h, h->i_vref.reserve(nh * sizeof(double)));
    CU_TRY(h, h->i_ridx.reserve(nh * sizeof(int)));
    CU_TRY(h, h->i_cur.reserve((size_t)n * sizeof(int)));
    CU_TRY(h, h->i_pred.reserve((size_t)n * PDMPC_MAX_PRED_LANELETS * sizeof(int)));
    CU_TRY(h, h->i_pre.reserve((size_t)n * sizeof(int)));
    CU_TRY(h, h->i_cnt.reserve((size_t)2 * n * sizeof(int)));
    CU_TRY(h, h->i_lptr.reserve(((size_t)2 * n + 1) * sizeof(int)));
    CU_TRY(h, h->i_lx.reserve(std::max<size_t>(lane_capacity, 1) * sizeof(double)));
    CU_TRY(h, h->i_ly.reserve(std::max<size_t>(lane_capacity, 1) * sizeof(double)));
    InputsDev in;
    in.n = n; in.Hp = Hp; in.dt = dt_seconds;
    in.path_id = h->i_pid.as<int>(); in.x = h->i_x.as<double>(); in.y = h->i_y.as<double>(); in.speed = h->i_speed.as<double>();
    in.ref_x = h->i_refx.as<double>(); in.ref_y = h->i_refy.as<double>(); in.v_ref = h->i_vref.as<double>();
    in.ref_index = h->i_ridx.as<int>(); in.current_index = h->i_cur.as<int>(); in.pred_lanelets = h->i_pred.as<int>();
    in.pre_lanelet = h->i_pre.as<int>(); in.lane_cnt = h->i_cnt.as<int>(); in.lane_ptr = h->i_lptr.as<int>();
    in.lane_x = h->i_lx.as<double>(); in.lane_y = h->i_ly.as<double>();
    const int blocks = (n + 3) / 4;   // 4 warps per block
    CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
    sample_inputs_kernel<<<blocks, 128, 0, h->stream>>>(h->road, in);
    scan_counts_kernel<<<1, 1024, 0, h->stream>>>(in.lane_cnt, in.lane_ptr, 2 * n);
    copy_bounds_kernel<<<blocks, 128, 0, h->stream>>>(h->road, in, lane_capacity);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    h->timing_pending_kernel = true;
    h->stats.kernel_launches = 3;
    return PDMPC_OK;
}

int pdmpc_sample_inputs(pdmpc_handle *h, int32_t n, const int32_t *path_id, const double *x, const double *y,
                        const double *speed, double dt_seconds, pdmpc_inputs_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "sample_inputs: call pdmpc_upload_mpa first (Hp)");
    if (!h->has_road) return fail(h, PDMPC_ERR_BAD_INPUT, "sample_inputs: call pdmpc_upload_road first");
    if (n < 0 || !out || (n && (!path_id || !x || !y || !speed)) || out->lane_capacity < 0)
        return fail(h, PDMPC_ERR_BAD_INPUT, "sample_inputs: NULL argument");
    for (int i = 0; i < n; ++i)
        if (path_id[i] < 0 || path_id[i] >= h->road.n_paths)
            return fail(h, PDMPC_ERR_BAD_INPUT, "sample_inputs: path_id out of range");
    if (n == 0) {
        if (out->lane_ptr) out->lane_ptr[0] = 0;
        return PDMPC_OK;
    }
    int rc_run = run_sample_inputs(h, n, path_id, x, y, speed, dt_seconds, out->lane_capacity);
    if (rc_run != PDMPC_OK) return rc_run;
    const int Hp = h->mpa.Hp;
    const size_t nh = (size_t)n * Hp;
    const int *d_lane_ptr = h->i_lptr.as<int>();
    int total = 0;
    CU_TRY(h, cudaMemcpyAsync(&total, d_lane_ptr + 2 * n, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    DOWN(h, out->ref_x, h->i_refx, nh);
    DOWN(h, out->ref_y, h->i_refy, nh);
    DOWN(h, out->v_ref, h->i_vref, nh);
    DOWN(h, out->ref_index, h->i_ridx, nh);
    DOWN(h, out->current_index, h->i_cur, n);
    DOWN(h, out->predicted_lanelets, h->i_pred, (size_t)n * PDMPC_MAX_PRED_LANELETS);
    DOWN(h, out->lane_ptr, h->i_lptr, 2 * (size_t)n + 1);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    if (total > out->lane_capacity)
        return fail(h, PDMPC_ERR_CAPACITY, "sample_inputs: the lanelet bounds need " + std::to_string(total) +
                                               " points, lane_capacity is " + std::to_string(out->lane_capacity));
    DOWN(h, out->lane_x, h->i_lx, total);
    DOWN(h, out->lane_y, h->i_ly, total);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return PDMPC_OK;
}

// ---- obstacle assembly of a time step (pdmpc_obstacles.cuh) -----------------------------------------------
int pdmpc_upload_reachable_sets(pdmpc_handle *h, const pdmpc_reach_desc *r) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!r || r->n_trims < 1 || r->Hp < 1 || !r->ptr || !r->x || !r->y)
        return fail(h, PDMPC_ERR_BAD_INPUT, "upload_reachable_sets: NULL table or empty automaton");
    h->has_reach = false;
    const int m = r->n_trims * r->Hp;
    if (r->ptr[0] != 0) return fail(h, PDMPC_ERR_BAD_INPUT, "upload_reachable_sets: ptr[0] must be 0");
    for (int i = 0; i < m; ++i) {
        const int a = r->ptr[i], b = r->ptr[i + 1];
        if (b - a < 2) return fail(h, PDMPC_ERR_BAD_INPUT, "upload_reachable_sets: a reachable set needs at least two points");
        // vectorize_all_obstacles.m:71-76 check_closeness: InterX needs closed polygons
        if (!(r->x[a] == r->x[b - 1] && r->y[a] == r->y[b - 1]))
            return fail(h, PDMPC_ERR_BAD_INPUT, "upload_reachable_sets: reachable set is not closed (first point != last)");
    }
    CU_TRY(h, cudaSetDevice(h->device));
    UP(h, h->q_rptr, r->ptr, m + 1);
    UP(h, h->q_rx, r->x, r->ptr[m]);
    UP(h, h->q_ry, r->y, r->ptr[m]);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    h->reach.nT = r->n_trims; h->reach.Hp = r->Hp;
    h->reach_max_pts = 0;
    for (int i = 0; i < m; ++i) h->reach_max_pts = std::max(h->reach_max_pts, r->ptr[i + 1] - r->ptr[i]);
    h->reach.ptr = h->q_rptr.as<int>(); h->reach.x = h->q_rx.as<double>(); h->reach.y = h->q_ry.as<double>();
    h->has_reach = true;
    return PDMPC_OK;
}

// Validation + the device side of pdmpc_assemble_obstacles; results stay in the handle's q_* buffers, the totals
// (polygons, vertices) come back in totals[2].
static int run_assemble_obstacles(pdmpc_handle *h, const pdmpc_coupling_in *in, int poly_capacity, int vert_capacity, int totals[2]) {
    const int n = in->n, Hp = h->mpa.Hp;
    if (in->succ_ptr[0] != 0 || in->par_ptr[0] != 0) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: CSR must start at 0");
    for (int i = 0; i < n; ++i)
        if (in->succ_ptr[i + 1] < in->succ_ptr[i] || in->par_ptr[i + 1] < in->par_ptr[i])
            return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: CSR not monotone");
    const int ns = in->succ_ptr[n], npar = in->par_ptr[n];
    if ((ns && !in->succ_idx) || (npar && !in->par_idx)) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: NULL index array");
    for (int q = 0; q < ns; ++q)
        if (in->succ_idx[q] < 0 || in->succ_idx[q] >= n) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: successor index out of range");
    for (int q = 0; q < npar; ++q)
        if (in->par_idx[q] < 0 || in->par_idx[q] >= n) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: predecessor index out of range");
    if (npar) {
        if (!h->has_reach) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: call pdmpc_upload_reachable_sets first");
        if (h->reach.Hp != Hp || h->reach.nT != h->mpa.nT)
            return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: the reachable sets belong to another automaton (n_trims, Hp)");
    }
    for (int i = 0; i < n; ++i)
        if (in->trim[i] < 1 || in->trim[i] > h->mpa.nT) return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: trim out of range");
    CU_TRY(h, cudaSetDevice(h->device));
    const int S = n * (Hp + 1);
    UP(h, h->q_x, in->x, n);
    UP(h, h->q_y, in->y, n);
    UP(h, h->q_yaw, in->yaw, n);
    UP(h, h->q_speed, in->speed, n);
    UP(h, h->q_trim, in->trim, n);
    UP(h, h->q_sptr, in->succ_ptr, n + 1);
    UP(h, h->q_sidx, in->succ_idx, ns);
    UP(h, h->q_pptr, in->par_ptr, n + 1);
    UP(h, h->q_pidx, in->par_idx, npar);
    CU_TRY(h, h->q_cs.reserve((size_t)n * sizeof(double2)));
    CU_TRY(h, h->q_cntp.reserve((size_t)S * sizeof(int)));
    CU_TRY(h, h->q_cntv.reserve((size_t)S * sizeof(int)));
    CU_TRY(h, h->q_slot.reserve(((size_t)S + 1) * sizeof(int)));
    CU_TRY(h, h->q_vbase.reserve(((size_t)S + 1) * sizeof(int)));
    CU_TRY(h, h->q_poly.reserve(((size_t)poly_capacity + 1) * sizeof(int)));
    CU_TRY(h, h->q_vx.reserve(std::max<size_t>(vert_capacity, 1) * sizeof(double)));
    CU_TRY(h, h->q_vy.reserve(std::max<size_t>(vert_capacity, 1) * sizeof(double)));
    CouplingDev c;
    c.n = n; c.Hp = Hp;
    c.x = h->q_x.as<double>(); c.y = h->q_y.as<double>(); c.yaw = h->q_yaw.as<double>(); c.speed = h->q_speed.as<double>();
    c.trim = h->q_trim.as<int>();
    c.succ_ptr = h->q_sptr.as<int>(); c.succ_idx = h->q_sidx.as<int>();
    c.par_ptr = h->q_pptr.as<int>(); c.par_idx = h->q_pidx.as<int>();
    c.half_len = in->half_length; c.half_wid = in->half_width;
    c.cs = h->q_cs.as<double2>();
    c.cnt_poly = h->q_cntp.as<int>(); c.cnt_vert = h->q_cntv.as<int>();
    c.slot_ptr = h->q_slot.as<int>(); c.vert_base = h->q_vbase.as<int>();
    c.poly_ptr = h->q_poly.as<int>(); c.vert_x = h->q_vx.as<double>(); c.vert_y = h->q_vy.as<double>();
    count_obstacles_kernel<<<(S + 127) / 128, 128, 0, h->stream>>>(h->reach, c);
    scan_counts_kernel<<<1, 1024, 0, h->stream>>>(c.cnt_poly, c.slot_ptr, S);
    scan_counts_kernel<<<1, 1024, 0, h->stream>>>(c.cnt_vert, c.vert_base, S);
    fill_obstacles_kernel<<<(S + 3) / 4, 128, 0, h->stream>>>(h->reach, c, poly_capacity, vert_capacity);
    CU_TRY(h, cudaGetLastError());
    CU_TRY(h, cudaMemcpyAsync(&totals[0], c.slot_ptr + S, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU_TRY(h, cudaMemcpyAsync(&totals[1], c.vert_base + S, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    return PDMPC_OK;
}

int pdmpc_assemble_obstacles(pdmpc_handle *h, const pdmpc_coupling_in *in, pdmpc_obstacles_out *out) {
    if (!h) return PDMPC_ERR_BAD_INPUT;
    if (!h->has_mpa) return fail(h, PDMPC_ERR_NO_MPA, "assemble_obstacles: call pdmpc_upload_mpa first (Hp)");
    if (!in || !out || in->n < 0 || out->poly_capacity < 0 || out->vert_capacity < 0 || !out->slot_ptr ||
        (in->n && (!in->x || !in->y || !in->yaw || !in->speed || !in->trim || !in->succ_ptr || !in->par_ptr)))
        return fail(h, PDMPC_ERR_BAD_INPUT, "assemble_obstacles: NULL argument");
    const int n = in->n, Hp = h->mpa.Hp;
    if (n == 0) {
        out->slot_ptr[0] = 0;
        if (out->poly_ptr) out->poly_ptr[0] = 0;
        return PDMPC_OK;
    }
    const int S = n * (Hp + 1);
    h->stats.h2d_bytes = 0;
    h->stats.d2h_bytes = 0;
    CU_TRY(h, cudaEventRecord(h->ev[2], h->stream));
    int totals[2] = {0, 0};
    int rc = run_assemble_obstacles(h, in, out->poly_capacity, out->vert_capacity, totals);
    if (rc != PDMPC_OK) return rc;
    CU_TRY(h, cudaEventRecord(h->ev[3], h->stream));
    h->timing_pending_kernel = true;
    h->stats.kernel_launches = 4;
    DOWN(h, out->slot_ptr, h->q_slot, (size_t)S + 1);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    out->n_polys = totals[0];
    out->n_verts = totals[1];
    if (totals[0] > out->poly_capacity || totals[1] > out->vert_capacity)
        return fail(h, PDMPC_ERR_CAPACITY, "assemble_obstacles: " + std::to_string(totals[0]) + " polygons / " + std::to_string(totals[1]) +
                                               " vertices do not fit poly_capacity " + std::to_string(out->poly_capacity) +
                                               " / vert_capacity " + std::to_string(out->vert_capacity));
    DOWN(h, out->poly_ptr, h->q_poly, (size_t)totals[0] + 1);
    DOWN(h, out->vert_x, h->q_vx, totals[1]);
    DOWN(h, out->vert_y, h->q_vy, totals[1]);
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    return PDMPC_OK;
}

int pdmpc_get_stats(pdmpc_handle *h, pdmpc_stats *out) {
    if (!h || !out) return PDMPC_ERR_BAD_INPUT;
    CU_TRY(h, cudaSetDevice(h->device));
    CU_TRY(h, cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    if (h->timing_pending_h2d && cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]) == cudaSuccess) h->stats.h2d_ms = ms;
    if (h->timing_pending_kernel && cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]) == cudaSuccess) h->stats.kernel_ms = ms;
    if (h->timing_pending_d2h && cudaEventElapsedTime(&ms, h->ev[4], h->ev[5]) == cudaSuccess) h->stats.d2h_ms = ms;
    *out = h->stats;
    return PDMPC_OK;
}

}  // extern "C"
