// pdmpc_fallback.cuh — the output side of a time step on the device (SURVEY.md §8(f) rank 4): what a vehicle does, and
// publishes, when its search is exhausted, and the closed-loop state that needs.
//
//   handle_graph_search_exhaustion   hlc/controller/prioritized/PrioritizedController.m:568-621  (standstill: the vehicle
//                                    keeps its pose for Hp steps, its area = the offset rectangle at that pose,
//                                    get_occupied_areas.m:21-25 / transformed_rectangle)
//   plan_fallback                    PrioritizedController.m:678-718  (the previous plan shifted by one step, last step
//                                    repeated: del_first_rpt_last on trims, y_predicted, shapes)
//
// The fallback plan of a vehicle depends only on the PREVIOUS time step, so it is known before the searches of this one
// start: make_fallback_kernel builds it for every vehicle from the plans kept on the device (ClosedLoopDev, one slot per
// vehicle of every scenario); the dependency-ordered search kernels read the AREAS of exhausted predecessors from it
// (DepsDev.fb_*), finalize_closed_loop_kernel then replaces the outputs of exhausted searches by the fallback plan and
// stores every vehicle's final plan as the next step's "previous plan".  No plan leaves the device between time steps.
#pragma once

#include "pdmpc_kernels.cuh"

namespace pdmpc {

struct ClosedLoopDev {             // per slot: the plan executed / published in the previous time step
    int n_slots, Hp;
    double half_len, half_wid;     // Length / 2 + offset, Width / 2 + offset of the standstill rectangle
    int *valid;                    // [slots] 0: no previous plan
    int *trims;                    // [slots * Hp]
    double *traj;                  // [slots * Hp * 3]
    int *npts;                     // [slots * Hp]
    double *sx, *sy;               // [slots * Hp * kAreaStride]
};

struct FallbackDev {               // per row of the call
    const int *slot;               // [n]
    const unsigned char *still;    // [n] the vehicle stands (|speed of its trim| < 0.01)
    int *fb_npts;                  // [n * Hp]
    double *fb_x, *fb_y;           // [n * Hp * kAreaStride]
    double *fb_traj;               // [n * Hp * 3]
    int *fb_trims;                 // [n * Hp]
    const unsigned char *commit = nullptr;   // [n] finalize stores row r in its slot iff commit[r] (null: every row)
};

// one thread per (row, step)
__global__ void make_fallback_kernel(BatchDev b, ClosedLoopDev st, FallbackDev fb) {
    const int Hp = st.Hp;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= b.n * Hp) return;
    const int row = idx / Hp, k = idx % Hp;
    const int s = fb.slot[row];
    const size_t o = (size_t)row * Hp + k;
    if (!st.valid[s] || fb.still[row]) {
        // :568-621 standstill — the closed 5-point rectangle of get_occupied_areas.m:21-25 at the current pose
        const double x = b.x0[row], y = b.y0[row], yaw = b.yaw0[row];
        double sn, cs;
        sincos_ref(yaw, sn, cs);
        const double sxl[5] = {-1.0, -1.0, 1.0, 1.0, -1.0}, syl[5] = {-1.0, 1.0, 1.0, -1.0, -1.0};
        for (int i = 0; i < kAreaStride; ++i) {
            double px = 0.0, py = 0.0;
            if (i < 5) {
                const double xl = sxl[i] * st.half_len, yl = syl[i] * st.half_wid;
                px = cs * xl - sn * yl + x;
                py = sn * xl + cs * yl + y;
            }
            fb.fb_x[o * kAreaStride + i] = px;
            fb.fb_y[o * kAreaStride + i] = py;
        }
        fb.fb_npts[o] = 5;
        fb.fb_traj[o * 3 + 0] = x; fb.fb_traj[o * 3 + 1] = y; fb.fb_traj[o * 3 + 2] = yaw;
        fb.fb_trims[o] = b.trim0[row];
    } else {
        // :678-718 previous plan, first step dropped, last step repeated
        const size_t p = (size_t)s * Hp + min(k + 1, Hp - 1);
        for (int i = 0; i < kAreaStride; ++i) {
            fb.fb_x[o * kAreaStride + i] = st.sx[p * kAreaStride + i];
            fb.fb_y[o * kAreaStride + i] = st.sy[p * kAreaStride + i];
        }
        fb.fb_npts[o] = st.npts[p];
        for (int c = 0; c < 3; ++c) fb.fb_traj[o * 3 + c] = st.traj[p * 3 + c];
        fb.fb_trims[o] = st.trims[p];
    }
}

// one thread per (row, step): exhausted searches take their fallback plan; every final plan (every committed one, when
// fb.commit is set) becomes the slot's state
__global__ void finalize_closed_loop_kernel(int n, OutDev o, ClosedLoopDev st, FallbackDev fb) {
    const int Hp = st.Hp;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * Hp) return;
    const int row = idx / Hp, k = idx % Hp;
    const size_t os = (size_t)row * Hp + k;
    if (o.is_exhausted[row]) {
        o.trims[(size_t)row * (Hp + 1) + k + 1] = fb.fb_trims[os];
        for (int c = 0; c < 3; ++c) o.y_predicted[os * 3 + c] = fb.fb_traj[os * 3 + c];
        o.shape_npts[os] = fb.fb_npts[os];
        for (int i = 0; i < kAreaStride; ++i) {
            o.shape_x[os * kAreaStride + i] = fb.fb_x[os * kAreaStride + i];
            o.shape_y[os * kAreaStride + i] = fb.fb_y[os * kAreaStride + i];
        }
    }
    if (fb.commit && !fb.commit[row]) return;
    const size_t p = (size_t)fb.slot[row] * Hp + k;
    st.trims[p] = o.trims[(size_t)row * (Hp + 1) + k + 1];
    for (int c = 0; c < 3; ++c) st.traj[p * 3 + c] = o.y_predicted[os * 3 + c];
    st.npts[p] = o.shape_npts[os];
    for (int i = 0; i < kAreaStride; ++i) {
        st.sx[p * kAreaStride + i] = o.shape_x[os * kAreaStride + i];
        st.sy[p * kAreaStride + i] = o.shape_y[os * kAreaStride + i];
    }
    if (k == 0) st.valid[fb.slot[row]] = 1;
}

}  // namespace pdmpc
