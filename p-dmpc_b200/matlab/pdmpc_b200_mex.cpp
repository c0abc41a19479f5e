// pdmpc_b200_mex.cpp — thin MEX shim: MATLAB arrays <-> the C ABI of include/pdmpc_b200.h.
//
// Plays the role priority_queue_interface_mex.cpp plays in the reference
// (hlc/optimizer/graph_search/priority_queue/priority_queue_interface_mex.cpp:33-108):
// a command dispatcher, first argument = command, handles owned by the MEX.  It only
// marshals; every computation happens behind pdmpc_* on the GPU.  Called by
// GraphSearchCuda.m; built by compile_pdmpc_b200.m (mex -R2018a, C Matrix API).
//
//   h = mex(CREATE, device_id)
//       mex(DESTROY, h)
//       mex(UPLOAD_MPA, h, transition_matrix_single [nT x nT x Hp], maneuvers {nT x nT})
//   [is_exhausted, n_expanded, trims, y_pred, g_path, h_path, shapes] =
//       mex(PLAN, h, x0 [1x3], trim, ref [Hp x 2], v_ref [1 x Hp], obstacles {n_s},
//           dynamic_obstacle_area {n_d x Hp}, left [2 x nL], right [2 x nR], checker, dt)
//   [same outputs] = mex(PLAN_SAMPLED, h, <the ten PLAN arguments>, seed, n_expansions_max)
//       MonteCarloTreeSearch.run_optimizer: seed = time_step + vehicle_index (MonteCarloTreeSearch.m:31)
//   s = mex(STATS, h)
//   [is_exhausted (1 x N), n_expanded (1 x N), trims (N x Hp+1), y_pred (3 x Hp*N), shapes {N x Hp}] =
//       mex(PLAN_TIMESTEP, h, x0 [N x 3], trims [N x 1], ref [N x Hp x 2], v_ref [N x Hp],
//           obstacles {N x S}, dynamic_obstacle_area {N x R*Hp} (row r of step k at column r + R*(k-1)),
//           left {N x 1}, right {N x 1}, checker, dt, directed_coupling_sequential [N x N],
//           fallback_shapes {N x Hp})
//       ALL vehicles of one time step in one call (plan_timestep_cuda.m): replaces the level loop of
//       PrioritizedSequentialController.controller (PrioritizedSequentialController.m:74-92); vehicle i
//       waits on the device for the vehicles j with directed_coupling_sequential(j, i) ~= 0 and takes
//       their planned areas as dynamic obstacles (PrioritizedController.m:449-506); empty cells are skipped.
//   [same outputs] = mex(PLAN_TIMESTEP_SAMPLED, h, <the thirteen PLAN_TIMESTEP arguments>, seeds [N], n_expansions_max)
//       the same time step with MonteCarloTreeSearch as the optimizer (plan_timestep_cuda.m with a
//       MonteCarloTreeSearchCuda optimizer): seeds(i) = time_step + vehicle_index of vehicle i (MonteCarloTreeSearch.m:31).
//       A search whose roll-outs run out of random numbers is reported exhausted, like one without a valid leaf.
//   [is_exhausted, n_expanded, trims (nV x Hp+1), y_pred (3 x Hp*nV), shapes {nV x Hp}, g_path (1 x Hp+1), h_path] =
//       mex(PLAN_JOINT, h, x0 [nV x 3], trims [nV x 1], ref [nV x Hp x 2], v_ref [nV x Hp], obstacles {nV x S},
//           dynamic_obstacle_area {nV x R*Hp}, left {nV x 1}, right {nV x 1}, checker (0 = SAT), dt)
//       ONE centralized search over nV vehicles (CentralizedController.m:33-59, GraphSearchCuda.run_optimizer with
//       iter.amount > 1): iter.obstacles / iter.dynamic_obstacle_area go into ROW 1 of the two cell arrays.
//       mex(UPLOAD_ROAD, h, lanelet_boundaries {nL x 2} (left, right; each n x 2), reference_paths {nP x 1} (n x 2),
//           lanelets_index {nP x 1}, points_index {nP x 1}, is_loop [nP], reference_speed [nP])
//   [ref (N x Hp x 2), v_ref (N x Hp), points_index (N x Hp), current_point_index (N x 1), predicted_lanelets {N x 1},
//    left {N x 1} (2 x n), right {N x 1} (2 x n)] = mex(SAMPLE_INPUTS, h, path_id [N] (1-based), x [N], y [N], speed [N], dt)
//       reference trajectories and lanelet boundaries of ALL vehicles of a time step in one call
//       (sample_inputs_cuda.m): get_reference_trajectory / sample_reference_trajectory / get_predicted_lanelets /
//       get_lanelets_boundary of hlc/controller/common, as HighLevelController fills them into iter.
//       mex(UPLOAD_REACHABLE_SETS, h, local_reachable_sets {nT x Hp} (2 x m closed polygons: the Vertices of
//           mpa.local_reachable_sets_conv{trim, t} with the first vertex repeated))
//   [obstacles {N x 1} of {s_i x 1} (2 x 5), dynamic_obstacle_area {N x 1} of {p_i x Hp} (2 x m)] =
//       mex(ASSEMBLE_OBSTACLES, h, x0 [N x 4] (x, y, yaw, speed), trims [N], successors {N x 1} (1-based indices),
//           parallel_predecessors {N x 1}, half_length, half_width)
//       the obstacles of ALL vehicles of a time step that do not depend on this time step's plans
//       (assemble_obstacles_cuda.m): standing successors' occupied areas (PrioritizedController.m:508-540,
//       get_occupied_areas.m:19-25) and parallel predecessors' reachable sets (:391-407,
//       MotionPrimitiveAutomaton.m:649-687).
//   [adjacency (N x N), overlap_area (N x N)] = mex(COUPLE, h, x0 [N x 3] (x, y, yaw), trims [N])
//       ReachableSetCoupler.couple for ONE scenario (couple_cuda.m, needs UPLOAD_REACHABLE_SETS): adjacency(i, j) = 1 iff
//       the step-Hp reachable sets of vehicles i and j overlap by more than 1e-3 (ReachableSetCoupler.m:39-42), N <= 64.
//       The prioritizer classes stay MATLAB's.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "mex.h"
#include "pdmpc_b200.h"

namespace {

enum Command { CREATE = 0, DESTROY = 1, UPLOAD_MPA = 2, PLAN = 3, STATS = 4, PLAN_SAMPLED = 5, PLAN_TIMESTEP = 6, PLAN_JOINT = 7, UPLOAD_ROAD = 8,
               SAMPLE_INPUTS = 9, UPLOAD_REACHABLE_SETS = 10, ASSEMBLE_OBSTACLES = 11, COUPLE = 12, PLAN_TIMESTEP_SAMPLED = 13 };

std::vector<pdmpc_handle *> g_handles;   // released at `clear mex` (HighLevelController.m:284-303)
bool g_at_exit_registered = false;

void release_all() {
    for (pdmpc_handle *h : g_handles)
        if (h) pdmpc_destroy(h);
    g_handles.clear();
}

[[noreturn]] void fail(const char *id, const std::string &msg) {
    mexErrMsgIdAndTxt(id, "%s", msg.c_str());
    throw 0;   // not reached: mexErrMsgIdAndTxt does not return
}

pdmpc_handle *handle_of(const mxArray *a) {
    const uint64_t idx = static_cast<uint64_t>(mxGetScalar(a));
    if (idx == 0 || idx > g_handles.size() || !g_handles[idx - 1]) fail("pdmpc:handle", "invalid planner handle");
    return g_handles[idx - 1];
}

void check(pdmpc_handle *h, int rc, const char *what) {
    if (rc == PDMPC_OK) return;
    const char *txt = pdmpc_last_error(h);
    fail("pdmpc:status", std::string(what) + " failed (" + std::to_string(rc) + "): " + (txt ? txt : ""));
}

// Append a 2 x n polygon (column-major: x0 y0 x1 y1 ...) to the vertex pool.
void append_polygon(const mxArray *p, std::vector<double> &vx, std::vector<double> &vy, std::vector<int32_t> &poly_ptr) {
    if (!p || mxIsEmpty(p)) return;   // empty cells contribute nothing (SearchBatch.from_iters does the same)
    if (mxGetM(p) != 2) fail("pdmpc:input", "obstacle polygons must be 2 x n");
    const double *d = mxGetDoubles(p);
    const size_t n = mxGetN(p);
    for (size_t i = 0; i < n; ++i) {
        vx.push_back(d[2 * i]);
        vy.push_back(d[2 * i + 1]);
    }
    poly_ptr.push_back(static_cast<int32_t>(vx.size()));
}

void upload_mpa(pdmpc_handle *h, const mxArray *trans, const mxArray *maneuvers) {
    // mpa.transition_matrix_single: nT x nT x Hp, column-major (t1, t2, k)
    const mwSize nd = mxGetNumberOfDimensions(trans);
    const mwSize *dims = mxGetDimensions(trans);
    const int nT = static_cast<int>(dims[0]);
    const int Hp = nd >= 3 ? static_cast<int>(dims[2]) : 1;
    if (static_cast<int>(dims[1]) != nT) fail("pdmpc:input", "transition_matrix_single must be nT x nT x Hp");
    const double *t = mxGetDoubles(trans);
    std::vector<uint8_t> transition(static_cast<size_t>(Hp) * nT * nT);
    for (int k = 0; k < Hp; ++k)
        for (int t1 = 0; t1 < nT; ++t1)
            for (int t2 = 0; t2 < nT; ++t2)
                transition[(static_cast<size_t>(k) * nT + t1) * nT + t2] =
                    t[t1 + static_cast<size_t>(nT) * t2 + static_cast<size_t>(nT) * nT * k] != 0.0;
    // mpa.maneuvers{t1, t2}: struct with dx, dy, dyaw, area, area_without_offset, area_large_offset
    std::vector<int32_t> from, to, npts;
    std::vector<double> dx, dy, dyaw, ax, ay;
    static const char *kAreas[3] = {"area", "area_without_offset", "area_large_offset"};
    for (int t1 = 0; t1 < nT; ++t1)
        for (int t2 = 0; t2 < nT; ++t2) {
            const mxArray *m = mxGetCell(maneuvers, t1 + static_cast<size_t>(nT) * t2);
            if (!m || mxIsEmpty(m)) continue;
            from.push_back(t1 + 1);
            to.push_back(t2 + 1);
            // maneuvers are structs (generate_maneuver.m) or objects with the same property names
            auto get = [&](const char *name) -> const mxArray * {
                const mxArray *f = mxIsStruct(m) ? mxGetField(m, 0, name) : mxGetProperty(m, 0, name);
                if (!f) fail("pdmpc:input", std::string("maneuver without field ") + name);
                return f;
            };
            dx.push_back(mxGetScalar(get("dx")));
            dy.push_back(mxGetScalar(get("dy")));
            dyaw.push_back(mxGetScalar(get("dyaw")));
            for (const char *name : kAreas) {
                const mxArray *a = get(name);
                const size_t n = mxGetN(a);
                if (mxGetM(a) != 2 || n > PDMPC_AREA_STRIDE) fail("pdmpc:input", "maneuver area must be 2 x n, n <= 8");
                const double *d = mxGetDoubles(a);
                npts.push_back(static_cast<int32_t>(n));
                for (size_t i = 0; i < PDMPC_AREA_STRIDE; ++i) {
                    ax.push_back(i < n ? d[2 * i] : 0.0);
                    ay.push_back(i < n ? d[2 * i + 1] : 0.0);
                }
            }
        }
    pdmpc_mpa_desc d;
    d.n_trims = nT;
    d.Hp = Hp;
    d.n_edges = static_cast<int32_t>(from.size());
    d.transition = transition.data();
    d.edge_from = from.data();
    d.edge_to = to.data();
    d.edge_dx = dx.data();
    d.edge_dy = dy.data();
    d.edge_dyaw = dyaw.data();
    d.area_npts = npts.data();
    d.area_x = ax.data();
    d.area_y = ay.data();
    check(h, pdmpc_upload_mpa(h, &d), "pdmpc_upload_mpa");
}

// PLAN (sampled == false): GraphSearch; PLAN_SAMPLED: MonteCarloTreeSearch with two more
// arguments, the RandStream seed (time_step + vehicle_index) and n_expansions_max.
void plan(pdmpc_handle *h, int nlhs, mxArray *plhs[], const mxArray *prhs[], bool sampled) {
    const mxArray *x0 = prhs[2], *ref = prhs[4], *vref = prhs[5], *obst = prhs[6], *dyn = prhs[7];
    const mxArray *left = prhs[8], *right = prhs[9];
    const int Hp = static_cast<int>(mxGetNumberOfElements(vref));
    if (Hp != pdmpc_get_hp(h)) fail("pdmpc:input", "v_ref holds " + std::to_string(Hp) + " steps, the uploaded MPA has Hp = " + std::to_string(pdmpc_get_hp(h)));
    if (mxGetNumberOfElements(x0) < 3 || mxGetNumberOfElements(ref) != static_cast<size_t>(2 * Hp))
        fail("pdmpc:input", "x0 must hold (x, y, yaw) and ref must be Hp x 2");
    const double *px0 = mxGetDoubles(x0);
    const double *pref = mxGetDoubles(ref);   // Hp x 2 column-major: x(1..Hp), y(1..Hp)
    const double *pv = mxGetDoubles(vref);
    int32_t trim0 = static_cast<int32_t>(mxGetScalar(prhs[3]));

    // obstacle CSR, slot 0 = iter.obstacles, slot k = iter.dynamic_obstacle_area(:, k)
    std::vector<int32_t> slot_ptr(1, 0), poly_ptr(1, 0);
    std::vector<double> vx, vy;
    const size_t n_static = mxIsCell(obst) ? mxGetNumberOfElements(obst) : 0;
    for (size_t i = 0; i < n_static; ++i) append_polygon(mxGetCell(obst, i), vx, vy, poly_ptr);
    slot_ptr.push_back(static_cast<int32_t>(poly_ptr.size() - 1));
    const size_t n_rows = mxIsCell(dyn) ? mxGetM(dyn) : 0;
    const size_t n_cols = mxIsCell(dyn) ? mxGetN(dyn) : 0;
    for (int k = 0; k < Hp; ++k) {
        if (static_cast<size_t>(k) < n_cols)   // vectorize_all_obstacles.m:39-43
            for (size_t r = 0; r < n_rows; ++r) append_polygon(mxGetCell(dyn, r + n_rows * k), vx, vy, poly_ptr);
        slot_ptr.push_back(static_cast<int32_t>(poly_ptr.size() - 1));
    }
    // lanelet bounds: open polylines
    std::vector<int32_t> lane_ptr(1, 0);
    std::vector<double> lx, ly;
    for (const mxArray *side : {left, right}) {
        if (side && !mxIsEmpty(side)) {
            if (mxGetM(side) != 2) fail("pdmpc:input", "lanelet bounds must be 2 x n");
            const double *d = mxGetDoubles(side);
            for (size_t i = 0; i < mxGetN(side); ++i) {
                lx.push_back(d[2 * i]);
                ly.push_back(d[2 * i + 1]);
            }
        }
        lane_ptr.push_back(static_cast<int32_t>(lx.size()));
    }

    pdmpc_batch_in in;
    std::memset(&in, 0, sizeof(in));
    in.n_searches = 1;
    in.checker = static_cast<int32_t>(mxGetScalar(prhs[10]));
    in.dt_seconds = mxGetScalar(prhs[11]);
    in.x0 = &px0[0];
    in.y0 = &px0[1];
    in.yaw0 = &px0[2];
    in.trim0 = &trim0;
    in.ref_x = pref;
    in.ref_y = pref + Hp;
    in.v_ref = pv;
    in.slot_ptr = slot_ptr.data();
    in.poly_ptr = poly_ptr.data();
    in.vert_x = vx.data();
    in.vert_y = vy.data();
    in.lane_ptr = lane_ptr.data();
    in.lane_x = lx.data();
    in.lane_y = ly.data();

    int32_t status = -1, n_expanded = 0;
    uint8_t exhausted = 0;
    std::vector<int32_t> trims(Hp + 1), shape_npts(Hp);
    std::vector<double> ypred(3 * Hp), g(Hp + 1), hh(Hp + 1), sx(Hp * PDMPC_AREA_STRIDE), sy(Hp * PDMPC_AREA_STRIDE);
    pdmpc_batch_out out;
    std::memset(&out, 0, sizeof(out));
    out.status = &status;
    out.is_exhausted = &exhausted;
    out.n_expanded = &n_expanded;
    out.trims = trims.data();
    out.y_predicted = ypred.data();
    out.g_path = g.data();
    out.h_path = hh.data();
    out.shape_npts = shape_npts.data();
    out.shape_x = sx.data();
    out.shape_y = sy.data();
    if (sampled) {
        const uint32_t seed = static_cast<uint32_t>(mxGetScalar(prhs[12]));
        pdmpc_mcts_params prm;
        prm.n_expansions_max = static_cast<int32_t>(mxGetScalar(prhs[13]));
        prm.seed = &seed;
        check(h, pdmpc_mcts_plan_batch(h, &in, &prm, &out), "pdmpc_mcts_plan_batch");
    } else {
        check(h, pdmpc_plan_batch(h, &in, &out), "pdmpc_plan_batch");
    }
    if (status != PDMPC_OK)   // e.g. PDMPC_ERR_CAPACITY: loud, never a silently truncated search
        fail("pdmpc:search", "search failed with status " + std::to_string(status));

    plhs[0] = mxCreateLogicalScalar(exhausted != 0);
    if (nlhs > 1) plhs[1] = mxCreateDoubleScalar(n_expanded);
    if (nlhs > 2) {
        plhs[2] = mxCreateDoubleMatrix(1, Hp + 1, mxREAL);
        for (int k = 0; k <= Hp; ++k) mxGetDoubles(plhs[2])[k] = trims[k];
    }
    if (nlhs > 3) {   // 3 x Hp: (x, y, yaw) per step, the layout of info.y_predicted(:, :, 1)
        plhs[3] = mxCreateDoubleMatrix(3, Hp, mxREAL);
        std::memcpy(mxGetDoubles(plhs[3]), ypred.data(), sizeof(double) * 3 * Hp);
    }
    if (nlhs > 4) {
        plhs[4] = mxCreateDoubleMatrix(1, Hp + 1, mxREAL);
        std::memcpy(mxGetDoubles(plhs[4]), g.data(), sizeof(double) * (Hp + 1));
    }
    if (nlhs > 5) {
        plhs[5] = mxCreateDoubleMatrix(1, Hp + 1, mxREAL);
        std::memcpy(mxGetDoubles(plhs[5]), hh.data(), sizeof(double) * (Hp + 1));
    }
    if (nlhs > 6) {   // info.shapes: 1 x Hp cell of 2 x n
        plhs[6] = mxCreateCellMatrix(1, Hp);
        for (int k = 0; k < Hp; ++k) {
            const int n = shape_npts[k];
            mxArray *s = mxCreateDoubleMatrix(2, n, mxREAL);
            double *d = mxGetDoubles(s);
            for (int i = 0; i < n; ++i) {
                d[2 * i] = sx[k * PDMPC_AREA_STRIDE + i];
                d[2 * i + 1] = sy[k * PDMPC_AREA_STRIDE + i];
            }
            mxSetCell(plhs[6], k, s);
        }
    }
}

// PLAN_TIMESTEP: N vehicles, one pdmpc_plan_timestep call.  PLAN_JOINT (joint == true): the same N rows as ONE
// centralized search (pdmpc_joint_plan_batch), no coupling / fallback arguments.  PLAN_TIMESTEP_SAMPLED (sampled == true):
// pdmpc_mcts_plan_timestep with seeds and n_expansions_max after the PLAN_TIMESTEP arguments.
void plan_timestep(pdmpc_handle *h, int nlhs, mxArray *plhs[], const mxArray *prhs[], bool joint, bool sampled = false) {
    const mxArray *x0 = prhs[2], *trim = prhs[3], *ref = prhs[4], *vref = prhs[5], *obst = prhs[6], *dyn = prhs[7];
    const mxArray *left = prhs[8], *right = prhs[9], *coupling = joint ? nullptr : prhs[12];
    const mxArray *fallback = joint ? nullptr : prhs[13];
    const size_t N = mxGetM(x0);
    if (N == 0 || mxGetN(x0) < 3) fail("pdmpc:input", "x0 must be N x 3");
    if (mxGetM(vref) != N) fail("pdmpc:input", "v_ref must be N x Hp");
    const int Hp = static_cast<int>(mxGetN(vref));
    if (Hp != pdmpc_get_hp(h)) fail("pdmpc:input", "v_ref holds " + std::to_string(Hp) + " steps, the uploaded MPA has Hp = " + std::to_string(pdmpc_get_hp(h)));
    if (mxGetNumberOfElements(ref) != N * Hp * 2 || mxGetNumberOfElements(trim) != N)
        fail("pdmpc:input", "ref must be N x Hp x 2 and trims N x 1");
    if (!joint && (mxGetM(coupling) != N || mxGetN(coupling) != N))
        fail("pdmpc:input", "directed_coupling_sequential must be N x N");
    const double *px0 = mxGetDoubles(x0), *pref = mxGetDoubles(ref), *pv = mxGetDoubles(vref), *ptrim = mxGetDoubles(trim);
    const double *pc = joint ? nullptr : mxGetDoubles(coupling);

    std::vector<double> xs(N), ys(N), yaws(N), rx(N * Hp), ry(N * Hp), vr(N * Hp);
    std::vector<int32_t> trims(N), slot_ptr(1, 0), poly_ptr(1, 0), lane_ptr(1, 0);
    std::vector<double> vx, vy, lx, ly;
    const size_t S = mxIsCell(obst) && mxGetM(obst) == N ? mxGetN(obst) : 0;
    const size_t RH = mxIsCell(dyn) && mxGetM(dyn) == N ? mxGetN(dyn) : 0;
    if (RH % Hp != 0) fail("pdmpc:input", "dynamic_obstacle_area must be N x (R*Hp)");
    const size_t R = RH / Hp;
    for (size_t i = 0; i < N; ++i) {
        xs[i] = px0[i]; ys[i] = px0[i + N]; yaws[i] = px0[i + 2 * N];
        trims[i] = static_cast<int32_t>(ptrim[i]);
        for (int k = 0; k < Hp; ++k) {
            rx[i * Hp + k] = pref[i + N * k];
            ry[i * Hp + k] = pref[i + N * k + N * Hp];
            vr[i * Hp + k] = pv[i + N * k];
        }
        for (size_t s = 0; s < S; ++s) append_polygon(mxGetCell(obst, i + N * s), vx, vy, poly_ptr);
        slot_ptr.push_back(static_cast<int32_t>(poly_ptr.size() - 1));
        for (int k = 0; k < Hp; ++k) {
            for (size_t r = 0; r < R; ++r) append_polygon(mxGetCell(dyn, i + N * (r + R * k)), vx, vy, poly_ptr);
            slot_ptr.push_back(static_cast<int32_t>(poly_ptr.size() - 1));
        }
        for (const mxArray *sides : {left, right}) {
            const mxArray *side = (mxIsCell(sides) && mxGetNumberOfElements(sides) == N) ? mxGetCell(sides, i) : nullptr;
            if (side && !mxIsEmpty(side)) {
                if (mxGetM(side) != 2) fail("pdmpc:input", "lanelet bounds must be 2 x n");
                const double *d = mxGetDoubles(side);
                for (size_t q = 0; q < mxGetN(side); ++q) {
                    lx.push_back(d[2 * q]);
                    ly.push_back(d[2 * q + 1]);
                }
            }
            lane_ptr.push_back(static_cast<int32_t>(lx.size()));
        }
    }
    // predecessors of vehicle i: find(directed_coupling_sequential(:, i)) (PrioritizedController.m:309)
    std::vector<int32_t> pred_ptr(1, 0), pred_idx;
    for (size_t i = 0; i < N; ++i) {
        for (size_t j = 0; j < N && pc; ++j)
            if (pc[j + N * i] != 0.0) pred_idx.push_back(static_cast<int32_t>(j));
        pred_ptr.push_back(static_cast<int32_t>(pred_idx.size()));
    }
    if (pred_idx.empty()) pred_idx.push_back(0);
    // what an exhausted vehicle publishes (plan_fallback / handle_graph_search_exhaustion)
    std::vector<int32_t> fb_npts(N * Hp, 0);
    std::vector<double> fbx(N * Hp * PDMPC_AREA_STRIDE, 0.0), fby(N * Hp * PDMPC_AREA_STRIDE, 0.0);
    const bool has_fb = fallback && mxIsCell(fallback) && mxGetM(fallback) == N && mxGetN(fallback) == static_cast<size_t>(Hp);
    if (has_fb)
        for (size_t i = 0; i < N; ++i)
            for (int k = 0; k < Hp; ++k) {
                const mxArray *a = mxGetCell(fallback, i + N * k);
                if (!a || mxIsEmpty(a)) continue;
                const size_t m = mxGetN(a);
                if (mxGetM(a) != 2 || m >= PDMPC_AREA_STRIDE) fail("pdmpc:input", "fallback shapes must be 2 x m, m <= 7");
                const double *d = mxGetDoubles(a);
                fb_npts[i * Hp + k] = static_cast<int32_t>(m);
                for (size_t q = 0; q < m; ++q) {
                    fbx[(i * Hp + k) * PDMPC_AREA_STRIDE + q] = d[2 * q];
                    fby[(i * Hp + k) * PDMPC_AREA_STRIDE + q] = d[2 * q + 1];
                }
            }

    pdmpc_batch_in in;
    std::memset(&in, 0, sizeof(in));
    in.n_searches = static_cast<int32_t>(N);
    in.checker = static_cast<int32_t>(mxGetScalar(prhs[10]));
    in.dt_seconds = mxGetScalar(prhs[11]);
    in.x0 = xs.data(); in.y0 = ys.data(); in.yaw0 = yaws.data(); in.trim0 = trims.data();
    in.ref_x = rx.data(); in.ref_y = ry.data(); in.v_ref = vr.data();
    in.slot_ptr = slot_ptr.data(); in.poly_ptr = poly_ptr.data(); in.vert_x = vx.data(); in.vert_y = vy.data();
    in.lane_ptr = lane_ptr.data(); in.lane_x = lx.data(); in.lane_y = ly.data();
    pdmpc_timestep_deps deps;
    std::memset(&deps, 0, sizeof(deps));
    deps.pred_ptr = pred_ptr.data();
    deps.pred_idx = pred_idx.data();
    if (has_fb) { deps.fb_npts = fb_npts.data(); deps.fb_x = fbx.data(); deps.fb_y = fby.data(); }

    std::vector<int32_t> status(N, -1), n_expanded(N, 0), out_trims(N * (Hp + 1)), shape_npts(N * Hp);
    std::vector<uint8_t> exhausted(N, 0);
    std::vector<double> ypred(N * Hp * 3), sx(N * Hp * PDMPC_AREA_STRIDE), sy(N * Hp * PDMPC_AREA_STRIDE);
    std::vector<double> g(N * (Hp + 1)), hh(N * (Hp + 1));
    pdmpc_batch_out out;
    std::memset(&out, 0, sizeof(out));
    out.status = status.data(); out.is_exhausted = exhausted.data(); out.n_expanded = n_expanded.data();
    out.trims = out_trims.data(); out.y_predicted = ypred.data();
    out.g_path = g.data(); out.h_path = hh.data();
    out.shape_npts = shape_npts.data(); out.shape_x = sx.data(); out.shape_y = sy.data();
    if (joint) {
        check(h, pdmpc_joint_plan_batch(h, &in, static_cast<int32_t>(N), &out), "pdmpc_joint_plan_batch");
    } else if (sampled) {
        // mxGetDoubles is NULL for any class but double (e.g. uint32(time_step + (1:N)))
        const double *ps = mxGetDoubles(prhs[14]);
        if (!ps || mxGetNumberOfElements(prhs[14]) != N)
            fail("pdmpc:input", "seeds must be N doubles (time_step + vehicle_index)");
        if (mxGetNumberOfElements(prhs[15]) != 1) fail("pdmpc:input", "n_expansions_max must be a scalar");
        std::vector<uint32_t> seeds(N);
        for (size_t i = 0; i < N; ++i) {
            const double v = ps[i];
            if (!(v >= 0.0 && v <= 4294967295.0) || v != static_cast<double>(static_cast<uint32_t>(v)))
                fail("pdmpc:input", "seeds must be integers in 0 .. 2^32 - 1");
            seeds[i] = static_cast<uint32_t>(v);
        }
        pdmpc_mcts_params prm;
        prm.n_expansions_max = static_cast<int32_t>(mxGetScalar(prhs[15]));
        prm.seed = seeds.data();
        check(h, pdmpc_mcts_plan_timestep(h, &in, &deps, &prm, &out), "pdmpc_mcts_plan_timestep");
    } else {
        check(h, pdmpc_plan_timestep(h, &in, &deps, &out), "pdmpc_plan_timestep");
    }
    for (size_t i = 0; i < N && !sampled; ++i)   // a sampled search out of random numbers is an exhausted row
        if (status[i] != PDMPC_OK) fail("pdmpc:search", "search " + std::to_string(i + 1) + " failed with status " + std::to_string(status[i]));

    plhs[0] = mxCreateDoubleMatrix(1, N, mxREAL);
    for (size_t i = 0; i < N; ++i) mxGetDoubles(plhs[0])[i] = exhausted[i];
    if (nlhs > 1) {
        plhs[1] = mxCreateDoubleMatrix(1, N, mxREAL);
        for (size_t i = 0; i < N; ++i) mxGetDoubles(plhs[1])[i] = n_expanded[i];
    }
    if (nlhs > 2) {
        plhs[2] = mxCreateDoubleMatrix(N, Hp + 1, mxREAL);
        for (size_t i = 0; i < N; ++i)
            for (int k = 0; k <= Hp; ++k) mxGetDoubles(plhs[2])[i + N * k] = out_trims[i * (Hp + 1) + k];
    }
    if (nlhs > 3) {   // 3 x (Hp*N): reshape(y, 3, Hp, N) gives info.y_predicted of vehicle i in (:, :, i)
        plhs[3] = mxCreateDoubleMatrix(3, Hp * N, mxREAL);
        std::memcpy(mxGetDoubles(plhs[3]), ypred.data(), sizeof(double) * 3 * Hp * N);
    }
    if (nlhs > 4) {
        plhs[4] = mxCreateCellMatrix(N, Hp);
        for (size_t i = 0; i < N; ++i)
            for (int k = 0; k < Hp; ++k) {
                const int n = shape_npts[i * Hp + k];
                mxArray *sh = mxCreateDoubleMatrix(2, n, mxREAL);
                double *d = mxGetDoubles(sh);
                for (int q = 0; q < n; ++q) {
                    d[2 * q] = sx[(i * Hp + k) * PDMPC_AREA_STRIDE + q];
                    d[2 * q + 1] = sy[(i * Hp + k) * PDMPC_AREA_STRIDE + q];
                }
                mxSetCell(plhs[4], i + N * k, sh);
            }
    }
    for (int q = 0; q < 2 && nlhs > 5 + q; ++q) {
        // cost to come / cost to go along the path: tree.g, tree.h of next_nodes (NodeInfo columns 5, 6), which
        // PrioritizedExplorativeController.compute_solution_cost reads through tree.get_cost (:100-104).
        // PLAN_TIMESTEP: N x (Hp+1), row i = vehicle i.  PLAN_JOINT: 1 x (Hp+1), the joint cost (row 1 of the search).
        const size_t rows = joint ? 1 : N;
        const std::vector<double> &src = q == 0 ? g : hh;
        plhs[5 + q] = mxCreateDoubleMatrix(rows, Hp + 1, mxREAL);
        for (size_t i = 0; i < rows; ++i)
            for (int k = 0; k <= Hp; ++k) mxGetDoubles(plhs[5 + q])[i + rows * k] = src[i * (Hp + 1) + k];
    }
}

// UPLOAD_ROAD: the map's lanelet boundaries and every vehicle's reference path -> pdmpc_upload_road
void upload_road(pdmpc_handle *h, const mxArray *prhs[]) {
    const mxArray *bounds = prhs[2], *paths = prhs[3], *lidx = prhs[4], *pidx = prhs[5], *loop = prhs[6], *speed = prhs[7];
    if (!mxIsCell(bounds) || mxGetN(bounds) < 2) fail("pdmpc:input", "lanelet_boundaries must be an nL x 2 cell (left, right)");
    const size_t nL = mxGetM(bounds), nP = mxGetNumberOfElements(paths);
    if (!mxIsCell(paths) || !mxIsCell(lidx) || !mxIsCell(pidx) || mxGetNumberOfElements(lidx) != nP ||
        mxGetNumberOfElements(pidx) != nP || mxGetNumberOfElements(loop) != nP || mxGetNumberOfElements(speed) != nP)
        fail("pdmpc:input", "reference_paths, lanelets_index, points_index, is_loop, reference_speed must have one entry per path");
    std::vector<int32_t> bptr(1, 0), pptr(1, 0), lptr(1, 0), li, pi;
    std::vector<double> bx, by, px, py, spd(nP);
    std::vector<uint8_t> lp(nP);
    auto append_rows = [&](const mxArray *a, std::vector<double> &x, std::vector<double> &y) {   // n x 2, column-major
        if (!a || mxGetN(a) != 2) fail("pdmpc:input", "polylines must be n x 2");
        const size_t n = mxGetM(a);
        const double *d = mxGetDoubles(a);
        for (size_t i = 0; i < n; ++i) { x.push_back(d[i]); y.push_back(d[i + n]); }
        return static_cast<int32_t>(n);
    };
    for (size_t l = 0; l < nL; ++l)
        for (size_t side = 0; side < 2; ++side)
            bptr.push_back(bptr.back() + append_rows(mxGetCell(bounds, l + nL * side), bx, by));
    for (size_t p = 0; p < nP; ++p) {
        pptr.push_back(pptr.back() + append_rows(mxGetCell(paths, p), px, py));
        const mxArray *a = mxGetCell(lidx, p), *b = mxGetCell(pidx, p);
        if (!a || !b || mxGetNumberOfElements(a) != mxGetNumberOfElements(b)) fail("pdmpc:input", "lanelets_index / points_index mismatch");
        for (size_t j = 0; j < mxGetNumberOfElements(a); ++j) {
            li.push_back(static_cast<int32_t>(mxGetDoubles(a)[j]));
            pi.push_back(static_cast<int32_t>(mxGetDoubles(b)[j]));
        }
        lptr.push_back(static_cast<int32_t>(li.size()));
        lp[p] = mxGetDoubles(loop)[p] != 0;
        spd[p] = mxGetDoubles(speed)[p];
    }
    pdmpc_road_desc d;
    std::memset(&d, 0, sizeof(d));
    d.n_lanelets = static_cast<int32_t>(nL); d.bound_ptr = bptr.data(); d.bound_x = bx.data(); d.bound_y = by.data();
    d.n_paths = static_cast<int32_t>(nP); d.path_ptr = pptr.data(); d.path_x = px.data(); d.path_y = py.data();
    d.lan_ptr = lptr.data(); d.lanelets_index = li.data(); d.points_index = pi.data();
    d.is_loop = lp.data(); d.reference_speed = spd.data();
    check(h, pdmpc_upload_road(h, &d), "pdmpc_upload_road");
}

// SAMPLE_INPUTS: reference trajectories + lanelet boundaries of N vehicles -> pdmpc_sample_inputs
void sample_inputs(pdmpc_handle *h, int nlhs, mxArray *plhs[], const mxArray *prhs[]) {
    const size_t N = mxGetNumberOfElements(prhs[2]);
    if (mxGetNumberOfElements(prhs[3]) != N || mxGetNumberOfElements(prhs[4]) != N || mxGetNumberOfElements(prhs[5]) != N)
        fail("pdmpc:input", "path_id, x, y, speed must have N entries each");
    const int Hp = pdmpc_get_hp(h);
    std::vector<int32_t> pid(N), ridx(N * Hp), cur(N), pred(N * PDMPC_MAX_PRED_LANELETS), lane_ptr(2 * N + 1);
    for (size_t i = 0; i < N; ++i) pid[i] = static_cast<int32_t>(mxGetDoubles(prhs[2])[i]) - 1;
    std::vector<double> rx(N * Hp), ry(N * Hp), vr(N * Hp), lx(512 * N + 1), ly(512 * N + 1);
    pdmpc_inputs_out out;
    std::memset(&out, 0, sizeof(out));
    out.ref_x = rx.data(); out.ref_y = ry.data(); out.v_ref = vr.data(); out.ref_index = ridx.data();
    out.current_index = cur.data(); out.predicted_lanelets = pred.data(); out.lane_ptr = lane_ptr.data();
    out.lane_x = lx.data(); out.lane_y = ly.data(); out.lane_capacity = static_cast<int32_t>(512 * N);
    check(h, pdmpc_sample_inputs(h, static_cast<int32_t>(N), pid.data(), mxGetDoubles(prhs[3]), mxGetDoubles(prhs[4]),
                                 mxGetDoubles(prhs[5]), mxGetScalar(prhs[6]), &out), "pdmpc_sample_inputs");
    const size_t dims[3] = {N, static_cast<size_t>(Hp), 2};
    plhs[0] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);      // iter.reference_trajectory_points
    for (size_t i = 0; i < N; ++i)
        for (int k = 0; k < Hp; ++k) {
            mxGetDoubles(plhs[0])[i + N * k] = rx[i * Hp + k];
            mxGetDoubles(plhs[0])[i + N * k + N * Hp] = ry[i * Hp + k];
        }
    auto matrix = [&](int slot, const double *src_d, const int32_t *src_i, size_t cols) {
        if (nlhs <= slot) return;
        plhs[slot] = mxCreateDoubleMatrix(N, cols, mxREAL);
        for (size_t i = 0; i < N; ++i)
            for (size_t k = 0; k < cols; ++k)
                mxGetDoubles(plhs[slot])[i + N * k] = src_d ? src_d[i * cols + k] : static_cast<double>(src_i[i * cols + k]);
    };
    matrix(1, vr.data(), nullptr, Hp);
    matrix(2, nullptr, ridx.data(), Hp);
    matrix(3, nullptr, cur.data(), 1);
    if (nlhs > 4) {
        plhs[4] = mxCreateCellMatrix(N, 1);
        for (size_t i = 0; i < N; ++i) {
            size_t m = 0;
            while (m < PDMPC_MAX_PRED_LANELETS && pred[i * PDMPC_MAX_PRED_LANELETS + m]) ++m;
            mxArray *a = mxCreateDoubleMatrix(1, m, mxREAL);
            for (size_t j = 0; j < m; ++j) mxGetDoubles(a)[j] = pred[i * PDMPC_MAX_PRED_LANELETS + j];
            mxSetCell(plhs[4], i, a);
        }
    }
    for (int side = 0; side < 2 && nlhs > 5 + side; ++side) {               // predicted_lanelet_boundary{i, 1:2}
        plhs[5 + side] = mxCreateCellMatrix(N, 1);
        for (size_t i = 0; i < N; ++i) {
            const int a = lane_ptr[2 * i + side], b = lane_ptr[2 * i + side + 1];
            mxArray *m = mxCreateDoubleMatrix(2, b - a, mxREAL);
            for (int j = a; j < b; ++j) {
                mxGetDoubles(m)[2 * (j - a)] = lx[j];
                mxGetDoubles(m)[2 * (j - a) + 1] = ly[j];
            }
            mxSetCell(plhs[5 + side], i, m);
        }
    }
}

// UPLOAD_REACHABLE_SETS: mpa.local_reachable_sets_conv as closed 2 x m polygons -> pdmpc_upload_reachable_sets
void upload_reachable_sets(pdmpc_handle *h, const mxArray *prhs[]) {
    const mxArray *sets = prhs[2];
    if (!mxIsCell(sets)) fail("pdmpc:input", "local_reachable_sets must be an nT x Hp cell");
    const size_t nT = mxGetM(sets), Hp = mxGetN(sets);
    std::vector<int32_t> ptr(1, 0);
    std::vector<double> x, y;
    for (size_t i = 0; i < nT; ++i)
        for (size_t t = 0; t < Hp; ++t) {
            const mxArray *p = mxGetCell(sets, i + nT * t);
            if (!p || mxGetM(p) != 2) fail("pdmpc:input", "a reachable set must be a 2 x m polygon");
            const double *d = mxGetDoubles(p);
            for (size_t j = 0; j < mxGetN(p); ++j) {
                x.push_back(d[2 * j]);
                y.push_back(d[2 * j + 1]);
            }
            ptr.push_back(static_cast<int32_t>(x.size()));
        }
    pdmpc_reach_desc r;
    r.n_trims = static_cast<int32_t>(nT); r.Hp = static_cast<int32_t>(Hp);
    r.ptr = ptr.data(); r.x = x.data(); r.y = y.data();
    check(h, pdmpc_upload_reachable_sets(h, &r), "pdmpc_upload_reachable_sets");
}

// ASSEMBLE_OBSTACLES: standing successors' areas + parallel predecessors' reachable sets -> pdmpc_assemble_obstacles
void assemble_obstacles(pdmpc_handle *h, int nlhs, mxArray *plhs[], const mxArray *prhs[]) {
    const size_t N = mxGetM(prhs[2]);
    if (mxGetN(prhs[2]) < 4 || mxGetNumberOfElements(prhs[3]) != N || !mxIsCell(prhs[4]) || !mxIsCell(prhs[5]) ||
        mxGetNumberOfElements(prhs[4]) != N || mxGetNumberOfElements(prhs[5]) != N)
        fail("pdmpc:input", "ASSEMBLE_OBSTACLES: x0 [N x 4], trims [N], successors {N x 1}, parallel_predecessors {N x 1}");
    const int Hp = pdmpc_get_hp(h);
    const double *x0 = mxGetDoubles(prhs[2]);
    std::vector<int32_t> trim(N), sp(1, 0), si, pp(1, 0), pi;
    for (size_t i = 0; i < N; ++i) trim[i] = static_cast<int32_t>(mxGetDoubles(prhs[3])[i]);
    auto csr = [&](const mxArray *cells, std::vector<int32_t> &ptr, std::vector<int32_t> &idx) {
        for (size_t i = 0; i < N; ++i) {
            const mxArray *c = mxGetCell(cells, i);
            const size_t m = c ? mxGetNumberOfElements(c) : 0;
            for (size_t j = 0; j < m; ++j) idx.push_back(static_cast<int32_t>(mxGetDoubles(c)[j]) - 1);
            ptr.push_back(static_cast<int32_t>(idx.size()));
        }
    };
    csr(prhs[4], sp, si);
    csr(prhs[5], pp, pi);
    pdmpc_coupling_in in;
    std::memset(&in, 0, sizeof(in));
    in.n = static_cast<int32_t>(N);
    in.x = x0; in.y = x0 + N; in.yaw = x0 + 2 * N; in.speed = x0 + 3 * N;      // column-major N x 4
    in.trim = trim.data();
    in.succ_ptr = sp.data(); in.succ_idx = si.data(); in.par_ptr = pp.data(); in.par_idx = pi.data();
    in.half_length = mxGetScalar(prhs[6]); in.half_width = mxGetScalar(prhs[7]);
    std::vector<int32_t> slot(N * (Hp + 1) + 1), poly(si.size() + static_cast<size_t>(Hp) * pi.size() + 1);
    std::vector<double> vx(5 * si.size() + 256 * static_cast<size_t>(Hp) * pi.size() + 1), vy(vx.size());
    pdmpc_obstacles_out out;
    std::memset(&out, 0, sizeof(out));
    out.slot_ptr = slot.data(); out.poly_ptr = poly.data(); out.vert_x = vx.data(); out.vert_y = vy.data();
    out.poly_capacity = static_cast<int32_t>(poly.size() - 1); out.vert_capacity = static_cast<int32_t>(vx.size() - 1);
    check(h, pdmpc_assemble_obstacles(h, &in, &out), "pdmpc_assemble_obstacles");
    auto polygon = [&](int p) {
        const int a = poly[p], b = poly[p + 1];
        mxArray *m = mxCreateDoubleMatrix(2, b - a, mxREAL);
        for (int j = a; j < b; ++j) {
            mxGetDoubles(m)[2 * (j - a)] = vx[j];
            mxGetDoubles(m)[2 * (j - a) + 1] = vy[j];
        }
        return m;
    };
    plhs[0] = mxCreateCellMatrix(N, 1);
    if (nlhs > 1) plhs[1] = mxCreateCellMatrix(N, 1);
    for (size_t i = 0; i < N; ++i) {
        const int32_t *s = slot.data() + i * (Hp + 1);
        mxArray *st = mxCreateCellMatrix(s[1] - s[0], 1);                   // iter.obstacles rows
        for (int p = s[0]; p < s[1]; ++p) mxSetCell(st, p - s[0], polygon(p));
        mxSetCell(plhs[0], i, st);
        if (nlhs > 1) {
            const int rows = s[2] - s[1];                                   // one row per parallel predecessor
            mxArray *dy = mxCreateCellMatrix(rows, Hp);                     // iter.dynamic_obstacle_area rows
            for (int k = 1; k <= Hp; ++k)
                for (int q = 0; q < rows; ++q) mxSetCell(dy, q + static_cast<size_t>(rows) * (k - 1), polygon(s[k] + q));
            mxSetCell(plhs[1], i, dy);
        }
    }
}

// COUPLE: the reachable-set coupling of one scenario -> pdmpc_couple; adjacency = every coupled pair in either direction
void couple(pdmpc_handle *h, int nlhs, mxArray *plhs[], const mxArray *prhs[]) {
    const size_t N = mxGetM(prhs[2]);
    if (mxGetN(prhs[2]) < 3 || mxGetNumberOfElements(prhs[3]) != N) fail("pdmpc:input", "COUPLE: x0 [N x 3], trims [N]");
    const double *x0 = mxGetDoubles(prhs[2]);
    std::vector<int32_t> trim(N), sp = {0, static_cast<int32_t>(N)}, ptr[3], idx[3], level(N + 1);
    for (size_t i = 0; i < N; ++i) trim[i] = static_cast<int32_t>(mxGetDoubles(prhs[3])[i]);
    for (int k = 0; k < 3; ++k) {
        ptr[k].resize(N + 1);
        idx[k].resize(N * N + 1);
    }
    pdmpc_couple_params prm;
    prm.n_scenarios = 1; prm.scenario_ptr = sp.data(); prm.prioritizer = PDMPC_PRIORITY_CONSTANT; prm.max_num_CLs = 1;
    std::vector<double> area(N * N + 1);                   // symmetric: row-major == column-major
    pdmpc_couple_out out;
    std::memset(&out, 0, sizeof(out));
    out.succ_ptr = ptr[0].data(); out.succ_idx = idx[0].data(); out.par_ptr = ptr[1].data(); out.par_idx = idx[1].data();
    out.pred_ptr = ptr[2].data(); out.pred_idx = idx[2].data(); out.idx_capacity = static_cast<int32_t>(N * N + 1);
    out.level = level.data(); out.overlap_area = area.data();
    check(h, pdmpc_couple(h, static_cast<int32_t>(N), x0, x0 + N, x0 + 2 * N, trim.data(), &prm, &out), "pdmpc_couple");
    plhs[0] = mxCreateDoubleMatrix(N, N, mxREAL);
    double *adj = mxGetDoubles(plhs[0]);
    for (int k = 0; k < 3; ++k)
        for (size_t i = 0; i < N; ++i)
            for (int q = ptr[k][i]; q < ptr[k][i + 1]; ++q) {
                adj[i + N * idx[k][q]] = 1.0;
                adj[idx[k][q] + N * i] = 1.0;
            }
    if (nlhs > 1) {
        plhs[1] = mxCreateDoubleMatrix(N, N, mxREAL);
        std::copy(area.begin(), area.end() - 1, mxGetDoubles(plhs[1]));
    }
}

}  // namespace

void mexFunction(int nlhs, mxArray *plhs[], int nrhs, const mxArray *prhs[]) {
    if (nrhs < 1) fail("pdmpc:usage", "first argument must be the command");
    if (!g_at_exit_registered) {
        mexAtExit(release_all);
        g_at_exit_registered = true;
    }
    const int cmd = static_cast<int>(mxGetScalar(prhs[0]));
    if (cmd == CREATE) {
        const int dev = nrhs > 1 ? static_cast<int>(mxGetScalar(prhs[1])) : 0;
        pdmpc_handle *h = nullptr;
        const int rc = pdmpc_create(dev, &h);
        if (rc != PDMPC_OK) {
            const char *txt = pdmpc_last_error(nullptr);
            fail("pdmpc:create", std::string("pdmpc_create failed: ") + (txt ? txt : ""));
        }
        // valid-only queue wherever the CTA shape runs (one search per call, PLAN_TIMESTEP): 2-3x lower latency on
        // collision-rich searches; every field the shim returns is unaffected (pop_hash, which it does not return,
        // then covers the popped nodes that passed their check)
        pdmpc_set_cta_queue(h, 1);
        g_handles.push_back(h);
        plhs[0] = mxCreateNumericMatrix(1, 1, mxUINT64_CLASS, mxREAL);
        *static_cast<uint64_t *>(mxGetData(plhs[0])) = g_handles.size();   // 1-based; 0 = none
        return;
    }
    if (nrhs < 2) fail("pdmpc:usage", "second argument must be the planner handle");
    pdmpc_handle *h = handle_of(prhs[1]);
    switch (cmd) {
    case DESTROY: {
        const uint64_t idx = static_cast<uint64_t>(mxGetScalar(prhs[1]));
        pdmpc_destroy(h);
        g_handles[idx - 1] = nullptr;
        return;
    }
    case UPLOAD_MPA:
        if (nrhs < 4) fail("pdmpc:usage", "UPLOAD_MPA needs transition_matrix_single and maneuvers");
        upload_mpa(h, prhs[2], prhs[3]);
        return;
    case PLAN:
        if (nrhs < 12) fail("pdmpc:usage", "PLAN needs 12 arguments");
        plan(h, nlhs, plhs, prhs, false);
        return;
    case PLAN_SAMPLED:
        if (nrhs < 14) fail("pdmpc:usage", "PLAN_SAMPLED needs 14 arguments");
        plan(h, nlhs, plhs, prhs, true);
        return;
    case PLAN_TIMESTEP:
        if (nrhs < 14) fail("pdmpc:usage", "PLAN_TIMESTEP needs 14 arguments");
        plan_timestep(h, nlhs, plhs, prhs, false);
        return;
    case PLAN_TIMESTEP_SAMPLED:
        if (nrhs < 16) fail("pdmpc:usage", "PLAN_TIMESTEP_SAMPLED needs 16 arguments");
        plan_timestep(h, nlhs, plhs, prhs, false, true);
        return;
    case PLAN_JOINT:
        if (nrhs < 12) fail("pdmpc:usage", "PLAN_JOINT needs 12 arguments");
        plan_timestep(h, nlhs, plhs, prhs, true);
        return;
    case UPLOAD_ROAD:
        if (nrhs < 8) fail("pdmpc:usage", "UPLOAD_ROAD needs 8 arguments");
        upload_road(h, prhs);
        return;
    case SAMPLE_INPUTS:
        if (nrhs < 7) fail("pdmpc:usage", "SAMPLE_INPUTS needs 7 arguments");
        sample_inputs(h, nlhs, plhs, prhs);
        return;
    case UPLOAD_REACHABLE_SETS:
        if (nrhs < 3) fail("pdmpc:usage", "UPLOAD_REACHABLE_SETS needs 3 arguments");
        upload_reachable_sets(h, prhs);
        return;
    case ASSEMBLE_OBSTACLES:
        if (nrhs < 8) fail("pdmpc:usage", "ASSEMBLE_OBSTACLES needs 8 arguments");
        assemble_obstacles(h, nlhs, plhs, prhs);
        return;
    case COUPLE:
        if (nrhs < 4) fail("pdmpc:usage", "COUPLE needs 4 arguments");
        couple(h, nlhs, plhs, prhs);
        return;
    case STATS: {
        pdmpc_stats st;
        check(h, pdmpc_get_stats(h, &st), "pdmpc_get_stats");
        static const char *names[] = {"kernel_ms", "h2d_ms", "d2h_ms", "total_pops", "total_nodes", "total_obstacle_cols"};
        plhs[0] = mxCreateStructMatrix(1, 1, 6, names);
        const double vals[] = {st.kernel_ms, st.h2d_ms, st.d2h_ms, static_cast<double>(st.total_pops),
                               static_cast<double>(st.total_nodes), static_cast<double>(st.total_obstacle_cols)};
        for (int i = 0; i < 6; ++i) mxSetField(plhs[0], 0, names[i], mxCreateDoubleScalar(vals[i]));
        return;
    }
    default:
        fail("pdmpc:usage", "unknown command");
    }
}
