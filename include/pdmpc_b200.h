/*
 * pdmpc_b200.h — C ABI of the B200-native drop-in for p-dmpc's per-vehicle
 * trajectory optimizer (hlc/optimizer graph search over the motion-primitive
 * automaton, MPA).
 *
 * This is the boundary a MATLAB MEX shim (see INTEGRATION.md and
 * p-dmpc_b200/matlab/) binds.  It replaces, for the hot path only:
 *
 *   reference interface                                      file:line
 *   -------------------------------------------------------  ------------------------------------------------------
 *   OptimizerInterface.run_optimizer(veh, iter, mpa, opt, k) hlc/optimizer/OptimizerInterface.m:14
 *   GraphSearch.do_graph_search / eval_edge_exact            hlc/optimizer/graph_search/GraphSearch.m:23-196
 *   expand_node                                              hlc/optimizer/graph_search/expand_node.m:1-91
 *   are_constraints_satisfied_sat / intersect_sat            hlc/optimizer/graph_search/are_constraints_satisfied_sat.m:1-68,
 *                                                            hlc/optimizer/graph_search/intersect_sat.m:1-42
 *   intersect_lanelet_boundary                               hlc/optimizer/common/intersect_lanelet_boundary.m:1-56
 *   are_constraints_satisfied_interx / InterX                hlc/optimizer/graph_search/are_constraints_satisfied_interx.m:1-39,
 *                                                            hlc/optimizer/graph_search/InterX.m:48-110
 *   vectorize_all_obstacles                                  hlc/optimizer/graph_search/vectorize_all_obstacles.m:1-76
 *   priority_queue_interface_mex (NEW/PUSH/POP)              hlc/optimizer/graph_search/priority_queue/priority_queue_interface_mex.cpp:19-108
 *   return_path_to / return_path_area                        hlc/optimizer/graph_search/return_path_to.m:1-27, return_path_area.m:1-8
 *   MonteCarloTreeSearch.run_optimizer / do_graph_search     hlc/optimizer/graph_search/MonteCarloTreeSearch.m:29-251
 *   the same search with iter.amount > 1 (joint)             hlc/controller/centralized/CentralizedController.m:33-59,
 *                                                            expand_node.m:15-75, are_constraints_satisfied_sat.m:37-44
 *   level loop + hand-over of predecessors' areas            hlc/controller/prioritized/PrioritizedSequentialController.m:74-92,
 *   (pdmpc_plan_timestep, optional)                          PrioritizedController.m:297-324,355-364,449-506
 *   simultaneous prioritizations: permuted relations, costs, hlc/controller/prioritized/PrioritizedExplorativeController.m:
 *   choice and commit (pdmpc_plan_timestep_explorative)      55-78,94-176
 *
 * Conventions
 *   - plain C, no C++ types, no exceptions cross this boundary; every call
 *     returns an int status (PDMPC_OK == 0) and pdmpc_last_error() gives text.
 *   - all host buffers are caller-owned; the library owns device memory.
 *   - trims and node ids are 1-BASED, exactly as MATLAB passes / expects them
 *     (Tree.m:18,61: root id 1, parent(root) = 0).
 *   - all floating point is IEEE double; the device path computes with the
 *     same operation order as the reference and with FMA contraction off.
 *   - one handle per host thread / process (MATLAB calls MEX from its main
 *     thread; parallel_threads = separate processes, utility/get_parallel_pool.m:37).
 *   - there is NO CPU fallback: without a CUDA device pdmpc_create fails with
 *     PDMPC_ERR_CUDA.
 */
#ifndef PDMPC_B200_H
#define PDMPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDMPC_ABI_VERSION 2

/* A maneuver area polygon has 5 (straight), 6 (turn, convex build) or 7 (turn,
 * non-convex build) closed points: generate_maneuver.m:73-103.  Fixed stride. */
#define PDMPC_AREA_STRIDE 8
/* Upper bound on the prediction horizon accepted by the library (Config.m:33
 * default 6; eval_phd.m:14-19 uses up to 10). */
#define PDMPC_MAX_HP 16
/* Upper bound on the number of trims (realistic MPA: 71). */
#define PDMPC_MAX_TRIMS 128
/* Most vehicles of one centralized (joint) search (pdmpc_joint_plan_batch). */
#define PDMPC_MAX_JOINT 4
#define PDMPC_MAX_PRED_LANELETS 8   /* predicted lanelets per vehicle: at most Hp + 1 distinct ones */

enum pdmpc_status {
    PDMPC_OK = 0,
    PDMPC_ERR_BAD_INPUT = 1,   /* null pointer, sizes out of range, malformed CSR, open polygon */
    PDMPC_ERR_CUDA = 2,        /* CUDA runtime error (text in pdmpc_last_error) */
    PDMPC_ERR_CAPACITY = 3,    /* a search outgrew the node arena / heap: never truncated silently */
    PDMPC_ERR_NO_MPA = 4,      /* plan called before pdmpc_upload_mpa */
    PDMPC_ERR_ALLOC = 5
};

/* Which constraint checker the search uses (OptimizerInterface.m:36-46,
 * Config.m:71-87): SAT for circle / non-prioritized, InterX otherwise. */
enum pdmpc_checker {
    PDMPC_CHECKER_SAT = 0,
    PDMPC_CHECKER_INTERX = 1
};

/* area kinds of one maneuver (generate_maneuver.m:39-64) */
enum pdmpc_area_kind {
    PDMPC_AREA_NORMAL = 0,         /* maneuver.area               (offset 0.01 all round) */
    PDMPC_AREA_WITHOUT_OFFSET = 1, /* maneuver.area_without_offset                         */
    PDMPC_AREA_LARGE_OFFSET = 2    /* maneuver.area_large_offset  (+0.05 in length)        */
};

typedef struct pdmpc_handle pdmpc_handle;

/* ---- MPA tables: what the search reads of MotionPrimitiveAutomaton
 *      (MotionPrimitiveAutomaton.m:5-17) ------------------------------------ */
typedef struct pdmpc_mpa_desc {
    int32_t n_trims;            /* numel(mpa.trims) */
    int32_t Hp;                 /* size(transition_matrix_single, 3) */
    int32_t n_edges;            /* number of non-empty mpa.maneuvers{t1,t2} */
    /* transition_matrix_single(t1,t2,k) != 0, laid out [k-1][t1-1][t2-1] */
    const uint8_t *transition;  /* Hp * n_trims * n_trims */
    const int32_t *edge_from;   /* [n_edges] t1, 1-based */
    const int32_t *edge_to;     /* [n_edges] t2, 1-based */
    const double *edge_dx;      /* [n_edges] maneuver.dx   */
    const double *edge_dy;      /* [n_edges] maneuver.dy   */
    const double *edge_dyaw;    /* [n_edges] maneuver.dyaw */
    const int32_t *area_npts;   /* [n_edges*3] points per area kind (closed: first == last) */
    const double *area_x;       /* [n_edges*3*PDMPC_AREA_STRIDE] local-frame x */
    const double *area_y;       /* [n_edges*3*PDMPC_AREA_STRIDE] local-frame y */
} pdmpc_mpa_desc;

/* ---- One batch of independent searches (vehicle x permutation x scenario).
 *      Each search is what PrioritizedController.plan hands to run_optimizer
 *      (PrioritizedController.m:297-341) reduced to the IterationData fields
 *      the search reads (IterationData.m:4-33), nV == 1. -------------------- */
typedef struct pdmpc_batch_in {
    int32_t n_searches;
    int32_t checker;            /* enum pdmpc_checker, same for the whole batch */
    double dt_seconds;          /* options.dt_seconds */
    const double *x0;           /* [n] iter.x0(:,1) */
    const double *y0;           /* [n] iter.x0(:,2) */
    const double *yaw0;         /* [n] iter.x0(:,3) */
    const int32_t *trim0;       /* [n] iter.trim_indices, 1-based */
    const double *ref_x;        /* [n*Hp] iter.reference_trajectory_points(1,k,1) */
    const double *ref_y;        /* [n*Hp] iter.reference_trajectory_points(1,k,2) */
    const double *v_ref;        /* [n*Hp] iter.v_ref(1,k) */
    /* Obstacle polygons as a three-level CSR.  Slot s = search*(Hp+1) + k:
     *   k = 0      -> iter.obstacles{:}               (static, checked at every step)
     *   k = 1..Hp  -> iter.dynamic_obstacle_area{:,k} (checked at step k)
     * slot_ptr[s]..slot_ptr[s+1] are polygon indices, poly_ptr[p]..poly_ptr[p+1]
     * are vertex indices into vert_x/vert_y.  Polygons are closed (first vertex
     * repeated last), as vectorize_all_obstacles.m:71-76 asserts. */
    const int32_t *slot_ptr;    /* [n*(Hp+1)+1] */
    const int32_t *poly_ptr;    /* [n_polys+1]  */
    const double *vert_x;       /* [n_verts] */
    const double *vert_y;       /* [n_verts] */
    /* iter.predicted_lanelet_boundary{1,1:2}: open polylines.  lane_ptr[2*i] ..
     * lane_ptr[2*i+1] = left bound of search i, lane_ptr[2*i+1]..lane_ptr[2*i+2]
     * = right bound.  Empty ranges = no lanelets (circle scenario). */
    const int32_t *lane_ptr;    /* [2n+1] */
    const double *lane_x;       /* [n_lane_pts] */
    const double *lane_y;       /* [n_lane_pts] */
} pdmpc_batch_in;

/* ---- Results, caller-allocated, SoA over the batch.  Field meaning follows
 *      ControlResultsInfo (ControlResultsInfo.m:5-17) and the flat outputs
 *      OptimizerInterface.create_control_results_info_from_mex consumes
 *      (OptimizerInterface.m:63-101).  Any pointer may be NULL = not wanted,
 *      except status. --------------------------------------------------------- */
typedef struct pdmpc_batch_out {
    int32_t *status;        /* [n] per-search pdmpc_status */
    uint8_t *is_exhausted;  /* [n] info.is_exhausted */
    int32_t *n_expanded;    /* [n] info.n_expanded == tree.size() at exit (GraphSearch.m:58,89) */
    int32_t *n_pops;        /* [n] number of pq.pop() that returned a node */
    uint64_t *pop_hash;     /* [n] FNV-1a over the popped node ids, in pop order (parity trace; launch shape 5:
                             *     over the popped ids that passed their edge check, see pdmpc_set_variant) */
    int32_t *trims;         /* [n*(Hp+1)] current_and_predicted_trims, 1-based; zeros after col 1 if exhausted */
    int32_t *tree_path;     /* [n*(Hp+1)] node ids root..goal in the full tree; zeros if exhausted */
    double *y_predicted;    /* [n*Hp*3] (x,y,yaw) per step; NaN if exhausted */
    double *g_path;         /* [n*(Hp+1)] tree.g along the path (cost to come); NaN if exhausted */
    double *h_path;         /* [n*(Hp+1)] tree.h along the path; NaN if exhausted */
    int32_t *shape_npts;    /* [n*Hp] points of info.shapes{1,k}; 0 if exhausted */
    double *shape_x;        /* [n*Hp*PDMPC_AREA_STRIDE] */
    double *shape_y;        /* [n*Hp*PDMPC_AREA_STRIDE] */
} pdmpc_batch_out;

/* Device-side counters of the last plan call (for roofline accounting,
 * SURVEY.md §8(d)). */
typedef struct pdmpc_stats {
    double kernel_ms;        /* CUDA-event time of the search kernel(s) */
    double h2d_ms;           /* host->device staging */
    double d2h_ms;           /* device->host results */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t total_pops;
    int64_t total_nodes;
    int64_t total_obstacle_cols; /* sum over pops of (V_k + L) columns tested */
    int32_t kernel_launches;
    int32_t handed_over;     /* shape 5: searches re-run with the exact queue after a non-unique minimum */
    int32_t shape;           /* the launch shape that actually ran (1..5, see pdmpc_set_variant): a requested
                              * shape that cannot serve a batch falls back, and says so here */
    int32_t escalated;       /* shapes 2, 3: searches given up after pdmpc_set_escalation pops and run by the CTA shape */
} pdmpc_stats;

/* Create a planner bound to CUDA device `device_id`.  Fails (PDMPC_ERR_CUDA)
 * when no such device exists: there is no CPU path. */
int pdmpc_create(int device_id, pdmpc_handle **out);
int pdmpc_destroy(pdmpc_handle *h);
const char *pdmpc_last_error(const pdmpc_handle *h);
int pdmpc_abi_version(void);
/* Hp of the uploaded MPA (0: none).  pdmpc_batch_in carries no Hp: every per-step array of a batch is indexed
 * with this one, so a binding must check its arrays against it before a plan call (the MEX shim and the ctypes
 * binding do). */
int pdmpc_get_hp(const pdmpc_handle *h);

/* Node-arena capacity (nodes per concurrently running search).  Default is the
 * full-tree bound of the uploaded MPA when it is below 2^20, else 2^20.  A
 * search that needs more returns PDMPC_ERR_CAPACITY in its status. */
int pdmpc_set_node_capacity(pdmpc_handle *h, int32_t max_nodes_per_search);

/* Launch shape of the search kernel: 0 = choose from the batch size (default);
 * 1 = one search per one-warp CTA (lowest latency of the warp shapes; every checker);
 * 2 = tiles, TWO searches per warp, 3 = tiles, FOUR searches per warp (p-dmpc_b200/csrc/pdmpc_tiles.cuh: the
 *     throughput shapes — one iteration of a warp pops one node for each of its searches, so the warp-uniform
 *     work is issued once for all of them; InterX batches only, SAT batches fall back to 1);
 * 4 = cta (one 16-warp CTA per search: a master warp owns queue and tree, checker warps validate the children
 *     of every expansion ahead of their pop; chosen automatically for batches of at most one search per SM;
 *     falls back to 1 when the full search tree of the MPA exceeds 32768 nodes);
 * 5 = shape 4 with a VALID-ONLY QUEUE: children whose edge check failed are not pushed; before every pop the
 *     minimum must be unique, otherwise the search is re-run with the exact queue (p-dmpc_b200/csrc/
 *     pdmpc_cta.cuh has the argument why every output then equals the reference's).
 * 0 picks 4 for n <= #SMs, 2 when there are more searches than shape 1 keeps in flight, else 1.
 * pdmpc_stats.shape reports the shape that actually ran.
 * Results do not depend on the shape, with ONE exception: pop_hash, a parity trace that is not
 * part of the reference's ControlResultsInfo, covers the popped nodes that passed their edge
 * check only in shape 5 (n_pops is exact in every shape). */
int pdmpc_set_variant(pdmpc_handle *h, int32_t variant);

/* The queue of the CTA shape whenever that shape runs (chosen automatically for small batches and by
 * pdmpc_plan_timestep, or forced with shape 4): 0 = the reference's lazy queue (default: pop_hash covers every
 * pop), 1 = the valid-only queue of shape 5 (2-3x lower latency on collision-rich searches; pop_hash covers
 * the valid pops; pdmpc_stats.shape then reports 5).  The MATLAB drop-in turns it on. */
int pdmpc_set_cta_queue(pdmpc_handle *h, int32_t valid_only);

/* Shapes 2, 3 only: ESCALATION of the longest searches.  A tile warp needs ~5 us per pop, so one search of
 * 8000 pops (1 in 10^5 of the road-network records) would hold a whole launch open for 40 ms.  A search that
 * reaches `pops` pops in a tile kernel is given up there and run from scratch by the CTA shape (4, or 5 after
 * pdmpc_set_cta_queue(1)) behind the tile kernel on the same stream.  0 = never; -1 (default) = by batch size:
 * 2560 pops, 3072 from 120 000 and 4096 from 300 000 searches per call, fewer for the searches that start late
 * in the work order (pdmpc_escalation_budgets; a pops > 0 is one budget for every search).  A list of at
 * most `short_list_max` searches (-1 = default, 3 per SM) runs with one master warp per CTA, all checker warps
 * serving it — the launch then ends with its longest search at 0.65 us per pop —, a longer one with several
 * masters per CTA.  Results do not depend on either; pdmpc_stats.escalated counts the searches that took this
 * route. */
int pdmpc_set_escalation(pdmpc_handle *h, int32_t pops, int32_t short_list_max);

/* Shapes 2, 3 only: polyline points (lanelet bounds + obstacles of all steps) a tile stages in shared
 * memory per search (0 = what the kernel holds, 256); polylines beyond it are read from HBM/L2.  Test knob:
 * results do not depend on it. */
int pdmpc_set_tile_points(pdmpc_handle *h, int32_t points);

/* Shape 4 only: heap entries kept in shared memory (0 = default 4096, even); the rest of the
 * queue spills to the HBM arena.  Tuning/test knob: results do not depend on it. */
int pdmpc_set_cta_heap_smem(pdmpc_handle *h, int32_t entries);

/* pdmpc_plan_batch on large host batches (>= 16384 searches, launch shapes 0..3) runs as a chunked
 * pipeline: host->device copies, searches and device->host copies of consecutive chunks overlap.
 * chunks: 0 = choose from the batch size (default: ~60 k searches per chunk, 2..12 chunks), 1 = off, 2..16 = that many chunks for any batch
 * of at least 2*chunks searches.  Tuning/test knob: results do not depend on it. */
int pdmpc_set_pipeline_chunks(pdmpc_handle *h, int32_t chunks);

/* The chunk boundaries pdmpc_plan_batch uses for a batch of n_searches (host-only, needs no device): chunk c = searches
 * [bounds[c], bounds[c+1]).  chunks = 0: the default (~60 000 searches per chunk, 2..12 chunks); chunks = 2..16: what
 * pdmpc_set_pipeline_chunks(chunks) gives.  Chunks are of equal size, the first one half of that.
 * bounds: cap >= *n_chunks + 1 entries (PDMPC_ERR_CAPACITY otherwise, *n_chunks is still set). */
int pdmpc_pipeline_bounds(int32_t n_searches, int32_t chunks, int32_t cap, int32_t *bounds, int32_t *n_chunks);

/* The pop budgets of the throughput shapes under the default escalation threshold (pdmpc_set_escalation(-1, ..)) in a
 * batch of n_searches (host-only, needs no device): budgets[i] = the pops after which the search at work position
 * positions[i] (0 <= positions[i] < n_searches) is given up and run again by the CTA shape (0 = never).  A search that
 * starts late in the work order gets fewer pops than one that starts early. */
int pdmpc_escalation_budgets(int32_t n_searches, int32_t count, const int32_t *positions, int32_t *budgets);

/* Diagnostics: the timeline of the LAST pipelined pdmpc_plan_batch call, per chunk: host_ms = host time since the start
 * of the call at which the chunk's copies and kernel had been enqueued (after its validation), in_ms / done_ms = device
 * time since the first copy started at which its inputs had landed / its searches were done.  Arrays of `cap` entries
 * (NULL = not wanted); *n_chunks = chunks of that call (0: the last call was not pipelined). */
int pdmpc_get_pipeline_timeline(pdmpc_handle *h, int32_t cap, double *host_ms, double *in_ms, double *done_ms, int32_t *n_chunks);

/* Stage the MPA tables in HBM (once per MPA; cached in the handle). */
int pdmpc_upload_mpa(pdmpc_handle *h, const pdmpc_mpa_desc *mpa);

/* Plan a batch whose inputs/outputs are HOST buffers: stage -> search -> fetch. */
int pdmpc_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, pdmpc_batch_out *out);

/* Device-resident variant for throughput runs: stage once, run many, fetch once. */
int pdmpc_stage_batch(pdmpc_handle *h, const pdmpc_batch_in *in);
int pdmpc_run_staged(pdmpc_handle *h);                 /* launches on the handle's stream, no host sync */
int pdmpc_sync(pdmpc_handle *h);
int pdmpc_fetch_staged(pdmpc_handle *h, pdmpc_batch_out *out);

int pdmpc_get_stats(pdmpc_handle *h, pdmpc_stats *out);

/* ---- OptimizerType.MatlabSampled: MonteCarloTreeSearch.run_optimizer
 *      (hlc/optimizer/graph_search/MonteCarloTreeSearch.m:29-251), selected by
 *      OptimizerInterface.get_optimizer (hlc/optimizer/OptimizerInterface.m:28-30).
 *      Same per-search inputs and the same constraint checkers as the graph
 *      search; random roll-outs from the root, at most n_expansions_max node
 *      expansions, the cheapest valid leaf at depth Hp wins. ------------------ */
typedef struct pdmpc_mcts_params {
    int32_t n_expansions_max;   /* MonteCarloTreeSearch.m:8 (default 250); 1 .. PDMPC_MCTS_MAX_EXPANSIONS */
    const uint32_t *seed;       /* [n] RandStream('mt19937ar', Seed = time_step + vehicle_index), :31 */
} pdmpc_mcts_params;
#define PDMPC_MCTS_MAX_EXPANSIONS 1023
#define PDMPC_MCTS_MAX_BRANCH 16   /* mpa.maximum_branching_factor() accepted by the sampled optimizer */

/* Host buffers in, host buffers out (like pdmpc_plan_batch).  Output fields as
 * for the graph search with these differences, all following the reference:
 *   n_expanded  = n_expansions (:199)            n_pops = n_traversals (random numbers consumed)
 *   pop_hash    = FNV-1a over ((node_id << 8) | child_position) of every roll-out step taken
 *   tree_path   = node ids in the sampled tree (root 1, ids in order of creation, :177)
 *   g_path      = -1 except the goal leaf, which carries the solution cost (:211,239); h_path = -1
 * A search whose roll-outs would read past the Hp * n_expansions_max random numbers drawn at
 * :52 (MATLAB raises an index error there) reports PDMPC_ERR_CAPACITY. */
int pdmpc_mcts_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_mcts_params *prm,
                          pdmpc_batch_out *out);
/* Device-resident form: inputs staged with pdmpc_stage_batch, results read with pdmpc_fetch_staged. */
int pdmpc_mcts_run_staged(pdmpc_handle *h, const pdmpc_mcts_params *prm);

/* ---- One whole time step (or many) in ONE call: the part of
 *      PrioritizedController.plan that hands the plans of higher-priority
 *      vehicles to the vehicles planning after them
 *      (hlc/controller/prioritized/PrioritizedController.m:297-324, consider_predecessors
 *      :449-506, publish_predictions :355-364) moves onto the device.  The searches of the
 *      batch form a DAG: search i waits for its sequential predecessors pred_idx[pred_ptr[i] ..
 *      pred_ptr[i+1]) — searches of the SAME batch — and sees, at step k, the area
 *      info_j.shapes{1,k} each of them has just planned as one more row of
 *      iter.dynamic_obstacle_area (appended after the rows the caller passed in `in`; the
 *      checkers only ask whether ANY obstacle is hit, so the row order changes no result).
 *      A predecessor whose search is exhausted publishes its fallback areas instead: what
 *      plan_fallback (:678-718, del_first_rpt_last of the previous plan's shapes) or
 *      handle_graph_search_exhaustion (:568-621, the standstill rectangle) would publish.  Both
 *      depend only on the previous time step, so the caller passes them up front.
 *      Computation levels are not needed: every search starts the moment its own predecessors
 *      are done (flags in HBM, one persistent launch), which is never later than its level. ---- */
typedef struct pdmpc_timestep_deps {
    const int32_t *pred_ptr;  /* [n+1] CSR over the searches of the batch, pred_ptr[0] == 0 */
    const int32_t *pred_idx;  /* [pred_ptr[n]] 0-based search indices; the relation must be acyclic */
    /* areas search i publishes when it is exhausted; NULL = an exhausted search publishes nothing */
    const int32_t *fb_npts;   /* [n*Hp] closed points per step, 0 (nothing) or 2..PDMPC_AREA_STRIDE-1 */
    const double *fb_x;       /* [n*Hp*PDMPC_AREA_STRIDE] */
    const double *fb_y;       /* [n*Hp*PDMPC_AREA_STRIDE] */
} pdmpc_timestep_deps;
/* Most sequential predecessors one search may have: Hp * PDMPC_AREA_STRIDE columns each must fit the
 * tile that holds them (PDMPC_TIMESTEP_COLS columns; shared memory in the CTA kernel). */
#define PDMPC_TIMESTEP_COLS 2048

/* Host buffers in, host buffers out (like pdmpc_plan_batch): one host->device copy, one launch,
 * one device->host copy for the whole DAG.  Every output equals what level-by-level calls of
 * pdmpc_plan_batch with host-side obstacle assembly return.  Launch shape: one CTA per search for up to
 * 48 searches per SM, one warp per search beyond that and for MPAs whose full search tree exceeds the
 * 32768 nodes the CTA kernel holds (pdmpc_set_variant 1..3 / 4..5 force either; results do not depend on
 * it).  Errors: PDMPC_ERR_BAD_INPUT for a cyclic or out-of-range relation or too many predecessors. */
int pdmpc_plan_timestep(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                        pdmpc_batch_out *out);

/* ---- Centralized (joint) search: GraphSearch.do_graph_search with iter.amount = n_vehicles > 1, what
 *      CentralizedController.controller calls (hlc/controller/centralized/CentralizedController.m:33-59):
 *      successors = Cartesian product of the vehicles' successors, first vehicle fastest
 *      (expand_node.m:15-26), costs summed over the vehicles in order (:43-75), every vehicle of a popped
 *      node checked in order against the static and dynamic obstacles, the vehicles before it and its own
 *      lanelet boundary (GraphSearch.m:150-192, are_constraints_satisfied_sat.m:15-53).  SAT checker only
 *      (are_constraints_satisfied_interx.m:12 asserts a single vehicle).
 *      Rows of `in` / `out` are (search, vehicle): r = search * n_vehicles + v, in->n_searches = number of
 *      ROWS.  iter.obstacles / iter.dynamic_obstacle_area of a search go into the slots of its first row
 *      (the other rows' slots must be empty); lanelet bounds, poses, trims, references are per row.  Per-row
 *      outputs: trims, y_predicted, shapes; status, is_exhausted, n_expanded, n_pops, pop_hash, tree_path,
 *      g_path and h_path (joint values) are repeated on every row of a search.  Node capacity per search: what
 *      pdmpc_set_node_capacity says, else what 2 GiB of arena give every resident search (at least 2^17, at
 *      most 2^28 - 1 nodes: branching is up to 12^n_vehicles per expansion); PDMPC_ERR_CAPACITY beyond it. ---- */
int pdmpc_joint_plan_batch(pdmpc_handle *h, const pdmpc_batch_in *in, int32_t n_vehicles, pdmpc_batch_out *out);

/* Diagnostics: the FP64 pipe peak of the handle's device, measured with register-only kernels
 * (no memory traffic): tera-operations/s of separate multiply + add (what the search executes: FMA
 * contraction is off for bit-exactness) and TFLOP/s of fused multiply-add.  The denominators of the
 * FP64 roofline fraction bench.py reports next to the HBM one. */
int pdmpc_measure_fp64_peak(pdmpc_handle *h, double *mul_add_tops, double *fma_tflops);

/* The plans of the LAST plan call as flat rows in DEVICE memory, ready for a collective — BASELINE configs[2]
 * (simultaneous prioritizations): the ranks exchange the cost of every vehicle in every permutation and the
 * winners' plans (PrioritizedExplorativeController.m:94-109 compute_solution_cost, :124-176 receive / choose /
 * publish) with one all_gather on these rows; nothing is routed through the host before the exchange.
 * Row r (search r of the call), L = 2 + 21*Hp doubles:
 *   [0] cost = g_path[r][Hp] (tree.get_cost of the goal node)   [1] 1.0 if the row is a fallback plan, else 0.0
 *   [2 .. 2+Hp) trims of steps 1..Hp   [.. +3Hp) y_predicted   [.. +Hp) shape_npts   [.. +8Hp) shape_x   [.. +8Hp) shape_y
 * For an exhausted search the row of vehicle (r mod n_vehicles) of `fallback_rows` [n_vehicles * L] (host; the
 * fallback plan and its cost are known before the time step, PrioritizedController.m:678-718) is taken instead
 * (zeros if fallback_rows is NULL).  `device_dst`: n_rows * L doubles of device memory on the handle's device
 * (e.g. a torch tensor's data pointer); complete when the call returns. */
int pdmpc_pack_plan_rows(pdmpc_handle *h, int32_t n_rows, int32_t n_vehicles, const double *fallback_rows,
                         void *device_dst);

/* ---- The input side of a time step on the device (SURVEY.md 8(f) rank 4): per vehicle the reference trajectory over
 *      the horizon and the lanelet boundary of the predicted lanelets — what HighLevelController fills into
 *      iter.reference_trajectory_points / v_ref / predicted_lanelets / predicted_lanelet_boundary before the
 *      optimizer runs (get_reference_trajectory.m:28-46, sample_reference_trajectory.m:24-97,
 *      get_arc_distance_to_endpoint.m:41-113, projection_2d.m, get_predicted_lanelets.m:25-62,
 *      get_lanelets_boundary.m:19-68).  Road + reference paths are uploaded once (cached in the handle). ----- */
typedef struct pdmpc_road_desc {
    int32_t n_lanelets;
    const int32_t *bound_ptr;       /* [2*n_lanelets+1]: left bound of lanelet l (0-based) at [bound_ptr[2l], bound_ptr[2l+1]),
                                     *   right bound at [bound_ptr[2l+1], bound_ptr[2l+2]) — lanelet_boundaries{l}{1:2} */
    const double *bound_x, *bound_y;
    int32_t n_paths;                /* reference paths (one per vehicle of every scenario) */
    const int32_t *path_ptr;        /* [n_paths+1] into path_x / path_y: reference_path (n x 2) */
    const double *path_x, *path_y;
    const int32_t *lan_ptr;         /* [n_paths+1] into lanelets_index / points_index */
    const int32_t *lanelets_index;  /* lanelet ids (1-based) along the path: reference_path_struct.lanelets_index */
    const int32_t *points_index;    /* 1-based index of the last path point of each of them: .points_index */
    const uint8_t *is_loop;         /* [n_paths] */
    const double *reference_speed;  /* [n_paths] */
} pdmpc_road_desc;

typedef struct pdmpc_inputs_out {   /* caller-owned host buffers; NULL fields are not copied back */
    double *ref_x, *ref_y, *v_ref;  /* [n*Hp] iter.reference_trajectory_points(:, :, 1:2), iter.v_ref */
    int32_t *ref_index;             /* [n*Hp] reference_trajectory_struct.points_index (1-based) */
    int32_t *current_index;         /* [n] current_point_index */
    int32_t *predicted_lanelets;    /* [n*PDMPC_MAX_PRED_LANELETS] 1-based lanelet ids, 0 padded */
    int32_t *lane_ptr;              /* [2n+1] as pdmpc_batch_in.lane_ptr */
    double *lane_x, *lane_y;        /* [lane_capacity] as pdmpc_batch_in.lane_x / lane_y */
    int32_t lane_capacity;          /* PDMPC_ERR_CAPACITY if the bounds need more points */
} pdmpc_inputs_out;

int pdmpc_upload_road(pdmpc_handle *h, const pdmpc_road_desc *road);
/* Row i: the vehicle on reference path path_id[i] (0-based) stands at (x[i], y[i]) and drives at speed[i]
 * (mpa.trims(trim).speed).  Needs an uploaded MPA (Hp) and road.  One warp per row. */
int pdmpc_sample_inputs(pdmpc_handle *h, int32_t n, const int32_t *path_id, const double *x, const double *y,
                        const double *speed, double dt_seconds, pdmpc_inputs_out *out);

/* ---- Obstacle assembly of a time step on the device (SURVEY.md 8(f) rank 1, the part that does not depend on this
 *      time step's plans): what PrioritizedController.plan puts into iter_v.obstacles / iter_v.dynamic_obstacle_area
 *      before the optimizer runs, for all vehicles (of all scenarios) in one call:
 *        - a coupled vehicle of LOWER priority that stands (|speed| < 0.01) is a static obstacle, its area the offset
 *          rectangle at its pose (consider_successors with ConstraintFromSuccessor.area_of_standstill,
 *          hlc/controller/prioritized/PrioritizedController.m:508-540; get_occupied_areas.m:19-25);
 *        - a coupled vehicle of HIGHER priority that plans in PARALLEL enters through its reachable sets, one dynamic
 *          obstacle per step (parallel_coupling_reachability :391-407 via consider_predecessors :449-506): the local
 *          reachable sets of its current trim placed at its pose (MotionPrimitiveAutomaton.reachable_sets_at_pose,
 *          hlc/model/motion_primitive_automaton/MotionPrimitiveAutomaton.m:649-687, utility/translate_global.m:20-23).
 *      (The areas of SEQUENTIAL predecessors are handed over inside pdmpc_plan_timestep.)  The reference also clips a
 *      reachable set by the predicted lanelets' polyshape (HighLevelController.m:241-246, a MATLAB polyshape
 *      intersection): not done here, the caller uploads the sets it wants placed. ---- */
typedef struct pdmpc_reach_desc {    /* mpa.local_reachable_sets_conv{trim, t} as closed polygons (first point repeated) */
    int32_t n_trims, Hp;             /* must equal the uploaded MPA's */
    const int32_t *ptr;              /* [n_trims*Hp+1] into x / y: set of (trim i, step t) (0-based) at ptr[i*Hp+t] */
    const double *x, *y;
} pdmpc_reach_desc;
int pdmpc_upload_reachable_sets(pdmpc_handle *h, const pdmpc_reach_desc *sets);

typedef struct pdmpc_coupling_in {
    int32_t n;                       /* rows: the vehicles of every scenario of the time step */
    const double *x, *y, *yaw;       /* [n] measured pose (iter.x0(:, 1:3)) */
    const double *speed;             /* [n] iter.x0(:, 4) */
    const int32_t *trim;             /* [n] iter.trim_indices, 1-based */
    const int32_t *succ_ptr;         /* [n+1] CSR: coupled rows of lower priority (directed_coupling(i, :)) */
    const int32_t *succ_idx;
    const int32_t *par_ptr;          /* [n+1] CSR: coupled rows of higher priority in another group (they plan in parallel) */
    const int32_t *par_idx;
    double half_length, half_width;  /* Length/2 + offset, Width/2 + offset (get_occupied_areas.m:21-22) */
} pdmpc_coupling_in;

typedef struct pdmpc_obstacles_out { /* caller-owned host buffers in the layout of pdmpc_batch_in's obstacle CSR */
    int32_t *slot_ptr;               /* [n*(Hp+1)+1]: slot i*(Hp+1) = standing successors of row i (in succ order), slot
                                      *   i*(Hp+1)+k = step-k reachable set of every parallel predecessor (in par order) */
    int32_t *poly_ptr;               /* [poly_capacity+1] */
    double *vert_x, *vert_y;         /* [vert_capacity] */
    int32_t poly_capacity, vert_capacity;   /* PDMPC_ERR_CAPACITY if the time step needs more (n_polys / n_verts say how much) */
    int32_t n_polys, n_verts;        /* out: polygons and vertices written */
} pdmpc_obstacles_out;
int pdmpc_assemble_obstacles(pdmpc_handle *h, const pdmpc_coupling_in *in, pdmpc_obstacles_out *out);

/* ---- The output side of a time step on the device (SURVEY.md 8(f) rank 4): the plan a vehicle falls back to when
 *      its search is exhausted — standstill at its pose (handle_graph_search_exhaustion,
 *      PrioritizedController.m:568-621, area = get_occupied_areas.m:21-25) or the previous plan shifted by one step
 *      (plan_fallback :678-718, del_first_rpt_last) — needs the previous time step's plans; they stay on the device,
 *      one SLOT per vehicle (of every scenario the handle serves).
 *      pdmpc_closed_loop_reset: forget all plans (scenario start).  half_length / half_width = Length/2 + offset,
 *      Width/2 + offset of the standstill rectangle.
 *      pdmpc_plan_timestep_closed_loop = pdmpc_plan_timestep, except that (i) deps->fb_* are ignored: the fallback
 *      areas exhausted predecessors publish are built on the device from the slots' previous plans (standstill[i] != 0,
 *      or no previous plan: the standstill rectangle at (x0, y0, yaw0), trims = trim0), (ii) on return trims[1..Hp],
 *      y_predicted and shape_* of an exhausted row hold its FALLBACK plan (is_exhausted still says so; g_path, h_path,
 *      tree_path keep their "no plan" values), (iii) every row's final plan is stored in its slot for the next call. */
int pdmpc_closed_loop_reset(pdmpc_handle *h, int32_t n_slots, double half_length, double half_width);
int pdmpc_plan_timestep_closed_loop(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                                    const int32_t *slot, const uint8_t *standstill, pdmpc_batch_out *out);

/* ---- One whole time step from the vehicles' MEASURED STATES in one call: pdmpc_sample_inputs, pdmpc_assemble_obstacles
 *      and pdmpc_plan_timestep_closed_loop chained on the device — the reference trajectories, lanelet boundaries and
 *      obstacle polygons never visit the host; what the host still supplies is what it decides: coupling and priorities
 *      (HighLevelController / PrioritizedController up to :324), as three relations over the rows.
 *      Needs pdmpc_upload_mpa, pdmpc_upload_road, pdmpc_upload_reachable_sets (if any row has parallel predecessors) and
 *      pdmpc_closed_loop_reset.  Outputs as pdmpc_plan_timestep_closed_loop: an exhausted row holds its fallback plan.
 *      The lanelet bounds of a vehicle may have at most 512 points (PDMPC_ERR_CAPACITY). ---- */
typedef struct pdmpc_timestep_states {
    int32_t n;                       /* rows: the vehicles of every scenario of the time step */
    const int32_t *path_id;          /* [n] 0-based reference path of the row (pdmpc_upload_road) */
    const double *x, *y, *yaw;       /* [n] measured pose */
    const double *speed;             /* [n] speed of the current trim; |speed| < 0.01 = the vehicle stands */
    const int32_t *trim;             /* [n] current trim, 1-based */
    const int32_t *succ_ptr, *succ_idx;   /* CSR: coupled rows of lower priority (pdmpc_coupling_in) */
    const int32_t *par_ptr, *par_idx;     /* CSR: coupled rows of higher priority that plan in parallel */
    const int32_t *pred_ptr, *pred_idx;   /* CSR: sequential predecessors (pdmpc_timestep_deps) */
    const int32_t *slot;             /* [n] closed-loop slot of the row (pdmpc_closed_loop_reset) */
    double half_length, half_width;  /* Length/2 + offset, Width/2 + offset */
    double dt_seconds;
    int32_t checker;                 /* PDMPC_CHECKER_* */
} pdmpc_timestep_states;
int pdmpc_plan_timestep_from_states(pdmpc_handle *h, const pdmpc_timestep_states *states, pdmpc_batch_out *out);

/* ---- Time steps with the sampled optimizer (MonteCarloTreeSearch.run_optimizer as the optimizer of
 *      PrioritizedController.plan, DESIGN.md §4.14): pdmpc_plan_timestep, pdmpc_plan_timestep_closed_loop and
 *      pdmpc_plan_timestep_from_states with one warp per sampled search (pdmpc_mcts_plan_batch's kernel) instead of the
 *      graph search.  prm->seed[i] is row i's RandStream seed (time_step + vehicle_index, both 1-based), the same
 *      n_expansions_max for every row.  A row is exhausted when no valid depth-Hp leaf was found or its status is not
 *      PDMPC_OK (PDMPC_ERR_CAPACITY: the roll-outs would read past the Hp * n_expansions_max random numbers); it then
 *      publishes its fallback areas like an exhausted graph search, and its status is reported.  Output fields as
 *      pdmpc_mcts_plan_batch; every one equals level-by-level pdmpc_mcts_plan_batch calls with host-side obstacle
 *      assembly.  The relation checks, the work order, the fallback plans and the closed-loop slots are those of the
 *      graph-search calls.  No node arena; pdmpc_set_variant has no effect and pdmpc_stats.shape reports 1.
 *      Errors (before anything is launched): those of the graph-search call, PDMPC_ERR_BAD_INPUT for n_expansions_max
 *      outside 1..PDMPC_MCTS_MAX_EXPANSIONS, NULL seeds with n > 0 or a branching factor above PDMPC_MCTS_MAX_BRANCH,
 *      PDMPC_ERR_CAPACITY when the sampled tree does not fit in shared memory. ---- */
int pdmpc_mcts_plan_timestep(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                             const pdmpc_mcts_params *prm, pdmpc_batch_out *out);
int pdmpc_mcts_plan_timestep_closed_loop(pdmpc_handle *h, const pdmpc_batch_in *in, const pdmpc_timestep_deps *deps,
                                         const int32_t *slot, const uint8_t *standstill,
                                         const pdmpc_mcts_params *prm, pdmpc_batch_out *out);
int pdmpc_mcts_plan_timestep_from_states(pdmpc_handle *h, const pdmpc_timestep_states *st,
                                         const pdmpc_mcts_params *prm, pdmpc_batch_out *out);

/* ---- Coupling, priorities and computation levels of a time step on the device: what the host decides before
 *      pdmpc_plan_timestep_from_states, for every scenario of the time step in one call (DESIGN.md §4.12).
 *        - coupling (ReachableSetCoupler.m:5-54): rows i, j of one scenario are coupled iff the step-Hp reachable sets of
 *          their current trims (reachable_sets{i, end}, pdmpc_upload_reachable_sets) placed at their poses overlap by more
 *          than 1e-3 (:39-42).  [dev] the overlap is the Sutherland-Hodgman clipping of DESIGN.md §4.12 in FP64 (the
 *          sets are convex), not polyshape intersect; the lanelet clipping of HighLevelController.m:241-246 is not done;
 *        - priorities: PDMPC_PRIORITY_CONSTANT (ConstantPrioritizer.m:6-18, the lower row first) or
 *          PDMPC_PRIORITY_COLORING (ColoringPrioritizer.m:11-153); directed coupling D(i, j) = coupled and prio(i) < prio(j);
 *        - sequential relation seq: the predecessors of row j that stay sequential so that no row sits deeper than
 *          max_num_CLs computation levels (equal to D when max_num_CLs >= the depth); level = kahn(seq), 1-based;
 *        - the three relations of pdmpc_timestep_states: successors = D(i, :), parallel = D(:, i) & ~seq(:, i),
 *          predecessors = seq(:, i); global 0-based rows, ascending within each list. ---- */
#define PDMPC_PRIORITY_CONSTANT 0      /* ConstantPrioritizer.m:6-18 */
#define PDMPC_PRIORITY_COLORING 1      /* ColoringPrioritizer.m:11-153 */
#define PDMPC_COUPLE_MAX_VEHICLES 64   /* rows per scenario */
typedef struct pdmpc_couple_params {
    int32_t n_scenarios;
    const int32_t *scenario_ptr;   /* [n_scenarios+1]: rows of scenario s are [ptr[s], ptr[s+1]), ptr[0] == 0, ptr[n_scenarios] == n */
    int32_t prioritizer;           /* PDMPC_PRIORITY_* */
    int32_t max_num_CLs;           /* >= 1 */
} pdmpc_couple_params;
typedef struct pdmpc_couple_out {  /* caller-owned host buffers; NULL fields are not copied back */
    int32_t *succ_ptr, *succ_idx;  /* [n+1], [idx_capacity]: as pdmpc_timestep_states */
    int32_t *par_ptr, *par_idx;
    int32_t *pred_ptr, *pred_idx;
    int32_t idx_capacity;          /* entries of each *_idx array; PDMPC_ERR_CAPACITY if a relation has more */
    int32_t *level;                /* [n] 1-based computation level */
    double *overlap_area;          /* [sum of n_s^2] per scenario an n_s x n_s row-major matrix; 0.0 on the diagonal */
} pdmpc_couple_out;
/* Needs pdmpc_upload_mpa and pdmpc_upload_reachable_sets (of that automaton; at most 129 points per set).  x, y, yaw,
 * trim: [n] measured pose and current trim (1-based) of every row.  Errors: PDMPC_ERR_BAD_INPUT for a missing or foreign
 * reachable-set table, a trim out of range, a malformed scenario_ptr, a scenario of more than PDMPC_COUPLE_MAX_VEHICLES
 * rows, an unknown prioritizer or max_num_CLs < 1; PDMPC_ERR_CAPACITY when idx_capacity is too small. */
int pdmpc_couple(pdmpc_handle *h, int32_t n, const double *x, const double *y, const double *yaw, const int32_t *trim,
                 const pdmpc_couple_params *prm, pdmpc_couple_out *out);
/* pdmpc_plan_timestep_from_states with the three relations decided by pdmpc_couple first (same call, one small
 * device->host copy of the relations in between): st's succ / par / pred pointers must be NULL (PDMPC_ERR_BAD_INPUT
 * otherwise).  The relations used are returned in `rel` (may be NULL); PDMPC_ERR_CAPACITY, before anything is planned,
 * when they do not fit rel->idx_capacity. */
int pdmpc_plan_timestep_from_states_coupled(pdmpc_handle *h, const pdmpc_timestep_states *st, const pdmpc_couple_params *prm,
                                            pdmpc_couple_out *rel, pdmpc_batch_out *out);

/* ---- Simultaneous prioritizations (PrioritizedExplorativeController, hlc/controller/prioritized/
 *      PrioritizedExplorativeController.m:21-176) for every scenario of the time step in ONE call (DESIGN.md §4.13):
 *      every permutation of the computation levels is planned from the measured states as in
 *      pdmpc_plan_timestep_from_states, the cheapest permutation per weakly connected sub-graph is chosen on the device
 *      and its plans become the vehicles' closed-loop state.
 *        - st: the n base rows (one per vehicle) as for pdmpc_plan_timestep_from_states; st->succ_ptr / succ_idx = the
 *          directed coupling D (coupled rows of lower priority, pdmpc_couple's succ); st->par_* and st->pred_* must be
 *          NULL (they are derived per permutation); base slots distinct.
 *        - permuted relation (:55-78): lev_p(i) = perm_p[level(i) - 1]; an edge i -> j of D with lev_p(i) > lev_p(j) is
 *          reversed.  level(i) < level(j) must hold on every edge of D, so every permuted relation is acyclic.  Per row:
 *          standing successors from the permuted relation's row, sequential predecessors from its column, no parallel
 *          predecessors (the controller has no level cut); fallback plans from the slot of the vehicle (read only).
 *        - cost of a row (compute_solution_cost :94-109): g_path[Hp]; an exhausted row the squared distance of its
 *          fallback trajectory to the reference trajectory, summed in numpy's pairwise order (DESIGN.md §4.13).
 *        - choice (:124-176): per (permutation, sub-graph) the row costs summed in vehicle order from 0.0, rounded
 *          sign(y) * floor(|y| + 0.5) / 1e8 with y = x * 1e8, first minimum over the permutations.
 *        - commit: per vehicle the row of its sub-graph's chosen permutation becomes its slot's state; no other row
 *          touches a slot.  An input error is reported before anything is launched and leaves the slots as they were.
 *      rows_out: rows = sum_s P_s * n_s, row (s, p, v) = sum_{t<s} P_t * n_t + p * n_s + (v - scenario_ptr[s]); outputs as
 *      pdmpc_plan_timestep_closed_loop (an exhausted row holds its fallback plan).
 *      Errors (PDMPC_ERR_BAD_INPUT): malformed scenario_ptr / perm_ptr / perm_val_ptr, P_s < 1, a perm row that is not a
 *      permutation of 1..L_s, a level < 1 or not increasing along an edge of D, an edge across scenarios or repeated,
 *      repeated base slots, relations passed in, a vehicle with more predecessors in some permutation than
 *      PDMPC_TIMESTEP_COLS allows, no pdmpc_closed_loop_reset. ---- */
typedef struct pdmpc_explorative_in {
    int32_t n_scenarios;            /* >= 1 */
    const int32_t *scenario_ptr;    /* [S+1] base rows of scenario s: [ptr[s], ptr[s+1]), ptr[0] == 0, ptr[S] == n */
    const int32_t *level;           /* [n] 1-based computation level of every base row; L_s = max level of scenario s */
    const int32_t *perm_ptr;        /* [S+1] permutations of scenario s: [perm_ptr[s], perm_ptr[s+1]), at least one */
    const int32_t *perm_val_ptr;    /* [S+1] values of scenario s in perm: [perm_val_ptr[s], perm_val_ptr[s+1]), P_s * L_s */
    const int32_t *perm;            /* row-major P_s x L_s per scenario: row p = the new position (1..L_s) of level 1..L_s
                                     * (computation_level_permutations; row 0 of the reference = identity) */
} pdmpc_explorative_in;

typedef struct pdmpc_explorative_out {   /* caller-owned host buffers; NULL fields are not copied back */
    int32_t *belonging;      /* [n] 1-based weakly connected sub-graph of the base row within its scenario */
    int32_t *chosen;         /* [n] 0-based permutation whose plan the base row executes */
    int32_t *applied_row;    /* [n] row of rows_out holding that plan */
    double *row_cost;        /* [rows] cost of every (permutation, vehicle) row, before rounding */
    double *solution_cost;   /* [rows] per scenario a P_s x n_s block; (p, g-1) = rounded sum of sub-graph g; columns >= G_s are 0 */
} pdmpc_explorative_out;

int pdmpc_plan_timestep_explorative(pdmpc_handle *h, const pdmpc_timestep_states *st, const pdmpc_explorative_in *ex,
                                    pdmpc_batch_out *rows_out, pdmpc_explorative_out *eo);

/* Pinned host buffers for callers that want full-rate host<->device copies. */
int pdmpc_host_alloc(void **p, size_t bytes);
int pdmpc_host_free(void *p);

/* Parity/debug aid: re-run the staged batch and record the node ids search
 * `search` pops, in order (the reference's pq.pop() sequence, GraphSearch.m:55). */
int pdmpc_trace_staged(pdmpc_handle *h, int32_t search, int64_t *ids, int64_t cap, int64_t *n_out);

/* The CUDA stream the kernels are launched on (cudaStream_t as void*), so a
 * host harness can record its own events on it. */
void *pdmpc_stream(pdmpc_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* PDMPC_B200_H */
