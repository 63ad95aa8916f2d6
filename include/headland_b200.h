/*
 * headland_b200.h -- C ABI of the B200 (sm_100a) warm-start search library.
 *
 * The reference (AgRoboticsResearch/headland_trajectory_planning) is pure Python and
 * has no FFI layer; its boundary for this path is a set of duck-typed Python call
 * signatures (SURVEY.md section 8b).  Each entry point below names the reference
 * call it replaces (paths relative to the reference checkout).  The Python mirror
 * classes in headland_trajectory_planning_b200/ bind these with ctypes; a
 * reference maintainer binds them the same way (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; hl_last_error()
 *     returns a thread-local message for the last failure;
 *   - pointers named d_* are DEVICE pointers, h_* are HOST pointers; the caller
 *     owns every buffer (no ownership transfer);
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream);
 *     calls are asynchronous with respect to the host unless the name ends in _host;
 *   - no global state besides the opaque hl_ctx (one per device).  Every entry point selects the context's
 *     device itself and REJECTS (non-zero + hl_last_error) an environment batch of another device / context and
 *     a probed d_* argument that is host memory or lives on another device -- it never launches on the wrong GPU;
 *   - entry points may be called from any host thread.  Searches (hl_hybrid_astar_batch) share one per-context
 *     workspace: calls on different streams/threads of one context are serialised on the device (event wait),
 *     everything else is independent per stream;
 *   - there is NO CPU fallback: without a CUDA device hl_ctx_create fails.
 */
#ifndef HEADLAND_B200_H
#define HEADLAND_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HL_ABI_VERSION 5

/* ---- limits (compile-time capacities of the kernels) ---------------------- */
#define HL_MAX_PRIMS        16   /* motion primitives per expansion (King: 14, Pawn: 8) */
#define HL_MAX_ROLLOUT      16   /* poses of one primitive rollout (round(L/res)+1)      */
#define HL_CAPSULE_VERTS    66   /* GEOS round-cap buffer of a 2-point line, quad_segs=16 */
#define HL_RS_CANDIDATES    46   /* Reeds-Shepp candidate words, reeds_shepp.py:565-582   */
#define HL_RS_MAX_SEGS       5

/* ---- check flags (orchard_geometry_environment.py:423-425, hybrid_a_star_search.py:412-427) */
#define HL_CHECK_OBSTACLES  1u   /* body vs obstacle + tree-row polygons (always on in the reference) */
#define HL_CHECK_BOUNDARY   2u   /* boundary_check=True: footprint inside field_range_poly */
#define HL_CHECK_AUX        4u   /* aux_check=True: implement rectangles at poses 0,2,4,.. */
#define HL_CHECK_LANE       8u   /* ReferenceLineHeuristic.check_path_feasibility (body inside lane) */

/* ---- per-scenario status (hybrid_a_star_search.py:516-555) ----------------- */
enum {
    HL_STATUS_OK                 = 0,  /* goal reached (RS shot free, or within tolerance) */
    HL_STATUS_START_GOAL_BLOCKED = 1,  /* :516-519 -> ([],[],[],[],[],0)                    */
    HL_STATUS_OPEN_EMPTY         = 2,  /* :537-539 "No solution is available"               */
    HL_STATUS_MAX_NODES          = 3,  /* :526-529 "drop the planner"                       */
    HL_STATUS_CAPACITY           = 4,  /* device workspace exhausted (never silent)         */
    HL_STATUS_RS_ASSERT          = 5   /* reeds_shepp.py:84 `assert path.L >= 0.01` would raise */
};

typedef struct hl_ctx hl_ctx;
typedef struct hl_env_batch hl_env_batch;

/* One environment + vehicle + guide, host side.  Built by the Python mirror of
 * OrchardGeometryEnvironment.__init__ (orchard_geometry_environment.py:15-32,
 * 277-353), CarModel.get_car_poly (car_model.py:75-162) and
 * ReferenceLineHeuristic.get_guide_line / create_segment_lengths
 * (reference_line_heuristic.py:50-96).  All polygons counter-clockwise, not closed. */
typedef struct {
    int32_t n_obs;           /* convex obstacle quads (obstacle squares + tree-row rectangles) */
    const double* obs_xy;    /* [n_obs][4][2]                                              */
    int32_t n_field;         /* field_range_poly vertices (simple polygon, may be non-convex) */
    const double* field_xy;  /* [n_field][2]                                               */
    int32_t n_seg;           /* guide segments = lane capsules (0 = no lane / heuristic)    */
    const double* seg_xy;    /* [n_seg][2][2] waypoint pairs                               */
    const double* seg_poly;  /* [n_seg][HL_CAPSULE_VERTS][2] capsule polygons               */
    const double* seg_len;   /* [n_seg] search length per segment (1.5 / 1.0)               */
    int32_t n_crit;          /* vertices of the lane union's boundary (pairwise crossings)  */
    const double* crit_xy;   /* [n_crit][2]                                                */
    int32_t n_guide;         /* guide polyline samples                                     */
    const double* guide;     /* [n_guide][4] x, y, yaw, s                                  */
    double default_search_length;  /* reference_line_heuristic.py:24 (1.5)                 */
    double body_ext[4];      /* body rectangle in base_link: x0, x1, y0, y1                 */
    int32_t n_aux;           /* implement rectangles (car_model.py:146-162)                 */
    const double* aux_ext;   /* [n_aux][4]                                                 */
} HlEnvHost;

/* Search parameters shared by a batch (HybridAStarSearch.__init__ + class constants,
 * hybrid_a_star_search.py:28-74; primitive table :331-354 computed on the host with
 * numpy so that arange/tan rounding is the reference's own). */
typedef struct {
    double plan_resolution;            /* :47  */
    double yaw_resolution;             /* :46  */
    double maxc;                       /* car_model.curvature, car_model.py:34 */
    double max_steer;                  /* car_model.MAX_STEER                  */
    double wheel_base;
    int32_t n_prims;
    double prim_steer[HL_MAX_PRIMS];   /* motion_steers[:,0]                    */
    double prim_dir[HL_MAX_PRIMS];     /* motion_steers[:,1] (+1/-1)            */
    double prim_yaw_step[HL_MAX_PRIMS];/* dir*res/WB*tan(steer), :370-375       */
    double prim_curv[HL_MAX_PRIMS];    /* np.tan(steer)/WB, :402                */
    double prim_steer_eff[HL_MAX_PRIMS];/* math.atan(curv*WB), :322             */
    int32_t steps_default;             /* informational only: the kernels take the per-environment search length from
                                          HlEnvHost.default_search_length and HlEnvHost.seg_len (the heuristic's values,
                                          reference_line_heuristic.py:120-131) and round it per node like :369 */
    int32_t steps_large;               /* informational only, see steps_default */
    double steer_cost, delta_steer_cost, direction_change_cost, reverse_cost, hybrid_cost;
    double min_length_to_goal;         /* :36 */
    int32_t max_nodes;                 /* hybrid_a_star_search(max_nodes=..), :497 */
    int32_t max_path_poses;            /* capacity of one scenario's output path */
    int32_t motion_type;               /* 0 = "King" (Reeds-Shepp goal extension, :232-287), 1 = "Pawn" (forward primitives
                                          :331-341, Dubins goal extension :184-230; pydubins parity unpinned) */
    int32_t dubins_capacity;           /* Pawn: samples / course rows the Dubins scratch of one scenario holds (0 = 2048) */
} HlSearchParams;

/* One search problem: HybridAStarSearch(start_pose, goal_pose, env, car, heuristic). */
typedef struct {
    int32_t env_id;
    int32_t reserved;
    double start[3];
    double goal[3];
} HlScenario;

/* Fixed-stride result record (one per scenario). */
typedef struct {
    int32_t status;        /* HL_STATUS_*                                            */
    int32_t counter;       /* the reference's `counter` (expansions incl. the last)   */
    int32_t n_expanded;    /* popped nodes written to expanded_keys                   */
    int32_t arrival;       /* 0 none, 1 Reeds-Shepp shot, 2 tolerance arrival (:483-493) */
    int32_t path_len;      /* poses in this scenario's slice of the path buffers      */
    int32_t rs_word;       /* candidate row (0..45) of the accepted shot, else -1     */
    int64_t path_offset;   /* first pose of the slice                                 */
    double  goal_cost;     /* cost of the goal node                                   */
    int64_t n_pose_checks; /* footprint checks executed (primitives + shots)          */
    int64_t n_exact;       /* of which escalated to the float64 predicates            */
    int64_t keys_offset;   /* first row of this scenario's slice of the pooled expanded-key buffer */
    int64_t cycles;        /* SM clock cycles this scenario occupied its CTA (the reference prints
                              `hybrid search time`, hybrid_a_star_search.py:603)       */
    int64_t n_pose_checks_ref; /* ALGORITHMIC pose checks: what the reference tests for the same search =
                              sum over tried words of their sampled poses (:273-276) + n_prims*(n+1) per
                              expansion (:412-427); n_pose_checks <= this thanks to early exits          */
} HlPlanResult;

/* Reeds-Shepp word record: hl_rs_all_paths output, one row per accepted word. */
typedef struct {
    int32_t cand;          /* row of the 46-candidate table, evaluation order          */
    int32_t n_seg;
    int32_t npts;          /* samples generate_local_course would emit                 */
    int32_t collide;       /* filled by hl_rs_all_paths when an environment is given   */
    double  L;             /* total length (metres)                                    */
    double  cost;          /* calculate_reeds_shepp_path_cost with node cost 0         */
    double  len[HL_RS_MAX_SEGS];  /* signed segment lengths (metres) = PATH.lengths    */
    double  nlen[HL_RS_MAX_SEGS]; /* the same lengths x maxc (normalised), as sampled  */
} HlRsWord;

/* ---- context ---------------------------------------------------------------- */
const char* hl_last_error(void);
int hl_abi_version(void);
int hl_ctx_create(hl_ctx** out, int device);
void hl_ctx_destroy(hl_ctx* ctx);
int hl_ctx_sm_count(const hl_ctx* ctx);
int hl_ctx_device(const hl_ctx* ctx);              /* CUDA device ordinal of the context (-1 for NULL)          */
/* Search-kernel variant for A/B runs (results are identical): 0 = two warps per scenario with the analytic shot
 * decoupled (default), 1 = one warp per scenario, 2 = level-synchronous graph.  The environment variable
 * HL_ASTAR_VARIANT (spec|warp|level) is read once, at hl_ctx_create. */
int hl_ctx_set_astar_variant(hl_ctx* ctx, int variant);

/* ---- environments ----------------------------------------------------------- */
/* Replaces the geometry that OrchardGeometryEnvironment / CarModel /
 * ReferenceLineHeuristic hold as shapely objects.  Host -> device, synchronous. */
int hl_env_upload(hl_ctx* ctx, const HlEnvHost* h_envs, int32_t n_env, hl_env_batch** out);
void hl_env_free(hl_env_batch* envs);
int32_t hl_env_count(const hl_env_batch* envs);
int hl_env_device(const hl_env_batch* envs);       /* device the batch was uploaded to                           */

/* ---- K1 footprint collision --------------------------------------------------
 * Replaces OrchardGeometryEnvironment.check_path_feasibility
 * (orchard_geometry_environment.py:423-458) [+ CarModel.get_path_poly, car_model.py:39-73]
 * and, with HL_CHECK_LANE, ReferenceLineHeuristic.check_path_feasibility
 * (reference_line_heuristic.py:105-118), per pose.
 *   d_env_id   [N] int32 environment of each pose (NULL = all poses use env 0)
 *   d_poses    [N][3] float64 x, y, yaw
 *   d_path_id  [N] int32 path each pose belongs to, or NULL; aux rectangles are
 *              tested at every 2nd pose OF ITS PATH (car_model.py:58), so with
 *              HL_CHECK_AUX the caller passes d_pose_idx [N] = index within the path
 *   d_out      [N] uint8, 1 = infeasible pose
 *   d_n_exact  optional device counter (int64) of float64 escalations, or NULL      */
int hl_collision_check(hl_ctx* ctx, const hl_env_batch* envs, const int32_t* d_env_id,
                       const double* d_poses, const int32_t* d_pose_idx, int64_t n,
                       uint32_t flags, uint8_t* d_out, unsigned long long* d_n_exact,
                       void* stream);

/* Per-path reduction: d_path_bad[p] = OR of d_pose_bad over [d_path_start[p], d_path_start[p+1]).
 * This is the boolean check_path_feasibility returns (negated). */
int hl_path_reduce(hl_ctx* ctx, const uint8_t* d_pose_bad, const int64_t* d_path_start,
                   int64_t n_paths, uint8_t* d_path_bad, void* stream);

/* ---- K5 Y-type parking candidates (SURVEY.md 8(f) rank 1) ------------------------
 * Replaces the loop body of search_y_type_parking_path
 * (path_planner/headland_path_planning.py:405-427): get_y_type_parking_path (:488-516, two
 * calculate_motion_path rollouts :455-485) + get_path_in_odom (:519-527) for EVERY candidate
 * of one or many sweeps in one launch.
 *   d_cand    [n][8] float64: backward_length, forward_length, backward_steer (signed),
 *             forward_steer (signed), end_x, end_y, end_yaw, wheel_base
 *   d_offsets [n+1] int64: first pose of each candidate in d_poses;
 *             offsets[i+1]-offsets[i] must be round(bl/step) + round(fl/step) + 2
 *             (Python round); a mismatching candidate is written as NaN poses (= infeasible)
 *   d_poses   [offsets[n]][3] float64 out: x, y, yaw in the odom frame, in the reference's row
 *             order (forward arc reversed, then backward arc reversed, ending on the end pose)
 * Feed d_poses to hl_collision_check and d_offsets to hl_path_reduce; the first feasible
 * candidate in loop order is the reference's result. */
int hl_ypark_paths(hl_ctx* ctx, const double* d_cand, const int64_t* d_offsets, int64_t n, double step,
                   double* d_poses, void* stream);

/* Single-arc rollouts of CarModel.calculate_motion_path (path_planner/car_model.py:202-234), the candidate
 * generator of get_offset_pose (path_planner/safety_forward_path_plan.py:248-283; SURVEY.md 8(f) rank 2).
 *   d_cand    [n][8] float64: init_x, init_y, init_yaw, steer (signed), direction (+1/-1),
 *             search_length (= delta_yaw / curvature), wheel_base, unused
 *   d_offsets [n+1] int64; offsets[i+1]-offsets[i] must be round(search_length/step) + 1
 *   d_poses   out: the init pose followed by the arc poses (NaN rows on a count mismatch)             */
int hl_arc_paths(hl_ctx* ctx, const double* d_cand, const int64_t* d_offsets, int64_t n, double step,
                 double* d_poses, void* stream);

/* ---- K8 warm-start path -> OBCA initial guess (SURVEY.md 8(f) rank 4) -------------
 * Replaces get_init_ref_path (obca_py/util.py:62-113) + calc_spline_course / Spline2D
 * (path_planner/utils/cubic_spline.py:19-112) for many paths at once.  Input = the pooled path
 * arrays of hl_hybrid_astar_batch (x, y, direction) with per-path offsets.
 *   hl_ref_path_count: d_counts[p] = rows of path p's trajectory (0 and d_status[p] = 1 when a
 *                      direction piece has fewer than 2 distinct poses -- the reference raises there);
 *                      the caller turns the counts into d_out_offsets [n+1] (exclusive prefix sum)
 *   hl_ref_path_fill:  d_out [offsets[n]][5] float64 rows (x, y, v, yaw, steer), yaw unwrapped along
 *                      each path (process_angle, util.py:16-44); d_workspace = 8 doubles per INPUT pose */
int hl_ref_path_count(hl_ctx* ctx, const double* d_x, const double* d_y, const int8_t* d_dir,
                      const int64_t* d_in_offsets, int64_t n_paths, double ds, int64_t* d_counts,
                      int32_t* d_status, void* stream);
int hl_ref_path_fill(hl_ctx* ctx, const double* d_x, const double* d_y, const int8_t* d_dir,
                     const int64_t* d_in_offsets, const int64_t* d_out_offsets, const int32_t* d_status,
                     int64_t n_paths, double wheel_base, double desired_v, double ds, double* d_workspace,
                     double* d_out, void* stream);

/* ---- K9 Dubins paths + spline course (SURVEY.md 8(f) ranks 2-3) ---------------------------
 * Replaces, for MANY pose pairs at once, get_dubins_path (path_planner/utils/navigation_utils.py:206-215:
 * dubins.shortest_path(q0, q1, rho) + sample_many(step)) followed by calc_spline_course(x, y, ds)
 * (path_planner/utils/cubic_spline.py:92-112) = get_dubins_path_full (path_planner/safety_forward_path_plan.py:286-297)
 * and, with append_goal = 1, HybridAStarSearch.get_dubins_path (path_planner/hybrid_a_star_search.py:289-304).
 * pydubins is un-vendored and un-pinned (requirements.txt:14): the published dubins.c algorithm is restated,
 * parity unpinned.
 *   hl_dubins_count: d_slots[p] = workspace slots of pair p (samples + 1, 0 = no path), d_word[p] = 0..5
 *                    (LSL LSR RSL RSR RLR LRL), d_length[p] = path length; the caller turns d_slots into
 *                    d_slot_offsets [n+1] (exclusive prefix sum) and provides 9 doubles per slot of workspace
 *   hl_dubins_knots: samples every path, builds the spline knots in the workspace; d_n_knots[p] (0 = a spline
 *                    cannot be built: the reference raises), d_n_rows[p] = rows of the course
 *   hl_dubins_fill:  d_out [row_offsets[n]][4] float64 rows (x, y, yaw, curvature)                             */
int hl_dubins_count(hl_ctx* ctx, const double* d_pairs, int64_t n, double rho, double step, double ds,
                    int32_t append_goal, int64_t* d_slots, int32_t* d_word, double* d_length, void* stream);
int hl_dubins_knots(hl_ctx* ctx, const double* d_pairs, int64_t n, double rho, double step, double ds,
                    int32_t append_goal, const int64_t* d_slot_offsets, double* d_workspace,
                    int32_t* d_n_knots, int64_t* d_n_rows, double* d_samples /* optional [slots][3]: the raw
                    sample_many configurations (x, y, yaw) of pair p at slot_offsets[p] .. +slots[p]-1 */, void* stream);
int hl_dubins_fill(hl_ctx* ctx, int64_t n, double ds, const int64_t* d_slot_offsets, const int64_t* d_row_offsets,
                   const int32_t* d_n_knots, double* d_workspace, double* d_out, void* stream);

/* ---- K10 distance of a swept path to the field boundary (SURVEY.md 8(f) rank 2) -----------------
 * Replaces OrchardGeometryEnvironment.get_min_distance_to_boundary (path_planner/orchard_geometry_environment.py:
 * 393-412): smallest signed distance (negative outside the field) from the exterior vertices of the swept footprint
 * unions (body at every pose; with_aux: every implement rectangle at every 2nd pose, car_model.py:39-73) to the
 * ring of field_range_poly.  One value per path; GEOS unavailable, parity unpinned.
 *   d_env_id [n_paths] or NULL; d_poses pooled [.,3]; d_path_start [n_paths+1]; d_out [n_paths] float64          */
int hl_min_boundary_distance(hl_ctx* ctx, const hl_env_batch* envs, const int32_t* d_env_id, const double* d_poses,
                             const int64_t* d_path_start, int64_t n_paths, int32_t with_aux, double* d_out, void* stream);

/* ---- K11 corridor test (SURVEY.md 8(f) rank 3) ---------------------------------------------------
 * Replaces the per-word test of classic_circle_back_turning_path (path_planner/safety_forward_path_plan.py:811-822):
 * LineString(xy).buffer(radius, cap_style=flat, join_style=round) intersects the obstacle / tree-row polygons.
 *   d_points pooled [.,2] float64 polyline vertices; d_line_start [n_lines+1]; d_out [n_lines] uint8 (1 = meets)  */
int hl_corridor_hits(hl_ctx* ctx, const hl_env_batch* envs, const int32_t* d_env_id, const double* d_points,
                     const int64_t* d_line_start, int64_t n_lines, double radius, uint8_t* d_out, void* stream);

/* ---- K2/K3 Reeds-Shepp --------------------------------------------------------
 * Replaces reeds_shepp.calc_all_paths (path_planner/utils/reeds_shepp.py:39-65):
 * generate_path + set_path dedup (:565-582, :68-87) and the sample count of
 * generate_local_course (:471-530).  If envs != NULL every word is also sampled and
 * collision-checked (hybrid_a_star_search.py:273-276) with `flags`.
 *   d_start_goal [N][6] float64 (sx,sy,syaw,gx,gy,gyaw)
 *   d_env_id     [N] or NULL
 *   d_words      [N][HL_RS_CANDIDATES] HlRsWord, first d_count[i] rows valid, reference order
 *   d_count      [N] int32 (-1 = the reference would raise at reeds_shepp.py:84)
 *   d_order      [N][HL_RS_CANDIDATES] int32: heapdict pop order of the rows by `cost`
 *                (hybrid_a_star_search.py:265-271), or NULL                             */
int hl_rs_all_paths(hl_ctx* ctx, const hl_env_batch* envs, const int32_t* d_env_id,
                    const double* d_start_goal, int64_t n, double maxc, double step,
                    double max_steer, uint32_t flags, HlRsWord* d_words, int32_t* d_count,
                    int32_t* d_order, void* stream);

/* Sample one word per request (generate_local_course + world transform,
 * reeds_shepp.py:46-63, 471-562).
 *   d_start [M][3]; d_words [M] (len/n_seg/cand used); d_offset [M+1] int64 output slices
 *   (from npts); outputs x,y,yaw,cs float64 and dir int8 of total length d_offset[M]. */
int hl_rs_sample(hl_ctx* ctx, const double* d_start, const HlRsWord* d_words, int64_t m,
                 double maxc, double step, const int64_t* d_offset, double* d_x, double* d_y,
                 double* d_yaw, double* d_cs, int8_t* d_dir, void* stream);

/* ---- K4 batched Hybrid A* -----------------------------------------------------
 * Replaces HybridAStarSearch(...).hybrid_a_star_search(max_nodes)
 * (path_planner/hybrid_a_star_search.py:497-607), King mode, one CTA per scenario.
 *   d_scen          [B] HlScenario
 *   d_results       [B] HlPlanResult
 *   d_expanded_keys pooled [keys_capacity][3] int32: popped grid indices in pop order, one slice per
 *                   scenario (HlPlanResult.keys_offset, n_expanded); keys_capacity = B*(max_nodes+1) always fits
 *   d_keys_cursor   device int64 bump allocator for that pool, zeroed by the callee
 *   d_path_*        pooled output path (x,y,yaw,k float64, dir int8), capacity
 *                   path_capacity poses in total; slices via HlPlanResult.path_offset
 *   d_path_cursor   device int64 bump allocator, zeroed by the callee                 */
int hl_hybrid_astar_batch(hl_ctx* ctx, const hl_env_batch* envs, const HlScenario* d_scen,
                          int32_t n_scen, const HlSearchParams* h_params,
                          HlPlanResult* d_results, int32_t* d_expanded_keys, int64_t keys_capacity,
                          unsigned long long* d_keys_cursor, double* d_path_x, double* d_path_y, double* d_path_yaw,
                          double* d_path_k, int8_t* d_path_dir, int64_t path_capacity,
                          unsigned long long* d_path_cursor, void* stream);
/* Bytes of scratch the search keeps per resident CTA, and how many CTAs it launches
 * (for capacity planning / reporting). */
int64_t hl_hybrid_astar_workspace_bytes(const hl_ctx* ctx, const HlSearchParams* h_params);
/* Phase timers of the search kernel (thread-0 cycles between barriers, summed over all scenarios since
 * the last reset) -- the device analogue of the reference's three accumulating timers
 * (hybrid_a_star_search.py:91-94).  Order: pop, rs_candidates, rs_select, rs_plan, rs_sample, arrival,
 * rollout, filter, exact, cost_heuristic, merge, setup, output. */
#define HL_ASTAR_N_PHASES 13
int hl_astar_phase_cycles(hl_ctx* ctx, uint64_t* h_out, int32_t n, int32_t reset);

/* ---- K6 grid distance field ---------------------------------------------------
 * Replaces holonomic_costs_with_obstacles (path_planner/utils/a_star_utils.py:75-142), the reference's index
 * wrap-around included (:49-64: validity is abs(index) < dim and the arrays are indexed with Python's negative
 * indices, so on a map with free border cells the search continues onto aliased cells and a cell reports the cost
 * of its last-closed alias -- e.g. 11.31 at the goal of a free 8 x 8 grid).  Maps whose border is occupied take
 * the plain tiled wavefront; any other map runs the same wavefront on the (2W-1) x (2H-1) extended grid plus the
 * closing-order pass (csrc/hl_grid.cu).  Results are bit-identical to the reference in float64.
 *   d_occ [W][H] uint8 (non-zero = occupied), row-major like obstacles[i][j]
 *   d_out [W][H] float64, +inf where unreachable
 *   motion_type 0 = King (8 moves, :8-21), 1 = Pawn (5 moves, :24-34)
 *   h_sweeps optional host int: relaxation launches used.  Synchronises the stream.                    */
int hl_distance_field(hl_ctx* ctx, const uint8_t* d_occ, int32_t w, int32_t h, int32_t gi,
                      int32_t gj, int32_t motion_type, double* d_out, int32_t* h_sweeps,
                      void* stream);

/* One field of a batch: a [w][h] occupancy grid (row-major, non-zero = occupied, like hl_distance_field) and a goal cell. */
typedef struct {
    int64_t occ_offset;   /* first byte of this field's grid in d_occ; several fields may share one grid        */
    int64_t out_offset;   /* first element of this field's [w][h] float64 result in d_out; slices must not overlap */
    int32_t w, h;
    int32_t gi, gj;       /* goal cell, 0 <= gi < w, 0 <= gj < h                                                  */
} HlGridField;

/* Distance fields of n_fields (grid, goal) pairs in one tiled wavefront: every relaxation launch serves all fields, so
 * a batch costs about the depth of its deepest field rather than the sum.  Each output slice is bit-identical to what
 * hl_distance_field returns for that grid and goal (wrap-around included).  motion_type is shared by the batch.
 *   h_fields  [n_fields] HOST array; checked before anything launches (bounds against occ_bytes / out_elems,
 *             overlapping output slices, goals, sizes): a failure names the field index in hl_last_error
 *   h_sweeps  optional host int: relaxation launches used (shared by the batch).  n_fields == 0 launches nothing.
 *   Synchronises the stream.                                                                              */
int hl_distance_field_batch(hl_ctx* ctx, const uint8_t* d_occ, int64_t occ_bytes,
                            const HlGridField* h_fields, int32_t n_fields, int32_t motion_type,
                            double* d_out, int64_t out_elems, int32_t* h_sweeps, void* stream);

/* ---- K7 occupancy-grid footprint ---------------------------------------------
 * The grid-based footprint check the reference intended
 * (orchard_geometry_environment.py:8,35-43,460-461; grid layout of
 * occupancy_grid_utils.py:70-101: cell (i,j) covers [i*res,(i+1)*res) x [j*res,(j+1)*res)).
 * No reference implementation exists (parity unpinned): a pose is infeasible iff the
 * closed body rectangle (float64 corners (c*lx - s*ly) + x, (s*lx + c*ly) + y, no fused
 * multiply-add) meets the closed square [fl(i*res), fl((i+1)*res)] x [fl(j*res), fl((j+1)*res)]
 * of some occupied cell (i, j); touching counts.  A pose with a NaN or infinite x, y or yaw
 * is infeasible (out = 1) whatever the grid holds.
 *   d_occ_bits  bit-packed grid, bit (i*H + j); res metres per cell                   */
int hl_grid_pack(hl_ctx* ctx, const uint8_t* d_occ, int32_t w, int32_t h, uint32_t* d_bits,
                 void* stream);
int hl_grid_footprint_check(hl_ctx* ctx, const uint32_t* d_occ_bits, int32_t w, int32_t h,
                            double res, const double* d_poses, int64_t n,
                            const double body_ext[4], uint8_t* d_out, void* stream);
/* The same check on a grid whose cell (0, 0) has the global index (i0, j0): cell (i, j) is the closed square
 * [fl((i0+i)*res), fl((i0+i+1)*res)] x [fl((j0+j)*res), fl((j0+j+1)*res)], so a grid may cover negative coordinates
 * (hl_env_rasterize's windows).  hl_grid_footprint_check is this call with i0 = j0 = 0.  Rejects w or h below 1,
 * i0 + w or j0 + h beyond int32, res not finite or not positive, and grid edges that are not finite.             */
int hl_grid_footprint_check_at(hl_ctx* ctx, const uint32_t* d_occ_bits, int32_t w, int32_t h, int32_t i0, int32_t j0,
                               double res, const double* d_poses, int64_t n, const double body_ext[4],
                               uint8_t* d_out, void* stream);

/* ---- K12 occupancy grids from environment geometry ------------------------------------------------
 * Rasterises the obstacle / tree-row quads and the field polygon of an environment batch into [w][h] uint8 grids
 * (byte i*h + j, 1 = occupied, 0 = free: hl_distance_field's layout; hl_grid_pack makes K7's bits), many grids of
 * many environments in one launch.  No reference implementation exists (the reference's grid path is commented
 * out, orchard_geometry_environment.py:8,35-43,460-461): the grids are defined by the closed-set rule below.
 *
 * Cell rule.  Let S be the closed square of cell (i, j) of a grid, with edges the float64 products
 * fl((i0+i)*res), fl((i0+i+1)*res), fl((j0+j)*res), fl((j0+j+1)*res) (exactly K7's edges).
 *   - HL_CHECK_OBSTACLES: occupied iff S meets some closed obstacle or tree-row quad;
 *   - HL_CHECK_BOUNDARY:  occupied iff S is not contained in the closed field polygon (GEOS contains: touching the
 *                         ring from inside is still contained; an environment without field vertices is all occupied);
 *   - both flags: occupied if either test fires.
 * Both tests are K1's float64 predicates applied to the identity pose (x, y, cos, sin) = (0, 0, 1, 0) with the
 * cell's edges as the rectangle: under that pose the corners and pose-frame coordinates reproduce the edges bit
 * for bit, so every byte is the boolean hl_collision_check's float64 path gives for that rectangle.  A float32
 * filter with K1's band decides the cells clear of the band; the rest go to those predicates (d_n_exact counts them).
 *   h_grids    [n_grids] HOST array; checked before anything launches (a failure names the grid index): env_id
 *              outside the batch, w or h below 1, i0 + w or j0 + h beyond int32, grid edges that are not finite,
 *              output slices outside out_elems or overlapping.  n_grids == 0 launches nothing.
 *   res        metres per cell, finite and positive
 *   flags      HL_CHECK_OBSTACLES and / or HL_CHECK_BOUNDARY, nothing else
 *   d_n_exact  optional device counter (int64) of cells decided by the float64 predicates, or NULL           */
typedef struct {
    int64_t out_offset;   /* first byte of this grid's [w][h] uint8 slice in d_out; slices must not overlap */
    int32_t env_id;       /* environment of the batch                                                      */
    int32_t w, h;         /* cells                                                                        */
    int32_t i0, j0;       /* global index of cell (0, 0)                                                  */
} HlRasterGrid;

int hl_env_rasterize(hl_ctx* ctx, const hl_env_batch* envs, const HlRasterGrid* h_grids, int32_t n_grids,
                     double res, uint32_t flags, uint8_t* d_out, int64_t out_elems,
                     unsigned long long* d_n_exact, void* stream);

/* ---- micro-benchmarks used for roofline denominators ------------------------- */
/* Measured FP32 FMA peak of this device in TFLOP/s (dependent-chain-free FFMA loop). */
int hl_measure_fp32_peak(hl_ctx* ctx, double* h_tflops);

#ifdef __cplusplus
}
#endif
#endif /* HEADLAND_B200_H */
