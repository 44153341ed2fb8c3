/* bpgeo.h -- C ABI of libbpgeo.so, the B200-native geometry core for BoundPlanner.
 *
 * The reference (Thieso/BoundPlanner) is pure Python and has no FFI of its own:
 * the seam is the Python object boundary between the planner / BoundMPC and
 *   - ConvexSetFinder            bound_planner/BoundPlanner/ConvexSetFinder.py:102-766
 *   - BoundPlanner.set_intersection / add_edges
 *                                bound_planner/BoundPlanner/BoundPlanner.py:774-798
 *   - RobotModel.fk*             bound_planner/RobotModel/RobotModel.py:146-231
 * Every entry point below names the reference call it replaces.  The Python
 * stubs that bind it are in boundplanner_b200/_lib.py; the one-line changes a
 * reference maintainer would make are in INTEGRATION.md.
 *
 * Conventions
 *   - fp64 everywhere, row-major.
 *   - "dev" pointers are CUDA device pointers owned by the caller; "host"
 *     pointers are ordinary host memory.  The library owns only bp_scene.
 *   - All kernels are enqueued on `stream` (a cudaStream_t passed as void*);
 *     no hidden synchronisation, no hidden allocation: scratch comes from the
 *     caller through (workspace, workspace_bytes), sized by the *_workspace_bytes
 *     query.
 *   - Return value: 0 on success, non-zero on error; bp_last_error_string()
 *     describes the last error of the calling thread.
 *   - Per-item status codes (int32, one per seed / segment):
 *       BP_OK 0, BP_ELLIPSE_VIOLATION 1 (ConvexSetFinder.py:433-438 RuntimeError),
 *       BP_ROW_OVERFLOW 2 (more than m_max rows), BP_MVIE_NO_INTERIOR 3,
 *       BP_MVIE_NOT_CONVERGED 4, BP_ROW_CAP 5 (more rows than row_cap in an IRIS pass),
 *       BP_NOT_A_POLYTOPE 6 (bp_polytope_vertices: unbounded / empty set).
 *   - There is NO CPU fallback: every compute entry point needs a CUDA device.
 */
#ifndef BPGEO_H
#define BPGEO_H

#ifdef __cplusplus
extern "C" {
#endif

#define BPGEO_ABI_VERSION 7
#define BP_MAX_ROWS 48 /* hard cap on rows per convex set (reference MVIE cap: 20, quirk Q5) */

typedef struct bp_scene bp_scene;

int bpgeo_abi_version(void);
const char* bp_last_error_string(void);

/* ---- obstacle scene ---------------------------------------------------------
 * Replaces BoundPlanner.make_box / add_obstacle_reps (BoundPlanner.py:126-152):
 * box k = [lbx,lby,lbz,ubx,uby,ubz]; the library stores lb - inflate, ub + inflate
 * (b += obs_size_increase, :141) as SoA columns in HBM.  boxes_host: [n,6]. */
int bp_scene_create(const double* boxes_host, int n, double inflate, bp_scene** out);
/* A batch of scenes stored back to back (one per planning query, BASELINE config C3): scene k owns boxes
 * [offsets[k], offsets[k+1]) of boxes_host.  Use with the *_ms entry points, which take the scene index of
 * every seed / segment. */
int bp_scene_create_batch(const double* boxes_host, const int* offsets_host /*[n_scenes+1]*/, int n_scenes,
                          double inflate, bp_scene** out);
/* General convex polytope obstacles (util_functions.compute_polytope_vertices / the obs_sets + obs_points_sets
 * a caller hands to ConvexSetFinder): rows_host [n,15,4] = (a0,a1,a2,b) per row, real rows first, then zero rows
 * with b = 10 (normalize_set_size padding, util_functions.py:119-133); nrows_host [n]; verts_host [n,vmax,3] with
 * nverts_host [n] vertices each.  Rows are taken as given (already inflated).  Supported by bp_closest_points(_line),
 * bp_polyhedron, bp_build_sets_point, bp_build_sets_around_line, bp_build_sets_line and bp_sample_filter; at most
 * 16384 obstacles per scene (bp_build_sets_around_line: 8192).  While
 * the closest points of all obstacles fit in shared memory (3072 obstacles) they are cached there; beyond that the
 * winner of every pick is re-solved (same bits). */
int bp_scene_create_polytopes(const double* rows_host, const int* nrows_host, const double* verts_host,
                              const int* nverts_host, int n, int vmax, bp_scene** out);
/* A batch of polytope scenes stored back to back (scene k owns obstacles [offsets[k], offsets[k+1]) of the four
 * arrays); use with the *_ms entry points like bp_scene_create_batch. */
int bp_scene_create_polytopes_batch(const double* rows_host, const int* nrows_host, const double* verts_host,
                                    const int* nverts_host, const int* offsets_host /*[n_scenes+1]*/, int n_scenes,
                                    int vmax, bp_scene** out);
int bp_scene_update(bp_scene* scene, const double* boxes_host, int n, double inflate, void* stream);
/* Rewrite a resident scene batch in place with new obstacles (ABI 5; an MPC loop whose obstacles move): the inputs of
 * the matching *_create_*batch, n_scenes equal to the batch's, the per-scene obstacle counts free to change (boxes:
 * down to 0; polytopes: at least one obstacle in all).  One host-to-device copy of the packed inputs through a staging
 * buffer owned by the scene (pinned host + device, grown on demand), a short kernel chain on `stream` that writes the
 * same bits as a freshly created batch, and a synchronisation of `stream` at the end; work on other streams that reads
 * the scene must have finished.  verts_host NULL: the vertices are enumerated on the device (bp_polytope_vertices, at
 * most 64 per obstacle, from the given rows) and vmax is ignored; vmax becomes the largest vertex count either way.
 * All or nothing: a wrong kind of batch, another n_scenes, decreasing offsets, an obstacle without 1..15 rows (or
 * 1..vmax vertices), a failed allocation or an enumerated obstacle that is not a polytope or has more than 64 vertices
 * fail the call and leave the scene as it was. */
int bp_scene_update_batch(bp_scene* scene, const double* boxes_host, const int* offsets_host /*[n_scenes+1]*/,
                          int n_scenes, double inflate, void* stream);
int bp_scene_update_polytopes_batch(bp_scene* scene, const double* rows_host, const int* nrows_host,
                                    const double* verts_host /*NULL: enumerate*/, const int* nverts_host,
                                    const int* offsets_host /*[n_scenes+1]*/, int n_scenes, int vmax, void* stream);
int bp_scene_destroy(bp_scene* scene);
int bp_scene_size(const bp_scene* scene);

/* ---- K1: closest points in the ellipsoid metric -----------------------------
 * Replaces ConvexSetFinder.compute_set_projs (:465-489; OSQP QP :10-49) for
 * S (p0, q_inv) pairs at once.  y_out[S,N,3] = E x* + p0, dist_out[S,N] =
 * || q_inv^-1 (y - p0) ||  (the `dists` of compute_polyhedron, :429). */
int bp_closest_points(const bp_scene* scene, const double* seeds_dev /*[S,3]*/, const double* q_inv_dev /*[S,3,3]*/,
                      int S, double* y_out_dev, double* dist_out_dev, void* stream);

/* ---- K2: closest points to a segment ----------------------------------------
 * Replaces ConvexSetFinder.compute_set_projs_line (:491-510; qpOASES QP :52-99).
 * x_out[S,N,3], phi_out[S,N]; obstacles are shrunk by 0.001 as at :496. */
int bp_closest_points_line(const bp_scene* scene, const double* p0_dev /*[S,3]*/, const double* p1_dev /*[S,3]*/,
                           int S, double* x_out_dev, double* phi_out_dev, void* stream);

/* ---- K3: one greedy separating-halfspace pass --------------------------------
 * Replaces ConvexSetFinder.compute_polyhedron (:423-463) for S seeds.
 * init_rows_dev: [S,6,4] rows (a0,a1,a2,b) that start every set (init_halfspaces).
 * Output rows A[S,m_max,3], b[S,m_max], m[S], status[S]. */
int bp_polyhedron(const bp_scene* scene, const double* seeds_dev, const double* q_inv_dev, const double* q_ellipse_dev,
                  const double* init_rows_dev, int S, int m_max, double* A_dev, double* b_dev, int* m_dev,
                  int* status_dev, void* stream);

/* ---- K4: maximum-volume inscribed ellipsoid -----------------------------------
 * Replaces ConvexSetFinder.mvie_socp (:512-537, free_centre=1; centre_dev is an
 * interior start hint) and mvie_socp_fixed_mid (:539-562, free_centre=0;
 * centre_dev is the fixed centre).  q_inv_out = L L^T [S,3,3], q_ellipse_out =
 * its inverse [S,3,3], centre_out [S,3]. */
int bp_mvie(const double* A_dev /*[S,m_max,3]*/, const double* b_dev /*[S,m_max]*/, const int* m_dev /*[S]*/, int S,
            int m_max, int free_centre, const double* centre_dev /*[S,3]*/, double* q_inv_out_dev,
            double* q_ellipse_out_dev, double* centre_out_dev, int* status_dev, int* newton_iters_dev /*or NULL*/,
            void* stream);

/* Replaces ConvexSetFinder.mvie_socp_fixed_r (:564-588): rotation r_ellipse_dev [S,3,3] (columns = axes) and
 * centre fixed, first semi-axis >= a_lb_dev[S].  q_inv_out = R diag(x^2) R^T, q_ellipse_out = R diag(1/x^2) R^T,
 * eigs_out [S,3] = x.  status BP_MVIE_NO_INTERIOR when the centre is not strictly inside or a_lb cannot be met
 * (the reference's SOCP is infeasible there). */
int bp_mvie_fixed_r(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max,
                    const double* centre_dev /*[S,3]*/, const double* r_ellipse_dev /*[S,3,3]*/,
                    const double* a_lb_dev /*[S]*/, double* q_inv_out_dev, double* q_ellipse_out_dev,
                    double* eigs_out_dev, int* status_dev, int* newton_iters_dev /*or NULL*/, void* stream);

/* ---- K5: the whole IRIS loop ---------------------------------------------------
 * Replaces ConvexSetFinder.find_set_around_point (:190-240) for S seeds.
 * ws_min/ws_max (host, 3 each) are the workspace box of init_halfspaces (:377-398).
 * Outputs: A[S,m_max,3], b[S,m_max], m[S] (6 + picked rows, NOT reduced),
 * q_ellipse[S,3,3], p_mid[S,3], status[S], iters[S] (k of the while loop). */
size_t bp_build_sets_workspace_bytes(int S);
int bp_build_sets_point(const bp_scene* scene, const double* seeds_dev, int S, const double* ws_min_host,
                        const double* ws_max_host, int fixed_mid, int optimize, int max_iter, int m_max,
                        double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev, double* p_mid_dev,
                        int* status_dev, int* iters_dev,
                        int* rows_peak_dev /* NULL or [S]: largest row count of any pass */,
                        int row_cap /* 0, or: a pass with more rows ends the seed with BP_ROW_CAP, like the
                                       reference's 20-row MVIE buffers do (ValueError, quirk Q5) */,
                        void* workspace_dev, size_t workspace_bytes, void* stream);

/* Same over a scene batch: seed_scene_dev[S] (int32) = scene index of every seed. */
int bp_build_sets_point_ms(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                           const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                           int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                           double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                           void* workspace_dev, size_t workspace_bytes, void* stream);

/* The same with two optional deliveries from the kernel's epilogue (rows still in shared memory):
 *   aabb_dev [S,6]    the exact bounding box of every finished set (what bp_set_aabb computes) -- hand it to
 *                     bp_pair_feasible as aabb_in_dev;
 *   peer tables       world > 0: rows, row count and box of set s are also stored into the global tables
 *                     A[S_glob,m_max,3] | b | m | aabb of EVERY rank at row slot0 + s through peer_base_dev[world]
 *                     (see bp_scatter_sets_peers); the caller synchronises the ranks afterwards.
 * Replaces find_set_around_point (ConvexSetFinder.py:190-240) + the exchange step of SURVEY 8e. */
int bp_build_sets_point_x(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                          const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                          int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                          double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                          double* aabb_dev, const unsigned long long* peer_base_dev, int world, int slot0,
                          size_t off_A, size_t off_b, size_t off_m, size_t off_aabb, void* workspace_dev,
                          size_t workspace_bytes, void* stream);

/* ---- pair tests in the tail of the set build -------------------------------------------------------------
 * With a bp_tail the CTAs of the fused set build do not exit when their set is finished: each appends its set to
 * the arrival log of every rank (a counter + a ring of set ids in the tables) and tests its set against every set
 * that is logged after it -- bounding-box
 * test, margin pre-test and LP of bp_pair_feasible, results OR-ed into row min(i,j) of the adjacency of every rank.
 * When the kernel ends on every rank the adjacency is complete: no pair kernels, no barrier between build and
 * pairs; what is left after the last set of the job arrives is one pair per waiting CTA.  Needs aabb_dev, the
 * fused path, and S <= the CTAs resident at once (checked).  bp_step_begin starts a step: it clears the adjacency
 * buffer and bumps *epoch (multi-GPU: two buffers [2][S_glob][words] alternate by the parity of the epoch and the
 * buffer of the NEXT step is the one cleared, so that no rank can clear bits a faster rank has already written;
 * the ranks synchronise once per step, after the kernel).  Tables: this rank's copies of A[S_glob,m_max,3] |
 * b | m | aabb (single GPU: the set build's own outputs); off_*: offsets of counter / log / bits in the symmetric
 * allocation of every rank (multi-GPU).  Replaces BoundPlanner.set_intersection over all pairs
 * (BoundPlanner.py:774-798) as a stage of its own. */
typedef struct {
  int S_glob, words;
  const double* A;
  const double* b;
  const int* m;
  const double* aabb;
  unsigned int* count;     /* arrival counter of this rank's log, 0 at allocation (grows by S_glob per step) */
  unsigned long long* log; /* [S_glob] ring of (epoch << 32 | set id), 0 at allocation */
  unsigned int* bits;      /* [S_glob, words] (single GPU) or [2, S_glob, words] */
  int* epoch;              /* device int, 0 at allocation */
  size_t off_count, off_log, off_bits;
  double tol;
} bp_tail;
int bp_step_begin(const bp_tail* tail, int double_buffered, void* stream);
int bp_build_sets_point_tail(const bp_scene* scene, const int* seed_scene_dev, const double* seeds_dev, int S,
                             const double* ws_min_host, const double* ws_max_host, int fixed_mid, int optimize,
                             int max_iter, int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                             double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                             double* aabb_dev, const unsigned long long* peer_base_dev, int world, int slot0,
                             size_t off_A, size_t off_b, size_t off_m, size_t off_aabb, const bp_tail* tail,
                             void* workspace_dev, size_t workspace_bytes, void* stream);

/* Replaces ConvexSetFinder.find_set_around_line (:242-307) for S segments p0 .. p0 + dp1: the IRIS loop around
 * the segment midpoint with the fixed-rotation MVIE (not called by the reference planner on main,
 * BoundPlanner.py:378-380, but part of ConvexSetFinder's surface).  optimize == 0: one pass + one free-centre
 * MVIE (:278-282).  p_mid = the midpoint (optimize) or the free MVIE's centre. */
int bp_build_sets_around_line(const bp_scene* scene, const double* p0_dev, const double* dp1_dev, int S,
                              const double* ws_min_host, const double* ws_max_host, int optimize, int max_iter,
                              int m_max, double* A_dev, double* b_dev, int* m_dev, double* q_ellipse_dev,
                              double* p_mid_dev, int* status_dev, int* iters_dev, int* rows_peak_dev, int row_cap,
                              void* stream);

/* Replaces ConvexSetFinder.find_set_collision_avoidance (:309-375) for S segments.
 * limit_space selects init_halfspaces_point(p0, e_max) (:400-421).  collision[S]
 * is the reference's `collision` flag (:336-345).  q_ellipse / p_mid are written
 * only when compute_ellipsoid != 0. */
int bp_build_sets_line(const bp_scene* scene, const double* p0_dev, const double* p1_dev, int S,
                       const double* ws_min_host, const double* ws_max_host, int limit_space, double e_max,
                       int compute_ellipsoid, int m_max, double* A_dev, double* b_dev, int* m_dev,
                       double* q_ellipse_dev, double* p_mid_dev, int* collision_dev, int* status_dev,
                       void* workspace_dev, size_t workspace_bytes, void* stream);

int bp_build_sets_line_ms(const bp_scene* scene, const int* seg_scene_dev, const double* p0_dev, const double* p1_dev,
                          int S, const double* ws_min_host, const double* ws_max_host, int limit_space, double e_max,
                          int compute_ellipsoid, int m_max, double* A_dev, double* b_dev, int* m_dev,
                          double* q_ellipse_dev, double* p_mid_dev, int* collision_dev, int* status_dev,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- K6: pairwise set-intersection test -----------------------------------------
 * Replaces BoundPlanner.set_intersection (BoundPlanner.py:774-787) as called by
 * add_edges with tol = 0.01 (:796-798), for every pair (i, j), i in
 * [row_begin,row_end), j in (i, S).  adj_bits_dev: [(row_end-row_begin), words]
 * uint32 words, words = (S+31)/32; bit j of row i is 1 iff sets i and j intersect.
 * Bits with j <= i are 0. */
/* bp_set_aabb: exact axis-aligned bounding boxes of S sets, aabb_out[S,6] = (lo xyz | hi xyz); the
 * rigorous pre-filter of bp_pair_feasible.  Pass them back through aabb_in_dev (or NULL to have
 * bp_pair_feasible compute them), e.g. after all-gathering them together with the sets. */
int bp_set_aabb(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double* aabb_out_dev,
                void* stream);
size_t bp_pair_workspace_bytes(int S, int rows /* row_end - row_begin */);
int bp_pair_feasible(const double* A_dev /*[S,m_max,3]*/, const double* b_dev /*[S,m_max]*/, const int* m_dev /*[S]*/,
                     int S, int m_max, double tol, int row_begin, int row_end, unsigned int* adj_bits_dev,
                     double* x_feas_dev /* NULL or [rows,S,3]: a point of the intersection where the bit is 1
                                           (the reference's sol_lin.x, BoundPlanner.py:785) */,
                     const double* aabb_in_dev /* NULL or [S,6] from bp_set_aabb */,
                     void* workspace_dev, size_t workspace_bytes, void* stream);

/* Diagnostics (bench.py's per-stage breakdown): the same launches as bp_pair_feasible with CUDA events between
 * them; synchronises and writes ms_host[3] = { k_set_aabb (0 when aabb_in_dev is given), k_pair_filter, k_pair_lp }. */
int bp_pair_feasible_stages(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                            int row_begin, int row_end, unsigned int* adj_bits_dev, const double* aabb_in_dev,
                            void* workspace_dev, size_t workspace_bytes, void* stream, float* ms_host);

/* The same test over an explicit list of pairs (i, j) (pairs_dev [P,2] int32): result[P] = 1/0,
 * x_feas[P,3] (or NULL).  Workspace: 6*S doubles. */
int bp_pairs_feasible_list(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double tol,
                           const int* pairs_dev, int P, int* result_dev, double* x_feas_dev, void* workspace_dev,
                           size_t workspace_bytes, void* stream);

/* ---- set-obstacle hit test (ABI 7): are planned sets still free after the obstacles moved? ----------------
 * For S sets (A[S,m_max,3] | b | m, padded rows A = 0, b = 10 accepted), first_hit[s] = the lowest obstacle index,
 * local to the set's scene, of an obstacle that set s intersects in the sense of BoundPlanner.set_intersection
 * (BoundPlanner.py:774-787): the set and the obstacle, each shrunk by tol, share a point -- the decision of an edge of
 * the set graph.  -1: no obstacle of the scene does; -2: set_scene_dev[s] lies outside [0, n_scenes) (checked on the
 * device, nothing out of range is read).  The obstacle rows are the scene's: a box gives [I; -I] x <= [ub; -lb] of
 * the inflated columns (the reference's make_box + obs_size_increase rows, bit for bit), a polytope its rows.
 * set_scene_dev [S] or NULL (every set in scene 0; a single scene has n_scenes = 1).  Box and polytope scenes, single
 * scenes and batches.  A set whose box (bp_set_aabb) misses an obstacle's box is not tested against it; the others
 * go through the LP of bp_pair_feasible in index order and the first hit ends the set's search.  Workspace:
 * bp_sets_obstacles_workspace_bytes(S) (the set boxes).  Fails for m_max outside 1 .. 48 and for a negative or
 * non-finite tol.  Used by an MPC loop to replan only the queries whose corridor (sets_via_prev) an obstacle entered. */
size_t bp_sets_obstacles_workspace_bytes(int S);
int bp_sets_obstacles(const bp_scene* scene, const int* set_scene_dev /*[S] or NULL: scene 0*/, const double* A_dev,
                      const double* b_dev, const int* m_dev, int S, int m_max, double tol, int* first_hit_dev /*[S]*/,
                      void* workspace_dev, size_t workspace_bytes, void* stream);

/* ---- K8 (next row 1): redundancy removal ---------------------------------------------
 * Replaces reduce_ineqs (bound_planner/utils/util_functions.py:82-88, cddlib
 * matrix_redundancy_remove) for S sets.  Kept rows keep their order and coefficients;
 * A_out/b_out are padded with A = 0, b = 10; keep_out[S,m_max] (or NULL) flags kept rows;
 * status[S] (or NULL) is BP_ROW_OVERFLOW when the vertex table overflowed (rows all kept). */
int bp_reduce_ineqs(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, double* A_out_dev,
                    double* b_out_dev, int* m_out_dev, unsigned char* keep_out_dev, int* status_dev, void* stream);

/* ---- K9 / K10 (next row 2): end-effector fit and projection on intersection sets ------
 * pairs_dev: [P,2] int32 (i, j) set indices; the intersection set is the stacked rows of
 * set i and set j (i == j: the set itself).
 * bp_check_fit replaces BoundPlanner.check_intersection (BoundPlanner.py:745-772):
 * l_ee_samples_host [n_samples,3] are the rotated offsets Rodrigues(omega_hat, |omega| k/19) l_ee
 * (n_samples = 20), margin = 0.001; fits[P] = 1/0 (-1: too many rows), first_sample[P] = the
 * first k that fits or -1; x0_dev (or NULL) [P,3] start points; active_dev lets the result of
 * bp_pairs_feasible_list gate the check on the device (add_edges only checks pairs that intersect).
 * bp_project_points replaces the projection QP of add_edges (BoundPlanner.py:842-864):
 * x_out[P,3] = argmin |x - xd|^2 over the intersection set. */
int bp_check_fit(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, const int* pairs_dev,
                 int P, const double* x0_dev, const int* active_dev /* NULL or [P]: 0 = skip the pair (fits = 0) */,
                 const double* l_ee_samples_host, int n_samples, double margin, int* fits_dev, int* first_sample_dev,
                 void* stream);
int bp_project_points(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max,
                      const int* pairs_dev, int P, const double* xd_dev, double* x_out_dev, int* status_dev,
                      void* stream);

/* ---- K11 - K13 (next rows 3-4): the planner loop's own tests, batched over queries -------------
 * bp_sample_filter replaces the rejection loop of plan_convex_set_path (BoundPlanner.py:459-478) for Q queries:
 * cand_dev [Q,C,3] are each query's candidate points in draw order (the caller draws them from the query's own
 * generator so the stream is the reference's); a candidate is rejected when max(A x - b) < 1e-3 for an inflated
 * obstacle of the query's scene (:467-471) or for one of its known sets (:472-476): sets set_off[q] .. set_off[q+1]-1
 * of A[.,m_max,3], b, m (set_off_dev NULL: no sets).  first_ok[Q] = index of the first accepted candidate or -1;
 * flags_dev (or NULL) [Q,C]: bit 0 in collision, bit 1 in a known set (every candidate is classified when given).
 * bp_dedupe_distance replaces the duplicate test (:505-512): dmin[P] = min over nodes node_off[i] .. node_off[i+1]-1
 * of |Q_new - Q_v|_F + |p_new - p_v| (+inf without nodes), argmin (or NULL) the node's local index.
 * bp_shortest_paths replaces nx.shortest_path(inter_graph, 0, 1, weight="weight") (:434) for G graphs in CSR form:
 * graph g owns nodes node_off[g] .. node_off[g+1]-1 (at most 1024), node v's edges are edge_off[v] .. edge_off[v+1]-1
 * with LOCAL destination ids edge_dst and weights edge_w (both directions listed); src/dst [G] local ids.
 * path[G,max_len] local node ids, path_len[G] (-1: unreachable; > max_len: path not written), cost[G]. */
int bp_sample_filter(const bp_scene* scene, const int* item_scene_dev, const double* cand_dev, int Q, int C,
                     const double* A_dev, const double* b_dev, const int* m_dev, int m_max, const int* set_off_dev,
                     int* first_ok_dev, unsigned char* flags_dev, void* stream);
int bp_dedupe_distance(const double* q_new_dev, const double* p_new_dev, int P, const double* q_nodes_dev,
                       const double* p_nodes_dev, const int* node_off_dev, double* dmin_dev, int* argmin_dev,
                       void* stream);

/* The same two tests over per-query TABLES that stay resident on the device (the lock-step planner driver keeps
 * every query's known sets and node ellipsoids in fixed-size blocks): the known sets of query q are rows
 * set_begin[q] .. set_begin[q]+set_count[q]-1 of (A, b, m); the nodes of item i are node_begin[i] ..
 * node_begin[i]+node_count[i]-1. */
int bp_sample_filter_tables(const bp_scene* scene, const int* item_scene_dev, const double* cand_dev, int Q, int C,
                            const double* A_dev, const double* b_dev, const int* m_dev, int m_max,
                            const int* set_begin_dev, const int* set_count_dev, int* first_ok_dev, void* stream);
int bp_dedupe_distance_tables(const double* q_new_dev, const double* p_new_dev, int P, const double* q_nodes_dev,
                              const double* p_nodes_dev, const int* node_begin_dev, const int* node_count_dev,
                              double* dmin_dev, int* argmin_dev, void* stream);
int bp_shortest_paths(const int* node_off_dev, const int* edge_off_dev, const int* edge_dst_dev,
                      const double* edge_w_dev, const int* src_dev, const int* dst_dev, int G, int max_len,
                      int* path_dev, int* path_len_dev, double* cost_dev, void* stream);

/* ---- native lock-step planner driver (SURVEY 8f; BASELINE config C3) ---------------------------------------
 * bp_plan_run plans Q independent queries, one scene each (a scene batch), in lock step: the per-query loop of
 * BoundPlanner.plan_convex_set_path (BoundPlanner.py:174-584, replanning branch :231-276 and the start-in-collision
 * fallbacks :296-324 included) up to the planned set
 * sequence, add_edges (:789-896) and compute_via_points (:586-743, no rotations) run as C++ state machines on the
 * host (csrc/bp_planner.h); every round, the pending requests of all queries are answered by ONE chain of the
 * kernels above (K11 -> K5 -> K12 -> K8 for sampling rounds, K6 + K9 for add_edges, K10, K13) against per-query
 * node tables resident on the device, with one H2D and one D2H copy per round.  Each query consumes its own
 * numpy-compatible PCG64 stream exactly as the reference's rng.uniform calls would.
 * The caller provides what involves rotations (scipy's as_rotvec in the reference, :207-219): l_ee, l_ee_end and
 * the 20 rotated offsets of check_intersection (:745-772) per query.
 * Obstacles come in one of two forms, the form of the plan's scene batch: boxes (obs_rows NULL; the batch from
 * bp_scene_create_batch) or general convex polytopes (obs_rows set, boxes may be NULL; the batch from
 * bp_scene_create_polytopes_batch).  bp_plan_run fails when the form of `in` is not the batch's, or when a query's
 * obstacle count is not its scene's: the host-side push-out of `end` (:199-204) and the device scene must agree.
 * Replanning (an MPC loop calling the planner again): a query with replanning[q] builds its start set around the
 * segment start .. p_horizon[idx], idx the horizon index of :231-266 over the query's previous sets; the previous
 * sets (what the reference keeps in sets_via_prev between calls) also serve the fallback of a start segment in
 * collision (:296-324): reduce_ineqs of the last one, or IndexError without any (err_kind 3); with new_obs a start
 * set around `start`, or AttributeError when `start` lies in an inflated obstacle (quirk Q12, err_kind 4).  All
 * replanning fields may be NULL: no query replans, none has previous sets.  Malformed offsets (not starting at 0,
 * decreasing), more than 64 sets per query or a set with no row or more than 48 rows fail the call before any
 * round runs. */
typedef struct {
  int Q;
  const double* boxes;        /* all scenes back to back [sum n_obs, 6] (lb, ub), as given to bp_scene_create_batch;
                                 NULL when obs_rows is set */
  const int* box_off;         /* [Q+1] obstacle offsets of every query (boxes or polytopes); for a plan from
                                 bp_plan_create_mapped [n_scenes+1] offsets of every scene, whose obstacles boxes /
                                 obs_rows hold once however many queries plan in it */
  double inflate;             /* obs_size_increase */
  const double* ws_min;       /* [3] */
  const double* ws_max;       /* [3] */
  const double* starts;       /* [Q,3] */
  const double* ends;         /* [Q,3] */
  const double* l_ee;         /* [Q,3]   r0 @ (-length_ee, 0, 0) */
  const double* l_ee_end;     /* [Q,3]   r1 @ (-length_ee, 0, 0) */
  const double* ee_samples;   /* [Q,20,3] Rodrigues(omega_hat, |omega| k/19) l_ee */
  const unsigned long long* rng; /* [Q,4] PCG64 (state_hi, state_lo, inc_hi, inc_lo) of every query's generator */
  const int* has_first;       /* [Q] or NULL */
  const double* first_sample; /* [Q,3] or NULL */
  int sample_chunk;           /* candidates drawn ahead per sampling request (<= 0: 32; at most 64) */
  int max_rounds;             /* <= 0: default (4000) */
  const double* obs_rows;     /* [sum n_obs, 15, 4] (a, b) rows of inflated polytope obstacles, or NULL: boxes */
  /* replanning (ABI 4); every field may be NULL */
  const int* replanning;      /* [Q] 1: replanning call (:231-276) */
  const int* new_obs;         /* [Q] the reference's new_obs flag */
  const int* horizon_off;     /* [Q+1] MPC horizon points of every query in p_horizon */
  const double* p_horizon;    /* [sum H, 3] */
  const int* prev_off;        /* [Q+1] previous sets of every query (at most 64 per query), oldest first */
  const int* prev_row_off;    /* [n_prev+1] rows of every previous set in prev_rows (1 .. 48 per set) */
  const double* prev_rows;    /* [sum rows, 4] (a0, a1, a2, b) */
} bp_plan_in;

typedef struct {
  int* err_kind;              /* [Q] 0 planned, 1 RuntimeError, 2 ValueError, 3 IndexError, 4 AttributeError
                                 (the reference's exits) */
  char* err_msg;              /* [Q,160] */
  int* path;                  /* [Q,64] intersection-graph node ids of the shortest path */
  int* path_len;              /* [Q] */
  int* set_ids;               /* [Q,64] planned set sequence (graph node ids) */
  int* n_ids;                 /* [Q] */
  double* p_via;              /* [Q,66,3] via points (start, projections, end) */
  int* n_via;                 /* [Q] */
  unsigned long long* rng_out; /* [Q,4] generator state after the query (or NULL) */
  int* n_nodes;               /* [Q] graph nodes */
  int* n_inter;               /* [Q] intersection-graph nodes */
  int* n_edges;               /* [Q] intersection-graph edges */
  int* finish_round;          /* [Q] lock-step round in which the query was answered */
  double* finish_ms;          /* [Q] or NULL: wall time since the start of the run at the end of that round */
  double* node_A;             /* [Q,64,24,3] or NULL: every graph node's reduced set */
  double* node_b;             /* [Q,64,24]   or NULL */
  int* node_m;                /* [Q,64]      or NULL */
  long long* stats;           /* [8] or NULL: rounds, set requests, pair tests, projections, shortest paths,
                                 kernel chains launched, microseconds spent waiting for the device */
  double* p_horizon_max;      /* [Q,3] or NULL (ABI 4): p_horizon[idx] of every replanning query */
} bp_plan_out;

/* bp_plan_create takes a box or a polytope scene batch with one scene per query (query q plans in scene q: the
 * identity map of bp_plan_create_mapped); the per-scene limits of the kernels
 * the rounds launch are checked here, not in the middle of a run (polytope scenes: at most 16384 obstacles).  The plan
 * keeps the scene batch, not a copy: after bp_scene_update_batch / bp_scene_update_polytopes_batch, bp_plan_run plans
 * against the new obstacles, checks its inputs against the batch's current offsets and re-checks the limit.
 * bp_plan_create_mapped (ABI 6) plans many queries over shared scenes: query q plans in scene query_scene_host[q] of a
 * batch of any n_scenes >= 1 (scenes no query uses are allowed); every entry must lie in [0, n_scenes), else the call
 * fails and names the query.  The plan keeps a copy of the map.  bp_plan_run then takes every scene's obstacles once
 * (bp_plan_in::box_off of n_scenes + 1 entries, checked scene by scene against the batch); every other field of
 * bp_plan_in stays per query.  A query planned in a shared scene gives the same results, bit for bit, as the same query
 * in a scene batch of one copy per query. */
typedef struct bp_plan bp_plan;
int bp_plan_create(const bp_scene* scene_batch, int Q, bp_plan** out);
int bp_plan_create_mapped(const bp_scene* scene_batch, int Q, const int* query_scene_host /*[Q]*/, bp_plan** out);
int bp_plan_run(bp_plan* plan, const bp_plan_in* in, bp_plan_out* out, void* stream);
/* bp_plan_run_active (ABI 7) plans the queries q with active_host[q] != 0 only (NULL: all, as bp_plan_run), e.g. the
 * queries of an MPC step whose corridor bp_sets_obstacles found hit.  `in` and `out` are the whole batch's, checked as
 * by bp_plan_run.  A skipped query gets no state machine, no request and no table write; its outputs are left as they
 * are, except finish_round[q] = -1, and stats count the active queries only.  An active query's outputs are bit for
 * bit the ones bp_plan_run gives it over the whole batch (generator state and errors included), on plans from
 * bp_plan_create and bp_plan_create_mapped.  The active queries are dealt to the lanes in turn (k-th -> lane k mod L). */
int bp_plan_run_active(bp_plan* plan, const bp_plan_in* in, const int* active_host /*[Q] or NULL*/, bp_plan_out* out,
                       void* stream);
int bp_plan_destroy(bp_plan* plan);

/* ---- multi-GPU exchange by peer stores (SURVEY 8e) -------------------------------------------------------
 * The owner of S_loc sets writes them into the global tables A[S,m_max,3] | b[S,m_max] | m[S] | aabb[S,6] of EVERY
 * rank at rows slot0 .. slot0+S_loc-1, through the peers' mapped addresses: peer_base_dev[world] holds the base
 * address of each rank's symmetric allocation (identical layout everywhere, e.g. torch symmetric memory or
 * cudaIpc / VMM mappings), off_* are the byte offsets of the tables inside it.  bp_scatter_rows_peers does the same
 * for a block of adjacency rows (rows x words uint32 at global row row0).  The caller synchronises the ranks after
 * each call (signal-pad barrier); replaces pack + ncclAllGather + unpack. */
int bp_scatter_sets_peers(const double* A_dev, const double* b_dev, const int* m_dev, const double* aabb_dev, int S_loc,
                          int m_max, int slot0, const unsigned long long* peer_base_dev, int world, size_t off_A,
                          size_t off_b, size_t off_m, size_t off_aabb, void* stream);
int bp_scatter_rows_peers(const unsigned int* rows_dev, int rows, int words, int row0,
                          const unsigned long long* peer_base_dev, int world, size_t off_bits, void* stream);

/* ---- K7: iiwa14 forward kinematics -----------------------------------------------
 * Replaces the numeric branch of RobotModel.fk_pos (RobotModel.py:146-160),
 * fk_pos_col (:162-181), hom_transform_endeffector (:197-211), jacobian_fk
 * (:213-231).  q[B,7]; p_ee[B,3]; p_col[B,7,3] (joint_3..7, link4_col, ee_col);
 * T_ee[B,4,4] or NULL; jac[B,6,7] or NULL. */
int bp_fk_iiwa14(const double* q_dev, int B, double* p_ee_dev, double* p_col_dev, double* T_ee_dev, double* jac_dev,
                 void* stream);

/* RobotModel.forward_kinematics(q, dq) (RobotModel.py:70-77; callers MPCNode.py:38,118, util_functions.py:57),
 * jacobian_fk (:213-231) and djacobian_fk (:233-251, pin.getFrameJacobianTimeVariation, LOCAL_WORLD_ALIGNED) for
 * B (q, dq) pairs: T_ee[B,4,4], jac[B,6,7], djac[B,6,7] (= d/dt jac along dq; NULL with dq_dev NULL: skip). */
int bp_fk_iiwa14_kin(const double* q_dev, const double* dq_dev, int B, double* T_ee_dev, double* jac_dev,
                     double* djac_dev, void* stream);

/* compute_polytope_vertices (bound_planner/utils/util_functions.py:66-79, cddlib): vertices of S polytopes
 * {A x <= b}: V[S,vmax,3] (first nv[s] rows valid, deterministic order), status[s] = BP_OK, BP_NOT_A_POLYTOPE (the
 * reference raises ValueError("Polyhedron is not a polytope")) or BP_ROW_OVERFLOW (more than vmax vertices). */
int bp_polytope_vertices(const double* A_dev, const double* b_dev, const int* m_dev, int S, int m_max, int vmax,
                         double* V_dev, int* nv_dev, int* status_dev, void* stream);

/* Diagnostics: out_host[0] = polyhedron passes (since the last reset) that overflowed the closest-point shell of
 * the box-scene pass and were redone in the per-pick form; further entries reserved (0).  Synchronises the device. */
int bp_debug_counters(unsigned long long* out_host, int n, int reset);

/* ---- diagnostics: FP64 pipe probe (roofline denominator in bench.py) ------------
 * Launches blocks x threads threads, each running `chains` (1, 4 or 8)
 * independent chains of `iters` dependent DFMAs; out_dev: [blocks*threads]. */
int bp_probe_fp64(int chains, int blocks, int threads, int iters, double* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BPGEO_H */
