/*
 * rrtqx_b200.h -- C ABI of librrtqx_b200.so: the B200 (sm_100a) implementation
 * of RRTQX_3D's geometric inner loop (batched kd-tree neighbour queries and
 * batched edge/node-vs-obstacle collision checks).
 *
 * This is the drop-in boundary.  The reference (Julia) has no FFI for this
 * path today; each entry point below names the Julia function(s) whose work it
 * takes over, as file:line under /root/reference/code_RRTQx_3D/.  The Julia
 * binding a maintainer adds is julia/RRTQXGpu.jl (see INTEGRATION.md); the
 * Python ctypes mirror used by the tests is rrtqx_3d_b200/_abi.py.
 *
 * Conventions
 *  - Every function returns rrtqx_status (0 = ok).  The message of the last
 *    failure is available from rrtqx_last_error(ctx) (ctx may be NULL for
 *    failures of rrtqx_ctx_create).  The reference signals errors with Julia
 *    error(...) exceptions; the Julia wrapper re-raises non-zero statuses.
 *  - Plain pointers and sizes only.  Input/output array pointers may be host
 *    (pageable or pinned) or CUDA device pointers; the library detects which
 *    (cudaPointerGetAttributes) and copies only when needed.  Arrays are
 *    row-major: an n x d position array is n consecutive rows of d doubles,
 *    which is the memory image of Julia's 1xd `position` matrices stacked.
 *  - Node indices are 0-based int32 in insertion order (index i = the i-th
 *    kdInsert).  Julia wrappers add 1.
 *  - Single caller thread per context, blocking calls (results are ready on
 *    return) unless a function says "async".  There is NO CPU fallback: if no
 *    CUDA device is usable, rrtqx_ctx_create fails with RRTQX_ERR_CUDA.
 *  - All arithmetic that decides membership / collision is IEEE binary64 in
 *    the reference's operation order, never fused (SURVEY.md appendix A).
 */
#ifndef RRTQX_B200_H
#define RRTQX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define RRTQX_API __declspec(dllexport)
#else
#define RRTQX_API __attribute__((visibility("default")))
#endif

typedef int32_t rrtqx_status;
enum {
  RRTQX_OK = 0,
  RRTQX_ERR_INVALID = 1,     /* bad argument */
  RRTQX_ERR_CUDA = 2,        /* CUDA runtime / no device */
  RRTQX_ERR_NOMEM = 3,       /* device or host allocation failed */
  RRTQX_ERR_EMPTY_TREE = 4,  /* query on an empty tree (the reference would
                                dereference an undefined root,
                                kdTree_general.jl:359,895) */
  RRTQX_ERR_UNSUPPORTED = 5,
  RRTQX_ERR_STATE = 6        /* result object not filled yet, etc. */
};

typedef struct rrtqx_ctx rrtqx_ctx;
typedef struct rrtqx_tree rrtqx_tree;
typedef struct rrtqx_spheres rrtqx_spheres;
typedef struct rrtqx_polygons rrtqx_polygons;
typedef struct rrtqx_edges rrtqx_edges;
typedef struct rrtqx_range_result rrtqx_range_result;
typedef struct rrtqx_sweep_result rrtqx_sweep_result;
typedef struct rrtqx_dubins_result rrtqx_dubins_result;

/* ---------------------------------------------------------------- context */

RRTQX_API const char *rrtqx_version(void);
/* device: CUDA ordinal.  cuda_stream: a cudaStream_t to launch on (e.g. the
 * caller's current stream) or NULL for a private non-blocking stream.  The
 * handle of CUDA's DEFAULT stream is 0 == NULL: a caller that wants its own
 * work ordered with the library's (timing events, cache flushes, tensors it
 * fills before a call) must hand over a stream it created, not the default
 * one (PyTorch: torch.cuda.Stream(), not torch.cuda.current_stream() of a
 * fresh process, whose cuda_stream is 0) -- or CUDA's explicit names for the
 * default streams, cudaStreamLegacy ((void *)0x1) / cudaStreamPerThread
 * ((void *)0x2), which are non-zero handles and are used verbatim. */
RRTQX_API rrtqx_status rrtqx_ctx_create(int32_t device, void *cuda_stream,
                                        rrtqx_ctx **out);
RRTQX_API rrtqx_status rrtqx_ctx_destroy(rrtqx_ctx *ctx);
RRTQX_API const char *rrtqx_last_error(const rrtqx_ctx *ctx);
/* The diagnostic RRTQX_* environment switches (DESIGN.md section 5) are read
 * once, by rrtqx_ctx_create; this re-reads them for `ctx` (tests and A/B runs
 * that change a switch between calls).  No call on the hot path touches the
 * environment. */
RRTQX_API rrtqx_status rrtqx_ctx_reload_tuning(rrtqx_ctx *ctx);
RRTQX_API rrtqx_status rrtqx_ctx_sync(rrtqx_ctx *ctx);
/* Page-locked ("pinned") host memory for query / result arrays.  Every entry
 * point accepts ordinary (pageable) host pointers too -- Julia `Vector`s under
 * GC.@preserve -- but the driver then stages the copies at a fraction of the
 * PCIe rate; arrays that are reused across calls should live here (in Julia:
 * unsafe_wrap(Array, Ptr{T}(p), n) over the returned pointer).  Free with
 * rrtqx_host_free (ctx may be NULL there). */
RRTQX_API rrtqx_status rrtqx_host_alloc(rrtqx_ctx *ctx, int64_t bytes,
                                        void **out);
RRTQX_API rrtqx_status rrtqx_host_free(rrtqx_ctx *ctx, void *p);
/* number of kernels this context has launched so far (bench.py gpu_launches) */
RRTQX_API rrtqx_status rrtqx_ctx_kernel_launches(const rrtqx_ctx *ctx,
                                                 int64_t *out);
/* CUDA-event timing of the context's most recent named phase, in ms; phase is
 * one of "range_query", "nearest", "edge_check", "node_check", "add_sweep",
 * "remove_sweep", "tree_build".  Measured on the context's stream. */
/* measured FP64 FMA throughput of the device (TFLOP/s, 2 flop per FMA): the roofline denominator of the
 * FP64-bound collision kernels, taken in the same run as the numbers it normalises */
RRTQX_API rrtqx_status rrtqx_ctx_measure_fp64_peak(rrtqx_ctx *ctx,
                                                   double *tflops);
RRTQX_API rrtqx_status rrtqx_ctx_last_phase_ms(rrtqx_ctx *ctx,
                                               const char *phase, float *ms);

/* ------------------------------------------------------------------- tree */
/* KDTree{T}(d, f) / KDTree{T}(d, f, wraps, wrapPoints)
 * (kdTree_general.jl:94-112).  The metric f is always KDdist = euclidianDist
 * in both edge files (DRRT_SimpleEdge_functions.jl:51,
 * DRRT_DubinsEdge_functions.jl:52), so it is not a parameter.  d in 2..4.
 * wraps: 0-based dimension indices that wrap around, period wrap_points[i]
 * (space assumed to start at 0, kdTree_general.jl:101-102). */
RRTQX_API rrtqx_status rrtqx_tree_create(rrtqx_ctx *ctx, int32_t d,
                                         int32_t num_wraps,
                                         const int32_t *wraps,
                                         const double *wrap_points,
                                         rrtqx_tree **out);
RRTQX_API rrtqx_status rrtqx_tree_destroy(rrtqx_tree *tree);
/* kdInsert (kdTree_general.jl:121-170) for n nodes in order.  The resulting
 * kd topology (parent / children / split) is exactly the one sequential
 * insertion produces.  *first_index_out = index of positions[0]. */
RRTQX_API rrtqx_status rrtqx_tree_insert_batch(rrtqx_tree *tree,
                                               const double *positions,
                                               int64_t n,
                                               int32_t *first_index_out);
/* kdInsert of one node (the planner's per-iteration insert, DRRT_Q.jl:2575).
 * A host position is read during the call and inserted by ONE asynchronous
 * launch (position passed by value): the call does not wait for the device;
 * every later call on the same context sees the node (stream order). */
RRTQX_API rrtqx_status rrtqx_tree_insert(rrtqx_tree *tree,
                                         const double *position,
                                         int32_t *index_out);
RRTQX_API rrtqx_status rrtqx_tree_size(const rrtqx_tree *tree, int64_t *n);
/* kd fields of nodes [first, first+count) so the caller can keep
 * RRTNode.kdParent/kdChildL/kdChildR/kdSplit populated
 * (DRRT_data_structures.jl:25-33,68-72).  -1 = absent; split is 0-based.
 * Any output pointer may be NULL. */
RRTQX_API rrtqx_status rrtqx_tree_kd_fields(rrtqx_tree *tree, int64_t first,
                                            int64_t count, int32_t *parent,
                                            int32_t *child_l, int32_t *child_r,
                                            int32_t *split);
/* Copies positions of nodes [first, first+count) back (row-major). */
/* order_out[k] = node visited k-th by the reference's recursive kd traversal (node, kdChildL subtree,
 * kdChildR subtree): the row order of saveRRTNodes / saveRRTTree / saveRRTGraph (DRRT_Q.jl:252-337).
 * order_out: host array of tree-size entries. */
RRTQX_API rrtqx_status rrtqx_tree_preorder(rrtqx_tree *tree,
                                           int32_t *order_out);
RRTQX_API rrtqx_status rrtqx_tree_positions(rrtqx_tree *tree, int64_t first,
                                            int64_t count, double *out);
/* Tuning knob of the device index: mean points per grid cell the next
 * (re)build aims for (default 8).  Does not change any result. */
RRTQX_API rrtqx_status rrtqx_tree_set_cell_occupancy(rrtqx_tree *tree,
                                                     double points_per_cell);
/* Force the device index to absorb the unsorted tail of recent inserts now. */
RRTQX_API rrtqx_status rrtqx_tree_reindex(rrtqx_tree *tree);

/* -------------------------------------------------------- range queries */
/* kdFindWithinRange(tree, range, q) (kdTree_general.jl:889-919), batched.
 * For each query: every node with euclid(q,node) < range (strict), the root
 * (node 0) being admitted with <= (:896-898); with wrap dimensions also the
 * nodes within range of the ghost identities (ghostPoint.jl:60-111), keyed by
 * the first identity that reaches them.  `ranges` = one radius per query, or
 * NULL to use `range` for all.  The result lives on the device inside *result
 * (created when *result == NULL, otherwise reused).  The per-query lists are
 * SETS: their order is the device traversal order, not the reference's LIFO
 * order (SURVEY.md appendix B3). */
enum {
  RRTQX_RANGE_WANT_DIST = 1u, /* also produce the JList keys (distances) */
  RRTQX_RANGE_COUNT_ONLY = 2u /* only counts and total */
};
RRTQX_API rrtqx_status rrtqx_range_query_batch(rrtqx_tree *tree,
                                               const double *queries,
                                               int64_t n_queries, double range,
                                               const double *ranges,
                                               uint32_t flags,
                                               rrtqx_range_result **result,
                                               int64_t *total_out);
RRTQX_API rrtqx_status rrtqx_range_result_destroy(rrtqx_range_result *r);
RRTQX_API rrtqx_status rrtqx_range_result_sizes(const rrtqx_range_result *r,
                                                int64_t *n_queries,
                                                int64_t *total);
/* counts[q] (int32, n_queries) and offsets[q] (int64, n_queries): query q's
 * list is idx[offsets[q] .. offsets[q]+counts[q]).  Lists are disjoint and
 * tightly packed (sum counts == total).  Output pointers: host or device. */
RRTQX_API rrtqx_status rrtqx_range_result_layout(rrtqx_range_result *r,
                                                 int32_t *counts,
                                                 int64_t *offsets);
/* idx (int32, total) and dist (double, total; NULL allowed).  dist requires
 * RRTQX_RANGE_WANT_DIST at query time. */
RRTQX_API rrtqx_status rrtqx_range_result_fetch(rrtqx_range_result *r,
                                                int32_t *idx, double *dist);
/* Device views (valid until the result is reused or destroyed). */
RRTQX_API rrtqx_status rrtqx_range_result_device(const rrtqx_range_result *r,
                                                 const int32_t **counts,
                                                 const int64_t **offsets,
                                                 const int32_t **idx,
                                                 const double **dist);

/* kdFindNearest(tree, q) (kdTree_general.jl:357-385), batched: index and
 * distance of the nearest node (ghost identities included).  On exact
 * distance ties the reference returns the first minimiser in its traversal
 * order; this library returns the minimiser with the smallest index
 * (documented tie, SURVEY.md appendix A6).  The distance is bit-exact. */
RRTQX_API rrtqx_status rrtqx_nearest_batch(rrtqx_tree *tree,
                                           const double *queries,
                                           int64_t n_queries, int32_t *idx_out,
                                           double *dist_out);

/* ------------------------------------------------------- sphere obstacles */
/* CSpace.obstacles :: List{SphereObstacle} (DRRT_data_structures.jl:267-316)
 * flattened: centres n x 3, radii n, active n (uint8).  active[i] must be
 * !(obstacleUnused || lifeSpan <= 0), the early-out predicate of
 * explicitEdgeCheck3D / explicitPointCheck2D (DRRT_Q.jl:1777,1467). */
RRTQX_API rrtqx_status rrtqx_spheres_create(rrtqx_ctx *ctx,
                                            rrtqx_spheres **out);
RRTQX_API rrtqx_status rrtqx_spheres_destroy(rrtqx_spheres *s);
RRTQX_API rrtqx_status rrtqx_spheres_upload(rrtqx_spheres *s,
                                            const double *centers,
                                            const double *radii,
                                            const uint8_t *active, int64_t n);
/* In-place update of obstacles [first, first+count): radius (obstacle
 * augmentation, obstacleAugmentation.jl:106-114) and/or active flag.  Either
 * pointer may be NULL. */
RRTQX_API rrtqx_status rrtqx_spheres_update(rrtqx_spheres *s, int64_t first,
                                            int64_t count, const double *radii,
                                            const uint8_t *active);
RRTQX_API rrtqx_status rrtqx_spheres_size(const rrtqx_spheres *s, int64_t *n);

/* ------------------------------------------------------ collision checks */
enum {
  RRTQX_CHECK_FMA_DOT = 1u,       /* evaluate the 3-term dot of
                                     distancePointToSegment with fused
                                     multiply-adds (OpenBLAS build variant,
                                     SURVEY.md 8c); default unfused */
  RRTQX_CHECK_IGNORE_ACTIVE = 2u, /* treat every obstacle as active */
  RRTQX_CHECK_QUICK_PASS = 4u     /* node check: run the quickCheck pass first
                                     (explicitPointCheck, DRRT_Q.jl:1520) as
                                     opposed to explicitPointCheck3D (:1558) */
};
/* explicitEdgeCheck(S, edge) (DRRT_Q.jl:1802-1826) for SimpleEdge
 * (DRRT_SimpleEdge_functions.jl:210 -> explicitEdgeCheck3D DRRT_Q.jl:1775 ->
 * distancePointToSegment :1205), batched over edges between tree nodes:
 * collide_out[e] = OR over all active spheres.  Edge e runs from node src[e]
 * to node dst[e]; the test is NOT symmetric in (src,dst). */
RRTQX_API rrtqx_status rrtqx_edge_check_batch(rrtqx_tree *tree,
                                              const rrtqx_spheres *spheres,
                                              const int32_t *src,
                                              const int32_t *dst,
                                              int64_t n_edges,
                                              double robot_radius,
                                              uint32_t flags,
                                              uint8_t *collide_out);
/* Same for segments given by explicit end points (a sample that is not in the
 * tree yet, the robot edge R.robotEdge DRRT_Q.jl:3287): starts/ends n x 3. */
RRTQX_API rrtqx_status rrtqx_segment_check_batch(rrtqx_ctx *ctx,
                                                 const rrtqx_spheres *spheres,
                                                 const double *starts,
                                                 const double *ends,
                                                 int64_t n_segments,
                                                 double robot_radius,
                                                 uint32_t flags,
                                                 uint8_t *collide_out);
/* explicitPointCheck / explicitNodeCheck (DRRT_Q.jl:1520-1556,1594) and the
 * 3D twins (:1558-1590,1595), batched: collide_out[i] and the certificate
 * cert_out[i] (min clearance; 0.0 on collision; NULL allowed). points n x 3. */
RRTQX_API rrtqx_status rrtqx_node_check_batch(rrtqx_ctx *ctx,
                                              const rrtqx_spheres *spheres,
                                              const double *points, int64_t n,
                                              double robot_radius,
                                              uint32_t flags,
                                              uint8_t *collide_out,
                                              double *cert_out);

/* The planner's per-iteration geometric work in ONE launch (rrtqx.jl:926-950,
 * extend() DRRT_Q.jl:2546-2641) for the new sample `point` (d doubles, host):
 *   kdFindNearest            -> nearest_idx / nearest_dist
 *   explicitNodeCheck(3D)    -> point_collides / point_cert (RRTQX_CHECK_QUICK_PASS selects :1520 vs :1558)
 *   kdFindWithinRange(range) -> *n_neighbors, nbr_idx[], nbr_dist[] (JList keys)
 *   explicitEdgeCheck of edge(new -> n) and edge(n -> new) for every neighbour n
 *                            -> fwd_collide[], rev_collide[]  (the test is not symmetric)
 * `capacity` = length of the four neighbour arrays; *n_neighbors receives the
 * full count (if it exceeds capacity only the first `capacity` are written).
 * At most 768 ACTIVE obstacles (inactive entries of an ever-growing list are
 * compacted away, once per obstacle-set change); d == 3 for the edge checks
 * (other d: flags are 0).  Trees with wrap-around dimensions are refused with
 * RRTQX_ERR_UNSUPPORTED: the launch searches the real point only, without the
 * ghost identities of kdFindNearest / kdFindWithinRange; use
 * rrtqx_nearest_batch and rrtqx_range_query_batch there, or, on the
 * DubinsEdge tree [x y t theta], rrtqx_extend_query_dubins below.
 * Non-finite input, as in kdFindNearest, which starts from the root: a sample
 * whose every radicand is NaN or +inf (a NaN coordinate, 1e200) and any sample
 * whose radicand to the root is NaN get nearest_idx = 0 with the root's
 * distance (never -1).  Nearest ties go to the smallest node index.
 * Results arrive through mapped pinned memory: one launch, one synchronise. */
RRTQX_API rrtqx_status rrtqx_extend_query(
    rrtqx_tree *tree, const rrtqx_spheres *spheres, const double *point,
    double range, double robot_radius, uint32_t flags, int32_t capacity,
    int32_t *nearest_idx, double *nearest_dist, uint8_t *point_collides,
    double *point_cert, int32_t *n_neighbors, int32_t *nbr_idx,
    double *nbr_dist, uint8_t *fwd_collide, uint8_t *rev_collide);

/* The DubinsEdge counterpart (config C4: a 4-D tree [x y t theta] whose
 * dimension 3 wraps with period 2 pi = 6.283185307179586; every other layout
 * fails with RRTQX_ERR_UNSUPPORTED) for the new sample `point` (4 doubles,
 * host), in the reference's order:
 *   kdFindNearest(KD, point), ghost identity included -> nearest_idx /
 *       nearest_dist (ties and non-finite input as rrtqx_nearest_batch)
 *   with RRTQX_EXTEND_SATURATE: saturate(point, nearest, delta)
 *       (DRRT_DubinsEdge_functions.jl:70-95), written back into `point`;
 *       without it the point is used as given (delta unused)
 *   kdFindWithinRange(KD, range, point), ghost identity included
 *       -> *n_neighbors, nbr_idx[], nbr_dist[] (as rrtqx_range_query_batch)
 *   for neighbour i: edge 2i = new -> nbr (findBestParent, DRRT_Q.jl:1949-1960)
 *   and edge 2i+1 = nbr -> new (:2600-2603): calculateTrajectory -> edge_dist[]
 *   and edge_type[] (codes of rrtqx_dubins_trajectory_batch), Dubins
 *   explicitEdgeCheck OR-ed over the polygon set -> edge_collide[]
 *   (as rrtqx_dubins_edge_check_batch; RRTQX_CHECK_IGNORE_ACTIVE honoured).
 * `capacity` = length of nbr_idx / nbr_dist; the edge arrays hold 2*capacity.
 * *n_neighbors is the full count; only the first `capacity` neighbours and
 * their edges are produced.  Any output pointer may be NULL.  With
 * trajectories != NULL the rows of the 2*min(count, capacity) edges are left,
 * in edge order, in that rrtqx_dubins_result (created when *trajectories is
 * NULL); read them with rrtqx_dubins_result_sizes / _fetch / _device.
 * The polygon-world node check is not part of this call.
 * Three launches and one host wait on mapped pinned memory; a call whose rows
 * outgrow the grow-only scratch grows it and runs once more. */
enum { RRTQX_EXTEND_SATURATE = 8u }; /* same flags word as the RRTQX_CHECK_* */
RRTQX_API rrtqx_status rrtqx_extend_query_dubins(
    rrtqx_tree *tree, const rrtqx_polygons *polygons, double *point,
    double delta, double range, double robot_radius, double min_turn_radius,
    uint32_t flags, int32_t capacity, int32_t *nearest_idx,
    double *nearest_dist, int32_t *n_neighbors, int32_t *nbr_idx,
    double *nbr_dist, double *edge_dist, int32_t *edge_type,
    uint8_t *edge_collide, rrtqx_dubins_result **trajectories);

/* ------------------------------------------------- resident edge set + sweeps */
/* Device mirror of the planner's out-edge lists: for node v the reference
 * iterates InitialNeighborListOut then rrtNeighborsOut
 * (DRRT_Q.jl:2408-2431); the caller uploads those edges as (src,dst) pairs in
 * any order (edge id = position in the upload) and optionally parent[v]
 * (index of rrtParentEdge.endNode, -1 when !rrtParentUsed). */
RRTQX_API rrtqx_status rrtqx_edges_create(rrtqx_tree *tree, rrtqx_edges **out);
RRTQX_API rrtqx_status rrtqx_edges_destroy(rrtqx_edges *e);
RRTQX_API rrtqx_status rrtqx_edges_upload(rrtqx_edges *e, const int32_t *src,
                                          const int32_t *dst, int64_t n_edges,
                                          const int32_t *parent,
                                          int64_t n_parent);
/* Neighbour-graph residency (SURVEY 8f-2).  rrtqx_edges_append adds n_new edges behind the existing ones
 * (edge id = position, continuing the upload order): the edges the planner creates in one iteration
 * (makeNeighborOf / makeInitialOutNeighborOf, DRRT_Q.jl:2589-2593); endpoints may be nodes inserted into the
 * tree since the upload.  rrtqx_edges_set_parents re-points parent edges (makeParentOf, DRRT_Q.jl:1841-1856):
 * parent_ids[i] becomes the parent of node_ids[i], -1 = rrtParentUsed false; nodes never mentioned have no
 * parent edge (which of these calls need new Dubins trajectories: rrtqx_edges_solve_trajectories).
 * Neither call re-uploads the graph; the device CSR is rebuilt before the next sweep.  Edges
 * are never deleted: results for edges the planner has culled are ignored by the caller. */
RRTQX_API rrtqx_status rrtqx_edges_append(rrtqx_edges *e, const int32_t *src,
                                          const int32_t *dst, int64_t n_new);
RRTQX_API rrtqx_status rrtqx_edges_set_parents(rrtqx_edges *e,
                                               const int32_t *node_ids,
                                               const int32_t *parent_ids,
                                               int64_t n);
RRTQX_API rrtqx_status rrtqx_edges_size(const rrtqx_edges *e, int64_t *n_edges);
/* explicitEdgeCheck(S, edge) (DRRT_Q.jl:1802-1826) of EVERY resident out-edge:
 * collide_out[e] for edge id e (n_edges entries, host or device).  Same
 * result as rrtqx_edge_check_batch on the same (src, dst) pairs; the resident
 * form streams per-edge records prepared when the set was built instead of
 * gathering the end points of every edge on every call. */
RRTQX_API rrtqx_status rrtqx_edges_check_batch(rrtqx_edges *e,
                                               const rrtqx_spheres *spheres,
                                               double robot_radius,
                                               uint32_t flags,
                                               uint8_t *collide_out);

/* addNewObstacle (DRRT_Q.jl:3220-3290) geometric part, batched over obstacles
 * ob_ids[0..n_obs) of `spheres` (treated as active, :3222).  For obstacle o:
 * candidate nodes = kdFindWithinRange(KD, (robot_radius+delta)+radius_o,
 * centre_o) (:3195-3204); every out-edge of a candidate that collides with o
 * is "blocked" (edge.dist = Inf, :3248-3249); every candidate whose parent
 * edge collides is an "orphan" (:3257-3270).  Only edges whose START node is
 * a candidate are tested, as in the reference.
 * Results (OR over the given obstacles): the set of blocked edge ids, the set
 * of orphaned node ids, and the same as per-edge / per-node byte flags. */
RRTQX_API rrtqx_status rrtqx_obstacle_add_sweep(rrtqx_edges *edges,
                                                const rrtqx_spheres *spheres,
                                                const int32_t *ob_ids,
                                                int64_t n_obs,
                                                double robot_radius,
                                                double delta, uint32_t flags,
                                                rrtqx_sweep_result **result);
/* removeObstacle (DRRT_Q.jl:3295-3362, DRRT.jl:3202-3268) geometric part for
 * ONE obstacle ob_id.  edge_dist_inf[e] = (edge.dist == Inf).  An edge is
 * "restored" if it is flagged, collides with ob_id and with none of the
 * obstacles in other_ids (the caller evaluates the reference's time-window
 * predicate :3330 to build that list).  QX behaviour (obstacle disabled before
 * the loop, nothing restored, SURVEY.md appendix B11) is the caller passing
 * RRTQX_SWEEP_REMOVED_INACTIVE. */
enum {
  RRTQX_SWEEP_REMOVED_INACTIVE = 16u,
  RRTQX_SWEEP_STATS = 32u /* add sweep: also count candidate nodes and (edge, obstacle) pairs (node-centric
                             kernel, slower); without it n_candidates / n_pair_tests are reported as -1 */
};
RRTQX_API rrtqx_status rrtqx_obstacle_remove_sweep(
    rrtqx_edges *edges, const rrtqx_spheres *spheres, int32_t ob_id,
    const int32_t *other_ids, int64_t n_others, const uint8_t *edge_dist_inf,
    double robot_radius, double delta, uint32_t flags,
    rrtqx_sweep_result **result);
RRTQX_API rrtqx_status rrtqx_sweep_result_destroy(rrtqx_sweep_result *r);
/* n_edge_hits = number of distinct edges reported (blocked / restored),
 * n_node_hits = number of distinct nodes reported (orphans / requeue),
 * n_candidates = sum over obstacles of candidate nodes (start-node filter),
 * n_pair_tests = (edge, obstacle) pairs that passed the start-node filter, the
 * "edge checks" unit of BASELINE.json (parent edges included). */
RRTQX_API rrtqx_status rrtqx_sweep_result_sizes(const rrtqx_sweep_result *r,
                                                int64_t *n_edge_hits,
                                                int64_t *n_node_hits,
                                                int64_t *n_candidates,
                                                int64_t *n_pair_tests);
/* ascending edge ids (n_edge_hits) and node ids (n_node_hits).  Pointers:
 * host or device, NULL ok. */
RRTQX_API rrtqx_status rrtqx_sweep_result_fetch(rrtqx_sweep_result *r,
                                                int32_t *edge_ids,
                                                int32_t *node_ids);
/* byte flags: edge_flag[e] (n_edges), node_flag[v] (nodes at edge upload). */
RRTQX_API rrtqx_status rrtqx_sweep_result_flags(rrtqx_sweep_result *r,
                                                uint8_t *edge_flag,
                                                uint8_t *node_flag);

/* ------------------------------------------- 2-D polygon world (DubinsEdge) */
/* Obstacle kinds 1 (ball) and 3 (polygon) of the Otte generation
 * (DRRT_data_structures.jl:135-265) flattened: kind[n], centres n x 2 and
 * radii n of the bounding circles (for polygons: bbox midpoint / farthest
 * vertex, :229-241, computed by the caller exactly as the constructor does),
 * active[n] = !(obstacleUnused || lifeSpan <= 0), polygon vertices as CSR
 * (vert_ptr[n+1] host array, verts nv x 2). */
RRTQX_API rrtqx_status rrtqx_polygons_create(rrtqx_ctx *ctx,
                                             rrtqx_polygons **out);
RRTQX_API rrtqx_status rrtqx_polygons_destroy(rrtqx_polygons *p);
RRTQX_API rrtqx_status rrtqx_polygons_upload(rrtqx_polygons *p,
                                             const int32_t *kind,
                                             const double *centers,
                                             const double *radii,
                                             const uint8_t *active,
                                             const int64_t *vert_ptr,
                                             const double *verts, int64_t n);
/* explicitEdgeCheck2D (DRRT.jl:1523-1578, via distanceSqrdPointToSegment
 * :1060-1083 and segmentDistSqrd :1144-1202) OR-ed over the obstacle list
 * (explicitEdgeCheck(C,edge) DRRT.jl:1660-1678) for n segments given by
 * starts/ends (n x 2) and the robot radius `radius`. */
RRTQX_API rrtqx_status rrtqx_segment_check_2d_batch(rrtqx_polygons *p,
                                                    const double *starts,
                                                    const double *ends,
                                                    int64_t n, double radius,
                                                    uint32_t flags,
                                                    uint8_t *collide_out);
/* Dubins explicitEdgeCheck(S, edge, ob) (DRRT_DubinsEdge_functions.jl:750-774)
 * OR-ed over the obstacle list: coarse start->end segment test with radius
 * robot_radius + 2*min_turn_radius, then every consecutive pair of trajectory
 * points with robot_radius.  Trajectories (edge.trajectory[:,1:2]) are a CSR:
 * traj_ptr[n_edges+1], traj_xy npts x 2.  Collision booleans are bit-exact
 * GIVEN the trajectory points (SURVEY.md appendix A14). */
RRTQX_API rrtqx_status rrtqx_dubins_edge_check_batch(
    rrtqx_polygons *p, const double *starts, const double *ends,
    const int64_t *traj_ptr, const double *traj_xy, int64_t n_edges,
    double robot_radius, double min_turn_radius, uint32_t flags,
    uint8_t *collide_out);

/* ------------------------------------- Otte / Dubins obstacle sweeps (DRRT.jl) */
/* addNewObstacle / removeObstacle of the Otte generation with DubinsEdge
 * (DRRT.jl:3127-3197, 3202-3268; candidates findPointsInConflictWithObstacle
 * :3048-3122; edge test = Dubins explicitEdgeCheck,
 * DRRT_DubinsEdge_functions.jl:750-774) over a resident edge set
 * (rrtqx_edges_upload / _append / _set_parents on a 4-D [x y t theta] tree with
 * the theta wrap, or a plain 2-D tree).
 *
 * The sweeps work on ITEMS: item e < n_edges is out-edge e (upload order),
 * item n_edges + v is the parent edge of node v (skipped when parent[v] < 0).
 * Every item needs its trajectory (edge.trajectory[:,1:2]) resident on the
 * device, as a CSR over the items: traj_ptr[n_edges + n_nodes + 1] (host or
 * device), traj_xy rows x 2.  Either upload the planner's own trajectories
 * (bit-exact booleans GIVEN the trajectory points, SURVEY.md appendix A14) ...*/
RRTQX_API rrtqx_status rrtqx_edges_set_trajectories(rrtqx_edges *e,
                                                    const int64_t *traj_ptr,
                                                    const double *traj_xy);
/* ... or have the device solve every item with calculateTrajectory
 * (DRRT_DubinsEdge_functions.jl:329-709; d == 4): start / end poses are the
 * resident node positions.  *n_rows_out = total trajectory rows.  Both calls
 * must be repeated after the edge set or the tree size change, and after a
 * rrtqx_edges_set_parents call that gives some node a parent (>= 0) other than
 * its current one, the first parents of an edge set uploaded without them
 * included; until then the sweeps fail with RRTQX_ERR_STATE.  Setting parents
 * to -1 keeps the trajectories valid: the item of a node without a parent edge
 * is never read. */
RRTQX_API rrtqx_status rrtqx_edges_solve_trajectories(rrtqx_edges *e,
                                                      double min_turn_radius,
                                                      int64_t *n_rows_out);
/* device views of the resident trajectories (RRTQX_ERR_STATE when none) */
RRTQX_API rrtqx_status rrtqx_edges_trajectories_device(
    const rrtqx_edges *e, const int64_t **traj_ptr, const double **traj_xy,
    int64_t *n_items, int64_t *n_rows);
/* copies them out: traj_ptr (n_items + 1) and traj_xy (n_rows x 2), host or
 * device destinations, either may be NULL */
RRTQX_API rrtqx_status rrtqx_edges_trajectories_fetch(rrtqx_edges *e,
                                                      int64_t *traj_ptr,
                                                      double *traj_xy);
/* Add sweep for obstacles ob_ids[0..n_obs) of `polygons` (treated as active,
 * DRRT.jl:3129).  For obstacle o the candidate nodes are
 *   kdFindWithinRange(KD, ((rho+delta)+radius_o)+pi, [x_o y_o 0.0 pi])  (d == 4)
 *   kdFindWithinRange(KD,  (rho+delta)+radius_o,     [x_o y_o])         (d == 2)
 * ghost identities of the wrapped heading included; out-edges of candidates
 * that collide are "blocked" (:3156-3158), candidates whose parent edge
 * collides are "orphans" (:3164-3177).  Result as rrtqx_obstacle_add_sweep
 * (n_candidates / n_pair_tests are reported as -1). */
RRTQX_API rrtqx_status rrtqx_obstacle_add_sweep_2d(
    rrtqx_edges *edges, const rrtqx_polygons *polygons, const int32_t *ob_ids,
    int64_t n_obs, double robot_radius, double delta, double min_turn_radius,
    uint32_t flags, rrtqx_sweep_result **result);
/* Remove sweep for ONE obstacle ob_id, Otte semantics (the obstacle is still
 * active while tested, :3228 vs :3267): a flagged edge (edge_dist_inf[e]) whose
 * start node is a candidate, that collides with ob_id and with none of
 * other_ids (the caller evaluates :3238) is "restored"; its start node is
 * reported for the LMC recompute. */
RRTQX_API rrtqx_status rrtqx_obstacle_remove_sweep_2d(
    rrtqx_edges *edges, const rrtqx_polygons *polygons, int32_t ob_id,
    const int32_t *other_ids, int64_t n_others, const uint8_t *edge_dist_inf,
    double robot_radius, double delta, double min_turn_radius, uint32_t flags,
    rrtqx_sweep_result **result);

/* ------------------------------------------------ Dubins solver on the device */
/* calculateTrajectory(S, edge::DubinsEdge), space without time
 * (DRRT_DubinsEdge_functions.jl:329-709; rightTurnDist / leftTurnDist
 * DRRT_distance_functions.jl:62-80) for n_edges edges: starts / goals are n x 4
 * rows [x y t theta] (edge.startNode.position / edge.endNode.position).
 * Produces per edge: dist (= edge.dist = edge.Wdist = edge.distOriginal; Inf
 * when no word applies), type (edge.dubinsType: 0 "rsl", 1 "rsr", 2 "rlr",
 * 3 "lsr", 4 "lsl", 5 "lrl", -1 "xxx") and edge.trajectory[:,1:2] as a CSR
 * (traj_ptr[n_edges+1], traj_xy n_rows x 2) that can be handed to
 * rrtqx_dubins_edge_check_batch without leaving the device.
 * *result may point to NULL (a result object is created) or to a result of an
 * earlier call (its buffers are reused).  Parity with the reference is by
 * tolerance (1e-9 relative; Julia libm and twice-precision ranges, SURVEY.md
 * appendix A14). */
RRTQX_API rrtqx_status rrtqx_dubins_trajectory_batch(
    rrtqx_ctx *ctx, const double *starts, const double *goals, int64_t n_edges,
    double min_turn_radius, rrtqx_dubins_result **result);
RRTQX_API rrtqx_status rrtqx_dubins_result_destroy(rrtqx_dubins_result *r);
RRTQX_API rrtqx_status rrtqx_dubins_result_sizes(const rrtqx_dubins_result *r,
                                                 int64_t *n_edges,
                                                 int64_t *n_rows);
/* copies to host or device arrays; any pointer may be NULL */
RRTQX_API rrtqx_status rrtqx_dubins_result_fetch(rrtqx_dubins_result *r,
                                                 double *dist, int32_t *type,
                                                 int64_t *traj_ptr,
                                                 double *traj_xy);
/* device views, valid until the next call that reuses the result */
RRTQX_API rrtqx_status rrtqx_dubins_result_device(
    const rrtqx_dubins_result *r, const double **dist, const int32_t **type,
    const int64_t **traj_ptr, const double **traj_xy);
/* saturate(newPoint, closestPoint, delta), DubinsEdge version
 * (DRRT_DubinsEdge_functions.jl:70-95, dist = R3SDist
 * DRRT_distance_functions.jl:41): in place on new_points (n x 4). */
RRTQX_API rrtqx_status rrtqx_dubins_saturate_batch(rrtqx_ctx *ctx,
                                                   double *new_points,
                                                   const double *closest,
                                                   int64_t n, double delta);

/* ------------------------------------------------------------ multi-GPU */
/* The path shards embarrassingly (SURVEY.md 8e): tree and obstacles are
 * replicated per GPU, rank g owns a contiguous slice of a batch, and the only
 * exchange is the gather of fixed-size results.  A communicator spans the
 * ranks of the job; this process drives n_local of them:
 *   rrtqx_comm_init_local -- ONE process holding one context per device (what
 *     a Julia host does; the reference is one process, rrtqx.jl:331).  When all
 *     devices have peer access the flag gather of the sharded check is fused
 *     into its packing kernel (direct stores into the peers' buffers over
 *     NVLink), otherwise NCCL gathers.
 *   rrtqx_comm_init_rank  -- one process per GPU (torchrun): every rank passes
 *     the 128-byte id rank 0 obtained from rrtqx_comm_unique_id (moved between
 *     the processes by the caller), its rank and the rank count.  Ranks of one
 *     node map each other's result windows through CUDA IPC (the handles
 *     travel over NCCL at init) and the gathers become direct stores into the
 *     peers' windows plus an epoch word per (destination, source); ranks on
 *     several nodes, RRTQX_COMM_NO_IPC=1 or parts larger than a window slot
 *     (RRTQX_COMM_IPC_MB, default 64): NCCL gathers.
 * NCCL (libnccl.so.2) is loaded on first use; without it these calls fail with
 * RRTQX_ERR_UNSUPPORTED and nothing else is affected. */
typedef struct rrtqx_comm rrtqx_comm;
RRTQX_API rrtqx_status rrtqx_comm_init_local(rrtqx_ctx *const *ctxs, int32_t n,
                                             rrtqx_comm **out);
RRTQX_API rrtqx_status rrtqx_comm_unique_id(void *id128);
RRTQX_API rrtqx_status rrtqx_comm_init_rank(rrtqx_ctx *ctx, const void *id128,
                                            int32_t rank, int32_t n_ranks,
                                            rrtqx_comm **out);
RRTQX_API rrtqx_status rrtqx_comm_destroy(rrtqx_comm *comm);
/* any output pointer may be NULL.  peer_stores = 1: the fused store path is
 * active.  nccl_version: NCCL_VERSION_CODE of the loaded library (0 when the
 * communicator has one rank and NCCL was never loaded). */
RRTQX_API rrtqx_status rrtqx_comm_info(const rrtqx_comm *comm, int32_t *n_ranks,
                                       int32_t *n_local, int32_t *first_rank,
                                       int32_t *peer_stores,
                                       int32_t *nccl_version);
/* All-gather of bytes_per_rank bytes per rank (fixed-size results: per-query
 * counts, nearest idx/dist): send[i] / recv[i] are device pointers of local
 * rank i, recv holds n_ranks * bytes_per_rank bytes in rank order.  Queued on
 * the contexts' streams, or (on_side_stream != 0) on the communicator's side
 * streams behind what the main streams hold so far, so that the next step does
 * not wait for it; rrtqx_comm_join makes the main streams wait for every
 * gather queued that way.  Asynchronous: synchronise the contexts to read. */
RRTQX_API rrtqx_status rrtqx_comm_allgather(rrtqx_comm *comm,
                                            const void *const *send,
                                            void *const *recv,
                                            int64_t bytes_per_rank,
                                            int32_t on_side_stream);
RRTQX_API rrtqx_status rrtqx_comm_join(rrtqx_comm *comm);
/* explicitEdgeCheck(S, edge) (DRRT_Q.jl:1802-1826) for ONE edge batch sharded
 * over the ranks: every rank holds the same device-resident edge list
 * (src[i] / dst[i], n_edges entries) next to its replica of the tree and the
 * obstacles; rank g checks the edges of word shard g and every rank ends up
 * with ALL flags, bit-packed: edge e is bit (e % 32) of word e / 32 of
 * packed_out[i] (device, rrtqx_comm_packed_words() words: G equal shards).
 * Blocking. */
RRTQX_API rrtqx_status rrtqx_comm_packed_words(const rrtqx_comm *comm,
                                               int64_t n_edges,
                                               int64_t *words_total,
                                               int64_t *words_per_rank);
RRTQX_API rrtqx_status rrtqx_edge_check_batch_sharded(
    rrtqx_comm *comm, rrtqx_tree *const *trees,
    const rrtqx_spheres *const *spheres, const int32_t *const *src,
    const int32_t *const *dst, int64_t n_edges, double robot_radius,
    uint32_t flags, uint32_t *const *packed_out);

#ifdef __cplusplus
}
#endif
#endif /* RRTQX_B200_H */
