// sweep2d.cu -- obstacle add / remove sweeps of the Otte generation with DubinsEdge (DRRT.jl):
//   findPointsInConflictWithObstacle   DRRT.jl:3048-3122   (kinds 1-5, space without time)
//   addNewObstacle                     DRRT.jl:3127-3197
//   removeObstacle                     DRRT.jl:3202-3268
//   edge test = Dubins explicitEdgeCheck(S, edge, ob)  DRRT_DubinsEdge_functions.jl:750-774
// over the resident edge set (out-edges in upload order followed by one parent edge per node) and its resident
// trajectories (uploaded edge.trajectory rows, or solved on the device by the Dubins solver of dubins.cu).
//
// Candidate rule.  The reference tests only the out-edges / parent edge of the nodes that
// kdFindWithinRange(KD, searchRange, centre) returns, with
//     searchRange = ((rho + delta) + ob.radius) + pi,  centre = [ob.x ob.y 0.0 pi]     (spaceHasTheta, :3061-3064)
//     searchRange =  (rho + delta) + ob.radius,        centre = ob.position             (plain 2-D,     :3058-3059)
// over the theta-wrapped tree, i.e. node v is a candidate iff  euclid(centre, v) < searchRange  (root: <=,
// kdTree_general.jl:896-898) or  euclid(ghost(centre), v) < searchRange  when the ghost identity is used
// (ghostPoint.jl:60-111).  The membership is evaluated per (item, obstacle) from the start node's position with the
// exact radicand test s < T_lt(searchRange); it is the same set the device range query returns.
//
// One warp per item; the obstacle loop is dubins_collide_warp (polygon.cuh), whose selector carries the
// start-node filter.  Only the geometric decisions are made here; the caller applies the list surgery.
#include "objects.cuh"
#include "polygon.cuh"

namespace rrtqx {

// range.cu's ghost construction, restated for one wrap dimension (ghostPoint.jl:76-104)
struct Sweep2dFilter {  // per listed obstacle
  double q[4];          // real identity of the query centre
  double g[4];          // ghost identity (valid when ghost_used)
  double T, sr;         // T_lt(searchRange), searchRange
  int ghost_used;
  int pad;
};

__global__ void sweep2d_table_kernel(PolyView P, const int32_t *__restrict__ ids, int n, int has_theta, WrapInfo wrap,
                                     double robot_radius, double delta, Sweep2dFilter *__restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int o = ids[k];
  const double2 c = P.center[o];
  Sweep2dFilter f;
  double sr = __dadd_rn(__dadd_rn(robot_radius, delta), P.radius[o]);  // left to right, DRRT.jl:3058
  f.q[0] = c.x; f.q[1] = c.y; f.q[2] = 0.0; f.q[3] = 0.0;
  if (has_theta) {
    sr = __dadd_rn(sr, 3.141592653589793);                             // + pi, :3062
    f.q[3] = 3.141592653589793;                                        // [x y 0.0 pi], :3063
  }
  f.sr = sr;
  f.T = sqrt_thresh_lt(sr);
  f.ghost_used = 0;
  for (int d = 0; d < 4; ++d) f.g[d] = f.q[d];
  if (wrap.num_wraps == 1) {  // getNextGhostPoint for one wrap dimension
    const int dim = wrap.wraps[0];
    const double Pw = wrap.wrap_points[0];
    double gv, cv;
    if (f.q[dim] < Pw / 2.0) { gv = __dadd_rn(f.q[dim], Pw); cv = Pw; }   // ghostPoint.jl:82-85
    else                     { gv = __dsub_rn(f.q[dim], Pw); cv = 0.0; }  // :86-89
    f.g[dim] = gv;
    // the ghost is used iff !(dist(closestUnwrappedPoint, ghost) > bestDist) (:104); they differ in `dim` only
    const double dd = __dsub_rn(cv, gv);
    f.ghost_used = !(__dsqrt_rn(__dmul_rn(dd, dd)) > sr) ? 1 : 0;
  }
  f.pad = 0;
  out[k] = f;
}

template <int D>
__device__ __forceinline__ bool sweep2d_candidate(const Sweep2dFilter &f, const double4 &p, int v) {
  const double s = sqdist<D>(f.q, p.x, p.y, p.z, p.w);
  if (s < f.T) return true;
  if (v == 0 && __dsqrt_rn(s) <= f.sr) return true;  // root admitted with <= by the real identity
  return f.ghost_used && sqdist<D>(f.g, p.x, p.y, p.z, p.w) < f.T;
}

template <int D>
struct ListedObstacles {  // the obstacles of the call, each with the start-node filter of the item's start node
  const int32_t *ids;
  const Sweep2dFilter *filt;  // nullptr: no filter (the "other obstacles" of removeObstacle)
  int n;
  double4 pv;
  int v;
  __device__ __forceinline__ int count() const { return n; }
  __device__ __forceinline__ int id(int k) const { return ids[k]; }
  __device__ __forceinline__ bool admit(int k) const { return !filt || sweep2d_candidate<D>(filt[k], pv, v); }
};

constexpr int SWEEP2D_BLOCKS_PER_SM = 6;  // as DUBINS_CHECK_BLOCKS_PER_SM (polygon.cu): latency-bound FP64 chains, 48 warps per SM (16.7 -> 10.5 ms on the C4 graph)
constexpr int SWEEP2D_SELECT_MAX_OBS = 8;  // more listed obstacles admit nearly every item: no list
// Few listed obstacles (the planner's call: ONE): the start-node filter admits a few per cent of the items, so a
// thread-per-item pass lists them first and the warp-per-item kernels below run over that list only (a device-side
// count, persistent warps) instead of spending a warp on every item of the graph.
// MODE 0: addNewObstacle items (out-edges, then parent edges), any of the n_f filters; MODE 1: removeObstacle edges
// (edge.dist == Inf only), filter 0.
template <int D, int MODE>
__global__ void __launch_bounds__(256)
sweep2d_select_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src, int64_t n_edges,
                      const int32_t *__restrict__ parent, const uint8_t *__restrict__ edge_dist_inf,
                      const Sweep2dFilter *__restrict__ filt, int n_f, int32_t *__restrict__ cand, int32_t *__restrict__ n_cand) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t items = MODE == 0 ? n_edges + n_nodes : n_edges;
  bool keep = false;
  if (i < items) {
    int v;
    bool live = true;
    if (i >= n_edges) { v = (int)(i - n_edges); live = parent && parent[v] >= 0; }
    else { v = src[i]; if (MODE == 1) live = edge_dist_inf[i] != 0; }
    if (live) {
      const double4 a = pos[v];
      for (int k = 0; k < n_f && !keep; ++k) keep = sweep2d_candidate<D>(filt[k], a, v);
    }
  }
  const unsigned m = __ballot_sync(FULL, keep);
  if (m) {
    int base = 0;
    if (lane_id() == 0) base = atomicAdd(n_cand, __popc(m));
    base = __shfl_sync(FULL, base, 0);
    if (keep) cand[base + __popc(m & lanemask_lt())] = (int32_t)i;
  }
}

// addNewObstacle: item i < n_edges is out-edge i (src[i] -> dst[i]); item n_edges + v is the parent edge of node v.
// cand == nullptr: one warp per item of the graph; otherwise persistent warps over the listed items.
template <int D>
__global__ void __launch_bounds__(256, SWEEP2D_BLOCKS_PER_SM)
add_sweep_2d_kernel(PolyView P, const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                    const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
                    const int64_t *__restrict__ tptr, const double *__restrict__ traj, const int32_t *__restrict__ ids,
                    const Sweep2dFilter *__restrict__ filt, int n_obs, double rho, double rho_coarse,
                    uint8_t *__restrict__ edge_flag, uint8_t *__restrict__ node_flag,
                    const int32_t *__restrict__ cand, const int32_t *__restrict__ n_cand) {
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_w = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t total = cand ? (int64_t)*n_cand : n_edges + n_nodes;
  for (int64_t k = w0; k < total; k += n_w) {
    const int64_t i = cand ? (int64_t)cand[k] : k;
    int v, w;
    if (i >= n_edges) {
      v = (int)(i - n_edges);
      w = parent ? parent[v] : -1;
      if (w < 0) continue;  // !rrtParentUsed (:3164)
    } else {
      v = src[i];
      w = dst[i];
    }
    const double4 a = pos[v], b = pos[w];
    const ListedObstacles<D> sel{ids, filt, n_obs, a, v};
    // the obstacles of an add sweep count as active (ob.obstacleUnused = false, :3129)
    const bool hit = dubins_collide_warp(P, true, sel, a.x, a.y, b.x, b.y, traj, tptr[i], tptr[i + 1], rho, rho_coarse);
    if (hit && lane_id() == 0) {
      if (i >= n_edges) node_flag[v] = 1;  // :3164-3177 orphan
      else edge_flag[i] = 1;               // :3156-3158 edge.dist = Inf
    }
  }
}

// removeObstacle: ids[0] = the removed obstacle (still active while tested, :3228 vs :3267), ids[1..] = the others.
template <int D>
__global__ void __launch_bounds__(256, SWEEP2D_BLOCKS_PER_SM)
remove_sweep_2d_kernel(PolyView P, const double4 *__restrict__ pos, const int32_t *__restrict__ src,
                       const int32_t *__restrict__ dst, int64_t n_edges, const uint8_t *__restrict__ edge_dist_inf,
                       const int64_t *__restrict__ tptr, const double *__restrict__ traj, const int32_t *__restrict__ ids,
                       const Sweep2dFilter *__restrict__ filt, int n_ids, double rho, double rho_coarse,
                       uint8_t *__restrict__ edge_flag, uint8_t *__restrict__ node_flag,
                       const int32_t *__restrict__ cand, const int32_t *__restrict__ n_cand) {
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_w = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t total = cand ? (int64_t)*n_cand : n_edges;
  for (int64_t k = w0; k < total; k += n_w) {
    const int64_t e = cand ? (int64_t)cand[k] : k;
    if (!edge_dist_inf[e]) continue;  // neighborEdge.dist == Inf (:3228)
    const int v = src[e], w = dst[e];
    const double4 a = pos[v], b = pos[w];
    const ListedObstacles<D> removed{ids, filt, 1, a, v};
    if (!dubins_collide_warp(P, true, removed, a.x, a.y, b.x, b.y, traj, tptr[e], tptr[e + 1], rho, rho_coarse)) continue;
    const ListedObstacles<D> others{ids + 1, nullptr, n_ids - 1, a, v};  // :3234-3246
    if (dubins_collide_warp(P, true, others, a.x, a.y, b.x, b.y, traj, tptr[e], tptr[e + 1], rho, rho_coarse)) continue;
    if (lane_id() == 0) {  // :3249-3264
      edge_flag[e] = 1;
      node_flag[v] = 1;
    }
  }
}

// items -> Dubins solver inputs: [x y t theta] of the start and of the end node (rows of 4 doubles); a node without
// parent edge gets a zero-length item that the sweeps never read
__global__ void sweep2d_gather_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                                      const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
                                      double *__restrict__ starts, double *__restrict__ goals) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_edges + n_nodes) return;
  int v, w;
  if (i >= n_edges) {
    v = (int)(i - n_edges);
    w = parent ? parent[v] : -1;
    if (w < 0) w = v;
  } else {
    v = src[i];
    w = dst[i];
  }
  const double4 a = pos[v], b = pos[w];
  reinterpret_cast<double4 *>(starts)[i] = a;
  reinterpret_cast<double4 *>(goals)[i] = b;
}

static int64_t sweep2d_items(rrtqx_edges *E) {
  if (E->dirty || E->tree->n != E->n_nodes) edges_rebuild(E);  // appended edges / parents / new nodes
  return E->n_edges + E->n_nodes;
}

void edges_set_trajectories(rrtqx_edges *E, const int64_t *traj_ptr, const double *traj_xy) {
  rrtqx_ctx *ctx = E->tree->ctx;
  cudaStream_t st = ctx->stream;
  const int64_t items = sweep2d_items(E);
  RQ_REQUIRE(traj_ptr != nullptr, "traj_ptr is NULL");
  int64_t rows = 0;
  if (is_device_ptr(traj_ptr)) RQ_CUDA(cudaMemcpy(&rows, traj_ptr + items, sizeof(int64_t), cudaMemcpyDeviceToHost));
  else {
    for (int64_t i = 0; i < items; ++i) RQ_REQUIRE(traj_ptr[i] <= traj_ptr[i + 1] && traj_ptr[i] >= 0, "traj_ptr must be non-decreasing");
    rows = traj_ptr[items];
  }
  RQ_REQUIRE(rows >= 0 && (rows == 0 || traj_xy), "bad trajectory arrays");
  E->traj_ptr.ensure((size_t)items + 1, st);
  E->traj_xy.ensure((size_t)rows * 2 + 2, st);
  RQ_CUDA(cudaMemcpyAsync(E->traj_ptr.p, traj_ptr, sizeof(int64_t) * (items + 1), cudaMemcpyDefault, st));
  if (rows) RQ_CUDA(cudaMemcpyAsync(E->traj_xy.p, traj_xy, sizeof(double) * 2 * rows, cudaMemcpyDefault, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  E->traj_items = items;
  E->traj_rows = rows;
  E->d_traj_ptr = E->traj_ptr.p;
  E->d_traj_xy = E->traj_xy.p;
}

void edges_solve_trajectories(rrtqx_edges *E, double min_turn_radius) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(t->d == 4, "the Dubins solver needs [x y t theta] positions (d == 4)");
  const int64_t items = sweep2d_items(E);
  E->traj_items = -1;
  if (items == 0) { E->traj_items = 0; E->traj_rows = 0; return; }
  E->solve_starts.ensure((size_t)items * 4, st);
  E->solve_goals.ensure((size_t)items * 4, st);
  sweep2d_gather_kernel<<<div_up(items, 256), 256, 0, st>>>(t->pos.p, E->n_nodes, E->src.p, E->dst.p, E->n_edges,
                                                            E->has_parent ? E->parent.p : nullptr, E->solve_starts.p,
                                                            E->solve_goals.p);
  post_launch(ctx);
  const rrtqx_status rc = rrtqx_dubins_trajectory_batch(ctx, E->solve_starts.p, E->solve_goals.p, items, min_turn_radius, &E->solved);
  if (rc != RRTQX_OK) throw Error(rc, ctx->err);
  const int64_t *dptr = nullptr;
  const double *dxy = nullptr;
  int64_t n_e = 0, n_rows = 0;
  rrtqx_dubins_result_device(E->solved, nullptr, nullptr, &dptr, &dxy);
  rrtqx_dubins_result_sizes(E->solved, &n_e, &n_rows);
  E->d_traj_ptr = dptr;
  E->d_traj_xy = dxy;
  E->traj_items = items;
  E->traj_rows = n_rows;
}

static void sweep2d_prepare(rrtqx_edges *E, const rrtqx_polygons *Pg, const int32_t *ids_host, int64_t n_ids,
                            double robot_radius, double delta, rrtqx_sweep_result *R) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(Pg->ctx == ctx, "obstacle set belongs to another context");
  RQ_REQUIRE(t->d == 2 || t->d == 4, "the Otte / Dubins sweeps need a 2-D ([x y]) or a Dubins ([x y t theta]) tree");
  RQ_REQUIRE(t->wrap.num_wraps <= 1, "at most one wrap-around dimension (the Dubins heading)");
  const int64_t items = sweep2d_items(E);
  if (E->traj_items != items)
    throw Error(RRTQX_ERR_STATE, "trajectories are not resident for the current edge set "
                                 "(rrtqx_edges_set_trajectories / rrtqx_edges_solve_trajectories after the last change)");
  for (int64_t i = 0; i < n_ids; ++i) RQ_REQUIRE(ids_host[i] >= 0 && ids_host[i] < Pg->n, "obstacle id out of range");
  R->ids_stage2.ensure((size_t)n_ids + 1, st);
  R->filt2d.ensure((size_t)n_ids * sizeof(Sweep2dFilter) + 16, st);
  R->cand2d.ensure((size_t)items + 1, st);   // candidate list of the two-stage form (grow-only: allocated once per graph size)
  R->cand2d_n.ensure(4, st);
  if (n_ids) {
    RQ_CUDA(cudaMemcpyAsync(R->ids_stage2.p, ids_host, sizeof(int32_t) * n_ids, cudaMemcpyHostToDevice, st));
    RQ_CUDA(cudaStreamSynchronize(st));  // ids_host may be a temporary of the caller
    sweep2d_table_kernel<<<div_up(n_ids, 128), 128, 0, st>>>(Pg->view(), R->ids_stage2.p, (int)n_ids, t->d == 4 ? 1 : 0, t->wrap,
                                                             robot_radius, delta, (Sweep2dFilter *)R->filt2d.p);
    post_launch(ctx);
  }
}

void obstacle_add_sweep_2d(rrtqx_edges *E, const rrtqx_polygons *Pg, const int32_t *ob_ids, int64_t n_obs,
                           double robot_radius, double delta, double min_turn_radius, uint32_t flags,
                           rrtqx_sweep_result *R) {
  (void)flags;
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(n_obs >= 0 && n_obs < (1 << 24), "n_obs out of range");
  std::vector<int32_t> ids((size_t)n_obs);
  if (n_obs) {
    if (is_device_ptr(ob_ids)) RQ_CUDA(cudaMemcpy(ids.data(), ob_ids, sizeof(int32_t) * n_obs, cudaMemcpyDeviceToHost));
    else memcpy(ids.data(), ob_ids, sizeof(int32_t) * n_obs);
  }
  sweep2d_prepare(E, Pg, ids.data(), n_obs, robot_radius, delta, R);
  PhaseScope ph(ctx, "add_sweep_2d");
  sweep_prepare_result(E, R);
  const int64_t items = E->n_edges + E->n_nodes;
  if (n_obs > 0 && items > 0) {
    const double rho_coarse = robot_radius + 2 * min_turn_radius;  // DRRT_DubinsEdge_functions.jl:758
    const int32_t *par = E->has_parent ? E->parent.p : nullptr;
    // few obstacles: list the admitted items first (thread per item), then persistent warps over the list
    const bool two_stage = n_obs <= SWEEP2D_SELECT_MAX_OBS && items < ((int64_t)1 << 31);
    const int32_t *cand = nullptr, *n_cand = nullptr;
    unsigned blocks = (unsigned)div_up(items * 32, 256);
    if (two_stage) {
      RQ_CUDA(cudaMemsetAsync(R->cand2d_n.p, 0, sizeof(int32_t), st));
      if (t->d == 4)
        sweep2d_select_kernel<4, 0><<<(unsigned)div_up(items, 256), 256, 0, st>>>(t->pos.p, E->n_nodes, E->src.p, E->n_edges, par, nullptr,
                                                                               (const Sweep2dFilter *)R->filt2d.p, (int)n_obs, R->cand2d.p, R->cand2d_n.p);
      else
        sweep2d_select_kernel<2, 0><<<(unsigned)div_up(items, 256), 256, 0, st>>>(t->pos.p, E->n_nodes, E->src.p, E->n_edges, par, nullptr,
                                                                               (const Sweep2dFilter *)R->filt2d.p, (int)n_obs, R->cand2d.p, R->cand2d_n.p);
      post_launch(ctx);
      cand = R->cand2d.p;
      n_cand = R->cand2d_n.p;
      blocks = (unsigned)std::min<int64_t>(blocks, (int64_t)ctx->sm_count * SWEEP2D_BLOCKS_PER_SM);
    }
#define RQ_ADD2D(D_)                                                                                                   \
  add_sweep_2d_kernel<D_><<<blocks, 256, 0, st>>>(Pg->view(), t->pos.p, E->n_nodes, E->src.p, E->dst.p, E->n_edges, par, \
                                                  E->d_traj_ptr, E->d_traj_xy, R->ids_stage2.p,                        \
                                                  (const Sweep2dFilter *)R->filt2d.p, (int)n_obs, robot_radius,        \
                                                  rho_coarse, R->edge_flag.p, R->node_flag.p, cand, n_cand)
    if (t->d == 4) RQ_ADD2D(4); else RQ_ADD2D(2);
#undef RQ_ADD2D
    post_launch(ctx);
  }
  sweep_finish(ctx, R);
  R->n_candidates = -1;
  R->n_pair_tests = -1;
}

void obstacle_remove_sweep_2d(rrtqx_edges *E, const rrtqx_polygons *Pg, int32_t ob_id, const int32_t *other_ids,
                              int64_t n_others, const uint8_t *edge_dist_inf, double robot_radius, double delta,
                              double min_turn_radius, uint32_t flags, rrtqx_sweep_result *R) {
  (void)flags;
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(n_others >= 0 && n_others < (1 << 24), "n_others out of range");
  RQ_REQUIRE(edge_dist_inf != nullptr || E->n_edges == 0, "edge_dist_inf is NULL");
  std::vector<int32_t> ids((size_t)n_others + 1);
  ids[0] = ob_id;
  if (n_others) {
    if (is_device_ptr(other_ids)) RQ_CUDA(cudaMemcpy(ids.data() + 1, other_ids, sizeof(int32_t) * n_others, cudaMemcpyDeviceToHost));
    else memcpy(ids.data() + 1, other_ids, sizeof(int32_t) * n_others);
  }
  sweep2d_prepare(E, Pg, ids.data(), (int64_t)ids.size(), robot_radius, delta, R);
  const uint8_t *dinf = to_device(ctx, edge_dist_inf, (size_t)E->n_edges, R->inf_stage);
  PhaseScope ph(ctx, "remove_sweep_2d");
  sweep_prepare_result(E, R);
  if (E->n_edges > 0) {
    const double rho_coarse = robot_radius + 2 * min_turn_radius;
    // the removed obstacle's filter admits a few per cent of the edges: list them first, then persistent warps
    const bool two_stage = E->n_edges < ((int64_t)1 << 31);
    const int32_t *cand = nullptr, *n_cand = nullptr;
    unsigned blocks = (unsigned)div_up(E->n_edges * 32, 256);
    if (two_stage) {
      RQ_CUDA(cudaMemsetAsync(R->cand2d_n.p, 0, sizeof(int32_t), st));
      if (t->d == 4)
        sweep2d_select_kernel<4, 1><<<(unsigned)div_up(E->n_edges, 256), 256, 0, st>>>(t->pos.p, E->n_nodes, E->src.p, E->n_edges, nullptr, dinf,
                                                                                    (const Sweep2dFilter *)R->filt2d.p, 1, R->cand2d.p, R->cand2d_n.p);
      else
        sweep2d_select_kernel<2, 1><<<(unsigned)div_up(E->n_edges, 256), 256, 0, st>>>(t->pos.p, E->n_nodes, E->src.p, E->n_edges, nullptr, dinf,
                                                                                    (const Sweep2dFilter *)R->filt2d.p, 1, R->cand2d.p, R->cand2d_n.p);
      post_launch(ctx);
      cand = R->cand2d.p;
      n_cand = R->cand2d_n.p;
      blocks = (unsigned)std::min<int64_t>(blocks, (int64_t)ctx->sm_count * SWEEP2D_BLOCKS_PER_SM);
    }
#define RQ_REM2D(D_)                                                                                                  \
  remove_sweep_2d_kernel<D_><<<blocks, 256, 0, st>>>(Pg->view(), t->pos.p, E->src.p, E->dst.p, E->n_edges, dinf,     \
                                                     E->d_traj_ptr, E->d_traj_xy, R->ids_stage2.p,                   \
                                                     (const Sweep2dFilter *)R->filt2d.p, (int)ids.size(),            \
                                                     robot_radius, rho_coarse, R->edge_flag.p, R->node_flag.p, cand, n_cand)
    if (t->d == 4) RQ_REM2D(4); else RQ_REM2D(2);
#undef RQ_REM2D
    post_launch(ctx);
  }
  sweep_finish(ctx, R);
  R->n_candidates = -1;
  R->n_pair_tests = -1;
}

}  // namespace rrtqx
