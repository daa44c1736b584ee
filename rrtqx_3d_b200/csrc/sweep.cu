// sweep.cu -- resident out-edge lists and the obstacle add / remove sweeps
// (addNewObstacle DRRT_Q.jl:3220-3290, removeObstacle :3295-3362,
// findPointsInConflictWithObstacle :3195-3215).
//
// Only the geometric decisions are made here; the Julia side applies the list
// surgery (edge.dist = Inf, orphaning, queue pushes) to the returned id sets.
#include "objects.cuh"
#include "scan.cuh"
#include "collide_queue.cuh"

namespace rrtqx {

// ------------------------------------------------------------ CSR build
__global__ void edge_hist_kernel(const int32_t *__restrict__ src, int64_t ne, int32_t *__restrict__ cnt) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < ne) atomicAdd(&cnt[src[e]], 1);
}
__global__ void edge_scatter_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t ne,
                                    const int32_t *__restrict__ row_ptr, int32_t *__restrict__ cursor,
                                    int32_t *__restrict__ csr_eid) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  int v = src[e];
  csr_eid[row_ptr[v] + atomicAdd(&cursor[v], 1)] = (int32_t)e;
}
// per row: ascending edge id (deterministic), then dst and the node's cull data
__global__ void edge_rows_kernel(const double4 *__restrict__ pos, const int32_t *__restrict__ dst,
                                 const int32_t *__restrict__ row_ptr, int32_t *__restrict__ csr_eid,
                                 int32_t *__restrict__ csr_dst, const int32_t *__restrict__ parent, int64_t n_nodes,
                                 double *__restrict__ lmax, uint8_t *__restrict__ degenerate) {
  int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_nodes) return;
  int a = row_ptr[v], b = row_ptr[v + 1];
  if (b - a <= 256)
    for (int i = a + 1; i < b; ++i) {
      int x = csr_eid[i];
      int j = i - 1;
      while (j >= a && csr_eid[j] > x) { csr_eid[j + 1] = csr_eid[j]; --j; }
      csr_eid[j + 1] = x;
    }
  double4 p = pos[v];
  double lm = 0.0;
  bool degen = false;
  for (int i = a; i < b; ++i) {
    int w = dst[csr_eid[i]];
    csr_dst[i] = w;
    double4 q = pos[w];
    SegPre s = seg_prepare(p.x, p.y, p.z, q.x, q.y, q.z);
    if (!s.cullable) degen = true; else lm = fmax(lm, s.len);
  }
  if (parent && parent[v] >= 0) {
    double4 q = pos[parent[v]];
    SegPre s = seg_prepare(p.x, p.y, p.z, q.x, q.y, q.z);
    if (!s.cullable) degen = true; else lm = fmax(lm, s.len);
  }
  lmax[v] = lm;
  degenerate[v] = degen ? 1 : 0;
}

// (Re)build the CSR by start node and the per-node cull data from the resident src / dst / parent arrays for
// the CURRENT tree size.  Runs on the device; called lazily by the sweeps after appends / parent updates.
void edges_rebuild(rrtqx_edges *E) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  const int64_t ne = E->n_edges, nn = t->n;
  RQ_REQUIRE(nn >= E->n_nodes, "the tree shrank under a resident edge set");
  E->csr_dst.ensure((size_t)ne + 1, st);
  E->csr_eid.ensure((size_t)ne + 1, st);
  E->row_ptr.ensure((size_t)nn + 2, st);
  E->cursor.ensure((size_t)nn + 2, st);
  E->lmax.ensure((size_t)nn + 1, st);
  E->degenerate.ensure((size_t)nn + 1, st);
  if (E->has_parent && nn > E->n_parent) {  // nodes inserted since the last parent update: no parent edge yet
    E->parent.ensure((size_t)nn + 1, st, (size_t)E->n_parent);
    RQ_CUDA(cudaMemsetAsync(E->parent.p + E->n_parent, 0xff, sizeof(int32_t) * (size_t)(nn - E->n_parent), st));
    E->n_parent = nn;
  }
  E->n_nodes = nn;
  const int TB = 256;
  RQ_CUDA(cudaMemsetAsync(E->cursor.p, 0, sizeof(int32_t) * ((size_t)nn + 1), st));
  if (ne) { edge_hist_kernel<<<div_up(ne, TB), TB, 0, st>>>(E->src.p, ne, E->cursor.p); post_launch(ctx); }
  exclusive_scan<int32_t, int32_t>(ctx, E->cursor.p, nn, E->row_ptr.p, E->scan_tmp);
  RQ_CUDA(cudaMemsetAsync(E->cursor.p, 0, sizeof(int32_t) * ((size_t)nn + 1), st));
  if (ne) {
    edge_scatter_kernel<<<div_up(ne, TB), TB, 0, st>>>(E->src.p, E->dst.p, ne, E->row_ptr.p, E->cursor.p, E->csr_eid.p);
    post_launch(ctx);
  }
  if (nn) {
    edge_rows_kernel<<<div_up(nn, TB), TB, 0, st>>>(t->pos.p, E->dst.p, E->row_ptr.p, E->csr_eid.p, E->csr_dst.p,
                                                    E->has_parent ? E->parent.p : nullptr, nn, E->lmax.p, E->degenerate.p);
    post_launch(ctx);
  }
  if (t->d == 3 && ne + nn > 0) {  // per-item records of the two-stage sphere-world kernels: one pass over the node table
    E->item_frec.ensure((size_t)(ne + nn) + 1, st);
    E->item_exact.ensure(3 * (size_t)(ne + nn) + 3, st);
    item_records_kernel<<<div_up(ne + nn, TB), TB, 0, st>>>(t->pos.p, nn, E->src.p, E->dst.p, ne,
                                                            E->has_parent ? E->parent.p : nullptr, E->item_frec.p, E->item_exact.p);
    post_launch(ctx);
    // and the items sorted by midpoint cell for the obstacle-centric kernels (item_grid.cuh)
    item_grid_build_levels(ctx, E->igrid, E->igrid1, t->pos.p, nn, E->src.p, E->dst.p, ne, E->has_parent ? E->parent.p : nullptr);
  } else {
    E->igrid.valid = false;
  }
  E->dirty = false;
}

__global__ void validate_endpoints_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t ne,
                                          int64_t nn, int32_t *__restrict__ bad) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= ne) return;
  const int a = src[e], b = dst[e];
  if (a < 0 || a >= nn || b < 0 || b >= nn) atomicAdd(bad, 1);
}

// Host arrays are checked on the host, device arrays by a small kernel: a bad index fails the call with
// RRTQX_ERR_INVALID before it can reach the histogram atomics or the position gathers.
static void validate_endpoints(rrtqx_tree *t, const int32_t *src, const int32_t *dst, int64_t ne, int64_t nn) {
  if (!ne) return;
  if (!is_device_ptr(src) && !is_device_ptr(dst)) {
    for (int64_t e = 0; e < ne; ++e)
      RQ_REQUIRE(src[e] >= 0 && src[e] < nn && dst[e] >= 0 && dst[e] < nn, "edge endpoint out of range");
    return;
  }
  RQ_REQUIRE(is_device_ptr(src) && is_device_ptr(dst), "src and dst must both be host or both be device arrays");
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  t->flagbuf.ensure(8, st);
  RQ_CUDA(cudaMemsetAsync(t->flagbuf.p, 0, sizeof(int32_t), st));
  validate_endpoints_kernel<<<div_up(ne, 256), 256, 0, st>>>(src, dst, ne, nn, t->flagbuf.p);
  post_launch(ctx);
  int32_t bad = 0;
  RQ_CUDA(cudaMemcpyAsync(&bad, t->flagbuf.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  RQ_REQUIRE(bad == 0, "edge endpoint out of range");
}

void edges_upload(rrtqx_edges *E, const int32_t *src, const int32_t *dst, int64_t ne, const int32_t *parent,
                  int64_t n_parent) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(ne >= 0 && ne < (int64_t)0x7fffffff, "n_edges out of range");
  E->traj_items = -1;  // resident trajectories belong to the previous edge set
  const int64_t nn = t->n;
  RQ_REQUIRE(parent == nullptr || n_parent == nn, "parent array must have one entry per tree node");
  validate_endpoints(t, src, dst, ne, nn);
  E->n_edges = ne;
  E->n_nodes = 0;
  E->has_parent = parent != nullptr;
  E->n_parent = parent ? nn : 0;
  E->src.ensure((size_t)ne + 1, st);
  E->dst.ensure((size_t)ne + 1, st);
  E->parent.ensure((size_t)nn + 1, st);
  if (ne) {
    RQ_CUDA(cudaMemcpyAsync(E->src.p, src, sizeof(int32_t) * ne, cudaMemcpyDefault, st));
    RQ_CUDA(cudaMemcpyAsync(E->dst.p, dst, sizeof(int32_t) * ne, cudaMemcpyDefault, st));
  }
  if (parent) RQ_CUDA(cudaMemcpyAsync(E->parent.p, parent, sizeof(int32_t) * nn, cudaMemcpyDefault, st));
  edges_rebuild(E);
  RQ_CUDA(cudaStreamSynchronize(st));
}

// Neighbour-graph residency (SURVEY 8f-2): the planner appends the edges it creates per iteration
// (makeNeighborOf / makeInitialOutNeighborOf, DRRT_Q.jl:2589-2593; edge id = position, continuing the upload
// order) and re-points parent edges (makeParentOf :1841-1856) without re-uploading the graph.  The CSR is
// rebuilt on the device before the next sweep.
void edges_append(rrtqx_edges *E, const int32_t *src, const int32_t *dst, int64_t n_new) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(n_new >= 0 && E->n_edges + n_new < (int64_t)0x7fffffff, "n_edges out of range");
  if (n_new == 0) return;
  validate_endpoints(t, src, dst, n_new, t->n);
  const size_t old = (size_t)E->n_edges;
  E->src.ensure(old + (size_t)n_new + 1, st, old);
  E->dst.ensure(old + (size_t)n_new + 1, st, old);
  RQ_CUDA(cudaMemcpyAsync(E->src.p + old, src, sizeof(int32_t) * n_new, cudaMemcpyDefault, st));
  RQ_CUDA(cudaMemcpyAsync(E->dst.p + old, dst, sizeof(int32_t) * n_new, cudaMemcpyDefault, st));
  E->n_edges += n_new;
  E->dirty = true;
  RQ_CUDA(cudaStreamSynchronize(st));  // the caller's arrays may be reused on return
}

// flags[0]: entries out of range; flags[1]: some node got a parent edge (p >= 0) other than the one it had
__global__ void parent_scatter_kernel(const int32_t *__restrict__ nodes, const int32_t *__restrict__ parents, int64_t n,
                                      int64_t n_nodes, int32_t *__restrict__ parent, int32_t *__restrict__ flags) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int v = nodes[i], p = parents[i];
  if (v < 0 || v >= n_nodes || p < -1 || p >= n_nodes) { atomicAdd(&flags[0], 1); return; }
  if (p >= 0 && parent[v] != p) flags[1] = 1;
  parent[v] = p;  // -1: rrtParentUsed = false
}

void edges_set_parents(rrtqx_edges *E, const int32_t *nodes, const int32_t *parents, int64_t n) {
  rrtqx_tree *t = E->tree;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(n >= 0 && (n == 0 || (nodes && parents)), "bad arguments");
  const int64_t nn = t->n;
  if (!E->has_parent) {  // first parent information: every node starts without a parent edge
    E->parent.ensure((size_t)nn + 1, st);
    RQ_CUDA(cudaMemsetAsync(E->parent.p, 0xff, sizeof(int32_t) * ((size_t)nn + 1), st));
    E->has_parent = true;
    E->n_parent = nn;
  } else if (nn > E->n_parent) {
    E->parent.ensure((size_t)nn + 1, st, (size_t)E->n_parent);
    RQ_CUDA(cudaMemsetAsync(E->parent.p + E->n_parent, 0xff, sizeof(int32_t) * (size_t)(nn - E->n_parent), st));
    E->n_parent = nn;
  }
  if (n == 0) return;
  const int32_t *dn = to_device(ctx, nodes, (size_t)n, ctx->stage_i32a);
  const int32_t *dp = to_device(ctx, parents, (size_t)n, ctx->stage_i32b);
  t->flagbuf.ensure(8, st);
  RQ_CUDA(cudaMemsetAsync(t->flagbuf.p, 0, 2 * sizeof(int32_t), st));
  parent_scatter_kernel<<<div_up(n, 256), 256, 0, st>>>(dn, dp, n, nn, E->parent.p, t->flagbuf.p);
  post_launch(ctx);
  int32_t flags[2] = {0, 0};
  RQ_CUDA(cudaMemcpyAsync(flags, t->flagbuf.p, sizeof(flags), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  E->dirty = true;
  // a parent edge now runs to another node: its resident trajectory (item n_edges + v) is the old edge's.  Clearing
  // parents keeps them valid, since the sweeps never read the item of a node without a parent edge.
  if (flags[1]) E->traj_items = -1;
  RQ_REQUIRE(flags[0] == 0, "node / parent index out of range");
}

// ------------------------------------------------------ sweep obstacle table
__global__ void sweep_table_kernel(const double4 *__restrict__ rec, const int32_t *__restrict__ ids, int n,
                                   double robot_radius, double delta, double4 *__restrict__ out_rec,
                                   double4 *__restrict__ out_par, double2 *__restrict__ out_thr,
                                   double2 *__restrict__ out_ext) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double4 r = rec[ids[i]];
  double thr = __dadd_rn(robot_radius, r.w);                       // DRRT_Q.jl:1790
  double sr = __dadd_rn(__dadd_rn(robot_radius, delta), r.w);     // :3203 searchRange, left to right
  out_rec[i] = r;
  const double4 par = make_double4(thr, sqrt_thresh_le(thr), sqrt_thresh_lt(sr), sr);
  out_par[i] = par;
  if (out_thr) { out_thr[i] = make_double2(par.x, par.y); out_ext[i] = make_double2(par.z, par.w); }
}

constexpr int SW_TILE = 256;  // obstacles per shared-memory tile

// addNewObstacle: one warp per node.  Lanes first sweep the obstacle tile
// (candidate = start-node filter, then a conservative bound using the node's
// longest edge); surviving obstacles are processed cooperatively, lanes over
// the node's out-edges + parent edge with the exact predicate.
template <bool FMA_DOT>
__global__ void __launch_bounds__(256)
add_sweep_kernel(const double4 *__restrict__ pos, int n_nodes, const int32_t *__restrict__ row_ptr,
                 const int32_t *__restrict__ csr_dst, const int32_t *__restrict__ csr_eid,
                 const int32_t *__restrict__ parent, const double *__restrict__ lmax,
                 const uint8_t *__restrict__ degenerate, const double4 *__restrict__ ob_rec,
                 const double4 *__restrict__ ob_par, int n_obs, uint8_t *__restrict__ edge_flag,
                 uint8_t *__restrict__ node_flag, unsigned long long *__restrict__ stats) {
  __shared__ alignas(128) double4 s_rec[SW_TILE];
  __shared__ alignas(128) double4 s_par[SW_TILE];
  __shared__ unsigned long long s_stats[2];
  __shared__ alignas(8) unsigned long long s_bar;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  unsigned phase = 0;
  const int lane = lane_id();
  const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  unsigned long long ncand = 0, ntests = 0;
  if (threadIdx.x < 2) s_stats[threadIdx.x] = 0;

  for (int t0 = 0; t0 < n_obs; t0 += SW_TILE) {
    const int tn = min(SW_TILE, n_obs - t0);
    // obstacle tile (records + parameters, tn x 32 B each) -> shared memory by the TMA engine
    tma_stage_tile(s_rec, ob_rec + t0, (unsigned)tn * 32u, s_par, ob_par + t0, (unsigned)tn * 32u, &s_bar, phase);
    for (int v = warp0; v < n_nodes; v += nwarps) {
      const double4 p = pos[v];
      const int ra = row_ptr[v], rb = row_ptr[v + 1];
      const int par = parent ? parent[v] : -1;
      const int deg = (rb - ra) + (par >= 0 ? 1 : 0);
      const double lm = lmax[v];
      const bool degen = degenerate[v] != 0;
      // lane's first edge, prepared lazily
      SegPre pre;
      bool have_pre = false;
      for (int o0 = 0; o0 < tn; o0 += 32) {
        const int o = o0 + lane;
        bool need = false;
        if (o < tn) {
          const double4 c = s_rec[o];
          const double4 pr = s_par[o];
          const double q[3] = {c.x, c.y, c.z};
          const double s = sqdist<3>(q, p.x, p.y, p.z, 0.0);  // euclid(ob.position, node.position)
          if (start_node_in_range(s, pr.z, pr.w, v == 0)) {
            ncand += 1;
            ntests += (unsigned long long)deg;
            if (deg > 0) {
              const double lim = (pr.x + lm) * (1.0 + 1e-9);
              need = degen || !(s > lim * lim) || !isfinite(lim);
            }
          }
        }
        unsigned m = __ballot_sync(FULL, need);
        while (m) {
          const int ol = __ffs(m) - 1;
          m &= m - 1;
          const double4 c = s_rec[o0 + ol];
          const double4 pr = s_par[o0 + ol];
          for (int k0 = 0; k0 < deg; k0 += 32) {
            const int k = k0 + lane;
            if (k < deg) {
              const bool is_parent = k >= (rb - ra);
              const int w = is_parent ? par : csr_dst[ra + k];
              SegPre cur;
              if (k0 == 0 && have_pre) {
                cur = pre;
              } else {
                const double4 e = pos[w];
                cur = seg_prepare(p.x, p.y, p.z, e.x, e.y, e.z);
                if (k0 == 0) { pre = cur; have_pre = true; }
              }
              if (seg_sphere_collide<FMA_DOT>(cur, c.x, c.y, c.z, pr.x, pr.y)) {
                if (is_parent) node_flag[v] = 1;          // :3257-3270 orphan
                else edge_flag[csr_eid[ra + k]] = 1;      // :3248-3249 edge.dist = Inf
              }
            }
          }
        }
      }
    }
  }
  // block-aggregated statistics: one global atomic pair per block
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ncand += __shfl_xor_sync(FULL, ncand, o);
    ntests += __shfl_xor_sync(FULL, ntests, o);
  }
  __syncthreads();
  if (lane == 0) {
    atomicAdd(&s_stats[0], ncand);
    atomicAdd(&s_stats[1], ntests);
  }
  __syncthreads();
  if (threadIdx.x < 2) atomicAdd(&stats[threadIdx.x], s_stats[threadIdx.x]);
}

// addNewObstacle, edge-centric form (no statistics; collide_queue.cuh), the sweep's obstacles binned into the
// obstacle grid: items are the out-edges followed by one parent edge per node; a colliding (edge, obstacle) pair
// counts only if the edge's START node passes the obstacle's start-node filter, the reference's candidate rule.  The
// filter is evaluated only for the few obstacles that actually collide.
struct SweepEdgeSrc {
  static constexpr bool RESIDENT = true;   // item records built with the edge set (collide_queue.cuh: ItemRecords)
  ItemRecords rec;
  int64_t n_edges;
  const int32_t *src;
  const double2 *ext;
  uint8_t *edge_flag, *node_flag;
  __device__ __forceinline__ float4 frec(int64_t i) const { return rec.frec[i]; }
  __device__ __forceinline__ bool endpoints(int64_t i, double a[3], double b[3], int &v) const {
    const double2 p0 = rec.exact[3 * i], p1 = rec.exact[3 * i + 1], p2 = rec.exact[3 * i + 2];
    a[0] = p0.x; a[1] = p0.y; a[2] = p1.x;
    b[0] = p1.y; b[1] = p2.x; b[2] = p2.y;
    v = i >= n_edges ? (int)(i - n_edges) : src[i];   // start node (the root is admitted with <= by accept())
    return true;
  }
  __device__ __forceinline__ void clear(int64_t) const {}  // flags are zeroed by sweep_prepare_result
  __device__ __forceinline__ bool accept(int o, const double4 &r, const double a[3], int v) const {
    const double q[3] = {r.x, r.y, r.z};
    const double s = sqdist<3>(q, a[0], a[1], a[2], 0.0);  // euclid(ob.position, startNode.position)
    const double2 e = ext[o];
    return start_node_in_range(s, e.x, e.y, [&] { return v == 0; });
  }
  __device__ __forceinline__ void mark(int64_t i) const {
    if (i >= n_edges) node_flag[i - n_edges] = 1; else edge_flag[i] = 1;
  }
};

// Sink of the obstacle-centric add sweep (item_grid.cuh): a colliding (item, obstacle) pair counts only if the item's
// START node passes the obstacle's start-node filter dist(c_o, v) < searchRange_o (root: <=), the reference's
// candidate rule (findPointsInConflictWithObstacle, DRRT_Q.jl:3195-3204).
struct SweepGridSink {
  int64_t n_edges;
  const int32_t *src;
  uint8_t *edge_flag, *node_flag;
  bool fast_ok;   // delta >= 0: a segment that lies within thr of the centre has its start node within searchRange
  __device__ __forceinline__ bool wants(int) const { return true; }
  __device__ __forceinline__ bool accept(const IgObstacle &o, const double a[3], int it) const {
    const double q[3] = {o.cx, o.cy, o.cz};
    const double s = sqdist<3>(q, a[0], a[1], a[2], 0.0);  // euclid(ob.position, startNode.position)
    return start_node_in_range(s, o.ext_t, o.ext_r, [&] { return (it >= n_edges ? (int)(it - n_edges) : src[it]) == 0; });
  }
  __device__ __forceinline__ void mark(int it) const {
    if (it >= n_edges) node_flag[it - n_edges] = 1; else edge_flag[it] = 1;
  }
};

// removeObstacle: one thread per edge (upload order).  ob = table entry 0,
// others = entries 1..n_tab-1 (thr / thr_le only).
template <bool FMA_DOT>
__global__ void __launch_bounds__(256)
remove_sweep_kernel(const double4 *__restrict__ pos, const int32_t *__restrict__ src, const int32_t *__restrict__ dst,
                    int64_t n_edges, const uint8_t *__restrict__ edge_dist_inf, const double4 *__restrict__ ob_rec,
                    const double4 *__restrict__ ob_par, int n_tab, int removed_inactive,
                    uint8_t *__restrict__ edge_flag, uint8_t *__restrict__ node_flag,
                    unsigned long long *__restrict__ stats) {
  __shared__ alignas(128) double4 s_rec[SW_TILE];
  __shared__ alignas(128) double4 s_par[SW_TILE];
  __shared__ unsigned s_cnt;
  __shared__ alignas(8) unsigned long long s_bar;
  if (threadIdx.x == 0) { s_cnt = 0; mbar_init(&s_bar, 1); }
  unsigned phase = 0;
  __syncthreads();
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = e < n_edges;
  const double4 c0 = ob_rec[0];
  const double4 p0 = ob_par[0];
  bool pending = false;  // flagged edge that collides with the removed obstacle
  SegPre pre;
  int v = 0;
  if (valid) {
    v = src[e];
    const double4 p = pos[v];
    const double q[3] = {c0.x, c0.y, c0.z};
    const double s = sqdist<3>(q, p.x, p.y, p.z, 0.0);
    if (start_node_in_range(s, p0.z, p0.w, v == 0)) {
      atomicAdd(&s_cnt, 1u);  // (edge, obstacle) pairs that pass the start-node filter
      if (edge_dist_inf[e] && !removed_inactive) {  // DRRT_Q.jl:3319 (QX: obstacle already unused -> false)
        const double4 w = pos[dst[e]];
        pre = seg_prepare(p.x, p.y, p.z, w.x, w.y, w.z);
        pending = seg_sphere_collide<FMA_DOT>(pre, c0.x, c0.y, c0.z, p0.x, p0.y);
      }
    }
  }
  bool conflicts = false;
  for (int t0 = 1; t0 < n_tab; t0 += SW_TILE) {  // :3326-3337 every other active obstacle
    const int tn = min(SW_TILE, n_tab - t0);
    tma_stage_tile(s_rec, ob_rec + t0, (unsigned)tn * 32u, s_par, ob_par + t0, (unsigned)tn * 32u, &s_bar, phase);
    if (pending && !conflicts)
      for (int k = 0; k < tn; ++k)
        if (seg_sphere_collide<FMA_DOT>(pre, s_rec[k].x, s_rec[k].y, s_rec[k].z, s_par[k].x, s_par[k].y)) {
          conflicts = true;
          break;
        }
  }
  if (pending && !conflicts) {  // :3340-3346
    edge_flag[e] = 1;
    node_flag[v] = 1;
  }
  __syncthreads();
  if (threadIdx.x == 0 && s_cnt) atomicAdd(&stats[1], (unsigned long long)s_cnt);
}

// ------------------------------------------------------- flag compaction
// Ordered compaction of the two byte-flag arrays (edges, nodes) into ascending id lists: tile counts, then one launch
// in which every block sums the counts of its predecessors itself (a few thousand words, all loads in flight at once:
// cheaper than a separate scan launch and than a single-pass look-back, whose spin / ticket traffic measured 40 us
// here), ranks its tile in shared memory and writes the ids coalesced.  Tiles [0, tiles_a) belong to the edge array,
// the rest to the node array, whose prefix restarts at tiles_a.
//   * the second kernel ZEROES every flag it found set: the arrays are clean again when the call returns, so the
//     next call needs no 10 MB memset (rrtqx_sweep_result_flags rebuilds the byte view from the lists);
//   * its last block to finish stores the totals, the sweep statistics (which it zeroes for the next call) and
//     one optional extra word (the item grid's overflow flag) into the context's mapped mailbox and publishes the
//     call number: the host spins on that word instead of three D2H copies and a stream synchronisation.
constexpr int FC_THREADS = 256, FC_ITEMS = 16, FC_TILE = FC_THREADS * FC_ITEMS;
__device__ __forceinline__ int fc_load(const uint8_t *__restrict__ flag, int64_t base, int64_t n, uint32_t (&w)[4]) {
  w[0] = w[1] = w[2] = w[3] = 0u;
  if (base + FC_ITEMS <= n) {
    const uint4 v = *reinterpret_cast<const uint4 *>(flag + base);
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
  } else {
    for (int k = 0; k < FC_ITEMS; ++k)
      if (base + k < n && flag[base + k]) w[k >> 2] |= 1u << (8 * (k & 3));
  }
  int cnt = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) { w[k] = __vcmpne4(w[k], 0u) & 0x01010101u; cnt += __popc(w[k]); }
  return cnt;
}
__global__ void __launch_bounds__(FC_THREADS)
flag_tile_counts_kernel(const uint8_t *__restrict__ fa, int64_t na, int tiles_a, const uint8_t *__restrict__ fb, int64_t nb,
                        int32_t *__restrict__ counts) {
  __shared__ int32_t sm[FC_THREADS / 32];
  const bool second = (int)blockIdx.x >= tiles_a;
  const int tile = second ? blockIdx.x - tiles_a : blockIdx.x;
  uint32_t w[4];
  int32_t cnt = fc_load(second ? fb : fa, (int64_t)tile * FC_TILE + (int64_t)threadIdx.x * FC_ITEMS, second ? nb : na, w);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(FULL, cnt, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    int32_t t = 0;
#pragma unroll
    for (int k = 0; k < FC_THREADS / 32; ++k) t += sm[k];
    counts[blockIdx.x] = t;
  }
}
__device__ __forceinline__ void sweep_publish(int32_t tot_a, int32_t tot_b, int tiles_a, int tiles_b,
                                              unsigned long long *__restrict__ stats, const int32_t *__restrict__ extra,
                                              HostMail::Block *__restrict__ mail, unsigned long long seq) {
  mail->v[0] = tiles_a ? tot_a : 0;
  mail->v[1] = tiles_b ? tot_b : 0;
  mail->v[2] = stats ? (long long)*(volatile unsigned long long *)&stats[0] : 0;
  mail->v[3] = stats ? (long long)*(volatile unsigned long long *)&stats[1] : 0;
  mail->v[4] = extra ? *(volatile const int32_t *)extra : 0;
  if (stats) { stats[0] = 0ull; stats[1] = 0ull; }
  __threadfence_system();
  *(volatile unsigned long long *)&mail->seq = seq;
}
__global__ void __launch_bounds__(FC_THREADS, 8)
flag_compact_kernel(uint8_t *__restrict__ fa, int64_t na, int tiles_a, int32_t *__restrict__ out_a,
                    uint8_t *__restrict__ fb, int64_t nb, int tiles_b, int32_t *__restrict__ out_b,
                    const int32_t *__restrict__ counts, int32_t *__restrict__ totals /* [2] totals, [2] done counter */,
                    unsigned long long *__restrict__ stats, const int32_t *__restrict__ extra,
                    HostMail::Block *__restrict__ mail, unsigned long long seq) {
  __shared__ int32_t sm[33];
  __shared__ int32_t s_prefix;
  __shared__ int32_t s_ids[FC_TILE];
  const int tile_g = blockIdx.x;
  const bool second = tile_g >= tiles_a;
  const int first = second ? tiles_a : 0;
  const int tile = tile_g - first;
  uint8_t *flag = second ? fb : fa;
  const int64_t n = second ? nb : na;
  int32_t *out = second ? out_b : out_a;
  if (threadIdx.x == 0) s_prefix = 0;
  // sum of the predecessors' counts: independent loads, all in flight before the first use
  int32_t part = 0;
  for (int j = first + (int)threadIdx.x; j < tile_g; j += FC_THREADS) part += counts[j];
  const int64_t base = (int64_t)tile * FC_TILE + (int64_t)threadIdx.x * FC_ITEMS;
  uint32_t w[4];
  const int32_t cnt = fc_load(flag, base, n, w);
  if (cnt) {   // clean up behind ourselves
    if (base + FC_ITEMS <= n) *reinterpret_cast<uint4 *>(flag + base) = make_uint4(0u, 0u, 0u, 0u);
    else for (int k = 0; k < FC_ITEMS; ++k) if (base + k < n) flag[base + k] = 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(FULL, part, o);
  int32_t tot;
  const int32_t ex = block_exclusive_scan<int32_t>(cnt, sm, &tot);   // (its barriers order the s_prefix initialisation)
  if ((threadIdx.x & 31) == 0 && part) atomicAdd(&s_prefix, part);
  {
    int32_t p = ex;
#pragma unroll
    for (int k = 0; k < FC_ITEMS; ++k)
      if ((w[k >> 2] >> (8 * (k & 3))) & 1u) s_ids[p++] = (int32_t)(base + k);
  }
  __syncthreads();
  const int32_t prefix = s_prefix;
  if (threadIdx.x == 0 && tile == (second ? tiles_b : tiles_a) - 1) totals[second ? 1 : 0] = prefix + tot;
  for (int j = threadIdx.x; j < tot; j += FC_THREADS) out[prefix + j] = s_ids[j];
  // the last block to finish publishes the call's small results (and resets the counter for the next call)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&totals[2], 1) == tiles_a + tiles_b - 1) {
      __threadfence();
      totals[2] = 0;
      sweep_publish(*(volatile int32_t *)&totals[0], *(volatile int32_t *)&totals[1], tiles_a, tiles_b, stats, extra, mail, seq);
    }
  }
}
__global__ void sweep_publish_kernel(unsigned long long *__restrict__ stats, const int32_t *__restrict__ extra,
                                     HostMail::Block *__restrict__ mail, unsigned long long seq) {   // empty edge set
  if (threadIdx.x == 0) sweep_publish(0, 0, 0, 0, stats, extra, mail, seq);
}

// list -> byte flags (rrtqx_sweep_result_flags: the compaction leaves the flag arrays clean)
__global__ void flags_from_list_kernel(const int32_t *__restrict__ list, int64_t n, uint8_t *__restrict__ flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) flag[list[i]] = 1;
}

struct FlagCompactBufs {   // per context
  DevBuf<int32_t> counts, totals;
};
static FlagCompactBufs &flag_compact_bufs(rrtqx_ctx *ctx) {
  static const char tag = 0;
  return ctx->scratch.get<FlagCompactBufs>(&tag);
}

// Flags -> ascending id lists + counts (+ one extra device word, returned in *extra_out).  The lists are allocated
// for the worst case (every edge / node); two launches back to back (tile counts, compaction whose last block
// publishes), results through the context's mailbox.
void sweep_finish(rrtqx_ctx *ctx, rrtqx_sweep_result *R, const int32_t *extra_dev, int32_t *extra_out) {
  cudaStream_t st = ctx->stream;
  const int64_t et = (R->n_edges + FC_TILE - 1) / FC_TILE, nt = (R->n_nodes + FC_TILE - 1) / FC_TILE;
  R->edge_list.ensure((size_t)R->n_edges + 1, st);
  R->node_list.ensure((size_t)R->n_nodes + 1, st);
  FlagCompactBufs &B = flag_compact_bufs(ctx);
  B.counts.ensure((size_t)(et + nt) + 1, st);
  if (!B.totals.p) {
    B.totals.ensure(4, st);
    RQ_CUDA(cudaMemsetAsync(B.totals.p, 0, 4 * sizeof(int32_t), st));   // [2]: blocks finished (reset by the last one)
  }
  HostMail &M = host_mail(ctx);
  const unsigned long long seq = ++M.seq;
  if (et + nt > 0) {
    flag_tile_counts_kernel<<<(unsigned)(et + nt), FC_THREADS, 0, st>>>(R->edge_flag.p, R->n_edges, (int)et, R->node_flag.p,
                                                                        R->n_nodes, B.counts.p);
    flag_compact_kernel<<<(unsigned)(et + nt), FC_THREADS, 0, st>>>(R->edge_flag.p, R->n_edges, (int)et, R->edge_list.p,
                                                                    R->node_flag.p, R->n_nodes, (int)nt, R->node_list.p,
                                                                    B.counts.p, B.totals.p, R->stats.p, extra_dev, M.d, seq);
    post_launch(ctx, 2);
  } else {
    sweep_publish_kernel<<<1, 32, 0, st>>>(R->stats.p, extra_dev, M.d, seq);
    post_launch(ctx);
  }
  M.wait(st, seq);
  R->n_edge_hits = M.h->v[0];
  R->n_node_hits = M.h->v[1];
  R->n_candidates = M.h->v[2];
  R->n_pair_tests = M.h->v[3];
  if (extra_out) *extra_out = (int32_t)M.h->v[4];
  R->flags_clean = true;
}

// Byte-flag view of the last result, rebuilt from the id lists (the compaction cleaned the arrays); the arrays are
// dirty afterwards and the next sweep clears them with a memset.
void sweep_result_rebuild_flags(rrtqx_ctx *ctx, rrtqx_sweep_result *R) {
  cudaStream_t st = ctx->stream;
  if (!R->flags_clean) return;   // still hold the flags of the last call (or nothing was ever swept)
  if (R->n_edge_hits > 0) flags_from_list_kernel<<<div_up(R->n_edge_hits, 256), 256, 0, st>>>(R->edge_list.p, R->n_edge_hits, R->edge_flag.p);
  if (R->n_node_hits > 0) flags_from_list_kernel<<<div_up(R->n_node_hits, 256), 256, 0, st>>>(R->node_list.p, R->n_node_hits, R->node_flag.p);
  post_launch(ctx, 2);
  R->flags_clean = false;
}

void sweep_prepare_result(rrtqx_edges *E, rrtqx_sweep_result *R) {
  rrtqx_ctx *ctx = E->tree->ctx;
  cudaStream_t st = ctx->stream;
  R->ctx = ctx;
  R->n_edges = E->n_edges;
  R->n_nodes = E->n_nodes;
  const uint8_t *pe = R->edge_flag.p, *pn = R->node_flag.p;
  const unsigned long long *ps = R->stats.p;
  R->edge_flag.ensure((size_t)E->n_edges + 1, st);
  R->node_flag.ensure((size_t)E->n_nodes + 1, st);
  R->stats.ensure(4, st);
  // the compaction leaves flags and statistics zeroed: clear only new allocations and arrays left dirty by a failed
  // call or by rrtqx_sweep_result_flags (whole capacity, so a later, larger edge set finds zeros too)
  const bool dirty = !R->flags_clean;
  if (dirty || pe != R->edge_flag.p) RQ_CUDA(cudaMemsetAsync(R->edge_flag.p, 0, R->edge_flag.cap, st));
  if (dirty || pn != R->node_flag.p) RQ_CUDA(cudaMemsetAsync(R->node_flag.p, 0, R->node_flag.cap, st));
  if (dirty || ps != R->stats.p) RQ_CUDA(cudaMemsetAsync(R->stats.p, 0, 4 * sizeof(unsigned long long), st));
  R->flags_clean = false;   // until sweep_finish has run
}

void obstacle_add_sweep(rrtqx_edges *E, const rrtqx_spheres *S, const int32_t *ob_ids, int64_t n_obs,
                        double robot_radius, double delta, uint32_t flags, rrtqx_sweep_result *R) {
  rrtqx_ctx *ctx = E->tree->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(E->tree->d == 3, "the sphere-world sweeps need a 3-D tree (SimpleEdge); Dubins trees use the *_2d sweeps");
  RQ_REQUIRE(n_obs >= 0 && n_obs < (1 << 24), "n_obs out of range");
  if (!is_device_ptr(ob_ids))
    for (int64_t i = 0; i < n_obs; ++i) RQ_REQUIRE(ob_ids[i] >= 0 && ob_ids[i] < S->n, "obstacle id out of range");
  const int32_t *dids = to_device(ctx, ob_ids, (size_t)n_obs, R->ids_stage);
  if (E->dirty || E->tree->n != E->n_nodes) edges_rebuild(E);  // appended edges / parents / new nodes
  PhaseScope ph(ctx, "add_sweep");
  sweep_prepare_result(E, R);
  if (n_obs == 0 || E->n_nodes == 0) {
    sweep_finish(ctx, R);
    return;
  }
  R->ob_rec.ensure((size_t)n_obs, st);
  R->ob_par.ensure((size_t)n_obs, st);
  R->ob_thr.ensure((size_t)n_obs, st);
  R->ob_ext.ensure((size_t)n_obs, st);
  const int TB = 256;
  sweep_table_kernel<<<div_up(n_obs, TB), TB, 0, st>>>(S->rec.p, dids, (int)n_obs, robot_radius, delta, R->ob_rec.p, R->ob_par.p, R->ob_thr.p, R->ob_ext.p);
  post_launch(ctx);
  const bool fma = flags & RRTQX_CHECK_FMA_DOT;
  const int32_t *par = E->has_parent ? E->parent.p : nullptr;
  if (flags & RRTQX_SWEEP_STATS) {  // node-centric, the only form with candidate / pair statistics
    const int blocks = std::max(1, std::min(div_up(E->n_nodes * 32, TB), ctx->sm_count * 8));
    if (fma)
      add_sweep_kernel<true><<<blocks, TB, 0, st>>>(E->tree->pos.p, (int)E->n_nodes, E->row_ptr.p, E->csr_dst.p, E->csr_eid.p, par,
                                                    E->lmax.p, E->degenerate.p, R->ob_rec.p, R->ob_par.p, (int)n_obs,
                                                    R->edge_flag.p, R->node_flag.p, R->stats.p);
    else
      add_sweep_kernel<false><<<blocks, TB, 0, st>>>(E->tree->pos.p, (int)E->n_nodes, E->row_ptr.p, E->csr_dst.p, E->csr_eid.p, par,
                                                     E->lmax.p, E->degenerate.p, R->ob_rec.p, R->ob_par.p, (int)n_obs,
                                                     R->edge_flag.p, R->node_flag.p, R->stats.p);
    post_launch(ctx);
    sweep_finish(ctx, R);
    return;
  }
  if (E->igrid.valid && !ctx->tune.no_item_grid) {
    // obstacle-centric sweep over the items sorted by midpoint cell: only the cells an obstacle can reach are read
    SweepGridSink K{E->n_edges, E->src.p, R->edge_flag.p, R->node_flag.p, delta >= 0.0};
    const int32_t *ovf_dev;
    if (fma)
      ovf_dev = item_grid_run<true>(ctx, E->igrid, &E->igrid1, R->ob_rec.p, R->ob_thr.p, R->ob_ext.p, nullptr, (int)n_obs, K,
                                    E->tree->pos.p, E->n_nodes, E->src.p, E->dst.p, E->n_edges, par);
    else
      ovf_dev = item_grid_run<false>(ctx, E->igrid, &E->igrid1, R->ob_rec.p, R->ob_thr.p, R->ob_ext.p, nullptr, (int)n_obs, K,
                                     E->tree->pos.p, E->n_nodes, E->src.p, E->dst.p, E->n_edges, par);
    // the overflow flag (more work units than the list holds: huge obstacles) is read together with the counts;
    // on overflow nothing was marked and the edge-centric kernels repeat the sweep (below)
    int32_t ovf = 0;
    sweep_finish(ctx, R, ovf_dev, &ovf);
    R->n_candidates = R->n_pair_tests = -1;
    if (ovf == 0) return;
    sweep_prepare_result(E, R);
  }
  // edge-centric sweep over the binned obstacles
  const int64_t work = E->n_edges + E->n_nodes;
  const bool use_queue = work >= cover_min_items(ctx, PQ_MIN_ITEMS_SWEEP) && work < ((int64_t)1 << 32);
  const BinnedObstacles T = bin_obstacles(ctx, R->binned, R->ob_rec.p, R->ob_thr.p, R->ob_ext.p, nullptr, (int)n_obs,
                                          use_queue && n_obs <= COV_MAX_OBSTACLES);
  const SweepEdgeSrc Q{ItemRecords{E->item_frec.p, E->item_exact.p}, E->n_edges, E->src.p, T.ext, R->edge_flag.p, R->node_flag.p};
  if (use_queue) { if (fma) pq_launch<true>(ctx, Q, work, T); else pq_launch<false>(ctx, Q, work, T); }
  else           { if (fma) pq_item_launch<true>(ctx, Q, work, T); else pq_item_launch<false>(ctx, Q, work, T); }
  sweep_finish(ctx, R);
  R->n_candidates = R->n_pair_tests = -1;
}

void obstacle_remove_sweep(rrtqx_edges *E, const rrtqx_spheres *S, int32_t ob_id, const int32_t *other_ids,
                           int64_t n_others, const uint8_t *edge_dist_inf, double robot_radius, double delta,
                           uint32_t flags, rrtqx_sweep_result *R) {
  rrtqx_ctx *ctx = E->tree->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(E->tree->d == 3, "the sphere-world sweeps need a 3-D tree (SimpleEdge); Dubins trees use the *_2d sweeps");
  RQ_REQUIRE(ob_id >= 0 && ob_id < S->n, "obstacle id out of range");
  RQ_REQUIRE(n_others >= 0 && n_others < (1 << 24), "n_others out of range");
  RQ_REQUIRE(edge_dist_inf != nullptr || E->n_edges == 0, "edge_dist_inf is NULL");
  if (E->dirty || E->tree->n != E->n_nodes) edges_rebuild(E);
  // table = [ob_id, others...]
  std::vector<int32_t> ids((size_t)n_others + 1);
  ids[0] = ob_id;
  if (n_others) {
    if (is_device_ptr(other_ids))
      RQ_CUDA(cudaMemcpy(ids.data() + 1, other_ids, sizeof(int32_t) * n_others, cudaMemcpyDeviceToHost));
    else
      memcpy(ids.data() + 1, other_ids, sizeof(int32_t) * n_others);
  }
  for (size_t i = 0; i < ids.size(); ++i) RQ_REQUIRE(ids[i] >= 0 && ids[i] < S->n, "obstacle id out of range");
  R->ids_stage2.ensure(ids.size(), st);
  RQ_CUDA(cudaMemcpyAsync(R->ids_stage2.p, ids.data(), sizeof(int32_t) * ids.size(), cudaMemcpyHostToDevice, st));
  RQ_CUDA(cudaStreamSynchronize(st));  // ids is a local vector
  const uint8_t *dinf = to_device(ctx, edge_dist_inf, (size_t)E->n_edges, R->inf_stage);
  PhaseScope ph(ctx, "remove_sweep");
  sweep_prepare_result(E, R);
  const int n_tab = (int)ids.size();
  R->ob_rec.ensure((size_t)n_tab, st);
  R->ob_par.ensure((size_t)n_tab, st);
  const int TB = 256;
  sweep_table_kernel<<<div_up(n_tab, TB), TB, 0, st>>>(S->rec.p, R->ids_stage2.p, n_tab, robot_radius, delta, R->ob_rec.p, R->ob_par.p, nullptr, nullptr);
  post_launch(ctx);
  if (E->n_edges > 0) {
    const int removed_inactive = (flags & RRTQX_SWEEP_REMOVED_INACTIVE) ? 1 : 0;
    if (flags & RRTQX_CHECK_FMA_DOT)
      remove_sweep_kernel<true><<<div_up(E->n_edges, TB), TB, 0, st>>>(E->tree->pos.p, E->src.p, E->dst.p, E->n_edges, dinf, R->ob_rec.p,
                                                                      R->ob_par.p, n_tab, removed_inactive, R->edge_flag.p,
                                                                      R->node_flag.p, R->stats.p);
    else
      remove_sweep_kernel<false><<<div_up(E->n_edges, TB), TB, 0, st>>>(E->tree->pos.p, E->src.p, E->dst.p, E->n_edges, dinf, R->ob_rec.p,
                                                                       R->ob_par.p, n_tab, removed_inactive, R->edge_flag.p,
                                                                       R->node_flag.p, R->stats.p);
    post_launch(ctx);
  }
  sweep_finish(ctx, R);
}

}  // namespace rrtqx
