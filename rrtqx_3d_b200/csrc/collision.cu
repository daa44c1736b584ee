// collision.cu -- batched explicitEdgeCheck / explicitPointCheck against the
// sphere obstacle list (DRRT_Q.jl:1434-1595, 1775-1826).
#include <cstdlib>

#include "objects.cuh"
#include "collide_queue.cuh"

namespace rrtqx {

// Active-obstacle table for one call: centre+radius, thr = robotRadius+radius,
// thr_le = sqrt_thresh_le(thr).  Ordered compaction by a single block (the
// obstacle list is small: tens to a few thousand entries).
struct SphereTable {
  const double4 *rec;   // (cx,cy,cz,R)
  const double2 *thr;   // (thr, thr_le)
  int n;
};

__global__ void sphere_table_kernel(const double4 *__restrict__ rec, const uint8_t *__restrict__ active, int n,
                                    int ignore_active, double robot_radius, double4 *__restrict__ out_rec,
                                    double2 *__restrict__ out_thr, int32_t *__restrict__ out_n) {
  __shared__ int warp_cnt[32];
  __shared__ int base_s;
  if (threadIdx.x == 0) base_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int b = 0; b < n; b += blockDim.x) {
    int i = b + threadIdx.x;
    bool keep = i < n && (ignore_active || active[i]);
    unsigned m = __ballot_sync(FULL, keep);
    if (lane == 0) warp_cnt[warp] = __popc(m);
    __syncthreads();
    int off = base_s;
    for (int w = 0; w < warp; ++w) off += warp_cnt[w];
    if (keep) {
      int o = off + __popc(m & lanemask_lt());
      double4 r = rec[i];
      double thr = __dadd_rn(robot_radius, r.w);  // robotRadius + thisObstacle.radius (DRRT_Q.jl:1790)
      out_rec[o] = r;
      out_thr[o] = make_double2(thr, sqrt_thresh_le(thr));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < nw; ++w) tot += warp_cnt[w];
      base_s += tot;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *out_n = base_s;
}

struct SphereTableBufs {
  DevBuf<double4> rec;
  DevBuf<double2> thr;
  DevBuf<int32_t> n;
  DevBuf<int32_t> bad;         // device counter of out-of-range edge endpoints
  BinnedObstacleBufs binned;   // the table binned for the large-batch kernels
  // what the buffers currently hold: the table of obstacle set `key_version` for (robot radius, ignore flag);
  // grid_level 0: table only, 1: + obstacle grid, 2: + cover lists (build `cover_id` of the context's cover
  // buffers).  An unchanged obstacle set is not re-binned on every call (the planner checks thousands of edge
  // batches between two obstacle events).
  uint64_t key_version = 0, key_rho = 0, cover_id = 0;
  int key_ignore = -1, grid_level = 0;
};

static SphereTableBufs &table_bufs(rrtqx_ctx *ctx) {  // owned by the context, freed in rrtqx_ctx_destroy
  static const char tag = 0;
  return ctx->scratch.get<SphereTableBufs>(&tag);
}

// Builds the table on the stream; returns it with n = upper bound (all
// obstacles) and writes the live count to *n_dev_out (device) for kernels.
SphereTable build_sphere_table(rrtqx_ctx *ctx, const rrtqx_spheres *s, double robot_radius, uint32_t flags,
                               const int32_t **n_dev_out) {
  SphereTableBufs &b = table_bufs(ctx);
  cudaStream_t st = ctx->stream;
  size_t n = (size_t)s->n;
  b.rec.ensure(n + 1, st);
  b.thr.ensure(n + 1, st);
  b.n.ensure(4, st);
  const int ignore = (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0;
  uint64_t rho_bits;
  memcpy(&rho_bits, &robot_radius, sizeof(rho_bits));
  if (!(s->version != 0 && b.key_version == s->version && b.key_rho == rho_bits && b.key_ignore == ignore)) {
    sphere_table_kernel<<<1, 1024, 0, st>>>(s->rec.p, s->active.p, (int)n, ignore, robot_radius, b.rec.p, b.thr.p, b.n.p);
    post_launch(ctx);
    b.key_version = s->version; b.key_rho = rho_bits; b.key_ignore = ignore; b.grid_level = 0;
  }
  SphereTable t;
  t.rec = b.rec.p;
  t.thr = b.thr.p;
  t.n = (int)n;
  *n_dev_out = b.n.p;
  return t;
}

// The table binned for the large-batch kernels, with the cover lists if want_cover; re-binned only when the table or
// the cover lists changed (SphereTableBufs::grid_level).
static BinnedObstacles binned_table(rrtqx_ctx *ctx, const SphereTable &tab, const int32_t *n_live, bool want_cover) {
  SphereTableBufs &b = table_bufs(ctx);
  const int want_level = want_cover ? 2 : 1;
  if (!(b.grid_level == want_level && (!want_cover || cover_bufs(ctx).build_id == b.cover_id))) {
    bin_obstacles(ctx, b.binned, tab.rec, tab.thr, nullptr, n_live, tab.n, want_cover);
    b.grid_level = want_level;
    if (want_cover) b.cover_id = cover_bufs(ctx).build_id;
  }
  return b.binned.view();
}

// Item source of the binned-table kernels of the per-call check (collide_queue.cuh).
template <bool SRC_TREE>
struct BatchEdgeSrc {
  static constexpr bool RESIDENT = false;   // end points are gathered per call (no prepared item records)
  __device__ __forceinline__ float4 frec(int64_t) const { return make_float4(0.f, 0.f, 0.f, -1.f); }
  const double4 *pos;
  const int32_t *src, *dst;
  const double *starts, *ends;
  uint8_t *out;
  int n_nodes;
  int32_t *bad;  // count of edges with an endpoint outside [0, n_nodes): the call fails with RRTQX_ERR_INVALID
  __device__ __forceinline__ bool endpoints(int64_t i, double a[3], double b[3], int &v) const {
    v = 0;
    if (SRC_TREE) {
      const int ia = src[i], ib = dst[i];
      if ((unsigned)ia >= (unsigned)n_nodes || (unsigned)ib >= (unsigned)n_nodes) {
        atomicAdd(bad, 1);
        out[i] = 0;
        return false;
      }
      const double4 pa = pos[ia], pb = pos[ib];
      a[0] = pa.x; a[1] = pa.y; a[2] = pa.z;
      b[0] = pb.x; b[1] = pb.y; b[2] = pb.z;
    } else {
      const double *pa = starts + 3 * i, *pb = ends + 3 * i;
      a[0] = pa[0]; a[1] = pa[1]; a[2] = pa[2];
      b[0] = pb[0]; b[1] = pb[1]; b[2] = pb[2];
    }
    return true;
  }
  __device__ __forceinline__ void clear(int64_t i) const { out[i] = 0; }
  __device__ __forceinline__ bool accept(int, const double4 &, const double *, int) const { return true; }
  __device__ __forceinline__ void mark(int64_t i) const { out[i] = 1; }
};

// Sink of the obstacle-centric resident check (item_grid.cuh): explicitEdgeCheck(S, edge) has no extra condition;
// parent-edge items of the grid are not part of the result.
struct CheckGridSink {
  int64_t n_edges;
  uint8_t *out;
  bool fast_ok;
  __device__ __forceinline__ bool wants(int it) const { return it < n_edges; }
  __device__ __forceinline__ bool accept(const IgObstacle &, const double *, int) const { return true; }
  __device__ __forceinline__ void mark(int it) const { out[it] = 1; }
};

// Resident form: every out-edge of an rrtqx_edges set, item records prepared when the set was built.
struct ResidentEdgeSrc {
  static constexpr bool RESIDENT = true;
  ItemRecords rec;
  uint8_t *out;
  __device__ __forceinline__ float4 frec(int64_t i) const { return rec.frec[i]; }
  __device__ __forceinline__ bool endpoints(int64_t i, double a[3], double b[3], int &v) const {
    const double2 p0 = rec.exact[3 * i], p1 = rec.exact[3 * i + 1], p2 = rec.exact[3 * i + 2];
    a[0] = p0.x; a[1] = p0.y; a[2] = p1.x;
    b[0] = p1.y; b[1] = p2.x; b[2] = p2.y;
    v = 0;
    return true;
  }
  __device__ __forceinline__ void clear(int64_t i) const { out[i] = 0; }
  __device__ __forceinline__ bool accept(int, const double4 &, const double *, int) const { return true; }
  __device__ __forceinline__ void mark(int64_t i) const { out[i] = 1; }
};

constexpr int SPH_TILE = 512;

// One thread per edge; obstacle table staged through shared memory in tiles.
// SRC_TREE: endpoints are gathered from the node table by index; otherwise
// they are read from explicit start/end arrays (n x 3 row-major).
template <bool FMA_DOT, bool SRC_TREE>
__global__ void __launch_bounds__(256)
edge_check_kernel(const double4 *__restrict__ pos, const int32_t *__restrict__ src, const int32_t *__restrict__ dst,
                  const double *__restrict__ starts, const double *__restrict__ ends, int64_t n_edges,
                  SphereTable tab, const int32_t *__restrict__ n_live, uint8_t *__restrict__ out, int n_nodes,
                  int32_t *__restrict__ bad) {
  __shared__ alignas(128) double4 s_rec[SPH_TILE];
  __shared__ alignas(128) double2 s_thr[SPH_TILE];
  __shared__ alignas(8) unsigned long long s_bar;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  unsigned phase = 0;
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_obs = *n_live;
  SegPre pre;
  bool valid = e < n_edges;
  if (valid) {
    if (SRC_TREE) {
      const int ia = src[e], ib = dst[e];
      if ((unsigned)ia >= (unsigned)n_nodes || (unsigned)ib >= (unsigned)n_nodes) {  // reported as RRTQX_ERR_INVALID
        atomicAdd(bad, 1);
        out[e] = 0;
        valid = false;
      } else {
        const double4 a = pos[ia], b = pos[ib];
        pre = seg_prepare(a.x, a.y, a.z, b.x, b.y, b.z);
      }
    } else {
      const double *a = starts + 3 * e, *b = ends + 3 * e;
      pre = seg_prepare(a[0], a[1], a[2], b[0], b[1], b[2]);
    }
  }
  bool hit = false;
  for (int t0 = 0; t0 < n_obs; t0 += SPH_TILE) {
    const int tn = min(SPH_TILE, n_obs - t0);
    // obstacle tile -> shared memory by the TMA engine (regular tile: tn x 32 B + tn x 16 B, contiguous)
    tma_stage_tile(s_rec, tab.rec + t0, (unsigned)tn * 32u, s_thr, tab.thr + t0, (unsigned)tn * 16u, &s_bar, phase);
    if (valid && !hit) {
      for (int k = 0; k < tn; ++k) {
        double4 o = s_rec[k];
        double2 th = s_thr[k];
        if (seg_sphere_collide<FMA_DOT>(pre, o.x, o.y, o.z, th.x, th.y)) { hit = true; break; }
      }
    }
  }
  if (valid) out[e] = hit ? 1 : 0;
}

// Everything of the batched check except the final synchronisation: kernels and the copy of the flags to a host
// destination are queued on the context's stream; *bad_dev (if not NULL) receives the device counter of
// out-of-range endpoints (valid when the tree path ran, else NULL).  The sharded multi-GPU form queues this on
// every device before it waits for any of them.
void edge_check_launch(rrtqx_ctx *ctx, const rrtqx_tree *tree, const rrtqx_spheres *spheres, const int32_t *src,
                       const int32_t *dst, const double *starts, const double *ends, int64_t n_edges,
                       double robot_radius, uint32_t flags, uint8_t *collide_out, const int32_t **bad_dev) {
  if (bad_dev) *bad_dev = nullptr;
  if (n_edges <= 0) return;
  cudaStream_t st = ctx->stream;
  const bool from_tree = tree != nullptr;
  const int32_t *dsrc = nullptr, *ddst = nullptr;
  const double *dstarts = nullptr, *dends = nullptr;
  if (from_tree) {
    dsrc = to_device(ctx, src, (size_t)n_edges, ctx->stage_i32a);
    ddst = to_device(ctx, dst, (size_t)n_edges, ctx->stage_i32b);
  } else {
    dstarts = to_device(ctx, starts, (size_t)n_edges * 3, ctx->stage_f64);
    dends = to_device(ctx, ends, (size_t)n_edges * 3, ctx->stage_f64b);
  }
  const bool out_dev = is_device_ptr(collide_out);
  uint8_t *dout = collide_out;
  if (!out_dev) { ctx->stage_u8.ensure((size_t)n_edges, st); dout = ctx->stage_u8.p; }
  // endpoint indices are validated on the device (host arrays were already checked by the caller, device arrays
  // cannot be): a bad index never reaches the position gather, it is counted and the call fails
  SphereTableBufs &tb = table_bufs(ctx);
  tb.bad.ensure(4, st);
  int32_t *dbad = tb.bad.p;
  const int n_nodes = from_tree ? (int)tree->n : 0;
  if (from_tree) RQ_CUDA(cudaMemsetAsync(dbad, 0, sizeof(int32_t), st));
  {
    PhaseScope ph(ctx, "edge_check");
    const int32_t *n_live = nullptr;
    SphereTable tab = build_sphere_table(ctx, spheres, robot_radius, flags, &n_live);
    const int TB = 256;
    const unsigned blocks = (unsigned)div_up(n_edges, TB);
    const double4 *pos = from_tree ? tree->pos.p : nullptr;
    const bool fma = flags & RRTQX_CHECK_FMA_DOT;
    if (n_edges >= 4096 && spheres->n >= 16) {
      // large batch: bin the obstacles once, then each edge meets only the obstacles around it
      const bool use_queue = n_edges >= cover_min_items(ctx, PQ_MIN_ITEMS_BATCH) && n_edges < ((int64_t)1 << 32);
      const BinnedObstacles T = binned_table(ctx, tab, n_live, use_queue && spheres->n <= COV_MAX_OBSTACLES);
      auto run = [&](const auto &S) {
        if (use_queue) { if (fma) pq_launch<true>(ctx, S, n_edges, T); else pq_launch<false>(ctx, S, n_edges, T); }
        else           { if (fma) pq_item_launch<true>(ctx, S, n_edges, T); else pq_item_launch<false>(ctx, S, n_edges, T); }
      };
      if (from_tree) run(BatchEdgeSrc<true>{pos, dsrc, ddst, nullptr, nullptr, dout, n_nodes, dbad});
      else           run(BatchEdgeSrc<false>{nullptr, nullptr, nullptr, dstarts, dends, dout, 0, dbad});
    } else if (from_tree) {
      if (fma) edge_check_kernel<true, true><<<blocks, TB, 0, st>>>(pos, dsrc, ddst, nullptr, nullptr, n_edges, tab, n_live, dout, n_nodes, dbad);
      else     edge_check_kernel<false, true><<<blocks, TB, 0, st>>>(pos, dsrc, ddst, nullptr, nullptr, n_edges, tab, n_live, dout, n_nodes, dbad);
      post_launch(ctx);
    } else {
      if (fma) edge_check_kernel<true, false><<<blocks, TB, 0, st>>>(pos, nullptr, nullptr, dstarts, dends, n_edges, tab, n_live, dout, n_nodes, dbad);
      else     edge_check_kernel<false, false><<<blocks, TB, 0, st>>>(pos, nullptr, nullptr, dstarts, dends, n_edges, tab, n_live, dout, n_nodes, dbad);
      post_launch(ctx);
    }
  }
  if (!out_dev) from_device(ctx, collide_out, dout, (size_t)n_edges);
  if (bad_dev && from_tree) *bad_dev = dbad;
}

void edge_check(rrtqx_ctx *ctx, const rrtqx_tree *tree, const rrtqx_spheres *spheres, const int32_t *src,
                const int32_t *dst, const double *starts, const double *ends, int64_t n_edges, double robot_radius,
                uint32_t flags, uint8_t *collide_out) {
  if (n_edges <= 0) return;
  const int32_t *dbad = nullptr;
  edge_check_launch(ctx, tree, spheres, src, dst, starts, ends, n_edges, robot_radius, flags, collide_out, &dbad);
  int32_t n_bad = 0;
  if (dbad) RQ_CUDA(cudaMemcpyAsync(&n_bad, dbad, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  RQ_REQUIRE(n_bad == 0, "edge endpoint out of range");
}

// explicitEdgeCheck(S, edge) (DRRT_Q.jl:1802-1826) of EVERY out-edge of a resident edge set: the two-stage kernels
// over the set's prepared item records (no per-call gathers of node positions in the collect stage).
void edges_check(rrtqx_edges *E, const rrtqx_spheres *spheres, double robot_radius, uint32_t flags, uint8_t *collide_out) {
  rrtqx_tree *tree = E->tree;
  rrtqx_ctx *ctx = tree->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(tree->d == 3, "SimpleEdge checks need a 3-D tree (explicitEdgeCheck3D)");
  RQ_REQUIRE(spheres->ctx == ctx, "obstacle set of another context");
  if (E->dirty || tree->n != E->n_nodes) edges_rebuild(E);
  const int64_t n = E->n_edges;
  if (n <= 0) return;
  RQ_REQUIRE(collide_out != nullptr, "collide_out is NULL");
  const bool out_dev = is_device_ptr(collide_out);
  uint8_t *dout = collide_out;
  if (!out_dev) { ctx->stage_u8.ensure((size_t)n, st); dout = ctx->stage_u8.p; }
  {
    PhaseScope ph(ctx, "edges_check");
    const int32_t *n_live = nullptr;
    SphereTable tab = build_sphere_table(ctx, spheres, robot_radius, flags, &n_live);
    if (E->igrid.valid && !ctx->tune.no_item_grid) {
      // obstacle-centric: only the cells of the item grid an active obstacle can reach are read
      RQ_CUDA(cudaMemsetAsync(dout, 0, (size_t)n, st));
      CheckGridSink K{n, dout, true};
      const int32_t *par = E->has_parent ? E->parent.p : nullptr;
      const int32_t *ovf_dev;
      if (flags & RRTQX_CHECK_FMA_DOT)
        ovf_dev = item_grid_run<true>(ctx, E->igrid, &E->igrid1, tab.rec, tab.thr, nullptr, n_live, (int)spheres->n, K, tree->pos.p,
                                      E->n_nodes, E->src.p, E->dst.p, n, par);
      else
        ovf_dev = item_grid_run<false>(ctx, E->igrid, &E->igrid1, tab.rec, tab.thr, nullptr, n_live, (int)spheres->n, K, tree->pos.p,
                                       E->n_nodes, E->src.p, E->dst.p, n, par);
      // the overflow word travels to pinned memory behind the kernels; the flags are copied out right behind it, so
      // the common case costs ONE synchronisation (an overflowed call marked nothing and is repeated below)
      HostMail &M = host_mail(ctx);
      RQ_CUDA(cudaMemcpyAsync(&M.h->aux[0], ovf_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      if (!out_dev) from_device(ctx, collide_out, dout, (size_t)n);
      RQ_CUDA(cudaStreamSynchronize(st));
      if (*(volatile int32_t *)&M.h->aux[0] == 0) return;   // the PhaseScope destructor records the end event
    }
    // no item grid, or it overflowed: the edge-centric two-stage kernels
    const BinnedObstacles T = binned_table(ctx, tab, n_live, spheres->n <= COV_MAX_OBSTACLES);
    const ResidentEdgeSrc S{ItemRecords{E->item_frec.p, E->item_exact.p}, dout};
    if (flags & RRTQX_CHECK_FMA_DOT) pq_launch<true>(ctx, S, n, T);
    else                             pq_launch<false>(ctx, S, n, T);
  }
  if (!out_dev) from_device(ctx, collide_out, dout, (size_t)n);
  RQ_CUDA(cudaStreamSynchronize(st));
}

// explicitPointCheck (DRRT_Q.jl:1520-1556) / explicitPointCheck3D (:1558-1590),
// one thread per point, literal sequential semantics over the active list.
template <bool QUICK>
__global__ void __launch_bounds__(256)
node_check_kernel(const double *__restrict__ pts, int64_t n, SphereTable tab, const int32_t *__restrict__ n_live,
                  double robot_radius, uint8_t *__restrict__ out, double *__restrict__ cert_out) {
  __shared__ alignas(128) double4 s_rec[SPH_TILE];
  __shared__ alignas(8) unsigned long long s_bar;
  if (threadIdx.x == 0) mbar_init(&s_bar, 1);
  unsigned phase = 0;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_obs = *n_live;
  const bool valid = i < n;
  double p[3] = {0, 0, 0};
  if (valid) { p[0] = pts[3 * i]; p[1] = pts[3 * i + 1]; p[2] = pts[3 * i + 2]; }
  bool hit = false;
  if (QUICK) {  // quickCheck :1434-1452 -> quickCheck2D :1402-1415
    for (int t0 = 0; t0 < n_obs; t0 += SPH_TILE) {
      const int tn = min(SPH_TILE, n_obs - t0);
      tma_stage_tile(s_rec, tab.rec + t0, (unsigned)tn * 32u, nullptr, nullptr, 0u, &s_bar, phase);
      if (valid && !hit)
        for (int k = 0; k < tn; ++k) {
          double4 o = s_rec[k];
          double c[3] = {o.x, o.y, o.z};
          double dd = __dsqrt_rn(sqdist<3>(c, p[0], p[1], p[2], 0.0));
          if (!(dd > o.w)) { hit = true; break; }
        }
    }
  }
  double ret_cert = INFINITY;
  for (int t0 = 0; t0 < n_obs; t0 += SPH_TILE) {
    const int tn = min(SPH_TILE, n_obs - t0);
    tma_stage_tile(s_rec, tab.rec + t0, (unsigned)tn * 32u, nullptr, nullptr, 0u, &s_bar, phase);
    if (valid && !hit)
      for (int k = 0; k < tn; ++k) {  // explicitPointCheck2D :1463-1487
        double4 o = s_rec[k];
        double c[3] = {o.x, o.y, o.z};
        double this_dist = __dsub_rn(__dsqrt_rn(sqdist<3>(c, p[0], p[1], p[2], 0.0)), robot_radius);
        if (__dsub_rn(this_dist, o.w) > ret_cert) continue;
        this_dist = __dsub_rn(this_dist, o.w);
        if (this_dist < 0.0) { hit = true; break; }
        double this_cert = jl_min(ret_cert, this_dist);
        if (this_cert < ret_cert) ret_cert = this_cert;  // :1545-1547
      }
  }
  if (valid) {
    out[i] = hit ? 1 : 0;
    if (cert_out) cert_out[i] = hit ? 0.0 : ret_cert;
  }
}

void node_check(rrtqx_ctx *ctx, const rrtqx_spheres *spheres, const double *points, int64_t n, double robot_radius,
                uint32_t flags, uint8_t *collide_out, double *cert_out) {
  if (n <= 0) return;
  cudaStream_t st = ctx->stream;
  const double *dp = to_device(ctx, points, (size_t)n * 3, ctx->stage_f64);
  const bool out_dev = is_device_ptr(collide_out), cert_dev = cert_out && is_device_ptr(cert_out);
  uint8_t *dout = collide_out;
  double *dcert = cert_out;
  if (!out_dev) { ctx->stage_u8.ensure((size_t)n, st); dout = ctx->stage_u8.p; }
  if (cert_out && !cert_dev) { ctx->stage_f64b.ensure((size_t)n, st); dcert = ctx->stage_f64b.p; }
  {
    PhaseScope ph(ctx, "node_check");
    const int32_t *n_live = nullptr;
    SphereTable tab = build_sphere_table(ctx, spheres, robot_radius, flags, &n_live);
    const int TB = 256;
    const unsigned blocks = (unsigned)div_up(n, TB);
    if (flags & RRTQX_CHECK_QUICK_PASS)
      node_check_kernel<true><<<blocks, TB, 0, st>>>(dp, n, tab, n_live, robot_radius, dout, dcert);
    else
      node_check_kernel<false><<<blocks, TB, 0, st>>>(dp, n, tab, n_live, robot_radius, dout, dcert);
    post_launch(ctx);
  }
  if (!out_dev) from_device(ctx, collide_out, dout, (size_t)n);
  if (cert_out && !cert_dev) from_device(ctx, cert_out, dcert, (size_t)n);
  RQ_CUDA(cudaStreamSynchronize(st));
}

}  // namespace rrtqx
