// extend_dubins.cuh -- the Dubins planner's per-iteration geometric work (DRRT.jl / DRRT_Q.jl extend() with
// DubinsEdge, config C4: 4-D tree [x y t theta], theta wrapped at 2 pi) in one call with one host wait
// (included by range.cu, inside namespace rrtqx):
//     (closest, d) = kdFindNearest(KD, p)                          ghost identity included
//     saturate(p, closest, delta)                                  DRRT_DubinsEdge_functions.jl:70-95 (optional)
//     nodeList     = kdFindWithinRange(KD, r, p)                   ghost identity included
//     calculateTrajectory + explicitEdgeCheck of edge(new -> n)    DRRT_Q.jl:1949-1960 (findBestParent)
//     calculateTrajectory + explicitEdgeCheck of edge(n -> new)    DRRT_Q.jl:2600-2603
// Three launches on the stream, no host round trip between them:
//   A  one 512-thread block: warp 0 runs nearest_warp (the body of nearest_kernel), lane 0 saturates, all warps
//      scan the ball's rows.  theta is off the grid, so the real and the ghost identity share the same (x, y, z)
//      rows and both radicands are evaluated per candidate, with the rules of range_query_kernel's WRAP path.
//      Then one thread per edge solves its Dubins word (dubins.cuh) and keeps the row layout; a block scan of
//      the row counts gives the CSR pointers.
//   B  a persistent grid, one warp per edge: the lanes emit the edge's rows (word_row, dubins.cuh).
//   C  a persistent grid, one warp per edge: dubins_collide_warp over the polygon set (polygon.cuh); the last
//      block to finish publishes the call number in mapped pinned memory.
// Emission and check are separate launches because the check reads the rows through the read-only data path,
// which is coherent only with writes of earlier launches.  Per-neighbour and per-edge results go straight to
// mapped pinned memory; the host spins on the completion word.  B and C read the edge count and the row total
// from device memory, so the host never sizes them; when the rows exceed the scratch, B and C skip their work
// and the host grows the scratch and repeats the call once.

constexpr int EXD_THREADS = 512;
constexpr int EXD_WARPS = EXD_THREADS / 32;
constexpr int64_t EXD_INITIAL_ROWS = 16384;

struct ExtendDubinsHeader {   // mapped pinned, written by launch A except `seq`
  double point[4];            // the (saturated) sample
  int32_t count;              // neighbours found (may exceed capacity)
  int32_t nearest_idx;
  double nearest_dist;
  int64_t rows;               // trajectory rows of the 2 * min(count, capacity) edges
  unsigned long long seq;     // written LAST by launch C (after a system-scope fence): the host polls it
};
struct ExtendDubinsDev {      // device memory: what launch A hands to launches B and C
  double p[4];
  int64_t rows;
  int32_t n_edges;
  uint32_t done;              // blocks of launch C finished; the last one resets it
};
struct ExtendDubinsParams {
  double p[4];
  double delta, r, r_turn;
  int32_t capacity, saturate;
  unsigned long long seq;
};
struct ExtendDubinsOut {
  int32_t *nbr;                        // device, capacity: neighbour node ids
  int32_t *h_idx;                      // mapped, capacity
  double *h_dist;                      // mapped, capacity
  double *dist;                        // device, 2 capacity (the trajectory result's per-edge arrays)
  int32_t *type;
  int64_t *ptr;                        // device, 2 capacity + 1
  double *h_edist;                     // mapped, 2 capacity
  int32_t *h_etype;
  WordRows *layout;                    // device, 2 capacity
};

__global__ void __launch_bounds__(EXD_THREADS, 1)
extend_dubins_query_kernel(GridView g, WrapInfo wrap, const ExtendDubinsParams prm, ExtendDubinsOut o,
                           ExtendDubinsDev *__restrict__ dev, ExtendDubinsHeader *__restrict__ hdr) {
  __shared__ double s_p[4];
  __shared__ int s_count, s_nearest;
  __shared__ double s_nearest_dist;
  __shared__ long long s_wsum[EXD_WARPS];
  __shared__ long long s_carry;
  const int lane = lane_id(), warp = threadIdx.x >> 5, tid = threadIdx.x;
  const unsigned lt = lanemask_lt();

  // ---- nearest of the sample as given, then saturate toward it ----------------------------------------------------
  if (warp == 0) {
    int nn;
    double nd;
    nearest_warp<4, true>(g, wrap, prm.p, nn, nd);
    if (lane == 0) {
      double p[4] = {prm.p[0], prm.p[1], prm.p[2], prm.p[3]};
      if (prm.saturate) {
        const double4 c4 = g.pos[nn];
        const double c[4] = {c4.x, c4.y, c4.z, c4.w};
        dubins_saturate_point(p, c, prm.delta);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) s_p[k] = p[k];
      s_nearest = nn;
      s_nearest_dist = nd;
      s_count = 0;
      s_carry = 0;
    }
  }
  __syncthreads();
  const double q[4] = {s_p[0], s_p[1], s_p[2], s_p[3]};

  // ---- ball: range_query_kernel's WRAP path with both identities per candidate -----------------------------------
  const double r = prm.r, T = sqrt_thresh_lt(r);
  const double4 p0 = g.pos[0];
  const double s0 = sqdist<4>(q, p0.x, p0.y, p0.z, p0.w);
  const bool root_hit = __dsqrt_rn(s0) <= r;   // the root is admitted with <= by the real identity only (:896-898)
  auto emit = [&](bool hit, int node, double s) {
    const unsigned m = __ballot_sync(FULL, hit);
    int base = 0;
    if (lane == 0 && m) base = atomicAdd(&s_count, __popc(m));
    base = __shfl_sync(FULL, base, 0);
    if (hit) {
      const int k = base + __popc(m & lt);
      if (k < prm.capacity) {
        const double key = __dsqrt_rn(s);
        o.nbr[k] = node;
        o.h_idx[k] = node;
        o.h_dist[k] = key;
      }
    }
  };
  if (warp == 0) emit(lane == 0 && root_hit, 0, s0);
  if (r > 0.0) {   // r <= 0 or NaN: no strict hit is possible
    double qg[4];
    const bool ghost = make_ghost<4>(wrap, q, 1, r, qg);
    // the key comes from the first identity that reaches the node: the real one, then the ghost
    // (addToRangeList dedup, :765-771)
    auto test = [&](double px, double py, double pz, double pw, int node, double &s) -> bool {
      if (node == 0 && root_hit) return false;  // already listed
      s = sqdist<4>(q, px, py, pz, pw);
      if (s < T) return true;
      if (!ghost) return false;
      s = sqdist<4>(qg, px, py, pz, pw);
      return s < T;
    };
    if (g.n_sorted > 0) {
      const double r_infl = r * (1.0 + 1e-9);
      const double r2_infl = r_infl * r_infl;
      const int cy0 = cell_of(q[1] - r_infl, g.lo[1], g.inv[1], g.ny);
      const int cy1 = cell_of(q[1] + r_infl, g.lo[1], g.inv[1], g.ny);
      const int cz0 = cell_of(q[2] - r_infl, g.lo[2], g.inv[2], g.nz);
      const int cz1 = cell_of(q[2] + r_infl, g.lo[2], g.inv[2], g.nz);
      const int wy = cy1 - cy0 + 1;
      const int nrows = wy * (cz1 - cz0 + 1);
      for (int row = warp; row < nrows; row += EXD_WARPS) {
        const RowSpan sp = row_span<4>(g, q, r2_infl, cy0 + row % wy, cz0 + row / wy);
        for (int j0 = sp.start; j0 < sp.end; j0 += 32) {
          const int j = j0 + lane;
          bool hit = false;
          int node = 0;
          double s = 0.0;
          if (j < sp.end) {
            node = g.sperm[j];
            hit = test(g.sx[j], g.sy[j], g.sz[j], g.sw[j], node, s);
          }
          emit(hit, node, s);
        }
      }
    }
    for (int j0 = g.n_sorted + warp * 32; j0 < g.n_total; j0 += EXD_WARPS * 32) {   // unsorted tail
      const int j = j0 + lane;
      bool hit = false;
      double s = 0.0;
      if (j < g.n_total) {
        const double4 pp = g.pos[j];
        hit = test(pp.x, pp.y, pp.z, pp.w, j, s);
      }
      emit(hit, j, s);
    }
  }
  __syncthreads();
  const int count = s_count;
  const int n_edges = 2 * min(count, prm.capacity);

  // ---- edges: 2i = new -> nbr i, 2i+1 = nbr i -> new; one thread solves one word, a block scan places the rows ----
  for (int c0 = 0; c0 < n_edges; c0 += EXD_THREADS) {
    const int e = c0 + tid;
    int rows = 0;
    if (e < n_edges) {
      const double4 pn = g.pos[o.nbr[e >> 1]];
      const double nb[4] = {pn.x, pn.y, pn.z, pn.w};
      const bool rev = e & 1;
      double a[4], b[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) { a[k] = rev ? nb[k] : q[k]; b[k] = rev ? q[k] : nb[k]; }
      const Word w = solve(a, b, prm.r_turn);
      const WordRows L = word_layout(w, a, b);
      rows = L.total;
      o.layout[e] = L;
      o.dist[e] = w.dist;
      o.type[e] = w.type;
      o.h_edist[e] = w.dist;
      o.h_etype[e] = w.type;
    }
    int x = rows;   // inclusive scan within the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(FULL, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) s_wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {   // inclusive scan of the warp totals
      long long v = lane < EXD_WARPS ? s_wsum[lane] : 0;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(FULL, v, d);
        if (lane >= d) v += y;
      }
      if (lane < EXD_WARPS) s_wsum[lane] = v;
    }
    __syncthreads();
    const long long base = s_carry + (warp ? s_wsum[warp - 1] : 0);
    if (e < n_edges) o.ptr[e] = base + x - rows;
    __syncthreads();
    if (tid == 0) s_carry += s_wsum[EXD_WARPS - 1];
    __syncthreads();
  }
  if (tid == 0) {
    const long long total = s_carry;
    o.ptr[n_edges] = total;
#pragma unroll
    for (int k = 0; k < 4; ++k) dev->p[k] = q[k];
    dev->rows = total;
    dev->n_edges = n_edges;
    ExtendDubinsHeader h;
#pragma unroll
    for (int k = 0; k < 4; ++k) h.point[k] = q[k];
    h.count = count;
    h.nearest_idx = s_nearest;
    h.nearest_dist = s_nearest_dist;
    h.rows = total;
    h.seq = prm.seq - 1;  // the value the host still holds: unchanged until launch C's completion store
    *hdr = h;
  }
  __threadfence_system();
}

// launch B: the rows of every edge, one warp per edge (persistent grid)
__global__ void __launch_bounds__(256)
extend_dubins_emit_kernel(const ExtendDubinsDev *__restrict__ dev, const WordRows *__restrict__ layout,
                          const int64_t *__restrict__ ptr, double r_turn, int64_t row_cap, double2 *__restrict__ traj) {
  const int n_edges = dev->n_edges;
  if (dev->rows > row_cap) return;   // the host grows the scratch and repeats the call
  const int lane = lane_id();
  const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int e = warp0; e < n_edges; e += nwarps) {
    const WordRows L = layout[e];
    double2 *out = traj + ptr[e];
    for (int k = lane; k < L.total; k += 32) out[k] = word_row(L, r_turn, k);
  }
}

// launch C: Dubins explicitEdgeCheck of every edge OR-ed over the polygon set, one warp per edge (persistent grid);
// the last block to finish publishes the call number
__global__ void __launch_bounds__(256)
extend_dubins_check_kernel(GridView g, PolyView P, int ignore_active, const ExtendDubinsDev *__restrict__ dev,
                           const int32_t *__restrict__ nbr, const int64_t *__restrict__ ptr,
                           const double2 *__restrict__ traj, int64_t row_cap, double rho, double rho_coarse,
                           uint8_t *__restrict__ h_collide, uint32_t *done, unsigned long long seq,
                           ExtendDubinsHeader *hdr) {
  const int n_edges = dev->n_edges;
  if (dev->rows <= row_cap) {
    const double px = dev->p[0], py = dev->p[1];
    const int lane = lane_id();
    const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int e = warp0; e < n_edges; e += nwarps) {
      const double4 pn = g.pos[nbr[e >> 1]];
      const bool rev = e & 1;
      const double sx = rev ? pn.x : px, sy = rev ? pn.y : py, ex = rev ? px : pn.x, ey = rev ? py : pn.y;
      const bool collide = dubins_collide_warp(P, ignore_active != 0, AllObstacles{P.n}, sx, sy, ex, ey,
                                               (const double *)traj, ptr[e], ptr[e + 1], rho, rho_coarse);
      if (lane == 0) h_collide[e] = collide ? 1 : 0;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(done, 1u) == gridDim.x - 1) {
    *done = 0;
    __threadfence_system();
    *(volatile unsigned long long *)&hdr->seq = seq;
    __threadfence_system();
  }
}

struct ExtendDubinsState {   // per tree: mapped pinned result buffers + device scratch
  ExtendDubinsHeader *h_hdr = nullptr, *d_hdr = nullptr;
  int32_t *h_idx = nullptr, *d_idx = nullptr;
  double *h_dist = nullptr, *d_dist = nullptr;
  double *h_edist = nullptr, *d_edist = nullptr;
  int32_t *h_etype = nullptr, *d_etype = nullptr;
  uint8_t *h_ecol = nullptr, *d_ecol = nullptr;
  DevBuf<ExtendDubinsDev> dev;
  DevBuf<int32_t> nbr;
  DevBuf<WordRows> layout;
  rrtqx_dubins_result own;   // per-edge results and rows when the caller keeps no trajectories
  int capacity = 0;
  unsigned long long seq = 0;  // calls issued
  void free_arrays() {
    for (void *p : {(void *)h_idx, (void *)h_dist, (void *)h_edist, (void *)h_etype, (void *)h_ecol})
      if (p) cudaFreeHost(p);
    h_idx = nullptr; h_dist = nullptr; h_edist = nullptr; h_etype = nullptr; h_ecol = nullptr;
  }
  ~ExtendDubinsState() {
    if (h_hdr) cudaFreeHost(h_hdr);
    free_arrays();
  }
  void ensure(int cap, cudaStream_t st) {
    if (!h_hdr) {
      mapped_alloc(h_hdr, d_hdr, 1);
      memset(h_hdr, 0, sizeof(ExtendDubinsHeader));
      dev.ensure(1, st);
      RQ_CUDA(cudaMemsetAsync(dev.p, 0, sizeof(ExtendDubinsDev), st));
    }
    if (cap > capacity) {
      if (h_idx) { RQ_CUDA(cudaStreamSynchronize(st)); free_arrays(); }
      const int nc = std::max(cap, std::max(4096, 2 * capacity));
      mapped_alloc(h_idx, d_idx, (size_t)nc);
      mapped_alloc(h_dist, d_dist, (size_t)nc);
      mapped_alloc(h_edist, d_edist, 2 * (size_t)nc);
      mapped_alloc(h_etype, d_etype, 2 * (size_t)nc);
      mapped_alloc(h_ecol, d_ecol, 2 * (size_t)nc);
      capacity = nc;
    }
    nbr.ensure((size_t)capacity, st);
    layout.ensure(2 * (size_t)capacity, st);
  }
};

static ExtendDubinsState &extend_dubins_state(rrtqx_tree *t) {  // owned by the tree, freed in rrtqx_tree_destroy
  static const char tag = 0;
  return t->scratch.get<ExtendDubinsState>(&tag);
}

void extend_query_dubins(rrtqx_tree *t, const rrtqx_polygons *P, double *point, double delta, double range,
                         double robot_radius, double min_turn_radius, uint32_t flags, int32_t capacity,
                         int32_t *nearest_idx, double *nearest_dist, int32_t *n_neighbors, int32_t *nbr_idx,
                         double *nbr_dist, double *edge_dist, int32_t *edge_type, uint8_t *edge_collide,
                         rrtqx_dubins_result **trajectories) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(point != nullptr && !is_device_ptr(point), "point must be a host array");
  RQ_REQUIRE(capacity >= 0, "capacity is negative");
  RQ_REQUIRE(P->ctx == ctx, "polygons belong to another context");
  // the kernels know one layout: the DubinsEdge tree [x y t theta] with theta wrapped at 2 pi (DRRT.jl)
  const WrapInfo &w = t->wrap;
  if (!(t->d == 4 && w.num_wraps == 1 && w.wraps[0] == 3 && w.wrap_points[0] == 6.283185307179586))
    throw Error(RRTQX_ERR_UNSUPPORTED, "Dubins extend query needs d == 4 with one wrap: dimension 3, period 2 pi");
  if (t->n == 0) throw Error(RRTQX_ERR_EMPTY_TREE, "extend query on an empty tree");
  rrtqx_dubins_result *E = nullptr;
  if (trajectories) {
    E = *trajectories;
    if (!E) {
      E = new rrtqx_dubins_result();
      E->ctx = ctx;
      *trajectories = E;
    }
    RQ_REQUIRE(E->ctx == ctx, "result belongs to another context");
  }
  tree_prepare_query(t);
  ExtendDubinsState *es = &extend_dubins_state(t);
  es->ensure(std::max(capacity, 1), st);
  if (!E) E = &es->own;
  const size_t ne = 2 * (size_t)es->capacity;
  E->dist.ensure(ne, st);
  E->type.ensure(ne, st);
  E->ptr.ensure(ne + 1, st);
  E->traj.ensure((size_t)EXD_INITIAL_ROWS, st);
  ExtendDubinsParams prm;
  for (int c = 0; c < 4; ++c) prm.p[c] = point[c];
  prm.delta = delta;
  prm.r = range;
  prm.r_turn = min_turn_radius;
  prm.capacity = capacity;
  prm.saturate = (flags & RRTQX_EXTEND_SATURATE) ? 1 : 0;
  const int ignore_active = (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0;
  const double rho_coarse = robot_radius + 2 * min_turn_radius;  // S.robotRadius + 2*S.minTurningRadius (:758)
  // B and C: one warp per edge, at most 2 * capacity edges
  const int grid = std::max(1, std::min(ctx->sm_count * 4, div_up(2 * (int64_t)std::max(capacity, 1), 8)));
  ExtendDubinsOut o;
  o.nbr = es->nbr.p;
  o.h_idx = es->d_idx;
  o.h_dist = es->d_dist;
  o.dist = E->dist.p;
  o.type = E->type.p;
  o.ptr = E->ptr.p;
  o.h_edist = es->d_edist;
  o.h_etype = es->d_etype;
  o.layout = es->layout.p;
  ExtendDubinsHeader h;
  for (int attempt = 0;; ++attempt) {
    const int64_t row_cap = (int64_t)E->traj.cap;
    prm.seq = ++es->seq;
    GridView g = t->view();
    extend_dubins_query_kernel<<<1, EXD_THREADS, 0, st>>>(g, t->wrap, prm, o, es->dev.p, es->d_hdr);
    post_launch(ctx);
    extend_dubins_emit_kernel<<<grid, 256, 0, st>>>(es->dev.p, es->layout.p, E->ptr.p, min_turn_radius, row_cap,
                                                    E->traj.p);
    post_launch(ctx);
    extend_dubins_check_kernel<<<grid, 256, 0, st>>>(g, P->view(), ignore_active, es->dev.p, es->nbr.p, E->ptr.p,
                                                     E->traj.p, row_cap, robot_radius, rho_coarse, es->d_ecol,
                                                     &es->dev.p->done, prm.seq, es->d_hdr);
    post_launch(ctx);
    // wait for launch C's completion word (mapped pinned memory); a stream query every few thousand spins turns a
    // faulted launch into an error instead of a hang
    {
      volatile unsigned long long *seqp = &es->h_hdr->seq;
      for (unsigned spins = 0; *seqp != prm.seq; ++spins) {
        if ((spins & 0xfff) == 0xfff) {
          cudaError_t qe = cudaStreamQuery(st);
          if (qe == cudaSuccess) break;  // kernels finished: the word is visible on the next read
          if (qe != cudaErrorNotReady) RQ_CUDA(qe);
        }
      }
      std::atomic_thread_fence(std::memory_order_acquire);
      if (*seqp != prm.seq) RQ_CUDA(cudaStreamSynchronize(st));
    }
    h = *es->h_hdr;
    if (h.rows <= row_cap) break;
    // rare: the rows do not fit the grow-only scratch; grow it and repeat the call once
    RQ_REQUIRE(attempt == 0, "trajectory rows exceed the grown scratch");
    E->traj.ensure((size_t)h.rows, st);
  }
  if (nearest_idx) *nearest_idx = h.nearest_idx;
  if (nearest_dist) *nearest_dist = h.nearest_dist;
  if (n_neighbors) *n_neighbors = h.count;
  if (prm.saturate)
    for (int c = 0; c < 4; ++c) point[c] = h.point[c];
  const int m = std::min(h.count, capacity);
  for (int k = 0; k < m; ++k) {
    if (nbr_idx) nbr_idx[k] = es->h_idx[k];
    if (nbr_dist) nbr_dist[k] = es->h_dist[k];
  }
  for (int e = 0; e < 2 * m; ++e) {
    if (edge_dist) edge_dist[e] = es->h_edist[e];
    if (edge_type) edge_type[e] = es->h_etype[e];
    if (edge_collide) edge_collide[e] = es->h_ecol[e];
  }
  if (trajectories) {
    E->n_edges = 2 * m;
    E->n_rows = h.rows;
  }
}
