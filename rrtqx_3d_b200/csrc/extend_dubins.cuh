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

// Launch A's work for one instance, run by one block of EXD_THREADS threads: nearest, saturate, the ball, the edges'
// words and their row layout; thread 0 stores the point, the counts and the row total in *dev and *hdr.
__device__ __forceinline__ void extend_dubins_block(GridView g, WrapInfo wrap, const ExtendDubinsParams prm,
                                                    ExtendDubinsOut o, ExtendDubinsDev *__restrict__ dev,
                                                    ExtendDubinsHeader *__restrict__ hdr) {
  __shared__ double s_p[4];
  __shared__ int s_count, s_nearest;
  __shared__ double s_nearest_dist;
  __shared__ long long s_wsum[EXD_WARPS];
  __shared__ long long s_carry;
  // both query kernels run blocks of EXD_THREADS threads (their launch bounds); an inlined device function does not
  // inherit that range of threadIdx.x, and the index arithmetic is tighter with it
  __builtin_assume(threadIdx.x < EXD_THREADS);
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
}

__global__ void __launch_bounds__(EXD_THREADS, 1)
extend_dubins_query_kernel(GridView g, WrapInfo wrap, const ExtendDubinsParams prm, ExtendDubinsOut o,
                           ExtendDubinsDev *__restrict__ dev, ExtendDubinsHeader *__restrict__ hdr) {
  extend_dubins_block(g, wrap, prm, o, dev, hdr);
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

// ---- rrtqx_extend_query_dubins_multi: one iteration of n independent Dubins planners, same three launches ----------
//   A  one block per instance runs extend_dubins_block on that instance's descriptor and scratch slices; the last
//      block to finish (device ticket, reset for the next call) scans the instances' edge counts and row totals into
//      edge_base / row_base (n + 1 entries each, the totals last).
//   B  one warp per edge of the packed edge index space of all instances: the instance is found from edge_base, the
//      rows go to row_base[i] + the instance's own CSR pointer, and the packed dist / type / ptr of the trajectory
//      result are written.
//   C  one warp per packed edge: dubins_collide_warp over that instance's polygon set; the last block publishes the
//      call number.
// As in the single call, B and C skip their work when the rows exceed the scratch; the host grows it and repeats.

struct ExtendDubinsInstance {   // one instance of the multi call, staged in pinned memory and copied once per call
  GridView g;
  WrapInfo wrap;
  ExtendDubinsParams prm;
  ExtendDubinsOut o;            // the instance's slices of the context's scratch and mapped buffers
  PolyView P;
};

struct ExtendDubinsMultiDev {   // device memory: launch A's totals for B and C, and the two tickets
  int64_t rows;                 // rows of all instances
  int32_t n_edges;              // edges of all instances
  uint32_t ticket;              // blocks of launch A finished; the last one resets it
  uint32_t done;                // blocks of launch C finished; the last one resets it
};

// the instance whose edges [base[i], base[i+1]) hold packed edge e: the last i with base[i] <= e (empty instances
// share their base with the next one)
__device__ __forceinline__ int instance_of(const int32_t *__restrict__ base, int n, int e) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (base[mid] <= e) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(EXD_THREADS, 1)
extend_dubins_query_multi_kernel(const ExtendDubinsInstance *__restrict__ inst, ExtendDubinsDev *dev,
                                 ExtendDubinsHeader *__restrict__ hdr, ExtendDubinsMultiDev *md,
                                 int32_t *__restrict__ edge_base, int64_t *__restrict__ row_base,
                                 int64_t *__restrict__ ptr /* packed CSR pointers of the trajectory result */) {
  __shared__ ExtendDubinsInstance s_inst;
  __shared__ bool s_last;
  static_assert(sizeof(ExtendDubinsInstance) % sizeof(unsigned long long) == 0, "descriptor copied as 8-byte words");
  constexpr int WORDS = sizeof(ExtendDubinsInstance) / sizeof(unsigned long long);
  static_assert(WORDS <= EXD_THREADS, "one word per thread");
  if (threadIdx.x < WORDS)
    reinterpret_cast<unsigned long long *>(&s_inst)[threadIdx.x] =
        reinterpret_cast<const unsigned long long *>(inst + blockIdx.x)[threadIdx.x];
  __syncthreads();
  extend_dubins_block(s_inst.g, s_inst.wrap, s_inst.prm, s_inst.o, dev + blockIdx.x, hdr + blockIdx.x);
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&md->ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last || threadIdx.x >= 32) return;
  // exclusive scans of the edge counts and row totals, 32 instances per step (other blocks' stores: read past L1)
  const int lane = threadIdx.x, n = gridDim.x;
  int e_carry = 0;
  long long r_carry = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    const int i = i0 + lane;
    int e = 0;
    long long r = 0;
    if (i < n) {
      e = __ldcg(&dev[i].n_edges);
      r = __ldcg(reinterpret_cast<const long long *>(&dev[i].rows));
    }
    int ei = e;
    long long ri = r;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int ey = __shfl_up_sync(FULL, ei, d);
      const long long ry = __shfl_up_sync(FULL, ri, d);
      if (lane >= d) { ei += ey; ri += ry; }
    }
    if (i < n) {
      edge_base[i] = e_carry + ei - e;
      row_base[i] = r_carry + ri - r;
    }
    e_carry += __shfl_sync(FULL, ei, 31);
    r_carry += __shfl_sync(FULL, ri, 31);
  }
  if (lane == 0) {
    edge_base[n] = e_carry;
    row_base[n] = r_carry;
    ptr[e_carry] = r_carry;
    md->n_edges = e_carry;
    md->rows = r_carry;
    md->ticket = 0;
  }
}

// launch B of the multi call: the rows and the packed per-edge arrays, one warp per packed edge (persistent grid)
__global__ void __launch_bounds__(256)
extend_dubins_emit_multi_kernel(const ExtendDubinsMultiDev *__restrict__ md, const int32_t *__restrict__ edge_base,
                                const int64_t *__restrict__ row_base, int n, int64_t edge_stride,
                                const WordRows *__restrict__ layout, const int64_t *__restrict__ lptr,
                                const double *__restrict__ ldist, const int32_t *__restrict__ ltype, double r_turn,
                                int64_t row_cap, double2 *__restrict__ traj, double *__restrict__ dist,
                                int32_t *__restrict__ type, int64_t *__restrict__ ptr) {
  const int n_edges = md->n_edges;
  if (md->rows > row_cap) return;   // the host grows the scratch and repeats the call
  const int lane = lane_id();
  const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int e = warp0; e < n_edges; e += nwarps) {
    const int i = instance_of(edge_base, n, e);
    const int64_t s = i * edge_stride + (e - edge_base[i]);
    const WordRows L = layout[s];
    const int64_t at = row_base[i] + lptr[s];
    double2 *out = traj + at;
    for (int k = lane; k < L.total; k += 32) out[k] = word_row(L, r_turn, k);
    if (lane == 0) {
      dist[e] = ldist[s];
      type[e] = ltype[s];
      ptr[e] = at;
    }
  }
}

// launch C of the multi call: Dubins explicitEdgeCheck of every packed edge over its instance's polygon set, one warp
// per edge (persistent grid); the last block to finish publishes the call number
__global__ void __launch_bounds__(256)
extend_dubins_check_multi_kernel(const ExtendDubinsInstance *__restrict__ inst, const ExtendDubinsDev *__restrict__ dev,
                                 ExtendDubinsMultiDev *md, const int32_t *__restrict__ edge_base, int n,
                                 int64_t nbr_stride, int64_t edge_stride, int ignore_active,
                                 const int32_t *__restrict__ nbr, const int64_t *__restrict__ ptr,
                                 const double2 *__restrict__ traj, int64_t row_cap, double rho, double rho_coarse,
                                 uint8_t *__restrict__ h_collide, unsigned long long *h_done, unsigned long long seq) {
  const int n_edges = md->n_edges;
  if (md->rows <= row_cap) {
    const int lane = lane_id();
    const int warp0 = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int e = warp0; e < n_edges; e += nwarps) {
      const int i = instance_of(edge_base, n, e);
      const int el = e - edge_base[i];
      const PolyView P = inst[i].P;
      const double4 pn = inst[i].g.pos[nbr[i * nbr_stride + (el >> 1)]];
      const double px = dev[i].p[0], py = dev[i].p[1];
      const bool rev = el & 1;
      const double sx = rev ? pn.x : px, sy = rev ? pn.y : py, ex = rev ? px : pn.x, ey = rev ? py : pn.y;
      const bool collide = dubins_collide_warp(P, ignore_active != 0, AllObstacles{P.n}, sx, sy, ex, ey,
                                               (const double *)traj, ptr[e], ptr[e + 1], rho, rho_coarse);
      if (lane == 0) h_collide[i * edge_stride + el] = collide ? 1 : 0;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(&md->done, 1u) == gridDim.x - 1) {
    md->done = 0;
    __threadfence_system();
    *(volatile unsigned long long *)h_done = seq;
    __threadfence_system();
  }
}

struct ExtendDubinsMultiState {   // per context: descriptors, scratch and mapped results of the multi call
  ExtendDubinsInstance *h_inst = nullptr;               // pinned staging of the descriptors
  DevBuf<ExtendDubinsInstance> inst;
  ExtendDubinsHeader *h_hdr = nullptr, *d_hdr = nullptr;  // mapped pinned, one per instance
  DevBuf<ExtendDubinsDev> dev;                          // one per instance
  DevBuf<int32_t> edge_base;                            // n + 1
  DevBuf<int64_t> row_base;                             // n + 1
  DevBuf<ExtendDubinsMultiDev> md;
  unsigned long long *h_done = nullptr, *d_done = nullptr;  // mapped pinned completion word
  // per-instance slices: neighbours with stride ns = max(capacity, 1), edges with stride es = 2 ns + 1
  int32_t *h_idx = nullptr, *d_idx = nullptr;           // mapped
  double *h_dist = nullptr, *d_dist = nullptr;
  double *h_edist = nullptr, *d_edist = nullptr;
  int32_t *h_etype = nullptr, *d_etype = nullptr;
  uint8_t *h_ecol = nullptr, *d_ecol = nullptr;
  DevBuf<int32_t> nbr;
  DevBuf<WordRows> layout;
  DevBuf<double> dist;
  DevBuf<int32_t> type;
  DevBuf<int64_t> ptr;
  rrtqx_dubins_result own;   // packed per-edge results and rows when the caller keeps no trajectories
  int n_inst = 0;
  size_t n_nbr = 0, n_edge = 0;
  unsigned long long seq = 0;  // calls issued
  void free_instances() {
    for (void *p : {(void *)h_inst, (void *)h_hdr})
      if (p) cudaFreeHost(p);
    h_inst = nullptr; h_hdr = nullptr;
  }
  void free_slices() {
    for (void *p : {(void *)h_idx, (void *)h_dist, (void *)h_edist, (void *)h_etype, (void *)h_ecol})
      if (p) cudaFreeHost(p);
    h_idx = nullptr; h_dist = nullptr; h_edist = nullptr; h_etype = nullptr; h_ecol = nullptr;
  }
  ~ExtendDubinsMultiState() {
    free_instances();
    free_slices();
    if (h_done) cudaFreeHost(h_done);
  }
  // grow-only; every call waits for its own completion, so the buffers are idle between calls
  void ensure(int n, size_t nbrs, size_t edges, cudaStream_t st) {
    if (!h_done) {
      mapped_alloc(h_done, d_done, 1);
      *h_done = 0;
      md.ensure(1, st);
      RQ_CUDA(cudaMemsetAsync(md.p, 0, sizeof(ExtendDubinsMultiDev), st));
    }
    if (n > n_inst) {
      if (h_inst) { RQ_CUDA(cudaStreamSynchronize(st)); free_instances(); }
      const int nc = std::max(n, 2 * n_inst);
      RQ_CUDA(cudaHostAlloc((void **)&h_inst, sizeof(ExtendDubinsInstance) * (size_t)nc, cudaHostAllocDefault));
      mapped_alloc(h_hdr, d_hdr, (size_t)nc);
      inst.ensure((size_t)nc, st);
      dev.ensure((size_t)nc, st);
      edge_base.ensure((size_t)nc + 1, st);
      row_base.ensure((size_t)nc + 1, st);
      n_inst = nc;
    }
    if (nbrs > n_nbr || edges > n_edge) {
      if (h_idx) { RQ_CUDA(cudaStreamSynchronize(st)); free_slices(); }
      n_nbr = std::max(nbrs, n_nbr);
      n_edge = std::max(edges, n_edge);
      mapped_alloc(h_idx, d_idx, n_nbr);
      mapped_alloc(h_dist, d_dist, n_nbr);
      mapped_alloc(h_edist, d_edist, n_edge);
      mapped_alloc(h_etype, d_etype, n_edge);
      mapped_alloc(h_ecol, d_ecol, n_edge);
    }
    nbr.ensure(n_nbr, st);
    layout.ensure(n_edge, st);
    dist.ensure(n_edge, st);
    type.ensure(n_edge, st);
    ptr.ensure(n_edge, st);
  }
};

static ExtendDubinsMultiState &extend_dubins_multi_state(rrtqx_ctx *ctx) {  // owned by the context
  static const char tag = 0;
  return ctx->scratch.get<ExtendDubinsMultiState>(&tag);
}

void extend_query_dubins_multi(rrtqx_tree *const *trees, const rrtqx_polygons *const *polygons, int n, double *points,
                               const double *ranges, double delta, double robot_radius, double min_turn_radius,
                               uint32_t flags, int32_t capacity, int32_t *nearest_idx, double *nearest_dist,
                               int32_t *n_neighbors, int32_t *nbr_idx, double *nbr_dist, double *edge_dist,
                               int32_t *edge_type, uint8_t *edge_collide, rrtqx_dubins_result **trajectories) {
  RQ_REQUIRE(n >= 0, "n_instances is negative");
  if (n == 0) return;
  RQ_REQUIRE(trees != nullptr && polygons != nullptr, "trees / polygons is NULL");
  RQ_REQUIRE(capacity >= 0, "capacity is negative");
  RQ_REQUIRE(points != nullptr && !is_device_ptr(points), "points must be a host array");
  RQ_REQUIRE(ranges != nullptr && !is_device_ptr(ranges), "ranges must be a host array");
  rrtqx_ctx *ctx = trees[0] ? trees[0]->ctx : nullptr;
  std::set<const rrtqx_tree *> seen;
  for (int i = 0; i < n; ++i) {
    const rrtqx_tree *t = trees[i];
    if (!t || !polygons[i]) throw Error(RRTQX_ERR_INVALID, instance_msg(i, "NULL tree or polygon set"));
    if (t->ctx != ctx || polygons[i]->ctx != ctx) throw Error(RRTQX_ERR_INVALID, instance_msg(i, "handle of another context"));
    if (!seen.insert(t).second) throw Error(RRTQX_ERR_INVALID, instance_msg(i, "the same tree appears twice"));
  }
  for (int i = 0; i < n; ++i) {
    const rrtqx_tree *t = trees[i];
    const WrapInfo &w = t->wrap;
    if (!(t->d == 4 && w.num_wraps == 1 && w.wraps[0] == 3 && w.wrap_points[0] == 6.283185307179586))
      throw Error(RRTQX_ERR_UNSUPPORTED,
                  instance_msg(i, "Dubins extend query needs d == 4 with one wrap: dimension 3, period 2 pi"));
    if (t->n == 0) throw Error(RRTQX_ERR_EMPTY_TREE, instance_msg(i, "extend query on an empty tree"));
  }
  rrtqx_dubins_result *E = nullptr;
  if (trajectories) {
    E = *trajectories;
    RQ_REQUIRE(!E || E->ctx == ctx, "result belongs to another context");
  }
  cudaStream_t st = ctx->stream;
  const int64_t ns = std::max(capacity, 1), es = 2 * ns + 1;   // slice strides
  ExtendDubinsMultiState &ms = extend_dubins_multi_state(ctx);
  ms.ensure(n, (size_t)(ns * n), (size_t)(es * n), st);
  if (trajectories && !E) {
    E = new rrtqx_dubins_result();
    E->ctx = ctx;
    *trajectories = E;
  }
  if (!E) E = &ms.own;
  for (int i = 0; i < n; ++i) tree_prepare_query(trees[i]);
  const size_t ne = 2 * (size_t)ns * (size_t)n;   // packed edges of the call, at most
  E->dist.ensure(ne, st);
  E->type.ensure(ne, st);
  E->ptr.ensure(ne + 1, st);
  E->traj.ensure((size_t)EXD_INITIAL_ROWS, st);
  const int saturate = (flags & RRTQX_EXTEND_SATURATE) ? 1 : 0;
  const int ignore_active = (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0;
  const double rho_coarse = robot_radius + 2 * min_turn_radius;  // S.robotRadius + 2*S.minTurningRadius (:758)
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->sm_count * 4, div_up((int64_t)ne, 8)));
  for (int i = 0; i < n; ++i) {
    ExtendDubinsInstance &I = ms.h_inst[i];
    I.g = trees[i]->view();
    I.wrap = trees[i]->wrap;
    ExtendDubinsParams &prm = I.prm;
    for (int c = 0; c < 4; ++c) prm.p[c] = points[(size_t)i * 4 + c];
    prm.delta = delta;
    prm.r = ranges[i];
    prm.r_turn = min_turn_radius;
    prm.capacity = capacity;
    prm.saturate = saturate;
    prm.seq = 0;   // the per-instance header's seq is not polled: the call publishes one completion word
    ExtendDubinsOut &o = I.o;
    o.nbr = ms.nbr.p + ns * i;
    o.h_idx = ms.d_idx + ns * i;
    o.h_dist = ms.d_dist + ns * i;
    o.dist = ms.dist.p + es * i;
    o.type = ms.type.p + es * i;
    o.ptr = ms.ptr.p + es * i;
    o.h_edist = ms.d_edist + es * i;
    o.h_etype = ms.d_etype + es * i;
    o.layout = ms.layout.p + es * i;
    I.P = polygons[i]->view();
  }
  RQ_CUDA(cudaMemcpyAsync(ms.inst.p, ms.h_inst, sizeof(ExtendDubinsInstance) * (size_t)n, cudaMemcpyHostToDevice, st));
  int64_t rows = 0;
  for (int attempt = 0;; ++attempt) {
    const int64_t row_cap = (int64_t)E->traj.cap;
    const unsigned long long seq = ++ms.seq;
    extend_dubins_query_multi_kernel<<<n, EXD_THREADS, 0, st>>>(ms.inst.p, ms.dev.p, ms.d_hdr, ms.md.p,
                                                                ms.edge_base.p, ms.row_base.p, E->ptr.p);
    post_launch(ctx);
    extend_dubins_emit_multi_kernel<<<grid, 256, 0, st>>>(ms.md.p, ms.edge_base.p, ms.row_base.p, n, es,
                                                          ms.layout.p, ms.ptr.p, ms.dist.p, ms.type.p,
                                                          min_turn_radius, row_cap, E->traj.p, E->dist.p, E->type.p,
                                                          E->ptr.p);
    post_launch(ctx);
    extend_dubins_check_multi_kernel<<<grid, 256, 0, st>>>(ms.inst.p, ms.dev.p, ms.md.p, ms.edge_base.p, n, ns, es,
                                                           ignore_active, ms.nbr.p, E->ptr.p, E->traj.p, row_cap,
                                                           robot_radius, rho_coarse, ms.d_ecol, ms.d_done, seq);
    post_launch(ctx);
    wait_published(ms.h_done, seq, st);
    rows = 0;
    for (int i = 0; i < n; ++i) rows += ms.h_hdr[i].rows;
    if (rows <= row_cap) break;
    // rare: the rows do not fit the grow-only scratch; grow it and repeat the call once
    RQ_REQUIRE(attempt == 0, "trajectory rows exceed the grown scratch");
    E->traj.ensure((size_t)rows, st);
  }
  int64_t edges = 0;
  for (int i = 0; i < n; ++i) {
    const ExtendDubinsHeader h = ms.h_hdr[i];
    if (nearest_idx) nearest_idx[i] = h.nearest_idx;
    if (nearest_dist) nearest_dist[i] = h.nearest_dist;
    if (n_neighbors) n_neighbors[i] = h.count;
    if (saturate)
      for (int c = 0; c < 4; ++c) points[(size_t)i * 4 + c] = h.point[c];
    const int m = std::min(h.count, capacity);
    const size_t o = (size_t)capacity * i, oe = 2 * (size_t)capacity * i;
    for (int k = 0; k < m; ++k) {
      if (nbr_idx) nbr_idx[o + k] = ms.h_idx[ns * i + k];
      if (nbr_dist) nbr_dist[o + k] = ms.h_dist[ns * i + k];
    }
    for (int e = 0; e < 2 * m; ++e) {
      if (edge_dist) edge_dist[oe + e] = ms.h_edist[es * i + e];
      if (edge_type) edge_type[oe + e] = ms.h_etype[es * i + e];
      if (edge_collide) edge_collide[oe + e] = ms.h_ecol[es * i + e];
    }
    edges += 2 * m;
  }
  if (trajectories) {
    E->n_edges = edges;
    E->n_rows = rows;
  }
}
