// extend.cuh -- the planner's per-iteration geometric work in ONE launch (included by range.cu,
// inside namespace rrtqx):  rrtqx.jl:926-950 + extend() DRRT_Q.jl:2546-2641
//     (closest, d)  = kdFindNearest(KD, p)                       rrtqx.jl:926
//     explicitNodeCheck(S, newNode)                              rrtqx.jl:940
//     nodeList      = kdFindWithinRange(KD, r, p)                DRRT_Q.jl:2551
//     explicitEdgeCheck(S, edge(new -> n)) for n in nodeList     DRRT_Q.jl:1960   (findBestParent)
//     explicitEdgeCheck(S, edge(n -> new)) for n in nodeList     DRRT_Q.jl:2602   (reverse direction)
// One block works on the single query: warps split the candidate rows; hits are appended with a
// warp-aggregated shared counter; the obstacle table is prepared in shared memory by the same
// kernel; results are written straight into mapped pinned host memory, so an iteration costs one
// launch and one stream synchronisation (no staging copies).

constexpr int EXT_WARPS = 16;
constexpr int EXT_MAX_SPHERES = 768;

struct FGrid {
  float inv[3], cell[3];
};

__device__ __forceinline__ int clampi(float v, int n) {  // floor + clamp to [0, n-1]; NaN -> 0
  return (int)fminf(fmaxf(floorf(v), 0.0f), (float)(n - 1));
}

// Conservative cell range [cxa, cxb] of row (cy,cz) that can hold a point within r of the query at
// ff (cell units); false if the row is out of reach.
template <int D>
__device__ __forceinline__ bool row_cells(const GridView &g, const FGrid &fg, const float *ff, float r2f, int cy, int cz,
                                          int &cxa, int &cxb) {
  // lower bounds of |p.y - q.y|, |p.z - q.z| in cell units; boundary rows also
  // hold the points clamped in from beyond the grid, so they give no bound on
  // that side.  1e-3 cells of slack covers the FP32 error of ff (coordinates
  // up to 1024 cells: ulp 6e-5) and the FP64 rounding of cell_of().
  const float ninf = -INFINITY;
  float dyc = fmaxf(cy == 0 ? ninf : (float)cy - ff[1], cy == g.ny - 1 ? ninf : ff[1] - (float)(cy + 1));
  dyc = fmaxf(dyc - 1e-3f, 0.0f);
  const float dy = dyc * fg.cell[1];
  float rem = r2f - dy * dy;
  if (D >= 3) {
    float dzc = fmaxf(cz == 0 ? ninf : (float)cz - ff[2], cz == g.nz - 1 ? ninf : ff[2] - (float)(cz + 1));
    dzc = fmaxf(dzc - 1e-3f, 0.0f);
    const float dz = dzc * fg.cell[2];
    rem -= dz * dz;
  }
  if (isinf(r2f)) {  // unbounded query: whole row
    cxa = 0;
    cxb = g.nx - 1;
    return true;
  }
  if (!(rem >= 0.0f)) return false;
  const float xc = sqrtf(rem) * (1.0f + 1e-5f) * fg.inv[0] + 1e-3f;
  cxa = clampi(ff[0] - xc, g.nx);
  cxb = clampi(ff[0] + xc, g.nx);
  return true;
}

struct ExtendEntry {   // 16 bytes
  int32_t node;
  uint8_t fwd, rev;
  uint16_t pad;
  double dist;
};
struct ExtendHeader {
  int32_t count;          // neighbours found (may exceed capacity -> overflow)
  int32_t nearest_idx;
  double nearest_dist;
  int32_t point_collides;
  int32_t overflow;
  double cert;
  unsigned long long seq;  // written LAST by the kernel (after a system-scope fence): the host polls it
};
struct ExtendParams {
  double p[4];
  double r, T, rho;
  int32_t capacity;
  int32_t quick_pass, ignore_active, fma_dot;
  unsigned long long seq;  // call number, echoed into the header when every result is visible to the host
};

template <int D, bool FMA_DOT>
__global__ void __launch_bounds__(EXT_WARPS * 32, 1)
extend_query_kernel(GridView g, const ExtendParams prm, const double4 *__restrict__ sph_rec,
                    const uint8_t *__restrict__ sph_active, int n_sph, ExtendHeader *__restrict__ hdr,
                    ExtendEntry *__restrict__ ent /* device scratch */, ExtendEntry *__restrict__ ent_out /* mapped host */) {
  __shared__ double4 s_rec[EXT_MAX_SPHERES];
  __shared__ double2 s_thr[EXT_MAX_SPHERES];
  __shared__ int s_nsph, s_count;
  __shared__ double s_best_s[EXT_WARPS];
  __shared__ int s_best_n[EXT_WARPS];
  const int lane = lane_id(), warp = threadIdx.x >> 5, tid = threadIdx.x;
  const unsigned lt = lanemask_lt();
  if (tid == 0) { s_nsph = 0; s_count = 0; }
  __syncthreads();
  const double r = prm.r, T = prm.T, rho = prm.rho;
  double q[D];
#pragma unroll
  for (int c = 0; c < D; ++c) q[c] = prm.p[c];

  // obstacle table (active spheres, thr = rho + R, thr_le) -- order is irrelevant for OR / min
  for (int i = tid; i < n_sph; i += blockDim.x) {
    if (prm.ignore_active || sph_active[i]) {
      const int o = atomicAdd(&s_nsph, 1);
      const double4 rec = sph_rec[i];
      const double thr = __dadd_rn(rho, rec.w);
      s_rec[o] = rec;
      s_thr[o] = make_double2(thr, sqrt_thresh_le(thr));
    }
  }

  // ---- range search: warps split the rows -----------------------------------------------------
  double bs = INFINITY;   // per-lane best radicand / node among the hits (nearest = argmin over hits)
  int bn = 0x7fffffff;
  auto emit = [&](bool hit, int node, double s) {
    const unsigned m = __ballot_sync(FULL, hit);
    int base = 0;
    if (lane == 0 && m) base = atomicAdd(&s_count, __popc(m));
    base = __shfl_sync(FULL, base, 0);
    if (hit) {
      const int o = base + __popc(m & lt);
      if (o < prm.capacity) {
        ExtendEntry e;
        e.node = node; e.fwd = 0; e.rev = 0; e.pad = 0; e.dist = __dsqrt_rn(s);
        ent[o] = e;
      }
      if (s < bs || (s == bs && node < bn)) { bs = s; bn = node; }
    }
  };
  const double4 p0 = g.pos[0];
  const double s0 = sqdist<D>(q, p0.x, p0.y, p0.z, p0.w);
  const bool root_extra = !(s0 < T) && (__dsqrt_rn(s0) <= r);   // root admitted with <= (kdTree_general.jl:896-898)
  if (warp == 0) emit(lane == 0 && root_extra, 0, s0);

  if (r > 0.0) {
    if (g.n_sorted > 0) {
      FGrid fg;
#pragma unroll
      for (int c = 0; c < 3; ++c) { fg.inv[c] = (float)g.inv[c]; fg.cell[c] = (float)g.cell[c]; }
      float ff[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) ff[c] = c < D ? (float)((q[c] - g.lo[c]) * g.inv[c]) : 0.0f;
      const double ri = r * (1.0 + 1e-9);
      const float rf = __double2float_ru(ri) * (1.0f + 1e-6f);
      const float r2f = __double2float_ru(ri * ri) * (1.0f + 1e-5f);
      const int cy0 = clampi(ff[1] - (rf * fg.inv[1] + 1e-3f), g.ny), cy1 = clampi(ff[1] + (rf * fg.inv[1] + 1e-3f), g.ny);
      const int cz0 = D >= 3 ? clampi(ff[2] - (rf * fg.inv[2] + 1e-3f), g.nz) : 0;
      const int cz1 = D >= 3 ? clampi(ff[2] + (rf * fg.inv[2] + 1e-3f), g.nz) : 0;
      const int wy = cy1 - cy0 + 1;
      const int nrows = wy * (cz1 - cz0 + 1);
      for (int row = warp; row < nrows; row += EXT_WARPS) {
        const int cy = cy0 + row % wy, cz = cz0 + row / wy;
        int ca, cb;
        if (!row_cells<D>(g, fg, ff, r2f, cy, cz, ca, cb)) continue;
        const int rbase = (cz * g.ny + cy) * g.nx;
        const int a = g.cell_start[rbase + ca], b = g.cell_start[rbase + cb + 1];
        for (int j0 = a; j0 < b; j0 += 32) {
          const int j = j0 + lane;
          bool hit = false;
          double s = 0.0;
          int node = 0;
          if (j < b) {
            s = sqdist<D>(q, g.sx[j], g.sy[j], D >= 3 ? g.sz[j] : 0.0, D >= 4 ? g.sw[j] : 0.0);
            hit = s < T;
            if (hit) node = g.sperm[j];
          }
          emit(hit, node, s);
        }
      }
    }
    for (int j0 = g.n_sorted + warp * 32; j0 < g.n_total; j0 += EXT_WARPS * 32) {   // unsorted tail
      const int j = j0 + lane;
      bool hit = false;
      double s = 0.0;
      if (j < g.n_total) {
        const double4 pp = g.pos[j];
        s = sqdist<D>(q, pp.x, pp.y, pp.z, pp.w);
        hit = s < T;
      }
      emit(hit, j, s);
    }
  }
  __syncthreads();
  const int count = s_count;

  // ---- nearest ----------------------------------------------------------------------------------
  if (count == 0) {   // empty ball: brute force over the whole node table (rare: early planning only)
    for (int j = tid; j < g.n_total; j += blockDim.x) {
      const double4 pp = g.pos[j];
      const double s = sqdist<D>(q, pp.x, pp.y, pp.z, pp.w);
      if (s < bs || (s == bs && j < bn)) { bs = s; bn = j; }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double os = __shfl_xor_sync(FULL, bs, o);
    const int on = __shfl_xor_sync(FULL, bn, o);
    if (os < bs || (os == bs && on < bn)) { bs = os; bn = on; }
  }
  if (lane == 0) { s_best_s[warp] = bs; s_best_n[warp] = bn; }
  __syncthreads();

  // ---- node check of p (DRRT_Q.jl:1520-1556 / 1558-1590), evaluated by warp 0 in parallel -------------
  // The reference walks the list keeping retCert = running minimum of t_k = (dist_k - rho) - R_k, skips k
  // when t_k > retCert and returns a collision at the first t_k < 0.  A skipped k can neither lower the
  // minimum nor be negative (retCert >= 0 while no collision was found), and NaN never wins jl_min's `<`
  // update, so: collision <=> any t_k < 0 (or, in the quick pass, any !(dist_k > R_k)); certificate = minimum
  // of the non-NaN t_k.  Same values, evaluated by one lane per sphere.
  const int nsph = s_nsph;
  if (warp == 0) {
    for (int w = 1; w < EXT_WARPS; ++w)
      if (s_best_s[w] < bs || (s_best_s[w] == bs && s_best_n[w] < bn)) { bs = s_best_s[w]; bn = s_best_n[w]; }
    bool hit = false;
    double cert = INFINITY;
    for (int k0 = 0; k0 < nsph; k0 += 32) {
      const int k = k0 + lane;
      if (k < nsph) {
        const double c[3] = {s_rec[k].x, s_rec[k].y, s_rec[k].z};
        const double dist = __dsqrt_rn(sqdist<3>(c, q[0], q[1], D >= 3 ? q[2] : 0.0, 0.0));
        if (prm.quick_pass && !(dist > s_rec[k].w)) hit = true;
        const double t = __dsub_rn(__dsub_rn(dist, rho), s_rec[k].w);
        if (t < 0.0) hit = true;
        if (t < cert) cert = t;
      }
    }
    hit = __any_sync(FULL, hit);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cert = fmin(cert, __shfl_xor_sync(FULL, cert, o));
    // kdFindNearest keeps its first candidate, the root, when no radicand compares below +inf (NaN or huge sample
    // coordinates) and when the root's radicand is NaN (nothing compares below it): kdTree_general.jl:359-379
    if (bn == 0x7fffffff || s0 != s0) { bn = 0; bs = s0; }
    if (lane == 0) {
      ExtendHeader h;
      h.count = count;
      h.nearest_idx = bn;
      h.nearest_dist = __dsqrt_rn(bs);
      h.point_collides = hit ? 1 : 0;
      h.overflow = count > prm.capacity ? 1 : 0;
      h.cert = hit ? 0.0 : cert;
      h.seq = prm.seq - 1;  // the value the host still holds: unchanged until the completion store below
      *hdr = h;
    }
  }

  // ---- forward / reverse edge checks of every neighbour (SimpleEdge, 3-D): one thread per (neighbour,
  //      direction); the even lane of each pair writes the finished entry to the mapped host buffer with
  //      one 16-byte store (the host memory is never read back)
  const int m = min(count, prm.capacity);
  for (int t0 = 0; t0 < 2 * m; t0 += blockDim.x) {
    const int t = t0 + tid, k = t >> 1;
    const bool reverse = t & 1;
    bool h = false;
    ExtendEntry e;
    e.node = 0; e.fwd = 0; e.rev = 0; e.pad = 0; e.dist = 0.0;
    if (k < m) {
      e = ent[k];
      if (D == 3) {
        const double4 pn = g.pos[e.node];
        // new -> neighbour / neighbour -> new: the predicate is not symmetric in (start, end)
        const SegPre seg = reverse ? seg_prepare(pn.x, pn.y, pn.z, q[0], q[1], q[2]) : seg_prepare(q[0], q[1], q[2], pn.x, pn.y, pn.z);
        for (int o = 0; o < nsph && !h; ++o)
          h = seg_sphere_collide<FMA_DOT>(seg, s_rec[o].x, s_rec[o].y, s_rec[o].z, s_thr[o].x, s_thr[o].y);
      }
    }
    const bool h_other = __shfl_xor_sync(FULL, h, 1);
    if (k < m && !reverse) {
      e.fwd = h ? 1 : 0;
      e.rev = h_other ? 1 : 0;
      ent_out[k] = e;
    }
  }
  // completion: every thread's stores to the mapped host buffers are fenced to system scope, then one thread
  // publishes the call number; the host spins on that word instead of paying a stream synchronisation
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    *(volatile unsigned long long *)&hdr->seq = prm.seq;
    __threadfence_system();
  }
}

// Active obstacles compacted into a dense table (order irrelevant: the kernel takes an OR and a minimum over it).
// The reference's obstacle list only grows (expired agent obstacles stay in it with obstacleUnused = true,
// rrtqx.jl:462-530), so the 768-entry shared-memory table of the kernel is filled from the ACTIVE ones only.
__global__ void extend_compact_kernel(const double4 *__restrict__ rec, const uint8_t *__restrict__ active, int n,
                                      int ignore_active, double4 *__restrict__ out, int32_t *__restrict__ out_n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && (ignore_active || active[i])) out[atomicAdd(out_n, 1)] = rec[i];
}

struct ExtendState {   // per tree: mapped pinned result buffers + device scratch
  DevBuf<double4> act_rec;            // compacted active obstacles of the set last used
  DevBuf<int32_t> act_n;
  uint64_t act_version = 0;           // content stamp of that set (rrtqx_spheres::version); 0: none
  int act_ignore = -1, n_act = 0;
  ExtendHeader *h_hdr = nullptr, *d_hdr = nullptr;     // mapped pinned (host / device views)
  ExtendEntry *h_ent = nullptr, *d_ent_out = nullptr;  // mapped pinned
  DevBuf<ExtendEntry> scratch;
  int capacity = 0;
  unsigned long long seq = 0;  // calls issued
  ~ExtendState() {
    if (h_hdr) cudaFreeHost(h_hdr);
    if (h_ent) cudaFreeHost(h_ent);
  }
  void ensure(int cap, cudaStream_t st) {
    if (!h_hdr) {
      RQ_CUDA(cudaHostAlloc((void **)&h_hdr, sizeof(ExtendHeader), cudaHostAllocMapped));
      RQ_CUDA(cudaHostGetDevicePointer((void **)&d_hdr, h_hdr, 0));
      memset(h_hdr, 0, sizeof(ExtendHeader));
    }
    if (cap > capacity) {
      if (h_ent) { RQ_CUDA(cudaStreamSynchronize(st)); cudaFreeHost(h_ent); h_ent = nullptr; }
      int nc = std::max(cap, std::max(4096, 2 * capacity));
      RQ_CUDA(cudaHostAlloc((void **)&h_ent, sizeof(ExtendEntry) * (size_t)nc, cudaHostAllocMapped));
      RQ_CUDA(cudaHostGetDevicePointer((void **)&d_ent_out, h_ent, 0));
      capacity = nc;
    }
    scratch.ensure((size_t)capacity, st);
  }
};

static ExtendState &extend_state(rrtqx_tree *t) {  // owned by the tree, freed in rrtqx_tree_destroy
  static const char tag = 0;
  return t->scratch.get<ExtendState>(&tag);
}

void extend_query(rrtqx_tree *t, const rrtqx_spheres *S, const double *point, double range, double robot_radius,
                  uint32_t flags, int32_t capacity, int32_t *nearest_idx, double *nearest_dist,
                  uint8_t *point_collides, double *point_cert, int32_t *n_neighbors, int32_t *nbr_idx,
                  double *nbr_dist, uint8_t *fwd_collide, uint8_t *rev_collide) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(point != nullptr && !is_device_ptr(point), "point must be a host array");
  RQ_REQUIRE(capacity >= 0, "capacity is negative");
  // the kernel searches the real query point only: on a wrap-around tree its nearest node and neighbour list would
  // miss the ghost identities that kdFindNearest / kdFindWithinRange visit (ghostPoint.jl:60-111)
  if (t->wrap.num_wraps > 0)
    throw Error(RRTQX_ERR_UNSUPPORTED, "extend query on a wrap-around tree (use the batched nearest / range calls)");
  if (t->n == 0) throw Error(RRTQX_ERR_EMPTY_TREE, "extend query on an empty tree");
  tree_prepare_query(t);
  ExtendState *es = &extend_state(t);
  es->ensure(std::max(capacity, 1), st);
  const int ignore_active = (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0;
  if (es->act_version != S->version || es->act_ignore != ignore_active) {  // obstacle set changed since the last call
    es->act_rec.ensure((size_t)S->n + 1, st);
    es->act_n.ensure(4, st);
    RQ_CUDA(cudaMemsetAsync(es->act_n.p, 0, sizeof(int32_t), st));
    if (S->n > 0) {
      extend_compact_kernel<<<div_up(S->n, 256), 256, 0, st>>>(S->rec.p, S->active.p, (int)S->n, ignore_active, es->act_rec.p, es->act_n.p);
      post_launch(ctx);
    }
    int32_t na = 0;
    RQ_CUDA(cudaMemcpyAsync(&na, es->act_n.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    RQ_CUDA(cudaStreamSynchronize(st));
    es->n_act = na;
    es->act_version = S->version;
    es->act_ignore = ignore_active;
  }
  RQ_REQUIRE(es->n_act <= EXT_MAX_SPHERES, "extend_query supports at most 768 ACTIVE obstacles; use the batched calls");
  ExtendParams prm;
  for (int c = 0; c < 4; ++c) prm.p[c] = c < t->d ? point[c] : 0.0;
  prm.r = range;
  prm.T = host_sqrt_thresh_lt(range);
  prm.rho = robot_radius;
  prm.capacity = capacity;
  prm.quick_pass = (flags & RRTQX_CHECK_QUICK_PASS) ? 1 : 0;
  prm.ignore_active = 1;  // the table handed to the kernel holds the active obstacles only
  prm.fma_dot = (flags & RRTQX_CHECK_FMA_DOT) ? 1 : 0;
  prm.seq = ++es->seq;
  GridView g = t->view();
  {
    // no phase events here: two event records would cost more host time than the kernel's launch
#define RQ_EXT(D_, F_)                                                                                           \
  extend_query_kernel<D_, F_><<<1, EXT_WARPS * 32, 0, st>>>(g, prm, es->act_rec.p, nullptr, es->n_act, es->d_hdr, \
                                                            es->scratch.p, es->d_ent_out)
    const bool fma = prm.fma_dot;
    switch (t->d) {
      case 2: if (fma) RQ_EXT(2, true); else RQ_EXT(2, false); break;
      case 3: if (fma) RQ_EXT(3, true); else RQ_EXT(3, false); break;
      case 4: if (fma) RQ_EXT(4, true); else RQ_EXT(4, false); break;
      default: throw Error(RRTQX_ERR_UNSUPPORTED, "d must be 2, 3 or 4");
    }
#undef RQ_EXT
    post_launch(ctx);
  }
  // wait for the kernel's completion word (mapped pinned memory); a stream query every few thousand spins
  // turns a faulted launch into an error instead of a hang
  {
    volatile unsigned long long *seqp = &es->h_hdr->seq;
    for (unsigned spins = 0; *seqp != prm.seq; ++spins) {
      if ((spins & 0xfff) == 0xfff) {
        cudaError_t qe = cudaStreamQuery(st);
        if (qe == cudaSuccess) break;  // kernel finished: the word is visible on the next read
        if (qe != cudaErrorNotReady) RQ_CUDA(qe);
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (*seqp != prm.seq) RQ_CUDA(cudaStreamSynchronize(st));
  }
  const ExtendHeader h = *es->h_hdr;
  if (nearest_idx) *nearest_idx = h.nearest_idx;
  if (nearest_dist) *nearest_dist = h.nearest_dist;
  if (point_collides) *point_collides = (uint8_t)h.point_collides;
  if (point_cert) *point_cert = h.cert;
  if (n_neighbors) *n_neighbors = h.count;
  const int m = std::min(h.count, capacity);
  for (int k = 0; k < m; ++k) {
    const ExtendEntry &e = es->h_ent[k];
    if (nbr_idx) nbr_idx[k] = e.node;
    if (nbr_dist) nbr_dist[k] = e.dist;
    if (fwd_collide) fwd_collide[k] = e.fwd;
    if (rev_collide) rev_collide[k] = e.rev;
  }
}
