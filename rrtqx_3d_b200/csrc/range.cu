// range.cu -- batched kdFindWithinRange (kdTree_general.jl:889-919) and
// kdFindNearest (:357-385) over the cell-sorted SoA index.
//
// Result semantics (SURVEY.md appendix A4/A6): the reference's pruned kd
// traversal returns exactly { n : fl(sqrt(s(q,n))) < r } (root admitted with
// <=), s being the left-to-right radicand of euclidianDist.  We evaluate the
// same s for every candidate the grid cannot exclude, and decide membership
// with the sqrt-free but equivalent test s < T_lt(r).  sqrt is paid on hits
// only (the returned JList key).
#include <atomic>
#include <cmath>
#include <cstdlib>

#include "dubins.cuh"
#include "objects.cuh"
#include "polygon.cuh"
#include "scan.cuh"

namespace rrtqx {

// ------------------------------------------------- sort queries by grid cell
// Sort key of a query: supercell-major (S x S x S blocks of grid cells), cell
// within the supercell minor.  Consecutive sorted queries are then spatial
// neighbours in ALL three directions, so the queries a block works on at any
// time share one compact candidate region (L1 reuse), and the two queries of a
// group have almost identical candidate rows.
template <int D>
__global__ void query_key_kernel(GridView g, int S, int F, int nsx, int nsy, const double *__restrict__ q, int64_t nq,
                                 int32_t *__restrict__ key, int32_t *__restrict__ hist) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const double *r = q + i * D;
  // sub-cell coordinates: F sub-cells per grid cell and direction
  const double f = (double)F;
  int cx = cell_of(r[0], g.lo[0], g.inv[0] * f, g.nx * F);
  int cy = cell_of(r[1], g.lo[1], g.inv[1] * f, g.ny * F);
  int cz = D >= 3 ? cell_of(r[2], g.lo[2], g.inv[2] * f, g.nz * F) : 0;
  const int SF = S * F;
  int sc = ((cz / SF) * nsy + cy / SF) * nsx + cx / SF;
  int local = ((cz % SF) * SF + cy % SF) * SF + cx % SF;
  int c = sc * (SF * SF * SF) + local;
  key[i] = c;
  atomicAdd(&hist[c], 1);
}

// Scatter into sorted order; also writes the query coordinates in sorted order so that the range
// kernel reads its queries with coalesced, L1-friendly loads (one dependent load less per group).
// `hist` still holds the bin counts of the key pass: every query takes the slot start[c] + (old count - 1) and
// counts its bin down, so the histogram is all-zero again when the kernel ends (no memset before the next sort).
template <int D>
__global__ void query_scatter_kernel(const int32_t *__restrict__ key, const double *__restrict__ q, int64_t nq,
                                     const int32_t *__restrict__ start, int32_t *__restrict__ hist,
                                     int32_t *__restrict__ order, double *__restrict__ qsorted) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  int c = key[i];
  const int pos = start[c] + atomicSub(&hist[c], 1) - 1;
  order[pos] = (int32_t)i;
#pragma unroll
  for (int k = 0; k < D; ++k) qsorted[(int64_t)pos * D + k] = q[i * D + k];
}

__global__ void iota_kernel(int32_t *__restrict__ a, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = (int32_t)i;
}

// Order in which warps pick up queries: grouped by the cell that contains the
// query so that neighbouring warps touch the same candidate slices (L1/L2 reuse).
template <int D>
static void sort_queries(rrtqx_tree *t, rrtqx_range_result *r, const double *dq, int64_t nq) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  const int TB = 256;
  r->qorder.ensure((size_t)nq, st);
  const int S = ctx->tune.qsort_s, F = ctx->tune.qsort_f;
  const int nsx = (t->nx + S - 1) / S, nsy = (t->ny + S - 1) / S, nsz = (t->nz + S - 1) / S;
  const int64_t nbins = (int64_t)nsx * nsy * nsz * S * S * S * F * F * F;
  r->qbins = 0;
  if (t->n_sorted == 0 || nq < 2048 || nbins > (int64_t)(1 << 28)) {
    iota_kernel<<<div_up(nq, TB), TB, 0, st>>>(r->qorder.p, nq);
    post_launch(ctx);
    return;
  }
  r->qbins = nbins;
  const int ncell = (int)nbins;
  r->qkey.ensure((size_t)nq, st);
  // the histogram is self-cleaning (query_scatter_kernel counts it back to zero): zero it only when the buffer is
  // new or a previous sort did not run to its end
  const bool fresh = r->qhist.cap < (size_t)ncell + 1 || !r->qhist_clean;
  r->qhist.ensure((size_t)ncell + 1, st);
  r->qstart.ensure((size_t)ncell + 1, st);
  if (fresh) RQ_CUDA(cudaMemsetAsync(r->qhist.p, 0, sizeof(int32_t) * r->qhist.cap, st));
  r->qhist_clean = false;
  GridView g = t->view();
  query_key_kernel<D><<<div_up(nq, TB), TB, 0, st>>>(g, S, F, nsx, nsy, dq, nq, r->qkey.p, r->qhist.p);
  post_launch(ctx);
  exclusive_scan<int32_t, int32_t>(ctx, r->qhist.p, ncell, r->qstart.p, r->scan_tmp32);
  r->qsorted.ensure((size_t)nq * D, st);
  query_scatter_kernel<D><<<div_up(nq, TB), TB, 0, st>>>(r->qkey.p, dq, nq, r->qstart.p, r->qhist.p, r->qorder.p, r->qsorted.p);
  post_launch(ctx);
  r->qhist_clean = true;
}

// --------------------------------------------------------- query identities
// The real query point plus its ghost identities in the order of
// getNextGhostPoint (ghostPoint.jl:60-111): pattern p = 1 .. 2^w-1, bit b of p
// wraps dimension wraps[w-1-b]; a ghost is used iff
// !(euclid(closestUnwrappedPoint, ghost) > bound) (:104).
template <int D>
__device__ inline bool make_ghost(const WrapInfo &w, const double *q, int pattern, double bound, double *ghost) {
  double closest[D];
#pragma unroll
  for (int k = 0; k < D; ++k) { ghost[k] = q[k]; closest[k] = q[k]; }
  for (int b = 0; b < w.num_wraps; ++b) {
    if (!((pattern >> b) & 1)) continue;
    int wi = w.num_wraps - 1 - b;
    int dim = w.wraps[wi];
    double P = w.wrap_points[wi];
    double gv, cv;
    if (q[dim] < P / 2.0) { gv = __dadd_rn(q[dim], P); cv = P; }   // :82-85
    else                  { gv = __dsub_rn(q[dim], P); cv = 0.0; } // :86-89
#pragma unroll
    for (int k = 0; k < D; ++k) if (k == dim) { ghost[k] = gv; closest[k] = cv; }
  }
  double s = sqdist<D>(closest, ghost[0], ghost[1], D >= 3 ? ghost[2] : 0.0, D >= 4 ? ghost[3] : 0.0);
  return !(__dsqrt_rn(s) > bound);
}

// ------------------------------------------------------------ range kernel
struct RowSpan { int start, end; };

// Conservative slice of row (cy,cz) that can contain points within r of q.
template <int D>
__device__ __forceinline__ RowSpan row_span(const GridView &g, const double *q, double r2_infl, int cy, int cz) {
  // lower bounds of |p.y-q.y| and |p.z-q.z| for points stored in this row;
  // boundary rows extend to infinity (clamped cells hold everything beyond).
  double dy = 0.0, dz = 0.0;
  {
    double ylo = g.lo[1] + cy * g.cell[1], yhi = ylo + g.cell[1];
    double a = (cy == 0) ? -INFINITY : ylo - q[1];
    double b = (cy == g.ny - 1) ? -INFINITY : q[1] - yhi;
    dy = fmax(0.0, fmax(a, b) - 1e-9 * g.cell[1] - 1e-12 * fabs(q[1]));
  }
  if (D >= 3) {
    double zlo = g.lo[2] + cz * g.cell[2], zhi = zlo + g.cell[2];
    double a = (cz == 0) ? -INFINITY : zlo - q[2];
    double b = (cz == g.nz - 1) ? -INFINITY : q[2] - zhi;
    dz = fmax(0.0, fmax(a, b) - 1e-9 * g.cell[2] - 1e-12 * fabs(q[2]));
  }
  RowSpan s;
  double rem = r2_infl - dy * dy - dz * dz;
  if (!(rem >= 0.0)) { s.start = 0; s.end = 0; return s; }
  double xr = isinf(rem) ? rem : sqrt(rem) * (1.0 + 1e-9) + 1e-12 * fabs(q[0]);
  int cxa = cell_of(q[0] - xr, g.lo[0], g.inv[0], g.nx);
  int cxb = cell_of(q[0] + xr, g.lo[0], g.inv[0], g.nx);
  int base = (cz * g.ny + cy) * g.nx;
  s.start = g.cell_start[base + cxa];
  s.end = g.cell_start[base + cxb + 1];
  return s;
}

// One warp per query.  FILL = false: count hits.  FILL = true: write idx/dist
// at offsets[q].  WRAP: tree has wrap-around dimensions (ghost identities).
template <int D, bool FILL, bool WRAP>
__global__ void __launch_bounds__(256)
range_query_kernel(GridView g, WrapInfo wrap, const double *__restrict__ queries, const int32_t *__restrict__ qorder,
                   int64_t nq, double r_uniform, const double *__restrict__ ranges, int32_t *__restrict__ counts,
                   const int64_t *__restrict__ offsets, int32_t *__restrict__ out_idx, double *__restrict__ out_dist) {
  const int lane = lane_id();
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const unsigned lt = lanemask_lt();

  for (int64_t qi = warp0; qi < nq; qi += nwarps) {
    const int qid = qorder[qi];
    const double r = ranges ? ranges[qid] : r_uniform;
    double q0[D];
#pragma unroll
    for (int k = 0; k < D; ++k) q0[k] = queries[(int64_t)qid * D + k];
    const double T = sqrt_thresh_lt(r);
    int64_t wbase = FILL ? offsets[qid] : 0;  // next free output slot
    int cnt = 0;                              // per-lane hit count (COUNT mode)

    // The root (node 0) is admitted with <= by the real identity only (:896-898).
    bool root_hit = false;
    {
      double4 p0 = g.pos[0];
      double s0 = sqdist<D>(q0, p0.x, p0.y, p0.z, p0.w);
      root_hit = (__dsqrt_rn(s0) <= r);
      if (root_hit) {
        if (FILL) {
          if (lane == 0) {
            out_idx[wbase] = 0;
            if (out_dist) out_dist[wbase] = __dsqrt_rn(s0);
          }
          wbase += 1;
        } else if (lane == 0) {
          cnt += 1;
        }
      }
    }
    if (!(r > 0.0)) {  // r <= 0 or NaN: no strict hit is possible
      if (!FILL) {
        cnt = __reduce_add_sync(FULL, cnt);
        if (lane == 0) counts[qid] = cnt;
      }
      continue;
    }

    const int n_ident = WRAP ? (1 << wrap.num_wraps) : 1;
    double qprev[WRAP ? ((1 << MAX_WRAPS) - 1) : 1][D];  // identities already searched
    int n_prev = 0;
    for (int ident = 0; ident < n_ident; ++ident) {
      double q[D];
      if (ident == 0) {
#pragma unroll
        for (int k = 0; k < D; ++k) q[k] = q0[k];
      } else {
        if (!make_ghost<D>(wrap, q0, ident, r, q)) continue;
      }
      // candidate test for one point; returns true if this identity is the
      // first to reach it
      auto test = [&](double px, double py, double pz, double pw, int node, double &s) -> bool {
        s = sqdist<D>(q, px, py, pz, pw);
        if (!(s < T)) return false;
        if (node == 0 && root_hit) return false;  // already listed
        if (WRAP) {
          for (int m = 0; m < n_prev; ++m) {
            double sm = sqdist<D>(qprev[m], px, py, pz, pw);
            if (sm < T) return false;  // an earlier identity found it (addToRangeList dedup, :765-771)
          }
        }
        return true;
      };
      auto emit = [&](bool hit, int node, double s) {
        if (FILL) {
          unsigned m = __ballot_sync(FULL, hit);
          if (hit) {
            int64_t o = wbase + __popc(m & lt);
            out_idx[o] = node;
            if (out_dist) out_dist[o] = __dsqrt_rn(s);
          }
          wbase += __popc(m);
        } else {
          cnt += hit ? 1 : 0;
        }
      };

      if (g.n_sorted > 0) {
        const double r_infl = r * (1.0 + 1e-9);
        const double r2_infl = r_infl * r_infl;
        const int cy0 = cell_of(q[1] - r_infl, g.lo[1], g.inv[1], g.ny);
        const int cy1 = cell_of(q[1] + r_infl, g.lo[1], g.inv[1], g.ny);
        const int cz0 = D >= 3 ? cell_of(q[2] - r_infl, g.lo[2], g.inv[2], g.nz) : 0;
        const int cz1 = D >= 3 ? cell_of(q[2] + r_infl, g.lo[2], g.inv[2], g.nz) : 0;
        const int wy = cy1 - cy0 + 1;
        const int nrows = wy * (cz1 - cz0 + 1);
        for (int rb = 0; rb < nrows; rb += 32) {
          RowSpan sp{0, 0};
          int row = rb + lane;
          if (row < nrows) sp = row_span<D>(g, q, r2_infl, cy0 + row % wy, cz0 + row / wy);
          const int lim = min(32, nrows - rb);
          for (int t = 0; t < lim; ++t) {
            const int a = __shfl_sync(FULL, sp.start, t);
            const int b = __shfl_sync(FULL, sp.end, t);
            for (int j0 = a; j0 < b; j0 += 32) {
              const int j = j0 + lane;
              bool hit = false;
              int node = 0;
              double s = 0.0;
              if (j < b) {
                node = g.sperm[j];
                hit = test(g.sx[j], g.sy[j], D >= 3 ? g.sz[j] : 0.0, D >= 4 ? g.sw[j] : 0.0, node, s);
              }
              emit(hit, node, s);
            }
          }
        }
      }
      // unsorted tail of recent inserts
      for (int j0 = g.n_sorted; j0 < g.n_total; j0 += 32) {
        const int j = j0 + lane;
        bool hit = false;
        double s = 0.0;
        if (j < g.n_total) {
          double4 p = g.pos[j];
          hit = test(p.x, p.y, p.z, p.w, j, s);
        }
        emit(hit, j, s);
      }
      // qprev holds 2^MAX_WRAPS - 1 identities: the last one is never needed (nothing is searched after it), and
      // storing it would write past the array with MAX_WRAPS wrap dimensions
      if (WRAP && ident + 1 < n_ident) {
#pragma unroll
        for (int k = 0; k < D; ++k) qprev[n_prev][k] = q[k];
        n_prev++;
      }
    }
    if (!FILL) {
      cnt = __reduce_add_sync(FULL, cnt);
      if (lane == 0) counts[qid] = cnt;
    }
  }
}

template <int D>
static void launch_range(rrtqx_tree *t, bool fill, const double *dq, const int32_t *qorder, int64_t nq, double r,
                         const double *ranges, int32_t *counts, const int64_t *offsets, int32_t *idx, double *dist) {
  rrtqx_ctx *ctx = t->ctx;
  GridView g = t->view();
  const int TB = 256;
  int64_t warps_needed = nq;
  int blocks = (int)std::min<int64_t>((warps_needed * 32 + TB - 1) / TB, (int64_t)ctx->sm_count * 8);
  if (blocks < 1) blocks = 1;
  const bool wrap = t->wrap.num_wraps > 0;
#define RQ_LAUNCH(FILL, WRAP)                                                                          \
  range_query_kernel<D, FILL, WRAP><<<blocks, TB, 0, ctx->stream>>>(g, t->wrap, dq, qorder, nq, r, ranges, counts, \
                                                                    offsets, idx, dist)
  if (fill) { if (wrap) RQ_LAUNCH(true, true); else RQ_LAUNCH(true, false); }
  else      { if (wrap) RQ_LAUNCH(false, true); else RQ_LAUNCH(false, false); }
#undef RQ_LAUNCH
  post_launch(ctx);
}

#include "range_v5.cuh"
#include "extend.cuh"

template <int D>
static void range_query_impl(rrtqx_tree *t, const double *queries, int64_t nq, double r, const double *ranges,
                             uint32_t flags, rrtqx_range_result *res) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  tree_prepare_query(t);
  const double *dq = to_device(ctx, queries, (size_t)nq * D, ctx->stage_f64);
  const double *dr = ranges ? to_device(ctx, ranges, (size_t)nq, ctx->stage_f64b) : nullptr;
  PhaseScope ph(ctx, "range_query");
  res->counts.ensure((size_t)nq + 1, st);
  res->offsets.ensure((size_t)nq + 1, st);
  // the single-pass kernels pack (slot << 4 | count) into 32-bit octet-table entries: slots below 2^27
  // ... and wrap-around trees when the identities' hit sets are provably disjoint (one wrap dimension, one radius
  // r <= period / 2: see ghost_expand_kernel); everything else takes the two-pass kernel with explicit dedup
  const bool ghost_ok = t->wrap.num_wraps == 1 && !ranges && std::isfinite(r) && r > 0.0 &&
                        r <= 0.5 * t->wrap.wrap_points[0] && nq < ((int64_t)1 << 29);
  if ((t->wrap.num_wraps == 0 || ghost_ok) && !ctx->tune.range_two_pass && t->n_sorted < ((int64_t)1 << 27)) {
    range_query_fused<D>(t, dq, dr, nq, r, flags, res);
    return;
  }
  {
    PhaseScope p2(ctx, "range_sort");
    sort_queries<D>(t, res, dq, nq);
  }
  {
    PhaseScope p2(ctx, "range_count");
    launch_range<D>(t, false, dq, res->qorder.p, nq, r, dr, res->counts.p, nullptr, nullptr, nullptr);
  }
  {
    PhaseScope p2(ctx, "range_scan");
    exclusive_scan<int32_t, int64_t>(ctx, res->counts.p, nq, res->offsets.p, res->scan_tmp64);
  }
  int64_t total = 0;
  RQ_CUDA(cudaMemcpyAsync(&total, res->offsets.p + nq, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  res->n_queries = nq;
  res->total = total;
  res->has_dist = false;
  res->has_lists = false;
  if (flags & RRTQX_RANGE_COUNT_ONLY) return;
  const bool want_dist = flags & RRTQX_RANGE_WANT_DIST;
  res->idx.ensure((size_t)total + 1, st, 0, 1.0);
  if (want_dist) res->dist.ensure((size_t)total + 1, st, 0, 1.0);
  {
    PhaseScope p2(ctx, "range_fill");
    launch_range<D>(t, true, dq, res->qorder.p, nq, r, dr, res->counts.p, res->offsets.p, res->idx.p,
                    want_dist ? res->dist.p : nullptr);
  }
  res->has_dist = want_dist;
  res->has_lists = true;
}

void range_query(rrtqx_tree *t, const double *queries, int64_t nq, double r, const double *ranges, uint32_t flags,
                 rrtqx_range_result *res) {
  RQ_REQUIRE(nq >= 0 && nq < (int64_t)0x7fffffff, "n_queries out of range");
  if (t->n == 0) throw Error(RRTQX_ERR_EMPTY_TREE, "range query on an empty tree (reference dereferences an undefined root)");
  if (nq == 0) {
    res->n_queries = 0;
    res->total = 0;
    res->has_lists = true;
    res->has_dist = flags & RRTQX_RANGE_WANT_DIST;
    return;
  }
  switch (t->d) {
    case 2: range_query_impl<2>(t, queries, nq, r, ranges, flags, res); break;
    case 3: range_query_impl<3>(t, queries, nq, r, ranges, flags, res); break;
    case 4: range_query_impl<4>(t, queries, nq, r, ranges, flags, res); break;
    default: throw Error(RRTQX_ERR_UNSUPPORTED, "d must be 2, 3 or 4");
  }
}

// ---------------------------------------------------------- nearest kernel
// One warp per query; cube of cells of growing half-width rho around the
// query's cell until no unseen cell can hold a closer point.
// nearest_warp: kdFindNearest of one query q0 by one warp (all 32 lanes take part); the result is warp-uniform.
// Shared by nearest_kernel and the fused Dubins extend query (extend_dubins.cuh).
template <int D, bool WRAP>
__device__ inline void nearest_warp(const GridView &g, const WrapInfo &wrap, const double *q0, int &out_node,
                                    double &out_dist) {
  const int lane = lane_id();
  {
    // best over all identities so far (distance = sqrt of radicand; strict <
    // replacement, kdTree_general.jl:375-379)
    double best_dist = INFINITY;
    int best_node = -1;

    const int n_ident = WRAP ? (1 << wrap.num_wraps) : 1;
    for (int ident = 0; ident < n_ident; ++ident) {
      double q[D];
      if (ident == 0) {
#pragma unroll
        for (int k = 0; k < D; ++k) q[k] = q0[k];
      } else {
        if (!make_ghost<D>(wrap, q0, ident, best_dist, q)) continue;
      }
      // per-lane running minimum of the radicand for this identity
      double bs = INFINITY;
      int bn = 0x7fffffff;
      auto consider = [&](double px, double py, double pz, double pw, int node) {
        double s = sqdist<D>(q, px, py, pz, pw);
        if (s < bs || (s == bs && node < bn)) { bs = s; bn = node; }
      };
      auto warp_min = [&]() {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          double os = __shfl_xor_sync(FULL, bs, o);
          int on = __shfl_xor_sync(FULL, bn, o);
          if (os < bs || (os == bs && on < bn)) { bs = os; bn = on; }
        }
      };
      // tail first (also seeds the bound)
      for (int j = g.n_sorted + lane; j < g.n_total; j += 32) {
        double4 p = g.pos[j];
        consider(p.x, p.y, p.z, p.w, j);
      }
      if (g.n_sorted > 0) {
        const int cx = cell_of(q[0], g.lo[0], g.inv[0], g.nx);
        const int cy = cell_of(q[1], g.lo[1], g.inv[1], g.ny);
        const int cz = D >= 3 ? cell_of(q[2], g.lo[2], g.inv[2], g.nz) : 0;
        const int max_rho = max(g.nx, max(g.ny, g.nz));
        for (int rho = 0; rho <= max_rho; ++rho) {
          const int x0 = max(cx - rho, 0), x1 = min(cx + rho, g.nx - 1);
          const int y0 = max(cy - rho, 0), y1 = min(cy + rho, g.ny - 1);
          const int z0 = max(cz - rho, 0), z1 = min(cz + rho, g.nz - 1);
          for (int z = z0; z <= z1; ++z)
            for (int y = y0; y <= y1; ++y) {
              const int base = (z * g.ny + y) * g.nx;
              // shell only: interior rows contribute just their two end cells
              const bool edge_row = (rho == 0) || (y == cy - rho) || (y == cy + rho) ||
                                    (D >= 3 && ((z == cz - rho) || (z == cz + rho)));
              if (edge_row) {
                const int a = g.cell_start[base + x0], b = g.cell_start[base + x1 + 1];
                for (int j = a + lane; j < b; j += 32)
                  consider(g.sx[j], g.sy[j], D >= 3 ? g.sz[j] : 0.0, D >= 4 ? g.sw[j] : 0.0, g.sperm[j]);
              } else {
                if (cx - rho >= 0) {
                  const int a = g.cell_start[base + cx - rho], b = g.cell_start[base + cx - rho + 1];
                  for (int j = a + lane; j < b; j += 32)
                    consider(g.sx[j], g.sy[j], D >= 3 ? g.sz[j] : 0.0, D >= 4 ? g.sw[j] : 0.0, g.sperm[j]);
                }
                if (cx + rho <= g.nx - 1) {
                  const int a = g.cell_start[base + cx + rho], b = g.cell_start[base + cx + rho + 1];
                  for (int j = a + lane; j < b; j += 32)
                    consider(g.sx[j], g.sy[j], D >= 3 ? g.sz[j] : 0.0, D >= 4 ? g.sw[j] : 0.0, g.sperm[j]);
                }
              }
            }
          warp_min();
          // lower bound on the distance of any point outside the scanned cube
          // (faces at the grid boundary do not count: nothing lies beyond).
          double bound = INFINITY;
          bool unseen = false;  // cells left outside the cube (their bound may be +inf for an infinite query)
          {
            double f;
            if (cx - rho > 0)          { f = q[0] - (g.lo[0] + (cx - rho) * g.cell[0]); bound = fmin(bound, f); unseen = true; }
            if (cx + rho < g.nx - 1)   { f = (g.lo[0] + (cx + rho + 1) * g.cell[0]) - q[0]; bound = fmin(bound, f); unseen = true; }
            if (cy - rho > 0)          { f = q[1] - (g.lo[1] + (cy - rho) * g.cell[1]); bound = fmin(bound, f); unseen = true; }
            if (cy + rho < g.ny - 1)   { f = (g.lo[1] + (cy + rho + 1) * g.cell[1]) - q[1]; bound = fmin(bound, f); unseen = true; }
            if (D >= 3) {
              if (cz - rho > 0)        { f = q[2] - (g.lo[2] + (cz - rho) * g.cell[2]); bound = fmin(bound, f); unseen = true; }
              if (cz + rho < g.nz - 1) { f = (g.lo[2] + (cz + rho + 1) * g.cell[2]) - q[2]; bound = fmin(bound, f); unseen = true; }
            }
          }
          // whole grid scanned.  An infinite bound alone does not end the search: a query with an infinite
          // coordinate has radicand +inf to every node, and the tie rule needs the smallest index among them all
          if (!unseen) break;
          // conservative: shrink the bound by the cell-geometry slack
          double slack = 1e-9 * fmax(g.cell[0], fmax(g.cell[1], g.cell[2])) +
                         1e-12 * (fabs(q[0]) + fabs(q[1]) + (D >= 3 ? fabs(q[2]) : 0.0));
          double bd = bound - slack;
          if (bd > 0.0 && bd * bd * (1.0 - 1e-9) > bs) break;
        }
      } else {
        warp_min();
      }
      if (g.n_sorted > 0 && g.n_total > g.n_sorted) warp_min();
      double dd = __dsqrt_rn(bs);
      if (bn != 0x7fffffff && (best_node < 0 || dd < best_dist)) {
        best_dist = dd;
        best_node = bn;
      }
    }
    {
      // the reference seeds its best distance with the root's (kdTree_general.jl:359-361) and replaces it only by
      // a strictly smaller one: it keeps the root when no radicand compared below +inf (NaN or infinite query
      // coordinates) and when the root's radicand is NaN (then nothing compares below it, ghosts included)
      const double4 p0 = g.pos[0];
      const double s0 = sqdist<D>(q0, p0.x, p0.y, p0.z, p0.w);
      if (best_node < 0 || s0 != s0) {
        best_node = 0;
        best_dist = __dsqrt_rn(s0);
      }
    }
    out_node = best_node;
    out_dist = best_dist;
  }
}

template <int D, bool WRAP>
__global__ void __launch_bounds__(256)
nearest_kernel(GridView g, WrapInfo wrap, const double *__restrict__ queries, const int32_t *__restrict__ qorder,
               int64_t nq, int32_t *__restrict__ out_idx, double *__restrict__ out_dist) {
  const int lane = lane_id();
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;

  for (int64_t qi = warp0; qi < nq; qi += nwarps) {
    const int qid = qorder[qi];
    double q0[D];
#pragma unroll
    for (int k = 0; k < D; ++k) q0[k] = queries[(int64_t)qid * D + k];
    int best_node;
    double best_dist;
    nearest_warp<D, WRAP>(g, wrap, q0, best_node, best_dist);
    if (lane == 0) {
      out_idx[qid] = best_node;
      if (out_dist) out_dist[qid] = best_dist;
    }
  }
}


// Thread-per-query nearest for large batches over a fully indexed tree (no unsorted tail, no wrap-around):
// a query needs its home cell and the few neighbouring cells closer than the best distance so far -- a dozen
// points -- so a warp per query idles 30 lanes.  The home cell (or the 3^3 block around an empty one) seeds
// the best radicand; the box of cells within that distance is then scanned, each cell skipped when a
// conservative lower bound of its distance exceeds the best radicand.  Queries whose box is wider than
// 2*NN_RHO_MAX+1 cells (far outside the grid, empty regions) are handed to the warp-per-query kernel.
// Result semantics identical to nearest_kernel: minimum radicand, ties to the smallest node index; a NaN radicand
// to the root answers (root, NaN).
constexpr int NN_RHO_MAX = 3;

template <int D>
__global__ void __launch_bounds__(128)
nearest_tpq_kernel(GridView g, const double *__restrict__ queries, const int32_t *__restrict__ qorder, int64_t nq,
                   int32_t *__restrict__ out_idx, double *__restrict__ out_dist, int32_t *__restrict__ unresolved,
                   int32_t *__restrict__ n_unresolved) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nq) return;
  const int qid = qorder[i];
  double q[D];
#pragma unroll
  for (int k = 0; k < D; ++k) q[k] = queries[(int64_t)qid * D + k];
  {
    // NaN radicand to the root: the reference's best distance starts as NaN and nothing compares below it
    const double4 p0 = g.pos[0];
    const double s0 = sqdist<D>(q, p0.x, p0.y, p0.z, p0.w);
    if (s0 != s0) {
      out_idx[qid] = 0;
      if (out_dist) out_dist[qid] = s0;
      return;
    }
  }
  double bs = INFINITY;
  int bn = 0x7fffffff;
  const int cx = cell_of(q[0], g.lo[0], g.inv[0], g.nx);
  const int cy = cell_of(q[1], g.lo[1], g.inv[1], g.ny);
  const int cz = D >= 3 ? cell_of(q[2], g.lo[2], g.inv[2], g.nz) : 0;
  const double slack = 1e-9 * fmax(g.cell[0], fmax(g.cell[1], g.cell[2])) +
                       1e-12 * (fabs(q[0]) + fabs(q[1]) + (D >= 3 ? fabs(q[2]) : 0.0));
  // conservative lower bound of |p_c - q_c| for a point stored in cell k of axis c (n cells).  Boundary cells are
  // open on their outer side: cell_of clamps into them whatever lies beyond the grid, and an axis whose bbox is not
  // finite (a +-inf node, an overflowing extent) is one cell [lo, lo + 1] that holds every point
  auto gap = [&](int c, int k, int n) {
    const double lo_k = g.lo[c] + k * g.cell[c], hi_k = lo_k + g.cell[c];
    const double a = (k == 0) ? -INFINITY : lo_k - q[c];
    const double b = (k == n - 1) ? -INFINITY : q[c] - hi_k;
    return fmax(0.0, fmax(a, b) - slack);
  };
  auto scan_cell = [&](int x, int y, int z) {
    const double gx = gap(0, x, g.nx), gy = gap(1, y, g.ny), gz = D >= 3 ? gap(2, z, g.nz) : 0.0;
    if ((gx * gx + gy * gy + gz * gz) * (1.0 - 1e-9) > bs) return;  // cannot beat (or tie) the best
    const int c = (z * g.ny + y) * g.nx + x;
    const int a = g.cell_start[c], b = g.cell_start[c + 1];
    for (int j = a; j < b; ++j) {
      const double4 p = g.d4[j];
      const int node = D <= 3 ? (int)__double_as_longlong(p.w) : g.sperm[j];
      const double s = sqdist<D>(q, p.x, p.y, p.z, p.w);
      if (s < bs || (s == bs && node < bn)) { bs = s; bn = node; }
    }
  };
  // 1. seed: the home cell, else (empty home cell) the 3 x 3 x 3 block around it
  bool done = false;
  scan_cell(cx, cy, cz);
  if (bn == 0x7fffffff) {
    for (int z = max(cz - 1, 0); z <= min(cz + 1, g.nz - 1); ++z)
      for (int y = max(cy - 1, 0); y <= min(cy + 1, g.ny - 1); ++y)
        for (int x = max(cx - 1, 0); x <= min(cx + 1, g.nx - 1); ++x)
          if (x != cx || y != cy || z != cz) scan_cell(x, y, z);
  }
  if (bn != 0x7fffffff) {
    // 2. every point that can beat or tie the seed lies within d = sqrt(bs) of q, hence (cell_of is monotone)
    // in the cells of the box [cell_of(q - d), cell_of(q + d)]; scan that box when it is small
    const double d = __dsqrt_rn(bs) * (1.0 + 1e-9) + slack;
    const int xa = cell_of(q[0] - d, g.lo[0], g.inv[0], g.nx), xb = cell_of(q[0] + d, g.lo[0], g.inv[0], g.nx);
    const int ya = cell_of(q[1] - d, g.lo[1], g.inv[1], g.ny), yb = cell_of(q[1] + d, g.lo[1], g.inv[1], g.ny);
    const int za = D >= 3 ? cell_of(q[2] - d, g.lo[2], g.inv[2], g.nz) : 0;
    const int zb = D >= 3 ? cell_of(q[2] + d, g.lo[2], g.inv[2], g.nz) : 0;
    if (xb - xa <= 2 * NN_RHO_MAX && yb - ya <= 2 * NN_RHO_MAX && zb - za <= 2 * NN_RHO_MAX && isfinite(d)) {
      for (int z = za; z <= zb; ++z)
        for (int y = ya; y <= yb; ++y)
          for (int x = xa; x <= xb; ++x) scan_cell(x, y, z);   // cells already seen are re-pruned or re-scanned (idempotent)
      done = true;
    }
  }
  if (done && bn != 0x7fffffff) {
    out_idx[qid] = bn;
    if (out_dist) out_dist[qid] = __dsqrt_rn(bs);
  } else {
    unresolved[atomicAdd(n_unresolved, 1)] = qid;  // finished by the warp-per-query kernel
  }
}

struct NearestScratch {
  rrtqx_range_result sortbuf;  // reuses the query sort buffers
  DevBuf<int32_t> idx;
  DevBuf<double> dist;
};

template <int D>
static void nearest_impl(rrtqx_tree *t, rrtqx_range_result *sortbuf, const double *queries, int64_t nq,
                         int32_t *idx_out, double *dist_out, DevBuf<int32_t> &idx_stage, DevBuf<double> &dist_stage) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  tree_prepare_query(t);
  const double *dq = to_device(ctx, queries, (size_t)nq * D, ctx->stage_f64);
  const bool idx_dev = is_device_ptr(idx_out), dist_dev = dist_out && is_device_ptr(dist_out);
  int32_t *didx = idx_out;
  double *ddist = dist_out;
  if (!idx_dev) { idx_stage.ensure((size_t)nq, st); didx = idx_stage.p; }
  if (dist_out && !dist_dev) { dist_stage.ensure((size_t)nq, st); ddist = dist_stage.p; }
  {
    // large batches over a tree without wrap-around: index the tail first, then one thread per query
    const bool tpq = t->wrap.num_wraps == 0 && nq >= 4096 && !ctx->tune.nearest_warp;
    if (tpq && t->n_sorted < t->n) tree_reindex(t);
    PhaseScope ph(ctx, "nearest");
    sort_queries<D>(t, sortbuf, dq, nq);
    GridView g = t->view();
    const int TB = 256;
    auto warp_kernel = [&](const int32_t *order, int64_t n) {
      int blocks = (int)std::min<int64_t>((n * 32 + TB - 1) / TB, (int64_t)ctx->sm_count * 8);
      if (blocks < 1) blocks = 1;
      if (t->wrap.num_wraps > 0)
        nearest_kernel<D, true><<<blocks, TB, 0, st>>>(g, t->wrap, dq, order, n, didx, ddist);
      else
        nearest_kernel<D, false><<<blocks, TB, 0, st>>>(g, t->wrap, dq, order, n, didx, ddist);
      post_launch(ctx);
    };
    if (tpq && t->n_sorted > 0) {
      sortbuf->qkey.ensure((size_t)nq + 1, st);          // free after the sort: list of unresolved queries
      t->flagbuf.ensure(8, st);
      RQ_CUDA(cudaMemsetAsync(t->flagbuf.p, 0, sizeof(int32_t), st));
      nearest_tpq_kernel<D><<<div_up(nq, 128), 128, 0, st>>>(g, dq, sortbuf->qorder.p, nq, didx, ddist, sortbuf->qkey.p,
                                                            t->flagbuf.p);
      post_launch(ctx);
      int32_t n_unres = 0;
      RQ_CUDA(cudaMemcpyAsync(&n_unres, t->flagbuf.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      RQ_CUDA(cudaStreamSynchronize(st));
      if (n_unres > 0) warp_kernel(sortbuf->qkey.p, n_unres);
    } else {
      warp_kernel(sortbuf->qorder.p, nq);
    }
  }
  if (!idx_dev) from_device(ctx, idx_out, didx, (size_t)nq);
  if (dist_out && !dist_dev) from_device(ctx, dist_out, ddist, (size_t)nq);
  RQ_CUDA(cudaStreamSynchronize(st));
}

void nearest_query(rrtqx_tree *t, rrtqx_range_result *sortbuf, const double *queries, int64_t nq, int32_t *idx_out,
                   double *dist_out, DevBuf<int32_t> &idx_stage, DevBuf<double> &dist_stage) {
  RQ_REQUIRE(nq >= 0 && nq < (int64_t)0x7fffffff, "n_queries out of range");
  RQ_REQUIRE(idx_out != nullptr || nq == 0, "idx_out is NULL");
  if (t->n == 0) throw Error(RRTQX_ERR_EMPTY_TREE, "nearest query on an empty tree (reference dereferences an undefined root)");
  if (nq == 0) return;
  switch (t->d) {
    case 2: nearest_impl<2>(t, sortbuf, queries, nq, idx_out, dist_out, idx_stage, dist_stage); break;
    case 3: nearest_impl<3>(t, sortbuf, queries, nq, idx_out, dist_out, idx_stage, dist_stage); break;
    case 4: nearest_impl<4>(t, sortbuf, queries, nq, idx_out, dist_out, idx_stage, dist_stage); break;
    default: throw Error(RRTQX_ERR_UNSUPPORTED, "d must be 2, 3 or 4");
  }
}

#include "extend_dubins.cuh"

}  // namespace rrtqx
