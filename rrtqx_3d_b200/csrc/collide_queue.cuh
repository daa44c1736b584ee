// collide_queue.cuh -- two-stage form of "does edge i collide with any binned sphere obstacle"
// (explicitEdgeCheck over the obstacle list, DRRT_Q.jl:1775-1826; the edge part of addNewObstacle,
// DRRT_Q.jl:3220-3290), used by the large-batch edge check and the edge-centric add sweep.
//
// The thread-per-edge kernels ran the long exact FP64 test (2 sqrt + 1 div, DRRT_Q.jl:1205-1210) under
// divergence: any lane that survived the cheap reject made the whole warp wait.  Here the stages are separate
// kernels.  pq_collect_kernel: one thread per edge finds the candidate obstacles of ITS edge and applies the
// FP32 conservative reject; surviving (edge, obstacle) pairs go through a per-block queue in shared memory to
// a global pair list (one atomic per block).  pq_test_kernel: one thread per pair runs the exact test (edge
// invariants recomputed from the endpoints) and marks the edge -- every lane busy, high occupancy.  The result
// is an OR over pairs, so order and duplicates do not matter.  Edges the scheme does not fit -- degenerate ones
// (no reject possible: the reference collides them with every active obstacle) and edges with more than
// PQ_KEEP surviving candidates -- are listed as items and decided by pq_slow_kernel with early exit.  Below the
// measured break-even the same pq_slow_kernel runs over every item instead (whole-range mode, one thread per item),
// so the thread-per-edge check and the two-stage one share the per-item walk of the binned table.  bin_obstacles
// bins an obstacle table for both forms and builds the cover lists.
//
// Cover lists: edges whose half length is at most G.cov_cap (half a cover cell) do not walk the coarse rows;
// they read the list of the one cover cell that holds their midpoint.  Obstacle o is on the list of cell c iff
// dist(c_o, box(c)) <= thr_o + cov_cap (+ margin), which contains every obstacle with |c_o - mid| <= thr_o +
// half for any midpoint in the cell; border cells extend to infinity, so midpoints outside the grid are
// covered too.  C3: about 1.3 candidates per edge instead of 16.  Lists have a fixed capacity per cell (one
// build pass, no scan; an entry is the 16-byte FP32 reject record with the obstacle number packed into it);
// an obstacle set too dense for that, or with more than 65536 obstacles, switches the cover off and every
// edge walks the coarse rows, as longer edges always do.
#pragma once
#include "collision.cuh"
#include <cstdlib>
#include <map>

namespace rrtqx {

#ifdef __CUDACC__

// ---------------------------------------------------------------- cover lists
constexpr int COV_CAPC = 32;  // entries per cover cell; a fuller cell switches the cover off (coarse rows instead)

struct SphCoverBufs {
  DevBuf<int32_t> cnt;                  // entries of each cover cell
  DevBuf<float4> list_f;                // COV_CAPC entries per cell: FP32 reject record with the obstacle number packed
                                        // into the low 16 bits of .w (threshold rounded up to the upper 16 bits)
  DevBuf<uint2> pairs;                  // (item, obstacle) pairs that survived the reject
  DevBuf<unsigned> slow;                // items decided by the slow kernels (list A, then list B)
  DevBuf<unsigned long long> n_pairs;   // [0] pairs, [1] slow list A, [2] slow list B
  uint64_t build_id = 0;                // renewed by every cover build (bin_obstacles): who built the lists last
};

// One warp per binned obstacle: append it to every cover cell it belongs to (fixed-capacity lists, so one pass,
// no scan).  cnt[] must be zero.
static __global__ void __launch_bounds__(256)
cover_register_kernel(const double4 *__restrict__ rec2, const double2 *__restrict__ thr2, const float4 *__restrict__ frec2,
                      const int32_t *__restrict__ cstart, SphGrid *__restrict__ Gp, int n_upper, int32_t *__restrict__ cnt,
                      float4 *__restrict__ list_f) {
  const int o = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (o >= n_upper) return;
  const SphGrid &G = *Gp;
  if (!G.cov_on) return;
  if (o >= cstart[G.nx * G.ny * G.nz]) return;  // the non-finite ones stay in the "always" bucket
  const double4 r = rec2[o];
  float4 fr = frec2[o];
  {  // .w = threshold, made coarser in the conservative direction (larger), + obstacle number (o < 65536)
    const unsigned b = __float_as_uint(fr.w);
    const unsigned up = (b >> 31) ? (b & 0xffff0000u) : ((b + 0xffffu) & 0xffff0000u);
    fr.w = __uint_as_float(up | (unsigned)o);
  }
  const double c[3] = {r.x, r.y, r.z};
  const double rho = (thr2[o].x + G.cov_cap) * (1.0 + 1e-9) + G.cov_margin;
  int a[3], n[3];
  for (int d = 0; d < 3; ++d) {
    a[d] = sg_cell(c[d] - rho, G.clo[d], G.cinv[d], COV_DIM);
    n[d] = sg_cell(c[d] + rho, G.clo[d], G.cinv[d], COV_DIM) - a[d] + 1;
  }
  const int total = n[0] * n[1] * n[2];
  for (int k = lane; k < total; k += 32) {
    const int i[3] = {a[0] + k % n[0], a[1] + (k / n[0]) % n[1], a[2] + k / (n[0] * n[1])};
    double d2 = 0.0;
    for (int d = 0; d < 3; ++d) {
      const double L = i[d] == 0 ? -INFINITY : G.clo[d] + i[d] * G.ccell[d];
      const double H = i[d] == COV_DIM - 1 ? INFINITY : G.clo[d] + (i[d] + 1) * G.ccell[d];
      const double g = fmax(fmax(L - c[d], c[d] - H), 0.0);
      d2 += g * g;
    }
    if (d2 <= rho * rho) {
      const int cell = (i[2] * COV_DIM + i[1]) * COV_DIM + i[0];
      const int p = atomicAdd(&cnt[cell], 1);
      if (p < COV_CAPC) {
        list_f[cell * COV_CAPC + p] = fr;
      } else {
        Gp->cov_on = 0;  // too dense for the cover: every consumer falls back to the coarse rows
      }
    }
  }
}

constexpr int COV_MAX_OBSTACLES = 65536;  // obstacle numbers are packed into 16 bits of the list entries

inline char g_cover_tag = 0;  // one key for all translation units (C++17 inline variable)
static inline SphCoverBufs &cover_bufs(rrtqx_ctx *ctx) {  // owned by the context, freed in rrtqx_ctx_destroy
  return ctx->scratch.get<SphCoverBufs>(&g_cover_tag);
}

// Bins an obstacle table (rec, thr and the optional payload ext; *n_live entries if n_live is not NULL, else n_upper)
// into B on the context's stream; cover: also (re)build the context's cover lists (n_upper <= COV_MAX_OBSTACLES).
static inline BinnedObstacles bin_obstacles(rrtqx_ctx *ctx, BinnedObstacleBufs &B, const double4 *rec, const double2 *thr,
                                            const double2 *ext, const int32_t *n_live, int n_upper, bool cover) {
  cudaStream_t st = ctx->stream;
  B.rec.ensure((size_t)n_upper + 1, st);
  B.thr.ensure((size_t)n_upper + 1, st);
  if (ext) B.ext.ensure((size_t)n_upper + 1, st);
  B.frec.ensure((size_t)n_upper + 1, st);
  B.cstart.ensure(SG_MAX_CELLS + 4, st);
  B.grid.ensure(sizeof(SphGrid) + 16, st);
  SphGrid *dG = (SphGrid *)B.grid.p;
  sphere_grid_kernel<<<1, 1024, 0, st>>>(rec, thr, ext, n_live, n_upper, B.rec.p, B.thr.p, ext ? B.ext.p : nullptr, B.cstart.p, dG,
                                         B.frec.p, cover ? 1 : 0);
  post_launch(ctx);
  if (cover) {
    SphCoverBufs &C = cover_bufs(ctx);
    C.build_id = next_content_stamp();
    C.cnt.ensure(COV_CELLS + 1, st);
    C.list_f.ensure((size_t)COV_CELLS * COV_CAPC, st);
    RQ_CUDA(cudaMemsetAsync(C.cnt.p, 0, (COV_CELLS + 1) * sizeof(int32_t), st));
    const unsigned blocks = (unsigned)div_up((int64_t)n_upper * 32, (int64_t)256);
    cover_register_kernel<<<blocks, 256, 0, st>>>(B.rec.p, B.thr.p, B.frec.p, B.cstart.p, dG, n_upper, C.cnt.p, C.list_f.p);
    post_launch(ctx);
  }
  return B.view();
}

// Batches below the threshold take the thread-per-item kernel (pq_item_launch): the cover build and the extra launches cost
// ~40 us, the two-stage path saves ~19 ns per 1000 edges in the batch check (break-even ~2e6 edges) and ~44 ns
// per 1000 items in the add sweep (break-even ~1e6).  The context's tuning (environment read at rrtqx_ctx_create /
// rrtqx_ctx_reload_tuning) can switch paths: RRTQX_EDGE_NO_QUEUE=1 forces the thread-per-item kernel,
// RRTQX_COVER_MIN_ITEMS=n moves the threshold.
constexpr int64_t PQ_MIN_ITEMS_BATCH = (int64_t)1 << 21, PQ_MIN_ITEMS_SWEEP = (int64_t)1 << 20;
static inline int64_t cover_min_items(const rrtqx_ctx *ctx, int64_t dflt) {
  if (ctx->tune.edge_no_queue) return INT64_MAX;
  return ctx->tune.cover_min_items >= 0 ? ctx->tune.cover_min_items : dflt;
}

// ---------------------------------------------------------------- per-item records of a resident edge set
// Built once per edge-set (re)build, in item order (out-edges in upload order, then one parent edge per node):
//   frec  = (fl32(mid.x), fl32(mid.y), fl32(mid.z), h)   h = FP32 upper bound of half the edge length;
//           h = -1: the item has no edge (node without parent); h = +inf: degenerate edge (zero length or non-finite
//           ends: the reference collides it with every active obstacle) -> decided by the slow kernel
//   exact = start.xyz, end.xyz as six doubles (three 16-byte loads)
// so the collect stage streams 16 bytes per item and never touches the node table, and the test stage reads the end
// points of the surviving pairs from consecutive records (pairs are listed in item order) instead of two random
// 32-byte gathers per pair.
struct ItemRecords {
  const float4 *frec;
  const double2 *exact;  // 3 per item
};

static __global__ void __launch_bounds__(256)
item_records_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                    const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
                    float4 *__restrict__ frec, double2 *__restrict__ exact) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_edges + n_nodes) return;
  int v, w;
  if (i >= n_edges) {
    v = (int)(i - n_edges);
    w = parent ? parent[v] : -1;
  } else {
    v = src[i];
    w = dst[i];
  }
  if (w < 0) {
    frec[i] = make_float4(0.f, 0.f, 0.f, -1.f);
    exact[3 * i] = exact[3 * i + 1] = exact[3 * i + 2] = make_double2(0.0, 0.0);
    return;
  }
  const double4 a = pos[v], b = pos[w];
  exact[3 * i] = make_double2(a.x, a.y);
  exact[3 * i + 1] = make_double2(a.z, b.x);
  exact[3 * i + 2] = make_double2(b.y, b.z);
  // the same quantities pq_collect_kernel derives from gathered end points
  const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y), dz = __dsub_rn(a.z, b.z);
  const double s2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  const double mx = 0.5 * (a.x + b.x), my = 0.5 * (a.y + b.y), mz = 0.5 * (a.z + b.z);
  float h;
  if (!(s2 > 0.0) || !isfinite(s2) || !isfinite(mx + my + mz)) {
    h = INFINITY;
  } else {
    float rt;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(__double2float_ru(s2)));
    h = 0.5f * (rt * 1.000001f) + 1e-19f;  // >= len / 2
  }
  frec[i] = make_float4(__double2float_rn(mx), __double2float_rn(my), __double2float_rn(mz), h);
}

// ---------------------------------------------------------------- pair queue
constexpr int PQ_THREADS = 128;  // collect kernel block
constexpr int PQ_KEEP = 4;       // pairs an item may put on the list; items with more go to the slow list
constexpr unsigned PQ_NONE = 0xffffffffu;  // filler pair (skipped by the test kernel)

// Src supplies the items:
//   static constexpr bool RESIDENT                                   true: per-item records were prepared when the edge
//                                                                    set was built (ItemRecords below): stage 1 streams
//                                                                    ONE coalesced 16-byte FP32 record per item instead
//                                                                    of gathering two node positions, and stage 2 reads
//                                                                    the exact end points from the item's own record
//   float4 frec(int64_t i)                                           (RESIDENT) FP32 record of item i
//   bool endpoints(int64_t i, double a[3], double b[3], int &v)   false: item has no edge (node without parent)
//   void clear(int64_t i)                                           item i is not hit (two-stage: before any test of it)
//   bool accept(int o, const double4 &rec, const double a[3], int v)  extra condition on a colliding pair
//   void mark(int64_t i)                                            some accepted obstacle collides with item i
//
// Stage 1: one thread per item.  Candidates that survive the FP32 reject are kept in registers (at most
// PQ_KEEP); at the end the thread publishes them as pairs through the block queue, or puts the ITEM on a slow
// list: list B (one warp per item) for degenerate edges (no reject possible, the reference collides them
// with every active obstacle) and long edges with more than PQ_KEEP survivors, list A (one thread per item)
// for short edges with more than PQ_KEEP survivors.  No exact arithmetic here, so the kernel stays small.
// The pair list holds `cap` pairs (2 per item); a block whose pairs do not fit any more turns its items into
// list A entries, so nothing is lost (each item is on at most one slow list, once).
template <class Src>
__global__ void __launch_bounds__(PQ_THREADS)
pq_collect_kernel(Src S, int64_t n_items, const float4 *__restrict__ frec, const int32_t *__restrict__ cstart,
                  const int32_t *__restrict__ cov_cnt,
                  const float4 *__restrict__ cov_frec, const SphGrid *__restrict__ Gp, uint2 *__restrict__ pairs,
                  unsigned long long cap, unsigned *__restrict__ slow_a, unsigned *__restrict__ slow_b,
                  unsigned long long *__restrict__ counters /* [0] pairs, [1] list A, [2] list B */) {
  const SphGrid &G = *Gp;  // uniform read-only loads
  __shared__ uint2 q[PQ_THREADS * PQ_KEEP];
  __shared__ int keep[PQ_KEEP][PQ_THREADS];  // surviving candidates of each thread
  __shared__ unsigned sq[PQ_THREADS];
  __shared__ unsigned qn, sna, snb;
  __shared__ unsigned long long qbase, sbase_a, sbase_b;
  if (threadIdx.x == 0) { qn = 0; sna = 0; snb = 0; }
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int nk = 0;
  bool to_slow = false, heavy = false;
  {
    double a[3], b[3];
    int v;
    // item invariants of this stage: midpoint (FP64 for the cell look-ups, FP32 for the reject), an FP32 upper
    // bound of the half length, and "degenerate" (no reject possible)
    bool have = false, degenerate = false;
    double mx = 0.0, my = 0.0, mz = 0.0;
    SegF32 sf;
    sf.mx = sf.my = sf.mz = sf.half = sf.bound = 0.f;
    sf.ok = false;
    if constexpr (Src::RESIDENT) {
      if (i < n_items) {
        const float4 fr = S.frec(i);      // ONE coalesced 16-byte load per item
        if (fr.w >= 0.f) {
          have = true;
          S.clear(i);
          degenerate = !(fr.w < INFINITY);
          sf.mx = fr.x; sf.my = fr.y; sf.mz = fr.z; sf.half = fr.w;
          mx = fr.x; my = fr.y; mz = fr.z;   // the FP32 midpoint picks the cells; its error goes into the margins below
        }
      }
    } else {
      if (i < n_items && S.endpoints(i, a, b, v)) {
        have = true;
        S.clear(i);
        // squared length as the reference's radicand (same operations as seg_prepare), so s2 == 0 / non-finite is
        // exactly len == 0 / non-finite; no FP64 sqrt: sqrt.approx upper bound
        const double dx = __dsub_rn(a[0], b[0]), dy = __dsub_rn(a[1], b[1]), dz = __dsub_rn(a[2], b[2]);
        const double s2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
        mx = 0.5 * (a[0] + b[0]); my = 0.5 * (a[1] + b[1]); mz = 0.5 * (a[2] + b[2]);
        degenerate = !(s2 > 0.0) || !isfinite(s2) || !isfinite(mx + my + mz);
        if (!degenerate) {
          sf.mx = __double2float_rn(mx); sf.my = __double2float_rn(my); sf.mz = __double2float_rn(mz);
          float rt;  // sqrt.approx: 1 ulp-level error, covered by the 1e-6 factor; + 1e-19 for flushed subnormals
          asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(__double2float_ru(s2)));
          sf.half = 0.5f * (rt * 1.000001f) + 1e-19f;  // >= len / 2
        }
      }
    }
    if (have) {
      if (degenerate) {
        to_slow = heavy = true;  // degenerate (or undecidable here): the slow kernel works it out exactly
      } else {
        sf.bound = 3.0e-7f * (G.cmax + fmaxf(fabsf(sf.mx), fmaxf(fabsf(sf.my), fabsf(sf.mz))));
        sf.ok = isfinite(sf.bound) && isfinite(sf.half);
        // cover lists serve edges with half length <= cov_cap.  RESIDENT: the midpoint used for the cell look-up is the
        // FP32 one, up to sf.bound / 3 away from the true midpoint per coordinate: that slack is part of cov_margin
        // only for the FP64 midpoint, so it is charged against the half length here.
        const float half_eff = Src::RESIDENT ? sf.half + sf.bound : sf.half;
        heavy = !(G.cov_on && (double)half_eff * (1.0 + 1e-6) <= G.cov_cap);
        auto visit = [&](int o, const float4 f) {
          if (seg_reject_f32(sf, f)) return;
          if (nk < PQ_KEEP) keep[nk][threadIdx.x] = o;
          ++nk;
        };
        const int ncell = G.nx * G.ny * G.nz;
        if (!heavy) {
          const int c = (sg_cell(mz, G.clo[2], G.cinv[2], COV_DIM) * COV_DIM + sg_cell(my, G.clo[1], G.cinv[1], COV_DIM)) * COV_DIM +
                        sg_cell(mx, G.clo[0], G.cinv[0], COV_DIM);
          const int k1 = c * COV_CAPC + cov_cnt[c];  // cov_on => no cell over capacity
          for (int k = c * COV_CAPC; k < k1; ++k) {
            float4 f = cov_frec[k];
            const unsigned w = __float_as_uint(f.w);
            f.w = __uint_as_float(w & 0xffff0000u);
            visit((int)(w & 0xffffu), f);
          }
        } else {
          const double R = ((double)half_eff + G.thr_max) * (1.0 + 1e-6) + 1e-300;  // half_eff >= len / 2 (+ midpoint slack)
          const int x0 = sg_cell(mx - R, G.lo[0], G.inv[0], G.nx), x1 = sg_cell(mx + R, G.lo[0], G.inv[0], G.nx);
          const int y0 = sg_cell(my - R, G.lo[1], G.inv[1], G.ny), y1 = sg_cell(my + R, G.lo[1], G.inv[1], G.ny);
          const int z0 = sg_cell(mz - R, G.lo[2], G.inv[2], G.nz), z1 = sg_cell(mz + R, G.lo[2], G.inv[2], G.nz);
          for (int z = z0; z <= z1; ++z)
            for (int y = y0; y <= y1; ++y) {
              const int cb = (z * G.ny + y) * G.nx;
              const int o1 = cstart[cb + x1 + 1];
              for (int o = cstart[cb + x0]; o < o1; ++o) visit(o, frec[o]);
            }
        }
        const int o1 = cstart[ncell + 1];
        for (int o = cstart[ncell]; o < o1; ++o) visit(o, frec[o]);  // non-finite obstacles: met by every edge
        to_slow = nk > PQ_KEEP;
      }
    }
  }
  __syncthreads();  // qn, sna, snb initialised
  if (to_slow) {  // list A from the front of sq, list B from its back
    if (heavy) sq[PQ_THREADS - 1 - atomicAdd(&snb, 1u)] = (unsigned)i;
    else       sq[atomicAdd(&sna, 1u)] = (unsigned)i;
  } else if (nk) {
    const unsigned k0 = atomicAdd(&qn, (unsigned)nk);
    for (int k = 0; k < nk; ++k) q[k0 + k] = make_uint2((unsigned)i, (unsigned)keep[k][threadIdx.x]);
  }
  __syncthreads();
  const unsigned n = qn, na = sna, nb = snb;
  if (threadIdx.x == 0 && n) qbase = atomicAdd(&counters[0], (unsigned long long)n);
  if (threadIdx.x == 32 && na) sbase_a = atomicAdd(&counters[1], (unsigned long long)na);
  if (threadIdx.x == 64 && nb) sbase_b = atomicAdd(&counters[2], (unsigned long long)nb);
  __syncthreads();
  if (n && qbase + n > cap) {  // pair list full: fillers into what is left of it, the items go to list A
    for (unsigned k = threadIdx.x; k < n; k += blockDim.x)
      if (qbase + k < cap) pairs[qbase + k] = make_uint2(PQ_NONE, 0u);
    if (nk && !to_slow) slow_a[atomicAdd(&counters[1], 1ull)] = (unsigned)i;
  } else {
    for (unsigned k = threadIdx.x; k < n; k += blockDim.x) pairs[qbase + k] = q[k];
  }
  if (threadIdx.x < na) slow_a[sbase_a + threadIdx.x] = sq[threadIdx.x];
  if (threadIdx.x < nb) slow_b[sbase_b + threadIdx.x] = sq[PQ_THREADS - 1 - threadIdx.x];
}

// Stage 2: one thread per pair, exact test (edge invariants recomputed from the endpoints).
template <bool FMA_DOT, class Src>
__global__ void __launch_bounds__(256)
pq_test_kernel(Src S, const double4 *__restrict__ rec, const double2 *__restrict__ thr, const uint2 *__restrict__ pairs,
               unsigned long long cap, const unsigned long long *__restrict__ counters) {
  const unsigned long long n = min(counters[0], cap);
  for (unsigned long long p = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; p < n;
       p += (unsigned long long)gridDim.x * blockDim.x) {
    const uint2 e = pairs[p];
    if (e.x == PQ_NONE) continue;
    double a[3], b[3];
    int v;
    S.endpoints((int64_t)e.x, a, b, v);
    const SegPre pre = seg_prepare(a[0], a[1], a[2], b[0], b[1], b[2]);
    const double4 r = rec[e.y];
    if (seg_sphere_collide_exact<FMA_DOT>(pre, r.x, r.y, r.z, thr[e.y].y) && S.accept((int)e.y, r, a, v)) S.mark((int64_t)e.x);
  }
}

// Items decided in place, every candidate of the item's rows, the item ends at its first hit.  ALL = false: the items
// of a slow list (*count of them), WARP = false: one thread per item (list A: short edges with many surviving
// candidates), WARP = true: one warp per item, the candidates of a row spread over the lanes (list B: degenerate and
// long edges, which may meet most of the table).  ALL = true (WARP = false): every item, one thread each, the p-th
// thread deciding item p (n_all of them) -- the thread-per-edge path of batches below the two-stage break-even; each
// item is marked or cleared, an item without an edge is skipped and never marked.  A separate instantiation, so that the
// list loop does not raise its register count.
template <bool FMA_DOT, bool WARP, class Src, bool ALL = false>
__global__ void __launch_bounds__(ALL ? 256 : 128)
pq_slow_kernel(Src S, BinnedObstacles T, const unsigned *__restrict__ slow, const unsigned long long *__restrict__ count,
               int64_t n_all) {
  static_assert(!(ALL && WARP), "whole-range mode is one thread per item");
  __shared__ SphGrid G;
  if (threadIdx.x == 0) G = *T.G;
  __syncthreads();
  const int lane = WARP ? (threadIdx.x & 31) : 0, step = WARP ? 32 : 1;
  auto collides = [&](const double a[3], const double b[3], int v) {
    const SegPre pre = seg_prepare(a[0], a[1], a[2], b[0], b[1], b[2]);
    const SegF32 sf = seg_f32(pre, G.cmax);
    return sg_walk(G, T.cstart, pre, [&](int lo, int hi) {
      bool h = false;  // warp-uniform when WARP
      for (int o0 = lo; o0 < hi && !h; o0 += step) {
        const int o = o0 + lane;
        bool ho = false;
        if (o < hi && !seg_reject_f32(sf, __ldg(&T.frec[o]))) {  // never rejects a degenerate edge (sf.ok false)
          const double2 cxy = __ldg(reinterpret_cast<const double2 *>(&T.rec[o]));  // (radius unused)
          const double4 r = make_double4(cxy.x, cxy.y, __ldg(&T.rec[o].z), 0.0);
          ho = seg_sphere_collide_exact<FMA_DOT>(pre, r.x, r.y, r.z, __ldg(&T.thr[o].y)) && S.accept(o, r, a, v);
        }
        h = WARP ? __any_sync(FULL, ho) : ho;
      }
      return h;
    });
  };
  double a[3], b[3];
  int v;
  if constexpr (ALL) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_all) return;
    if (!S.endpoints(i, a, b, v)) return;  // invalid end point index: counted and cleared by the source
    if constexpr (Src::RESIDENT)
      if (S.frec(i).w < 0.f) return;     // no edge (node without parent): its exact record is all zeros
    if (collides(a, b, v)) S.mark(i);
    else S.clear(i);
  } else {
    const unsigned long long n = *count;
    const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long nthr = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long p = WARP ? tid >> 5 : tid; p < n; p += WARP ? nthr >> 5 : nthr) {
      const int64_t i = (int64_t)slow[p];
      S.endpoints(i, a, b, v);
      if (collides(a, b, v) && lane == 0) S.mark(i);
    }
  }
}

// The four kernels of the two-stage form on the context's stream.  Requires n_items < 2^32 (32-bit item numbers in
// the lists) and the cover lists of T's table, if its header has them switched on.
template <bool FMA_DOT, class Src>
static inline void pq_launch(rrtqx_ctx *ctx, const Src &S, int64_t n_items, const BinnedObstacles &T) {
  cudaStream_t st = ctx->stream;
  SphCoverBufs &B = cover_bufs(ctx);
  const unsigned long long cap = 2ull * (unsigned long long)n_items + 1024;
  B.pairs.ensure((size_t)cap, st);
  B.slow.ensure(2 * (size_t)n_items + 2, st);
  B.n_pairs.ensure(4, st);
  unsigned *slow_a = B.slow.p, *slow_b = B.slow.p + n_items + 1;
  RQ_CUDA(cudaMemsetAsync(B.n_pairs.p, 0, 4 * sizeof(unsigned long long), st));
  pq_collect_kernel<Src><<<(unsigned)div_up(n_items, (int64_t)PQ_THREADS), PQ_THREADS, 0, st>>>(S, n_items, T.frec, T.cstart, B.cnt.p,
                                                                                                  B.list_f.p, T.G, B.pairs.p, cap, slow_a, slow_b, B.n_pairs.p);
  const unsigned tblocks = (unsigned)std::min<int64_t>(div_up((int64_t)cap, (int64_t)256), (int64_t)ctx->sm_count * 8);
  pq_test_kernel<FMA_DOT, Src><<<tblocks, 256, 0, st>>>(S, T.rec, T.thr, B.pairs.p, cap, B.n_pairs.p);
  const unsigned ablocks = (unsigned)std::min<int64_t>(div_up(n_items, (int64_t)128), (int64_t)ctx->sm_count * 4);
  pq_slow_kernel<FMA_DOT, false, Src><<<ablocks, 128, 0, st>>>(S, T, slow_a, B.n_pairs.p + 1, 0);
  const unsigned bblocks = (unsigned)std::min<int64_t>(div_up(n_items, (int64_t)4), (int64_t)ctx->sm_count * 8);
  pq_slow_kernel<FMA_DOT, true, Src><<<bblocks, 128, 0, st>>>(S, T, slow_b, B.n_pairs.p + 2, 0);
  post_launch(ctx, 4);
}

// Thread-per-item form (batches below the two-stage break-even): pq_slow_kernel over every item.
template <bool FMA_DOT, class Src>
static inline void pq_item_launch(rrtqx_ctx *ctx, const Src &S, int64_t n_items, const BinnedObstacles &T) {
  pq_slow_kernel<FMA_DOT, false, Src, true><<<(unsigned)div_up(n_items, (int64_t)256), 256, 0, ctx->stream>>>(S, T, nullptr, nullptr, n_items);
  post_launch(ctx);
}

#endif  // __CUDACC__

}  // namespace rrtqx
