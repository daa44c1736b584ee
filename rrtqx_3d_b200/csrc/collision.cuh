// collision.cuh -- sphere-obstacle table and the exact segment/point-vs-sphere
// predicates of the QX-3D generation (DRRT_Q.jl:1205-1210, 1402-1590,
// 1775-1826), shared by the batched checks and the obstacle sweeps.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace rrtqx {
// process-wide unique stamps for obstacle-set contents: caches of derived tables (active-obstacle table, obstacle
// grid, cover lists, the extend_query table) are keyed on the stamp, so an upload / update invalidates them and a
// new object at a recycled address can never match an old key
inline uint64_t next_content_stamp() {
  static std::mutex mu;
  static uint64_t counter = 0;
  std::lock_guard<std::mutex> lk(mu);
  return ++counter;
}
}  // namespace rrtqx

struct rrtqx_spheres {
  rrtqx_ctx *ctx = nullptr;
  int64_t n = 0;
  uint64_t version = 0;  // content stamp, renewed by rrtqx_spheres_upload / rrtqx_spheres_update
  // SoA-in-AoS: (cx, cy, cz, radius) as one 32-byte record + active byte
  rrtqx::DevBuf<double4> rec;
  rrtqx::DevBuf<uint8_t> active;
};

namespace rrtqx {

#ifdef __CUDACC__

// Per-edge invariants of distancePointToSegment (DRRT_Q.jl:1205-1210):
// edgeLen = dist(startPoint,endPoint) and b = endPoint - startPoint.
struct SegPre {
  double sx, sy, sz;
  double bx, by, bz;
  double len;
  // conservative cull helpers (midpoint and half length, any rounding is fine:
  // the cull margin dwarfs it)
  double mx, my, mz, half;
  bool cullable;  // false when the reference result does not follow geometry
                  // (len == 0 -> t = NaN -> "collides with every active
                  // obstacle", or non-finite inputs)
};

__device__ __forceinline__ SegPre seg_prepare(double sx, double sy, double sz, double ex, double ey, double ez) {
  SegPre p;
  p.sx = sx; p.sy = sy; p.sz = sz;
  // dist(startPoint,endPoint): (s-e).^2 summed left to right
  double dx = __dsub_rn(sx, ex), dy = __dsub_rn(sy, ey), dz = __dsub_rn(sz, ez);
  double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  p.len = __dsqrt_rn(s);
  p.bx = __dsub_rn(ex, sx); p.by = __dsub_rn(ey, sy); p.bz = __dsub_rn(ez, sz);
  p.mx = 0.5 * (sx + ex); p.my = 0.5 * (sy + ey); p.mz = 0.5 * (sz + ez);
  p.half = 0.5 * p.len;
  p.cullable = (p.len > 0.0) && isfinite(p.len) && isfinite(p.mx) && isfinite(p.my) && isfinite(p.mz);
  return p;
}

// Radicand of dist(point, closePt) for obstacle centre (px,py,pz); the edge
// collides with the sphere iff !(sqrt(result) > robotRadius + radius)
// (explicitEdgeCheck3D DRRT_Q.jl:1789-1794).
template <bool FMA_DOT>
__device__ __forceinline__ double seg_point_radicand(const SegPre &e, double px, double py, double pz) {
  double ax = __dsub_rn(px, e.sx), ay = __dsub_rn(py, e.sy), az = __dsub_rn(pz, e.sz);
  double dot;
  if (FMA_DOT) {
    dot = __fma_rn(e.bx, ax, 0.0);
    dot = __fma_rn(e.by, ay, dot);
    dot = __fma_rn(e.bz, az, dot);
  } else {  // OpenBLAS ddot scalar tail: dot = 0.0; dot += y[i]*x[i]
    dot = __dadd_rn(0.0, __dmul_rn(e.bx, ax));
    dot = __dadd_rn(dot, __dmul_rn(e.by, ay));
    dot = __dadd_rn(dot, __dmul_rn(e.bz, az));
  }
  double t = jl_max(0.0, jl_min(1.0, __ddiv_rn(dot, e.len)));
  double cx = __dadd_rn(e.sx, __dmul_rn(t, e.bx));
  double cy = __dadd_rn(e.sy, __dmul_rn(t, e.by));
  double cz = __dadd_rn(e.sz, __dmul_rn(t, e.bz));
  double ux = __dsub_rn(px, cx), uy = __dsub_rn(py, cy), uz = __dsub_rn(pz, cz);
  return __dadd_rn(__dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy)), __dmul_rn(uz, uz));
}

// Exact collision decision for one (segment, sphere) pair.
//   thr    = robotRadius + radius          (rounded once, that order)
//   thr_le = sqrt_thresh_le(thr)           (sqrt(s) > thr  <=>  s > thr_le)
template <bool FMA_DOT>
__device__ __forceinline__ bool seg_sphere_collide(const SegPre &e, double px, double py, double pz, double thr,
                                                   double thr_le) {
  // Conservative reject: closePt always lies on the segment, so the
  // reference's D is >= the true point-segment distance >= |p - mid| - len/2.
  if (e.cullable) {
    double ux = px - e.mx, uy = py - e.my, uz = pz - e.mz;
    double lim = (thr + e.half) * (1.0 + 1e-9) + 1e-300;
    if (ux * ux + uy * uy + uz * uz > lim * lim && isfinite(lim)) return false;
  }
  double s = seg_point_radicand<FMA_DOT>(e, px, py, pz);
  (void)thr;
  return !(s > thr_le);  // NaN radicand -> collides, as !(NaN > x) in the reference
}

// FP32 form of the conservative reject for the grid kernels (the reject is a filter: it may only say "cannot
// collide" when that is certain).  u^ = fl32(c) - fl32(mid) differs from c - mid by at most
// sqrt(3) 2^-24 (|c|max + |mid|max) + 2^-24 |u^| in norm; `bound` is three times the first term, the 1e-5 factors
// cover the roundings of d2, lim and of thr / half (both rounded up).  Not cullable / not finite => never rejects.
struct SegF32 {
  float mx, my, mz, half, bound;
  bool ok;
};
__device__ __forceinline__ SegF32 seg_f32(const SegPre &e, float cmax) {
  SegF32 f;
  f.mx = __double2float_rn(e.mx); f.my = __double2float_rn(e.my); f.mz = __double2float_rn(e.mz);
  f.half = __double2float_ru(e.half);
  f.bound = 3.0e-7f * (cmax + fmaxf(fabsf(f.mx), fmaxf(fabsf(f.my), fabsf(f.mz))));
  f.ok = e.cullable && isfinite(f.bound) && isfinite(f.half);
  return f;
}
__device__ __forceinline__ bool seg_reject_f32(const SegF32 &f, const float4 c /* centre, thr rounded up */) {
  const float ux = c.x - f.mx, uy = c.y - f.my, uz = c.z - f.mz;
  const float d2 = ux * ux + uy * uy + uz * uz;
  const float lim = ((c.w + f.half) + f.bound) * 1.00001f;
  return f.ok && d2 > lim * lim * 1.00001f;  // NaN anywhere: comparison false, no reject
}
// exact decision without the FP64 reject (the caller has run the FP32 one)
template <bool FMA_DOT>
__device__ __forceinline__ bool seg_sphere_collide_exact(const SegPre &e, double px, double py, double pz, double thr_le) {
  return !(seg_point_radicand<FMA_DOT>(e, px, py, pz) > thr_le);
}

// Start-node filter of the obstacle sweeps (findPointsInConflictWithObstacle, DRRT_Q.jl:3195-3204): node v at squared
// distance s from the obstacle's centre is a candidate iff dist < searchRange, i.e. s < t_lt = T_lt(searchRange); the
// root is admitted with dist <= searchRange (kdTree_general.jl:896).  is_root: a bool, or a callable evaluated only when
// s < t_lt fails (a sink that has to load the start node).  The bool form lets the node-centric sweeps test both
// conditions with one predicate in their inner loop (the C3 sweep with statistics ran 14 % slower with the callable
// form on a B200 at 1000 W).
template <class IsRoot>
__device__ __forceinline__ bool start_node_in_range(double s, double t_lt, double search_range, IsRoot is_root) {
  bool in = s < t_lt;
  if constexpr (std::is_same_v<IsRoot, bool>) {
    if (!in && is_root) in = __dsqrt_rn(s) <= search_range;
  } else {
    if (!in) in = is_root() && __dsqrt_rn(s) <= search_range;
  }
  return in;
}

// ---------------------------------------------------------------- obstacle grid
// For large edge batches the active-obstacle table is binned into a small uniform grid (cell >= 2 *
// max(robotRadius + radius), at most 16^3 cells), so that an edge only meets the obstacles whose centre
// lies within (half edge length + thr_max) of its midpoint.  Conservative: sphere o can only collide
// if |c_o - mid| <= thr_o + L/2 (closePt lies on the segment), and the same monotone cell function bins
// the centres and bounds the edge's box.  Obstacles with non-finite centre / threshold go to an
// "always tested" bucket (the reference collides them with everything: !(NaN > x)).
struct SphGrid {
  int n_total;     // entries in the sorted table (binned + always)
  int nx, ny, nz;  // cells; bucket nx*ny*nz is the "always" list
  double lo[3], inv[3];
  double thr_max;
  float cmax;      // max |centre component| of the binned obstacles (error bound of the FP32 reject)
  double hi[3];    // upper corner of the box of the finite centres (lo[] is the lower one when binned)
  // Cover lists for short edges (collide_queue.cuh): a fine grid whose cell c lists every binned obstacle o
  // with dist(c_o, box(c)) <= thr_o + cov_cap, so an edge with half length <= cov_cap only meets the list of
  // the cell that holds its midpoint.  cov_on = 0: not built / over budget, use the coarse rows.
  int cov_on;
  int cnx, cny, cnz;
  double clo[3], cinv[3], ccell[3];
  double cov_cap, cov_margin;
  double cov_len2;  // an edge with squared length <= cov_len2 has half length <= cov_cap
};
constexpr int SG_MAX_DIM = 16;
constexpr int SG_MAX_CELLS = SG_MAX_DIM * SG_MAX_DIM * SG_MAX_DIM;
constexpr int COV_DIM = 32;
constexpr int COV_CELLS = COV_DIM * COV_DIM * COV_DIM;

__device__ __forceinline__ int sg_cell(double v, double lo, double inv, int n) {
  const int c = __double2int_rd((v - lo) * inv);  // floor, saturating; NaN -> 0
  return min(max(c, 0), n - 1);
}

// The binned obstacles segment e can collide with: the coarse rows within half + thr_max of its midpoint, then the
// non-finite bucket; a segment that cannot be culled meets the whole table.  run(lo, hi) visits the sorted entries
// [lo, hi) and returns true on a hit, which ends the walk; the result is whether some visit hit.
template <class Run>
__device__ __forceinline__ bool sg_walk(const SphGrid &G, const int32_t *__restrict__ cstart, const SegPre &e, Run run) {
  if (!e.cullable) return run(0, G.n_total);  // degenerate edge: the reference collides it with every active obstacle
  const double R = (e.half + G.thr_max) * (1.0 + 1e-9) + 1e-300;
  const int x0 = sg_cell(e.mx - R, G.lo[0], G.inv[0], G.nx), x1 = sg_cell(e.mx + R, G.lo[0], G.inv[0], G.nx);
  const int y0 = sg_cell(e.my - R, G.lo[1], G.inv[1], G.ny), y1 = sg_cell(e.my + R, G.lo[1], G.inv[1], G.ny);
  const int z0 = sg_cell(e.mz - R, G.lo[2], G.inv[2], G.nz), z1 = sg_cell(e.mz + R, G.lo[2], G.inv[2], G.nz);
  for (int z = z0; z <= z1; ++z)
    for (int y = y0; y <= y1; ++y) {
      const int cb = (z * G.ny + y) * G.nx;
      if (run(__ldg(&cstart[cb + x0]), __ldg(&cstart[cb + x1 + 1]))) return true;
    }
  const int ncell = G.nx * G.ny * G.nz;
  return run(__ldg(&cstart[ncell]), __ldg(&cstart[ncell + 1]));  // non-finite obstacles
}

// An obstacle table binned by sphere_grid_kernel: records in cell order, (thr, thr_le), the optional payload (the
// sweeps' start-node filter (T_lt(searchRange), searchRange)), the FP32 reject records, the cell starts and the header.
struct BinnedObstacles {
  const double4 *rec;
  const double2 *thr, *ext;
  const float4 *frec;
  const int32_t *cstart;
  const SphGrid *G;
};
struct BinnedObstacleBufs {
  DevBuf<double4> rec;
  DevBuf<double2> thr, ext;
  DevBuf<float4> frec;
  DevBuf<int32_t> cstart;
  DevBuf<unsigned char> grid;  // SphGrid header
  BinnedObstacles view() const { return {rec.p, thr.p, ext.p, frec.p, cstart.p, (const SphGrid *)grid.p}; }
};

static __global__ void sphere_grid_kernel(const double4 *__restrict__ rec, const double2 *__restrict__ thr,
                                          const double2 *__restrict__ extra /* optional payload */,
                                          const int32_t *__restrict__ n_live, int n_fixed, double4 *__restrict__ rec2,
                                          double2 *__restrict__ thr2, double2 *__restrict__ extra2,
                                          int32_t *__restrict__ cstart, SphGrid *__restrict__ G,
                                          float4 *__restrict__ frec2 /* FP32 reject records, sorted order */,
                                          int cover = 0 /* also set up the cover grid (collide_queue.cuh) */) {
  __shared__ int hist[SG_MAX_CELLS + 2];
  __shared__ double red[8][32];
  __shared__ SphGrid g;
  const int n = n_live ? *n_live : n_fixed;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  // bounding box of the finite centres and the largest finite threshold
  double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY}, tm = 0.0, cm = 0.0;
  for (int i = tid; i < n; i += blockDim.x) {
    const double4 r = rec[i];
    const double t = thr[i].x;
    if (isfinite(r.x) && isfinite(r.y) && isfinite(r.z) && isfinite(t)) {
      mn[0] = fmin(mn[0], r.x); mx[0] = fmax(mx[0], r.x);
      mn[1] = fmin(mn[1], r.y); mx[1] = fmax(mx[1], r.y);
      mn[2] = fmin(mn[2], r.z); mx[2] = fmax(mx[2], r.z);
      tm = fmax(tm, t);
      cm = fmax(cm, fmax(fabs(r.x), fmax(fabs(r.y), fabs(r.z))));
    }
  }
  double v[8] = {mn[0], mn[1], mn[2], mx[0], mx[1], mx[2], tm, cm};
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    for (int o = 16; o > 0; o >>= 1) {
      const double w = __shfl_xor_sync(FULL, v[k], o);
      v[k] = k < 3 ? fmin(v[k], w) : fmax(v[k], w);
    }
    if (lane == 0) red[k][warp] = v[k];
  }
  for (int i = tid; i < SG_MAX_CELLS + 2; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  if (tid == 0) {
    double r7[8];
    for (int k = 0; k < 8; ++k) {
      r7[k] = red[k][0];
      for (int w = 1; w < nw; ++w) r7[k] = k < 3 ? fmin(r7[k], red[k][w]) : fmax(r7[k], red[k][w]);
    }
    g.thr_max = r7[6];
    g.cmax = __double2float_ru(r7[7]);
    g.n_total = n;
    int dims[3];
    for (int c = 0; c < 3; ++c) {
      const double ext = r7[3 + c] - r7[c];
      double cell = fmax(2.0 * g.thr_max * (1.0 + 1e-9), ext / SG_MAX_DIM);
      if (!(ext > 0.0) || !isfinite(ext) || !(cell > 0.0) || !isfinite(cell)) {
        dims[c] = 1; g.lo[c] = 0.0; g.inv[c] = 0.0;
      } else {
        dims[c] = min(SG_MAX_DIM, (int)floor(ext / cell) + 1);
        g.lo[c] = r7[c];
        g.inv[c] = 1.0 / cell;
      }
    }
    g.nx = dims[0]; g.ny = dims[1]; g.nz = dims[2];
    // cover grid: the box of the centres grown by 1.25 thr_max, COV_DIM cells per dimension
    g.cov_on = 0;
    g.cnx = g.cny = g.cnz = 1;
    g.cov_cap = 0.0;
    g.cov_margin = 0.0;
    g.cov_len2 = -1.0;
    double cap = INFINITY, span = 0.0;
    bool ok = g.thr_max > 0.0;
    for (int c = 0; c < 3; ++c) {
      g.hi[c] = r7[3 + c];
      const double pad = 1.25 * g.thr_max;
      const double lo2 = r7[c] - pad, ext2 = (r7[3 + c] - r7[c]) + 2.0 * pad;
      ok = ok && isfinite(lo2) && isfinite(ext2) && ext2 > 0.0;
      g.clo[c] = lo2;
      g.ccell[c] = ext2 / COV_DIM;
      g.cinv[c] = COV_DIM / ext2;
      cap = fmin(cap, 0.5 * g.ccell[c]);
      span = fmax(span, ext2);
    }
    if (ok && isfinite(cap) && cap > 0.0 && isfinite(g.cinv[0]) && isfinite(g.cinv[1]) && isfinite(g.cinv[2])) {
      g.cov_on = cover ? 1 : 0;
      g.cnx = g.cny = g.cnz = COV_DIM;
      g.cov_cap = cap;
      g.cov_margin = 1e-9 * (r7[7] + span + g.thr_max);
      g.cov_len2 = 4.0 * cap * cap * (1.0 - 1e-9);
    }
    *G = g;
  }
  __syncthreads();
  const int ncell = g.nx * g.ny * g.nz;
  auto bucket = [&](int i) {
    const double4 r = rec[i];
    const double t = thr[i].x;
    if (!(isfinite(r.x) && isfinite(r.y) && isfinite(r.z) && isfinite(t))) return ncell;  // always tested
    return (sg_cell(r.z, g.lo[2], g.inv[2], g.nz) * g.ny + sg_cell(r.y, g.lo[1], g.inv[1], g.ny)) * g.nx +
           sg_cell(r.x, g.lo[0], g.inv[0], g.nx);
  };
  for (int i = tid; i < n; i += blockDim.x) atomicAdd(&hist[bucket(i)], 1);
  __syncthreads();
  if (tid == 0) {  // exclusive scan (<= 4097 buckets)
    int acc = 0;
    for (int c = 0; c <= ncell; ++c) { const int h = hist[c]; hist[c] = acc; cstart[c] = acc; acc += h; }
    cstart[ncell + 1] = acc;
  }
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) {
    const int o = atomicAdd(&hist[bucket(i)], 1);
    const double4 rr = rec[i];
    rec2[o] = rr;
    thr2[o] = thr[i];
    if (extra) extra2[o] = extra[i];
    if (frec2)  // non-finite obstacles (the "always" bucket) get NaN / Inf here: never rejected
      frec2[o] = make_float4(__double2float_rn(rr.x), __double2float_rn(rr.y), __double2float_rn(rr.z),
                             __double2float_ru(thr[i].x));
  }
}

#endif  // __CUDACC__

}  // namespace rrtqx
