// item_grid.cuh -- obstacle-centric form of "which resident edges collide with these sphere obstacles"
// (explicitEdgeCheck over an obstacle list, DRRT_Q.jl:1775-1826; the edge part of addNewObstacle, DRRT_Q.jl:3220-3290).
//
// The edge-centric kernels (collide_queue.cuh) let every edge look for its obstacles: 10^7 threads, each with its own
// list look-up, its own handful of candidates and its own queue traffic -- 335 warp-instructions per 32 edges, most of
// them bookkeeping.  A resident edge set allows the opposite decomposition, because its items (out-edges, then one
// parent edge per node) do not change between obstacle events:
//
//   * at (re)build time the items are counting-sorted by the cell of their midpoint in a uniform grid (about 32 items
//     per cell) into sorted SoA records: the FP32 reject record (midpoint, half-length bound), the exact end points
//     (three 16-byte arrays) and the item number; every cell also keeps hmax = the largest half length of its items;
//   * a sweep enumerates WORK UNITS (obstacle o, cell c) with dist(c_o, box(c)) <= thr_o + hmax[c] (+ slack): only those
//     cells can hold an item that collides with o, because the reference's closest point lies ON the segment, so a
//     collision needs |c_o - mid| <= thr_o + len/2 (DRRT_Q.jl:1205-1210);
//   * one warp per unit streams the cell's records -- contiguous, coalesced, the obstacle in registers -- applies the
//     FP32 conservative reject and runs the exact FP64 test (distancePointToSegment, 2 sqrt + 1 div) in place: inside a
//     unit most items do collide, so there is no divergence worth a second stage, no pair list and no queue.
//
// A single new obstacle touches the few hundred cells around it instead of all 10^7 items; 256 obstacles at once (C3)
// touch each item 0.6 times on average.  The cell size follows the item density AND the edge lengths (at least twice
// the mean half length), and hmax is capped at one cell: the few items longer than that (parent edges across an empty
// region) would make their whole cell a candidate for far obstacles, so they go, together with the items no bound
// covers -- zero-length edges and non-finite end points, which the reference collides with EVERY active obstacle
// (t = 0/0 = NaN, !(NaN > x)) -- on a "loose" list that is tested against every obstacle of the call (FP32 reject
// first where it applies); obstacles with a non-finite centre or threshold take every cell.
// The result is an OR over (item, obstacle) pairs of exactly the predicate the edge-centric kernels evaluate.
#pragma once
#include "collision.cuh"
#include "scan.cuh"

namespace rrtqx {

#ifdef __CUDACC__

constexpr int IG_MAX_DIM = 128;
constexpr int IG_UNIT_ITEMS = 128;  // items per work unit (a warp's share: 4 trips, one 2 KB TMA tile); longer runs are split
constexpr int64_t IG_MAX_UNITS = (int64_t)1 << 23;  // work units a sweep may list (8 bytes each); more -> fall back

struct ItemGridView {
  int nx, ny, nz;
  double lo[3], inv[3], cell[3];
  double slack;                 // absolute slack of the cell-box bound (FP32 midpoints, cell function roundings)
  int64_t n_sorted;             // items in the grid
  int64_t n_degenerate;         // items on the loose ("every obstacle") list
  float hcap;                   // items with a half-length bound above this are loose (hmax <= hcap)
  const int32_t *cell_start;    // nx*ny*nz + 1
  const float *hmax;            // per cell: upper bound of the half lengths of its items
  const float4 *frec;           // sorted: (fl32 mid.xyz, half-length bound)
  const double2 *ex0, *ex1, *ex2;  // sorted: start.xy | start.z, end.x | end.yz
  const int32_t *item;          // sorted position -> item number
  const int32_t *degenerate;    // item numbers
};

struct ItemGridBufs {
  DevBuf<int32_t> cell_of, cell_start, cursor, item, degenerate, counters, scan_tmp;
  DevBuf<float> hmax;
  DevBuf<float4> frec;
  DevBuf<double2> ex0, ex1, ex2;
  DevBuf<double> bbox;  // 6 doubles
  int nx = 1, ny = 1, nz = 1;
  double lo[3] = {0, 0, 0}, inv[3] = {0, 0, 0}, cell[3] = {1, 1, 1}, slack = 0.0;
  float hcap = 0.f;
  int64_t n_sorted = 0, n_degenerate = 0, n_items = -1;
  bool valid = false;
  ItemGridView view() const {
    ItemGridView v;
    v.nx = nx; v.ny = ny; v.nz = nz;
    for (int c = 0; c < 3; ++c) { v.lo[c] = lo[c]; v.inv[c] = inv[c]; v.cell[c] = cell[c]; }
    v.slack = slack;
    v.hcap = hcap;
    v.n_sorted = n_sorted; v.n_degenerate = n_degenerate;
    v.cell_start = cell_start.p; v.hmax = hmax.p; v.frec = frec.p;
    v.ex0 = ex0.p; v.ex1 = ex1.p; v.ex2 = ex2.p; v.item = item.p; v.degenerate = degenerate.p;
    return v;
  }
};

// ---- build ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool ig_endpoints(const double4 *pos, int64_t n_nodes, const int32_t *src, const int32_t *dst,
                                             int64_t n_edges, const int32_t *parent, int64_t i, double4 &a, double4 &b) {
  int v, w;
  if (i >= n_edges) {
    v = (int)(i - n_edges);
    w = parent ? parent[v] : -1;
  } else {
    v = src[i];
    w = dst[i];
  }
  if (w < 0) return false;
  a = pos[v];
  b = pos[w];
  return true;
}

// midpoint / squared length of an item exactly as the per-call kernels derive them (collide_queue.cuh)
struct IgItem {
  double mx, my, mz, s2;
  bool has, degenerate;
};
__device__ __forceinline__ IgItem ig_item(const double4 &a, const double4 &b) {
  IgItem t;
  const double dx = __dsub_rn(a.x, b.x), dy = __dsub_rn(a.y, b.y), dz = __dsub_rn(a.z, b.z);
  t.s2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  t.mx = 0.5 * (a.x + b.x); t.my = 0.5 * (a.y + b.y); t.mz = 0.5 * (a.z + b.z);
  t.has = true;
  t.degenerate = !(t.s2 > 0.0) || !isfinite(t.s2) || !isfinite(t.mx + t.my + t.mz);
  return t;
}

// pass 1: bounding box of the finite midpoints (block partials -> 6 atomics on ordered-integer images of doubles)
__device__ __forceinline__ unsigned long long ig_ord(double x) {  // monotone map double -> uint64
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double ig_unord(unsigned long long u) {
  const unsigned long long b = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)b);
#else
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
#endif
}
static __global__ void __launch_bounds__(256)
ig_bbox_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
               const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
               unsigned long long *__restrict__ box /* min xyz, max xyz as ordered integers */,
               double *__restrict__ len_stats /* [0] sum of lengths, [1] count (cell-size heuristic only) */,
               const int32_t *__restrict__ ids /* NULL: items 0 .. n_edges + n_nodes */, int64_t n_ids) {
  // grid-stride: every thread folds its items, one set of atomics per BLOCK (same-address atomics serialise)
  __shared__ double s_red[8][8];
  const int64_t n_all = ids ? n_ids : n_edges + n_nodes;
  double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  double len = 0.0, cntv = 0.0;
  for (int64_t kk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; kk < n_all; kk += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = ids ? (int64_t)ids[kk] : kk;
    double4 a, b;
    if (ig_endpoints(pos, n_nodes, src, dst, n_edges, parent, i, a, b)) {
      const IgItem t = ig_item(a, b);
      if (!t.degenerate) {
        mn[0] = fmin(mn[0], t.mx); mx[0] = fmax(mx[0], t.mx);
        mn[1] = fmin(mn[1], t.my); mx[1] = fmax(mx[1], t.my);
        mn[2] = fmin(mn[2], t.mz); mx[2] = fmax(mx[2], t.mz);
        len += sqrt(t.s2);
        cntv += 1.0;
      }
    }
  }
  double v[8] = {mn[0], mn[1], mn[2], mx[0], mx[1], mx[2], len, cntv};
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    for (int o = 16; o > 0; o >>= 1) {
      const double w = __shfl_xor_sync(FULL, v[k], o);
      v[k] = k < 3 ? fmin(v[k], w) : (k < 6 ? fmax(v[k], w) : v[k] + w);
    }
    if (lane == 0) s_red[k][warp] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    const int k = threadIdx.x;
    double r = s_red[k][0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = k < 3 ? fmin(r, s_red[k][w]) : (k < 6 ? fmax(r, s_red[k][w]) : r + s_red[k][w]);
    if (k < 3) { if (r < INFINITY) atomicMin(&box[k], ig_ord(r)); }
    else if (k < 6) { if (r > -INFINITY) atomicMax(&box[k], ig_ord(r)); }
    else if (r > 0.0) atomicAdd(&len_stats[k - 6], r);
  }
}

__device__ __forceinline__ int ig_cell(double v, double lo, double inv, int n) {
  const int c = __double2int_rd((v - lo) * inv);  // floor, saturating; NaN -> 0
  return min(max(c, 0), n - 1);
}

// pass 2: cell of every item (-1: no edge, -2: degenerate), histogram, hmax
static __global__ void __launch_bounds__(256)
ig_assign_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                 const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent, ItemGridView G,
                 int32_t *__restrict__ cell_of, int32_t *__restrict__ hist, unsigned *__restrict__ hmax_bits,
                 int32_t *__restrict__ degenerate, int32_t *__restrict__ counters /* [0] degenerate items */,
                 const int32_t *__restrict__ ids, int64_t n_ids) {
  const int64_t kk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (kk >= (ids ? n_ids : n_edges + n_nodes)) return;
  const int64_t i = ids ? (int64_t)ids[kk] : kk;
  double4 a, b;
  if (!ig_endpoints(pos, n_nodes, src, dst, n_edges, parent, i, a, b)) { cell_of[kk] = -1; return; }
  const IgItem t = ig_item(a, b);
  float h = INFINITY;
  if (!t.degenerate) {
    float rt;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(__double2float_ru(t.s2)));
    h = 0.5f * (rt * 1.000001f) + 1e-19f;  // >= len / 2
  }
  if (t.degenerate || !(h <= G.hcap)) {   // no bound, or longer than a cell: the next level / the loose list
    cell_of[kk] = -2;
    degenerate[atomicAdd(&counters[0], 1)] = (int32_t)i;
    return;
  }
  // the record's midpoint is the FP32 one: it decides the cell, so the cell box bounds what the reject test sees
  const float fx = __double2float_rn(t.mx), fy = __double2float_rn(t.my), fz = __double2float_rn(t.mz);
  const int c = (ig_cell(fz, G.lo[2], G.inv[2], G.nz) * G.ny + ig_cell(fy, G.lo[1], G.inv[1], G.ny)) * G.nx +
                ig_cell(fx, G.lo[0], G.inv[0], G.nx);
  cell_of[kk] = c;
  atomicAdd(&hist[c], 1);
  atomicMax(&hmax_bits[c], __float_as_uint(h));      // h > 0: the bit patterns order like the values
  atomicMax(&hmax_bits[G.nx * G.ny * G.nz], __float_as_uint(h));  // and the largest of all (obstacle cell boxes)
}

// pass 3: scatter into sorted order
static __global__ void __launch_bounds__(256)
ig_scatter_kernel(const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                  const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
                  const int32_t *__restrict__ cell_of, const int32_t *__restrict__ cell_start, int32_t *__restrict__ cursor,
                  float4 *__restrict__ frec, double2 *__restrict__ ex0, double2 *__restrict__ ex1, double2 *__restrict__ ex2,
                  int32_t *__restrict__ item, const int32_t *__restrict__ ids, int64_t n_ids) {
  const int64_t kk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (kk >= (ids ? n_ids : n_edges + n_nodes)) return;
  const int64_t i = ids ? (int64_t)ids[kk] : kk;
  const int c = cell_of[kk];
  if (c < 0) return;
  double4 a, b;
  ig_endpoints(pos, n_nodes, src, dst, n_edges, parent, i, a, b);
  const IgItem t = ig_item(a, b);
  const int j = cell_start[c] + atomicAdd(&cursor[c], 1);
  float rt;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rt) : "f"(__double2float_ru(t.s2)));
  frec[j] = make_float4(__double2float_rn(t.mx), __double2float_rn(t.my), __double2float_rn(t.mz),
                        0.5f * (rt * 1.000001f) + 1e-19f);
  ex0[j] = make_double2(a.x, a.y);
  ex1[j] = make_double2(a.z, b.x);
  ex2[j] = make_double2(b.y, b.z);
  item[j] = (int32_t)i;
}

// ---- sweep ------------------------------------------------------------------------------------------------------
struct IgObstacle {      // per obstacle of the call
  double cx, cy, cz, thr, thr_le;
  double ext_t, ext_r;   // start-node filter: T_lt(searchRange), searchRange (unused by the plain check)
  float4 f;              // FP32 reject record: centre, threshold rounded UP
  float thr_dn;          // threshold rounded DOWN and shrunk by 2e-6: the FP32 certain-collision test
  float cmax;            // max |centre component| (error bound of the FP32 tests)
  int finite;            // 0: non-finite centre / threshold -> every cell, no FP32 shortcut
};

// Sink: what to do with a colliding (item, obstacle) pair.
//   bool wants(int item)                                            cheap filter on the item number
//   bool accept(const IgObstacle &o, const double a[3], int item)   exact extra condition (the sweeps' start-node filter)
//   bool fast_ok                                                    the FP32 certain-collision test also implies accept()
//   void mark(int item)

__device__ __forceinline__ IgObstacle ig_make_obstacle(const double4 r, const double2 t, const double2 *ext, int i) {
  IgObstacle o;
  o.cx = r.x; o.cy = r.y; o.cz = r.z; o.thr = t.x; o.thr_le = t.y;
  o.ext_t = ext ? ext[i].x : 0.0;
  o.ext_r = ext ? ext[i].y : 0.0;
  o.f = make_float4(__double2float_rn(r.x), __double2float_rn(r.y), __double2float_rn(r.z), __double2float_ru(t.x));
  o.thr_dn = __double2float_rd(t.x) * (1.0f - 2e-6f);
  o.cmax = __double2float_ru(fmax(fabs(r.x), fmax(fabs(r.y), fabs(r.z))));
  o.finite = (isfinite(r.x) && isfinite(r.y) && isfinite(r.z) && isfinite(t.x)) ? 1 : 0;
  return o;
}

// Work units of one obstacle in one level of the item grid: for every grid row (y, z) its box can reach, the run of
// slots of the cells [x0, x1] that can hold an item within thr + hcap of the centre (cells along x are contiguous in
// the sorted order), cut into pieces of at most IG_UNIT_ITEMS slots.  One block per (level, obstacle), threads <->
// rows; the block reserves its units with ONE atomic on the level's cursor.  The level-0 blocks also publish the
// obstacle records of the call (from (centre+R, (thr, thr_le)[, (T_lt(searchRange), searchRange)])) for the test and
// loose-item kernels: no separate launch for them.
static __global__ void __launch_bounds__(256)
ig_units_kernel(ItemGridView G0, ItemGridView G1, int n_upper, const double4 *__restrict__ rec, const double2 *__restrict__ thr,
                const double2 *__restrict__ ext, const int32_t *__restrict__ n_live, IgObstacle *__restrict__ obs,
                float4 *__restrict__ obs_f, float2 *__restrict__ obs_aux, int32_t *__restrict__ n_obs_out,
                unsigned long long *__restrict__ cursors, uint2 *__restrict__ units, int64_t cap, int32_t *__restrict__ overflow) {
  __shared__ int sm[33];
  __shared__ long long s_base;
  const int level = (int)blockIdx.x >= n_upper ? 1 : 0;
  const int o = (int)blockIdx.x - level * n_upper;
  const int n_obs = n_live ? *n_live : n_upper;
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_obs_out = n_obs;
  if (o >= n_obs) return;
  const IgObstacle ob = ig_make_obstacle(rec[o], thr[o], ext, o);
  if (level == 0 && threadIdx.x == 0) {
    obs[o] = ob;
    obs_f[o] = ob.f;
    obs_aux[o] = make_float2(ob.cmax, ob.finite ? 1.f : 0.f);
  }
  const ItemGridView &G = level ? G1 : G0;
  if (G.n_sorted <= 0) return;
  unsigned long long *cursor = cursors + level;
  uint2 *my_units = units + (int64_t)level * cap;
  const double c[3] = {ob.cx, ob.cy, ob.cz};
  const double R = (ob.thr + (double)G.hcap) * (1.0 + 1e-6) + G.slack;
  int y0 = 0, ny = G.ny, z0 = 0, nz = G.nz;
  if (ob.finite) {
    y0 = ig_cell(c[1] - R, G.lo[1], G.inv[1], G.ny); ny = ig_cell(c[1] + R, G.lo[1], G.inv[1], G.ny) - y0 + 1;
    z0 = ig_cell(c[2] - R, G.lo[2], G.inv[2], G.nz); nz = ig_cell(c[2] + R, G.lo[2], G.inv[2], G.nz) - z0 + 1;
  }
  const int rows = ny * nz;
  for (int r0 = 0; r0 < rows; r0 += blockDim.x) {
    const int r = r0 + threadIdx.x;
    int j0 = 0, j1 = 0;
    if (r < rows) {
      const int y = y0 + r % ny, z = z0 + r / ny;
      int x0 = 0, x1 = G.nx - 1;
      bool any = true;
      if (ob.finite) {
        // lower bounds of |c.y - m.y|, |c.z - m.z| for midpoints stored in this row; border rows are unbounded outwards
        const double yl = y == 0 ? -INFINITY : G.lo[1] + y * G.cell[1], yh = y == G.ny - 1 ? INFINITY : G.lo[1] + (y + 1) * G.cell[1];
        const double zl = z == 0 ? -INFINITY : G.lo[2] + z * G.cell[2], zh = z == G.nz - 1 ? INFINITY : G.lo[2] + (z + 1) * G.cell[2];
        const double dy = fmax(fmax(yl - c[1], c[1] - yh) - G.slack, 0.0), dz = fmax(fmax(zl - c[2], c[2] - zh) - G.slack, 0.0);
        const double rem = R * R - dy * dy - dz * dz;
        if (!(rem >= 0.0)) {
          any = false;
        } else {
          const double xr = sqrt(rem) * (1.0 + 1e-9) + G.slack;
          x0 = ig_cell(c[0] - xr, G.lo[0], G.inv[0], G.nx);
          x1 = ig_cell(c[0] + xr, G.lo[0], G.inv[0], G.nx);
        }
      }
      if (any) {
        const int base = (z * G.ny + y) * G.nx;
        j0 = G.cell_start[base + x0];
        j1 = G.cell_start[base + x1 + 1];
      }
    }
    const int chunks = (j1 - j0 + IG_UNIT_ITEMS - 1) / IG_UNIT_ITEMS;
    int tot;
    const int ex = block_exclusive_scan<int>(chunks, sm, &tot);
    if (threadIdx.x == 0) s_base = tot ? (long long)atomicAdd(cursor, (unsigned long long)tot) : 0;
    __syncthreads();
    const long long base_u = s_base;
    if (tot && base_u + tot > cap) {
      if (threadIdx.x == 0) *overflow = 1;   // more units than the list holds: the caller falls back to the edge-centric kernels
    } else {
      for (int q = 0; q < chunks; ++q) {
        const int a0 = j0 + q * IG_UNIT_ITEMS, n = min(IG_UNIT_ITEMS, j1 - a0);
        my_units[base_u + ex + q] = make_uint2((unsigned)o | ((unsigned)(n - 1) << 24), (unsigned)a0);   // o < 2^24
      }
    }
    __syncthreads();
  }
}

// One warp per unit, grid-stride over the unit list.  The unit's FP32 records arrive as ONE TMA bulk copy
// (cp.async.bulk + mbarrier, the next unit's tile in flight while the current one is classified).  Phase 1 sorts
// every item into: cannot collide (FP32 conservative reject) / certainly collides (the whole segment lies within the
// obstacle: |c - mid| + len/2 <= thr, so the reference's D, a distance to a point ON the segment, is <= thr) / needs the
// exact test; the last kind is compacted into a per-warp list.  Phase 2 runs the exact FP64 test
// (distancePointToSegment, 2 sqrt + 1 div) on that list with every lane busy.
// One wave of persistent blocks, 4 per SM at 64 registers (5 / 6 blocks per SM spill and are 10 / 23 % slower,
// 3 blocks 4 % slower).
constexpr int IG_BLOCKS_PER_SM = 4;
template <bool FMA_DOT, class Sink>
static __global__ void __launch_bounds__(256, IG_BLOCKS_PER_SM)
ig_test_kernel(ItemGridView G0, ItemGridView G1, const IgObstacle *__restrict__ obs, const uint2 *__restrict__ units_all,
               const unsigned long long *__restrict__ cursors, int64_t cap, const int32_t *__restrict__ overflow, Sink S) {
  // per warp: two TMA tiles of FP32 records (the unit being classified and the next one in flight), their mbarriers,
  // and the list of items that need the exact test
  __shared__ alignas(128) float4 s_frec[8][2][IG_UNIT_ITEMS];
  __shared__ alignas(8) unsigned long long s_bar[8][2];
  __shared__ unsigned short s_list[8][IG_UNIT_ITEMS];
  if (*overflow) return;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const unsigned lt = lanemask_lt();
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  if (lane == 0) { mbar_init(&s_bar[wib][0], 1); mbar_init(&s_bar[wib][1], 1); }
  __syncwarp();
  unsigned phase[2] = {0u, 0u};
  int buf = 0;
#pragma unroll 1
  for (int level = 0; level < 2; ++level) {   // the units of level 0, then those of level 1 (same warps, same tiles)
  if ((level ? G1.n_sorted : G0.n_sorted) <= 0) continue;
  // the level's arrays (kernel parameters: selected from the constant bank, nothing kept for the other level)
  const float4 *const g_frec = level ? G1.frec : G0.frec;
  const double2 *const g_ex0 = level ? G1.ex0 : G0.ex0, *const g_ex1 = level ? G1.ex1 : G0.ex1, *const g_ex2 = level ? G1.ex2 : G0.ex2;
  const int32_t *const g_item = level ? G1.item : G0.item;
  const uint2 *units = units_all + (int64_t)level * cap;
  const int64_t n_units = (int64_t)min(cursors[level], (unsigned long long)cap);
  // a unit's records are one contiguous, 16-byte aligned run of at most 2 KB: one bulk copy by the TMA engine
  auto issue = [&](const uint2 un, int buf) {
    if (lane == 0) {
      const unsigned bytes = ((un.x >> 24) + 1u) * 16u;
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the tile was read by ordinary loads before
      mbar_expect_tx(&s_bar[wib][buf], bytes);
      tma_load_1d(&s_frec[wib][buf][0], g_frec + un.y, bytes, &s_bar[wib][buf]);
    }
  };
  int64_t u = warp0;
  uint2 un = make_uint2(0u, 0u);
  if (u < n_units) { un = units[u]; issue(un, buf); }
  while (u < n_units) {
    const int64_t u_next = u + n_warps;
    uint2 un_next = make_uint2(0u, 0u);
    if (u_next < n_units) { un_next = units[u_next]; issue(un_next, buf ^ 1); }   // next tile in flight while this one is worked on
    const IgObstacle ob = obs[un.x & 0xffffffu];
    const int j0 = (int)un.y, n = (int)(un.x >> 24) + 1;
    mbar_wait(&s_bar[wib][buf], phase[buf]);
    phase[buf] ^= 1u;
    int n_ex = 0;
    for (int t = 0; t < n; t += 32) {
      const int k = t + lane;
      bool need = k < n;
      if (need && ob.finite) {
        const float4 fr = s_frec[wib][buf][k];
        const float ux = ob.f.x - fr.x, uy = ob.f.y - fr.y, uz = ob.f.z - fr.z;
        const float d2 = ux * ux + uy * uy + uz * uz;
        // |u^ - (c - mid)| <= bound (collision.cuh: seg_f32); NaN anywhere: every comparison false -> exact test
        const float bound = 3.0e-7f * (ob.cmax + fmaxf(fabsf(fr.x), fmaxf(fabsf(fr.y), fabsf(fr.z))));
        const float lim = ((ob.f.w + fr.w) + bound) * 1.00001f;
        if (d2 > lim * lim * 1.00001f) {
          need = false;                                       // cannot collide
        } else {
          const float far = (sqrtf(d2) * 1.000001f + fr.w + bound) * 1.00001f;   // >= max distance centre <-> segment
          if (S.fast_ok && far <= ob.thr_dn) {                // certainly collides (and passes the sink's filter)
            need = false;
            const int it = g_item[j0 + k];
            if (S.wants(it)) S.mark(it);
          }
        }
      }
      const unsigned m = __ballot_sync(FULL, need);
      if (need) s_list[wib][n_ex + __popc(m & lt)] = (unsigned short)k;
      n_ex += __popc(m);
    }
    __syncwarp();
    for (int e = lane; e < n_ex; e += 32) {
      const int j = j0 + (int)s_list[wib][e];
      const int it = g_item[j];
      if (!S.wants(it)) continue;
      const double2 p0 = g_ex0[j], p1 = g_ex1[j], p2 = g_ex2[j];
      const SegPre pre = seg_prepare(p0.x, p0.y, p1.x, p1.y, p2.x, p2.y);
      if (seg_sphere_collide_exact<FMA_DOT>(pre, ob.cx, ob.cy, ob.cz, ob.thr_le)) {
        const double a[3] = {p0.x, p0.y, p1.x};
        if (S.accept(ob, a, it)) S.mark(it);
      }
    }
    __syncwarp();   // the tile and the list are free again
    u = u_next;
    un = un_next;
    buf ^= 1;
  }
  }
}

// loose items (degenerate or longer than a cell): one WARP per item, lanes over the obstacles of the call, FP32 reject
// where it applies, exact test (a NaN radicand collides, as in the reference), the item ends at the first hit
template <bool FMA_DOT, class Sink>
static __global__ void __launch_bounds__(256)
ig_loose_kernel(ItemGridView G, const double4 *__restrict__ pos, int64_t n_nodes, const int32_t *__restrict__ src,
                const int32_t *__restrict__ dst, int64_t n_edges, const int32_t *__restrict__ parent,
                const IgObstacle *__restrict__ obs, const float4 *__restrict__ obs_f /* centre, thr up */,
                const float2 *__restrict__ obs_aux /* cmax, finite */, const int32_t *__restrict__ n_obs_dev, Sink S) {
  const int lane = threadIdx.x & 31;
  const int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (k >= G.n_degenerate) return;
  const int n_obs = *n_obs_dev;
  const int it = G.degenerate[k];
  if (!S.wants(it)) return;
  double4 a4, b4;
  if (!ig_endpoints(pos, n_nodes, src, dst, n_edges, parent, it, a4, b4)) return;
  const SegPre pre = seg_prepare(a4.x, a4.y, a4.z, b4.x, b4.y, b4.z);
  const double a[3] = {a4.x, a4.y, a4.z};
  bool hit = false;
  for (int o0 = 0; o0 < n_obs && !hit; o0 += 32) {
    const int o = o0 + lane;
    bool h = false;
    if (o < n_obs) {
      bool rejected = false;
      if (pre.cullable) {               // 24 bytes per obstacle for the reject, the full record only for survivors
        const float2 aux = obs_aux[o];
        if (aux.y != 0.f) rejected = seg_reject_f32(seg_f32(pre, aux.x), obs_f[o]);
      }
      if (!rejected) {
        const IgObstacle ob = obs[o];
        h = seg_sphere_collide_exact<FMA_DOT>(pre, ob.cx, ob.cy, ob.cz, ob.thr_le) && S.accept(ob, a, it);
      }
    }
    hit = __any_sync(FULL, h);
  }
  if (hit && lane == 0) S.mark(it);
}

#endif  // __CUDACC__

#ifdef __CUDACC__
// ---- host side --------------------------------------------------------------------------------------------------
struct IgRunBufs {  // per context (rrtqx_ctx::scratch)
  DevBuf<unsigned char> obs;   // IgObstacle[n]
  DevBuf<float4> obs_f;        // reject records of the same obstacles (loose-item kernel)
  DevBuf<float2> obs_aux;
  DevBuf<int32_t> cnt, flags;  // units per obstacle | [0] overflow, [1] obstacles of the call
  DevBuf<int64_t> off;         // unit offsets per obstacle, [n] = total
  DevBuf<uint2> units;
  DevBuf<unsigned long long> cursor;  // units listed so far
};
inline char g_ig_run_tag = 0;
static inline IgRunBufs &ig_run_bufs(rrtqx_ctx *ctx) { return ctx->scratch.get<IgRunBufs>(&g_ig_run_tag); }

// Sort the items of an edge set into the grid.  Synchronises the stream twice (bounding box, degenerate count): it
// runs with the edge-set (re)build, not inside a sweep.
// ids / n_ids: the items to sort (NULL: all of them); min_cell: lower bound of the cell length (level 1 of the
// hierarchy sorts the items that were too long for level 0 into cells 8 times larger).
static inline void item_grid_build(rrtqx_ctx *ctx, ItemGridBufs &B, const double4 *pos, int64_t n_nodes, const int32_t *src,
                                   const int32_t *dst, int64_t n_edges, const int32_t *parent, const int32_t *ids = nullptr,
                                   int64_t n_ids = 0, double min_cell = 0.0) {
  cudaStream_t st = ctx->stream;
  const int64_t n_items = ids ? n_ids : n_edges + n_nodes;
  B.valid = false;
  B.n_items = n_items;
  B.n_sorted = B.n_degenerate = 0;
  if (n_items <= 0 || n_items >= ((int64_t)1 << 31)) return;
  const int TB = 256;
  const unsigned blocks = (unsigned)div_up(n_items, TB);
  B.bbox.ensure(8, st);
  unsigned long long init[8] = {~0ull, ~0ull, ~0ull, 0ull, 0ull, 0ull, 0ull, 0ull};  // box, then two doubles (0.0)
  RQ_CUDA(cudaMemcpyAsync(B.bbox.p, init, sizeof(init), cudaMemcpyHostToDevice, st));
  ig_bbox_kernel<<<(unsigned)std::min<int64_t>(blocks, (int64_t)ctx->sm_count * 8), TB, 0, st>>>(
      pos, n_nodes, src, dst, n_edges, parent, (unsigned long long *)B.bbox.p, B.bbox.p + 6, ids, n_ids);
  post_launch(ctx);
  unsigned long long box[8];
  RQ_CUDA(cudaMemcpyAsync(box, B.bbox.p, sizeof(box), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  double len_sum, len_cnt;
  memcpy(&len_sum, &box[6], sizeof(double));
  memcpy(&len_cnt, &box[7], sizeof(double));
  const double mean_half = len_cnt > 0.0 ? 0.5 * len_sum / len_cnt : 0.0;
  double mn[3], mx[3];
  bool any = true;
  for (int c = 0; c < 3; ++c) {
    if (box[c] == ~0ull) { any = false; break; }
    mn[c] = ig_unord(box[c]); mx[c] = ig_unord(box[3 + c]);
  }
  // grid shape: about 32 items per cell, cubic cells, at most IG_MAX_DIM per axis
  int dims[3] = {1, 1, 1};
  double span = 0.0, mag = 0.0;
  if (any) {
    double ext[3], vol = 1.0;
    int nz_dims = 0;
    for (int c = 0; c < 3; ++c) {
      ext[c] = mx[c] - mn[c];
      span = std::max(span, ext[c]);
      mag = std::max(mag, std::max(std::fabs(mn[c]), std::fabs(mx[c])));
      if (ext[c] > 0.0 && std::isfinite(ext[c])) { vol *= ext[c]; nz_dims++; }
    }
    const double target_cells = std::max(1.0, (double)n_items / 32.0);
    double cell_len = nz_dims ? std::pow(vol / target_cells, 1.0 / nz_dims) : 1.0;
    // cells at least twice the mean half length: hmax is capped at one cell, so shorter cells would push most items
    // of a long-edged graph (early RRTx: edges up to the ball radius) onto the loose list
    if (std::isfinite(mean_half) && 2.0 * mean_half > cell_len) cell_len = 2.0 * mean_half;
    if (min_cell > cell_len) cell_len = min_cell;
    B.hcap = std::isfinite(cell_len) && cell_len > 0.0 ? (float)cell_len : 0.f;
    for (int c = 0; c < 3; ++c) {
      if (ext[c] > 0.0 && std::isfinite(ext[c]) && cell_len > 0.0 && std::isfinite(cell_len))
        dims[c] = (int)std::min<double>(IG_MAX_DIM, std::max(1.0, std::floor(ext[c] / cell_len) + 1.0));
      B.lo[c] = mn[c];
      B.cell[c] = dims[c] > 1 ? ext[c] / dims[c] : std::max(ext[c], 1.0);
      B.inv[c] = dims[c] > 1 ? dims[c] / ext[c] : 0.0;
    }
  } else {
    for (int c = 0; c < 3; ++c) { B.lo[c] = 0.0; B.cell[c] = 1.0; B.inv[c] = 0.0; }
    B.hcap = 0.f;
  }
  B.nx = dims[0]; B.ny = dims[1]; B.nz = dims[2];
  // FP32 midpoints (relative 2^-24 of their magnitude), the roundings of the cell function and of the box corners
  B.slack = 1e-6 * (mag + span) + 1e-300;
  const int64_t ncell = (int64_t)B.nx * B.ny * B.nz;
  B.cell_of.ensure((size_t)n_items + 1, st);
  B.cursor.ensure((size_t)ncell + 2, st);
  B.cell_start.ensure((size_t)ncell + 2, st);
  B.hmax.ensure((size_t)ncell + 2, st);
  B.degenerate.ensure((size_t)n_items + 1, st);
  B.counters.ensure(4, st);
  RQ_CUDA(cudaMemsetAsync(B.cursor.p, 0, sizeof(int32_t) * ((size_t)ncell + 2), st));
  RQ_CUDA(cudaMemsetAsync(B.hmax.p, 0, sizeof(float) * ((size_t)ncell + 2), st));
  RQ_CUDA(cudaMemsetAsync(B.counters.p, 0, sizeof(int32_t) * 4, st));
  ItemGridView G = B.view();
  ig_assign_kernel<<<blocks, TB, 0, st>>>(pos, n_nodes, src, dst, n_edges, parent, G, B.cell_of.p, B.cursor.p,
                                          (unsigned *)B.hmax.p, B.degenerate.p, B.counters.p, ids, n_ids);
  post_launch(ctx);
  exclusive_scan<int32_t, int32_t>(ctx, B.cursor.p, ncell, B.cell_start.p, B.scan_tmp);
  int32_t counts[2] = {0, 0};
  RQ_CUDA(cudaMemcpyAsync(&counts[0], B.counters.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaMemcpyAsync(&counts[1], B.cell_start.p + ncell, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  B.n_degenerate = counts[0];
  B.n_sorted = counts[1];
  B.frec.ensure((size_t)B.n_sorted + 1, st);
  B.ex0.ensure((size_t)B.n_sorted + 1, st);
  B.ex1.ensure((size_t)B.n_sorted + 1, st);
  B.ex2.ensure((size_t)B.n_sorted + 1, st);
  B.item.ensure((size_t)B.n_sorted + 1, st);
  RQ_CUDA(cudaMemsetAsync(B.cursor.p, 0, sizeof(int32_t) * ((size_t)ncell + 2), st));
  ig_scatter_kernel<<<blocks, TB, 0, st>>>(pos, n_nodes, src, dst, n_edges, parent, B.cell_of.p, B.cell_start.p, B.cursor.p,
                                           B.frec.p, B.ex0.p, B.ex1.p, B.ex2.p, B.item.p, ids, n_ids);
  post_launch(ctx);
  B.valid = true;
}

// The obstacle-centric check of every item of a grid against the obstacles (rec, thr[, ext]) of a call (live count on
// the device in *n_live, or n_upper when n_live is NULL).  Everything is queued on the stream; *overflow_dev (device
// flag) reads 1 afterwards if the call listed more than IG_MAX_UNITS work units -- then NOTHING was marked and the
// caller repeats the call through the edge-centric kernels.
template <bool FMA_DOT, class Sink>
static inline const int32_t *item_grid_run(rrtqx_ctx *ctx, const ItemGridBufs &B0, const ItemGridBufs *B1, const double4 *rec,
                                           const double2 *thr, const double2 *ext, const int32_t *n_live, int n_upper,
                                           const Sink &S, const double4 *pos, int64_t n_nodes, const int32_t *src,
                                           const int32_t *dst, int64_t n_edges, const int32_t *parent) {
  cudaStream_t st = ctx->stream;
  IgRunBufs &R = ig_run_bufs(ctx);
  R.obs.ensure(sizeof(IgObstacle) * ((size_t)n_upper + 1), st);
  R.obs_f.ensure((size_t)n_upper + 1, st);
  R.obs_aux.ensure((size_t)n_upper + 1, st);
  R.units.ensure((size_t)IG_MAX_UNITS, st);
  R.cursor.ensure(4, st);   // [0], [1]: units listed per level; [2]: two 32-bit words: overflow flag, obstacle count
  IgObstacle *obs = (IgObstacle *)R.obs.p;
  int32_t *overflow = (int32_t *)(R.cursor.p + 2), *n_obs = overflow + 1;
  // flags and the two unit cursors live in one buffer: a single memset per call
  static_assert(sizeof(unsigned long long) == 8, "");
  RQ_CUDA(cudaMemsetAsync(R.cursor.p, 0, sizeof(unsigned long long) * 4, st));
  if (n_upper <= 0) return overflow;
  // level 0: the items that fit its cells; level 1 (if built): the longer ones in cells 8 times larger; what fits
  // neither is the last level's loose list.  One launch lists the units of both levels (and publishes the obstacle
  // records), one launch tests them.
  const bool has1 = B1 && B1->valid;
  const ItemGridBufs *last = has1 ? B1 : &B0;
  ItemGridView G0 = B0.view(), G1 = has1 ? B1->view() : B0.view();
  if (!has1) G1.n_sorted = 0;
  const int64_t cap = IG_MAX_UNITS / 2;
  ig_units_kernel<<<(has1 ? 2 : 1) * n_upper, 256, 0, st>>>(G0, G1, n_upper, rec, thr, ext, n_live, obs, R.obs_f.p, R.obs_aux.p,
                                                          n_obs, R.cursor.p, R.units.p, cap, overflow);
  ig_test_kernel<FMA_DOT, Sink><<<ctx->sm_count * IG_BLOCKS_PER_SM, 256, 0, st>>>(G0, G1, obs, R.units.p, R.cursor.p, cap, overflow, S);
  post_launch(ctx, 2);
  if (last->n_degenerate > 0) {
    const ItemGridView G = last->view();
    ig_loose_kernel<FMA_DOT, Sink><<<div_up(last->n_degenerate * 32, 256), 256, 0, st>>>(G, pos, n_nodes, src, dst, n_edges, parent,
                                                                                       obs, R.obs_f.p, R.obs_aux.p, n_obs, S);
    post_launch(ctx);
  }
  return overflow;
}

// Both levels of an edge set: level 0 over all items, level 1 over what level 0 found too long (when that is more than
// a handful: a graph whose parent edges cross empty regions), in cells 8 times larger.
static inline void item_grid_build_levels(rrtqx_ctx *ctx, ItemGridBufs &B0, ItemGridBufs &B1, const double4 *pos, int64_t n_nodes,
                                          const int32_t *src, const int32_t *dst, int64_t n_edges, const int32_t *parent) {
  item_grid_build(ctx, B0, pos, n_nodes, src, dst, n_edges, parent);
  B1.valid = false;
  if (B0.valid && B0.n_degenerate >= 4096)
    item_grid_build(ctx, B1, pos, n_nodes, src, dst, n_edges, parent, B0.degenerate.p, B0.n_degenerate, 8.0 * (double)B0.hcap);
}

#endif  // __CUDACC__

}  // namespace rrtqx
