// tree.cu -- kd topology build (exactly the insertion-order tree of
// kdTree_general.jl:121-170, built level-parallel) and the uniform-grid query
// index (cell-sorted SoA).
#include <algorithm>
#include <cmath>

#include "scan.cuh"
#include "tree.cuh"

namespace rrtqx {

// ---------------------------------------------------------------- node table

__global__ void unpack_positions_kernel(const double *__restrict__ rows, int d, int64_t first, int64_t n_new,
                                        double4 *__restrict__ pos, unsigned *__restrict__ child,
                                        int32_t *__restrict__ parent, int8_t *__restrict__ split,
                                        int32_t *__restrict__ cur) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_new) return;
  const double *r = rows + k * d;
  double4 p;
  p.x = r[0];
  p.y = r[1];
  p.z = d >= 3 ? r[2] : 0.0;
  p.w = d >= 4 ? r[3] : 0.0;
  int64_t i = first + k;
  pos[i] = p;
  child[2 * i] = KD_EMPTY;
  child[2 * i + 1] = KD_EMPTY;
  parent[i] = -1;
  split[i] = 0;
  cur[i] = 0;  // every new node starts its descent at the root
}

__device__ __forceinline__ double coord(const double4 &p, int s) {
  return s == 0 ? p.x : (s == 1 ? p.y : (s == 2 ? p.z : p.w));
}

// One round of the level-parallel build.  Every unplaced node walks down
// through FINAL child links as far as they go (kdTree_general.jl:136-160: left
// iff node.pos[split] < parent.pos[split]) and bids for the empty slot it
// reaches with atomicMin(index | TENTATIVE).  All nodes whose sequential
// insertion path runs through a slot reach it in the same round (their common
// ancestors were fixed in earlier rounds), so the smallest bidder is exactly
// the node sequential insertion would have put there.
__global__ void kd_descend_claim_kernel(const double4 *__restrict__ pos, unsigned *__restrict__ child,
                                        const int8_t *__restrict__ split, int32_t *__restrict__ cur,
                                        int64_t first, int64_t n_new) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_new) return;
  int64_t i = first + k;
  int32_t p = cur[i];
  if (p < 0) return;  // placed
  if (i == 0) return; // root handled by resolve
  double4 me = pos[i];
  for (;;) {
    int s = split[p];
    int side = coord(me, s) < coord(pos[p], s) ? 0 : 1;
    unsigned c = child[2 * (int64_t)p + side];
    if (!(c & KD_TENTATIVE)) {  // final link (KD_EMPTY has the bit set)
      p = (int32_t)c;
      continue;
    }
    atomicMin(&child[2 * (int64_t)p + side], (unsigned)i | KD_TENTATIVE);
    break;
  }
  cur[i] = p;
}

__global__ void kd_resolve_kernel(const double4 *__restrict__ pos, unsigned *__restrict__ child,
                                  int32_t *__restrict__ parent, int8_t *__restrict__ split,
                                  int32_t *__restrict__ cur, int64_t first, int64_t n_new, int d,
                                  int32_t *__restrict__ remaining) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_new) return;
  int64_t i = first + k;
  int32_t p = cur[i];
  if (p < 0) return;
  if (i == 0) {  // kdTree_general.jl:127-132
    split[0] = 0;
    cur[0] = -1;
    return;
  }
  int s = split[p];
  int side = coord(pos[i], s) < coord(pos[p], s) ? 0 : 1;
  unsigned v = child[2 * (int64_t)p + side];
  if (v == ((unsigned)i | KD_TENTATIVE)) {
    child[2 * (int64_t)p + side] = (unsigned)i;
    parent[i] = p;
    split[i] = (int8_t)((s == d - 1) ? 0 : s + 1);  // :164-168
    cur[i] = -1;
  } else {
    atomicAdd(remaining, 1);
  }
}

// Sequential kdInsert of one node by one thread (the planner's per-iteration
// insert); the walk is ~log n dependent loads.
__global__ void kd_insert_one_kernel(const double4 *__restrict__ pos, unsigned *__restrict__ child,
                                     int32_t *__restrict__ parent, int8_t *__restrict__ split,
                                     int32_t *__restrict__ cur, int64_t i, int d) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  cur[i] = -1;
  if (i == 0) {
    split[0] = 0;
    return;
  }
  double4 me = pos[i];
  int32_t p = 0;
  for (;;) {
    int s = split[p];
    int side = coord(me, s) < coord(pos[p], s) ? 0 : 1;
    unsigned c = child[2 * (int64_t)p + side];
    if (c == KD_EMPTY) {
      child[2 * (int64_t)p + side] = (unsigned)i;
      parent[i] = p;
      split[i] = (int8_t)((s == d - 1) ? 0 : s + 1);
      return;
    }
    p = (int32_t)c;
  }
}

// The planner's per-iteration insert in ONE launch: the position travels as a kernel argument (no staging
// copy, nothing to wait for), the thread initialises the node's records and walks down to its slot.
__global__ void kd_insert_point_kernel(double4 p, double4 *__restrict__ pos, unsigned *__restrict__ child,
                                       int32_t *__restrict__ parent, int8_t *__restrict__ split, int32_t *__restrict__ cur,
                                       int64_t i, int d) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  pos[i] = p;
  child[2 * i] = KD_EMPTY;
  child[2 * i + 1] = KD_EMPTY;
  parent[i] = -1;
  split[i] = 0;
  cur[i] = -1;
  if (i == 0) return;  // root: split 0 (kdTree_general.jl:127-132)
  int32_t q = 0;
  for (;;) {
    const int s = split[q];
    const int side = coord(p, s) < coord(pos[q], s) ? 0 : 1;
    const unsigned c = child[2 * (int64_t)q + side];
    if (c == KD_EMPTY) {
      child[2 * (int64_t)q + side] = (unsigned)i;
      parent[i] = q;
      split[i] = (int8_t)((s == d - 1) ? 0 : s + 1);
      return;
    }
    q = (int32_t)c;
  }
}

// Single insert of a HOST position (rrtqx_tree_insert): asynchronous, one launch.
void tree_insert_point(rrtqx_tree *t, const double *position) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(t->n + 1 < (int64_t)0x7fffffff, "tree too large for int32 node indices");
  const int64_t first = t->n;
  const size_t need = (size_t)(first + 1);
  t->pos.ensure(need, st, (size_t)first);
  t->child.ensure(2 * need, st, 2 * (size_t)first);
  t->parent.ensure(need, st, (size_t)first);
  t->split.ensure(need, st, (size_t)first);
  t->cur.ensure(need, st, (size_t)first);
  double4 p;
  p.x = position[0];
  p.y = position[1];
  p.z = t->d >= 3 ? position[2] : 0.0;
  p.w = t->d >= 4 ? position[3] : 0.0;
  kd_insert_point_kernel<<<1, 32, 0, st>>>(p, t->pos.p, t->child.p, t->parent.p, t->split.p, t->cur.p, first, t->d);
  post_launch(ctx);
  t->n = first + 1;
}

void tree_insert_batch(rrtqx_tree *t, const double *positions, int64_t n_new) {
  if (n_new <= 0) return;
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  RQ_REQUIRE(t->n + n_new < (int64_t)0x7fffffff, "tree too large for int32 node indices");
  const int64_t first = t->n;
  const size_t need = (size_t)(first + n_new);
  t->pos.ensure(need, st, (size_t)first);
  t->child.ensure(2 * need, st, 2 * (size_t)first);
  t->parent.ensure(need, st, (size_t)first);
  t->split.ensure(need, st, (size_t)first);
  t->cur.ensure(need, st, (size_t)first);
  t->flagbuf.ensure(8, st);

  const double *rows = to_device(ctx, positions, (size_t)n_new * t->d, ctx->stage_f64);
  const int TB = 256;
  unpack_positions_kernel<<<div_up(n_new, TB), TB, 0, st>>>(rows, t->d, first, n_new, t->pos.p, t->child.p,
                                                            t->parent.p, t->split.p, t->cur.p);
  post_launch(ctx);

  if (n_new == 1) {
    kd_insert_one_kernel<<<1, 32, 0, st>>>(t->pos.p, t->child.p, t->parent.p, t->split.p, t->cur.p, first, t->d);
    post_launch(ctx);
  } else {
    // rounds until every node is placed; check the counter every few rounds
    int rounds_per_check = 8;
    int32_t remaining = 1;
    int64_t total_rounds = 0;
    while (remaining > 0) {
      RQ_CUDA(cudaMemsetAsync(t->flagbuf.p, 0, sizeof(int32_t), st));
      for (int r = 0; r < rounds_per_check; ++r) {
        if (r == rounds_per_check - 1) RQ_CUDA(cudaMemsetAsync(t->flagbuf.p, 0, sizeof(int32_t), st));
        kd_descend_claim_kernel<<<div_up(n_new, TB), TB, 0, st>>>(t->pos.p, t->child.p, t->split.p, t->cur.p,
                                                                  first, n_new);
        kd_resolve_kernel<<<div_up(n_new, TB), TB, 0, st>>>(t->pos.p, t->child.p, t->parent.p, t->split.p,
                                                            t->cur.p, first, n_new, t->d, t->flagbuf.p);
        post_launch(ctx, 2);
      }
      RQ_CUDA(cudaMemcpyAsync(&remaining, t->flagbuf.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      RQ_CUDA(cudaStreamSynchronize(st));
      total_rounds += rounds_per_check;
      if (total_rounds > 64) rounds_per_check = 32;  // deep (adversarial) trees: sync less often
    }
  }
  t->n = first + n_new;
}

// --------------------------------------------------------------- grid index

constexpr int BBOX_BLOCKS = 256;

__global__ void bbox_kernel(const double4 *__restrict__ pos, int64_t n, double *__restrict__ partial) {
  double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double4 p = pos[i];
    mn[0] = fmin(mn[0], p.x); mx[0] = fmax(mx[0], p.x);
    mn[1] = fmin(mn[1], p.y); mx[1] = fmax(mx[1], p.y);
    mn[2] = fmin(mn[2], p.z); mx[2] = fmax(mx[2], p.z);
  }
  __shared__ double sm[6][8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    for (int o = 16; o > 0; o >>= 1) {
      mn[k] = fmin(mn[k], __shfl_xor_sync(FULL, mn[k], o));
      mx[k] = fmax(mx[k], __shfl_xor_sync(FULL, mx[k], o));
    }
    if (lane == 0) { sm[k][warp] = mn[k]; sm[3 + k][warp] = mx[k]; }
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = sm[threadIdx.x][0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
      v = threadIdx.x < 3 ? fmin(v, sm[threadIdx.x][w]) : fmax(v, sm[threadIdx.x][w]);
    partial[blockIdx.x * 6 + threadIdx.x] = v;
  }
}

__global__ void cell_id_kernel(GridView g, int64_t n, int32_t *__restrict__ cell_id, int32_t *__restrict__ cell_count) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double4 p = g.pos[i];
  int cx = cell_of(p.x, g.lo[0], g.inv[0], g.nx);
  int cy = cell_of(p.y, g.lo[1], g.inv[1], g.ny);
  int cz = cell_of(p.z, g.lo[2], g.inv[2], g.nz);
  int c = (cz * g.ny + cy) * g.nx + cx;
  cell_id[i] = c;
  atomicAdd(&cell_count[c], 1);
}

__global__ void cell_scatter_kernel(const int32_t *__restrict__ cell_id, int64_t n,
                                    const int32_t *__restrict__ cell_start, int32_t *__restrict__ cursor,
                                    int32_t *__restrict__ sperm) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int c = cell_id[i];
  int slot = cell_start[c] + atomicAdd(&cursor[c], 1);
  sperm[slot] = (int32_t)i;
}

// Deterministic layout: inside a cell, ascending x (ties: ascending node index).  cell_of() is monotone in x, so a
// whole ROW of cells is then sorted by x: the neighbours of a query in a row are one nearly contiguous run of slots
// (fewer 128-byte lines per 32 gathered exact records in the range kernel's flush).  No kernel relies on the order
// inside a cell for its result.
__global__ void cell_sort_kernel(const int32_t *__restrict__ cell_start, int ncell, const double4 *__restrict__ pos,
                                 int32_t *__restrict__ sperm) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= ncell) return;
  int a = cell_start[c], b = cell_start[c + 1];
  if (b - a > 256) return;  // degenerate pile-up: order left as scattered (result sets unaffected)
  for (int i = a + 1; i < b; ++i) {
    const int v = sperm[i];
    const double xv = pos[v].x;
    int j = i - 1;
    while (j >= a) {
      const int u = sperm[j];
      const double xu = pos[u].x;
      if (!(xu > xv || (xu == xv && u > v))) break;   // NaN x: compares false, keeps its place
      sperm[j + 1] = u;
      --j;
    }
    sperm[j + 1] = v;
  }
}

// Also writes the two per-slot records of the v5 range kernel: the FP32 filter record (coordinates
// relative to the grid origin, so the rounding error is bounded by 2^-24 * extent) and the exact
// FP64 record, and accumulates max |component| of the filter records (bit pattern order of
// non-negative floats; a NaN/Inf component yields a non-finite maximum, which disables the filter).
__global__ void cell_gather_kernel(const double4 *__restrict__ pos, const int32_t *__restrict__ sperm, int64_t n, int d,
                                   double lox, double loy, double loz,
                                   double *__restrict__ sx, double *__restrict__ sy, double *__restrict__ sz,
                                   double *__restrict__ sw, float4 *__restrict__ f4, double4 *__restrict__ d4,
                                   float *__restrict__ fmaxabs) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float m = 0.0f;
  if (j >= n && j < n + 8) {  // the 8 padding slots behind the last record never hit: +inf filter coordinates
    f4[j] = make_float4(INFINITY, INFINITY, INFINITY, INFINITY);
    d4[j] = make_double4(INFINITY, INFINITY, INFINITY, __longlong_as_double(-1LL));
  }
  if (j < n) {
    const int node = sperm[j];
    double4 p = pos[node];
    sx[j] = p.x;
    sy[j] = p.y;
    sz[j] = p.z;
    sw[j] = p.w;
    float4 f;
    f.x = __double2float_rn(__dsub_rn(p.x, lox));
    f.y = __double2float_rn(__dsub_rn(p.y, loy));
    f.z = __double2float_rn(__dsub_rn(p.z, loz));
    f.w = __double2float_rn(p.w);
    f4[j] = f;
    double4 r = p;
    if (d <= 3) r.w = __longlong_as_double((long long)(unsigned)node);
    d4[j] = r;
    // NaN components never produce a hit (neither in FP32 nor in FP64) and are skipped by fmaxf;
    // infinities make the maximum infinite.
    m = fmaxf(fmaxf(fabsf(f.x), fabsf(f.y)), fmaxf(fabsf(f.z), fabsf(f.w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(FULL, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax((int *)fmaxabs, __float_as_int(m));
}

void tree_reindex(rrtqx_tree *t) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  const int64_t n = t->n;
  if (n == 0) {
    t->n_sorted = 0;
    return;
  }
  PhaseScope ph(ctx, "tree_build");
  // 1. bounding box of the first three coordinates
  t->bbox_partial.ensure(BBOX_BLOCKS * 6, st);
  bbox_kernel<<<BBOX_BLOCKS, 256, 0, st>>>(t->pos.p, n, t->bbox_partial.p);
  post_launch(ctx);
  std::vector<double> part(BBOX_BLOCKS * 6);
  RQ_CUDA(cudaMemcpyAsync(part.data(), t->bbox_partial.p, sizeof(double) * part.size(), cudaMemcpyDeviceToHost, st));
  RQ_CUDA(cudaStreamSynchronize(st));
  double mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int b = 0; b < BBOX_BLOCKS; ++b)
    for (int k = 0; k < 3; ++k) {
      mn[k] = std::fmin(mn[k], part[b * 6 + k]);
      mx[k] = std::fmax(mx[k], part[b * 6 + 3 + k]);
    }
  // 2. grid resolution: ~occupancy points per cell over the non-flat dimensions
  double ext[3];
  int nonflat = 0;
  double vol = 1.0;
  for (int k = 0; k < 3; ++k) {
    if (!std::isfinite(mn[k]) || !std::isfinite(mx[k])) { mn[k] = 0.0; mx[k] = 0.0; }
    ext[k] = mx[k] - mn[k];
    if (k >= t->d || !(ext[k] > 0.0) || !std::isfinite(ext[k])) ext[k] = 0.0;
    if (ext[k] > 0.0) { nonflat++; vol *= ext[k]; }
  }
  int dims[3] = {1, 1, 1};
  if (nonflat > 0) {
    double target_cells = std::max(1.0, (double)n / std::max(0.25, t->occupancy));
    double c = std::pow(vol / target_cells, 1.0 / nonflat);
    // Anisotropic cells: thin along x (the contiguous direction of a row of
    // cells), wide across, at constant cell volume.  Rows of a query then hold
    // ~100 candidates (3+ full warp trips) instead of ~35.
    double cs[3] = {c, c, c};
    if (ext[0] > 0.0 && nonflat >= 2 && t->aspect > 1.0) {
      cs[0] = c / std::pow(t->aspect, (nonflat - 1.0) / nonflat);
      for (int k = 1; k < 3; ++k) cs[k] = c * std::pow(t->aspect, 1.0 / nonflat);
    }
    for (int k = 0; k < 3; ++k)
      if (ext[k] > 0.0) {
        double m = std::ceil(ext[k] / cs[k]);
        if (!(m >= 1.0)) m = 1.0;
        if (m > 1024.0) m = 1024.0;
        dims[k] = (int)m;
      }
    while ((int64_t)dims[0] * dims[1] * dims[2] > (int64_t)(1 << 25)) {
      int k = (dims[0] >= dims[1] && dims[0] >= dims[2]) ? 0 : (dims[1] >= dims[2] ? 1 : 2);
      dims[k] = (dims[k] + 1) / 2;
    }
  }
  t->nx = dims[0]; t->ny = dims[1]; t->nz = dims[2];
  for (int k = 0; k < 3; ++k) {
    t->lo[k] = mn[k];
    if (ext[k] > 0.0) {
      t->cell[k] = ext[k] / dims[k];
      t->inv[k] = dims[k] / ext[k];
    } else {
      t->cell[k] = 1.0;
      t->inv[k] = 1.0;
    }
  }
  const int ncell = t->nx * t->ny * t->nz;
  // 3. counting sort by cell
  t->cell_start.ensure((size_t)ncell + 1, st);
  t->cell_cursor.ensure((size_t)ncell + 1, st);
  t->cell_id.ensure((size_t)n, st);
  t->sperm.ensure((size_t)n, st);
  t->sx.ensure((size_t)n + 8, st);
  t->sy.ensure((size_t)n + 8, st);
  t->sz.ensure((size_t)n + 8, st);
  t->sw.ensure((size_t)n + 8, st);
  t->f4.ensure((size_t)n + 8, st);
  t->d4.ensure((size_t)n + 8, st);
  t->fmaxabs.ensure(1, st);
  RQ_CUDA(cudaMemsetAsync(t->fmaxabs.p, 0, sizeof(float), st));
  RQ_CUDA(cudaMemsetAsync(t->cell_cursor.p, 0, sizeof(int32_t) * ((size_t)ncell + 1), st));
  t->n_sorted = n;  // view() below must describe the new grid
  GridView g = t->view();
  const int TB = 256;
  cell_id_kernel<<<div_up(n, TB), TB, 0, st>>>(g, n, t->cell_id.p, t->cell_cursor.p);
  post_launch(ctx);
  exclusive_scan<int32_t, int32_t>(ctx, t->cell_cursor.p, ncell, t->cell_start.p, t->scan_tmp);
  RQ_CUDA(cudaMemsetAsync(t->cell_cursor.p, 0, sizeof(int32_t) * ((size_t)ncell + 1), st));
  cell_scatter_kernel<<<div_up(n, TB), TB, 0, st>>>(t->cell_id.p, n, t->cell_start.p, t->cell_cursor.p, t->sperm.p);
  cell_sort_kernel<<<div_up(ncell, TB), TB, 0, st>>>(t->cell_start.p, ncell, t->pos.p, t->sperm.p);
  cell_gather_kernel<<<div_up(n + 8, TB), TB, 0, st>>>(t->pos.p, t->sperm.p, n, t->d, t->lo[0], t->lo[1], t->lo[2], t->sx.p, t->sy.p,
                                                   t->sz.p, t->sw.p, t->f4.p, t->d4.p, t->fmaxabs.p);
  post_launch(ctx, 3);
}

void tree_prepare_query(rrtqx_tree *t) {
  int64_t tail = t->n - t->n_sorted;
  int64_t limit = std::max<int64_t>(t->tail_limit, t->n_sorted / 64);
  if (t->n_sorted == 0 ? (t->n > 64) : (tail > limit)) tree_reindex(t);
}

}  // namespace rrtqx
