// tree.cuh -- GPU-resident point set of one KDTree (kdTree_general.jl:94-112):
//   * node table in insertion order: AoS double4 (one 32-byte sector per
//     gather) + the reference's kd topology (parent / children / split), kept
//     identical to what sequential kdInsert (kdTree_general.jl:121-170) builds;
//   * the query index: points re-ordered by uniform-grid cell (x fastest) into
//     SoA coordinate arrays so that a row of cells is ONE contiguous slice per
//     coordinate (coalesced, vectorisable), plus the permutation back to node
//     indices;
//   * an unsorted tail of recent inserts [n_sorted, n) that queries scan
//     linearly until the next re-index (LSM style), so the planner's one-node
//     inserts stay O(1).
#pragma once
#include "common.cuh"

namespace rrtqx {

constexpr int MAX_D = 4;
constexpr int MAX_WRAPS = 4;
constexpr unsigned KD_EMPTY = 0xffffffffu;
constexpr unsigned KD_TENTATIVE = 0x80000000u;

struct WrapInfo {
  int num_wraps;
  int wraps[MAX_WRAPS];
  double wrap_points[MAX_WRAPS];
};

// POD view handed to kernels by value.
struct GridView {
  int d;
  int n_sorted;  // points covered by the cell index
  int n_total;   // tree size
  int nx, ny, nz;
  double lo[3];
  double inv[3];   // 1 / cell size
  double cell[3];  // cell size
  const int *cell_start;  // nx*ny*nz + 1
  const double *sx, *sy, *sz, *sw;
  const int *sperm;        // sorted slot -> node index
  const double4 *pos;      // node index -> (x,y,z,w)
  // records of the v5 range kernel (range_v5.cuh)
  const float4 *f4;        // slot -> FP32 filter record ((x,y,z) - lo, w), round-to-nearest
  const double4 *d4;       // slot -> exact record (x, y, z, w); for d <= 3 the low word of .w holds the node index
  const float *fmaxabs;    // device scalar: max |component| over all f4 records (error bound of the FP32 filter)
};

#ifdef __CUDACC__
// Monotone non-decreasing map coordinate -> cell (clamped).  The SAME function
// assigns points to cells and bounds query ranges, so culling only relies on
// monotonicity, never on the exact position of cell boundaries.
__device__ __forceinline__ int cell_of(double x, double lo, double inv, int n) {
  double v = floor(__dmul_rn(__dsub_rn(x, lo), inv));
  v = fmin(fmax(v, 0.0), (double)(n - 1));  // NaN -> 0
  return (int)v;
}
#endif

}  // namespace rrtqx

struct rrtqx_tree {
  rrtqx_ctx *ctx = nullptr;
  int d = 3;
  rrtqx::WrapInfo wrap{};
  int64_t n = 0;         // tree size
  int64_t n_sorted = 0;  // covered by the grid index
  double occupancy = 4.0;
  double aspect = 2.0;   // cell width across rows / cell length along x (C2 sweep, scripts/tune_v5.sh: 1 / 1.5 / 2 / 3 / 4 -> 2.77 / 2.73 / 2.70 / 2.70 / 2.73 ms; 2 keeps kdFindNearest at 0.34 ms)
  int64_t tail_limit = 4096;
  rrtqx::ScratchMap scratch;  // per-tree scratch (nearest-query sort buffers, extend_query state)

  // node table (insertion order)
  rrtqx::DevBuf<double4> pos;
  rrtqx::DevBuf<unsigned> child;  // 2 per node: [2i] left, [2i+1] right; KD_EMPTY when absent
  rrtqx::DevBuf<int32_t> parent;
  rrtqx::DevBuf<int8_t> split;
  rrtqx::DevBuf<int32_t> cur;     // build scratch: current descent position
  rrtqx::DevBuf<int32_t> flagbuf; // small device counters

  // grid index
  int nx = 1, ny = 1, nz = 1;
  double lo[3] = {0, 0, 0}, inv[3] = {1, 1, 1}, cell[3] = {1, 1, 1};
  rrtqx::DevBuf<int32_t> cell_start, cell_cursor, cell_id, sperm;
  rrtqx::DevBuf<double> sx, sy, sz, sw;
  rrtqx::DevBuf<float4> f4;
  rrtqx::DevBuf<double4> d4;
  rrtqx::DevBuf<float> fmaxabs;
  rrtqx::DevBuf<double> bbox_partial;
  rrtqx::DevBuf<int32_t> scan_tmp;

  rrtqx::GridView view() const {
    rrtqx::GridView g;
    g.d = d;
    g.n_sorted = (int)n_sorted;
    g.n_total = (int)n;
    g.nx = nx; g.ny = ny; g.nz = nz;
    for (int i = 0; i < 3; ++i) { g.lo[i] = lo[i]; g.inv[i] = inv[i]; g.cell[i] = cell[i]; }
    g.cell_start = cell_start.p;
    g.sx = sx.p; g.sy = sy.p; g.sz = sz.p; g.sw = sw.p;
    g.sperm = sperm.p;
    g.pos = pos.p;
    g.f4 = f4.p; g.d4 = d4.p; g.fmaxabs = fmaxabs.p;
    return g;
  }
};

namespace rrtqx {
void tree_insert_batch(rrtqx_tree *t, const double *positions, int64_t n);
void tree_insert_point(rrtqx_tree *t, const double *host_position);  // one node, one launch, asynchronous
// one node into each of n distinct trees of one context (host positions, n x d), one launch, asynchronous
void tree_insert_multi(rrtqx_tree *const *trees, int n, const double *positions, int32_t *index_out);
void tree_reindex(rrtqx_tree *t);
// re-index if the unsorted tail has outgrown its limit
void tree_prepare_query(rrtqx_tree *t);
}  // namespace rrtqx
