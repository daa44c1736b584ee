// abi.cu -- extern "C" boundary of librrtqx_b200.so (include/rrtqx_b200.h).
// Every entry point converts C++ exceptions into a status + message; there is
// no CPU fallback anywhere behind this file.
#include <cstdlib>
#include <mutex>

#include "objects.cuh"
#include "polygon.cuh"

using namespace rrtqx;

static thread_local std::string g_last_error;

struct NearestScratchHolder {
  rrtqx_range_result sortbuf;
  DevBuf<int32_t> idx;
  DevBuf<double> dist;
};
static const char g_nearest_tag = 0;  // key of the per-tree nearest-query scratch (rrtqx_tree::scratch)

namespace rrtqx {
static std::set<const void *> g_live_handles;
static std::mutex g_live_mutex;
void handle_register(const void *h) { std::lock_guard<std::mutex> lk(g_live_mutex); g_live_handles.insert(h); }
void handle_unregister(const void *h) { std::lock_guard<std::mutex> lk(g_live_mutex); g_live_handles.erase(h); }
bool handle_live(const void *h) { std::lock_guard<std::mutex> lk(g_live_mutex); return g_live_handles.count(h) != 0; }
}  // namespace rrtqx

namespace {
// Destroy a child object whose parent context may already be gone (finalizers run in any order): with a live
// context the stream is drained first; without one the memory is simply released.
template <typename T>
rrtqx_status destroy_child(rrtqx_ctx *ctx, T *obj) {
  if (!obj) return RRTQX_OK;
  if (ctx && handle_live(ctx)) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
  } else {
    cudaDeviceSynchronize();
  }
  delete obj;
  cudaGetLastError();  // a failed synchronise of a dying context must not poison the next launch check
  return RRTQX_OK;
}

template <typename F>
rrtqx_status guarded(rrtqx_ctx *ctx, F &&f) {
  try {
    f();
    return RRTQX_OK;
  } catch (const Error &e) {
    g_last_error = e.what();
    if (ctx) ctx->err = e.what();
    return e.code;
  } catch (const std::bad_alloc &) {
    g_last_error = "host allocation failed";
    if (ctx) ctx->err = g_last_error;
    return RRTQX_ERR_NOMEM;
  } catch (const std::exception &e) {
    g_last_error = e.what();
    if (ctx) ctx->err = e.what();
    return RRTQX_ERR_INVALID;
  }
}
void bind_device(rrtqx_ctx *ctx) { RQ_CUDA(cudaSetDevice(ctx->device)); }
}  // namespace

extern "C" {

const char *rrtqx_version(void) { return "rrtqx-b200 0.1 (sm_100a)"; }

rrtqx_status rrtqx_ctx_create(int32_t device, void *cuda_stream, rrtqx_ctx **out) {
  return guarded(nullptr, [&] {
    RQ_REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
      throw Error(RRTQX_ERR_CUDA, std::string("no usable CUDA device (there is no CPU fallback): ") +
                                      (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    RQ_REQUIRE(device >= 0 && device < count, "device ordinal out of range");
    RQ_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RQ_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
      throw Error(RRTQX_ERR_CUDA, std::string("this library is built for sm_100a only; device is ") + prop.name);
    rrtqx_ctx *c = new rrtqx_ctx();
    c->tune.load();  // the only place (with rrtqx_ctx_reload_tuning) where the environment is read
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (cuda_stream) {
      c->stream = (cudaStream_t)cuda_stream;
      c->own_stream = false;
    } else {
      RQ_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
      c->own_stream = true;
    }
    handle_register(c);
    *out = c;
  });
}

rrtqx_status rrtqx_ctx_destroy(rrtqx_ctx *ctx) {
  if (!ctx || !handle_live(ctx)) return RRTQX_OK;
  handle_unregister(ctx);
  return guarded(nullptr, [&] {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &kv : ctx->phases) {
      if (kv.second.a) cudaEventDestroy(kv.second.a);
      if (kv.second.b) cudaEventDestroy(kv.second.b);
    }
    ctx->scratch.clear();  // device buffers of the collision / sweep paths, while the device is bound
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
  });
}

// Page-locked host memory for the caller's query / result arrays: the library accepts any host pointer, but
// copies from pageable memory are staged by the driver at a fraction of the PCIe rate.
rrtqx_status rrtqx_host_alloc(rrtqx_ctx *ctx, int64_t bytes, void **out) {
  if (!ctx || !out) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(bytes >= 0, "bytes is negative");
    *out = nullptr;
    if (bytes == 0) return;
    cudaError_t e = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); throw Error(RRTQX_ERR_NOMEM, std::string("cudaHostAlloc failed: ") + cudaGetErrorString(e)); }
  });
}

rrtqx_status rrtqx_host_free(rrtqx_ctx *ctx, void *p) {
  if (!p) return RRTQX_OK;
  cudaError_t e = cudaFreeHost(p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    if (ctx && handle_live(ctx)) ctx->err = std::string("cudaFreeHost failed: ") + cudaGetErrorString(e);
    return RRTQX_ERR_INVALID;
  }
  return RRTQX_OK;
}

rrtqx_status rrtqx_ctx_reload_tuning(rrtqx_ctx *ctx) {
  if (!ctx) return RRTQX_ERR_INVALID;
  ctx->tune.load();
  return RRTQX_OK;
}

const char *rrtqx_last_error(const rrtqx_ctx *ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

rrtqx_status rrtqx_ctx_sync(rrtqx_ctx *ctx) {
  if (!ctx) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] { bind_device(ctx); RQ_CUDA(cudaStreamSynchronize(ctx->stream)); });
}

rrtqx_status rrtqx_ctx_kernel_launches(const rrtqx_ctx *ctx, int64_t *out) {
  if (!ctx || !out) return RRTQX_ERR_INVALID;
  *out = ctx->launches;
  return RRTQX_OK;
}

rrtqx_status rrtqx_ctx_last_phase_ms(rrtqx_ctx *ctx, const char *phase, float *ms) {
  if (!ctx) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    RQ_REQUIRE(phase && ms, "NULL argument");
    auto it = ctx->phases.find(phase);
    if (it == ctx->phases.end() || !it->second.valid) throw Error(RRTQX_ERR_STATE, "phase has not run");
    RQ_CUDA(cudaEventSynchronize(it->second.b));
    RQ_CUDA(cudaEventElapsedTime(ms, it->second.a, it->second.b));
  });
}

// ---------------------------------------------------------- measured FP64 peak
// Roofline denominator of the FP64-bound kernels (collision sweeps): 8 independent DFMA chains per thread,
// full occupancy, timed with events on the context's stream.  Not in MEASURED_PEAKS.json, so it is measured
// in the bench run itself (SURVEY.md section 7, "measure it").
namespace rrtqx {
__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = __fma_rn(x0, a, b); x1 = __fma_rn(x1, a, b); x2 = __fma_rn(x2, a, b); x3 = __fma_rn(x3, a, b);
    x4 = __fma_rn(x4, a, b); x5 = __fma_rn(x5, a, b); x6 = __fma_rn(x6, a, b); x7 = __fma_rn(x7, a, b);
  }
  const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
  if (s == 12345.678) out[0] = s;  // never true: keeps the chains alive
}
}  // namespace rrtqx

rrtqx_status rrtqx_ctx_measure_fp64_peak(rrtqx_ctx *ctx, double *tflops) {
  if (!ctx || !tflops) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    bind_device(ctx);
    cudaStream_t st = ctx->stream;
    ctx->stage_f64.ensure(16, st);
    const int iters = 4096, blocks = ctx->sm_count * 8, threads = 256;
    cudaEvent_t a, b;
    RQ_CUDA(cudaEventCreate(&a));
    RQ_CUDA(cudaEventCreate(&b));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
      RQ_CUDA(cudaEventRecord(a, st));
      fp64_peak_kernel<<<blocks, threads, 0, st>>>(ctx->stage_f64.p, iters, 0.999999, 1e-9);
      post_launch(ctx);
      RQ_CUDA(cudaEventRecord(b, st));
      RQ_CUDA(cudaEventSynchronize(b));
      float ms = 0.f;
      RQ_CUDA(cudaEventElapsedTime(&ms, a, b));
      if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    const double flop = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
    *tflops = flop / ((double)best * 1e-3) / 1e12;
  });
}

// ------------------------------------------------------------------- tree
rrtqx_status rrtqx_tree_create(rrtqx_ctx *ctx, int32_t d, int32_t num_wraps, const int32_t *wraps,
                               const double *wrap_points, rrtqx_tree **out) {
  if (!ctx) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    RQ_REQUIRE(out != nullptr, "out is NULL");
    RQ_REQUIRE(d >= 2 && d <= MAX_D, "d must be 2, 3 or 4");
    RQ_REQUIRE(num_wraps >= 0 && num_wraps <= MAX_WRAPS, "num_wraps out of range");
    RQ_REQUIRE(num_wraps == 0 || (wraps && wrap_points), "wraps / wrap_points is NULL");
    rrtqx_tree *t = new rrtqx_tree();
    t->ctx = ctx;
    t->d = d;
    t->wrap.num_wraps = num_wraps;
    if (ctx->tune.grid_occupancy > 0.0) t->occupancy = ctx->tune.grid_occupancy;
    if (ctx->tune.grid_aspect >= 1.0) t->aspect = ctx->tune.grid_aspect;
    for (int i = 0; i < num_wraps; ++i) {
      if (wraps[i] < 0 || wraps[i] >= d) { delete t; throw Error(RRTQX_ERR_INVALID, "wrap dimension out of range"); }
      t->wrap.wraps[i] = wraps[i];
      t->wrap.wrap_points[i] = wrap_points[i];
    }
    handle_register(t);
    *out = t;
  });
}

rrtqx_status rrtqx_tree_destroy(rrtqx_tree *tree) {
  if (!tree || !handle_live(tree)) return RRTQX_OK;
  handle_unregister(tree);
  return destroy_child(tree->ctx, tree);  // frees the per-tree scratch (nearest sort buffers, extend_query state) with it
}

rrtqx_status rrtqx_tree_insert_batch(rrtqx_tree *tree, const double *positions, int64_t n, int32_t *first_index_out) {
  if (!tree) return RRTQX_ERR_INVALID;
  return guarded(tree->ctx, [&] {
    bind_device(tree->ctx);
    RQ_REQUIRE(n >= 0, "n is negative");
    RQ_REQUIRE(positions != nullptr || n == 0, "positions is NULL");
    if (first_index_out) *first_index_out = (int32_t)tree->n;
    tree_insert_batch(tree, positions, n);
    RQ_CUDA(cudaStreamSynchronize(tree->ctx->stream));
  });
}

rrtqx_status rrtqx_tree_insert(rrtqx_tree *tree, const double *position, int32_t *index_out) {
  if (!tree) return RRTQX_ERR_INVALID;
  if (position && is_device_ptr(position)) return rrtqx_tree_insert_batch(tree, position, 1, index_out);
  return guarded(tree->ctx, [&] {
    bind_device(tree->ctx);
    RQ_REQUIRE(position != nullptr, "position is NULL");
    if (index_out) *index_out = (int32_t)tree->n;
    tree_insert_point(tree, position);  // stream-ordered: later calls on this context see the node
  });
}

rrtqx_status rrtqx_tree_size(const rrtqx_tree *tree, int64_t *n) {
  if (!tree || !n) return RRTQX_ERR_INVALID;
  *n = tree->n;
  return RRTQX_OK;
}

__global__ void kd_fields_kernel(const unsigned *__restrict__ child, const int32_t *__restrict__ parent,
                                 const int8_t *__restrict__ split, int64_t first, int64_t count,
                                 int32_t *__restrict__ o_parent, int32_t *__restrict__ o_l, int32_t *__restrict__ o_r,
                                 int32_t *__restrict__ o_split) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  int64_t i = first + k;
  o_parent[k] = parent[i];
  unsigned l = child[2 * i], r = child[2 * i + 1];
  o_l[k] = (l == KD_EMPTY) ? -1 : (int32_t)l;
  o_r[k] = (r == KD_EMPTY) ? -1 : (int32_t)r;
  o_split[k] = split[i];
}

__global__ void positions_kernel(const double4 *__restrict__ pos, int d, int64_t first, int64_t count,
                                 double *__restrict__ out) {
  int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= count) return;
  double4 p = pos[first + k];
  double *o = out + k * d;
  o[0] = p.x;
  o[1] = p.y;
  if (d >= 3) o[2] = p.z;
  if (d >= 4) o[3] = p.w;
}

rrtqx_status rrtqx_tree_kd_fields(rrtqx_tree *tree, int64_t first, int64_t count, int32_t *parent, int32_t *child_l,
                                  int32_t *child_r, int32_t *split) {
  if (!tree) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(first >= 0 && count >= 0 && first + count <= tree->n, "node range out of bounds");
    if (count == 0) return;
    cudaStream_t st = ctx->stream;
    ctx->stage_i32a.ensure((size_t)count * 4, st);
    int32_t *b = ctx->stage_i32a.p;
    kd_fields_kernel<<<div_up(count, 256), 256, 0, st>>>(tree->child.p, tree->parent.p, tree->split.p, first, count, b,
                                                         b + count, b + 2 * count, b + 3 * count);
    post_launch(ctx);
    from_device(ctx, parent, b, (size_t)count);
    from_device(ctx, child_l, b + count, (size_t)count);
    from_device(ctx, child_r, b + 2 * count, (size_t)count);
    from_device(ctx, split, b + 3 * count, (size_t)count);
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

// Visit order of the reference's recursive kd traversals (saveRRTSubNodes / saveRRTSubTree / saveRRTSubGraph,
// DRRT_Q.jl:252-337: node, then kdChildL subtree, then kdChildR subtree).  One bulk copy of the child links, then
// an explicit-stack walk on the host: export for the visualisation dumps, not a hot path.
rrtqx_status rrtqx_tree_preorder(rrtqx_tree *tree, int32_t *order_out) {
  if (!tree) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    const int64_t n = tree->n;
    RQ_REQUIRE(order_out != nullptr || n == 0, "order_out is NULL");
    RQ_REQUIRE(!is_device_ptr(order_out), "order_out must be a host array");
    if (n == 0) return;
    std::vector<unsigned> child(2 * (size_t)n);
    RQ_CUDA(cudaMemcpyAsync(child.data(), tree->child.p, sizeof(unsigned) * 2 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
    std::vector<int32_t> stack;
    stack.push_back(0);
    int64_t k = 0;
    while (!stack.empty()) {
      const int32_t v = stack.back();
      stack.pop_back();
      RQ_REQUIRE(k < n, "kd links are inconsistent");
      order_out[k++] = v;
      const unsigned l = child[2 * (size_t)v], r = child[2 * (size_t)v + 1];
      if (r != KD_EMPTY) stack.push_back((int32_t)r);  // right is visited after the whole left subtree
      if (l != KD_EMPTY) stack.push_back((int32_t)l);
    }
    RQ_REQUIRE(k == n, "kd links do not reach every node");
  });
}

rrtqx_status rrtqx_tree_positions(rrtqx_tree *tree, int64_t first, int64_t count, double *out) {
  if (!tree) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(first >= 0 && count >= 0 && first + count <= tree->n, "node range out of bounds");
    RQ_REQUIRE(out != nullptr || count == 0, "out is NULL");
    if (count == 0) return;
    cudaStream_t st = ctx->stream;
    ctx->stage_f64.ensure((size_t)count * tree->d, st);
    positions_kernel<<<div_up(count, 256), 256, 0, st>>>(tree->pos.p, tree->d, first, count, ctx->stage_f64.p);
    post_launch(ctx);
    from_device(ctx, out, ctx->stage_f64.p, (size_t)count * tree->d);
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_tree_set_cell_occupancy(rrtqx_tree *tree, double points_per_cell) {
  if (!tree) return RRTQX_ERR_INVALID;
  return guarded(tree->ctx, [&] {
    RQ_REQUIRE(points_per_cell > 0.0 && points_per_cell <= 4096.0, "points_per_cell out of range");
    tree->occupancy = points_per_cell;
  });
}

rrtqx_status rrtqx_tree_reindex(rrtqx_tree *tree) {
  if (!tree) return RRTQX_ERR_INVALID;
  return guarded(tree->ctx, [&] {
    bind_device(tree->ctx);
    tree_reindex(tree);
    RQ_CUDA(cudaStreamSynchronize(tree->ctx->stream));
  });
}

// ---------------------------------------------------------- range / nearest
rrtqx_status rrtqx_range_query_batch(rrtqx_tree *tree, const double *queries, int64_t n_queries, double range,
                                     const double *ranges, uint32_t flags, rrtqx_range_result **result,
                                     int64_t *total_out) {
  if (!tree) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(result != nullptr, "result is NULL");
    RQ_REQUIRE(queries != nullptr || n_queries == 0, "queries is NULL");
    if (!*result) {
      *result = new rrtqx_range_result();
      (*result)->ctx = ctx;
    }
    range_query(tree, queries, n_queries, range, ranges, flags, *result);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
    if (total_out) *total_out = (*result)->total;
  });
}

rrtqx_status rrtqx_range_result_destroy(rrtqx_range_result *r) { return r ? destroy_child(r->ctx, r) : RRTQX_OK; }

rrtqx_status rrtqx_range_result_sizes(const rrtqx_range_result *r, int64_t *n_queries, int64_t *total) {
  if (!r) return RRTQX_ERR_INVALID;
  if (n_queries) *n_queries = r->n_queries;
  if (total) *total = r->total;
  return RRTQX_OK;
}

rrtqx_status rrtqx_range_result_layout(rrtqx_range_result *r, int32_t *counts, int64_t *offsets) {
  if (!r) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = r->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    from_device(ctx, counts, r->counts.p, (size_t)r->n_queries);
    from_device(ctx, offsets, r->offsets.p, (size_t)r->n_queries);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_range_result_fetch(rrtqx_range_result *r, int32_t *idx, double *dist) {
  if (!r) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = r->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    if (!r->has_lists) throw Error(RRTQX_ERR_STATE, "result holds counts only (RRTQX_RANGE_COUNT_ONLY)");
    if (dist && !r->has_dist) throw Error(RRTQX_ERR_STATE, "distances were not requested (RRTQX_RANGE_WANT_DIST)");
    from_device(ctx, idx, r->idx.p, (size_t)r->total);
    from_device(ctx, dist, r->dist.p, (size_t)r->total);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_range_result_device(const rrtqx_range_result *r, const int32_t **counts, const int64_t **offsets,
                                       const int32_t **idx, const double **dist) {
  if (!r) return RRTQX_ERR_INVALID;
  if (counts) *counts = r->counts.p;
  if (offsets) *offsets = r->offsets.p;
  if (idx) *idx = r->has_lists ? r->idx.p : nullptr;
  if (dist) *dist = r->has_dist ? r->dist.p : nullptr;
  return RRTQX_OK;
}

rrtqx_status rrtqx_nearest_batch(rrtqx_tree *tree, const double *queries, int64_t n_queries, int32_t *idx_out,
                                 double *dist_out) {
  if (!tree) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(queries != nullptr || n_queries == 0, "queries is NULL");
    NearestScratchHolder *h = &tree->scratch.get<NearestScratchHolder>(&g_nearest_tag);
    h->sortbuf.ctx = ctx;
    nearest_query(tree, &h->sortbuf, queries, n_queries, idx_out, dist_out, h->idx, h->dist);
  });
}

rrtqx_status rrtqx_extend_query(rrtqx_tree *tree, const rrtqx_spheres *spheres, const double *point, double range,
                                double robot_radius, uint32_t flags, int32_t capacity, int32_t *nearest_idx,
                                double *nearest_dist, uint8_t *point_collides, double *point_cert,
                                int32_t *n_neighbors, int32_t *nbr_idx, double *nbr_dist, uint8_t *fwd_collide,
                                uint8_t *rev_collide) {
  if (!tree || !spheres) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    extend_query(tree, spheres, point, range, robot_radius, flags, capacity, nearest_idx, nearest_dist, point_collides,
                 point_cert, n_neighbors, nbr_idx, nbr_dist, fwd_collide, rev_collide);
  });
}

rrtqx_status rrtqx_extend_query_dubins(rrtqx_tree *tree, const rrtqx_polygons *polygons, double *point, double delta,
                                       double range, double robot_radius, double min_turn_radius, uint32_t flags,
                                       int32_t capacity, int32_t *nearest_idx, double *nearest_dist,
                                       int32_t *n_neighbors, int32_t *nbr_idx, double *nbr_dist, double *edge_dist,
                                       int32_t *edge_type, uint8_t *edge_collide,
                                       rrtqx_dubins_result **trajectories) {
  if (!tree || !polygons) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    extend_query_dubins(tree, polygons, point, delta, range, robot_radius, min_turn_radius, flags, capacity,
                        nearest_idx, nearest_dist, n_neighbors, nbr_idx, nbr_dist, edge_dist, edge_type, edge_collide,
                        trajectories);
  });
}

// ---------------------------------------------------------------- spheres
rrtqx_status rrtqx_spheres_create(rrtqx_ctx *ctx, rrtqx_spheres **out) {
  if (!ctx) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    RQ_REQUIRE(out != nullptr, "out is NULL");
    rrtqx_spheres *s = new rrtqx_spheres();
    s->ctx = ctx;
    *out = s;
  });
}

rrtqx_status rrtqx_spheres_destroy(rrtqx_spheres *s) { return s ? destroy_child(s->ctx, s) : RRTQX_OK; }

__global__ void spheres_pack_kernel(const double *__restrict__ centers, const double *__restrict__ radii, int64_t first,
                                    int64_t n, double4 *__restrict__ rec) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double4 r = rec[first + i];
  if (centers) { r.x = centers[3 * i]; r.y = centers[3 * i + 1]; r.z = centers[3 * i + 2]; }
  if (radii) r.w = radii[i];
  rec[first + i] = r;
}

rrtqx_status rrtqx_spheres_upload(rrtqx_spheres *s, const double *centers, const double *radii, const uint8_t *active,
                                  int64_t n) {
  if (!s) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = s->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(n >= 0 && n < (1 << 24), "n out of range");
    RQ_REQUIRE(n == 0 || (centers && radii), "centers / radii is NULL");
    cudaStream_t st = ctx->stream;
    s->rec.ensure((size_t)n + 1, st);
    s->active.ensure((size_t)n + 1, st);
    s->n = n;
    s->version = next_content_stamp();
    if (n == 0) return;
    const double *dc = to_device(ctx, centers, (size_t)n * 3, ctx->stage_f64);
    const double *dr = to_device(ctx, radii, (size_t)n, ctx->stage_f64b);
    spheres_pack_kernel<<<div_up(n, 256), 256, 0, st>>>(dc, dr, 0, n, s->rec.p);
    post_launch(ctx);
    if (active) RQ_CUDA(cudaMemcpyAsync(s->active.p, active, (size_t)n, cudaMemcpyDefault, st));
    else RQ_CUDA(cudaMemsetAsync(s->active.p, 1, (size_t)n, st));
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_spheres_update(rrtqx_spheres *s, int64_t first, int64_t count, const double *radii,
                                  const uint8_t *active) {
  if (!s) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = s->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(first >= 0 && count >= 0 && first + count <= s->n, "obstacle range out of bounds");
    if (count == 0) return;
    s->version = next_content_stamp();
    cudaStream_t st = ctx->stream;
    if (radii) {
      const double *dr = to_device(ctx, radii, (size_t)count, ctx->stage_f64b);
      spheres_pack_kernel<<<div_up(count, 256), 256, 0, st>>>(nullptr, dr, first, count, s->rec.p);
      post_launch(ctx);
    }
    if (active) RQ_CUDA(cudaMemcpyAsync(s->active.p + first, active, (size_t)count, cudaMemcpyDefault, st));
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_spheres_size(const rrtqx_spheres *s, int64_t *n) {
  if (!s || !n) return RRTQX_ERR_INVALID;
  *n = s->n;
  return RRTQX_OK;
}

// ------------------------------------------------------------ collision
rrtqx_status rrtqx_edge_check_batch(rrtqx_tree *tree, const rrtqx_spheres *spheres, const int32_t *src,
                                    const int32_t *dst, int64_t n_edges, double robot_radius, uint32_t flags,
                                    uint8_t *collide_out) {
  if (!tree || !spheres) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(tree->d == 3, "SimpleEdge checks need a 3-D tree (explicitEdgeCheck3D)");
    RQ_REQUIRE(n_edges >= 0, "n_edges is negative");
    RQ_REQUIRE(n_edges == 0 || (src && dst && collide_out), "NULL array");
    // endpoint indices are validated on the device, inside the kernels that gather the positions (host and
    // device arrays alike): a bad index fails the call with RRTQX_ERR_INVALID
    edge_check(ctx, tree, spheres, src, dst, nullptr, nullptr, n_edges, robot_radius, flags, collide_out);
  });
}

rrtqx_status rrtqx_segment_check_batch(rrtqx_ctx *ctx, const rrtqx_spheres *spheres, const double *starts,
                                       const double *ends, int64_t n_segments, double robot_radius, uint32_t flags,
                                       uint8_t *collide_out) {
  if (!ctx || !spheres) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(n_segments >= 0, "n_segments is negative");
    RQ_REQUIRE(n_segments == 0 || (starts && ends && collide_out), "NULL array");
    edge_check(ctx, nullptr, spheres, nullptr, nullptr, starts, ends, n_segments, robot_radius, flags, collide_out);
  });
}

rrtqx_status rrtqx_node_check_batch(rrtqx_ctx *ctx, const rrtqx_spheres *spheres, const double *points, int64_t n,
                                    double robot_radius, uint32_t flags, uint8_t *collide_out, double *cert_out) {
  if (!ctx || !spheres) return RRTQX_ERR_INVALID;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(n >= 0, "n is negative");
    RQ_REQUIRE(n == 0 || (points && collide_out), "NULL array");
    node_check(ctx, spheres, points, n, robot_radius, flags, collide_out, cert_out);
  });
}

// ------------------------------------------------------------ edges + sweeps
rrtqx_status rrtqx_edges_create(rrtqx_tree *tree, rrtqx_edges **out) {
  if (!tree) return RRTQX_ERR_INVALID;
  return guarded(tree->ctx, [&] {
    RQ_REQUIRE(out != nullptr, "out is NULL");
    rrtqx_edges *e = new rrtqx_edges();
    e->tree = tree;
    *out = e;
  });
}

rrtqx_status rrtqx_edges_destroy(rrtqx_edges *e) {
  if (!e) return RRTQX_OK;
  rrtqx_ctx *ctx = handle_live(e->tree) ? e->tree->ctx : nullptr;  // the tree may have been finalized first
  if (e->solved) rrtqx_dubins_result_destroy(e->solved);
  return destroy_child(ctx, e);
}

rrtqx_status rrtqx_edges_upload(rrtqx_edges *e, const int32_t *src, const int32_t *dst, int64_t n_edges,
                                const int32_t *parent, int64_t n_parent) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(n_edges == 0 || (src && dst), "src / dst is NULL");
    edges_upload(e, src, dst, n_edges, parent, n_parent);
  });
}

rrtqx_status rrtqx_edges_append(rrtqx_edges *e, const int32_t *src, const int32_t *dst, int64_t n_new) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(n_new == 0 || (src && dst), "src / dst is NULL");
    edges_append(e, src, dst, n_new);
  });
}

rrtqx_status rrtqx_edges_set_parents(rrtqx_edges *e, const int32_t *node_ids, const int32_t *parent_ids, int64_t n) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    edges_set_parents(e, node_ids, parent_ids, n);
  });
}

rrtqx_status rrtqx_edges_check_batch(rrtqx_edges *e, const rrtqx_spheres *spheres, double robot_radius, uint32_t flags,
                                     uint8_t *collide_out) {
  if (!e || !spheres) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    edges_check(e, spheres, robot_radius, flags, collide_out);
  });
}

rrtqx_status rrtqx_edges_size(const rrtqx_edges *e, int64_t *n_edges) {
  if (!e || !n_edges) return RRTQX_ERR_INVALID;
  *n_edges = e->n_edges;
  return RRTQX_OK;
}

rrtqx_status rrtqx_obstacle_add_sweep(rrtqx_edges *edges, const rrtqx_spheres *spheres, const int32_t *ob_ids,
                                      int64_t n_obs, double robot_radius, double delta, uint32_t flags,
                                      rrtqx_sweep_result **result) {
  if (!edges || !spheres) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = edges->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(result != nullptr, "result is NULL");
    RQ_REQUIRE(ob_ids != nullptr || n_obs == 0, "ob_ids is NULL");
    if (!*result) *result = new rrtqx_sweep_result();
    obstacle_add_sweep(edges, spheres, ob_ids, n_obs, robot_radius, delta, flags, *result);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_obstacle_remove_sweep(rrtqx_edges *edges, const rrtqx_spheres *spheres, int32_t ob_id,
                                         const int32_t *other_ids, int64_t n_others, const uint8_t *edge_dist_inf,
                                         double robot_radius, double delta, uint32_t flags,
                                         rrtqx_sweep_result **result) {
  if (!edges || !spheres) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = edges->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(result != nullptr, "result is NULL");
    RQ_REQUIRE(other_ids != nullptr || n_others == 0, "other_ids is NULL");
    if (!*result) *result = new rrtqx_sweep_result();
    obstacle_remove_sweep(edges, spheres, ob_id, other_ids, n_others, edge_dist_inf, robot_radius, delta, flags, *result);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

// ------------------------------------------- Otte / Dubins sweeps (2-D polygon world)
rrtqx_status rrtqx_edges_set_trajectories(rrtqx_edges *e, const int64_t *traj_ptr, const double *traj_xy) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    edges_set_trajectories(e, traj_ptr, traj_xy);
  });
}

rrtqx_status rrtqx_edges_solve_trajectories(rrtqx_edges *e, double min_turn_radius, int64_t *n_rows_out) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    edges_solve_trajectories(e, min_turn_radius);
    if (n_rows_out) *n_rows_out = e->traj_rows;
  });
}

rrtqx_status rrtqx_edges_trajectories_device(const rrtqx_edges *e, const int64_t **traj_ptr, const double **traj_xy,
                                             int64_t *n_items, int64_t *n_rows) {
  if (!e) return RRTQX_ERR_INVALID;
  if (e->traj_items < 0) return RRTQX_ERR_STATE;
  if (traj_ptr) *traj_ptr = e->d_traj_ptr;
  if (traj_xy) *traj_xy = e->d_traj_xy;
  if (n_items) *n_items = e->traj_items;
  if (n_rows) *n_rows = e->traj_rows;
  return RRTQX_OK;
}

rrtqx_status rrtqx_edges_trajectories_fetch(rrtqx_edges *e, int64_t *traj_ptr, double *traj_xy) {
  if (!e) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = e->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    if (e->traj_items < 0) throw Error(RRTQX_ERR_STATE, "no trajectories are resident");
    from_device(ctx, traj_ptr, e->d_traj_ptr, (size_t)e->traj_items + 1);
    from_device(ctx, traj_xy, e->d_traj_xy, (size_t)e->traj_rows * 2);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_obstacle_add_sweep_2d(rrtqx_edges *edges, const rrtqx_polygons *polygons, const int32_t *ob_ids,
                                         int64_t n_obs, double robot_radius, double delta, double min_turn_radius,
                                         uint32_t flags, rrtqx_sweep_result **result) {
  if (!edges || !polygons) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = edges->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(result != nullptr, "result is NULL");
    RQ_REQUIRE(ob_ids != nullptr || n_obs == 0, "ob_ids is NULL");
    if (!*result) *result = new rrtqx_sweep_result();
    obstacle_add_sweep_2d(edges, polygons, ob_ids, n_obs, robot_radius, delta, min_turn_radius, flags, *result);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_obstacle_remove_sweep_2d(rrtqx_edges *edges, const rrtqx_polygons *polygons, int32_t ob_id,
                                            const int32_t *other_ids, int64_t n_others, const uint8_t *edge_dist_inf,
                                            double robot_radius, double delta, double min_turn_radius, uint32_t flags,
                                            rrtqx_sweep_result **result) {
  if (!edges || !polygons) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = edges->tree->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    RQ_REQUIRE(result != nullptr, "result is NULL");
    RQ_REQUIRE(other_ids != nullptr || n_others == 0, "other_ids is NULL");
    if (!*result) *result = new rrtqx_sweep_result();
    obstacle_remove_sweep_2d(edges, polygons, ob_id, other_ids, n_others, edge_dist_inf, robot_radius, delta,
                             min_turn_radius, flags, *result);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_sweep_result_destroy(rrtqx_sweep_result *r) { return r ? destroy_child(r->ctx, r) : RRTQX_OK; }

rrtqx_status rrtqx_sweep_result_sizes(const rrtqx_sweep_result *r, int64_t *n_edge_hits, int64_t *n_node_hits,
                                      int64_t *n_candidates, int64_t *n_pair_tests) {
  if (!r) return RRTQX_ERR_INVALID;
  if (n_edge_hits) *n_edge_hits = r->n_edge_hits;
  if (n_node_hits) *n_node_hits = r->n_node_hits;
  if (n_candidates) *n_candidates = r->n_candidates;
  if (n_pair_tests) *n_pair_tests = r->n_pair_tests;
  return RRTQX_OK;
}

rrtqx_status rrtqx_sweep_result_fetch(rrtqx_sweep_result *r, int32_t *edge_ids, int32_t *node_ids) {
  if (!r || !r->ctx) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = r->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    from_device(ctx, edge_ids, r->edge_list.p, (size_t)r->n_edge_hits);
    from_device(ctx, node_ids, r->node_list.p, (size_t)r->n_node_hits);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_sweep_result_flags(rrtqx_sweep_result *r, uint8_t *edge_flag, uint8_t *node_flag) {
  if (!r || !r->ctx) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = r->ctx;
  return guarded(ctx, [&] {
    bind_device(ctx);
    sweep_result_rebuild_flags(ctx, r);
    from_device(ctx, edge_flag, r->edge_flag.p, (size_t)r->n_edges);
    from_device(ctx, node_flag, r->node_flag.p, (size_t)r->n_nodes);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

}  // extern "C"
