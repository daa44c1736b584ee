// dubins.cu -- batched Dubins calculateTrajectory on the device
// (DRRT_DubinsEdge_functions.jl:329-709, space without time) and the DubinsEdge steering point
// (saturate, :70-95); the solver, the discretisation and saturate live in dubins.cuh.
//
// One thread solves one edge.  The solver runs twice per batch: a sizing pass (distance, word, number of
// trajectory rows), an exclusive scan of the row counts on the device, and an emission pass that writes
// edge.trajectory[:,1:2] rows into a CSR.
// Library built with -fmad=false: no contraction changes the operation order.
#include <cmath>

#include "common.cuh"
#include "dubins.cuh"
#include "scan.cuh"

namespace rrtqx {

namespace {

__global__ void dubins_size_kernel(const double *__restrict__ starts, const double *__restrict__ goals, int64_t n, double r,
                                   double *__restrict__ dist, int32_t *__restrict__ type, int32_t *__restrict__ rows) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const Word w = solve(starts + 4 * e, goals + 4 * e, r);
  if (dist) dist[e] = w.dist;
  if (type) type[e] = w.type;
  rows[e] = word_rows<false>(w, starts + 4 * e, goals + 4 * e, r, nullptr);
}

__global__ void dubins_emit_kernel(const double *__restrict__ starts, const double *__restrict__ goals, int64_t n, double r,
                                   const int64_t *__restrict__ ptr, double2 *__restrict__ traj) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const Word w = solve(starts + 4 * e, goals + 4 * e, r);
  word_rows<true>(w, starts + 4 * e, goals + 4 * e, r, traj + ptr[e]);
}

// saturate, DubinsEdge version (DRRT_DubinsEdge_functions.jl:70-95), in place on new_points (n x 4)
__global__ void dubins_saturate_kernel(double *__restrict__ pts, const double *__restrict__ closest, int64_t n, double delta) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  dubins_saturate_point(pts + 4 * i, closest + 4 * i, delta);
}

}  // namespace
}  // namespace rrtqx

using namespace rrtqx;

namespace {
template <typename F>
rrtqx_status guarded_d(rrtqx_ctx *ctx, F &&f) {
  try {
    f();
    return RRTQX_OK;
  } catch (const Error &e) {
    if (ctx) ctx->err = e.what();
    return e.code;
  } catch (const std::exception &e) {
    if (ctx) ctx->err = e.what();
    return RRTQX_ERR_INVALID;
  }
}
}  // namespace

extern "C" {

rrtqx_status rrtqx_dubins_trajectory_batch(rrtqx_ctx *ctx, const double *starts, const double *goals, int64_t n_edges,
                                           double min_turn_radius, rrtqx_dubins_result **result) {
  if (!ctx || !result) return RRTQX_ERR_INVALID;
  return guarded_d(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    RQ_REQUIRE(n_edges >= 0 && n_edges < (int64_t)0x7fffffff, "n_edges out of range");
    RQ_REQUIRE(n_edges == 0 || (starts && goals), "NULL array");
    rrtqx_dubins_result *R = *result;
    if (!R) {
      R = new rrtqx_dubins_result();
      R->ctx = ctx;
      *result = R;
    }
    RQ_REQUIRE(R->ctx == ctx, "result belongs to another context");
    cudaStream_t st = ctx->stream;
    R->n_edges = n_edges;
    R->n_rows = 0;
    if (n_edges == 0) return;
    const double *ds = to_device(ctx, starts, (size_t)n_edges * 4, R->starts);
    const double *dg = to_device(ctx, goals, (size_t)n_edges * 4, R->goals);
    R->dist.ensure((size_t)n_edges, st);
    R->type.ensure((size_t)n_edges, st);
    R->rows.ensure((size_t)n_edges + 1, st);
    R->ptr.ensure((size_t)n_edges + 1, st);
    const int TB = 128;
    {
      PhaseScope ph(ctx, "dubins_solve");
      dubins_size_kernel<<<div_up(n_edges, TB), TB, 0, st>>>(ds, dg, n_edges, min_turn_radius, R->dist.p, R->type.p, R->rows.p);
      post_launch(ctx);
      exclusive_scan<int32_t, int64_t>(ctx, R->rows.p, n_edges, R->ptr.p, R->scan_tmp64);
    }
    int64_t total = 0;
    RQ_CUDA(cudaMemcpyAsync(&total, R->ptr.p + n_edges, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    RQ_CUDA(cudaStreamSynchronize(st));
    R->n_rows = total;
    R->traj.ensure((size_t)total + 1, st, 0, 1.0);
    {
      PhaseScope ph(ctx, "dubins_emit");
      dubins_emit_kernel<<<div_up(n_edges, TB), TB, 0, st>>>(ds, dg, n_edges, min_turn_radius, R->ptr.p, R->traj.p);
      post_launch(ctx);
    }
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_dubins_result_destroy(rrtqx_dubins_result *r) {
  if (!r) return RRTQX_OK;
  rrtqx_ctx *ctx = r->ctx;
  if (ctx && handle_live(ctx)) {  // finalizers run in any order: the context may be gone already
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
  } else {
    cudaDeviceSynchronize();
  }
  delete r;
  cudaGetLastError();
  return RRTQX_OK;
}

rrtqx_status rrtqx_dubins_result_sizes(const rrtqx_dubins_result *r, int64_t *n_edges, int64_t *n_rows) {
  if (!r) return RRTQX_ERR_INVALID;
  if (n_edges) *n_edges = r->n_edges;
  if (n_rows) *n_rows = r->n_rows;
  return RRTQX_OK;
}

rrtqx_status rrtqx_dubins_result_fetch(rrtqx_dubins_result *r, double *dist, int32_t *type, int64_t *traj_ptr,
                                       double *traj_xy) {
  if (!r) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = r->ctx;
  return guarded_d(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)r->n_edges;
    if (n == 0) {
      if (traj_ptr && !is_device_ptr(traj_ptr)) traj_ptr[0] = 0;
      return;
    }
    from_device(ctx, dist, r->dist.p, n);
    from_device(ctx, type, r->type.p, n);
    from_device(ctx, traj_ptr, r->ptr.p, n + 1);
    from_device(ctx, traj_xy, (const double *)r->traj.p, 2 * (size_t)r->n_rows);
    RQ_CUDA(cudaStreamSynchronize(ctx->stream));
  });
}

rrtqx_status rrtqx_dubins_result_device(const rrtqx_dubins_result *r, const double **dist, const int32_t **type,
                                        const int64_t **traj_ptr, const double **traj_xy) {
  if (!r) return RRTQX_ERR_INVALID;
  if (dist) *dist = r->dist.p;
  if (type) *type = r->type.p;
  if (traj_ptr) *traj_ptr = r->ptr.p;
  if (traj_xy) *traj_xy = (const double *)r->traj.p;
  return RRTQX_OK;
}

rrtqx_status rrtqx_dubins_saturate_batch(rrtqx_ctx *ctx, double *new_points, const double *closest, int64_t n,
                                         double delta) {
  if (!ctx) return RRTQX_ERR_INVALID;
  return guarded_d(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    RQ_REQUIRE(n >= 0 && (n == 0 || (new_points && closest)), "bad arguments");
    if (n == 0) return;
    cudaStream_t st = ctx->stream;
    const bool pd = is_device_ptr(new_points);
    double *dp = new_points;
    if (!pd) {
      ctx->stage_f64.ensure((size_t)n * 4, st);
      RQ_CUDA(cudaMemcpyAsync(ctx->stage_f64.p, new_points, sizeof(double) * 4 * n, cudaMemcpyHostToDevice, st));
      dp = ctx->stage_f64.p;
    }
    const double *dc = to_device(ctx, closest, (size_t)n * 4, ctx->stage_f64b);
    dubins_saturate_kernel<<<div_up(n, 256), 256, 0, st>>>(dp, dc, n, delta);
    post_launch(ctx);
    if (!pd) RQ_CUDA(cudaMemcpyAsync(new_points, dp, sizeof(double) * 4 * n, cudaMemcpyDeviceToHost, st));
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
