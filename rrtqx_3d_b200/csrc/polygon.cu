// polygon.cu -- 2-D obstacle world of the Otte generation (DRRT.jl) used by DubinsEdge:
//   distanceSqrdPointToSegment   DRRT.jl:1060-1083
//   segmentDistSqrd              DRRT.jl:1144-1202
//   explicitEdgeCheck2D          DRRT.jl:1523-1578   (kinds 1 = ball, 3 = polygon; no time dimension)
//   Dubins explicitEdgeCheck     DRRT_DubinsEdge_functions.jl:750-774
//   explicitEdgeCheck(C, edge)   DRRT.jl:1660-1678   (OR over the obstacle list)
// Every operation is individually rounded FP64 in the reference's order.
#include <cstdlib>

#include "objects.cuh"
#include "polygon.cuh"

namespace rrtqx {

// explicitEdgeCheck2D OR-ed over all obstacles, one thread per segment
__global__ void __launch_bounds__(256)
segment_check_2d_kernel(PolyView P, int ignore_active, const double *__restrict__ starts,
                        const double *__restrict__ ends, int64_t n, double rad, uint8_t *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double sx = starts[2 * i], sy = starts[2 * i + 1], ex = ends[2 * i], ey = ends[2 * i + 1];
  bool hit = false;
  for (int o = 0; o < P.n && !hit; ++o) hit = edge_check_2d(P, o, ignore_active, sx, sy, ex, ey, rad);
  out[i] = hit ? 1 : 0;
}

// Dubins explicitEdgeCheck OR-ed over ALL obstacles of the set: one warp per edge (dubins_collide_warp, polygon.cuh).
constexpr int DUBINS_CHECK_BLOCKS_PER_SM = 6;  // FP64 dependency chains: latency-bound, 48 warps per SM beat 16 although 40 registers spill (0.93 -> 0.60 ms on C4)
__global__ void __launch_bounds__(256, DUBINS_CHECK_BLOCKS_PER_SM)
dubins_check_kernel(PolyView P, int ignore_active, const double *__restrict__ starts, const double *__restrict__ ends,
                    const int64_t *__restrict__ tptr, const double *__restrict__ traj, int64_t n_edges, double rho,
                    double rho_coarse, uint8_t *__restrict__ out) {
  const int64_t e = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (e >= n_edges) return;
  const bool collide = dubins_collide_warp(P, ignore_active != 0, AllObstacles{P.n}, starts[2 * e], starts[2 * e + 1],
                                           ends[2 * e], ends[2 * e + 1], traj, tptr[e], tptr[e + 1], rho, rho_coarse);
  if (lane_id() == 0) out[e] = collide ? 1 : 0;
}

}  // namespace rrtqx

using namespace rrtqx;

namespace {
template <typename F>
rrtqx_status guarded_p(rrtqx_ctx *ctx, F &&f) {
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

rrtqx_status rrtqx_polygons_create(rrtqx_ctx *ctx, rrtqx_polygons **out) {
  if (!ctx || !out) return RRTQX_ERR_INVALID;
  return guarded_p(ctx, [&] {
    rrtqx_polygons *p = new rrtqx_polygons();
    p->ctx = ctx;
    *out = p;
  });
}

rrtqx_status rrtqx_polygons_destroy(rrtqx_polygons *p) {
  if (!p) return RRTQX_OK;
  rrtqx_ctx *ctx = p->ctx;
  if (ctx && handle_live(ctx)) {  // finalizers run in any order: the context may be gone already
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
  } else {
    cudaDeviceSynchronize();
  }
  delete p;
  cudaGetLastError();
  return RRTQX_OK;
}

rrtqx_status rrtqx_polygons_upload(rrtqx_polygons *p, const int32_t *kind, const double *centers,
                                   const double *radii, const uint8_t *active, const int64_t *vert_ptr,
                                   const double *verts, int64_t n) {
  if (!p) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = p->ctx;
  return guarded_p(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    RQ_REQUIRE(n >= 0 && n < (1 << 24), "n out of range");
    RQ_REQUIRE(n == 0 || (kind && centers && radii && vert_ptr), "NULL array");
    RQ_REQUIRE(!is_device_ptr(vert_ptr), "vert_ptr must be a host array");
    cudaStream_t st = ctx->stream;
    const int64_t nv = n ? vert_ptr[n] : 0;
    RQ_REQUIRE(nv >= 0 && (nv == 0 || verts), "bad vertex arrays");
    for (int64_t i = 0; i < n; ++i) RQ_REQUIRE(vert_ptr[i] <= vert_ptr[i + 1], "vert_ptr must be non-decreasing");
    p->kind.ensure((size_t)n + 1, st); p->center.ensure((size_t)n + 1, st); p->radius.ensure((size_t)n + 1, st);
    p->active.ensure((size_t)n + 1, st); p->vptr.ensure((size_t)n + 2, st); p->verts.ensure((size_t)nv + 1, st);
    p->n = n; p->nv = nv;
    if (n == 0) return;
    RQ_CUDA(cudaMemcpyAsync(p->kind.p, kind, sizeof(int32_t) * n, cudaMemcpyDefault, st));
    RQ_CUDA(cudaMemcpyAsync(p->center.p, centers, sizeof(double) * 2 * n, cudaMemcpyDefault, st));
    RQ_CUDA(cudaMemcpyAsync(p->radius.p, radii, sizeof(double) * n, cudaMemcpyDefault, st));
    if (active) RQ_CUDA(cudaMemcpyAsync(p->active.p, active, (size_t)n, cudaMemcpyDefault, st));
    else RQ_CUDA(cudaMemsetAsync(p->active.p, 1, (size_t)n, st));
    RQ_CUDA(cudaMemcpyAsync(p->vptr.p, vert_ptr, sizeof(int64_t) * (n + 1), cudaMemcpyDefault, st));
    if (nv) RQ_CUDA(cudaMemcpyAsync(p->verts.p, verts, sizeof(double) * 2 * nv, cudaMemcpyDefault, st));
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_segment_check_2d_batch(rrtqx_polygons *p, const double *starts, const double *ends, int64_t n,
                                          double radius, uint32_t flags, uint8_t *collide_out) {
  if (!p) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = p->ctx;
  return guarded_p(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    RQ_REQUIRE(n >= 0 && (n == 0 || (starts && ends && collide_out)), "bad arguments");
    if (n == 0) return;
    cudaStream_t st = ctx->stream;
    const double *ds = to_device(ctx, starts, (size_t)n * 2, p->s_a);
    const double *de = to_device(ctx, ends, (size_t)n * 2, p->s_b);
    const bool od = is_device_ptr(collide_out);
    uint8_t *dout = collide_out;
    if (!od) { p->s_out.ensure((size_t)n, st); dout = p->s_out.p; }
    {
      PhaseScope ph(ctx, "edge_check_2d");
      segment_check_2d_kernel<<<div_up(n, 256), 256, 0, st>>>(p->view(), (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0, ds,
                                                              de, n, radius, dout);
      post_launch(ctx);
    }
    if (!od) from_device(ctx, collide_out, dout, (size_t)n);
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

rrtqx_status rrtqx_dubins_edge_check_batch(rrtqx_polygons *p, const double *starts, const double *ends,
                                           const int64_t *traj_ptr, const double *traj_xy, int64_t n_edges,
                                           double robot_radius, double min_turn_radius, uint32_t flags,
                                           uint8_t *collide_out) {
  if (!p) return RRTQX_ERR_INVALID;
  rrtqx_ctx *ctx = p->ctx;
  return guarded_p(ctx, [&] {
    RQ_CUDA(cudaSetDevice(ctx->device));
    RQ_REQUIRE(n_edges >= 0 && (n_edges == 0 || (starts && ends && traj_ptr && collide_out)), "bad arguments");
    if (n_edges == 0) return;
    cudaStream_t st = ctx->stream;
    int64_t npts = 0;
    if (is_device_ptr(traj_ptr)) RQ_CUDA(cudaMemcpy(&npts, traj_ptr + n_edges, sizeof(int64_t), cudaMemcpyDeviceToHost));
    else npts = traj_ptr[n_edges];
    RQ_REQUIRE(npts >= 0 && (npts == 0 || traj_xy), "bad trajectory arrays");
    const double *ds = to_device(ctx, starts, (size_t)n_edges * 2, p->s_a);
    const double *de = to_device(ctx, ends, (size_t)n_edges * 2, p->s_b);
    const int64_t *dp = to_device(ctx, traj_ptr, (size_t)n_edges + 1, p->s_ptr);
    const double *dt = to_device(ctx, traj_xy, (size_t)npts * 2, p->s_t);
    const bool od = is_device_ptr(collide_out);
    uint8_t *dout = collide_out;
    if (!od) { p->s_out.ensure((size_t)n_edges, st); dout = p->s_out.p; }
    {
      PhaseScope ph(ctx, "dubins_check");
      // S.robotRadius + 2*S.minTurningRadius (DRRT_DubinsEdge_functions.jl:758)
      const double rho_coarse = robot_radius + 2 * min_turn_radius;
      dubins_check_kernel<<<div_up(n_edges * 32, 256), 256, 0, st>>>(p->view(), (flags & RRTQX_CHECK_IGNORE_ACTIVE) ? 1 : 0,
                                                                    ds, de, dp, dt, n_edges, robot_radius, rho_coarse, dout);
      post_launch(ctx);
    }
    if (!od) from_device(ctx, collide_out, dout, (size_t)n_edges);
    RQ_CUDA(cudaStreamSynchronize(st));
  });
}

}  // extern "C"
