// polygon.cuh -- 2-D obstacle world of the Otte generation (DRRT.jl) used by DubinsEdge: the obstacle table and the
// exact predicates, shared by the batched checks (polygon.cu) and the Otte / Dubins obstacle sweeps (sweep2d.cu).
//   distanceSqrdPointToSegment   DRRT.jl:1060-1083
//   segmentDistSqrd              DRRT.jl:1144-1202
//   explicitEdgeCheck2D          DRRT.jl:1523-1578   (kinds 1 = ball, 3 = polygon; no time dimension)
// Every operation is individually rounded FP64 in the reference's order.
#pragma once
#include "common.cuh"

namespace rrtqx {

struct PolyView {
  const int32_t *kind;
  const double2 *center;
  const double *radius;
  const uint8_t *active;
  const int64_t *vptr;
  const double2 *verts;
  int n;
};

__device__ __forceinline__ double dist2_point_segment_2d(double px, double py, double sx, double sy, double ex,
                                                          double ey) {
  const double vx = __dsub_rn(px, sx), vy = __dsub_rn(py, sy);
  const double ux = __dsub_rn(ex, sx), uy = __dsub_rn(ey, sy);
  const double det = __dadd_rn(__dmul_rn(vx, ux), __dmul_rn(vy, uy));
  if (det <= 0) return __dadd_rn(__dmul_rn(vx, vx), __dmul_rn(vy, vy));
  const double len = __dadd_rn(__dmul_rn(ux, ux), __dmul_rn(uy, uy));
  if (det >= len) {
    const double ax = __dsub_rn(ex, px), ay = __dsub_rn(ey, py);
    return __dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay));
  }
  const double c = __dsub_rn(__dmul_rn(ux, vy), __dmul_rn(uy, vx));
  return __ddiv_rn(__dmul_rn(c, c), len);
}

// one side-of-line pre-test of segmentDistSqrd: false if Q lies strictly on one side of line(PA,PB)
__device__ __forceinline__ bool may_cross(double pax, double pay, double pbx, double pby, double qax, double qay,
                                          double qbx, double qby) {
  if (fabs(__dsub_rn(pbx, pax)) < .000001) {  // DRRT.jl:1152-1157
    if ((qax >= pax && qbx >= pax) || (qax <= pax && qbx <= pax)) return false;
  } else {  // :1158-1169
    const double m = __ddiv_rn(__dsub_rn(pby, pay), __dsub_rn(pbx, pax));
    const double diffA = __dsub_rn(__dadd_rn(__dmul_rn(m, __dsub_rn(qax, pax)), pay), qay);
    const double diffB = __dsub_rn(__dadd_rn(__dmul_rn(m, __dsub_rn(qbx, pax)), pay), qby);
    if ((diffA > 0.0 && diffB > 0.0) || (diffA < 0.0 && diffB < 0.0)) return false;
  }
  return true;
}

__device__ __forceinline__ double segment_dist2_2d(double pax, double pay, double pbx, double pby, double qax,
                                                   double qay, double qbx, double qby) {
  bool possible = may_cross(pax, pay, pbx, pby, qax, qay, qbx, qby);
  if (possible) possible = may_cross(qax, qay, qbx, qby, pax, pay, pbx, pby);  // :1172-1190
  if (possible) return 0.0;                                                      // :1192-1195
  double r = jl_min(dist2_point_segment_2d(pax, pay, qax, qay, qbx, qby),
                    dist2_point_segment_2d(pbx, pby, qax, qay, qbx, qby));       // :1199-1202, min folds left
  r = jl_min(r, dist2_point_segment_2d(qax, qay, pax, pay, pbx, pby));
  r = jl_min(r, dist2_point_segment_2d(qbx, qby, pax, pay, pbx, pby));
  return r;
}

// explicitEdgeCheck2D for one obstacle
__device__ inline bool edge_check_2d(const PolyView &P, int o, bool ignore_active, double sx, double sy, double ex,
                                     double ey, double rad) {
  if (!ignore_active && !P.active[o]) return false;  // obstacleUnused || lifeSpan <= 0
  const double2 c = P.center[o];
  const double d2 = dist2_point_segment_2d(c.x, c.y, sx, sy, ex, ey);  // :1536
  const double rr = __dadd_rn(rad, P.radius[o]);
  if (d2 > __dmul_rn(rr, rr)) return false;  // :1537-1539
  const int kind = P.kind[o];
  if (kind == 1) return true;
  if (kind != 3) return false;
  const int64_t v0 = P.vptr[o], v1 = P.vptr[o + 1];
  if (v1 - v0 < 2) return false;  // :1551-1553
  const double r2 = __dmul_rn(rad, rad);
  double2 A = P.verts[v1 - 1];
  for (int64_t i = v0; i < v1; ++i) {  // :1556-1578
    const double2 B = P.verts[i];
    if (segment_dist2_2d(sx, sy, ex, ey, A.x, A.y, B.x, B.y) < r2) return true;
    A = B;
  }
  return false;
}

// Dubins explicitEdgeCheck (DRRT_DubinsEdge_functions.jl:750-774) of ONE edge by ONE warp, OR-ed over the obstacles
// a selector names.  Sel: int count(); int id(int k) -> obstacle number; bool admit(int k) -> extra condition
// on obstacle k for this edge (the sweeps' start-node filter).  The circle part of the coarse start->end test
// (radius rho + 2 r_turn, :757-760) runs lane-parallel over 32 obstacles, the polygon part of the survivors is
// spread over the lanes (8 lanes per obstacle, one polygon edge each, 4 obstacles per round), and every obstacle
// that passed is tested against the trajectory segments, 32 segments per trip (:767-771).  The same predicates
// on the same operands as the reference; only the order of an OR changes.  Returns a warp-uniform flag.
template <class Sel>
__device__ __forceinline__ bool dubins_collide_warp(const PolyView &P, bool ignore_active, const Sel &sel, double sx,
                                                    double sy, double ex, double ey, const double *__restrict__ traj,
                                                    int64_t t0, int64_t t1, double rho, double rho_coarse) {
  const int lane = lane_id();
  const double rc2 = __dmul_rn(rho_coarse, rho_coarse);
  const int sub = lane >> 3, j0 = lane & 7;
  const int n_sel = sel.count();
  bool collide = false;
  for (int k0 = 0; k0 < n_sel && !collide; k0 += 32) {
    const int k = k0 + lane;
    const int o = k < n_sel ? sel.id(k) : -1;
    int st = 0;  // 0: coarse test fails, 1: passes (ball), 3: polygon part still to do
    if (o >= 0 && (ignore_active || P.active[o]) && sel.admit(k)) {
      const double2 c = P.center[o];
      const double d2 = dist2_point_segment_2d(c.x, c.y, sx, sy, ex, ey);  // :1536
      const double rr = __dadd_rn(rho_coarse, P.radius[o]);
      if (!(d2 > __dmul_rn(rr, rr))) {  // :1537-1539
        const int kind = P.kind[o];
        if (kind == 1) st = 1;
        else if (kind == 3 && P.vptr[o + 1] - P.vptr[o] >= 2) st = 3;  // :1551-1553
      }
    }
    unsigned pass = __ballot_sync(FULL, st == 1), pend = __ballot_sync(FULL, st == 3);
    while (pend) {  // polygon part of the coarse test, up to 4 obstacles per round
      unsigned mm = pend;
      int ob = -1;
      for (int q = 0; q <= sub && mm; ++q) {
        ob = __ffs(mm) - 1;
        mm &= mm - 1;
        if (q < sub) ob = -1;
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) pend &= pend - 1;  // the 4 lowest candidates are taken (x & (x-1) of 0 is 0)
      bool hit = false;
      const int oo = __shfl_sync(FULL, o, ob >= 0 ? ob : 0);  // obstacle number held by lane `ob` of this trip
      if (ob >= 0) {
        const int64_t v0 = P.vptr[oo], v1 = P.vptr[oo + 1];
        for (int64_t i = v0 + j0; i < v1 && !hit; i += 8) {  // polygon edge (verts[i-1], verts[i]), first one wraps
          const double2 A = P.verts[i == v0 ? v1 - 1 : i - 1], B = P.verts[i];
          hit = segment_dist2_2d(sx, sy, ex, ey, A.x, A.y, B.x, B.y) < rc2;
        }
      }
      const unsigned hm = __ballot_sync(FULL, hit);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int obq = __shfl_sync(FULL, ob, 8 * q);
        if (obq >= 0 && ((hm >> (8 * q)) & 0xffu)) pass |= 1u << obq;
      }
    }
    while (pass && !collide) {  // obstacles that passed the coarse test: every trajectory segment, 32 per trip
      const int ob = __shfl_sync(FULL, o, __ffs(pass) - 1);
      pass &= pass - 1;
      for (int64_t i0 = t0 + 1; i0 < t1 && !collide; i0 += 32) {  // for i = 2:size(trajectory,1)  :767-771
        const int64_t i = i0 + lane;
        bool hit = false;
        if (i < t1)
          hit = edge_check_2d(P, ob, true, traj[2 * (i - 1)], traj[2 * (i - 1) + 1], traj[2 * i], traj[2 * i + 1], rho);
        collide = __any_sync(FULL, hit);
      }
    }
  }
  return collide;
}

// selector of dubins_collide_warp: every obstacle of the set
struct AllObstacles {
  int n;
  __device__ __forceinline__ int count() const { return n; }
  __device__ __forceinline__ int id(int k) const { return k; }
  __device__ __forceinline__ bool admit(int) const { return true; }
};

}  // namespace rrtqx

struct rrtqx_polygons {
  rrtqx_ctx *ctx = nullptr;
  int64_t n = 0, nv = 0;
  rrtqx::DevBuf<int32_t> kind;
  rrtqx::DevBuf<double2> center, verts;
  rrtqx::DevBuf<double> radius;
  rrtqx::DevBuf<uint8_t> active;
  rrtqx::DevBuf<int64_t> vptr;
  rrtqx::DevBuf<double> s_a, s_b, s_t;
  rrtqx::DevBuf<int64_t> s_ptr;
  rrtqx::DevBuf<uint8_t> s_out;
  rrtqx::PolyView view() const {
    rrtqx::PolyView v;
    v.kind = kind.p; v.center = center.p; v.radius = radius.p; v.active = active.p; v.vptr = vptr.p; v.verts = verts.p;
    v.n = (int)n;
    return v;
  }
};

