// dubins.cuh -- Dubins calculateTrajectory (DRRT_DubinsEdge_functions.jl:329-709, space without time;
// rightTurnDist / leftTurnDist DRRT_distance_functions.jl:62-80) and the DubinsEdge steering point
// (saturate, :70-95) as device functions, shared by the batch kernels (dubins.cu) and the fused Dubins
// extend query (extend_dubins.cuh), so that both run the same code.
//
// solve(): the four turning circles, the six words tried in the reference's order (rsl, rsr, rlr, lsr,
// lsl, lrl) with its strict `bestDist > length` replacement.  word_layout() / word_row(): the
// discretisation of the winning word, arcs sampled every 0.1 rad from the start angle
// (collect(phi_start:+-0.1:phi_end)), a straight part as its two end points.  Row k of an edge depends on
// the layout and k only, so one thread or the lanes of a warp can emit the rows.
//
// Parity: the reference evaluates sin/cos/atan/acos with Julia's libm ports and builds the angle
// ranges in twice-precision arithmetic; this code uses the CUDA double-precision library and
// phi_start + i*0.1.  Results agree to a few ulp, so trajectories and lengths are compared at 1e-9
// relative (SURVEY.md appendix A14); the collision booleans computed FROM a trajectory are bit-exact.
// Library built with -fmad=false: no contraction changes the operation order below.
#pragma once
#include "common.cuh"

namespace rrtqx {

constexpr double DB_PI = 3.141592653589793;  // Julia's Float64(pi)
constexpr double DB_DPHI = 0.1;              // delta_phi, :506

struct P2 {
  double x, y;
};

#ifdef __CUDACC__
__device__ __forceinline__ double len2(P2 a, P2 b) {  // sqrt(sum((a - b).^2))
  const double dx = a.x - b.x, dy = a.y - b.y;
  return sqrt(dx * dx + dy * dy);
}
// arc length from a to b around c turning right / left (DRRT_distance_functions.jl:62-80)
__device__ __forceinline__ double turn_right(P2 a, P2 b, P2 c, double r) {
  double th = atan2(a.y - c.y, a.x - c.x) - atan2(b.y - c.y, b.x - c.x);
  if (th < 0) th = th + 2 * DB_PI;
  return th * r;
}
__device__ __forceinline__ double turn_left(P2 a, P2 b, P2 c, double r) {
  double th = atan2(b.y - c.y, b.x - c.x) - atan2(a.y - c.y, a.x - c.x);
  if (th < 0) th = th + 2 * DB_PI;
  return th * r;
}

// The winning word in a form the emission can walk: three pieces, each either an arc (centre, from,
// to, direction) or the straight segment between the two transition points.
struct Word {
  double dist;
  int type;      // 0 rsl, 1 rsr, 2 rlr, 3 lsr, 4 lsl, 5 lrl, -1 none
  P2 c1, cm, c3; // first / middle / last turning circle
  P2 t1, t2;     // transition points (tangent points, or the circle contact points of a CCC word)
};

__device__ inline Word solve(const double *s4, const double *g4, double r) {
  const P2 il = {s4[0], s4[1]}, gl = {g4[0], g4[1]};
  const double ith = s4[3], gth = g4[3];
  // :346-356  centres of the right / left turning circles at both ends
  const P2 irc = {il.x + r * cos(ith - DB_PI / 2.0), il.y + r * sin(ith - DB_PI / 2.0)};
  const P2 ilc = {il.x + r * cos(ith + DB_PI / 2.0), il.y + r * sin(ith + DB_PI / 2.0)};
  const P2 grc = {gl.x + r * cos(gth - DB_PI / 2.0), gl.y + r * sin(gth - DB_PI / 2.0)};
  const P2 glc = {gl.x + r * cos(gth + DB_PI / 2.0), gl.y + r * sin(gth + DB_PI / 2.0)};
  Word w;
  w.dist = INFINITY;
  w.type = -1;
  w.c1 = w.cm = w.c3 = w.t1 = w.t2 = P2{0.0, 0.0};
  auto offer = [&](double length, int type, P2 c1, P2 cm, P2 c3, P2 t1, P2 t2) {
    if (w.dist > length) {  // strict: the earlier word wins ties
      w.dist = length; w.type = type; w.c1 = c1; w.cm = cm; w.c3 = c3; w.t1 = t1; w.t2 = t2;
    }
  };
  // inner tangents between a first circle A and a last circle B (rsl: sign = -1, lsr: sign = +1)
  auto inner = [&](P2 A, P2 B, double sign, P2 &ta, P2 &tb) -> bool {
    const double D = len2(B, A);
    const double vx = (B.x - A.x) / D, vy = (B.y - A.y) / D;
    const double R = sign * 2.0 * r / D;
    if (fabs(R) > 1.0) return false;
    const double sq = sqrt(1.0 - R * R);
    if (sign < 0) {  // :373-377
      const double a = r * (R * vx + vy * sq), b = r * (R * vy - vx * sq);
      ta = P2{A.x - a, A.y - b};
      tb = P2{B.x + a, B.y + b};
    } else {         // :443-447
      const double a = R * vx + vy * sq, b = R * vy - vx * sq;
      ta = P2{A.x + a * r, A.y + b * r};
      tb = P2{B.x - a * r, B.y - b * r};
    }
    return true;
  };
  P2 ta, tb;
  // r-s-l :365-388
  if (inner(irc, glc, -1.0, ta, tb))
    offer(turn_right(il, ta, irc, r) + len2(tb, ta) + turn_left(tb, gl, glc, r), 0, irc, irc, glc, ta, tb);
  // r-s-r :394-409 and r-l-r :413-433 (same centre line)
  {
    const double D = len2(grc, irc);
    const double vx = (grc.x - irc.x) / D, vy = (grc.y - irc.y) / D;
    ta = P2{-r * vy + irc.x, r * vx + irc.y};
    tb = P2{-r * vy + grc.x, r * vx + grc.y};
    offer(turn_right(il, ta, irc, r) + len2(tb, ta) + turn_right(tb, gl, grc, r), 1, irc, irc, grc, ta, tb);
    if (D < 4.0 * r) {
      const double th = -acos(D / (4 * r)) + atan2(vy, vx);
      const P2 cm = {irc.x + 2 * r * cos(th), irc.y + 2 * r * sin(th)};
      ta = P2{(cm.x + irc.x) / 2.0, (cm.y + irc.y) / 2.0};
      tb = P2{(cm.x + grc.x) / 2.0, (cm.y + grc.y) / 2.0};
      offer(turn_right(il, ta, irc, r) + turn_left(ta, tb, cm, r) + turn_right(tb, gl, grc, r), 2, irc, cm, grc, ta, tb);
    }
  }
  // l-s-r :436-460
  if (inner(ilc, grc, 1.0, ta, tb))
    offer(turn_left(il, ta, ilc, r) + len2(tb, ta) + turn_right(tb, gl, grc, r), 3, ilc, ilc, grc, ta, tb);
  // l-s-l :463-478 and l-r-l :481-499
  {
    const double D = len2(glc, ilc);
    const double vx = (glc.x - ilc.x) / D, vy = (glc.y - ilc.y) / D;
    ta = P2{r * vy + ilc.x, -r * vx + ilc.y};
    tb = P2{r * vy + glc.x, -r * vx + glc.y};
    offer(turn_left(il, ta, ilc, r) + len2(tb, ta) + turn_left(tb, gl, glc, r), 4, ilc, ilc, glc, ta, tb);
    if (D < 4.0 * r) {
      const double th = acos(D / (4 * r)) + atan2(vy, vx);
      const P2 cm = {ilc.x + 2.0 * r * cos(th), ilc.y + 2.0 * r * sin(th)};
      ta = P2{(cm.x + ilc.x) / 2.0, (cm.y + ilc.y) / 2.0};
      tb = P2{(cm.x + glc.x) / 2.0, (cm.y + glc.y) / 2.0};
      offer(turn_left(il, ta, ilc, r) + turn_right(ta, tb, cm, r) + turn_left(tb, gl, glc, r), 5, ilc, cm, glc, ta, tb);
    }
  }
  return w;
}

// one arc piece: rows centre + r [cos(phi) sin(phi)], phi = phi_start, phi_start +- 0.1, ... up to phi_end
// (a single row when the two angles coincide)
struct Arc {
  P2 c;
  double ps, step;
  int rows;
};

__device__ __forceinline__ Arc arc_piece(P2 c, P2 from, P2 to, bool right) {
  Arc a;
  a.c = c;
  a.ps = atan2(from.y - c.y, from.x - c.x);
  double pe = atan2(to.y - c.y, to.x - c.x);
  if (right) {
    if (pe > a.ps) pe = pe - 2.0 * DB_PI;
    a.step = -DB_DPHI;
  } else {
    if (pe < a.ps) pe = pe + 2.0 * DB_PI;
    a.step = DB_DPHI;
  }
  a.rows = 1;
  if (pe != a.ps) {
    const double q = (pe - a.ps) / a.step;
    a.rows = q >= 0.0 ? (int)floor(q) + 1 : 0;
  }
  return a;
}

__device__ __forceinline__ double2 arc_point(const Arc &a, double r, int i) {
  const double phi = a.ps + (double)i * a.step;
  return make_double2(a.c.x + r * cos(phi), a.c.y + r * sin(phi));
}

// Row layout of a word's trajectory: first arc :508-548, then the middle arc of a CCC word or the straight
// part :552-570 (two rows, t1 and t2), then the last arc :606-655.
struct WordRows {
  Arc a1, am, a3;
  P2 t1, t2;
  int mid_arc;  // 1: CCC word (rlr / lrl), 0: straight middle part
  int total;
};

__device__ inline WordRows word_layout(const Word &w, const double *s4, const double *g4) {
  WordRows L;
  L.total = 0;
  L.mid_arc = 0;
  L.t1 = w.t1;
  L.t2 = w.t2;
  if (w.type < 0) {
    L.a1 = L.am = L.a3 = Arc{P2{0.0, 0.0}, 0.0, 0.0, 0};
    return L;
  }
  const bool first_right = w.type <= 2;                       // r**: 0,1,2
  const bool last_right = w.type == 1 || w.type == 2 || w.type == 3;  // **r: rsr, rlr, lsr
  const P2 il = {s4[0], s4[1]}, gl = {g4[0], g4[1]};
  L.a1 = arc_piece(w.c1, il, w.t1, first_right);
  if (w.type == 2 || w.type == 5) {                           // rlr: middle left turn, lrl: middle right turn
    L.am = arc_piece(w.cm, w.t1, w.t2, w.type == 5);
    L.mid_arc = 1;
  } else {
    L.am = Arc{P2{0.0, 0.0}, 0.0, 0.0, 2};
  }
  L.a3 = arc_piece(w.c3, w.t2, gl, last_right);
  L.total = L.a1.rows + L.am.rows + L.a3.rows;
  return L;
}

// row k (0 <= k < L.total) of the trajectory
__device__ __forceinline__ double2 word_row(const WordRows &L, double r, int k) {
  if (k < L.a1.rows) return arc_point(L.a1, r, k);
  k -= L.a1.rows;
  if (k < L.am.rows) {
    if (L.mid_arc) return arc_point(L.am, r, k);
    return k == 0 ? make_double2(L.t1.x, L.t1.y) : make_double2(L.t2.x, L.t2.y);
  }
  return arc_point(L.a3, r, k - L.am.rows);
}

// number of trajectory rows of the word; EMIT = true also writes them to out[0 ..)
template <bool EMIT>
__device__ inline int word_rows(const Word &w, const double *s4, const double *g4, double r, double2 *out) {
  const WordRows L = word_layout(w, s4, g4);
  if (EMIT)
    for (int k = 0; k < L.total; ++k) out[k] = word_row(L, r, k);
  return L.total;
}

// saturate, DubinsEdge version (DRRT_DubinsEdge_functions.jl:70-95), in place on p[4]; dist = R3SDist
// (:41 of the distance functions)
__device__ inline void dubins_saturate_point(double *p, const double *c, double delta) {
  // R3SDist: sqrt(sum((x[1:3]-y[1:3]).^2) + min(|x4-y4|, min(x4,y4) + 2pi - max(x4,y4))^2)
  const double dx = __dsub_rn(p[0], c[0]), dy = __dsub_rn(p[1], c[1]), dz = __dsub_rn(p[2], c[2]);
  const double a = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  const double w = jl_min(fabs(__dsub_rn(p[3], c[3])),
                          __dsub_rn(__dadd_rn(jl_min(p[3], c[3]), 6.283185307179586), jl_max(p[3], c[3])));
  const double d = __dsqrt_rn(__dadd_rn(a, __dmul_rn(w, w)));
  if (d > delta) {
    for (int k = 0; k < 3; ++k) p[k] = __dadd_rn(c[k], __ddiv_rn(__dmul_rn(__dsub_rn(p[k], c[k]), delta), d));
    if (fabs(__dsub_rn(p[3], c[3])) < DB_PI) {
      p[3] = __dadd_rn(c[3], __ddiv_rn(__dmul_rn(__dsub_rn(p[3], c[3]), delta), d));
    } else {
      p[3] = p[3] < DB_PI ? __dadd_rn(p[3], 2 * DB_PI) : __dsub_rn(p[3], 2 * DB_PI);
      p[3] = __dadd_rn(c[3], __ddiv_rn(__dmul_rn(__dsub_rn(p[3], c[3]), delta), d));
      p[3] = jl_max(jl_min(p[3], 2 * DB_PI), 0.0);
    }
  }
}
#endif  // __CUDACC__

}  // namespace rrtqx

// Result of a Dubins trajectory batch (rrtqx_dubins_trajectory_batch) or of the edges of a fused Dubins extend
// query (rrtqx_extend_query_dubins): per edge dist / type, the rows as a CSR (ptr, traj).
struct rrtqx_dubins_result {
  rrtqx_ctx *ctx = nullptr;
  int64_t n_edges = 0, n_rows = 0;
  rrtqx::DevBuf<double> starts, goals, dist;
  rrtqx::DevBuf<int32_t> type, rows, scan_tmp;
  rrtqx::DevBuf<int64_t> ptr, scan_tmp64;
  rrtqx::DevBuf<double2> traj;
};
