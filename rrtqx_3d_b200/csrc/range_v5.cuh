// range_v5.cuh -- single-pass batched kdFindWithinRange, fifth generation (included by range.cu,
// inside namespace rrtqx).
//
// One warp per pair of consecutive (cell-sorted) queries: the candidate rows of the pair are flattened
// into a shared-memory table of octets (start slot, 1..8 points), each 8-lane sub-group takes one octet
// per trip, hits are buffered per query and flushed densely after one atomic reserves the pair's output.
// The previous generation (v4) was instruction-issue bound (profiles/README.md, "what the range kernel is
// bound by": 2450 warp-instructions per query: 1160 in the candidate tests, 620 in the flush, 670 in
// set-up), so v5 removes instructions, not bytes:
//   * the candidate scan runs on an FP32 *filter*: slot records float4((x,y,z) - grid origin, w) are
//     fetched with ONE 128-bit load and both queries of the warp's pair are tested with packed
//     f32x2 arithmetic (sm_100 FADD2/FFMA2: 6 instructions for 2 x 32 tests).  The filter computes
//     s' ~ |q-p|^2 - T with a rigorous error bound M (derivation at v5_filter); s' < -M is a certain
//     hit, s' > M a certain miss, and a trip in which any lane lands in the band |s'| <= M is
//     re-decided in exact FP64 from the exact records.  The filter never decides a result on its own
//     unless the decision is provably the one the exact test s < T_lt(r) makes.
//   * the flush reads one 256-bit exact record per hit (x, y, z, node) instead of four gathers,
//     recomputes the reference's radicand in FP64, takes the correctly rounded sqrt with all lanes
//     busy and stores idx / dist coalesced;
//   * per-pair set-up is FP32 where it only culls; the exact FP64 query is reloaded where needed
//     instead of being kept in registers across the scan;
//   * rare cases (FP32 unusable for a query, hit-buffer overflow) go through one out-of-line exact
//     routine, so they cost no registers in the hot path.

constexpr int V5_TABPAD = 16;  // zero entries behind the last one (a trip group never tests bounds)
constexpr int V5_UNIT = 128;    // pairs per dynamically scheduled unit of work (a block's warps share one unit; C2 kernel time at 48 / 64 / 96 / 128 / 160 / 256 pairs: 2.78 / 2.69 / 2.70 / 2.665 / 2.664 / 2.70 ms)
constexpr int V5_RING = 64;     // published unit bases kept per block
constexpr int V5_U = 4;         // trips per loop iteration (loads in flight before the first test)

__device__ __forceinline__ void sts32(unsigned addr, int v) {
  asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ int lds32(unsigned addr) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
// keeps a value in a register (stops the compiler from re-deriving it from
// special registers inside the hot loop)
__device__ __forceinline__ unsigned pin_reg(unsigned v) {
  unsigned r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}
__device__ __forceinline__ unsigned long long pk2(float a, float b) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void upk2(unsigned long long r, float &a, float &b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(r));
}
__device__ __forceinline__ unsigned long long fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ unsigned long long sub2(unsigned long long a, unsigned long long b) {
  unsigned long long r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ void sts16(unsigned addr, unsigned v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ unsigned lds16(unsigned addr) {
  unsigned short v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ double4 ldg256(const double4 *p) {
  double4 v;
  asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
}

// Result stores of the flush.  Kept as calls: the same stores written inline change how the compiler schedules and
// spills range_v5_kernel (other spill counts and stack frames), and the code generated through these calls is the
// one that was measured.
__device__ __forceinline__ void v5_st(int32_t *p, int32_t v) { *p = v; }
__device__ __forceinline__ void v5_st(double *p, double v) { *p = v; }

// double -> float rounded up (host twin: nextafter of the nearest conversion when it fell below)
__host__ __device__ __forceinline__ float f32_up(double x) {
#ifdef __CUDA_ARCH__
  return __double2float_ru(x);
#else
  float f = (float)x;
  if ((double)f < x) f = nextafterf(f, INFINITY);
  return f;
#endif
}

// FP32 filter parameters of one query.
//
// Records hold F_c = fl32(p_c - lo_c) and the query side uses G_c = fl32(q_c - lo_c) (c < 3; the 4th
// coordinate is converted directly).  With u = 2^-24, A = max |record component|, B = max |G_c| and
// e = 1.01 u (A + B), every computed difference d^_c = fl32(G_c - F_c) satisfies
// |d^_c - (q_c - p_c)| <= e + u |q_c - p_c| (two input roundings, one subtraction rounding; 1.01 covers the
// FP64 roundings of p - lo and q - lo).  For S = sum (q_c - p_c)^2 <= 4T and e <= 2^-10 sqrt(T) this gives
// |sum d^_c^2 - S| <= 8.1 sqrt(T) e + 40 u T for up to four coordinates, the four FMA roundings add at most
// 4 u (S + T) <= 20.1 u T and |fl32(T) - T| <= u T, so the computed s' = sum d^_c^2 - fl32(T) is within
//   M = 12 sqrt(T) e + 64 u T
// of S - T; for S > 4T the same bounds give s' >= 2.9 T > M.  The reference's radicand differs from S by
// less than 2^-50 S, far inside M.  Hence s' < -M  =>  exact hit, s' > M  =>  exact miss.
// The filter is declared unusable (exact = true) when e > 2^-10 sqrt(T), when T is outside
// [1e-30, 1e30] (FP32 under/overflow of the squares) or when anything is not finite.
__host__ __device__ __forceinline__ void v5_filter(double T, float maxabs_sum, float &Tm, float &M, bool &exact) {
  const float e = maxabs_sum * 6.03e-8f;  // 1.01 * 2^-24 = 6.0201e-8
  const float Tf = f32_up(T);
  const float sT = sqrtf(Tf);
  Tm = (float)T;
  M = 12.0f * (sT * 1.000001f) * e + 3.9e-6f * Tf;  // 64 u = 3.8147e-6
  exact = !(e * 1024.0f <= sT * 0.999999f) || !(Tf < 1e30f) || !(Tf > 1e-30f);
}

// Exact (FP64 only) evaluation of one query by the whole warp: the same rows, exact records, test
// s < T.  WRITE = false returns the number of hits; WRITE = true writes idx/dist at base.  Used when the
// FP32 filter is unusable for a query and when a query overflowed its hit buffer.
template <int D, bool WRITE>
__device__ __noinline__ int v5_exact_query(const GridView *gp, const double *qptr, double T, double r, int64_t base,
                                           int32_t *__restrict__ out_idx, double *__restrict__ out_dist) {
  const GridView &g = *gp;
  const int lane = lane_id();
  const unsigned lt = lanemask_lt();
  double q[D];
#pragma unroll
  for (int c = 0; c < D; ++c) q[c] = qptr[c];
  int cnt = 0;
  auto visit = [&](bool valid, int node, double px, double py, double pz, double pw) {
    const double s = sqdist<D>(q, px, py, pz, pw);
    const bool hit = valid && (s < T);
    const unsigned m = __ballot_sync(FULL, hit);
    if (WRITE && hit) {
      const int64_t o = base + cnt + __popc(m & lt);
      out_idx[o] = node;
      if (out_dist) out_dist[o] = __dsqrt_rn(s);
    }
    cnt += __popc(m);
  };
  if (g.n_sorted > 0 && r > 0.0) {
    const double r_infl = r * (1.0 + 1e-9);
    const double r2_infl = r_infl * r_infl;
    const int cy0 = cell_of(q[1] - r_infl, g.lo[1], g.inv[1], g.ny);
    const int cy1 = cell_of(q[1] + r_infl, g.lo[1], g.inv[1], g.ny);
    const int cz0 = D >= 3 ? cell_of(q[2] - r_infl, g.lo[2], g.inv[2], g.nz) : 0;
    const int cz1 = D >= 3 ? cell_of(q[2] + r_infl, g.lo[2], g.inv[2], g.nz) : 0;
    const int wy = cy1 - cy0 + 1;
    const int nrows = wy * (cz1 - cz0 + 1);
    for (int rb = 0; rb < nrows; rb += 32) {
      RowSpan sp{0, 0};
      const int row = rb + lane;
      if (row < nrows) sp = row_span<D>(g, q, r2_infl, cy0 + row % wy, cz0 + row / wy);
      const int lim = min(32, nrows - rb);
      for (int t = 0; t < lim; ++t) {
        const int a = __shfl_sync(FULL, sp.start, t);
        const int b = __shfl_sync(FULL, sp.end, t);
        for (int j0 = a; j0 < b; j0 += 32) {
          const int j = j0 + lane;
          const bool v = j < b;
          double4 p = make_double4(0, 0, 0, 0);
          int node = 0;
          if (v) {
            p = g.d4[j];
            node = D <= 3 ? (int)__double_as_longlong(p.w) : g.sperm[j];
          }
          visit(v, node, p.x, p.y, p.z, p.w);
        }
      }
    }
  }
  if (r > 0.0)
    for (int j0 = g.n_sorted; j0 < g.n_total; j0 += 32) {  // unsorted tail of recent inserts
      const int j = j0 + lane;
      const bool v = j < g.n_total;
      double4 p = make_double4(0, 0, 0, 0);
      if (v) p = g.pos[j];
      visit(v, j, p.x, p.y, p.z, p.w);
    }
  return cnt;
}

// Dense flush of one query's buffered hits.  A hit is a 16-bit code: (octet-table entry << 3) | lane-in-octet,
// or 0x8000 | (node - n_sorted) for a node of the unsorted tail; the slot is recovered through the table.
template <int D, bool TAIL>
__device__ __forceinline__ void v5_flush(const GridView &g, const double *q, unsigned sbuf_k, unsigned stab, int n, int lane,
                                         int32_t *__restrict__ oi, double *__restrict__ od) {
  constexpr int U = 4;  // rows of 32 hits in flight per flush step
  auto fetch = [&](unsigned h, int &node, double4 &p) {
    if (!TAIL || !(h & 0x8000u)) {
      const int ent = lds32(stab + 4u * (h >> 3));
      const int slot = (ent >> 4) + (int)(h & 7u);
      p = ldg256(g.d4 + slot);
      node = D <= 3 ? (int)__double_as_longlong(p.w) : g.sperm[slot];
    } else {
      node = g.n_sorted + (int)(h & 0x7fffu);
      p = g.pos[node];
    }
  };
  const int n_full = (n / (32 * U)) * (32 * U);
  for (int h0 = lane; h0 < n_full; h0 += 32 * U) {  // full groups of U x 32 hits: no predicates
    int node[U];
    double4 p[U];
#pragma unroll
    for (int u = 0; u < U; ++u) fetch(lds16(sbuf_k + 2u * (unsigned)(h0 + 32 * u)), node[u], p[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      v5_st(oi + h0 + 32 * u, node[u]);
      if (od) v5_st(od + h0 + 32 * u, __dsqrt_rn(sqdist<D>(q, p[u].x, p[u].y, p[u].z, p[u].w)));
    }
  }
  // last, partial group: same shape (all loads in flight before the first use), predicated, and only as many rows
  // as the remainder needs (1, 2 or 4): a short list does not pay for four rows of FP64 work
  auto tail = [&](auto rows_tag) {
    constexpr int R = decltype(rows_tag)::value;
    const int h0 = n_full + lane;
    int node[R];
    double4 p[R];
#pragma unroll
    for (int u = 0; u < R; ++u) {
      // lanes past the end re-read hit 0 (always present here): no predicated loads, only predicated stores
      const int hh = h0 + 32 * u < n ? h0 + 32 * u : 0;
      fetch(lds16(sbuf_k + 2u * (unsigned)hh), node[u], p[u]);
    }
#pragma unroll
    for (int u = 0; u < R; ++u)
      if (h0 + 32 * u < n) {
        v5_st(oi + h0 + 32 * u, node[u]);
        if (od) v5_st(od + h0 + 32 * u, __dsqrt_rn(sqdist<D>(q, p[u].x, p[u].y, p[u].z, p[u].w)));
      }
  };
  const int rem = n - n_full;
  if (rem > 64) tail(std::integral_constant<int, 4>{});
  else if (rem > 32) tail(std::integral_constant<int, 2>{});
  else if (rem > 0) tail(std::integral_constant<int, 1>{});
}

// Trees with an unsorted tail (planner inserts since the last re-index) flush through an out-of-line copy, so the
// hot path carries one flush body only.
template <int D>
__device__ __noinline__ void v5_flush_tail(const GridView *gp, const double *qs, unsigned sbuf_k, unsigned stab, int n,
                                           int32_t *__restrict__ oi, double *__restrict__ od) {
  double q[D];
#pragma unroll
  for (int c = 0; c < D; ++c) q[c] = qs[c];
  v5_flush<D, true>(*gp, q, sbuf_k, stab, n, lane_id(), oi, od);
}

// Radius-dependent constants of the FP32 culling and filter (hoisted out of the pair loop when the
// batch has one radius).
struct V5Radius {
  float rf, r2f;     // inflated r, r^2 (round up)
  float Tm;          // fl32(T); -inf for a dead query (s' = +inf: never a hit, never in the band)
  float cM1, cM0;    // M = cM1 * (A + B) + cM0
  float sum_max;     // filter usable iff (A + B) <= sum_max
  bool live;
};
__host__ __device__ __forceinline__ V5Radius v5_radius(double r, double T, bool have) {
  V5Radius R;
  R.live = have && (r > 0.0);
  const double ri = r * (1.0 + 1e-9);
  R.rf = f32_up(ri) * (1.0f + 1e-6f);
  R.r2f = f32_up(ri * ri) * (1.0f + 1e-5f);
  float Tm, M;
  bool ex;
  v5_filter(T, 0.0f, Tm, M, ex);  // M at zero coordinate error = 64 u T
  const float Tf = f32_up(T), sT = sqrtf(Tf);
  R.Tm = Tm;
  R.cM0 = M;
  R.cM1 = 12.0f * (sT * 1.000001f) * 6.03e-8f * 1.000001f;
  // e * 1024 <= sT * 0.999999  <=>  sum <= sT * 0.999999 / (1024 * 6.03e-8)
  R.sum_max = ex ? -1.0f : sT * 0.999999f * (1.0f / (1024.0f * 6.03e-8f)) * 0.99999f;
  if (!R.live) { R.Tm = -INFINITY; R.r2f = -1.0f; R.cM0 = 0.0f; R.cM1 = 0.0f; R.sum_max = INFINITY; }
  return R;
}

// launch constants kept in the constant bank (no registers): uniform-radius parameters and FP32 grid scales
struct V5Params {
  V5Radius RU;
  float invx, invy, invz, celly, cellz;
  unsigned unit;  // pairs per dynamically scheduled unit of work
  int ghost_pairs;  // 1: query 2j+1 is the ghost identity of query 2j (wrap-around trees): no root `<=` rule for it
};

// floor + clamp to [0, n-1] through the integer converter (F2I.FLOOR saturates, NaN -> 0): 3 instructions
__device__ __forceinline__ int clampi_fast(float v, int n) { return min(max(__float2int_rd(v), 0), n - 1); }

__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <int D, int NW, int CAP, int TAB, bool UNIFORM>
__global__ void __launch_bounds__(NW * 32, 1)
range_v5_kernel(GridView g_param, V5Params P, const double *__restrict__ queries, const double *__restrict__ qsorted,
                const int32_t *__restrict__ qorder, int64_t nq, double r_uniform, double T_uniform,
                const double *__restrict__ ranges, const double *__restrict__ Tq, int32_t *__restrict__ counts,
                int64_t *__restrict__ offsets, int32_t *__restrict__ out_idx, double *__restrict__ out_dist,
                unsigned long long cap, unsigned long long *__restrict__ cursor, int write_lists) {
  extern __shared__ int s_buf[];  // [NW][2][CAP] 16-bit hit codes, then [NW][TAB + V5_TABPAD] octet tables
  __shared__ GridView s_g;        // for the out-of-line exact routine
  // barrier-free dynamic work distribution (see the ticket loop below)
  __shared__ unsigned s_ticket;
  __shared__ unsigned s_pub[V5_RING];
  __shared__ long long s_base[V5_RING];
  const GridView &g = g_param;
  if (threadIdx.x == 0) { s_g = g_param; s_ticket = 0; }
  if (threadIdx.x < V5_RING) s_pub[threadIdx.x] = 0;
  __syncthreads();
  const int lane = lane_id(), warp = threadIdx.x >> 5;
  const unsigned lt = lanemask_lt();
  const unsigned s0 = (unsigned)__cvta_generic_to_shared(s_buf);
  const unsigned sbuf = pin_reg(s0 + 2u * (unsigned)(warp * 2 * CAP));
  const unsigned stab = pin_reg(s0 + 2u * (unsigned)(NW * 2 * CAP) + 4u * (unsigned)(warp * (TAB + V5_TABPAD)));
  const float &invx = P.invx, &invy = P.invy, &invz = P.invz, &celly = P.celly, &cellz = P.cellz;
  const float fmaxabs = g.n_sorted > 0 ? *g.fmaxabs : 0.0f;
  const bool has_tail = g.n_total > g.n_sorted;
  const unsigned grp = pin_reg((unsigned)lane >> 3), sub = pin_reg((unsigned)lane & 7u);
  constexpr bool uniform = UNIFORM;

  // Work distribution.  Static striding of chunks over the 148 persistent blocks left the SMs 12 % idle on
  // average (sm__cycles_active avg / max = 0.88: boundary regions are cheaper, and chunk order correlates with
  // position).  Instead: the block draws UNITS of V5_UNIT consecutive (cell-sorted) pairs from a global
  // counter, and its warps draw pairs of the current unit one by one from a shared ticket counter -- no
  // barrier anywhere.  The warp whose ticket opens a unit fetches the unit's base from the global counter and
  // publishes it in a small ring; the other warps of that unit wait for the publication (one global atomic
  // away).  The warps of a block therefore always work on adjacent pairs (L1 locality as before), finish
  // together, and blocks take units until the batch is exhausted.
  const int64_t n_pairs = (nq + 1) >> 1;
  for (;;) {
    {
      unsigned tk = 0;
      if (lane == 0) tk = atomicAdd(&s_ticket, 1u);
      tk = __shfl_sync(FULL, tk, 0);
      const unsigned unit = tk / P.unit, off = tk - unit * P.unit, slot = unit % V5_RING;
      long long base = 0;
      if (lane == 0) {
        if (off == 0) {
          base = (long long)atomicAdd(&cursor[1], (unsigned long long)P.unit);
          s_base[slot] = base;
          __threadfence_block();
          atomicExch(&s_pub[slot], unit + 1u);
        } else {
          while (atomicAdd(&s_pub[slot], 0u) != unit + 1u) __nanosleep(32);
          base = *(volatile long long *)&s_base[slot];
        }
      }
      base = __shfl_sync(FULL, base, 0);
      if (base >= n_pairs) break;                 // batch exhausted (every later unit is beyond the end too)
      const int64_t qfirst = (base + off) * 2;
      if (qfirst >= nq) continue;                 // last, partial unit
      // ------------------------------------------------------------ per-pair set-up
      const bool have1 = qfirst + 1 < nq;
      const int qid0 = qorder[qfirst], qid1 = have1 ? qorder[qfirst + 1] : -1;
      const double *qs0 = qsorted ? qsorted + qfirst * D : queries + (int64_t)qid0 * D;
      const double *qs1 = !have1 ? qs0 : (qsorted ? qs0 + D : queries + (int64_t)qid1 * D);
      // uniform radius: the parameters stay in the constant bank; a missing second query (odd batch) is
      // scanned as a copy of the first and its results are dropped
      V5Radius Rq0, Rq1;
      if (!uniform) {
        Rq0 = v5_radius(ranges[qid0], Tq[qid0], true);
        Rq1 = have1 ? v5_radius(ranges[qid1], Tq[qid1], true) : Rq0;
      }
      const V5Radius &R0 = uniform ? P.RU : Rq0, &R1 = uniform ? P.RU : Rq1;
      // FP32 view of a query: coordinates relative to the grid origin and max |component|.  Recomputed per
      // phase from the (L1-resident) query instead of being carried in registers.
      auto fp32_query = [&](const double *qs, float (&qf)[4], float &mab) {
        mab = 0.0f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c < D) {
            const double v = qs[c];
            qf[c] = __double2float_rn(c < 3 ? __dsub_rn(v, g.lo[c < 3 ? c : 0]) : v);
            mab = fmaxf(mab, fabsf(qf[c]));  // fmaxf drops NaN; a NaN coordinate is flagged below
          } else {
            qf[c] = 0.0f;
          }
        }
        // a NaN coordinate: the query can never hit (NaN < T is false in FP32 and FP64 alike), so it needs no
        // rows and no exact path; flagged by mab = -1.  (Unused ghost identities of wrap-around trees arrive so.)
#pragma unroll
        for (int c = 0; c < D; ++c) if (qf[c] != qf[c]) mab = -1.0f;
      };
      // exact thresholds / radii for the rare exact paths (re-read, not kept in registers)
      auto exactT = [&](int k) { return uniform ? T_uniform : ((k == 0 || !have1) ? Tq[qid0] : Tq[qid1]); };
      auto exactR = [&](int k) { return uniform ? r_uniform : ((k == 0 || !have1) ? ranges[qid0] : ranges[qid1]); };

      int root_extra = 0;  // bit k: the root sits exactly at distance r of query k
      {
        // the root (node 0) is admitted with <= (kdTree_general.jl:896-898): it needs an explicit entry only
        // when it sits exactly at distance r; the sqrt is evaluated only in a 1e-6 band above T
        const double4 p0 = g.pos[0];
        double q0[D], q1[D];
#pragma unroll
        for (int c = 0; c < D; ++c) { q0[c] = qs0[c]; q1[c] = qs1[c]; }
        const double T0 = exactT(0), T1 = exactT(1);
        const double sr0 = sqdist<D>(q0, p0.x, p0.y, p0.z, p0.w), sr1 = sqdist<D>(q1, p0.x, p0.y, p0.z, p0.w);
        if (!(sr0 < T0) && sr0 <= T0 * 1.000001 && __dsqrt_rn(sr0) <= exactR(0)) root_extra |= 1;
        if (have1 && !P.ghost_pairs && !(sr1 < T1) && sr1 <= T1 * 1.000001 && __dsqrt_rn(sr1) <= exactR(1)) root_extra |= 2;
      }
      const bool live0 = R0.live, live1 = R1.live;
      bool exact_path = false;  // FP32 filter unusable, or the octet table overflowed
      int n_ent = 0;            // octets in the table
      // ---------------------------------------------------------------- phase B: rows -> octet table
      if (live0 || live1) {
        float qf0[4], qf1[4], mab0, mab1;
        fp32_query(qs0, qf0, mab0);
        fp32_query(qs1, qf1, mab1);
        const bool rows0 = live0 && !(mab0 < 0.0f), rows1 = live1 && !(mab1 < 0.0f);
        exact_path = (rows0 && !(fmaxabs + mab0 <= R0.sum_max)) || (rows1 && !(fmaxabs + mab1 <= R1.sum_max));
        if (!exact_path && g.n_sorted > 0 && (rows0 || rows1)) {
          // cell coordinates (FP32; relative error 2^-23 per operation, nx <= 1024: far inside the 1e-3 cell slack)
          float ff0[3], ff1[3];
          ff0[0] = qf0[0] * invx; ff0[1] = qf0[1] * invy; ff0[2] = D >= 3 ? qf0[2] * invz : 0.0f;
          ff1[0] = qf1[0] * invx; ff1[1] = qf1[1] * invy; ff1[2] = D >= 3 ? qf1[2] * invz : 0.0f;
          // union of the two queries' row ranges; lanes <-> rows through a power-of-two row stride
          const float ry0 = R0.rf * invy + 1e-3f, ry1 = R1.rf * invy + 1e-3f;
          const float rz0 = R0.rf * invz + 1e-3f, rz1 = R1.rf * invz + 1e-3f;
          int cy0 = 0x7fffffff, cy1 = -1, cz0 = 0, cz1 = 0;
          if (D >= 3) { cz0 = 0x7fffffff; cz1 = -1; }
          if (rows0) {
            cy0 = clampi_fast(ff0[1] - ry0, g.ny); cy1 = clampi_fast(ff0[1] + ry0, g.ny);
            if (D >= 3) { cz0 = clampi_fast(ff0[2] - rz0, g.nz); cz1 = clampi_fast(ff0[2] + rz0, g.nz); }
          }
          if (rows1) {
            cy0 = min(cy0, clampi_fast(ff1[1] - ry1, g.ny)); cy1 = max(cy1, clampi_fast(ff1[1] + ry1, g.ny));
            if (D >= 3) { cz0 = min(cz0, clampi_fast(ff1[2] - rz1, g.nz)); cz1 = max(cz1, clampi_fast(ff1[2] + rz1, g.nz)); }
          }
          const int wy = cy1 - cy0 + 1;
          const int sh = 32 - __clz(wy - 1);  // wy = 1 -> 0
          const int nslots = (cz1 - cz0 + 1) << sh;
          for (int rb = 0; rb < nslots; rb += 32) {
            int sa_ = 0, sb_ = 0;
            const int slot = rb + lane;
            const int ry = slot & ((1 << sh) - 1);
            if (slot < nslots && ry < wy) {
              const int cy = cy0 + ry, cz = cz0 + (slot >> sh);
              // lower bounds of |p.y - q.y|, |p.z - q.z| in cell units; boundary rows also hold the points
              // clamped in from beyond the grid, so they give no bound on that side.  Slack: 1e-6 relative +
              // 1e-3 cells covers the FP32 error of ff and the FP64 rounding of cell_of().
              const float ylo = cy == 0 ? -INFINITY : (float)cy, yhi = cy == g.ny - 1 ? INFINITY : (float)(cy + 1);
              const float zlo = cz == 0 ? -INFINITY : (float)cz, zhi = cz == g.nz - 1 ? INFINITY : (float)(cz + 1);
              int ca = 0x7fffffff, cb = -1;
              auto span = [&](const float *ff, float r2f) {
                float dy = fmaxf(fmaxf(ylo - ff[1], ff[1] - yhi) * (1.0f - 1e-6f) - 1e-3f, 0.0f) * celly;
                float rem = r2f - dy * dy;
                if (D >= 3) {
                  float dz = fmaxf(fmaxf(zlo - ff[2], ff[2] - zhi) * (1.0f - 1e-6f) - 1e-3f, 0.0f) * cellz;
                  rem -= dz * dz;
                }
                if (rem >= 0.0f) {
                  // sqrt.approx: 2 ulp, inside the 1e-5 inflation; an infinite r2f gives the whole row
                  const float xc = sqrt_approx(rem) * (1.0f + 1e-5f) * invx + 1e-3f;
                  ca = min(ca, clampi_fast(ff[0] - xc, g.nx));
                  cb = max(cb, clampi_fast(ff[0] + xc, g.nx));
                }
              };
              if (rows0) span(ff0, R0.r2f);
              if (rows1) span(ff1, R1.r2f);
              if (cb >= ca) {
                const int rbase = (cz * g.ny + cy) * g.nx;
                sa_ = g.cell_start[rbase + ca];
                sb_ = g.cell_start[rbase + cb + 1];
              }
            }
            // append this batch's octets to the table
            const int todo = (sb_ - sa_ + 7) >> 3;
            int incl = todo;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const int t = __shfl_up_sync(FULL, incl, o);
              if (lane >= o) incl += t;
            }
            const int sum = __shfl_sync(FULL, incl, 31);
            if (n_ent + sum > TAB) {  // region too large for the table: exact routine (rare, large-K variants exist)
              exact_path = true;
              break;
            }
            unsigned ta = stab + 4u * (unsigned)(n_ent + incl - todo);
            for (int i = 0; i < todo; ++i) {
              sts32(ta, (sa_ << 4) | min(8, sb_ - sa_));
              ta += 4u;
              sa_ += 8;
            }
            n_ent += sum;
          }
        }
      }
      int cnt0 = 0, cnt1 = 0;
      bool overflow = false;
      if (exact_path) {
        // exact count now, exact write after the allocation
        cnt0 = live0 ? v5_exact_query<D, false>(&s_g, qs0, exactT(0), exactR(0), 0, nullptr, nullptr) : 0;
        cnt1 = (live1 && have1) ? v5_exact_query<D, false>(&s_g, qs1, exactT(1), exactR(1), 0, nullptr, nullptr) : 0;
        overflow = true;
      } else if (live0 || live1) {
        // ---------------------------------------------------------- phase C: FP32 filter scan of the table
        float qf0[4], qf1[4], mab0, mab1;
        fp32_query(qs0, qf0, mab0);
        fp32_query(qs1, qf1, mab1);
        const unsigned long long qx2 = pk2(qf0[0], qf1[0]), qy2 = pk2(qf0[1], qf1[1]);
        const unsigned long long qz2 = pk2(qf0[2], qf1[2]), qw2 = pk2(qf0[3], qf1[3]);
        const unsigned long long nT2 = pk2(-R0.Tm, -R1.Tm);
        const float M = fmaxf(R0.cM1 * (fmaxabs + mab0) + R0.cM0, R1.cM1 * (fmaxabs + mab1) + R1.cM0) * 1.000001f;
        unsigned wp0 = sbuf, wp1 = sbuf + 2u * CAP;  // write pointers (bytes) into the two hit buffers
        const unsigned lim0 = sbuf + 2u * (CAP - 32 * V5_U), lim1 = sbuf + 2u * (2 * CAP - 32 * V5_U);

        // one group: V5_U trips of 32 candidate lanes (4 octets each) against both queries
        const unsigned goff = 4u * grp;
        const unsigned hv0 = (grp << 3) | sub;
        // The table walk is software-pipelined: the records of group i+1 are requested before the tests of
        // group i, so a warp always has V5_U 128-bit loads in flight while it computes.
        int jj[V5_U];
        float4 c[V5_U];
        const int dummy = g.n_sorted + 7;  // padding record of +inf coordinates: s' = +inf (miss, outside the band)
        auto load_group = [&](unsigned tb) {
          const unsigned taddr = tb + goff;
#pragma unroll
          for (int u = 0; u < V5_U; ++u) {
            const int ent = lds32(taddr + 16u * u);
            jj[u] = sub < (unsigned)(ent & 15) ? (ent >> 4) + (int)sub : dummy;  // lanes past the octet's end
          }
#pragma unroll
          for (int u = 0; u < V5_U; ++u) {
            c[u] = g.f4[jj[u]];
          }
        };
        auto test_group = [&](auto store_tag, unsigned tb, bool more) {
          constexpr bool STORE = decltype(store_tag)::value;
          const unsigned hv = hv0 + ((tb - stab) << 1);  // (entry index << 3) | lane-in-octet of trip 0
          float sa[V5_U], sb[V5_U];
          int jc[V5_U];
          float band = INFINITY;  // min |s'| over the group's tests of this lane
#pragma unroll
          for (int u = 0; u < V5_U; ++u) {
            unsigned long long s2 = sub2(qx2, pk2(c[u].x, c[u].x));
            s2 = fma2(s2, s2, nT2);
            unsigned long long d2 = sub2(qy2, pk2(c[u].y, c[u].y));
            s2 = fma2(d2, d2, s2);
            if (D >= 3) { d2 = sub2(qz2, pk2(c[u].z, c[u].z)); s2 = fma2(d2, d2, s2); }
            if (D >= 4) { d2 = sub2(qw2, pk2(c[u].w, c[u].w)); s2 = fma2(d2, d2, s2); }
            upk2(s2, sa[u], sb[u]);
            band = fminf(band, fminf(fabsf(sa[u]), fabsf(sb[u])));
            jc[u] = jj[u];
          }
          if (more) load_group(tb + 4u * 4 * V5_U);  // next group's records: in flight during the compaction
          if (__any_sync(FULL, band <= M)) {
            // some test of the group fell inside the error band of the filter: decide the whole group in
            // exact FP64 from the exact records (the decision is encoded as s' = -inf / +inf)
            double qa[D], qb[D];
#pragma unroll
            for (int cc = 0; cc < D; ++cc) { qa[cc] = qs0[cc]; qb[cc] = qs1[cc]; }
            const double Ta = exactT(0), Tb = exactT(1);
#pragma unroll
            for (int u = 0; u < V5_U; ++u) {
              if (sa[u] < INFINITY || sb[u] < INFINITY) {  // valid lane (an overflowed s' = +inf is a miss either way)
                const double4 p = g.d4[jc[u]];
                sa[u] = (live0 && sqdist<D>(qa, p.x, p.y, p.z, p.w) < Ta) ? -INFINITY : INFINITY;
                sb[u] = (live1 && sqdist<D>(qb, p.x, p.y, p.z, p.w) < Tb) ? -INFINITY : INFINITY;
              }
            }
          }
#pragma unroll
          for (int u = 0; u < V5_U; ++u) {
            const bool h0 = sa[u] < M;
            const unsigned m0 = __ballot_sync(FULL, h0);
            if (STORE && h0) sts16(wp0 + 2u * __popc(m0 & lt), hv + 32u * u);
            wp0 += 2u * __popc(m0);
            const bool h1 = sb[u] < M;
            const unsigned m1 = __ballot_sync(FULL, h1);
            if (STORE && h1) sts16(wp1 + 2u * __popc(m1 & lt), hv + 32u * u);
            wp1 += 2u * __popc(m1);
          }
        };
        if (n_ent > 0) {
          // zero entries behind the last one: groups never test bounds, and the pipelined load of the group
          // behind the last one reads zeros (slot 0: harmless)
          if (lane < V5_TABPAD) sts32(stab + 4u * (unsigned)(n_ent + lane), 0);
          __syncwarp();
          unsigned tb = stab;  // warp-uniform table cursor
          const unsigned tend = stab + 4u * (unsigned)n_ent;
          load_group(tb);
          while (tb < tend && wp0 <= lim0 && wp1 <= lim1) {
            const unsigned nb = tb + 4u * 4 * V5_U;
            test_group(std::true_type{}, tb, nb < tend);
            tb = nb;
          }
          if (tb < tend) {  // a buffer is nearly full: keep counting, re-scan exactly afterwards
            overflow = true;
            do {
              const unsigned nb = tb + 4u * 4 * V5_U;
              test_group(std::false_type{}, tb, nb < tend);
              tb = nb;
            } while (tb < tend);
          }
          __syncwarp();
        }
        if (has_tail && g.n_total - g.n_sorted > 0x8000) overflow = true;  // tail codes are 15 bits: exact routine
        if (has_tail) {  // unsorted tail of recent inserts: exact test, hit code 0x8000 | (node - n_sorted)
          double qa[D], qb[D];
#pragma unroll
          for (int cc = 0; cc < D; ++cc) { qa[cc] = qs0[cc]; qb[cc] = qs1[cc]; }
          const double Ta = exactT(0), Tb = exactT(1);
          for (int j0 = g.n_sorted; j0 < g.n_total; j0 += 32) {
            const int j = j0 + lane;
            const bool v = j < g.n_total;
            double4 p = make_double4(0, 0, 0, 0);
            if (v) p = g.pos[j];
            const bool h0 = v && live0 && (sqdist<D>(qa, p.x, p.y, p.z, p.w) < Ta);
            const bool h1 = v && live1 && (sqdist<D>(qb, p.x, p.y, p.z, p.w) < Tb);
            const unsigned m0 = __ballot_sync(FULL, h0);
            const unsigned o0 = wp0 + 2u * __popc(m0 & lt);
            if (h0 && o0 < sbuf + 2u * CAP) sts16(o0, 0x8000u | (unsigned)((j - g.n_sorted) & 0x7fff));
            wp0 += 2u * __popc(m0);
            const unsigned m1 = __ballot_sync(FULL, h1);
            const unsigned o1 = wp1 + 2u * __popc(m1 & lt);
            if (h1 && o1 < sbuf + 4u * CAP) sts16(o1, 0x8000u | (unsigned)((j - g.n_sorted) & 0x7fff));
            wp1 += 2u * __popc(m1);
          }
        }
        cnt0 = (int)((wp0 - sbuf) >> 1);
        cnt1 = (int)((wp1 - (sbuf + 2u * CAP)) >> 1);
        if (cnt0 > CAP || cnt1 > CAP) overflow = true;
      }
      const bool live1w = live1 && have1;
      if (!have1) cnt1 = 0;

      // ------------------------------------------- reserve the exact output range: one atomic per pair
      const int tot0 = cnt0 + (root_extra & 1), tot1 = cnt1 + ((root_extra >> 1) & 1);
      unsigned long long b0 = 0;
      if (lane == 0) b0 = atomicAdd(&cursor[0], (unsigned long long)(tot0 + tot1));
      b0 = __shfl_sync(FULL, b0, 0);
      if (lane == 0) {
        counts[qid0] = tot0;
        offsets[qid0] = (int64_t)b0;
        if (have1) {
          counts[qid1] = tot1;
          offsets[qid1] = (int64_t)(b0 + (unsigned long long)tot0);
        }
      }
      if (!write_lists || b0 + (unsigned long long)(tot0 + tot1) > cap) continue;  // counts only / lists do not fit
      __syncwarp();
      auto emit = [&](int k, const double *qs, int cnt, int64_t base, bool live_k) {
        if (!live_k) return;
        if (overflow) {
          v5_exact_query<D, true>(&s_g, qs, exactT(k), exactR(k), base, out_idx, out_dist);
        } else {
          const unsigned sb_k = sbuf + 2u * (unsigned)(k * CAP);
          if (has_tail) {
            v5_flush_tail<D>(&s_g, qs, sb_k, stab, cnt, out_idx + base, out_dist ? out_dist + base : nullptr);
          } else {
            double q[D];
#pragma unroll
            for (int c = 0; c < D; ++c) q[c] = qs[c];
            v5_flush<D, false>(g, q, sb_k, stab, cnt, lane, out_idx + base, out_dist ? out_dist + base : nullptr);
          }
        }
      };
      // one copy of the flush code for both queries (the warps of a block run unsynchronised, so code
      // size is instruction-cache pressure): a real loop, not two inlined bodies
#pragma unroll 1
      for (int k = 0; k < 2; ++k)
        emit(k, k ? qs1 : qs0, k ? cnt1 : cnt0, (int64_t)b0 + (k ? tot0 : 0), k ? live1w : live0);
      if (root_extra && lane == 0) {  // the root at exactly distance r: appended behind the strict hits
        const double4 p0 = g.pos[0];
        if (root_extra & 1) {
          double q[D];
#pragma unroll
          for (int c = 0; c < D; ++c) q[c] = qs0[c];
          out_idx[b0 + cnt0] = 0;
          if (out_dist) out_dist[b0 + cnt0] = __dsqrt_rn(sqdist<D>(q, p0.x, p0.y, p0.z, p0.w));
        }
        if (root_extra & 2) {
          double q[D];
#pragma unroll
          for (int c = 0; c < D; ++c) q[c] = qs1[c];
          out_idx[b0 + tot0 + cnt1] = 0;
          if (out_dist) out_dist[b0 + tot0 + cnt1] = __dsqrt_rn(sqdist<D>(q, p0.x, p0.y, p0.z, p0.w));
        }
      }
      __syncwarp();
    }
  }
}

// ---------------------------------------------------------------- wrap-around trees through the pair machinery
// One wrap dimension (the Dubins heading, period 2 pi) and r <= period / 2: the hit sets of the real query and of
// its ghost identity (ghostPoint.jl:60-111) are disjoint, so the reference's "first identity that reaches the node
// wins" dedup (kdTree_general.jl:903-916) never fires and the result is the concatenation of the two sets.  The
// batch is expanded into virtual queries 2j (real) and 2j+1 (ghost, or NaN -- a query that cannot hit -- when the ghost is
// not used): exactly the pair a warp works on, whose two lists it writes back to back.
template <int D>
__global__ void ghost_expand_kernel(WrapInfo wrap, const double *__restrict__ queries, const double *__restrict__ qsorted,
                                    const int32_t *__restrict__ qorder, int64_t nq, double r,
                                    double *__restrict__ vq, int32_t *__restrict__ vorder) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nq) return;
  const int qid = qorder[j];
  const double *src = qsorted ? qsorted + j * D : queries + (int64_t)qid * D;
  double q[D], gh[D];
#pragma unroll
  for (int k = 0; k < D; ++k) q[k] = src[k];
  const bool used = make_ghost<D>(wrap, q, 1, r, gh);
#pragma unroll
  for (int k = 0; k < D; ++k) {
    vq[(2 * j) * D + k] = q[k];
    vq[(2 * j + 1) * D + k] = used ? gh[k] : __longlong_as_double(0x7ff8000000000000LL);  // unused ghost: NaN, a dead query
  }
  vorder[2 * j] = 2 * qid;
  vorder[2 * j + 1] = 2 * qid + 1;
}
__global__ void ghost_merge_kernel(const int32_t *__restrict__ vcounts, const int64_t *__restrict__ voffsets, int64_t nq,
                                   int32_t *__restrict__ counts, int64_t *__restrict__ offsets) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nq) return;
  counts[q] = vcounts[2 * q] + vcounts[2 * q + 1];
  offsets[q] = voffsets[2 * q];  // the pair's lists are contiguous: real identity first, then the ghost
}

template <int D, int NW, int CAP, int TAB>
static void launch_v5(rrtqx_ctx *ctx, const GridView &g, const double *dq, const double *dqs, const int32_t *qorder,
                      int64_t nq, double r, double T, const double *dr, const double *dT, int32_t *counts,
                      int64_t *offsets, int32_t *idx, double *dist, unsigned long long cap, unsigned long long *cursor,
                      int write_lists, int ghost_pairs = 0) {
  const size_t smem = (size_t)NW * (CAP + TAB + V5_TABPAD) * sizeof(int);  // 16-bit hit codes: 2 * CAP * 2 bytes
  // the opt-in to > 48 KB of dynamic shared memory is per device: tracked per context, not per process
  if (ctx->smem_attr_done.insert((const void *)range_v5_kernel<D, NW, CAP, TAB, true>).second) {
    RQ_CUDA(cudaFuncSetAttribute(range_v5_kernel<D, NW, CAP, TAB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RQ_CUDA(cudaFuncSetAttribute(range_v5_kernel<D, NW, CAP, TAB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  V5Params P;
  P.RU = v5_radius(r, T, true);
  P.invx = (float)g.inv[0]; P.invy = (float)g.inv[1]; P.invz = (float)g.inv[2];
  P.celly = (float)g.cell[1]; P.cellz = (float)g.cell[2];
  P.unit = V5_UNIT;
  P.ghost_pairs = ghost_pairs;
  const int64_t n_units = ((nq + 1) / 2 + P.unit - 1) / P.unit;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>(n_units, (int64_t)ctx->sm_count));
  if (dr)
    range_v5_kernel<D, NW, CAP, TAB, false><<<blocks, NW * 32, smem, ctx->stream>>>(g, P, dq, dqs, qorder, nq, r, T, dr, dT, counts,
                                                                              offsets, idx, dist, cap, cursor, write_lists);
  else
    range_v5_kernel<D, NW, CAP, TAB, true><<<blocks, NW * 32, smem, ctx->stream>>>(g, P, dq, dqs, qorder, nq, r, T, dr, dT, counts,
                                                                             offsets, idx, dist, cap, cursor, write_lists);
  post_launch(ctx);
}

__global__ void thresh_kernel(const double *__restrict__ ranges, int64_t n, double *__restrict__ Tq) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) Tq[i] = sqrt_thresh_lt(ranges[i]);
}

template <int D>
static void range_query_fused(rrtqx_tree *t, const double *dq, const double *dr, int64_t nq, double r, uint32_t flags,
                              rrtqx_range_result *res) {
  rrtqx_ctx *ctx = t->ctx;
  cudaStream_t st = ctx->stream;
  const bool count_only = flags & RRTQX_RANGE_COUNT_ONLY;
  const bool want_dist = flags & RRTQX_RANGE_WANT_DIST;
  res->cursor.ensure(4, st);
  {
    PhaseScope p2(ctx, "range_sort");
    sort_queries<D>(t, res, dq, nq);
  }
  // wrap-around tree (one wrap dimension, r <= period / 2, checked by the caller): expand into (real, ghost) pairs
  const bool ghost = t->wrap.num_wraps == 1;
  const double *kq = dq, *kqs = res->qbins > 0 ? res->qsorted.p : nullptr;
  const int32_t *korder = res->qorder.p;
  int32_t *kcounts = res->counts.p;
  int64_t *koffsets = res->offsets.p;
  int64_t knq = nq;
  if (ghost) {
    res->vq.ensure((size_t)nq * 2 * D, st);
    res->vorder.ensure((size_t)nq * 2, st);
    res->vcounts.ensure((size_t)nq * 2 + 1, st);
    res->voffsets.ensure((size_t)nq * 2 + 1, st);
    ghost_expand_kernel<D><<<div_up(nq, 256), 256, 0, st>>>(t->wrap, dq, kqs, res->qorder.p, nq, r, res->vq.p, res->vorder.p);
    post_launch(ctx);
    kq = nullptr; kqs = res->vq.p; korder = res->vorder.p; kcounts = res->vcounts.p; koffsets = res->voffsets.p; knq = 2 * nq;
  }
  const double T = host_sqrt_thresh_lt(r);
  const double *dT = nullptr;
  if (dr) {
    res->tq.ensure((size_t)nq, st);
    thresh_kernel<<<div_up(nq, 256), 256, 0, st>>>(dr, nq, res->tq.p);
    post_launch(ctx);
    dT = res->tq.p;
  }
  // Output capacity: grow-only buffers sized by the previous results; if the
  // lists do not fit, the pass still yields exact counts + total and is
  // repeated once with the exact size (first call / growing workloads only).
  size_t cap = count_only ? 0 : res->idx.cap;
  if (!count_only && want_dist) cap = std::min(cap, res->dist.cap);
  if (!count_only && cap == 0) {
    cap = (size_t)nq * 64;
    res->idx.ensure(cap, st, 0, 1.0);
    if (want_dist) res->dist.ensure(cap, st, 0, 1.0);
    cap = want_dist ? std::min(res->idx.cap, res->dist.cap) : res->idx.cap;
  }
  // Expected neighbours per query (only selects the kernel variant): the uniform-density estimate
  // n * V_ball(r) / V_grid with a 15 % margin; per-query radii take the large-buffer variant.
  double k_est = 1e9;
  if (!dr && r > 0.0 && std::isfinite(r)) {
    double vol = 1.0;
    int dims = 0;
    const int nd[3] = {t->nx, t->ny, t->nz};
    for (int c = 0; c < 3; ++c)
      if (nd[c] > 1) { vol *= nd[c] * t->cell[c]; dims++; }
    const double ball = dims == 3 ? 4.18879 * r * r * r : (dims == 2 ? 3.14159 * r * r : 2.0 * r);
    k_est = dims ? 1.15 * (double)t->n * ball / vol : (double)t->n;
  } else if (!dr) {
    k_est = 0.0;
  }
  int variant = k_est <= 576.0 ? 0 : (k_est <= 1280.0 ? 1 : (k_est <= 2048.0 ? 2 : 3));
  if (ctx->tune.fused_variant >= 0) variant = ctx->tune.fused_variant;
  unsigned long long total = 0;
  for (int attempt = 0; attempt < 2; ++attempt) {
    GridView g = t->view();
    RQ_CUDA(cudaMemsetAsync(res->cursor.p, 0, 4 * sizeof(unsigned long long), st));
    {
      PhaseScope p2(ctx, "range_fill");
#define RQ_V5(NW_, CAP_, TAB_)                                                                                       \
  launch_v5<D, NW_, CAP_, TAB_>(ctx, g, kq, kqs, korder, knq, r, T, dr, dT, kcounts, koffsets, res->idx.p, \
                                want_dist ? res->dist.p : nullptr, (unsigned long long)cap, res->cursor.p, count_only ? 0 : 1, ghost ? 1 : 0)
      // hit buffers leave 32*V5_U entries of head-room; the octet table must hold a whole pair's region (else the
      // pair takes the exact routine)
      if (variant == 0) RQ_V5(24, 704, 256);          // 24 warps/SM (80 registers), 94 KB shared
      else if (variant == 1) RQ_V5(24, 1408, 512);    // 186 KB
      else if (variant == 2) RQ_V5(16, 2176, 1024);   // 205 KB
      else RQ_V5(8, 4224, 2048);                      // 201 KB
#undef RQ_V5
    }
    RQ_CUDA(cudaMemcpyAsync(&total, res->cursor.p, sizeof(total), cudaMemcpyDeviceToHost, st));
    RQ_CUDA(cudaStreamSynchronize(st));
    if (count_only || total <= cap) break;
    RQ_REQUIRE(attempt == 0, "internal: range output did not fit after resizing");
    cap = (size_t)total + (size_t)(total / 32) + 1024;
    res->idx.ensure(cap, st, 0, 1.0);
    if (want_dist) res->dist.ensure(cap, st, 0, 1.0);
    cap = want_dist ? std::min(res->idx.cap, res->dist.cap) : res->idx.cap;
  }
  if (ghost) {
    ghost_merge_kernel<<<div_up(nq, 256), 256, 0, st>>>(res->vcounts.p, res->voffsets.p, nq, res->counts.p, res->offsets.p);
    post_launch(ctx);
  }
  res->n_queries = nq;
  res->total = (int64_t)total;
  res->has_lists = !count_only;
  res->has_dist = !count_only && want_dist;
}
