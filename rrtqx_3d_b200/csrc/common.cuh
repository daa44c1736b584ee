// common.cuh -- shared host/device infrastructure of librrtqx_b200.so.
// sm_100a only; compiled with -fmad=false, and every arithmetic step that
// decides a result uses the explicit round-to-nearest intrinsics so that no
// FMA contraction can ever change a bit (SURVEY.md appendix A).
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rrtqx_b200.h"

namespace rrtqx {

// ------------------------------------------------------------------ errors
struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

#define RQ_CUDA(expr)                                                         \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess) {                                                  \
      char _b[512];                                                           \
      snprintf(_b, sizeof(_b), "%s failed: %s (%s:%d)", #expr,                \
               cudaGetErrorString(_e), __FILE__, __LINE__);                   \
      throw ::rrtqx::Error(_e == cudaErrorMemoryAllocation ? RRTQX_ERR_NOMEM  \
                                                           : RRTQX_ERR_CUDA,  \
                           _b);                                               \
    }                                                                         \
  } while (0)

#define RQ_REQUIRE(cond, msg)                                                 \
  do {                                                                        \
    if (!(cond)) throw ::rrtqx::Error(RRTQX_ERR_INVALID, msg);                \
  } while (0)

// --------------------------------------------------------- device buffers
// Grow-only typed device buffer.  Frees are deferred to destruction so that
// work already queued on the stream never loses its memory.
template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t cap = 0;
  std::vector<T *> graveyard;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    for (T *g : graveyard) cudaFree(g);
    graveyard.clear();
    p = nullptr;
    cap = 0;
  }
  // Ensure capacity >= n elements.  preserve = number of leading elements to
  // keep (copied on `stream`).
  void ensure(size_t n, cudaStream_t stream = 0, size_t preserve = 0,
              double growth = 1.5) {
    if (n <= cap) return;
    size_t nc = (size_t)((double)cap * growth);
    if (nc < n) nc = n;
    if (nc < 256) nc = 256;
    T *np = nullptr;
    RQ_CUDA(cudaMalloc((void **)&np, nc * sizeof(T)));
    if (p && preserve) {
      RQ_CUDA(cudaMemcpyAsync(np, p, preserve * sizeof(T),
                              cudaMemcpyDeviceToDevice, stream));
    }
    if (p) graveyard.push_back(p);
    p = np;
    cap = nc;
  }
  // Free retired allocations; only call after the stream has been synchronised.
  void collect() {
    for (T *g : graveyard) cudaFree(g);
    graveyard.clear();
  }
};

inline bool is_device_ptr(const void *p) {
  if (!p) return false;
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

}  // namespace rrtqx

// Diagnostic switches (DESIGN.md section 5).  The environment is read ONCE per context, at rrtqx_ctx_create
// (and again only on an explicit rrtqx_ctx_reload_tuning): no libc lock or string scan sits inside a planner
// iteration.  None of the switches selects a CPU path.
namespace rrtqx {
struct Tuning {
  bool edge_no_grid = false, edge_no_queue = false, range_two_pass = false, nearest_warp = false, no_item_grid = false;
  int64_t cover_min_items = -1;  // < 0: the measured break-even defaults
  int fused_variant = -1;        // < 0: chosen from the expected neighbour count
  int qsort_s = 2, qsort_f = 1;  // supercells of 2^3 cells with the 2:1 grid aspect (scripts/tune_v5.sh)
  bool comm_no_ipc = false;      // one process per GPU: gathers through NCCL even where IPC windows are possible
  int comm_ipc_mb = 64;          // bytes per slot of the IPC result window (two slots per rank), MiB
  int nccl_max_ctas = 0;         // cap on the CTAs NCCL may use for this library's gathers (0: NCCL's default; caps of 1-4 measured slower on 8 B200s)
  double grid_occupancy = 0.0, grid_aspect = 0.0;  // 0: the tree's defaults
  void load() {
    *this = Tuning();
    auto on = [](const char *n) { return getenv(n) != nullptr; };
    auto geti = [](const char *n, long long d) { const char *e = getenv(n); return e ? atoll(e) : d; };
    auto getd = [](const char *n) { const char *e = getenv(n); return e ? atof(e) : 0.0; };
    edge_no_grid = on("RRTQX_EDGE_NO_GRID");
    edge_no_queue = on("RRTQX_EDGE_NO_QUEUE");
    range_two_pass = on("RRTQX_RANGE_TWO_PASS");
    nearest_warp = on("RRTQX_NEAREST_WARP");
    no_item_grid = on("RRTQX_NO_ITEM_GRID");
    cover_min_items = geti("RRTQX_COVER_MIN_ITEMS", -1);
    fused_variant = (int)geti("RRTQX_FUSED_VARIANT", -1);
    nccl_max_ctas = (int)geti("RRTQX_NCCL_MAX_CTAS", 0);
    comm_no_ipc = on("RRTQX_COMM_NO_IPC");
    { const long long mb = geti("RRTQX_COMM_IPC_MB", 64); comm_ipc_mb = (int)(mb < 1 ? 1 : (mb > 4096 ? 4096 : mb)); }
    const long long s = geti("RRTQX_QSORT_S", 2), f = geti("RRTQX_QSORT_F", 1);
    qsort_s = (int)(s < 1 ? 1 : (s > 16 ? 16 : s));
    qsort_f = (int)(f < 1 ? 1 : (f > 8 ? 8 : f));
    const double o = getd("RRTQX_GRID_OCCUPANCY"), a = getd("RRTQX_GRID_ASPECT");
    grid_occupancy = o > 0.0 ? o : 0.0;
    grid_aspect = a >= 1.0 ? a : 0.0;
  }
};

// Scratch objects owned by a context or a tree, keyed by the address of a tag: created on first use, destroyed
// with their owner (rrtqx_ctx_destroy / rrtqx_tree_destroy), guarded by the owner's mutex.
struct ScratchMap {
  struct Slot { void *p; void (*del)(void *); };
  std::map<const void *, Slot> slots;
  std::mutex mu;
  template <class T>
  T &get(const void *key) {
    std::lock_guard<std::mutex> lk(mu);
    auto it = slots.find(key);
    if (it == slots.end())
      it = slots.emplace(key, Slot{new T(), [](void *q) { delete static_cast<T *>(q); }}).first;
    return *static_cast<T *>(it->second.p);
  }
  void clear() {
    std::lock_guard<std::mutex> lk(mu);
    for (auto &kv : slots) kv.second.del(kv.second.p);
    slots.clear();
  }
  ~ScratchMap() { clear(); }
};
}  // namespace rrtqx

// ------------------------------------------------------------------ context
struct rrtqx_ctx {
  int device = 0;
  rrtqx::Tuning tune;
  rrtqx::ScratchMap scratch;                 // per-context scratch buffers of the collision / sweep paths
  std::set<const void *> smem_attr_done;     // kernels whose dynamic shared memory opt-in is set on THIS device
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int sm_count = 148;
  std::string err;
  int64_t launches = 0;
  struct Phase {
    cudaEvent_t a = nullptr, b = nullptr;
    bool valid = false;
  };
  std::map<std::string, Phase> phases;
  // staging buffers for host<->device traffic of the batched calls
  rrtqx::DevBuf<double> stage_f64;
  rrtqx::DevBuf<int32_t> stage_i32a, stage_i32b;
  rrtqx::DevBuf<uint8_t> stage_u8;
  rrtqx::DevBuf<double> stage_f64b;

  void phase_begin(const char *name) {
    Phase &p = phases[name];
    if (!p.a) {
      cudaEventCreate(&p.a);
      cudaEventCreate(&p.b);
    }
    cudaEventRecord(p.a, stream);
    p.valid = false;
  }
  void phase_end(const char *name) {
    Phase &p = phases[name];
    cudaEventRecord(p.b, stream);
    p.valid = true;
  }
};

namespace rrtqx {

// Registry of live contexts and trees.  Garbage-collected hosts (Julia finalizers, Python __del__) destroy handles
// in arbitrary order, so a child (tree, obstacle set, edge set, result) may be destroyed AFTER its context / tree:
// the destroy entry points ask here before they touch the parent, and free the child's memory without it.
void handle_register(const void *h);
void handle_unregister(const void *h);
bool handle_live(const void *h);

// RAII phase timer
struct PhaseScope {
  rrtqx_ctx *c;
  const char *n;
  PhaseScope(rrtqx_ctx *c_, const char *n_) : c(c_), n(n_) { c->phase_begin(n); }
  ~PhaseScope() { c->phase_end(n); }
};

inline void post_launch(rrtqx_ctx *ctx, int n = 1) {
  ctx->launches += n;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    throw Error(RRTQX_ERR_CUDA, std::string("kernel launch failed: ") + cudaGetErrorString(e));
}

// Small results of a call (counts, flags) travel through one block of mapped pinned memory per context: the call's
// last kernel stores them and then a call number, and the host spins on that word -- no copy operations, no stream
// synchronisation (each of those costs 10-15 us on a call whose kernels take 40).  D2H copies of single words that
// cannot come from a kernel use `aux` as their pinned target.
struct HostMail {
  struct Block { unsigned long long seq; long long v[6]; int32_t aux[2]; };
  Block *h = nullptr, *d = nullptr;   // host / device views
  unsigned long long seq = 0;         // calls issued
  ~HostMail() { if (h) cudaFreeHost(h); }
  void ensure() {
    if (h) return;
    RQ_CUDA(cudaHostAlloc((void **)&h, sizeof(Block), cudaHostAllocMapped));
    RQ_CUDA(cudaHostGetDevicePointer((void **)&d, h, 0));
    memset(h, 0, sizeof(Block));
  }
  // spin until the device has published call `want`; a stream query every few thousand spins turns a faulted launch
  // into an error instead of a hang
  void wait(cudaStream_t st, unsigned long long want) {
    volatile unsigned long long *seqp = &h->seq;
    for (unsigned spins = 0; *seqp != want; ++spins) {
      if ((spins & 0xfff) == 0xfff) {
        cudaError_t qe = cudaStreamQuery(st);
        if (qe == cudaSuccess) break;
        if (qe != cudaErrorNotReady) RQ_CUDA(qe);
      }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    if (*seqp != want) RQ_CUDA(cudaStreamSynchronize(st));
  }
};
inline HostMail &host_mail(rrtqx_ctx *ctx) {
  static const char tag = 0;
  HostMail &m = ctx->scratch.get<HostMail>(&tag);
  m.ensure();
  return m;
}

// Input array that may live on host or device: returns a device pointer valid
// on ctx->stream, staging through `buf` when the source is host memory.
template <typename T>
const T *to_device(rrtqx_ctx *ctx, const T *src, size_t n, DevBuf<T> &buf) {
  if (n == 0 || src == nullptr) return nullptr;
  if (is_device_ptr(src)) return src;
  buf.ensure(n, ctx->stream);
  RQ_CUDA(cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
  return buf.p;
}

// Copy n elements from device memory to a host-or-device destination.
template <typename T>
void from_device(rrtqx_ctx *ctx, T *dst, const T *src_dev, size_t n) {
  if (n == 0 || dst == nullptr) return;
  RQ_CUDA(cudaMemcpyAsync(dst, src_dev, n * sizeof(T), cudaMemcpyDefault, ctx->stream));
}

inline int div_up(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------ device math
#ifdef __CUDACC__

constexpr unsigned FULL = 0xffffffffu;

// euclidianDist radicand (DRRT_distance_functions.jl:37): left-to-right sum of
// individually rounded squares of individually rounded differences.
template <int D>
__device__ __forceinline__ double sqdist(const double *q, double px, double py, double pz, double pw) {
  double dx = __dsub_rn(q[0], px);
  double dy = __dsub_rn(q[1], py);
  double s = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
  if (D >= 3) {
    double dz = __dsub_rn(q[2], pz);
    s = __dadd_rn(s, __dmul_rn(dz, dz));
  }
  if (D >= 4) {
    double dw = __dsub_rn(q[3], pw);
    s = __dadd_rn(s, __dmul_rn(dw, dw));
  }
  return s;
}

__device__ __forceinline__ double next_up(double x) {  // x finite, >= 0
  return __longlong_as_double(__double_as_longlong(x) + 1);
}
__device__ __forceinline__ double next_down(double x) {  // x finite, > 0
  return __longlong_as_double(__double_as_longlong(x) - 1);
}

// T_lt(r) = min{ t >= 0 : fl(sqrt(t)) >= r }  so that  sqrt(s) < r  <=>  s < T_lt
// (monotonicity of correctly rounded sqrt; SURVEY.md appendix A4).
__device__ inline double sqrt_thresh_lt(double r) {
  if (r != r) return r;            // NaN: s < NaN is false for every s
  if (r <= 0.0) return 0.0;        // sqrt(s) < r never holds
  if (isinf(r)) return r;          // every finite s qualifies
  double t = __dmul_rn(r, r);
  if (isinf(t)) {                  // r^2 overflows: search below DBL_MAX
    t = 1.7976931348623157e308;
    if (__dsqrt_rn(t) < r) return __longlong_as_double(0x7ff0000000000000LL);
  }
  while (t > 0.0 && __dsqrt_rn(t) >= r) t = next_down(t);
  while (__dsqrt_rn(t) < r) t = next_up(t);
  return t;
}

// Host twin of sqrt_thresh_lt (std::sqrt is correctly rounded, like __dsqrt_rn).
inline double host_sqrt_thresh_lt(double r) {
  if (r != r) return r;
  if (r <= 0.0) return 0.0;
  if (std::isinf(r)) return r;
  double t = r * r;
  if (std::isinf(t)) {
    t = 1.7976931348623157e308;
    if (std::sqrt(t) < r) return INFINITY;
  }
  while (t > 0.0 && std::sqrt(t) >= r) t = std::nextafter(t, -INFINITY);
  while (std::sqrt(t) < r) t = std::nextafter(t, INFINITY);
  return t;
}

// T_le(r) = max{ t : fl(sqrt(t)) <= r }  so that  sqrt(s) <= r <=> s <= T_le
// and  sqrt(s) > r <=> s > T_le.   Returns -1 if no t >= 0 qualifies.
__device__ inline double sqrt_thresh_le(double r) {
  if (r != r) return r;            // comparisons with NaN are false
  if (r < 0.0) return -1.0;
  if (isinf(r)) return r;
  double t = __dmul_rn(r, r);
  if (isinf(t)) t = 1.7976931348623157e308;
  while (__dsqrt_rn(t) <= r && t < 1.7976931348623157e308) t = next_up(t);
  while (t > 0.0 && __dsqrt_rn(t) > r) t = next_down(t);
  return t;
}

// Julia Base.min / Base.max on Float64: NaN-propagating, -0.0 < +0.0.
__device__ __forceinline__ double jl_min(double x, double y) {
  bool sy = __double_as_longlong(y) < 0, sx = __double_as_longlong(x) < 0;
  if ((y < x) || (sy && !sx)) return (x != x) ? x : y;
  return (y != y) ? y : x;
}
__device__ __forceinline__ double jl_max(double x, double y) {
  bool sy = __double_as_longlong(y) < 0, sx = __double_as_longlong(x) < 0;
  if ((y > x) || (!sy && sx)) return (x != x) ? x : y;
  return (y != y) ? y : x;
}

// ---- TMA (bulk asynchronous copy engine) staging of regular tiles: global -> shared, completion on an mbarrier.
// One thread arms the barrier with the byte count and issues the copies; every thread of the block waits on the
// barrier's phase.  No register round trip, no per-thread address arithmetic, and the LSU stays free while a tile is
// in flight.  Addresses and sizes must be multiples of 16 bytes (cudaMalloc'ed tables of 16 / 32-byte records are).
__device__ __forceinline__ unsigned smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *smem_dst, const void *gmem_src, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_addr(bar)), "r"(phase) : "memory");
}
// Stage `n` records of two parallel tables (recA: sizeA bytes each, recB optional) as one tile.  Called by ALL
// threads of the block: a block barrier protects the previous tile's readers, thread 0 issues, everybody waits.
__device__ __forceinline__ void tma_stage_tile(void *sA, const void *gA, unsigned bytesA, void *sB, const void *gB,
                                               unsigned bytesB, unsigned long long *bar, unsigned &phase) {
  __syncthreads();  // the previous tile is no longer read
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, bytesA + bytesB);
    tma_load_1d(sA, gA, bytesA, bar);
    if (bytesB) tma_load_1d(sB, gB, bytesB, bar);
  }
  mbar_wait(bar, phase);
  phase ^= 1u;
}

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

#endif  // __CUDACC__

}  // namespace rrtqx
