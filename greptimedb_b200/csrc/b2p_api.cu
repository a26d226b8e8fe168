// b2p_api.cu — C ABI of libb200promql.so (see include/b200promql.h).
// Host-side runtime: context, stream, device scratch, kernel dispatch, slow-path completion.
// There is NO CPU fallback anywhere in this file: every entry point either launches the CUDA
// kernels or returns an error.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/b200promql.h"
#include "b2p_aggregate.cuh"
#include "b2p_kernel_t.cuh"
#include "b2p_kernel_lean.cuh"
#include "b2p_kernels.cuh"

using namespace b2p;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU(x)                                                                                   \
  do {                                                                                          \
    cudaError_t e__ = (x);                                                                      \
    if (e__ != cudaSuccess) return fail(B2P_E_CUDA, "%s: %s (%s:%d)", #x, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

// NCCL, bound at run time: libnccl.so.2 is not a link dependency (single-GPU users never need it), and inside a
// process that already loaded an NCCL (e.g. the one bundled with torch) dlopen hands back that same library.
// Only the handful of entry points the by-label all-reduce needs; enum values are NCCL's ABI (nccl.h).
struct Nccl {
  typedef struct ncclComm* comm_t;
  struct unique_id { char internal[128]; };
  enum { kSum = 0, kMax = 2, kMin = 3 };
  enum { kUint32 = 3, kInt64 = 4, kUint64 = 5, kFloat64 = 8 };
  int (*GetUniqueId)(unique_id*) = nullptr;
  int (*CommInitRank)(comm_t*, int, unique_id, int) = nullptr;
  int (*CommDestroy)(comm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  void* handle = nullptr;
  bool load() {
    if (handle) return true;
    const char* names[] = {getenv("B2P_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) return false;
    bool ok = true;
    auto sym = [&](const char* n) { void* p = dlsym(handle, n); ok = ok && p; return p; };
    GetUniqueId = reinterpret_cast<decltype(GetUniqueId)>(sym("ncclGetUniqueId"));
    CommInitRank = reinterpret_cast<decltype(CommInitRank)>(sym("ncclCommInitRank"));
    CommDestroy = reinterpret_cast<decltype(CommDestroy)>(sym("ncclCommDestroy"));
    AllReduce = reinterpret_cast<decltype(AllReduce)>(sym("ncclAllReduce"));
    GroupStart = reinterpret_cast<decltype(GroupStart)>(sym("ncclGroupStart"));
    GroupEnd = reinterpret_cast<decltype(GroupEnd)>(sym("ncclGroupEnd"));
    GetErrorString = reinterpret_cast<decltype(GetErrorString)>(sym("ncclGetErrorString"));
    if (!ok) { handle = nullptr; }
    return ok;
  }
};
Nccl g_nccl;

#define NCCL_TRY(x)                                                                                          \
  do {                                                                                                       \
    int r__ = (x);                                                                                           \
    if (r__ != 0) return fail(B2P_E_CUDA, "%s: %s", #x, g_nccl.GetErrorString ? g_nccl.GetErrorString(r__) : "NCCL error"); \
  } while (0)


struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return B2P_OK;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      e = cudaMalloc(&p, bytes);
      want = bytes;
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(B2P_E_NOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    }
    cap = want;
    return B2P_OK;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

constexpr int kRing = 256;
constexpr int kBigRing = 1024;        // long-window instantiation of the warp-per-series kernel (one CTA per SM)
constexpr int kStatusSlots = 32;      // range calls that may be outstanding between two b2p_sync
constexpr int kSlowCtas = 148;        // slow-path grid (4 warps per CTA)
constexpr int kSlowWarps = kSlowCtas * 4;
constexpr size_t kArenaDefaultRows = 1u << 21;  // 32 MB: regions of 3 542 rows for the 592 slow-path warps

}  // namespace

// group -> member-series CSR of one gid[] assignment (b2p_group_index_create_dev), reusable across calls
struct b2p_group_index {
  uint32_t n_series = 0, n_groups = 0;
  uint32_t max_members = 0;      // size of the largest group
  uint32_t* gid = nullptr;       // [n_series] device copy
  uint32_t* goff = nullptr;      // [n_groups + 1]
  uint32_t* members = nullptr;   // [n_series] series ids ordered by (group, series id)
};

struct b2p_ctx {
  int device = 0;
  int num_sms = 148;
  cudaStream_t own_stream = nullptr, stream = nullptr;
  // Device-side status.  Every range call owns one slot of d_ring until b2p_sync has read it back, so any number
  // (<= kStatusSlots, then the library synchronises by itself) of *_dev range calls may be outstanding; the verdict
  // of the series-id scan (K0) is sticky in d_k0 until the next b2p_sync.
  Status* d_ring = nullptr;  // [kStatusSlots]
  Status* h_ring = nullptr;  // pinned mirror
  Status* d_k0 = nullptr;
  Status* h_k0 = nullptr;    // pinned
  int next_slot = 0;
  struct Pending {
    int slot; int fn; RangeArgs args; int lean_mode; bool thread_tier; bool used_lean; uint32_t n_series; bool verdict_taken;
    bool fused;  // by-label partials were added in place: only the slow kernel may be repeated
    bool merged; // ... and already all-reduced (or tiled): nothing can be repeated, an arena overflow is an error
  };
  std::vector<Pending> pending;
  DevBuf slow_list, w_list, b_list, arena_ts, arena_val, win_scratch;
  // multi-GPU (one process per GPU): communicator of the by-label all-reduce, its stream and join event
  Nccl::comm_t comm = nullptr;
  int comm_ranks = 1, comm_rank = 0;
  long long comm_headstart_cycles = 60000;  // ~30 us at 1.965 GHz (B2P_COMM_HEADSTART_US overrides)
  // SMs the fused tier leaves to the tile all-reduce (B2P_COMM_RESERVE_SMS).  Off: measured at 2 GPUs, 0 / 8 / 16 SMs
  // left free give 12.0 / 12.3 / 14.2 ms per step — the all-reduce of a tile still does not run beside the next tile's
  // kernel, the step only loses the SMs (DESIGN.md section 7)
  int comm_reserve_sms = 0;
  int comm_reserve_now = 0;                 // ... in effect for the launch being issued
  cudaStream_t s_comm = nullptr;
  cudaEvent_t ev_comm_in = nullptr, ev_comm_done = nullptr, ev_comm_go = nullptr;
  DevBuf m_tmp0, m_tmp1;             // scratch of the variance merge
  DevBuf w_skip, b_skip, slow_skip;  // fused by-label partials: steps already added, parallel to the work lists
  bool fused_pending = false;        // a fused call is outstanding: its work lists must survive until b2p_sync
  // K2T (thread per series) in front of K2 for rate/increase/delta.  Measured slower than K2 on B200
  // (28 vs 64 G samples/s, profiles/r1_thread_tier.md), so it is opt-in: B2P_ENABLE_THREAD_TIER=1.
  bool thread_tier = false;
  // K2L, the lean warp-per-series tier in front of K2 (default on; B2P_DISABLE_LEAN_TIER=1 turns it off)
  bool lean_tier = true;
  // adaptive tiering: when K2L handed more than half of the series of a call to K2 (e.g. every counter has resets),
  // the next calls skip it for a while; the verdict is taken wherever the status block is read back
  bool lean_force_flags = false;  // B2P_LEAN_FORCE_FLAGS=1: rate / increase always take the bit-word variant (tests)
  bool lean_adaptive = true;    // B2P_LEAN_ADAPTIVE=0 switches the back-off off (tests that pin the tier)
  // per range function: 0 = plain K2L; 1 = K2L with reset bit words (rate / increase after a call that handed most
  // series on); 2 = skip K2L.  `lean_backoff` counts the calls a non-zero mode still lasts.
  int lean_mode[B2P_FN__COUNT] = {};
  int lean_backoff[B2P_FN__COUNT] = {};
  int last_lean_mode = 0;
  int last_range_fn = 0;
  bool last_used_lean = false;  // the pending / last range call started with K2L
  uint32_t last_range_series = 0;
  int lean_blocks_per_sm[B2P_FN__COUNT][2][2] = {};  // [fn][FLAGS][UNI]
  // first-tier variant for equally spaced samples (rate / increase / delta): -1 = cadence_probe_kernel decides per call
  // on the device, 0 / 1 = forced (B2P_UNIFORM)
  int uniform_mode = -1;
  size_t arena_rows = 0;
  size_t arena_rows_wanted = 0;  // B2P_ARENA_ROWS: initial size of the slow-path arena (default kArenaDefaultRows)
  cudaEvent_t ev[5][2] = {};  // 0 K0, 1 range tiers, 2 slow kernel, 3 by-label aggregate, 4 all-reduce (last tile)
  bool ev_used[5] = {false, false, false, false, false};
  long long launches = 0;
  long long last_slow = 0;
  long long last_w = 0;
  // host-API staging
  DevBuf h_ts, h_val, h_sid, h_off, h_out, h_valid, h_aux0, h_aux1, h_aux2, h_aux3;
  // host-API pipeline (double-buffered staging, separate copy streams)
  bool pipe_ready = false;
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_h2d[2] = {}, ev_comp[2] = {}, ev_d2h[2] = {};
  DevBuf p_ts[2], p_val[2], p_sid[2], p_off[2], p_out[2], p_valid[2], p_status;
  DevBuf p_t0[2], p_cad[2];  // per-series (first timestamp, cadence) of a chunk whose timestamp column stays on the host
  // b2p_range_eval: scan every chunk on the host (worker threads, ahead of the copies) and, where all of its series are
  // equally spaced, send (offsets, t0, cadence) instead of the timestamp and id columns (B2P_HOST_TS_SCAN=0: never)
  bool host_ts_scan = true;
  long long last_h2d_bytes = 0;
  // uniform histogram layout -> fold index (b2p_histogram_quantile_dev)
  DevBuf hq_off, hq_series, hq_les;
  // group aggregate scratch
  DevBuf g_keys_in, g_keys_out, g_vals_in, g_vals_out, g_goff, g_tmp;
  // column reduce scratch
  DevBuf c_psum, c_pcnt;
  int fast_blocks_per_sm[B2P_FN__COUNT][2] = {};
  int big_blocks_per_sm[B2P_FN__COUNT] = {};
};

namespace {

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    int cur = -1;
    cudaGetDevice(&cur);
    if (prev >= 0 && cur != prev) cudaSetDevice(prev);
  }
};

void stage_begin(b2p_ctx* c, int stage) {
  cudaEventRecord(c->ev[stage][0], c->stream);
}
void stage_end(b2p_ctx* c, int stage) {
  cudaEventRecord(c->ev[stage][1], c->stream);
  c->ev_used[stage] = true;
}
void stage_begin_on(b2p_ctx* c, int stage, cudaStream_t s) { cudaEventRecord(c->ev[stage][0], s); }
void stage_end_on(b2p_ctx* c, int stage, cudaStream_t s) {
  cudaEventRecord(c->ev[stage][1], s);
  c->ev_used[stage] = true;
}

template <int FN, bool TS32>
int launch_fast_t(b2p_ctx* c, const RangeArgs& a) {
  constexpr size_t smem = (size_t)kWarpsPerCta * (2 * kRing * (8 + (TS32 ? 4 : 8)) + kRing / 8) + kRcpTable * 8;
  auto kern = range_fast_kernel<FN, kRing, TS32>;
  int& cached = c->fast_blocks_per_sm[FN][TS32 ? 1 : 0];
  if (cached == 0) {
    int nb = 0;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kWarpsPerCta * 32, smem));
    cached = nb > 0 ? nb : 1;
  }
  const unsigned need = (a.n_series + kWarpsPerCta - 1) / kWarpsPerCta;
  const unsigned cap = (unsigned)(c->num_sms * cached);
  const unsigned grid = need < cap ? need : cap;
  if (grid == 0) return B2P_OK;
  kern<<<grid, kWarpsPerCta * 32, smem, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

// Long-window instantiation (32-bit time domain only): RING = kBigRing, one CTA per SM, over RangeArgs::b_list.
template <int FN>
int launch_big(b2p_ctx* c, const RangeArgs& a0) {
  RangeArgs a = a0;
  a.use_w_list = 2;
  constexpr size_t smem = (size_t)kWarpsPerCta * (2 * kBigRing * (8 + 4) + kBigRing / 8) + kRcpTable * 8;
  auto kern = range_fast_kernel<FN, kBigRing, true>;
  int& cached = c->big_blocks_per_sm[FN];
  if (cached == 0) {
    int nb = 0;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kWarpsPerCta * 32, smem));
    cached = nb > 0 ? nb : 1;
  }
  kern<<<(unsigned)(c->num_sms * cached), kWarpsPerCta * 32, smem, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

// 32-bit relative timestamps when the whole query span (plus one lookback) fits 31 bits of ms.
bool fits_ts32(const RangeArgs& a) {
  const double span = (double)a.end - (double)a.start + (double)a.range;
  return span >= 0 && span < 2147483000.0 && a.interval < 2147483000ll && a.range < 2147483000ll;
}

template <int FN>
constexpr bool lean_supports() { return LeanTraits<FN>::kSupported; }

// Adaptive tiering verdict of a finished range call that started with K2L: more than half of the series handed on ->
// the next 32 calls of this function use the next mode (plain -> bit words for rate / increase -> skip).
void lean_verdict(b2p_ctx* c, int fn, uint64_t handed, uint64_t n_series) {
  if (!c->lean_adaptive || handed * 2 <= n_series) return;
  const bool counter = (fn == B2P_FN_RATE || fn == B2P_FN_INCREASE);
  c->lean_mode[fn] = (c->last_lean_mode == 0 && counter) ? 1 : 2;
  c->lean_backoff[fn] = 32;
}

bool lean_fn_supported(int fn) {
  switch (fn) {
#define X(N) case N: return lean_supports<N>();
    X(0) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19) X(20)
#undef X
  }
  return false;
}

bool lean_ok(const b2p_ctx* c, int fn, const RangeArgs& a) {
  if (!c->lean_tier || !lean_fn_supported(fn)) return false;
  if (!fits_ts32(a) || a.range < a.interval || a.start < 0) return false;
  if (fn == B2P_FN_RATE && a.rcp_rs == 0.0) return false;
  return (double)a.rel_max + 64.0 * (double)a.interval < 4294967295.0;
}

template <int FN>
int launch_fast(b2p_ctx* c, const RangeArgs& a) {
  return fits_ts32(a) ? launch_fast_t<FN, true>(c, a) : launch_fast_t<FN, false>(c, a);
}

// Lean first tier (K2L): rate / increase / delta in the 32-bit time domain.  The gates are what the kernel
// relies on: exact reciprocal division by range/1000, range >= interval (steps evaluated before the end of a
// series are below the trimmed end), start >= 0 (truncating division == floor in the end trim), and window
// ends of the 31 steps past the grid still below the 0xFFFFFFFF end sentinel.
bool lean_ok(const b2p_ctx* c, int fn, const RangeArgs& a);

// Functions whose first tier has a uniform-cadence variant: the probe (or B2P_UNIFORM) writes Status::uniform, then
// both variants are launched and the one the verdict does not name returns at once — no host round trip.
static int cadence_verdict(b2p_ctx* c, const RangeArgs& a) {
  if (c->uniform_mode < 0) {
    cadence_probe_kernel<<<1, kProbeThreads, 0, c->stream>>>(a);
    c->launches++;
    CU(cudaGetLastError());
  } else {
    CU(cudaMemsetAsync(&a.status->uniform, c->uniform_mode ? 1 : 0, sizeof(uint32_t), c->stream));
  }
  return B2P_OK;
}

template <int FN, bool FLAGS, bool UNI>
int launch_lean_variant(b2p_ctx* c, const RangeArgs& a) {
  constexpr size_t smem = lean_smem_bytes(UNI);
  auto kern = range_lean_kernel<FN, FLAGS, false, UNI>;
  int& cached = c->lean_blocks_per_sm[FN][FLAGS ? 1 : 0][UNI ? 1 : 0];
  if (cached == 0) {
    int nb = 0;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kLeanWarps * 32, smem));
    cached = nb > 0 ? nb : 1;
  }
  const unsigned need = (a.n_series + kLeanWarps - 1) / kLeanWarps;
  const unsigned cap = (unsigned)(c->num_sms * cached);
  const unsigned grid = need < cap ? need : cap;
  if (grid == 0) return B2P_OK;
  kern<<<grid, kLeanWarps * 32, smem, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

template <int FN, bool FLAGS>
int launch_lean(b2p_ctx* c, const RangeArgs& a) {
  if constexpr (kLeanUniform<FN, FLAGS>) {
    int rc = cadence_verdict(c, a);
    if (!rc && c->uniform_mode != 0) rc = launch_lean_variant<FN, FLAGS, true>(c, a);
    if (!rc && c->uniform_mode != 1) rc = launch_lean_variant<FN, FLAGS, false>(c, a);
    return rc;
  } else {
    return launch_lean_variant<FN, FLAGS, false>(c, a);
  }
}

// `with_flags`: the variant whose ring carries the reset / change bit words (always for resets() / changes(); for
// rate / increase when the adaptive policy picked it; never for the other functions).
template <int FN>
int launch_lean_if_supported(b2p_ctx* c, const RangeArgs& a, bool with_flags) {
  if constexpr (!LeanTraits<FN>::kSupported) {
    return fail(B2P_E_INVALID, "fn_id %d has no lean tier", FN);
  } else if constexpr (LeanTraits<FN>::kNeedsFlags) {
    return launch_lean<FN, true>(c, a);
  } else if constexpr (LeanTraits<FN>::kHasFlagsVariant) {
    return with_flags ? launch_lean<FN, true>(c, a) : launch_lean<FN, false>(c, a);
  } else {
    return launch_lean<FN, false>(c, a);
  }
}

// First tier of the fused by-label SUM: rate / increase / delta walk the series group by group and add into
// gsum / gcnt (range_lean_kernel<FN, FLAGS, GROUPED = true>).
template <int FN, bool FLAGS, bool UNI>
int launch_lean_grouped_variant(b2p_ctx* c, const RangeArgs& a) {
  constexpr size_t smem = lean_grouped_smem_bytes(UNI);
  auto kern = range_lean_kernel<FN, FLAGS, true, UNI>;
  static int cached_nb[16] = {};  // per device
  int& cached = cached_nb[c->device & 15];
  if (cached == 0) {
    int nb = 0;
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, kLeanWarps * 32, smem));
    cached = nb > 0 ? nb : 1;
  }
  const unsigned n_g = a.g_hi - a.g_lo;
  const unsigned need = (n_g + kLeanWarps - 1) / kLeanWarps;
  // The grid is one CTA per SM and takes its groups from a counter, so it can be any size: while tiles are being
  // all-reduced a few SMs are left to the collective's CTAs (they cannot be placed beside a resident 24-warp CTA).
  unsigned cap = (unsigned)(c->num_sms * cached);
  if (c->comm_reserve_now > 0 && cap > (unsigned)c->comm_reserve_now + 8u) cap -= (unsigned)c->comm_reserve_now;
  const unsigned grid = need < cap ? need : cap;
  if (grid == 0) return B2P_OK;
  kern<<<grid, kLeanWarps * 32, smem, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}
template <int FN, bool FLAGS>
int launch_lean_grouped(b2p_ctx* c, const RangeArgs& a) {
  if constexpr (kLeanUniform<FN, FLAGS>) {
    int rc = cadence_verdict(c, a);
    if (!rc && c->uniform_mode != 0) rc = launch_lean_grouped_variant<FN, FLAGS, true>(c, a);
    if (!rc && c->uniform_mode != 1) rc = launch_lean_grouped_variant<FN, FLAGS, false>(c, a);
    return rc;
  } else {
    return launch_lean_grouped_variant<FN, FLAGS, false>(c, a);
  }
}
bool lean_grouped_fn(int fn) { return fn == B2P_FN_RATE || fn == B2P_FN_INCREASE || fn == B2P_FN_DELTA; }
int dispatch_lean_grouped(b2p_ctx* c, int fn, const RangeArgs& a, bool with_flags) {
  switch (fn) {
    case B2P_FN_RATE: return with_flags ? launch_lean_grouped<B2P_FN_RATE, true>(c, a) : launch_lean_grouped<B2P_FN_RATE, false>(c, a);
    case B2P_FN_INCREASE: return with_flags ? launch_lean_grouped<B2P_FN_INCREASE, true>(c, a) : launch_lean_grouped<B2P_FN_INCREASE, false>(c, a);
    case B2P_FN_DELTA: return launch_lean_grouped<B2P_FN_DELTA, false>(c, a);
  }
  return fail(B2P_E_INVALID, "fn_id %d has no fused by-label tier", fn);
}

int dispatch_lean(b2p_ctx* c, int fn, const RangeArgs& a, bool with_flags) {
  switch (fn) {
#define X(N) case N: return launch_lean_if_supported<N>(c, a, with_flags);
    X(0) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19) X(20)
#undef X
  }
  return fail(B2P_E_INVALID, "unknown fn_id %d", fn);
}

template <int FN>
int launch_thread_tier(b2p_ctx* c, const RangeArgs& a) {
  const unsigned batches = (a.n_series + 31) / 32;
  const unsigned cap = (unsigned)c->num_sms * (unsigned)(220 * 1024 / (kTRing * 32 * 12 + 512));  // shared memory per 1-warp CTA
  const unsigned grid = batches < cap ? batches : cap;
  if (grid == 0) return B2P_OK;
  range_thread_kernel<FN><<<grid, 32, 0, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

template <int FN>
int launch_slow(b2p_ctx* c, const RangeArgs& a) {
  range_slow_kernel<FN><<<kSlowCtas, 128, 0, c->stream>>>(a);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

template <int FN>
int launch_udf(b2p_ctx* c, const int64_t* ts, const double* val, const int64_t* packed, const int64_t* eval_ts,
               uint64_t n_win, int64_t range_length, double p0, double p1, double* out, uint8_t* valid) {
  if (n_win == 0) return B2P_OK;
  uint64_t blocks = (n_win + 127) / 128;
  if (blocks > (uint64_t)c->num_sms * 32) blocks = (uint64_t)c->num_sms * 32;
  range_udf_kernel<FN><<<(unsigned)blocks, 128, 0, c->stream>>>(ts, val, packed, eval_ts, n_win, range_length, p0, p1,
                                                                 out, valid);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

#define B2P_FOR_EACH_FN(X) \
  X(0) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13) X(14) X(15) X(16) X(17) X(18) X(19) X(20)

int dispatch_fast(b2p_ctx* c, int fn, const RangeArgs& a) {
  switch (fn) {
#define X(N) case N: return launch_fast<N>(c, a);
    B2P_FOR_EACH_FN(X)
#undef X
  }
  return fail(B2P_E_INVALID, "unknown fn_id %d", fn);
}
int dispatch_big(b2p_ctx* c, int fn, const RangeArgs& a) {
  switch (fn) {
#define X(N) case N: return launch_big<N>(c, a);
    B2P_FOR_EACH_FN(X)
#undef X
  }
  return fail(B2P_E_INVALID, "unknown fn_id %d", fn);
}
int dispatch_slow(b2p_ctx* c, int fn, const RangeArgs& a) {
  switch (fn) {
#define X(N) case N: return launch_slow<N>(c, a);
    B2P_FOR_EACH_FN(X)
#undef X
  }
  return fail(B2P_E_INVALID, "unknown fn_id %d", fn);
}
int dispatch_udf(b2p_ctx* c, int fn, const int64_t* ts, const double* val, const int64_t* packed,
                 const int64_t* eval_ts, uint64_t n_win, int64_t range_length, double p0, double p1, double* out,
                 uint8_t* valid) {
  switch (fn) {
#define X(N) case N: return launch_udf<N>(c, ts, val, packed, eval_ts, n_win, range_length, p0, p1, out, valid);
    B2P_FOR_EACH_FN(X)
#undef X
  }
  return fail(B2P_E_INVALID, "unknown fn_id %d", fn);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_grid(const b2p_range_params* p, uint32_t n_series, int64_t* T_out) {
  if (!p) return fail(B2P_E_INVALID, "params is NULL");
  if (p->interval <= 0) return fail(B2P_E_INVALID, "interval must be > 0 (got %lld)", (long long)p->interval);
  if (p->range < 0) return fail(B2P_E_INVALID, "range must be >= 0");
  if (p->fn_id < 0 || p->fn_id >= B2P_FN__COUNT) return fail(B2P_E_INVALID, "unknown fn_id %d", p->fn_id);
  const int64_t T = b2p_num_steps(p->start, p->end, p->interval);
  if (T > (int64_t)0x7fffff00) return fail(B2P_E_TOO_LARGE, "%lld eval steps: trim [start,end] to the data extent first", (long long)T);
  if ((double)T * (double)n_series > 1.0e12) return fail(B2P_E_TOO_LARGE, "dense grid %lld x %u too large", (long long)T, n_series);
  *T_out = T;
  return B2P_OK;
}

int reset_status(b2p_ctx*) { return B2P_OK; }  // (every range call resets its own status slot; K0's verdict is sticky)

int ensure_slow_scratch(b2p_ctx* c, uint32_t n_series, int64_t T) {
  int rc;
  if ((rc = c->slow_list.ensure((size_t)(n_series ? n_series : 1) * 4))) return rc;
  if ((rc = c->w_list.ensure((size_t)(n_series ? n_series : 1) * 4))) return rc;
  if ((rc = c->b_list.ensure((size_t)(n_series ? n_series : 1) * 4))) return rc;
  if ((rc = c->win_scratch.ensure((size_t)kSlowWarps * (size_t)(T > 0 ? T : 1) * 8))) return rc;
  if (c->arena_rows == 0) {
    const size_t rows = c->arena_rows_wanted > kArenaDefaultRows ? c->arena_rows_wanted : kArenaDefaultRows;
    if ((rc = c->arena_ts.ensure(rows * 8))) return rc;
    if ((rc = c->arena_val.ensure(rows * 8))) return rc;
    c->arena_rows = rows;
  }
  return B2P_OK;
}

}  // namespace

extern "C" {

const char* b2p_last_error(void) { return g_err.c_str(); }
const char* b2p_version(void) { return "b200promql 0.1 (sm_100a)"; }

int64_t b2p_num_steps(int64_t start, int64_t end, int64_t interval) {
  if (interval <= 0 || end < start) return 0;
  return (end - start) / interval + 1;
}

b2p_ctx* b2p_create(int device) {
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    fail(B2P_E_CUDA, "no CUDA device: %s — libb200promql has no CPU fallback", cudaGetErrorString(e));
    cudaGetLastError();
    return nullptr;
  }
  if (device < 0 || device >= ndev) {
    fail(B2P_E_INVALID, "device %d out of range (have %d)", device, ndev);
    return nullptr;
  }
  b2p_ctx* c = new (std::nothrow) b2p_ctx();
  if (!c) {
    fail(B2P_E_NOMEM, "out of host memory");
    return nullptr;
  }
  c->device = device;
  DeviceGuard g(device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->num_sms = prop.multiProcessorCount;
  bool ok = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) == cudaSuccess;
  c->stream = c->own_stream;
  ok = ok && cudaMalloc(&c->d_ring, kStatusSlots * sizeof(Status)) == cudaSuccess;
  ok = ok && cudaMallocHost(&c->h_ring, kStatusSlots * sizeof(Status)) == cudaSuccess;
  ok = ok && cudaMalloc(&c->d_k0, sizeof(Status)) == cudaSuccess;
  ok = ok && cudaMallocHost(&c->h_k0, sizeof(Status)) == cudaSuccess;
  for (int i = 0; ok && i < 5; ++i)
    for (int j = 0; j < 2; ++j) ok = ok && cudaEventCreate(&c->ev[i][j]) == cudaSuccess;
  if (!ok) {
    fail(B2P_E_CUDA, "context creation failed: %s", cudaGetErrorString(cudaGetLastError()));
    b2p_destroy(c);
    return nullptr;
  }
  cudaMemset(c->d_ring, 0, kStatusSlots * sizeof(Status));
  cudaMemset(c->d_k0, 0, sizeof(Status));
  {
    double tab[kRcpTable];
    tab[0] = 0.0;
    for (int i = 1; i < kRcpTable; ++i) tab[i] = 1.0 / (double)i;
    if (cudaMemcpyToSymbol(c_rcp_table, tab, sizeof tab) != cudaSuccess) {
      fail(B2P_E_CUDA, "constant table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
      b2p_destroy(c);
      return nullptr;
    }
  }
  if (const char* e = getenv("B2P_ENABLE_THREAD_TIER")) c->thread_tier = (e[0] == '1');
  if (const char* e = getenv("B2P_DISABLE_LEAN_TIER")) c->lean_tier = !(e[0] == '1');
  if (const char* e = getenv("B2P_LEAN_ADAPTIVE")) c->lean_adaptive = !(e[0] == '0');
  if (const char* e = getenv("B2P_LEAN_FORCE_FLAGS")) c->lean_force_flags = (e[0] == '1');
  if (const char* e = getenv("B2P_HOST_TS_SCAN")) c->host_ts_scan = (e[0] != '0');
  if (const char* e = getenv("B2P_UNIFORM")) c->uniform_mode = (e[0] == '0') ? 0 : (e[0] == '1' ? 1 : -1);
  if (const char* e = getenv("B2P_COMM_RESERVE_SMS")) c->comm_reserve_sms = atoi(e);
  if (const char* e = getenv("B2P_COMM_HEADSTART_US")) c->comm_headstart_cycles = (long long)(atof(e) * 1965.0);
  if (const char* e = getenv("B2P_ARENA_ROWS")) c->arena_rows_wanted = (size_t)strtoull(e, nullptr, 10);
  return c;
}

void b2p_destroy(b2p_ctx* c) {
  if (!c) return;
  DeviceGuard g(c->device);
  if (c->own_stream) cudaStreamSynchronize(c->own_stream);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  if (c->s_comm) cudaStreamDestroy(c->s_comm);
  if (c->ev_comm_in) cudaEventDestroy(c->ev_comm_in);
  if (c->ev_comm_done) cudaEventDestroy(c->ev_comm_done);
  if (c->ev_comm_go) cudaEventDestroy(c->ev_comm_go);
  for (DevBuf* b : {&c->w_skip, &c->b_skip, &c->slow_skip, &c->m_tmp0, &c->m_tmp1, &c->hq_off, &c->hq_series, &c->hq_les}) b->release();
  for (DevBuf* b : {&c->slow_list, &c->w_list, &c->b_list, &c->arena_ts, &c->arena_val, &c->win_scratch, &c->h_ts, &c->h_val, &c->h_sid,
                    &c->h_off, &c->h_out, &c->h_valid, &c->h_aux0, &c->h_aux1, &c->h_aux2, &c->h_aux3,
                    &c->g_keys_in, &c->g_keys_out, &c->g_vals_in, &c->g_vals_out, &c->g_goff, &c->g_tmp, &c->c_psum,
                    &c->c_pcnt})
    b->release();
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 2; ++j)
      if (c->ev[i][j]) cudaEventDestroy(c->ev[i][j]);
  for (int i = 0; i < 2; ++i) {
    for (DevBuf* b : {&c->p_ts[i], &c->p_val[i], &c->p_sid[i], &c->p_off[i], &c->p_out[i], &c->p_valid[i]}) b->release();
    if (c->ev_h2d[i]) cudaEventDestroy(c->ev_h2d[i]);
    if (c->ev_comp[i]) cudaEventDestroy(c->ev_comp[i]);
    if (c->ev_d2h[i]) cudaEventDestroy(c->ev_d2h[i]);
  }
  c->p_status.release();
  if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
  if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
  if (c->d_ring) cudaFree(c->d_ring);
  if (c->h_ring) cudaFreeHost(c->h_ring);
  if (c->d_k0) cudaFree(c->d_k0);
  if (c->h_k0) cudaFreeHost(c->h_k0);
  if (c->own_stream) cudaStreamDestroy(c->own_stream);
  delete c;
}

int b2p_set_stream(b2p_ctx* c, void* cuda_stream) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);  // NULL == the legacy default stream
  return B2P_OK;
}

int b2p_use_own_stream(b2p_ctx* c) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  c->stream = c->own_stream;
  return B2P_OK;
}

int64_t b2p_last_slow_series(b2p_ctx* c) { return c ? c->last_slow : -1; }
int64_t b2p_last_h2d_bytes(b2p_ctx* c) { return c ? c->last_h2d_bytes : -1; }
int64_t b2p_last_warp_tier_series(b2p_ctx* c) { return c ? c->last_w : -1; }
int64_t b2p_launch_count(b2p_ctx* c) { return c ? c->launches : -1; }

double b2p_last_kernel_ms(b2p_ctx* c, int stage) {
  if (!c || stage < 0 || stage >= 5 || !c->ev_used[stage]) return -1.0;
  DeviceGuard g(c->device);
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, c->ev[stage][0], c->ev[stage][1]) != cudaSuccess) {
    cudaGetLastError();
    return -1.0;
  }
  return (double)ms;
}

__global__ void comm_marker_kernel() {}
// holds the compute stream back for a few microseconds so that the all-reduce released at the same instant on the
// communication stream has its CTAs placed before the persistent range kernel asks for every SM
__global__ void comm_headstart_kernel(long long cycles) {
  const long long t0 = clock64();
  while (clock64() - t0 < cycles) {}
}

// Launches every tier of one range call (first tier when `used_lean`/`thread_tier`, warp-per-series kernel, its
// long-window instantiation, exact slow kernel) on the context's stream.
static int launch_range_tiers(b2p_ctx* c, int fn, RangeArgs a, bool thread_tier, bool used_lean, int lean_mode,
                              bool later_tile = false) {
  int rc;
  if (!later_tile) {
    CU(cudaMemsetAsync(a.status, 0, sizeof(Status), c->stream));
  } else {  // a further tile of the same fused call: new work lists, same verdict (overflow / arena fields stay)
    CU(cudaMemsetAsync(&a.status->slow_count, 0, sizeof(uint32_t), c->stream));
    CU(cudaMemsetAsync(&a.status->w_count, 0, 3 * sizeof(uint32_t), c->stream));  // w_count, b_count, g_next
  }
  stage_begin(c, 1);
  if (thread_tier) {
    if (fn == B2P_FN_RATE) rc = launch_thread_tier<B2P_FN_RATE>(c, a);
    else if (fn == B2P_FN_INCREASE) rc = launch_thread_tier<B2P_FN_INCREASE>(c, a);
    else rc = launch_thread_tier<B2P_FN_DELTA>(c, a);
    if (rc) return rc;
    a.use_w_list = 1;
  } else if (used_lean) {
    if ((rc = a.gsum ? dispatch_lean_grouped(c, fn, a, lean_mode == 1) : dispatch_lean(c, fn, a, lean_mode == 1))) return rc;
    a.use_w_list = 1;
  }
  rc = dispatch_fast(c, fn, a);
  if (!rc && a.b_list) rc = dispatch_big(c, fn, a);
  stage_end(c, 1);
  if (rc) return rc;
  stage_begin(c, 2);
  rc = dispatch_slow(c, fn, a);
  stage_end(c, 2);
  return rc;
}

int b2p_sync(b2p_ctx* c) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  DeviceGuard g(c->device);
  for (int attempt = 0; attempt < 4; ++attempt) {
    CU(cudaMemcpyAsync(c->h_ring, c->d_ring, kStatusSlots * sizeof(Status), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(c->h_k0, c->d_k0, sizeof(Status), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const uint32_t k0 = c->h_k0->k0_errors;
    if (k0) {
      CU(cudaMemsetAsync(c->d_k0, 0, sizeof(Status), c->stream));
      c->pending.clear();
      if (k0 & 1u) return fail(B2P_E_UNSORTED, "series-id column is not non-decreasing");
      return fail(B2P_E_UNSORTED, "series id >= n_series");
    }
    // verdicts of the outstanding range calls, oldest first; a call whose slow path ran out of arena is redone
    // as a whole (all tiers, same modes) after the arena has grown to what the largest of them needs
    size_t need = 0;
    std::vector<b2p_ctx::Pending> redo;
    for (auto& pc : c->pending) {
      const Status st = c->h_ring[pc.slot];
      c->last_slow = st.slow_count;
      c->last_w = st.w_count;
      if (pc.used_lean && !pc.verdict_taken) {
        c->last_lean_mode = pc.lean_mode;
        lean_verdict(c, pc.fn, st.w_count, pc.n_series);
        pc.verdict_taken = true;
      }
      if (st.arena_overflow) {
        if ((size_t)st.arena_needed + 1024 > need) need = (size_t)st.arena_needed + 1024;
        redo.push_back(pc);
      }
    }
    c->pending.clear();
    c->fused_pending = false;
    if (redo.empty()) return B2P_OK;
    int rc;
    if ((rc = c->arena_ts.ensure(need * 8))) return rc;
    if ((rc = c->arena_val.ensure(need * 8))) return rc;
    c->arena_rows = need;
    for (auto& pc : redo) {
      pc.args.arena_ts = c->arena_ts.as<int64_t>();
      pc.args.arena_val = c->arena_val.as<double>();
      pc.args.arena_cap = need;
      if (pc.merged)
        return fail(B2P_E_TOO_LARGE, "a series of %llu+ rows needs the exact slow path but does not fit its arena region; "
                    "the merged partials are incomplete — set B2P_ARENA_ROWS >= %zu and repeat the query",
                    (unsigned long long)(need / (size_t)kSlowWarps), need);
      if (pc.fused) {
        // partials were added in place: only the slow kernel runs again, over its intact work list (a series that
        // did not fit the arena added nothing); no other range call was admitted while this one was outstanding
        Status patch = c->h_ring[pc.slot];
        patch.arena_overflow = 0; patch.arena_used = 0; patch.arena_needed = 0;
        c->h_ring[pc.slot] = patch;
        CU(cudaMemcpyAsync(c->d_ring + pc.slot, c->h_ring + pc.slot, sizeof(Status), cudaMemcpyHostToDevice, c->stream));
        if ((rc = dispatch_slow(c, pc.fn, pc.args))) return rc;
        c->pending.push_back(pc);
        CU(cudaStreamSynchronize(c->stream));
        continue;
      }
      if ((rc = launch_range_tiers(c, pc.fn, pc.args, pc.thread_tier, pc.used_lean, pc.lean_mode))) return rc;
      c->pending.push_back(pc);
      CU(cudaStreamSynchronize(c->stream));  // one redone call at a time: they share the arena from offset 0
    }
  }
  return fail(B2P_E_NOMEM, "slow-path arena could not be sized");
}

/* ---- device-pointer API ---------------------------------------------------------------------- */

static int series_offsets_impl(b2p_ctx* c, const uint32_t* sid, uint64_t n_rows, uint32_t n_series, uint32_t sid_base,
                               uint64_t* offsets);

int b2p_series_offsets_dev(b2p_ctx* c, const uint32_t* sid, uint64_t n_rows, uint32_t n_series, uint64_t* offsets) {
  return series_offsets_impl(c, sid, n_rows, n_series, 0u, offsets);
}

static int series_offsets_impl(b2p_ctx* c, const uint32_t* sid, uint64_t n_rows, uint32_t n_series, uint32_t sid_base,
                               uint64_t* offsets) {
  if (!c || !offsets || (!sid && n_rows)) return fail(B2P_E_INVALID, "NULL argument");
  if (!aligned16(sid)) return fail(B2P_E_INVALID, "sid must be 16-byte aligned");
  DeviceGuard g(c->device);
  uint64_t blocks = (n_rows / 16 + 255) / 256;
  const uint64_t cap = (uint64_t)c->num_sms * 16;
  if (blocks > cap) blocks = cap;
  if (blocks == 0) blocks = 1;
  stage_begin(c, 0);
  series_offsets_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(sid, n_rows, n_series, sid_base, offsets, c->d_k0);
  c->launches++;
  stage_end(c, 0);
  CU(cudaGetLastError());
  return B2P_OK;
}

// Target of a fused by-label SUM / COUNT (b2p_range_group_sum*_dev): groups [g_lo, g_hi) of an index.
struct GroupTarget {
  const b2p_group_index* idx;
  uint32_t g_lo, g_hi;
  double* gsum;
  uint32_t* gcnt;
  // > 0: the group range is processed in this many tiles and every tile's rows of gsum / gcnt are all-reduced over
  // the context's communicator as soon as the tile is complete, on the (high-priority) communication stream, while
  // the next tile computes
  int allreduce_tiles;
};

// Can this range call add its results straight into by-label partials?  (first tier available for the function and
// the query shape, and not switched off by the adaptive policy; groups balanced enough for group-exclusive warps)
static bool fused_group_ok(b2p_ctx* c, const b2p_range_params* p, int64_t T, const b2p_group_index* idx) {
  if (!lean_grouped_fn(p->fn_id) || c->thread_tier) return false;
  if (T > 32 * (int64_t)kLeanFullWords) return false;  // per-warp word counters of the first tier
  RangeArgs a{};
  a.start = p->start; a.end = p->end; a.interval = p->interval; a.range = p->range;
  a.T = T;
  a.rcp_rs = 1.0;
  if (fits_ts32(a)) a.rel_max = (uint32_t)(p->range + (T - 1) * p->interval + 1);
  {
    const double rs = (double)p->range / 1000.0;
    uint64_t bits;
    memcpy(&bits, &rs, 8);
    if (p->range <= 0 || (bits & 0x000fffffffffffffull) == 0x000fffffffffffffull) a.rcp_rs = 0.0;
  }
  if (!lean_ok(c, p->fn_id, a)) return false;
  if (c->lean_backoff[p->fn_id] > 0 && c->lean_mode[p->fn_id] == 2) return false;
  // a group is walked by ONE warp: the largest group may not exceed a few times a warp's fair share
  const uint64_t warps = (uint64_t)c->num_sms * B2P_LEAN_MIN_BLOCKS * kLeanWarps;
  const uint64_t share = idx->n_series / warps + 1;
  return (uint64_t)idx->max_members <= 8 * share + 64;
}

static int range_call(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                      const uint64_t* offsets, uint64_t n_rows, uint32_t n_series, double* out, uint32_t* valid_words,
                      const GroupTarget* gt);

int b2p_range_eval_dev(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                       const uint64_t* offsets, uint64_t n_rows, uint32_t n_series, double* out,
                       uint32_t* valid_words) {
  return range_call(c, p, ts, val, offsets, n_rows, n_series, out, valid_words, nullptr);
}

static int range_call(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                      const uint64_t* offsets, uint64_t n_rows, uint32_t n_series, double* out, uint32_t* valid_words,
                      const GroupTarget* gt) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  int64_t T = 0;
  int rc = check_grid(p, n_series, &T);
  if (rc) return rc;
  if (n_series == 0 || T == 0) return B2P_OK;
  if (!offsets || (!gt && (!out || !valid_words)) || ((!ts || !val) && n_rows)) return fail(B2P_E_INVALID, "NULL argument");
  if (!aligned16(ts) || !aligned16(val)) return fail(B2P_E_INVALID, "ts/val must be 16-byte aligned");
  DeviceGuard g(c->device);
  if ((rc = ensure_slow_scratch(c, n_series, T))) return rc;
  RangeArgs a{};
  a.start = p->start; a.end = p->end; a.interval = p->interval; a.range = p->range; a.offset = p->offset;
  a.p0 = p->param0; a.p1 = p->param1; a.filter_nan = p->filter_nan;
  a.T = T; a.Tw = (uint32_t)((T + 31) / 32);
  a.tb = p->start - p->range;
  a.rel_max = 0;
  if (fits_ts32(a)) a.rel_max = (uint32_t)(p->range + (T - 1) * p->interval + 1);
  {
    // exact two-FMA division by range/1000 needs RN(1/b) and a significand that is not all ones
    const double rs = (double)p->range / 1000.0;
    uint64_t bits;
    memcpy(&bits, &rs, 8);
    const bool all_ones = (bits & 0x000fffffffffffffull) == 0x000fffffffffffffull;
    a.rcp_rs = (p->range > 0 && !all_ones) ? 1.0 / rs : 0.0;
    a.range_secs = rs;
    a.rcp_interval = 1.0 / (double)p->interval;
    a.start_mod = p->start >= 0 ? (uint32_t)(p->start % p->interval) : 0u;
  }
  a.ts = ts; a.val = val; a.offsets = offsets; a.n_rows = n_rows; a.n_series = n_series;
  a.out = out; a.valid = valid_words;
  // a fused call keeps the work lists until its verdict is in: nothing else is admitted before that
  if (c->fused_pending && (rc = b2p_sync(c))) return rc;
  if (gt) {
    if (!c->pending.empty() && (rc = b2p_sync(c))) return rc;
    const size_t ns = n_series;
    if ((rc = c->w_skip.ensure(ns * 4)) || (rc = c->b_skip.ensure(ns * 4)) || (rc = c->slow_skip.ensure(ns * 4))) return rc;
    a.gsum = gt->gsum; a.gcnt = gt->gcnt; a.gid = gt->idx->gid; a.g_off = gt->idx->goff; a.g_members = gt->idx->members;
    a.n_groups = gt->idx->n_groups; a.g_lo = gt->g_lo; a.g_hi = gt->g_hi;
    a.w_skip = c->w_skip.as<uint32_t>(); a.b_skip = c->b_skip.as<uint32_t>(); a.slow_skip = c->slow_skip.as<uint32_t>();
  }
  // every call owns a status slot until b2p_sync has read it; with all slots taken the library synchronises itself
  if ((int)c->pending.size() >= kStatusSlots && (rc = b2p_sync(c))) return rc;
  const int slot = c->next_slot;
  c->next_slot = (c->next_slot + 1) % kStatusSlots;
  a.status = c->d_ring + slot; a.slow_list = c->slow_list.as<uint32_t>();
  a.w_list = c->w_list.as<uint32_t>();
  a.b_list = fits_ts32(a) ? c->b_list.as<uint32_t>() : nullptr;  // long windows: the 1024-sample ring (32-bit domain)
  a.use_w_list = 0;
  a.arena_ts = c->arena_ts.as<int64_t>(); a.arena_val = c->arena_val.as<double>(); a.arena_cap = c->arena_rows;
  a.win_scratch = c->win_scratch.as<unsigned long long>();
  // tier 1 (rate / increase / delta, 32-bit time domain): thread per series (opt-in) or the lean warp-per-series
  // kernel; what it declines goes to tier 2 (warp per series) through w_list, long windows from there to the
  // 1024-sample instantiation through b_list, and what that declines to the exact slow kernel
  const bool tier1 = c->thread_tier && fits_ts32(a) &&
                     (p->fn_id == B2P_FN_RATE || p->fn_id == B2P_FN_INCREASE || p->fn_id == B2P_FN_DELTA);
  bool used_lean = false;
  int mode = 0;
  if (!tier1 && lean_ok(c, p->fn_id, a)) {
    if (c->lean_backoff[p->fn_id] > 0) {
      c->lean_backoff[p->fn_id]--;
      mode = c->lean_mode[p->fn_id];
    }
    if (mode != 2) used_lean = true;
    if (mode == 0 && c->lean_force_flags) mode = 1;
  }
  if (gt && !used_lean) return fail(B2P_E_INVALID, "fused by-label call without its first tier (internal)");
  c->last_lean_mode = mode;
  c->last_used_lean = used_lean;
  c->last_range_series = n_series;
  c->last_range_fn = p->fn_id;
  if (gt && gt->allreduce_tiles > 0) {
    if (!c->comm && c->comm_ranks > 1) return fail(B2P_E_INVALID, "no communicator: call b2p_comm_init first");
    const uint32_t n_t = (uint32_t)gt->allreduce_tiles;
    const uint64_t span = (uint64_t)gt->g_hi - gt->g_lo;
    c->comm_reserve_now = (c->comm && n_t > 1) ? c->comm_reserve_sms : 0;
    for (uint32_t t = 0; t < n_t; ++t) {
      a.g_lo = gt->g_lo + (uint32_t)(span * t / n_t);
      a.g_hi = gt->g_lo + (uint32_t)(span * (t + 1) / n_t);
      if (a.g_hi == a.g_lo) continue;
      if ((rc = launch_range_tiers(c, p->fn_id, a, tier1, used_lean, mode, t > 0))) return rc;
      if (c->comm) {
        const size_t off = (size_t)a.g_lo * (size_t)T, cnt_n = (size_t)(a.g_hi - a.g_lo) * (size_t)T;
        CU(cudaEventRecord(c->ev_comm_in, c->stream));
        CU(cudaStreamWaitEvent(c->s_comm, c->ev_comm_in, 0));
        // The next tile's kernels are released by a marker that sits directly IN FRONT of the all-reduce on the
        // communication stream: when they become runnable the (few) NCCL CTAs are already next in line on the
        // high-priority stream and get their SMs first; the persistent first-tier kernel fills what is left and its
        // dynamic group counter keeps late CTAs from becoming a tail.
        comm_marker_kernel<<<1, 32, 0, c->s_comm>>>();
        CU(cudaEventRecord(c->ev_comm_go, c->s_comm));
        CU(cudaStreamWaitEvent(c->stream, c->ev_comm_go, 0));
        if (c->comm_headstart_cycles > 0) comm_headstart_kernel<<<1, 32, 0, c->stream>>>(c->comm_headstart_cycles);
        stage_begin_on(c, 4, c->s_comm);
        NCCL_TRY(g_nccl.GroupStart());
        NCCL_TRY(g_nccl.AllReduce(a.gsum + off, a.gsum + off, cnt_n, Nccl::kFloat64, Nccl::kSum, c->comm, c->s_comm));
        NCCL_TRY(g_nccl.AllReduce(a.gcnt + off, a.gcnt + off, cnt_n, Nccl::kUint32, Nccl::kSum, c->comm, c->s_comm));
        NCCL_TRY(g_nccl.GroupEnd());
        stage_end_on(c, 4, c->s_comm);
      }
    }
    c->comm_reserve_now = 0;
    if (c->comm) {  // everything after this call on the context's stream sees the merged partials
      CU(cudaEventRecord(c->ev_comm_done, c->s_comm));
      CU(cudaStreamWaitEvent(c->stream, c->ev_comm_done, 0));
    }
    a.g_lo = gt->g_lo; a.g_hi = gt->g_hi;
  } else if ((rc = launch_range_tiers(c, p->fn_id, a, tier1, used_lean, mode))) {
    return rc;
  }
  b2p_ctx::Pending pc{};
  pc.slot = slot; pc.fn = p->fn_id; pc.args = a; pc.lean_mode = mode; pc.thread_tier = tier1; pc.used_lean = used_lean;
  pc.n_series = n_series; pc.verdict_taken = false; pc.fused = gt != nullptr;
  pc.merged = gt && gt->allreduce_tiles > 0;
  c->pending.push_back(pc);
  if (gt) c->fused_pending = true;
  return B2P_OK;
}

int b2p_range_udf_dev(b2p_ctx* c, int32_t fn_id, const int64_t* ts, const double* val, uint64_t n_rows,
                      const int64_t* packed_ranges, const int64_t* eval_ts, uint64_t n_win, int64_t range_length,
                      double param0, double param1, double* out, uint8_t* valid) {
  (void)n_rows;
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_win == 0) return B2P_OK;
  if (!packed_ranges || !out || !valid) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  stage_begin(c, 1);
  int rc = dispatch_udf(c, fn_id, ts, val, packed_ranges, eval_ts, n_win, range_length, param0, param1, out, valid);
  stage_end(c, 1);
  return rc;
}

int b2p_instant_select_dev(b2p_ctx* c, int64_t start, int64_t end, int64_t interval, int64_t lookback, int64_t offset,
                           const int64_t* ts, const double* val, const uint64_t* offsets, uint64_t n_rows,
                           uint32_t n_series, double* out, uint32_t* valid_words) {
  (void)n_rows;
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  b2p_range_params p{};
  p.start = start; p.end = end; p.interval = interval; p.range = lookback;
  int64_t T = 0;
  int rc = check_grid(&p, n_series, &T);
  if (rc) return rc;
  if (n_series == 0 || T == 0) return B2P_OK;
  if (!offsets || !out || !valid_words) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  InstantArgs a{};
  a.start = start; a.end = end; a.interval = interval; a.lookback = lookback; a.offset = offset;
  a.T = T; a.Tw = (uint32_t)((T + 31) / 32);
  a.ts = ts; a.val = val; a.offsets = offsets; a.n_series = n_series; a.out = out; a.valid = valid_words;
  unsigned need = (n_series + kWarpsPerCta - 1) / kWarpsPerCta;
  unsigned cap = (unsigned)c->num_sms * 8;
  stage_begin(c, 1);
  instant_kernel<<<need < cap ? need : cap, kWarpsPerCta * 32, 0, c->stream>>>(a);
  c->launches++;
  stage_end(c, 1);
  CU(cudaGetLastError());
  return B2P_OK;
}

namespace {
// group -> member series CSR: stable radix sort of (gid, series index), then lower bounds per group
int build_group_csr(b2p_ctx* c, const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint32_t* goff,
                    uint32_t* members) {
  int rc;
  const size_t ns = n_series ? n_series : 1;
  if ((rc = c->g_vals_in.ensure(ns * 4))) return rc;
  if ((rc = c->g_keys_out.ensure(ns * 4))) return rc;
  iota_kernel<<<(unsigned)((ns + 255) / 256 < 1024 ? (ns + 255) / 256 : 1024), 256, 0, c->stream>>>(
      c->g_vals_in.as<uint32_t>(), n_series);
  c->launches++;
  size_t tmp_bytes = 0;
  CU(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, gid, c->g_keys_out.as<uint32_t>(), c->g_vals_in.as<uint32_t>(),
                                     members, (int)n_series, 0, 32, c->stream));
  if ((rc = c->g_tmp.ensure(tmp_bytes ? tmp_bytes : 16))) return rc;
  if (n_series > 0)
    CU(cub::DeviceRadixSort::SortPairs(c->g_tmp.p, tmp_bytes, gid, c->g_keys_out.as<uint32_t>(),
                                       c->g_vals_in.as<uint32_t>(), members, (int)n_series, 0, 32, c->stream));
  group_offsets_kernel<<<(n_groups + 1 + 255) / 256, 256, 0, c->stream>>>(c->g_keys_out.as<uint32_t>(), n_series,
                                                                          n_groups, goff);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

// accumulate = 1 (SUM / COUNT partials only): out_val / out_cnt are added to instead of overwritten
int group_aggregate_csr(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words, const uint32_t* goff,
                        const uint32_t* members, uint32_t n_groups, uint64_t T, double* out_val, uint32_t* out_cnt,
                        int accumulate, double* out_mean = nullptr) {
  GroupArgs a{};
  a.out_mean = out_mean;
  a.agg = agg; a.vals = vals; a.valid = valid_words; a.goff = goff;
  a.members = members; a.n_groups = n_groups; a.T = T; a.Tw = (uint32_t)((T + 31) / 32);
  a.out_val = out_val; a.out_cnt = out_cnt; a.accumulate = accumulate;
  const uint64_t warps = (uint64_t)n_groups * ((T + 31) / 32);
  uint64_t blocks = (warps + 7) / 8;
  const uint64_t cap = (uint64_t)c->num_sms * 32;
  if (blocks > cap) blocks = cap;
  switch (agg) {
    case B2P_AGG_SUM: group_aggregate_kernel<B2P_AGG_SUM><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    case B2P_AGG_AVG: group_aggregate_kernel<B2P_AGG_AVG><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    case B2P_AGG_COUNT: group_aggregate_kernel<B2P_AGG_COUNT><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    case B2P_AGG_MIN: group_aggregate_kernel<B2P_AGG_MIN><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    case B2P_AGG_MAX: group_aggregate_kernel<B2P_AGG_MAX><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    case B2P_AGG_STDVAR: group_aggregate_kernel<B2P_AGG_STDVAR><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
    default: group_aggregate_kernel<B2P_AGG_STDDEV><<<(unsigned)blocks, 256, 0, c->stream>>>(a); break;
  }
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

int group_aggregate_impl(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words, const uint32_t* gid,
                         uint32_t n_series, uint32_t n_groups, uint64_t T, double* out_val, uint32_t* out_cnt,
                         int accumulate, double* out_mean = nullptr) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (agg < 0 || agg > B2P_AGG_STDVAR) return fail(B2P_E_INVALID, "unknown aggregator %d", agg);
  if (n_groups == 0 || T == 0) return B2P_OK;
  if (!vals || !valid_words || !gid || !out_val || !out_cnt) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  int rc;
  const size_t ns = n_series ? n_series : 1;
  if ((rc = c->g_vals_out.ensure(ns * 4))) return rc;
  if ((rc = c->g_goff.ensure(((size_t)n_groups + 1) * 4))) return rc;
  stage_begin(c, 3);
  if ((rc = build_group_csr(c, gid, n_series, n_groups, c->g_goff.as<uint32_t>(), c->g_vals_out.as<uint32_t>()))) return rc;
  rc = group_aggregate_csr(c, agg, vals, valid_words, c->g_goff.as<uint32_t>(), c->g_vals_out.as<uint32_t>(), n_groups, T,
                           out_val, out_cnt, accumulate, out_mean);
  stage_end(c, 3);
  return rc;
}
}  // namespace

int b2p_group_aggregate_dev(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words,
                            const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint64_t T, double* out_val,
                            uint32_t* out_cnt) {
  return group_aggregate_impl(c, agg, vals, valid_words, gid, n_series, n_groups, T, out_val, out_cnt, 0);
}

int b2p_group_aggregate_partial_dev(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words,
                                    const uint32_t* gid, uint32_t n_series, uint32_t n_groups, uint64_t T,
                                    double* out_val, uint32_t* out_cnt, double* out_mean) {
  const bool var = agg == B2P_AGG_STDDEV || agg == B2P_AGG_STDVAR;
  if (var && !out_mean) return fail(B2P_E_INVALID, "stddev / stdvar partials need out_mean");
  if (agg == B2P_AGG_AVG) agg = B2P_AGG_SUM;  // the partial of an average is (sum, count)
  return group_aggregate_impl(c, agg, vals, valid_words, gid, n_series, n_groups, T, out_val, out_cnt, 0,
                              var ? out_mean : nullptr);
}

int b2p_group_index_create_dev(b2p_ctx* c, const uint32_t* gid, uint32_t n_series, uint32_t n_groups,
                               b2p_group_index** out_index) {
  if (!c || !out_index || (!gid && n_series)) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  b2p_group_index* ix = new (std::nothrow) b2p_group_index();
  if (!ix) return fail(B2P_E_NOMEM, "out of host memory");
  ix->n_series = n_series; ix->n_groups = n_groups;
  const size_t ns = n_series ? n_series : 1;
  bool ok = cudaMalloc(&ix->gid, ns * 4) == cudaSuccess && cudaMalloc(&ix->members, ns * 4) == cudaSuccess &&
            cudaMalloc(&ix->goff, ((size_t)n_groups + 1) * 4) == cudaSuccess;
  int rc = ok ? B2P_OK : fail(B2P_E_NOMEM, "cudaMalloc failed for the group index");
  if (!rc && n_series) {
    cudaMemcpyAsync(ix->gid, gid, (size_t)n_series * 4, cudaMemcpyDeviceToDevice, c->stream);
    rc = build_group_csr(c, ix->gid, n_series, n_groups, ix->goff, ix->members);
  }
  if (!rc) {
    // largest group (host-side scan of the offsets: the index is built once per label assignment)
    std::vector<uint32_t> h((size_t)n_groups + 1);
    cudaError_t e = cudaMemcpyAsync(h.data(), ix->goff, h.size() * 4, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) rc = fail(B2P_E_CUDA, "group index read-back: %s", cudaGetErrorString(e));
    for (uint32_t i = 0; !rc && i < n_groups; ++i)
      if (h[i + 1] - h[i] > ix->max_members) ix->max_members = h[i + 1] - h[i];
  }
  if (rc) {
    b2p_group_index_destroy(c, ix);
    return rc;
  }
  *out_index = ix;
  return B2P_OK;
}

void b2p_group_index_destroy(b2p_ctx* c, b2p_group_index* ix) {
  if (!ix) return;
  if (c) {
    DeviceGuard g(c->device);
    cudaStreamSynchronize(c->stream);
    if (ix->gid) cudaFree(ix->gid);
    if (ix->goff) cudaFree(ix->goff);
    if (ix->members) cudaFree(ix->members);
  }
  delete ix;
}

int b2p_group_aggregate_indexed_dev(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words,
                                    const b2p_group_index* ix, uint64_t T, double* out_val, uint32_t* out_cnt) {
  if (!c || !ix) return fail(B2P_E_INVALID, "NULL argument");
  if (agg < 0 || agg > B2P_AGG_STDVAR) return fail(B2P_E_INVALID, "unknown aggregator %d", agg);
  if (ix->n_groups == 0 || T == 0) return B2P_OK;
  if (!vals || !valid_words || !out_val || !out_cnt) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  stage_begin(c, 3);
  int rc = group_aggregate_csr(c, agg, vals, valid_words, ix->goff, ix->members, ix->n_groups, T, out_val, out_cnt, 0);
  stage_end(c, 3);
  return rc;
}

// sum by (..)(fn(..)) partials of groups [g_lo, g_hi) added into out_sum / out_cnt [n_groups x T].
// Fused (no [n_series x T] intermediate) for rate / increase / delta whenever the first tier applies; otherwise the
// range function is evaluated into context scratch and folded by the by-label kernel (two passes, synchronous).
int b2p_range_group_sum_indexed_dev(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                                    const uint64_t* offsets, uint64_t n_rows, uint32_t n_series,
                                    const b2p_group_index* ix, uint32_t g_lo, uint32_t g_hi, double* out_sum,
                                    uint32_t* out_cnt) {
  if (!c || !ix) return fail(B2P_E_INVALID, "NULL argument");
  if (ix->n_series != n_series) return fail(B2P_E_INVALID, "group index was built for %u series, call has %u", ix->n_series, n_series);
  if (g_hi > ix->n_groups) g_hi = ix->n_groups;
  int64_t T = 0;
  int rc = check_grid(p, n_series, &T);
  if (rc) return rc;
  if (n_series == 0 || T == 0 || g_lo >= g_hi) return B2P_OK;
  if (!out_sum || !out_cnt) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  if (fused_group_ok(c, p, T, ix)) {
    GroupTarget gt{ix, g_lo, g_hi, out_sum, out_cnt, 0};
    return range_call(c, p, ts, val, offsets, n_rows, n_series, nullptr, nullptr, &gt);
  }
  if (g_lo != 0 || g_hi != ix->n_groups)
    return fail(B2P_E_INVALID, "group ranges need the fused tier (rate / increase / delta in the 32-bit time domain)");
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  if ((rc = c->h_aux0.ensure((size_t)n_series * (size_t)T * 8))) return rc;
  if ((rc = c->h_aux1.ensure((size_t)n_series * Tw * 4))) return rc;
  if ((rc = b2p_range_eval_dev(c, p, ts, val, offsets, n_rows, n_series, c->h_aux0.as<double>(),
                               c->h_aux1.as<uint32_t>())))
    return rc;
  if ((rc = b2p_sync(c))) return rc;  // slow-path fix-ups must land before the aggregate reads
  stage_begin(c, 3);
  rc = group_aggregate_csr(c, B2P_AGG_SUM, c->h_aux0.as<double>(), c->h_aux1.as<uint32_t>(), ix->goff, ix->members,
                           ix->n_groups, (uint64_t)T, out_sum, out_cnt, 1);
  stage_end(c, 3);
  return rc;
}

// sum by over all ranks: the fused partials of this rank's series, tile by tile, each tile all-reduced over the
// communicator while the next one computes.  Falls back to partials + one all-reduce when the call cannot run fused.
int b2p_range_group_sum_allreduce_dev(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                                      const uint64_t* offsets, uint64_t n_rows, uint32_t n_series,
                                      const b2p_group_index* ix, int32_t n_tiles, double* out_sum, uint32_t* out_cnt) {
  if (!c || !ix) return fail(B2P_E_INVALID, "NULL argument");
  if (ix->n_series != n_series) return fail(B2P_E_INVALID, "group index was built for %u series, call has %u", ix->n_series, n_series);
  int64_t T = 0;
  int rc = check_grid(p, n_series, &T);
  if (rc) return rc;
  if (T == 0 || ix->n_groups == 0) return B2P_OK;
  if (!out_sum || !out_cnt) return fail(B2P_E_INVALID, "NULL argument");
  if (n_tiles < 1) n_tiles = 1;
  DeviceGuard g(c->device);
  if (n_series > 0 && fused_group_ok(c, p, T, ix)) {
    GroupTarget gt{ix, 0, ix->n_groups, out_sum, out_cnt, n_tiles};
    return range_call(c, p, ts, val, offsets, n_rows, n_series, nullptr, nullptr, &gt);
  }
  if (n_series > 0 &&
      (rc = b2p_range_group_sum_indexed_dev(c, p, ts, val, offsets, n_rows, n_series, ix, 0, ix->n_groups, out_sum, out_cnt)))
    return rc;
  return b2p_allreduce_partials_dev(c, B2P_AGG_SUM, out_sum, out_cnt, nullptr, (uint64_t)ix->n_groups * (uint64_t)T);
}

int b2p_range_group_sum_fused(b2p_ctx* c, const b2p_range_params* p, const b2p_group_index* ix) {
  if (!c || !ix || !p) return 0;
  int64_t T = b2p_num_steps(p->start, p->end, p->interval);
  return fused_group_ok(c, p, T, ix) ? 1 : 0;
}

int b2p_range_group_sum_dev(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                            const uint64_t* offsets, uint64_t n_rows, uint32_t n_series, const uint32_t* gid,
                            uint32_t n_groups, double* out_sum, uint32_t* out_cnt) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_series == 0 || n_groups == 0) return B2P_OK;
  b2p_group_index* ix = nullptr;
  int rc = b2p_group_index_create_dev(c, gid, n_series, n_groups, &ix);
  if (rc) return rc;
  rc = b2p_range_group_sum_indexed_dev(c, p, ts, val, offsets, n_rows, n_series, ix, 0, n_groups, out_sum, out_cnt);
  if (!rc) rc = b2p_sync(c);  // the temporary index must outlive the kernels that read it
  b2p_group_index_destroy(c, ix);
  return rc;
}

/* ---- multi-GPU: all-reduce of by-label partials over NCCL ----------------------------------------- */

int b2p_comm_unique_id(void* out_id, size_t bytes) {
  if (!out_id || bytes < sizeof(Nccl::unique_id)) return fail(B2P_E_INVALID, "need a %zu-byte buffer", sizeof(Nccl::unique_id));
  if (!g_nccl.load()) return fail(B2P_E_CUDA, "libnccl.so.2 not found (%s)", dlerror() ? dlerror() : "dlopen");
  Nccl::unique_id id;
  NCCL_TRY(g_nccl.GetUniqueId(&id));
  memcpy(out_id, &id, sizeof id);
  return B2P_OK;
}

int b2p_comm_init(b2p_ctx* c, const void* id_bytes, size_t bytes, int n_ranks, int rank) {
  if (!c || !id_bytes || bytes < sizeof(Nccl::unique_id) || n_ranks < 1 || rank < 0 || rank >= n_ranks)
    return fail(B2P_E_INVALID, "bad communicator arguments");
  if (c->comm) return fail(B2P_E_INVALID, "context already has a communicator");
  if (!g_nccl.load()) return fail(B2P_E_CUDA, "libnccl.so.2 not found (%s)", dlerror() ? dlerror() : "dlopen");
  DeviceGuard g(c->device);
  Nccl::unique_id id;
  memcpy(&id, id_bytes, sizeof id);
  // the tile all-reduces run next to the persistent range kernel: keep their footprint to a few SMs (an explicit
  // NCCL_MAX_CTAS / NCCL_MAX_NCHANNELS of the caller wins)
  setenv("NCCL_MAX_CTAS", "16", 0);
  setenv("NCCL_MAX_NCHANNELS", "16", 0);
  NCCL_TRY(g_nccl.CommInitRank(&c->comm, n_ranks, id, rank));
  c->comm_ranks = n_ranks;
  c->comm_rank = rank;
  int lo = 0, hi = 0;
  CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = numerically lowest = highest priority
  CU(cudaStreamCreateWithPriority(&c->s_comm, cudaStreamNonBlocking, hi));
  CU(cudaEventCreateWithFlags(&c->ev_comm_in, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_comm_done, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_comm_go, cudaEventDisableTiming));
  return B2P_OK;
}

int b2p_comm_destroy(b2p_ctx* c) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (!c->comm) return B2P_OK;
  DeviceGuard g(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->s_comm) cudaStreamSynchronize(c->s_comm);
  NCCL_TRY(g_nccl.CommDestroy(c->comm));
  c->comm = nullptr;
  c->comm_ranks = 1;
  return B2P_OK;
}

// One all-reduce of the by-label partials [n] of every rank, enqueued on the context's stream (asynchronous).
//   SUM / AVG / COUNT   val (plain sums) and cnt are added (the __sum_state / __sum_merge split of the reference,
//                       src/query/src/dist_plan/commutativity.rs:85-113); finalise afterwards (b2p_group_finalize_dev)
//   MIN / MAX           cnt is added, val is reduced as f64::total_cmp keys with int64 min / max (groups absent on a
//                       rank, cnt == 0, hold the neutral key); groups absent everywhere end up 0.0 again
//   STDDEV / STDVAR     inputs are per-rank (cnt, mean, M2 = val): the global mean comes from an all-reduce of
//                       cnt*mean, then M2 = sum_r [M2_r + cnt_r (mean_r - mean)^2] (commutativity.rs:158-191 merges
//                       the same state pairwise); on return mean / val hold the merged state on every rank
int b2p_allreduce_partials_dev(b2p_ctx* c, int32_t agg, double* val, uint32_t* cnt, double* mean, uint64_t n) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (agg < 0 || agg > B2P_AGG_STDVAR) return fail(B2P_E_INVALID, "unknown aggregator %d", agg);
  if (n == 0) return B2P_OK;
  if (!val || !cnt) return fail(B2P_E_INVALID, "NULL argument");
  const bool var = agg == B2P_AGG_STDDEV || agg == B2P_AGG_STDVAR;
  if (var && !mean) return fail(B2P_E_INVALID, "stddev / stdvar partials need the per-group means");
  if (!c->comm) {
    if (c->comm_ranks == 1) return B2P_OK;  // single rank: nothing to merge
    return fail(B2P_E_INVALID, "no communicator: call b2p_comm_init first");
  }
  DeviceGuard g(c->device);
  uint64_t blocks = (n + 255) / 256;
  if (blocks > (uint64_t)c->num_sms * 16) blocks = (uint64_t)c->num_sms * 16;
  if (agg == B2P_AGG_MIN || agg == B2P_AGG_MAX) {
    minmax_key_encode_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(agg == B2P_AGG_MIN, val, cnt, n);
    NCCL_TRY(g_nccl.GroupStart());
    NCCL_TRY(g_nccl.AllReduce(val, val, n, Nccl::kInt64, agg == B2P_AGG_MIN ? Nccl::kMin : Nccl::kMax, c->comm, c->stream));
    NCCL_TRY(g_nccl.AllReduce(cnt, cnt, n, Nccl::kUint32, Nccl::kSum, c->comm, c->stream));
    NCCL_TRY(g_nccl.GroupEnd());
    minmax_key_decode_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(val, cnt, n);
    c->launches += 2;
  } else if (var) {
    int rc;
    if ((rc = c->m_tmp0.ensure(n * 8)) || (rc = c->m_tmp1.ensure(n * 4))) return rc;
    double* wsum = c->m_tmp0.as<double>();    // cnt_r * mean_r -> global sum
    uint32_t* cnt_r = c->m_tmp1.as<uint32_t>();  // this rank's counts (cnt itself becomes the global count)
    variance_merge_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(0, val, cnt, mean, wsum, cnt_r, n);
    NCCL_TRY(g_nccl.GroupStart());
    NCCL_TRY(g_nccl.AllReduce(wsum, wsum, n, Nccl::kFloat64, Nccl::kSum, c->comm, c->stream));
    NCCL_TRY(g_nccl.AllReduce(cnt, cnt, n, Nccl::kUint32, Nccl::kSum, c->comm, c->stream));
    NCCL_TRY(g_nccl.GroupEnd());
    variance_merge_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(1, val, cnt, mean, wsum, cnt_r, n);
    NCCL_TRY(g_nccl.AllReduce(val, val, n, Nccl::kFloat64, Nccl::kSum, c->comm, c->stream));
    c->launches += 2;
  } else {
    stage_begin(c, 4);
    NCCL_TRY(g_nccl.GroupStart());
    NCCL_TRY(g_nccl.AllReduce(val, val, n, Nccl::kFloat64, Nccl::kSum, c->comm, c->stream));
    NCCL_TRY(g_nccl.AllReduce(cnt, cnt, n, Nccl::kUint32, Nccl::kSum, c->comm, c->stream));
    NCCL_TRY(g_nccl.GroupEnd());
    stage_end(c, 4);
  }
  CU(cudaGetLastError());
  return B2P_OK;
}

// config 5 (wide avg_over_time): per-column (sum f64, count u64) of every rank added in place
int b2p_allreduce_columns_dev(b2p_ctx* c, double* sum, uint64_t* cnt, uint32_t n_cols) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_cols == 0) return B2P_OK;
  if (!sum || !cnt) return fail(B2P_E_INVALID, "NULL argument");
  if (!c->comm) {
    if (c->comm_ranks == 1) return B2P_OK;
    return fail(B2P_E_INVALID, "no communicator: call b2p_comm_init first");
  }
  DeviceGuard g(c->device);
  stage_begin(c, 4);
  NCCL_TRY(g_nccl.GroupStart());
  NCCL_TRY(g_nccl.AllReduce(sum, sum, n_cols, Nccl::kFloat64, Nccl::kSum, c->comm, c->stream));
  NCCL_TRY(g_nccl.AllReduce(cnt, cnt, n_cols, Nccl::kUint64, Nccl::kSum, c->comm, c->stream));
  NCCL_TRY(g_nccl.GroupEnd());
  stage_end(c, 4);
  return B2P_OK;
}

int b2p_group_finalize_dev(b2p_ctx* c, int32_t agg, double* val, const uint32_t* cnt, uint64_t n) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n == 0) return B2P_OK;
  DeviceGuard g(c->device);
  uint64_t blocks = (n + 255) / 256;
  if (blocks > (uint64_t)c->num_sms * 16) blocks = (uint64_t)c->num_sms * 16;
  group_finalize_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(agg, val, cnt, n);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

// HistogramFold over an explicit (histogram -> buckets in le order) index; every pointer is a device pointer.
int b2p_histogram_fold_dev(b2p_ctx* c, double phi, const uint32_t* hist_off, const uint32_t* bucket_series,
                           const double* bucket_le, uint32_t n_hist, const double* rates, const uint32_t* valid_words,
                           uint64_t T, double* out, uint32_t* out_valid_words) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_hist == 0 || T == 0) return B2P_OK;
  if (!hist_off || !bucket_series || !bucket_le || !rates || !valid_words || !out || !out_valid_words)
    return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  HistFoldArgs a{};
  a.phi = phi; a.hist_off = hist_off; a.bucket_series = bucket_series; a.bucket_le = bucket_le; a.n_hist = n_hist;
  a.rates = rates; a.valid = valid_words; a.T = T; a.Tw = (uint32_t)((T + 31) / 32); a.out = out; a.out_valid = out_valid_words;
  const uint64_t warps = (uint64_t)n_hist * ((T + 31) / 32);
  uint64_t blocks = (warps + kHistWarps - 1) / kHistWarps;
  const uint64_t cap = (uint64_t)c->num_sms * 3;  // 72 KB of counters + slots per CTA: three CTAs per SM
  if (blocks > cap) blocks = cap;
  constexpr size_t smem = (size_t)kHistWarps * kHistSmemBuckets * 32 * (8 + 1);
  static bool attr_set[16] = {};
  if (!attr_set[c->device & 15]) {
    CU(cudaFuncSetAttribute(histogram_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set[c->device & 15] = true;
  }
  stage_begin(c, 3);
  histogram_fold_kernel<<<(unsigned)blocks, kHistWarps * 32, smem, c->stream>>>(a);
  c->launches++;
  stage_end(c, 3);
  CU(cudaGetLastError());
  return B2P_OK;
}

// Uniform layout: bucket b of histogram h is series h * n_buckets + b and every histogram has the bounds le[].
int b2p_histogram_quantile_dev(b2p_ctx* c, double phi, const double* le, uint32_t n_buckets, const double* rates,
                               const uint32_t* valid_words, uint32_t n_hist, uint64_t T, double* out,
                               uint32_t* out_valid_words) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_hist == 0 || T == 0) return B2P_OK;
  if (!le || !rates || !valid_words || !out || !out_valid_words || n_buckets == 0)
    return fail(B2P_E_INVALID, "NULL argument");
  if ((uint64_t)n_hist * n_buckets > 0xffffffffull) return fail(B2P_E_TOO_LARGE, "more than 2^32 bucket series");
  DeviceGuard g(c->device);
  int rc;
  const size_t nb = (size_t)n_hist * n_buckets;
  {  // the fold index of the uniform layout (12 B per bucket series, rebuilt per call: microseconds)
    if ((rc = c->hq_off.ensure(((size_t)n_hist + 1) * 4)) || (rc = c->hq_series.ensure(nb * 4)) || (rc = c->hq_les.ensure(nb * 8)))
      return rc;
    uint64_t blocks = (nb + 255) / 256;
    if (blocks > (uint64_t)c->num_sms * 16) blocks = (uint64_t)c->num_sms * 16;
    histogram_uniform_index_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(le, n_buckets, n_hist, c->hq_off.as<uint32_t>(),
                                                                            c->hq_series.as<uint32_t>(), c->hq_les.as<double>());
    c->launches++;
    CU(cudaGetLastError());
  }
  return b2p_histogram_fold_dev(c, phi, c->hq_off.as<uint32_t>(), c->hq_series.as<uint32_t>(), c->hq_les.as<double>(), n_hist,
                                rates, valid_words, T, out, out_valid_words);
}

int b2p_column_reduce_dev(b2p_ctx* c, const double* const* cols, uint32_t n_cols, uint64_t n_rows, double* out_sum,
                          uint64_t* out_cnt) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_cols == 0 || n_rows == 0) return B2P_OK;
  if (!cols || !out_sum || !out_cnt) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  unsigned bpc = (unsigned)((c->num_sms * 8 + n_cols - 1) / n_cols);
  if (bpc < 1) bpc = 1;
  const uint64_t max_useful = (n_rows + 511) / 512;
  if (bpc > max_useful) bpc = (unsigned)max_useful;
  int rc;
  if ((rc = c->c_psum.ensure((size_t)n_cols * bpc * 8))) return rc;
  if ((rc = c->c_pcnt.ensure((size_t)n_cols * bpc * 8))) return rc;
  stage_begin(c, 3);
  column_reduce_stage1<<<dim3(bpc, n_cols), 256, 0, c->stream>>>(cols, n_rows, c->c_psum.as<double>(),
                                                                 c->c_pcnt.as<unsigned long long>());
  column_reduce_stage2<<<n_cols, 32, 0, c->stream>>>(c->c_psum.as<double>(), c->c_pcnt.as<unsigned long long>(), bpc,
                                                     out_sum, reinterpret_cast<unsigned long long*>(out_cnt));
  c->launches += 2;
  stage_end(c, 3);
  CU(cudaGetLastError());
  return B2P_OK;
}

int b2p_synth_fill_dev(b2p_ctx* c, uint64_t series_begin, uint64_t n_series, uint32_t n_samples, int64_t t0,
                       int64_t scrape_ms, uint32_t jitter_ms, int32_t with_resets, uint64_t seed, int64_t* ts,
                       double* val, uint32_t* sid) {
  if (!c || !ts || !val) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  const uint64_t total = n_series * (uint64_t)n_samples;
  if (total == 0) return B2P_OK;
  uint64_t blocks = (total + 255) / 256;
  if (blocks > (uint64_t)c->num_sms * 32) blocks = (uint64_t)c->num_sms * 32;
  synth_fill_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(series_begin, n_series, n_samples, t0, scrape_ms,
                                                             jitter_ms, with_resets, seed, ts, val, sid);
  c->launches++;
  CU(cudaGetLastError());
  return B2P_OK;
}

/* ---- host-pointer API ------------------------------------------------------------------------ */

// One chunk, no overlap: H2D -> K0/K2 -> D2H on the context stream.  sid values are global ids
// (sid_base is subtracted on the device); offsets_host, when given, is already rebased to the chunk.
// Host-side SeriesDivide + cadence scan (see the header).  Plain sequential passes: memory bound, ~8-10 GB/s per thread;
// b2p_range_eval runs one of these per chunk on a few worker threads while earlier chunks are on the bus.
static int host_scan_series(const int64_t* ts, const uint32_t* sid, const uint64_t* offsets_in, uint64_t n_rows,
                            uint32_t n_series, uint32_t sid_base, uint64_t* offsets_out, int64_t* t0, int64_t* cadence,
                            int32_t* all_regular) {
  if (sid) {
    uint64_t r = 0;
    uint32_t prev = sid_base;
    offsets_out[0] = 0;
    uint32_t next = 0;  // next local series whose start is still to be written (offsets_out[next + 1 ..] pending)
    for (; r < n_rows; ++r) {
      const uint32_t id = sid[r];
      if (id < prev || id - sid_base >= n_series) return B2P_E_UNSORTED;
      const uint32_t local = id - sid_base;
      while (next < local) offsets_out[++next] = r;  // series without rows in between start (and end) here
      prev = id;
    }
    while (next < n_series) offsets_out[++next] = n_rows;
  } else {
    for (uint32_t s = 0; s <= n_series; ++s) offsets_out[s] = offsets_in[s] - offsets_in[0];
    for (uint32_t s = 0; s < n_series; ++s)
      if (offsets_out[s + 1] < offsets_out[s] || offsets_out[s + 1] > n_rows) return B2P_E_INVALID;
  }
  bool regular = true;
  for (uint32_t s = 0; s < n_series; ++s) {
    const uint64_t r0 = offsets_out[s], r1 = offsets_out[s + 1];
    const int64_t first = r1 > r0 ? ts[r0] : 0;
    // (wrapping arithmetic: the device rebuilds the column with the same operations)
    const int64_t step = r1 - r0 >= 2 ? (int64_t)((uint64_t)ts[r0 + 1] - (uint64_t)first) : 0;
    if (t0) t0[s] = first;
    if (cadence) cadence[s] = step;
    if (regular) {
      uint64_t expect = (uint64_t)first;
      for (uint64_t r = r0; r < r1; ++r) {
        if ((uint64_t)ts[r] != expect) { regular = false; break; }
        expect += (uint64_t)step;
      }
    }
    if (!regular && !t0 && !cadence) break;
  }
  if (all_regular) *all_regular = regular ? 1 : 0;
  return B2P_OK;
}

int b2p_host_scan_series(const int64_t* ts, const uint32_t* sid, const uint64_t* offsets_in, uint64_t n_rows,
                         uint32_t n_series, uint32_t sid_base, uint64_t* offsets_out, int64_t* t0, int64_t* cadence,
                         int32_t* all_regular) {
  if (!offsets_out || (!sid && !offsets_in) || (!ts && n_rows)) return fail(B2P_E_INVALID, "NULL argument");
  const int rc = host_scan_series(ts, sid, offsets_in, n_rows, n_series, sid_base, offsets_out, t0, cadence, all_regular);
  if (rc == B2P_E_UNSORTED) return fail(rc, "series-id column is not non-decreasing or out of range");
  if (rc) return fail(rc, "offsets are not non-decreasing or exceed n_rows");
  return rc;
}

static int range_eval_host_simple(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                                  const uint32_t* sid, uint32_t sid_base, const uint64_t* offsets_host, uint64_t n_rows,
                                  uint32_t n_series, int64_t T, double* out, uint32_t* valid_words) {
  int rc;
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  const size_t rows = n_rows ? n_rows : 1;
  if ((rc = c->h_ts.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_val.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_off.ensure(((size_t)n_series + 1) * 8))) return rc;
  if ((rc = c->h_out.ensure((size_t)n_series * (size_t)T * 8))) return rc;
  if ((rc = c->h_valid.ensure((size_t)n_series * Tw * 4))) return rc;
  if ((rc = reset_status(c))) return rc;
  c->last_h2d_bytes = (long long)(n_rows * 16 + (offsets_host ? ((size_t)n_series + 1) * 8 : n_rows * 4));
  CU(cudaMemcpyAsync(c->h_ts.p, ts, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_val.p, val, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  if (offsets_host) {
    CU(cudaMemcpyAsync(c->h_off.p, offsets_host, ((size_t)n_series + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  } else {
    if ((rc = c->h_sid.ensure(rows * 4 + 16))) return rc;
    CU(cudaMemcpyAsync(c->h_sid.p, sid, n_rows * 4, cudaMemcpyHostToDevice, c->stream));
    if ((rc = series_offsets_impl(c, c->h_sid.as<uint32_t>(), n_rows, n_series, sid_base, c->h_off.as<uint64_t>())))
      return rc;
  }
  if ((rc = b2p_range_eval_dev(c, p, c->h_ts.as<int64_t>(), c->h_val.as<double>(), c->h_off.as<uint64_t>(), n_rows,
                               n_series, c->h_out.as<double>(), c->h_valid.as<uint32_t>())))
    return rc;
  if ((rc = b2p_sync(c))) return rc;
  CU(cudaMemcpyAsync(out, c->h_out.p, (size_t)n_series * (size_t)T * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(valid_words, c->h_valid.p, (size_t)n_series * Tw * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

// first row whose id is >= key in a non-decreasing id column
static uint64_t lower_bound_sid(const uint32_t* sid, uint64_t n, uint64_t key) {
  uint64_t lo = 0, hi = n;
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    if ((uint64_t)sid[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

int b2p_range_eval(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val, const uint32_t* sid,
                   const uint64_t* offsets_host, uint64_t n_rows, uint32_t n_series, double* out,
                   uint32_t* valid_words, int64_t* out_ts) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  int64_t T = 0;
  int rc = check_grid(p, n_series, &T);
  if (rc) return rc;
  if (out_ts)
    for (int64_t k = 0; k < T; ++k) out_ts[k] = p->start + k * p->interval;
  if (n_series == 0 || T == 0) return B2P_OK;
  if (!sid && !offsets_host) return fail(B2P_E_INVALID, "need sid or offsets_host");
  if (!out || !valid_words || ((!ts || !val) && n_rows)) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  if (!c->pending.empty() && (rc = b2p_sync(c))) return rc;  // earlier asynchronous calls finish first
  const uint32_t Tw = (uint32_t)((T + 31) / 32);

  // ---- small inputs: one shot -------------------------------------------------------------------
  constexpr uint64_t kChunkRows = 4u << 20;  // ~84 MB of H2D per chunk
  if (n_rows <= kChunkRows + kChunkRows / 2 || n_series < 64)
    return range_eval_host_simple(c, p, ts, val, sid, 0u, offsets_host, n_rows, n_series, T, out, valid_words);

  // ---- large inputs: series chunks, double-buffered; H2D(i+1) | K0+K2(i) | D2H(i-1) overlap -----------
  const uint64_t avg_rows = n_rows / n_series + 1;
  uint32_t C = (uint32_t)(kChunkRows / avg_rows);
  if (C < 64) C = 64;
  const uint32_t n_chunks = (n_series + C - 1) / C;
  if (!c->pipe_ready) {
    bool ok = cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < 2; ++i) {
      ok = ok && cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&c->ev_comp[i], cudaEventDisableTiming) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&c->ev_d2h[i], cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) return fail(B2P_E_CUDA, "pipeline stream/event creation failed");
    c->pipe_ready = true;
  }
  if ((rc = c->p_status.ensure((size_t)n_chunks * sizeof(Status)))) return rc;  // device copies of each chunk's status
  Status* h_stat = nullptr;
  CU(cudaMallocHost(&h_stat, (size_t)n_chunks * sizeof(Status)));
  uint64_t* h_offs[2] = {nullptr, nullptr};
  if (offsets_host) {
    for (int i = 0; i < 2; ++i) CU(cudaMallocHost(&h_offs[i], ((size_t)C + 1) * 8));
  }
  struct Cleanup {
    Status* s; uint64_t* o0; uint64_t* o1;
    ~Cleanup() { if (s) cudaFreeHost(s); if (o0) cudaFreeHost(o0); if (o1) cudaFreeHost(o1); }
  } cleanup{h_stat, h_offs[0], h_offs[1]};

  // worst-case chunk row count (chunks are whole series)
  uint64_t max_rows = 0;
  std::vector<uint64_t> chunk_row(n_chunks + 1, 0);
  {
    uint64_t prev = 0;
    for (uint32_t i = 0; i < n_chunks; ++i) {
      const uint64_t s1 = (uint64_t)(i + 1) * C < n_series ? (uint64_t)(i + 1) * C : n_series;
      const uint64_t r1 = offsets_host ? offsets_host[s1] : lower_bound_sid(sid, n_rows, s1);
      if (r1 < prev) return fail(B2P_E_UNSORTED, "series-id column is not non-decreasing");
      if (r1 - prev > max_rows) max_rows = r1 - prev;
      prev = r1;
      chunk_row[i + 1] = r1;
    }
    if (!offsets_host && prev != n_rows) return fail(B2P_E_UNSORTED, "series id >= n_series");
  }
  // Host scan of every chunk, ahead of the copies (worker k takes chunks k, k + W, ..): 0 = not scanned yet, 1 = every
  // series of the chunk is equally spaced (its rebased offsets, first timestamps and cadences are in the pinned
  // descriptor arrays), 2 = take the ordinary route (ids out of order included: K0 reports those as before)
  // (only when the batch comes with its id column: then the descriptors replace 12 of the 20 B/row and K0; with offsets
  // handed over the call is already at 16 B/row, and the scan's per-call cost — pinned descriptor arrays, worker
  // threads — measured more than the 8 B/row it saves: 2.36 vs 3.0 G samples/s)
  const bool scan = c->host_ts_scan && !offsets_host;
  uint64_t* h_doff = nullptr;
  int64_t *h_t0 = nullptr, *h_cad = nullptr;
  std::unique_ptr<std::atomic<int>[]> scan_state;
  std::atomic<bool> scan_stop{false};
  std::vector<std::thread> scan_workers;
  struct ScanJoin {
    std::atomic<bool>& stop; std::vector<std::thread>& w; uint64_t*& a; int64_t*& b; int64_t*& d;
    ~ScanJoin() {
      stop.store(true);
      for (auto& t : w) if (t.joinable()) t.join();
      if (a) cudaFreeHost(a);
      if (b) cudaFreeHost(b);
      if (d) cudaFreeHost(d);
    }
  } scan_join{scan_stop, scan_workers, h_doff, h_t0, h_cad};
  if (scan) {
    CU(cudaMallocHost(&h_doff, ((size_t)n_series + n_chunks) * 8));
    CU(cudaMallocHost(&h_t0, (size_t)n_series * 8));
    CU(cudaMallocHost(&h_cad, (size_t)n_series * 8));
    scan_state.reset(new std::atomic<int>[n_chunks]);
    for (uint32_t i = 0; i < n_chunks; ++i) scan_state[i].store(0);
    unsigned hw = std::thread::hardware_concurrency();
    unsigned W = hw >= 64 ? 16u : (hw >= 8 ? hw / 4 : 1u);
    if (W > n_chunks) W = n_chunks;
    std::atomic<int>* state = scan_state.get();
    const uint64_t* rows = chunk_row.data();
    try {
    for (unsigned k = 0; k < W; ++k) {
      scan_workers.emplace_back([=, &scan_stop]() {
        for (uint32_t i = k; i < n_chunks && !scan_stop.load(std::memory_order_relaxed); i += W) {
          const uint32_t s0 = i * C;
          const uint32_t s1 = (uint64_t)s0 + C < n_series ? s0 + C : n_series;
          const uint64_t r0 = rows[i], nr = rows[i + 1] - rows[i];
          int32_t regular = 0;
          const int rc_scan = host_scan_series(ts + r0, sid ? sid + r0 : nullptr, offsets_host ? offsets_host + s0 : nullptr, nr,
                                               s1 - s0, s0, h_doff + s0 + i, h_t0 + s0, h_cad + s0, &regular);
          state[i].store((rc_scan == B2P_OK && regular) ? 1 : 2, std::memory_order_release);
        }
      });
    }
    } catch (...) {  // no threads to be had: every chunk the started workers do not reach takes the ordinary route
      scan_stop.store(true);
      for (auto& t : scan_workers) if (t.joinable()) t.join();
      for (uint32_t i = 0; i < n_chunks; ++i) {
        int zero = 0;
        state[i].compare_exchange_strong(zero, 2);
      }
    }
  }
  for (int i = 0; i < 2; ++i) {
    if (scan && (rc = c->p_t0[i].ensure((size_t)C * 8))) return rc;
    if (scan && (rc = c->p_cad[i].ensure((size_t)C * 8))) return rc;
    if ((rc = c->p_ts[i].ensure(max_rows * 8 + 16))) return rc;
    if ((rc = c->p_val[i].ensure(max_rows * 8 + 16))) return rc;
    if (!offsets_host && (rc = c->p_sid[i].ensure(max_rows * 4 + 16))) return rc;
    if ((rc = c->p_off[i].ensure(((size_t)C + 1) * 8))) return rc;
    if ((rc = c->p_out[i].ensure((size_t)C * (size_t)T * 8))) return rc;
    if ((rc = c->p_valid[i].ensure((size_t)C * Tw * 4))) return rc;
  }
  CU(cudaStreamSynchronize(c->stream));
  c->last_h2d_bytes = 0;
  uint64_t row_lo = 0;
  for (uint32_t i = 0; i < n_chunks; ++i) {
    const int b = (int)(i & 1);
    const uint32_t s0 = i * C;
    const uint32_t s1 = (uint64_t)s0 + C < n_series ? s0 + C : n_series;
    const uint32_t ns = s1 - s0;
    const uint64_t row_hi = offsets_host ? offsets_host[s1] : lower_bound_sid(sid, n_rows, s1);
    const uint64_t nr = row_hi - row_lo;
    int described = 2;  // 1: the chunk's timestamp (and id) column is described by (offsets, t0, cadence)
    if (scan)
      while ((described = scan_state[i].load(std::memory_order_acquire)) == 0) std::this_thread::yield();
    // H2D of chunk i may start once chunk i-2's kernels no longer read this buffer pair
    if (i >= 2) CU(cudaStreamWaitEvent(c->s_h2d, c->ev_comp[b], 0));
    CU(cudaMemcpyAsync(c->p_val[b].p, val + row_lo, nr * 8, cudaMemcpyHostToDevice, c->s_h2d));
    c->last_h2d_bytes += (long long)(nr * 8);
    if (described == 1) {
      c->last_h2d_bytes += (long long)(((size_t)ns + 1) * 8 + (size_t)ns * 16);
      CU(cudaMemcpyAsync(c->p_off[b].p, h_doff + s0 + i, ((size_t)ns + 1) * 8, cudaMemcpyHostToDevice, c->s_h2d));
      CU(cudaMemcpyAsync(c->p_t0[b].p, h_t0 + s0, (size_t)ns * 8, cudaMemcpyHostToDevice, c->s_h2d));
      CU(cudaMemcpyAsync(c->p_cad[b].p, h_cad + s0, (size_t)ns * 8, cudaMemcpyHostToDevice, c->s_h2d));
    } else {
    c->last_h2d_bytes += (long long)(nr * 8 + (offsets_host ? ((size_t)ns + 1) * 8 : nr * 4));
    CU(cudaMemcpyAsync(c->p_ts[b].p, ts + row_lo, nr * 8, cudaMemcpyHostToDevice, c->s_h2d));
    if (offsets_host) {
      if (i >= 2) CU(cudaEventSynchronize(c->ev_h2d[b]));  // the pinned rebase buffer is free again
      for (uint32_t q = 0; q <= ns; ++q) h_offs[b][q] = offsets_host[s0 + q] - row_lo;
      CU(cudaMemcpyAsync(c->p_off[b].p, h_offs[b], ((size_t)ns + 1) * 8, cudaMemcpyHostToDevice, c->s_h2d));
    } else {
      CU(cudaMemcpyAsync(c->p_sid[b].p, sid + row_lo, nr * 4, cudaMemcpyHostToDevice, c->s_h2d));
    }
    }
    CU(cudaEventRecord(c->ev_h2d[b], c->s_h2d));
    // compute: after its inputs landed and after chunk i-2's results left the output buffers
    CU(cudaStreamWaitEvent(c->stream, c->ev_h2d[b], 0));
    if (i >= 2) CU(cudaStreamWaitEvent(c->stream, c->ev_d2h[b], 0));
    if ((rc = reset_status(c))) return rc;
    if (described == 1) {
      unsigned blocks = (ns + 7) / 8;
      if (blocks > (unsigned)c->num_sms * 8u) blocks = (unsigned)c->num_sms * 8u;
      ts_expand_kernel<<<blocks, 256, 0, c->stream>>>(c->p_off[b].as<uint64_t>(), c->p_t0[b].as<int64_t>(),
                                                      c->p_cad[b].as<int64_t>(), ns, c->p_ts[b].as<int64_t>());
      c->launches++;
      CU(cudaGetLastError());
    } else if (!offsets_host &&
        (rc = series_offsets_impl(c, c->p_sid[b].as<uint32_t>(), nr, ns, s0, c->p_off[b].as<uint64_t>())))
      return rc;
    if ((rc = b2p_range_eval_dev(c, p, c->p_ts[b].as<int64_t>(), c->p_val[b].as<double>(), c->p_off[b].as<uint64_t>(),
                                 nr, ns, c->p_out[b].as<double>(), c->p_valid[b].as<uint32_t>())))
      return rc;
    {  // this chunk's verdict is read with all the others below: take the call out of the pending queue
      const int slot = c->pending.back().slot;
      c->pending.pop_back();
      CU(cudaMemcpyAsync(c->p_status.as<Status>() + i, c->d_ring + slot, sizeof(Status), cudaMemcpyDeviceToDevice, c->stream));
    }
    CU(cudaEventRecord(c->ev_comp[b], c->stream));
    // D2H
    CU(cudaStreamWaitEvent(c->s_d2h, c->ev_comp[b], 0));
    CU(cudaMemcpyAsync(out + (size_t)s0 * (size_t)T, c->p_out[b].p, (size_t)ns * (size_t)T * 8, cudaMemcpyDeviceToHost,
                       c->s_d2h));
    CU(cudaMemcpyAsync(valid_words + (size_t)s0 * Tw, c->p_valid[b].p, (size_t)ns * Tw * 4, cudaMemcpyDeviceToHost,
                       c->s_d2h));
    CU(cudaEventRecord(c->ev_d2h[b], c->s_d2h));
    row_lo = row_hi;
  }
  CU(cudaMemcpyAsync(h_stat, c->p_status.p, (size_t)n_chunks * sizeof(Status), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(c->h_k0, c->d_k0, sizeof(Status), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaStreamSynchronize(c->s_d2h));
  if (const uint32_t k0 = c->h_k0->k0_errors) {
    CU(cudaMemsetAsync(c->d_k0, 0, sizeof(Status), c->stream));
    if (k0 & 1u) return fail(B2P_E_UNSORTED, "series-id column is not non-decreasing");
    return fail(B2P_E_UNSORTED, "series id >= n_series");
  }
  // per-chunk verdicts; a chunk whose slow path ran out of arena is redone alone (b2p_sync grows the arena)
  long long slow_total = 0, w_total = 0;
  row_lo = 0;
  for (uint32_t i = 0; i < n_chunks; ++i) {
    const uint32_t s0 = i * C;
    const uint32_t s1 = (uint64_t)s0 + C < n_series ? s0 + C : n_series;
    const uint64_t row_hi = offsets_host ? offsets_host[s1] : lower_bound_sid(sid, n_rows, s1);
    const Status st = h_stat[i];
    slow_total += st.slow_count;
    w_total += st.w_count;
    if (st.arena_overflow) {
      std::string tmp_offs;
      const uint64_t* offs_chunk = nullptr;
      if (offsets_host) {
        tmp_offs.resize(((size_t)(s1 - s0) + 1) * 8);
        uint64_t* o = reinterpret_cast<uint64_t*>(&tmp_offs[0]);
        for (uint32_t q = 0; q <= s1 - s0; ++q) o[q] = offsets_host[s0 + q] - row_lo;
        offs_chunk = o;
      }
      if ((rc = range_eval_host_simple(c, p, ts + row_lo, val + row_lo, sid ? sid + row_lo : nullptr, s0, offs_chunk,
                                       row_hi - row_lo, s1 - s0, T, out + (size_t)s0 * (size_t)T,
                                       valid_words + (size_t)s0 * Tw)))
        return rc;
    }
    row_lo = row_hi;
  }
  c->last_slow = slow_total;
  c->last_w = w_total;
  if (c->last_used_lean) lean_verdict(c, p->fn_id, (uint64_t)w_total, n_series);
  return B2P_OK;
}

int b2p_range_udf(b2p_ctx* c, int32_t fn_id, const int64_t* ts, const double* val, uint64_t n_rows,
                  const int64_t* packed_ranges, const int64_t* eval_ts, uint64_t n_win, int64_t range_length,
                  double param0, double param1, double* out, uint8_t* valid) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_win == 0) return B2P_OK;
  if (!packed_ranges || !out || !valid) return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  int rc;
  const size_t rows = n_rows ? n_rows : 1;
  if ((rc = c->h_ts.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_val.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_aux0.ensure(n_win * 8))) return rc;
  if ((rc = c->h_aux1.ensure(n_win * 8))) return rc;
  if ((rc = c->h_out.ensure(n_win * 8))) return rc;
  if ((rc = c->h_valid.ensure(n_win))) return rc;
  if (n_rows) {
    CU(cudaMemcpyAsync(c->h_ts.p, ts, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemcpyAsync(c->h_val.p, val, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  }
  CU(cudaMemcpyAsync(c->h_aux0.p, packed_ranges, n_win * 8, cudaMemcpyHostToDevice, c->stream));
  if (eval_ts) CU(cudaMemcpyAsync(c->h_aux1.p, eval_ts, n_win * 8, cudaMemcpyHostToDevice, c->stream));
  if ((rc = b2p_range_udf_dev(c, fn_id, c->h_ts.as<int64_t>(), c->h_val.as<double>(), n_rows, c->h_aux0.as<int64_t>(),
                              eval_ts ? c->h_aux1.as<int64_t>() : nullptr, n_win, range_length, param0, param1,
                              c->h_out.as<double>(), c->h_valid.as<uint8_t>())))
    return rc;
  CU(cudaMemcpyAsync(out, c->h_out.p, n_win * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(valid, c->h_valid.p, n_win, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

int b2p_instant_select(b2p_ctx* c, int64_t start, int64_t end, int64_t interval, int64_t lookback, int64_t offset,
                       const int64_t* ts, const double* val, const uint32_t* sid, const uint64_t* offsets_host,
                       uint64_t n_rows, uint32_t n_series, double* out, uint32_t* valid_words) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  b2p_range_params p{};
  p.start = start; p.end = end; p.interval = interval; p.range = lookback;
  int64_t T = 0;
  int rc = check_grid(&p, n_series, &T);
  if (rc) return rc;
  if (n_series == 0 || T == 0) return B2P_OK;
  if (!sid && !offsets_host) return fail(B2P_E_INVALID, "need sid or offsets_host");
  DeviceGuard g(c->device);
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  const size_t rows = n_rows ? n_rows : 1;
  if ((rc = c->h_ts.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_val.ensure(rows * 8 + 16))) return rc;
  if ((rc = c->h_off.ensure(((size_t)n_series + 1) * 8))) return rc;
  if ((rc = c->h_out.ensure((size_t)n_series * (size_t)T * 8))) return rc;
  if ((rc = c->h_valid.ensure((size_t)n_series * Tw * 4))) return rc;
  if ((rc = reset_status(c))) return rc;
  CU(cudaMemcpyAsync(c->h_ts.p, ts, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_val.p, val, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  if (offsets_host) {
    CU(cudaMemcpyAsync(c->h_off.p, offsets_host, ((size_t)n_series + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  } else {
    if ((rc = c->h_sid.ensure(rows * 4 + 16))) return rc;
    CU(cudaMemcpyAsync(c->h_sid.p, sid, n_rows * 4, cudaMemcpyHostToDevice, c->stream));
    if ((rc = b2p_series_offsets_dev(c, c->h_sid.as<uint32_t>(), n_rows, n_series, c->h_off.as<uint64_t>()))) return rc;
  }
  if ((rc = b2p_instant_select_dev(c, start, end, interval, lookback, offset, c->h_ts.as<int64_t>(),
                                   c->h_val.as<double>(), c->h_off.as<uint64_t>(), n_rows, n_series,
                                   c->h_out.as<double>(), c->h_valid.as<uint32_t>())))
    return rc;
  if ((rc = b2p_sync(c))) return rc;
  CU(cudaMemcpyAsync(out, c->h_out.p, (size_t)n_series * (size_t)T * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(valid_words, c->h_valid.p, (size_t)n_series * Tw * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

int b2p_group_aggregate(b2p_ctx* c, int32_t agg, const double* vals, const uint32_t* valid_words, const uint32_t* gid,
                        uint32_t n_series, uint32_t n_groups, uint64_t T, double* out_val, uint32_t* out_cnt) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_groups == 0 || T == 0) return B2P_OK;
  DeviceGuard g(c->device);
  int rc;
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  const size_t ns = n_series ? n_series : 1;
  if ((rc = c->h_aux0.ensure(ns * T * 8))) return rc;
  if ((rc = c->h_aux1.ensure(ns * Tw * 4))) return rc;
  if ((rc = c->h_aux2.ensure(ns * 4))) return rc;
  if ((rc = c->h_out.ensure((size_t)n_groups * T * 8))) return rc;
  if ((rc = c->h_valid.ensure((size_t)n_groups * T * 4))) return rc;
  CU(cudaMemcpyAsync(c->h_aux0.p, vals, (size_t)n_series * T * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_aux1.p, valid_words, (size_t)n_series * Tw * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_aux2.p, gid, (size_t)n_series * 4, cudaMemcpyHostToDevice, c->stream));
  if ((rc = b2p_group_aggregate_dev(c, agg, c->h_aux0.as<double>(), c->h_aux1.as<uint32_t>(), c->h_aux2.as<uint32_t>(),
                                    n_series, n_groups, T, c->h_out.as<double>(), c->h_valid.as<uint32_t>())))
    return rc;
  CU(cudaMemcpyAsync(out_val, c->h_out.p, (size_t)n_groups * T * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(out_cnt, c->h_valid.p, (size_t)n_groups * T * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

int b2p_histogram_quantile(b2p_ctx* c, double phi, const double* le, uint32_t n_buckets, const double* rates,
                           const uint32_t* valid_words, uint32_t n_hist, uint64_t T, double* out,
                           uint32_t* out_valid_words) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  if (n_hist == 0 || T == 0) return B2P_OK;
  DeviceGuard g(c->device);
  int rc;
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  const size_t ns = (size_t)n_hist * n_buckets;
  if ((rc = c->h_aux0.ensure(ns * T * 8))) return rc;
  if ((rc = c->h_aux1.ensure(ns * Tw * 4))) return rc;
  if ((rc = c->h_aux2.ensure((size_t)n_buckets * 8))) return rc;
  if ((rc = c->h_out.ensure((size_t)n_hist * T * 8))) return rc;
  if ((rc = c->h_valid.ensure((size_t)n_hist * Tw * 4))) return rc;
  CU(cudaMemcpyAsync(c->h_aux0.p, rates, ns * T * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_aux1.p, valid_words, ns * Tw * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_aux2.p, le, (size_t)n_buckets * 8, cudaMemcpyHostToDevice, c->stream));
  if ((rc = b2p_histogram_quantile_dev(c, phi, c->h_aux2.as<double>(), n_buckets, c->h_aux0.as<double>(),
                                       c->h_aux1.as<uint32_t>(), n_hist, T, c->h_out.as<double>(),
                                       c->h_valid.as<uint32_t>())))
    return rc;
  CU(cudaMemcpyAsync(out, c->h_out.p, (size_t)n_hist * T * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(out_valid_words, c->h_valid.p, (size_t)n_hist * Tw * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

// histogram_quantile(phi, fn(bucket_series[range])) from host buffers to host rows without the dense [n_series x T]
// matrix ever leaving the device: H2D of the samples, series offsets, the range function into context scratch, the
// HistogramFold over the caller's (histogram -> buckets in le order) index, D2H of [n_hist x T] only.
int b2p_range_histogram_fold(b2p_ctx* c, const b2p_range_params* p, const int64_t* ts, const double* val,
                             const uint32_t* sid, const uint64_t* offsets_host, uint64_t n_rows, uint32_t n_series,
                             double phi, const uint32_t* hist_off, const uint32_t* bucket_series, const double* bucket_le,
                             uint32_t n_hist, double* out, uint32_t* out_valid_words) {
  if (!c) return fail(B2P_E_INVALID, "ctx is NULL");
  int64_t T = 0;
  int rc = check_grid(p, n_series, &T);
  if (rc) return rc;
  if (n_hist == 0 || T == 0) return B2P_OK;
  if (!sid && !offsets_host) return fail(B2P_E_INVALID, "need sid or offsets_host");
  if (!hist_off || !bucket_series || !bucket_le || !out || !out_valid_words || ((!ts || !val) && n_rows))
    return fail(B2P_E_INVALID, "NULL argument");
  DeviceGuard g(c->device);
  if (!c->pending.empty() && (rc = b2p_sync(c))) return rc;
  const uint32_t Tw = (uint32_t)((T + 31) / 32);
  const size_t rows = n_rows ? n_rows : 1;
  const size_t nb = hist_off[n_hist];
  if ((rc = c->h_ts.ensure(rows * 8 + 16)) || (rc = c->h_val.ensure(rows * 8 + 16)) ||
      (rc = c->h_off.ensure(((size_t)n_series + 1) * 8)) || (rc = c->h_out.ensure((size_t)n_series * (size_t)T * 8)) ||
      (rc = c->h_valid.ensure((size_t)n_series * Tw * 4)) || (rc = c->hq_off.ensure(((size_t)n_hist + 1) * 4)) ||
      (rc = c->hq_series.ensure((nb ? nb : 1) * 4)) || (rc = c->hq_les.ensure((nb ? nb : 1) * 8)) ||
      (rc = c->h_aux2.ensure((size_t)n_hist * (size_t)T * 8)) || (rc = c->h_aux3.ensure((size_t)n_hist * Tw * 4)))
    return rc;
  CU(cudaMemcpyAsync(c->h_ts.p, ts, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->h_val.p, val, n_rows * 8, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->hq_off.p, hist_off, ((size_t)n_hist + 1) * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->hq_series.p, bucket_series, nb * 4, cudaMemcpyHostToDevice, c->stream));
  CU(cudaMemcpyAsync(c->hq_les.p, bucket_le, nb * 8, cudaMemcpyHostToDevice, c->stream));
  if (offsets_host) {
    CU(cudaMemcpyAsync(c->h_off.p, offsets_host, ((size_t)n_series + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  } else {
    if ((rc = c->h_sid.ensure(rows * 4 + 16))) return rc;
    CU(cudaMemcpyAsync(c->h_sid.p, sid, n_rows * 4, cudaMemcpyHostToDevice, c->stream));
    if ((rc = series_offsets_impl(c, c->h_sid.as<uint32_t>(), n_rows, n_series, 0u, c->h_off.as<uint64_t>()))) return rc;
  }
  if ((rc = b2p_range_eval_dev(c, p, c->h_ts.as<int64_t>(), c->h_val.as<double>(), c->h_off.as<uint64_t>(), n_rows, n_series,
                               c->h_out.as<double>(), c->h_valid.as<uint32_t>())))
    return rc;
  if ((rc = b2p_sync(c))) return rc;  // slow-path fix-ups land before the fold reads
  if ((rc = b2p_histogram_fold_dev(c, phi, c->hq_off.as<uint32_t>(), c->hq_series.as<uint32_t>(), c->hq_les.as<double>(), n_hist,
                                   c->h_out.as<double>(), c->h_valid.as<uint32_t>(), (uint64_t)T, c->h_aux2.as<double>(),
                                   c->h_aux3.as<uint32_t>())))
    return rc;
  CU(cudaMemcpyAsync(out, c->h_aux2.p, (size_t)n_hist * (size_t)T * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaMemcpyAsync(out_valid_words, c->h_aux3.p, (size_t)n_hist * Tw * 4, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return B2P_OK;
}

}  // extern "C"
