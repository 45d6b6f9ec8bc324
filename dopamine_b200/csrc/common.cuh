// Shared helpers for libb200replay (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>

#include "b200_replay.h"

namespace b2r {

// ---- error plumbing ---------------------------------------------------------
std::string &last_error_slot();
int fail(int code, const char *fmt, ...);
extern std::atomic<int64_t> g_launches;

#define B2R_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t _e = (expr);                                                  \
    if (_e != cudaSuccess)                                                    \
      return ::b2r::fail(B2R_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,        \
                         cudaGetErrorString(_e), __FILE__, __LINE__);         \
  } while (0)

#define B2R_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != B2R_OK) return _s; \
  } while (0)

// Counts the launch and surfaces launch-configuration errors immediately.
#define B2R_LAUNCHED()                                                        \
  do {                                                                        \
    ::b2r::g_launches.fetch_add(1, std::memory_order_relaxed);                \
    B2R_CUDA(cudaGetLastError());                                             \
  } while (0)

static inline cudaStream_t as_stream(b2r_stream s) {
  return reinterpret_cast<cudaStream_t>(s);
}

// The refusals of the versioned state get / set pairs (b2r_sampler_state_*,
// b2r_exchange_state_*), checked before the handle or the device is touched.
static inline int check_state_words(int32_t version, int32_t known_version, int32_t n_words,
                                    int32_t known_words, const void *handle,
                                    const void *words) {
  if (version != known_version)
    return fail(B2R_ERR_INVALID_ARGUMENT, "state version %d is not %d", version,
                known_version);
  if (n_words != known_words)
    return fail(B2R_ERR_INVALID_ARGUMENT, "state of %d words, expected %d", n_words,
                known_words);
  if (!handle || !words) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  return B2R_OK;
}

// Pinned host <-> device bounce buffer that grows on demand.
struct Bounce {
  uint8_t *host = nullptr;
  uint8_t *dev = nullptr;
  size_t cap = 0;
  // A caller that returns before its copy out of `host` has run (b2r_set_priority with
  // host-validated inputs) marks the buffer busy; reserve() waits for that copy.
  cudaEvent_t busy = nullptr;
  bool pending = false;
  int reserve(size_t bytes);
  int mark_busy(cudaStream_t stream);
  void release();
};

// ---- programmatic dependent launch ---------------------------------------------
// The hot-path kernels of one step form a dependent chain of short launches; each
// is launched with programmatic stream serialization so that its launch latency
// overlaps the tail of its predecessor: a kernel lets its successor start
// launching right away (pdl_release) and touches global memory only after its
// own predecessor has completed and flushed (pdl_acquire).
bool pdl_enabled();

// Launch priority of the latency chain (sample -> loss -> write-back): when the
// HBM-bound frame copies of the same step run beside it on another stream, the
// block scheduler must hand freed SM slots to the chain's CTAs first, or the chain
// queues behind tens of thousands of copy CTAs.
int chain_priority();  // the device's greatest stream priority (numerically lowest)

// L2 residency of the sum tree.  The frame copies stream hundreds of MB through the
// 126 MB L2 beside the chain; without protection they evict the 16 MB tree that the
// sampler's descents and the write-back's read-modify-writes live on.  Chain kernels
// are launched with an access-policy window over the tree heap (persisting hits);
// the copy kernels use streaming loads / stores.  set_tree_window() is called by
// the launch sites that touch a tree; the window applies to the next launches made
// through launch() on this thread.
struct TreeWindow {
  void *base = nullptr;
  size_t bytes = 0;
};
TreeWindow &tree_window();
void set_tree_window(void *base, size_t bytes);  // also reserves the L2 set-aside once

// launch_prio_cluster options: launch without programmatic stream serialization even where
// pdl_enabled(); take the tree's L2 window at priority 0 too (the frame copies launch at
// priority 0 precisely so that they stay out of it).
constexpr unsigned kLaunchNoPdl = 1u, kLaunchTreeWindow = 2u;

template <unsigned kFlags = 0u, typename... Params, typename... Args>
cudaError_t launch_prio_cluster(void (*kernel)(Params...), dim3 grid, dim3 block,
                                size_t smem, cudaStream_t stream, int priority,
                                int cluster_x, Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[4];
  int n = 0;
  const TreeWindow &w = tree_window();
  if (w.base != nullptr && (priority != 0 || (kFlags & kLaunchTreeWindow))) {
    attr[n].id = cudaLaunchAttributeAccessPolicyWindow;
    attr[n].val.accessPolicyWindow.base_ptr = w.base;
    attr[n].val.accessPolicyWindow.num_bytes = w.bytes;
    attr[n].val.accessPolicyWindow.hitRatio = 1.0f;
    attr[n].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    attr[n].val.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    ++n;
  }
  if (pdl_enabled() && !(kFlags & kLaunchNoPdl)) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (priority != 0) {
    attr[n].id = cudaLaunchAttributePriority;
    attr[n].val.priority = priority;
    ++n;
  }
  if (cluster_x > 1) {  // the whole grid as thread-block clusters of cluster_x CTAs
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<Params>(args)...);
}

template <typename... Params, typename... Args>
cudaError_t launch_prio(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem,
                        cudaStream_t stream, int priority, Args &&...args) {
  return launch_prio_cluster(kernel, grid, block, smem, stream, priority, 1,
                             static_cast<Args &&>(args)...);
}

// Chain kernels (everything but the frame copies) run at chain priority.
template <typename... Params, typename... Args>
cudaError_t launch(void (*kernel)(Params...), dim3 grid, dim3 block, size_t smem,
                   cudaStream_t stream, Args &&...args) {
  return launch_prio(kernel, grid, block, smem, stream, chain_priority(),
                     static_cast<Args &&>(args)...);
}

// Lets `kernel` launch with up to `bytes` of dynamic shared memory per CTA (above the
// default 48 KB), on the current device.
template <typename K>
int allow_dynamic_smem(K kernel, int bytes) {
  B2R_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  return B2R_OK;
}
// The same once per kernel and process.
template <auto kKernel>
int allow_dynamic_smem_once(int bytes) {
  static bool done = false;
  if (!done) {
    B2R_TRY(allow_dynamic_smem(kKernel, bytes));
    done = true;
  }
  return B2R_OK;
}

// Barrier over the CTAs of a thread-block cluster with release / acquire semantics at
// cluster scope: what the threads of the cluster wrote before it (shared memory of any
// CTA of the cluster, global memory) is visible to all of them after it.
// (SASS: MEMBAR.ALL.GPU, UCGABAR_ARV, UCGABAR_WAIT, CCTL.IVALL — the release is a
// GPU-wide fence, as in cooperative_groups' cluster.sync(); a cheaper hand-over would
// send the few words through st.async onto an mbarrier of the receiving CTA.)
__device__ __forceinline__ void cluster_sync_relacq() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}

// ---- hand-over of a few words between the CTAs of a cluster without a fence ------------
// The receiving CTA owns an mbarrier; a sender stores its word into the receiver's shared
// memory with st.async, which completes `bytes` on that mbarrier when the word has landed;
// the receiver waits for the byte count it expects.  No release fence (barrier.cluster
// .arrive.release is a MEMBAR.ALL.GPU in SASS), only a relaxed cluster barrier at the
// start of the kernel so that nobody sends before the mbarrier exists.
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// The same with acquire at cluster scope: what the senders wrote before their st.async (whose
// complete-tx releases at cluster scope), global memory included, happens before what follows.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// word -> the same shared-memory location in CTA `rank` of the cluster, counted on that
// CTA's mbarrier (both given as THIS CTA's addresses of the corresponding variables)
__device__ __forceinline__ void st_async_u32(void *local_dst, uint32_t value, uint64_t *local_bar,
                                             int rank) {
  uint32_t dst, bar;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(dst) : "r"(smem_u32(local_dst)), "r"(rank));
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(bar) : "r"(smem_u32(local_bar)), "r"(rank));
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(dst),
               "r"(value), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void cluster_arrive_relaxed() {
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");
}

__device__ __forceinline__ void pdl_release() {
  asm volatile("griddepcontrol.launch_dependents;");
}
__device__ __forceinline__ void pdl_acquire() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ---- hand-over of a few words between kernels through global memory ---------------------
// A signaller publishes a word with release; its consumers poll it with acquire, and what
// the signaller wrote before the release is visible to them once they have seen the word.
__device__ __forceinline__ void st_release_u32(unsigned int *p, unsigned int v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int *p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Peer memory (NVLink / NVSwitch): relaxed at system scope.
__device__ __forceinline__ void st_sys_u64(uint64_t *p, uint64_t v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_sys_u64(const uint64_t *p) {
  uint64_t v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ uint64_t global_timer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// How long a consumer polls a hand-over word before it gives up: 4e9 clock64 cycles, about
// 2 s at the B200's clocks.  A signaller that never ran (its launch failed, and the caller has
// been told) must not hang the GPU; every consumer has a safe fallback, normally its
// griddepcontrol.wait.
constexpr long long kSpinLimit = 4000000000ll;

// Polls *word with acquire until ready(value) holds: false once kSpinLimit has passed.
// kBackoffNs > 0: a __nanosleep between polls.
template <int kBackoffNs = 0, typename Ready>
__device__ __forceinline__ bool poll_acquire(const unsigned int *word, Ready ready) {
  const long long t0 = clock64();
  while (!ready(ld_acquire_u32(word))) {
    if (clock64() - t0 > kSpinLimit) return false;
    if (kBackoffNs > 0) __nanosleep(kBackoffNs);
  }
  return true;
}

// Polls a peer-memory mailbox word until its low 32 bits carry step `seq`: true with the word
// in *w, false once timeout_ns of %globaltimer have passed.
__device__ __forceinline__ bool poll_tagged_word(const uint64_t *src, uint64_t seq,
                                                 int64_t timeout_ns, uint64_t *w) {
  const uint64_t t0 = global_timer_ns();
  for (;;) {
    *w = ld_sys_u64(src);
    if ((uint32_t)*w == (uint32_t)seq) return true;
    if (global_timer_ns() - t0 > (uint64_t)timeout_ns) return false;
  }
}

// Launch numbers from tickets: every CTA of a launch takes one ticket before it lets its
// dependents start, so the tickets of consecutive launches never interleave.  `launch` is the
// launch's number counted from 1, `arrival` the CTA's place within its launch.
struct LaunchTicket {
  unsigned int launch, arrival;
};
__device__ __forceinline__ LaunchTicket launch_ticket(unsigned long long *tickets,
                                                      unsigned int ctas) {
  const unsigned long long t = atomicAdd(tickets, 1ull);
  return {(unsigned int)(t / ctas) + 1u, (unsigned int)(t % ctas)};
}

// Last-CTA election, by thread 0 of every CTA of the launch: true in the CTA that arrives
// last.  rearm: that CTA resets the ticket for the next launch at once; a caller that passes
// false resets it itself, later (the next launch takes its tickets behind its own
// griddepcontrol.wait, so any point before this launch ends will do).
__device__ __forceinline__ bool arrive_last(unsigned int *ticket, bool rearm = true) {
  const bool last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  if (rearm && last) *ticket = 0u;
  return last;
}
// The same for the whole CTA (every thread calls it; s_last in shared memory): the CTA that
// arrives last sees everything the others wrote before they arrived.
__device__ __forceinline__ bool last_cta(unsigned int *ticket, bool *s_last, bool rearm = true) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) *s_last = arrive_last(ticket, rearm);
  __syncthreads();
  const bool last = *s_last;
  if (last) __threadfence();
  return last;
}

// ---- optional phase tracing (build with -DB2R_TRACE; never in the shipped .so) ---
#ifdef B2R_TRACE
// -DB2R_TRACE_GT: marks are %globaltimer nanoseconds (one clock for all kernels and
// SMs: a timeline of the whole step); otherwise clock64 cycles of the marking SM.
#ifdef B2R_TRACE_GT
__device__ __forceinline__ long long b2r_now() { return (long long)global_timer_ns(); }
#else
__device__ __forceinline__ long long b2r_now() { return clock64(); }
#endif
#define B2R_TRACE_DECL static __device__ long long g_trace[32];
#define B2R_MARK(i)                                              \
  do {                                                           \
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0)  \
      g_trace[i] = b2r_now();                                    \
  } while (0)
// mark from thread 0 of a chosen CTA (blockIdx.x == blk)
#define B2R_MARK_CTA(i, blk)                                 \
  do {                                                       \
    if ((int)blockIdx.x == (blk) && threadIdx.x == 0)        \
      g_trace[i] = b2r_now();                                \
  } while (0)
// mark from thread 0 of the CTA for which `cond` holds
#define B2R_MARK_IF(i, cond)                                 \
  do {                                                       \
    if ((cond) && threadIdx.x == 0) g_trace[i] = b2r_now();  \
  } while (0)
// mark from thread 0 of whichever CTA gets there (e.g. the last one to finish)
#define B2R_MARK_ANY(i)                        \
  do {                                         \
    if (threadIdx.x == 0) g_trace[i] = b2r_now(); \
  } while (0)
// the latest time any CTA passed here
#define B2R_MARK_END(i)                                                         \
  do {                                                                          \
    if (threadIdx.x == 0)                                                       \
      atomicMax(reinterpret_cast<unsigned long long *>(&g_trace[i]),            \
                (unsigned long long)b2r_now());                                 \
  } while (0)
#else
#define B2R_TRACE_DECL
#define B2R_MARK(i) \
  do {              \
  } while (0)
#define B2R_MARK_ANY(i) \
  do {                  \
  } while (0)
#define B2R_MARK_END(i) \
  do {                  \
  } while (0)
#define B2R_MARK_CTA(i, blk) \
  do {                       \
  } while (0)
#define B2R_MARK_IF(i, cond) \
  do {                       \
  } while (0)
#endif

// ---- device helpers ----------------------------------------------------------
__device__ __forceinline__ int64_t wrap_index(int64_t i, int64_t cap) {
  int64_t r = i % cap;
  return r < 0 ? r + cap : r;
}

// Philox4x32-10 (Salmon et al. 2011), counter = (lo, hi, stream, 0), key = seed.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1,
                                              uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1,
                                              uint32_t out[4]) {
  // Rolled on purpose: these kernels run once per launch on a cold instruction
  // cache, where every extra 128-byte line of straight-line code costs an L2 trip.
#pragma unroll 1
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// 53-bit uniform in [0,1) from draw number `n` of stream (seed, offset).
__device__ __forceinline__ double philox_uniform53(uint64_t seed, uint64_t offset,
                                                   uint64_t n) {
  uint32_t o[4];
  philox4x32_10((uint32_t)n, (uint32_t)(n >> 32), (uint32_t)offset,
                (uint32_t)(offset >> 32), (uint32_t)seed, (uint32_t)(seed >> 32),
                o);
  uint64_t a = o[0] >> 5, b = o[1] >> 6;  // 27 + 26 bits
  return (double)((a << 26) | b) * (1.0 / 9007199254740992.0);
}

// The same draw with the ten rounds unrolled and each 32 x 32 product taken once as a
// 64-bit multiply: a dependent chain of ~20 instructions instead of ~140.  For kernels
// where a lone warp waits on the draw (the warp sampler).
__device__ __forceinline__ double philox_uniform53_fast(uint64_t seed, uint64_t offset,
                                                        uint64_t n) {
  uint32_t c0 = (uint32_t)n, c1 = (uint32_t)(n >> 32), c2 = (uint32_t)offset,
           c3 = (uint32_t)(offset >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  const uint64_t hi = c0 >> 5, lo = c1 >> 6;  // 27 + 26 bits
  return (double)((hi << 26) | lo) * (1.0 / 9007199254740992.0);
}

}  // namespace b2r
