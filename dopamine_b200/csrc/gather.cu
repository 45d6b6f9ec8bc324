// Fused batch assembly: replaces the per-index Python loop of
// OutOfGraphReplayBuffer.sample_transition_batch (circular_replay_buffer.py:516-556,
// stacks via 338-375) and the sampling_probabilities fill of the prioritized
// buffer (prioritized_replay_buffer.py:193-200).
//
// Per sampled index i (one launch for the whole batch):
//   L         = 1 + offset of the first non-zero terminal in slots i..i+n-1, else n
//   state     = frames i-S+1..i,      stack axis innermost  (np.moveaxis, CRB:375)
//   next_state= frames i+L-S+1..i+L   (deterministic even when terminal, Q14)
//   reward    = np.sum(f32(gamma^k) * r[i+k], k < L)  in numpy's f32 order
//   next_action / next_reward = rows at (i+L) mod C; action/extras = rows at i
//   terminal  = any terminal in the trajectory; indices = i; priorities = leaf(i)
//
// HBM-bound byte movement: per transition (S=4, n=3, 84x84 u8) 7 unique frames are
// read (49 392 B, one contiguous span of the ring unless it wraps) and 2 x 28 224 B
// written.  Fast path (S=4, 1-byte pixels, frame % 16 == 0): each thread moves one
// 16-pixel column of the span — up to 7 x LDG.128, a PRMT byte-transpose into the
// [pixel][stack] interleave, 8 x STG.128 — with frames shared between state and
// next_state read once.
#include "gather.cuh"

#include <cstdlib>
#include <cstring>

namespace b2r {
namespace {

B2R_TRACE_DECL

struct GatherArgs {
  int64_t capacity;
  int32_t stack, horizon, batch;
  int64_t obs_bytes;
  int32_t obs_itemsize;
  const uint8_t *obs;
  const uint8_t *term_flag;
  const int32_t *indices;
  uint8_t *state, *next_state;
  int32_t scalar_rows;   // grid rows of appended scalar CTAs (0: frames only)
  ScalarArgs sc;
  const int32_t *count;  // nullable: device-side number of rows (<= batch)
  LaunchGate gate;         // the one-stream step (TMA copies only; done == nullptr: none)
};

// [a0 a1 a2 a3] x4 frames -> 4 words [a_p b_p c_p d_p], p = 0..3.
__device__ __forceinline__ uint4 interleave4(uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  const uint32_t ab_lo = __byte_perm(a, b, 0x5140);  // a0 b0 a1 b1
  const uint32_t ab_hi = __byte_perm(a, b, 0x7362);  // a2 b2 a3 b3
  const uint32_t cd_lo = __byte_perm(c, d, 0x5140);
  const uint32_t cd_hi = __byte_perm(c, d, 0x7362);
  uint4 o;
  o.x = __byte_perm(ab_lo, cd_lo, 0x5410);  // a0 b0 c0 d0
  o.y = __byte_perm(ab_lo, cd_lo, 0x7632);  // a1 b1 c1 d1
  o.z = __byte_perm(ab_hi, cd_hi, 0x5410);
  o.w = __byte_perm(ab_hi, cd_hi, 0x7632);
  return o;
}

__device__ __forceinline__ void store_stack16(uint8_t *dst, const uint4 f0,
                                              const uint4 f1, const uint4 f2,
                                              const uint4 f3) {
  uint4 *d = reinterpret_cast<uint4 *>(dst);
  __stcs(d + 0, interleave4(f0.x, f1.x, f2.x, f3.x));
  __stcs(d + 1, interleave4(f0.y, f1.y, f2.y, f3.y));
  __stcs(d + 2, interleave4(f0.z, f1.z, f2.z, f3.z));
  __stcs(d + 3, interleave4(f0.w, f1.w, f2.w, f3.w));
}

__device__ __forceinline__ uint4 load_frame16(const uint8_t *__restrict__ obs,
                                              int64_t slot, int64_t cap,
                                              int64_t obs_bytes, int chunk) {
  if (slot < 0) slot += cap;
  if (slot >= cap) slot -= cap;
  // streamed: every frame byte is read once per batch; keep L2 for the sum tree
  return __ldcs(reinterpret_cast<const uint4 *>(obs + slot * obs_bytes) + chunk);
}

// Fast path: stack 4, 1-byte pixels, obs_bytes % 16 == 0.
// grid = (ceil(chunks / blockDim), batch); thread = one 16-pixel column.
// SCALARS: the grid carries appended CTAs that write the scalar columns.
template <bool SCALARS>
__global__ void __launch_bounds__(128, 12) gather_stack4_u8_kernel(const __grid_constant__ GatherArgs a) {
  B2R_MARK(0);
  pdl_release();
  const int b = blockIdx.y;
  pdl_acquire();
  B2R_MARK(1);
  const int rows = a.count ? min(*a.count, a.batch) : a.batch;
  if (SCALARS && blockIdx.y >= a.batch) {  // appended scalar CTAs: one thread per transition
    const int r = ((blockIdx.y - a.batch) * gridDim.x + blockIdx.x) * blockDim.x +
                  threadIdx.x;
    if (r < rows) write_scalars(a.sc, r, a.indices[r]);
    return;
  }
  if (b >= rows) return;
  const int64_t i = a.indices[b];
  bool ends;
  const int length = trajectory_length(a.term_flag, i, a.horizon, a.capacity, &ends);
  B2R_MARK(2);

  const int chunks = (int)(a.obs_bytes >> 4);
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= chunks) return;

  // frames i-3 .. i
  const uint4 s0 = load_frame16(a.obs, i - 3, a.capacity, a.obs_bytes, c);
  const uint4 s1 = load_frame16(a.obs, i - 2, a.capacity, a.obs_bytes, c);
  const uint4 s2 = load_frame16(a.obs, i - 1, a.capacity, a.obs_bytes, c);
  const uint4 s3 = load_frame16(a.obs, i, a.capacity, a.obs_bytes, c);
  // frames i+L-3 .. i+L: the first 4-L of them are state frames already loaded.
  uint4 n0, n1, n2, n3;
  const int64_t j = i + length;  // < 2 * capacity
  if (length == 1) {
    n0 = s1; n1 = s2; n2 = s3;
    n3 = load_frame16(a.obs, j, a.capacity, a.obs_bytes, c);
  } else if (length == 2) {
    n0 = s2; n1 = s3;
    n2 = load_frame16(a.obs, j - 1, a.capacity, a.obs_bytes, c);
    n3 = load_frame16(a.obs, j, a.capacity, a.obs_bytes, c);
  } else if (length == 3) {
    n0 = s3;
    n1 = load_frame16(a.obs, j - 2, a.capacity, a.obs_bytes, c);
    n2 = load_frame16(a.obs, j - 1, a.capacity, a.obs_bytes, c);
    n3 = load_frame16(a.obs, j, a.capacity, a.obs_bytes, c);
  } else {
    n0 = load_frame16(a.obs, j - 3, a.capacity, a.obs_bytes, c);
    n1 = load_frame16(a.obs, j - 2, a.capacity, a.obs_bytes, c);
    n2 = load_frame16(a.obs, j - 1, a.capacity, a.obs_bytes, c);
    n3 = load_frame16(a.obs, j, a.capacity, a.obs_bytes, c);
  }
  const int64_t out_off = (int64_t)b * a.obs_bytes * 4 + (int64_t)c * 64;
  B2R_MARK(4);
  if (a.state) store_stack16(a.state + out_off, s0, s1, s2, s3);
  if (a.next_state) store_stack16(a.next_state + out_off, n0, n1, n2, n3);
  B2R_MARK(5);
  B2R_MARK_END(6);
}

// ---- TMA variant of the fast path ------------------------------------------------
// One CTA per transition.  An elected thread computes the trajectory length and
// issues one bulk asynchronous copy (cp.async.bulk, the 1-D form of TMA) per unique
// frame — 7 x 7 056 B for n = 3 — from the ring into shared memory, completing on
// an mbarrier; all threads then read the staged frames 4 bytes per frame at a time
// (conflict-free), interleave them into the [pixel][stack] order and write 16-byte
// chunks that consecutive threads place consecutively (fully coalesced stores).
// The ring is read in 7 KB bursts by the copy engine instead of by 16-byte loads
// held in registers, so few threads keep the whole transition in flight.
constexpr int kTmaThreads = 256;
constexpr int kTmaMaxFrames = 8;

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes,
                                         uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

template <bool SCALARS>
__global__ void __launch_bounds__(kTmaThreads)
gather_stack4_u8_tma_kernel(const __grid_constant__ GatherArgs a) {
  extern __shared__ __align__(128) uint8_t tma_smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ int s_length;
  __shared__ bool s_rows;
  B2R_MARK(0);
  pdl_release();
  // The one-stream step: the predecessor is the first half of the loss; the indices are
  // final once the sampler has counted its launch (StageGate::rows), and the
  // griddepcontrol.wait moves to the end (the copies have landed when the step's last
  // kernel completes).
  const bool gated = a.gate.done != nullptr;
  if (!(gated && cta_gate_wait<32>(a.gate, &s_rows))) pdl_acquire();
  B2R_MARK(1);
  const int rows = a.count ? min(*a.count, a.batch) : a.batch;
  if (SCALARS && (int)blockIdx.x >= a.batch) {  // appended scalar CTAs
    const int b = ((int)blockIdx.x - a.batch) * blockDim.x + threadIdx.x;
    if (b < rows) write_scalars(a.sc, b, a.indices[b]);
    return;
  }
  const int b = blockIdx.x;
  if (b >= rows) return;
  const uint32_t frame = (uint32_t)a.obs_bytes;
  if (threadIdx.x == 0) mbar_init(&bar, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    const int64_t i = a.indices[b];
    bool ends;
    const int length = trajectory_length(a.term_flag, i, a.horizon, a.capacity, &ends);
    const int shared_frames = length < 4 ? length : 4;  // next-state frames beyond `state`
    const int unique = 4 + shared_frames;
    s_length = length;
    mbar_expect_tx(&bar, (uint32_t)unique * frame);
    for (int k = 0; k < unique; ++k) {
      // slots 0..3: frames i-3..i; slots 4..: the frames of next_state not among them
      int64_t slot = k < 4 ? i - 3 + k : i + length - 3 + (k - shared_frames);
      if (slot < 0) slot += a.capacity;
      if (slot >= a.capacity) slot -= a.capacity;
      bulk_g2s(tma_smem + (size_t)k * frame, a.obs + slot * a.obs_bytes, frame, &bar);
    }
  }
  mbar_wait(&bar, 0);
  const int length = s_length;
  const int next_base = length < 4 ? length : 4;  // slot of next_state's first frame
  const int chunks = (int)(frame >> 2);           // 16-byte output chunks per stack
  uint8_t *out_state = a.state ? a.state + (int64_t)b * frame * 4 : nullptr;
  uint8_t *out_next = a.next_state ? a.next_state + (int64_t)b * frame * 4 : nullptr;
  const uint32_t *f = reinterpret_cast<const uint32_t *>(tma_smem);
  const uint32_t words = frame >> 2;  // 4-byte words per frame
#pragma unroll 2
  for (int o = threadIdx.x; o < chunks; o += kTmaThreads) {
    if (out_state) {
      const uint4 v = interleave4(f[o], f[words + o], f[2 * words + o], f[3 * words + o]);
      reinterpret_cast<uint4 *>(out_state)[o] = v;
    }
    if (out_next) {
      const uint32_t *g = f + (size_t)next_base * words;
      const uint4 v = interleave4(g[o], g[words + o], g[2 * words + o], g[3 * words + o]);
      reinterpret_cast<uint4 *>(out_next)[o] = v;
    }
  }
  B2R_MARK_END(6);
  if (gated) pdl_acquire();
}

// General path: any stack size / element size. thread = one observation element.
__global__ void __launch_bounds__(256) gather_generic_kernel(const __grid_constant__ GatherArgs a) {
  pdl_release();
  pdl_acquire();
  const int rows = a.count ? min(*a.count, a.batch) : a.batch;
  if (blockIdx.y >= a.batch) {  // appended scalar CTAs: one thread per transition
    const int b = ((blockIdx.y - a.batch) * gridDim.x + blockIdx.x) * blockDim.x +
                  threadIdx.x;
    if (b < rows) write_scalars(a.sc, b, a.indices[b]);
    return;
  }
  const int b = blockIdx.y;
  if (b >= rows) return;
  const int64_t i = a.indices[b];
  bool ends;
  const int length = trajectory_length(a.term_flag, i, a.horizon, a.capacity, &ends);

  const int es = a.obs_itemsize;
  const int64_t elems = a.obs_bytes / es;
  const int64_t j = i + length;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < elems;
       e += (int64_t)gridDim.x * blockDim.x) {
    for (int k = 0; k < a.stack; ++k) {
      const int64_t fs = wrap_index(i - a.stack + 1 + k, a.capacity);
      const int64_t fn = wrap_index(j - a.stack + 1 + k, a.capacity);
      const uint8_t *ps = a.obs + fs * a.obs_bytes + e * es;
      const uint8_t *pn = a.obs + fn * a.obs_bytes + e * es;
      const int64_t o = ((int64_t)b * elems * a.stack + e * a.stack + k) * es;
      for (int q = 0; q < es; ++q) {
        if (a.state) a.state[o + q] = ps[q];
        if (a.next_state) a.next_state[o + q] = pn[q];
      }
    }
  }
}

__global__ void get_priority_kernel(const double *__restrict__ leaves, int64_t n,
                                    const int32_t *__restrict__ indices,
                                    float *__restrict__ out) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) out[k] = (float)leaves[indices[k]];
}

}  // namespace

// 0: register path (LDG.128 -> PRMT -> STG.128), 1: TMA-staged path (cp.async.bulk into
// shared memory on an mbarrier), for a launch of `batch` rows.  B2R_GATHER = reg | tma
// forces one; the default follows the measurements (profiles/r2/README.md: CUDA-event
// times of the fused step and ncu --set full of both kernels at 32 / 256 / 1024 / 4096):
// the TMA kernel issues half the instructions and reaches 67 % of DRAM throughput at
// batch 4096 against 56 % (fused step 100 us against 111 us; 24.5 against 26.0 at 256).
// Between those sizes, where the copies run beside the next step's chain, the register
// kernel with its occupancy cap used to be the faster one (37.2 against 39.8 us at 1024)
// — while the write-back sorted on a side stream and needed the room.  With the
// write-back that groups ahead of its values (tree.cu, kEarly) the TMA kernel wins there
// too: 28.6 / 33.2 / 50.3 us at 768 / 1024 / 1536 rows against 33.5 / 36.8 / 57.2
// (profiles/r2/out/run71.txt .. run73.txt), so it is the default at every size.
int gather_variant(int batch) {
  static const int forced = [] {
    const char *e = std::getenv("B2R_GATHER");
    if (e == nullptr || std::strcmp(e, "auto") == 0) return -1;
    return std::strcmp(e, "tma") == 0 ? 1 : 0;
  }();
  if (forced >= 0) return forced;
  (void)batch;
  return 1;
}

void fill_scalar_args(const b2r_buffer *b, const b2r_batch *out, ScalarArgs *sc) {
  sc->capacity = b->cfg.capacity;
  sc->horizon = b->cfg.update_horizon;
  sc->term_flag = b->term_flag;
  sc->reward = b->col[2].dev;
  sc->reward_itemsize = b->cfg.reward_itemsize;
  sc->discounts = b->discounts;
  sc->ret = out->reward;
  sc->terminal_out = static_cast<uint8_t *>(out->terminal);
  sc->terminal_itemsize = b->cfg.terminal_itemsize;
  sc->indices_out = out->indices;
  sc->n_copies = 0;
  auto add_copy = [&](int column, void *dst, int at_next) {
    if (!dst) return;
    RowCopy &rc = sc->copies[sc->n_copies++];
    rc.src = b->col[column].dev;
    rc.dst = static_cast<uint8_t *>(dst);
    rc.row_bytes = (int32_t)b->col[column].row_bytes;
    rc.at_next = at_next;
  };
  add_copy(B2R_COL_ACTION, out->action, 0);
  add_copy(B2R_COL_ACTION, out->next_action, 1);
  add_copy(B2R_COL_REWARD, out->next_reward, 1);
  for (int e = 0; e < b->cfg.num_extras; ++e)
    add_copy(B2R_COL_EXTRA0 + e, out->extras[e], 0);
  sc->leaves = nullptr;
  sc->prio_out = nullptr;
  if (b->tree && out->sampling_probabilities) {
    sc->leaves = b->tree->heap + b->tree->leaves;
    sc->prio_out = out->sampling_probabilities;
  }
  sc->fast = b->cfg.update_horizon <= kFastHorizon && b->cfg.reward_itemsize == 4 &&
             b->cfg.terminal_itemsize == 1 && b->cfg.action_bytes == 4 &&
             b->cfg.num_extras == 0;
  sc->action_col = reinterpret_cast<const uint32_t *>(b->col[B2R_COL_ACTION].dev);
  sc->action_out = static_cast<uint32_t *>(out->action);
  sc->next_action_out = static_cast<uint32_t *>(out->next_action);
  sc->next_reward_out = static_cast<float *>(out->next_reward);
}

// Gated copies always launch this many CTAs (those beyond the batch only take their ticket):
// a launch's number is ticket / CTAs only while every launch has the same grid.
constexpr int kGatedCopyCtas = kTinyBatch;

bool gather_can_gate(const b2r_buffer *b, int32_t batch) {
  return batch <= kGatedCopyCtas && b->cfg.stack_size == 4 && b->cfg.obs_itemsize == 1 && (b->cfg.obs_bytes & 15) == 0 &&
         gather_variant(batch) == 1 &&
         (size_t)kTmaMaxFrames * (size_t)b->cfg.obs_bytes <= 200 * 1024;
}

int launch_gather(b2r_buffer *b, int32_t batch, const int32_t *indices_dev,
                  const b2r_batch *out, cudaStream_t stream,
                  const int32_t *count_dev, bool frames_only, const LaunchGate *gate) {
  if (gate != nullptr && (count_dev != nullptr || !frames_only || !gather_can_gate(b, batch)))
    return fail(B2R_ERR_INVALID_ARGUMENT, "only the TMA frame copies of a counted batch gate");
  GatherArgs a;
  if (gate != nullptr) a.gate = *gate;
  a.count = count_dev;
  a.capacity = b->cfg.capacity;
  a.stack = b->cfg.stack_size;
  a.horizon = b->cfg.update_horizon;
  a.batch = batch;
  a.obs_bytes = b->cfg.obs_bytes;
  a.obs_itemsize = b->cfg.obs_itemsize;
  a.obs = b->col[0].dev;
  a.term_flag = b->term_flag;
  a.indices = indices_dev;
  a.state = static_cast<uint8_t *>(out->state);
  a.next_state = static_cast<uint8_t *>(out->next_state);
  fill_scalar_args(b, out, &a.sc);
  if (frames_only && !a.state && !a.next_state) return B2R_OK;
  const bool fast = a.stack == 4 && a.obs_itemsize == 1 && (a.obs_bytes & 15) == 0;
  const size_t tma_bytes = (size_t)kTmaMaxFrames * (size_t)a.obs_bytes;
  if (fast && gather_variant(batch) == 1 && tma_bytes <= 200 * 1024) {
    B2R_TRY(allow_dynamic_smem_once<gather_stack4_u8_tma_kernel<true>>(200 * 1024));
    B2R_TRY(allow_dynamic_smem_once<gather_stack4_u8_tma_kernel<false>>(200 * 1024));
    a.scalar_rows = frames_only ? 0 : (batch + kTmaThreads - 1) / kTmaThreads;
    dim3 grid(gate != nullptr ? kGatedCopyCtas : batch + a.scalar_rows);
    if (frames_only)
      B2R_CUDA(launch_prio(gather_stack4_u8_tma_kernel<false>, grid, dim3(kTmaThreads),
                           tma_bytes, stream, 0, a));
    else
      B2R_CUDA(launch(gather_stack4_u8_tma_kernel<true>, grid, dim3(kTmaThreads),
                      tma_bytes, stream, a));
  } else if (fast) {
    const int chunks = (int)(a.obs_bytes >> 4);
    const int nx = (chunks + 127) / 128;
    // + rows of scalar CTAs (one thread per transition)
    a.scalar_rows = frames_only ? 0 : (batch + nx * 128 - 1) / (nx * 128);
    dim3 grid(nx, batch + a.scalar_rows);
    if (frames_only) {  // beside the chain: lowest priority
      // While the copies are short next to the chain (up to ~1.5k rows) each copy CTA
      // claims 56 KB of shared memory it does not use: at most 4 of them then share an
      // SM, which leaves the chain's CTAs their occupancy (65 -> 58 us per step at
      // batch 1024).  Beyond that the copies themselves bound the step and run
      // unrestricted (capping costs 146 -> 162 us at 4096).
      const int pad_kb = batch > 64 && batch <= 1536 ? 56 : 0;
      if (pad_kb > 0)
        B2R_TRY(allow_dynamic_smem_once<gather_stack4_u8_kernel<false>>(pad_kb * 1024));
      B2R_CUDA(launch_prio(gather_stack4_u8_kernel<false>, grid, dim3(128),
                           (size_t)pad_kb * 1024, stream, 0, a));
    }
    else
      B2R_CUDA(launch(gather_stack4_u8_kernel<true>, grid, dim3(128), 0, stream, a));
  } else {
    const int64_t elems = a.obs_bytes / a.obs_itemsize;
    int gx = (int)((elems + 255) / 256);
    if (gx > 32) gx = 32;
    a.scalar_rows = frames_only ? 0 : (batch + gx * 256 - 1) / (gx * 256);
    dim3 grid(gx, batch + a.scalar_rows);
    B2R_CUDA(launch_prio(gather_generic_kernel, grid, dim3(256), 0, stream,
                         frames_only ? 0 : chain_priority(), a));
  }
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" {

int32_t b2r_gather_variant(const b2r_buffer *b, int32_t batch) {
  if (!b) return -1;
  const bool fast = b->cfg.stack_size == 4 && b->cfg.obs_itemsize == 1 &&
                    (b->cfg.obs_bytes & 15) == 0;
  if (!fast) return 2;
  return b2r::gather_variant(batch) == 1 &&
                 (size_t)b2r::kTmaMaxFrames * (size_t)b->cfg.obs_bytes <= 200 * 1024
             ? 1 : 0;
}

int b2r_gather_device(b2r_buffer *b, int32_t batch, const int32_t *indices,
                      const b2r_batch *out, b2r_stream stream) {
  if (batch <= 0 || batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "batch must be in [1, 60000]");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  return b2r::launch_gather(b, batch, indices, out, as_stream(stream));
}

int b2r_gather_device_counted(b2r_buffer *b, int32_t max_batch,
                              const int32_t *count, const int32_t *indices,
                              const b2r_batch *out, b2r_stream stream) {
  if (max_batch <= 0 || max_batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "max_batch must be in [1, 60000]");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  return b2r::launch_gather(b, max_batch, indices, out, as_stream(stream), count);
}

namespace {

// Layout of every requested output column in ONE slab, 256-byte aligned segments in a
// fixed order, the indices the kernel reads first.  `want`: a non-null field = the
// column is wanted.  Fills `at` with pointers into `base` and returns the slab size.
size_t slab_layout(const b2r_buffer *b, int32_t batch, const b2r_batch *want,
                   uint8_t *base, b2r_batch *at, size_t *indices_off) {
  size_t total = 0;
  auto seg = [&](size_t bytes) -> uint8_t * {
    uint8_t *p = base + total;
    total += (bytes + 255) & ~(size_t)255;
    return p;
  };
  const size_t B = (size_t)batch;
  const size_t stack_bytes = (size_t)b->cfg.obs_bytes * b->cfg.stack_size;
  memset(at, 0, sizeof(*at));
  *indices_off = total;
  uint8_t *idx = seg(B * 4);
  if (want->state) at->state = seg(B * stack_bytes);
  if (want->action) at->action = seg(B * b->cfg.action_bytes);
  if (want->reward) at->reward = seg(B * b->cfg.reward_itemsize);
  if (want->next_state) at->next_state = seg(B * stack_bytes);
  if (want->next_action) at->next_action = seg(B * b->cfg.action_bytes);
  if (want->next_reward) at->next_reward = seg(B * b->cfg.reward_itemsize);
  if (want->terminal) at->terminal = seg(B * b->cfg.terminal_itemsize);
  // the kernel's index input doubles as the `indices` output column
  if (want->indices) at->indices = reinterpret_cast<int32_t *>(idx);
  for (int e = 0; e < b->cfg.num_extras; ++e)
    if (want->extras[e]) at->extras[e] = seg(B * b->cfg.extra_bytes[e]);
  if (want->sampling_probabilities)
    at->sampling_probabilities = reinterpret_cast<float *>(seg(B * 4));
  return total;
}

int ensure_out_scratch(b2r_buffer *b, size_t total) {
  if (total <= b->out_scratch_cap) return B2R_OK;
  if (b->out_scratch) cudaFree(b->out_scratch);
  b->out_scratch = nullptr;
  b->out_scratch_cap = 0;
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->out_scratch), total));
  b->out_scratch_cap = total;
  return B2R_OK;
}

}  // namespace

int b2r_gather(b2r_buffer *b, int32_t batch, const int32_t *indices,
               const b2r_batch *out, b2r_stream stream) {
  if (batch <= 0 || batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "batch must be in [1, 60000]");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  // Device scratch for every requested output, then one copy per column into the
  // caller's (pageable) arrays.  b2r_gather_slab is the fast form of this call.
  b2r_batch d;
  size_t off_idx = 0;
  const size_t total = slab_layout(b, batch, out, nullptr, &d, &off_idx);
  B2R_TRY(ensure_out_scratch(b, total));
  uint8_t *base = b->out_scratch;
  auto dev = [&](const void *p) -> uint8_t * {  // (offsets were laid out against nullptr)
    return base + reinterpret_cast<size_t>(p);
  };
  const size_t B = (size_t)batch;
  const size_t stack_bytes = (size_t)b->cfg.obs_bytes * b->cfg.stack_size;
  struct Copy { void *host; const uint8_t *dev; size_t bytes; };
  Copy copies[8 + B2R_MAX_EXTRAS + 2];
  int n = 0;
  b2r_batch k;
  memset(&k, 0, sizeof(k));
  auto col = [&](void *host, const void *at, size_t bytes) -> void * {
    if (!host) return nullptr;
    copies[n++] = {host, dev(at), bytes};
    return dev(at);
  };
  k.state = col(out->state, d.state, B * stack_bytes);
  k.action = col(out->action, d.action, B * b->cfg.action_bytes);
  k.reward = col(out->reward, d.reward, B * b->cfg.reward_itemsize);
  k.next_state = col(out->next_state, d.next_state, B * stack_bytes);
  k.next_action = col(out->next_action, d.next_action, B * b->cfg.action_bytes);
  k.next_reward = col(out->next_reward, d.next_reward, B * b->cfg.reward_itemsize);
  k.terminal = col(out->terminal, d.terminal, B * b->cfg.terminal_itemsize);
  if (out->indices) {
    copies[n++] = {out->indices, base + off_idx, B * 4};
    k.indices = nullptr;  // (the kernel's input already is that column)
  }
  for (int e = 0; e < b->cfg.num_extras; ++e)
    k.extras[e] = col(out->extras[e], d.extras[e], B * b->cfg.extra_bytes[e]);
  k.sampling_probabilities = static_cast<float *>(
      col(out->sampling_probabilities, d.sampling_probabilities, B * 4));
  B2R_CUDA(cudaMemcpyAsync(base + off_idx, indices, B * 4, cudaMemcpyHostToDevice, s));
  B2R_TRY(b2r::launch_gather(b, batch,
                             reinterpret_cast<const int32_t *>(base + off_idx), &k, s));
  for (int c = 0; c < n; ++c)
    B2R_CUDA(cudaMemcpyAsync(copies[c].host, copies[c].dev, copies[c].bytes,
                             cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  return B2R_OK;
}

int b2r_gather_slab(b2r_buffer *b, int32_t batch, const int32_t *indices,
                    int32_t indices_on_device, const b2r_batch *want, void *host_slab,
                    size_t slab_bytes, b2r_batch *host_out, size_t *needed,
                    b2r_stream stream) {
  if (!b || !want || !host_out || !needed)
    return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  if (batch <= 0 || batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "batch must be in [1, 60000]");
  size_t off_idx = 0;
  const size_t total =
      slab_layout(b, batch, want, static_cast<uint8_t *>(host_slab), host_out, &off_idx);
  *needed = total;
  if (host_slab == nullptr) return B2R_OK;  // (size query: *host_out holds the offsets)
  if (slab_bytes < total) {
    memset(host_out, 0, sizeof(*host_out));
    return fail(B2R_ERR_INVALID_ARGUMENT, "the slab holds %zu bytes, the batch needs %zu",
                slab_bytes, total);
  }
  if (!indices) return fail(B2R_ERR_INVALID_ARGUMENT, "indices is NULL");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  B2R_TRY(ensure_out_scratch(b, total));
  uint8_t *base = b->out_scratch;
  b2r_batch d;
  size_t unused = 0;
  slab_layout(b, batch, want, base, &d, &unused);
  d.indices = nullptr;  // (the kernel's input already is that column)
  B2R_CUDA(cudaMemcpyAsync(base + off_idx, indices, (size_t)batch * 4,
                           indices_on_device ? cudaMemcpyDeviceToDevice
                                             : cudaMemcpyHostToDevice, s));
  B2R_TRY(b2r::launch_gather(b, batch,
                             reinterpret_cast<const int32_t *>(base + off_idx), &d, s));
  B2R_CUDA(cudaMemcpyAsync(host_slab, base, total, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  return B2R_OK;
}

int b2r_sample_transition_batch_device(b2r_buffer *b, int32_t batch,
                                       uint64_t seed, uint64_t offset,
                                       const b2r_batch *out, b2r_stream stream) {
  if (!out->indices)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "out->indices is required (the sampled indices live there)");
  B2R_TRY(b2r_sample_indices_device(b, batch, seed, offset, out->indices, stream));
  return b2r::launch_gather(b, batch, out->indices, out, as_stream(stream));
}

int b2r_get_priority_device(b2r_buffer *b, int64_t n, const int32_t *indices,
                            float *out, b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  b2r::get_priority_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
      b->tree->heap + b->tree->leaves, n, indices, out);
  B2R_LAUNCHED();
  return B2R_OK;
}

int b2r_get_priority(b2r_buffer *b, int64_t n, const int32_t *indices, float *out,
                     b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (n <= 0) return B2R_OK;
  for (int64_t k = 0; k < n; ++k)
    if (indices[k] < 0 || indices[k] >= b->tree->leaves)
      return fail(B2R_ERR_INDEX_RANGE, "index %d is out of bounds", indices[k]);
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  B2R_TRY(b->bounce.reserve((size_t)n * 8 + 16));
  memcpy(b->bounce.host, indices, (size_t)n * 4);
  B2R_CUDA(cudaMemcpyAsync(b->bounce.dev, b->bounce.host, (size_t)n * 4,
                           cudaMemcpyHostToDevice, s));
  float *dout = reinterpret_cast<float *>(b->bounce.dev + (size_t)n * 4);
  b2r::get_priority_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
      b->tree->heap + b->tree->leaves, n,
      reinterpret_cast<const int32_t *>(b->bounce.dev), dout);
  B2R_LAUNCHED();
  B2R_CUDA(cudaMemcpyAsync(b->bounce.host + (size_t)n * 4, dout, (size_t)n * 4,
                           cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  memcpy(out, b->bounce.host + (size_t)n * 4, (size_t)n * 4);
  return B2R_OK;
}

}  // extern "C"

#ifdef B2R_TRACE
extern "C" int b2r_debug_trace_gather(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_trace, sizeof(long long) * 32);
}
#endif
