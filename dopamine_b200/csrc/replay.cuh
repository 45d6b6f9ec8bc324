// Replay buffer internals shared by replay.cu / sample.cu / gather.cu.
#pragma once

#include <vector>

#include "common.cuh"
#include "tree.cuh"

namespace b2r {

constexpr int kMaxColumns = 4 + B2R_MAX_EXTRAS;
constexpr int kMaxInvalid = 64;  // stack_size + update_horizon entries

// What is_valid_transition (circular_replay_buffer.py:381-414) needs, by value in
// kernel parameters: the host owns add_count / invalid_range (adds are host-driven).
struct ValidCtx {
  int64_t capacity;
  int64_t add_count;
  int64_t cursor;
  int32_t stack;
  int32_t horizon;
  int32_t n_invalid;
  int64_t invalid[kMaxInvalid];
  const uint8_t *term_flag;  // 1 byte per slot: terminal != 0
};

__device__ __forceinline__ bool is_valid_transition(const ValidCtx &c,
                                                    int64_t index) {
  if (index < 0 || index >= c.capacity) return false;
  bool ok = true;
  if (c.add_count < c.capacity)  // not full
    ok = index < c.cursor - c.horizon && index >= c.stack - 1;
  for (int k = 0; k < c.n_invalid; ++k) ok = ok && c.invalid[k] != index;
  // get_terminal_stack(index)[:-1].any(): all flags are loaded before any is
  // tested, so the check costs one memory round trip.
  unsigned any = 0;
#pragma unroll 4
  for (int k = 1; k < c.stack; ++k) {
    int64_t s = index - k;
    if (s < 0) s += c.capacity;
    any |= c.term_flag[s];
  }
  return ok && any == 0;
}

// Block-wide exclusive scan of a 0/1 flag (warp ballots + one shared array).
// Every thread of the block must call it.  Returns this thread's exclusive
// prefix; *total receives the block total.
__device__ __forceinline__ int block_scan_flag(bool flag, int *warp_counts,
                                               int *total) {
  const unsigned ballot = __ballot_sync(0xffffffffu, flag);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int within = __popc(ballot & ((1u << lane) - 1u));
  __syncthreads();  // protect warp_counts from the previous call's readers
  if (lane == 0) warp_counts[warp] = __popc(ballot);
  __syncthreads();
  int before = 0, all = 0;
  const int warps = (blockDim.x + 31) >> 5;
  for (int w = 0; w < warps; ++w) {
    const int c = warp_counts[w];
    if (w < warp) before += c;
    all += c;
  }
  *total = all;
  return before + within;
}

// Completion hand-shake between the first half of the C51 loss (c51.cu: c51_pre_*,
// launched on a forked stream beside the sampler because it needs the network outputs
// only) and the sampler of the same step.  The loss tail must follow BOTH; a kernel node
// with two parents loses its programmatic early launch (measured: 2.4 us from the end of
// the sampler to the first instruction of the tail, against 0.5 us with one parent), so
// the dependency on the first half goes through memory instead of through the graph:
// its last CTA bumps `done` (release), the sampler's closing thread waits for that bump
// (acquire) before the kernel ends, and the tail has the sampler as its only parent.
// The first half is a few microseconds of work that starts together with the sampler,
// so the wait normally finds the bump already there.
// Only the fork/join step needs this hand-shake for its ordering; the one-stream step
// (step.cu: train_step, StageGate::rows) orders the first half behind the sampler on the stream
// and keeps the sampler's wait only so that `done` and `seen` advance the same way on both
// paths, which may alternate on one buffer.
struct PreSync {
  unsigned int *done;    // first-half launches completed (monotone); nullptr: no hand-shake
  unsigned int *seen;    // ... consumed by a sampler (touched by its closing thread only)
  unsigned int *ticket;  // CTAs finished in the running first-half launch
};

// The agent's batch (at most 32 rows, no gradient): the loss tail stages what the first
// half left for it — the greedy action's probabilities and the online log-probabilities
// of EVERY action — while the sampler is still running, so that only the sampled scalars
// are fetched behind the sampler (c51.cu: c51_post_tree_kernel).  The tail is resident
// long before the first half of its step has ended and the scratch is rewritten every
// step, so it waits for a launch NUMBER, as the early write-back does (TreeGo): every
// staged first half counts itself in `done` when its last CTA leaves; every CTA of a
// staged tail takes a ticket before it lets its dependents start, so ticket / CTAs is
// the launch's number k (launches never interleave their tickets), and the CTA stages
// once done >= k + 1.  (The first halves of consecutive steps run on one stream, so they
// complete in order; with the trainer's direct I/O the next one may have completed too.)
// Staged first halves and staged tails are launched in pairs by the same host call.
// The scratch is two halves by step parity: the first half of step n + 1 writes the other
// half, and that of step n + 2 is ordered behind the tail of step n (stream order, or
// DirectIO::first_half_after) — no first half overwrites rows a tail may still read.
// The one-stream step (step.cu: train_step at the agent's batch with its frame copies joined
// and nothing else to wait for): sampler, first half, frame copies and tail run in this order
// on the caller's stream, each launched programmatically behind the one before, so that every
// kernel node of a captured step has ONE parent and keeps its early launch — the next step's
// sampler included.  The copies and the tail no longer learn from their predecessor's
// completion that the sampled rows are there: the sampler's closing thread counts its launch
// in `done` (release) once every row, the minimum and the counters are final, and every CTA
// of a gated copy or tail launch takes a ticket (ticket / CTAs = its launch number k, as in
// StageGate) and reads the rows once done >= k + 1.  Samplers, copies and tails of this kind
// are launched together by one host call, and only by it: the counts stay paired.
// Completion stays transitive: the first half, the copies and the tail each pass their
// griddepcontrol.wait before they exit (the first half after it has signalled the sampler),
// so "tail n complete" means all of step n is complete, the copies included.  The sampler lets
// its dependents launch only after its own griddepcontrol.wait: the first half of step n + 1
// then starts after the tail of step n has ended, never while it reads the scratch half.
// Both gates are LaunchGates: one opens for the launch numbered k (launch_ticket, counted
// from 1) once `done` >= k.
struct LaunchGate {
  unsigned int *done = nullptr;           // signaller launches completed (monotone)
  unsigned long long *tickets = nullptr;  // CTAs of the gated launches started (monotone)
};
struct StageGate {
  LaunchGate first_half;  // staged first halves completed / CTAs of staged tails started
  float *logp = nullptr;  // [rows][c51_logp_stride] log-probabilities, action-major
  // the one-stream step: sampler launches with final rows / CTAs of gated tails
  // (rows.done == nullptr: the fork/join step)
  LaunchGate rows;
};
// Row stride of StageGate::logp: whole 16-byte words, so a row moves as float4s.
__host__ __device__ __forceinline__ int c51_logp_stride(int actions, int atoms) {
  return (actions * atoms + 3) & ~3;
}

// The hand-over words of the fused step (step.cu), one set per buffer, zeroed at creation.
struct StepSync {
  unsigned int pre_done, pre_seen, pre_ticket;  // PreSync
  unsigned int tree_done;  // UpdateArgs::skip_flag of a shard's one-CTA write-back
  unsigned int stage_done, unused0;
  unsigned long long stage_tickets;  // StageGate::first_half
  unsigned int rows_done, unused1;   // StageGate::rows and the gated copies
  unsigned long long copy_tickets, tail_tickets;
  unsigned int sample_ticket;  // last-CTA election of the sample kernels
};
static_assert(offsetof(StepSync, stage_tickets) % 8 == 0 &&
                  offsetof(StepSync, copy_tickets) % 8 == 0 &&
                  offsetof(StepSync, tail_tickets) == 48 && sizeof(StepSync) == 64,
              "StepSync keeps its word order");

#ifdef __CUDACC__
// Last statement of a first-half CTA (every thread calls it).  staged_done (nullable):
// StageGate::first_half.done of a staged first half.
__device__ __forceinline__ void pre_sync_signal(const PreSync &p,
                                                unsigned int *staged_done = nullptr) {
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0 && arrive_last(p.ticket)) {
    __threadfence();
    if (staged_done != nullptr) st_release_u32(staged_done, *staged_done + 1u);
    st_release_u32(p.done, *p.done + 1u);
  }
}
// By thread 0 of every CTA of a gated launch, BEFORE the CTA lets its dependents start: takes
// the ticket and waits for the signaller of this launch's step.  False after kSpinLimit: the
// caller then falls back to its griddepcontrol.wait, which is behind the signaller's own
// completion or wait (correct, only late).  kBackoffNs: poll_acquire.
template <int kBackoffNs>
__device__ __forceinline__ bool gate_wait(const LaunchGate &g) {
  const unsigned int launch = launch_ticket(g.tickets, gridDim.x).launch;
  return poll_acquire<kBackoffNs>(g.done, [=](unsigned v) { return (int)(v - launch) >= 0; });
}
// The same for the whole CTA (every thread calls it; s_ok in shared memory).  The staged
// tail spins; the one-stream step's copies and tail back off 32 ns between polls (measured
// that way).
template <int kBackoffNs>
__device__ __forceinline__ bool cta_gate_wait(const LaunchGate &g, bool *s_ok) {
  if (threadIdx.x == 0) *s_ok = gate_wait<kBackoffNs>(g);
  __syncthreads();
  return *s_ok;
}
// The sampler's last word (StageGate::rows.done): release, no round trip.
__device__ __forceinline__ void rows_gate_publish(unsigned int *done) {
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(done) : "memory");
}
// Called by the sampler's closing thread (ONE thread) before the kernel ends.  Gives up
// after kSpinLimit: a first half that never ran must not hang the GPU (the tail then reads
// stale rows; the launch error that caused it has been reported to the caller).
__device__ __forceinline__ void pre_sync_consume(const PreSync &p) {
  if (p.done == nullptr) return;
  const unsigned int seen = *p.seen;
  poll_acquire(p.done, [=](unsigned v) { return v != seen; });
  *p.seen = seen + 1u;
}
// The same in two steps, so that the two loads are in flight long before the closing
// thread needs their answer (the first half is normally done by then: no spin at all).
struct PreSyncPeek {
  unsigned int seen, done;
};
__device__ __forceinline__ PreSyncPeek pre_sync_peek(const PreSync &p) {
  PreSyncPeek k = {0u, 1u};
  if (p.done != nullptr) {
    k.seen = *p.seen;
    k.done = ld_acquire_u32(p.done);
  }
  return k;
}
__device__ __forceinline__ void pre_sync_consume(const PreSync &p, const PreSyncPeek &k) {
  if (p.done == nullptr) return;
  if (k.done == k.seen)  // not yet when we looked: wait now
    poll_acquire(p.done, [=](unsigned v) { return v != k.seen; });
  *p.seen = k.seen + 1u;
}
#endif

// Staged rows -> ring (replay.cu: flush_queue).  In a header because the fused flush
// kernel of tree.cu runs it beside the priority update.
struct AddParams {
  int n_entries;
  int num_columns;
  int64_t row_stride;
  const int64_t *slots;     // device, per entry
  const int32_t *src_rows;  // device, per entry; -1 = all-zero padding transition
  const uint8_t *rows;      // device staged rows
  uint8_t *col_dev[kMaxColumns];
  int64_t col_bytes[kMaxColumns];
  int64_t col_qoff[kMaxColumns];
  uint8_t *term_flag;       // nullptr when it aliases the 1-byte terminal column
  int term_itemsize;
  const uint64_t *ctx_src;  // ValidCtx image in the staged header
  uint64_t *ctx_dst;        // the buffer's device ValidCtx
};

// One CTA of the row writer: entry e, chunk-block bx of nbx.
#ifdef __CUDACC__
__device__ __forceinline__ void add_rows_body(const AddParams &p, int e, int bx, int nbx) {
  const int64_t slot = p.slots[e];
  const int src = p.src_rows[e];
  const uint8_t *row = src >= 0 ? p.rows + (int64_t)src * p.row_stride : nullptr;

  // observation: coalesced 16-byte stores when the frame size allows it.
  const int64_t obs_bytes = p.col_bytes[0];
  uint8_t *dst = p.col_dev[0] + slot * obs_bytes;
  const int64_t tid = bx * (int64_t)blockDim.x + threadIdx.x;
  const int64_t nthreads = nbx * (int64_t)blockDim.x;
  if ((obs_bytes & 15) == 0) {
    const int64_t chunks = obs_bytes >> 4;
    const uint4 *s4 = reinterpret_cast<const uint4 *>(row);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
    for (int64_t c = tid; c < chunks; c += nthreads)
      d4[c] = row ? s4[c] : make_uint4(0, 0, 0, 0);
  } else {
    for (int64_t c = tid; c < obs_bytes; c += nthreads) dst[c] = row ? row[c] : 0;
  }

  // the validity context that goes with these rows
  if (bx == 0 && e == 0)
    for (int w = threadIdx.x; w < (int)(sizeof(ValidCtx) / 8); w += blockDim.x)
      p.ctx_dst[w] = p.ctx_src[w];

  // scalar columns: a handful of bytes, first block of the entry only.
  if (bx == 0) {
    for (int c = 1; c < p.num_columns; ++c) {
      const int64_t nb = p.col_bytes[c];
      uint8_t *d = p.col_dev[c] + slot * nb;
      const uint8_t *s = row ? row + p.col_qoff[c] : nullptr;
      for (int64_t b = threadIdx.x; b < nb; b += blockDim.x) d[b] = s ? s[b] : 0;
    }
    if (p.term_flag != nullptr && threadIdx.x == 0) {
      uint8_t any = 0;
      if (row)
        for (int b = 0; b < p.term_itemsize; ++b) any |= row[p.col_qoff[3] + b];
      p.term_flag[slot] = any ? 1 : 0;
    }
  }
}

#endif  // __CUDACC__

struct Column {
  int64_t row_bytes = 0;
  int64_t queue_offset = 0;  // byte offset inside a staged row
  uint8_t *dev = nullptr;
};

struct Staging {
  uint8_t *host = nullptr;  // pinned
  uint8_t *host_dev = nullptr;  // the same memory as the device sees it (zero-copy)
  uint8_t *dev = nullptr;
  cudaEvent_t done = nullptr;
  bool in_flight = false;
};

}  // namespace b2r

struct b2r_buffer {
  b2r_config cfg;
  int num_columns = 0;
  b2r::Column col[b2r::kMaxColumns];
  uint8_t *term_flag = nullptr;  // aliases the terminal column when it is 1 byte
  bool term_flag_owned = false;
  float *discounts = nullptr;    // f32(pow(gamma, k)), k < update_horizon
  std::vector<float> discounts_host;
  b2r_tree *tree = nullptr;

  // host bookkeeping (circular_replay_buffer.py:177-178, 284-287)
  int64_t add_count = 0;
  std::vector<int64_t> invalid_range;
  std::vector<uint8_t> term_is_one;  // host mirror of `terminal == 1` (CRB:255)

  // deferred-add queue: rows staged in pinned memory, applied by one kernel
  int queue_cap = 0;        // entries (real rows + zero pads)
  int64_t row_stride = 0;   // bytes of one staged row (16-byte aligned)
  int64_t header_bytes = 0; // SoA entry table in front of the rows
  b2r::Staging staging[2];
  int active = 0;
  int q_entries = 0, q_rows = 0;

  // scratch
  int32_t *inv_slots = nullptr;
  int64_t inv_slots_cap = 0;
  int32_t *info = nullptr;      // device [4]: status, fail slot, draws used, count
  int64_t *status = nullptr;    // device [2]: latched asynchronous error
  uint64_t *shard_counter = nullptr;  // device: like draw_counter, for sharded draws
                                      // (advances in lockstep on every rank)
  uint64_t *draw_counter = nullptr;  // device: bumps per Philox sample launch, so a
                                     // replayed CUDA graph draws fresh uniforms
  // fused step: the frame copies run on `side`, forked/joined with these events
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_pre = nullptr, ev_h2d = nullptr, ev_rows = nullptr;  // split flush
  // ... and the half of the C51 loss that needs the network outputs only on `side3`,
  // beside the sampler (c51.cu: c51_pre_kernel)
  cudaStream_t side3 = nullptr;
  cudaEvent_t ev_c51_fork = nullptr, ev_c51_pre = nullptr;
  float *c51_bestp = nullptr;  // device [2 halves][c51_bestp_rows][64 probabilities | 64 stats]
  int64_t c51_bestp_rows = 0;
  int c51_half = 0;            // half the next step's first half writes
  b2r::StepSync *sync = nullptr;     // device
  float *c51_logp = nullptr;         // device [2 halves][c51_logp_half]: StageGate::logp
  int64_t c51_logp_half = 0;
  // Deferred frame copies (b2r_set_deferred_frames): the copies of a fused step are not
  // joined into the caller's stream when the call returns but when b2r_join_frames is
  // called (or staged adds are flushed: they overwrite ring slots the copies may still
  // read), so the next step's sampler -> loss -> write-back chain runs BESIDE them.  The
  // copies read their indices from a private two-slot ring: the next sampler overwrites
  // the caller's `indices` while they are still running.
  bool deferred_frames = false;
  bool frames_pending = false;   // a copy was queued on `side` since the last join
  int frame_parity = 0;
  int32_t *idx_ring = nullptr;   // device [2][idx_ring_cap]
  int64_t idx_ring_cap = 0;
  // copies that read ring slot p have finished (a sampler may then overwrite it: the
  // chain runs at most one step ahead of the copies)
  cudaEvent_t ev_slot_free[2] = {nullptr, nullptr};
  bool slot_busy[2] = {false, false};
  float *min_prob = nullptr;    // device: min sampling probability of the last batch
  // Device copy of the validity context (add_count, cursor, invalid_range): the
  // prioritized sampler reads it from here, so a captured CUDA graph stays valid
  // while adds move the cursor.  Refreshed by every flush (the image rides in the
  // staging header) and lazily after b2r_set_state.
  b2r::ValidCtx *ctx_dev = nullptr;
  bool ctx_dirty = true;
  b2r::Bounce bounce;           // HOST-array calls
  uint8_t *out_scratch = nullptr;  // device outputs of b2r_gather (HOST variant)
  size_t out_scratch_cap = 0;
};

struct b2r_exchange {
  int world = 0, rank = 0;
  uint64_t *mailbox = nullptr;  // device, written by the peers
  uint64_t *seq = nullptr;      // device
  uint64_t *peer[b2r::kMaxShards] = {nullptr};
  bool opened[b2r::kMaxShards] = {false};  // peer[g] came from cudaIpcOpenMemHandle
  bool connected = false;
  int64_t timeout_ns = 2000000000ll;
  uint64_t *pub = nullptr;              // device [2]: ExchangeArgs::pub
  b2r::ExchangeArgs *args_dev = nullptr;  // device copy of the kernel arguments (the tree
                                          // kernels' publish hook reads it from there)
  // b2r_exchange_set_early_publish: the kernel that leaves the tree final for the next
  // sharded step publishes the shard total itself, and the staged adds of a step call are
  // flushed at the END of that call (they become visible to the next step's sampler).
  bool early_publish = false;
  // Latch of the buffer last sampled through b2r_sample_transition_batch_sharded_device:
  // where b2r_c51_loss_sharded reports a peer whose minimum never arrived.
  int64_t *latched = nullptr;
};

namespace b2r {
// Applies the staged adds.  split: the staged rows are copied and written to the
// ring on the buffer's side stream while the priorities go into the tree on
// `stream`; `stream` then waits for the rows, so callers see no difference.
// publish (nullable): the flush leaves the tree final for the next sharded step (see
// tree_apply).
int flush_queue(b2r_buffer *buf, cudaStream_t stream, bool split = false,
                const b2r_exchange *publish = nullptr);
// Keeps the host mirror of `terminal == 1` (CRB:255) and the 1-byte terminal flags in step
// with terminal rows [row0, row0 + nrows) of the store after they were overwritten.
int refresh_terminal_mirror(b2r_buffer *buf, int64_t row0, int64_t nrows,
                            cudaStream_t stream);
// Makes `stream` wait for every deferred frame copy queued so far (no-op otherwise).
int join_frames(b2r_buffer *buf, cudaStream_t stream);
void fill_exchange_args(const b2r_exchange *x, ExchangeArgs *out);
int launch_exchange_publish(const b2r_exchange *x, const b2r_buffer *buf,
                            cudaStream_t stream);
// One launch of the prioritized sampler (sample.cu), unsharded or one rank of a sharded
// global batch.  Every pointer is a device pointer.
struct SampleRequest {
  int32_t batch = 0;  // strata (the global batch when sharded)
  // A sharded call (also with one shard): this rank's rows go to out_slots / count_out, and
  // rows the range search cannot find (caller queries, one shard) are compacted by one CTA.
  bool sharded = false;
  int32_t num_shards = 1, rank = 0;
  // Shard totals from `shard_totals`, or, when `x` is set, from the peer-memory exchange.
  const double *shard_totals = nullptr;
  const b2r_exchange *x = nullptr;
  // Stratified queries in [0, 1] and retry uniforms (the reference's RNG stream);
  // query01 == nullptr: Philox draws (seed, offset + *counter).
  const double *query01 = nullptr;
  const double *retry_u01 = nullptr;
  int32_t max_attempts = 0;
  uint64_t seed = 0, offset = 0;
  // Philox: the device draw counter added to offset and advanced by the launch, so that a
  // captured CUDA graph draws fresh strata at every replay (b2r_buffer::draw_counter;
  // sharded calls: shard_counter, which advances in lockstep on all ranks as each makes the
  // same sequence of sharded calls).
  uint64_t *counter = nullptr;
  bool latch = true;       // report asynchronous errors in b2r_buffer::status
  int32_t *info = nullptr;  // [4]: status, fail slot, retry draws used, count
  int32_t *out_idx = nullptr;
  int32_t *out_slots = nullptr;  // nullable: each row's place in the global batch
  int32_t *count_out = nullptr;  // nullable: this rank's row count
  // > 0: rows the outputs hold — a rank whose share of a Philox batch is larger serves the
  // first out_cap and latches B2R_ERR_UNSUPPORTED (0: batch rows).
  int32_t out_cap = 0;
  // Scalar columns written as the rows become final, and the batch's smallest sampling
  // probability (both nullable).
  const b2r_batch *scalars = nullptr;
  float *min_prob_out = nullptr;
  const PreSync *pre = nullptr;  // nullable: the first half of the loss running beside
  bool publish_min = false;      // store the minimum into every peer's mailbox
  // nullable: StageGate::rows.done of the one-stream step (batches of the warp sampler,
  // with scalars and the minimum).
  unsigned int *rows_done = nullptr;
};
int launch_sample(b2r_buffer *buf, const SampleRequest &r, cudaStream_t stream);
// Sharded uniform sampling (sample.cu: uniform_sharded_kernel).  check_uniform_sharded:
// the host-side refusals shared by the sampling call and the publish-ahead.
// mode 0 / 1: publish-ahead of the span / the rejection list of the exchange's next step
// (ranks emulated by sequential launches); 2: the sampler, which closes the step.
int check_uniform_sharded(const b2r_buffer *buf, const b2r_exchange *x,
                          int32_t global_batch);
int launch_uniform_sharded(b2r_buffer *buf, const b2r_exchange *x, int32_t global_batch,
                           uint64_t seed, uint64_t offset, int mode, int32_t *out_idx,
                           int32_t *out_slots, int32_t *out_count, int32_t out_cap,
                           cudaStream_t stream);
void fill_valid_ctx(const b2r_buffer *buf, ValidCtx *ctx);
int ensure_ctx(b2r_buffer *buf, cudaStream_t stream);
// tree.cu: the fused flush launch (priorities of n new rows + their row writes, staging
// read zero-copy).
int flush_fused(b2r_tree *tree, int n, const int64_t *slots, const double *prio,
                const uint8_t *mode, const AddParams &rows, int row_blocks_per_entry,
                cudaStream_t stream, const b2r_exchange *publish = nullptr);
int ensure_inv_slots(b2r_buffer *buf, int64_t n);
// gate (nullable): frame copies of the one-stream step (StageGate::rows); only the TMA copies
// (gather_can_gate) take one.
int launch_gather(b2r_buffer *buf, int32_t batch, const int32_t *indices_dev,
                  const b2r_batch *out, cudaStream_t stream,
                  const int32_t *count_dev = nullptr, bool frames_only = false,
                  const LaunchGate *gate = nullptr);
bool gather_can_gate(const b2r_buffer *buf, int32_t batch);
}  // namespace b2r
