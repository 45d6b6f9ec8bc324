// The hot path as ONE call: what a sess.run of the Rainbow train op does around the
// network (SURVEY.md 3.2) — prioritized sample (prioritized_replay_buffer.py:142-201)
// -> C51 target / loss / new priorities (rainbow_agent.py:200-293) -> priority
// write-back (prioritized_replay_buffer.py:203-214) — plus the host-facing,
// pipelined trainer built on it.
//
// Dependencies inside a step: the loss needs only the SCALAR columns of the batch
// (action, n-step return, terminal, sampling probability) and the network outputs;
// the next step's sampler needs this step's write-back.  The frame stacks feed the
// network, not this chain.  So the sampler emits the scalar columns itself, the
// chain sample -> loss -> write-back runs on the caller's stream, and the HBM-bound
// frame copies run beside it on a forked stream, joined before the call returns —
// except at the agent's batch, where every kernel goes on the caller's stream
// (StageGate::rows, replay.cuh: a joined fork would give the next step's sampler three parents).
#include "gather.cuh"

#include <cmath>
#include <cstdlib>
#include <new>
#include <vector>

#include <chrono>

namespace b2r {

// Host-side cost of the trainer's driver calls, by segment (B2R_HOST_TRACE=1 prints
// the averages when a trainer is destroyed).  Off: one predictable branch per call.
struct HostTrace {
  bool on = std::getenv("B2R_HOST_TRACE") != nullptr;
  double acc[8] = {0};
  long calls = 0;
  std::chrono::steady_clock::time_point last;
  void start() { if (on) last = std::chrono::steady_clock::now(); }
  void lap(int k) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    acc[k] += std::chrono::duration<double, std::micro>(now - last).count();
    last = now;
  }
};
static HostTrace g_host_trace;

// Batch size above which the staged adds are flushed "split" (rows on the side
// stream beside the tree update).  Measured at batch 32 (e2e_breakdown.py): 49.7 us
// per update unsplit, 54.7 us split — the side stream also carries the forked frame
// copies, and the extra event hops cost more than the 3 us row kernel they hide.
constexpr int kSplitMin = 64;

// One shard of a sharded replay: `batch` is then the GLOBAL batch, this rank's rows
// are compacted at the front of `out` and counted on the device.
struct ShardSpec {
  const b2r_exchange *exchange;
  int32_t *out_slots;
  int32_t *out_count;
  // Rows the caller's outputs (and logits) hold: a bound on this rank's share of the
  // global batch.  Every launch behind the sampler is sized by it, not by the global
  // batch; 0 = global batch rows.
  int32_t max_rows;
  // b2r_sample_transition_batch_sharded_device: the step ends after the sampler and the
  // frame copies (no loss, no write-back); the sampler leaves its minimum sampling
  // probability in min_probability and publishes it to the peers.
  bool sample_only;
  float *min_probability;
};

// The host-facing trainer without copy calls: the first half of the loss reads both
// logits tensors straight from the caller's page-locked memory (and leaves a device copy
// of the online logits for the tail), the tail writes the per-row losses into the
// trainer's page-locked result slot.  Only with the loss in two halves.
struct DirectIO {
  const float *online_src;   // device-visible address of the caller's online logits
  float *online_copy;        // device buffer the tail reads (c51->online_logits)
  float *loss_host;          // device-visible address of the result slot
  cudaEvent_t first_half_after;  // nullable: what last read online_copy / the scratch half
  // online_src == nullptr: no direct I/O, only the trainer's EAGER launch order — the
  // logits are ready at `wait_before_loss`, nothing on `s` feeds them and nothing is being
  // captured, so the first half is neither forked from `s` nor joined back into it (its
  // hand-shake with the sampler goes through memory): four driver calls less per update.
};

// wait_before_loss / loss_done (nullable): events of the trainer's copy stream.
static int train_step(b2r_buffer *b, int32_t batch, uint64_t seed, uint64_t offset,
                      const b2r_batch *out, const b2r_c51_args *c51, cudaStream_t s,
                      cudaEvent_t wait_before_loss, cudaEvent_t loss_done,
                      const ShardSpec *shard = nullptr, const DirectIO *direct = nullptr) {
  const bool sample_only = shard != nullptr && shard->sample_only;
  if (!b || !out || (!c51 && !sample_only)) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (batch <= 0 || batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "batch must be in [1, 60000]");
  if (b->cfg.terminal_itemsize != 1 || b->cfg.reward_itemsize != 4 ||
      b->cfg.action_bytes != 4)
    return fail(B2R_ERR_UNSUPPORTED,
                "the fused step needs uint8 terminals, float32 rewards and scalar "
                "int32 actions");
  if (!out->indices || !out->action || !out->reward || !out->terminal ||
      !out->sampling_probabilities)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "out->indices, action, reward, terminal and sampling_probabilities "
                "are required");
  if (shard && (!shard->exchange || !shard->out_count))
    return fail(B2R_ERR_INVALID_ARGUMENT, "exchange and out_count are required");
  const int32_t *count = shard ? shard->out_count : nullptr;  // (deferred: a ring slot)
  // rows behind the sampler: the batch, or the capacity of a shard's outputs
  const int32_t rows_cap =
      shard && shard->max_rows > 0 && shard->max_rows < batch ? shard->max_rows : batch;
  g_host_trace.lap(1);
  b2r_c51_args loss = c51 ? *c51 : b2r_c51_args{};
  loss.batch = rows_cap;
  loss.actions = static_cast<const int32_t *>(out->action);
  loss.rewards = static_cast<const float *>(out->reward);
  loss.terminals = static_cast<const uint8_t *>(out->terminal);
  loss.sampling_probabilities = out->sampling_probabilities;
  float *const min_out = sample_only ? shard->min_probability : b->min_prob;
  loss.min_probability = min_out;
  loss.batch_count = count;
  if (count) loss.mean_weighted_loss = nullptr;
  // The half of the loss that needs the network outputs only (every action's softmax
  // and q-value, the greedy next action) starts now, on a forked stream beside the
  // sampler; the tail that needs the sampled rows follows the sampler (c51.cu).
  // (A shard does not know its row count before it has sampled: the first half covers
  // every row its logits hold.)
  const bool split_loss = !sample_only && c51_can_split(&loss);
  if (direct != nullptr && direct->online_src != nullptr && !split_loss)
    return fail(B2R_ERR_INVALID_ARGUMENT, "direct logits need the loss in two halves");
  const bool unjoined = direct != nullptr && split_loss;  // (see DirectIO)
  PreSync pre_sync = {nullptr, nullptr, nullptr};
  int have_stats = 0;
  float *scratch = nullptr;
  // The agent's batch: the tail stages the first half's rows ahead of the sampler's end
  // (StageGate, replay.cuh; the tail and the write-back are then one cluster, below).
  const bool staged = split_loss && !shard && c51_post_takes_tree(&loss, b->tree) &&
                      c51_tail_can_stage(&loss);
  // The one-stream step (StageGate::rows, replay.cuh): sampler -> first half -> frame copies ->
  // tail + write-back, all on `s`, every kernel launched programmatically behind the one
  // before — in a captured graph every node then has ONE parent, and the next step's
  // sampler keeps its early launch.  Only where nothing else joins the step: copies joined
  // before the call returns, no direct I/O, no event to wait for.  (Programmatic launch is
  // required: the sampler's closing thread waits for the first half, launched behind it.)
  const bool frames = out->state != nullptr || out->next_state != nullptr;
  const bool one_stream = staged && frames && !b->deferred_frames && direct == nullptr &&
                          wait_before_loss == nullptr && pdl_enabled() &&
                          gather_can_gate(b, rows_cap);
  LaunchGate copy_gate;
  StageGate stage;
  if (split_loss) {
    // (two halves of scratch: with direct I/O the first half of step n + 1 is not
    // ordered behind the tail of step n, which may still be reading its rows)
    if (b->c51_bestp_rows < rows_cap) {
      if (b->c51_bestp) {
        B2R_CUDA(cudaStreamSynchronize(b->side3));
        B2R_CUDA(cudaStreamSynchronize(s));
        cudaFree(b->c51_bestp);
      }
      b->c51_bestp = nullptr;
      b->c51_bestp_rows = 0;
      int64_t cap = 256;
      while (cap < rows_cap) cap *= 2;
      B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->c51_bestp),
                          2 * (size_t)cap * c51_scratch_floats_per_row() * sizeof(float)));
      b->c51_bestp_rows = cap;
    }
    scratch = b->c51_bestp + (size_t)(b->c51_half & 1) * (size_t)b->c51_bestp_rows *
                                 c51_scratch_floats_per_row();
    if (staged) {
      const int64_t half =
          (int64_t)rows_cap * c51_logp_stride(loss.num_actions, loss.num_atoms);
      if (b->c51_logp_half < half) {
        if (b->c51_logp) {
          B2R_CUDA(cudaStreamSynchronize(b->side3));
          B2R_CUDA(cudaStreamSynchronize(s));
          cudaFree(b->c51_logp);
        }
        b->c51_logp = nullptr;
        b->c51_logp_half = 0;
        B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->c51_logp),
                            2 * (size_t)half * sizeof(float)));
        b->c51_logp_half = half;
      }
      stage.first_half = {&b->sync->stage_done, &b->sync->stage_tickets};
      stage.logp = b->c51_logp + (size_t)(b->c51_half & 1) * (size_t)b->c51_logp_half;
      if (one_stream) {
        stage.rows = {&b->sync->rows_done, &b->sync->tail_tickets};
        copy_gate = {&b->sync->rows_done, &b->sync->copy_tickets};
      }
    }
    b->c51_half ^= 1;
    pre_sync = {&b->sync->pre_done, &b->sync->pre_seen, &b->sync->pre_ticket};
    if (one_stream) {
      // (launched behind the sampler, below)
    } else if (unjoined) {
      // nothing on `s` feeds the first half: it waits only for whoever last read the
      // buffers it writes (the tail two steps back) and for the logits
      if (direct->first_half_after)
        B2R_CUDA(cudaStreamWaitEvent(b->side3, direct->first_half_after, 0));
      if (wait_before_loss) B2R_CUDA(cudaStreamWaitEvent(b->side3, wait_before_loss, 0));
      B2R_TRY(c51_pre_launch(&loss, rows_cap, scratch, pre_sync, b->side3, &have_stats,
                             direct->online_src, direct->online_copy,
                             staged ? &stage : nullptr));
    } else {
      B2R_CUDA(cudaEventRecord(b->ev_c51_fork, s));
      B2R_CUDA(cudaStreamWaitEvent(b->side3, b->ev_c51_fork, 0));
      if (wait_before_loss) B2R_CUDA(cudaStreamWaitEvent(b->side3, wait_before_loss, 0));
      B2R_TRY(c51_pre_launch(&loss, rows_cap, scratch, pre_sync, b->side3, &have_stats,
                             nullptr, nullptr, staged ? &stage : nullptr));
      B2R_CUDA(cudaEventRecord(b->ev_c51_pre, b->side3));
    }
  }
  // Staged adds (rows on the side stream beside the tree update at larger batches).
  // Early publish (b2r_exchange_set_early_publish): whichever kernel of this call writes
  // the tree LAST publishes the shard total for the next step — so the adds staged before
  // this call are applied behind the write-back, at the end of the call, and are seen by
  // the next step's sampler: the order of effects on the tree stays the reference's
  // add, sample, set_priority, add, ... with the adds one call later.
  const b2r_exchange *early = shard && !sample_only && shard->exchange->early_publish &&
                                      shard->exchange->world > 1
                                  ? shard->exchange
                                  : nullptr;
  if (!early) B2R_TRY(flush_queue(b, s, batch > kSplitMin));
  const bool flush_behind = early != nullptr && b->q_entries > 0;
  g_host_trace.lap(2);
  // Deferred frame copies: the copies read their indices from a private ring slot (the
  // next step's sampler overwrites out->indices while they may still be running).
  // (A shard's copies also read its row count: that lives in the ring slot as well, and
  // the loss tail hands it on to the caller's out_count.)
  const bool deferred = b->deferred_frames && (!shard || split_loss);
  if (b->deferred_frames && !deferred) B2R_TRY(join_frames(b, s));
  int32_t *sample_idx = out->indices;
  int ring_slot = 0;
  if (deferred) {
    if (b->idx_ring_cap < rows_cap) {
      B2R_TRY(join_frames(b, s));
      B2R_CUDA(cudaStreamSynchronize(b->side));
      if (b->idx_ring) cudaFree(b->idx_ring);
      b->idx_ring = nullptr;
      b->idx_ring_cap = 0;
      int64_t cap = 256;
      while (cap < rows_cap) cap *= 2;
      // [2][cap] indices, then the two row counts
      B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->idx_ring), (size_t)(cap * 2 + 2) * 4));
      b->idx_ring_cap = cap;
    }
    ring_slot = b->frame_parity & 1;
    sample_idx = b->idx_ring + (size_t)ring_slot * b->idx_ring_cap;
    if (shard) {
      count = b->idx_ring + 2 * b->idx_ring_cap + ring_slot;
      loss.batch_count = count;
    }
    b->frame_parity ^= 1;
    // the copies of two steps ago read this slot
    if (b->slot_busy[ring_slot])
      B2R_CUDA(cudaStreamWaitEvent(s, b->ev_slot_free[ring_slot], 0));
  }
  SampleRequest req;
  req.batch = batch;
  req.max_attempts = b->cfg.max_sample_attempts;
  req.seed = seed;
  req.offset = offset;
  req.counter = shard ? b->shard_counter : b->draw_counter;
  req.info = b->info;
  req.out_idx = sample_idx;
  req.scalars = out;
  req.pre = split_loss ? &pre_sync : nullptr;
  if (shard) {
    req.sharded = true;
    req.num_shards = shard->exchange->world;
    req.rank = shard->exchange->rank;
    req.x = shard->exchange;
    req.out_slots = shard->out_slots;
    req.count_out = const_cast<int32_t *>(count);
    req.out_cap = rows_cap;
    req.min_prob_out = min_out;
    req.publish_min = sample_only;
  } else {
    req.min_prob_out = b->min_prob;
    req.rows_done = one_stream ? copy_gate.done : nullptr;
  }
  B2R_TRY(launch_sample(b, req, s));
  if (one_stream)
    B2R_TRY(c51_pre_launch(&loss, rows_cap, scratch, pre_sync, s, &have_stats, nullptr,
                           nullptr, &stage));
  g_host_trace.lap(3);
  int64_t expected_rows =
      shard ? (batch + shard->exchange->world - 1) / shard->exchange->world : -1;
  if (expected_rows > rows_cap) expected_rows = rows_cap;
  // Behind a split loss, up to 1024 rows (tree_early_takes): ONE write-back kernel behind
  // the loss tail that is resident early and groups the batch ahead of its values
  // (tree.cu, kEarly; the loss tail tells it when the indices are final — TreeGo).
  // (At 1024 rows, where the frame copies bound the step: 33.2 us with the TMA copies,
  // 36.8 us with a separate grouping kernel on a forked stream and the register copies
  // under their occupancy cap, 40.1 us with this kernel beside the capped register
  // copies — profiles/r2/out/run63.txt, run71.txt, run72.txt.)
  // Behind the one-kernel loss the write-back is the plain kFull launch: that kernel lets
  // its dependents start at its first instruction, while the sampler may still be writing
  // the indices.
  const bool early_tree = split_loss && tree_early_takes(rows_cap, expected_rows);
  const TreeGo tree_go = early_tree ? tree_go_of(b->tree) : TreeGo();
  if (one_stream) {
    B2R_TRY(launch_gather(b, rows_cap, sample_idx, out, s, nullptr, true, &copy_gate));
  } else if (frames) {
    B2R_CUDA(cudaEventRecord(b->ev_fork, s));
    B2R_CUDA(cudaStreamWaitEvent(b->side, b->ev_fork, 0));
    // (deferred: the first half of the loss rejoins through the copies' stream, so that
    // the next sampler's only parent in a captured graph is this step's write-back)
    if (deferred && split_loss && !unjoined)
      B2R_CUDA(cudaStreamWaitEvent(b->side, b->ev_c51_pre, 0));
    B2R_TRY(launch_gather(b, rows_cap, sample_idx, out, b->side, count, true));
    B2R_CUDA(cudaEventRecord(b->ev_join, b->side));
    if (deferred) {
      b->frames_pending = true;
      B2R_CUDA(cudaEventRecord(b->ev_slot_free[ring_slot], b->side));
      b->slot_busy[ring_slot] = true;
    }
  }
  g_host_trace.lap(4);
  if (sample_only) {
    if (frames) B2R_CUDA(cudaStreamWaitEvent(s, b->ev_join, 0));
    return B2R_OK;
  }
  // (Measured: waiting for the logits before the sampler, or recording "loss done"
  // after the write-back, serialises the input copy of the next step behind this
  // step's tail and costs 13 us per update.)
  // (The first half has signalled the sampler's closing thread by now — PreSync — so the
  // tail's only parent in a captured graph is the sampler: it keeps its programmatic
  // early launch.  Its stream rejoins below, with the frame copies.)
  if (!split_loss && wait_before_loss) B2R_CUDA(cudaStreamWaitEvent(s, wait_before_loss, 0));
  // (split loss, at most 32 rows: tail and write-back as one thread-block cluster)
  // A shard's step (row count on the device): the cluster applies the write-back when
  // the count turns out to be at most 32 and the one-CTA tree kernel launched behind it
  // then returns at once (`tree_done`).
  const bool tail_counted = split_loss && shard != nullptr && !flush_behind &&
                            c51_post_takes_tree(&loss, b->tree, expected_rows);
  const bool tail_writeback = split_loss && !shard && c51_post_takes_tree(&loss, b->tree);
  unsigned int *tree_done = tail_counted ? &b->sync->tree_done : nullptr;
  if (split_loss)
    B2R_TRY(c51_post_launch(&loss, scratch, have_stats, s, b->status,
                            shard && count != shard->out_count ? shard->out_count : nullptr,
                            tail_writeback || tail_counted ? b->tree : nullptr,
                            out->indices, tree_done, tail_counted ? early : nullptr,
                            direct ? direct->loss_host : nullptr,
                            early_tree ? &tree_go : nullptr, staged ? &stage : nullptr));
  else
    B2R_TRY(b2r_c51_loss(&loss, s));
  if (loss_done) B2R_CUDA(cudaEventRecord(loss_done, s));
  g_host_trace.lap(5);
  if (!tail_writeback)
    B2R_TRY((tree_apply<int32_t, float>(b->tree, rows_cap, out->indices, loss.priorities,
                                        nullptr, s, count, expected_rows,
                                        early_tree ? kEarly : kFull,
                                        flush_behind ? nullptr : early, tree_done,
                                        early_tree)));
  if (flush_behind) B2R_TRY(flush_queue(b, s, false, early));
  if (frames && !deferred && !one_stream) B2R_CUDA(cudaStreamWaitEvent(s, b->ev_join, 0));
  if (split_loss && !unjoined && !(deferred && frames) && !one_stream)
    B2R_CUDA(cudaStreamWaitEvent(s, b->ev_c51_pre, 0));
  g_host_trace.lap(6);
  return B2R_OK;
}

}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

struct b2r_trainer {
  b2r_buffer *buf = nullptr;
  b2r_trainer_config cfg;
  // device
  float *logits[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [set][online, target]
  float *support = nullptr;
  uint8_t *frames = nullptr;    // state | next_state
  uint8_t *scalars = nullptr;   // every other batch column and loss output
  b2r_batch batch;
  b2r_c51_args c51;
  // copies run on their own stream, double-buffered against the loss kernel
  cudaStream_t copy = nullptr;      // inputs (H2D of the logits)
  cudaStream_t copy_out = nullptr;  // results (D2H of the losses): a result copy waits
                                    // for its step, and must not hold up the inputs
                                    // of the next one
  cudaEvent_t ev_in[2] = {nullptr, nullptr};
  cudaEvent_t ev_loss[2] = {nullptr, nullptr};
  // sharded mode
  b2r_exchange *exchange = nullptr;
  int32_t *slots = nullptr;   // device [batch]: stratum of every local row
  // Per-row losses (+ the shard's row count behind them), one buffer per logits set:
  // step n's result copy reads its buffer on the result-copy stream while step n + 1's
  // loss kernel is already writing the other one.
  float *loss_buf[2] = {nullptr, nullptr};
  int32_t *count_buf[2] = {nullptr, nullptr};
  int32_t last_rows = 0;
  // graph mode: the step's kernels captured once per logits set
  cudaStream_t cap = nullptr;
  cudaGraphExec_t exec[2] = {nullptr, nullptr};
  // Direct I/O: logits read by the kernels from the caller's page-locked memory, losses
  // written by the kernels into the result ring — no copy calls, no copy streams (see
  // DirectIO).  Decided per call: it needs page-locked logits (checked once per pointer
  // pair) and the loss in two halves.  Default: only for the synchronous trainer
  // (pipeline_depth 0), where the host waits for every step and the saved calls count
  // (48.7 against 57.2 us per update with adds); a pipelined trainer is bound by the
  // device, whose first half of the loss then reads 235 KB over PCIe beside the flush
  // kernel's zero-copy reads (33.5 against 29.5 us).  B2R_TRAINER_DIRECT=0|1 forces it.
  bool direct_ok = true;
  const float *probed[2] = {nullptr, nullptr};  // last pointer pair looked up ...
  const float *probed_dev[2] = {nullptr, nullptr};  // ... and their device addresses
  float *ring_dev = nullptr;  // the result ring as the device sees it
  // results
  int ring = 1;
  float *ring_host = nullptr;  // pinned [ring][batch]
  std::vector<cudaEvent_t> ev_done;
  int64_t submitted = 0;
};

namespace {

// Captures one step (sampler, forked frame copies, loss, write-back) on the
// trainer's private stream; the graph is then launched into the caller's stream.
int capture_step(b2r_trainer *t, int set) {
  b2r_c51_args c51 = t->c51;
  c51.online_logits = t->logits[set][0];
  c51.target_logits = t->logits[set][1];
  c51.loss = t->loss_buf[set];
  cudaGraph_t graph = nullptr;
  B2R_CUDA(cudaStreamBeginCapture(t->cap, cudaStreamCaptureModeThreadLocal));
  const int status = b2r::train_step(t->buf, t->cfg.batch, t->cfg.seed, 0, &t->batch,
                                     &c51, t->cap, nullptr, nullptr);
  const cudaError_t end = cudaStreamEndCapture(t->cap, &graph);
  if (status != B2R_OK) {
    if (graph) cudaGraphDestroy(graph);
    return status;
  }
  if (end != cudaSuccess)
    return fail(B2R_ERR_CUDA, "stream capture of the step failed: %s",
                cudaGetErrorString(end));
  const cudaError_t inst = cudaGraphInstantiate(&t->exec[set], graph, 0);
  cudaGraphDestroy(graph);
  if (inst != cudaSuccess)
    return fail(B2R_ERR_CUDA, "graph instantiation failed: %s",
                cudaGetErrorString(inst));
  return B2R_OK;
}

int collect(b2r_trainer *t, int64_t step, float *loss_out, int64_t *loss_step) {
  if (step < 0) {
    if (loss_step) *loss_step = -1;
    return B2R_OK;
  }
  const int slot = (int)(step % t->ring);
  B2R_CUDA(cudaEventSynchronize(t->ev_done[slot]));
  const int rows = t->cfg.logit_rows;
  const float *row = t->ring_host + (size_t)slot * (rows + 1);
  if (loss_out) memcpy(loss_out, row, (size_t)rows * sizeof(float));
  t->last_rows = rows;
  if (t->exchange) memcpy(&t->last_rows, row + rows, sizeof(int32_t));
  if (loss_step) *loss_step = step;
  return B2R_OK;
}

}  // namespace

extern "C" {

int b2r_train_step_device(b2r_buffer *b, int32_t batch, uint64_t seed,
                          uint64_t offset, const b2r_batch *out,
                          const b2r_c51_args *c51, b2r_stream stream) {
  return b2r::train_step(b, batch, seed, offset, out, c51, as_stream(stream),
                         nullptr, nullptr);
}

int b2r_set_deferred_frames(b2r_buffer *b, int32_t on) {
  if (!b) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  b->deferred_frames = on != 0;
  return B2R_OK;
}

int b2r_join_frames(b2r_buffer *b, b2r_stream stream) {
  if (!b) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  return b2r::join_frames(b, as_stream(stream));
}

int b2r_train_step_sharded_device(b2r_buffer *b, b2r_exchange *x,
                                  int32_t global_batch, uint64_t seed,
                                  uint64_t offset, const b2r_batch *out,
                                  const b2r_c51_args *c51, int32_t *out_slots,
                                  int32_t *out_count, int32_t max_rows,
                                  b2r_stream stream) {
  if (max_rows < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "max_rows must be >= 0");
  b2r::ShardSpec shard = {x, out_slots, out_count, max_rows, false, nullptr};
  return b2r::train_step(b, global_batch, seed, offset, out, c51, as_stream(stream),
                         nullptr, nullptr, &shard);
}

int b2r_sample_transition_batch_sharded_device(b2r_buffer *b, b2r_exchange *x,
                                               int32_t global_batch, uint64_t seed,
                                               uint64_t offset, const b2r_batch *out,
                                               int32_t *out_slots, int32_t *out_count,
                                               int32_t max_rows, float *min_probability,
                                               b2r_stream stream) {
  if (global_batch < 1) return fail(B2R_ERR_INVALID_ARGUMENT, "global_batch must be >= 1");
  if (max_rows < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "max_rows must be >= 0");
  if (!b || !x || !out || !out_slots || !out_count || !min_probability)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "buffer, exchange, out, out_slots, out_count and min_probability are "
                "required");
  if (!x->connected) return fail(B2R_ERR_INVALID_ARGUMENT, "the exchange is not connected");
  // the sharded loss of this step latches a peer that never published into this buffer
  x->latched = b->status;
  b2r::ShardSpec shard = {x, out_slots, out_count, max_rows, true, min_probability};
  return b2r::train_step(b, global_batch, seed, offset, out, nullptr, as_stream(stream),
                         nullptr, nullptr, &shard);
}

int b2r_trainer_create(b2r_buffer *b, const b2r_trainer_config *cfg,
                       b2r_trainer **out) {
  if (!b || !cfg || !out) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  *out = nullptr;
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (cfg->batch <= 0 || cfg->batch > 60000 || cfg->num_actions <= 0 ||
      cfg->num_atoms < 2 || cfg->pipeline_depth < 0 || cfg->pipeline_depth > 64 ||
      cfg->logit_rows < 0 || cfg->logit_rows > cfg->batch)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad trainer configuration");
  b2r_trainer *t = new (std::nothrow) b2r_trainer();
  if (!t) return fail(B2R_ERR_INVALID_ARGUMENT, "out of host memory");
  t->buf = b;
  t->cfg = *cfg;
  if (t->cfg.logit_rows == 0) t->cfg.logit_rows = cfg->batch;
  if (const char *e = std::getenv("B2R_TRAINER_GRAPH")) t->cfg.use_graph = std::atoi(e);
  // Every buffer holds logit_rows rows: the batch, or (a shard's trainer) the bound on
  // this rank's share of the global batch — nothing here grows with the world size.
  const size_t B = (size_t)t->cfg.logit_rows, A = (size_t)cfg->num_actions,
               N = (size_t)cfg->num_atoms;
  const size_t logit_bytes = B * A * N * sizeof(float);
  for (int set = 0; set < 2; ++set)
    for (int k = 0; k < 2; ++k) {
      B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->logits[set][k]), logit_bytes));
      B2R_CUDA(cudaMemset(t->logits[set][k], 0, logit_bytes));
    }
  // tf.linspace(-vmax, vmax, N) as TF-1.x evaluates it: start + i * step in f32
  // (rainbow_agent.py:124-126, SURVEY.md Q23).
  std::vector<float> z(N);
  const float lo = -cfg->vmax;
  const float step = (cfg->vmax - lo) / (float)(N - 1);
  for (size_t i = 0; i < N; ++i) z[i] = lo + (float)i * step;
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->support), N * sizeof(float)));
  B2R_CUDA(cudaMemcpy(t->support, z.data(), N * sizeof(float), cudaMemcpyHostToDevice));

  const size_t stack_bytes = (size_t)b->cfg.obs_bytes * b->cfg.stack_size;
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->frames), 2 * B * stack_bytes));
  // scalar columns, 256-byte aligned segments
  size_t off = 0;
  auto seg = [&](size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~(size_t)255;
    return at;
  };
  const size_t o_action = seg(B * 4), o_reward = seg(B * 4), o_naction = seg(B * 4),
               o_nreward = seg(B * 4), o_term = seg(B), o_idx = seg(B * 4),
               o_prob = seg(B * 4), o_loss = seg((B + 1) * 4), o_loss1 = seg((B + 1) * 4),
               o_prio = seg(B * 4), o_w = seg(B * 4), o_slots = seg(B * 4);
  size_t o_extra[B2R_MAX_EXTRAS];
  for (int e = 0; e < b->cfg.num_extras; ++e)
    o_extra[e] = seg(B * (size_t)b->cfg.extra_bytes[e]);
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->scalars), off));
  B2R_CUDA(cudaMemset(t->scalars, 0, off));
  memset(&t->batch, 0, sizeof(t->batch));
  t->batch.state = t->frames;
  t->batch.next_state = t->frames + B * stack_bytes;
  t->batch.action = t->scalars + o_action;
  t->batch.reward = t->scalars + o_reward;
  t->batch.next_action = t->scalars + o_naction;
  t->batch.next_reward = t->scalars + o_nreward;
  t->batch.terminal = t->scalars + o_term;
  t->batch.indices = reinterpret_cast<int32_t *>(t->scalars + o_idx);
  t->batch.sampling_probabilities = reinterpret_cast<float *>(t->scalars + o_prob);
  for (int e = 0; e < b->cfg.num_extras; ++e) t->batch.extras[e] = t->scalars + o_extra[e];
  memset(&t->c51, 0, sizeof(t->c51));
  t->c51.batch = t->cfg.logit_rows;
  t->c51.num_actions = cfg->num_actions;
  t->c51.num_atoms = cfg->num_atoms;
  t->c51.cumulative_gamma = cfg->cumulative_gamma;
  t->c51.support = t->support;
  t->c51.loss = reinterpret_cast<float *>(t->scalars + o_loss);
  t->c51.priorities = reinterpret_cast<float *>(t->scalars + o_prio);
  t->c51.weights = reinterpret_cast<float *>(t->scalars + o_w);
  t->slots = reinterpret_cast<int32_t *>(t->scalars + o_slots);
  t->loss_buf[0] = t->c51.loss;
  t->loss_buf[1] = reinterpret_cast<float *>(t->scalars + o_loss1);
  for (int k = 0; k < 2; ++k)  // copied back with the losses
    t->count_buf[k] = reinterpret_cast<int32_t *>(t->loss_buf[k] + B);

  B2R_CUDA(cudaStreamCreateWithFlags(&t->copy, cudaStreamNonBlocking));
  B2R_CUDA(cudaStreamCreateWithFlags(&t->copy_out, cudaStreamNonBlocking));
  B2R_CUDA(cudaStreamCreateWithFlags(&t->cap, cudaStreamNonBlocking));
  for (int k = 0; k < 2; ++k) {
    B2R_CUDA(cudaEventCreateWithFlags(&t->ev_in[k], cudaEventDisableTiming));
    B2R_CUDA(cudaEventCreateWithFlags(&t->ev_loss[k], cudaEventDisableTiming));
  }
  t->ring = cfg->pipeline_depth + 1;
  B2R_CUDA(cudaMallocHost(reinterpret_cast<void **>(&t->ring_host),
                          (size_t)t->ring * (B + 1) * sizeof(float)));
  t->ev_done.resize(t->ring);
  for (int k = 0; k < t->ring; ++k)
    B2R_CUDA(cudaEventCreateWithFlags(&t->ev_done[k], cudaEventDisableTiming));
  {
    void *as_device = nullptr;
    if (cudaHostGetDevicePointer(&as_device, t->ring_host, 0) == cudaSuccess)
      t->ring_dev = static_cast<float *>(as_device);
    else
      cudaGetLastError();
    const char *e = std::getenv("B2R_TRAINER_DIRECT");
    t->direct_ok = t->ring_dev != nullptr &&
                   (e != nullptr ? std::atoi(e) != 0 : cfg->pipeline_depth == 0);
  }
  *out = t;
  return B2R_OK;
}

int b2r_trainer_destroy(b2r_trainer *t) {
  if (!t) return B2R_OK;
  cudaDeviceSynchronize();
  if (b2r::g_host_trace.on && b2r::g_host_trace.calls > 0) {
    static const char *names[8] = {"collect (wait + copy out)", "logits H2D + events",
                                   "flush staged adds", "sampler launch",
                                   "gather fork", "loss launch", "write-back + join",
                                   "loss D2H + events"};
    fprintf(stderr, "b2r host trace over %ld trainer steps (us per step):\n",
            b2r::g_host_trace.calls);
    for (int k = 1; k <= 8; ++k)
      fprintf(stderr, "  %-28s %6.2f\n", names[k % 8],
              b2r::g_host_trace.acc[k % 8] / b2r::g_host_trace.calls);
    b2r::g_host_trace = b2r::HostTrace();
  }
  for (int set = 0; set < 2; ++set)
    for (int k = 0; k < 2; ++k) cudaFree(t->logits[set][k]);
  cudaFree(t->support);
  cudaFree(t->frames);
  cudaFree(t->scalars);
  if (t->copy) cudaStreamDestroy(t->copy);
  if (t->copy_out) cudaStreamDestroy(t->copy_out);
  if (t->cap) cudaStreamDestroy(t->cap);
  for (int k = 0; k < 2; ++k)
    if (t->exec[k]) cudaGraphExecDestroy(t->exec[k]);
  for (int k = 0; k < 2; ++k) {
    if (t->ev_in[k]) cudaEventDestroy(t->ev_in[k]);
    if (t->ev_loss[k]) cudaEventDestroy(t->ev_loss[k]);
  }
  if (t->ring_host) cudaFreeHost(t->ring_host);
  for (cudaEvent_t e : t->ev_done) cudaEventDestroy(e);
  delete t;
  return B2R_OK;
}

int b2r_trainer_step_host(b2r_trainer *t, const float *online_logits,
                          const float *target_logits, float *loss_out,
                          int64_t *loss_step, b2r_stream stream) {
  if (!t || !online_logits || !target_logits)
    return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  if (!t->exchange && t->cfg.logit_rows != t->cfg.batch)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "logit_rows below the batch is for a shard's trainer (set the exchange)");
  cudaStream_t s = as_stream(stream);
  b2r::g_host_trace.start();
  const int64_t n = t->submitted;
  const int set = (int)(n & 1);
  // ---- direct I/O: no copies, the kernels reach into the caller's page-locked memory
  if (t->direct_ok && !t->cfg.use_graph) {
    if (t->probed[0] != online_logits || t->probed[1] != target_logits) {
      void *d0 = nullptr, *d1 = nullptr;
      const bool mapped =
          cudaHostGetDevicePointer(&d0, const_cast<float *>(online_logits), 0) == cudaSuccess &&
          cudaHostGetDevicePointer(&d1, const_cast<float *>(target_logits), 0) == cudaSuccess;
      if (!mapped) cudaGetLastError();  // pageable memory: the copy path below
      t->probed[0] = online_logits;
      t->probed[1] = target_logits;
      t->probed_dev[0] = mapped ? static_cast<const float *>(d0) : nullptr;
      t->probed_dev[1] = mapped ? static_cast<const float *>(d1) : nullptr;
    }
    b2r_c51_args c51 = t->c51;
    c51.batch = t->exchange ? t->cfg.logit_rows : t->cfg.batch;
    if (t->probed_dev[0] != nullptr && b2r::c51_can_split(&c51)) {
      const int slot = (int)(n % t->ring);
      c51.online_logits = t->logits[set][0];   // device copy left by the first half
      c51.target_logits = t->probed_dev[1];
      c51.loss = t->loss_buf[set];
      b2r::DirectIO io;
      io.online_src = t->probed_dev[0];
      io.online_copy = t->logits[set][0];
      io.loss_host = t->ring_dev + (size_t)slot * (t->cfg.logit_rows + 1);
      // the buffers of this set were last read by the tail of step n - 2
      io.first_half_after = n >= 2 ? t->ev_done[(size_t)((n - 2) % t->ring)] : nullptr;
      b2r::ShardSpec shard = {t->exchange, t->slots, t->count_buf[set], t->cfg.logit_rows,
                              false, nullptr};
      // (the result slot of step n is read by the host after ev_done[slot], recorded
      // behind the tail; with ring = depth + 1 slots it was collected before this call)
      B2R_TRY(b2r::train_step(t->buf, t->cfg.batch, t->cfg.seed, 0, &t->batch, &c51, s,
                              nullptr, t->ev_done[slot], t->exchange ? &shard : nullptr, &io));
      t->submitted = n + 1;
      b2r::g_host_trace.lap(7);
      const int status = collect(t, n - t->cfg.pipeline_depth, loss_out, loss_step);
      b2r::g_host_trace.lap(0);
      b2r::g_host_trace.calls += 1;
      return status;
    }
  }
  const size_t logit_bytes = (size_t)t->cfg.logit_rows * t->cfg.num_actions *
                             t->cfg.num_atoms * sizeof(float);
  // inputs: on the copy stream, beside the sampler; set `set` was last read by the
  // loss kernel of step n - 2.
  // (step n - 2's loss is done: ev_loss[set] in the copy path, the event behind its tail
  // — ev_done of its slot — when the kernel wrote the losses; waiting for the later of the
  // two records covers both)
  b2r_c51_args probe = t->c51;  // (c51.batch is the rows behind the sampler)
  const bool through_first_half = !t->cfg.use_graph && b2r::c51_can_split(&probe);
  const bool kernel_writes_losses = through_first_half && t->ring_dev != nullptr;
  if (n >= 2)
    B2R_CUDA(cudaStreamWaitEvent(
        t->copy, kernel_writes_losses ? t->ev_done[(size_t)((n - 2) % t->ring)]
                                      : t->ev_loss[set], 0));
  B2R_CUDA(cudaMemcpyAsync(t->logits[set][0], online_logits, logit_bytes,
                           cudaMemcpyHostToDevice, t->copy));
  B2R_CUDA(cudaMemcpyAsync(t->logits[set][1], target_logits, logit_bytes,
                           cudaMemcpyHostToDevice, t->copy));
  B2R_CUDA(cudaEventRecord(t->ev_in[set], t->copy));
  // The loss buffer of this set was last read by the result copy of step n - 2.  With a
  // pipeline of depth <= 1 the host has already waited for that copy (collect); deeper
  // pipelines order the step behind it on the device: the eager path through the first
  // half of the loss (which the sampler of this step waits for: `hints` below), the
  // graph-replayed path on `s`.
  const bool behind_copy = n >= 2 && t->cfg.pipeline_depth >= 2;
  b2r::DirectIO hints = {nullptr, nullptr, nullptr,
                         n >= 2 ? t->ev_done[(size_t)((n - 2) % t->ring)] : nullptr};
  // ... and then the tail writes the per-row losses into this step's page-locked result
  // slot itself (33 words over PCIe): no result copy, no result-copy stream; the event
  // the host collects on is recorded behind the tail.
  const int slot = (int)(n % t->ring);
  if (kernel_writes_losses)
    hints.loss_host = t->ring_dev + (size_t)slot * (t->cfg.logit_rows + 1);
  cudaEvent_t after_loss = kernel_writes_losses ? t->ev_done[slot] : t->ev_loss[set];
  if (behind_copy && !through_first_half)
    B2R_CUDA(cudaStreamWaitEvent(s, t->ev_done[(size_t)((n - 2) % t->ring)], 0));
  if (t->exchange) {
    b2r_c51_args c51 = t->c51;
    c51.online_logits = t->logits[set][0];
    c51.target_logits = t->logits[set][1];
    c51.loss = t->loss_buf[set];
    b2r::ShardSpec shard = {t->exchange, t->slots, t->count_buf[set], t->cfg.logit_rows,
                            false, nullptr};
    B2R_TRY(b2r::train_step(t->buf, t->cfg.batch, t->cfg.seed, 0, &t->batch, &c51, s,
                            t->ev_in[set], after_loss, &shard, &hints));
  } else if (t->cfg.use_graph && n >= 2) {
    // Everything host-dependent (staged adds, validity context) goes first, eagerly;
    // the replayed graph reads it from HBM.
    B2R_TRY(b2r::flush_queue(t->buf, s, t->cfg.batch > b2r::kSplitMin));
    B2R_TRY(b2r::ensure_ctx(t->buf, s));
    if (!t->exec[set]) B2R_TRY(capture_step(t, set));
    B2R_CUDA(cudaStreamWaitEvent(s, t->ev_in[set], 0));
    B2R_CUDA(cudaGraphLaunch(t->exec[set], s));
    b2r::g_launches.fetch_add(4, std::memory_order_relaxed);
    B2R_CUDA(cudaEventRecord(t->ev_loss[set], s));
  } else {
    b2r_c51_args c51 = t->c51;
    c51.online_logits = t->logits[set][0];
    c51.target_logits = t->logits[set][1];
    c51.loss = t->loss_buf[set];
    B2R_TRY(b2r::train_step(t->buf, t->cfg.batch, t->cfg.seed, 0, &t->batch, &c51, s,
                            t->ev_in[set], after_loss, nullptr, &hints));
  }
  if (!kernel_writes_losses) {
    // result: per-row losses into this step's pinned slot (copy stream, after the loss)
    B2R_CUDA(cudaStreamWaitEvent(t->copy_out, t->ev_loss[set], 0));
    B2R_CUDA(cudaMemcpyAsync(t->ring_host + (size_t)slot * (t->cfg.logit_rows + 1),
                             t->loss_buf[set],
                             (size_t)(t->cfg.logit_rows + 1) * sizeof(float),
                             cudaMemcpyDeviceToHost, t->copy_out));
    B2R_CUDA(cudaEventRecord(t->ev_done[slot], t->copy_out));
  }
  t->submitted = n + 1;
  b2r::g_host_trace.lap(7);
  const int status = collect(t, n - t->cfg.pipeline_depth, loss_out, loss_step);
  b2r::g_host_trace.lap(0);
  b2r::g_host_trace.calls += 1;
  return status;
}

int b2r_trainer_set_exchange(b2r_trainer *t, b2r_exchange *x) {
  if (!t || !x) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  if (t->submitted != 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "set the exchange before the first step");
  t->exchange = x;
  return B2R_OK;
}

int32_t b2r_trainer_last_rows(const b2r_trainer *t) { return t ? t->last_rows : 0; }

int b2r_trainer_drain(b2r_trainer *t, float *loss_out, int64_t *loss_step,
                      b2r_stream stream) {
  if (!t) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  B2R_CUDA(cudaStreamSynchronize(t->copy));
  B2R_CUDA(cudaStreamSynchronize(t->copy_out));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return collect(t, t->submitted - 1, loss_out, loss_step);
}

int b2r_trainer_views(b2r_trainer *t, b2r_batch *batch, b2r_c51_args *c51) {
  if (!t) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  if (batch) *batch = t->batch;
  if (c51) {
    *c51 = t->c51;
    const int set = (int)((t->submitted + 1) & 1);  // set of the last queued step
    c51->online_logits = t->logits[set][0];
    c51->target_logits = t->logits[set][1];
    c51->loss = t->loss_buf[set];
    c51->actions = static_cast<const int32_t *>(t->batch.action);
    c51->rewards = static_cast<const float *>(t->batch.reward);
    c51->terminals = static_cast<const uint8_t *>(t->batch.terminal);
    c51->sampling_probabilities = t->batch.sampling_probabilities;
  }
  return B2R_OK;
}

}  // extern "C"
