// HBM-resident circular replay storage: replaces the numpy `_store` and the add
// path of OutOfGraphReplayBuffer (circular_replay_buffer.py:98-336) and of
// OutOfGraphPrioritizedReplayBuffer (prioritized_replay_buffer.py:117-140).
//
// Layout in HBM: one dense array per storage element, row = slot:
//   observation  capacity x obs_bytes   (7 056 B per Atari frame = 441 x 16 B, so
//                                         every frame is 16-byte aligned)
//   action / reward / terminal / extras  capacity x row_bytes
//   term_flag    capacity x 1 B          (terminal != 0; what validity and the
//                                         n-step cut test)
// Adds are host-driven (the agent calls add once per env step), so rows are staged
// in pinned memory and written by ONE kernel per flush with 16-byte vector stores;
// every reader flushes first, so deferral is unobservable.
#include "replay.cuh"

#include <cmath>
#include <cstdlib>
#include <new>

namespace b2r {
namespace {

// grid = (x: 16-byte chunks of the observation, y: entries).
__global__ void __launch_bounds__(256) add_rows_kernel(AddParams p) {
  add_rows_body(p, blockIdx.y, blockIdx.x, gridDim.x);
}

__global__ void valid_mask_kernel(ValidCtx ctx, int64_t n,
                                  const int64_t *__restrict__ indices,
                                  uint8_t *__restrict__ out) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) out[k] = is_valid_transition(ctx, indices[k]) ? 1 : 0;
}

__global__ void term_flag_rebuild_kernel(const uint8_t *__restrict__ terminal,
                                         int itemsize, int64_t row0, int64_t n,
                                         uint8_t *__restrict__ flag) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  uint8_t any = 0;
  for (int b = 0; b < itemsize; ++b) any |= terminal[(row0 + k) * itemsize + b];
  flag[row0 + k] = any ? 1 : 0;
}

int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

bool terminal_equals_one(const void *p, int itemsize) {
  switch (itemsize) {
    case 1: return *static_cast<const uint8_t *>(p) == 1;
    case 2: { uint16_t v; memcpy(&v, p, 2); return v == 1; }
    case 4: { uint32_t v; memcpy(&v, p, 4); return v == 1; }
    default: { uint64_t v; memcpy(&v, p, 8); return v == 1; }
  }
}

// SoA entry table at the front of a staging buffer.
struct Header {
  int64_t *slots;
  double *prio;
  int32_t *src_rows;
  uint8_t *mode;
};

Header header_of(uint8_t *base, int cap) {
  Header h;
  h.slots = reinterpret_cast<int64_t *>(base);
  h.prio = reinterpret_cast<double *>(base + (size_t)cap * 8);
  h.src_rows = reinterpret_cast<int32_t *>(base + (size_t)cap * 16);
  h.mode = base + (size_t)cap * 20;
  return h;
}

void recompute_invalid_range(b2r_buffer *b) {
  // circular_replay_buffer.py:53-77 with the post-increment cursor (CRB:284-287).
  const int64_t cap = b->cfg.capacity;
  const int64_t cursor = b->add_count % cap;
  const int n = b->cfg.stack_size + b->cfg.update_horizon;
  b->invalid_range.resize(n);
  for (int i = 0; i < n; ++i) {
    int64_t v = (cursor - b->cfg.update_horizon + i) % cap;
    if (v < 0) v += cap;
    b->invalid_range[i] = v;
  }
}

int wait_staging(Staging *s) {
  if (s->in_flight) {
    B2R_CUDA(cudaEventSynchronize(s->done));
    s->in_flight = false;
  }
  return B2R_OK;
}

// Appends one entry (a real row when `row` is set, else a zero transition).
int enqueue(b2r_buffer *b, bool real, const void *const *cols, double priority,
            int mode, cudaStream_t stream) {
  if (b->q_entries == b->queue_cap) B2R_TRY(flush_queue(b, stream));
  Staging *s = &b->staging[b->active];
  if (b->q_entries == 0) B2R_TRY(wait_staging(s));
  Header h = header_of(s->host, b->queue_cap);
  const int64_t slot = b->add_count % b->cfg.capacity;
  const int e = b->q_entries++;
  h.slots[e] = slot;
  h.prio[e] = priority;
  h.mode[e] = (uint8_t)mode;
  if (real) {
    uint8_t *row = s->host + b->header_bytes + (int64_t)b->q_rows * b->row_stride;
    for (int c = 0; c < b->num_columns; ++c)
      memcpy(row + b->col[c].queue_offset, cols[c], (size_t)b->col[c].row_bytes);
    h.src_rows[e] = b->q_rows++;
    b->term_is_one[slot] =
        terminal_equals_one(cols[3], b->cfg.terminal_itemsize) ? 1 : 0;
  } else {
    h.src_rows[e] = -1;
    b->term_is_one[slot] = 0;
  }
  b->add_count += 1;
  return B2R_OK;
}

}  // namespace

// Largest flush that goes out as the one fused launch (its tree half is the one-CTA
// kernel body, which copes with up to 256 entries but is only quick for a few dozen).
constexpr int kFusedFlushMax = 64;

int join_frames(b2r_buffer *b, cudaStream_t stream) {
  if (!b->frames_pending) return B2R_OK;
  B2R_CUDA(cudaStreamWaitEvent(stream, b->ev_join, 0));
  b->frames_pending = false;
  b->slot_busy[0] = b->slot_busy[1] = false;  // (the copies run in order)
  return B2R_OK;
}

int flush_queue(b2r_buffer *b, cudaStream_t stream, bool split,
                const b2r_exchange *publish) {
  if (b->q_entries == 0) return B2R_OK;
  // the new rows overwrite ring slots that deferred frame copies may still be reading
  B2R_TRY(join_frames(b, stream));
  if (b->deferred_frames) split = false;  // (`side` is the copies' stream)
  Staging *s = &b->staging[b->active];
  const size_t bytes = (size_t)b->header_bytes + (size_t)b->q_rows * b->row_stride;
  // the validity context as of these adds travels in the header
  const size_t ctx_off = (size_t)b->header_bytes - sizeof(ValidCtx);
  fill_valid_ctx(b, reinterpret_cast<ValidCtx *>(s->host + ctx_off));
  // split: rows (H2D + ring writes) on the side stream, ordered after everything
  // already queued on `stream` (earlier readers of the ring), beside the tree update.
  // Small flushes of a prioritized buffer (the agent's add loop: a handful of rows
  // per update): ONE launch that reads the staging buffer straight from pinned host
  // memory — tree update in CTA 0, row writes in the others (tree.cu).
  if (b->tree != nullptr && !split && s->host_dev != nullptr &&
      b->q_entries <= kFusedFlushMax) {
    Header hh = header_of(s->host_dev, b->queue_cap);
    AddParams p;
    p.n_entries = b->q_entries;
    p.num_columns = b->num_columns;
    p.row_stride = b->row_stride;
    p.slots = hh.slots;
    p.src_rows = hh.src_rows;
    p.rows = s->host_dev + b->header_bytes;
    for (int c = 0; c < b->num_columns; ++c) {
      p.col_dev[c] = b->col[c].dev;
      p.col_bytes[c] = b->col[c].row_bytes;
      p.col_qoff[c] = b->col[c].queue_offset;
    }
    p.term_flag = b->term_flag_owned ? b->term_flag : nullptr;
    p.term_itemsize = b->cfg.terminal_itemsize;
    p.ctx_src = reinterpret_cast<const uint64_t *>(s->host_dev + ctx_off);
    p.ctx_dst = reinterpret_cast<uint64_t *>(b->ctx_dev);
    const int64_t chunks = (b->cfg.obs_bytes & 15) == 0 ? b->cfg.obs_bytes >> 4
                                                         : b->cfg.obs_bytes;
    const int threads = 32 * (b->tree->depth + 1);
    int per_entry = (int)((chunks + threads - 1) / threads);
    if (per_entry < 1) per_entry = 1;
    if (per_entry > 8) per_entry = 8;
    B2R_TRY(flush_fused(b->tree, b->q_entries, hh.slots, hh.prio, hh.mode, p, per_entry,
                        stream, publish));
    b->ctx_dirty = false;
    B2R_CUDA(cudaEventRecord(s->done, stream));
    s->in_flight = true;
    b->active ^= 1;
    b->q_entries = 0;
    b->q_rows = 0;
    return B2R_OK;
  }
  cudaStream_t data = stream;
  if (split) {
    data = b->side;
    B2R_CUDA(cudaEventRecord(b->ev_pre, stream));
    B2R_CUDA(cudaStreamWaitEvent(data, b->ev_pre, 0));
  }
  B2R_CUDA(cudaMemcpyAsync(s->dev, s->host, bytes, cudaMemcpyHostToDevice, data));
  if (split) {
    B2R_CUDA(cudaEventRecord(b->ev_h2d, data));
    B2R_CUDA(cudaStreamWaitEvent(stream, b->ev_h2d, 0));
  }
  Header hd = header_of(s->dev, b->queue_cap);
  if (b->tree != nullptr) {
    // prioritized_replay_buffer.py:139-140: sum_tree.set(cursor, priority) per row,
    // in add order (zero transitions carry priority 0).
    B2R_TRY((tree_apply<int64_t, double>(b->tree, b->q_entries, hd.slots, hd.prio,
                                         hd.mode, stream, nullptr, -1, 0, publish)));
  }
  AddParams p;
  p.n_entries = b->q_entries;
  p.num_columns = b->num_columns;
  p.row_stride = b->row_stride;
  p.slots = hd.slots;
  p.src_rows = hd.src_rows;
  p.rows = s->dev + b->header_bytes;
  for (int c = 0; c < b->num_columns; ++c) {
    p.col_dev[c] = b->col[c].dev;
    p.col_bytes[c] = b->col[c].row_bytes;
    p.col_qoff[c] = b->col[c].queue_offset;
  }
  p.term_flag = b->term_flag_owned ? b->term_flag : nullptr;
  p.term_itemsize = b->cfg.terminal_itemsize;
  p.ctx_src = reinterpret_cast<const uint64_t *>(s->dev + ctx_off);
  p.ctx_dst = reinterpret_cast<uint64_t *>(b->ctx_dev);
  b->ctx_dirty = false;
  const int64_t work = (b->cfg.obs_bytes & 15) == 0 ? b->cfg.obs_bytes >> 4
                                                    : b->cfg.obs_bytes;
  int gx = (int)((work + 255) / 256);
  if (gx < 1) gx = 1;
  if (gx > 64) gx = 64;
  add_rows_kernel<<<dim3(gx, b->q_entries), 256, 0, data>>>(p);
  B2R_LAUNCHED();
  if (split) {
    B2R_CUDA(cudaEventRecord(b->ev_rows, data));
    B2R_CUDA(cudaStreamWaitEvent(stream, b->ev_rows, 0));
  }
  B2R_CUDA(cudaEventRecord(s->done, stream));
  s->in_flight = true;
  b->active ^= 1;
  b->q_entries = 0;
  b->q_rows = 0;
  return B2R_OK;
}

void fill_valid_ctx(const b2r_buffer *b, ValidCtx *ctx) {
  ctx->capacity = b->cfg.capacity;
  ctx->add_count = b->add_count;
  ctx->cursor = b->add_count % b->cfg.capacity;
  ctx->stack = b->cfg.stack_size;
  ctx->horizon = b->cfg.update_horizon;
  ctx->n_invalid = (int)b->invalid_range.size();
  for (int i = 0; i < ctx->n_invalid; ++i) ctx->invalid[i] = b->invalid_range[i];
  ctx->term_flag = b->term_flag;
}

int ensure_ctx(b2r_buffer *b, cudaStream_t stream) {
  if (!b->ctx_dirty) return B2R_OK;
  ValidCtx image;
  fill_valid_ctx(b, &image);
  // pageable source: the runtime stages it before returning, `image` may go away
  B2R_CUDA(cudaMemcpyAsync(b->ctx_dev, &image, sizeof(image), cudaMemcpyHostToDevice,
                           stream));
  b->ctx_dirty = false;
  return B2R_OK;
}

int ensure_inv_slots(b2r_buffer *b, int64_t n) {
  if (n <= b->inv_slots_cap) return B2R_OK;
  if (b->inv_slots) cudaFree(b->inv_slots);
  b->inv_slots = nullptr;
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->inv_slots), (size_t)n * 4));
  b->inv_slots_cap = n;
  return B2R_OK;
}

}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

namespace b2r {
int refresh_terminal_mirror(b2r_buffer *b, int64_t row0, int64_t nrows, cudaStream_t s) {
  // `in` of a store write may be a device pointer, and a checkpoint load writes the
  // column from a kernel, so the rows are read back from the store itself.
  const int64_t rb = b->col[B2R_COL_TERMINAL].row_bytes;
  std::vector<uint8_t> rows((size_t)(nrows * rb));
  B2R_CUDA(cudaMemcpyAsync(rows.data(), b->col[B2R_COL_TERMINAL].dev + row0 * rb,
                           rows.size(), cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  for (int64_t k = 0; k < nrows; ++k)
    b->term_is_one[row0 + k] = terminal_equals_one(rows.data() + k * rb,
                                                   b->cfg.terminal_itemsize);
  if (b->term_flag_owned && nrows > 0) {
    term_flag_rebuild_kernel<<<(unsigned)((nrows + 255) / 256), 256, 0, s>>>(
        b->col[B2R_COL_TERMINAL].dev, b->cfg.terminal_itemsize, row0, nrows, b->term_flag);
    B2R_LAUNCHED();
  }
  return B2R_OK;
}
}  // namespace b2r

extern "C" {

int b2r_create(const b2r_config *cfg, b2r_buffer **out) {
  if (!cfg || !out) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  *out = nullptr;
  if (cfg->capacity < (int64_t)cfg->update_horizon + cfg->stack_size)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "There is not enough capacity to cover update_horizon and "
                "stack_size.");
  if (cfg->stack_size < 1 || cfg->update_horizon < 1)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "stack_size and update_horizon must be positive");
  if (cfg->stack_size + cfg->update_horizon > b2r::kMaxInvalid)
    return fail(B2R_ERR_UNSUPPORTED,
                "stack_size + update_horizon above %d is not supported",
                b2r::kMaxInvalid);
  if (cfg->num_extras < 0 || cfg->num_extras > B2R_MAX_EXTRAS)
    return fail(B2R_ERR_UNSUPPORTED, "at most %d extra storage types",
                B2R_MAX_EXTRAS);
  if (cfg->reward_itemsize != 4 && cfg->reward_itemsize != 8)
    return fail(B2R_ERR_UNSUPPORTED, "reward must be float32 or float64");
  if (cfg->terminal_itemsize != 1 && cfg->terminal_itemsize != 2 &&
      cfg->terminal_itemsize != 4 && cfg->terminal_itemsize != 8)
    return fail(B2R_ERR_UNSUPPORTED, "terminal must be a 1/2/4/8-byte integer");
  if (cfg->obs_bytes <= 0 || cfg->obs_itemsize <= 0 ||
      cfg->obs_bytes % cfg->obs_itemsize != 0 || cfg->action_bytes <= 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad observation/action size");
  if (cfg->capacity > (1ll << 30))
    return fail(B2R_ERR_UNSUPPORTED, "capacity above 2^30 is not supported");
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count == 0)
    return fail(B2R_ERR_CUDA,
                "no CUDA device: libb200replay has no CPU fallback");

  b2r_buffer *b = new (std::nothrow) b2r_buffer();
  if (!b) return fail(B2R_ERR_INVALID_ARGUMENT, "out of host memory");
  b->cfg = *cfg;
  b->num_columns = 4 + cfg->num_extras;
  b->col[0].row_bytes = cfg->obs_bytes;
  b->col[1].row_bytes = cfg->action_bytes;
  b->col[2].row_bytes = cfg->reward_itemsize;
  b->col[3].row_bytes = cfg->terminal_itemsize;
  for (int e = 0; e < cfg->num_extras; ++e) {
    if (cfg->extra_bytes[e] <= 0) {
      delete b;
      return fail(B2R_ERR_INVALID_ARGUMENT, "extra %d has no bytes", e);
    }
    b->col[4 + e].row_bytes = cfg->extra_bytes[e];
  }
  int64_t off = 0;
  for (int c = 0; c < b->num_columns; ++c) {
    b->col[c].queue_offset = off;
    off = b2r::align_up(off + b->col[c].row_bytes, c == 0 ? 16 : 8);
  }
  b->row_stride = b2r::align_up(off, 16);
  b->queue_cap = cfg->add_queue_rows > 0 ? cfg->add_queue_rows : 128;
  // One flush never holds two rows for the same slot (the row kernel writes
  // entries concurrently), so the queue is no longer than the ring.
  if (b->queue_cap > cfg->capacity) b->queue_cap = (int)cfg->capacity;
  b->header_bytes = b2r::align_up(
      (int64_t)b->queue_cap * 21 + 64 + 16 + (int64_t)sizeof(b2r::ValidCtx), 256);

  for (int c = 0; c < b->num_columns; ++c) {
    const size_t bytes = (size_t)cfg->capacity * (size_t)b->col[c].row_bytes;
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->col[c].dev), bytes));
    // The reference uses np.empty (garbage); zero-filling is allowed, nothing may
    // depend on it (SURVEY.md Q1).
    B2R_CUDA(cudaMemset(b->col[c].dev, 0, bytes));
  }
  if (cfg->terminal_itemsize == 1) {
    b->term_flag = b->col[3].dev;
  } else {
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->term_flag),
                        (size_t)cfg->capacity));
    B2R_CUDA(cudaMemset(b->term_flag, 0, (size_t)cfg->capacity));
    b->term_flag_owned = true;
  }
  // circular_replay_buffer.py:181-183: float32(math.pow(gamma, k)).
  b->discounts_host.resize(cfg->update_horizon);
  for (int k = 0; k < cfg->update_horizon; ++k)
    b->discounts_host[k] = (float)std::pow(cfg->gamma, (double)k);
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->discounts),
                      (size_t)cfg->update_horizon * 4));
  B2R_CUDA(cudaMemcpy(b->discounts, b->discounts_host.data(),
                      (size_t)cfg->update_horizon * 4, cudaMemcpyHostToDevice));
  if (cfg->prioritized) {
    int st = b2r_tree_create(cfg->capacity, &b->tree);
    if (st != B2R_OK) return st;
  }
  b->term_is_one.assign((size_t)cfg->capacity, 0);
  b->invalid_range.assign((size_t)cfg->stack_size, 0);  // np.zeros(stack) CRB:178
  const size_t staging_bytes =
      (size_t)b->header_bytes + (size_t)b->queue_cap * (size_t)b->row_stride;
  for (int k = 0; k < 2; ++k) {
    B2R_CUDA(cudaMallocHost(reinterpret_cast<void **>(&b->staging[k].host),
                            staging_bytes));
    void *as_device = nullptr;
    if (cudaHostGetDevicePointer(&as_device, b->staging[k].host, 0) == cudaSuccess)
      b->staging[k].host_dev = static_cast<uint8_t *>(as_device);
    else
      cudaGetLastError();
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->staging[k].dev),
                        staging_bytes));
    B2R_CUDA(cudaEventCreateWithFlags(&b->staging[k].done,
                                      cudaEventDisableTiming));
  }
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->info), 64));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->status), 16));
  B2R_CUDA(cudaMemset(b->status, 0, 16));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->shard_counter), 8));
  B2R_CUDA(cudaMemset(b->shard_counter, 0, 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->draw_counter), 8));
  B2R_CUDA(cudaMemset(b->draw_counter, 0, 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->ctx_dev), sizeof(b2r::ValidCtx)));
  B2R_CUDA(cudaMemset(b->ctx_dev, 0, sizeof(b2r::ValidCtx)));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->min_prob), 4));
  B2R_CUDA(cudaMemset(b->min_prob, 0, 4));
  B2R_CUDA(cudaStreamCreateWithFlags(&b->side, cudaStreamNonBlocking));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming));
  {
    int least = 0, greatest = 0;
    cudaDeviceGetStreamPriorityRange(&least, &greatest);
    B2R_CUDA(cudaStreamCreateWithPriority(&b->side3, cudaStreamNonBlocking, greatest));
  }
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&b->sync), sizeof(b2r::StepSync)));
  B2R_CUDA(cudaMemset(b->sync, 0, sizeof(b2r::StepSync)));
  for (int k = 0; k < 2; ++k)
    B2R_CUDA(cudaEventCreateWithFlags(&b->ev_slot_free[k], cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_c51_fork, cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_c51_pre, cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_pre, cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_h2d, cudaEventDisableTiming));
  B2R_CUDA(cudaEventCreateWithFlags(&b->ev_rows, cudaEventDisableTiming));
  *out = b;
  return B2R_OK;
}

int b2r_destroy(b2r_buffer *b) {
  if (!b) return B2R_OK;
  cudaDeviceSynchronize();
  for (int c = 0; c < b->num_columns; ++c) cudaFree(b->col[c].dev);
  if (b->term_flag_owned) cudaFree(b->term_flag);
  cudaFree(b->discounts);
  if (b->tree) b2r_tree_destroy(b->tree);
  for (int k = 0; k < 2; ++k) {
    if (b->staging[k].host) cudaFreeHost(b->staging[k].host);
    if (b->staging[k].dev) cudaFree(b->staging[k].dev);
    if (b->staging[k].done) cudaEventDestroy(b->staging[k].done);
  }
  if (b->inv_slots) cudaFree(b->inv_slots);
  cudaFree(b->info);
  cudaFree(b->status);
  cudaFree(b->draw_counter);
  cudaFree(b->shard_counter);
  cudaFree(b->min_prob);
  cudaFree(b->ctx_dev);
  if (b->side) cudaStreamDestroy(b->side);
  if (b->ev_fork) cudaEventDestroy(b->ev_fork);
  if (b->ev_join) cudaEventDestroy(b->ev_join);
  if (b->side3) cudaStreamDestroy(b->side3);
  if (b->ev_c51_fork) cudaEventDestroy(b->ev_c51_fork);
  if (b->ev_c51_pre) cudaEventDestroy(b->ev_c51_pre);
  if (b->c51_bestp) cudaFree(b->c51_bestp);
  if (b->c51_logp) cudaFree(b->c51_logp);
  if (b->sync) cudaFree(b->sync);
  if (b->idx_ring) cudaFree(b->idx_ring);
  for (int k = 0; k < 2; ++k)
    if (b->ev_slot_free[k]) cudaEventDestroy(b->ev_slot_free[k]);
  if (b->ev_pre) cudaEventDestroy(b->ev_pre);
  if (b->ev_h2d) cudaEventDestroy(b->ev_h2d);
  if (b->ev_rows) cudaEventDestroy(b->ev_rows);
  if (b->out_scratch) cudaFree(b->out_scratch);
  b->bounce.release();
  delete b;
  return B2R_OK;
}

b2r_tree *b2r_buffer_tree(b2r_buffer *b) { return b ? b->tree : nullptr; }

int b2r_add(b2r_buffer *b, const void *observation, const void *action,
            const void *reward, const void *terminal, const void *const *extras,
            double priority, int priority_mode, b2r_stream stream) {
  if (stream == B2R_STREAM_NONE) {
    // worst case stack_size - 1 zero transitions + the row itself
    if (b->q_entries + b->cfg.stack_size > b->queue_cap) return B2R_QUEUE_FULL;
    stream = nullptr;  // no launch can happen below
  }
  cudaStream_t s = as_stream(stream);
  const void *cols[b2r::kMaxColumns] = {observation, action, reward, terminal};
  for (int e = 0; e < b->cfg.num_extras; ++e) cols[4 + e] = extras[e];
  for (int c = 0; c < b->num_columns; ++c)
    if (cols[c] == nullptr)
      return fail(B2R_ERR_INVALID_ARGUMENT, "add: column %d is NULL", c);
  // circular_replay_buffer.py:255-259: stack_size-1 zero transitions when the
  // buffer is empty or the previous slot closed an episode (terminal == 1).
  const int64_t cap = b->cfg.capacity;
  const int64_t prev = ((b->add_count % cap) - 1 + cap) % cap;
  if (b->add_count == 0 || b->term_is_one[prev]) {
    for (int k = 0; k < b->cfg.stack_size - 1; ++k)
      B2R_TRY(b2r::enqueue(b, false, nullptr, 0.0, B2R_PRIORITY_EXPLICIT, s));
  }
  if (b->cfg.stack_size > 1) b2r::recompute_invalid_range(b);
  // sum_tree.set raises before the row is written (PRB:139, ST:191-193); the
  // zero transitions above have already been committed by then.
  if (b->tree && priority_mode == B2R_PRIORITY_EXPLICIT && priority < 0.0)
    return fail(B2R_ERR_NEGATIVE_PRIORITY,
                "Sum tree values should be nonnegative. Got %g", priority);
  B2R_TRY(b2r::enqueue(b, true, cols, priority, priority_mode, s));
  b2r::recompute_invalid_range(b);
  return B2R_OK;
}

int b2r_add_atari(b2r_buffer *b, const void *observation, int32_t action,
                  float reward, uint8_t terminal, double priority,
                  int priority_mode, b2r_stream stream) {
  if (b->cfg.action_bytes != 4 || b->cfg.reward_itemsize != 4 ||
      b->cfg.terminal_itemsize != 1 || b->cfg.num_extras != 0)
    return fail(B2R_ERR_UNSUPPORTED, "b2r_add_atari: not the Atari storage layout");
  return b2r_add(b, observation, &action, &reward, &terminal, nullptr, priority,
                 priority_mode, stream);
}

int b2r_add_batch(b2r_buffer *b, int64_t n, const void *observations,
                  const void *actions, const void *rewards, const void *terminals,
                  const void *const *extras, const double *priorities, int priority_mode,
                  int64_t *added, b2r_stream stream) {
  if (added) *added = 0;
  if (!b || n < 0 || (n > 0 && (!observations || !actions || !rewards || !terminals)))
    return fail(B2R_ERR_INVALID_ARGUMENT, "add_batch: bad argument");
  if (stream == B2R_STREAM_NONE)
    return fail(B2R_ERR_INVALID_ARGUMENT, "add_batch needs a stream: it may have to flush");
  if (b->tree && priority_mode == B2R_PRIORITY_EXPLICIT && n > 0 && !priorities)
    return fail(B2R_ERR_INVALID_ARGUMENT, "add_batch: explicit priorities are NULL");
  const uint8_t *col[4] = {static_cast<const uint8_t *>(observations),
                           static_cast<const uint8_t *>(actions),
                           static_cast<const uint8_t *>(rewards),
                           static_cast<const uint8_t *>(terminals)};
  const size_t stride[4] = {(size_t)b->cfg.obs_bytes, (size_t)b->cfg.action_bytes,
                            (size_t)b->cfg.reward_itemsize,
                            (size_t)b->cfg.terminal_itemsize};
  const void *extra_rows[B2R_MAX_EXTRAS] = {nullptr};
  for (int64_t k = 0; k < n; ++k) {
    for (int e = 0; e < b->cfg.num_extras; ++e)
      extra_rows[e] = static_cast<const uint8_t *>(extras[e]) +
                      (size_t)k * (size_t)b->cfg.extra_bytes[e];
    B2R_TRY(b2r_add(b, col[0] + k * stride[0], col[1] + k * stride[1],
                    col[2] + k * stride[2], col[3] + k * stride[3],
                    b->cfg.num_extras ? extra_rows : nullptr,
                    priorities ? priorities[k] : 0.0, priority_mode, stream));
    if (added) *added = k + 1;
  }
  return B2R_OK;
}

int b2r_flush(b2r_buffer *b, b2r_stream stream) {
  return b2r::flush_queue(b, as_stream(stream));
}

int64_t b2r_add_count(const b2r_buffer *b) { return b->add_count; }

int64_t b2r_cursor(const b2r_buffer *b) { return b->add_count % b->cfg.capacity; }

int b2r_get_invalid_range(const b2r_buffer *b, int64_t *out, int32_t *n) {
  *n = (int32_t)b->invalid_range.size();
  for (size_t i = 0; i < b->invalid_range.size(); ++i) out[i] = b->invalid_range[i];
  return B2R_OK;
}

int b2r_set_state(b2r_buffer *b, int64_t add_count, const int64_t *invalid_range,
                  int32_t n) {
  if (add_count < 0 || n < 0 || n > b2r::kMaxInvalid)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad state");
  b->add_count = add_count;
  b->invalid_range.assign(invalid_range, invalid_range + n);
  b->ctx_dirty = true;
  return B2R_OK;
}

int b2r_valid_mask(b2r_buffer *b, int64_t n, const int64_t *indices, uint8_t *out,
                   b2r_stream stream) {
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  B2R_TRY(b->bounce.reserve((size_t)n * 9 + 16));
  memcpy(b->bounce.host, indices, (size_t)n * 8);
  B2R_CUDA(cudaMemcpyAsync(b->bounce.dev, b->bounce.host, (size_t)n * 8,
                           cudaMemcpyHostToDevice, s));
  b2r::ValidCtx ctx;
  b2r::fill_valid_ctx(b, &ctx);
  uint8_t *dout = b->bounce.dev + (size_t)n * 8;
  b2r::valid_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
      ctx, n, reinterpret_cast<const int64_t *>(b->bounce.dev), dout);
  B2R_LAUNCHED();
  B2R_CUDA(cudaMemcpyAsync(b->bounce.host + (size_t)n * 8, dout, (size_t)n,
                           cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  memcpy(out, b->bounce.host + (size_t)n * 8, (size_t)n);
  return B2R_OK;
}

int b2r_store_read(b2r_buffer *b, int32_t column, int64_t row0, int64_t nrows,
                   void *out, b2r_stream stream) {
  if (column < 0 || column >= b->num_columns || row0 < 0 || nrows < 0 ||
      row0 + nrows > b->cfg.capacity)
    return fail(B2R_ERR_INVALID_ARGUMENT, "store_read out of range");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  const int64_t rb = b->col[column].row_bytes;
  B2R_CUDA(cudaMemcpyAsync(out, b->col[column].dev + row0 * rb,
                           (size_t)(nrows * rb), cudaMemcpyDefault, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  return B2R_OK;
}

int b2r_store_write(b2r_buffer *b, int32_t column, int64_t row0, int64_t nrows,
                    const void *in, b2r_stream stream) {
  if (column < 0 || column >= b->num_columns || row0 < 0 || nrows < 0 ||
      row0 + nrows > b->cfg.capacity)
    return fail(B2R_ERR_INVALID_ARGUMENT, "store_write out of range");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  const int64_t rb = b->col[column].row_bytes;
  B2R_CUDA(cudaMemcpyAsync(b->col[column].dev + row0 * rb, in,
                           (size_t)(nrows * rb), cudaMemcpyDefault, s));
  if (column == B2R_COL_TERMINAL) B2R_TRY(b2r::refresh_terminal_mirror(b, row0, nrows, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  return B2R_OK;
}


const void *b2r_store_device_ptr(b2r_buffer *b, int32_t column) {
  if (column < 0 || column >= b->num_columns) return nullptr;
  return b->col[column].dev;
}

const double *b2r_total_device_ptr(b2r_buffer *b) {
  return b->tree ? b->tree->heap + 1 : nullptr;  // root of the 1-based heap
}

int b2r_check(b2r_buffer *b, b2r_stream stream) {
  cudaStream_t s = as_stream(stream);
  int64_t st[2];
  B2R_CUDA(cudaMemcpyAsync(st, b->status, 16, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  if (st[0] != 0) {
    B2R_CUDA(cudaMemsetAsync(b->status, 0, 16, s));
    if (st[0] == B2R_ERR_EMPTY_TREE)
      return fail(B2R_ERR_EMPTY_TREE, "Cannot sample from an empty sum tree.");
    if (st[0] == B2R_ERR_STALE_TOTAL)
      return fail(B2R_ERR_STALE_TOTAL,
                  "the sum tree changed between the early publish of this shard's total "
                  "and the next sharded step (b2r_exchange_set_early_publish)");
    if (st[0] == B2R_ERR_EXCHANGE)
      return fail(B2R_ERR_EXCHANGE,
                  "shard %lld did not publish its priority total in time",
                  (long long)st[1]);
    if (st[0] == B2R_ERR_UNSUPPORTED)
      return fail(B2R_ERR_UNSUPPORTED,
                  "a sharded step's share of the global batch (%lld strata) outgrew the "
                  "rows its outputs hold (max_rows)", (long long)st[1]);
    if (st[0] == B2R_ERR_TOO_FEW_TRANSITIONS)
      return fail(B2R_ERR_TOO_FEW_TRANSITIONS,
                  "Cannot sample a batch: no shard holds more than stack size (%d) + "
                  "update_horizon (%d) transitions.",
                  b->cfg.stack_size, b->cfg.update_horizon);
    if (st[0] == B2R_ERR_INDEX_RANGE)
      return fail(B2R_ERR_INDEX_RANGE,
                  "row %lld of the batch holds an action outside [0, num_actions)",
                  (long long)st[1]);
    return fail((int)st[0],
                "Max sample attempts: Tried %d times but only sampled %lld valid "
                "indices.",
                b->cfg.max_sample_attempts, (long long)st[1]);
  }
  if (b->tree) return b2r_tree_check(b->tree, stream);
  return B2R_OK;
}

int b2r_set_priority(b2r_buffer *b, int64_t n, const int32_t *indices,
                     const double *priorities, int64_t *bad_pos,
                     b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (bad_pos) *bad_pos = -1;
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  b2r_tree *t = b->tree;
  B2R_TRY(b->bounce.reserve((size_t)n * 12 + 16));
  memcpy(b->bounce.host, priorities, (size_t)n * 8);
  memcpy(b->bounce.host + (size_t)n * 8, indices, (size_t)n * 4);
  B2R_CUDA(cudaMemcpyAsync(b->bounce.dev, b->bounce.host, (size_t)n * 12,
                           cudaMemcpyHostToDevice, s));
  B2R_TRY((b2r::tree_apply<int32_t, double>(
      t, n, reinterpret_cast<const int32_t *>(b->bounce.dev + (size_t)n * 8),
      reinterpret_cast<const double *>(b->bounce.dev), nullptr, s)));
  // What the device could refuse — a negative value (sum_tree.py:191-193), an index
  // outside the tree — is visible on the host: when there is nothing of the kind the
  // update cannot fail and the call returns without waiting for it.
  bool clean = true;
  for (int64_t k = 0; k < n && clean; ++k)
    clean = priorities[k] >= 0.0 && indices[k] >= 0 && (int64_t)indices[k] < t->leaves;
  if (clean) return b->bounce.mark_busy(s);
  int64_t st[2];
  B2R_CUDA(cudaMemcpyAsync(st, t->status, 16, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  if (st[0] != 0) {
    B2R_CUDA(cudaMemsetAsync(t->status, 0, 16, s));
    if (bad_pos) *bad_pos = st[1];
    if (st[0] == B2R_ERR_NEGATIVE_PRIORITY)
      return fail(B2R_ERR_NEGATIVE_PRIORITY,
                  "Sum tree values should be nonnegative. Got %g",
                  priorities[st[1]]);
    return fail((int)st[0], "index %d is out of range", (int)indices[st[1]]);
  }
  return B2R_OK;
}

int b2r_set_priority_device(b2r_buffer *b, int64_t n, const int32_t *indices,
                            const float *priorities, b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  return b2r_tree_set_device(b->tree, n, indices, priorities, stream);
}

int b2r_set_priority_device_counted(b2r_buffer *b, int64_t max_n,
                                    const int32_t *count, const int32_t *indices,
                                    const float *priorities, b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (max_n <= 0) return B2R_OK;
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  // the count is a fraction of max_n (a shard's part of a global batch)
  return b2r::tree_apply<int32_t, float>(b->tree, max_n, indices, priorities,
                                         nullptr, as_stream(stream), count,
                                         max_n <= 256 ? 0 : -1);
}

int b2r_copy_total_device(b2r_buffer *b, double *dst, b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  B2R_CUDA(cudaMemcpyAsync(dst, b->tree->heap + 1, 8, cudaMemcpyDeviceToDevice,
                           as_stream(stream)));
  return B2R_OK;
}

int b2r_sampler_state_get(b2r_buffer *b, int32_t version, uint64_t *words, int32_t n_words,
                          b2r_stream stream) {
  B2R_TRY(b2r::check_state_words(version, B2R_SAMPLER_STATE_VERSION, n_words,
                                 B2R_SAMPLER_STATE_WORDS, b, words));
  cudaStream_t s = as_stream(stream);
  B2R_CUDA(cudaMemcpyAsync(words, b->draw_counter, 8, cudaMemcpyDefault, s));
  B2R_CUDA(cudaMemcpyAsync(words + 1, b->shard_counter, 8, cudaMemcpyDefault, s));
  return B2R_OK;
}

int b2r_sampler_state_set(b2r_buffer *b, int32_t version, const uint64_t *words,
                          int32_t n_words, b2r_stream stream) {
  B2R_TRY(b2r::check_state_words(version, B2R_SAMPLER_STATE_VERSION, n_words,
                                 B2R_SAMPLER_STATE_WORDS, b, words));
  cudaStream_t s = as_stream(stream);
  B2R_CUDA(cudaMemcpyAsync(b->draw_counter, words, 8, cudaMemcpyDefault, s));
  B2R_CUDA(cudaMemcpyAsync(b->shard_counter, words + 1, 8, cudaMemcpyDefault, s));
  return B2R_OK;
}

}  // extern "C"
