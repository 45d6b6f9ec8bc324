// Shard-total exchange over peer memory: set-up of the mailboxes that the sharded
// sampling kernel (sample.cu: exchange_publish / exchange_collect) writes and polls.
// SURVEY.md section 8e: the only cross-GPU step of the path is an all-gather of one
// fp64 per rank; here every rank stores its total straight into its peers' HBM over
// NVLink from inside the kernel that needs the totals, instead of calling a
// collective library between two launches.
#include "replay.cuh"

#include <new>

using b2r::fail;

namespace {
// totals [2][kMaxShards][2 words], then local minima [2][kMaxShards], then the uniform
// sampler's rejection lists [2][kMaxShards][1 + kRejListWords] (tree.cuh)
constexpr size_t kMailboxBytes = b2r::kMailboxWords * sizeof(uint64_t);
}

namespace {
// The kernel arguments as the tree kernels' publish hook reads them (device memory).
int upload_args(b2r_exchange *x) {
  b2r::ExchangeArgs a;
  b2r::fill_exchange_args(x, &a);
  B2R_CUDA(cudaMemcpy(x->args_dev, &a, sizeof(a), cudaMemcpyHostToDevice));
  return B2R_OK;
}
}  // namespace

extern "C" {

int b2r_exchange_create(int32_t world, int32_t rank, b2r_exchange **out) {
  if (!out) return fail(B2R_ERR_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  if (world < 1 || world > b2r::kMaxShards || rank < 0 || rank >= world)
    return fail(B2R_ERR_INVALID_ARGUMENT, "world must be in [1, %d], rank in [0, world)",
                b2r::kMaxShards);
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count == 0)
    return fail(B2R_ERR_CUDA, "no CUDA device: libb200replay has no CPU fallback");
  b2r_exchange *x = new (std::nothrow) b2r_exchange();
  if (!x) return fail(B2R_ERR_INVALID_ARGUMENT, "out of host memory");
  x->world = world;
  x->rank = rank;
  // cudaMalloc memory can be exported with cudaIpcGetMemHandle.
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&x->mailbox), kMailboxBytes));
  B2R_CUDA(cudaMemset(x->mailbox, 0, kMailboxBytes));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&x->seq), 8));
  B2R_CUDA(cudaMemset(x->seq, 0, 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&x->pub), 16));
  B2R_CUDA(cudaMemset(x->pub, 0, 16));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&x->args_dev), sizeof(b2r::ExchangeArgs)));
  B2R_CUDA(cudaDeviceSynchronize());
  x->connected = world == 1;
  *out = x;
  return world == 1 ? upload_args(x) : B2R_OK;
}

int b2r_exchange_destroy(b2r_exchange *x) {
  if (!x) return B2R_OK;
  cudaDeviceSynchronize();
  for (int g = 0; g < b2r::kMaxShards; ++g)
    if (x->opened[g] && x->peer[g]) cudaIpcCloseMemHandle(x->peer[g]);
  cudaFree(x->mailbox);
  cudaFree(x->seq);
  cudaFree(x->pub);
  cudaFree(x->args_dev);
  delete x;
  return B2R_OK;
}

int b2r_exchange_local_handle(b2r_exchange *x, void *handle_out) {
  if (!x || !handle_out) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == B2R_IPC_HANDLE_BYTES,
                "IPC handle size");
  cudaIpcMemHandle_t h;
  B2R_CUDA(cudaIpcGetMemHandle(&h, x->mailbox));
  memcpy(handle_out, &h, sizeof(h));
  return B2R_OK;
}

int b2r_exchange_connect(b2r_exchange *x, const void *handles) {
  if (!x || !handles) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  const uint8_t *bytes = static_cast<const uint8_t *>(handles);
  for (int g = 0; g < x->world; ++g) {
    if (g == x->rank) {
      x->peer[g] = x->mailbox;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, bytes + (size_t)g * B2R_IPC_HANDLE_BYTES, sizeof(h));
    void *p = nullptr;
    B2R_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    x->peer[g] = static_cast<uint64_t *>(p);
    x->opened[g] = true;
  }
  x->connected = true;
  return upload_args(x);
}

int b2r_exchange_connect_pointers(b2r_exchange *x, void *const *mailboxes) {
  if (!x || !mailboxes) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  for (int g = 0; g < x->world; ++g)
    x->peer[g] = g == x->rank ? x->mailbox : static_cast<uint64_t *>(mailboxes[g]);
  x->connected = true;
  return upload_args(x);
}

void *b2r_exchange_mailbox(b2r_exchange *x) { return x ? x->mailbox : nullptr; }

int b2r_exchange_set_timeout(b2r_exchange *x, double seconds) {
  if (!x || !(seconds > 0.0))
    return fail(B2R_ERR_INVALID_ARGUMENT, "timeout must be positive");
  x->timeout_ns = (int64_t)(seconds * 1e9);
  return x->connected ? upload_args(x) : B2R_OK;
}

int b2r_exchange_set_early_publish(b2r_exchange *x, int32_t on) {
  if (!x) return fail(B2R_ERR_INVALID_ARGUMENT, "NULL argument");
  x->early_publish = on != 0;
  return B2R_OK;
}

int b2r_exchange_state_get(b2r_exchange *x, int32_t version, uint64_t *words,
                           int32_t n_words, b2r_stream stream) {
  B2R_TRY(b2r::check_state_words(version, B2R_EXCHANGE_STATE_VERSION, n_words,
                                 B2R_EXCHANGE_STATE_WORDS, x, words));
  B2R_CUDA(cudaMemcpyAsync(words, x->seq, 8, cudaMemcpyDefault, b2r::as_stream(stream)));
  return B2R_OK;
}

int b2r_exchange_state_set(b2r_exchange *x, int32_t version, const uint64_t *words,
                           int32_t n_words, b2r_stream stream) {
  B2R_TRY(b2r::check_state_words(version, B2R_EXCHANGE_STATE_VERSION, n_words,
                                 B2R_EXCHANGE_STATE_WORDS, x, words));
  cudaStream_t s = b2r::as_stream(stream);
  B2R_CUDA(cudaMemcpyAsync(x->seq, words, 8, cudaMemcpyDefault, s));
  // every tag in the mailbox becomes 0, and pub[0] = 0 "nothing published": the steps
  // after any restored step number are >= 1
  B2R_CUDA(cudaMemsetAsync(x->mailbox, 0, kMailboxBytes, s));
  B2R_CUDA(cudaMemsetAsync(x->pub, 0, 16, s));
  return B2R_OK;
}

int b2r_exchange_publish_device(b2r_exchange *x, b2r_buffer *buf, b2r_stream stream) {
  if (!x || !buf || !buf->tree) return fail(B2R_ERR_INVALID_ARGUMENT, "bad argument");
  if (!x->connected) return fail(B2R_ERR_INVALID_ARGUMENT, "the exchange is not connected");
  B2R_TRY(b2r::flush_queue(buf, b2r::as_stream(stream)));
  return b2r::launch_exchange_publish(x, buf, b2r::as_stream(stream));
}

int b2r_exchange_publish_uniform_device(b2r_exchange *x, b2r_buffer *buf,
                                        int32_t global_batch, uint64_t seed,
                                        uint64_t offset, int32_t phase, b2r_stream stream) {
  B2R_TRY(b2r::check_uniform_sharded(buf, x, global_batch));
  if (phase != 0 && phase != 1) return fail(B2R_ERR_INVALID_ARGUMENT, "phase must be 0 or 1");
  return b2r::launch_uniform_sharded(buf, x, global_batch, seed, offset, phase, nullptr,
                                     nullptr, nullptr, 0, b2r::as_stream(stream));
}

}  // extern "C"
