// DQN's Bellman target and Huber loss: replaces the TF ops of
// dopamine/agents/dqn/dqn_agent.py:283-322 (_build_target_q_op, _build_train_op):
//   target_b = r_b + gamma^n * max_a Q_target(s'_b, a) * (1 - terminal_b)
//   loss_b   = huber(target_b, Q_online(s_b, a_b)),  delta = 1  (tf.losses.huber_loss:
//              e = prediction - label; q = min(|e|, 1); loss = 0.5 q^2 + (|e| - q))
// plus d mean(loss) / d Q_online for the optimizer.  One thread per row (a row is
// num_actions floats per network: 72 B for Atari); f32 with explicit round-to-nearest
// intrinsics where TF evaluates separate ops (no FMA contraction).
//
// Sharded mode (b2r_dqn_loss_sharded): the rows are one rank's share of a global batch.
// The gradient divides by the global batch instead of the row count, so a computed row's
// loss, target and gradient row are the bits b2r_dqn_loss gives that row on the whole
// global batch; rows past the count get loss 0 and zero gradient rows.  The mean is this
// rank's part of the global mean: its rows' losses summed in f64, divided by the global
// batch, rounded once.
#include "common.cuh"

namespace b2r {
namespace {

struct DqnArgs {
  b2r_dqn_args u;
  float *row_loss;   // scratch when u.loss is NULL but the mean is wanted
  int global_batch;  // > 0: sharded mode, the divisor of the gradient
};

__global__ void __launch_bounds__(256) dqn_loss_kernel(DqnArgs a) {
  pdl_release();
  pdl_acquire();
  const int rows = a.u.batch_count ? min(*a.u.batch_count, a.u.batch) : a.u.batch;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int A = a.u.num_actions;
  if (b >= rows) {
    if (a.global_batch > 0 && b < a.u.batch) {  // a padded row of a shard
      if (a.u.loss) a.u.loss[b] = 0.f;
      if (a.row_loss) a.row_loss[b] = 0.f;
      if (a.u.grad_q)
        for (int k = 0; k < A; ++k) a.u.grad_q[(size_t)b * A + k] = 0.f;
    }
    return;
  }
  const float *qt = a.u.target_q + (size_t)b * A;
  const float *qo = a.u.online_q + (size_t)b * A;
  const int action = a.u.actions[b];
  float best = qt[0];  // tf.reduce_max over the action axis
  for (int k = 1; k < A; ++k) best = fmaxf(best, qt[k]);
  const float live = __fsub_rn(1.0f, (float)a.u.terminals[b]);
  const float target =
      __fadd_rn(a.u.rewards[b], __fmul_rn(__fmul_rn(a.u.cumulative_gamma, best), live));
  const float chosen = qo[action];  // sum(q * one_hot(action))
  const float err = __fsub_rn(chosen, target);
  const float abs_err = fabsf(err);
  const float quad = fminf(abs_err, 1.0f);
  const float lin = __fsub_rn(abs_err, quad);
  const float loss = __fadd_rn(__fmul_rn(0.5f, __fmul_rn(quad, quad)), lin);
  if (a.u.loss) a.u.loss[b] = loss;
  if (a.row_loss) a.row_loss[b] = loss;
  if (a.u.target) a.u.target[b] = target;
  if (a.u.grad_q) {
    // d mean(loss) / d q[b, k]: clip(e, -1, 1) / rows (sharded: / global batch) on the
    // chosen action
    const float g = __fdiv_rn(fminf(fmaxf(err, -1.0f), 1.0f),
                              (float)(a.global_batch > 0 ? a.global_batch : rows));
    for (int k = 0; k < A; ++k) a.u.grad_q[(size_t)b * A + k] = k == action ? g : 0.f;
  }
}

// Fixed-order mean (one CTA): the same bits on every run.
__global__ void __launch_bounds__(1024) dqn_mean_kernel(const float *row_loss, int batch,
                                                        const int32_t *count,
                                                        float *mean_out) {
  __shared__ float partial[1024];
  pdl_release();
  pdl_acquire();
  const int rows = count ? min(*count, batch) : batch;
  float acc = 0.f;
  for (int k = threadIdx.x; k < rows; k += blockDim.x) acc = __fadd_rn(acc, row_loss[k]);
  partial[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s)
      partial[threadIdx.x] = __fadd_rn(partial[threadIdx.x], partial[threadIdx.x + s]);
    __syncthreads();
  }
  if (threadIdx.x == 0) *mean_out = rows > 0 ? __fdiv_rn(partial[0], (float)rows) : 0.f;
}

// Sharded mean (one CTA): f64 sum of this rank's rows in a fixed order, over the global
// batch, rounded once.
__global__ void __launch_bounds__(256) dqn_mean_sharded_kernel(const float *row_loss,
                                                               int batch, const int32_t *count,
                                                               int global_batch,
                                                               float *mean_out) {
  __shared__ double partial[256];
  pdl_release();
  pdl_acquire();
  const int rows = min(max(*count, 0), batch);
  double acc = 0.0;
  for (int k = threadIdx.x; k < rows; k += blockDim.x) acc += (double)row_loss[k];
  partial[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) partial[threadIdx.x] += partial[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) *mean_out = (float)(partial[0] / (double)global_batch);
}

float *g_row_loss = nullptr;
int g_row_loss_cap = 0;

// The checks and the launches of both entry points; global_batch 0: unsharded.
int dqn_launch(const b2r_dqn_args *args, int global_batch, cudaStream_t s) {
  if (!args || args->batch <= 0 || args->num_actions <= 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad DQN shape");
  if (!args->target_q || !args->online_q || !args->actions || !args->rewards ||
      !args->terminals)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a required DQN pointer is NULL");
  DqnArgs a;
  a.u = *args;
  a.row_loss = nullptr;
  a.global_batch = global_batch;
  if (args->mean_loss && !args->loss) {
    if (args->batch > g_row_loss_cap) {
      if (g_row_loss) cudaFree(g_row_loss);
      g_row_loss = nullptr;
      int cap = 4096;
      while (cap < args->batch) cap *= 2;
      B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&g_row_loss), (size_t)cap * 4));
      g_row_loss_cap = cap;
    }
    a.row_loss = g_row_loss;
  }
  B2R_CUDA(launch(dqn_loss_kernel, dim3((args->batch + 255) / 256), dim3(256), 0, s, a));
  B2R_LAUNCHED();
  if (args->mean_loss) {
    const float *rows = args->loss ? args->loss : a.row_loss;
    if (global_batch > 0)
      B2R_CUDA(launch(dqn_mean_sharded_kernel, dim3(1), dim3(256), 0, s, rows, args->batch,
                      args->batch_count, global_batch, args->mean_loss));
    else
      B2R_CUDA(launch(dqn_mean_kernel, dim3(1), dim3(1024), 0, s, rows, args->batch,
                      args->batch_count, args->mean_loss));
    B2R_LAUNCHED();
  }
  return B2R_OK;
}

}  // namespace
}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" int b2r_dqn_loss(const b2r_dqn_args *args, b2r_stream stream) {
  return b2r::dqn_launch(args, 0, as_stream(stream));
}

extern "C" int b2r_dqn_loss_sharded(const b2r_dqn_args *args, int32_t global_batch,
                                    b2r_stream stream) {
  if (!args) return fail(B2R_ERR_INVALID_ARGUMENT, "args is NULL");
  if (!args->batch_count)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a shard's loss needs args->batch_count");
  if (global_batch < 1) return fail(B2R_ERR_INVALID_ARGUMENT, "global_batch must be >= 1");
  return b2r::dqn_launch(args, global_batch, as_stream(stream));
}
