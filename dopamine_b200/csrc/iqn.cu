// IQN's target quantile values and quantile-Huber loss: replaces the TensorFlow ops of
// ImplicitQuantileAgent (dopamine/agents/implicit_quantile/implicit_quantile_agent.py):
//   :176-188  q(s', a) = mean_k Z_action[k*B + b, a]; a* = first argmax
//   :190-231  target[t'] = r + gamma^n (1 - terminal) * Z_target[t'*B + b, a*]
//   :233-315  delta = target[t'] - Z_online[t*B + b, action];  two-case Huber(kappa);
//             |tau_t - 1[delta < 0]| * huber / kappa;  sum over t, mean over t'
// plus d mean_b(loss) / d Z_online for the optimizer (the indicator is behind
// tf.stop_gradient, :304).  All network outputs keep the reference's layout:
// (samples x batch) rows, sample-major, num_actions columns.
//
// One CTA of 4 warps per batch row.  The K action samples are summed by warp (k mod
// 4), the N' targets of the row are built into shared memory by all threads, and warp
// w takes the targets t' = w (mod 4) against the online samples t = lane, lane + 32,
// ... it owns; per-sample partial sums meet in shared memory.  A row costs N * N'
// error terms (4 096 for the paper's 64 x 64) on 3 * 64 gathered values:
// arithmetic-bound, ~20 instructions per term, latency-bound at the agent's batch of
// 32 (hence the split of one row over 4 warps).  Every term is formed in f32 exactly
// as the reference's elementwise ops form it (no FMA contraction); the sums over t and
// t' are accumulated in f64 in a fixed order and rounded once, which is within 1 ulp
// of any f32 summation order the reference's reductions may use.
//
// Sharded mode (b2r_iqn_loss_sharded): the rows are one rank's share of a global batch.
// Only the first min(*count, batch) CTAs compute a row, and the gradient scale and the
// mean divide by the global batch instead of `batch`.  Per row that is the arithmetic of
// the unsharded launch on the whole global batch, so a computed row's loss, next_action
// and gradient rows are the same bits; CTAs past the count write zero gradient rows and
// loss 0.  The mean is this rank's part of the global mean.  An unsharded launch is the
// case count = NULL, global_batch = batch.
#include "common.cuh"

namespace b2r {
namespace {

constexpr int kIqnWarps = 4;
constexpr int kIqnMaxSamples = 256;  // N, N' <= 256

struct IqnArgs {
  b2r_iqn_args u;
  const int32_t *count;  // nullable: rows = min(*count, batch), else batch
  int global_batch;      // divisor of the mean and of its gradient
  unsigned int *ticket;
};

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- mean over the batch (:315): the last CTA to finish sums loss[0, rows) in a fixed
// order and divides by the global batch (every CTA calls; s_red, s_last in shared memory).
__device__ __forceinline__ void iqn_mean(const IqnArgs &a, int rows, double *s_red,
                                         bool *s_last) {
  if (a.u.mean_loss == nullptr || !last_cta(a.ticket, s_last, false)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double acc = 0.0;
  for (int k = threadIdx.x; k < rows; k += blockDim.x) acc += (double)__ldcg(a.u.loss + k);
  acc = warp_sum_f64(acc);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double total = 0.0;
    for (int k = 0; k < kIqnWarps; ++k) total += s_red[k];
    *a.u.mean_loss = (float)(total / (double)a.global_batch);
    *a.ticket = 0u;  // ready for the next launch
  }
}

__global__ void __launch_bounds__(kIqnWarps * 32) iqn_loss_kernel(IqnArgs a) {
  __shared__ float s_target[kIqnMaxSamples];
  __shared__ double s_q[kIqnWarps][32];
  __shared__ double s_acc[kIqnWarps][kIqnMaxSamples];
  __shared__ double s_gacc[kIqnWarps][kIqnMaxSamples];
  __shared__ int s_best;
  __shared__ double s_red[kIqnWarps];
  __shared__ bool s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = a.u.batch, A = a.u.num_actions;
  const int N = a.u.num_tau_samples, NP = a.u.num_tau_prime_samples;
  const int K = a.u.num_quantile_samples;
  pdl_release();
  pdl_acquire();
  const int b = blockIdx.x;
  const int rows = a.count ? min(*a.count, B) : B;
  if (b >= rows) {  // a padded row of a shard: zero gradient rows, loss 0, no next_action
    if (a.u.grad_quantile_values)
      for (int k = threadIdx.x; k < N * A; k += blockDim.x) {
        const int t = k / A;
        a.u.grad_quantile_values[((size_t)t * B + b) * A + (k - t * A)] = 0.f;
      }
    if (threadIdx.x == 0) a.u.loss[b] = 0.f;
    iqn_mean(a, rows, s_red, &s_last);
    return;
  }

  // ---- greedy next action (:176-188): mean over the K samples, first maximum.
  // Warp w sums the samples k = w (mod 4) of 32 actions at a time; warp 0 adds the four
  // partial sums in warp order, divides and keeps the running first maximum.  A lane
  // takes its first action whatever its q, so a row whose means are all -inf or NaN
  // still yields an action in [0, A) (all -inf: action 0, as argmax gives) and never
  // gathers the target at the sentinel's column.
  constexpr int kNoAction = 0x7fffffff;
  float best_q = -INFINITY;
  int best_a = kNoAction;
  for (int base = 0; base < A; base += 32) {
    const int act = base + lane;
    double sum = 0.0;
    if (act < A)
      for (int k = warp; k < K; k += kIqnWarps)
        sum += (double)a.u.action_quantile_values[((size_t)k * B + b) * A + act];
    s_q[warp][lane] = sum;
    __syncthreads();
    if (warp == 0 && act < A) {
      double total = s_q[0][lane];
#pragma unroll
      for (int w = 1; w < kIqnWarps; ++w) total += s_q[w][lane];
      const float q = __fdiv_rn((float)total, (float)K);
      // ascending act: strict > keeps the first maximum
      if (best_a == kNoAction || q > best_q) {
        best_q = q;
        best_a = act;
      }
    }
    __syncthreads();
  }
  if (warp == 0) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float q2 = __shfl_xor_sync(0xffffffffu, best_q, o);
      const int a2 = __shfl_xor_sync(0xffffffffu, best_a, o);
      // & and | rather than && and ||: one predicate, no branch in each step
      if ((a2 != kNoAction) &
          ((best_a == kNoAction) | (q2 > best_q) | ((q2 == best_q) & (a2 < best_a)))) {
        best_q = q2;
        best_a = a2;
      }
    }
    if (lane == 0) {
      s_best = best_a;
      if (a.u.next_action) a.u.next_action[b] = best_a;
    }
  }
  __syncthreads();
  best_a = s_best;

  // ---- target quantile values (:196-231)
  const float r = a.u.rewards[b];
  const float live = __fsub_rn(1.0f, (float)a.u.terminals[b]);
  const float gwt = __fmul_rn(a.u.cumulative_gamma, live);
  for (int tp = threadIdx.x; tp < NP; tp += blockDim.x) {
    const float z = a.u.target_quantile_values[((size_t)tp * B + b) * A + best_a];
    s_target[tp] = __fadd_rn(r, __fmul_rn(gwt, z));
  }
  __syncthreads();

  // ---- quantile Huber loss (:278-311) and its gradient
  const int action = a.u.actions[b];
  const float kappa = a.u.kappa;
  const bool unit_kappa = kappa == 1.0f;  // x / 1 is x: the default needs no division
  const float half_kappa = __fmul_rn(0.5f, kappa);
  for (int t = lane; t < N; t += 32) {
    const size_t row = (size_t)t * B + b;
    const float chosen = a.u.online_quantile_values[row * A + action];
    const float tau = a.u.quantiles[row];
    double acc = 0.0, gacc = 0.0;
#pragma unroll 4
    for (int tp = warp; tp < NP; tp += kIqnWarps) {
      const float err = __fsub_rn(s_target[tp], chosen);
      const float abs_err = fabsf(err);
      const bool small = abs_err <= kappa;
      // to_float(|e| <= k) * 0.5 * e^2  +  to_float(|e| > k) * k * (|e| - 0.5 k)
      const float huber = small ? __fmul_rn(0.5f, __fmul_rn(err, err))
                                : __fmul_rn(kappa, __fsub_rn(abs_err, half_kappa));
      const float weight = fabsf(__fsub_rn(tau, err < 0.f ? 1.0f : 0.0f));
      const float wh = __fmul_rn(weight, huber);
      acc += (double)(unit_kappa ? wh : __fdiv_rn(wh, kappa));
      const float dh = small ? err : copysignf(kappa, err);
      gacc += (double)__fmul_rn(weight, dh);
    }
    s_acc[warp][t] = acc;
    s_gacc[warp][t] = gacc;
  }
  __syncthreads();
  if (warp == 0) {
    const double grad_scale = -1.0 / ((double)kappa * (double)NP * (double)a.global_batch);
    double row_sum = 0.0;
    for (int t = lane; t < N; t += 32) {
      double acc = s_acc[0][t], gacc = s_gacc[0][t];
#pragma unroll
      for (int w = 1; w < kIqnWarps; ++w) {
        acc += s_acc[w][t];
        gacc += s_gacc[w][t];
      }
      row_sum += acc;
      if (a.u.grad_quantile_values) {
        float *g = a.u.grad_quantile_values + ((size_t)t * B + b) * A;
        const float gv = (float)(gacc * grad_scale);
        for (int act = 0; act < A; ++act) g[act] = act == action ? gv : 0.f;
      }
    }
    row_sum = warp_sum_f64(row_sum);
    if (lane == 0) a.u.loss[b] = (float)(row_sum / (double)NP);
  }

  iqn_mean(a, rows, s_red, &s_last);
}

unsigned int *g_iqn_ticket = nullptr;

// The checks and the launch of both entry points; count = NULL: unsharded.
int iqn_launch(const b2r_iqn_args *args, const int32_t *count, int global_batch,
               cudaStream_t stream) {
  if (!args || args->batch <= 0 || args->num_actions <= 0 || args->num_tau_samples <= 0 ||
      args->num_tau_prime_samples <= 0 || args->num_quantile_samples <= 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad IQN shape");
  if (args->num_tau_samples > kIqnMaxSamples || args->num_tau_prime_samples > kIqnMaxSamples)
    return fail(B2R_ERR_UNSUPPORTED, "more than 256 tau samples are not supported");
  if (!(args->kappa > 0.f))
    return fail(B2R_ERR_INVALID_ARGUMENT, "kappa must be positive");
  if (!args->action_quantile_values || !args->target_quantile_values ||
      !args->online_quantile_values || !args->quantiles || !args->actions ||
      !args->rewards || !args->terminals || !args->loss)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a required IQN pointer is NULL");
  if (!g_iqn_ticket) {
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&g_iqn_ticket), 4));
    B2R_CUDA(cudaMemset(g_iqn_ticket, 0, 4));
  }
  IqnArgs a;
  a.u = *args;
  a.count = count;
  a.global_batch = global_batch;
  a.ticket = g_iqn_ticket;
  B2R_CUDA(launch(iqn_loss_kernel, dim3(args->batch), dim3(kIqnWarps * 32), 0, stream, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // namespace
}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" int b2r_iqn_loss(const b2r_iqn_args *args, b2r_stream stream) {
  return b2r::iqn_launch(args, nullptr, args ? args->batch : 0, as_stream(stream));
}

extern "C" int b2r_iqn_loss_sharded(const b2r_iqn_args *args, const int32_t *count,
                                    int32_t global_batch, b2r_stream stream) {
  if (!args) return fail(B2R_ERR_INVALID_ARGUMENT, "args is NULL");
  if (!count) return fail(B2R_ERR_INVALID_ARGUMENT, "a shard's loss needs count");
  if (global_batch < 1) return fail(B2R_ERR_INVALID_ARGUMENT, "global_batch must be >= 1");
  return b2r::iqn_launch(args, count, global_batch, as_stream(stream));
}
