// C51 distributional Bellman target, projection, cross-entropy, priorities and IS
// weights: replaces the TensorFlow graph built by RainbowAgent
// (rainbow_agent.py:200-305) and project_distribution (rainbow_agent.py:340-494).
//
// Two kernels share the arithmetic.  Batches below 128 rows (latency-bound): one CTA per
// row, one warp per action (c51_loss_kernel).  From 128 rows (bound by instruction
// issue): one WARP per row, 8 lanes per action (c51_loss_rows_kernel) — a third of the
// instructions per row.  In both, atoms are strided over lanes, reductions are warp
// shuffles, the (Bellman support, probability) pairs of a row sit in shared memory so
// that each output atom is accumulated over all j exactly as the dense [B, N, N] form
// does — without ever materialising it.  All arithmetic is f32 with explicit
// round-to-nearest intrinsics where TF evaluates separate ops (no FMA contraction),
// true division and IEEE sqrt.
//
// Traffic per row (A=18, N=51): 3 672 B of target logits + 204 B of online logits
// read, <= 204 B target + 12 B scalars written (+3 672 B if grad_logits is asked).
#include "replay.cuh"

#include <cooperative_groups.h>

#include <cstdlib>

namespace b2r {
namespace {

B2R_TRACE_DECL

constexpr int kWarpsPerBlock = 4;

// UNROLLED = false keeps the reductions as 5-trip loops (compact code for the
// latency-bound small-batch instance); true unrolls them: the large-batch instance
// is bound by instruction issue and the loop control is 2/3 of a rolled reduction.
template <bool UNROLLED = false>
__device__ __forceinline__ float warp_max(float v) {
  if (UNROLLED) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  } else {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  }
  return v;
}
template <bool UNROLLED = false>
__device__ __forceinline__ float warp_sum(float v) {
  if (UNROLLED) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  } else {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  }
  return v;
}

// The first output atom whose projection interval is open above.  Bellman atoms at or
// above zlast clip to it, and reach atom i wherever zlast - z_i < dz: the last atom, and
// also atom N - 2 on the f32 supports whose last spacing rounds below dz = z[1] - z[0]
// (vmax 10 at 64 or 101 atoms, not at 51).  Their hat there is a few millionths, but
// the dense form adds it.
__device__ __forceinline__ int clipped_reach_below_last(float zprev, float zlast, float dz,
                                                        int n) {
  return __fsub_rn(zlast, zprev) < dz ? n - 2 : n - 1;
}

// out[i] = sum_j clip(1 - |clip(s_j, z0, zlast) - z_i| / dz, 0, 1) * w_j
// (rainbow_agent.py:424-492); s, w in shared memory, i strided over lanes.
__device__ __forceinline__ float project_atom(const float *s, const float *w,
                                              int n, float z_i, float z0,
                                              float zlast, float dz) {
  float acc = 0.f;
  for (int j = 0; j < n; ++j) {
    const float clipped = fminf(fmaxf(s[j], z0), zlast);
    const float gap = fabsf(__fsub_rn(clipped, z_i));
    float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
    hat = fminf(fmaxf(hat, 0.f), 1.f);
    acc = __fadd_rn(acc, __fmul_rn(hat, w[j]));
  }
  return acc;
}

__global__ void __launch_bounds__(kWarpsPerBlock * 32)
c51_project_kernel(int batch, int n, const float *__restrict__ supports,
                   const float *__restrict__ weights,
                   const float *__restrict__ z, float *__restrict__ out) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kWarpsPerBlock + warp;
  if (b >= batch) return;
  float *s = smem + (size_t)warp * 2 * n;
  float *w = s + n;
  for (int j = lane; j < n; j += 32) {
    s[j] = supports[(size_t)b * n + j];
    w[j] = weights[(size_t)b * n + j];
  }
  __syncwarp();
  const float z0 = z[0], zlast = z[n - 1];
  const float dz = __fsub_rn(z[1], z[0]);  // rainbow_agent.py:381-383
  for (int i = lane; i < n; i += 32)
    out[(size_t)b * n + i] = project_atom(s, w, n, z[i], z0, zlast, dz);
}

// b2r_c51_loss_sharded: this rank's rows of a global batch of global_batch strata.  The
// IS normaliser is the minimum over the G ranks' local minima (the rank's own one is
// args->min_probability, the peers' are polled from the local mailbox for the step the
// sampler has just closed), the mean and its gradient use global_batch as the divisor and
// rows >= count get zero gradients: summed over the ranks, the means and the gradients
// are those of the whole global batch.
struct ShardedLoss {
  int global_batch = 0;        // 0: not sharded
  int world = 1, rank = 0;
  const uint64_t *mins = nullptr;  // this rank's mailbox, local-minimum region
  const uint64_t *seq = nullptr;   // device step counter (advanced by the sampler)
  int64_t timeout_ns = 0;
  int64_t *latched = nullptr;      // nullable: B2R_ERR_EXCHANGE on a peer's timeout
};

struct LossArgs {
  b2r_c51_args u;
  ShardedLoss sh;
  float *weighted;        // scratch (B,): w_b * loss_b, reduced by the last CTA
  unsigned int *ticket;   // scratch: CTAs finished (self-resetting)
  int warps;              // warps per CTA = min(num_actions, 32)
  // c51_post_tree_kernel: the priority write-back that the cluster applies behind the
  // tail (batches of at most 32 rows: the fused step at the agent's batch size)
  UpdateArgs<int32_t, float> tree;
  int64_t *err;  // nullable: asynchronous error latch (an action outside [0, A))
  int32_t *count_copy;  // nullable: receives the row count (c51_post_kernel)
  // c51_post_tree_kernel with a device-side row count (a shard's step): set to 1 when the
  // kernel has applied the write-back itself (at most 32 rows), so that the one-CTA tree
  // kernel launched behind it returns at once; left alone otherwise.
  unsigned int *tree_done;
  // nullable: a second copy of the per-row losses (and of the row count behind them, at
  // [batch]) in the caller's page-locked memory: the host-facing trainer's result slot,
  // written by the kernel instead of copied by a call.
  float *loss_host;
  // The write-back behind this kernel is resident already and waits to hear that the
  // sampled indices are final (tree.cuh: TreeGo); go.go == nullptr: nobody does.
  TreeGo go;
  // c51_post_tree_kernel<true>: where the first half left the log-probabilities, and the
  // word that says it has (replay.cuh)
  StageGate stage;
};

// Minimum of `own` and the peers' local minima of the current step (see ShardedLoss).  A
// peer's word carries the step number in-band: a stale or early word is waited on, never
// read as a value.  A peer that does not publish within the timeout latches
// B2R_ERR_EXCHANGE (later launches then skip the wait) and is left out.
__device__ __noinline__ float sharded_min_probability(const ShardedLoss &x, float own) {
  const uint64_t seq = *x.seq;
  const uint64_t *box = x.mins + (size_t)(seq & 1) * x.world;
  float m = own;
  for (int g = 0; g < x.world; ++g) {
    if (g == x.rank || x.timeout_ns <= 0 ||
        (x.latched != nullptr && x.latched[0] == B2R_ERR_EXCHANGE))
      continue;
    uint64_t w;
    if (poll_tagged_word(box + g, seq, x.timeout_ns, &w)) {
      m = fminf(m, __uint_as_float((uint32_t)(w >> 32)));
    } else if (x.latched != nullptr) {
      x.latched[0] = B2R_ERR_EXCHANGE;
      x.latched[1] = g;
    }
  }
  return m;
}

// By the last CTA: sum of weighted[0, n) in a fixed order (thread t takes k = t mod
// blockDim, butterfly per warp, warps in order) / divisor into *out.
__device__ __forceinline__ void mean_of_weighted(const float *weighted, int n, float divisor,
                                                 float *s_red, float *out) {
  float acc = 0.f;
  for (int k = threadIdx.x; k < n; k += blockDim.x) acc = __fadd_rn(acc, __ldcg(weighted + k));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, o));
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float total = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) total = __fadd_rn(total, s_red[w]);
    *out = __fdiv_rn(total, divisor);
  }
}

// A sharded launch's rows past the count: zero gradient rows, and the CTA still takes its
// ticket so that the last CTA forms this rank's part of the mean.
__device__ void sharded_padding(const LossArgs &a, int b0, int nrows, int rows, float *s_red,
                                bool *s_last) {
  const int AN = a.u.num_actions * a.u.num_atoms;
  if (a.u.grad_logits != nullptr)
    for (int r = 0; r < nrows; ++r) {
      const int b = b0 + r;
      if (b < rows || b >= a.u.batch) continue;
      float *g = a.u.grad_logits + (size_t)b * AN;
      for (int k = threadIdx.x; k < AN; k += blockDim.x) g[k] = 0.f;
    }
  if (a.u.mean_weighted_loss == nullptr) return;
  if (!last_cta(a.ticket, s_last)) return;
  mean_of_weighted(a.weighted, rows, (float)a.sh.global_batch, s_red, a.u.mean_weighted_loss);
}

// One CTA per batch row, one warp per action (rainbow_agent.py:200-293):
//   A. every warp: softmax of its action's target logits, q = sum z*p
//      (atari_lib.py:141-143); meanwhile the CTA finds min(sampling_probabilities)
//      for the IS-weight normalisation.
//   B. first argmax over actions (RA:238-248); Bellman support r + g^n(1-t) z
//      (RA:229-235); projection, `parts` threads per output atom (RA:381-494).
//   C. warp 0: cross-entropy vs the chosen online logits (RA:262-271), priority
//      sqrt(loss + 1e-10) (RA:290), weight 1/sqrt(p + 1e-10) / max (RA:279-280).
//   D. all threads: gradient row; the last CTA to finish sums w*loss in a fixed
//      order for mean_weighted_loss (RA:293, 305).
constexpr int kMaxAtomsPerLane = 4;  // num_atoms <= 128

// PL = atoms per lane (2 covers C51's 51 atoms; fewer unrolled copies = less
// straight-line code to fetch on a cold instruction cache).
template <int PL>
__global__ void __launch_bounds__(1024, 1) c51_loss_kernel(LossArgs a) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x;
  const int N = a.u.num_atoms, A = a.u.num_actions, W = a.warps;
  float *bestp = smem + (size_t)warp * N;        // [W][N] best action's probs
  float *sup = smem + (size_t)W * N;             // [N] Bellman support
  float *tgt = sup + N;                          // [N] projected target
  float *onl = tgt + N;                          // [N] chosen online logits
  float *zs = onl + N;                           // [N] the support, staged
  float *lgp = zs + N;                           // [N] log_softmax of the chosen logits
  __shared__ float s_q[32];
  __shared__ int s_a[32];
  __shared__ float s_red[32];
  __shared__ float s_scalar[4];  // tsum, w_b, m, denom
  __shared__ float s_ce;
  __shared__ bool s_last;
  const float *z = a.u.support;
  B2R_MARK(0);
  pdl_release();
  pdl_acquire();
  // (the sampler has ended: the write-back behind this kernel may read its indices)
  if (blockIdx.x == 0 && threadIdx.x == 0) tree_go_signal(a.go);
  B2R_MARK(1);
  const int rows = a.u.batch_count ? min(*a.u.batch_count, a.u.batch) : a.u.batch;
  const bool sharded = a.sh.global_batch > 0;
  if (b >= rows) {  // (mean_weighted_loss with batch_count: sharded only)
    if (sharded) sharded_padding(a, b, 1, rows, s_red, &s_last);
    return;
  }

  // ---- every global load the row needs is issued here, before the first use:
  // the kernel is latency-bound at batch 32 and this keeps it to one round trip.
  // an action outside [0, A) (tf.gather_nd raises): the row is evaluated for action 0,
  // reports a zero loss and latches B2R_ERR_INDEX_RANGE where the caller gave a latch
  const int chosen_raw = a.u.actions[b];
  const bool bad_action = chosen_raw < 0 || chosen_raw >= A;
  const int chosen = bad_action ? 0 : chosen_raw;
  const float r = a.u.rewards[b];
  const float term = (float)a.u.terminals[b];
  const float my_prob = a.u.sampling_probabilities ? a.u.sampling_probabilities[b] : 1.f;
  // min over the batch of the sampling probabilities (IS-weight normaliser):
  // handed in by the sampler when it produced the batch, else reduced here.
  float pmin = INFINITY;
  if (a.u.min_probability)
    pmin = *a.u.min_probability;
  else if (a.u.sampling_probabilities)
    for (int k = threadIdx.x; k < rows; k += blockDim.x)
      pmin = fminf(pmin, a.u.sampling_probabilities[k]);
  float zl[PL], xt[PL], xo[PL];
  const int act0 = warp;  // first (usually only) action of this warp
  const float *__restrict__ trow = a.u.target_logits + (size_t)b * A * N;
  const float *__restrict__ orow = a.u.online_logits + (size_t)b * A * N;
#pragma unroll
  for (int t = 0; t < PL; ++t) {
    const int i = lane + 32 * t;
    const bool ok = i < N && act0 < A;
    zl[t] = i < N ? z[i] : 0.f;
    xt[t] = ok ? trow[act0 * N + i] : -INFINITY;
    xo[t] = ok ? orow[act0 * N + i] : 0.f;
  }

  B2R_MARK(2);
  // ---- A. per-action softmax + q-value (atari_lib.py:141-143)
  float best_q = 0.f;
  int best_a = -1;
  for (int act = warp; act < A; act += W) {
    if (act != act0) {  // more actions than warps: later rounds load as they go
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        const int i = lane + 32 * t;
        xt[t] = i < N ? trow[act * N + i] : -INFINITY;
        // only the chosen action's online logits are ever used
        xo[t] = (i < N && act == chosen) ? orow[act * N + i] : 0.f;
      }
    }
    if (act == chosen) {
      // log_softmax of the chosen action's online logits (rainbow_agent.py:262-271),
      // by the warp that holds them, while the other warps do their softmaxes
      float mo = -INFINITY;
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (lane + 32 * t < N) mo = fmaxf(mo, xo[t]);
      mo = warp_max(mo);
      float ps = 0.f;
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (lane + 32 * t < N) ps = __fadd_rn(ps, expf(__fsub_rn(xo[t], mo)));
      const float den_o = warp_sum(ps);
      const float lse = logf(den_o);
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        if (lane + 32 * t < N) {
          onl[lane + 32 * t] = xo[t];
          lgp[lane + 32 * t] = __fsub_rn(__fsub_rn(xo[t], mo), lse);
        }
      }
      if (lane == 0) {
        s_scalar[2] = mo;
        s_scalar[3] = den_o;
      }
    }
    float m = -INFINITY;
#pragma unroll
    for (int t = 0; t < PL; ++t) m = fmaxf(m, xt[t]);
    m = warp_max(m);
    float e[PL];
    float psum = 0.f;
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      const bool ok = lane + 32 * t < N;
      e[t] = ok ? expf(__fsub_rn(xt[t], m)) : 0.f;
      if (ok) psum = __fadd_rn(psum, e[t]);
    }
    const float denom = warp_sum(psum);
    float qpart = 0.f;
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      if (lane + 32 * t < N) {
        e[t] = __fdiv_rn(e[t], denom);
        qpart = __fadd_rn(qpart, __fmul_rn(zl[t], e[t]));
      }
    }
    const float q = warp_sum(qpart);
    if (best_a < 0 || q > best_q) {  // strict > keeps the first maximum
      best_q = q;
      best_a = act;
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (lane + 32 * t < N) bestp[lane + 32 * t] = e[t];
    }
  }
  B2R_MARK(3);
  if (lane == 0) {
    s_q[warp] = best_q;
    s_a[warp] = best_a;
  }
  // min over the batch of the sampling probabilities: 1/sqrt(p + 1e-10) is
  // monotone under round-to-nearest, so max_b w_b == w(min_b p_b) exactly.
  if (a.u.sampling_probabilities) {
    pmin = -warp_max(-pmin);
    if (lane == 0) s_red[warp] = pmin;
  }
  // Bellman support (rainbow_agent.py:229-235)
  const float live = __fsub_rn(1.0f, term);
  const float gwt = __fmul_rn(a.u.cumulative_gamma, live);
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float zj = z[j];
    zs[j] = zj;
    sup[j] = __fadd_rn(r, __fmul_rn(gwt, zj));
  }
  __syncthreads();

  B2R_MARK(4);
  // ---- B. argmax action (first maximum, RA:238-248), projection (RA:381-494)
  // every warp reduces the per-warp bests itself (5 shuffle steps instead of a
  // serial scan of shared memory): highest q, ties to the smaller action index
  int win = lane;
  {
    float q = lane < W ? s_q[lane] : 0.f;
    int act = lane < W ? s_a[lane] : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float q2 = __shfl_xor_sync(0xffffffffu, q, o);
      const int act2 = __shfl_xor_sync(0xffffffffu, act, o);
      const int win2 = __shfl_xor_sync(0xffffffffu, win, o);
      if (act2 >= 0 && (act < 0 || q2 > q || (q2 == q && act2 < act))) {
        q = q2;
        act = act2;
        win = win2;
      }
    }
  }
  const float *next_p = smem + (size_t)win * N;
  const float z0 = zs[0], zlast = zs[N - 1];
  const float dz = __fsub_rn(zs[1], zs[0]);
  const int open_above = clipped_reach_below_last(zs[N - 2], zlast, dz, N);
  // The dense form sums hat(i, j) * p_j over all j, but hat is exactly 0 unless
  // |clip(s_j) - z_i| < dz.  The Bellman atoms s_j = r + g * z_j are non-decreasing
  // in j (g = gamma^n (1 - terminal) >= 0), so the j that can reach atom i form one
  // interval: those with s_j inside (z_i - dz, z_i + dz), open-ended below for the
  // first atom and above for the atoms from open_above up (clipping).  Each thread
  // evaluates the reference's expression over a conservative superset of its interval
  // (two extra positions either side cover any rounding of the bounds; terminal rows,
  // where all s_j coincide, take the whole range) in ascending j.  Skipped terms are
  // zeros of the dense form, so the sum is its sum in the same order.
#pragma unroll 1
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    const float zi = zs[i];
    int jl = 0, jh = N - 1;
    if (gwt > 0.f) {
      // s_j > zi - dz  <=>  j > ((zi - dz - r) / g - z0) / dz
      const float inv = __fdividef(1.0f, gwt * dz);
      const float lo = (zi - dz - r - gwt * z0) * inv;
      const float hi = (zi + dz - r - gwt * z0) * inv;
      if (i > 0 && lo > 2.f) jl = min(N - 1, (int)fminf(lo, 1e6f) - 2);
      if (i < open_above && hi < (float)(N - 3))
        jh = min(N - 1, max(0, (int)fmaxf(hi, -1e6f) + 3));  // (N <= 3: hi may be < 0)
    }
    float acc = 0.f;
#pragma unroll 1
    for (int j = jl; j <= jh; ++j) {
      const float clipped = fminf(fmaxf(sup[j], z0), zlast);
      const float gap = fabsf(__fsub_rn(clipped, zi));
      if (gap < dz) {
        float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
        hat = fminf(fmaxf(hat, 0.f), 1.f);
        acc = __fadd_rn(acc, __fmul_rn(hat, next_p[j]));
      }
    }
    tgt[i] = acc;
    if (a.u.target) a.u.target[(size_t)b * N + i] = acc;
  }
  __syncthreads();

  B2R_MARK(5);
  // ---- C. cross entropy (RA:262-271), priority (RA:290), weight (RA:279-280)
  const float *x = onl;
  if (warp == 0) {
    float ce_part = 0.f, tsum_part = 0.f;
#pragma unroll 1
    for (int i = lane; i < N; i += 32) {
      const float t = tgt[i];
      const float logp = lgp[i];
      ce_part = __fadd_rn(ce_part, __fmul_rn(t, logp));
      tsum_part = __fadd_rn(tsum_part, t);
    }
    float ce = -warp_sum(ce_part);
    const float tsum = warp_sum(tsum_part);
    if (bad_action) {
      ce = 0.f;
      if (lane == 0 && a.err != nullptr && a.err[0] == 0) {
        a.err[0] = B2R_ERR_INDEX_RANGE;
        a.err[1] = b;
      }
    }
    if (lane == 0) {
      a.u.loss[b] = ce;
      a.u.priorities[b] = sqrtf(__fadd_rn(ce, 1e-10f));
      s_scalar[0] = tsum;
      s_ce = ce;
    }
  }
  // importance weight (RA:279-280), by another warp beside the cross entropy
  if (warp == (W > 1 ? 1 : 0) && lane == 0) {
    float w = 1.f;
    if (a.u.sampling_probabilities) {
      float mn = pmin;  // handed over by the sampler, or reduced per warp above
      if (sharded) mn = sharded_min_probability(a.sh, mn);
      if (!a.u.min_probability) {
        mn = s_red[0];
#pragma unroll 1
        for (int k = 1; k < (int)(blockDim.x >> 5); ++k) mn = fminf(mn, s_red[k]);
      }
      const float wmax = __fdiv_rn(1.0f, sqrtf(__fadd_rn(mn, 1e-10f)));
      const float raw = __fdiv_rn(1.0f, sqrtf(__fadd_rn(my_prob, 1e-10f)));
      w = __fdiv_rn(raw, wmax);
    }
    if (a.u.weights) a.u.weights[b] = w;
    s_scalar[1] = w;
  }
  __syncthreads();
  if (threadIdx.x == 0) a.weighted[b] = __fmul_rn(s_scalar[1], s_ce);

  B2R_MARK(6);
  // ---- D. gradient of mean(w * ce) w.r.t. the online logits
  if (a.u.grad_logits) {
    const float tsum = s_scalar[0], w = s_scalar[1], m = s_scalar[2], denom = s_scalar[3];
    const float scale = __fmul_rn(w, __fdiv_rn(1.0f, (float)(sharded ? a.sh.global_batch : rows)));
    float *g = a.u.grad_logits + (size_t)b * A * N;
    for (int k = threadIdx.x; k < A * N; k += blockDim.x) {
      const int act = k / N, i = k - act * N;
      float v = 0.f;
      if (act == chosen) {
        const float p = __fdiv_rn(expf(__fsub_rn(x[i], m)), denom);
        v = __fmul_rn(__fsub_rn(__fmul_rn(p, tsum), tgt[i]), scale);
      }
      g[k] = v;
    }
  }

  B2R_MARK(7);
  B2R_MARK_END(8);
  // ---- the last CTA to finish: mean weighted loss, reduced in a fixed order
  if (a.u.mean_weighted_loss == nullptr || !last_cta(a.ticket, &s_last)) return;
  mean_of_weighted(a.weighted, sharded ? rows : a.u.batch,
                   (float)(sharded ? a.sh.global_batch : a.u.batch), s_red,
                   a.u.mean_weighted_loss);
}

// ---- throughput instance (batches above 256 rows, num_atoms <= 64) ----------
// One WARP per batch row, kRowWarps rows per CTA.  The CTA-per-row kernel above
// spends most of its issue slots on 5-step shuffle reductions whose lanes are 80 %
// idle on the second atom pass (51 atoms over 32 lanes) and on block barriers: 6 300
// warp instructions per row at A = 18, N = 51.  Here G lanes share an action and hold
// 64 / G atoms each, so one warp instruction serves 32 / G actions, a reduction is
// log2(G) shuffle steps, and nothing but __syncwarp separates the phases.  The
// arithmetic is the same f32 sequence per element (exp of the max-shifted logit,
// probabilities by true division, q = sum z p, first maximum); only the order in which
// a row's 51 terms are summed differs between the instances.
constexpr int kRowWarps = 4;
constexpr int kRowAtoms = 64;

template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Pad value of the lanes beyond num_atoms (and of the groups beyond num_actions):
// finite, so max-shifting never forms inf - inf, and exp(pad - max) is exactly 0.
constexpr float kLogitPad = -1e30f;

// NC = num_atoms at compile time (51: the lanes' bounds tests fold away), 0 = runtime.
template <int G, int NC>
__global__ void __launch_bounds__(kRowWarps * 32)
c51_loss_rows_kernel(LossArgs a) {
  constexpr int PL = NC ? (NC + G - 1) / G : kRowAtoms / G;  // atoms per lane
  constexpr int GROUPS = 32 / G;     // actions per warp instruction
  __shared__ float s_bestp[kRowWarps][kRowAtoms];  // greedy action's probabilities
  __shared__ float s_sup[kRowWarps][kRowAtoms];    // Bellman support
  __shared__ float s_red[kRowWarps];
  __shared__ bool s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = lane / G, l = lane % G;
  const int N = NC ? NC : a.u.num_atoms, A = a.u.num_actions;
  const float *__restrict__ z = a.u.support;
  B2R_MARK(10);
  pdl_release();
  pdl_acquire();
  // (the sampler has ended: the write-back behind this kernel may read its indices)
  if (blockIdx.x == 0 && threadIdx.x == 0) tree_go_signal(a.go);
  B2R_MARK(11);
  const int rows = a.u.batch_count ? min(*a.u.batch_count, a.u.batch) : a.u.batch;
  const bool sharded = a.sh.global_batch > 0;
  if ((int)blockIdx.x * kRowWarps >= rows) {  // (mean loss with batch_count: sharded only)
    if (sharded) sharded_padding(a, blockIdx.x * kRowWarps, kRowWarps, rows, s_red, &s_last);
    return;
  }
  const int b = blockIdx.x * kRowWarps + warp;
  const bool row_ok = b < rows;

  // min over the batch of the sampling probabilities (IS-weight normaliser): handed
  // in by the sampler when it produced the batch, else reduced by the CTA.
  float pmin = INFINITY;
  if (a.u.sampling_probabilities) {
    if (a.u.min_probability) {
      pmin = *a.u.min_probability;
      if (sharded) pmin = sharded_min_probability(a.sh, pmin);
    } else {
      for (int k = threadIdx.x; k < rows; k += blockDim.x)
        pmin = fminf(pmin, a.u.sampling_probabilities[k]);
      pmin = -group_max<32>(-pmin);
      if (lane == 0) s_red[warp] = pmin;
      __syncthreads();
      pmin = s_red[0];
#pragma unroll
      for (int k = 1; k < kRowWarps; ++k) pmin = fminf(pmin, s_red[k]);
      __syncthreads();  // s_red is reused by the mean-loss reduction
    }
  }

  if (row_ok) {
    const int chosen_raw = a.u.actions[b];
    const bool bad_action = chosen_raw < 0 || chosen_raw >= A;  // (see c51_loss_kernel)
    const int chosen = bad_action ? 0 : chosen_raw;
    const float r = a.u.rewards[b];
    const float term = (float)a.u.terminals[b];
    const float my_prob = a.u.sampling_probabilities ? a.u.sampling_probabilities[b] : 1.f;
    const float *__restrict__ trow = a.u.target_logits + (size_t)b * A * N;
    const float *__restrict__ orow = a.u.online_logits + (size_t)b * A * N;
    float zl[PL], xn[PL];
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      const int i = l + G * t;
      zl[t] = i < N ? z[i] : 0.f;
      xn[t] = (i < N && grp < A) ? trow[grp * N + i] : kLogitPad;
    }
    float xo[2];  // the chosen action's online logits, atoms lane and lane + 32
#pragma unroll
    for (int t = 0; t < 2; ++t)
      xo[t] = lane + 32 * t < N ? orow[chosen * N + lane + 32 * t] : kLogitPad;

    // ---- A. per-action softmax + q-value (atari_lib.py:141-143), GROUPS actions per
    // round; the next round's logits are in flight while this one is reduced
    float best_q = 0.f;
    int best_a = -1;
    float bp[PL];
#pragma unroll
    for (int t = 0; t < PL; ++t) bp[t] = 0.f;
    const int rounds = (A + GROUPS - 1) / GROUPS;
#pragma unroll 1
    for (int rd = 0; rd < rounds; ++rd) {
      const int act = rd * GROUPS + grp;
      const bool valid = act < A;
      float xt[PL];
#pragma unroll
      for (int t = 0; t < PL; ++t) xt[t] = xn[t];
      const int nact = act + GROUPS;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        const int i = l + G * t;
        xn[t] = (i < N && nact < A) ? trow[nact * N + i] : kLogitPad;
      }
      float m = xt[0];
#pragma unroll
      for (int t = 1; t < PL; ++t) m = fmaxf(m, xt[t]);
      m = group_max<G>(m);
      float e[PL];
      float psum = 0.f;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        e[t] = expf(__fsub_rn(xt[t], m));  // pads: exactly 0
        psum = __fadd_rn(psum, e[t]);
      }
      const float denom = group_sum<G>(psum);  // >= 1: the maximum contributes 1
      float qpart = 0.f;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        e[t] = __fdiv_rn(e[t], denom);
        qpart = __fadd_rn(qpart, __fmul_rn(zl[t], e[t]));
      }
      const float q = group_sum<G>(qpart);
      if (valid && (best_a < 0 || q > best_q)) {  // strict > keeps the first maximum
        best_q = q;
        best_a = act;
#pragma unroll
        for (int t = 0; t < PL; ++t) bp[t] = e[t];
      }
    }
    // first maximum over the groups (RA:238-248): highest q, ties to the smaller action
    const int own_a = best_a;
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      const float q2 = __shfl_xor_sync(0xffffffffu, best_q, o);
      const int a2 = __shfl_xor_sync(0xffffffffu, best_a, o);
      if (a2 >= 0 && (best_a < 0 || q2 > best_q || (q2 == best_q && a2 < best_a))) {
        best_q = q2;
        best_a = a2;
      }
    }
    if (own_a == best_a && own_a >= 0) {
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (l + G * t < N) s_bestp[warp][l + G * t] = bp[t];
    }

    // log_softmax of the chosen action's online logits (rainbow_agent.py:262-271):
    // atoms lane, lane + 32 — the layout of the projection below
    float mo = fmaxf(xo[0], xo[1]);
    mo = group_max<32>(mo);
    const float eo0 = expf(__fsub_rn(xo[0], mo)), eo1 = expf(__fsub_rn(xo[1], mo));
    const float den_o = group_sum<32>(__fadd_rn(eo0, eo1));  // pads add exactly 0
    const float lse = logf(den_o);
    const float lgp[2] = {__fsub_rn(__fsub_rn(xo[0], mo), lse),
                          __fsub_rn(__fsub_rn(xo[1], mo), lse)};
    // Bellman support (rainbow_agent.py:229-235)
    const float live = __fsub_rn(1.0f, term);
    const float gwt = __fmul_rn(a.u.cumulative_gamma, live);
    for (int j = lane; j < N; j += 32) s_sup[warp][j] = __fadd_rn(r, __fmul_rn(gwt, z[j]));
    __syncwarp();

    // ---- B. projection (RA:381-494).  hat(i, j) is exactly 0 unless
    // |clip(s_j) - z_i| < dz, and the Bellman atoms s_j = r + g z_j are non-decreasing
    // in j (g >= 0), so the j that reach atom i form one interval: s_j inside
    // (z_i - dz, z_i + dz), i.e. lo < j < hi in units of atoms, open-ended below for
    // the first atom and above for the atoms from open_above up (clipping).  Each lane
    // sums the reference's expression in ascending j over [floor(lo), floor(hi) + 1]:
    // one spare position either side, against a rounding error of lo / hi below 1e-4.
    // Skipped terms are zeros of the dense form, so the sum is its sum in the same order.
    const float *sup = s_sup[warp], *next_p = s_bestp[warp];
    const float z0 = z[0], zlast = z[N - 1];
    const float dz = __fsub_rn(z[1], z0);
    const int open_above = clipped_reach_below_last(z[N - 2], zlast, dz, N);
    float tg[2] = {0.f, 0.f};
    float ce_part = 0.f, tsum_part = 0.f;
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int i = lane + 32 * t;
      if (i < N) {
        const float zi = z[i];
        float acc = 0.f;
        if (gwt == 0.f) {
          // terminal row: every s_j is r, so hat(i, .) is one number, and it is 0 for
          // all but the (at most two) atoms next to clip(r)
          const float clipped = fminf(fmaxf(sup[0], z0), zlast);
          const float gap = fabsf(__fsub_rn(clipped, zi));
          if (gap < dz) {
            float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
            hat = fminf(fmaxf(hat, 0.f), 1.f);
#pragma unroll 1
            for (int j = 0; j < N; ++j) acc = __fadd_rn(acc, __fmul_rn(hat, next_p[j]));
          }
        } else {
          int jl = 0, jh = N - 1;
          if (gwt > 0.f) {
            const float inv = __fdividef(1.0f, gwt * dz);
            const float lo = (zi - dz - r - gwt * z0) * inv;
            const float hi = (zi + dz - r - gwt * z0) * inv;
            if (i > 0 && lo > 0.f) jl = min(N - 1, (int)fminf(lo, 1e6f));
            if (i < open_above && hi < (float)(N - 2)) jh = max(0, (int)fmaxf(hi, -1e6f) + 1);
          }
#pragma unroll 1
          for (int j = jl; j <= jh; ++j) {
            const float clipped = fminf(fmaxf(sup[j], z0), zlast);
            const float gap = fabsf(__fsub_rn(clipped, zi));
            if (gap < dz) {
              float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
              hat = fminf(fmaxf(hat, 0.f), 1.f);
              acc = __fadd_rn(acc, __fmul_rn(hat, next_p[j]));
            }
          }
        }
        tg[t] = acc;
        if (a.u.target) a.u.target[(size_t)b * N + i] = acc;
        ce_part = __fadd_rn(ce_part, __fmul_rn(acc, lgp[t]));
        tsum_part = __fadd_rn(tsum_part, acc);
      }
    }

    // ---- C. cross entropy (RA:262-271), priority (RA:290), weight (RA:279-280)
    float ce = -group_sum<32>(ce_part);
    const float tsum = group_sum<32>(tsum_part);
    if (bad_action) {
      ce = 0.f;
      if (lane == 0 && a.err != nullptr && a.err[0] == 0) {
        a.err[0] = B2R_ERR_INDEX_RANGE;
        a.err[1] = b;
      }
    }
    float w = 1.f;
    if (a.u.sampling_probabilities) {
      const float wmax = __fdiv_rn(1.0f, sqrtf(__fadd_rn(pmin, 1e-10f)));
      const float raw = __fdiv_rn(1.0f, sqrtf(__fadd_rn(my_prob, 1e-10f)));
      w = __fdiv_rn(raw, wmax);
    }
    if (lane == 0) {
      a.u.loss[b] = ce;
      a.u.priorities[b] = sqrtf(__fadd_rn(ce, 1e-10f));
      if (a.u.weights) a.u.weights[b] = w;
      a.weighted[b] = __fmul_rn(w, ce);
    }

    // ---- D. gradient of mean(w * ce) w.r.t. the online logits
    if (a.u.grad_logits) {
      const float scale =
          __fmul_rn(w, __fdiv_rn(1.0f, (float)(sharded ? a.sh.global_batch : rows)));
      float *g = a.u.grad_logits + (size_t)b * A * N;
      float v[2] = {0.f, 0.f};
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int i = lane + 32 * t;
        if (i < N) {
          const float p = __fdiv_rn(t == 0 ? eo0 : eo1, den_o);
          v[t] = __fmul_rn(__fsub_rn(__fmul_rn(p, tsum), tg[t]), scale);
        }
      }
      for (int act = 0; act < A; ++act) {
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const int i = lane + 32 * t;
          if (i < N) g[act * N + i] = act == chosen ? v[t] : 0.f;
        }
      }
    }
  } else if (sharded && a.u.grad_logits != nullptr && b < a.u.batch) {
    float *g = a.u.grad_logits + (size_t)b * A * N;  // a padded row of this CTA
    for (int k = lane; k < A * N; k += 32) g[k] = 0.f;
  }

  B2R_MARK_END(12);
  // ---- mean weighted loss: the last CTA to finish reduces in a fixed order.
  if (a.u.mean_weighted_loss == nullptr) return;
  if (!last_cta(a.ticket, &s_last)) return;
  mean_of_weighted(a.weighted, sharded ? rows : a.u.batch,
                   (float)(sharded ? a.sh.global_batch : a.u.batch), s_red,
                   a.u.mean_weighted_loss);
}

// ---- the loss in two halves (the fused step) --------------------------------------
// What a row's loss needs from the NETWORK OUTPUTS alone — softmax and q-value of every
// action's target logits, the greedy next action and its probabilities, the log-sum-exp
// of every action's online logits — does not depend on which transitions were sampled;
// what depends on the sample (action, n-step return, terminal, sampling probability) is
// a short tail: Bellman support, projection of ONE distribution, cross entropy against
// ONE row of online logits.  The fused step runs the first half (c51_pre_*) beside the
// sampler and the tail (c51_post_kernel) behind it (PreSync, replay.cuh, says how the two
// meet).  The arithmetic is that of c51_loss_kernel, element by element.
//
// Scratch per row (kPreRow floats): [0, 64) probabilities of the greedy next action,
// [64, 128) online softmax statistics, (max, log of the denominator) per action for the
// first 32 actions (c51_pre_kernel only; stats == 0 in PostArgs: the tail computes them).
// A staged tail (StageGate) also gets the online log-probabilities of every action, in a
// buffer of their own (PreArgs::logp).
constexpr int kPreRow = 2 * kRowAtoms;

struct PreArgs {
  const float *target_logits;
  const float *online_logits;
  const float *support;
  float *scratch;  // [rows][kPreRow]
  int rows, num_actions, num_atoms, warps;
  PreSync sync;
  // nullable: device copy of the online logits, written as they are read.  The host-facing
  // trainer lets this kernel read both logits tensors straight from the caller's
  // page-locked memory (no copy calls on the host); the tail then reads its one row of
  // online logits per transition from this copy instead of crossing PCIe again.
  float *online_copy;
  // nullable (c51_pre_kernel): [rows][c51_logp_stride] log_softmax of every action's online
  // logits, and StageGate::first_half.done, counted when they are all there
  float *logp;
  unsigned int *staged_done;
  // The one-stream step (StageGate::rows): launched behind the sampler, which waits for this
  // launch's signal before it ends, so the griddepcontrol.wait comes after the signal.
  int wait_late;
};

// CTA per row, warp per action (rows below 128: latency-bound).
template <int PL>
__global__ void __launch_bounds__(1024) c51_pre_kernel(PreArgs a) {
  __shared__ float s_q[32];
  __shared__ int s_a[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x;
  const int N = a.num_atoms, A = a.num_actions, W = a.warps;
  B2R_MARK(0);
  pdl_release();
  if (!a.wait_late) pdl_acquire();
  B2R_MARK(1);
  const float *__restrict__ trow = a.target_logits + (size_t)b * A * N;
  const float *__restrict__ orow = a.online_logits + (size_t)b * A * N;
  float zl[PL], xt[PL], xo[PL], bp[PL];
#pragma unroll
  for (int t = 0; t < PL; ++t) {
    const int i = lane + 32 * t;
    zl[t] = i < N ? a.support[i] : 0.f;
    xt[t] = (i < N && warp < A) ? trow[warp * N + i] : -INFINITY;
    xo[t] = (i < N && warp < A) ? orow[warp * N + i] : -INFINITY;
    bp[t] = 0.f;
  }
  float *__restrict__ ocopy =
      a.online_copy != nullptr ? a.online_copy + (size_t)b * A * N : nullptr;
  float best_q = 0.f;
  int best_a = -1;
  for (int act = warp; act < A; act += W) {
    if (act != warp) {
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        const int i = lane + 32 * t;
        xt[t] = i < N ? trow[act * N + i] : -INFINITY;
        xo[t] = i < N ? orow[act * N + i] : -INFINITY;
      }
    }
    if (ocopy != nullptr) {
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (lane + 32 * t < N) ocopy[act * N + lane + 32 * t] = xo[t];
    }
    // the two softmaxes interleave: their reductions do not depend on each other
    float m = -INFINITY, mo = -INFINITY;
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      m = fmaxf(m, xt[t]);
      mo = fmaxf(mo, xo[t]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
      mo = fmaxf(mo, __shfl_xor_sync(0xffffffffu, mo, o));
    }
    float e[PL];
    float psum = 0.f, osum = 0.f;
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      const bool ok = lane + 32 * t < N;
      e[t] = ok ? expf(__fsub_rn(xt[t], m)) : 0.f;
      if (ok) psum = __fadd_rn(psum, e[t]);
      if (ok) osum = __fadd_rn(osum, expf(__fsub_rn(xo[t], mo)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      psum = __fadd_rn(psum, __shfl_xor_sync(0xffffffffu, psum, o));
      osum = __fadd_rn(osum, __shfl_xor_sync(0xffffffffu, osum, o));
    }
    const float denom = psum;
    // log_softmax(x) = (x - max) - log(sum exp(x - max))   (rainbow_agent.py:262-271)
    if (lane == 0 && act < 32) {
      float2 st;
      st.x = mo;
      st.y = logf(osum);
      *reinterpret_cast<float2 *>(a.scratch + (size_t)b * kPreRow + kRowAtoms + 2 * act) = st;
    }
    if (a.logp != nullptr) {  // (the tail's expression, with the statistics above)
      const float lse = logf(osum);
      float *lrow = a.logp + (size_t)b * c51_logp_stride(A, N) + act * N;
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (lane + 32 * t < N) lrow[lane + 32 * t] = __fsub_rn(__fsub_rn(xo[t], mo), lse);
    }
    float qpart = 0.f;
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      if (lane + 32 * t < N) {
        e[t] = __fdiv_rn(e[t], denom);
        qpart = __fadd_rn(qpart, __fmul_rn(zl[t], e[t]));
      }
    }
    const float q = warp_sum<true>(qpart);
    if (best_a < 0 || q > best_q) {  // strict > keeps the first maximum
      best_q = q;
      best_a = act;
#pragma unroll
      for (int t = 0; t < PL; ++t) bp[t] = e[t];
    }
  }
  if (lane == 0) {
    s_q[warp] = best_q;
    s_a[warp] = best_a;
  }
  __syncthreads();
  // first maximum over the actions (RA:238-248): highest q, ties to the smaller action
  int win = lane;
  {
    float q = lane < W ? s_q[lane] : 0.f;
    int act = lane < W ? s_a[lane] : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float q2 = __shfl_xor_sync(0xffffffffu, q, o);
      const int act2 = __shfl_xor_sync(0xffffffffu, act, o);
      const int win2 = __shfl_xor_sync(0xffffffffu, win, o);
      if (act2 >= 0 && (act < 0 || q2 > q || (q2 == q && act2 < act))) {
        q = q2;
        act = act2;
        win = win2;
      }
    }
  }
  if (warp == win) {
#pragma unroll
    for (int t = 0; t < PL; ++t)
      if (lane + 32 * t < N) a.scratch[(size_t)b * kPreRow + lane + 32 * t] = bp[t];
  }
  B2R_MARK_END(8);
  pre_sync_signal(a.sync, a.staged_done);
  if (a.wait_late) pdl_acquire();
}

// Warp per row, G lanes per action (rows from 128 up: bound by instruction issue).
template <int G, int NC>
__global__ void __launch_bounds__(kRowWarps * 32) c51_pre_rows_kernel(PreArgs a) {
  constexpr int PL = NC ? (NC + G - 1) / G : kRowAtoms / G;
  constexpr int GROUPS = 32 / G;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = lane / G, l = lane % G;
  const int N = NC ? NC : a.num_atoms, A = a.num_actions;
  B2R_MARK(0);
  pdl_release();
  pdl_acquire();
  B2R_MARK(1);
  const int b = blockIdx.x * kRowWarps + warp;
  if (b < a.rows) {
    if (a.online_copy != nullptr) {
      const float *__restrict__ src = a.online_logits + (size_t)b * A * N;
      float *__restrict__ dst = a.online_copy + (size_t)b * A * N;
      for (int k = lane; k < A * N; k += 32) dst[k] = src[k];
    }
    const float *__restrict__ trow = a.target_logits + (size_t)b * A * N;
    float zl[PL], xn[PL];
#pragma unroll
    for (int t = 0; t < PL; ++t) {
      const int i = l + G * t;
      zl[t] = i < N ? a.support[i] : 0.f;
      xn[t] = (i < N && grp < A) ? trow[grp * N + i] : kLogitPad;
    }
    float best_q = 0.f;
    int best_a = -1;
    float bp[PL];
#pragma unroll
    for (int t = 0; t < PL; ++t) bp[t] = 0.f;
    const int rounds = (A + GROUPS - 1) / GROUPS;
#pragma unroll 1
    for (int rd = 0; rd < rounds; ++rd) {
      const int act = rd * GROUPS + grp;
      const bool valid = act < A;
      float xt[PL];
#pragma unroll
      for (int t = 0; t < PL; ++t) xt[t] = xn[t];
      const int nact = act + GROUPS;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        const int i = l + G * t;
        xn[t] = (i < N && nact < A) ? trow[nact * N + i] : kLogitPad;
      }
      float m = xt[0];
#pragma unroll
      for (int t = 1; t < PL; ++t) m = fmaxf(m, xt[t]);
      m = group_max<G>(m);
      float e[PL];
      float psum = 0.f;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        e[t] = expf(__fsub_rn(xt[t], m));  // pads: exactly 0
        psum = __fadd_rn(psum, e[t]);
      }
      const float denom = group_sum<G>(psum);  // >= 1: the maximum contributes 1
      float qpart = 0.f;
#pragma unroll
      for (int t = 0; t < PL; ++t) {
        e[t] = __fdiv_rn(e[t], denom);
        qpart = __fadd_rn(qpart, __fmul_rn(zl[t], e[t]));
      }
      const float q = group_sum<G>(qpart);
      if (valid && (best_a < 0 || q > best_q)) {
        best_q = q;
        best_a = act;
#pragma unroll
        for (int t = 0; t < PL; ++t) bp[t] = e[t];
      }
    }
    const int own_a = best_a;
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      const float q2 = __shfl_xor_sync(0xffffffffu, best_q, o);
      const int a2 = __shfl_xor_sync(0xffffffffu, best_a, o);
      if (a2 >= 0 && (best_a < 0 || q2 > best_q || (q2 == best_q && a2 < best_a))) {
        best_q = q2;
        best_a = a2;
      }
    }
    if (own_a == best_a && own_a >= 0) {
#pragma unroll
      for (int t = 0; t < PL; ++t)
        if (l + G * t < N) a.scratch[(size_t)b * kPreRow + l + G * t] = bp[t];
    }
  }
  B2R_MARK_END(8);
  pre_sync_signal(a.sync);
}

constexpr int kProjTerms = 5;  // Bellman atoms within dz of an output atom, with slack
                              // (gamma^n >= 2/3: 2 / (gamma^n) + 2 <= 5; wider, or atom
                              // N - 2 open above with clipped mass beyond: the loop)

// The part of a row's tail that follows its scalars and the log-probabilities of its
// chosen action: Bellman support, projection, cross entropy and the row's outputs.
// LEAN: neither the projected target nor a gradient row is asked for (compile-time: the
// staged instance the fused step runs at the agent's batch).
template <bool LEAN>
__device__ __forceinline__ float c51_post_finish(const LossArgs &a, int b, int rows, int lane,
                                                 const float (&zl)[2], float r, float term,
                                                 float w, const float (&lgp)[2],
                                                 bool bad_action, int chosen, float eo0,
                                                 float eo1, float den_o,
                                                 const float *bestp_row, float *sup_row) {
  const int N = a.u.num_atoms, A = a.u.num_actions;
  float prio_out = 0.f;
  // Bellman support (rainbow_agent.py:229-235)
  const float live = __fsub_rn(1.0f, term);
  const float gwt = __fmul_rn(a.u.cumulative_gamma, live);
#pragma unroll
  for (int t = 0; t < 2; ++t)
    if (lane + 32 * t < N) sup_row[lane + 32 * t] = __fadd_rn(r, __fmul_rn(gwt, zl[t]));
  __syncwarp();

  // projection (RA:381-494): see c51_loss_rows_kernel for the interval argument
  const float *sup = sup_row, *next_p = bestp_row;
  const float z0 = __shfl_sync(0xffffffffu, zl[0], 0);
  const float z1 = __shfl_sync(0xffffffffu, zl[0], 1);
  const float zlast = __shfl_sync(0xffffffffu, N > 32 ? zl[1] : zl[0], (N - 1) & 31);
  const float zprev = __shfl_sync(0xffffffffu, N > 33 ? zl[1] : zl[0], (N - 2) & 31);
  const float dz = __fsub_rn(z1, z0);
  const int open_above = clipped_reach_below_last(zprev, zlast, dz, N);
  float tg[2] = {0.f, 0.f};
  if (gwt == 0.f) {
    // terminal row: every s_j is r, so hat(i, .) is one number, and it is 0 for all but
    // the (at most two) atoms next to clip(r)
    const float clipped = fminf(fmaxf(sup[0], z0), zlast);
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int i = lane + 32 * t;
      const float gap = fabsf(__fsub_rn(clipped, zl[t]));
      if (i < N && gap < dz) {
        float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
        hat = fminf(fmaxf(hat, 0.f), 1.f);
        float acc = 0.f;
#pragma unroll 1
        for (int j = 0; j < N; ++j) acc = __fadd_rn(acc, __fmul_rn(hat, next_p[j]));
        tg[t] = acc;
      }
    }
  } else {
    int jl[2], jh[2];
    const float inv = __fdividef(1.0f, gwt * dz);
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int i = lane + 32 * t;
      jl[t] = 0;
      jh[t] = i < N ? N - 1 : -1;
      if (gwt > 0.f && i < N) {
        const float lo = (zl[t] - dz - r - gwt * z0) * inv;
        const float hi = (zl[t] + dz - r - gwt * z0) * inv;
        if (i > 0 && lo > 0.f) jl[t] = min(N - 1, (int)fminf(lo, 1e6f));
        if (i < open_above && hi < (float)(N - 2)) jh[t] = max(0, (int)fmaxf(hi, -1e6f) + 1);
      }
    }
    const bool narrow = jh[0] - jl[0] < kProjTerms && jh[1] - jl[1] < kProjTerms;
    if (__all_sync(0xffffffffu, narrow)) {
      float term_v[2][kProjTerms];
      bool term_on[2][kProjTerms];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
#pragma unroll
        for (int k = 0; k < kProjTerms; ++k) {
          const int j = jl[t] + k;
          const bool in = j <= jh[t];
          const int jj = in ? j : 0;
          const float clipped = fminf(fmaxf(sup[jj], z0), zlast);
          const float gap = fabsf(__fsub_rn(clipped, zl[t]));
          float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
          hat = fminf(fmaxf(hat, 0.f), 1.f);
          term_v[t][k] = __fmul_rn(hat, next_p[jj]);
          term_on[t][k] = in && gap < dz;
        }
      }
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < kProjTerms; ++k)
          if (term_on[t][k]) acc = __fadd_rn(acc, term_v[t][k]);
        tg[t] = acc;
      }
    } else {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        float acc = 0.f;
#pragma unroll 1
        for (int j = jl[t]; j <= jh[t]; ++j) {
          const float clipped = fminf(fmaxf(sup[j], z0), zlast);
          const float gap = fabsf(__fsub_rn(clipped, zl[t]));
          if (gap < dz) {
            float hat = __fsub_rn(1.0f, __fdiv_rn(gap, dz));
            hat = fminf(fmaxf(hat, 0.f), 1.f);
            acc = __fadd_rn(acc, __fmul_rn(hat, next_p[j]));
          }
        }
        tg[t] = acc;
      }
    }
  }
  float ce_part = 0.f, tsum_part = 0.f;
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int i = lane + 32 * t;
    if (i < N) {
      if (!LEAN && a.u.target) a.u.target[(size_t)b * N + i] = tg[t];
      ce_part = __fadd_rn(ce_part, __fmul_rn(tg[t], lgp[t]));
      tsum_part = __fadd_rn(tsum_part, tg[t]);
    }
  }

  // cross entropy (RA:262-271), priority (RA:290), weight (RA:279-280)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ce_part = __fadd_rn(ce_part, __shfl_xor_sync(0xffffffffu, ce_part, o));
    tsum_part = __fadd_rn(tsum_part, __shfl_xor_sync(0xffffffffu, tsum_part, o));
  }
  float ce = -ce_part;
  const float tsum = tsum_part;
  if (bad_action) {
    ce = 0.f;
    if (lane == 0 && a.err != nullptr && a.err[0] == 0) {
      a.err[0] = B2R_ERR_INDEX_RANGE;
      a.err[1] = b;
    }
  }
  prio_out = sqrtf(__fadd_rn(ce, 1e-10f));
  if (lane == 0) {
    a.u.loss[b] = ce;
    if (a.loss_host != nullptr) a.loss_host[b] = ce;
    a.u.priorities[b] = prio_out;
    if (a.u.weights) a.u.weights[b] = w;
    a.weighted[b] = __fmul_rn(w, ce);
  }
  if (!LEAN && a.u.grad_logits) {
    const float scale = __fmul_rn(w, __fdiv_rn(1.0f, (float)rows));
    float *g = a.u.grad_logits + (size_t)b * A * N;
    float v[2] = {0.f, 0.f};
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int i = lane + 32 * t;
      if (i < N) {
        const float p = __fdiv_rn(t == 0 ? eo0 : eo1, den_o);
        v[t] = __fmul_rn(__fsub_rn(__fmul_rn(p, tsum), tg[t]), scale);
      }
    }
    for (int act = 0; act < A; ++act) {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const int i = lane + 32 * t;
        if (i < N) g[act * N + i] = act == chosen ? v[t] : 0.f;
      }
    }
  }
  return prio_out;
}

// One row of the tail by one warp.  bestp_row / sup_row: this warp's shared-memory rows
// ([kRowAtoms] floats each).  Writes the row's outputs and returns its new priority.
__device__ __forceinline__ float c51_post_row(const LossArgs &a,
                                              const float *__restrict__ scratch,
                                              int have_stats, int b, int rows, int lane,
                                              float pmin, float *bestp_row, float *sup_row) {
  const int N = a.u.num_atoms, A = a.u.num_actions;
  const float *__restrict__ z = a.u.support;
  // ---- round trip 1
  int chosen = a.u.actions[b];
  const float r = a.u.rewards[b];
  const float term = (float)a.u.terminals[b];
  const float my_prob = a.u.sampling_probabilities ? a.u.sampling_probabilities[b] : 1.f;
  float zl[2], bp[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int i = lane + 32 * t;
    zl[t] = i < N ? z[i] : 0.f;
    bp[t] = i < N ? scratch[(size_t)b * kPreRow + i] : 0.f;
  }
  float2 st = make_float2(0.f, 0.f);  // lane = action: (max, log denominator)
  if (have_stats && lane < A)
    st = *reinterpret_cast<const float2 *>(scratch + (size_t)b * kPreRow + kRowAtoms + 2 * lane);
  // importance weight (RA:279-280): needs the probabilities only — two square roots and
  // three divisions that are in flight while the second round trip and the projection run
  float w = 1.f;
  if (a.u.sampling_probabilities) {
    const float wmax = __fdiv_rn(1.0f, sqrtf(__fadd_rn(pmin, 1e-10f)));
    const float raw = __fdiv_rn(1.0f, sqrtf(__fadd_rn(my_prob, 1e-10f)));
    w = __fdiv_rn(raw, wmax);
  }
  B2R_MARK(13);
  // an action outside [0, A) (tf.gather_nd raises): evaluated for action 0, zero loss,
  // B2R_ERR_INDEX_RANGE latched
  const bool bad_action = chosen < 0 || chosen >= A;
  if (bad_action) chosen = 0;
  // ---- round trip 2
  const float *__restrict__ orow = a.u.online_logits + ((size_t)b * A + chosen) * N;
  float xo[2];
#pragma unroll
  for (int t = 0; t < 2; ++t) xo[t] = lane + 32 * t < N ? orow[lane + 32 * t] : kLogitPad;
#pragma unroll
  for (int t = 0; t < 2; ++t)
    if (lane + 32 * t < N) bestp_row[lane + 32 * t] = bp[t];
  // log_softmax of the chosen action's online logits (rainbow_agent.py:262-271)
  float mo, lse, eo0 = 0.f, eo1 = 0.f, den_o = 1.f;
  if (have_stats && chosen < 32) {
    mo = __shfl_sync(0xffffffffu, st.x, chosen);
    lse = __shfl_sync(0xffffffffu, st.y, chosen);
    if (a.u.grad_logits) {
      eo0 = expf(__fsub_rn(xo[0], mo));
      eo1 = expf(__fsub_rn(xo[1], mo));
      den_o = group_sum<32>(__fadd_rn(eo0, eo1));
    }
  } else {
    mo = group_max<32>(fmaxf(xo[0], xo[1]));
    eo0 = expf(__fsub_rn(xo[0], mo));
    eo1 = expf(__fsub_rn(xo[1], mo));
    den_o = group_sum<32>(__fadd_rn(eo0, eo1));  // pads add exactly 0
    lse = logf(den_o);
  }
  const float lgp[2] = {__fsub_rn(__fsub_rn(xo[0], mo), lse),
                        __fsub_rn(__fsub_rn(xo[1], mo), lse)};
  B2R_MARK(14);
  return c51_post_finish<false>(a, b, rows, lane, zl, r, term, w, lgp, bad_action, chosen,
                                eo0, eo1, den_o, bestp_row, sup_row);
}

// A staged row (c51_post_tree_kernel<true>), ahead of the sampler's end: the greedy
// action's probabilities into bestp_row, the log-probabilities of all actions into
// logp_row ([c51_logp_stride / 4] float4s), the support into zl.  L2 loads (__ldcg): the
// first half's rows arrive through memory, not across a kernel boundary.
__device__ __forceinline__ void c51_stage_row(const LossArgs &a, const float *scratch, int b,
                                              int lane, float *bestp_row, float4 *logp_row,
                                              float (&zl)[2]) {
  const int N = a.u.num_atoms;
  const int words = c51_logp_stride(a.u.num_actions, N) / 4;
  const float4 *src = reinterpret_cast<const float4 *>(a.stage.logp) + (size_t)b * words;
  constexpr int kBurst = 8;  // float4 loads in flight per lane
  for (int base = 0; base < words; base += 32 * kBurst) {
    float4 v[kBurst];
#pragma unroll
    for (int u = 0; u < kBurst; ++u) {
      const int k = base + 32 * u + lane;
      if (k < words) v[u] = __ldcg(src + k);
    }
#pragma unroll
    for (int u = 0; u < kBurst; ++u) {
      const int k = base + 32 * u + lane;
      if (k < words) logp_row[k] = v[u];
    }
  }
#pragma unroll
  for (int t = 0; t < 2; ++t) {
    const int i = lane + 32 * t;
    zl[t] = i < N ? __ldcg(a.u.support + i) : 0.f;
    if (i < N) bestp_row[i] = __ldcg(scratch + (size_t)b * kPreRow + i);
  }
  __syncwarp();  // (the chosen action's row is read across lanes)
}

// The rest of a staged row, behind the sampler: ONE round trip for the sampled scalars,
// then the chosen action's log-probabilities from shared memory.
__device__ __forceinline__ float c51_post_staged_row(const LossArgs &a, int b, int rows,
                                                     int lane, const float (&zl)[2],
                                                     const float *bestp_row, float *sup_row,
                                                     const float *logp_row) {
  const int N = a.u.num_atoms, A = a.u.num_actions;
  int chosen = a.u.actions[b];
  const float r = a.u.rewards[b];
  const float term = (float)a.u.terminals[b];
  float w = 1.f;
  if (a.u.sampling_probabilities) {  // (RA:279-280)
    const float pmin = *a.u.min_probability;
    const float my_prob = a.u.sampling_probabilities[b];
    const float wmax = __fdiv_rn(1.0f, sqrtf(__fadd_rn(pmin, 1e-10f)));
    const float raw = __fdiv_rn(1.0f, sqrtf(__fadd_rn(my_prob, 1e-10f)));
    w = __fdiv_rn(raw, wmax);
  }
  // (as in c51_post_row: an action outside [0, A) is evaluated for action 0)
  const bool bad_action = chosen < 0 || chosen >= A;
  if (bad_action) chosen = 0;
  B2R_MARK_CTA(13, 1);
  const float lgp[2] = {lane < N ? logp_row[chosen * N + lane] : 0.f,
                        lane + 32 < N ? logp_row[chosen * N + lane + 32] : 0.f};
  return c51_post_finish<true>(a, b, rows, lane, zl, r, term, w, lgp, bad_action, chosen, 0.f,
                               0.f, 1.f, bestp_row, sup_row);
}

// The tail: one warp per row, kRowWarps rows per CTA, lanes own atoms lane and lane + 32.
// Everything a row needs arrives in two memory round trips (the row's scalars, the
// greedy action's probabilities and the statistics of all actions; then the chosen
// action's online logits); the candidate terms of a projected atom are evaluated side by
// side and added in ascending j, as the dense form adds them.

__global__ void __launch_bounds__(kRowWarps * 32)
c51_post_kernel(LossArgs a, const float *__restrict__ scratch, int have_stats) {
  __shared__ float s_bestp[kRowWarps][kRowAtoms];
  __shared__ float s_sup[kRowWarps][kRowAtoms];
  __shared__ float s_red[kRowWarps];
  __shared__ bool s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  B2R_MARK(10);
  pdl_release();
  pdl_acquire();
  // (the sampler has ended: the write-back behind this kernel may read its indices)
  if (blockIdx.x == 0 && threadIdx.x == 0) tree_go_signal(a.go);
  B2R_MARK(11);
  const int rows = a.u.batch_count ? min(*a.u.batch_count, a.u.batch) : a.u.batch;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const int all = a.u.batch_count ? *a.u.batch_count : a.u.batch;
    if (a.count_copy != nullptr) *a.count_copy = all;
    if (a.loss_host != nullptr) reinterpret_cast<int32_t *>(a.loss_host)[a.u.batch] = all;
  }
  if ((int)blockIdx.x * kRowWarps >= rows) return;  // (no mean loss with batch_count)
  const int b = blockIdx.x * kRowWarps + warp;
  const bool row_ok = b < rows;

  float pmin = INFINITY;
  if (a.u.sampling_probabilities) {
    if (a.u.min_probability) {
      pmin = *a.u.min_probability;
    } else {
      for (int k = threadIdx.x; k < rows; k += blockDim.x)
        pmin = fminf(pmin, a.u.sampling_probabilities[k]);
      pmin = -group_max<32>(-pmin);
      if (lane == 0) s_red[warp] = pmin;
      __syncthreads();
      pmin = s_red[0];
#pragma unroll
      for (int k = 1; k < kRowWarps; ++k) pmin = fminf(pmin, s_red[k]);
      __syncthreads();  // s_red is reused by the mean-loss reduction
    }
  }

  if (row_ok)
    c51_post_row(a, scratch, have_stats, b, rows, lane, pmin, s_bestp[warp], s_sup[warp]);
  B2R_MARK_END(12);

  // ---- mean weighted loss: the last CTA to finish reduces in a fixed order.
  if (a.u.mean_weighted_loss == nullptr || !last_cta(a.ticket, &s_last, false)) return;
  float acc = 0.f;
  for (int k = threadIdx.x; k < a.u.batch; k += blockDim.x)
    acc = __fadd_rn(acc, __ldcg(a.weighted + k));
  acc = group_sum<32>(acc);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float total = 0.f;
    for (int k = 0; k < kRowWarps; ++k) total = __fadd_rn(total, s_red[k]);
    *a.u.mean_weighted_loss = __fdiv_rn(total, (float)a.u.batch);
    *a.ticket = 0u;  // ready for the next launch
  }
}

// The agent's batch (<= 32 rows): the tail and the priority write-back
// (prioritized_replay_buffer.py:203-214) as ONE thread-block cluster of 8 CTAs.  CTAs 1..7
// compute five rows each (one warp per row); CTA 0 is the tree's: its warp l owns tree
// level l, and what that needs from the sampled indices alone — node loads, grouping of
// the entries by node — runs while the rows are projected (tree_update_tiny_issue).  The
// new priorities go from the row warps' registers into CTA 0's shared memory (distributed
// shared memory), one cluster barrier replaces the kernel boundary, and CTA 0 finishes
// the update (tree_update_tiny_finish).  Measured (profiles/r2/README.md): 15.3 us per
// step at batch 32 against 16.3 us with the tail and the write-back as two kernels.
// STAGED (c51_tail_can_stage, no row count on the device): every row CTA stages its rows'
// inputs from the first half (StageGate) BEFORE its griddepcontrol.wait, while the
// sampler still runs, and is left with one round trip for the sampled scalars behind it.
constexpr int kPostClusterCtas = 8;
constexpr int kPostRowWarps = 5;  // rows per row CTA: 7 row CTAs x 5 >= 32 rows

template <bool STAGED>
__global__ void __launch_bounds__(1024)
c51_post_tree_kernel(LossArgs a, const float *__restrict__ scratch, int have_stats) {
  __shared__ float s_bestp[kPostRowWarps][kRowAtoms];
  __shared__ float s_sup[kPostRowWarps][kRowAtoms];
  __shared__ float s_prio[kTinyBatch];      // (CTA 0's copy is the one that is used)
  __shared__ float s_weighted[kTinyBatch];
  __shared__ __align__(8) uint64_t s_arrived;  // mbarrier: the rows' words have landed
  __shared__ bool s_gate, s_rows;
  extern __shared__ float4 s_logp[];  // STAGED: [kPostRowWarps][c51_logp_stride / 4]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool tree_cta = blockIdx.x == 0;
  B2R_MARK(10);
  if (tree_cta && threadIdx.x == 0) mbar_init(&s_arrived, 1);
  cluster_arrive_relaxed();  // (nobody sends before the mbarrier exists: waited for below)
  // STAGED: the row this warp owns (at most 32 rows: one per row warp), staged ahead of the
  // sampler's end once the first half of this step has ended (StageGate; the ticket is
  // taken before the dependents may start, and they start once it has ended: the tails of
  // later steps do not pile up resident behind this one)
  float zl[2] = {0.f, 0.f};
  float4 *logp_row = s_logp + (size_t)warp * (c51_logp_stride(a.u.num_actions, a.u.num_atoms) / 4);
  const int srow = (int)(blockIdx.x - 1) * kPostRowWarps + warp;
  const bool stages = STAGED && !tree_cta && warp < kPostRowWarps && srow < a.u.batch;
  const bool early = STAGED && cta_gate_wait<0>(a.stage.first_half, &s_gate);
  pdl_release();
  if (early && stages) c51_stage_row(a, scratch, srow, lane, s_bestp[warp], logp_row, zl);
  if (STAGED) B2R_MARK_CTA(15, 1);
  // The one-stream step: the predecessor is the frame copies, not the sampler — the rows
  // are there once the sampler has counted its launch (StageGate::rows); the griddepcontrol.wait
  // moves to the exits.  (Either gate timed out: behind the wait, the safe order.)
  const bool gated = STAGED && a.stage.rows.done != nullptr;
  if (!(gated && cta_gate_wait<32>(a.stage.rows, &s_rows) && early)) pdl_acquire();
  if (STAGED && !early && stages) c51_stage_row(a, scratch, srow, lane, s_bestp[warp], logp_row, zl);
  B2R_MARK(11);
  // (a shard's step: the row count is on the device, and the write-back rides along only
  // when it turns out to be at most 32 rows — else the tree kernel behind this one does it)
  const int rows = a.u.batch_count ? min(*a.u.batch_count, a.u.batch) : a.u.batch;
  const bool with_tree = rows <= kTinyBatch;
  const bool want_mean = a.u.mean_weighted_loss != nullptr;
  // CTA 0 is the tree's: warp l owns level l, loads its nodes and groups its entries now.
  // CTAs 1..7 are the rows': warps 0..4 compute one row each (and stride on).
  TinyLoads tl;
  float prio = 0.f, weighted = 0.f;
  int my_row = -1;
  if (tree_cta) {
    if (a.count_copy != nullptr && threadIdx.x == 0) *a.count_copy = rows;
    if (a.loss_host != nullptr && threadIdx.x == 0)
      reinterpret_cast<int32_t *>(a.loss_host)[a.u.batch] = rows;
    if (with_tree) {
      // one word per row (two with the mean loss) will arrive
      if (threadIdx.x == 0) mbar_arrive_expect(&s_arrived, (uint32_t)rows * (want_mean ? 8u : 4u));
      tree_update_tiny_issue(a.tree, warp, lane, &tl);
    }
  } else if (STAGED) {
    if (stages) {
      prio = c51_post_staged_row(a, srow, rows, lane, zl, s_bestp[warp], s_sup[warp],
                                 reinterpret_cast<const float *>(logp_row));
      my_row = srow;
      if (want_mean) weighted = a.weighted[srow];
    }
  } else if (warp < kPostRowWarps) {
    const float pmin = a.u.sampling_probabilities ? *a.u.min_probability : INFINITY;
    for (int b = ((int)blockIdx.x - 1) * kPostRowWarps + warp; b < rows;
         b += (kPostClusterCtas - 1) * kPostRowWarps) {
      __syncwarp();  // (this warp's shared rows are free again)
      prio = c51_post_row(a, scratch, have_stats, b, rows, lane, pmin, s_bestp[warp],
                          s_sup[warp]);
      my_row = b;  // (with the tree riding along there are at most 32 rows: one per warp)
      if (want_mean) weighted = a.weighted[b];
    }
  }
  B2R_MARK_END(12);
  cluster_wait();
  if (!with_tree) {
    if (gated) pdl_acquire();
    return;
  }
  if (!tree_cta) {
    // the row's priority (and weighted loss) into CTA 0's shared memory, counted on its
    // mbarrier: no fence, no second barrier
    if (my_row >= 0 && lane == 0) {
      st_async_u32(&s_prio[my_row], __float_as_uint(prio), &s_arrived, 0);
      if (want_mean) st_async_u32(&s_weighted[my_row], __float_as_uint(weighted), &s_arrived, 0);
    }
    if (gated) pdl_acquire();
    return;
  }
  mbar_wait(&s_arrived, 0);
  const double v = (tl.in && !tl.use_max) ? (double)s_prio[lane] : 0.0;
  tree_update_tiny_finish(a.tree, warp, lane, tl, v);
  if (a.tree_done != nullptr && threadIdx.x == 0) *a.tree_done = 1u;
  B2R_MARK_END(9);
  if (want_mean && warp == 0) {
    // fixed order: row k in lane k, butterfly, as the other instances reduce
    float acc = lane < rows ? s_weighted[lane] : 0.f;
    acc = group_sum<32>(acc);
    if (lane == 0) *a.u.mean_weighted_loss = __fdiv_rn(acc, (float)rows);
  }
  if (gated) pdl_acquire();
}

float *g_weighted = nullptr;
unsigned int *g_ticket = nullptr;
int g_weighted_cap = 0;

}  // namespace
}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" {

int b2r_c51_project(int32_t batch, int32_t num_atoms, const float *supports,
                    const float *weights, const float *target_support, float *out,
                    b2r_stream stream) {
  if (batch <= 0 || num_atoms < 2)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "project_distribution needs batch > 0 and at least 2 atoms");
  const size_t smem = (size_t)b2r::kWarpsPerBlock * 2 * num_atoms * 4;
  if (smem > 48 * 1024)
    return fail(B2R_ERR_UNSUPPORTED, "num_atoms too large");
  const int blocks = (batch + b2r::kWarpsPerBlock - 1) / b2r::kWarpsPerBlock;
  b2r::c51_project_kernel<<<blocks, b2r::kWarpsPerBlock * 32, smem,
                            as_stream(stream)>>>(batch, num_atoms, supports,
                                                 weights, target_support, out);
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // extern "C"

namespace b2r {
int launch_loss(const b2r_c51_args *args, cudaStream_t s, const ShardedLoss &sh);
}  // namespace b2r

extern "C" {

int b2r_c51_loss(const b2r_c51_args *args, b2r_stream stream) {
  return b2r::launch_loss(args, as_stream(stream), b2r::ShardedLoss());
}

int b2r_c51_loss_sharded(const b2r_c51_args *args, b2r_exchange *exchange,
                         int32_t global_batch, b2r_stream stream) {
  if (!args) return fail(B2R_ERR_INVALID_ARGUMENT, "args is NULL");
  if (!args->batch_count)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a shard's loss needs batch_count");
  if (global_batch < 1) return fail(B2R_ERR_INVALID_ARGUMENT, "global_batch must be >= 1");
  if (args->sampling_probabilities && !args->min_probability)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "sampling_probabilities need the sampler's min_probability");
  if (!exchange) return fail(B2R_ERR_INVALID_ARGUMENT, "exchange is NULL");
  if (!exchange->connected)
    return fail(B2R_ERR_INVALID_ARGUMENT, "the exchange is not connected");
  b2r::ShardedLoss sh;
  sh.global_batch = global_batch;
  sh.world = exchange->world;
  sh.rank = exchange->rank;
  sh.mins = exchange->mailbox + b2r::kMinWordsOffset;
  sh.seq = exchange->seq;
  sh.timeout_ns = exchange->timeout_ns;
  sh.latched = exchange->latched;
  return b2r::launch_loss(args, as_stream(stream), sh);
}

}  // extern "C"

namespace b2r {

static int ensure_loss_scratch(int batch) {
  if (batch > g_weighted_cap) {
    if (g_weighted) cudaFree(g_weighted);
    g_weighted = nullptr;
    int cap = 4096;
    while (cap < batch) cap *= 2;
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&g_weighted), (size_t)cap * 4));
    g_weighted_cap = cap;
  }
  if (!g_ticket) {
    B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&g_ticket), 4));
    B2R_CUDA(cudaMemset(g_ticket, 0, 4));
  }
  return B2R_OK;
}

// ---- the loss in two halves (see c51_pre_kernel) ----
// Largest batch that splits.  Measured per step, one kernel against two halves
// (profiles/r2/README.md): 16.8 / 16.0 us at batch 32, 27.9 / 25.7 at 256, 39.5 / 37.1 at
// 1024 (deferred copies), but 111 / 119 at 4096, where the first half's 1024 CTAs take
// issue slots from the sampler that everything else waits for.
constexpr int kC51SplitMax = 2048;

bool c51_can_split(const b2r_c51_args *args) {
  return args->batch <= kC51SplitMax && args->num_atoms >= 2 &&
         args->num_atoms <= kRowAtoms && args->num_actions > 0;
}

int c51_scratch_floats_per_row() { return kPreRow; }

// The staged tail (c51_post_tree_kernel<true>) is the lean instance — no target, no
// gradient — over at most 32 rows, and keeps every action's log-probabilities of its five
// rows in shared memory (at most 40 KB: 32 actions x 64 atoms).
bool c51_tail_can_stage(const b2r_c51_args *args) {
  return args->batch <= kTinyBatch && args->batch_count == nullptr &&
         args->grad_logits == nullptr && args->target == nullptr &&
         args->num_actions <= 32 && args->num_atoms <= kRowAtoms;
}

// First half over `rows` rows of logits; scratch: device [rows][kPreRow] floats.  Sets
// *have_stats when the launch leaves the online softmax statistics in the scratch.
int c51_pre_launch(const b2r_c51_args *args, int rows, float *scratch, const PreSync &sync,
                   cudaStream_t s, int *have_stats, const float *online_src,
                   float *online_copy, const StageGate *stage) {
  if (!args || rows <= 0 || !scratch || !args->target_logits || !args->online_logits ||
      !args->support)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad C51 arguments");
  if (stage != nullptr && (rows >= 128 || !stage->first_half.done || !stage->logp))
    return fail(B2R_ERR_INVALID_ARGUMENT, "a staged first half covers fewer than 128 rows");
  PreArgs a;
  a.target_logits = args->target_logits;
  a.online_logits = online_src != nullptr ? online_src : args->online_logits;
  a.online_copy = online_copy;
  a.support = args->support;
  a.scratch = scratch;
  a.rows = rows;
  a.num_actions = args->num_actions;
  a.num_atoms = args->num_atoms;
  a.warps = args->num_actions < 32 ? args->num_actions : 32;
  a.sync = sync;
  a.logp = stage != nullptr ? stage->logp : nullptr;
  a.staged_done = stage != nullptr ? stage->first_half.done : nullptr;
  a.wait_late = stage != nullptr && stage->rows.done != nullptr ? 1 : 0;
  if (rows >= 128) {
    const dim3 grid((rows + kRowWarps - 1) / kRowWarps), block(kRowWarps * 32);
    if (args->num_atoms == 51)
      B2R_CUDA(launch(c51_pre_rows_kernel<8, 51>, grid, block, 0, s, a));
    else
      B2R_CUDA(launch(c51_pre_rows_kernel<8, 0>, grid, block, 0, s, a));
    *have_stats = 0;
  } else {
    B2R_CUDA(launch(c51_pre_kernel<2>, dim3(rows), dim3(a.warps * 32), 0, s, a));
    *have_stats = 1;
  }
  B2R_LAUNCHED();
  return B2R_OK;
}

// The tail over the sampled rows.
// expected_rows < 0: the host knows the rows (args->batch); else a shard's step, whose
// device-side count is expected to be about that many.
bool c51_post_takes_tree(const b2r_c51_args *args, const b2r_tree *tree,
                         int64_t expected_rows) {
  const bool counted = args->batch_count != nullptr;
  const bool small = counted ? (expected_rows >= 0 && expected_rows <= kTinyBatch &&
                                args->batch <= 256 && args->mean_weighted_loss == nullptr)
                             : args->batch <= kTinyBatch;
  return tree != nullptr && small && tree->depth + 1 <= 32 &&
         (args->sampling_probabilities == nullptr || args->min_probability != nullptr);
}

int c51_post_launch(const b2r_c51_args *args, const float *scratch, int have_stats,
                    cudaStream_t s, int64_t *err, int32_t *count_copy, b2r_tree *tree,
                    const int32_t *indices, unsigned int *tree_done,
                    const b2r_exchange *publish, float *loss_host, const TreeGo *go,
                    const StageGate *stage) {
  if (!args || args->batch <= 0 || !scratch)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad C51 shape");
  if (args->batch_count && args->mean_weighted_loss)
    return fail(B2R_ERR_UNSUPPORTED,
                "mean_weighted_loss cannot be combined with batch_count");
  if (!args->support || !args->online_logits || !args->actions || !args->rewards ||
      !args->terminals || !args->loss || !args->priorities)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a required C51 pointer is NULL");
  LossArgs a;
  a.u = *args;
  a.err = err;
  a.count_copy = count_copy;
  a.tree_done = nullptr;
  a.loss_host = loss_host;
  if (go != nullptr) a.go = *go;
  if (stage != nullptr) {
    if (tree == nullptr || !c51_tail_can_stage(args) || !stage->first_half.done ||
        !stage->first_half.tickets || !stage->logp)
      return fail(B2R_ERR_INVALID_ARGUMENT, "this tail cannot stage its inputs");
    a.stage = *stage;
  }
  a.warps = 0;
  B2R_TRY(ensure_loss_scratch(args->batch));
  a.weighted = g_weighted;
  a.ticket = g_ticket;
  if (tree != nullptr) {
    if (args->batch_count != nullptr && tree_done == nullptr)
      return fail(B2R_ERR_INVALID_ARGUMENT, "a counted batch needs the tree_done flag");
    set_tree_window(tree->heap, (size_t)tree->leaves * 16);
    a.tree_done = tree_done;
    a.tree.heap = tree->heap;
    a.tree.depth = tree->depth;
    a.tree.leaves = tree->leaves;
    a.tree.n = args->batch < kTinyBatch ? args->batch : kTinyBatch;
    a.tree.padded = 32;
    a.tree.indices = indices;
    a.tree.values = args->priorities;
    a.tree.mode = nullptr;
    a.tree.k_base = 0;
    a.tree.delta = tree->delta;
    a.tree.max_rec = tree->max_rec;
    a.tree.status = tree->status;
    a.tree.n_dev = args->batch_count;
    if (publish != nullptr && publish->world > 1 && publish->connected) {
      a.tree.publish = publish->args_dev;
      a.tree.publish_world = publish->world;
      a.tree.publish_rank = publish->rank;
    }
    int warps = tree->depth + 1;
    if (warps < kPostRowWarps) warps = kPostRowWarps;
    if (stage != nullptr) {
      const size_t smem = (size_t)kPostRowWarps *
                          c51_logp_stride(args->num_actions, args->num_atoms) * sizeof(float);
      B2R_CUDA(launch_prio_cluster(c51_post_tree_kernel<true>, dim3(kPostClusterCtas),
                                   dim3(warps * 32), smem, s, chain_priority(),
                                   kPostClusterCtas, a, scratch, have_stats));
    } else {
      B2R_CUDA(launch_prio_cluster(c51_post_tree_kernel<false>, dim3(kPostClusterCtas),
                                   dim3(warps * 32), 0, s, chain_priority(),
                                   kPostClusterCtas, a, scratch, have_stats));
    }
    B2R_LAUNCHED();
    return B2R_OK;
  }
  const dim3 grid((args->batch + kRowWarps - 1) / kRowWarps), block(kRowWarps * 32);
  B2R_CUDA(launch(c51_post_kernel, grid, block, 0, s, a, scratch, have_stats));
  B2R_LAUNCHED();
  return B2R_OK;
}

// From 128 rows up: one warp per row (c51_loss_rows_kernel).  Measured with 10 launches
// per graph (profiles/r1/README.md): at batch 32 the CTA-per-row kernel and a rows
// kernel tie (5.95 us), at 256 the rows kernel wins once the logits no longer sit in L2
// (10.2 -> 7.0 us).
constexpr int kC51RowsMin = 128;

int launch_loss(const b2r_c51_args *args, cudaStream_t s, const ShardedLoss &sh) {
  if (!args || args->batch <= 0 || args->num_atoms < 2 || args->num_actions <= 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad C51 shape");
  if (args->batch_count && args->mean_weighted_loss && sh.global_batch == 0)
    return fail(B2R_ERR_UNSUPPORTED,
                "mean_weighted_loss cannot be combined with batch_count");
  if (!args->support || !args->target_logits || !args->online_logits ||
      !args->actions || !args->rewards || !args->terminals || !args->loss ||
      !args->priorities)
    return fail(B2R_ERR_INVALID_ARGUMENT, "a required C51 pointer is NULL");
  b2r::LossArgs a;
  a.u = *args;
  a.sh = sh;
  a.err = nullptr;
  a.count_copy = nullptr;
  a.tree_done = nullptr;
  a.loss_host = nullptr;
  // Small batches are latency-bound: one warp per action.  Large batches are
  // throughput-bound: a third of that, so more rows are resident per SM.
  a.warps = args->num_actions < 32 ? args->num_actions : 32;
  if (args->batch > 256) a.warps = (a.warps + 2) / 3;
  const int threads = a.warps * 32;
  const size_t smem = ((size_t)a.warps + 5) * args->num_atoms * sizeof(float);
  if (smem > 48 * 1024 || args->num_atoms > 32 * b2r::kMaxAtomsPerLane)
    return fail(B2R_ERR_UNSUPPORTED, "num_atoms above 128 is not supported");
  B2R_TRY(ensure_loss_scratch(args->batch));
  a.weighted = b2r::g_weighted;
  a.ticket = b2r::g_ticket;
  if (args->batch >= kC51RowsMin && args->num_atoms <= b2r::kRowAtoms) {
    const int blocks = (args->batch + b2r::kRowWarps - 1) / b2r::kRowWarps;
    const dim3 grid(blocks), block(b2r::kRowWarps * 32);
    if (args->num_atoms == 51)
      B2R_CUDA(b2r::launch(b2r::c51_loss_rows_kernel<8, 51>, grid, block, 0, s, a));
    else
      B2R_CUDA(b2r::launch(b2r::c51_loss_rows_kernel<8, 0>, grid, block, 0, s, a));
    B2R_LAUNCHED();
    return B2R_OK;
  }
  if (args->num_atoms <= 64)
    B2R_CUDA(b2r::launch(b2r::c51_loss_kernel<2>, dim3(args->batch), dim3(threads), smem,
                         s, a));
  else
    B2R_CUDA(b2r::launch(b2r::c51_loss_kernel<4>, dim3(args->batch), dim3(threads), smem,
                         s, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // namespace b2r

#ifdef B2R_TRACE
extern "C" int b2r_debug_trace_c51(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_trace, sizeof(long long) * 32);
}
#endif
