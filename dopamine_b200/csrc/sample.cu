// Index sampling: replaces sample_index_batch of OutOfGraphReplayBuffer
// (circular_replay_buffer.py:436-477) and OutOfGraphPrioritizedReplayBuffer
// (prioritized_replay_buffer.py:142-171), incl. SumTree.stratified_sample
// (sum_tree.py:143-166).
//
// A batch is at most a few thousand independent root-to-leaf descents (20 dependent
// fp64 loads each at capacity 1M): one CTA up to 256 strata, tiles of 128 strata over
// many CTAs above.  The sequential parts of the reference — "the j-th invalid slot
// takes the j-th valid retry draw", "stop after max_sample_attempts failures" — become
// block-wide prefix scans (warp ballots + shuffles) over windows evaluated
// speculatively in parallel, by the last CTA to finish.  Levels 0..10 of the tree are
// staged in shared memory first.  The prioritized kernel can also write the scalar
// columns of the batch (gather.cuh) and exchange shard totals over peer memory.
#include "gather.cuh"

#include <cooperative_groups.h>

#include <cstddef>
#include <cstdlib>
#include <cstring>

namespace cg = cooperative_groups;

namespace b2r {
namespace {

B2R_TRACE_DECL

constexpr int kMaxTiles = 2048;  // batch / tile size (>= 32 strata per tile)

struct PerSampleArgs {
  const double *heap;
  int depth;
  const ValidCtx *valid_dev;  // the buffer's device validity context
  int batch;          // strata (global batch when sharded)
  int max_attempts;
  // uniforms: host-provided (reference RNG stream) or Philox (throughput mode)
  int use_philox;
  uint64_t seed, offset;
  uint64_t *counter;            // nullable: device draw counter added to offset
  uint32_t zero;                // always 0 (see descend_levels)
  const double *strat_query01;  // [batch]  final query values in [0,1]
  const double *retry_u01;      // [max_attempts]
  // outputs
  int32_t *out_idx;
  int32_t *inv_slots;  // scratch [n_tiles * tile_size]: per-tile invalid slots
  int32_t *tile_counts;        // scratch [n_tiles]
  unsigned int *ticket;        // scratch: CTAs finished (self-resetting)
  int32_t *info;       // [0] status, [1] fail slot, [2] retry draws used, [3] count
  int64_t *latched;    // nullable: asynchronous error latch
  // sharding (num_shards == 1: plain buffer)
  int num_shards, rank;
  const double *shard_totals;
  int32_t *out_slots;  // nullable
  // fused scalar outputs (with_scalars): every row's n-step return, terminal,
  // actions, ... are written here as soon as its index is final, and the minimum
  // sampling probability of the batch (the IS-weight normaliser) is reduced.
  int with_scalars;
  ScalarArgs sc;
  float *tile_min;      // scratch [n_tiles]
  float *min_prob_out;  // nullable
  int32_t *count_out;   // nullable: number of rows this launch produced
  // Sharded + Philox + large batch: stratified queries grow with the stratum index
  // and the rank-order scan is monotone, so a rank's strata are ONE index range
  // [lo, hi).  Every CTA finds the range with a parallel k-ary search and then works
  // on a tile of it: the sharded sampler scales over CTAs like the plain one.
  int shard_ranges;
  // Shard totals over peer memory instead of shard_totals (see exchange_totals).
  ExchangeArgs xchg;
  // 1.0 / batch as IEEE double division gives it (np.linspace's step), computed on the
  // host: an fp64 division is a ~500-cycle subroutine on the device.
  double step;
  // Fused step: the first half of the C51 loss runs beside this kernel; the closing
  // thread waits for it before the kernel ends (PreSync; done == nullptr: nothing to wait
  // for).
  PreSync pre;
  // Rows the caller's outputs hold (a sharded step sizes them by a bound on its share of
  // the global batch): rows beyond it are dropped and B2R_ERR_UNSUPPORTED is latched.
  int out_cap;
  // Exchange mode: the closing thread also stores min_prob_out's value into every peer's
  // mailbox for this step (b2r_sample_transition_batch_sharded_device).
  int publish_min;
  // nullable: StageGate::rows.done of the one-stream step (replay.cuh), counted by the closing
  // thread when rows, minimum and counters are final.  The kernel then lets its dependents
  // launch only after its own griddepcontrol.wait.
  unsigned int *rows_done;
};

// The local minimum of step `seq`, for the peers' sharded loss (b2r_c51_loss_sharded).
__device__ __forceinline__ void publish_local_min(const PerSampleArgs &a, bool exchange,
                                                  float m, uint64_t seq) {
  if (a.publish_min && exchange) exchange_publish_min(a.xchg, a.num_shards, a.rank, m, seq);
}

// Receiving half of the all-gather of shard totals (tree.cuh: exchange_publish): thread g
// polls this rank's mailbox for rank g's total of step `seq`.  A peer that does not answer
// within the timeout latches B2R_ERR_EXCHANGE (and later launches skip the wait), so a
// lost rank cannot hang the GPU.
// The sampler's sending half: nothing to do when the kernel that last changed the tree
// has published this step's total already (its bits must then be the root's: anything
// else changed the tree behind the publisher's back, and the ranks would apportion the
// batch from different totals — latched as B2R_ERR_STALE_TOTAL).
__device__ __forceinline__ void exchange_publish_if_needed(const ExchangeArgs &x, int world,
                                                           int rank, double local_total,
                                                           uint64_t seq, int64_t *latched) {
  if (x.pub != nullptr && x.pub[0] == seq) {
    if ((threadIdx.x & 31) == rank && x.pub[1] != (uint64_t)__double_as_longlong(local_total) &&
        latched != nullptr && latched[0] == 0) {
      latched[0] = B2R_ERR_STALE_TOTAL;
      latched[1] = rank;
    }
    return;
  }
  exchange_publish(x, world, rank, local_total, seq);
}

__device__ __forceinline__ void exchange_collect(const ExchangeArgs &x, int world,
                                                 int rank, double local_total,
                                                 uint64_t seq, double *totals,
                                                 int64_t *latched) {
  const int g = threadIdx.x;
  if (g >= world) return;
  double got = local_total;
  if (g != rank && x.timeout_ns > 0) {
    const uint32_t tag = (uint32_t)seq;
    const uint64_t *src = x.local + ((size_t)(seq & 1) * world + g) * 2;
    const bool broken = latched != nullptr && latched[0] == B2R_ERR_EXCHANGE;
    const uint64_t t0 = global_timer_ns();
    uint64_t r0 = 0, r1 = 0;
    bool ok = false;
    while (!broken) {
      r0 = ld_sys_u64(src);
      r1 = ld_sys_u64(src + 1);
      ok = (uint32_t)r0 == tag && (uint32_t)r1 == tag;
      if (ok || global_timer_ns() - t0 > (uint64_t)x.timeout_ns) break;
    }
    if (ok) {
      got = __longlong_as_double((long long)((r0 & 0xffffffff00000000ull) | (r1 >> 32)));
    } else {
      got = 0.0;
      if (latched != nullptr) {
        latched[0] = B2R_ERR_EXCHANGE;
        latched[1] = g;
      }
    }
  }
  totals[g] = got;
}

// Block-wide minimum; every thread of the block must call it.
__device__ __forceinline__ float block_min(float v, float *scratch) {
#pragma unroll 1
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float m = INFINITY;
  const int warps = (blockDim.x + 31) >> 5;
  for (int w = 0; w < warps; ++w) m = fminf(m, scratch[w]);
  return m;
}

// Slot of the ord-th invalid stratum: the per-tile lists are concatenated in tile
// order (tile_start[] is the exclusive prefix of the per-tile counts).
__device__ __forceinline__ int invalid_slot(const PerSampleArgs &a, const int *tile_start,
                                            int n_tiles, int tile_size, int ord) {
  int t = 0;
  while (t + 1 < n_tiles && tile_start[t + 1] <= ord) ++t;
  return a.inv_slots[(size_t)t * tile_size + (ord - tile_start[t])];
}

// grid = 1 CTA (small batches, sharded sampling) or one CTA per tile of blockDim
// strata (large batches).  The stratified picks are independent; what the
// reference does sequentially — the j-th invalid slot takes the j-th valid retry
// draw out of a shared budget — is done by the last CTA to finish, on per-tile
// ordered lists of invalid slots, with block-wide prefix scans over windows of
// retry draws evaluated speculatively in parallel.
template <int K, int MAX_THREADS>
__global__ void __launch_bounds__(MAX_THREADS) per_sample_kernel(const __grid_constant__ PerSampleArgs a) {
  __shared__ double top[2 << kTopLevels];
  __shared__ int warp_counts[32];
  __shared__ float warp_mins[32];
  __shared__ double s_totals[kMaxShards];
  __shared__ int s_first[2];
  __shared__ int s_draws_used, s_last_idx, s_last_valid;
  __shared__ bool s_is_last;
  __shared__ int tile_start[kMaxTiles + 1];

  __shared__ ValidCtx s_valid;
  const ValidCtx &valid_ctx = s_valid;

  B2R_MARK(0);
  pdl_release();
  pdl_acquire();
  B2R_MARK(1);
  // validity context: from HBM (it moves with every add), visible after the
  // barrier inside stage_top_levels
  for (int w = threadIdx.x; w < (int)(sizeof(ValidCtx) / 8); w += blockDim.x)
    reinterpret_cast<uint64_t *>(&s_valid)[w] =
        reinterpret_cast<const uint64_t *>(a.valid_dev)[w];
  const uint64_t draws_before = a.counter ? *a.counter : 0ull;
  const uint64_t draw_offset = a.offset + draws_before;
  // Peer exchange (one CTA): the totals are on the wire while the top levels are
  // staged.
  const bool exchange = a.xchg.local != nullptr && a.num_shards > 1;
  uint64_t xseq = 0;
  if (exchange) {
    xseq = *a.xchg.seq + 1;
    if (blockIdx.x == 0 && threadIdx.x < 32)
      exchange_publish_if_needed(a.xchg, a.num_shards, a.rank, a.heap[1], xseq, a.latched);
  }
  const int top_depth = stage_top_levels(a.heap, a.depth, top);
  B2R_MARK(2);
  const double local_total = top[1];  // root of the 1-based heap
  // The first tile's uniforms need no totals: drawn while the peers' totals travel.
  const int first_i = blockIdx.x * blockDim.x + threadIdx.x;
  double first_u = 0.0;
  if (a.use_philox && first_i < a.batch)
    first_u = philox_uniform53(a.seed, draw_offset, (uint64_t)first_i);
  const double *shard_totals = a.shard_totals;
  if (exchange) {
    exchange_collect(a.xchg, a.num_shards, a.rank, local_total, xseq, s_totals,
                     a.latched);
    __syncthreads();
    shard_totals = s_totals;
  }
  // Mass the strata are spread over: the root, or all shards' roots summed in
  // rank order (fp64, left to right).
  double grand_total = local_total;
  if (a.num_shards > 1) {
    grand_total = 0.0;
    for (int g = 0; g < a.num_shards; ++g)
      grand_total = __dadd_rn(grand_total, shard_totals[g]);
  }
  if (grand_total == 0.0 || (a.num_shards == 1 && local_total == 0.0)) {
    // sum_tree.py:159-160 (every CTA takes this branch together; the last one to
    // arrive advances the step counters, which every CTA read on entry)
    if (threadIdx.x == 0 && (gridDim.x == 1 || arrive_last(a.ticket))) {
      a.info[0] = B2R_ERR_EMPTY_TREE;
      a.info[1] = 0; a.info[2] = 0; a.info[3] = 0;
      if (a.count_out) *a.count_out = 0;
      if (a.min_prob_out) *a.min_prob_out = INFINITY;
      publish_local_min(a, exchange, INFINITY, xseq);
      if (a.counter) *a.counter = draws_before + 1;  // ranks stay in lockstep
      pre_sync_consume(a.pre);
      if (exchange) *a.xchg.seq = xseq;
      if (a.latched && a.latched[0] == 0) a.latched[0] = B2R_ERR_EMPTY_TREE;
    }
    return;
  }
  if (threadIdx.x == 0) {
    s_draws_used = 0;
    s_last_idx = -1;
    s_last_valid = 0;
  }

  // ---- stratified pass (sum_tree.py:162-166 + prioritized_replay_buffer.py:155)
  const int tile_size = blockDim.x;
  const double step = 1.0 / (double)a.batch;  // np.linspace(0, 1, batch + 1)
  // Owner of stratum i under the rank-order scan (ST:128-139 applied to the shard
  // totals) and the mass left inside the owning shard.
  auto stratum_owner = [&](int i, double u, double *residual) {
    double q01;
    if (a.use_philox) {
      const double lo = __dmul_rn((double)i, step);
      const double hi = (i + 1 == a.batch) ? 1.0 : __dmul_rn((double)(i + 1), step);
      q01 = __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u));  // random.uniform
    } else {
      q01 = a.strat_query01[i];
    }
    double mass = __dmul_rn(q01, grand_total);
    int owner = 0;
    for (; owner < a.num_shards - 1; ++owner) {
      const double left = shard_totals[owner];
      if (mass < left) break;
      mass = __dsub_rn(mass, left);
    }
    *residual = mass;
    return owner;
  };
  // This rank's strata: everything, or (shard_ranges) the range [lo, hi) found by two
  // simultaneous k-ary searches for the first stratum owned by a rank >= ours and the
  // first owned by a rank > ours; blockDim candidates per round.
  int range_lo = 0, range_hi = a.batch;
  if (a.shard_ranges) {
    int base[2] = {0, 0}, limit[2] = {a.batch, a.batch};
    while (base[0] < limit[0] || base[1] < limit[1]) {
      if (threadIdx.x < 2) s_first[threadIdx.x] = tile_size;
      __syncthreads();
      int cand[2], stride[2];
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        const int width = limit[w] - base[w];
        stride[w] = (width + tile_size - 1) / tile_size;
        cand[w] = base[w] + (int)threadIdx.x * stride[w];
        if (width > 0) {
          bool hit = cand[w] >= limit[w];  // at or past the known upper bound
          if (!hit) {
            double unused;
            const int owner = stratum_owner(
                cand[w], philox_uniform53(a.seed, draw_offset, (uint64_t)cand[w]),
                &unused);
            hit = w == 0 ? owner >= a.rank : owner > a.rank;
          }
          if (hit) atomicMin(&s_first[w], (int)threadIdx.x);
        }
      }
      __syncthreads();
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        if (base[w] >= limit[w]) continue;
        const int t = s_first[w];  // first candidate that satisfies the predicate
        const int hit = base[w] + t * stride[w];
        const int new_limit = hit < limit[w] ? hit : limit[w];
        // the answer lies in (previous candidate, new_limit]
        base[w] = t == 0 ? new_limit : base[w] + (t - 1) * stride[w] + 1;
        if (base[w] > new_limit) base[w] = new_limit;
        limit[w] = new_limit;
      }
      __syncthreads();
    }
    range_lo = base[0];
    range_hi = base[1];
  }
  const int n_all = range_hi - range_lo;
  // strata walked by this launch's tiles (shard_ranges: at most the output capacity)
  const int n_mine = a.shard_ranges && n_all > a.out_cap ? a.out_cap : n_all;
  const int n_tiles = (n_mine + tile_size - 1) / tile_size;
  range_hi = range_lo + n_mine;
  int mine_base = 0;  // running output position (single-CTA sharded mode)
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int i = range_lo + tile * tile_size + threadIdx.x;
    bool mine = false, valid = true;
    int64_t idx = 0;
    ScalarLoads row;
    const bool fast_scalars = a.with_scalars && a.sc.fast;
    if (i < range_hi) {
      double u = 0.0;
      if (a.use_philox)
        u = i == first_i ? first_u : philox_uniform53(a.seed, draw_offset, (uint64_t)i);
      double mass;
      const int owner = stratum_owner(i, u, &mass);
      mine = (owner == a.rank);
      B2R_MARK(3);
      if (mine) {
        idx = tree_descend_staged<K>(a.heap, top, top_depth, a.depth, mass, a.zero);
        B2R_MARK(4);
        // the row's scalar inputs travel with the validity flags: one round trip
        if (fast_scalars) load_scalars(a.sc, idx, &row);
        valid = is_valid_transition(valid_ctx, idx);
        B2R_MARK(5);
      }
    }
    int pos = i - range_lo, tile_mine = 0, tile_inv;
    if (a.num_shards > 1 && !a.shard_ranges) {  // compact (grid is 1 CTA here)
      pos = mine_base + block_scan_flag(mine, warp_counts, &tile_mine);
      mine_base += tile_mine;
      if (pos >= a.out_cap) mine = false;  // beyond the outputs: dropped, latched below
    }
    // The usual case of the agent's batch — one CTA, one tile, every pick valid —
    // needs none of the machinery below (slot lists, ticket, retries): one barrier
    // says so, the rows are written and thread 0 closes the launch.
    if (gridDim.x == 1 && n_tiles == 1 && __syncthreads_or(mine && !valid) == 0) {
      float row_prio = INFINITY;
      if (mine) {
        a.out_idx[pos] = (int32_t)idx;
        if (a.out_slots) a.out_slots[pos] = i;
        if (fast_scalars) row_prio = finish_scalars(a.sc, pos, idx, row);
        else if (a.with_scalars) row_prio = write_scalars(a.sc, pos, idx);
      }
      const bool want_min = a.with_scalars && a.min_prob_out != nullptr;
      const float m = want_min ? block_min(row_prio, warp_mins) : INFINITY;
      if (threadIdx.x == 0) {
        const int all = a.shard_ranges ? n_all : (a.num_shards > 1 ? mine_base : a.batch);
        const int rows = all < a.out_cap ? all : a.out_cap;
        if (a.counter) *a.counter = draws_before + 1;
        if (exchange) *a.xchg.seq = xseq;
        a.info[0] = all > rows ? B2R_ERR_UNSUPPORTED : B2R_OK;
        a.info[1] = 0;
        a.info[2] = 0;
        a.info[3] = rows;
        if (a.count_out) *a.count_out = rows;
        if (want_min) *a.min_prob_out = m;
        if (want_min) publish_local_min(a, exchange, m, xseq);
        if (all > rows && a.latched && a.latched[0] == 0) {  // the share outgrew the buffers
          a.latched[0] = B2R_ERR_UNSUPPORTED;
          a.latched[1] = all;
        }
        pre_sync_consume(a.pre);
      }
      B2R_MARK(8);
      return;
    }
    const int ipos = block_scan_flag(mine && !valid, warp_counts, &tile_inv);
    float my_prio = INFINITY;
    if (mine) {
      a.out_idx[pos] = (int32_t)idx;
      if (a.out_slots) a.out_slots[pos] = i;
      if (!valid) a.inv_slots[(size_t)tile * tile_size + ipos] = pos;
      else if (fast_scalars) my_prio = finish_scalars(a.sc, pos, idx, row);
      else if (a.with_scalars) my_prio = write_scalars(a.sc, pos, idx);
    }
    if (a.with_scalars) {
      const float m = block_min(my_prio, warp_mins);
      if (threadIdx.x == 0) a.tile_min[tile] = m;
    }
    if (threadIdx.x == 0) a.tile_counts[tile] = tile_inv;
  }
  B2R_MARK(6);
  const int count_all = a.shard_ranges ? n_all : (a.num_shards > 1 ? mine_base : a.batch);
  const int count = count_all < a.out_cap ? count_all : a.out_cap;

  // ---- only the last CTA to finish goes on
  if (gridDim.x > 1) {
    if (!last_cta(a.ticket, &s_is_last, false)) return;
  } else {
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    int run = 0;
    for (int t = 0; t < n_tiles; ++t) {
      tile_start[t] = run;
      run += *(volatile int *)(a.tile_counts + t);
    }
    tile_start[n_tiles] = run;
    if (gridDim.x > 1) *a.ticket = 0u;  // ready for the next launch
  }
  __syncthreads();
  const int num_invalid = tile_start[n_tiles];
  B2R_MARK(7);

  // ---- in-order replacement of invalid slots (prioritized_replay_buffer.py:156-170)
  int found = 0, drawn = 0;
  float fix_min = INFINITY;  // sampling probabilities of the rows replaced below
  const int budget = a.max_attempts;
  while (num_invalid > 0 && found < num_invalid && drawn < budget) {
    const int r = drawn + threadIdx.x;
    const bool active = r < budget;
    bool valid = false;
    int64_t idx = 0;
    ScalarLoads row;
    const bool fast_scalars = a.with_scalars && a.sc.fast;
    if (active) {
      // Philox retry stream: rank-private (strata streams are shared by all ranks)
      const double u = (a.use_philox || a.retry_u01 == nullptr)
                           ? philox_uniform53(a.seed + 0x9E3779B97F4A7C15ull * (uint64_t)(a.rank + 1),
                                              draw_offset,
                                              (uint64_t)a.batch + (uint64_t)r)
                           : a.retry_u01[r];
      // sum_tree.py:123-124: query = random.random() * total
      idx = tree_descend_staged<K>(a.heap, top, top_depth, a.depth,
                                   __dmul_rn(u, local_total), a.zero);
      if (fast_scalars) load_scalars(a.sc, idx, &row);
      valid = is_valid_transition(valid_ctx, idx);
    }
    int tile_valid;
    const int ord = found + block_scan_flag(active && valid, warp_counts, &tile_valid);
    if (active && valid && ord < num_invalid) {
      const int slot = invalid_slot(a, tile_start, n_tiles, tile_size, ord);
      a.out_idx[slot] = (int32_t)idx;
      if (fast_scalars)
        fix_min = fminf(fix_min, finish_scalars(a.sc, slot, idx, row));
      else if (a.with_scalars)
        fix_min = fminf(fix_min, write_scalars(a.sc, slot, idx));
      if (ord == num_invalid - 1) s_draws_used = r + 1;
    }
    if (active && r == budget - 1) {
      s_last_idx = (int)idx;
      s_last_valid = valid ? 1 : 0;
    }
    found += tile_valid;
    drawn += blockDim.x;
    __syncthreads();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int status = B2R_OK, fail_slot = 0, used = 0;
    if (num_invalid > 0) {
      if (found >= num_invalid) {
        used = s_draws_used;
      } else {
        // Every one of the `budget` draws was consumed; `found` slots were fixed.
        used = budget;
        const int next = found;  // first invalid slot still unresolved
        const int next_slot = invalid_slot(a, tile_start, n_tiles, tile_size, next);
        if (budget == 0 || s_last_valid) {
          // budget already 0 when this slot is reached -> PRB:159-163
          status = B2R_ERR_SAMPLE_ATTEMPTS;
          fail_slot = next_slot;
        } else {
          // the slot burnt the rest of the budget and keeps its last (invalid)
          // draw; only a FURTHER invalid slot raises (SURVEY.md Q10).
          a.out_idx[next_slot] = s_last_idx;
          if (a.with_scalars && s_last_idx >= 0 && s_last_idx < valid_ctx.capacity)
            fix_min = fminf(fix_min, write_scalars(a.sc, next_slot, s_last_idx));
          if (num_invalid > next + 1) {
            status = B2R_ERR_SAMPLE_ATTEMPTS;
            fail_slot = invalid_slot(a, tile_start, n_tiles, tile_size, next + 1);
          }
        }
      }
    }
    const bool outgrew = count_all > count && status == B2R_OK;
    if (outgrew) status = B2R_ERR_UNSUPPORTED;  // a sharded step outgrew its buffers
    if (a.counter) *a.counter = draws_before + 1;
    if (exchange) *a.xchg.seq = xseq;
    a.info[0] = status;
    a.info[1] = outgrew ? count_all
                        : (a.out_slots ? (status ? a.out_slots[fail_slot] : 0) : fail_slot);
    if (outgrew) fail_slot = count_all;
    a.info[2] = used;
    a.info[3] = count;
    if (a.count_out) *a.count_out = count;
    if (status != B2R_OK && a.latched && a.latched[0] == 0) {
      a.latched[0] = status;
      a.latched[1] = fail_slot;
    }
  }
  if (a.with_scalars && a.min_prob_out) {
    float m = block_min(fix_min, warp_mins);
    if (threadIdx.x == 0) {
      for (int t = 0; t < n_tiles; ++t)
        m = fminf(m, *(volatile float *)(a.tile_min + t));
      *a.min_prob_out = m;
      publish_local_min(a, exchange, m, xseq);
    }
  }
  if (threadIdx.x == 0) pre_sync_consume(a.pre);
  B2R_MARK(8);
}

// ---- warp-per-stratum sampler -------------------------------------------------------
// The kernel above gives a stratum to a THREAD and stages tree levels 0..10 in shared
// memory first (one DRAM/L2 round trip, 3.2 k cycles, before any descent starts), then
// walks three levels per round trip.  Here a stratum belongs to a WARP
// (tree_descend_warp: five levels per round trip, nothing staged, the first round's
// nodes fetched with the prologue), and the replacement draws for invalid picks are
// evaluated SPECULATIVELY by extra warps of the same grid, so that the last CTA to
// finish only has to match the j-th invalid slot with the j-th valid draw.  A batch of B
// strata is B warps spread over B / warps-per-CTA CTAs: the sampler's latency is that of
// ONE descent whatever the batch — three dependent L2 round trips for a 1M-leaf tree.
//
// The validity context (ValidCtx, 70 words) is read by the warp as 3 coalesced words
// per lane and stays in registers: scalars come out by shuffle, `index in
// invalid_range` is one compare per lane and a vote.
constexpr int kCtxWords = (int)(sizeof(ValidCtx) / 8);
static_assert(sizeof(ValidCtx) == 560 && offsetof(ValidCtx, invalid) == 40 &&
              offsetof(ValidCtx, term_flag) == 552 && offsetof(ValidCtx, stack) == 24 &&
              offsetof(ValidCtx, n_invalid) == 32,
              "WarpCtx picks ValidCtx fields by word");

struct WarpCtx {
  uint64_t w[3];  // words lane, lane + 32, lane + 64 of the ValidCtx image
  int64_t capacity, add_count, cursor;
  int stack, horizon, n_invalid;
  const uint8_t *term_flag;
};

__device__ __forceinline__ void warp_ctx_issue(const ValidCtx *src, int lane, WarpCtx *c) {
  const uint64_t *p = reinterpret_cast<const uint64_t *>(src);
#pragma unroll
  for (int r = 0; r < 3; ++r)
    c->w[r] = lane + 32 * r < kCtxWords ? p[lane + 32 * r] : 0ull;
}

__device__ __forceinline__ void warp_ctx_finish(WarpCtx *c) {
  const unsigned full = 0xffffffffu;
  c->capacity = (int64_t)__shfl_sync(full, c->w[0], 0);
  c->add_count = (int64_t)__shfl_sync(full, c->w[0], 1);
  c->cursor = (int64_t)__shfl_sync(full, c->w[0], 2);
  const uint64_t sh = __shfl_sync(full, c->w[0], 3);
  c->stack = (int)(uint32_t)sh;
  c->horizon = (int)(uint32_t)(sh >> 32);
  c->n_invalid = (int)(uint32_t)__shfl_sync(full, c->w[0], 4);
  c->term_flag = reinterpret_cast<const uint8_t *>(__shfl_sync(full, c->w[2], 5));
}

// is_valid_transition (circular_replay_buffer.py:381-414) by a warp; the same answer in
// every lane.
__device__ __forceinline__ bool warp_is_valid(const WarpCtx &c, int64_t index, int lane) {
  if (index < 0 || index >= c.capacity) return false;
  bool ok = true;
  if (c.add_count < c.capacity)  // not full
    ok = index < c.cursor - c.horizon && index >= c.stack - 1;
  bool bad = false;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int k = lane + 32 * r - 5;  // invalid[k] is word 5 + k
    bad = bad || (k >= 0 && k < c.n_invalid && (int64_t)c.w[r] == index);
  }
  // get_terminal_stack(index)[:-1].any()
  for (int k = lane + 1; k < c.stack; k += 32) {
    int64_t s = index - k;
    if (s < 0) s += c.capacity;
    bad = bad || c.term_flag[s] != 0;
  }
  return ok && !__any_sync(0xffffffffu, bad);
}

// Thread-per-draw descent from the root with nothing staged (the rare later rounds of
// the retry loop); out of line so that its registers do not burden the warp path.
static __device__ __noinline__ int64_t descend_from_root(const double *heap, int depth,
                                                         double q, uint32_t zero) {
  return tree_descend_staged<3>(heap, nullptr, 0, depth, q, zero);
}

constexpr int kSpecMax = 64;  // speculative replacement draws per launch

// Scratch of the warp sampler (carved out of b2r_buffer::inv_slots by the host).
struct WarpScratch {
  uint8_t *inv_flag;    // [cap, padded to 16]: 1 = the stratified pick of this position
                        // is invalid
  int32_t *inv_list;    // [cap]: positions of the invalid picks in order (last CTA)
  int32_t *spec_idx;    // [kSpecMax]: leaf of replacement draw r
  int32_t *spec_valid;  // [kSpecMax]: 1 = that leaf is a valid transition
  float *cta_min;       // [grid]: smallest sampling probability a CTA wrote
  int cap;              // rows the caller's outputs hold
  int spec;             // replacement draws evaluated up front (0: none)
  int cluster;          // the grid is one thread-block cluster (host-side switch)
};

// grid = ceil((strata + spec) / warps per CTA) CTAs (sharded: an estimate of this rank's
// share; the warps stride over whatever the share turns out to be).
//
// CLUSTER (batches of a few dozen strata, the agent's batch of 32): the whole grid is
// ONE thread-block cluster.  Flags, speculative draws and minima go straight into the
// shared memory of CTA 0 (distributed shared memory) and a cluster barrier replaces the
// fence + atomic ticket + L2 round trip by which the last CTA of a plain grid finds out
// that it is the last: ~0.6 k instead of ~3 k cycles on the critical path.
constexpr int kClusterCap = 1024;  // output rows a clustered launch can flag in smem

template <bool CLUSTER, typename T>
__device__ __forceinline__ T ld_scratch(const T *p) {
  if (CLUSTER) return *p;  // shared memory of this CTA
  return __ldcg(p);
}

template <int MIN_CTAS, bool CLUSTER>
__global__ void __launch_bounds__(256, MIN_CTAS)
per_sample_warp_kernel(const __grid_constant__ PerSampleArgs a,
                       const __grid_constant__ WarpScratch ws_in) {
  __shared__ __align__(16) uint8_t s_flag[CLUSTER ? kClusterCap : 16];
  __shared__ uint32_t s_flag32[CLUSTER ? kClusterCap : 1];  // as the words arrive
  __shared__ int s_cl_spec_idx[kSpecMax], s_cl_spec_valid[kSpecMax];
  __shared__ float s_cl_min[16];
  __shared__ __align__(8) uint64_t s_arrived;  // CLUSTER: mbarrier of CTA 0
  WarpScratch ws = ws_in;
  if (CLUSTER) {
    // Everybody's flags, speculative draws and minima go into CTA 0's shared memory as
    // 32-bit words sent with st.async and counted on CTA 0's mbarrier: CTA 0 waits for the
    // bytes it expects, nobody fences (common.cuh).  The relaxed barrier only keeps the
    // senders behind the mbarrier's initialisation; it is waited for where the first
    // word is sent, a microsecond later.
    if (blockIdx.x == 0 && threadIdx.x == 0) mbar_init(&s_arrived, 1);
    cluster_arrive_relaxed();
  }
  __shared__ double s_totals[kMaxShards];
  __shared__ int s_first[2];
  __shared__ float s_wmin[8];
  __shared__ int warp_counts[32];
  __shared__ float warp_mins[32];
  __shared__ int s_draw_of[kSpecMax], s_spec_idx[kSpecMax];
  __shared__ int s_draws_used, s_last_idx, s_last_valid;
  __shared__ bool s_is_last;
  __shared__ ValidCtx s_valid;  // thread-per-draw retry rounds only

  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int warps = blockDim.x >> 5;
  B2R_MARK(10);
  if (a.rows_done == nullptr) pdl_release();
  pdl_acquire();
  if (a.rows_done != nullptr) pdl_release();
  B2R_MARK(11);
  // every load of the prologue is issued before the first one is used; the nodes of
  // the first descent round (levels 1..5 under the root) ride along
  WarpCtx ctx;
  warp_ctx_issue(a.valid_dev, lane, &ctx);
  const uint64_t draws_before = a.counter ? *a.counter : 0ull;
  const bool exchange = a.xchg.local != nullptr && a.num_shards > 1;
  uint64_t xseq = 0;
  if (exchange) xseq = *a.xchg.seq + 1;
  const double local_total = a.heap[1];  // root of the 1-based heap
  double c_top = warp_candidate(a.heap, 1, a.depth < 5 ? a.depth : 5, lane);
  const uint64_t draw_offset = a.offset + draws_before;
  if (exchange && blockIdx.x == 0 && threadIdx.x < 32)
    exchange_publish_if_needed(a.xchg, a.num_shards, a.rank, local_total, xseq, a.latched);
  const double *shard_totals = a.shard_totals;
  if (exchange) {
    exchange_collect(a.xchg, a.num_shards, a.rank, local_total, xseq, s_totals,
                     a.latched);
    __syncthreads();
    shard_totals = s_totals;
  }
  warp_ctx_finish(&ctx);
  B2R_MARK(12);
  double grand_total = local_total;
  if (a.num_shards > 1) {
    grand_total = 0.0;
    for (int g = 0; g < a.num_shards; ++g)
      grand_total = __dadd_rn(grand_total, shard_totals[g]);
  }
  if (grand_total == 0.0 || (a.num_shards == 1 && local_total == 0.0)) {
    // sum_tree.py:159-160; every CTA takes this branch, the last to arrive closes
    if (threadIdx.x == 0 &&
        (CLUSTER ? blockIdx.x == 0 : (gridDim.x == 1 || arrive_last(a.ticket)))) {
      a.info[0] = B2R_ERR_EMPTY_TREE;
      a.info[1] = 0; a.info[2] = 0; a.info[3] = 0;
      if (a.count_out) *a.count_out = 0;
      if (a.min_prob_out) *a.min_prob_out = INFINITY;
      publish_local_min(a, exchange, INFINITY, xseq);
      if (a.counter) *a.counter = draws_before + 1;
      if (exchange) *a.xchg.seq = xseq;
      if (a.latched && a.latched[0] == 0) a.latched[0] = B2R_ERR_EMPTY_TREE;
      pre_sync_consume(a.pre);
      if (a.rows_done != nullptr) rows_gate_publish(a.rows_done);
    }
    if (CLUSTER) cluster_wait();
    return;
  }

  const double step = a.step;  // np.linspace(0, 1, batch + 1)
  auto stratum_owner = [&](int i, double u, double *residual) {
    double q01;
    if (a.use_philox) {
      const double lo = __dmul_rn((double)i, step);
      const double hi = (i + 1 == a.batch) ? 1.0 : __dmul_rn((double)(i + 1), step);
      q01 = __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u));  // random.uniform
    } else {
      q01 = a.strat_query01[i];
    }
    double mass = __dmul_rn(q01, grand_total);
    int owner = 0;
    for (; owner < a.num_shards - 1; ++owner) {
      const double left = shard_totals[owner];
      if (mass < left) break;
      mass = __dsub_rn(mass, left);
    }
    *residual = mass;
    return owner;
  };
  // This rank's strata: all of them, or (shard_ranges: Philox strata grow with the
  // stratum index and the rank-order scan is monotone) the range [lo, hi) found by two
  // simultaneous k-ary searches, blockDim candidates per round.
  int range_lo = 0, range_hi = a.batch;
  bool ranges_found = false;
  if (a.shard_ranges) {
    // Both ends sit within a stratum or two of (totals before this rank) / total * batch
    // and (totals through this rank) / total * batch: every warp tests a window of 16
    // candidates around each estimate — lanes 0..15 the lower end, 16..31 the upper — with
    // the exact owner rule, one draw per lane and no block barrier.  A window that does
    // not bracket its boundary (never seen; the estimates are off by rounding only) falls
    // back to the search below, so the result is the search's in every case.
    double before = 0.0;
    for (int g = 0; g < a.rank; ++g) before = __dadd_rn(before, shard_totals[g]);
    const double through = __dadd_rn(before, shard_totals[a.rank]);
    // (an estimate: single precision is plenty, and an fp64 division is a ~500-cycle
    // subroutine)
    const int which = lane >> 4;
    const float est = __fdividef((float)(which == 0 ? before : through), (float)grand_total) *
                      (float)a.batch;
    const int win_base = (est < (float)a.batch ? (int)est : a.batch) - 7;
    const int cand = win_base + (lane & 15);
    bool pred = cand >= a.batch;  // at or past the end
    if (cand >= 0 && cand < a.batch) {
      double unused;
      const int owner = stratum_owner(
          cand, philox_uniform53_fast(a.seed, draw_offset, (uint64_t)cand), &unused);
      pred = which == 0 ? owner >= a.rank : owner > a.rank;
    }
    const unsigned votes = __ballot_sync(full, pred);
    const unsigned v_lo = votes & 0xffffu, v_hi = votes >> 16;
    const int base_lo = __shfl_sync(full, win_base, 0), base_hi = __shfl_sync(full, win_base, 16);
    const bool ok_lo = (v_lo & 0x8000u) != 0 && ((v_lo & 1u) == 0 || base_lo <= 0);
    const bool ok_hi = (v_hi & 0x8000u) != 0 && ((v_hi & 1u) == 0 || base_hi <= 0);
    if (ok_lo && ok_hi) {
      range_lo = base_lo + __ffs(v_lo) - 1;
      range_hi = base_hi + __ffs(v_hi) - 1;
      if (range_lo < 0) range_lo = 0;
      if (range_hi < range_lo) range_hi = range_lo;
      ranges_found = true;
    }
  }
  if (a.shard_ranges && !ranges_found) {
    const int fan = blockDim.x;
    int base[2] = {0, 0}, limit[2] = {a.batch, a.batch};
    while (base[0] < limit[0] || base[1] < limit[1]) {
      if (threadIdx.x < 2) s_first[threadIdx.x] = fan;
      __syncthreads();
      int stride[2];
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        const int width = limit[w] - base[w];
        stride[w] = (width + fan - 1) / fan;
        const int cand = base[w] + (int)threadIdx.x * stride[w];
        if (width > 0) {
          bool hit = cand >= limit[w];
          if (!hit) {
            double unused;
            const int owner = stratum_owner(
                cand, philox_uniform53(a.seed, draw_offset, (uint64_t)cand), &unused);
            hit = w == 0 ? owner >= a.rank : owner > a.rank;
          }
          if (hit) atomicMin(&s_first[w], (int)threadIdx.x);
        }
      }
      __syncthreads();
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        if (base[w] >= limit[w]) continue;
        const int t = s_first[w];
        const int hit = base[w] + t * stride[w];
        const int new_limit = hit < limit[w] ? hit : limit[w];
        base[w] = t == 0 ? new_limit : base[w] + (t - 1) * stride[w] + 1;
        if (base[w] > new_limit) base[w] = new_limit;
        limit[w] = new_limit;
      }
      __syncthreads();
    }
    range_lo = base[0];
    range_hi = base[1];
  }
  const int n_all = range_hi - range_lo;
  // rows beyond the output capacity of a sharded step are dropped and latched
  const int n_mine = n_all < ws.cap ? n_all : ws.cap;
  const bool fast_scalars = a.with_scalars && a.sc.fast;
  const bool want_min = a.with_scalars && a.min_prob_out != nullptr;
  const int budget = a.max_attempts;
  const int n_spec = ws.spec < budget ? ws.spec : budget;  // draws evaluated up front
  const uint64_t retry_seed = a.seed + 0x9E3779B97F4A7C15ull * (uint64_t)(a.rank + 1);
  auto retry_uniform = [&](int r) {
    // Philox retry stream: rank-private (strata streams are shared by all ranks)
    return (a.use_philox || a.retry_u01 == nullptr)
               ? philox_uniform53_fast(retry_seed, draw_offset,
                                       (uint64_t)a.batch + (uint64_t)r)
               : a.retry_u01[r];
  };

  // ---- stratified pass (sum_tree.py:162-166 + prioritized_replay_buffer.py:155) and,
  // by the warps behind it, the first n_spec replacement draws (sum_tree.py:123-124:
  // query = random.random() * total), whether or not they will be needed
  float my_min = INFINITY;
  bool first_item = true;
  if (CLUSTER) {
    cluster_wait();
    // one word per stratum, two per speculative draw, one minimum per CTA
    if (blockIdx.x == 0 && threadIdx.x == 0)
      mbar_arrive_expect(&s_arrived,
                         4u * (uint32_t)(n_mine + 2 * n_spec + (want_min ? (int)gridDim.x : 0)));
  }
#pragma unroll 1
  for (int pos = blockIdx.x * warps + warp; pos < n_mine + n_spec;
       pos += gridDim.x * warps) {
    const bool stratum = pos < n_mine;
    double mass;
    if (stratum) {
      const int i = range_lo + pos;
      const double u =
          a.use_philox ? philox_uniform53_fast(a.seed, draw_offset, (uint64_t)i) : 0.0;
      stratum_owner(i, u, &mass);  // (inside the range the owner is this rank)
    } else {
      mass = __dmul_rn(retry_uniform(pos - n_mine), local_total);
    }
    B2R_MARK(13);
    if (!first_item) c_top = warp_candidate(a.heap, 1, a.depth < 5 ? a.depth : 5, lane);
    first_item = false;
    const int64_t idx = tree_descend_warp(a.heap, a.depth, mass, lane, c_top);
    B2R_MARK(14);
    ScalarLoads row;
    if (stratum && fast_scalars && lane == 0) load_scalars(a.sc, idx, &row);
    const bool valid = warp_is_valid(ctx, idx, lane);
    B2R_MARK(15);
    if (lane == 0) {
      if (stratum) {
        a.out_idx[pos] = (int32_t)idx;
        if (a.out_slots) a.out_slots[pos] = range_lo + pos;
        if (CLUSTER) st_async_u32(&s_flag32[pos], valid ? 0u : 1u, &s_arrived, 0);
        else ws.inv_flag[pos] = valid ? 0 : 1;
        if (valid) {
          float p = INFINITY;
          if (fast_scalars) p = finish_scalars(a.sc, pos, idx, row);
          else if (a.with_scalars) p = write_scalars(a.sc, pos, idx);
          my_min = fminf(my_min, p);
        }
      } else if (CLUSTER) {
        st_async_u32(&s_cl_spec_idx[pos - n_mine], (uint32_t)(int32_t)idx, &s_arrived, 0);
        st_async_u32(&s_cl_spec_valid[pos - n_mine], valid ? 1u : 0u, &s_arrived, 0);
      } else {
        ws.spec_idx[pos - n_mine] = (int32_t)idx;
        ws.spec_valid[pos - n_mine] = valid ? 1 : 0;
      }
    }
  }
  // The one-stream step: the copies and the tail read these rows once the closing thread has
  // counted the launch (StageGate::rows), not behind the kernel's completion.  The order comes
  // without a fence per row: every CTA sends its minimum word behind the barrier below,
  // after all of its rows; the complete-tx of an st.async releases at cluster scope; CTA 0
  // waits for every word with acquire at cluster scope (mbar_wait_cluster); and the closing
  // thread counts the launch with a release at GPU scope, which passes on what it has
  // acquired.  (Plain grids: the fence + ticket election below orders the rows before the
  // last CTA.)
  B2R_MARK(16);
  if (want_min) {
    if (lane == 0) s_wmin[warp] = my_min;
    __syncthreads();
    if (threadIdx.x == 0) {
      float m = s_wmin[0];
      for (int w = 1; w < warps; ++w) m = fminf(m, s_wmin[w]);
      if (CLUSTER) st_async_u32(&s_cl_min[blockIdx.x], __float_as_uint(m), &s_arrived, 0);
      else ws.cta_min[blockIdx.x] = m;
    }
  }

  // ---- only the last CTA to finish goes on (CLUSTER: CTA 0, after the barrier)
  if (CLUSTER) {
    if (blockIdx.x != 0) return;  // (its words are on their way to CTA 0)
    // (the closing thread's look at the first half of the loss travels with the wait)
    PreSyncPeek peek = {0u, 1u};
    if (threadIdx.x == 0) peek = pre_sync_peek(a.pre);
    if (a.rows_done != nullptr)
      mbar_wait_cluster(&s_arrived, 0);
    else
      mbar_wait(&s_arrived, 0);
    ws.inv_flag = s_flag;
    ws.spec_idx = s_cl_spec_idx;
    ws.spec_valid = s_cl_spec_valid;
    ws.cta_min = s_cl_min;
    // The usual case at the agent's batch — every stratified pick valid, nothing to
    // replace — is closed by warp 0 alone: a vote over the flags, a shuffle minimum over
    // the CTAs' minima, the launch's counters; no block scan, no list, one barrier.
    __shared__ int s_slow;
    if (warp == 0) {
      bool bad = false;
      for (int p = lane; p < n_mine; p += 32) bad = bad || s_flag32[p] != 0u;
      const bool slow = __any_sync(full, bad) || n_all > n_mine;
      if (lane == 0) s_slow = slow ? 1 : 0;
    }
    __syncthreads();
    if (s_slow == 0) {
      if (warp != 0) return;
      float m = INFINITY;
      if (want_min) {
        for (int c = lane; c < (int)gridDim.x; c += 32) m = fminf(m, s_cl_min[c]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fminf(m, __shfl_xor_sync(full, m, o));
      }
      if (lane == 0) {
        if (want_min) *a.min_prob_out = m;
        // (rows and minimum are final: the count goes first, its release waits for them only)
        if (a.rows_done != nullptr) rows_gate_publish(a.rows_done);
        if (a.counter) *a.counter = draws_before + 1;
        if (exchange) *a.xchg.seq = xseq;
        a.info[0] = B2R_OK;
        a.info[1] = 0;
        a.info[2] = 0;
        a.info[3] = n_mine;
        if (a.count_out) *a.count_out = n_mine;
        if (want_min) publish_local_min(a, exchange, m, xseq);
        pre_sync_consume(a.pre, peek);
      }
      B2R_MARK_ANY(20);
      return;
    }
    // the slow path below reads the flags as bytes
    for (int p = threadIdx.x; p < n_mine; p += blockDim.x) s_flag[p] = (uint8_t)s_flag32[p];
    __syncthreads();
  } else if (gridDim.x > 1) {
    if (!last_cta(a.ticket, &s_is_last, false)) return;
  } else {
    __syncthreads();
  }
  B2R_MARK_ANY(17);
  if (threadIdx.x == 0) {
    s_draws_used = 0;
    s_last_idx = -1;
    s_last_valid = 0;
    if (!CLUSTER && gridDim.x > 1) *a.ticket = 0u;  // ready for the next launch
  }
  // Ordered list of the invalid positions (16 flag bytes per thread and round) and, in
  // the same block scan, the order of the valid speculative draws: every load of this
  // phase is issued before the first one is used.
  float min_seen = INFINITY;
  if (want_min)
    for (int c = threadIdx.x; c < (int)gridDim.x; c += blockDim.x)
      min_seen = fminf(min_seen, ld_scratch<CLUSTER>(ws.cta_min + c));
  const bool spec_mine = (int)threadIdx.x < n_spec;
  const int spec_v = spec_mine ? ld_scratch<CLUSTER>(ws.spec_valid + threadIdx.x) : 0;
  if (spec_mine) s_spec_idx[threadIdx.x] = ld_scratch<CLUSTER>(ws.spec_idx + threadIdx.x);
  int num_invalid = 0, spec_good = 0;
  for (int base = 0; base < n_mine || base == 0; base += 16 * (int)blockDim.x) {
    const int p0 = base + 16 * (int)threadIdx.x;
    uint32_t f[4] = {0, 0, 0, 0};
    if (p0 < n_mine) {
      const uint4 v = ld_scratch<CLUSTER>(reinterpret_cast<const uint4 *>(ws.inv_flag + p0));
      f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
#pragma unroll
      for (int k = 0; k < 4; ++k) {  // bytes at or beyond n_mine are stale
        const int left = n_mine - (p0 + 4 * k);
        f[k] &= left >= 4 ? 0x01010101u : (left <= 0 ? 0u : (0x01010101u >> (8 * (4 - left))));
      }
    }
    const int mine_inv = __popc(f[0]) + __popc(f[1]) + __popc(f[2]) + __popc(f[3]);
    const int mine_spec = base == 0 && spec_v == 1 ? 1 : 0;
    const int mine_packed = mine_inv | (mine_spec << 20);  // two counts, one scan
    int inc = mine_packed;  // inclusive scan over the block
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(full, inc, o);
      if (lane >= o) inc += v;
    }
    __syncthreads();  // (warp_counts of the previous round has been read)
    if (lane == 31) warp_counts[warp] = inc;
    __syncthreads();
    int before = inc - mine_packed, total = 0;
    for (int w = 0; w < warps; ++w) {
      const int cnt = warp_counts[w];
      if (w < warp) before += cnt;
      total += cnt;
    }
    int slot_at = num_invalid + (before & 0xfffff);
    if (mine_inv > 0) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if ((f[k] >> (8 * b)) & 1u) ws.inv_list[slot_at++] = p0 + 4 * k + b;
    }
    if (mine_spec) s_draw_of[before >> 20] = threadIdx.x;
    num_invalid += total & 0xfffff;
    if (base == 0) spec_good = total >> 20;
  }
  __syncthreads();  // inv_list (global), s_draw_of and the shared scalars are visible
  B2R_MARK_ANY(18);

  // ---- in-order replacement of invalid slots (prioritized_replay_buffer.py:156-170):
  // the j-th invalid slot takes the j-th valid draw out of a shared budget.
  int found = 0, drawn = 0;
  float fix_min = INFINITY;
  if (num_invalid > 0 && budget > 0) {
    int spec_done = n_spec;
    if (spec_done == 0) {
      // nothing was evaluated up front (single-CTA launches): one warp per draw, now
      spec_done = warps < budget ? warps : budget;
      if (warp < spec_done) {
        const double c0 = warp_candidate(a.heap, 1, a.depth < 5 ? a.depth : 5, lane);
        const int64_t idx = tree_descend_warp(
            a.heap, a.depth, __dmul_rn(retry_uniform(warp), local_total), lane, c0);
        const bool valid = warp_is_valid(ctx, idx, lane);
        if (lane == 0) {
          ws.spec_idx[warp] = (int32_t)idx;
          ws.spec_valid[warp] = valid ? 1 : 0;
        }
      }
      __syncthreads();
      const bool v = (int)threadIdx.x < spec_done && ws.spec_valid[threadIdx.x] == 1;
      const int ord = block_scan_flag(v, warp_counts, &spec_good);
      if (v) s_draw_of[ord] = threadIdx.x;
      __syncthreads();
    }
    // draw r fills invalid slot number (valid draws before r)
    const int fixed = num_invalid < spec_good ? num_invalid : spec_good;
    for (int j = threadIdx.x; j < fixed; j += blockDim.x) {
      const int r = s_draw_of[j];
      const int idx = n_spec > 0 ? s_spec_idx[r] : ld_scratch<CLUSTER>(ws.spec_idx + r);
      const int slot = ws.inv_list[j];
      a.out_idx[slot] = idx;
      if (fast_scalars) {  // one round trip for every input of the row
        ScalarLoads row;
        load_scalars(a.sc, idx, &row);
        fix_min = fminf(fix_min, finish_scalars(a.sc, slot, idx, row));
      } else if (a.with_scalars) {
        fix_min = fminf(fix_min, write_scalars(a.sc, slot, idx));
      }
      if (j == num_invalid - 1) s_draws_used = r + 1;
    }
    if (threadIdx.x == 0 && spec_done == budget) {
      s_last_idx = ld_scratch<CLUSTER>(ws.spec_idx + budget - 1);
      s_last_valid = ld_scratch<CLUSTER>(ws.spec_valid + budget - 1) == 1 ? 1 : 0;
    }
    found = fixed;
    drawn = spec_done;
    if (found < num_invalid && drawn < budget) {
      // (rare) the speculative draws did not suffice: windows of blockDim draws, a
      // thread per draw, validity against a shared-memory copy of the context
      for (int w = threadIdx.x; w < kCtxWords; w += blockDim.x)
        reinterpret_cast<uint64_t *>(&s_valid)[w] =
            reinterpret_cast<const uint64_t *>(a.valid_dev)[w];
      __syncthreads();
    }
    while (found < num_invalid && drawn < budget) {
      const int r = drawn + threadIdx.x;
      const bool active = r < budget;
      bool valid = false;
      int64_t idx = 0;
      if (active) {
        idx = descend_from_root(a.heap, a.depth,
                                __dmul_rn(retry_uniform(r), local_total), a.zero);
        valid = is_valid_transition(s_valid, idx);
      }
      int tile_valid;
      const int ord = found + block_scan_flag(active && valid, warp_counts, &tile_valid);
      if (active && valid && ord < num_invalid) {
        const int slot = ws.inv_list[ord];
        a.out_idx[slot] = (int32_t)idx;
        if (fast_scalars) {
          ScalarLoads row;
          load_scalars(a.sc, idx, &row);
          fix_min = fminf(fix_min, finish_scalars(a.sc, slot, idx, row));
        } else if (a.with_scalars) {
          fix_min = fminf(fix_min, write_scalars(a.sc, slot, idx));
        }
        if (ord == num_invalid - 1) s_draws_used = r + 1;
      }
      if (active && r == budget - 1) {
        s_last_idx = (int)idx;
        s_last_valid = valid ? 1 : 0;
      }
      found += tile_valid;
      drawn += blockDim.x;
      __syncthreads();
    }
  }
  if (a.rows_done != nullptr) __threadfence();  // (the fix-ups, before the count)
  __syncthreads();
  B2R_MARK_ANY(19);
  if (threadIdx.x == 0) {
    int status = B2R_OK, fail_slot = 0, used = 0;
    if (num_invalid > 0) {
      if (found >= num_invalid) {
        used = s_draws_used;
      } else {
        // Every one of the `budget` draws was consumed; `found` slots were fixed.
        used = budget;
        const int next_slot = ws.inv_list[found];  // first invalid slot still unresolved
        if (budget == 0 || s_last_valid) {
          // budget already 0 when this slot is reached -> PRB:159-163
          status = B2R_ERR_SAMPLE_ATTEMPTS;
          fail_slot = next_slot;
        } else {
          // the slot burnt the rest of the budget and keeps its last (invalid) draw;
          // only a FURTHER invalid slot raises (SURVEY.md Q10).
          a.out_idx[next_slot] = s_last_idx;
          if (a.with_scalars && s_last_idx >= 0 && s_last_idx < ctx.capacity) {
            // (the reference hands this invalid index on: so do the consumers' rows)
            if (fast_scalars) {
              ScalarLoads row;
              load_scalars(a.sc, s_last_idx, &row);
              fix_min = fminf(fix_min, finish_scalars(a.sc, next_slot, s_last_idx, row));
            } else {
              fix_min = fminf(fix_min, write_scalars(a.sc, next_slot, s_last_idx));
            }
          }
          if (num_invalid > found + 1) {
            status = B2R_ERR_SAMPLE_ATTEMPTS;
            fail_slot = ws.inv_list[found + 1];
          }
        }
      }
    }
    if (n_all > n_mine && status == B2R_OK) {  // a sharded step outgrew its buffers
      status = B2R_ERR_UNSUPPORTED;
      fail_slot = n_all;  // (reported: the size of the share)
    }
    if (a.counter) *a.counter = draws_before + 1;
    if (exchange) *a.xchg.seq = xseq;
    a.info[0] = status;
    a.info[1] = a.out_slots ? (status ? a.out_slots[fail_slot < n_mine ? fail_slot : 0] : 0)
                            : fail_slot;
    a.info[2] = used;
    a.info[3] = n_mine;
    if (a.count_out) *a.count_out = n_mine;
    if (status != B2R_OK && a.latched && a.latched[0] == 0) {
      a.latched[0] = status;
      a.latched[1] = fail_slot;
    }
  }
  if (want_min) {
    const float m = block_min(fminf(min_seen, fix_min), warp_mins);
    if (threadIdx.x == 0) {
      *a.min_prob_out = m;
      publish_local_min(a, exchange, m, xseq);
    }
  }
  if (threadIdx.x == 0) {
    pre_sync_consume(a.pre);
    if (a.rows_done != nullptr) rows_gate_publish(a.rows_done);
  }
  B2R_MARK_ANY(20);
}

struct UniformSampleArgs {
  // read from HBM (refreshed by every flush), not passed by value: a captured CUDA graph
  // samples over the transitions added since the capture
  const ValidCtx *valid_dev;
  int batch;
  int max_attempts;
  int use_philox;
  uint64_t seed, offset;
  uint64_t *counter;
  int n_cand;                  // host mode: number of supplied candidates
  const int64_t *candidates;   // np.random.randint(min_id, max_id) draws
  int32_t *out_idx;
  int32_t *counters;           // in/out: [0] accepted, [1] rejected; out: [2] draws used
  int64_t *latched;
};

// circular_replay_buffer.py:462-470 over a window of candidate draws.
__global__ void __launch_bounds__(1024) uniform_sample_kernel(UniformSampleArgs a) {
  __shared__ int warp_counts[32];
  __shared__ ValidCtx s_valid;
  pdl_release();
  pdl_acquire();
  for (int w = threadIdx.x; w < (int)(sizeof(ValidCtx) / 8); w += blockDim.x)
    reinterpret_cast<uint64_t *>(&s_valid)[w] =
        reinterpret_cast<const uint64_t *>(a.valid_dev)[w];
  int accepted = a.counters[0], rejected = a.counters[1], used = 0;
  const uint64_t draws_before = a.counter ? *a.counter : 0ull;
  const uint64_t draw_offset = a.offset + draws_before;
  __syncthreads();
  const ValidCtx &c = s_valid;
  // Philox mode: uniform_bounds (CRB:449-460) on the device; the host has checked that
  // the span is not empty
  const int64_t min_id = c.add_count >= c.capacity ? c.cursor - c.capacity + c.stack - 1
                                                   : c.stack - 1;
  const int64_t span = c.cursor - c.horizon - min_id;
  int base = 0;
  while (accepted < a.batch && rejected < a.max_attempts &&
         (a.use_philox || base < a.n_cand)) {
    const int p = base + threadIdx.x;
    const bool active = a.use_philox || p < a.n_cand;
    bool valid = false;
    int64_t idx = 0;
    if (active) {
      int64_t cand;
      if (a.use_philox) {
        const double u = philox_uniform53(a.seed, draw_offset, (uint64_t)p);
        int64_t off = (int64_t)(u * (double)span);
        if (off >= span) off = span - 1;
        cand = min_id + off;
      } else {
        cand = a.candidates[p];
      }
      idx = wrap_index(cand, c.capacity);  // `% replay_capacity`, CRB:466
      valid = is_valid_transition(c, idx);
    }
    int tile_acc, tile_rej, tile_done;
    const int acc_before = accepted + block_scan_flag(active && valid, warp_counts, &tile_acc);
    const int rej_before = rejected + block_scan_flag(active && !valid, warp_counts, &tile_rej);
    // A draw happens only while both loop conditions still hold (CRB:464-465).
    const bool processed =
        active && acc_before < a.batch && rej_before < a.max_attempts;
    if (processed && valid) a.out_idx[acc_before] = (int32_t)idx;
    block_scan_flag(processed, warp_counts, &tile_done);
    int done_acc, done_rej;
    block_scan_flag(processed && valid, warp_counts, &done_acc);
    block_scan_flag(processed && !valid, warp_counts, &done_rej);
    accepted += done_acc;
    rejected += done_rej;
    used += tile_done;
    base += blockDim.x;
  }
  if (threadIdx.x == 0) {
    a.counters[0] = accepted;
    a.counters[1] = rejected;
    a.counters[2] = used;
    if (a.counter) *a.counter = draws_before + 1;
    if (a.use_philox && accepted < a.batch && a.latched && a.latched[0] == 0) {
      a.latched[0] = B2R_ERR_SAMPLE_ATTEMPTS;
      a.latched[1] = accepted;
    }
  }
}

int uniform_bounds(const b2r_buffer *b, int64_t *lo, int64_t *hi) {
  // circular_replay_buffer.py:449-460
  const int64_t cap = b->cfg.capacity;
  const int64_t cursor = b->add_count % cap;
  if (b->add_count >= cap) {
    *lo = cursor - cap + b->cfg.stack_size - 1;
    *hi = cursor - b->cfg.update_horizon;
  } else {
    *lo = b->cfg.stack_size - 1;
    *hi = cursor - b->cfg.update_horizon;
    if (*hi <= *lo)
      return fail(B2R_ERR_TOO_FEW_TRANSITIONS,
                  "Cannot sample a batch with fewer than stack size (%d) + "
                  "update_horizon (%d) transitions.",
                  b->cfg.stack_size, b->cfg.update_horizon);
  }
  return B2R_OK;
}

int sample_threads(int n) {
  int t = 32;
  while (t < n && t < 1024) t <<= 1;
  return t;
}

// The request of the b2r_sample_indices_sharded_* entry points, but for the totals.
SampleRequest sharded_indices_request(b2r_buffer *b, int32_t global_batch,
                                      const double *query01, int32_t n_retry,
                                      const double *retry_u01, uint64_t seed,
                                      uint64_t offset, int32_t *out_slots,
                                      int32_t *out_indices, int32_t *out_count) {
  SampleRequest r;
  r.batch = global_batch;
  r.sharded = true;
  r.query01 = query01;
  r.retry_u01 = retry_u01;
  r.max_attempts = n_retry;
  r.seed = seed;
  r.offset = offset;
  r.counter = b->shard_counter;
  r.info = b->info;
  r.out_idx = out_indices;
  r.out_slots = out_slots;
  r.count_out = out_count;
  return r;
}

// uniform_sample_kernel over the caller's `candidates` (n_cand of them; no latch, counters
// in/out) or, candidates == nullptr, over Philox draws of (seed, offset + the buffer's draw
// counter).
int launch_uniform_sample(b2r_buffer *b, int batch, uint64_t seed, uint64_t offset,
                          int n_cand, const int64_t *candidates, int32_t *out_idx,
                          int32_t *counters, cudaStream_t stream) {
  const bool philox = candidates == nullptr;
  UniformSampleArgs a;
  a.valid_dev = b->ctx_dev;
  a.batch = batch;
  a.max_attempts = b->cfg.max_sample_attempts;
  a.use_philox = philox ? 1 : 0;
  a.seed = seed;
  a.offset = offset;
  a.counter = philox ? b->draw_counter : nullptr;
  a.n_cand = n_cand;
  a.candidates = candidates;
  a.out_idx = out_idx;
  a.counters = counters;
  a.latched = philox ? b->status : nullptr;
  B2R_CUDA(launch(uniform_sample_kernel, dim3(1), dim3(sample_threads(philox ? batch : n_cand)),
                  0, stream, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // namespace

// Largest number of strata the warp sampler (per_sample_warp_kernel) takes; above, a
// thread per stratum over shared-memory-staged top levels (per_sample_kernel).  Every
// instruction of the warp sampler serves ONE stratum, so from a few thousand strata on it
// is bound by instruction issue (4096 warps x ~2 k instructions = 14 k cycles on 592
// schedulers) and the thread-per-stratum kernel, 32 strata per instruction, is the faster
// one again: measured in the fused step at 4096, 116 us against 109 us
// (profiles/r2/README.md).  Caller-supplied queries of a SHARDED batch always take the
// thread kernel: their owners need not be monotone in the stratum index, so the rank's
// rows are compacted by one CTA.
constexpr int kSamplerWarpMax = 2048;

// Grid and scratch of the warp sampler for `strata` expected strata and outputs of
// `cap` rows.
static int warp_sampler_setup(b2r_buffer *b, int strata, int cap, WarpScratch *ws,
                              int *threads, int *ctas) {
  int warps = strata <= 64 ? 4 : 8;
  // replacement draws evaluated up front: a pick is invalid with probability ~0.3 % in
  // an Atari-like memory (a terminal among the three frames before it)
  int spec = strata / 64;
  if (spec < 4) spec = 4;
  if (spec > kSpecMax) spec = kSpecMax;
  ws->cluster = 0;
  if (strata + 4 <= 64 && cap <= kClusterCap) {
    // one cluster of 8 CTAs; the warps left over after the strata draw replacements
    ws->cluster = 1;
    *ctas = 8;
    warps = (strata + 4 + 7) / 8;
    spec = 8 * warps - strata;
  } else {
    *ctas = (strata + spec + warps - 1) / warps;
    if (*ctas > 8192) *ctas = 8192;  // the warps stride
  }
  *threads = warps * 32;
  const int64_t flag_words = ((int64_t)cap + 15) / 16 * 4;
  B2R_TRY(ensure_inv_slots(b, flag_words + cap + 2 * kSpecMax + *ctas + 16));
  ws->inv_flag = reinterpret_cast<uint8_t *>(b->inv_slots);
  ws->inv_list = b->inv_slots + flag_words;
  ws->spec_idx = ws->inv_list + cap;
  ws->spec_valid = ws->spec_idx + kSpecMax;
  ws->cta_min = reinterpret_cast<float *>(ws->spec_valid + kSpecMax);
  ws->cap = cap;
  ws->spec = spec;
  return B2R_OK;
}

// Two register budgets: 126 registers (no spills, 16 warps per SM) while every warp of
// the launch is resident anyway; 64 registers (a few spills outside the descent, 32 warps
// per SM) for the batches that would otherwise need a second wave: 296 CTAs, two per SM.
constexpr int kSamplerWaveCtas = 296;

int launch_sample(b2r_buffer *b, const SampleRequest &r, cudaStream_t stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (r.batch <= 0 || r.num_shards <= 0 || r.num_shards > kMaxShards || r.rank < 0 ||
      r.rank >= r.num_shards)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad sharding arguments");
  if (r.x && !r.x->connected && r.x->world > 1)
    return fail(B2R_ERR_INVALID_ARGUMENT, "the exchange is not connected");
  const bool philox = r.query01 == nullptr;
  const int cap = r.out_cap > 0 && r.out_cap < r.batch ? r.out_cap : r.batch;
  // The warp sampler up to kSamplerWarpMax strata (sharded: of a rank's expected share,
  // not of the global batch), over this rank's stratum range for Philox strata (see
  // shard_ranges).  Sharded caller queries (any order): one CTA of the thread kernel walks
  // every tile and compacts this rank's strata with block scans; Philox strata above
  // kSamplerWarpMax: tiles of 128 over many CTAs with the range search.
  const bool by_warp = (philox || !r.sharded) && r.batch / r.num_shards <= kSamplerWarpMax;
  const bool ranges = philox && r.num_shards > 1 && (by_warp || r.batch > 256);
  if (r.rows_done != nullptr && (!by_warp || !r.scalars || !r.min_prob_out))
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "only the warp sampler with scalars and the minimum counts its rows");
  PerSampleArgs a = {};
  WarpScratch ws;
  int threads, ctas;
  if (by_warp) {
    // grid for the expected share plus a margin; the warps stride over the rest
    int expect = r.num_shards > 1
                     ? r.batch / r.num_shards + r.batch / (4 * r.num_shards) + 8
                     : r.batch;
    if (expect > cap) expect = cap;
    B2R_TRY(warp_sampler_setup(b, expect, cap, &ws, &threads, &ctas));
  } else {
    // Threads per CTA (= strata per tile).  Small batches: one CTA (at least 256 threads,
    // so that staging the top levels is two rounds of loads).  Large batches: tiles of 128
    // strata, so that the descents spread over many SMs (with ranges, tiles of this rank's
    // range: the grid follows the capacity of the outputs, not the global batch), or the
    // one CTA of 1024 threads that compacts a rank's rows.
    const bool one_cta = r.sharded && !ranges;
    threads = r.batch <= 256 ? 256 : (one_cta ? 1024 : 128);
    ctas = ((one_cta ? r.batch : cap) + threads - 1) / threads;
    if (ctas > kMaxTiles)
      return r.sharded ? fail(B2R_ERR_UNSUPPORTED, "global batch too large")
                       : fail(B2R_ERR_UNSUPPORTED, "batch above %d is not supported",
                              kMaxTiles * 128);
    B2R_TRY(ensure_inv_slots(b, (int64_t)ctas * threads + 2 * kMaxTiles + 8));
    a.inv_slots = b->inv_slots;
    a.tile_counts = b->inv_slots + (int64_t)ctas * threads;
    a.tile_min = reinterpret_cast<float *>(a.tile_counts + kMaxTiles);
  }
  a.heap = b->tree->heap;
  a.depth = b->tree->depth;
  B2R_TRY(ensure_ctx(b, stream));
  a.valid_dev = b->ctx_dev;
  a.batch = r.batch;
  a.step = 1.0 / (double)r.batch;
  a.max_attempts = r.max_attempts;
  a.use_philox = philox ? 1 : 0;
  a.seed = r.seed;
  a.offset = r.offset;
  a.counter = philox ? r.counter : nullptr;
  a.strat_query01 = r.query01;
  a.retry_u01 = r.retry_u01;
  a.out_idx = r.out_idx;
  a.ticket = &b->sync->sample_ticket;
  a.info = r.info;
  a.latched = r.latch ? b->status : nullptr;
  a.num_shards = r.num_shards;
  a.rank = r.rank;
  a.shard_totals = r.shard_totals;
  a.out_slots = r.out_slots;
  a.with_scalars = r.scalars != nullptr;
  a.min_prob_out = r.min_prob_out;
  a.count_out = r.count_out;
  a.shard_ranges = ranges ? 1 : 0;
  a.out_cap = cap;
  a.publish_min = r.publish_min ? 1 : 0;
  a.rows_done = r.rows_done;
  if (r.pre != nullptr) a.pre = *r.pre;
  if (r.x && r.x->world > 1) fill_exchange_args(r.x, &a.xchg);
  if (r.scalars) {
    fill_scalar_args(b, r.scalars, &a.sc);
    if (a.sc.indices_out == r.out_idx) a.sc.indices_out = nullptr;
  }
  set_tree_window(b->tree->heap, (size_t)b->tree->leaves * 16);
  if (by_warp && ws.cluster)
    B2R_CUDA(launch_prio_cluster(per_sample_warp_kernel<2, true>, dim3(ctas), dim3(threads),
                                 0, stream, chain_priority(), ctas, a, ws));
  else if (by_warp && ctas > kSamplerWaveCtas)
    B2R_CUDA(launch(per_sample_warp_kernel<4, false>, dim3(ctas), dim3(threads), 0, stream,
                    a, ws));
  else if (by_warp)
    B2R_CUDA(launch(per_sample_warp_kernel<2, false>, dim3(ctas), dim3(threads), 0, stream,
                    a, ws));
  else if (threads != 1024)  // 3 tree levels per memory round trip (more would bloat the
                             // straight-line code, and a cold instruction cache costs more
                             // than the saved round trips)
    B2R_CUDA(launch(per_sample_kernel<3, 256>, dim3(ctas), dim3(threads), 0, stream, a));
  else
    B2R_CUDA(launch(per_sample_kernel<3, 1024>, dim3(1), dim3(threads), 0, stream, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

void fill_exchange_args(const b2r_exchange *x, ExchangeArgs *out) {
  out->local = x->mailbox;
  for (int g = 0; g < kMaxShards; ++g) out->peer[g] = x->peer[g];
  out->seq = x->seq;
  out->timeout_ns = x->timeout_ns;
  out->pub = x->pub;
  // Profiling switch (never set in production): B2R_DEBUG_XCHG_NOWAIT=1 takes this rank's
  // own total for every peer instead of waiting for theirs — the step time without the
  // cross-GPU coupling, i.e. the bound of what any change to the exchange can gain.  The
  // ranks' strata then no longer partition the batch.
  static const bool nowait = std::getenv("B2R_DEBUG_XCHG_NOWAIT") != nullptr;
  if (nowait) out->timeout_ns = 0;
}

// Publishes a rank's total for the next exchange step without consuming it.
__global__ void exchange_publish_kernel(ExchangeArgs x, int world, int rank,
                                        const double *heap) {
  exchange_publish(x, world, rank, heap[1], *x.seq + 1);  // (also records x.pub)
}

int launch_exchange_publish(const b2r_exchange *x, const b2r_buffer *b,
                            cudaStream_t s) {
  ExchangeArgs xa;
  fill_exchange_args(x, &xa);
  exchange_publish_kernel<<<1, 32, 0, s>>>(xa, x->world, x->rank, b->tree->heap);
  B2R_LAUNCHED();
  return B2R_OK;
}

// ---- Sharded UNIFORM sampling: one global batch of circular_replay_buffer.py:462-470 over
// a virtual buffer whose index range is the concatenation of the shards' ranges.
//
// Rank g's span is n_g = max(0, max_id_g - min_id_g) (CRB:449-460, from the device
// validity context, so a replayed graph sees new adds); N = sum of the spans.  Draw j is
// u_j = philox_uniform53(seed, offset + step, j) with `step` the exchange's step number,
// o_j = min((int64)(u_j N), N - 1), owned by the rank the scan `o < n_g ? g : o -= n_g`
// stops at, candidate (min_id_owner + o) mod capacity.  The draws are processed in order
// while accepted < batch and rejected < max_sample_attempts; the k-th accepted draw is
// global row k.  Only the owner of a draw knows whether it is valid, so the ranks agree on
// the accepted draws in two rounds over the mailbox:
//   1. spans: the totals words (exchange_publish / exchange_collect, f64 payload);
//   2. rejections: every rank evaluates the draws it owns in [0, batch + max_attempts) —
//      every draw the loop could process — and publishes the ascending ordinals of its
//      invalid ones, the first max_attempts of them (kRejWordsOffset region).
// With rejects_before(j) summed over the G lists (binary searches), an owned valid draw j
// is kept iff j - rejects_before(j) < batch and rejects_before(j) < max_attempts, as row
// j - rejects_before(j).  Both quantities only grow with j, so the kept draws are a
// prefix of the rank's valid draws.  A rank stops evaluating once it has `batch` valid
// draws (a later draw's row is >= batch) or max_attempts invalid ones (a later draw has
// rejects_before >= max_attempts): what it leaves out of its list changes no decision.
namespace {

constexpr int kUniformShardThreads = 1024;
enum { kUniformPublishSpan = 0, kUniformPublishRejections = 1, kUniformSample = 2 };

struct UniformShardArgs {
  const ValidCtx *valid_dev;
  ExchangeArgs xchg;
  int world, rank;
  int batch;  // global batch
  int max_attempts;
  uint64_t seed, offset;
  int mode;
  int out_cap;
  int32_t *out_idx, *out_slots, *count_out;
  int32_t *own_j, *own_idx;  // scratch [batch]: this rank's valid draws, ascending
  int32_t *lists;            // scratch [world * kRejListWords]: the collected lists
  int64_t *latched;
};

__device__ __forceinline__ uint64_t rej_word(int32_t value, uint64_t seq) {
  return ((uint64_t)(uint32_t)value << 32) | (uint32_t)seq;
}

// Polls one mailbox word until it carries step `seq` (value returned) or the timeout
// passes (latches B2R_ERR_EXCHANGE for rank g, returns `missing`).
__device__ __forceinline__ int32_t poll_rej_word(const ExchangeArgs &x, const uint64_t *src,
                                                 uint64_t seq, int g, int32_t missing,
                                                 int64_t *latched) {
  if (x.timeout_ns <= 0) return missing;
  const bool broken = latched != nullptr && latched[0] == B2R_ERR_EXCHANGE;
  uint64_t w;
  if (!broken && poll_tagged_word(src, seq, x.timeout_ns, &w)) return (int32_t)(w >> 32);
  if (latched != nullptr) {
    latched[0] = B2R_ERR_EXCHANGE;
    latched[1] = g;
  }
  return missing;
}

__global__ void __launch_bounds__(kUniformShardThreads)
    uniform_sharded_kernel(const __grid_constant__ UniformShardArgs a) {
  __shared__ ValidCtx s_valid;
  __shared__ double s_spans[kMaxShards];
  __shared__ int64_t s_span[kMaxShards];
  __shared__ int warp_counts[32];
  __shared__ int32_t s_rej[kRejListWords];
  __shared__ int s_start[kMaxShards + 1];
  __shared__ int s_published, s_stale, s_kept;
  pdl_release();
  pdl_acquire();  // (everything below publishes: after griddepcontrol.wait)
  for (int w = threadIdx.x; w < (int)(sizeof(ValidCtx) / 8); w += blockDim.x)
    reinterpret_cast<uint64_t *>(&s_valid)[w] =
        reinterpret_cast<const uint64_t *>(a.valid_dev)[w];
  const uint64_t xseq = *a.xchg.seq + 1;
  if (threadIdx.x == 0) {
    s_published = 0;
    s_stale = 0;
    s_kept = 0;
  }
  __syncthreads();
  const ValidCtx &c = s_valid;
  // uniform_bounds (CRB:449-460) on the device
  int64_t min_id, max_id;
  if (c.add_count >= c.capacity) {
    min_id = c.cursor - c.capacity + c.stack - 1;
    max_id = c.cursor - c.horizon;
  } else {
    min_id = c.stack - 1;
    max_id = c.cursor - c.horizon;
  }
  const int64_t span = max_id > min_id ? max_id - min_id : 0;

  // ---- round 1: spans
  if (threadIdx.x < 32) {
    if (a.mode == kUniformPublishSpan)
      exchange_publish(a.xchg, a.world, a.rank, (double)span, xseq);
    else
      exchange_publish_if_needed(a.xchg, a.world, a.rank, (double)span, xseq, a.latched);
  }
  if (a.mode == kUniformPublishSpan) return;
  exchange_collect(a.xchg, a.world, a.rank, (double)span, xseq, s_spans, a.latched);
  __syncthreads();
  if (threadIdx.x < a.world) s_span[threadIdx.x] = (int64_t)s_spans[threadIdx.x];
  __syncthreads();
  int64_t total = 0;
  for (int g = 0; g < a.world; ++g) total += s_span[g];
  if (total == 0) {  // CRB:457-460 on every shard
    if (threadIdx.x == 0 && a.mode == kUniformSample) {
      *a.count_out = 0;
      if (a.latched && a.latched[0] == 0) {
        a.latched[0] = B2R_ERR_TOO_FEW_TRANSITIONS;
        a.latched[1] = 0;
      }
      *a.xchg.seq = xseq;
    }
    return;
  }

  // ---- this rank's draws of the window: ordinals of the invalid ones, valid ones
  const uint64_t draw_offset = a.offset + xseq;
  const int window = a.batch + a.max_attempts;
  int n_rej = 0, n_ok = 0;  // (block-uniform)
  for (int base = 0; base < window && n_rej < a.max_attempts && n_ok < a.batch;
       base += blockDim.x) {
    const int j = base + threadIdx.x;
    bool mine = false, ok = false;
    int64_t idx = 0;
    if (j < window) {
      const double u = philox_uniform53(a.seed, draw_offset, (uint64_t)j);
      int64_t o = (int64_t)(u * (double)total);
      if (o >= total) o = total - 1;
      int g = 0;
      while (g < a.world - 1 && o >= s_span[g]) o -= s_span[g++];
      if (g == a.rank) {
        mine = true;
        idx = wrap_index(min_id + o, c.capacity);  // `% replay_capacity`, CRB:466
        ok = is_valid_transition(c, idx);
      }
    }
    int tile_rej, tile_ok;
    const int rej_pos = n_rej + block_scan_flag(mine && !ok, warp_counts, &tile_rej);
    const int ok_pos = n_ok + block_scan_flag(mine && ok, warp_counts, &tile_ok);
    if (mine && !ok && rej_pos < a.max_attempts) s_rej[rej_pos] = j;
    if (mine && ok && ok_pos < a.batch && a.mode == kUniformSample) {
      a.own_j[ok_pos] = j;
      a.own_idx[ok_pos] = (int32_t)idx;
    }
    n_rej = min(n_rej + tile_rej, a.max_attempts);
    n_ok = min(n_ok + tile_ok, a.batch);
  }
  __syncthreads();

  // ---- round 2: the rejection list, unless a publish-ahead of this step has sent it
  const size_t parity_base = kRejWordsOffset + (size_t)(xseq & 1) * kMaxShards * kRejSlotWords;
  const size_t my_slot = parity_base + (size_t)a.rank * kRejSlotWords;
  if (a.mode == kUniformSample) {
    if (threadIdx.x == 0) {
      const uint64_t w = ld_sys_u64(a.xchg.local + my_slot);
      if ((uint32_t)w == (uint32_t)xseq) {
        s_published = 1;
        if ((int32_t)(w >> 32) != n_rej) s_stale = 1;
      }
    }
    __syncthreads();
    // published ahead: it must be what this launch found (else the buffer changed in
    // between and the peers decided on another list)
    if (s_published)
      for (int k = threadIdx.x; k < n_rej; k += blockDim.x)
        if (ld_sys_u64(a.xchg.local + my_slot + 1 + k) != rej_word(s_rej[k], xseq)) s_stale = 1;
  }
  if (!s_published) {
    const int words = 1 + n_rej;
    for (int t = threadIdx.x; t < a.world * words; t += blockDim.x) {
      const int g = t / words, k = t - g * words;
      uint64_t *box = g == a.rank ? a.xchg.local : a.xchg.peer[g];
      st_sys_u64(box + my_slot + k, rej_word(k == 0 ? n_rej : s_rej[k - 1], xseq));
    }
  }
  if (a.mode == kUniformPublishRejections) return;
  __syncthreads();
  if (threadIdx.x == 0 && s_stale && a.latched && a.latched[0] == 0) {
    a.latched[0] = B2R_ERR_STALE_TOTAL;
    a.latched[1] = a.rank;
  }

  // ---- the peers' lists: counts, then every ordinal (each word polled for its tag)
  if (threadIdx.x < a.world) {
    const int g = threadIdx.x;
    int cnt = n_rej;
    if (g != a.rank) {
      cnt = poll_rej_word(a.xchg, a.xchg.local + parity_base + (size_t)g * kRejSlotWords,
                          xseq, g, 0, a.latched);
      cnt = min(max(cnt, 0), a.max_attempts);
    }
    s_start[g + 1] = cnt;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    s_start[0] = 0;
    for (int g = 0; g < a.world; ++g) s_start[g + 1] += s_start[g];
  }
  __syncthreads();
  const int n_lists = s_start[a.world];
  for (int t = threadIdx.x; t < n_lists; t += blockDim.x) {
    int g = 0;
    while (s_start[g + 1] <= t) ++g;
    const int k = t - s_start[g];
    a.lists[t] = g == a.rank
                     ? s_rej[k]
                     : poll_rej_word(a.xchg,
                                     a.xchg.local + parity_base + (size_t)g * kRejSlotWords +
                                         1 + k,
                                     xseq, g, window, a.latched);
  }
  __syncthreads();
  // invalid draws before draw j, over every rank's list
  auto rejects_before = [&](int j) {
    int r = 0;
    for (int g = 0; g < a.world; ++g) {
      int lo = s_start[g], hi = s_start[g + 1];
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a.lists[mid] < j) lo = mid + 1; else hi = mid;
      }
      r += lo - s_start[g];
    }
    return r;
  };

  // ---- this rank's rows: the kept prefix of its valid draws
  int kept = 0;
  for (int k = threadIdx.x; k < n_ok; k += blockDim.x) {
    const int j = a.own_j[k];
    const int rb = rejects_before(j);
    if (j - rb < a.batch && rb < a.max_attempts) {
      ++kept;
      if (k < a.out_cap) {
        a.out_slots[k] = j - rb;
        a.out_idx[k] = a.own_idx[k];
      }
    }
  }
  if (kept) atomicAdd(&s_kept, kept);
  __syncthreads();
  if (threadIdx.x == 0) {
    // Did the loop end short (CRB:471-475)?  It stops at the max_attempts-th rejection
    // j_A - 1 if that comes before the batch is full: j_A - max_attempts accepted.
    int accepted = a.batch;
    if (n_lists >= a.max_attempts) {
      int lo = 0, hi = window;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (rejects_before(mid) >= a.max_attempts) hi = mid; else lo = mid + 1;
      }
      if (rejects_before(lo) >= a.max_attempts) accepted = min(accepted, lo - a.max_attempts);
    }
    const int rows = s_kept;
    *a.count_out = min(rows, a.out_cap);
    if (a.latched && a.latched[0] == 0) {
      if (accepted < a.batch) {
        a.latched[0] = B2R_ERR_SAMPLE_ATTEMPTS;
        a.latched[1] = accepted;
      } else if (rows > a.out_cap) {  // a share beyond the caller's outputs
        a.latched[0] = B2R_ERR_UNSUPPORTED;
        a.latched[1] = rows;
      }
    }
    *a.xchg.seq = xseq;
  }
}

}  // namespace

int check_uniform_sharded(const b2r_buffer *b, const b2r_exchange *x, int32_t global_batch) {
  if (!b) return fail(B2R_ERR_INVALID_ARGUMENT, "buffer is NULL");
  if (!x) return fail(B2R_ERR_INVALID_ARGUMENT, "exchange is NULL");
  if (global_batch < 1 || global_batch > 60000)
    return fail(B2R_ERR_INVALID_ARGUMENT, "global_batch must be in [1, 60000]");
  if (x->early_publish)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "the exchange has early publish on: it would send tree totals where the "
                "uniform sampler exchanges spans");
  if (!x->connected) return fail(B2R_ERR_INVALID_ARGUMENT, "the exchange is not connected");
  if (b->cfg.max_sample_attempts > kRejListWords)
    return fail(B2R_ERR_UNSUPPORTED,
                "max_sample_attempts %d is above %d, the rejection list a shard can publish",
                b->cfg.max_sample_attempts, kRejListWords);
  return B2R_OK;
}

int launch_uniform_sharded(b2r_buffer *b, const b2r_exchange *x, int32_t global_batch,
                           uint64_t seed, uint64_t offset, int mode, int32_t *out_idx,
                           int32_t *out_slots, int32_t *out_count, int32_t out_cap,
                           cudaStream_t s) {
  B2R_TRY(flush_queue(b, s));
  B2R_TRY(ensure_ctx(b, s));
  B2R_TRY(ensure_inv_slots(b, 2 * (int64_t)global_batch + (int64_t)x->world * kRejListWords));
  UniformShardArgs a;
  a.valid_dev = b->ctx_dev;
  fill_exchange_args(x, &a.xchg);
  a.world = x->world;
  a.rank = x->rank;
  a.batch = global_batch;
  a.max_attempts = b->cfg.max_sample_attempts > 0 ? b->cfg.max_sample_attempts : 0;
  a.seed = seed;
  a.offset = offset;
  a.mode = mode;
  a.out_cap = out_cap;
  a.out_idx = out_idx;
  a.out_slots = out_slots;
  a.count_out = out_count;
  a.own_j = b->inv_slots;
  a.own_idx = a.own_j + global_batch;
  a.lists = a.own_idx + global_batch;
  a.latched = b->status;
  B2R_CUDA(launch(uniform_sharded_kernel, dim3(1), dim3(kUniformShardThreads), 0, s, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" {

int b2r_uniform_bounds(const b2r_buffer *b, int64_t *min_id, int64_t *max_id) {
  return b2r::uniform_bounds(b, min_id, max_id);
}

int b2r_sample_indices_uniform(b2r_buffer *b, int32_t batch, int32_t n_cand,
                               const int64_t *candidates, int32_t *out_indices,
                               int32_t *accepted, int32_t *rejected,
                               int32_t *draws_used, b2r_stream stream) {
  if (batch <= 0 || n_cand < 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad batch / candidate count");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  // bounce layout: [candidates n_cand*8][out batch*4][counters 16]
  const size_t off_out = (size_t)n_cand * 8;
  const size_t off_cnt = off_out + (((size_t)batch * 4 + 15) & ~(size_t)15);
  B2R_TRY(b->bounce.reserve(off_cnt + 16));
  memcpy(b->bounce.host, candidates, (size_t)n_cand * 8);
  // Earlier windows already filled out_indices[0 .. *accepted).
  memcpy(b->bounce.host + off_out, out_indices, (size_t)batch * 4);
  int32_t cnt[4] = {*accepted, *rejected, 0, 0};
  memcpy(b->bounce.host + off_cnt, cnt, 16);
  B2R_CUDA(cudaMemcpyAsync(b->bounce.dev, b->bounce.host, off_cnt + 16,
                           cudaMemcpyHostToDevice, s));
  B2R_TRY(b2r::ensure_ctx(b, s));
  B2R_TRY(b2r::launch_uniform_sample(
      b, batch, 0, 0, n_cand, reinterpret_cast<const int64_t *>(b->bounce.dev),
      reinterpret_cast<int32_t *>(b->bounce.dev + off_out),
      reinterpret_cast<int32_t *>(b->bounce.dev + off_cnt), s));
  B2R_CUDA(cudaMemcpyAsync(b->bounce.host + off_out, b->bounce.dev + off_out,
                           off_cnt + 16 - off_out, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  memcpy(out_indices, b->bounce.host + off_out, (size_t)batch * 4);
  memcpy(cnt, b->bounce.host + off_cnt, 16);
  *accepted = cnt[0];
  *rejected = cnt[1];
  *draws_used = cnt[2];
  return B2R_OK;
}

int b2r_sample_indices_prioritized(b2r_buffer *b, int32_t batch,
                                   const double *strat_query01, int32_t n_retry,
                                   const double *retry_u01,
                                   int32_t *out_indices, int32_t *draws_used,
                                   int32_t *fail_slot, b2r_stream stream) {
  if (!b->tree) return fail(B2R_ERR_UNSUPPORTED, "not a prioritized buffer");
  if (batch <= 0 || n_retry < 0)
    return fail(B2R_ERR_INVALID_ARGUMENT, "bad batch / retry count");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  // bounce layout: [strat batch*8][retry n_retry*8][out batch*4][info 16]
  const size_t off_retry = (size_t)batch * 8;
  const size_t off_out = off_retry + (size_t)n_retry * 8;
  const size_t off_info = off_out + (((size_t)batch * 4 + 15) & ~(size_t)15);
  B2R_TRY(b->bounce.reserve(off_info + 16));
  memcpy(b->bounce.host, strat_query01, (size_t)batch * 8);
  if (n_retry) memcpy(b->bounce.host + off_retry, retry_u01, (size_t)n_retry * 8);
  B2R_CUDA(cudaMemcpyAsync(b->bounce.dev, b->bounce.host, off_out,
                           cudaMemcpyHostToDevice, s));
  b2r::SampleRequest r;
  r.batch = batch;
  r.query01 = reinterpret_cast<const double *>(b->bounce.dev);
  r.retry_u01 = reinterpret_cast<const double *>(b->bounce.dev + off_retry);
  r.max_attempts = n_retry;
  r.latch = false;
  r.info = reinterpret_cast<int32_t *>(b->bounce.dev + off_info);
  r.out_idx = reinterpret_cast<int32_t *>(b->bounce.dev + off_out);
  B2R_TRY(b2r::launch_sample(b, r, s));
  B2R_CUDA(cudaMemcpyAsync(b->bounce.host + off_out, b->bounce.dev + off_out,
                           off_info + 16 - off_out, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  int32_t info[4];
  memcpy(info, b->bounce.host + off_info, 16);
  memcpy(out_indices, b->bounce.host + off_out, (size_t)batch * 4);
  *draws_used = info[2];
  *fail_slot = info[1];
  if (info[0] == B2R_ERR_EMPTY_TREE)
    return fail(B2R_ERR_EMPTY_TREE, "Cannot sample from an empty sum tree.");
  if (info[0] == B2R_ERR_SAMPLE_ATTEMPTS)
    return fail(B2R_ERR_SAMPLE_ATTEMPTS,
                "Max sample attempts: Tried %d times but only sampled %d valid "
                "indices. Batch size is %d",
                b->cfg.max_sample_attempts, info[1], batch);
  return B2R_OK;
}

int b2r_sample_indices_device(b2r_buffer *b, int32_t batch, uint64_t seed,
                              uint64_t offset, int32_t *out_indices,
                              b2r_stream stream) {
  if (batch <= 0) return fail(B2R_ERR_INVALID_ARGUMENT, "bad batch");
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::flush_queue(b, s));
  if (b->tree) {
    b2r::SampleRequest r;
    r.batch = batch;
    r.max_attempts = b->cfg.max_sample_attempts;
    r.seed = seed;
    r.offset = offset;
    r.counter = b->draw_counter;
    r.info = b->info;
    r.out_idx = out_indices;
    return b2r::launch_sample(b, r, s);
  }
  int64_t min_id, max_id;  // (the kernel recomputes them from the device context)
  B2R_TRY(b2r::uniform_bounds(b, &min_id, &max_id));
  B2R_TRY(b2r::ensure_ctx(b, s));
  B2R_CUDA(cudaMemsetAsync(b->info, 0, 16, s));
  return b2r::launch_uniform_sample(b, batch, seed, offset, 0, nullptr, out_indices, b->info,
                                    s);
}

int b2r_sample_indices_sharded_device(b2r_buffer *b, int32_t global_batch,
                                      int32_t num_shards, int32_t rank,
                                      const double *shard_totals,
                                      const double *query01, int32_t n_retry,
                                      const double *retry_u01, uint64_t seed,
                                      uint64_t offset, int32_t *out_slots,
                                      int32_t *out_indices, int32_t *out_count,
                                      b2r_stream stream) {
  if (!shard_totals) return fail(B2R_ERR_INVALID_ARGUMENT, "shard_totals is NULL");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  b2r::SampleRequest r = b2r::sharded_indices_request(
      b, global_batch, query01, n_retry, retry_u01, seed, offset, out_slots, out_indices,
      out_count);
  r.num_shards = num_shards;
  r.rank = rank;
  r.shard_totals = shard_totals;
  return b2r::launch_sample(b, r, as_stream(stream));
}

int b2r_sample_indices_sharded_p2p_device(b2r_buffer *b, b2r_exchange *x,
                                          int32_t global_batch,
                                          const double *query01, int32_t n_retry,
                                          const double *retry_u01, uint64_t seed,
                                          uint64_t offset, int32_t *out_slots,
                                          int32_t *out_indices, int32_t *out_count,
                                          b2r_stream stream) {
  if (!x) return fail(B2R_ERR_INVALID_ARGUMENT, "exchange is NULL");
  B2R_TRY(b2r::flush_queue(b, as_stream(stream)));
  b2r::SampleRequest r = b2r::sharded_indices_request(
      b, global_batch, query01, n_retry, retry_u01, seed, offset, out_slots, out_indices,
      out_count);
  r.num_shards = x->world;
  r.rank = x->rank;
  r.x = x;
  return b2r::launch_sample(b, r, as_stream(stream));
}

int b2r_sample_transition_batch_uniform_sharded_device(
    b2r_buffer *b, b2r_exchange *x, int32_t global_batch, uint64_t seed, uint64_t offset,
    const b2r_batch *out, int32_t *out_slots, int32_t *out_count, int32_t max_rows,
    b2r_stream stream) {
  if (!b) return fail(B2R_ERR_INVALID_ARGUMENT, "buffer is NULL");
  if (!x) return fail(B2R_ERR_INVALID_ARGUMENT, "exchange is NULL");
  if (!out || !out->indices)
    return fail(B2R_ERR_INVALID_ARGUMENT, "out and out->indices are required");
  if (!out_slots) return fail(B2R_ERR_INVALID_ARGUMENT, "out_slots is NULL");
  if (!out_count) return fail(B2R_ERR_INVALID_ARGUMENT, "out_count is NULL");
  if (max_rows < 0) return fail(B2R_ERR_INVALID_ARGUMENT, "max_rows must be >= 0");
  B2R_TRY(b2r::check_uniform_sharded(b, x, global_batch));
  const int32_t cap = max_rows > 0 && max_rows < global_batch ? max_rows : global_batch;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(b2r::launch_uniform_sharded(b, x, global_batch, seed, offset,
                                      b2r::kUniformSample, out->indices, out_slots,
                                      out_count, cap, s));
  return b2r::launch_gather(b, cap, out->indices, out, s, out_count);
}

}  // extern "C"

#ifdef B2R_TRACE
extern "C" int b2r_debug_trace_sample(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_trace, sizeof(long long) * 32);
}
#endif
