// GPU sum tree internals shared by tree.cu and replay.cu.
#pragma once

#include "common.cuh"

// Nodes live in ONE fp64 heap array in HBM, 1-based: node (level l, position i)
// at h = 2^l + i (root at 1, element 0 unused).  Level l is the contiguous slice
// [2^l, 2^(l+1)) and is exactly the reference's `nodes[l]` (sum_tree.py:79-87);
// the children of h are 2h and 2h+1, and the 4 grandchildren / 8
// great-grandchildren of a node start on 32 B / 64 B boundaries, which the
// speculative descent below relies on.  16 MB for capacity 1M: L2-resident.
namespace b2r {
// The tree kernels' hand-over words (tree.cu), zeroed at creation; each protocol re-arms
// its words for the next launch.
struct TreeSync {
  // tree_update_kernel: levels handed out in order of arrival, the leaf CTA's one-way
  // barrier flag and the count of levels past it
  unsigned int role_ticket, leaf_flag, level_arrivals, unused0;
  long long pending[2];  // failure of the leaf CTA: stop code, first entry not applied
  // tree_update_early_kernel: the leaf CTA's list of duplicates is out, CTAs that have
  // left, level CTAs that have their leaves; the launches' tickets (launch_ticket)
  unsigned int list_flag, ended, fetched, unused1;
  unsigned long long early_tickets;
  unsigned int go, completed;  // TreeGo
};
static_assert(offsetof(TreeSync, pending) % 8 == 0 &&
                  offsetof(TreeSync, early_tickets) % 8 == 0 &&
                  offsetof(TreeSync, go) == 56 && sizeof(TreeSync) == 64,
              "TreeSync keeps its word order");
}  // namespace b2r

struct b2r_tree {
  int64_t capacity = 0;
  int depth = 0;          // levels = depth + 1
  int64_t leaves = 0;     // 2^depth; leaf i sits at heap[leaves + i]
  double *heap = nullptr;
  double *max_rec = nullptr;   // device scalar: max_recorded_priority
  int64_t *status = nullptr;   // device [2]: latched error code, offending position
  double *delta = nullptr;     // device scratch: per-element leaf deltas of a chunk
  uint32_t *sorted = nullptr;  // device scratch: the early write-back's list of
                               // duplicate leaves (tree.cu: kEarly, DupInfo)
  b2r::TreeSync *sync = nullptr;  // device
  b2r::Bounce bounce;
};

struct b2r_exchange;

namespace b2r {

constexpr int kTreeChunk = 4096;   // elements sorted per CTA (64 KB of smem)
constexpr int kTopLevels = 10;     // levels 0..10 (heap[1..2048), 16 KB) staged in smem

// One step of sum_tree.py:128-139: strict `<` against the stored left child,
// subtract when going right.  __dsub_rn pins the rounding (no contraction).
__device__ __forceinline__ void descend_step(int64_t &h, double &q, double left) {
  if (q < left) {
    h = 2 * h;
  } else {
    h = 2 * h + 1;
    q = __dsub_rn(q, left);
  }
}

// K levels in ONE memory round trip: the left-child values of the next K levels
// (1 + 2 + ... + 2^(K-1) candidates; the 1-based layout keeps each level's
// candidates inside 2^(K-d) adjacent 32-byte sectors) are fetched together, then the
// K decisions are taken one after the other exactly as the reference takes them.
// Candidates are picked with unrolled selects, so everything stays in registers.
template <int COUNT>
__device__ __forceinline__ double select_candidate(const double (&c)[COUNT], int w) {
  double r = c[0];
#pragma unroll
  for (int j = 1; j < COUNT; ++j) r = (w == j) ? c[j] : r;
  return r;
}

// Loads issued through volatile asm keep their program order and cannot be sunk
// below the selects by the compiler, which is the whole point: all candidates of a
// round are in flight before the first decision is taken.
struct GlobalNodes {
  const double *base;
  __device__ __forceinline__ double operator()(int64_t h) const {
    double v;
    asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(base + h));
    return v;
  }
};
struct SharedNodes {
  uint32_t base;  // shared-space address of element 0
  __device__ __forceinline__ double operator()(int64_t h) const {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(base + (uint32_t)h * 8u));
    return v;
  }
};

__device__ __forceinline__ uint32_t low_bits(double v) {
  return (uint32_t)__double2loint(v);
}

// `zero` is a run-time 0 the compiler cannot see through: q is made to depend on the
// bits of every candidate (q.lo ^= xor(all) & zero), so neither nvcc nor ptxas can
// take the first decision - and stall the in-order issue - before all loads of the
// round have been issued.
template <int K, typename Nodes>
__device__ __forceinline__ void descend_levels(const Nodes &nodes, int64_t &h,
                                               double &q, uint32_t zero) {
  static_assert(K >= 1 && K <= 5, "K levels per round trip");
  const int64_t h0 = h;
  const double c1 = nodes(2 * h0);
  double c2[2], c3[4], c4[8], c5[16];
  if (K >= 2) {
#pragma unroll
    for (int j = 0; j < 2; ++j) c2[j] = nodes(4 * h0 + 2 * j);
  }
  if (K >= 3) {
#pragma unroll
    for (int j = 0; j < 4; ++j) c3[j] = nodes(8 * h0 + 2 * j);
  }
  if (K >= 4) {
#pragma unroll
    for (int j = 0; j < 8; ++j) c4[j] = nodes(16 * h0 + 2 * j);
  }
  if (K >= 5) {
#pragma unroll
    for (int j = 0; j < 16; ++j) c5[j] = nodes(32 * h0 + 2 * j);
  }
  if (K >= 3) {
    uint32_t g = low_bits(c1);
#pragma unroll
    for (int j = 0; j < 2; ++j) g ^= low_bits(c2[j]);
#pragma unroll
    for (int j = 0; j < 4; ++j) g ^= low_bits(c3[j]);
    if (K >= 4) {
#pragma unroll
      for (int j = 0; j < 8; ++j) g ^= low_bits(c4[j]);
    }
    if (K >= 5) {
#pragma unroll
      for (int j = 0; j < 16; ++j) g ^= low_bits(c5[j]);
    }
    q = __hiloint2double(__double2hiint(q), __double2loint(q) ^ (int)(g & zero));
  }
  descend_step(h, q, c1);
  if (K >= 2) descend_step(h, q, select_candidate<2>(c2, (int)(h - 2 * h0)));
  if (K >= 3) descend_step(h, q, select_candidate<4>(c3, (int)(h - 4 * h0)));
  if (K >= 4) descend_step(h, q, select_candidate<8>(c4, (int)(h - 8 * h0)));
  if (K >= 5) descend_step(h, q, select_candidate<16>(c5, (int)(h - 16 * h0)));
}

template <int K, typename Nodes>
__device__ __forceinline__ void descend_span(const Nodes &nodes, int64_t &h,
                                             double &q, int levels, uint32_t zero) {
#pragma unroll 1
  while (levels >= K) {
    descend_levels<K>(nodes, h, q, zero);
    levels -= K;
  }
  if (K > 4 && levels == 4) { descend_levels<4>(nodes, h, q, zero); levels = 0; }
  if (K > 3 && levels == 3) { descend_levels<3>(nodes, h, q, zero); levels = 0; }
  if (K > 2 && levels == 2) { descend_levels<2>(nodes, h, q, zero); levels = 0; }
  if (K > 1 && levels == 1) { descend_levels<1>(nodes, h, q, zero); levels = 0; }
}

// Root-to-leaf descent (sum_tree.py:126-141).  `top` is a shared-memory copy of
// heap[0 .. 2^(top_depth+1)): those levels are walked two per shared-memory round
// trip, the rest K per global-memory round trip.
template <int K>
__device__ __forceinline__ int64_t tree_descend_staged(
    const double *__restrict__ heap, const double *top, int top_depth, int depth,
    double q, uint32_t zero) {
  int64_t h = 1;
  const SharedNodes staged{(uint32_t)__cvta_generic_to_shared(top)};
  const GlobalNodes global{heap};
  descend_span<2>(staged, h, q, top_depth, zero);
  descend_span<K>(global, h, q, depth - top_depth, zero);
  return h - (((int64_t)1) << depth);
}

// Root-to-leaf descent by a whole WARP (sum_tree.py:126-141), up to 5 levels per
// memory round trip and nothing staged.  A round below node h0 needs the left children
// of 1 + 2 + 4 + 8 + 16 = 31 nodes: lane L fetches the one numbered L in breadth-first
// order (ONE load instruction for the warp).  Then lane p takes the K-bit path p as a
// hypothesis and replays the reference's K decisions along it — `q < left` goes left,
// else `q -= left` (rounded, __dsub_rn) goes right — checking at every level that the
// comparison agrees with its bit.  The decisions are deterministic, so exactly one lane
// is consistent on all K levels: its path is the reference's, its residual the
// reference's q.  The K subtractions of a lane depend on each other, the shuffles that
// feed them do not: a round costs one L2 round trip plus ~K dependent fp64 operations,
// against K dependent round trips for the textbook walk.  All lanes return the leaf.
// warp_candidate: the node lane `lane` fetches for a round of K levels below h.
__device__ __forceinline__ double warp_candidate(const double *__restrict__ heap,
                                                 int64_t h, int K, int lane) {
  const int d_me = 32 - __clz(lane + 1);               // level below h of my candidate
  const int prefix_me = lane + 1 - (1 << (d_me - 1));  // its position on that level
  return d_me <= K ? heap[(h << d_me) + 2 * prefix_me] : 0.0;
}

// One round: K levels walked from (h, q) over the candidates `c` of warp_candidate.
__device__ __forceinline__ void warp_walk(double c, int K, int lane, int64_t &h,
                                          double &q) {
  const unsigned full = 0xffffffffu;
  double r = q;
  bool ok;
  if (K == 5) {  // the usual round: sources and bits are per-lane constants
    ok = true;
    const double l1 = __shfl_sync(full, c, 0);
    const double l2 = __shfl_sync(full, c, 1 + (lane >> 4));
    const double l3 = __shfl_sync(full, c, 3 + (lane >> 3));
    const double l4 = __shfl_sync(full, c, 7 + (lane >> 2));
    const double l5 = __shfl_sync(full, c, 15 + (lane >> 1));
    const double left[5] = {l1, l2, l3, l4, l5};
#pragma unroll
    for (int d = 0; d < 5; ++d) {
      const bool lt = r < left[d];
      if ((lane >> (4 - d)) & 1) {
        ok = ok && !lt;
        r = __dsub_rn(r, left[d]);
      } else {
        ok = ok && lt;
      }
    }
  } else {
    ok = lane < (1 << K);
#pragma unroll
    for (int d = 1; d <= 4; ++d) {
      if (d <= K) {
        const int pre = lane >> (K - d + 1);  // the first d - 1 decisions of path `lane`
        const double left = __shfl_sync(full, c, ((1 << (d - 1)) - 1 + pre) & 31);
        if ((lane >> (K - d)) & 1) {
          ok = ok && !(r < left);
          r = __dsub_rn(r, left);
        } else {
          ok = ok && (r < left);
        }
      }
    }
  }
  const int w = __ffs(__ballot_sync(full, ok)) - 1;
  h = (h << K) + w;
  q = __shfl_sync(full, r, w);
}

// c_first: warp_candidate(heap, 1, min(depth, 5), lane), fetched by the caller ahead of
// time (it does not depend on q).
__device__ __forceinline__ int64_t tree_descend_warp(const double *__restrict__ heap,
                                                     int depth, double q, int lane,
                                                     double c_first) {
  int64_t h = 1;
  int level = 0;
  double c = c_first;
#pragma unroll 1
  while (true) {
    const int K = depth - level < 5 ? depth - level : 5;
    warp_walk(c, K, lane, h, q);
    level += K;
    if (level >= depth) break;
    c = warp_candidate(heap, h, depth - level < 5 ? depth - level : 5, lane);
  }
  return h - (((int64_t)1) << depth);
}

// Cooperative copy of heap[0 .. 2^(min(depth, kTopLevels)+1)) into shared memory:
// every thread issues all of its loads before the first store, so staging costs one
// memory round trip (needs blockDim.x >= 128).
__device__ __forceinline__ int stage_top_levels(const double *__restrict__ heap,
                                                int depth, double *top) {
  const int top_depth = depth < kTopLevels ? depth : kTopLevels;
  const int count = 2 << top_depth;
  // 8 independent loads in flight per thread and iteration: 256 threads stage the
  // 2048 nodes of levels 0..10 in ONE round trip (two with 4 loads per iteration).
#pragma unroll 1
  for (int i0 = threadIdx.x; i0 < count; i0 += 8 * blockDim.x) {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = i0 + j * blockDim.x;
      r[j] = i < count ? heap[i] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = i0 + j * blockDim.x;
      if (i < count) top[i] = r[j];
    }
  }
  __syncthreads();
  return top_depth;
}

// Shard totals exchanged through peer memory (sample.cu: exchange_collect; exchange.cu).
constexpr int kMaxShards = 16;
struct ExchangeArgs {
  uint64_t *local;             // this rank's mailbox [2 parities][world][2 words];
                               // nullptr: no exchange
  uint64_t *peer[kMaxShards];  // the peers' mailboxes (peer-mapped device pointers)
  uint64_t *seq;               // device step counter, in lockstep on all ranks
  int64_t timeout_ns;
  // [0] the step number this rank's total has been published for, [1] the published
  // bits.  A kernel that leaves the tree in its final state for the next sharded step
  // (the write-back, or the flush of staged adds behind it) publishes the new root right
  // away — the wire latency then hides behind the rest of that kernel, the kernel
  // boundary and the next sampler's prologue — and the sampler publishes only if nobody
  // has (pub[0] != its step number).
  uint64_t *pub;
};

#ifdef __CUDACC__
// All-gather of one fp64 per rank through peer memory (NVLink / NVSwitch), sending half:
// thread g (= threadIdx.x & 31 < world) stores this rank's root total straight into rank
// g's mailbox.  Each total travels as two 8-byte words that carry half of the payload and
// the step number in their low 32 bits (the flag is in-band, as in NCCL's LL protocol), so
// no fence or ordering between the stores is needed.  Mailbox slots alternate with the
// parity of the step: a rank can only be one step ahead of a peer, which has then
// finished reading the other parity.  The lane of this rank's own index records what was
// published (x.pub).
__device__ __forceinline__ void exchange_publish(const ExchangeArgs &x, int world,
                                                 int rank, double local_total,
                                                 uint64_t seq) {
  const int g = threadIdx.x & 31;
  if (g >= world) return;
  const uint64_t bits = (uint64_t)__double_as_longlong(local_total);
  if (g == rank) {
    if (x.pub != nullptr) {
      x.pub[1] = bits;
      x.pub[0] = seq;
    }
    return;
  }
  const uint32_t tag = (uint32_t)seq;
  uint64_t *dst = x.peer[g] + ((size_t)(seq & 1) * world + rank) * 2;
  st_sys_u64(dst, (bits & 0xffffffff00000000ull) | tag);
  st_sys_u64(dst + 1, (bits << 32) | tag);
}
#endif  // __CUDACC__

// Second region of a mailbox: the ranks' local minimum sampling probabilities of a step
// (the IS-weight normaliser of a sharded batch, read by b2r_c51_loss_sharded).  Layout
// [2 parities][world] words after the totals; a word is the f32 value in the high half
// and the step number in the low half, written with ONE 8-byte store.
constexpr int kMinWordsOffset = 2 * kMaxShards * 2;
// Third region: the rejection lists of the sharded uniform sampler (sample.cu:
// uniform_sharded_kernel).  Layout [2 parities][kMaxShards][1 count word + kRejListWords
// ordinal words]; every word is (value:32 | step:32), written with ONE 8-byte store, so a
// reader polls each word it needs until it carries the step's number.  kRejListWords
// bounds a buffer's max_sample_attempts (the reference's default is 1000).
constexpr int kRejWordsOffset = kMinWordsOffset + 2 * kMaxShards;
constexpr int kRejListWords = 1024;
constexpr int kRejSlotWords = 1 + kRejListWords;
constexpr int kMailboxWords = kRejWordsOffset + 2 * kMaxShards * kRejSlotWords;

#ifdef __CUDACC__
// Called by ONE thread: stores this rank's local minimum of step `seq` into every peer's
// mailbox (the own value stays with the caller: its min_probability).
__device__ __forceinline__ void exchange_publish_min(const ExchangeArgs &x, int world,
                                                     int rank, float local_min,
                                                     uint64_t seq) {
  const uint64_t word = ((uint64_t)__float_as_uint(local_min) << 32) | (uint32_t)seq;
  for (int g = 0; g < world; ++g)
    if (g != rank) st_sys_u64(x.peer[g] + kMinWordsOffset + (seq & 1) * world + rank, word);
}
#endif  // __CUDACC__

// "The sampled indices are final": what the kernel in front of the early write-back
// (tree.cu, kEarly) tells it through memory, so that the write-back can be resident and
// start on the indices the moment they are — a programmatic dependent launch would only
// START it then, 1.5 us later.  Every early write-back counts itself in `completed` when
// its last CTA leaves; the kernel in front — which runs when the write-back before this
// one has ended and this one cannot have — stores completed + 1, the number of the coming
// launch, in `go`; the CTAs of that launch know their number from the tickets they take
// (each before it lets ITS dependents start, so launches never interleave) and wait for
// exactly it.
struct TreeGo {
  const unsigned int *completed = nullptr;
  unsigned int *go = nullptr;  // nullptr: nothing to signal
};
#ifdef __CUDACC__
// (by one thread of the kernel in front, behind its griddepcontrol.wait)
__device__ __forceinline__ void tree_go_signal(const TreeGo &g) {
  if (g.go == nullptr) return;
  const unsigned int launch = *reinterpret_cast<const volatile unsigned int *>(g.completed) + 1u;
  st_release_u32(g.go, launch);
}
#endif

#ifdef __CUDACC__
// Arguments of the batched-set kernels (tree.cu; the tiny body below also runs in the
// C51 loss tail's cluster, c51.cu).
template <typename I, typename V>
struct UpdateArgs {
  double *heap;
  int depth;
  int64_t leaves;
  int n, padded;
  const I *indices;
  const V *values;
  const uint8_t *mode;
  int64_t k_base;
  double *delta;      // global scratch [n]: leaf deltas, produced by the leaf CTA
  double *max_rec;
  int64_t *status;
  const int32_t *n_dev;  // nullable: device-side element count of the whole batch
  // internal levels whose average chain (n >> level) is at least this long run their
  // ordered add-chains as a verified scan (chains_by_verified_scan); 0 = never
  int scan_min_chain = 0;
  // kFull: the whole update in tree_update_kernel.  kEarly (tree_update_early_kernel): ONE
  // launch that does the work that needs the INDICES only (grouping the entries by node)
  // ahead of its griddepcontrol.wait, beside the kernel that produces the values.  The
  // caller promises that the indices (and n_dev) were final before that kernel let its
  // dependents start.
  int phase = 0;
  // kEarly: the launch's tickets (always) and, when the kernel in front signals "indices
  // final" through memory instead of through its end, the word to wait on (TreeGo)
  unsigned long long *tickets = nullptr;
  unsigned int *go = nullptr;
  uint32_t *sorted = nullptr;  // kEarly: b2r_tree::sorted
  TreeSync *sync = nullptr;
  // Sharded replay: this launch leaves the tree final for the next sharded step, so the
  // warp that writes the root publishes it to the peers (ExchangeArgs::pub; one-CTA
  // kernels only).  nullptr: nothing to publish.
  const ExchangeArgs *publish = nullptr;
  int publish_world = 0, publish_rank = 0;
  // One-CTA kernels: *skip_flag != 0 — the update has been applied already (the loss tail
  // of a shard's step did it, c51.cu) — means return at once, re-arming the flag.
  unsigned int *skip_flag = nullptr;
};

// Called by every lane of the warp that owns tree level 0, after its store of the root.
template <typename I, typename V>
__device__ __forceinline__ void publish_root(const UpdateArgs<I, V> &a) {
  if (a.publish == nullptr) return;
  __syncwarp();
  const double root = *reinterpret_cast<volatile double *>(a.heap + 1);
  exchange_publish(*a.publish, a.publish_world, a.publish_rank, root, *a.publish->seq + 1);
}
constexpr int kFull = 0, kEarly = 3;

// At most 32 sets (the agent's batch, an add flush): entry k lives in lane k of every
// warp, warp l owns tree level l, and nothing is sorted.  __match_any_sync groups the
// lanes whose entries share a node; the lowest lane of a group adds the group's deltas
// in lane (= batch) order, fed by shuffles that do not depend on the running sum, so a
// level costs its longest chain of DADDs and no more.  The leaf warp resolves duplicate
// leaves the same way (delta = value - leaf; leaf += delta, sum_tree.py:196-202) and
// publishes the deltas through shared memory; every other warp has its node values in
// flight before that barrier.
constexpr int kTinyBatch = 32;

// The update in two halves, so that a kernel which PRODUCES the values (c51.cu: the
// loss tail of the fused step) can have every tree load in flight before it starts on
// them: tiny_issue needs the indices only; tiny_finish takes the entry's value.
struct TinyLoads {
  int n;
  int64_t latched, idx, node;
  bool in, use_max, idx_ok;
  double node_val;
  double recorded;    // max_recorded_priority as stored (leaf warp)
  unsigned same_all;  // lanes whose entries share this lane's node, all in-range entries
                      // taken as applied (the usual case; else regrouped in the finish)
};

template <typename I, typename V>
__device__ __forceinline__ void tree_update_tiny_issue(const UpdateArgs<I, V> &a, int level,
                                                       int lane, TinyLoads *t) {
  t->n = a.n;
  if (a.n_dev) t->n = min(t->n, max(*a.n_dev, 0));
  t->latched = a.status[0];
  const int shift = a.depth - level;
  const int64_t base = ((int64_t)1) << level;
  t->in = lane < t->n && level <= a.depth;
  t->idx = t->in ? (int64_t)a.indices[lane] : 0;
  t->use_max = t->in && a.mode != nullptr && a.mode[lane] != 0;
  t->idx_ok = t->in && t->idx >= 0 && t->idx < a.leaves;
  // every lane fetches the node its entry sits under (group mates fetch the same word)
  t->node = t->idx_ok ? (t->idx >> shift) : 0;
  t->node_val = t->idx_ok ? a.heap[base + t->node] : 0.0;
  t->recorded = (level == a.depth && lane == 0) ? *a.max_rec : 0.0;
  // grouping needs the indices only: done here, off the path that waits for the values
  t->same_all = __match_any_sync(0xffffffffu, t->idx_ok ? (long long)t->node : -1ll - lane);
}

// Every warp of the block must call this (one block barrier inside); warps whose level
// lies beyond the tree's depth only take part in the barrier.
template <typename I, typename V>
__device__ __forceinline__ void tree_update_tiny_finish(const UpdateArgs<I, V> &a, int level,
                                                        int lane, const TinyLoads &t,
                                                        double explicit_v) {
  __shared__ double s_delta[kTinyBatch];
  __shared__ int s_stop;
  const unsigned full = 0xffffffffu;
  const int n = t.n;
  const bool is_leaf = level == a.depth;
  const bool skip = level > a.depth || t.latched != 0;  // an earlier chunk failed: the
                                                        // sequence stopped there
  const int64_t base = ((int64_t)1) << (level <= a.depth ? level : 0);
  const bool in = t.in, use_max = t.use_max, idx_ok = t.idx_ok;
  const int64_t idx = t.idx, node = t.node;
  const double node_val = t.node_val;
  // (leaf warp, kept for after the barrier: what the other levels do not wait for)
  double v = explicit_v, recorded = 0.0;
  int n_eff_leaf = n;
  unsigned bad_mask = 0;

  if (is_leaf && !skip) {
    // v_k = mode ? max(max_recorded, explicit values before k) : value_k
    // (stage_mode_values), the first entry the reference would raise on, and
    // max_recorded_priority over the applied prefix.
    recorded = __shfl_sync(full, t.recorded, 0);
    if (a.mode != nullptr) {
      double x = (in && !use_max) ? explicit_v : -INFINITY;  // inclusive prefix max
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(full, x, o);
        if (lane >= o) x = fmax(x, y);
      }
      double before = __shfl_up_sync(full, x, 1);
      if (lane == 0) before = -INFINITY;
      v = use_max ? fmax(recorded, before) : explicit_v;
    }
    const bool bad = in && (v < 0.0 || !idx_ok);
    bad_mask = __ballot_sync(full, bad);
    const int n_eff = bad_mask ? __ffs(bad_mask) - 1 : n;
    n_eff_leaf = n_eff;
    const bool live = lane < n_eff;
    // lanes that share a leaf: the lowest walks the group in batch order
    unsigned same = t.same_all;
    if (bad_mask != 0)  // (entries from the first refused one on are not applied)
      same = __match_any_sync(full, live ? (long long)idx : -1ll - lane);
    double delta = __dsub_rn(v, node_val);
    double leaf = __dadd_rn(node_val, delta);
    if (__any_sync(full, live && (same & (same - 1)) != 0)) {
      // duplicate leaves: every lane replays its group's chain from the stored leaf
      double run = node_val;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const double vj = __shfl_sync(full, v, j);
        if ((same >> j) & 1u) {
          const double dj = __dsub_rn(vj, run);
          run = __dadd_rn(run, dj);
          if (j == lane) delta = dj;
        }
      }
      leaf = run;  // the group's final leaf, in every lane of the group
    }
    if (live) {
      s_delta[lane] = delta;
      if (lane == __ffs(same) - 1) a.heap[base + idx] = leaf;
    }
    if (lane == 0) s_stop = n_eff;
  }
  __syncthreads();  // deltas and n_eff are in shared memory
  if (skip) return;
  if (is_leaf) {
    // max_recorded_priority over the applied prefix and the code of the failure: value
    // first (sum_tree.py:191-193), else the index — nobody waits for these
    const bool live = lane < n_eff_leaf;
    double vmax = live ? v : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(full, vmax, o));
    const double bad_v = __shfl_sync(full, v, bad_mask ? __ffs(bad_mask) - 1 : 0);
    if (lane == 0) {
      if (n_eff_leaf > 0 && vmax > recorded) *a.max_rec = vmax;
      if (n_eff_leaf < n) {
        a.status[0] = bad_v < 0.0 ? B2R_ERR_NEGATIVE_PRIORITY : B2R_ERR_INDEX_RANGE;
        a.status[1] = a.k_base + n_eff_leaf;
      }
    }
    return;
  }
  const int n_eff = s_stop;
  const bool live = lane < n_eff;
  const double d = live ? s_delta[lane] : 0.0;
  unsigned same = t.same_all;
  if (n_eff < n)  // a refused entry: regroup over the applied prefix
    same = __match_any_sync(full, live ? (long long)node : -1ll - lane);
  double acc = __dadd_rn(node_val, d);
  if (__any_sync(full, live && (same & (same - 1)) != 0)) {
    acc = node_val;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const double dj = __shfl_sync(full, d, j);
      if ((same >> j) & 1u) acc = __dadd_rn(acc, dj);
    }
  }
  if (live && lane == __ffs(same) - 1) a.heap[base + node] = acc;
  if (level == 0) publish_root(a);
}

// PDL: the body opens a kernel of its own (programmatic dependent launch hand-shake);
// false when it runs at the tail of another kernel.
template <bool PDL, typename I, typename V>
__device__ __forceinline__ void tree_update_tiny_body(const UpdateArgs<I, V> &a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (PDL) {
    pdl_release();
    pdl_acquire();
  }
  TinyLoads t;
  tree_update_tiny_issue(a, warp, lane, &t);
  const double explicit_v = (t.in && !t.use_max) ? (double)a.values[lane] : 0.0;
  tree_update_tiny_finish(a, warp, lane, t, explicit_v);
}

#endif  // __CUDACC__

// Applies n sets in array order (device arrays).  mode (nullable): 1 = use the
// running max_recorded_priority instead of values[k].
// n_dev (nullable): device count, the effective n is min(n, *n_dev).
// expected_n (>= 0): how many entries the caller expects when only the device knows
// (n_dev); picks between the one-CTA and the cooperative kernel.
// phase: kFull = the whole update; kEarly = the early write-back, resident ahead of the
// values (tree_early_takes says whether this batch can; see UpdateArgs::phase).
// publish (nullable, one-CTA kernels only): the launch leaves the tree final for the next
// sharded step and publishes the new root to the exchange's peers.
template <typename I, typename V>
int tree_apply(b2r_tree *t, int64_t n, const I *indices, const V *values,
               const uint8_t *mode, cudaStream_t stream,
               const int32_t *n_dev = nullptr, int64_t expected_n = -1, int phase = 0,
               const b2r_exchange *publish = nullptr, unsigned int *skip_flag = nullptr,
               bool go_by_flag = false);
// What the kernel in front of an early write-back of `t` signals (go_by_flag).
TreeGo tree_go_of(b2r_tree *t);
bool tree_early_takes(int64_t n, int64_t expected_n);
// c51.cu: the loss in two halves (the fused step): what depends on the network outputs
// alone, over `rows` rows, into scratch ([rows][c51_scratch_floats_per_row()] floats),
// signalling `sync` when done ...
struct PreSync;
struct StageGate;
bool c51_can_split(const b2r_c51_args *args);
int c51_scratch_floats_per_row();
// Can the tail of this batch stage its inputs ahead of the sampler's end (StageGate)?
// (Also needs the tail and the write-back as one cluster: c51_post_takes_tree.)
bool c51_tail_can_stage(const b2r_c51_args *args);
// online_src / online_copy (nullable): read the online logits from there (the caller's
// page-locked host memory) and leave a device copy for the tail.
// stage (nullable): also leave every action's log-probabilities for a staged tail.
int c51_pre_launch(const b2r_c51_args *args, int rows, float *scratch, const PreSync &sync,
                   cudaStream_t stream, int *have_stats, const float *online_src = nullptr,
                   float *online_copy = nullptr, const StageGate *stage = nullptr);
// ... and the tail over the sampled rows.  err (nullable): asynchronous error latch.
// tree != nullptr (c51_post_takes_tree: batches of at most 32 rows): the tail and
// set_priority(indices, priorities) as one thread-block cluster.
// (expected_rows >= 0: a shard's step with a device-side row count — the cluster applies
// the write-back when the count turns out to be at most 32 and says so in *tree_done; the
// one-CTA tree kernel launched behind it with the same flag then returns at once.)
bool c51_post_takes_tree(const b2r_c51_args *args, const b2r_tree *tree,
                         int64_t expected_rows = -1);
int c51_post_launch(const b2r_c51_args *args, const float *scratch, int have_stats,
                    cudaStream_t stream, int64_t *err, int32_t *count_copy = nullptr,
                    b2r_tree *tree = nullptr, const int32_t *indices = nullptr,
                    unsigned int *tree_done = nullptr,
                    const b2r_exchange *publish = nullptr, float *loss_host = nullptr,
                    const TreeGo *go = nullptr, const StageGate *stage = nullptr);

}  // namespace b2r
