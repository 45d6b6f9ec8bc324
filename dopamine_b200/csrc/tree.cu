// GPU sum tree: replaces dopamine/replay_memory/sum_tree.py (SumTree).
//
// Bit-exactness contract.  The reference's `set` (sum_tree.py:178-205) computes
// delta = value - leaf once and adds it to the node on every level, so internal
// nodes are history-dependent fp64 sums, not left+right.  A batch of sets
// (prioritized_replay_buffer.py:213-214) is a sequential loop, so for every node
// the deltas of the batch elements below it must be added IN BATCH ORDER.
//
// ONE cooperative launch per chunk of <= 4096 sets, one CTA per tree level (see
// tree_update_kernel): every CTA groups the entries by node with a stable radix
// sort in shared memory, the leaf CTA resolves duplicate leaves as chains and
// publishes delta[k], a grid barrier, then each internal CTA adds the deltas of every
// touched node in batch order: as a prefix scan that is kept only if it reproduces the
// sequential recurrence bit for bit on the upper levels (chains_by_verified_scan),
// as serial fp64 add-chains elsewhere and whenever the scan does not verify.
//
// The root's chain of n dependent DADDs used to be the critical path (25 us at
// n = 4096); with the verified scan it is the deepest levels' radix sort before the
// barrier.  Bandwidth is irrelevant here (n * depth * 16 bytes).
//
// The fused step's write-back of 33 .. 512 rows is a second kernel over the same pieces
// (tree_update_early_kernel, further down): resident beside the loss kernel, it does
// everything that needs the indices only ahead of the values and nothing that needs
// another CTA behind them.
#include "replay.cuh"

#include <cooperative_groups.h>
#include <cub/block/block_radix_sort.cuh>

#include <cstdlib>
#include <new>

namespace cg = cooperative_groups;

namespace b2r {
namespace {

B2R_TRACE_DECL

constexpr uint64_t kPadKey = ~0ull;

// (trace builds) a mark by the CTA that took tree level `lv` in tree_update_kernel
#define B2R_MARK_LVL(i, lv) B2R_MARK_IF(i, level == (lv))
// (trace builds) per-level times of the write-back: [what][level]
#ifdef B2R_TRACE
static __device__ unsigned long long g_trace_count[8];
#define B2R_TRACE_COUNT(i, cond)                                          \
  do {                                                                    \
    if ((cond) && threadIdx.x == 0) atomicAdd(&g_trace_count[i], 1ull);  \
  } while (0)
static __device__ long long g_level_trace[4][32];
static __device__ long long g_phase_trace[2][16];
// who: 0 = the leaf CTA, 1 = the CTA of level 10, else not traced
#define B2R_PHASE(who, i)                                                          \
  do {                                                                             \
    if (threadIdx.x == 0 && (unsigned)(who) < 2u) g_phase_trace[who][i] = b2r_now(); \
  } while (0)
#define B2R_LEVEL_TIME(what, lv)                                      \
  do {                                                                \
    if (threadIdx.x == 0) g_level_trace[what][(lv) & 31] = b2r_now(); \
  } while (0)
#else
#define B2R_LEVEL_TIME(what, lv) \
  do {                           \
  } while (0)
#define B2R_TRACE_COUNT(i, cond) \
  do {                           \
  } while (0)
#define B2R_PHASE(who, i) \
  do {                    \
  } while (0)
#endif




// Add-path batches may ask for "whatever max_recorded_priority is when this entry
// is applied" (mode[k] != 0, rainbow_agent.py:330-334).  Sequentially that is
//   v = mode ? running : value;  stop if v < 0 or the index is out of range;
//   running = max(running, v)
// Entries that take the running maximum never raise it, so v_k = mode_k ?
// max(max_rec, explicit values before k) : value_k: an exclusive prefix maximum,
// evaluated by warp 0 with shuffles, 32 entries per round (one round trip of loads
// instead of a chain of dependent ones).
template <typename I, typename V>
__device__ __forceinline__ void stage_mode_values(const UpdateArgs<I, V> &a, int n,
                                                  double *vals, int *s_stop,
                                                  int *s_stop_code) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  double running = *a.max_rec;
  for (int base = 0; base < n; base += 32) {
    const int k = base + lane;
    const bool in = k < n;
    const bool use_max = in && a.mode[k] != 0;
    const double v = (in && !use_max) ? (double)a.values[k] : 0.0;
    const int64_t idx = in ? (int64_t)a.indices[k] : 0;
    double x = (in && !use_max) ? v : -INFINITY;  // inclusive prefix max of explicit values
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x = fmax(x, y);
    }
    double before = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) before = -INFINITY;
    const double vk = use_max ? fmax(running, before) : v;
    const bool bad = in && (vk < 0.0 || idx < 0 || idx >= a.leaves);
    const unsigned bad_mask = __ballot_sync(0xffffffffu, bad);
    if (in) vals[k] = vk;
    if (bad_mask) {
      const int first = __ffs(bad_mask) - 1;
      if (lane == first) {
        *s_stop = base + first;
        *s_stop_code = vk < 0.0 ? B2R_ERR_NEGATIVE_PRIORITY : B2R_ERR_INDEX_RANGE;
      }
      break;
    }
    running = fmax(running, __shfl_sync(0xffffffffu, x, 31));
  }
}

// ONE cooperative launch, grid = depth + 1 CTAs (CTA l owns level l, CTA `depth`
// the leaves).  Every CTA groups the chunk's elements by their node on its level
// with a STABLE block radix sort over the node index only (the elements start in
// batch order, so each group stays in batch order; level l sorts l bits, the root
// nothing); the leaf CTA then resolves the per-leaf chains and publishes delta[k];
// after one grid-wide barrier each internal CTA adds the deltas that fall under
// each of its nodes in batch order.  Critical path: the leaf CTA's sort + the
// root's chain of n dependent DADDs.
// Geometry of the cooperative kernel: THREADS x ITEMS entries per chunk.  Two
// instances: 1024 x 4 for chunks of up to 4096 entries, 256 x 4 for batches of up to
// 1024 (a radix pass over 1024 slots costs a fraction of one over 4096, and every
// level pays its passes before it can apply the deltas).
template <int THREADS, int ITEMS>
struct BigCfg {
  static constexpr int kThreads = THREADS;
  static constexpr int kItems = ITEMS;
  static constexpr int kChunk = THREADS * ITEMS;
  static constexpr int kHashSlots = 2 * kChunk;  // load factor <= 0.5
  static constexpr int kHashBits = kChunk == 4096 ? 13 : (kChunk == 1024 ? 11 : -1);
  static_assert(kHashBits > 0 && (1 << kHashBits) == kHashSlots, "hash size");
  // duplicate-leaf entries the hashed leaf pass handles (one thread ranks each)
  static constexpr int kMaxDup = THREADS < 512 ? THREADS : 512;
  using Sort = cub::BlockRadixSort<uint32_t, THREADS, ITEMS, uint32_t>;
  struct GroupSmem {
    typename Sort::TempStorage sort;
    uint32_t node[kChunk];  // node index on this level, grouped
    uint32_t elem[kChunk];  // batch position k of the same entry
  };
  struct HashSmem {
    uint32_t key[kHashSlots];    // leaf index owning the slot
    uint32_t count[kHashSlots];  // entries of the chunk that hit it
  };
  struct Smem {
    union {
      GroupSmem g;
      HashSmem h;           // leaf CTA only, before (instead of) the sort
    };
    double vals[kChunk];    // value -> leaf delta (leaf CTA) / deltas in group order
  };
  // tree_update_early_kernel: what it stages ahead of the values, per entry k
  struct EarlySmem : Smem {
    uint32_t place[kChunk]; // its place in the list of duplicate leaves / all ones
    double leafv[kChunk];   // its leaf's value before the batch
    double nodev[kChunk];   // its node's value on the CTA's level
  };
};
using BigCfg4096 = BigCfg<1024, 4>;
using BigCfg1024 = BigCfg<256, 4>;
// kEarly, up to 1024 entries: one entry per thread.  These kernels are chains of dependent
// instructions (ncu: 13 cycles per instruction and warp, 2 warps per scheduler with
// 256 x 4); a thread with one entry runs a quarter of them and the schedulers have eight
// warps to pick from.
using BigCfgWide = BigCfg<1024, 1>;
static_assert(BigCfg4096::kChunk == kTreeChunk, "chunk size");

// Leaf pass without sorting.  The leaf deltas gate every other level (the root's
// chain of n dependent adds starts when they are published), so the leaf CTA avoids
// the 20-bit sort whenever it can: a shared-memory hash set finds the entries whose
// leaf occurs more than once in the chunk; all others are independent
// (delta = value - leaf, leaf += delta, sum_tree.py:196-202), and the few duplicates
// are ordered by (leaf, batch position) with a counting rank and walked as chains.
// Returns false (nothing written) when more than C::kMaxDup entries share leaves; the
// caller then takes the sorted path.
template <typename C, typename I, typename V>
__device__ __forceinline__ bool leaf_deltas_hashed(const UpdateArgs<I, V> &a, int n_eff,
                                                   typename C::HashSmem &h,
                                                   double *vals) {
  constexpr int kBigItems = C::kItems, kBigThreads = C::kThreads;
  constexpr int kHashSlots = C::kHashSlots, kHashBits = C::kHashBits;
  constexpr int kMaxDup = C::kMaxDup;
  __shared__ uint32_t d_idx[kMaxDup], d_k[kMaxDup], ds_idx[kMaxDup], ds_k[kMaxDup];
  __shared__ int s_ndup;
  constexpr uint32_t kEmpty = 0xffffffffu;
  // every global load of the pass is issued before the hash set is touched: the
  // indices first, then the leaves they point at (in flight while the set fills)
  uint32_t my_idx[kBigItems], my_slot[kBigItems];
  double my_leaf[kBigItems];
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    const int k = threadIdx.x + j * kBigThreads;
    my_idx[j] = k < n_eff ? (uint32_t)a.indices[k] : kEmpty;
  }
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    my_leaf[j] = 0.0;
    my_slot[j] = 0;
    if (my_idx[j] != kEmpty) my_leaf[j] = a.heap[a.leaves + my_idx[j]];
  }
  for (int i = threadIdx.x; i < kHashSlots; i += blockDim.x) {
    h.key[i] = kEmpty;
    h.count[i] = 0;
  }
  if (threadIdx.x == 0) s_ndup = 0;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    if (my_idx[j] != kEmpty) {
      const uint32_t idx = my_idx[j];
      uint32_t slot = (idx * 2654435761u) >> (32 - kHashBits);
      while (true) {
        const uint32_t old = atomicCAS(&h.key[slot], kEmpty, idx);
        if (old == kEmpty || old == idx) break;
        slot = (slot + 1) & (kHashSlots - 1);
      }
      atomicAdd(&h.count[slot], 1u);
      my_slot[j] = slot;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    if (my_idx[j] != kEmpty && h.count[my_slot[j]] > 1) {
      const int pos = atomicAdd(&s_ndup, 1);
      if (pos < kMaxDup) {
        d_idx[pos] = my_idx[j];
        d_k[pos] = (uint32_t)(threadIdx.x + j * kBigThreads);
      }
    }
  }
  __syncthreads();
  const int ndup = s_ndup;
  if (ndup > kMaxDup) return false;
  // entries whose leaf is theirs alone
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    if (my_idx[j] != kEmpty && h.count[my_slot[j]] == 1) {
      const int k = threadIdx.x + j * kBigThreads;
      const double d = __dsub_rn(vals[k], my_leaf[j]);
      a.heap[a.leaves + my_idx[j]] = __dadd_rn(my_leaf[j], d);
      vals[k] = d;
    }
  }
  // duplicates: order by (leaf, batch position), one chain per leaf
  if ((int)threadIdx.x < ndup) {
    const uint64_t me = ((uint64_t)d_idx[threadIdx.x] << 32) | d_k[threadIdx.x];
    int rank = 0;
    for (int j = 0; j < ndup; ++j)
      rank += ((((uint64_t)d_idx[j] << 32) | d_k[j]) < me) ? 1 : 0;
    ds_idx[rank] = d_idx[threadIdx.x];
    ds_k[rank] = d_k[threadIdx.x];
  }
  __syncthreads();
  const int p = threadIdx.x;
  if (p < ndup && (p == 0 || ds_idx[p - 1] != ds_idx[p])) {
    const uint32_t idx = ds_idx[p];
    double leaf = a.heap[a.leaves + idx];
    for (int q = p; q < ndup && ds_idx[q] == idx; ++q) {
      const uint32_t k = ds_k[q];
      const double d = __dsub_rn(vals[k], leaf);
      leaf = __dadd_rn(leaf, d);
      vals[k] = d;
    }
    a.heap[a.leaves + idx] = leaf;
  }
  return true;
}

// Ordered fp64 add-chains without the serial dependence, when the data allow it.
//
// For every node the reference adds the deltas below it in batch order, rounding
// after each add (sum_tree.py:198-205); at the root that is a chain of n dependent
// DADDs (25 us at n = 4096), and fp64 addition is not associative, so a parallel
// prefix sum has no right to the same bits.  But it usually HAS them: priorities are
// f32 numbers cast to f64, so the deltas are multiples of 2^-32 or coarser while a
// node worth 2^20 has an ulp of 2^-33 — no add in the chain rounds at all, and any
// summation order gives the sequential result.  So: run a segmented prefix scan
// (segment = node, base = the node's stored value), then CHECK the sequential
// recurrence  P[p] == fl(P[p-1] + d[p])  at every position, bit for bit.  Positions
// inside a thread satisfy it by construction (the thread re-walks its ITEMS entries
// from its carry-in); what is checked is each thread's carry-in against the value its
// left neighbour actually ended on.  If all hold, induction from the segment heads
// makes P the sequential chain.  A carry that fails is replaced by a fresh segment
// head  fl(P[p-1] + d[p])  taken from the neighbour's verified value and the scan is
// repeated (every round fixes at least the first failure of each segment); after
// kScanRounds rounds the caller falls back to the serial chains, which have read and
// written nothing yet.  Returns true when the nodes were written.
constexpr int kScanRounds = 3;

template <typename C>
__device__ __forceinline__ bool chains_by_verified_scan(double *__restrict__ level_nodes,
                                                        const double *node_val,
                                                        const uint32_t *node,
                                                        const double *sorted_delta,
                                                        int n_eff) {
  constexpr int T = C::kThreads, ITEMS = C::kItems, WARPS = T / 32;
  static_assert(WARPS <= 32, "one warp scans the warp totals");
  __shared__ double s_last[T];
  __shared__ double s_wv[32];
  __shared__ int s_wf[32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  double d[ITEMS], hv[ITEMS], P[ITEMS];
  uint32_t nd[ITEMS];
  bool head[ITEMS];
  const int p0 = t * ITEMS;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const int p = p0 + j;
    const bool in = p < n_eff;
    nd[j] = in ? node[p] : 0xffffffffu;
    d[j] = in ? sorted_delta[p] : 0.0;
    const uint32_t before = j > 0 ? nd[j - 1] : (p > 0 && in ? node[p - 1] : 0xfffffffeu);
    head[j] = !in || before != nd[j];   // (pads are heads worth 0: they carry nothing)
    hv[j] = 0.0;
  }
#pragma unroll
  for (int j = 0; j < ITEMS; ++j)  // node_val[j]: the stored value of a head's node
    if (head[j] && p0 + j < n_eff) hv[j] = __dadd_rn(node_val[j], d[j]);
  const bool checked = t > 0 && p0 < n_eff && !head[0];  // takes a carry from the left
  bool promoted = false;
  bool ok = false;
#pragma unroll 1
  for (int round = 0; round < kScanRounds; ++round) {
    // the thread's entries as one scan element: (value, "contains a head")
    double v = head[0] ? hv[0] : d[0];
    int f = head[0] ? 1 : 0;
#pragma unroll
    for (int j = 1; j < ITEMS; ++j) {
      if (head[j]) {
        v = hv[j];
        f = 1;
      } else {
        v = __dadd_rn(v, d[j]);
      }
    }
    // inclusive segmented scan over the warp, then over the warp totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double v2 = __shfl_up_sync(0xffffffffu, v, o);
      const int f2 = __shfl_up_sync(0xffffffffu, f, o);
      if (lane >= o) {
        if (!f) v = __dadd_rn(v2, v);
        f |= f2;
      }
    }
    if (lane == 31) {
      s_wv[warp] = v;
      s_wf[warp] = f;
    }
    const double ev = __shfl_up_sync(0xffffffffu, v, 1);  // lanes before this one
    const int ef = __shfl_up_sync(0xffffffffu, f, 1);
    __syncthreads();
    if (warp == 0) {
      double wv = lane < WARPS ? s_wv[lane] : 0.0;
      int wf = lane < WARPS ? s_wf[lane] : 1;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double v2 = __shfl_up_sync(0xffffffffu, wv, o);
        const int f2 = __shfl_up_sync(0xffffffffu, wf, o);
        if (lane >= o) {
          if (!wf) wv = __dadd_rn(v2, wv);
          wf |= f2;
        }
      }
      s_wv[lane] = wv;
    }
    __syncthreads();
    double carry = 0.0;  // (thread 0 starts on a head and never uses it)
    if (lane > 0)
      carry = (ef || warp == 0) ? ev : __dadd_rn(s_wv[warp - 1], ev);
    else if (warp > 0)
      carry = s_wv[warp - 1];
    double acc = carry;
#pragma unroll
    for (int j = 0; j < ITEMS; ++j) {
      acc = head[j] ? hv[j] : __dadd_rn(acc, d[j]);
      P[j] = acc;
    }
    s_last[t] = acc;
    __syncthreads();
    bool bad = false;
    if (checked) {
      const double left = s_last[t - 1];
      if (promoted) {
        const double need = __dadd_rn(left, d[0]);
        if (__double_as_longlong(need) != __double_as_longlong(hv[0])) {
          hv[0] = need;
          bad = true;
        }
      } else if (__double_as_longlong(carry) != __double_as_longlong(left)) {
        promoted = true;
        head[0] = true;
        hv[0] = __dadd_rn(left, d[0]);
        bad = true;
      }
    }
    if (!__syncthreads_or(bad)) {
      ok = true;
      break;
    }
  }
  if (!ok) return false;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const int p = p0 + j;
    if (p < n_eff) {
      const uint32_t after = p + 1 < n_eff ? (j + 1 < ITEMS ? nd[j + 1] : node[p + 1])
                                           : 0xffffffffu;
      if (after != nd[j]) level_nodes[nd[j]] = P[j];
    }
  }
  return true;
}

// ---- the one-way barrier between the leaf CTA and the level CTAs ---------------------
// A failure is latched by the LAST level to pass (every CTA has read the latch by
// then: CTAs start whenever an SM has room, and one that started after the latch was
// set would skip the launch — and the barrier).
template <typename I, typename V>
__device__ __forceinline__ void leaf_publishes(const UpdateArgs<I, V> &a, int n, int n_eff,
                                               int stop_code) {
  long long *pending = a.sync->pending;
  if (threadIdx.x == 0) {
    pending[0] = n_eff < n ? stop_code : 0;
    pending[1] = a.k_base + n_eff;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) st_release_u32(&a.sync->leaf_flag, 1u);
  B2R_MARK_ANY(10);
}

// Returns (to every thread) the number of entries the leaf CTA applied.
template <typename I, typename V>
__device__ __forceinline__ int levels_wait_for_leaf(const UpdateArgs<I, V> &a) {
  const long long *pending = a.sync->pending;
  __shared__ int s_applied;
  if (threadIdx.x == 0) {
    const bool seen = poll_acquire(&a.sync->leaf_flag, [](unsigned v) { return v != 0u; });
    if (!seen && a.status[0] == 0) a.status[0] = B2R_ERR_CUDA;
    s_applied = seen ? (int)(pending[1] - a.k_base) : 0;
    // the last level to leave re-arms the flag for the next launch
    if (atomicInc(&a.sync->level_arrivals, (unsigned)a.depth - 1) == (unsigned)a.depth - 1) {
      a.sync->leaf_flag = 0u;
      if (pending[0] != 0 && a.status[0] == 0) {
        a.status[0] = pending[0];
        a.status[1] = pending[1];
      }
    }
  }
  __syncthreads();
  return s_applied;
}

// ---- an internal level behind the barrier: deltas in group order, then one ordered
// chain per node (sm.g.node / sm.g.elem hold the level's grouping, node_val the stored
// values of the nodes whose groups start at this thread's positions).
template <typename C, typename I, typename V>
__device__ __forceinline__ void internal_level_chains(const UpdateArgs<I, V> &a, int level,
                                                      int n_eff, typename C::Smem &sm,
                                                      const double *node_val) {
  constexpr int kBigItems = C::kItems;
  const int64_t base = ((int64_t)1) << level;
  double *vals = sm.vals;
  double *sorted_delta = vals;
  {
    double d[kBigItems];
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      const int p = threadIdx.x + j * C::kThreads;
      d[j] = p < n_eff ? __ldcg(a.delta + sm.g.elem[p]) : 0.0;
    }
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      const int p = threadIdx.x + j * C::kThreads;
      if (p < n_eff) sorted_delta[p] = d[j];
    }
  }
  __syncthreads();
  B2R_MARK_LVL(3, 0);
  B2R_MARK_LVL(20, 1);
  B2R_MARK_LVL(26, a.depth - 1);
  // long chains (the upper levels): verified scan; it declines when adds round
  if (a.scan_min_chain > 0 && (n_eff >> level) >= a.scan_min_chain &&
      chains_by_verified_scan<C>(a.heap + base, node_val, sm.g.node, sorted_delta,
                                 n_eff)) {
    B2R_MARK_LVL(4, 0);
    B2R_MARK_LVL(21, 1);
    B2R_MARK_LVL(27, a.depth - 1);
    B2R_MARK_END(15);
    return;
  }
  // serial chains: the thread that owns a group's first position walks the group
  int seg_end[kBigItems];
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    const int p = threadIdx.x * kBigItems + j;
    seg_end[j] = p;  // (empty: not a group start)
    if (p < n_eff) {
      const uint32_t node = sm.g.node[p];
      if (p == 0 || sm.g.node[p - 1] != node) {
        // first position whose node is larger: the neighbour, else a binary search
        int lo = p + 1, hi = n_eff;
        if (lo < hi && sm.g.node[lo] > node) hi = lo;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (sm.g.node[mid] > node) hi = mid; else lo = mid + 1;
        }
        seg_end[j] = lo;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    const int p = threadIdx.x * kBigItems + j;
    if (seg_end[j] > p) {
      double acc = node_val[j];
#pragma unroll 8
      for (int q = p; q < seg_end[j]; ++q) acc = __dadd_rn(acc, sorted_delta[q]);
      a.heap[base + sm.g.node[p]] = acc;
    }
  }
  B2R_MARK_LVL(4, 0);
  B2R_MARK_LVL(21, 1);
  B2R_MARK_LVL(27, a.depth - 1);
  B2R_MARK_END(15);
}


template <typename I, typename V, typename C>
__global__ void __launch_bounds__(C::kThreads) tree_update_kernel(UpdateArgs<I, V> a) {
  constexpr int kBigItems = C::kItems;
  using BigSort = typename C::Sort;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  typename C::Smem &sm = *reinterpret_cast<typename C::Smem *>(smem_raw);
  double *vals = sm.vals;
  __shared__ int s_stop;       // first position that must not be applied
  __shared__ int s_stop_code;
  __shared__ double s_max[32];

  // Levels are handed out in order of arrival, the leaf level first: the other CTAs
  // wait for its deltas at a flag (below), so the CTA they wait for is always one that
  // is already running — no cooperative launch, which would keep this kernel from
  // sharing the GPU with the frame copies of the same step (a cooperative grid starts
  // only once every CTA of it can be resident).
  __shared__ int s_role;
  B2R_MARK(13);
  pdl_release();
  pdl_acquire();
  if (threadIdx.x == 0) s_role = (int)atomicInc(&a.sync->role_ticket, (unsigned)a.depth);
  __syncthreads();
  const int level = s_role == 0 ? a.depth : s_role - 1;
  const bool is_leaf = level == a.depth;
  B2R_MARK_LVL(0, 0);
  B2R_MARK_LVL(16, a.depth);
  B2R_MARK_LVL(22, a.depth - 1);
  int n = a.n;
  if (a.n_dev) {
    const int64_t left = (int64_t)*a.n_dev - a.k_base;
    n = left < n ? (left > 0 ? (int)left : 0) : n;
  }
  // An earlier chunk failed: the reference's loop stopped there.  The latch is
  // only written after the grid barrier, so every CTA takes the same branch.
  if (a.status[0] != 0) return;
  // A chunk beyond the device-side count (sharded replay: the host launches for the
  // largest possible count) has nothing to do; every CTA sees the same n.
  if (n <= 0) return;
  if (threadIdx.x == 0) {
    s_stop = n;
    s_stop_code = 0;
  }
  __syncthreads();

  // 1. stage values; find the first element the reference would have raised on.
  //    (Redundant in every CTA: cheaper than a second barrier.)
  if (a.mode != nullptr) {
    // add-path batches may ask for "current max_recorded_priority": needs the
    // running maximum in order.  These batches are tiny; one thread walks them.
    stage_mode_values(a, n, vals, &s_stop, &s_stop_code);
  } else {
    // (every load of a thread is in flight before the first is used: one round trip)
    double v[kBigItems];
    int64_t ix[kBigItems];
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      const int k = threadIdx.x + j * C::kThreads;
      v[j] = k < n ? (double)a.values[k] : 0.0;
      ix[j] = k < n ? (int64_t)a.indices[k] : 0;
    }
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      const int k = threadIdx.x + j * C::kThreads;
      if (k < n) {
        vals[k] = v[j];
        if (v[j] < 0.0 || ix[j] < 0 || ix[j] >= a.leaves) atomicMin(&s_stop, k);
      }
    }
  }
  __syncthreads();
  const int n_eff = s_stop;
  if (a.mode == nullptr && n_eff < n && threadIdx.x == 0)
    s_stop_code = (vals[n_eff] < 0.0) ? B2R_ERR_NEGATIVE_PRIORITY
                                      : B2R_ERR_INDEX_RANGE;

  // 2. leaf CTA: the sort-free pass when duplicates are few (the usual case)
  B2R_MARK_LVL(17, a.depth);
  B2R_MARK_LVL(23, a.depth - 1);
  B2R_MARK_LVL(29, 0);
  bool leaf_done = false;
  if (is_leaf) {
    // max_recorded_priority = max(value, current) over the applied prefix
    // (before vals[] turns into deltas).
    double local_max = 0.0;
    for (int k = threadIdx.x; k < n_eff; k += blockDim.x)
      local_max = fmax(local_max, vals[k]);
    for (int off = 16; off > 0; off >>= 1)
      local_max = fmax(local_max, __shfl_xor_sync(0xffffffffu, local_max, off));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = local_max;
    leaf_done = leaf_deltas_hashed<C>(a, n_eff, sm.h, vals);
    __syncthreads();
  }

  // 3. group by node: thread t holds entries 4t .. 4t+3 (batch order); pads carry
  //    all-ones keys and sit behind every real entry, so they stay last.
  const int shift = a.depth - level;
  if (!leaf_done) {
    uint32_t key[kBigItems], val[kBigItems];
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      const int k = threadIdx.x * kBigItems + j;
      key[j] = k < n_eff ? (uint32_t)((int64_t)a.indices[k] >> shift) : 0xffffffffu;
      val[j] = (uint32_t)k;
    }
    if (level != 0) BigSort(sm.g.sort).Sort(key, val, 0, level);
#pragma unroll
    for (int j = 0; j < kBigItems; ++j) {
      sm.g.node[threadIdx.x * kBigItems + j] = key[j];
      sm.g.elem[threadIdx.x * kBigItems + j] = val[j];
    }
  }
  __syncthreads();
  B2R_MARK_LVL(18, a.depth);

  if (is_leaf) {
    if (!leaf_done) {
      // many duplicates: one thread per distinct leaf walks its chain in batch order
      //   delta = value - leaf; leaf += delta   (sum_tree.py:196-202, last level).
      // (the leaves of a thread's group heads are fetched together)
      double leaf0[kBigItems];
      bool head[kBigItems];
#pragma unroll
      for (int j = 0; j < kBigItems; ++j) {
        const int p = threadIdx.x + j * C::kThreads;
        head[j] = p < n_eff && (p == 0 || sm.g.node[p - 1] != sm.g.node[p]);
        leaf0[j] = head[j] ? a.heap[a.leaves + sm.g.node[p]] : 0.0;
      }
#pragma unroll
      for (int j = 0; j < kBigItems; ++j) {
        if (!head[j]) continue;
        const int p = threadIdx.x + j * C::kThreads;
        const uint32_t node = sm.g.node[p];
        double leaf = leaf0[j];
        for (int q = p; q < n_eff && sm.g.node[q] == node; ++q) {
          const uint32_t k = sm.g.elem[q];
          const double d = __dsub_rn(vals[k], leaf);
          leaf = __dadd_rn(leaf, d);
          vals[k] = d;
        }
        a.heap[a.leaves + node] = leaf;
      }
      __syncthreads();
    }
    for (int k = threadIdx.x; k < n_eff; k += blockDim.x) a.delta[k] = vals[k];
  }

  // Internal levels: thread t owns the grouped positions 4t .. 4t+3; the stored value
  // of every node whose group starts there is fetched now, so that its DRAM round
  // trip hides behind the wait for the leaf deltas (only this CTA writes this level).
  const int64_t base = ((int64_t)1) << level;
  double node_val[kBigItems];
#pragma unroll
  for (int j = 0; j < kBigItems; ++j) {
    const int p = threadIdx.x * kBigItems + j;
    node_val[j] = 0.0;
    if (!is_leaf && p < n_eff) {
      const uint32_t node = sm.g.node[p];
      if (p == 0 || sm.g.node[p - 1] != node) node_val[j] = a.heap[base + node];
    }
  }

  B2R_MARK_LVL(1, 0);
  B2R_MARK_LVL(19, a.depth);
  B2R_MARK_LVL(24, a.depth - 1);
  // ---- one-way barrier: the leaf CTA's deltas (and leaf writes) are published
  if (is_leaf) {
    leaf_publishes(a, n, n_eff, s_stop_code);
  } else {
    levels_wait_for_leaf(a);
    B2R_MARK_END(11);
  }
  B2R_MARK_LVL(2, 0);
  B2R_MARK_LVL(25, a.depth - 1);
  B2R_MARK_LVL(28, a.depth);

  if (is_leaf) {
    if (threadIdx.x == 0) {
      double m = *a.max_rec;
      for (int w = 0; w < (int)((blockDim.x + 31) >> 5); ++w)
        if (s_max[w] > m) m = s_max[w];
      if (n_eff > 0) *a.max_rec = m;
      if (n_eff < n && a.depth == 0) {  // (a one-node tree has no other level to latch)
        a.status[0] = s_stop_code;
        a.status[1] = a.k_base + n_eff;
      }
    }
    B2R_MARK_END(15);
    return;
  }

  // 3. internal level: deltas in group order, then one ordered chain per node.
  internal_level_chains<C>(a, level, n_eff, sm, node_val);
}

// ---- the same update with everything that needs only the INDICES done ahead of the
// values, and no hand-over between the CTAs behind them (kEarly).
//
// In the fused step the indices are final when the sampler ends and the values are what
// the loss tail between the sampler and this kernel produces.  This kernel is launched
// programmatically from the tail's first instruction, so it is RESIDENT while the tail
// works; the tail's first thread tells it through memory when the sampler has ended
// (TreeGo, tree.cuh).  Ahead of its own griddepcontrol.wait every CTA
//   * reads the indices and at once, per entry, its leaf and its node on the CTA's level;
//   * finds the entries that share a leaf with another entry, ordered by leaf and batch
//     position (the "list"), and groups the batch by node on its level.
//     The usual batch is grouped by leaf already but for a few entries
//     (nearly_sorted_analyse): two block scans and a binary search per moved entry, and
//     every CTA makes the list for itself (leaf_list_from_sorted).  Any other batch: the
//     leaf CTA makes the list with a hash set and hands it to the level CTAs through HBM
//     and a flag — a hand-over nobody is waiting for yet — while they group by radix sort.
// Behind the wait a level CTA needs nothing from any other CTA: an entry's delta is
// value - leaf (sum_tree.py:196-202) with the leaf as it was before the batch; the few
// entries that share leaves are chains  delta = value - leaf; leaf += delta  that every CTA
// walks for itself from the list.  One round trip for the values, the deltas, the ordered
// chains (or the verified scan), the stores.  (The plain kernel's leaf CTA publishes the
// deltas through HBM behind a fence and a flag: 4-5 us of that kernel's 11 at 1024.)
// When the list does not serve — more duplicates than it holds, or an entry the
// reference's loop would have raised on (negative priority, index out of range), so that
// only a prefix is applied — every CTA sees that for itself and the kernel goes on as the
// plain one does: leaf pass over the prefix, deltas through HBM, flag, regrouped levels.
// Only for callers that can promise that the indices are final when they say so
// (phase == kEarly: train_step, whose loss tail signals; or a predecessor that is not a
// programmatic launch at all, such as the copy in front of b2r_tree_set's test hook).
template <typename C>
struct LeafDupSmem {
  uint32_t d_idx[C::kMaxDup], d_k[C::kMaxDup], ds_idx[C::kMaxDup], ds_k[C::kMaxDup];
  int ndup;
};

// What the leaf CTA leaves in HBM for the level CTAs (words of UpdateArgs::sorted).
template <typename C>
struct DupInfo {
  static constexpr uint32_t kOverflow = 0xffffffffu;
  static constexpr int kCount = 0;                     // [1]: entries in the list / kOverflow
  static constexpr int kIdx = 16;                      // [kMaxDup]: leaf, in chain order
  static constexpr int kK = kIdx + C::kMaxDup;         // [kMaxDup]: batch position
  static constexpr int kOf = kK + C::kMaxDup;          // [chunk]: k -> place in the list / -1
  static constexpr int kLeaf = kOf + C::kChunk;        // [chunk] doubles: k -> its leaf's value
  static constexpr int kWords = kLeaf + 2 * C::kChunk;
  static_assert(kLeaf % 2 == 0, "doubles");
};

template <typename C>
struct LeafPrep {
  uint32_t idx[C::kItems];  // leaf index / 0xffffffff (pad, out of range)
  uint32_t k[C::kItems];    // batch position
  double leaf[C::kItems];   // the leaf's value
  bool single[C::kItems];   // no other entry of the batch has this leaf
};

// ---- a batch that is ALREADY grouped, but for a few entries.  The fused step's batch
// is: stratified queries grow with the stratum (sum_tree.py:162-166), the descent is
// monotone in the query, so row k's leaf — and with it its node on every level — never
// decreases with k; the exceptions are the rows whose pick was invalid and was drawn
// again (prioritized_replay_buffer.py:155-170), ~0.3 % of them.  Grouping by (node, k)
// is then the identity with a handful of entries moved, and costs two block scans and a
// few binary searches instead of a radix sort (5 passes at the deepest levels: what made
// the index-only half of this kernel longer than the loss kernel it runs beside).
//   * suspects: every entry that is larger than its right neighbour or smaller than its
//     left one (both ends of every descent: the culprit and, possibly, an innocent);
//   * the rest must be non-decreasing — checked against its running maximum, else (or
//     with more than kMaxMoved suspects) the caller sorts;
//   * a suspect's place: entries of the rest that sort before (key, k) — two binary
//     searches in the rest with the suspects' slots filled by the running maximum — plus
//     the suspects that do; an entry of the rest moves by the suspects that cross it.
constexpr int kMaxMoved = 64;

struct ScanSmem {
  // two sets, used in turn: a scan may start while slow warps still read the one before
  uint32_t wmax[2][32];
  int wsum[2][32];
};

// Exclusive block scan of (max, sum) over thread totals; *total = the sum of all.  ONE
// block barrier: every warp scans the 32 warp totals for itself.  `which`: 0, 1, 0, ...
// on successive calls of a kernel.
template <int T>
__device__ __forceinline__ void block_scan_max_sum(uint32_t tm, int ts, ScanSmem &ss,
                                                   int which, uint32_t *pm, int *ps,
                                                   int *total) {
  constexpr int WARPS = T / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t im = tm;
  int is = ts;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t um = __shfl_up_sync(0xffffffffu, im, o);
    const int us = __shfl_up_sync(0xffffffffu, is, o);
    if (lane >= o) {
      im = max(im, um);
      is += us;
    }
  }
  uint32_t em = __shfl_up_sync(0xffffffffu, im, 1);
  int es = __shfl_up_sync(0xffffffffu, is, 1);
  if (lane == 0) {
    em = 0u;
    es = 0;
  }
  if (lane == 31) {
    ss.wmax[which][warp] = im;
    ss.wsum[which][warp] = is;
  }
  __syncthreads();
  uint32_t wm = lane < WARPS ? ss.wmax[which][lane] : 0u;
  int ws = lane < WARPS ? ss.wsum[which][lane] : 0;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t um = __shfl_up_sync(0xffffffffu, wm, o);
    const int us = __shfl_up_sync(0xffffffffu, ws, o);
    if (lane >= o) {
      wm = max(wm, um);
      ws += us;
    }
  }
  const uint32_t before_m = __shfl_sync(0xffffffffu, wm, warp > 0 ? warp - 1 : 0);
  const int before_s = __shfl_sync(0xffffffffu, ws, warp > 0 ? warp - 1 : 0);
  *pm = warp > 0 ? max(before_m, em) : em;
  *ps = warp > 0 ? before_s + es : es;
  *total = __shfl_sync(0xffffffffu, ws, 31);
}

// What a thread keeps of the analysis for its entries kItems * t + j.
template <typename C>
struct NearlySorted {
  bool moved[C::kItems];
  int before_moved[C::kItems];  // suspects in front of the entry
  int n_moved;
};

// key[j]: the key of entry kItems * t + j (pads: all ones, behind every real entry).
// True: the batch is of that kind; `scratch` (at least kChunk + 2 * kMaxMoved words of
// shared memory) then holds the rest's keys with the suspects' slots filled, and the
// suspects.
template <typename C>
__device__ __forceinline__ bool nearly_sorted_analyse(const uint32_t *key, uint32_t *scratch,
                                                      ScanSmem &ss, NearlySorted<C> *ns) {
  constexpr int kItems = C::kItems, T = C::kThreads, kChunk = C::kChunk;
  uint32_t *c = scratch, *moved_k = scratch + kChunk, *moved_key = moved_k + kMaxMoved;
  const int k0 = threadIdx.x * kItems;
#pragma unroll
  for (int j = 0; j < kItems; ++j) c[k0 + j] = key[j];
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = k0 + j;
    const uint32_t left = j > 0 ? key[j - 1] : (k > 0 ? c[k - 1] : 0u);
    const uint32_t right = j + 1 < kItems ? key[j + 1] : (k + 1 < kChunk ? c[k + 1] : 0xffffffffu);
    ns->moved[j] = key[j] < left || key[j] > right;
  }
  // running maximum of the rest, running count of the suspects
  uint32_t before_max[kItems];
  uint32_t tm = 0u;
  int ts = 0;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    before_max[j] = tm;
    ns->before_moved[j] = ts;
    if (ns->moved[j]) ++ts; else tm = max(tm, key[j]);
  }
  uint32_t pm;
  int ps;
  block_scan_max_sum<T>(tm, ts, ss, 0, &pm, &ps, &ns->n_moved);  // (its barrier: c[] is read)
  bool unsorted = false;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    before_max[j] = max(before_max[j], pm);
    ns->before_moved[j] += ps;
    unsorted |= !ns->moved[j] && key[j] < before_max[j];
  }
  if (__syncthreads_or(unsorted || ns->n_moved > kMaxMoved)) return false;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (ns->moved[j]) {
      c[k0 + j] = before_max[j];
      moved_k[ns->before_moved[j]] = (uint32_t)(k0 + j);
      moved_key[ns->before_moved[j]] = key[j];
    }
  }
  __syncthreads();
  return true;
}

// Where the entries go when the batch is ordered by (key >> shift, k): the rest is in
// that order for every shift, and any superset of a level's suspects will do for it.
// A suspect's INSERTION POINT is the first slot of the batch that sorts behind it (slots
// of the rest carry their keys, the suspects' slots the running maximum: one monotone
// predicate, one binary search); an entry of the rest at slot k has exactly the suspects
// with an insertion point <= k in front of it, and a suspect the rest in front of its
// insertion point plus the suspects that sort before it.
// Two shifts at once (the leaves and the CTA's own level; the searches interleave):
// first nearly_sorted_insertions by every thread (a block barrier inside), then
// nearly_sorted_positions for either shift.
template <typename C>
__device__ __forceinline__ void nearly_sorted_insertions(const uint32_t *key, int shift_a,
                                                         int shift_b,
                                                         const NearlySorted<C> &ns,
                                                         uint32_t *scratch) {
  constexpr int kItems = C::kItems, kChunk = C::kChunk;
  const uint32_t *c = scratch;
  uint32_t *ip_a = scratch + kChunk + 2 * kMaxMoved, *ip_b = ip_a + kMaxMoved;
  const int k0 = threadIdx.x * kItems;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (!ns.moved[j]) continue;
    const int k = k0 + j;
    const uint32_t xa = key[j] >> shift_a, xb = key[j] >> shift_b;
    int lo_a = 0, hi_a = kChunk, lo_b = 0, hi_b = kChunk;
    while (lo_a < hi_a || lo_b < hi_b) {  // (same number of steps: same range)
      const int mid_a = (lo_a + hi_a) >> 1, mid_b = (lo_b + hi_b) >> 1;
      const uint32_t ca = c[mid_a < kChunk ? mid_a : kChunk - 1] >> shift_a;
      const uint32_t cb = c[mid_b < kChunk ? mid_b : kChunk - 1] >> shift_b;
      if (lo_a < hi_a) {
        if (ca > xa || (ca == xa && mid_a > k)) hi_a = mid_a; else lo_a = mid_a + 1;
      }
      if (lo_b < hi_b) {
        if (cb > xb || (cb == xb && mid_b > k)) hi_b = mid_b; else lo_b = mid_b + 1;
      }
    }
    ip_a[ns.before_moved[j]] = (uint32_t)lo_a;
    ip_b[ns.before_moved[j]] = (uint32_t)lo_b;
  }
  __syncthreads();
}

// pos[j]: where entry kItems * t + j goes (which = 0: shift_a's order, 1: shift_b's).
template <typename C>
__device__ __forceinline__ void nearly_sorted_positions(const uint32_t *key, int shift,
                                                        int which,
                                                        const NearlySorted<C> &ns,
                                                        const uint32_t *scratch, int *pos) {
  constexpr int kItems = C::kItems, kChunk = C::kChunk;
  const uint32_t *moved_k = scratch + kChunk, *moved_key = moved_k + kMaxMoved;
  const uint32_t *ip = scratch + kChunk + 2 * kMaxMoved + which * kMaxMoved;
  const int k0 = threadIdx.x * kItems;
  const int n_moved = ns.n_moved;
  bool any_moved = false;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    pos[j] = k0 + j - ns.before_moved[j];
    any_moved |= ns.moved[j];
  }
  for (int o = 0; o < n_moved; ++o) {  // (one load per suspect for the thread's entries)
    const int at = (int)ip[o];
#pragma unroll
    for (int j = 0; j < kItems; ++j) pos[j] += at <= k0 + j ? 1 : 0;
  }
  if (any_moved) {
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      if (!ns.moved[j]) continue;
      const uint32_t k = (uint32_t)(k0 + j), mine = key[j] >> shift;
      const int at = (int)ip[ns.before_moved[j]];
      int p = at;
      for (int o = 0; o < n_moved; ++o) {
        const uint32_t ok = moved_key[o] >> shift, kk = moved_k[o];
        p -= (int)kk < at ? 1 : 0;  // (a suspect's slot in front of the insertion point)
        p += (ok < mine || (ok == mine && kk < k)) ? 1 : 0;
      }
      pos[j] = p;
    }
  }
}

// Leaves the entries in sm.g.node / sm.g.elem at the given positions (a block barrier
// behind the stores).
template <typename C>
__device__ __forceinline__ void nearly_sorted_store(const uint32_t *key, int shift,
                                                    const int *pos, typename C::Smem &sm) {
  constexpr int kItems = C::kItems;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    sm.g.node[pos[j]] = key[j] >> shift;
    sm.g.elem[pos[j]] = (uint32_t)(threadIdx.x * kItems + j);
  }
  __syncthreads();
}

template <typename C>
__device__ __forceinline__ bool group_nearly_sorted(const uint32_t *key,
                                                    typename C::Smem &sm, uint32_t *scratch,
                                                    ScanSmem &ss) {
  NearlySorted<C> ns;
  if (!nearly_sorted_analyse<C>(key, scratch, ss, &ns)) return false;
  int pos[C::kItems];
  nearly_sorted_insertions<C>(key, 0, 0, ns, scratch);
  nearly_sorted_positions<C>(key, 0, 0, ns, scratch, pos);
  nearly_sorted_store<C>(key, 0, pos, sm);
  return true;
}

// The leaf CTA ahead of the values (first half of leaf_deltas_hashed): needs a.indices
// and the tree only.  Entries whose index is out of range lower *s_stop (initialised by
// the caller) and stay out of the set.  Leaves dup.ds_idx / ds_k / ndup in shared memory
// and the same, plus every entry's place in the list, in `info`.  False: more duplicates
// than the list holds (info says so too).
template <typename C, typename I, typename V>
__device__ __forceinline__ bool leaf_hashed_prepare(const UpdateArgs<I, V> &a, int n,
                                                    typename C::HashSmem &h,
                                                    LeafDupSmem<C> &dup, LeafPrep<C> *r,
                                                    int *s_stop, uint32_t *info) {
  constexpr int kItems = C::kItems, T = C::kThreads;
  constexpr int kHashSlots = C::kHashSlots, kHashBits = C::kHashBits;
  constexpr int kMaxDup = C::kMaxDup;
  constexpr uint32_t kEmpty = 0xffffffffu;
  using Info = DupInfo<C>;
  uint32_t slot_of[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x + j * T;
    r->idx[j] = kEmpty;
    r->k[j] = (uint32_t)k;
    if (k < n) {
      const int64_t ix = (int64_t)a.indices[k];
      if (ix >= 0 && ix < a.leaves) r->idx[j] = (uint32_t)ix;
      else atomicMin(s_stop, k);
    }
  }
#pragma unroll
  for (int j = 0; j < kItems; ++j) {  // (first used behind the values)
    r->leaf[j] = 0.0;
    slot_of[j] = 0;
    if (r->idx[j] != kEmpty) r->leaf[j] = a.heap[a.leaves + r->idx[j]];
  }
  for (int i = threadIdx.x; i < kHashSlots; i += blockDim.x) {
    h.key[i] = kEmpty;
    h.count[i] = 0;
  }
  if (threadIdx.x == 0) dup.ndup = 0;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    if (r->idx[j] != kEmpty) {
      const uint32_t idx = r->idx[j];
      uint32_t slot = (idx * 2654435761u) >> (32 - kHashBits);
      while (true) {
        const uint32_t old = atomicCAS(&h.key[slot], kEmpty, idx);
        if (old == kEmpty || old == idx) break;
        slot = (slot + 1) & (kHashSlots - 1);
      }
      atomicAdd(&h.count[slot], 1u);
      slot_of[j] = slot;
    }
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x + j * T;
    r->single[j] = r->idx[j] != kEmpty && h.count[slot_of[j]] == 1;
    if (r->idx[j] != kEmpty && h.count[slot_of[j]] > 1) {
      const int pos = atomicAdd(&dup.ndup, 1);
      if (pos < kMaxDup) {
        dup.d_idx[pos] = r->idx[j];
        dup.d_k[pos] = (uint32_t)k;
      }
    } else if (k < n) {
      info[Info::kOf + k] = 0xffffffffu;  // its leaf is its alone
    }
    // (the level CTAs take the leaves from here, not from the tree: this CTA may be
    // writing the new ones while a level CTA that got an SM late is still fetching)
    if (k < n) reinterpret_cast<double *>(info + Info::kLeaf)[k] = r->leaf[j];
  }
  __syncthreads();
  const int ndup = dup.ndup;
  if (ndup > kMaxDup) {
    if (threadIdx.x == 0) info[Info::kCount] = Info::kOverflow;
    return false;
  }
  // duplicates: order by (leaf, batch position), one chain per leaf
  if ((int)threadIdx.x < ndup) {
    const uint64_t me = ((uint64_t)dup.d_idx[threadIdx.x] << 32) | dup.d_k[threadIdx.x];
    int rank = 0;
    for (int j = 0; j < ndup; ++j)
      rank += ((((uint64_t)dup.d_idx[j] << 32) | dup.d_k[j]) < me) ? 1 : 0;
    dup.ds_idx[rank] = dup.d_idx[threadIdx.x];
    dup.ds_k[rank] = dup.d_k[threadIdx.x];
    info[Info::kIdx + rank] = dup.d_idx[threadIdx.x];
    info[Info::kK + rank] = dup.d_k[threadIdx.x];
    info[Info::kOf + dup.d_k[threadIdx.x]] = (uint32_t)rank;
  }
  if (threadIdx.x == 0) info[Info::kCount] = (uint32_t)ndup;
  __syncthreads();
  return true;
}

// What a level CTA holds for the grouped positions kItems * t .. kItems * t + kItems - 1
// of thread t (sm.g.node / sm.g.elem hold the grouping itself).
template <typename C>
struct LevelPrep {
  double node_val[C::kItems];  // group starts here: the node's stored value
  double leaf[C::kItems];      // the leaf the entry points at (from the leaf CTA's list)
  uint32_t k[C::kItems];       // the entry's batch position
  uint32_t dup_of[C::kItems];  // its place in the leaf CTA's list / 0xffffffff
};

// What LevelPrep holds, but for leaf and dup_of, from the grouping in sm.g (behind a block
// barrier).
template <typename C, typename I, typename V>
__device__ __forceinline__ void level_prefetch(const UpdateArgs<I, V> &a, int level,
                                               int count, typename C::EarlySmem &sm,
                                               LevelPrep<C> *r, bool staged = false) {
  constexpr int kItems = C::kItems;
  const int64_t base = ((int64_t)1) << level;
  uint32_t key[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    key[j] = sm.g.node[threadIdx.x * kItems + j];
    r->k[j] = sm.g.elem[threadIdx.x * kItems + j];
  }
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int p = threadIdx.x * kItems + j;
    r->node_val[j] = 0.0;
    r->leaf[j] = 0.0;
    r->dup_of[j] = 0xffffffffu;
    if (p >= count || (int64_t)key[j] >= base) continue;
    // (staged: every entry fetched its node's value when its index arrived, sm.nodev)
    if (p == 0 || sm.g.node[p - 1] != key[j])
      r->node_val[j] = staged ? sm.nodev[r->k[j]] : a.heap[base + key[j]];
  }
}

// Groups the first `count` entries by their node on `level` into sm.g (as a batch that is
// grouped already but for a few entries, else by a stable radix sort on the level's bits;
// entries that are pads or out of range sort as all-ones keys and lower *s_stop) and
// fetches what LevelPrep holds, but for leaf and dup_of.  sm.vals is scratch here.
template <typename C, typename I, typename V>
__device__ __forceinline__ void group_level(const UpdateArgs<I, V> &a, int level, int count,
                                            typename C::EarlySmem &sm, LevelPrep<C> *r,
                                            int *s_stop, ScanSmem &ss) {
  constexpr int kItems = C::kItems;
  using Sort = typename C::Sort;
  const int shift = a.depth - level;
  uint32_t key[kItems], val[kItems];
  int64_t ix[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x * kItems + j;
    ix[j] = k < count ? (int64_t)a.indices[k] : 0;
  }
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x * kItems + j;
    key[j] = 0xffffffffu;
    if (k < count) {
      if (ix[j] >= 0 && ix[j] < a.leaves) key[j] = (uint32_t)(ix[j] >> shift);
      else atomicMin(s_stop, k);
    }
    val[j] = (uint32_t)k;
  }
  if (level != 0 &&
      !group_nearly_sorted<C>(key, sm, reinterpret_cast<uint32_t *>(sm.vals), ss)) {
    Sort(sm.g.sort).Sort(key, val, 0, level);
    __syncthreads();  // (the sort's storage overlaps nothing below, but keep the order)
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      sm.g.node[threadIdx.x * kItems + j] = key[j];
      sm.g.elem[threadIdx.x * kItems + j] = val[j];
    }
  } else if (level == 0) {
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      sm.g.node[threadIdx.x * kItems + j] = key[j];
      sm.g.elem[threadIdx.x * kItems + j] = val[j];
    }
  }
  __syncthreads();
  level_prefetch<C>(a, level, count, sm, r);
}

// EVERY CTA ahead of the values when the batch is grouped by leaf already, but for a few
// entries (nearly_sorted_analyse): entries that share a leaf are neighbours then, and the
// list of them is what is left of the grouped batch without the leaves that occur once —
// no hash set, and nothing to hand from the leaf CTA to the others: each CTA makes the
// list for itself.  idx[j]: leaf of entry kItems * t + j / all ones (pads, out of range).
// 1: dup.ds_idx / ds_k / ndup and sm.place hold the list, own_pos the entries' places in
// the order of the CTA's own level (keys >> own_shift; for nearly_sorted_store); 0: the
// batch is not of that kind; -1: more duplicates than the list holds.  (sm.g is
// overwritten.)
template <typename C, typename I, typename V>
__device__ __forceinline__ int leaf_list_from_sorted(const UpdateArgs<I, V> &a, int n,
                                                     typename C::EarlySmem &sm,
                                                     LeafDupSmem<C> &dup,
                                                     const uint32_t *idx,
                                                     NearlySorted<C> *ns, uint32_t *scratch,
                                                     ScanSmem &ss, int own_shift,
                                                     int *own_pos, int who = -1) {
  constexpr int kItems = C::kItems, T = C::kThreads;
  constexpr int kMaxDup = C::kMaxDup;
  constexpr uint32_t kEmpty = 0xffffffffu;
  (void)who;
  B2R_PHASE(who, 1);
  if (!nearly_sorted_analyse<C>(idx, scratch, ss, ns)) return 0;
  B2R_PHASE(who, 2);
  // (own_pos: the entries' places on the CTA's own level, for nearly_sorted_store later)
  int pos[kItems];
  nearly_sorted_insertions<C>(idx, 0, own_shift, *ns, scratch);
  nearly_sorted_positions<C>(idx, 0, 0, *ns, scratch, pos);
  nearly_sorted_positions<C>(idx, own_shift, 1, *ns, scratch, own_pos);
  nearly_sorted_store<C>(idx, 0, pos, sm);
  B2R_PHASE(who, 3);
  // entries that share their leaf with a neighbour, compacted in (leaf, k) order
  bool shares[kItems];
  int mine = 0;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int p = threadIdx.x * kItems + j;
    const uint32_t node = sm.g.node[p];
    shares[j] = p < n && node != kEmpty &&
                ((p > 0 && sm.g.node[p - 1] == node) || (p + 1 < n && sm.g.node[p + 1] == node));
    mine += shares[j] ? 1 : 0;
  }
  uint32_t unused;
  int at, ndup;
  block_scan_max_sum<T>(0u, mine, ss, 1, &unused, &at, &ndup);
  B2R_PHASE(who, 4);
  if (ndup > kMaxDup) return -1;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int p = threadIdx.x * kItems + j;
    if (p >= n) continue;
    const uint32_t k = sm.g.elem[p];
    if (shares[j]) {
      dup.ds_idx[at] = sm.g.node[p];
      dup.ds_k[at] = k;
      sm.place[k] = (uint32_t)at;
      ++at;
    } else {
      sm.place[k] = kEmpty;
    }
  }
  if (threadIdx.x == 0) dup.ndup = ndup;
  __syncthreads();
  return 1;
}

// The ordered chains of one level over deltas that are in shared memory already
// (sm.vals, in group order, behind a block barrier).
template <typename C, typename I, typename V>
__device__ __forceinline__ void level_chains_grouped(const UpdateArgs<I, V> &a, int level,
                                                     int n, typename C::Smem &sm,
                                                     const LevelPrep<C> &r) {
  constexpr int kItems = C::kItems;
  const int64_t base = ((int64_t)1) << level;
  const double *sorted_delta = sm.vals;
  // long chains (the upper levels): verified scan; it declines when adds round
  if (a.scan_min_chain > 0 && (n >> level) >= a.scan_min_chain &&
      chains_by_verified_scan<C>(a.heap + base, r.node_val, sm.g.node, sorted_delta, n))
    return;
  // serial chains: the thread that owns a group's first position walks the group
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int p = threadIdx.x * kItems + j;
    if (p >= n) continue;
    const uint32_t node = sm.g.node[p];
    if ((int64_t)node >= base || (p > 0 && sm.g.node[p - 1] == node)) continue;
    double acc = r.node_val[j];
    for (int q = p; q < n && sm.g.node[q] == node; ++q) acc = __dadd_rn(acc, sorted_delta[q]);
    a.heap[base + node] = acc;
  }
}

template <typename I, typename V, typename C>
__global__ void __launch_bounds__(C::kThreads) tree_update_early_kernel(UpdateArgs<I, V> a) {
  constexpr int kItems = C::kItems, T = C::kThreads;
  constexpr uint32_t kEmpty = 0xffffffffu;
  using Sort = typename C::Sort;
  using Info = DupInfo<C>;
  static_assert(Info::kWords <= DupInfo<BigCfgWide>::kWords, "scratch (ensure_sorted)");
  extern __shared__ __align__(16) uint8_t smem_raw[];
  typename C::EarlySmem &sm = *reinterpret_cast<typename C::EarlySmem *>(smem_raw);
  double *vals = sm.vals;
  __shared__ LeafDupSmem<C> s_dup;
  __shared__ double s_dupd[C::kMaxDup];  // deltas of the entries that share leaves
  __shared__ int s_stop;                 // first position that must not be applied
  __shared__ int s_stop_code;
  __shared__ double s_max[32];
  __shared__ int s_role;
  __shared__ uint32_t s_listed;
  __shared__ ScanSmem s_scan;
  uint32_t *info = a.sorted;
  TreeSync &sync = *a.sync;
  B2R_MARK(13);
  // The last CTA to leave re-arms the list's flag and the count of level CTAs that have
  // their leaves (everybody is past both then), and counts the launch (TreeGo).
  auto leave = [&]() {
    if (threadIdx.x == 0 && atomicInc(&sync.ended, (unsigned)a.depth) == (unsigned)a.depth) {
      sync.list_flag = 0u;
      sync.fetched = 0u;
      atomicAdd(&sync.completed, 1u);
    }
  };
  // A ticket first, dependents second: the next early write-back can only start once
  // every CTA of this one has its ticket, so ticket / CTAs is the launch's number and
  // ticket % CTAs the order of arrival within it.  Dependents only when the indices are
  // final, too: released at once, the kernels of the NEXT steps would all become resident
  // behind each other (each lets the next start from its first instruction) and sit on
  // the SMs waiting — bounded to one step ahead this way.
  if (threadIdx.x == 0) {
    const LaunchTicket t = launch_ticket(a.tickets, (unsigned)a.depth + 1u);
    s_role = (int)t.arrival;
    s_listed = 1u;
    // resident ahead of the indices: wait to hear that they are final (TreeGo)
    if (a.go != nullptr)
      s_listed = poll_acquire(a.go, [&](unsigned v) { return v == t.launch; }) ? 1u : 0u;
  }
  __syncthreads();
  pdl_release();
  if (s_listed == 0u) {  // (nobody said go: touch nothing, say so)
    pdl_acquire();
    if (threadIdx.x == 0 && a.status[0] == 0) a.status[0] = B2R_ERR_CUDA;
    leave();
    return;
  }
  int n = a.n;
  if (a.n_dev) {
    const int64_t left = (int64_t)*a.n_dev - a.k_base;
    n = left < n ? (left > 0 ? (int)left : 0) : n;
  }
  if (threadIdx.x == 0) {
    s_stop = n;
    s_stop_code = 0;
  }
  __syncthreads();
  // Levels are handed out in order of arrival, the leaf level first: the CTA the others
  // wait for (its list ahead of the values; its deltas when the list does not serve) is
  // always one that is already running.
  const int level = s_role == 0 ? a.depth : s_role - 1;
  const bool is_leaf = level == a.depth;
  B2R_MARK_LVL(0, 0);
  B2R_MARK_LVL(16, a.depth);
  B2R_MARK_LVL(22, a.depth - 1);
  if (n <= 0) {  // (every CTA sees the same n)
    pdl_acquire();
    leave();
    return;
  }

  // ---- ahead of the values
  LeafPrep<C> leaf_prep;
  LevelPrep<C> prep;
  bool listed = false;  // a list of the duplicate leaves serves
  int ndup = 0;
  double chain_leaf = 0.0;
  uint32_t *scratch = reinterpret_cast<uint32_t *>(sm.vals);
  uint32_t lidx[kItems];
  NearlySorted<C> ns;
  // own_list: the batch is grouped by leaf already but for a few entries — every CTA makes
  // the list for itself and takes its leaves from the tree; else the leaf CTA makes it
  // with a hash set and hands it (and the leaves) to the others.
  const int who = is_leaf ? 0 : (level == 10 ? 1 : -1);
  (void)who;
  B2R_PHASE(who, 0);
  // The indices; then, at once and for every entry, the loads that need nothing else: its
  // leaf and (level CTAs) its node on this level — they fly while the batch is analysed.
  int first_bad = n;
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x * kItems + j;
    lidx[j] = kEmpty;
    if (k < n) {
      const int64_t ix = (int64_t)a.indices[k];
      if (ix >= 0 && ix < a.leaves) lidx[j] = (uint32_t)ix;
      else first_bad = min(first_bad, k);
    }
  }
  double leaf_k[kItems], node_k[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    leaf_k[j] = node_k[j] = 0.0;
    if (lidx[j] == kEmpty) continue;
    leaf_k[j] = a.heap[a.leaves + lidx[j]];
    if (!is_leaf)
      node_k[j] = a.heap[(((int64_t)1) << level) + (lidx[j] >> (a.depth - level))];
  }
  if (first_bad < n) atomicMin(&s_stop, first_bad);
  int own_pos[kItems];
  const bool own_list = leaf_list_from_sorted<C>(a, n, sm, s_dup, lidx, &ns, scratch, s_scan,
                                                 a.depth - level, own_pos, who) == 1;
  B2R_PHASE(who, 5);
  B2R_TRACE_COUNT(0, is_leaf);
  B2R_TRACE_COUNT(1, is_leaf && own_list);
  if (own_list) {
    listed = true;
    ndup = s_dup.ndup;
    // (the grouping by leaf has been read by everybody: leaf_list_from_sorted ends on a
    // barrier; the one behind these stores is the one below)
    if (!is_leaf) {
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        sm.g.node[own_pos[j]] = lidx[j] >> (a.depth - level);
        sm.g.elem[own_pos[j]] = (uint32_t)(threadIdx.x * kItems + j);
      }
    }
    B2R_PHASE(who, 6);
    // The leaf CTA writes the new leaves only once every level CTA HAS the old ones: a
    // value that is in shared memory has landed.
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      sm.leafv[threadIdx.x * kItems + j] = leaf_k[j];
      if (!is_leaf) sm.nodev[threadIdx.x * kItems + j] = node_k[j];
    }
    B2R_PHASE(who, 8);
    __syncthreads();
    if (!is_leaf && threadIdx.x == 0) atomicAdd(&sync.fetched, 1u);
    B2R_PHASE(who, 9);
    const bool head = (int)threadIdx.x < ndup &&
                      (threadIdx.x == 0 ||
                       s_dup.ds_idx[threadIdx.x - 1] != s_dup.ds_idx[threadIdx.x]);
    if (head) chain_leaf = sm.leafv[s_dup.ds_k[threadIdx.x]];
    if (is_leaf) {
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        const int k = threadIdx.x * kItems + j;
        leaf_prep.idx[j] = lidx[j];
        leaf_prep.k[j] = (uint32_t)k;
        leaf_prep.single[j] = k < n && lidx[j] != kEmpty && sm.place[k] == kEmpty;
        leaf_prep.leaf[j] = leaf_k[j];
      }
    } else {
      level_prefetch<C>(a, level, n, sm, &prep, true);
#pragma unroll
      for (int j = 0; j < kItems; ++j)
        if (threadIdx.x * kItems + j < n) prep.dup_of[j] = sm.place[prep.k[j]];
      B2R_PHASE(who, 7);
    }
  } else if (is_leaf) {
    listed = leaf_hashed_prepare<C>(a, n, sm.h, s_dup, &leaf_prep, &s_stop, info);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) st_release_u32(&sync.list_flag, 1u);
    ndup = listed ? s_dup.ndup : 0;
  } else {
    group_level<C>(a, level, n, sm, &prep, &s_stop, s_scan);
    B2R_LEVEL_TIME(0, level);
    if (threadIdx.x == 0) {
      const bool seen = poll_acquire(&sync.list_flag, [](unsigned v) { return v != 0u; });
      s_listed = seen ? __ldcg(info + Info::kCount) : Info::kOverflow;
    }
    __syncthreads();
    listed = s_listed != Info::kOverflow;
    ndup = listed ? (int)s_listed : 0;
    if (listed) {
      for (int q = threadIdx.x; q < ndup; q += T) {
        s_dup.ds_idx[q] = __ldcg(info + Info::kIdx + q);
        s_dup.ds_k[q] = __ldcg(info + Info::kK + q);
      }
      const double *leaves_then = reinterpret_cast<const double *>(info + Info::kLeaf);
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        if (threadIdx.x * kItems + j < n) {
          prep.dup_of[j] = __ldcg(info + Info::kOf + prep.k[j]);
          prep.leaf[j] = __ldcg(leaves_then + prep.k[j]);
        }
      }
      __syncthreads();
    }
  }
  // heads of the duplicates' chains (every CTA walks them all): the leaf they start from
  const bool chain_head = (int)threadIdx.x < ndup &&
                          (threadIdx.x == 0 ||
                           s_dup.ds_idx[threadIdx.x - 1] != s_dup.ds_idx[threadIdx.x]);
  if (chain_head && !own_list)
    chain_leaf = __ldcg(reinterpret_cast<const double *>(info + Info::kLeaf) +
                        s_dup.ds_k[threadIdx.x]);
  B2R_MARK_LVL(17, a.depth);
  B2R_MARK_LVL(23, a.depth - 1);
  B2R_MARK_LVL(29, 0);
  B2R_LEVEL_TIME(1, level);
  B2R_PHASE(who, 10);
  pdl_acquire();
  B2R_PHASE(who, 11);
  B2R_LEVEL_TIME(2, level);
  B2R_MARK_LVL(18, a.depth);
  B2R_MARK_LVL(1, 0);
  B2R_MARK_LVL(24, a.depth - 1);
  // An earlier chunk (or the kernel that produced the values) failed: the reference's
  // loop stopped there.  This kernel's own latch is only written once every level has
  // passed the plain kernel's flag, so every CTA takes the same branch.
  if (a.status[0] != 0) {
    leave();
    return;
  }

  // ---- the values: every CTA reads all of them, and finds the first entry the reference
  // would have raised on for itself
  double v[kItems];
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x + j * T;
    v[j] = k < n ? (double)a.values[k] : 0.0;
  }
#pragma unroll
  for (int j = 0; j < kItems; ++j) {
    const int k = threadIdx.x + j * T;
    if (k < n) {
      vals[k] = v[j];
      if (v[j] < 0.0) atomicMin(&s_stop, k);
    }
  }
  __syncthreads();
  const int n_eff = s_stop;

  // (own lists: the level CTAs take the old leaves from the tree, so the new ones wait
  // until all of them have theirs — which they have had since before the values came)
  if (own_list && is_leaf) {
    if (threadIdx.x == 0 &&
        !poll_acquire(&sync.fetched, [&](unsigned v) { return v >= (unsigned)a.depth; }) &&
        a.status[0] == 0)
      a.status[0] = B2R_ERR_CUDA;
    __syncthreads();
  }
  B2R_TRACE_COUNT(2, is_leaf && listed && n_eff == n);
  if (listed && n_eff == n) {
    // ---- nothing to wait for.  Chains of the entries that share leaves:
    //   delta = value - leaf; leaf += delta   (sum_tree.py:196-202, last level)
    if (chain_head) {
      const uint32_t idx = s_dup.ds_idx[threadIdx.x];
      double leaf = chain_leaf;
      for (int q = threadIdx.x; q < ndup && s_dup.ds_idx[q] == idx; ++q) {
        const double d = __dsub_rn(vals[s_dup.ds_k[q]], leaf);
        leaf = __dadd_rn(leaf, d);
        s_dupd[q] = d;
      }
      if (is_leaf) a.heap[a.leaves + idx] = leaf;
    }
    if (is_leaf) {
#pragma unroll
      for (int j = 0; j < kItems; ++j) {
        if (leaf_prep.single[j]) {
          const double d = __dsub_rn(vals[leaf_prep.k[j]], leaf_prep.leaf[j]);
          a.heap[a.leaves + leaf_prep.idx[j]] = __dadd_rn(leaf_prep.leaf[j], d);
        }
      }
      // max_recorded_priority = max(value, current)
      double local_max = 0.0;
#pragma unroll
      for (int j = 0; j < kItems; ++j) local_max = fmax(local_max, v[j]);
      for (int off = 16; off > 0; off >>= 1)
        local_max = fmax(local_max, __shfl_xor_sync(0xffffffffu, local_max, off));
      if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = local_max;
      __syncthreads();
      if (threadIdx.x == 0) {
        double m = *a.max_rec;
        for (int w = 0; w < T / 32; ++w)
          if (s_max[w] > m) m = s_max[w];
        *a.max_rec = m;
      }
      B2R_LEVEL_TIME(3, level);
      B2R_MARK_END(15);
      leave();
      return;
    }
    double vp[kItems];
#pragma unroll
    for (int j = 0; j < kItems; ++j)
      vp[j] = threadIdx.x * kItems + j < n ? vals[prep.k[j]] : 0.0;
    __syncthreads();  // (vals turns into the deltas in group order)
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int p = threadIdx.x * kItems + j;
      if (p < n)
        vals[p] = prep.dup_of[j] != kEmpty
                      ? s_dupd[prep.dup_of[j]]
                      : __dsub_rn(vp[j], own_list ? sm.leafv[prep.k[j]] : prep.leaf[j]);
    }
    __syncthreads();
    B2R_MARK_LVL(3, 0);
    B2R_MARK_LVL(20, 1);
    B2R_MARK_LVL(26, a.depth - 1);
    level_chains_grouped<C>(a, level, n, sm, prep);
    B2R_MARK_LVL(4, 0);
    B2R_MARK_LVL(21, 1);
    B2R_MARK_LVL(27, a.depth - 1);
    B2R_LEVEL_TIME(3, level);
    B2R_MARK_END(15);
    leave();
    return;
  }

  // ---- the list does not serve: on as the plain kernel
  if (!is_leaf) {
    const int applied = levels_wait_for_leaf(a);
    B2R_MARK_END(11);
    if (applied != n) group_level<C>(a, level, applied, sm, &prep, &s_stop, s_scan);
    if (applied > 0) internal_level_chains<C>(a, level, applied, sm, prep.node_val);
    leave();
    return;
  }
  if (n_eff < n && threadIdx.x == 0)
    s_stop_code = (vals[n_eff] < 0.0) ? B2R_ERR_NEGATIVE_PRIORITY : B2R_ERR_INDEX_RANGE;
  {
    double local_max = 0.0;
#pragma unroll
    for (int j = 0; j < kItems; ++j)
      if (threadIdx.x + j * T < n_eff) local_max = fmax(local_max, v[j]);
    for (int off = 16; off > 0; off >>= 1)
      local_max = fmax(local_max, __shfl_xor_sync(0xffffffffu, local_max, off));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = local_max;
  }
  __syncthreads();
  if (!leaf_deltas_hashed<C>(a, n_eff, sm.h, vals)) {
    __syncthreads();
    uint32_t key[kItems], val[kItems];
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      const int k = threadIdx.x * kItems + j;
      key[j] = k < n_eff ? (uint32_t)a.indices[k] : 0xffffffffu;
      val[j] = (uint32_t)k;
    }
    if (a.depth != 0) Sort(sm.g.sort).Sort(key, val, 0, a.depth);
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
      sm.g.node[threadIdx.x * kItems + j] = key[j];
      sm.g.elem[threadIdx.x * kItems + j] = val[j];
    }
    __syncthreads();
    // one thread per distinct leaf walks its chain in batch order
    for (int p = threadIdx.x; p < n_eff; p += T) {
      if (p != 0 && sm.g.node[p - 1] == sm.g.node[p]) continue;
      const uint32_t node = sm.g.node[p];
      double leaf = a.heap[a.leaves + node];
      for (int q = p; q < n_eff && sm.g.node[q] == node; ++q) {
        const uint32_t k = sm.g.elem[q];
        const double d = __dsub_rn(vals[k], leaf);
        leaf = __dadd_rn(leaf, d);
        vals[k] = d;
      }
      a.heap[a.leaves + node] = leaf;
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < n_eff; k += T) a.delta[k] = vals[k];
  B2R_MARK_LVL(19, a.depth);
  leaf_publishes(a, n, n_eff, s_stop_code);
  B2R_MARK_LVL(28, a.depth);
  if (threadIdx.x == 0) {
    double m = *a.max_rec;
    for (int w = 0; w < T / 32; ++w)
      if (s_max[w] > m) m = s_max[w];
    if (n_eff > 0) *a.max_rec = m;
    if (n_eff < n && a.depth == 0) {  // (a one-node tree has no other level to latch)
      a.status[0] = s_stop_code;
      a.status[1] = a.k_base + n_eff;
    }
  }
  B2R_MARK_END(15);
  leave();
}

constexpr int kSmallBatch = 256;  // largest batch the single-CTA kernel takes

// Warp-level bitonic sort of `padded` (<= 256) keys in shared memory.
__device__ __forceinline__ void warp_bitonic_sort(uint64_t *keys, int padded, int lane) {
#pragma unroll 1
  for (int k = 2; k <= padded; k <<= 1) {
#pragma unroll 1
    for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll 1
      for (int t = lane; t < padded; t += 32) {
        const int partner = t ^ j;
        if (partner > t) {
          const uint64_t a = keys[t], b = keys[partner];
          const bool ascending = (t & k) == 0;
          if ((a > b) == ascending) {
            keys[t] = b;
            keys[partner] = a;
          }
        }
      }
      __syncwarp();
    }
  }
}

// Latency path for small batches (<= 256 sets: the agent's batch 32): ONE CTA,
// one WARP per tree level, so the only synchronisation between the leaf pass and
// the internal levels is a __syncthreads.  Each warp sorts its own (node, k) keys
// with shuffled-free warp-synchronous bitonic steps while the leaf warp resolves
// the leaf chains; internal warps prefetch their node values before the barrier.
template <bool PDL = true, typename I, typename V>
__device__ __forceinline__ void tree_update_small_body(const UpdateArgs<I, V> &a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int levels = a.depth + 1;
  double *vals = reinterpret_cast<double *>(smem_raw);            // [padded] value -> delta
  uint64_t *all_keys = reinterpret_cast<uint64_t *>(smem_raw) + a.padded;
  uint64_t *keys = all_keys + (size_t)warp * a.padded;            // this level's keys
  double *all_sorted = reinterpret_cast<double *>(all_keys + (size_t)levels * a.padded);
  double *sorted_delta = all_sorted + (size_t)warp * a.padded;
  __shared__ int s_stop, s_stop_code;

  if (PDL) {
    B2R_MARK(0);
    pdl_release();
    pdl_acquire();
    B2R_MARK(1);
  }
  int n = a.n;
  if (a.n_dev) n = min(n, max(*a.n_dev, 0));
  const int64_t latched = a.status[0];
  if (threadIdx.x == 0) {
    s_stop = n;
    s_stop_code = 0;
  }
  __syncthreads();
  if (latched != 0) return;  // an earlier chunk failed: the sequence stopped there

  if (a.mode != nullptr) {
    stage_mode_values(a, n, vals, &s_stop, &s_stop_code);
  } else {
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
      const double v = (double)a.values[k];
      const int64_t idx = (int64_t)a.indices[k];
      vals[k] = v;
      if (v < 0.0 || idx < 0 || idx >= a.leaves) atomicMin(&s_stop, k);
    }
  }
  __syncthreads();
  const int n_eff = s_stop;
  if (a.mode == nullptr && n_eff < n && threadIdx.x == 0)
    s_stop_code = (vals[n_eff] < 0.0) ? B2R_ERR_NEGATIVE_PRIORITY
                                      : B2R_ERR_INDEX_RANGE;

  B2R_MARK(2);
  const int level = warp;
  const bool is_leaf = level == a.depth;
  const int shift = a.depth - level;
  // The leaf warp gates every other level (they wait for its deltas at the barrier
  // below).  With at most one entry per lane it needs no sort: __match_any_sync finds
  // the lanes that share a leaf, the lowest of them walks its group in lane (= batch)
  // order; the leaf values are already in flight when the groups are formed.
  const bool leaf_by_match = is_leaf && n_eff <= 32;
  const int64_t base = ((int64_t)1) << level;
  int p2 = 32;
  while (p2 < n_eff) p2 <<= 1;
  if (!leaf_by_match) {
    for (int k = lane; k < p2; k += 32)
      keys[k] = k < n_eff
                    ? (((uint64_t)((int64_t)a.indices[k] >> shift)) << 32) | (uint32_t)k
                    : kPadKey;
    __syncwarp();
  }
  B2R_MARK(3);
  if (level != 0 && !leaf_by_match) warp_bitonic_sort(keys, p2, lane);
  B2R_MARK(4);

  // (Loops below stay rolled: compact code beats unrolling in these one-shot phases.)
  if (is_leaf) {
    // (loaded here, not where it is compared: one memory round trip less at the end)
    const double recorded_max = lane == 0 ? *a.max_rec : 0.0;
    double local_max = 0.0;
#pragma unroll 1
    for (int k = lane; k < n_eff; k += 32) local_max = fmax(local_max, vals[k]);
#pragma unroll 1
    for (int off = 16; off > 0; off >>= 1)
      local_max = fmax(local_max, __shfl_xor_sync(0xffffffffu, local_max, off));
    if (leaf_by_match) {
      const bool in = lane < n_eff;
      // lanes without an entry get distinct keys that no leaf index can take
      const long long idx = in ? (long long)a.indices[lane] : -1ll - lane;
      double leaf = in ? a.heap[base + idx] : 0.0;
      const unsigned same = __match_any_sync(0xffffffffu, idx);
      if (in && lane == __ffs(same) - 1) {
        unsigned rest = same;
#pragma unroll 1
        while (rest) {
          const int k = __ffs(rest) - 1;
          rest &= rest - 1;
          const double d = __dsub_rn(vals[k], leaf);
          leaf = __dadd_rn(leaf, d);
          vals[k] = d;
        }
        a.heap[base + idx] = leaf;
      }
    } else {
#pragma unroll 1
      for (int p = lane; p < n_eff; p += 32) {
        const uint32_t node = (uint32_t)(keys[p] >> 32);
        if (p > 0 && (uint32_t)(keys[p - 1] >> 32) == node) continue;
        double leaf = a.heap[base + node];
#pragma unroll 1
        for (int q = p; q < n_eff && (uint32_t)(keys[q] >> 32) == node; ++q) {
          const uint32_t k = (uint32_t)keys[q];
          const double d = __dsub_rn(vals[k], leaf);
          leaf = __dadd_rn(leaf, d);
          vals[k] = d;
        }
        a.heap[base + node] = leaf;
      }
    }
    if (lane == 0) {
      if (n_eff > 0 && local_max > recorded_max) *a.max_rec = local_max;
      if (n_eff < n) {
        a.status[0] = s_stop_code;
        a.status[1] = a.k_base + n_eff;
      }
    }
  }
  B2R_MARK(5);
  __syncthreads();  // deltas are in vals[]
  B2R_MARK(6);
  if (is_leaf || warp >= levels) return;

#pragma unroll 1
  for (int p = lane; p < n_eff; p += 32) sorted_delta[p] = vals[(uint32_t)keys[p]];
  __syncwarp();
  B2R_MARK(8);
#pragma unroll 1
  for (int p = lane; p < n_eff; p += 32) {
    const uint32_t node = (uint32_t)(keys[p] >> 32);
    if (p > 0 && (uint32_t)(keys[p - 1] >> 32) == node) continue;
    double acc = a.heap[base + node];  // issued before the search below
    int lo = p + 1, hi = n_eff;
#pragma unroll 1
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((uint32_t)(keys[mid] >> 32) > node) hi = mid; else lo = mid + 1;
    }
    B2R_MARK(9);
#pragma unroll 4
    for (int q = p; q < lo; ++q) acc = __dadd_rn(acc, sorted_delta[q]);
    B2R_MARK(10);
    a.heap[base + node] = acc;
  }
  if (level == 0) publish_root(a);
  B2R_MARK(7);
}

// tiny_ok: when the device-side count (a sharded step's rows: the launch is sized for the
// bound on the share, the rows are usually far fewer) turns out to be at most 32, the
// match-based body runs instead — the decision the host makes from n when it knows n.
template <typename I, typename V>
__global__ void __launch_bounds__(1024) tree_update_small_kernel(UpdateArgs<I, V> a,
                                                                 int tiny_ok) {
  B2R_MARK(0);
  pdl_release();
  pdl_acquire();
  B2R_MARK(1);
  if (a.skip_flag != nullptr) {
    const unsigned int done = *a.skip_flag;
    __syncthreads();  // (every thread has read the flag before it is re-armed)
    if (done != 0u) {
      if (threadIdx.x == 0) *a.skip_flag = 0u;
      return;
    }
  }
  if (tiny_ok) {
    int n = a.n;
    if (a.n_dev) n = min(n, max(*a.n_dev, 0));
    if (n <= kTinyBatch) {
      tree_update_tiny_body<false>(a);
      B2R_MARK_END(7);
      return;
    }
  }
  tree_update_small_body<false>(a);
}

template <typename I, typename V>
__global__ void __launch_bounds__(1024) tree_update_tiny_kernel(UpdateArgs<I, V> a) {
  B2R_MARK(30);
  tree_update_tiny_body<true>(a);
  B2R_MARK_END(7);
}

// The flush of staged adds as ONE launch: CTA 0 applies the priorities of the new
// rows to the tree (the body above), the other CTAs write the rows into the ring
// (replay.cuh: add_rows_body).  Both read the staging buffer straight from pinned
// host memory (zero-copy), so an add flush puts one kernel on the stream instead of
// a copy and two kernels.
__global__ void __launch_bounds__(1024)
flush_fused_kernel(UpdateArgs<int64_t, double> a, AddParams p, int row_blocks_per_entry,
                   int tiny) {
  if (blockIdx.x == 0) {
    if (tiny)
      tree_update_tiny_body<true>(a);
    else
      tree_update_small_body(a);
    return;
  }
  pdl_release();
  pdl_acquire();
  const int r = blockIdx.x - 1;
  add_rows_body(p, r / row_blocks_per_entry, r % row_blocks_per_entry,
                row_blocks_per_entry);
}

__global__ void tree_get_kernel(const double *__restrict__ heap, int64_t leaves,
                                int64_t n, const int64_t *__restrict__ indices,
                                double *__restrict__ out) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = indices[k];
  out[k] = (i >= 0 && i < leaves) ? heap[leaves + i] : 0.0;
}

__global__ void tree_query_kernel(const double *__restrict__ heap, int depth,
                                  int64_t n, const double *__restrict__ query01,
                                  int64_t *__restrict__ out,
                                  double *__restrict__ total_out, uint32_t zero) {
  extern __shared__ double top[];
  const int top_depth = stage_top_levels(heap, depth, top);
  const double total = top[1];
  if (blockIdx.x == 0 && threadIdx.x == 0) *total_out = total;
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k >= n) return;
  // sum_tree.py:123-124: query_value *= total
  out[k] = tree_descend_staged<3>(heap, top, top_depth, depth,
                               __dmul_rn(query01[k], total), zero);
}

__global__ void tree_set_scalar_kernel(double *dst, double v) { *dst = v; }

int padded_size(int n) {
  int p = 32;
  while (p < n) p <<= 1;
  return p;
}

// One chunk of the cooperative kernel with geometry C: tree_update_kernel, or (EARLY,
// kEarly) tree_update_early_kernel.
template <typename C, bool EARLY, typename I, typename V>
int launch_big_chunk(const UpdateArgs<I, V> &a, int depth, cudaStream_t stream) {
  constexpr auto kernel = [] {  // (only the kernel used is instantiated)
    if constexpr (EARLY)
      return tree_update_early_kernel<I, V, C>;
    else
      return tree_update_kernel<I, V, C>;
  }();
  constexpr int smem = EARLY ? sizeof(typename C::EarlySmem) : sizeof(typename C::Smem);
  B2R_TRY(allow_dynamic_smem_once<kernel>(smem));
  // Launched early (programmatic dependent launch) only in the 256 x 4 geometry: 21
  // early CTAs of 1024 threads would sit on 21 SMs for the whole loss kernel.
  // (kEarly: starting early is the point — its CTAs are sorting meanwhile.)
  constexpr unsigned flags =
      kLaunchTreeWindow | (C::kThreads <= 256 || EARLY ? 0u : kLaunchNoPdl);
  B2R_CUDA(launch_prio_cluster<flags>(kernel, dim3(depth + 1), dim3(C::kThreads), smem,
                                      stream, chain_priority(), 1, a));
  B2R_LAUNCHED();
  return B2R_OK;
}

// What every write-back of `t` takes; the launch adds its chunk of the batch and its own
// fields.  publish: see tree_apply.
template <typename I, typename V>
UpdateArgs<I, V> update_args(const b2r_tree *t, const b2r_exchange *publish) {
  UpdateArgs<I, V> a;
  a.heap = t->heap;
  a.depth = t->depth;
  a.leaves = t->leaves;
  a.delta = t->delta;
  a.max_rec = t->max_rec;
  a.status = t->status;
  a.sync = t->sync;
  if (publish != nullptr && publish->world > 1 && publish->connected) {
    a.publish = publish->args_dev;
    a.publish_world = publish->world;
    a.publish_rank = publish->rank;
  }
  return a;
}

}  // namespace

// The one-CTA kernel sorts per warp (cost ~ n log^2 n): it wins for the agent's batch
// of 32 (4.9 us) and already loses to the 256 x 4 cooperative kernel at 64 entries
// (10.5 vs 9.2 us; at 256: 43 vs 9.8 us — measured with 10 launches per graph,
// profiles/r1/README.md).  Largest batch it takes.
constexpr int kTreeSmallMax = 32;

// Shortest average chain (entries per touched node of a level) that is worth the
// verified scan: a round costs about as much as 60-80 dependent DADDs.
constexpr int kTreeScanMinChain = 32;

// The one-CTA kernels' dynamic shared memory for kSmallBatch entries at the deepest tree
// (32 levels).
static int allow_small_smem() {
  constexpr int bytes = kSmallBatch * 8 * (1 + 2 * 32);
  B2R_TRY((allow_dynamic_smem_once<tree_update_small_kernel<int64_t, double>>(bytes)));
  B2R_TRY((allow_dynamic_smem_once<tree_update_small_kernel<int32_t, float>>(bytes)));
  B2R_TRY((allow_dynamic_smem_once<tree_update_small_kernel<int32_t, double>>(bytes)));
  return allow_dynamic_smem_once<flush_fused_kernel>(bytes);
}

int flush_fused(b2r_tree *t, int n, const int64_t *slots, const double *prio,
                const uint8_t *mode, const AddParams &rows, int row_blocks_per_entry,
                cudaStream_t stream, const b2r_exchange *publish) {
  set_tree_window(t->heap, (size_t)t->leaves * 16);
  B2R_TRY(allow_small_smem());
  const int padded = padded_size(n);
  const size_t smem = (size_t)padded * 8 * (1 + 2 * (size_t)(t->depth + 1));
  UpdateArgs<int64_t, double> a = update_args<int64_t, double>(t, publish);
  a.n = n;
  a.padded = padded;
  a.indices = slots;
  a.values = prio;
  a.mode = mode;
  a.k_base = 0;
  a.n_dev = nullptr;
  B2R_CUDA(launch(flush_fused_kernel, dim3(1 + n * row_blocks_per_entry),
                  dim3(32 * (t->depth + 1)), smem, stream, a, rows,
                  row_blocks_per_entry, (int)(n <= kTinyBatch)));
  B2R_LAUNCHED();
  return B2R_OK;
}

// Can the early write-back (kEarly) take a batch of n sets (expected_n as in
// tree_apply)?  It is the cooperative kernel in ONE chunk of its geometry: batches above
// the one-CTA kernel's and up to 1024 sets.  Beyond that the frame copies bound the step
// and the write-back hides behind them anyway.
// (A launch sized for more entries than are expected — a sharded step's bound on its
// share — groups its first chunk early, where the expected entries are; chunks behind
// it, normally empty, run as kFull.)
bool tree_early_takes(int64_t n, int64_t expected_n) {
  const int64_t likely = expected_n >= 0 ? expected_n : n;
  if (n <= kSmallBatch && likely <= kTreeSmallMax) return false;
  return likely <= BigCfgWide::kChunk;
}

static int ensure_sorted(b2r_tree *t) {
  if (t->sorted) return B2R_OK;
  // (kEarly: the leaf CTA's list of duplicate leaves)
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->sorted),
                      (size_t)DupInfo<BigCfgWide>::kWords * sizeof(uint32_t)));
  return B2R_OK;
}

template <typename I, typename V>
int tree_apply(b2r_tree *t, int64_t n, const I *indices, const V *values,
               const uint8_t *mode, cudaStream_t stream, const int32_t *n_dev,
               int64_t expected_n, int phase, const b2r_exchange *publish,
               unsigned int *skip_flag, bool go_by_flag) {
  set_tree_window(t->heap, (size_t)t->leaves * 16);
  if (phase == kEarly) {
    if (!tree_early_takes(n, expected_n) || mode != nullptr)
      return fail(B2R_ERR_INVALID_ARGUMENT, "this batch cannot take the early write-back");
    B2R_TRY(ensure_sorted(t));
  }
  // A device-side count (sharded replay) is only bounded by n on the host: the
  // caller's expectation decides, the one-CTA kernel copes with up to kSmallBatch.
  const int64_t likely = expected_n >= 0 ? expected_n : n;
  if (n <= kSmallBatch && likely <= kTreeSmallMax) {
    // latency path: one CTA, one warp per level
    const int padded = padded_size((int)n);
    const size_t smem = (size_t)padded * 8 * (1 + 2 * (size_t)(t->depth + 1));
    B2R_TRY(allow_small_smem());
    UpdateArgs<I, V> a = update_args<I, V>(t, publish);
    a.n = (int)n;
    a.padded = padded;
    a.indices = indices;
    a.values = values;
    a.mode = mode;
    a.k_base = 0;
    a.n_dev = n_dev;
    a.skip_flag = skip_flag;
    if (n <= kTinyBatch && skip_flag == nullptr)
      B2R_CUDA(launch(tree_update_tiny_kernel<I, V>, dim3(1), dim3(32 * (t->depth + 1)),
                      0, stream, a));
    else
      B2R_CUDA(launch(tree_update_small_kernel<I, V>, dim3(1),
                      dim3(32 * (t->depth + 1)), smem, stream, a,
                      (int)(n_dev != nullptr && t->depth + 1 <= 32)));
    B2R_LAUNCHED();
    return B2R_OK;
  }
  // Up to 1024 entries (known on the host): the 256 x 4 geometry; above, chunks of
  // 4096 through the 1024 x 4 one.
  const bool compact = likely <= BigCfg1024::kChunk;
  const int64_t chunk = compact ? BigCfg1024::kChunk : BigCfg4096::kChunk;
  for (int64_t base = 0; base < n; base += chunk) {
    const int len = (int)((n - base) < chunk ? (n - base) : chunk);
    UpdateArgs<I, V> a = update_args<I, V>(t, publish);
    a.n = len;
    a.padded = (int)chunk;
    a.indices = indices + base;
    a.values = values + base;
    a.mode = mode ? mode + base : nullptr;
    a.k_base = base;
    a.n_dev = n_dev;
    a.scan_min_chain = kTreeScanMinChain;
    a.phase = base == 0 ? phase : kFull;
    a.tickets = &t->sync->early_tickets;
    a.go = go_by_flag && a.phase == kEarly ? &t->sync->go : nullptr;
    a.sorted = t->sorted;
    if (a.phase == kEarly)  // (tree_early_takes: compact)
      B2R_TRY((launch_big_chunk<BigCfgWide, true>(a, t->depth, stream)));
    else if (compact)
      B2R_TRY((launch_big_chunk<BigCfg1024, false>(a, t->depth, stream)));
    else
      B2R_TRY((launch_big_chunk<BigCfg4096, false>(a, t->depth, stream)));
  }
  return B2R_OK;
}

template int tree_apply<int64_t, double>(b2r_tree *, int64_t, const int64_t *,
                                         const double *, const uint8_t *,
                                         cudaStream_t, const int32_t *, int64_t, int,
    const b2r_exchange *, unsigned int *, bool);
template int tree_apply<int32_t, float>(b2r_tree *, int64_t, const int32_t *,
                                        const float *, const uint8_t *,
                                        cudaStream_t, const int32_t *, int64_t, int,
    const b2r_exchange *, unsigned int *, bool);
template int tree_apply<int32_t, double>(b2r_tree *, int64_t, const int32_t *,
                                         const double *, const uint8_t *,
                                         cudaStream_t, const int32_t *, int64_t, int,
    const b2r_exchange *, unsigned int *, bool);

TreeGo tree_go_of(b2r_tree *t) {
  TreeGo g;
  g.completed = &t->sync->completed;
  g.go = &t->sync->go;
  return g;
}

}  // namespace b2r

using b2r::as_stream;
using b2r::fail;

extern "C" {

int b2r_tree_create(int64_t capacity, b2r_tree **out) {
  if (out == nullptr) return fail(B2R_ERR_INVALID_ARGUMENT, "out is NULL");
  *out = nullptr;
  if (capacity <= 0)
    return fail(B2R_ERR_INVALID_ARGUMENT,
                "Sum tree capacity should be positive. Got: %lld",
                (long long)capacity);
  if (capacity > (1ll << 30))
    return fail(B2R_ERR_UNSUPPORTED, "capacity above 2^30 is not supported");
  int device_count = 0;
  if (cudaGetDeviceCount(&device_count) != cudaSuccess || device_count == 0)
    return fail(B2R_ERR_CUDA,
                "no CUDA device: libb200replay has no CPU fallback");
  b2r_tree *t = new (std::nothrow) b2r_tree();
  if (!t) return fail(B2R_ERR_INVALID_ARGUMENT, "out of host memory");
  t->capacity = capacity;
  int depth = 0;
  while ((1ll << depth) < capacity) ++depth;  // ceil(log2(capacity)), ST:81
  t->depth = depth;
  t->leaves = 1ll << depth;
  const size_t nodes = (size_t)(2 * t->leaves);  // 1-based heap, element 0 unused
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->heap), nodes * 8));
  B2R_CUDA(cudaMemset(t->heap, 0, nodes * 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->max_rec), 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->status), 16));
  B2R_CUDA(cudaMemset(t->status, 0, 16));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->delta), b2r::kTreeChunk * 8));
  B2R_CUDA(cudaMalloc(reinterpret_cast<void **>(&t->sync), sizeof(b2r::TreeSync)));
  B2R_CUDA(cudaMemset(t->sync, 0, sizeof(b2r::TreeSync)));
  const double one = 1.0;  // ST:89
  B2R_CUDA(cudaMemcpy(t->max_rec, &one, 8, cudaMemcpyHostToDevice));
  *out = t;
  return B2R_OK;
}

int b2r_tree_destroy(b2r_tree *t) {
  if (!t) return B2R_OK;
  cudaFree(t->heap);
  cudaFree(t->max_rec);
  cudaFree(t->status);
  cudaFree(t->delta);
  if (t->sorted) cudaFree(t->sorted);
  cudaFree(t->sync);
  t->bounce.release();
  delete t;
  return B2R_OK;
}

int b2r_tree_depth(const b2r_tree *t) { return t ? t->depth : -1; }

int b2r_tree_check(b2r_tree *t, b2r_stream stream) {
  int64_t st[2];
  B2R_CUDA(cudaMemcpyAsync(st, t->status, 16, cudaMemcpyDeviceToHost,
                           as_stream(stream)));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  if (st[0] == 0) return B2R_OK;
  B2R_CUDA(cudaMemsetAsync(t->status, 0, 16, as_stream(stream)));
  if (st[0] == B2R_ERR_NEGATIVE_PRIORITY)
    return fail(B2R_ERR_NEGATIVE_PRIORITY,
                "Sum tree values should be nonnegative (element %lld)",
                (long long)st[1]);
  return fail((int)st[0], "sum tree index out of range (element %lld)",
              (long long)st[1]);
}

int b2r_tree_set(b2r_tree *t, int64_t n, const int64_t *indices,
                 const double *values, int64_t *bad_pos, b2r_stream stream) {
  if (bad_pos) *bad_pos = -1;
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(t->bounce.reserve((size_t)n * 16 + 16));
  memcpy(t->bounce.host, indices, (size_t)n * 8);
  memcpy(t->bounce.host + (size_t)n * 8, values, (size_t)n * 8);
  B2R_CUDA(cudaMemcpyAsync(t->bounce.dev, t->bounce.host, (size_t)n * 16,
                           cudaMemcpyHostToDevice, s));
  // (tests: B2R_TREE_SET_PHASE=3 sends this call through the kernel that groups ahead of
  // its values, as the fused step does; indices and values come from a copy here, so its
  // promise holds trivially)
  const char *phase_env = std::getenv("B2R_TREE_SET_PHASE");
  const int phase = phase_env != nullptr && std::atoi(phase_env) == b2r::kEarly &&
                            b2r::tree_early_takes(n, -1)
                        ? b2r::kEarly
                        : b2r::kFull;
  B2R_TRY((b2r::tree_apply<int64_t, double>(
      t, n, reinterpret_cast<const int64_t *>(t->bounce.dev),
      reinterpret_cast<const double *>(t->bounce.dev + (size_t)n * 8), nullptr,
      s, nullptr, -1, phase)));
  int64_t st[2];
  B2R_CUDA(cudaMemcpyAsync(st, t->status, 16, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  if (st[0] != 0) {
    B2R_CUDA(cudaMemsetAsync(t->status, 0, 16, s));
    if (bad_pos) *bad_pos = st[1];
    if (st[0] == B2R_ERR_NEGATIVE_PRIORITY)
      return fail(B2R_ERR_NEGATIVE_PRIORITY,
                  "Sum tree values should be nonnegative. Got %g",
                  values[st[1]]);
    return fail((int)st[0], "index %lld is out of range for a tree of %lld leaves",
                (long long)indices[st[1]], (long long)t->leaves);
  }
  return B2R_OK;
}

int b2r_tree_set_device(b2r_tree *t, int64_t n, const int32_t *indices,
                        const float *values, b2r_stream stream) {
  if (n <= 0) return B2R_OK;
  return b2r::tree_apply<int32_t, float>(t, n, indices, values, nullptr,
                                         as_stream(stream));
}

int b2r_tree_get(b2r_tree *t, int64_t n, const int64_t *indices, double *out,
                 b2r_stream stream) {
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  for (int64_t k = 0; k < n; ++k)
    if (indices[k] < 0 || indices[k] >= t->leaves)
      return fail(B2R_ERR_INDEX_RANGE,
                  "index %lld is out of bounds for a tree of %lld leaves",
                  (long long)indices[k], (long long)t->leaves);
  B2R_TRY(t->bounce.reserve((size_t)n * 16));
  memcpy(t->bounce.host, indices, (size_t)n * 8);
  B2R_CUDA(cudaMemcpyAsync(t->bounce.dev, t->bounce.host, (size_t)n * 8,
                           cudaMemcpyHostToDevice, s));
  double *dout = reinterpret_cast<double *>(t->bounce.dev + (size_t)n * 8);
  b2r::tree_get_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(
      t->heap, t->leaves, n, reinterpret_cast<const int64_t *>(t->bounce.dev),
      dout);
  B2R_LAUNCHED();
  B2R_CUDA(cudaMemcpyAsync(t->bounce.host + (size_t)n * 8, dout, (size_t)n * 8,
                           cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  memcpy(out, t->bounce.host + (size_t)n * 8, (size_t)n * 8);
  return B2R_OK;
}

int b2r_tree_total(b2r_tree *t, double *out, b2r_stream stream) {
  B2R_CUDA(cudaMemcpyAsync(out, t->heap + 1, 8, cudaMemcpyDeviceToHost,
                           as_stream(stream)));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return B2R_OK;
}

int b2r_tree_max_recorded(b2r_tree *t, double *out, b2r_stream stream) {
  B2R_CUDA(cudaMemcpyAsync(out, t->max_rec, 8, cudaMemcpyDeviceToHost,
                           as_stream(stream)));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return B2R_OK;
}

int b2r_tree_set_max_recorded(b2r_tree *t, double value, b2r_stream stream) {
  b2r::tree_set_scalar_kernel<<<1, 1, 0, as_stream(stream)>>>(t->max_rec, value);
  B2R_LAUNCHED();
  return B2R_OK;
}

int b2r_tree_sample(b2r_tree *t, int64_t n, const double *query01, int64_t *out,
                    b2r_stream stream) {
  if (n <= 0) return B2R_OK;
  cudaStream_t s = as_stream(stream);
  B2R_TRY(t->bounce.reserve((size_t)n * 16 + 8));
  memcpy(t->bounce.host, query01, (size_t)n * 8);
  B2R_CUDA(cudaMemcpyAsync(t->bounce.dev, t->bounce.host, (size_t)n * 8,
                           cudaMemcpyHostToDevice, s));
  int64_t *dout = reinterpret_cast<int64_t *>(t->bounce.dev + (size_t)n * 8);
  double *dtotal = reinterpret_cast<double *>(t->bounce.dev + (size_t)n * 16);
  const size_t smem = ((size_t)2 << b2r::kTopLevels) * 8;
  b2r::tree_query_kernel<<<(unsigned)((n + 255) / 256), 256, smem, s>>>(
      t->heap, t->depth, n, reinterpret_cast<const double *>(t->bounce.dev),
      dout, dtotal, 0u);
  B2R_LAUNCHED();
  B2R_CUDA(cudaMemcpyAsync(t->bounce.host + (size_t)n * 8, dout,
                           (size_t)n * 8 + 8, cudaMemcpyDeviceToHost, s));
  B2R_CUDA(cudaStreamSynchronize(s));
  double total;
  memcpy(&total, t->bounce.host + (size_t)n * 16, 8);
  if (total == 0.0)
    return fail(B2R_ERR_EMPTY_TREE, "Cannot sample from an empty sum tree.");
  memcpy(out, t->bounce.host + (size_t)n * 8, (size_t)n * 8);
  return B2R_OK;
}

int b2r_tree_read_level(b2r_tree *t, int level, double *out, b2r_stream stream) {
  if (level < 0 || level > t->depth)
    return fail(B2R_ERR_INVALID_ARGUMENT, "level %d out of range", level);
  const size_t count = (size_t)1 << level;
  B2R_CUDA(cudaMemcpyAsync(out, t->heap + count, count * 8,
                           cudaMemcpyDeviceToHost, as_stream(stream)));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return B2R_OK;
}

int b2r_tree_write_level(b2r_tree *t, int level, const double *in,
                         b2r_stream stream) {
  if (level < 0 || level > t->depth)
    return fail(B2R_ERR_INVALID_ARGUMENT, "level %d out of range", level);
  const size_t count = (size_t)1 << level;
  B2R_CUDA(cudaMemcpyAsync(t->heap + count, in, count * 8,
                           cudaMemcpyHostToDevice, as_stream(stream)));
  B2R_CUDA(cudaStreamSynchronize(as_stream(stream)));
  return B2R_OK;
}

}  // extern "C"

#ifdef B2R_TRACE
extern "C" int b2r_debug_trace_tree(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_trace, sizeof(long long) * 32);
}
// [4][32]: per tree level — grouped, parent ended, released (leaf: deltas written), done
extern "C" int b2r_debug_trace_tree_levels(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_level_trace, sizeof(long long) * 128);
}
// [8]: launches of the early write-back, ... with every CTA's own list, ... that needed no
// hand-over behind the values
extern "C" int b2r_debug_trace_tree_phases(long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_phase_trace, sizeof(long long) * 32);
}
extern "C" int b2r_debug_trace_tree_counts(unsigned long long *out) {
  return (int)cudaMemcpyFromSymbol(out, b2r::g_trace_count, sizeof(unsigned long long) * 8);
}
#endif
