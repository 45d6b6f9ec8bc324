/*
 * b200_replay.h — C ABI of libb200replay.so: Dopamine's replay-and-update hot path
 * on one B200 (sm_100a).  Plain pointers and sizes only; no torch types.
 *
 * The reference (K-Kielak/dopamine) is pure Python and has no FFI; the entry points
 * below are what a binding for its hot path would call.  Each one names the
 * reference interface it replaces (paths relative to the reference root):
 *   ST  = dopamine/replay_memory/sum_tree.py
 *   CRB = dopamine/replay_memory/circular_replay_buffer.py
 *   PRB = dopamine/replay_memory/prioritized_replay_buffer.py
 *   RA  = dopamine/agents/rainbow/rainbow_agent.py
 *
 * Conventions
 *   - every function returns a b2r_status; b2r_last_error() gives the text of the
 *     last failure on the calling thread.
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream).  Work is
 *     stream-ordered; a call synchronises the stream only when it has to hand a
 *     result back in HOST memory (documented per function).
 *   - "_device" variants take/return DEVICE pointers owned by the caller and never
 *     synchronise.  The others take HOST pointers.
 *   - handles are not thread-safe (neither is the reference: one host thread per
 *     buffer, see SURVEY.md section 8b).
 *   - there is no CPU fallback: without a CUDA device every create call fails.
 */
#ifndef B200_REPLAY_H_
#define B200_REPLAY_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b2r_tree b2r_tree;     /* GPU sum tree            (ST:30)  */
typedef struct b2r_buffer b2r_buffer; /* GPU circular replay     (CRB:80, PRB:36) */
typedef void *b2r_stream;             /* cudaStream_t */

typedef enum {
  B2R_OK = 0,
  B2R_ERR_INVALID_ARGUMENT = 1,
  B2R_ERR_CUDA = 2,
  B2R_ERR_NEGATIVE_PRIORITY = 3, /* ST:191-193 ValueError                     */
  B2R_ERR_EMPTY_TREE = 4,        /* ST:116-117, 159-160 Exception             */
  B2R_ERR_SAMPLE_ATTEMPTS = 5,   /* CRB:471-475 / PRB:160-163 RuntimeError    */
  B2R_ERR_TOO_FEW_TRANSITIONS = 6, /* CRB:457-460 RuntimeError                */
  B2R_ERR_INDEX_RANGE = 7,
  B2R_ERR_UNSUPPORTED = 8,
  B2R_ERR_EXCHANGE = 9,          /* a peer shard did not publish its total in time */
  B2R_QUEUE_FULL = 10,           /* b2r_add with B2R_STREAM_NONE: flush, then retry */
  B2R_ERR_STALE_TOTAL = 11       /* early publish: the tree changed after the shard's total
                                    for the next step had been given to the peers        */
} b2r_status;

/* Stream argument of b2r_add / b2r_add_atari meaning "never launch from this call":
 * if the staging queue has no room the call changes nothing and returns
 * B2R_QUEUE_FULL; the caller then calls b2r_flush(buf, stream) and adds again.
 * Lets a host loop add rows without looking up its current stream every time. */
#define B2R_STREAM_NONE ((b2r_stream)(intptr_t)-1)

const char *b2r_last_error(void);
/* Version of this header's structs and signatures; a binding compares it with the
 * version it was written against when it loads the library (dopamine_b200/_native.py). */
#define B2R_ABI_VERSION 3
int b2r_abi_version(void);
/* Number of kernels this library has launched in this process (for bench.py's
 * gpu_launches claim). */
int64_t b2r_launch_count(void);

/* ------------------------------------------------------------------------- */
/* Sum tree — replaces sum_tree.SumTree (ST:30-205).                          */
/* fp64 nodes, one 1-based heap array: node (level l, position i) at 2^l + i.  */
/* ------------------------------------------------------------------------- */

/* SumTree.__init__ (ST:65-89). capacity <= 0 -> B2R_ERR_INVALID_ARGUMENT. */
int b2r_tree_create(int64_t capacity, b2r_tree **out);
int b2r_tree_destroy(b2r_tree *tree);
/* len(SumTree.nodes) - 1 (ST:81). */
int b2r_tree_depth(const b2r_tree *tree);

/* n x SumTree.set applied IN ARRAY ORDER (ST:178-205 as looped by PRB:213-214):
 * duplicates chain, every ancestor receives the deltas in order, so all fp64 nodes
 * are bit-identical to the reference's.  A negative value at position k applies
 * elements [0,k) and returns B2R_ERR_NEGATIVE_PRIORITY (*bad_pos = k).
 * HOST arrays; synchronises. */
int b2r_tree_set(b2r_tree *tree, int64_t n, const int64_t *indices,
                 const double *values, int64_t *bad_pos, b2r_stream stream);
/* Same, DEVICE arrays (int32 indices, f32 values: what the loss kernel emits).
 * Asynchronous; a negative value latches an error reported by b2r_tree_check. */
int b2r_tree_set_device(b2r_tree *tree, int64_t n, const int32_t *indices,
                        const float *values, b2r_stream stream);
/* Returns (and clears) a latched asynchronous error. Synchronises. */
int b2r_tree_check(b2r_tree *tree, b2r_stream stream);

/* SumTree.get (ST:168-176). HOST arrays; synchronises. */
int b2r_tree_get(b2r_tree *tree, int64_t n, const int64_t *indices, double *out,
                 b2r_stream stream);
/* SumTree._total_priority (ST:91-97) and .max_recorded_priority (ST:89, 194). */
int b2r_tree_total(b2r_tree *tree, double *out, b2r_stream stream);
int b2r_tree_max_recorded(b2r_tree *tree, double *out, b2r_stream stream);
int b2r_tree_set_max_recorded(b2r_tree *tree, double value, b2r_stream stream);

/* SumTree.sample (ST:99-141) for n explicit query values in [0,1] (the caller
 * draws them, so the reference's RNG stream can be reproduced):
 * out[k] = leaf reached by descending with query01[k] * root.
 * Empty tree -> B2R_ERR_EMPTY_TREE. HOST arrays; synchronises. */
int b2r_tree_sample(b2r_tree *tree, int64_t n, const double *query01,
                    int64_t *out, b2r_stream stream);

/* SumTree.nodes[level] (ST:79-87): 2^level doubles. HOST; synchronises. */
int b2r_tree_read_level(b2r_tree *tree, int level, double *out,
                        b2r_stream stream);
int b2r_tree_write_level(b2r_tree *tree, int level, const double *in,
                         b2r_stream stream);

/* ------------------------------------------------------------------------- */
/* Replay buffer — replaces OutOfGraphReplayBuffer (CRB:80-687) and            */
/* OutOfGraphPrioritizedReplayBuffer (PRB:36-252).                             */
/* ------------------------------------------------------------------------- */

#define B2R_MAX_EXTRAS 8
#define B2R_COL_OBSERVATION 0
#define B2R_COL_ACTION 1
#define B2R_COL_REWARD 2
#define B2R_COL_TERMINAL 3
#define B2R_COL_EXTRA0 4

typedef struct {
  int64_t capacity;            /* replay_capacity                    CRB:101 */
  int32_t stack_size;          /* CRB:100                                    */
  int32_t update_horizon;      /* CRB:103                                    */
  double gamma;                /* CRB:104 (discounts = f32(pow(gamma,k)) CRB:181) */
  int32_t max_sample_attempts; /* CRB:105                                    */
  int32_t prioritized;         /* 0: CRB:80, 1: PRB:36 (owns a b2r_tree)     */
  int64_t obs_bytes;           /* bytes of one observation                   */
  int32_t obs_itemsize;        /* bytes of one observation element           */
  int32_t action_bytes;        /* bytes of one action row                    */
  int32_t reward_itemsize;     /* 4 = float32, 8 = float64 (scalar rewards)  */
  int32_t terminal_itemsize;   /* 1/2/4/8-byte integer                       */
  int32_t num_extras;          /* extra_storage_types               CRB:106  */
  int32_t extra_bytes[B2R_MAX_EXTRAS]; /* bytes of one row of each extra     */
  int32_t add_queue_rows;      /* rows staged on the host before an automatic
                                  flush; 0 = library default                 */
} b2r_config;

int b2r_create(const b2r_config *config, b2r_buffer **out);
int b2r_destroy(b2r_buffer *buf);
/* The PER buffer's tree (`memory.sum_tree`, PRB:98); NULL for the uniform buffer. */
b2r_tree *b2r_buffer_tree(b2r_buffer *buf);

/* Priority argument of add(): an explicit value, or "whatever
 * sum_tree.max_recorded_priority is when the row is applied" (RA:330-334),
 * resolved on the device so the caller never has to read it back. */
#define B2R_PRIORITY_EXPLICIT 0
#define B2R_PRIORITY_MAX_RECORDED 1

/* OutOfGraphReplayBuffer.add (CRB:234-260) incl. the stack_size-1 zero
 * transitions at episode starts (CRB:255-259), and for PER the
 * sum_tree.set(cursor, priority) that precedes each row (PRB:139-140).
 * All pointers are HOST rows already cast to the storage dtypes.  Rows are staged
 * in pinned memory and applied by one kernel at the next flush; every call below
 * that reads buffer state flushes first, so the deferral is not observable. */
int b2r_add(b2r_buffer *buf, const void *observation, const void *action,
            const void *reward, const void *terminal,
            const void *const *extras, double priority, int priority_mode,
            b2r_stream stream);
/* b2r_add for the Atari layout (scalar int32 action, float32 reward, uint8 terminal,
 * no extras) with the scalars passed by value: one call, no host-side row buffers.
 * Other layouts -> B2R_ERR_UNSUPPORTED. */
int b2r_add_atari(b2r_buffer *buf, const void *observation, int32_t action,
                  float reward, uint8_t terminal, double priority,
                  int priority_mode, b2r_stream stream);
/* n consecutive add()s of ONE trajectory stream in one call (the loop of
 * DQNAgent._store_transition over a chunk of steps: an actor that hands over the steps of
 * an environment in blocks, a vectorised environment with one replay shard per
 * environment — the frame stacks of a buffer are built from CONSECUTIVE slots, so the
 * steps of different environments never share one).  Column arrays hold n rows each in
 * the storage dtypes, HOST.  Exactly the effects of n b2r_add calls in array order
 * (zero transitions after every terminal == 1, invalid_range, PER priorities;
 * priorities == NULL with B2R_PRIORITY_MAX_RECORDED), staged together and applied by as
 * few flush kernels as the staging buffer allows.  A negative explicit priority stops at
 * its row like the reference's loop would (*added = rows committed before it). */
int b2r_add_batch(b2r_buffer *buf, int64_t n, const void *observations,
                  const void *actions, const void *rewards, const void *terminals,
                  const void *const *extras, const double *priorities, int priority_mode,
                  int64_t *added, b2r_stream stream);
int b2r_flush(b2r_buffer *buf, b2r_stream stream);

/* add_count (CRB:177), cursor() (CRB:334-336), invalid_range (CRB:53-77, 285-287). */
int64_t b2r_add_count(const b2r_buffer *buf);
int64_t b2r_cursor(const b2r_buffer *buf);
int b2r_get_invalid_range(const b2r_buffer *buf, int64_t *out, int32_t *n);
/* For load() (CRB:656-687): overwrite the bookkeeping after the stores. */
int b2r_set_state(b2r_buffer *buf, int64_t add_count,
                  const int64_t *invalid_range, int32_t n);

/* is_valid_transition (CRB:381-414) evaluated on the device for n indices.
 * HOST arrays; synchronises. */
int b2r_valid_mask(b2r_buffer *buf, int64_t n, const int64_t *indices,
                   uint8_t *out, b2r_stream stream);

/* Uniform sample_index_batch (CRB:436-477).
 * b2r_uniform_bounds: min_id/max_id of CRB:449-460 (TOO_FEW_TRANSITIONS as there).
 * b2r_sample_indices_uniform consumes, in order, `candidates` =
 * np.random.randint(min_id, max_id) draws made by the caller: each is reduced
 * mod capacity, accepted if valid, otherwise counted as a failed attempt, until
 * `batch` are accepted or max_sample_attempts failed (CRB:464-470).  The counters
 * are in/out so a caller can feed several windows.  HOST arrays; synchronises. */
int b2r_uniform_bounds(const b2r_buffer *buf, int64_t *min_id, int64_t *max_id);
int b2r_sample_indices_uniform(b2r_buffer *buf, int32_t batch, int32_t n_cand,
                               const int64_t *candidates, int32_t *out_indices,
                               int32_t *accepted, int32_t *rejected,
                               int32_t *draws_used, b2r_stream stream);

/* Prioritized sample_index_batch (PRB:142-171) with the caller's uniforms:
 * strat_query01[i] = random.uniform(bounds[i], bounds[i+1]) (ST:162-165);
 * retry_u01[r] = the r-th random.random() a retry would draw (ST:123), n_retry
 * should be max_sample_attempts.  Reproduces the shared attempt budget, the
 * in-order replacement of invalid slots and the "last slot may stay invalid"
 * quirk.  *draws_used = retry draws the reference would have consumed.
 * On B2R_ERR_SAMPLE_ATTEMPTS *fail_slot is the `i` of PRB:160-163.
 * HOST arrays; synchronises. */
int b2r_sample_indices_prioritized(b2r_buffer *buf, int32_t batch,
                                   const double *strat_query01, int32_t n_retry,
                                   const double *retry_u01,
                                   int32_t *out_indices, int32_t *draws_used,
                                   int32_t *fail_slot, b2r_stream stream);

/* Throughput mode: indices drawn on the device with Philox4x32-10 keyed by
 * (seed, offset); same sampling rules, not stream-compatible with Python's RNG.
 * Uniform or prioritized according to the buffer.  DEVICE output; asynchronous;
 * attempt exhaustion latches an error reported by b2r_check. */
int b2r_sample_indices_device(b2r_buffer *buf, int32_t batch, uint64_t seed,
                              uint64_t offset, int32_t *out_indices,
                              b2r_stream stream);
int b2r_check(b2r_buffer *buf, b2r_stream stream);

/* Outputs of sample_transition_batch in get_transition_elements order
 * (CRB:571-590, PRB:246-252).  Any pointer may be NULL to skip that output. */
typedef struct {
  void *state;          /* (B, obs..., stack)  observation dtype */
  void *action;         /* (B, action...)                        */
  void *reward;         /* (B,) n-step discounted return         */
  void *next_state;     /* (B, obs..., stack)                    */
  void *next_action;    /* (B, action...)                        */
  void *next_reward;    /* (B,)                                  */
  void *terminal;       /* (B,) terminal dtype, 0/1              */
  int32_t *indices;     /* (B,)                                  */
  void *extras[B2R_MAX_EXTRAS];
  float *sampling_probabilities; /* (B,) PER only: f32(leaf)  PRB:193-200 */
} b2r_batch;

/* The per-index body of sample_transition_batch (CRB:516-556): frame stacks with
 * the stack axis innermost, n-step return cut at the first terminal, next_* taken
 * at (i + L) mod capacity, terminal mask, indices, extras, raw leaf priorities.
 * DEVICE pointers; asynchronous. */
int b2r_gather_device(b2r_buffer *buf, int32_t batch, const int32_t *indices,
                      const b2r_batch *out, b2r_stream stream);
/* Which frame-copy kernel a launch of `batch` rows takes: 0 gather_stack4_u8_kernel
 * (registers: LDG.128 -> PRMT -> STG.128), 1 gather_stack4_u8_tma_kernel (frames staged
 * through cp.async.bulk into shared memory), 2 gather_generic_kernel (other layouts). */
int32_t b2r_gather_variant(const b2r_buffer *buf, int32_t batch);
/* Same with HOST indices and HOST outputs (copies inside); synchronises. */
int b2r_gather(b2r_buffer *buf, int32_t batch, const int32_t *indices,
               const b2r_batch *out, b2r_stream stream);
/* The OutOfGraph return convention (host arrays, CRB:479-558) at PCIe speed: the batch
 * is built in a device slab and shipped with ONE copy into `host_slab`, which the
 * caller allocates page-locked (b2r_gather moves every column into pageable memory with
 * a copy of its own).  `want`: a non-NULL field means the column is wanted, its value is
 * ignored.  *host_out receives pointers INTO host_slab for the wanted columns (256-byte
 * aligned segments); *needed the bytes the slab must hold — call with host_slab == NULL
 * to ask for the size and the layout only (*host_out then holds the columns' OFFSETS in
 * the slab; nothing is sampled or copied).  indices: HOST, or DEVICE when indices_on_device != 0 (a
 * batch sampled by b2r_sample_indices_device never visits the host before the copy).
 * Synchronises: the arrays are ready when the call returns. */
int b2r_gather_slab(b2r_buffer *buf, int32_t batch, const int32_t *indices,
                    int32_t indices_on_device, const b2r_batch *want, void *host_slab,
                    size_t slab_bytes, b2r_batch *host_out, size_t *needed,
                    b2r_stream stream);
/* Device-RNG sampling + gather in one call (two launches). DEVICE; asynchronous. */
int b2r_sample_transition_batch_device(b2r_buffer *buf, int32_t batch,
                                       uint64_t seed, uint64_t offset,
                                       const b2r_batch *out, b2r_stream stream);

/* set_priority / get_priority (PRB:203-235) — b2r_tree_set/get on the buffer's
 * tree after flushing pending adds. */
int b2r_set_priority(b2r_buffer *buf, int64_t n, const int32_t *indices,
                     const double *priorities, int64_t *bad_pos,
                     b2r_stream stream);
int b2r_set_priority_device(b2r_buffer *buf, int64_t n, const int32_t *indices,
                            const float *priorities, b2r_stream stream);
int b2r_get_priority(b2r_buffer *buf, int64_t n, const int32_t *indices,
                     float *out, b2r_stream stream);
int b2r_get_priority_device(b2r_buffer *buf, int64_t n, const int32_t *indices,
                            float *out, b2r_stream stream);

/* Raw access to `_store[name]` rows for save()/load() (CRB:596-687) and tests.
 * HOST memory; synchronises. */
int b2r_store_read(b2r_buffer *buf, int32_t column, int64_t row0, int64_t nrows,
                   void *out, b2r_stream stream);
int b2r_store_write(b2r_buffer *buf, int32_t column, int64_t row0,
                    int64_t nrows, const void *in, b2r_stream stream);
/* Device address of a column (read-only use by callers that stay on the GPU). */
const void *b2r_store_device_ptr(b2r_buffer *buf, int32_t column);

/* Checkpoint files of a store column as blocked gzip (save() / load(), CRB:593-687).
 * The column's bytes (capacity x row bytes) are cut into 65280-byte slices; slice k-1 is
 * gzip member k, compressed on the device by one CTA: header 1f 8b 08, FLG FEXTRA, MTIME
 * 0, XFL 0, OS 255, one BGZF extra subfield 'B' 'C' with BSIZE = member size - 1; a raw
 * deflate body of one fixed-Huffman block, or one stored block where that is smaller
 * (matches stay inside the member, distances <= 32768); CRC-32 and ISIZE.  Member 0, the
 * .npy header, is the caller's.  Any gzip reader inflates the whole file as one stream.
 * Work goes through fixed windows of 1024 members, double-buffered, so device and pinned
 * scratch do not grow with the capacity and the file I/O overlaps the kernels.
 *
 * b2r_ckpt_save_column appends members 1..M to `fd` at its current position and sets
 * *bytes_out to the bytes appended.  verify_only != 0: writes nothing; every member is
 * compressed, inflated again on the device and compared with the column (any difference
 * -> B2R_ERR_INVALID_ARGUMENT), *bytes_out the size the members would take.
 * b2r_ckpt_load_column reads members 1..M from `fd` at byte `offset` (pread: the file
 * position does not move) and inflates them straight into the column.  Only members in
 * the format above are accepted; anything else — a bad header or BSIZE, another block type,
 * a bad code or distance, a CRC-32 or ISIZE that does not match, a missing member, bytes
 * after the last one — returns B2R_ERR_INVALID_ARGUMENT naming the member, never a device
 * fault.  A member is written only after its own checks pass; verify_only != 0 runs every
 * check and writes nothing, so a caller that verifies first never leaves a column half
 * loaded.  Both synchronise. */
int b2r_ckpt_save_column(b2r_buffer *buf, int32_t column, int32_t fd, int32_t verify_only,
                         int64_t *bytes_out, b2r_stream stream);
int b2r_ckpt_load_column(b2r_buffer *buf, int32_t column, int32_t fd, int64_t offset,
                         int32_t verify_only, b2r_stream stream);

/* The sampler state of a buffer that only the device holds, for a checkpoint that resumes
 * the same draws: word 0 the draw counter of the Philox samplers, word 1 the counter of
 * the sharded prioritized sampler (it advances in lockstep on every rank).  `words` is
 * B2R_SAMPLER_STATE_WORDS uint64 in host or device memory.  _get copies the counters
 * into `words` and _set copies `words` into them, both with cudaMemcpyAsync on `stream`
 * (host memory: synchronise `stream` before reading what _get wrote).  _set refuses a
 * version or word count other than these before it touches the buffer or the device. */
#define B2R_SAMPLER_STATE_VERSION 1
#define B2R_SAMPLER_STATE_WORDS 2
int b2r_sampler_state_get(b2r_buffer *buf, int32_t version, uint64_t *words,
                          int32_t n_words, b2r_stream stream);
int b2r_sampler_state_set(b2r_buffer *buf, int32_t version, const uint64_t *words,
                          int32_t n_words, b2r_stream stream);

/* Sharded replay (SURVEY.md section 8e): one buffer per GPU; shard_totals[g] is
 * rank g's root priority (device array, e.g. straight out of an NCCL all-gather).
 * For each of the global_batch strata i (query01[i] in [0,1], DEVICE), mass =
 * query01[i] * (sum of totals, rank order); the owner is found by the same
 * "q < left ? left : (q -= left, right)" rule as ST:128-139 applied to the G
 * totals in rank order, and only the owning rank descends its tree with the
 * residual.  out_slots/out_indices receive this rank's strata (ascending i) and
 * *out_count their number.  Invalid picks are redrawn locally from retry_u01
 * exactly as in PRB:156-170.  query01 / retry_u01 may be NULL: the uniforms then
 * come from Philox keyed by (seed, offset) — the strata stream is identical on all
 * ranks, the retry stream is rank-private (n_retry = attempt budget); the draw
 * number is offset + a device counter that every such call advances, so all ranks
 * must make the same sequence of sharded calls.
 * DEVICE pointers; asynchronous. */
int b2r_sample_indices_sharded_device(b2r_buffer *buf, int32_t global_batch,
                                      int32_t num_shards, int32_t rank,
                                      const double *shard_totals,
                                      const double *query01, int32_t n_retry,
                                      const double *retry_u01, uint64_t seed,
                                      uint64_t offset, int32_t *out_slots,
                                      int32_t *out_indices, int32_t *out_count,
                                      b2r_stream stream);
/* Shard totals over peer memory (NVLink / NVSwitch) instead of a collective
 * library: every rank owns a small device mailbox; inside the sharded sampling
 * kernel each rank stores its root total straight into every peer's mailbox and
 * polls its own, so the "all-gather" costs one NVLink write latency and no extra
 * launch.  Set-up: create on every rank, exchange the 64-byte handles by any
 * transport (torch.distributed, MPI, a file), connect.  All ranks must then make
 * the same sequence of exchange-based calls (each call is one step of a device
 * counter).  A peer that does not answer within the timeout (default 2 s) latches
 * B2R_ERR_EXCHANGE, reported by b2r_check; later calls then skip the wait. */
typedef struct b2r_exchange b2r_exchange;
#define B2R_IPC_HANDLE_BYTES 64
int b2r_exchange_create(int32_t world, int32_t rank, b2r_exchange **out);
int b2r_exchange_destroy(b2r_exchange *exchange);
/* cudaIpcMemHandle_t of this rank's mailbox (B2R_IPC_HANDLE_BYTES bytes, HOST). */
int b2r_exchange_local_handle(b2r_exchange *exchange, void *handle_out);
/* handles: world x B2R_IPC_HANDLE_BYTES in rank order (the own entry is ignored);
 * opens the peers' mailboxes with peer access enabled. */
int b2r_exchange_connect(b2r_exchange *exchange, const void *handles);
/* Same-process variant for ranks emulated on one device (tests): mailboxes[g] is
 * rank g's b2r_exchange_mailbox(). */
int b2r_exchange_connect_pointers(b2r_exchange *exchange, void *const *mailboxes);
void *b2r_exchange_mailbox(b2r_exchange *exchange);
int b2r_exchange_set_timeout(b2r_exchange *exchange, double seconds);
/* Early publish.  By default a rank publishes its shard total at the start of the
 * sampling kernel that needs the peers' totals, so every step waits one NVLink store
 * latency inside that kernel.  With on != 0 the kernel that leaves the tree in its final
 * state for the NEXT sharded step — the priority write-back of
 * b2r_train_step_sharded_device, or the flush of staged add()s when there is one —
 * publishes the new root the moment it is written (one-CTA tree kernels: shares of up
 * to 256 rows; larger write-backs keep publishing from the sampler).  Consequences the
 * caller accepts with the switch: (i) add()s staged before a step call are applied at the
 * END of that call, behind its write-back, and become visible to the next step's sampler
 * (the order of effects on the tree stays add, sample, set_priority, add, ...); (ii)
 * between two sharded steps nothing else may change the tree (set_priority, a flush
 * forced by another call): the next sampler finds the root different from what was
 * published and latches B2R_ERR_STALE_TOTAL instead of letting the ranks apportion
 * the batch from different totals.  Every rank of an exchange must use the same setting. */
int b2r_exchange_set_early_publish(b2r_exchange *exchange, int32_t on);
/* The step number of an exchange, for a checkpoint: word 0 is the step counter (its
 * parity picks the mailbox slot of the next step, its low 32 bits + 1 the tag a peer
 * polls for).  `words` is B2R_EXCHANGE_STATE_WORDS uint64 in host or device memory,
 * copied with cudaMemcpyAsync on `stream` as in b2r_sampler_state_get / _set, which also
 * refuse what these refuse.  _set also clears this rank's mailbox and its record of what
 * it has published, so that no word written before the restore can carry the tag of a
 * step after it.  That is safe because every rank restores the same step number: no peer
 * has published for a step beyond it, and none may do so before every rank's _set has
 * run (the caller holds the ranks at a barrier in between). */
#define B2R_EXCHANGE_STATE_VERSION 1
#define B2R_EXCHANGE_STATE_WORDS 1
int b2r_exchange_state_get(b2r_exchange *exchange, int32_t version, uint64_t *words,
                           int32_t n_words, b2r_stream stream);
int b2r_exchange_state_set(b2r_exchange *exchange, int32_t version, const uint64_t *words,
                           int32_t n_words, b2r_stream stream);
/* Publishes this rank's total for the NEXT step without consuming the step (the
 * sampling call publishes again, identically).  Only needed when ranks are
 * emulated by sequential launches on one device, where a launch cannot wait for a
 * later one.  Asynchronous. */
int b2r_exchange_publish_device(b2r_exchange *exchange, b2r_buffer *buf,
                                b2r_stream stream);
/* b2r_sample_indices_sharded_device with the totals taken from the exchange. */
int b2r_sample_indices_sharded_p2p_device(b2r_buffer *buf, b2r_exchange *exchange,
                                          int32_t global_batch,
                                          const double *query01, int32_t n_retry,
                                          const double *retry_u01, uint64_t seed,
                                          uint64_t offset, int32_t *out_slots,
                                          int32_t *out_indices, int32_t *out_count,
                                          b2r_stream stream);

/* The first half of b2r_train_step_sharded_device alone: the sharded sampler (totals
 * over the exchange, this rank's strata compacted at the front of `out`, *out_count of
 * them, out_slots[r] = stratum of row r; the scalar columns written by the sampler) and
 * the frame copies, joined into `stream` before the call returns.  No loss, no
 * write-back: a learner runs its networks on the max_rows rows of `out` next, then
 * b2r_c51_loss_sharded and b2r_set_priority_device_counted.  *min_probability
 * (DEVICE) receives the minimum sampling probability of this rank's rows, and the
 * sampler publishes it to every peer of the exchange for this step.  max_rows as in
 * b2r_train_step_sharded_device (0 = global_batch); a share above it latches
 * B2R_ERR_UNSUPPORTED (b2r_check).  Early publish is not used by this call.
 * DEVICE pointers; asynchronous; can be captured in a CUDA graph. */
int b2r_sample_transition_batch_sharded_device(b2r_buffer *buf, b2r_exchange *exchange,
                                               int32_t global_batch, uint64_t seed,
                                               uint64_t offset, const b2r_batch *out,
                                               int32_t *out_slots, int32_t *out_count,
                                               int32_t max_rows, float *min_probability,
                                               b2r_stream stream);

/* Sharded UNIFORM replay: this rank's share of ONE global batch of `global_batch`
 * transitions drawn as OutOfGraphReplayBuffer draws them (CRB:436-477) from a virtual
 * buffer whose index range is the concatenation of the shards' ranges.  Rank g's span is
 * n_g = max(0, max_id_g - min_id_g) (CRB:449-460, read on the device), N = sum of the
 * spans.  Draw j is u_j = philox_uniform53(seed, offset + step, j), with `step` the
 * exchange's step number (its step counter + 1; every sampling call over the exchange
 * closes one step); o_j = min((int64)(u_j * N), N - 1); the owner is the rank the scan
 * "o < n_g ? g : o -= n_g" in rank order stops at; the candidate is
 * (min_id_owner + o) mod capacity.  Draws are processed in order while accepted <
 * global_batch and rejected < max_sample_attempts (CRB:464-470); draw j is accepted iff
 * it is a valid transition of its owner's shard, and the k-th accepted draw is global
 * row k.  For one rank this is the mapping of b2r_sample_indices_device.
 * The ranks agree on the accepted draws in two rounds over the exchange's mailboxes,
 * inside the sampling kernel: the spans, then each rank's ordinals of rejected draws.
 * This rank's rows are its accepted draws in row order: out->indices[r] the index,
 * out_slots[r] the global row, *out_count (DEVICE) their number; the scalar columns and
 * frames of those rows are gathered into `out` (rows past the count are left alone).
 * max_rows: rows the outputs hold (0 = global_batch); a larger share serves max_rows rows
 * and latches B2R_ERR_UNSUPPORTED.  No shard with enough transitions latches
 * B2R_ERR_TOO_FEW_TRANSITIONS, a loop that ends short B2R_ERR_SAMPLE_ATTEMPTS (on every
 * rank alike), a peer that does not answer in time B2R_ERR_EXCHANGE (b2r_check).
 * Refused before any device work: a buffer with max_sample_attempts above 1024, an
 * exchange with early publish on.  DEVICE pointers; asynchronous; can be captured in a
 * CUDA graph. */
int b2r_sample_transition_batch_uniform_sharded_device(
    b2r_buffer *buf, b2r_exchange *exchange, int32_t global_batch, uint64_t seed,
    uint64_t offset, const b2r_batch *out, int32_t *out_slots, int32_t *out_count,
    int32_t max_rows, b2r_stream stream);
/* Publish-ahead of the uniform sampler's rounds for the exchange's NEXT step, for ranks
 * emulated by sequential launches on one device: phase 0 publishes this rank's span;
 * phase 1 (after every rank's phase 0) collects the spans and publishes the rank's
 * rejection list.  The sampling call then republishes nothing (a list published ahead
 * that no longer matches the buffer latches B2R_ERR_STALE_TOTAL).  Same arguments as the
 * sampling call.  Asynchronous. */
int b2r_exchange_publish_uniform_device(b2r_exchange *exchange, b2r_buffer *buf,
                                        int32_t global_batch, uint64_t seed,
                                        uint64_t offset, int32_t phase, b2r_stream stream);

/* Variants whose element count lives on the DEVICE (*count <= max_...): what a
 * shard serves of a global batch is only known there.  Rows past *count are
 * skipped.  Asynchronous. */
int b2r_gather_device_counted(b2r_buffer *buf, int32_t max_batch,
                              const int32_t *count, const int32_t *indices,
                              const b2r_batch *out, b2r_stream stream);
int b2r_set_priority_device_counted(b2r_buffer *buf, int64_t max_n,
                                    const int32_t *count, const int32_t *indices,
                                    const float *priorities, b2r_stream stream);
/* Copies the buffer's root total into dst (device), e.g. the send buffer of the
 * all-gather.  Asynchronous. */
int b2r_copy_total_device(b2r_buffer *buf, double *dst, b2r_stream stream);
/* Device address of the buffer's root total (input of the all-gather). */
const double *b2r_total_device_ptr(b2r_buffer *buf);

/* ------------------------------------------------------------------------- */
/* C51 — replaces the TF graph of RA:200-305 and project_distribution          */
/* (RA:340-494).  f32, DEVICE pointers, asynchronous.                          */
/* ------------------------------------------------------------------------- */

/* project_distribution(supports, weights, target_support) (RA:340-494):
 * out[b,i] = sum_j clip(1 - |clip(s[b,j], z0, zN-1) - z_i| / (z1 - z0), 0, 1) * w[b,j] */
int b2r_c51_project(int32_t batch, int32_t num_atoms, const float *supports,
                    const float *weights, const float *target_support,
                    float *out, b2r_stream stream);

typedef struct {
  int32_t batch, num_actions, num_atoms;
  float cumulative_gamma;       /* f32(pow(gamma, n))               DQ:175, RA:232 */
  const float *support;         /* (N,)                             RA:126 */
  const float *target_logits;   /* (B, A, N) target net on next_state  RA:238-248 */
  const float *online_logits;   /* (B, A, N) online net on state       RA:262-267 */
  const int32_t *actions;       /* (B,)                                          */
  const float *rewards;         /* (B,) n-step returns                 RA:221 */
  const uint8_t *terminals;     /* (B,)                                RA:229 */
  const float *sampling_probabilities; /* (B,) or NULL (uniform scheme) RA:278 */
  float *target;                /* (B, N) projected target or NULL     RA:250 */
  float *loss;                  /* (B,) cross entropy                  RA:269 */
  float *priorities;            /* (B,) sqrt(loss + 1e-10)             RA:290 */
  float *weights;               /* (B,) IS weights / max or NULL       RA:279-280 */
  float *mean_weighted_loss;    /* scalar or NULL                      RA:293, 305 */
  float *grad_logits;           /* (B, A, N) d mean(w*loss)/d online_logits or NULL */
  const int32_t *batch_count;   /* NULL, or DEVICE count <= batch of rows to process */
  const float *min_probability; /* NULL, or DEVICE scalar min_b sampling_probabilities[b]
                                   (what b2r_train_step_device's sampler leaves behind);
                                   NULL: reduced inside the kernel                  */
} b2r_c51_args;

/* Bellman target + projection + softmax cross-entropy + new priorities + IS
 * weights in one launch (RA:200-293). */
int b2r_c51_loss(const b2r_c51_args *args, b2r_stream stream);

/* The loss of one shard of a global batch of `global_batch` strata, sampled by
 * b2r_sample_transition_batch_sharded_device over the same exchange (the call that
 * closed the exchange's current step).  The same arithmetic per row as b2r_c51_loss;
 * args->batch is the rank's max_rows, args->batch_count (required) its row count and
 * args->min_probability (required with sampling_probabilities) the sampler's local
 * minimum.  The IS-weight normaliser is the minimum over every rank's published local
 * minimum, so the weights are those of the whole global batch (RA:279-280);
 * mean_weighted_loss = (sum over this rank's rows of w * loss) / global_batch and
 * grad_logits its derivative, with rows >= count written as zeros.  Summed over the
 * ranks, the means and the gradients are the global batch's (RA:293).  A peer whose
 * minimum does not arrive within the exchange's timeout latches B2R_ERR_EXCHANGE in
 * the sampled buffer (b2r_check).  DEVICE pointers; asynchronous. */
int b2r_c51_loss_sharded(const b2r_c51_args *args, b2r_exchange *exchange,
                         int32_t global_batch, b2r_stream stream);

/* DQN (dqn_agent.py:283-322): Bellman target r + gamma^n max_a Q_target(s') (1 - t),
 * Huber loss (delta 1) against Q_online(s, a), optional mean and gradient.  f32,
 * DEVICE pointers, asynchronous. */
typedef struct {
  int32_t batch, num_actions;
  float cumulative_gamma;       /* f32(pow(gamma, n))               DQ:175 */
  const float *target_q;        /* (B, A) target net on next_state  DQ:291-292 */
  const float *online_q;        /* (B, A) online net on state       DQ:308-312 */
  const int32_t *actions;       /* (B,)                                         */
  const float *rewards;         /* (B,) n-step returns                          */
  const uint8_t *terminals;     /* (B,)                                         */
  float *loss;                  /* (B,) Huber loss per row or NULL  DQ:315-316  */
  float *target;                /* (B,) Bellman target or NULL      DQ:299-300  */
  float *mean_loss;             /* scalar or NULL                   DQ:321      */
  float *grad_q;                /* (B, A) d mean(loss)/d online_q or NULL       */
  const int32_t *batch_count;   /* NULL, or DEVICE count <= batch of rows       */
} b2r_dqn_args;
int b2r_dqn_loss(const b2r_dqn_args *args, b2r_stream stream);
/* The loss of one shard of a global batch of `global_batch` transitions, as
 * b2r_sample_transition_batch_uniform_sharded_device samples it.  args->batch is the
 * rank's max_rows and args->batch_count (DEVICE, required) its row count.  Rows b < count
 * get the loss, target and gradient row b2r_dqn_loss gives that transition on the whole
 * global batch (gradient clip(e, -1, 1) / global_batch); rows b >= count get loss 0 and
 * zero gradient rows, their target is not written.  mean_loss = (sum over this rank's
 * rows of loss, in f64, rounded once) / global_batch: summed over the ranks, the means and
 * the gradients are the global batch's (DQ:321).  DEVICE pointers; asynchronous. */
int b2r_dqn_loss_sharded(const b2r_dqn_args *args, int32_t global_batch,
                         b2r_stream stream);

/* ------------------------------------------------------------------------- */
/* The whole hot path in one call (SURVEY.md 3.2: what one sess.run(train_op)   */
/* does around the network): PRB:142-201 -> RA:200-293 -> PRB:203-214.          */
/* ------------------------------------------------------------------------- */

/* Prioritized sample (device Philox, as b2r_sample_indices_device) -> batch
 * assembly -> C51 loss / new priorities -> priority write-back.  The sampler
 * writes the scalar columns of the batch itself (n-step return, terminal, actions,
 * sampling_probabilities and their minimum), so the loss and the write-back follow
 * it directly on `stream`, while the frame-stack copies (state / next_state) run
 * beside them on an internal stream that forks after the sampler and joins
 * `stream` again before the call returns: later work on `stream` sees the whole
 * batch.  In `c51`, actions / rewards / terminals / sampling_probabilities /
 * min_probability and batch are taken from `out` (whatever the caller put there is
 * ignored).  out->indices, reward, terminal, action and (prioritized buffers)
 * sampling_probabilities are required.  DEVICE pointers; asynchronous; can be
 * captured in a CUDA graph.
 * The logits in `c51` are inputs that exist before the batch is sampled: row r of them
 * meets whatever transition the sampler draws for row r.  This is the path measured
 * without a network in the middle; a learner runs b2r_sample_transition_batch_device,
 * its networks, b2r_c51_loss and b2r_set_priority_device in that order (RA:253-305). */
int b2r_train_step_device(b2r_buffer *buf, int32_t batch, uint64_t seed,
                          uint64_t offset, const b2r_batch *out,
                          const b2r_c51_args *c51, b2r_stream stream);

/* Deferred frame copies.  By default the frame-stack copies of b2r_train_step_device are
 * joined into `stream` before the call returns.  With on != 0 they are joined only by
 * b2r_join_frames (or by the next flush of staged add()s, which overwrite ring slots the
 * copies may still read): the NEXT step's sampler -> loss -> write-back chain, which
 * needs this step's priorities but not its frames, then runs beside the HBM-bound copies
 * of this step — the analogue of the reference's staged prefetch (use_staging,
 * CRB:728-779), except that the tree sees exactly the sequential order sample(n),
 * set_priority(n), sample(n+1).  The copies of consecutive steps stay in order among
 * themselves (they share the output buffers in `out`).  The caller joins before it
 * reads state / next_state, before it ends a stream capture, and before destroying
 * `out`'s buffers.  out->indices is valid as soon as the step's sampler has run; the
 * copies read a private copy of it. */
int b2r_set_deferred_frames(b2r_buffer *buf, int32_t on);
int b2r_join_frames(b2r_buffer *buf, b2r_stream stream);

/* The same for one shard of a sharded replay (SURVEY.md section 8e): global
 * stratified batch of `global_batch` strata over `exchange`'s ranks, this rank's
 * rows compacted at the front of `out` (*out_count of them, device; out_slots[r] =
 * stratum of row r), loss and write-back over those rows only.  The single
 * exchange of shard totals happens inside the sampling kernel.
 * max_rows: rows that `out`, `out_slots`, the logits and the outputs of `c51` hold — a
 * bound on this rank's share of the global batch chosen by the caller (its expected
 * share is global_batch / world when the shards' totals are alike); every launch
 * behind the sampler and every buffer is sized by it, so a rank's memory and grids do
 * not grow with the number of ranks.  A step whose share exceeds it serves its first
 * max_rows strata and latches B2R_ERR_UNSUPPORTED (b2r_check).  0 = global_batch. */
int b2r_train_step_sharded_device(b2r_buffer *buf, b2r_exchange *exchange,
                                  int32_t global_batch, uint64_t seed,
                                  uint64_t offset, const b2r_batch *out,
                                  const b2r_c51_args *c51, int32_t *out_slots,
                                  int32_t *out_count, int32_t max_rows,
                                  b2r_stream stream);

/* Host-facing, pipelined form of the same step: what an agent's training loop
 * calls once per update with the network outputs in HOST memory
 * (dqn_agent.py:359-442 around rainbow_agent.py:253-305).  The trainer owns the
 * device copies of the logits, the batch outputs and a ring of pinned result
 * slots. */
typedef struct b2r_trainer b2r_trainer;

typedef struct {
  int32_t batch, num_actions, num_atoms;
  float vmax;              /* support = linspace(-vmax, vmax, N) in f32 (RA:126)   */
  float cumulative_gamma;  /* f32(pow(gamma, update_horizon))       (DQ:175)       */
  uint64_t seed;           /* Philox key of the sampler                            */
  int32_t pipeline_depth;  /* 0: each call returns its own losses (synchronous);
                              d > 0: the losses of the step queued d calls earlier */
  int32_t use_graph;       /* != 0: after two eager steps the kernels of a step are
                              replayed as one captured CUDA graph per call          */
  int32_t logit_rows;      /* rows of each logits tensor copied per step; 0 = batch.
                              A sharded trainer's batch is the GLOBAL batch, but a
                              rank's network only produces logits for the rows it
                              serves: the caller passes (logit_rows, A, N) tensors.
                              It is the max_rows of b2r_train_step_sharded_device:
                              every device buffer, the loss_out of a step and the
                              launches behind the sampler are sized by it, and a step
                              whose share exceeds it latches B2R_ERR_UNSUPPORTED     */
} b2r_trainer_config;

int b2r_trainer_create(b2r_buffer *buf, const b2r_trainer_config *config,
                       b2r_trainer **out);
int b2r_trainer_destroy(b2r_trainer *trainer);

/* One training iteration.  Applies the staged add()s, copies both logits tensors
 * ((B, A, N) f32, HOST; page-locked memory keeps the copies asynchronous and must
 * then stay untouched until the step has run), runs b2r_train_step_device and
 * copies the per-row losses back.  loss_out (B floats, HOST) receives the losses
 * of step number *loss_step (0-based; -1 and untouched while the pipeline fills).
 * The host only ever waits for a step queued pipeline_depth calls ago. */
int b2r_trainer_step_host(b2r_trainer *trainer, const float *online_logits,
                          const float *target_logits, float *loss_out,
                          int64_t *loss_step, b2r_stream stream);
/* Sharded trainer (one per rank): the configured batch becomes the GLOBAL batch of
 * b2r_train_step_sharded_device, this rank's rows are compacted at the front of the
 * batch and of loss_out, and b2r_trainer_last_rows() tells how many of them the step
 * reported by the last step_host / drain call had.  Call before the first step; the
 * sharded trainer always launches eagerly (use_graph is ignored). */
int b2r_trainer_set_exchange(b2r_trainer *trainer, b2r_exchange *exchange);
int32_t b2r_trainer_last_rows(const b2r_trainer *trainer);
/* Waits for everything queued; loss_out / *loss_step describe the last step. */
int b2r_trainer_drain(b2r_trainer *trainer, float *loss_out, int64_t *loss_step,
                      b2r_stream stream);
/* Device views of the trainer's batch (valid for the last step that has run) and
 * of its loss outputs (loss, priorities, weights in a b2r_c51_args). */
int b2r_trainer_views(b2r_trainer *trainer, b2r_batch *batch, b2r_c51_args *c51);

/* Actor side of the path (the step before add): DQNAgent.state, a (1, H, W, S)
 * frame stack with the stack index innermost, and the two methods that change it
 * (dqn_agent.py:444-458 _record_observation: np.roll(state, -1, axis=-1) then
 * state[0, ..., -1] = observation; dqn_agent.py:474-476 _reset_state: fill(0)).
 * `state` is the caller's DEVICE tensor (pixels * stack_size elements of elem_size
 * bytes); the handle owns a ring of `slots` pinned host frames (0 = default) that
 * b2r_actor_record copies the HOST observation into and that ONE kernel reads
 * zero-copy while it rolls the stack.  A slot is reused only after the launch that
 * read it has completed, so the call never waits unless `slots` records are in
 * flight. */
typedef struct b2r_actor b2r_actor;
int b2r_actor_create(int64_t pixels, int32_t elem_size, int32_t stack_size,
                     int32_t slots, b2r_actor **out);
int b2r_actor_destroy(b2r_actor *actor);
int b2r_actor_reset(b2r_actor *actor, void *state, b2r_stream stream);
int b2r_actor_record(b2r_actor *actor, void *state, const void *observation,
                     b2r_stream stream);

/* The network's input cast (atari_lib.py:124-125: tf.cast(state, tf.float32) followed by
 * tf.div(net, 255.)) fused with the layout change the first convolution needs: uint8
 * frame stacks (images, pixels, stack_size), stack axis innermost — the replay batch's
 * `state` / `next_state`, the actor's state — to (images, stack_size, pixels) planes of
 * float32 (half_out == 0: float(u8) / 255 by true division, the reference's values bit
 * for bit) or float16 (the same quotient rounded once).  One pass over the data instead
 * of a permute, a cast and a division.  DEVICE pointers; asynchronous. */
int b2r_stack_to_planes_device(const void *stacks, void *planes, int64_t images,
                                int64_t pixels, int32_t stack_size, int32_t half_out,
                                b2r_stream stream);

/* IQN (implicit_quantile_agent.py:166-315): greedy next action from the action
 * network's K quantile samples (:176-188), target quantile values
 * r + gamma^n (1 - t) Z_target[., a*] (:190-231), the quantile-Huber loss of every
 * (target sample t', online sample t) pair, summed over t and averaged over t'
 * (:278-311), its mean over the batch (:315) and d mean / d Z_online.  All network
 * outputs are DEVICE (samples * batch, num_actions) f32 matrices with the
 * reference's sample-major row order (row = sample * batch + b).  One launch. */
typedef struct {
  int32_t batch, num_actions;
  int32_t num_tau_samples;        /* N : online samples  (:233-262)              */
  int32_t num_tau_prime_samples;  /* N': target samples  (:196-231)              */
  int32_t num_quantile_samples;   /* K : samples behind the greedy action (:166) */
  float cumulative_gamma;         /* f32(pow(gamma, update_horizon))  (DQ:175)   */
  float kappa;                    /* Huber threshold, > 0             (:283-289) */
  int32_t reserved;
  const float *action_quantile_values; /* (K * B, A): target net, or online net with
                                          double_dqn (:166-175)                   */
  const float *target_quantile_values; /* (N' * B, A)                             */
  const float *online_quantile_values; /* (N * B, A)                              */
  const float *quantiles;              /* (N * B): tau of each online row         */
  const int32_t *actions;              /* (B)                                     */
  const float *rewards;                /* (B)                                     */
  const uint8_t *terminals;            /* (B)                                     */
  float *loss;                         /* (B) out                                 */
  float *mean_loss;                    /* scalar out, nullable                    */
  float *grad_quantile_values;         /* (N * B, A) out, nullable                */
  int32_t *next_action;                /* (B) out, nullable: a*                   */
} b2r_iqn_args;
int b2r_iqn_loss(const b2r_iqn_args *args, b2r_stream stream);

/* The loss of one shard of a global batch of `global_batch` strata, as
 * b2r_sample_transition_batch_sharded_device samples it (IQN's replay is the prioritized
 * buffer with unit priorities, implicit_quantile.gin:23-24).  The same arithmetic per
 * row as b2r_iqn_loss; args->batch is the rank's max_rows (the row stride of every
 * (samples * batch, A) matrix) and *count (DEVICE, required) its row count.  Rows
 * b < count get the loss, next_action and gradient rows b2r_iqn_loss gives that
 * transition on the whole global batch (the gradient scale is
 * -1 / (kappa * N' * global_batch)); rows b >= count get loss 0 and zero gradient rows,
 * and their next_action is not written.  mean_loss = (sum over this rank's rows of
 * loss) / global_batch.  IQN has no importance weights, so nothing is exchanged:
 * summed over the ranks, the means and the gradients are the global batch's (:315).
 * DEVICE pointers; asynchronous; can be captured in a CUDA graph. */
int b2r_iqn_loss_sharded(const b2r_iqn_args *args, const int32_t *count,
                         int32_t global_batch, b2r_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_REPLAY_H_ */
