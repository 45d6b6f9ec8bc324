"""Replay sharded over the GPUs of one box (SURVEY.md section 8e).

The reference is single-process; this is the only multi-GPU piece of the path.
Every rank owns a complete `OutOfGraphPrioritizedReplayBuffer` shard (its own
cursor, validity window and sum tree) fed by its own actors.  A GLOBAL stratified
batch is drawn as if the G shard trees hung under one more tree level:

  1. each rank publishes its root priority total (one fp64) — the only collective
     on the path, an all-gather of G x 8 bytes over NCCL/NVLink;
  2. every rank scans the G totals in rank order with SumTree's own rule
     (`q < left ? descend : q -= left`, sum_tree.py:128-139) for each of the B
     strata and keeps those that land in its shard;
  3. it descends its local tree with the residual mass, fixes invalid picks with
     local retries exactly like prioritized_replay_buffer.py:156-170, and gathers
     its part of the batch.  No frame ever crosses NVLink.

The number of strata a shard serves is data dependent and stays on the device
(`count`); downstream kernels take it from there.

`ShardedUniformReplay` does the same for the uniform `OutOfGraphReplayBuffer`
(circular_replay_buffer.py:436-477): one global batch of uniform draws over the
concatenated index ranges of the shards.
"""
import ctypes

import numpy as np

from dopamine_b200 import _native


def all_gather_totals(local_total, group=None):
  """All-gathers one fp64 per rank into a (world,) tensor on the same device.

  Works with NCCL (CUDA tensors) and gloo (CPU tensors, used by the CPU tests)."""
  import torch
  import torch.distributed as dist
  world = dist.get_world_size(group)
  out = torch.empty(world, dtype=torch.float64, device=local_total.device)
  dist.all_gather_into_tensor(out, local_total.reshape(1), group=group)
  return out


class PeerExchange(object):
  """Shard totals over peer memory (NVLink) instead of an NCCL all-gather.

  Every rank owns a small device mailbox (`b2r_exchange_*` in the C ABI); the
  sharded sampling kernel stores its root total straight into the peers' mailboxes
  and polls its own, so the exchange costs one NVLink write latency inside a
  kernel that runs anyway.  `torch.distributed` is only used once, here, to swap
  the 64-byte CUDA IPC handles of the mailboxes.
  """

  def __init__(self, rank=None, world_size=None, group=None, timeout_s=2.0):
    import torch
    import torch.distributed as dist
    self._lib = _native.lib()
    self.rank = dist.get_rank(group) if rank is None else rank
    self.world = dist.get_world_size(group) if world_size is None else world_size
    handle = ctypes.c_void_p()
    _native.check(self._lib.b2r_exchange_create(self.world, self.rank,
                                                ctypes.byref(handle)))
    self._h = handle
    _native.check(self._lib.b2r_exchange_set_timeout(self._h, float(timeout_s)))
    if self.world > 1:
      mine = np.zeros(_native.IPC_HANDLE_BYTES, dtype=np.uint8)
      _native.check(self._lib.b2r_exchange_local_handle(self._h, _native.ptr(mine)))
      device = 'cuda' if dist.get_backend(group) == 'nccl' else 'cpu'
      send = torch.as_tensor(mine, device=device)
      recv = torch.empty(self.world * _native.IPC_HANDLE_BYTES, dtype=torch.uint8,
                         device=device)
      dist.all_gather_into_tensor(recv, send, group=group)
      handles = np.ascontiguousarray(recv.cpu().numpy())
      _native.check(self._lib.b2r_exchange_connect(self._h, _native.ptr(handles)))
      dist.barrier(group)  # every mailbox is mapped before anyone writes

  @classmethod
  def emulated(cls, world):
    """`world` exchanges on ONE device wired to each other by raw pointers: ranks
    emulated by sequential launches (tests)."""
    lib = _native.lib()
    out = []
    for rank in range(world):
      x = cls.__new__(cls)
      x._lib, x.rank, x.world = lib, rank, world
      handle = ctypes.c_void_p()
      _native.check(lib.b2r_exchange_create(world, rank, ctypes.byref(handle)))
      x._h = handle
      out.append(x)
    boxes = (ctypes.c_void_p * world)(*[lib.b2r_exchange_mailbox(x._h) for x in out])
    for x in out:
      _native.check(lib.b2r_exchange_connect_pointers(x._h, boxes))
    return out

  def set_early_publish(self, on=True):
    """The kernel that leaves the tree final for the next sharded step (write-back, or
    the flush of staged adds behind it) publishes the shard total itself; see
    b2r_exchange_set_early_publish for what the caller accepts with it."""
    _native.check(self._lib.b2r_exchange_set_early_publish(self._h, 1 if on else 0))

  def publish(self, memory):
    """Publishes `memory`'s total for the next step ahead of the sampling call
    (needed only when the ranks are emulated by sequential launches)."""
    _native.check(self._lib.b2r_exchange_publish_device(
        self._h, memory._h, _native.current_stream()))  # pylint: disable=protected-access

  def publish_uniform(self, memory, global_batch, seed, phase):
    """Publish-ahead of the uniform sampler's rounds for the next step (ranks emulated by
    sequential launches): phase 0 sends `memory`'s span; phase 1, once every rank has
    run phase 0, sends its rejection list (b2r_exchange_publish_uniform_device).
    `global_batch` and `seed` are those of the coming `ShardedUniformReplay` call."""
    _native.check(self._lib.b2r_exchange_publish_uniform_device(
        self._h, memory._h, int(global_batch), int(seed), 0, int(phase),  # pylint: disable=protected-access
        _native.current_stream()))

  def state(self):
    """The exchange's step number (b2r_exchange_state_get) as a dict of plain ints."""
    import torch
    words = np.zeros(_native.EXCHANGE_STATE_WORDS, dtype=np.uint64)
    _native.check(self._lib.b2r_exchange_state_get(
        self._h, _native.EXCHANGE_STATE_VERSION, _native.ptr(words), len(words),
        _native.current_stream()))
    torch.cuda.current_stream().synchronize()
    return {'version': _native.EXCHANGE_STATE_VERSION, 'words': [int(w) for w in words]}

  def set_state(self, state):
    """Restores what `state` returned and clears this rank's mailbox
    (b2r_exchange_state_set).  Every rank must restore the same step number, and none
    may start a step before every rank has restored."""
    words = np.ascontiguousarray(state['words'], dtype=np.uint64)
    _native.check(self._lib.b2r_exchange_state_set(
        self._h, int(state['version']), _native.ptr(words), len(words),
        _native.current_stream()))

  def __del__(self):
    if getattr(self, '_h', None):
      self._lib.b2r_exchange_destroy(self._h)
      self._h = None


def global_index(rank, shard_capacity, local_indices):
  """Index in the virtual replay of world * shard_capacity transitions."""
  return rank * shard_capacity + local_indices


class ShardedPrioritizedReplay(object):
  """Global stratified sampling over one local shard per rank."""

  def __init__(self, memory, rank=None, world_size=None, group=None, seed=0,
               exchange=None):
    import torch
    import torch.distributed as dist
    self.memory = memory
    self.group = group
    self.exchange = exchange  # PeerExchange, or None: NCCL / gloo all-gather
    self.rank = dist.get_rank(group) if rank is None else rank
    self.world = dist.get_world_size(group) if world_size is None else world_size
    self.seed = int(seed)
    self._lib = _native.lib()
    self._h = memory._h  # pylint: disable=protected-access
    self._send = torch.zeros(1, dtype=torch.float64, device='cuda')
    self._count = torch.zeros(1, dtype=torch.int32, device='cuda')
    self._torch = torch

  def local_total(self):
    """This shard's root priority as a 1-element CUDA tensor (no host sync)."""
    _native.check(self._lib.b2r_copy_total_device(
        self._h, self._send.data_ptr(), _native.current_stream()))
    return self._send

  def totals(self):
    return all_gather_totals(self.local_total(), self.group)

  def sample_index_batch(self, global_batch, totals=None, queries01=None,
                         retry_u01=None):
    """Returns (slots, indices, count): CUDA int32 tensors of length global_batch
    whose first `count` (device scalar) entries are this rank's strata."""
    torch = self._torch
    slots = torch.empty(global_batch, dtype=torch.int32, device='cuda')
    indices = torch.zeros(global_batch, dtype=torch.int32, device='cuda')
    n_retry = (len(retry_u01) if retry_u01 is not None else
               self.memory._max_sample_attempts)  # pylint: disable=protected-access
    if totals is None and self.exchange is not None:
      _native.check(self._lib.b2r_sample_indices_sharded_p2p_device(
          self._h, self.exchange._h, global_batch,  # pylint: disable=protected-access
          queries01.data_ptr() if queries01 is not None else None, n_retry,
          retry_u01.data_ptr() if retry_u01 is not None else None, self.seed, 0,
          slots.data_ptr(), indices.data_ptr(), self._count.data_ptr(),
          _native.current_stream()))
      return slots, indices, self._count
    if totals is None:
      totals = self.totals()
    _native.check(self._lib.b2r_sample_indices_sharded_device(
        self._h, global_batch, self.world, self.rank, totals.data_ptr(),
        queries01.data_ptr() if queries01 is not None else None, n_retry,
        retry_u01.data_ptr() if retry_u01 is not None else None, self.seed,
        0, slots.data_ptr(), indices.data_ptr(),
        self._count.data_ptr(), _native.current_stream()))
    return slots, indices, self._count

  def sample_transition_batch(self, global_batch, **kwargs):
    """(slots, count, batch tuple): batch rows [0, count) are valid."""
    slots, indices, count = self.sample_index_batch(global_batch, **kwargs)
    mem = self.memory
    _, arrays, batch = mem._alloc_outputs(global_batch, True)  # pylint: disable=protected-access
    _native.check(self._lib.b2r_gather_device_counted(
        self._h, global_batch, count.data_ptr(), indices.data_ptr(),
        ctypes.byref(batch), _native.current_stream()))
    return slots, count, tuple(arrays)

  def sample_transition_batch_sharded(self, global_batch, max_rows=None):
    """This rank's share of a global batch in one call over the peer exchange
    (b2r_sample_transition_batch_sharded_device): sharded sampler, scalar columns and
    frame copies.  Returns (slots, count, batch tuple, min_probability), CUDA tensors
    sized by `max_rows` rows (default `share_bound`); rows [0, count) are this rank's
    strata in ascending order, the rest are left from earlier calls.  min_probability
    (1,) is the minimum sampling probability of this rank's rows; the sampler has also
    published it to the peers for `rainbow_agent.c51_loss(..., sharded=...)`.  The
    tensors are reused by every call with the same sizes (static for CUDA graphs)."""
    if self.exchange is None:
      raise ValueError('sample_transition_batch_sharded needs a PeerExchange')
    torch = self._torch
    global_batch = int(global_batch)
    rows = (share_bound(global_batch, self.world) if max_rows is None
            else min(int(max_rows), global_batch))
    key = (global_batch, rows)
    if getattr(self, '_share_out', None) is None or self._share_out[0] != key:
      _, arrays, batch = self.memory._alloc_outputs(rows, True)  # pylint: disable=protected-access
      self._share_out = (key, torch.zeros(rows, dtype=torch.int32, device='cuda'),
                         tuple(arrays), batch,
                         torch.zeros(1, dtype=torch.float32, device='cuda'))
    _, slots, arrays, batch, min_probability = self._share_out
    _native.check(self._lib.b2r_sample_transition_batch_sharded_device(
        self._h, self.exchange._h, global_batch, self.seed, 0,  # pylint: disable=protected-access
        ctypes.byref(batch), slots.data_ptr(), self._count.data_ptr(), rows,
        min_probability.data_ptr(), _native.current_stream()))
    return slots, self._count, arrays, min_probability

  def flush(self):
    """Applies the staged adds (before a CUDA graph replay)."""
    self.memory._flush()  # pylint: disable=protected-access

  def check(self):
    """Raises the error latched by an earlier asynchronous call (a share beyond
    max_rows, a peer that did not answer in time, ...).  Synchronises."""
    _native.check(self._lib.b2r_check(self._h, _native.current_stream()))

  def set_priority(self, indices, priorities, count):
    """Batched priority write-back for the first `count` (device) entries."""
    _native.check(self._lib.b2r_set_priority_device_counted(
        self._h, indices.numel(), count.data_ptr(), indices.data_ptr(),
        priorities.data_ptr(), _native.current_stream()))


class ShardedUniformReplay(object):
  """ONE global uniform batch over one `OutOfGraphReplayBuffer` shard per rank.

  The batch is the reference's uniform batch (circular_replay_buffer.py:436-477) of a
  virtual buffer whose index range is the concatenation of the shards' ranges: every rank
  draws the same Philox candidates over the summed spans, each candidate belongs to the
  shard its offset lands in, and the ranks agree on which draws were accepted by
  exchanging their spans and the ordinals of their rejected draws over the peer mailboxes
  inside the sampling kernel (b2r_sample_transition_batch_uniform_sharded_device).  The
  result is uniform over the union of the shards' valid transitions."""

  def __init__(self, memory, rank, world_size, seed, exchange):
    import torch
    if exchange is None:
      raise ValueError('ShardedUniformReplay needs a PeerExchange')
    self.memory = memory
    self.exchange = exchange
    self.rank = int(rank)
    self.world = int(world_size)
    self.seed = int(seed)
    self._lib = _native.lib()
    self._h = memory._h  # pylint: disable=protected-access
    self._count = torch.zeros(1, dtype=torch.int32, device='cuda')
    self._torch = torch
    self._share_out = None

  def sample_transition_batch_sharded(self, global_batch, max_rows=None):
    """This rank's share of a global uniform batch in one call: sampler, scalar columns
    and frame copies.  Returns (slots, count, batch tuple), CUDA tensors sized by
    `max_rows` rows (default `share_bound`); rows [0, count) are this rank's accepted
    draws in global row order, slots[r] their global row, the rest are left from earlier
    calls.  The tensors are reused by every call with the same sizes (static for CUDA
    graphs)."""
    torch = self._torch
    global_batch = int(global_batch)
    rows = (share_bound(global_batch, self.world) if max_rows is None
            else min(int(max_rows), global_batch))
    key = (global_batch, rows)
    if self._share_out is None or self._share_out[0] != key:
      _, arrays, batch = self.memory._alloc_outputs(rows, True)  # pylint: disable=protected-access
      self._share_out = (key, torch.zeros(rows, dtype=torch.int32, device='cuda'),
                         tuple(arrays), batch)
    _, slots, arrays, batch = self._share_out
    _native.check(self._lib.b2r_sample_transition_batch_uniform_sharded_device(
        self._h, self.exchange._h, global_batch, self.seed, 0,  # pylint: disable=protected-access
        ctypes.byref(batch), slots.data_ptr(), self._count.data_ptr(), rows,
        _native.current_stream()))
    return slots, self._count, arrays

  def publish(self, global_batch, phase):
    """`PeerExchange.publish_uniform` for this shard (emulated ranks)."""
    self.exchange.publish_uniform(self.memory, global_batch, self.seed, phase)

  def flush(self):
    """Applies the staged adds (before a CUDA graph replay)."""
    _native.check(self._lib.b2r_flush(self._h, _native.current_stream()))

  def check(self):
    """Raises the error latched by an earlier asynchronous call (a share beyond
    max_rows, attempts exhausted, too few transitions, a peer that did not answer in
    time, ...).  Synchronises."""
    _native.check(self._lib.b2r_check(self._h, _native.current_stream()))


def share_bound(global_batch, world, slack=1.5, extra=32):
  """Rows a rank provides for its share of a global batch: `slack` times the even share
  plus `extra`, never more than the global batch.  A shard serves
  global_batch * total_g / sum(totals) strata, so shards fed alike stay within a few rows
  of the even share; a step that outgrows the bound latches B2R_ERR_UNSUPPORTED."""
  even = -(-int(global_batch) // int(world))
  return min(int(global_batch), int(np.ceil(slack * even)) + int(extra))


class ShardedStep(object):
  """bench.py's N>1 step: all-gather totals -> sharded sample -> gather -> C51
  loss/priorities -> write-back, for a global batch spread over the ranks."""

  def __init__(self, workload, global_batch, world, rank, dist, exchange=None,
               max_rows=None):
    import torch
    self.wl = workload
    self.global_batch = global_batch
    self.dist = dist
    self.exchange = exchange
    self.sharded = ShardedPrioritizedReplay(
        workload.mem, rank=rank, world_size=world, seed=1234, exchange=exchange)
    # Outputs, logits and launches are sized by a bound on the LOCAL share (peer
    # exchange path), so that a rank's memory and grids do not grow with the world size.
    self.max_rows = global_batch
    if exchange is not None:
      self.max_rows = (share_bound(global_batch, world) if max_rows is None
                       else min(int(max_rows), global_batch))
    t, b, c = workload.plan(self.max_rows)
    self.t, self.b, self.c = t, b, c
    self.slots = torch.empty(self.max_rows, dtype=torch.int32, device='cuda')
    c.batch_count = self.sharded._count.data_ptr()  # pylint: disable=protected-access
    c.mean_weighted_loss = None
    self.lib = workload.lib
    self.h = workload.h
    self._launches = None

  def step(self):
    nat, lib, sh = self.wl.native, self.lib, self.sharded
    stream = nat.current_stream()
    count_ptr = sh._count.data_ptr()  # pylint: disable=protected-access
    if self.exchange is not None:
      # one call: totals exchanged over peer memory inside the sampling kernel,
      # scalar columns from the sampler, frame copies on the forked stream
      nat.check(lib.b2r_train_step_sharded_device(
          self.h, self.exchange._h, self.global_batch, sh.seed, 0,  # pylint: disable=protected-access
          ctypes.byref(self.b), ctypes.byref(self.c), self.slots.data_ptr(),
          count_ptr, self.max_rows, stream))
      return
    totals = sh.totals()
    nat.check(lib.b2r_sample_indices_sharded_device(
        self.h, self.global_batch, sh.world, sh.rank, totals.data_ptr(), None,
        sh.memory._max_sample_attempts, None, sh.seed, 0,  # pylint: disable=protected-access
        self.slots.data_ptr(), self.t['indices'].data_ptr(), count_ptr, stream))
    nat.check(lib.b2r_gather_device_counted(
        self.h, self.global_batch, count_ptr, self.t['indices'].data_ptr(),
        ctypes.byref(self.b), stream))
    nat.check(lib.b2r_c51_loss(ctypes.byref(self.c), stream))
    nat.check(lib.b2r_set_priority_device_counted(
        self.h, self.global_batch, count_ptr, self.t['indices'].data_ptr(),
        self.t['priorities'].data_ptr(), stream))

  def check_partition(self, max_valid_checks=512):
    """After a step has run on EVERY rank: all-gathers each rank's (count, strata) and
    asserts that the ranks' strata partition range(global_batch) exactly — no stratum
    served twice or by nobody — and that this rank's rows are valid transitions of its
    own shard (circular_replay_buffer.py:381-414).  This is the check of the real
    multi-process exchange (CUDA-IPC mailboxes over NVLink): the ranks agree on the
    apportioning only if every one of them read the same G totals.  Returns the row
    counts of all ranks."""
    import torch
    dist, world = self.dist, self.sharded.world
    torch.cuda.synchronize()
    count = int(self.sharded._count.item())  # pylint: disable=protected-access
    cap = int(self.slots.numel())
    assert 0 <= count <= cap, (count, cap)
    send = torch.full((cap + 1,), -1, dtype=torch.int32, device='cuda')
    send[0] = count
    send[1:1 + count] = self.slots[:count]
    recv = torch.empty(world * (cap + 1), dtype=torch.int32, device='cuda')
    dist.all_gather_into_tensor(recv, send)
    recv = recv.cpu().numpy().reshape(world, cap + 1)
    counts = [int(c) for c in recv[:, 0]]
    strata = np.concatenate([recv[g, 1:1 + counts[g]] for g in range(world)])
    assert sum(counts) == self.global_batch, (counts, self.global_batch)
    assert np.array_equal(np.sort(strata), np.arange(self.global_batch)), (
        'the ranks\' strata do not partition the global batch')
    for g in range(world):  # rank-order scan: a rank's strata are ascending
      mine = recv[g, 1:1 + counts[g]]
      assert np.all(np.diff(mine) > 0), g
    indices = self.t['indices'][:count].cpu().numpy()
    mem = self.sharded.memory
    for index in indices[:max_valid_checks]:
      assert mem.is_valid_transition(int(index)), int(index)
    return counts

  def launches_per_step(self):
    if self._launches is None:
      before = self.lib.b2r_launch_count()
      self.step()
      self._launches = self.lib.b2r_launch_count() - before
    return self._launches
