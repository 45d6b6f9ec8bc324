"""What the learners share beyond their loss: the update replayed as one CUDA graph, the
rank plumbing of a data-parallel learner on ONE global batch sharded over the ranks
(`agent.ShardedRainbowLearner`, `learner.ShardedIQNLearner`,
`learner.ShardedDQNLearner`), and its checkpoints (`ShardedLearner.save` / `restore`)."""
import hashlib
import json
import os

# Checkpoint files of the iteration this many before the one written are removed, as the
# replay buffer does with its own (circular_replay_buffer.CHECKPOINT_DURATION).
CHECKPOINT_DURATION = 4
CHECKPOINT_FORMAT = 1


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


class CheckpointError(ValueError):
  """A sharded checkpoint that cannot be restored into these learners.  Raised before
  anything is changed."""


def load_optimizer_state(optimizer, state_dict):
  """`Optimizer.load_state_dict` that copies into the optimizer's existing state tensors
  when it has them, so that a captured CUDA graph keeps reading them; an optimizer that
  has not stepped yet takes the state as torch's loader gives it."""
  torch = _torch()
  params = [p for group in optimizer.param_groups for p in group['params']]
  saved = state_dict['state']
  have = [optimizer.state.get(p) for p in params]
  if not saved or not all(have):
    torch.optim.Optimizer.load_state_dict(optimizer, state_dict)
    return
  if sorted(saved) != list(range(len(params))) or any(
      sorted(saved[i]) != sorted(have[i]) for i in range(len(params))):
    raise ValueError('the saved optimizer state does not match this optimizer')
  with torch.no_grad():
    for i, p in enumerate(params):
      for key, tensor in have[i].items():
        tensor.copy_(saved[i][key])
  for group, loaded in zip(optimizer.param_groups, state_dict['param_groups']):
    group.update({k: v for k, v in loaded.items() if k != 'params'})


def _write_atomically(path, data):
  tmp = path + '.tmp'
  with open(tmp, 'wb') as f:
    f.write(data)
  os.replace(tmp, path)


def _remove(path):
  try:
    os.remove(path)
  except FileNotFoundError:
    pass


class _Files(object):
  """Where a sharded checkpoint of one iteration lives:
    checkpoint_dir/manifest_ckpt.<it>.json          rank 0: what the run is
    checkpoint_dir/learner_ckpt.<it>.pt             rank 0: networks, optimizer, counters
    checkpoint_dir/sentinel_checkpoint_complete.<it>   rank 0, after every rank has written
    checkpoint_dir/rank_<g>/...                     rank g: its shard, reference layout
    checkpoint_dir/rank_<g>/sharded_state_ckpt.<it>.json   rank g: sampler + exchange words"""

  def __init__(self, checkpoint_dir, iteration):
    self.dir, self.iteration = checkpoint_dir, int(iteration)
    name = lambda fmt: os.path.join(checkpoint_dir, fmt.format(self.iteration))
    self.manifest = name('manifest_ckpt.{}.json')
    self.learner = name('learner_ckpt.{}.pt')
    self.sentinel = name('sentinel_checkpoint_complete.{}')

  def rank_dir(self, rank):
    return os.path.join(self.dir, 'rank_{}'.format(rank))

  def rank_state(self, rank):
    return os.path.join(self.rank_dir(rank),
                        'sharded_state_ckpt.{}.json'.format(self.iteration))


def _params_sha256(online_state, target_state):
  """Checksum of the online and target networks' tensors, in state_dict order."""
  digest = hashlib.sha256()
  for state in (online_state, target_state):
    for name, tensor in state.items():
      digest.update(name.encode('utf-8'))
      digest.update(tensor.detach().cpu().contiguous().numpy().tobytes())
  return digest.hexdigest()


class GraphedUpdate(object):
  """`train_step()` runs `_update()` eagerly, or with `_cuda_graph` replays ONE CUDA
  graph of it captured on the first call: one launch per update instead of ~150 eager
  ones.  Staged adds are flushed before every replay; the sampler's validity context and
  draw counter live on the device, so the replayed graph sees new transitions and draws
  fresh strata.  The learner sets `_cuda_graph`, `_graph` (None) and `_static_loss`, and
  lists in `_graph_generators()` the torch generators its update draws from."""

  def train_step(self):
    """One update; returns the scalar training loss (a CUDA tensor, no sync)."""
    if not self._cuda_graph:
      return self._update()
    if self._graph is None:
      self._capture()
    self._flush_replay()
    self._graph.replay()
    self.updates += 1
    return self._static_loss

  def _graph_generators(self):
    return ()

  def _flush_replay(self):
    """Applies the replay's staged adds (the graph's sampler reads the ring)."""
    self.memory._flush()  # pylint: disable=protected-access

  def _capture(self):
    torch = _torch()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
      for _ in range(3):  # lazy allocations, cuDNN algorithm selection, Adam state
        self._update()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    self._flush_replay()
    self._graph = torch.cuda.CUDAGraph()
    for generator in self._graph_generators():  # each replay draws fresh numbers
      self._graph.register_generator_state(generator)
    with torch.cuda.graph(self._graph):
      self._static_loss = self._update()


class ShardedLearner(GraphedUpdate):
  """The rank plumbing of a learner whose `batch_size` is the GLOBAL batch, drawn over
  the ranks' replay shards (`ShardedPrioritizedReplay`, `ShardedUniformReplay`).  Every
  rank owns one shard and a peer-memory exchange; parameters start as rank 0's; every
  gradient views one flat buffer whose last entry is the partial loss, so `reduce()` is
  ONE all-reduce.  The learner calls `_connect()` before, and `_shard()` after, the
  single-GPU learner's constructor, and provides `loss_backward()`, `apply()` and
  `_update()`.  Pass `exchange` (`PeerExchange.emulated`) to run the phases of several
  ranks on one device without torch.distributed (tests); `reduce()` then is the
  caller's."""

  def _connect(self, exchange, group, exchange_timeout_s, ddp):
    """The exchange of this rank: `exchange`, or one over torch.distributed's group."""
    import torch.distributed as dist  # pylint: disable=g-import-not-at-top
    from dopamine_b200.replay_memory import sharded_replay  # pylint: disable=g-import-not-at-top
    if ddp:
      raise ValueError('the sharded learner reduces its gradients itself (ddp=False)')
    self._dist = dist if exchange is None else None
    if exchange is None:
      if not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError('{} needs torch.distributed initialised'.format(
            type(self).__name__))
      exchange = sharded_replay.PeerExchange(group=group, timeout_s=exchange_timeout_s)
    self._group = group
    return exchange

  def _shard(self, exchange, max_rows, seed, replay_class):
    """The sharded replay over `self.memory` (`replay_class`: `ShardedPrioritizedReplay`
    or `ShardedUniformReplay`), rank 0's parameters (and target) on every rank, and the
    flat gradient buffer."""
    torch = _torch()
    from dopamine_b200.replay_memory import sharded_replay  # pylint: disable=g-import-not-at-top
    self.exchange = exchange
    self.rank, self.world = exchange.rank, exchange.world
    self.sharded = replay_class(self.memory, rank=self.rank, world_size=self.world,
                                seed=seed, exchange=exchange)
    self.max_rows = (sharded_replay.share_bound(self.batch_size, self.world)
                     if max_rows is None else min(int(max_rows), int(self.batch_size)))
    params = list(self.online.parameters())
    if self._dist is not None:
      with torch.no_grad():
        for p in params:
          self._dist.broadcast(p, 0, group=self._group)
      super(ShardedLearner, self).sync_target()
    # every gradient views one flat buffer; the partial loss rides at its end
    total = sum(p.numel() for p in params)
    self._flat = torch.zeros(total + 1, dtype=torch.float32, device='cuda')
    offset = 0
    for p in params:
      p.grad = self._flat[offset:offset + p.numel()].view_as(p)
      offset += p.numel()
    self.loss = self._flat[total:]
    self._sample = None

  def _flush_replay(self):
    self.sharded.flush()

  # -- phases ------------------------------------------------------------------------
  def sample(self):
    """This rank's share: (slots, count, batch tuple) and, from a prioritized shard,
    min_probability."""
    self._sample = self.sharded.sample_transition_batch_sharded(self.batch_size,
                                                                self.max_rows)
    return self._sample

  def reduce(self):
    """The one all-reduce of the update: gradients and loss summed over the ranks."""
    self._dist.all_reduce(self._flat, group=self._group)

  def check(self):
    """Raises what the device latched since the last check (synchronises); also
    verifies that backward left every gradient in the flat buffer."""
    lo, hi = self._flat.data_ptr(), self._flat.data_ptr() + 4 * self._flat.numel()
    for p in self.online.parameters():
      if p.grad is None or not lo <= p.grad.data_ptr() < hi:
        raise RuntimeError('a gradient left the all-reduced buffer')
    self.sharded.check()

  def sync_target(self):
    self.check()
    super(ShardedLearner, self).sync_target()

  # -- checkpoints -------------------------------------------------------------------
  # Every rank writes its shard into checkpoint_dir/rank_<g>/ through the buffer's own
  # `save` (each rank's GPU compresses its shard), and beside it the device words that
  # decide its next draws; rank 0 also writes the learner state and the manifest.  The
  # checkpoint counts as complete once the sentinel exists, written after every rank has
  # written (`finish_save`).  A restore validates everything on every rank, the shards'
  # device verify pass included, before any rank changes anything, then copies into the
  # existing tensors: a learner whose update was captured as a CUDA graph keeps replaying
  # it.  Ranks emulated on one device: `save_ranks` / `restore_ranks`.

  def _kind(self):
    scheme = getattr(self, 'replay_scheme', None)
    return type(self).__name__ + ('' if scheme is None else ':' + scheme)

  def _manifest(self):
    return {'format': CHECKPOINT_FORMAT, 'kind': self._kind(), 'world_size': self.world,
            'global_batch': int(self.batch_size), 'max_rows': int(self.max_rows),
            'shard_capacity': int(self.memory._replay_capacity),  # pylint: disable=protected-access
            'update_horizon': int(self.memory._update_horizon),  # pylint: disable=protected-access
            'seed': int(self.sharded.seed)}

  def _learner_state(self):
    """Networks, optimizer (its step count included) and counters, as saved."""
    return {'online': self.online.state_dict(), 'target': self.target.state_dict(),
            'optimizer': self.optimizer.state_dict(),
            'training_steps': int(self.training_steps), 'updates': int(self.updates)}

  def _load_learner_state(self, state):
    """The inverse of `_learner_state`, copying into the existing tensors."""
    self.online.load_state_dict(state['online'])
    self.target.load_state_dict(state['target'])
    self.optimizer.load_state_dict(state['optimizer'])
    self.training_steps = int(state['training_steps'])
    self.updates = int(state['updates'])

  def _rank_state(self):
    """What each rank saves of its own: the words that decide its next draws."""
    return {'rank': self.rank, 'world_size': self.world,
            'sampler': self.memory.sampler_state(), 'exchange': self.exchange.state()}

  def _load_rank_state(self, state):
    self.memory.set_sampler_state(state['sampler'])
    self.exchange.set_state(state['exchange'])

  def _agree(self, ok):
    """True on every rank iff `ok` on every rank (one all-reduce); emulated ranks: ok."""
    if self._dist is None:
      return ok
    torch = _torch()
    device = 'cuda' if self._dist.get_backend(self._group) == 'nccl' else 'cpu'
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=device)
    self._dist.all_reduce(flag, op=self._dist.ReduceOp.MIN, group=self._group)
    return bool(flag.item())

  def save(self, checkpoint_dir, iteration):
    """Writes this rank's part of checkpoint `iteration`: staged adds flushed, deferred
    frame copies joined and latched errors raised first.  Over torch.distributed every
    rank calls it, and rank 0 then writes the sentinel; emulated ranks: `save_ranks`."""
    from dopamine_b200 import _native  # pylint: disable=g-import-not-at-top
    files = _Files(checkpoint_dir, iteration)
    error = None
    try:
      if self.rank == 0:  # an iteration written again is incomplete until it is done
        _remove(files.sentinel)
      self._flush_replay()
      _native.check(_native.lib().b2r_join_frames(self.memory._h,  # pylint: disable=protected-access
                                                  _native.current_stream()))
      self.check()
      rank_dir = files.rank_dir(self.rank)
      os.makedirs(rank_dir, exist_ok=True)
      self.memory.save(rank_dir, files.iteration)
      _write_atomically(files.rank_state(self.rank),
                        json.dumps(self._rank_state()).encode('utf-8'))
      _remove(_Files(checkpoint_dir, files.iteration - CHECKPOINT_DURATION).rank_state(
          self.rank))
      if self.rank == 0:
        self._save_learner(files)
    except Exception as e:  # pylint: disable=broad-except
      error = e
    if not self._agree(error is None):
      raise error or RuntimeError('another rank failed to write checkpoint {}'.format(
          files.iteration))
    if self._dist is not None and self.rank == 0:
      self.finish_save(checkpoint_dir, iteration)

  def _save_learner(self, files):
    torch = _torch()
    import io  # pylint: disable=g-import-not-at-top
    state = self._learner_state()
    manifest = dict(self._manifest(), iteration=files.iteration,
                    training_steps=state['training_steps'], updates=state['updates'],
                    params_sha256=_params_sha256(state['online'], state['target']))
    blob = io.BytesIO()
    torch.save(state, blob)
    _write_atomically(files.learner, blob.getvalue())
    _write_atomically(files.manifest, json.dumps(manifest, indent=1).encode('utf-8'))

  def finish_save(self, checkpoint_dir, iteration):
    """Marks checkpoint `iteration` complete (rank 0, once every rank's `save` has
    returned) and removes the files of the iteration CHECKPOINT_DURATION before it."""
    files = _Files(checkpoint_dir, iteration)
    missing = [g for g in range(self.world) if not os.path.exists(files.rank_state(g))]
    if missing or not os.path.exists(files.manifest):
      raise CheckpointError('checkpoint {} is not written by every rank (missing: {})'.
                            format(files.iteration, missing or 'manifest'))
    _write_atomically(files.sentinel, b'complete\n')
    stale = _Files(checkpoint_dir, files.iteration - CHECKPOINT_DURATION)
    for path in (stale.sentinel, stale.manifest, stale.learner):
      _remove(path)

  def _prepare_restore(self, checkpoint_dir, iteration):
    """Reads and checks everything `_apply_restore` writes; changes nothing."""
    torch = _torch()
    files = _Files(checkpoint_dir, iteration)
    where = 'checkpoint {} in {}'.format(files.iteration, checkpoint_dir)
    if not os.path.exists(files.manifest):
      raise CheckpointError('{}: no manifest'.format(where))
    if not os.path.exists(files.sentinel):
      raise CheckpointError('{} is not complete: no {}'.format(
          where, os.path.basename(files.sentinel)))
    with open(files.manifest, 'rb') as f:
      manifest = json.loads(f.read().decode('utf-8'))
    mine = self._manifest()
    for key in ('format', 'kind', 'world_size', 'shard_capacity', 'global_batch',
                'update_horizon'):
      if manifest.get(key) != mine[key]:
        raise CheckpointError('{}: {} is {!r}, this learner has {!r}{}'.format(
            where, key, manifest.get(key), mine[key],
            ' (a restore onto another world size is not supported)'
            if key == 'world_size' else ''))
    for g in range(self.world):
      if not os.path.exists(files.rank_state(g)):
        raise CheckpointError('{}: rank {} is missing ({})'.format(
            where, g, files.rank_state(g)))
    with open(files.rank_state(self.rank), 'rb') as f:
      rank_state = json.loads(f.read().decode('utf-8'))
    if rank_state.get('rank') != self.rank or rank_state.get('world_size') != self.world:
      raise CheckpointError('{}: {} is not rank {} of {}'.format(
          where, files.rank_state(self.rank), self.rank, self.world))
    learner = torch.load(files.learner, map_location='cpu', weights_only=True)
    if _params_sha256(learner['online'], learner['target']) != manifest['params_sha256']:
      raise CheckpointError('{}: the saved parameters do not match the manifest\'s '
                            'checksum'.format(where))
    for name in ('online', 'target'):
      have = getattr(self, name).state_dict()
      saved = learner[name]
      if sorted(have) != sorted(saved) or any(
          tuple(have[k].shape) != tuple(saved[k].shape) for k in have):
        raise CheckpointError('{}: the {} network does not match this learner'.format(
            where, name))
    memory = self.memory._load_prepare(files.rank_dir(self.rank), files.iteration)  # pylint: disable=protected-access
    return {'memory': memory, 'rank_state': rank_state, 'learner': learner}

  def _apply_restore(self, prepared):
    """Writes what `_prepare_restore` read, in place, and waits for the copies."""
    self._flush_replay()
    self.memory._load_apply(prepared['memory'])  # pylint: disable=protected-access
    self._load_rank_state(prepared['rank_state'])
    self._load_learner_state(prepared['learner'])
    _torch().cuda.current_stream().synchronize()

  def restore(self, checkpoint_dir, iteration):
    """Restores checkpoint `iteration` written by learners of the same kind, world size,
    global batch and shard capacity.  Over torch.distributed every rank calls it: the
    ranks agree that every rank's checks passed before any rank writes, and none returns
    before every rank has restored.  A refused restore raises `CheckpointError` (or the
    replay's own error for a damaged shard file) and leaves learner, replay and exchange
    as they were.  Emulated ranks: `restore_ranks`."""
    prepared, error = None, None
    try:
      prepared = self._prepare_restore(checkpoint_dir, iteration)
    except Exception as e:  # pylint: disable=broad-except
      error = e
    if not self._agree(error is None):
      raise error or CheckpointError(
          'checkpoint {} in {}: another rank refused it'.format(iteration, checkpoint_dir))
    self._apply_restore(prepared)
    if self._dist is not None:  # no rank publishes into a mailbox not yet cleared
      self._dist.barrier(group=self._group)

  @staticmethod
  def save_ranks(learners, checkpoint_dir, iteration):
    """`save` of ranks emulated on one device: every rank's part, then the sentinel."""
    for learner in learners:
      learner.save(checkpoint_dir, iteration)
    learners[0].finish_save(checkpoint_dir, iteration)

  @staticmethod
  def restore_ranks(learners, checkpoint_dir, iteration):
    """`restore` of ranks emulated on one device: every rank's checks before any write."""
    prepared = [l._prepare_restore(checkpoint_dir, iteration) for l in learners]  # pylint: disable=protected-access
    for learner, p in zip(learners, prepared):
      learner._apply_restore(p)  # pylint: disable=protected-access
