"""What the learners share beyond their loss: the update replayed as one CUDA graph, and
the rank plumbing of a data-parallel learner on ONE global batch sharded over the ranks
(`agent.ShardedRainbowLearner`, `learner.ShardedIQNLearner`,
`learner.ShardedDQNLearner`)."""


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


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
