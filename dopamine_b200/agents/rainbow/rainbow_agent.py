"""Rainbow's C51 target / loss math as fused CUDA kernels.

Drop-in for the hot-path pieces of `dopamine/agents/rainbow/rainbow_agent.py`:
  * `project_distribution(supports, weights, target_support, validate_args)`
    (rainbow_agent.py:340-494) — same argument meaning and validation errors,
    over torch CUDA tensors (numpy arrays are accepted and round-tripped);
  * `build_target_distribution` / `c51_loss` — the n-step distributional Bellman
    target, projection, softmax cross-entropy, `sqrt(loss + 1e-10)` priorities
    and `1/sqrt(p + 1e-10) / max` importance weights of
    `_build_target_distribution` (rainbow_agent.py:200-251) and `_build_train_op`
    (rainbow_agent.py:253-305), in one launch (+ a one-CTA finalize);
  * `C51Loss` — the same as a differentiable torch op, so the conv Q-network
    (cuDNN through PyTorch, the only dense contraction on the path) trains on it.

  * `train_step` / `ReplayTrainer` — the whole replay-and-update step as one native
    call on device tensors, and as one pipelined host-facing call per update.

The learner that puts the conv network, Adam and the target sync around these
(`RainbowLearner`) lives in `dopamine_b200/agents/rainbow/agent.py`.
"""
import ctypes
import math

import numpy as np

from dopamine_b200 import _native


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def make_support(vmax, num_atoms, device='cuda'):
  """`tf.linspace(-vmax, vmax, num_atoms)` in f32 (rainbow_agent.py:124-126).

  TF-1.x evaluates `start + i * step` in f32 (SURVEY.md Q23).
  """
  torch = _torch()
  vmax = np.float32(float(vmax))
  if num_atoms == 1:
    host = np.array([-vmax], dtype=np.float32)
  else:
    step = (vmax - (-vmax)) / np.float32(num_atoms - 1)
    host = (-vmax + np.arange(num_atoms, dtype=np.float32) * step).astype(
        np.float32)
  return torch.as_tensor(host, device=device)


def _as_cuda_f32(x):
  torch = _torch()
  if isinstance(x, torch.Tensor):
    return x.to(device='cuda', dtype=torch.float32).contiguous(), False
  return torch.as_tensor(np.asarray(x, dtype=np.float32), device='cuda'), True


def project_distribution(supports, weights, target_support,
                         validate_args=False):
  """Projects a batch of (support, weights) onto target_support (Eq. 7 of C51).

  Args:
    supports: (batch_size, num_dims) supports of the source distributions.
    weights: (batch_size, num_dims) weights on those supports.
    target_support: (num_dims,) equally spaced, increasing target support.
    validate_args: also check monotonicity / equal spacing of target_support
      (a device->host read), as the reference's tf.Assert ops do.

  Returns:
    (batch_size, num_dims) projection; a CUDA tensor, or a numpy array if the
    inputs were numpy.

  Raises:
    ValueError: on incompatible shapes or an invalid target_support.
  """
  torch = _torch()
  supports, from_numpy = _as_cuda_f32(supports)
  weights, _ = _as_cuda_f32(weights)
  target_support, _ = _as_cuda_f32(target_support)
  if target_support.dim() == 0:
    raise ValueError('Index out of range: target_support has no dimensions')
  if target_support.dim() != 1:
    raise ValueError('target_support must have rank 1, index out of bounds '
                     'for rank {}'.format(target_support.dim()))
  if supports.dim() != 2 or tuple(supports.shape) != tuple(weights.shape):
    raise ValueError('Shapes {} and {} are incompatible'.format(
        tuple(supports.shape), tuple(weights.shape)))
  if supports.shape[1] != target_support.shape[0]:
    raise ValueError('Shapes {} and {} are incompatible'.format(
        tuple(supports.shape[1:]), tuple(target_support.shape)))
  if target_support.shape[0] < 2:
    raise ValueError('target_support needs at least two atoms')
  if validate_args:
    deltas = (target_support[1:] - target_support[:-1]).cpu()
    if not bool((deltas > 0).all()):
      raise ValueError('assertion failed: target_support must be increasing')
    if not bool((deltas == deltas[0]).all()):
      raise ValueError('assertion failed: target_support must be equally spaced')
  out = torch.empty_like(supports)
  _native.check(_native.lib().b2r_c51_project(
      supports.shape[0], supports.shape[1], supports.data_ptr(),
      weights.data_ptr(), target_support.data_ptr(), out.data_ptr(),
      _native.current_stream()))
  return out.cpu().numpy() if from_numpy else out


def c51_loss(online_logits, target_logits, actions, rewards, terminals,
             sampling_probabilities, support, cumulative_gamma,
             want_target=False, want_grad=False, want_mean=True, out=None,
             sharded=None):
  """Fused Rainbow update math for one batch, all on the device.

  Args:
    online_logits: (B, A, N) f32, online network on `state`.
    target_logits: (B, A, N) f32, target network on `next_state`.
    actions: (B,) int32; rewards: (B,) f32 n-step returns; terminals: (B,) uint8.
    sampling_probabilities: (B,) f32 raw priorities from the replay batch, or
      None for the 'uniform' replay scheme (rainbow_agent.py:273-295).
    support: (N,) f32 (see make_support); cumulative_gamma: gamma ** n.
  Returns:
    dict with 'loss' (B,), 'priorities' (B,) = sqrt(loss + 1e-10), 'weights'
    (B,), 'mean_weighted_loss' (scalar tensor) and optionally 'target' (B, N),
    'grad_logits' (B, A, N) = d mean_weighted_loss / d online_logits.
    `out` (a dict returned by an earlier call with the same shapes) is reused
    instead of allocating.
    sharded: (exchange, global_batch, count, min_probability) — the rows are one
    rank's share of a global batch of `global_batch` strata, as
    `ShardedPrioritizedReplay.sample_transition_batch_sharded` returns it
    (b2r_c51_loss_sharded): the first `count` (device) rows are valid, the weights are
    normalised over every rank's minimum sampling probability, and the mean and its
    gradient are this rank's part of the global batch's (divisor global_batch; padded
    rows get zero gradients).
  """
  torch = _torch()
  b, a, n = online_logits.shape
  assert tuple(target_logits.shape) == (b, a, n)
  assert online_logits.dtype == torch.float32 and online_logits.is_cuda
  assert target_logits.dtype == torch.float32 and target_logits.is_cuda
  assert actions.dtype == torch.int32 and rewards.dtype == torch.float32
  assert terminals.dtype == torch.uint8 and support.dtype == torch.float32
  online_logits = online_logits.contiguous()
  target_logits = target_logits.contiguous()
  dev = online_logits.device
  if out is None:
    out = {
        'loss': torch.empty(b, dtype=torch.float32, device=dev),
        'priorities': torch.empty(b, dtype=torch.float32, device=dev),
        'weights': torch.empty(b, dtype=torch.float32, device=dev),
    }
    if want_mean:
      out['mean_weighted_loss'] = torch.empty((), dtype=torch.float32, device=dev)
    if want_target:
      out['target'] = torch.empty(b, n, dtype=torch.float32, device=dev)
    if want_grad:
      out['grad_logits'] = torch.empty(b, a, n, dtype=torch.float32, device=dev)
  want_mean = 'mean_weighted_loss' in out
  want_target = 'target' in out
  want_grad = 'grad_logits' in out
  args = _native.C51Args()
  args.batch, args.num_actions, args.num_atoms = b, a, n
  args.cumulative_gamma = float(np.float32(cumulative_gamma))
  args.support = support.data_ptr()
  args.target_logits = target_logits.data_ptr()
  args.online_logits = online_logits.data_ptr()
  args.actions = actions.contiguous().data_ptr()
  args.rewards = rewards.contiguous().data_ptr()
  args.terminals = terminals.contiguous().data_ptr()
  args.sampling_probabilities = (
      sampling_probabilities.contiguous().data_ptr()
      if sampling_probabilities is not None else None)
  args.target = out['target'].data_ptr() if want_target else None
  args.loss = out['loss'].data_ptr()
  args.priorities = out['priorities'].data_ptr()
  args.weights = out['weights'].data_ptr()
  args.mean_weighted_loss = (out['mean_weighted_loss'].data_ptr()
                             if want_mean else None)
  args.grad_logits = out['grad_logits'].data_ptr() if want_grad else None
  if sharded is None:
    _native.check(_native.lib().b2r_c51_loss(ctypes.byref(args),
                                             _native.current_stream()))
    return out
  exchange, global_batch, count, min_probability = sharded
  args.batch_count = count.data_ptr()
  if sampling_probabilities is not None:
    args.min_probability = min_probability.data_ptr()
  _native.check(_native.lib().b2r_c51_loss_sharded(
      ctypes.byref(args), exchange._h, int(global_batch),  # pylint: disable=protected-access
      _native.current_stream()))
  return out


def build_target_distribution(rewards, terminals, target_logits, support,
                              cumulative_gamma):
  """The projected C51 target of `_build_target_distribution`
  (rainbow_agent.py:200-251) for a batch, given the target net's logits."""
  torch = _torch()
  b, a, _ = target_logits.shape
  zeros_i = torch.zeros(b, dtype=torch.int32, device=target_logits.device)
  out = c51_loss(target_logits, target_logits, zeros_i, rewards, terminals, None,
                 support, cumulative_gamma, want_target=True)
  del a
  return out['target']


def cumulative_gamma(gamma, update_horizon):
  """dqn_agent.py:175."""
  return math.pow(gamma, update_horizon)


class C51Loss(object):
  """Differentiable wrapper: `loss, aux = C51Loss.apply(online_logits, ...)`.

  Forward runs the fused kernel once (it also produces the gradient w.r.t. the
  online logits); backward scales that gradient by the upstream scalar.
  """

  _fn = None

  @classmethod
  def _function(cls):
    if cls._fn is None:
      torch = _torch()

      class _Fn(torch.autograd.Function):

        @staticmethod
        def forward(ctx, online_logits, target_logits, actions, rewards,
                    terminals, probs, support, gamma_n, sharded):
          out = c51_loss(online_logits.detach(), target_logits.detach(), actions,
                         rewards, terminals, probs, support, gamma_n,
                         want_grad=True, sharded=sharded)
          ctx.save_for_backward(out['grad_logits'])
          ctx.mark_non_differentiable(out['priorities'], out['loss'],
                                      out['weights'])
          return (out['mean_weighted_loss'], out['priorities'], out['loss'],
                  out['weights'])

        @staticmethod
        def backward(ctx, grad_mean, *unused):
          (grad_logits,) = ctx.saved_tensors
          return (grad_logits * grad_mean, None, None, None, None, None, None,
                  None, None)

      cls._fn = _Fn
    return cls._fn

  @classmethod
  def apply(cls, online_logits, target_logits, actions, rewards, terminals,
            sampling_probabilities, support, gamma_n):
    return cls._function().apply(online_logits, target_logits, actions, rewards,
                                 terminals, sampling_probabilities, support,
                                 gamma_n, None)


class ShardedC51Loss(C51Loss):
  """`C51Loss` over one rank's share of a sharded global batch (b2r_c51_loss_sharded):
  `mean, priorities, loss, weights = ShardedC51Loss.apply(..., sharded)` with `sharded`
  as in `c51_loss`.  `mean` is this rank's partial mean (its rows' weighted losses over
  the global batch size) and backward gives its gradient; summed over the ranks both
  are the global batch's."""

  @classmethod
  def apply(cls, online_logits, target_logits, actions, rewards, terminals,
            sampling_probabilities, support, gamma_n, sharded):
    return cls._function().apply(online_logits, target_logits, actions, rewards,
                                 terminals, sampling_probabilities, support,
                                 gamma_n, tuple(sharded))


# ---------------------------------------------------------------------------
# The whole hot path in one native call (include/b200_replay.h, "The whole hot
# path in one call"): what one sess.run of the train op does around the network.
# ---------------------------------------------------------------------------
def train_step(memory, online_logits, target_logits, support, cumulative_gamma,
               batch_size=None, out=None):
  """Prioritized sample -> C51 loss -> priority write-back in ONE native call.

  Equivalent to `memory.sample_transition_batch()` (device RNG), `c51_loss(...)`
  and `memory.set_priority(indices, priorities)`, but the sampler writes the
  scalar columns of the batch itself and the frame-stack copies run on a forked
  stream beside the loss and the write-back (they rejoin the current stream
  before this returns).

  NOTE — what this call is for.  The logits are INPUTS: row b of both tensors is paired
  with whatever transition the sampler draws for row b, so they cannot be the networks'
  outputs ON that transition (the reference runs the networks on the sampled batch,
  rainbow_agent.py:253-305).  This is the replay-and-update path of north_star measured
  without a network in the middle (bench.py's `value` / `e2e`, and the parity tests, which
  only need the arithmetic); priorities written by it are meaningful only if the caller's
  logits do not depend on the batch.  A learner uses the same kernels in the reference's
  order — `memory.sample_transition_batch()` -> networks -> `c51_loss` ->
  `memory.set_priority` — as `agent.RainbowLearner._update` does; bench.py reports that
  loop as `full_train_step`.

  Args:
    memory: OutOfGraphPrioritizedReplayBuffer (uint8 terminals, f32 rewards,
      scalar int32 actions).
    online_logits, target_logits: (B, A, N) f32 CUDA tensors.
    out: dict returned by an earlier call with the same shapes (reused).
  Returns:
    (transition tuple in get_transition_elements() order, dict with 'loss',
    'priorities', 'weights' (B,) CUDA tensors).
  """
  torch = _torch()
  b, a, n = online_logits.shape
  batch_size = b if batch_size is None else batch_size
  assert b == batch_size and tuple(target_logits.shape) == (b, a, n)
  assert online_logits.dtype == torch.float32 and online_logits.is_cuda
  assert target_logits.dtype == torch.float32 and target_logits.is_cuda
  _, arrays, batch = memory._alloc_outputs(batch_size, True)  # pylint: disable=protected-access
  if out is None:
    out = {k: torch.empty(b, dtype=torch.float32, device='cuda')
           for k in ('loss', 'priorities', 'weights')}
  args = _native.C51Args()
  args.batch, args.num_actions, args.num_atoms = b, a, n
  args.cumulative_gamma = float(np.float32(cumulative_gamma))
  args.support = support.data_ptr()
  args.target_logits = target_logits.contiguous().data_ptr()
  args.online_logits = online_logits.contiguous().data_ptr()
  args.loss = out['loss'].data_ptr()
  args.priorities = out['priorities'].data_ptr()
  args.weights = out['weights'].data_ptr()
  status = _native.lib().b2r_train_step_device(
      memory._h, batch_size, memory._seed, memory._next_offset(),  # pylint: disable=protected-access
      ctypes.byref(batch), ctypes.byref(args), _native.current_stream())
  if status == _native.ERR_UNSUPPORTED:
    raise NotImplementedError(_native.last_error())
  _native.check(status)
  return tuple(arrays), out


class _DeviceView(object):
  """A device buffer owned by the native library, for torch.as_tensor."""

  def __init__(self, pointer, shape, typestr):
    self.__cuda_array_interface__ = {
        'shape': tuple(shape), 'typestr': typestr, 'data': (int(pointer), False),
        'version': 2, 'strides': None}


class ReplayTrainer(object):
  """Pipelined host-facing training iteration (b2r_trainer_* in the C ABI).

  `step(online_logits, target_logits)` takes the two network outputs as HOST
  float32 arrays of shape (B, A, N) (page-locked memory keeps the copies
  asynchronous: do not overwrite it before the step has run), applies the staged
  `memory.add()`s, runs sample -> C51 loss -> priority write-back on the device and
  hands back the per-row losses of the step queued `pipeline_depth` calls earlier,
  so the host never waits for the step it has just queued.

  Like `train_step`, this takes the logits as inputs BEFORE the batch is sampled: it is
  the host-facing harness of the replay-and-update path (bench.py's `e2e`), not a
  learner — see the note in `train_step`; `agent.RainbowLearner` is the learner.
  """

  def __init__(self, memory, num_actions, num_atoms=51, vmax=10.,
               batch_size=None, pipeline_depth=2, seed=0, use_graph=False,
               logit_rows=None):
    self._memory = memory
    self._lib = _native.lib()
    cfg = _native.TrainerConfig()
    cfg.batch = memory._batch_size if batch_size is None else batch_size  # pylint: disable=protected-access
    cfg.num_actions, cfg.num_atoms = num_actions, num_atoms
    cfg.vmax = float(vmax)
    cfg.cumulative_gamma = float(np.float32(math.pow(
        memory._gamma, memory._update_horizon)))  # pylint: disable=protected-access
    cfg.seed = int(seed)
    cfg.pipeline_depth = int(pipeline_depth)
    cfg.use_graph = int(bool(use_graph))
    cfg.logit_rows = int(logit_rows or 0)
    self.logit_rows = int(logit_rows or cfg.batch)
    self.batch_size, self.num_actions, self.num_atoms = (
        cfg.batch, num_actions, num_atoms)
    handle = ctypes.c_void_p()
    status = self._lib.b2r_trainer_create(memory._h, ctypes.byref(cfg),  # pylint: disable=protected-access
                                          ctypes.byref(handle))
    if status == _native.ERR_UNSUPPORTED:
      raise NotImplementedError(_native.last_error())
    _native.check(status)
    self._h = handle
    self._loss = np.empty(self.logit_rows, dtype=np.float32)
    self._loss_ptr = self._loss.ctypes.data
    self._step = ctypes.c_int64(-1)
    self._step_ref = ctypes.byref(self._step)
    self._step_addr = ctypes.addressof(self._step)
    self._fast_step = _native.fast().trainer_step
    self._h_int = self._h.value

  def __del__(self):
    if getattr(self, '_h', None):
      self._lib.b2r_trainer_destroy(self._h)
      self._h = None

  def set_exchange(self, exchange):
    """Makes this the trainer of one shard of a sharded replay
    (`sharded_replay.PeerExchange`): `batch_size` becomes the GLOBAL batch, this
    rank's rows come first and `last_rows` counts them."""
    _native.check(self._lib.b2r_trainer_set_exchange(self._h, exchange._h))  # pylint: disable=protected-access
    self._exchange = exchange  # keep it alive

  @property
  def last_rows(self):
    """Rows of the step reported by the last step() / drain()."""
    return int(self._lib.b2r_trainer_last_rows(self._h))

  def step_pointers(self, online_ptr, target_ptr, stream=None):
    """As `step`, from raw host addresses (no per-call Python work)."""
    status = self._fast_step(
        self._h_int, online_ptr, target_ptr, self._loss_ptr, self._step_addr,
        _native.current_stream() if stream is None else stream)
    if status:
      _native.check(status)
    return self._step.value

  def step(self, online_logits, target_logits):
    """Queues one iteration; returns (losses or None, step number or -1)."""
    shape = (self.logit_rows, self.num_actions, self.num_atoms)
    pointers = []
    for x in (online_logits, target_logits):
      if hasattr(x, 'data_ptr'):  # torch CPU tensor (e.g. pinned)
        assert not x.is_cuda and tuple(x.shape) == shape and x.is_contiguous()
        pointers.append(x.data_ptr())
      else:
        assert x.dtype == np.float32 and x.shape == shape
        pointers.append(_native.ptr(x))
    done = self.step_pointers(pointers[0], pointers[1])
    return (self._loss.copy() if done >= 0 else None), done

  def drain(self):
    """Waits for every queued step; returns (losses of the last one, its number)."""
    _native.check(self._lib.b2r_trainer_drain(
        self._h, self._loss_ptr, self._step_ref, _native.current_stream()))
    done = self._step.value
    return (self._loss.copy() if done >= 0 else None), done

  def views(self):
    """The trainer's device buffers as torch tensors: (transition dict, loss dict)."""
    torch = _torch()
    batch, c51 = _native.Batch(), _native.C51Args()
    _native.check(self._lib.b2r_trainer_views(self._h, ctypes.byref(batch),
                                              ctypes.byref(c51)))
    mem, b = self._memory, self.logit_rows
    obs = tuple(mem._observation_shape) + (mem._stack_size,)  # pylint: disable=protected-access

    def view(pointer, shape, typestr):
      return torch.as_tensor(_DeviceView(pointer, shape, typestr), device='cuda')

    transition = {
        'state': view(batch.state, (b,) + obs, '|u1'),
        'action': view(batch.action, (b,), '<i4'),
        'reward': view(batch.reward, (b,), '<f4'),
        'next_state': view(batch.next_state, (b,) + obs, '|u1'),
        'next_action': view(batch.next_action, (b,), '<i4'),
        'next_reward': view(batch.next_reward, (b,), '<f4'),
        'terminal': view(batch.terminal, (b,), '|u1'),
        'indices': view(batch.indices, (b,), '<i4'),
        'sampling_probabilities': view(batch.sampling_probabilities, (b,), '<f4'),
    }
    losses = {
        'loss': view(c51.loss, (b,), '<f4'),
        'priorities': view(c51.priorities, (b,), '<f4'),
        'weights': view(c51.weights, (b,), '<f4'),
    }
    return transition, losses
