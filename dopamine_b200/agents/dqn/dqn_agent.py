"""DQN's target / loss math as a fused CUDA kernel.

Drop-in for the hot-path pieces of `dopamine/agents/dqn/dqn_agent.py`:
`_build_target_q_op` (dqn_agent.py:283-300) and the Huber loss of `_build_train_op`
(dqn_agent.py:302-322), over torch CUDA tensors, in one launch (+ a one-CTA
fixed-order mean).  The replay side is `OutOfGraphReplayBuffer` /
`WrappedReplayBuffer` of `dopamine_b200.replay_memory.circular_replay_buffer`
(uniform sampling, BASELINE config 1).

Also the actor side of the agent (SURVEY.md section 8f, row 3): the epsilon
schedules (dqn_agent.py:45-88), `ActorState` — `DQNAgent.state` kept in HBM, rolled
and refilled by one kernel per environment step (`_record_observation`,
dqn_agent.py:444-458) — and `ActingLoop`, the episode interface the reference's
runner drives (`begin_episode` / `step` / `end_episode` / `_select_action` /
`_train_step` / `bundle_and_checkpoint` / `unbundle`, dqn_agent.py:341-442, 480-560).
"""
import ctypes
import math
import os
import random

import numpy as np

from dopamine_b200 import _native


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def cumulative_gamma(gamma, update_horizon):
  """dqn_agent.py:175."""
  return math.pow(gamma, update_horizon)


def dqn_loss(online_q, target_q, actions, rewards, terminals, cumulative_gamma,  # pylint: disable=redefined-outer-name
             want_target=False, want_grad=False, want_mean=True, out=None, sharded=None):
  """Bellman target + Huber loss for one batch, on the device.

  Args:
    online_q: (B, A) f32 CUDA, online network on `state`.
    target_q: (B, A) f32 CUDA, target network on `next_state`.
    actions: (B,) int32; rewards: (B,) f32 n-step returns; terminals: (B,) uint8.
    cumulative_gamma: gamma ** update_horizon.
    sharded: (global_batch, count) — the B rows are one rank's share of a global batch
      of `global_batch` transitions, as `ShardedUniformReplay.sample_transition_batch_
      sharded` returns it (b2r_dqn_loss_sharded): the first `count` rows ((1,) int32
      CUDA tensor) are valid, the mean and its gradient are this rank's part of the
      global batch's (divisor global_batch), rows past the count get loss 0 and zero
      gradients.
  Returns:
    dict with 'loss' (B,), optionally 'mean_loss' (scalar), 'target' (B,),
    'grad_q' (B, A) = d mean(loss) / d online_q.
  """
  torch = _torch()
  b, a = online_q.shape
  assert tuple(target_q.shape) == (b, a)
  assert online_q.dtype == torch.float32 and online_q.is_cuda
  assert target_q.dtype == torch.float32 and target_q.is_cuda
  assert actions.dtype == torch.int32 and rewards.dtype == torch.float32
  assert terminals.dtype == torch.uint8
  if sharded is not None:
    global_batch, count = sharded
    if (not isinstance(count, torch.Tensor) or count.dtype != torch.int32 or
        not count.is_cuda or tuple(count.shape) != (1,)):
      raise ValueError('count must be a (1,) int32 CUDA tensor')
    if int(global_batch) < 1:
      raise ValueError('global_batch must be >= 1, got {}'.format(global_batch))
  dev = online_q.device
  if out is None:
    out = {'loss': torch.empty(b, dtype=torch.float32, device=dev)}
    if want_mean:
      out['mean_loss'] = torch.empty((), dtype=torch.float32, device=dev)
    if want_target:
      out['target'] = torch.empty(b, dtype=torch.float32, device=dev)
    if want_grad:
      out['grad_q'] = torch.empty(b, a, dtype=torch.float32, device=dev)
  # the contiguous copies of strided inputs live until the launch: a copy freed at once
  # goes back to torch's allocator, which hands its memory to the next input's copy
  keep = [target_q.contiguous(), online_q.contiguous(), actions.contiguous(),
          rewards.contiguous(), terminals.contiguous()]
  args = _native.DqnArgs()
  args.batch, args.num_actions = b, a
  args.cumulative_gamma = float(np.float32(cumulative_gamma))
  args.target_q = keep[0].data_ptr()
  args.online_q = keep[1].data_ptr()
  args.actions = keep[2].data_ptr()
  args.rewards = keep[3].data_ptr()
  args.terminals = keep[4].data_ptr()
  args.loss = out['loss'].data_ptr()
  args.target = out['target'].data_ptr() if 'target' in out else None
  args.mean_loss = out['mean_loss'].data_ptr() if 'mean_loss' in out else None
  args.grad_q = out['grad_q'].data_ptr() if 'grad_q' in out else None
  if sharded is None:
    _native.check(_native.lib().b2r_dqn_loss(ctypes.byref(args),
                                             _native.current_stream()))
    return out
  args.batch_count = count.data_ptr()
  _native.check(_native.lib().b2r_dqn_loss_sharded(ctypes.byref(args), int(global_batch),
                                                   _native.current_stream()))
  return out


class DQNLoss(object):
  """Differentiable wrapper: `mean_loss, loss = DQNLoss.apply(online_q, ...)`."""

  _fn = None

  @classmethod
  def _function(cls):
    if cls._fn is None:
      torch = _torch()

      class _Fn(torch.autograd.Function):

        @staticmethod
        def forward(ctx, online_q, target_q, actions, rewards, terminals, gamma_n,  # pylint: disable=redefined-outer-name
                    sharded):
          out = dqn_loss(online_q.detach(), target_q.detach(), actions, rewards,
                         terminals, gamma_n, want_grad=True, sharded=sharded)
          ctx.save_for_backward(out['grad_q'])
          ctx.mark_non_differentiable(out['loss'])
          return out['mean_loss'], out['loss']

        @staticmethod
        def backward(ctx, grad_mean, *unused):
          (grad_q,) = ctx.saved_tensors
          return (grad_q * grad_mean,) + (None,) * 6

      cls._fn = _Fn
    return cls._fn

  @classmethod
  def apply(cls, online_q, target_q, actions, rewards, terminals, gamma_n):
    return cls._function().apply(online_q, target_q, actions, rewards, terminals, gamma_n,
                                 None)


class ShardedDQNLoss(DQNLoss):
  """`DQNLoss` over one rank's share of a sharded global batch (b2r_dqn_loss_sharded):
  `mean, loss = ShardedDQNLoss.apply(..., gamma_n, sharded)` with `sharded` =
  (global_batch, count) as in `dqn_loss`.  `mean` is this rank's partial mean (its rows'
  losses over the global batch size) and backward gives its gradient; summed over the
  ranks both are the global batch's."""

  @classmethod
  def apply(cls, online_q, target_q, actions, rewards, terminals, gamma_n, sharded):  # pylint: disable=arguments-differ
    return cls._function().apply(online_q, target_q, actions, rewards, terminals, gamma_n,
                                 tuple(sharded))


# ------------------------------------------------------------- actor side ----
def linearly_decaying_epsilon(decay_period, step, warmup_steps, epsilon):
  """The Nature-DQN schedule of dqn_agent.py:45-67: 1.0 until `warmup_steps`, a straight
  line down to `epsilon` over the next `decay_period` steps, `epsilon` from then on
  (same operation order as the reference, so the same doubles)."""
  remaining = decay_period + warmup_steps - step
  extra = (1.0 - epsilon) * remaining / decay_period
  return epsilon + min(max(extra, 0.), 1. - epsilon)


def identity_epsilon(unused_decay_period, unused_step, unused_warmup_steps, epsilon):
  """dqn_agent.py:70-88."""
  return epsilon


class ActorState(object):
  """`DQNAgent.state` (dqn_agent.py:181-184): the (1,) + observation_shape +
  (stack_size,) frame stack the online network acts on, as a CUDA tensor.

  `record(observation)` is `_record_observation` (dqn_agent.py:444-458) and
  `reset()` is `_reset_state` (dqn_agent.py:474-476); both are one launch of
  `b2r_actor_record` / `b2r_actor_reset` (csrc/actor.cu), the observation going
  through a pinned slot that the kernel reads in place."""

  def __init__(self, observation_shape, stack_size, observation_dtype=np.uint8,
               slots=4):
    from dopamine_b200.replay_memory import circular_replay_buffer  # pylint: disable=g-import-not-at-top
    torch = _torch()
    self.observation_shape = tuple(observation_shape)
    self.stack_size = int(stack_size)
    self.observation_dtype = np.dtype(observation_dtype)
    self.tensor = torch.zeros(
        (1,) + self.observation_shape + (self.stack_size,),
        dtype=circular_replay_buffer._torch_dtype(self.observation_dtype),  # pylint: disable=protected-access
        device='cuda')
    self._lib = _native.lib()
    self._h = ctypes.c_void_p()
    pixels = int(np.prod(self.observation_shape, dtype=np.int64))
    _native.check(self._lib.b2r_actor_create(
        pixels, self.observation_dtype.itemsize, self.stack_size, slots,
        ctypes.byref(self._h)))

  def reset(self):
    _native.check(self._lib.b2r_actor_reset(self._h, self.tensor.data_ptr(),
                                            _native.current_stream()))

  def record(self, observation):
    """Rolls the stack and appends `observation`; returns the frame as stored
    (`DQNAgent._observation`: reshaped to observation_shape, cast by assignment)."""
    frame = np.ascontiguousarray(
        np.reshape(observation, self.observation_shape).astype(
            self.observation_dtype, copy=False))
    _native.check(self._lib.b2r_actor_record(
        self._h, self.tensor.data_ptr(), frame.ctypes.data,
        _native.current_stream()))
    return frame

  def numpy(self):
    return self.tensor.cpu().numpy()

  def close(self):
    if getattr(self, '_h', None) is not None and self._h:
      self._lib.b2r_actor_destroy(self._h)
      self._h = None

  def __del__(self):
    try:
      self.close()
    except Exception:  # pylint: disable=broad-except
      pass


class ActingLoop(object):
  """The episode interface of `DQNAgent` (dqn_agent.py:341-442, 480-560) for a
  learner that provides `num_actions`, `memory` (the replay buffer), `q_values(state)`,
  `train_step()`, `sync_target()` and `_store_transition(...)`.

  Same attribute names and the same order of effects as the reference: `state`
  (here a CUDA tensor), `_observation`, `_last_observation`, `action`, `eval_mode`,
  `training_steps`.  Random numbers come from Python's `random` module exactly as in
  `_select_action` (dqn_agent.py:397-416), so a seeded run picks the same exploratory
  actions."""

  def _init_acting(self, observation_shape, stack_size, observation_dtype=np.uint8,
                   min_replay_history=20000, update_period=4,
                   target_update_period=8000,
                   epsilon_fn=linearly_decaying_epsilon, epsilon_train=0.01,
                   epsilon_eval=0.001, epsilon_decay_period=250000,
                   allow_partial_reload=False):
    self.observation_shape = tuple(observation_shape)
    self.stack_size = stack_size
    self.min_replay_history = min_replay_history
    self.update_period = update_period
    self.target_update_period = target_update_period
    self.epsilon_fn = epsilon_fn
    self.epsilon_train = epsilon_train
    self.epsilon_eval = epsilon_eval
    self.epsilon_decay_period = epsilon_decay_period
    self.allow_partial_reload = allow_partial_reload
    self.eval_mode = False
    self.training_steps = 0
    self.action = None
    self._observation = None
    self._last_observation = None
    self._actor_state = self._make_actor_state(observation_shape, stack_size,
                                               observation_dtype)

  def _make_actor_state(self, observation_shape, stack_size, observation_dtype):
    return ActorState(observation_shape, stack_size, observation_dtype)

  @property
  def state(self):
    return self._actor_state.tensor

  def begin_episode(self, observation):
    """dqn_agent.py:341-358: clear the stack, then the common tail without a
    transition to store."""
    self._reset_state()
    return self._observe_and_act(observation, finished=None)

  def step(self, reward, observation):
    """dqn_agent.py:360-381: the observation before this one is stored together with
    the reward it earned."""
    self._last_observation = self._observation
    return self._observe_and_act(observation, finished=(self._last_observation, reward))

  def _observe_and_act(self, observation, finished):
    """What begin_episode and step share, in the reference's order: record the frame;
    in training mode store the finished (observation, action, reward) and run the
    train-step cadence; pick the next action."""
    self._record_observation(observation)
    if not self.eval_mode:
      if finished is not None:
        self._store_transition(finished[0], self.action, finished[1], False)
      self._train_step()
    self.action = self._select_action()
    return self.action

  def end_episode(self, reward):
    """dqn_agent.py:383-393: the episode's last observation closes it."""
    if not self.eval_mode:
      self._store_transition(self._observation, self.action, reward, True)

  def _select_action(self):
    """dqn_agent.py:395-416."""
    if self.eval_mode:
      epsilon = self.epsilon_eval
    else:
      epsilon = self.epsilon_fn(self.epsilon_decay_period, self.training_steps,
                                self.min_replay_history, self.epsilon_train)
    if random.random() <= epsilon:
      return random.randint(0, self.num_actions - 1)
    return int(self.q_values(self.state).argmax(dim=1)[0])

  def _train_step(self):
    """dqn_agent.py:418-442."""
    if self.memory.add_count > self.min_replay_history:
      if self.training_steps % self.update_period == 0:
        self.train_step()
      if self.training_steps % self.target_update_period == 0:
        self.sync_target()
    self.training_steps += 1

  def _record_observation(self, observation):
    """dqn_agent.py:444-458."""
    self._observation = self._actor_state.record(observation)

  def _reset_state(self):
    """dqn_agent.py:474-476."""
    self._actor_state.reset()

  def _store_transition(self, last_observation, action, reward, is_terminal):
    """dqn_agent.py:460-472."""
    self.memory.add(last_observation, action, reward, is_terminal)

  # -- checkpointing (dqn_agent.py:480-560) ------------------------------------------
  def _network_state(self):
    """What the reference's tf.train.Saver holds: every variable of the graph."""
    return {'online': self.online.state_dict(), 'target': self.target.state_dict(),
            'optimizer': self.optimizer.state_dict()}

  def _load_network_state(self, blob):
    self.online.load_state_dict(blob['online'])
    self.target.load_state_dict(blob['target'])
    self.optimizer.load_state_dict(blob['optimizer'])

  def bundle_and_checkpoint(self, checkpoint_dir, iteration_number):
    if not os.path.exists(checkpoint_dir):
      return None
    torch = _torch()
    torch.save(self._network_state(),
               os.path.join(checkpoint_dir, 'torch_ckpt-{}'.format(iteration_number)))
    self.memory.save(checkpoint_dir, iteration_number)
    return {'state': self._actor_state.numpy(), 'training_steps': self.training_steps}

  def unbundle(self, checkpoint_dir, iteration_number, bundle_dictionary):
    torch = _torch()
    try:
      self.memory.load(checkpoint_dir, iteration_number)
    except (IOError, OSError):  # the reference catches tf.errors.NotFoundError
      if not self.allow_partial_reload:
        return False
    if bundle_dictionary is not None:
      if 'state' in bundle_dictionary:
        self.state.copy_(torch.as_tensor(np.asarray(bundle_dictionary['state'])))
      for key in self.__dict__:
        if key in bundle_dictionary and key != 'state':
          self.__dict__[key] = bundle_dictionary[key]
    elif not self.allow_partial_reload:
      return False
    self._load_network_state(torch.load(
        os.path.join(checkpoint_dir, 'torch_ckpt-{}'.format(iteration_number))))
    return True
