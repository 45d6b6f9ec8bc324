"""The learner half of the Rainbow agent on top of the B200 replay path.

Mirrors what `RainbowAgent` builds around the replay memory
(dopamine/agents/rainbow/rainbow_agent.py:93-337 on dqn_agent.py:341-442): the
convolutional distribution network (atari_lib.py:108-144, cuDNN through PyTorch —
the only dense contraction on the path, so the only part that is NOT a hand-written
kernel here), the C51 train op, Adam with the reference's hyper-parameters
(rainbow.gin:21-25), priority write-back and the target-network sync.
`RainbowLearner` is that half alone (the caller feeds `store_transition` exactly as
the reference's `_store_transition` feeds `add`); `RainbowAgent` adds the episode
interface the reference's runner drives (`dqn_agent.ActingLoop`: epsilon-greedy
acting on a frame stack kept in HBM, the `_train_step` cadence, checkpoint bundles).

One `train_step()`:
  sample + gather (one fused call, batch stays in HBM) -> online net on `state`,
  target net on `next_state` -> fused C51 loss kernel (also yields d loss / d logits)
  -> backward + Adam -> batched priority write-back.
With `ddp=True` every rank owns its own replay shard and the gradients are averaged
by torch DistributedDataParallel over NCCL (SURVEY.md section 8e, config 5).
"""
import math

import numpy as np

from dopamine_b200.agents import sharded_learner
from dopamine_b200.agents.dqn import dqn_agent
from dopamine_b200.agents.rainbow import rainbow_agent
from dopamine_b200.replay_memory import prioritized_replay_buffer
from dopamine_b200.replay_memory import sharded_replay


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def _same_pad(size, kernel, stride):
  """TensorFlow 'SAME' padding (before, after) for one spatial dimension."""
  out = -(-size // stride)
  total = max((out - 1) * stride + kernel - size, 0)
  return total // 2, total - total // 2


def network_input(state, half=False):
  """uint8 (B, H, W, stack) CUDA frame stacks -> (B, stack, H, W) float32 (or float16)
  planes of value / 255: the reference's `tf.cast(state, tf.float32)`, `tf.div(net,
  255.)` (atari_lib.py:124-125) and the layout of the first cuDNN convolution in ONE
  hand-written pass (b2r_stack_to_planes_device) instead of permute + cast + division."""
  torch = _torch()
  from dopamine_b200 import _native  # pylint: disable=g-import-not-at-top
  assert state.is_cuda and state.dtype == torch.uint8 and state.dim() == 4
  state = state.contiguous()
  b, h, w, stack = state.shape
  out = torch.empty((b, stack, h, w), device=state.device,
                    dtype=torch.float16 if half else torch.float32)
  _native.check(_native.lib().b2r_stack_to_planes_device(
      state.data_ptr(), out.data_ptr(), b, h * w, stack, int(bool(half)),
      _native.current_stream()))
  return out


def make_rainbow_network(num_actions, num_atoms, observation_shape=(84, 84),
                         stack_size=4):
  """atari_lib.rainbow_network (atari_lib.py:108-144): uint8 (B, H, W, stack) in,
  (B, num_actions, num_atoms) logits out; conv 32x8x8/4, 64x4x4/2, 64x3x3/1 with
  SAME padding, FC 512, FC A*N; uniform variance-scaling init, factor 1/sqrt(3),
  fan-in (atari_lib.py:122-123)."""
  torch = _torch()
  nn = torch.nn

  class RainbowNetwork(nn.Module):

    def __init__(self):
      super().__init__()
      h, w = observation_shape
      specs = [(stack_size, 32, 8, 4), (32, 64, 4, 2), (64, 64, 3, 1)]
      self.convs = nn.ModuleList()
      self.pads = []
      for cin, cout, k, s in specs:
        ph, pw = _same_pad(h, k, s), _same_pad(w, k, s)
        self.pads.append((pw[0], pw[1], ph[0], ph[1]))
        self.convs.append(nn.Conv2d(cin, cout, k, stride=s))
        h, w = -(-h // s), -(-w // s)
      self.fc1 = nn.Linear(h * w * 64, 512)
      self.fc2 = nn.Linear(512, num_actions * num_atoms)
      for m in list(self.convs) + [self.fc1, self.fc2]:
        fan_in = m.weight[0].numel()
        # variance_scaling_initializer(factor, 'FAN_IN', uniform=True):
        # limit = sqrt(3 * factor / fan_in)
        limit = math.sqrt(3.0 * (1.0 / math.sqrt(3.0)) / fan_in)
        nn.init.uniform_(m.weight, -limit, limit)
        nn.init.zeros_(m.bias)

    def forward(self, state):
      x = network_input(state)  # atari_lib.py:124-125 (cast, / 255) + NCHW, one kernel
      for pad, conv in zip(self.pads, self.convs):
        x = torch.relu(conv(torch.nn.functional.pad(x, pad)))
      # slim.flatten works on NHWC; keep that ordering of the 7 744 features
      x = x.permute(0, 2, 3, 1).flatten(1)
      x = torch.relu(self.fc1(x))
      return self.fc2(x).view(-1, num_actions, num_atoms)

  return RainbowNetwork()


def make_tf_adam(params, lr, beta1=0.9, beta2=0.999, epsilon=1e-8, capturable=False):
  """tf.train.AdamOptimizer as the reference configures it (rainbow_agent.py:69-71,
  rainbow.gin:21-25: learning_rate 6.25e-5, epsilon 1.5e-4).

  TensorFlow 1.x applies   lr_t = lr * sqrt(1 - beta2^t) / (1 - beta1^t),
                           theta -= lr_t * m_t / (sqrt(v_t) + epsilon)
  — its `epsilon` is the "epsilon hat" of Kingma & Ba, added to the UNcorrected sqrt(v_t).
  torch.optim.Adam adds eps to the bias-corrected sqrt(v_t / (1 - beta2^t)) instead, which
  with Rainbow's large epsilon makes the first thousands of updates up to 30x larger
  (t = 1: sqrt(1 - beta2) = 0.032).  This optimizer implements TensorFlow's form with
  multi-tensor (`_foreach`) ops; with `capturable` the step count lives on the device so
  that the update can be captured in a CUDA graph, otherwise lr_t is a host float."""
  torch = _torch()

  class TFAdam(torch.optim.Optimizer):

    def __init__(self):
      super().__init__(list(params), dict(lr=lr, beta1=beta1, beta2=beta2,
                                          epsilon=epsilon))
      self._t = None
      self._host_t = 0

    @torch.no_grad()
    def step(self, closure=None):
      assert closure is None
      for group in self.param_groups:
        ps = [p for p in group['params'] if p.grad is not None]
        if not ps:
          continue
        grads = [p.grad for p in ps]
        ms, vs = [], []
        for p in ps:
          state = self.state[p]
          if not state:
            state['m'] = torch.zeros_like(p)
            state['v'] = torch.zeros_like(p)
          ms.append(state['m'])
          vs.append(state['v'])
        b1, b2 = group['beta1'], group['beta2']
        if capturable:
          if self._t is None:
            self._t = torch.zeros((), dtype=torch.float64, device=ps[0].device)
          self._t += 1
          # lr_t in float64 on the device, applied as a float32 scalar tensor
          lr_t = (group['lr'] * torch.sqrt(1.0 - b2 ** self._t) /
                  (1.0 - b1 ** self._t)).to(torch.float32)
        else:
          self._host_t += 1
          lr_t = float(np.float32(group['lr'] * math.sqrt(1.0 - b2 ** self._host_t) /
                                  (1.0 - b1 ** self._host_t)))
        torch._foreach_mul_(ms, b1)
        torch._foreach_add_(ms, grads, alpha=1.0 - b1)
        torch._foreach_mul_(vs, b2)
        torch._foreach_addcmul_(vs, grads, grads, value=1.0 - b2)
        denom = torch._foreach_sqrt(vs)
        torch._foreach_add_(denom, group['epsilon'])
        update = torch._foreach_div(ms, denom)
        torch._foreach_mul_(update, lr_t)
        torch._foreach_sub_(ps, update)
      return None

    def state_dict(self):
      """Also holds the step count t, as TensorFlow saves beta1_power / beta2_power."""
      out = super().state_dict()
      out['step'] = int(self._t.item()) if capturable and self._t is not None else (
          self._host_t)
      return out

    def load_state_dict(self, state_dict):
      """In place (sharded_learner.load_optimizer_state), the step count included: a
      captured update keeps reading the same moments and device step count."""
      state_dict = dict(state_dict)
      step = state_dict.pop('step', None)
      sharded_learner.load_optimizer_state(self, state_dict)
      if step is None:  # a bundle written before the step count was saved
        return
      self._host_t = int(step)
      if capturable:
        if self._t is None:
          self._t = torch.zeros((), dtype=torch.float64,
                                device=self.param_groups[0]['params'][0].device)
        self._t.fill_(float(step))

  return TFAdam()


class RainbowLearner(sharded_learner.GraphedUpdate):
  """Replay + train op of RainbowAgent (rainbow_agent.py:93-337)."""

  def __init__(self, num_actions, observation_shape=(84, 84), stack_size=4,
               num_atoms=51, vmax=10., gamma=0.99, update_horizon=3,
               replay_capacity=1000000, batch_size=32, target_update_period=8000,
               update_period=4, replay_scheme='prioritized', learning_rate=6.25e-5,
               adam_epsilon=1.5e-4, seed=0, ddp=False, memory=None,
               cuda_graph=False):
    torch = _torch()
    if replay_scheme not in ('prioritized', 'uniform'):
      raise ValueError('Invalid replay scheme: {}'.format(replay_scheme))
    self.num_actions, self.num_atoms = num_actions, num_atoms
    self.batch_size = batch_size
    self.replay_scheme = replay_scheme
    self.update_period = update_period
    self.target_update_period = target_update_period
    # rainbow_agent.py:188-198: the prioritized buffer is used for both schemes.
    self.memory = memory or prioritized_replay_buffer.OutOfGraphPrioritizedReplayBuffer(
        observation_shape, stack_size, replay_capacity, batch_size,
        update_horizon=update_horizon, gamma=gamma, output='torch', rng='device',
        seed=seed, reuse_outputs=True)
    self.support = rainbow_agent.make_support(vmax, num_atoms)
    self.cumulative_gamma = math.pow(gamma, update_horizon)  # dqn_agent.py:175
    torch.manual_seed(seed)
    self.online = make_rainbow_network(num_actions, num_atoms, observation_shape,
                                       stack_size).cuda()
    self.target = make_rainbow_network(num_actions, num_atoms, observation_shape,
                                       stack_size).cuda()
    self.target.load_state_dict(self.online.state_dict())
    for p in self.target.parameters():
      p.requires_grad_(False)
    self._net = self.online
    if ddp:
      from torch.nn.parallel import DistributedDataParallel  # pylint: disable=g-import-not-at-top
      self._net = DistributedDataParallel(
          self.online, device_ids=[torch.cuda.current_device()])
    # cuda_graph: the whole update (replay kernels, both networks, backward, Adam,
    # write-back) is captured once and replayed: one launch per update instead of
    # ~150 eager ones.  Staged adds are flushed before every replay; the sampler's
    # validity context and draw counter live on the device, so the replayed graph
    # sees new transitions and draws fresh strata.
    if cuda_graph and ddp:
      raise NotImplementedError('cuda_graph is not combined with ddp')
    self._cuda_graph = bool(cuda_graph)
    self._graph = None
    self._static_loss = None
    self.optimizer = make_tf_adam(self.online.parameters(), lr=learning_rate,
                                  epsilon=adam_epsilon,  # rainbow.gin:21-25
                                  capturable=self._cuda_graph)
    self.training_steps = 0
    self.updates = 0

  # -- the add side (rainbow_agent.py:307-337) -------------------------------------
  def store_transition(self, last_observation, action, reward, is_terminal,
                       priority=None):
    if priority is None:
      priority = (1. if self.replay_scheme == 'uniform' else
                  prioritized_replay_buffer.MAX_RECORDED_PRIORITY)
    self.memory.add(last_observation, action, reward, is_terminal, priority)

  def q_values(self, state):
    """(B, A) expected values of the online network (atari_lib.py:141-143)."""
    torch = _torch()
    with torch.no_grad():
      probs = torch.softmax(self.online(state), dim=2)
      return (probs * self.support).sum(dim=2)

  # -- the train op (rainbow_agent.py:253-305); train_step() is GraphedUpdate's ------
  def _update(self):
    torch = _torch()
    batch = self.memory.sample_transition_batch(self.batch_size)
    (state, action, reward, next_state, _, _, terminal, indices, probs) = batch[:9]
    with torch.no_grad():
      target_logits = self.target(next_state)
    online_logits = self._net(state)
    scheme_probs = probs if self.replay_scheme == 'prioritized' else None
    loss, priorities, _, _ = rainbow_agent.C51Loss.apply(
        online_logits, target_logits, action, reward, terminal, scheme_probs,
        self.support, self.cumulative_gamma)
    self.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    self.optimizer.step()
    if self.replay_scheme == 'prioritized':  # rainbow_agent.py:289-295
      self.memory.set_priority(indices, priorities)
    if not self._cuda_graph or self._graph is None:
      self.updates += 1
    return loss

  def sync_target(self):
    self.target.load_state_dict(self.online.state_dict())

  def step_cadence(self):
    """dqn_agent.py:418-442: called once per environment step by the acting loop;
    trains every `update_period` steps and syncs the target network every
    `target_update_period` steps."""
    loss = None
    if self.training_steps % self.update_period == 0:
      loss = self.train_step()
    if self.training_steps % self.target_update_period == 0:
      self.sync_target()
    self.training_steps += 1
    return loss


class RainbowAgent(RainbowLearner, dqn_agent.ActingLoop):
  """`RainbowAgent` (rainbow_agent.py:50-337) as the reference's runner sees it:
  `begin_episode(observation)`, `step(reward, observation)`, `end_episode(reward)`,
  `eval_mode`, `bundle_and_checkpoint`, `unbundle`.  Constructor arguments keep the
  reference's names and defaults (rainbow_agent.py:53-87); `sess`, `tf_device`,
  `use_staging`, `optimizer` and the summary arguments have no meaning here."""

  def __init__(self, sess=None, num_actions=None, observation_shape=(84, 84),
               observation_dtype=np.uint8, stack_size=4, num_atoms=51, vmax=10.,
               gamma=0.99, update_horizon=1, min_replay_history=20000,
               update_period=4, target_update_period=8000,
               epsilon_fn=dqn_agent.linearly_decaying_epsilon, epsilon_train=0.01,
               epsilon_eval=0.001, epsilon_decay_period=250000,
               replay_scheme='prioritized', replay_capacity=1000000, batch_size=32,
               learning_rate=6.25e-5, adam_epsilon=1.5e-4, seed=0,
               allow_partial_reload=False, memory=None, cuda_graph=False):
    del sess
    if num_actions is None:
      raise ValueError('num_actions is required')
    if np.dtype(observation_dtype) != np.uint8:
      raise NotImplementedError('the convolutional network takes uint8 frames')
    RainbowLearner.__init__(
        self, num_actions, observation_shape=observation_shape,
        stack_size=stack_size, num_atoms=num_atoms, vmax=vmax, gamma=gamma,
        update_horizon=update_horizon, replay_capacity=replay_capacity,
        batch_size=batch_size, target_update_period=target_update_period,
        update_period=update_period, replay_scheme=replay_scheme,
        learning_rate=learning_rate, adam_epsilon=adam_epsilon, seed=seed,
        memory=memory, cuda_graph=cuda_graph)
    self._init_acting(observation_shape, stack_size, observation_dtype,
                      min_replay_history=min_replay_history,
                      update_period=update_period,
                      target_update_period=target_update_period,
                      epsilon_fn=epsilon_fn, epsilon_train=epsilon_train,
                      epsilon_eval=epsilon_eval,
                      epsilon_decay_period=epsilon_decay_period,
                      allow_partial_reload=allow_partial_reload)

  def _store_transition(self, last_observation, action, reward, is_terminal,
                        priority=None):
    """rainbow_agent.py:307-337 (the default priority of the prioritized scheme,
    "the maximum ever seen", is resolved on the device when the row is applied)."""
    if not self.eval_mode:
      self.store_transition(last_observation, action, reward, is_terminal, priority)


class ShardedRainbowLearner(sharded_learner.ShardedLearner, RainbowLearner):
  """`RainbowLearner` on ONE global prioritized batch sharded over the ranks of
  torch.distributed (SURVEY.md section 8(d), config 5 fed by config 4's sampler).

  Every rank owns one replay shard of `replay_capacity` transitions and a peer-memory
  exchange.  `batch_size` is the GLOBAL batch: its strata are apportioned over the
  shards by their priority totals (`ShardedPrioritizedReplay`), so the update is the
  reference's update (rainbow_agent.py:253-305) on that global batch, up to the order of
  floating-point sums.  One update:
    1. `sample()`: sharded sampler + frame copies into `max_rows` rows (default
       `share_bound`; the rank's share is counted on the device);
    2. `loss_backward()`: both networks on all `max_rows` rows, the sharded C51 loss
       (IS weights normalised over every rank's minimum, mean over the global batch,
       zero gradients for padded rows) and backward into one flat buffer;
    3. `reduce()`: ONE all-reduce (sum) of that buffer — every parameter's gradient
       and, appended, the partial loss, so the reported loss is the global mean;
    4. `apply()`: TF-form Adam and the counted priority write-back.
  The shapes are static, so `cuda_graph=True` captures the whole update, all-reduce
  included.  Errors latched on the device (a share beyond `max_rows`, a peer that did not
  answer) are raised by `check()`, which `sync_target()` calls.  Pass `exchange`
  (`PeerExchange.emulated`) to run the phases of several ranks on one device without
  torch.distributed (tests); `reduce()` then is the caller's.  The rank plumbing is
  `sharded_learner.ShardedLearner`'s.
  """

  def __init__(self, num_actions, batch_size=32, max_rows=None, exchange=None,
               group=None, exchange_timeout_s=2.0, ddp=False, **kwargs):
    exchange = self._connect(exchange, group, exchange_timeout_s, ddp)
    RainbowLearner.__init__(self, num_actions, batch_size=batch_size, **kwargs)
    self._shard(exchange, max_rows, kwargs.get('seed', 0),
                sharded_replay.ShardedPrioritizedReplay)

  # -- phases (sample, reduce: ShardedLearner's) ----------------------------------------
  def loss_backward(self):
    """Networks, sharded loss and backward: the flat buffer holds this rank's partial
    gradients and partial mean.  Returns the per-row priorities."""
    torch = _torch()
    _, count, batch, min_probability = self._sample
    (state, action, reward, next_state, _, _, terminal, _, probs) = batch[:9]
    with torch.no_grad():
      target_logits = self.target(next_state)
    online_logits = self.online(state)
    scheme_probs = probs if self.replay_scheme == 'prioritized' else None
    mean, priorities, _, _ = rainbow_agent.ShardedC51Loss.apply(
        online_logits, target_logits, action, reward, terminal, scheme_probs,
        self.support, self.cumulative_gamma,
        (self.exchange, self.batch_size, count, min_probability))
    self._flat.zero_()
    mean.backward()  # (accumulates into the views of the flat buffer)
    self.loss.copy_(mean.detach().view(1))
    return priorities

  def apply(self, priorities):
    """Adam on the reduced gradients, then this rank's priority write-back."""
    self.optimizer.step()
    if self.replay_scheme == 'prioritized':  # rainbow_agent.py:289-295
      slots, count, batch, _ = self._sample
      del slots
      self.sharded.set_priority(batch[7], priorities, count)

  def _update(self):
    self.sample()
    priorities = self.loss_backward()
    self.reduce()
    self.apply(priorities)
    if not self._cuda_graph or self._graph is None:
      self.updates += 1
    return self.loss
