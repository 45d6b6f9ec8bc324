"""The learner half of DQNAgent on top of the B200 replay path.

What `DQNAgent` builds around its replay memory (dopamine/agents/dqn/dqn_agent.py:237-322,
defaults of :79-108 and dqn.gin): the Nature DQN network (atari_lib.py:85-105, cuDNN
through PyTorch behind the hand-written input kernel), the uniform replay buffer, the
Bellman target + Huber loss as ONE kernel (`dqn_loss`, csrc/dqn.cu), TensorFlow's centred
RMSProp with the reference's numbers, and the target sync.  Same structure as
`agents/rainbow/agent.RainbowLearner`; the acting side is `dqn_agent.ActingLoop`, and
`DQNAgent` joins the two as the reference's runner creates it for dqn.gin.
`ShardedDQNLearner` trains on one global uniform batch drawn over the GPUs' replay shards.
"""
import math

import numpy as np

from dopamine_b200.agents import sharded_learner
from dopamine_b200.agents.dqn import dqn_agent
from dopamine_b200.agents.rainbow import agent as conv
from dopamine_b200.replay_memory import circular_replay_buffer
from dopamine_b200.replay_memory import sharded_replay


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def xavier_uniform_(torch, module):
  """tf.contrib.slim's default weights_initializer, xavier_initializer(uniform=True) =
  variance_scaling(factor 1, FAN_AVG, uniform): limit sqrt(6 / (fan_in + fan_out));
  biases zero (slim's default biases_initializer)."""
  w = module.weight
  receptive = w[0][0].numel() if w.dim() > 2 else 1
  fan_in, fan_out = w.shape[1] * receptive, w.shape[0] * receptive
  limit = math.sqrt(6.0 / (fan_in + fan_out))
  torch.nn.init.uniform_(w, -limit, limit)
  torch.nn.init.zeros_(module.bias)


def conv_trunk(torch, observation_shape, stack_size, init):
  """The three SAME-padded convolutions every Atari network of the reference starts
  with (32x8x8/4, 64x4x4/2, 64x3x3/1; atari_lib.py:97-99, 126-131, 169-174).  Returns
  (module list, pads, flattened feature size)."""
  nn = torch.nn
  h, w = observation_shape
  convs, pads = nn.ModuleList(), []
  for cin, cout, k, s in [(stack_size, 32, 8, 4), (32, 64, 4, 2), (64, 64, 3, 1)]:
    ph, pw = conv._same_pad(h, k, s), conv._same_pad(w, k, s)  # pylint: disable=protected-access
    pads.append((pw[0], pw[1], ph[0], ph[1]))
    layer = nn.Conv2d(cin, cout, k, stride=s)
    init(torch, layer)
    convs.append(layer)
    h, w = -(-h // s), -(-w // s)
  return convs, pads, h * w * 64


def run_trunk(torch, convs, pads, state):
  """uint8 (B, H, W, stack) -> (B, features) in slim.flatten's NHWC order."""
  x = conv.network_input(state)  # atari_lib.py:95-96: cast, / 255 (+ NCHW), one kernel
  for pad, layer in zip(pads, convs):
    x = torch.relu(layer(torch.nn.functional.pad(x, pad)))
  return x.permute(0, 2, 3, 1).flatten(1)


def make_nature_dqn_network(num_actions, observation_shape=(84, 84), stack_size=4):
  """atari_lib.nature_dqn_network (atari_lib.py:85-105): convolutions, FC 512 (ReLU),
  FC num_actions; slim's default (Xavier uniform) initialisation."""
  torch = _torch()
  nn = torch.nn

  class NatureDQNNetwork(nn.Module):

    def __init__(self):
      super().__init__()
      self.convs, self.pads, features = conv_trunk(torch, observation_shape, stack_size,
                                                   xavier_uniform_)
      self.fc1 = nn.Linear(features, 512)
      self.fc2 = nn.Linear(512, num_actions)
      xavier_uniform_(torch, self.fc1)
      xavier_uniform_(torch, self.fc2)

    def forward(self, state):
      x = run_trunk(torch, self.convs, self.pads, state)
      return self.fc2(torch.relu(self.fc1(x)))

  return NatureDQNNetwork()


def make_tf_rmsprop(params, lr=0.00025, decay=0.95, momentum=0.0, epsilon=0.00001,
                    centered=True):
  """tf.train.RMSPropOptimizer as DQNAgent configures it (dqn_agent.py:100-105,
  dqn.gin:19-25).  TensorFlow 1.x (ApplyCenteredRMSProp):
      mg  = decay mg + (1 - decay) g          (centered)
      ms  = decay ms + (1 - decay) g^2        (ms starts at ONE, not zero)
      mom = momentum mom + lr g / sqrt(ms - mg^2 + epsilon)
      theta -= mom
  torch.optim.RMSprop adds epsilon OUTSIDE the square root and starts ms at zero, which
  at this epsilon changes the first updates by orders of magnitude."""
  torch = _torch()

  class TFRMSProp(torch.optim.Optimizer):

    def __init__(self):
      super().__init__(list(params), dict(lr=lr, decay=decay, momentum=momentum,
                                          epsilon=epsilon, centered=centered))

    @torch.no_grad()
    def step(self, closure=None):
      assert closure is None
      for group in self.param_groups:
        ps = [p for p in group['params'] if p.grad is not None]
        if not ps:
          continue
        grads = [p.grad for p in ps]
        ms, mg, mom = [], [], []
        for p in ps:
          state = self.state[p]
          if not state:
            state['ms'] = torch.ones_like(p)
            state['mg'] = torch.zeros_like(p)
            state['mom'] = torch.zeros_like(p)
          ms.append(state['ms'])
          mg.append(state['mg'])
          mom.append(state['mom'])
        rho = group['decay']
        torch._foreach_mul_(ms, rho)
        torch._foreach_addcmul_(ms, grads, grads, value=1.0 - rho)
        denom = [m.clone() for m in ms]
        if group['centered']:
          torch._foreach_mul_(mg, rho)
          torch._foreach_add_(mg, grads, alpha=1.0 - rho)
          torch._foreach_addcmul_(denom, mg, mg, value=-1.0)
        torch._foreach_add_(denom, group['epsilon'])
        torch._foreach_sqrt_(denom)
        update = torch._foreach_div(grads, denom)
        torch._foreach_mul_(update, group['lr'])
        if group['momentum']:
          torch._foreach_mul_(mom, group['momentum'])
          torch._foreach_add_(mom, update)
          update = mom
        torch._foreach_sub_(ps, update)
      return None

    def load_state_dict(self, state_dict):
      """In place: a captured update keeps reading the same accumulators."""
      sharded_learner.load_optimizer_state(self, state_dict)

  return TFRMSProp()


class DQNLearner(sharded_learner.GraphedUpdate):
  """Replay + train op of DQNAgent (dqn_agent.py:237-322).  With `cuda_graph=True` the
  whole update (uniform sampler, frame copies, both networks, loss, backward, RMSProp)
  is captured once and replayed as one CUDA graph (`GraphedUpdate`)."""

  def __init__(self, num_actions, observation_shape=(84, 84), stack_size=4, gamma=0.99,
               update_horizon=1, replay_capacity=1000000, batch_size=32,
               target_update_period=8000, update_period=4, seed=0, memory=None,
               cuda_graph=False):
    torch = _torch()
    self.num_actions = num_actions
    self.batch_size = batch_size
    self.update_period = update_period
    self.target_update_period = target_update_period
    # dqn_agent.py:265-281: the uniform buffer
    self.memory = memory or circular_replay_buffer.OutOfGraphReplayBuffer(
        observation_shape, stack_size, replay_capacity, batch_size,
        update_horizon=update_horizon, gamma=gamma, output='torch', rng='device',
        seed=seed, reuse_outputs=True)
    self.cumulative_gamma = dqn_agent.cumulative_gamma(gamma, update_horizon)
    torch.manual_seed(seed)
    self.online = make_nature_dqn_network(num_actions, observation_shape, stack_size).cuda()
    self.target = make_nature_dqn_network(num_actions, observation_shape, stack_size).cuda()
    self.target.load_state_dict(self.online.state_dict())
    for p in self.target.parameters():
      p.requires_grad_(False)
    self.optimizer = make_tf_rmsprop(self.online.parameters())
    self._cuda_graph = bool(cuda_graph)
    self._graph = None
    self._static_loss = None
    self.training_steps = 0
    self.updates = 0

  def store_transition(self, last_observation, action, reward, is_terminal):
    """dqn_agent.py:460-472."""
    self.memory.add(last_observation, action, reward, is_terminal)

  def q_values(self, state):
    with _torch().no_grad():
      return self.online(state)

  # train_step() is GraphedUpdate's
  def _update(self):
    """dqn_agent.py:283-322: sample -> target net on next_state, online net on state ->
    Bellman target + Huber loss (one kernel) -> backward -> RMSProp.  Returns the mean
    loss (a CUDA tensor, no sync)."""
    torch = _torch()
    batch = self.memory.sample_transition_batch(self.batch_size)
    state, action, reward, next_state, _, _, terminal = batch[:7]
    with torch.no_grad():
      target_q = self.target(next_state)
    online_q = self.online(state)
    loss, _ = dqn_agent.DQNLoss.apply(online_q, target_q, action, reward, terminal,
                                      self.cumulative_gamma)
    self.optimizer.zero_grad(set_to_none=True)
    loss.backward()
    self.optimizer.step()
    if not self._cuda_graph or self._graph is None:
      self.updates += 1
    return loss

  def sync_target(self):
    self.target.load_state_dict(self.online.state_dict())

  def step_cadence(self):
    """dqn_agent.py:418-442."""
    loss = None
    if self.training_steps % self.update_period == 0:
      loss = self.train_step()
    if self.training_steps % self.target_update_period == 0:
      self.sync_target()
    self.training_steps += 1
    return loss


class DQNAgent(DQNLearner, dqn_agent.ActingLoop):
  """`DQNAgent` (dqn_agent.py:76-560) as the reference's runner sees it:
  `begin_episode(observation)`, `step(reward, observation)`, `end_episode(reward)`,
  `eval_mode`, `bundle_and_checkpoint`, `unbundle`.  Constructor arguments keep the
  reference's names and defaults (dqn_agent.py:76-108); `sess`, `tf_device`,
  `use_staging`, `max_tf_checkpoints_to_keep`, `optimizer` (always TensorFlow's centred
  RMSProp with dqn.gin's numbers, `make_tf_rmsprop`) and the summary arguments have no
  meaning here.  `replay_capacity` and `batch_size` are the replay buffer's
  (`_build_replay_buffer`, dqn_agent.py:265-281, binds them through gin); `seed`,
  `memory` and `cuda_graph` are `DQNLearner`'s.  Lives here rather than in
  `dqn_agent.py` because this module imports that one."""

  def __init__(self, sess=None, num_actions=None, observation_shape=(84, 84),
               observation_dtype=np.uint8, stack_size=4, gamma=0.99, update_horizon=1,
               min_replay_history=20000, update_period=4, target_update_period=8000,
               epsilon_fn=dqn_agent.linearly_decaying_epsilon, epsilon_train=0.01,
               epsilon_eval=0.001, epsilon_decay_period=250000, tf_device='/cpu:*',
               use_staging=True, max_tf_checkpoints_to_keep=4, optimizer=None,
               summary_writer=None, summary_writing_frequency=500,
               replay_capacity=1000000, batch_size=32, seed=0,
               allow_partial_reload=False, memory=None, cuda_graph=False):
    del sess, tf_device, use_staging, max_tf_checkpoints_to_keep, optimizer
    del summary_writer, summary_writing_frequency
    if num_actions is None:
      raise ValueError('num_actions is required')
    if np.dtype(observation_dtype) != np.uint8:
      raise NotImplementedError('the convolutional network takes uint8 frames')
    DQNLearner.__init__(
        self, num_actions, observation_shape=observation_shape, stack_size=stack_size,
        gamma=gamma, update_horizon=update_horizon, replay_capacity=replay_capacity,
        batch_size=batch_size, target_update_period=target_update_period,
        update_period=update_period, seed=seed, memory=memory, cuda_graph=cuda_graph)
    self._init_acting(observation_shape, stack_size, observation_dtype,
                      min_replay_history=min_replay_history,
                      update_period=update_period,
                      target_update_period=target_update_period,
                      epsilon_fn=epsilon_fn, epsilon_train=epsilon_train,
                      epsilon_eval=epsilon_eval,
                      epsilon_decay_period=epsilon_decay_period,
                      allow_partial_reload=allow_partial_reload)

  def _store_transition(self, last_observation, action, reward, is_terminal):
    """dqn_agent.py:460-472: the uniform buffer takes no priority."""
    if not self.eval_mode:
      self.store_transition(last_observation, action, reward, is_terminal)


class ShardedDQNLearner(sharded_learner.ShardedLearner, DQNLearner):
  """`DQNLearner` on ONE global batch sharded over the ranks of torch.distributed.

  Every rank owns one uniform replay shard of `replay_capacity` transitions (the
  reference's `OutOfGraphReplayBuffer`, dqn_agent.py:265-281) and a peer-memory exchange.
  `batch_size` is the GLOBAL batch: the reference's uniform draws with rejection
  (circular_replay_buffer.py:436-477) over a virtual buffer whose index range is the
  concatenation of the shards' ranges (`ShardedUniformReplay`), so the update is the
  reference's update (dqn_agent.py:283-322) on one batch uniform over the union of the
  shards' valid transitions.  One update:
    1. `sample()`: sharded uniform sampler + frame copies into `max_rows` rows (default
       `share_bound`);
    2. `loss_backward()`: the target net on `next_state`, the online net on `state`, both
       on `max_rows` rows, then the sharded Bellman target + Huber loss (mean and
       gradient over the global batch, zero gradients for padded rows) and backward into
       one flat buffer;
    3. `reduce()`: ONE all-reduce (sum) of that buffer — every gradient and, appended,
       the partial loss, so the reported loss is the global mean;
    4. `apply()`: TF-form centred RMSProp.  There are no priorities to write back.
  `cuda_graph=True` captures the whole update, all-reduce included; `step_cadence()` is
  `DQNLearner`'s.  Errors latched on the device are raised by `check()`, which
  `sync_target()` calls.  Pass `exchange` (`PeerExchange.emulated`) to run the phases of
  several ranks on one device without torch.distributed (tests): each rank's sampler then
  needs the two publish-ahead phases of every rank first (`self.sharded.publish`), and
  `reduce()` is the caller's.
  """

  def __init__(self, num_actions, batch_size=32, max_rows=None, exchange=None,
               group=None, exchange_timeout_s=2.0, ddp=False, cuda_graph=False,
               **kwargs):
    exchange = self._connect(exchange, group, exchange_timeout_s, ddp)
    DQNLearner.__init__(self, num_actions, batch_size=batch_size, cuda_graph=cuda_graph,
                        **kwargs)
    self._shard(exchange, max_rows, kwargs.get('seed', 0),
                sharded_replay.ShardedUniformReplay)

  # -- phases (sample, reduce: ShardedLearner's) ----------------------------------------
  def loss_backward(self):
    """Networks, sharded loss and backward: the flat buffer holds this rank's partial
    gradients and partial mean.  Returns the per-row losses."""
    torch = _torch()
    _, count, batch = self._sample
    state, action, reward, next_state, _, _, terminal = batch[:7]
    with torch.no_grad():
      target_q = self.target(next_state)
    online_q = self.online(state)
    mean, rows = dqn_agent.ShardedDQNLoss.apply(online_q, target_q, action, reward,
                                                terminal, self.cumulative_gamma,
                                                (self.batch_size, count))
    self._flat.zero_()
    mean.backward()  # (accumulates into the views of the flat buffer)
    self.loss.copy_(mean.detach().view(1))
    return rows

  def apply(self):
    """RMSProp on the reduced gradients."""
    self.optimizer.step()

  def _update(self):
    self.sample()
    self.loss_backward()
    self.reduce()
    self.apply()
    if not self._cuda_graph or self._graph is None:
      self.updates += 1
    return self.loss
