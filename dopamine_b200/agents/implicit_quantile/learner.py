"""The learner half of ImplicitQuantileAgent on top of the B200 replay path.

What the reference builds around its replay memory
(dopamine/agents/implicit_quantile/implicit_quantile_agent.py:120-321,
implicit_quantile.gin): the implicit quantile network (atari_lib.py:147-199: state
features tiled over the quantile samples, times a cosine embedding of the sampled taus),
the target quantile values and the quantile-Huber loss as ONE kernel
(`quantile_huber_loss`, csrc/iqn.cu), TensorFlow's Adam with the reference's numbers, the
target sync.  Uniform replay through the prioritized buffer class, as the reference does
("IQN currently does not support prioritized replay", implicit_quantile.gin:23-24).
`ImplicitQuantileAgent` joins `IQNLearner` to the episode interface
(`dqn_agent.ActingLoop`) as the reference's runner creates it for implicit_quantile.gin.
"""
import math

import numpy as np

from dopamine_b200.agents import sharded_learner
from dopamine_b200.agents.dqn import dqn_agent
from dopamine_b200.agents.dqn import learner as dqn_learner
from dopamine_b200.agents.implicit_quantile import implicit_quantile_agent as iqn
from dopamine_b200.agents.rainbow import agent as conv
from dopamine_b200.replay_memory import prioritized_replay_buffer
from dopamine_b200.replay_memory import sharded_replay


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def _variance_scaling_(torch, module):
  """variance_scaling_initializer(1 / sqrt(3), FAN_IN, uniform) (atari_lib.py:160-161)."""
  fan_in = module.weight[0].numel()
  limit = math.sqrt(3.0 * (1.0 / math.sqrt(3.0)) / fan_in)
  torch.nn.init.uniform_(module.weight, -limit, limit)
  torch.nn.init.zeros_(module.bias)


def make_implicit_quantile_network(num_actions, quantile_embedding_dim=64,
                                   observation_shape=(84, 84), stack_size=4):
  """atari_lib.implicit_quantile_network (atari_lib.py:147-199).  forward(state,
  num_quantiles) -> (quantile_values (num_quantiles * B, A), quantiles (num_quantiles * B,
  1)); rows are sample-major (tf.tile of the state features, :176), the layout
  `quantile_huber_loss` takes."""
  torch = _torch()
  nn = torch.nn

  class ImplicitQuantileNetwork(nn.Module):

    def __init__(self):
      super().__init__()
      self.convs, self.pads, features = dqn_learner.conv_trunk(
          torch, observation_shape, stack_size, _variance_scaling_)
      self.embed = nn.Linear(quantile_embedding_dim, features)
      self.fc1 = nn.Linear(features, 512)
      self.fc2 = nn.Linear(512, num_actions)
      for m in (self.embed, self.fc1, self.fc2):
        _variance_scaling_(torch, m)
      # tf.range(1, dim + 1) * pi  (atari_lib.py:184-186), float32
      self.register_buffer(
          'multiples', torch.arange(1, quantile_embedding_dim + 1, dtype=torch.float32) *
          torch.tensor(math.pi, dtype=torch.float32))

    def forward(self, state, num_quantiles, quantiles=None):
      features = dqn_learner.run_trunk(torch, self.convs, self.pads, state)
      batch = features.shape[0]
      tiled = features.repeat(num_quantiles, 1)                      # :176
      if quantiles is None:                                          # :180-181
        quantiles = torch.rand(num_quantiles * batch, 1, device=features.device)
      embedding = torch.relu(self.embed(torch.cos(self.multiples * quantiles)))  # :183-189
      x = torch.relu(self.fc1(tiled * embedding))                    # :191-194
      return self.fc2(x), quantiles

  return ImplicitQuantileNetwork()


class IQNLearner(sharded_learner.GraphedUpdate):
  """Replay + train op of ImplicitQuantileAgent (implicit_quantile_agent.py:120-321).

  Eagerly the networks draw their taus with `torch.rand` (atari_lib.py:180-181).  With
  `cuda_graph=True` the whole update is captured once and replayed as one CUDA graph
  (`GraphedUpdate`); its taus are then drawn into three static buffers, `online_taus`
  (N * B, 1), `target_taus` (N' * B, 1) and `action_taus` (K * B, 1), refilled in place
  at every update from a CUDA generator of the learner seeded from `seed`, so that every
  replay draws fresh ones.  `q_values` (acting) keeps drawing its own taus and does not
  move that generator."""

  def __init__(self, num_actions, observation_shape=(84, 84), stack_size=4, kappa=1.0,
               num_tau_samples=32, num_tau_prime_samples=32, num_quantile_samples=32,
               quantile_embedding_dim=64, double_dqn=False, gamma=0.99, update_horizon=3,
               replay_capacity=1000000, batch_size=32, target_update_period=8000,
               update_period=4, learning_rate=0.00005, adam_epsilon=0.0003125, seed=0,
               memory=None, cuda_graph=False):
    torch = _torch()
    self.num_actions = num_actions
    self.kappa = kappa
    self.num_tau_samples = num_tau_samples
    self.num_tau_prime_samples = num_tau_prime_samples
    self.num_quantile_samples = num_quantile_samples
    self.double_dqn = double_dqn
    self.batch_size = batch_size
    self.update_period = update_period
    self.target_update_period = target_update_period
    self.memory = memory or prioritized_replay_buffer.OutOfGraphPrioritizedReplayBuffer(
        observation_shape, stack_size, replay_capacity, batch_size,
        update_horizon=update_horizon, gamma=gamma, output='torch', rng='device',
        seed=seed, reuse_outputs=True)
    self.cumulative_gamma = iqn.cumulative_gamma(gamma, update_horizon)
    torch.manual_seed(seed)
    make = lambda: make_implicit_quantile_network(
        num_actions, quantile_embedding_dim, observation_shape, stack_size).cuda()
    self.online, self.target = make(), make()
    self.target.load_state_dict(self.online.state_dict())
    for p in self.target.parameters():
      p.requires_grad_(False)
    self._cuda_graph = bool(cuda_graph)
    self._graph = None
    self._static_loss = None
    # with cuda_graph, Adam's step count lives on the device so that it can be captured
    self.optimizer = conv.make_tf_adam(self.online.parameters(), lr=learning_rate,
                                       epsilon=adam_epsilon,  # implicit_quantile.gin:26-29
                                       capturable=self._cuda_graph)
    self._generator = None
    if self._cuda_graph:
      self._init_taus(batch_size, [seed])
    self.training_steps = 0
    self.updates = 0

  def _init_taus(self, rows, entropy):
    """The three static tau buffers for `rows` batch rows and the CUDA generator that
    refills them, seeded from `entropy` (a list of ints)."""
    torch = _torch()
    self._generator = torch.Generator(device='cuda')
    self._generator.manual_seed(
        int(np.random.SeedSequence([int(e) for e in entropy]).generate_state(1)[0]))
    taus = lambda samples: torch.zeros(samples * rows, 1, device='cuda')
    self.online_taus = taus(self.num_tau_samples)
    self.target_taus = taus(self.num_tau_prime_samples)
    self.action_taus = taus(self.num_quantile_samples)

  def _draw_taus(self):
    """Fresh taus in the static buffers (atari_lib.py:180-181)."""
    for t in (self.online_taus, self.target_taus, self.action_taus):
      t.uniform_(0., 1., generator=self._generator)

  def _graph_generators(self):
    return (self._generator,)

  def store_transition(self, last_observation, action, reward, is_terminal):
    """rainbow_agent.py:307-337 with the uniform scheme: priority 1."""
    self.memory.add(last_observation, action, reward, is_terminal, 1.0)

  def q_values(self, state):
    """implicit_quantile_agent.py:148-164: mean over num_quantile_samples."""
    torch = _torch()
    with torch.no_grad():
      values, _ = self.online(state, self.num_quantile_samples)
      return values.view(self.num_quantile_samples, -1, self.num_actions).mean(0)

  # train_step() is GraphedUpdate's
  def _update(self):
    """implicit_quantile_agent.py:166-321: online net on `state` with N taus, target net
    on `next_state` with N' taus, the action-picking net with K taus (target net; online
    with double_dqn) -> greedy next action, target quantile values and quantile-Huber
    loss (one kernel) -> backward -> Adam.  Returns the mean loss (a CUDA tensor)."""
    torch = _torch()
    batch = self.memory.sample_transition_batch(self.batch_size)
    state, action, reward, next_state, _, _, terminal = batch[:7]
    online_taus = target_taus = action_taus = None  # eager: drawn inside the networks
    if self._generator is not None:
      self._draw_taus()
      online_taus, target_taus = self.online_taus, self.target_taus
      action_taus = self.action_taus
    with torch.no_grad():
      target_values, _ = self.target(next_state, self.num_tau_prime_samples, target_taus)
      picker = self.online if self.double_dqn else self.target
      action_values, _ = picker(next_state, self.num_quantile_samples, action_taus)
    online_values, quantiles = self.online(state, self.num_tau_samples, online_taus)
    loss, _ = iqn.QuantileHuberLoss.apply(
        online_values, quantiles, target_values, action_values, action, reward, terminal,
        self.cumulative_gamma, self.kappa)
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


class ImplicitQuantileAgent(IQNLearner, dqn_agent.ActingLoop):
  """`ImplicitQuantileAgent` (implicit_quantile_agent.py, on the acting loop of
  dqn_agent.py:341-560) as the reference's runner sees it: `begin_episode(observation)`,
  `step(reward, observation)`, `end_episode(reward)`, `eval_mode`,
  `bundle_and_checkpoint`, `unbundle`.  IQN's own arguments keep the reference's names
  and defaults; the `RainbowAgent` arguments the reference forwards through `**kwargs`
  are explicit here, with implicit_quantile.gin's numbers as `IQNLearner` has them.
  `sess`, `tf_device`, `use_staging`, `optimizer` (always TensorFlow's Adam,
  `learning_rate` / `adam_epsilon`) and the summary arguments have no meaning here.
  Replay is uniform (implicit_quantile.gin:23-24): transitions are stored with priority
  1.  The greedy action is the first argmax of the mean over `num_quantile_samples`
  quantile values (`IQNLearner.q_values`, implicit_quantile_agent.py:148-164)."""

  def __init__(self, sess=None, num_actions=None, kappa=1.0, num_tau_samples=32,
               num_tau_prime_samples=32, num_quantile_samples=32,
               quantile_embedding_dim=64, double_dqn=False, summary_writer=None,
               summary_writing_frequency=500, observation_shape=(84, 84),
               observation_dtype=np.uint8, stack_size=4, gamma=0.99, update_horizon=3,
               min_replay_history=20000, update_period=4, target_update_period=8000,
               epsilon_fn=dqn_agent.linearly_decaying_epsilon, epsilon_train=0.01,
               epsilon_eval=0.001, epsilon_decay_period=250000, tf_device='/cpu:*',
               use_staging=True, optimizer=None, replay_capacity=1000000, batch_size=32,
               learning_rate=0.00005, adam_epsilon=0.0003125, seed=0,
               allow_partial_reload=False, memory=None, cuda_graph=False):
    del sess, summary_writer, summary_writing_frequency, tf_device, use_staging
    del optimizer
    if num_actions is None:
      raise ValueError('num_actions is required')
    if np.dtype(observation_dtype) != np.uint8:
      raise NotImplementedError('the convolutional network takes uint8 frames')
    IQNLearner.__init__(
        self, num_actions, observation_shape=observation_shape, stack_size=stack_size,
        kappa=kappa, num_tau_samples=num_tau_samples,
        num_tau_prime_samples=num_tau_prime_samples,
        num_quantile_samples=num_quantile_samples,
        quantile_embedding_dim=quantile_embedding_dim, double_dqn=double_dqn,
        gamma=gamma, update_horizon=update_horizon, replay_capacity=replay_capacity,
        batch_size=batch_size, target_update_period=target_update_period,
        update_period=update_period, learning_rate=learning_rate,
        adam_epsilon=adam_epsilon, seed=seed, memory=memory, cuda_graph=cuda_graph)
    self._init_acting(observation_shape, stack_size, observation_dtype,
                      min_replay_history=min_replay_history,
                      update_period=update_period,
                      target_update_period=target_update_period,
                      epsilon_fn=epsilon_fn, epsilon_train=epsilon_train,
                      epsilon_eval=epsilon_eval,
                      epsilon_decay_period=epsilon_decay_period,
                      allow_partial_reload=allow_partial_reload)

  def _store_transition(self, last_observation, action, reward, is_terminal):
    """rainbow_agent.py:307-337 with the uniform scheme: priority 1."""
    if not self.eval_mode:
      self.store_transition(last_observation, action, reward, is_terminal)


class ShardedIQNLearner(sharded_learner.ShardedLearner, IQNLearner):
  """`IQNLearner` on ONE global batch sharded over the ranks of torch.distributed.

  Every rank owns one replay shard of `replay_capacity` transitions (unit priorities, as
  the reference's IQN uses its prioritized buffer, implicit_quantile.gin:23-24) and a
  peer-memory exchange.  `batch_size` is the GLOBAL batch: its strata are apportioned
  over the shards by their totals, i.e. by their transition counts, so the update is the
  reference's update (implicit_quantile_agent.py:166-321) on one uniform batch of a
  virtual replay of every shard's transitions.  One update:
    1. `sample()`: sharded sampler + frame copies into `max_rows` rows (default
       `share_bound`), then fresh taus for the three networks;
    2. `loss_backward()`: the online net on `state` with N taus, the target net on
       `next_state` with N' taus and the action-picking net (target net; online net with
       `double_dqn`) with K taus, all on `max_rows` rows, then the sharded
       quantile-Huber loss (mean and gradient over the global batch, zero gradients for
       padded rows) and backward into one flat buffer;
    3. `reduce()`: ONE all-reduce (sum) of that buffer — every gradient and, appended,
       the partial loss, so the reported loss is the global mean;
    4. `apply()`: TF-form Adam.  Priorities stay 1: there is no write-back.
  IQN has no importance weights, so the loss exchanges nothing between the ranks.  The
  taus are drawn into three static buffers, `online_taus` (N * max_rows, 1),
  `target_taus` (N' * max_rows, 1) and `action_taus` (K * max_rows, 1), refilled in
  place by every `sample()` from a CUDA generator seeded with (seed, rank): an emulated
  rank and a process of the same rank draw the same taus, and a replayed graph draws
  fresh ones.  `cuda_graph=True` captures the whole update, all-reduce included.  Errors
  latched on the device are raised by `check()`, which `sync_target()` calls.  Pass
  `exchange` (`PeerExchange.emulated`) to run the phases of several ranks on one device
  without torch.distributed (tests); `reduce()` then is the caller's.
  """

  def __init__(self, num_actions, batch_size=32, max_rows=None, exchange=None,
               group=None, exchange_timeout_s=2.0, ddp=False, cuda_graph=False,
               **kwargs):
    exchange = self._connect(exchange, group, exchange_timeout_s, ddp)
    IQNLearner.__init__(self, num_actions, batch_size=batch_size, **kwargs)
    self._cuda_graph = bool(cuda_graph)
    self._graph = None
    self._static_loss = None
    if self._cuda_graph:  # Adam's step count on the device, so that it can be captured
      adam = self.optimizer.param_groups[0]
      self.optimizer = conv.make_tf_adam(self.online.parameters(), lr=adam['lr'],
                                         epsilon=adam['epsilon'], capturable=True)
    seed = kwargs.get('seed', 0)
    self._shard(exchange, max_rows, seed, sharded_replay.ShardedPrioritizedReplay)
    self._init_taus(self.max_rows, [seed, self.rank])

  # -- phases (reduce: ShardedLearner's) ----------------------------------------------
  def sample(self):
    """This rank's share of the global batch, then fresh taus (:180-181)."""
    sample = super(ShardedIQNLearner, self).sample()
    self._draw_taus()
    return sample

  def loss_backward(self):
    """Networks, sharded loss and backward: the flat buffer holds this rank's partial
    gradients and partial mean.  Returns the per-row losses."""
    torch = _torch()
    _, count, batch, _ = self._sample
    state, action, reward, next_state, _, _, terminal = batch[:7]
    with torch.no_grad():
      target_values, _ = self.target(next_state, self.num_tau_prime_samples,
                                     self.target_taus)
      picker = self.online if self.double_dqn else self.target
      action_values, _ = picker(next_state, self.num_quantile_samples, self.action_taus)
    online_values, _ = self.online(state, self.num_tau_samples, self.online_taus)
    mean, rows = iqn.ShardedQuantileHuberLoss.apply(
        online_values, self.online_taus, target_values, action_values, action, reward,
        terminal, self.cumulative_gamma, self.kappa, (self.batch_size, count))
    self._flat.zero_()
    mean.backward()  # (accumulates into the views of the flat buffer)
    self.loss.copy_(mean.detach().view(1))
    return rows

  def apply(self):
    """Adam on the reduced gradients."""
    self.optimizer.step()

  # -- checkpoints (ShardedLearner's, with this rank's tau generator) ------------------
  def _rank_state(self):
    state = super(ShardedIQNLearner, self)._rank_state()
    state['tau_generator'] = bytes(self._generator.get_state().numpy()).hex()
    return state

  def _load_rank_state(self, state):
    torch = _torch()
    super(ShardedIQNLearner, self)._load_rank_state(state)
    words = bytearray.fromhex(state['tau_generator'])
    self._generator.set_state(torch.frombuffer(words, dtype=torch.uint8))  # (in place)

  def _update(self):
    self.sample()
    self.loss_backward()
    self.reduce()
    self.apply()
    if not self._cuda_graph or self._graph is None:
      self.updates += 1
    return self.loss
