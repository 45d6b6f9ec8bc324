"""The DQN and implicit-quantile agents: `learner.DQNAgent` and
`learner.ImplicitQuantileAgent`, the episode interface the reference's runner drives
(`dqn_agent.ActingLoop`) around `DQNLearner` / `IQNLearner`, and both learners' update
replayed as one CUDA graph.

The agent tests restate tests/dopamine/agents/dqn/dqn_agent_test.py (testBeginEpisode
:103, testStepEval :139, testStepTrain :174, testBundling :346) and hold both agents to
tests/golden/actor_episodes.npz, which the reference's own DQNAgent methods wrote."""
import inspect
import random
import zlib

import numpy as np
import pytest

from tests import golden_cases

AGENTS = ['dqn', 'iqn']


def _agent_class(kind):
  if kind == 'dqn':
    from dopamine_b200.agents.dqn import learner
    return learner.DQNAgent
  from dopamine_b200.agents.implicit_quantile import learner
  return learner.ImplicitQuantileAgent


# IQN's network is smaller here than implicit_quantile.gin's: the tests are about the
# agent, not the network, and fewer taus keep them quick
_SMALL_IQN = dict(num_tau_samples=8, num_tau_prime_samples=8, num_quantile_samples=4)


def _small(kind):
  return dict(_SMALL_IQN) if kind == 'iqn' else {}


# ------------------------------------------------------------------ CPU side ----
@pytest.mark.parametrize('kind', AGENTS)
def test_constructor_refusals(kind):
  """num_actions is required; the Nature network's input kernel takes uint8 frames."""
  cls = _agent_class(kind)
  with pytest.raises(ValueError, match='num_actions is required'):
    cls()
  with pytest.raises(NotImplementedError, match='uint8'):
    cls(num_actions=4, observation_dtype=np.float32)


def _defaults(cls):
  return {name: p.default for name, p in inspect.signature(cls.__init__).parameters.items()
          if p.default is not inspect.Parameter.empty}


def test_reference_defaults():
  """dqn_agent.py:76-108 (dqn.gin's RMSProp numbers are make_tf_rmsprop's defaults);
  implicit_quantile_agent.py's own arguments and implicit_quantile.gin's values of the
  forwarded ones (update_horizon 3, Adam 5e-5 / 3.125e-4)."""
  from dopamine_b200.agents.dqn import dqn_agent
  from dopamine_b200.agents.dqn import learner as dqn_learner
  from dopamine_b200.agents.implicit_quantile import learner as iqn_learner
  acting = dict(observation_shape=(84, 84), observation_dtype=np.uint8, stack_size=4,
                gamma=0.99, min_replay_history=20000, update_period=4,
                target_update_period=8000,
                epsilon_fn=dqn_agent.linearly_decaying_epsilon, epsilon_train=0.01,
                epsilon_eval=0.001, epsilon_decay_period=250000, replay_capacity=1000000,
                batch_size=32, allow_partial_reload=False, cuda_graph=False)
  dqn = _defaults(dqn_learner.DQNAgent)
  for name, want in dict(acting, update_horizon=1).items():
    assert dqn[name] == want, name
  assert dqn['num_actions'] is None
  iqn = _defaults(iqn_learner.ImplicitQuantileAgent)
  for name, want in dict(acting, update_horizon=3, kappa=1.0, num_tau_samples=32,
                         num_tau_prime_samples=32, num_quantile_samples=32,
                         quantile_embedding_dim=64, double_dqn=False,
                         learning_rate=0.00005, adam_epsilon=0.0003125).items():
    assert iqn[name] == want, name
  # the same numbers as the learner underneath
  learner = _defaults(iqn_learner.IQNLearner)
  for name in ('kappa', 'num_tau_samples', 'num_tau_prime_samples',
               'num_quantile_samples', 'quantile_embedding_dim', 'double_dqn', 'gamma',
               'update_horizon', 'learning_rate', 'adam_epsilon', 'replay_capacity',
               'batch_size'):
    assert iqn[name] == learner[name], name


@pytest.mark.parametrize('kind', AGENTS)
def test_tf_only_arguments_are_accepted(kind):
  """The reference's TensorFlow plumbing is accepted and ignored: the call gets as far
  as the argument checks (no TypeError)."""
  cls = _agent_class(kind)
  tf_only = dict(sess=object(), tf_device='/gpu:0', use_staging=False, optimizer=object(),
                 summary_writer=object(), summary_writing_frequency=10)
  if kind == 'dqn':
    tf_only['max_tf_checkpoints_to_keep'] = 2
  with pytest.raises(ValueError, match='num_actions is required'):
    cls(**tf_only)


# ------------------------------------------------------------------ GPU side ----
@pytest.fixture(scope='module')
def torch():
  import torch as torch_module
  if not torch_module.cuda.is_available():
    pytest.fail('-m gpu tests need a CUDA device (no CPU fallback exists)')
  return torch_module


class _LoggedMemory(object):
  """Forwards add() to the agent's replay memory after logging what was stored."""

  def __init__(self, memory, log):
    self._memory, self._log = memory, log

  def add(self, obs, action, reward, terminal, *rest):
    self._log['stored'].append((zlib.crc32(np.ascontiguousarray(obs).tobytes()),
                                int(action), float(reward), int(terminal)))
    self._memory.add(obs, action, reward, terminal, *rest)

  def __getattr__(self, name):
    return getattr(self._memory, name)


class _MockMemory(object):
  """test_utils.MockReplayBuffer: records the calls to add()."""

  def __init__(self):
    self.add_count = 0
    self.calls = []

  def add(self, *args):
    self.calls.append(args)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', AGENTS)
@pytest.mark.parametrize('name', sorted(golden_cases.ACTOR_CASES))
def test_agent_matches_reference_fixture(torch, kind, name):
  """The agent with its frame stack in HBM and its own replay memory behind it
  reproduces what the reference's DQNAgent methods wrote: actions, every intermediate
  state, every stored transition, train and sync steps, add_count and the position of
  Python's random stream afterwards."""
  cls = _agent_class(kind)

  def make_agent(shape, stack, num_actions, params, log):

    class Agent(cls):

      def q_values(self, state):
        q = torch.zeros(1, num_actions, device='cuda')
        q[0, golden_cases.greedy_rule(state, num_actions)] = 1.0
        return q

      def train_step(self):
        log['train'].append(self.training_steps)

      def sync_target(self):
        log['sync'].append(self.training_steps)

    agent = Agent(num_actions=num_actions, observation_shape=shape, stack_size=stack,
                  update_horizon=1, replay_capacity=200, batch_size=8, **params)
    agent.memory = _LoggedMemory(agent.memory, log)
    return agent

  golden_cases.check_actor(make_agent, name)


def _test_agent(torch, kind, **kw):
  """dqn_agent_test.py:53-90: a network that always prefers action 0, no exploration,
  eval mode."""
  cls = _agent_class(kind)

  class MockAgent(cls):

    def q_values(self, state):
      q = torch.arange(self.num_actions, 0, -1, dtype=torch.float32, device='cuda')
      return (q + 1.0).repeat(state.shape[0], 1)

  args = dict(num_actions=4, min_replay_history=6, update_period=2,
              target_update_period=4, epsilon_fn=lambda w, x, y, z: 0.0,
              epsilon_eval=0.0, replay_capacity=1000, batch_size=8, update_horizon=3)
  args.update(_small(kind))
  args.update(kw)
  agent = MockAgent(**args)
  agent.eval_mode = True
  return agent


@pytest.mark.gpu
@pytest.mark.parametrize('kind', AGENTS)
def test_begin_episode(torch, kind):
  """dqn_agent_test.py:103-137."""
  agent = _test_agent(torch, kind)
  shape = (84, 84)
  agent.state.fill_(9)
  first = np.ones(shape + (1,))
  assert agent.begin_episode(first) == 0
  want = np.zeros((1,) + shape + (4,), np.uint8)
  want[:, :, :, -1] = 1
  assert np.array_equal(agent.state.cpu().numpy(), want)
  assert np.array_equal(agent._observation, first[:, :, 0])
  assert agent.training_steps == 0  # no training in eval mode
  agent.eval_mode = False
  second = np.ones(shape + (1,)) * 2
  agent.begin_episode(second)
  want[:, :, :, -1] = 2
  assert np.array_equal(agent.state.cpu().numpy(), want)
  assert np.array_equal(agent._observation, second[:, :, 0])
  assert agent.training_steps == 1
  assert agent.updates == 0  # add_count below min_replay_history: no train op


@pytest.mark.gpu
@pytest.mark.parametrize('kind', AGENTS)
def test_step_eval(torch, kind):
  """dqn_agent_test.py:139-172."""
  agent = _test_agent(torch, kind)
  shape = (84, 84)
  base = np.ones(shape + (1,))
  agent.begin_episode(base)
  agent.memory = _MockMemory()
  want = np.zeros((1,) + shape + (4,), np.uint8)
  num_steps = 10
  for step in range(1, num_steps + 1):
    observation = base * step
    assert agent.step(reward=1, observation=observation) == 0
    stack_pos = step - num_steps - 1
    if stack_pos >= -4:
      want[:, :, :, stack_pos] = step
  assert np.array_equal(agent.state.cpu().numpy(), want)
  assert np.array_equal(agent._last_observation, np.ones(shape) * (num_steps - 1))
  assert np.array_equal(agent._observation, observation[:, :, 0])
  assert agent.training_steps == 0
  assert not agent.memory.calls


@pytest.mark.gpu
@pytest.mark.parametrize('kind,priority', [('dqn', ()), ('iqn', (1.0,))])
def test_step_train(torch, kind, priority):
  """dqn_agent_test.py:174-223 with each agent's own add: no priority on DQN's uniform
  buffer (dqn_agent.py:460-472), priority 1 on IQN's (the uniform scheme)."""
  agent = _test_agent(torch, kind)
  agent.eval_mode = False
  shape = (84, 84)
  base = np.ones(shape + (1,))
  agent.memory = _MockMemory()
  agent.begin_episode(base)
  observation = base
  want = np.zeros((1,) + shape + (4,), np.uint8)
  num_steps = 10
  for step in range(1, num_steps + 1):
    last_observation = observation
    observation = base * step
    assert agent.step(reward=1, observation=observation) == 0
    stack_pos = step - num_steps - 1
    if stack_pos >= -4:
      want[:, :, :, stack_pos] = step
    assert len(agent.memory.calls) == step
    args = agent.memory.calls[-1]
    assert np.array_equal(last_observation[:, :, 0], args[0])
    assert args[1] == 0 and args[2] == 1 and not args[3]
    assert args[4:] == priority
  assert np.array_equal(agent.state.cpu().numpy(), want)
  assert np.array_equal(agent._last_observation, np.full(shape, num_steps - 1))
  assert agent.training_steps == num_steps + 1
  agent.end_episode(reward=1)
  assert len(agent.memory.calls) == num_steps + 1
  args = agent.memory.calls[-1]
  assert np.array_equal(observation[:, :, 0], args[0])
  assert args[1] == 0 and args[2] == 1 and args[3]
  assert args[4:] == priority


def _q_values(torch, agent, state, kind):
  """The agent's q-values; IQN's draw their taus from the default CUDA generator, which
  is seeded first so that two agents see the same taus."""
  if kind == 'iqn':
    torch.manual_seed(123)
  return agent.q_values(state)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', AGENTS)
def test_train_cadence_exploration_and_bundle(torch, kind, tmp_path):
  """A real agent over a few episodes: the train op runs on exactly the steps where
  add_count > min_replay_history and training_steps is a multiple of update_period, the
  target sync likewise every target_update_period steps (dqn_agent.py:430-441); the
  exploratory actions are Python's random stream (dqn_agent.py:411-413); a bundle
  restores state, counters, replay contents and every parameter (dqn_agent.py:480-560),
  and the restored agent's q-values are the original's."""
  cls = _agent_class(kind)
  log = dict(cadence=[], train=[], sync=[])

  class Agent(cls):

    def _train_step(self):
      log['cadence'].append((int(self.memory.add_count), self.training_steps))
      super(Agent, self)._train_step()

    def train_step(self):
      log['train'].append(self.training_steps)
      return super(Agent, self).train_step()

    def sync_target(self):
      log['sync'].append(self.training_steps)
      super(Agent, self).sync_target()

  rng = np.random.RandomState(1)
  kw = dict(num_actions=5, min_replay_history=40, update_period=2,
            target_update_period=8, epsilon_fn=lambda *unused: 0.3,
            replay_capacity=500, batch_size=8, update_horizon=3, seed=1)
  kw.update(_small(kind))
  agent = Agent(**kw)
  random.seed(11)
  actions = []
  for _ in range(3):
    actions.append(agent.begin_episode(rng.randint(0, 256, size=(84, 84, 1))))
    for _ in range(30):
      actions.append(agent.step(float(rng.randn()), rng.randint(0, 256, size=(84, 84, 1))))
    agent.end_episode(1.0)
  assert all(0 <= a < 5 for a in actions)
  assert len(set(actions)) > 1  # epsilon 0.3: some exploration
  assert agent.training_steps == 3 * 31
  # adds: 30 steps + 1 terminal per episode, + 3 pads at each episode start
  assert int(agent.memory.add_count) == 3 * (31 + 3)
  assert log['train'] == [t for c, t in log['cadence'] if c > 40 and t % 2 == 0]
  assert log['sync'] == [t for c, t in log['cadence'] if c > 40 and t % 8 == 0]
  assert log['train'] and log['sync']
  assert agent.updates == len(log['train'])
  # the random stream is the reference's: epsilon test, then randint
  greedy = int(_q_values(torch, agent, agent.state, kind).argmax(dim=1)[0])
  assert 0 <= greedy < 5
  random.seed(5)
  if kind == 'iqn':
    torch.manual_seed(123)
  picked = agent._select_action()
  random.seed(5)
  if random.random() <= 0.3:
    assert picked == random.randint(0, 4)
  else:
    assert picked == greedy
  bundle = agent.bundle_and_checkpoint(str(tmp_path), 7)
  assert set(bundle) == {'state', 'training_steps'}
  assert agent.bundle_and_checkpoint(str(tmp_path / 'missing'), 7) is None
  clone = cls(**dict(kw, seed=2))
  assert not clone.unbundle(str(tmp_path), 8, bundle)  # no such iteration
  assert clone.unbundle(str(tmp_path), 7, bundle)
  assert clone.training_steps == agent.training_steps
  assert torch.equal(clone.state, agent.state)
  assert int(clone.memory.add_count) == int(agent.memory.add_count)
  assert np.array_equal(clone.memory.invalid_range, agent.memory.invalid_range)
  for column in ('observation', 'action', 'reward', 'terminal'):
    assert np.array_equal(clone.memory._store[column], agent.memory._store[column]), column
  for a, b in zip(list(agent.online.parameters()) + list(agent.target.parameters()),
                  list(clone.online.parameters()) + list(clone.target.parameters())):
    assert torch.equal(a, b)
  x = agent.state
  assert torch.equal(_q_values(torch, agent, x, kind), _q_values(torch, clone, x, kind))


@pytest.mark.gpu
def test_iqn_greedy_action_is_first_argmax_of_the_quantile_mean(torch):
  """implicit_quantile_agent.py:148-164: the greedy action is the first argmax of the
  mean over num_quantile_samples quantile values.  The taus q_values draws are the ones
  a seeded torch.rand gives, so the network is re-run on those fixed taus; two actions
  with identical output weights tie, and the lower index wins."""
  cls = _agent_class('iqn')
  k, num_actions = 5, 6
  agent = cls(num_actions=num_actions, num_quantile_samples=k, replay_capacity=100,
              batch_size=8, epsilon_eval=0.0, seed=3)
  agent.eval_mode = True
  rng = np.random.RandomState(2)

  def expected(seed):
    torch.manual_seed(seed)
    taus = torch.rand(k, 1, device='cuda')
    with torch.no_grad():
      values, used = agent.online(agent.state, k, taus)
    assert torch.equal(used, taus)
    assert tuple(values.shape) == (k, num_actions)
    mean = values.view(k, 1, num_actions).mean(0)[0].cpu().numpy()
    return int(np.argmax(mean)), mean  # numpy's argmax: the first maximum

  def act(seed, observation):
    agent.begin_episode(observation)
    torch.manual_seed(seed)
    return agent._select_action()

  picks = set()
  for seed in range(6):
    observation = rng.randint(0, 256, size=(84, 84, 1))
    got = act(seed, observation)
    want, _ = expected(seed)
    assert got == want
    picks.add(got)
  with torch.no_grad():  # actions 1 and 4 tie, above every other
    agent.online.fc2.weight[4].copy_(agent.online.fc2.weight[1])
    agent.online.fc2.bias[1] = agent.online.fc2.bias[4] = 50.0
  got = act(7, rng.randint(0, 256, size=(84, 84, 1)))
  want, mean = expected(7)
  assert mean[1] == mean[4] and want == 1
  assert got == 1


def _graph_equals_eager(torch, make, capacity, batch_size, steps=12):
  """tests/test_learner.py:test_graph_replayed_learner_equals_eager for a learner made
  by `make(cuda_graph)`: adds between the updates, the eager learner fed what the
  graphed one sees (its 3 warm-up updates at capture, the sampler's draw offset)."""
  rng = np.random.RandomState(2)
  total = 500 + 4 * steps
  frames = rng.randint(0, 256, size=(total, 84, 84)).astype(np.uint8)
  acts = rng.randint(0, 5, size=total)
  rews = np.clip(rng.randn(total), -1, 1)
  terms = rng.rand(total) < 0.02

  def run(cuda_graph):
    torch.manual_seed(0)
    learner = make(cuda_graph)
    k = 0
    for _ in range(500):
      learner.store_transition(frames[k], int(acts[k]), float(rews[k]), int(terms[k]))
      k += 1
    losses, indices = [], []
    for it in range(steps):
      for _ in range(4):
        learner.store_transition(frames[k], int(acts[k]), float(rews[k]), int(terms[k]))
        k += 1
      if not cuda_graph:
        if it == 0:
          for _ in range(3):  # the graphed learner warms up with 3 updates at capture
            learner.train_step()
        else:
          # the captured sampler keeps the host draw offset of the capture call (4)
          # and advances only the device counter: give the eager run the same stream
          learner.memory._draw_counter = 3
      losses.append(float(learner.train_step().detach()))
      batch = learner.memory._output_cache[(batch_size, True)][1]
      indices.append(batch[7].cpu().numpy().copy())
    torch.cuda.synchronize()
    assert learner.updates == steps + 3
    params = [p.detach().cpu().numpy().copy() for p in learner.online.parameters()]
    return losses, params, indices

  eager = run(False)
  graphed = run(True)
  # the replayed sampler sees the adds made since the capture (with `capacity` below
  # the number of adds, also the wrap of the cursor): the same indices, update by update
  for a, b in zip(graphed[2], eager[2]):
    assert np.array_equal(a, b)
  np.testing.assert_allclose(graphed[0], eager[0], rtol=2e-3)
  for a, b in zip(graphed[1], eager[1]):
    np.testing.assert_allclose(a, b, rtol=2e-3, atol=5e-4)


@pytest.mark.gpu
def test_dqn_graph_replayed_learner_equals_eager(torch):
  """DQNLearner(cuda_graph=True): the uniform sampler, the frame copies, both networks,
  the Huber kernel, backward and RMSProp replayed as one graph equal the eager
  learner fed identically, with the replay wrapping around during the run."""
  from dopamine_b200.agents.dqn import learner as dqn_learner
  make = lambda cuda_graph: dqn_learner.DQNLearner(
      5, replay_capacity=520, batch_size=16, seed=7, cuda_graph=cuda_graph)
  _graph_equals_eager(torch, make, 520, 16)


@pytest.mark.gpu
def test_iqn_graph_replayed_learner_equals_eager(torch):
  """IQNLearner(cuda_graph=True) draws its taus into static buffers from its own
  generator; the eager learner given the same generator (`_init_taus` with the same
  seed) computes the same updates.  Acting between updates does not move that stream."""
  from dopamine_b200.agents.implicit_quantile import learner as iqn_learner

  def make(cuda_graph):
    learner = iqn_learner.IQNLearner(5, replay_capacity=1000, batch_size=16, seed=7,
                                     cuda_graph=cuda_graph, **_SMALL_IQN)
    if not cuda_graph:
      learner._init_taus(16, [7])
    original = learner.train_step

    def train_step_after_acting():
      learner.q_values(torch.zeros(1, 84, 84, 4, dtype=torch.uint8, device='cuda'))
      return original()

    learner.train_step = train_step_after_acting
    return learner

  _graph_equals_eager(torch, make, 1000, 16)

