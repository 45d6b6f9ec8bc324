"""Checkpoints of the data-parallel learners (ShardedLearner.save / restore,
b2r_sampler_state_*, b2r_exchange_state_*) and Adam's step count in TFAdam.state_dict.
CPU tests check the ABI's refusals, the restore's checks that need no device and the
optimizer's state; the GPU tests (`pytest -m gpu`) check that a restored run continues
bit for bit, with ranks emulated on one device, with an update captured as CUDA graphs
before the restore, and with real processes, that each rank directory is a plain replay
checkpoint, and that every refused restore leaves every rank as it was."""
import gzip
import hashlib
import json
import os
import shutil
import socket

import numpy as np
import pytest

from dopamine_b200 import _native

FRAME = 84 * 84
ACTIONS = 6
CAP = 2000
BATCH = 64
HORIZON = 3
K_UPDATES, M_UPDATES = 2, 3
KINDS = ['rainbow-prioritized', 'rainbow-uniform', 'iqn', 'dqn']
STORE = '$store$_'


# -- CPU -----------------------------------------------------------------------------
def test_state_words_are_refused_without_a_device():
  """A version or word count other than the header's is refused before the handle or
  the device is looked at."""
  lib = _native.lib()
  words = np.zeros(4, dtype=np.uint64)
  for fn, version, n in ((lib.b2r_sampler_state_set, _native.SAMPLER_STATE_VERSION,
                          _native.SAMPLER_STATE_WORDS),
                         (lib.b2r_sampler_state_get, _native.SAMPLER_STATE_VERSION,
                          _native.SAMPLER_STATE_WORDS),
                         (lib.b2r_exchange_state_set, _native.EXCHANGE_STATE_VERSION,
                          _native.EXCHANGE_STATE_WORDS),
                         (lib.b2r_exchange_state_get, _native.EXCHANGE_STATE_VERSION,
                          _native.EXCHANGE_STATE_WORDS)):
    assert fn(None, version + 1, _native.ptr(words), n, None) == _native.ERR_INVALID_ARGUMENT
    assert 'version' in _native.last_error()
    assert fn(None, version, _native.ptr(words), n + 1, None) == _native.ERR_INVALID_ARGUMENT
    assert 'words' in _native.last_error()
    assert fn(None, version, _native.ptr(words), n, None) == _native.ERR_INVALID_ARGUMENT
    assert 'NULL' in _native.last_error()


def test_adam_state_dict_carries_the_step_count_and_loads_in_place():
  import torch
  from dopamine_b200.agents.rainbow import agent
  torch.manual_seed(0)
  params = [torch.nn.Parameter(torch.randn(5)), torch.nn.Parameter(torch.randn(3, 2))]
  adam = agent.make_tf_adam(params, lr=0.1)
  for _ in range(4):
    for p in params:
      p.grad = torch.randn_like(p)
    adam.step()
  saved = adam.state_dict()
  assert saved['step'] == 4
  fresh_params = [torch.nn.Parameter(p.detach().clone()) for p in params]
  fresh = agent.make_tf_adam(fresh_params, lr=0.1)
  for p in fresh_params:
    p.grad = torch.zeros_like(p)
  fresh.step()
  held = [fresh.state[p]['m'] for p in fresh_params]
  fresh.load_state_dict(saved)
  assert fresh._host_t == 4
  for p, q, m in zip(params, fresh_params, held):
    assert fresh.state[q]['m'] is m  # in place
    assert torch.equal(m, adam.state[p]['m'])
    assert torch.equal(fresh.state[q]['v'], adam.state[p]['v'])
  grads = [torch.randn_like(p) for p in params]
  for ps, opt in ((params, adam), (fresh_params, fresh)):
    for p, g in zip(ps, grads):
      p.grad = g.clone()
    opt.step()
  for p, q in zip(params, fresh_params):
    assert torch.equal(p, q)


class _Stub(object):
  """What ShardedLearner's checks read, without a device."""

  def __init__(self, world=2, rank=0, capacity=CAP, batch=BATCH, scheme='prioritized'):
    from dopamine_b200.agents import sharded_learner
    self.cls = sharded_learner.ShardedLearner
    self.world, self.rank, self.batch_size, self.max_rows = world, rank, batch, 64
    self.replay_scheme = scheme
    self.memory = type('M', (), dict(_replay_capacity=capacity, _update_horizon=HORIZON))()
    self.sharded = type('S', (), dict(seed=3))()

  def prepare(self, path, iteration):
    learner = self.cls.__new__(self.cls)
    learner.__dict__.update(self.__dict__)
    return learner._prepare_restore(path, iteration)


def _fake_checkpoint(path, world=2, **changes):
  from dopamine_b200.agents import sharded_learner
  stub = _Stub(world=world)
  learner = stub.cls.__new__(stub.cls)
  learner.__dict__.update(stub.__dict__)
  manifest = dict(learner._manifest(), **changes)
  files = sharded_learner._Files(str(path), 7)
  with open(files.manifest, 'w') as f:
    json.dump(manifest, f)
  with open(files.sentinel, 'w') as f:
    f.write('complete\n')
  for g in range(world):
    os.makedirs(files.rank_dir(g))
    with open(files.rank_state(g), 'w') as f:
      json.dump({'rank': g, 'world_size': world}, f)
  return files


@pytest.mark.parametrize('change,stub,word', [
    ('manifest', {}, 'no manifest'),
    ('sentinel', {}, 'not complete'),
    ('rank', {}, 'rank 1 is missing'),
    (None, dict(world=3), 'world_size'),
    (None, dict(capacity=CAP // 2), 'shard_capacity'),
    (None, dict(scheme='uniform'), 'kind'),
    (None, dict(batch=2 * BATCH), 'global_batch'),
])
def test_restore_checks_that_need_no_device(tmp_path, change, stub, word):
  from dopamine_b200.agents import sharded_learner
  files = _fake_checkpoint(tmp_path)
  if change == 'manifest':
    os.remove(files.manifest)
  elif change == 'sentinel':
    os.remove(files.sentinel)
  elif change == 'rank':
    shutil.rmtree(files.rank_dir(1))
  with pytest.raises(sharded_learner.CheckpointError, match=word):
    _Stub(**stub).prepare(str(tmp_path), 7)


# -- GPU: learners on emulated ranks ----------------------------------------------------
def _deterministic_convs(torch):
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False


def _fill(mem, seed, cap):
  rng = np.random.RandomState(seed)
  pattern = rng.randint(0, 256, size=(257, FRAME)).astype(np.uint8)
  mem._store['observation'] = pattern[np.arange(cap) % 257].reshape(cap, 84, 84)
  mem._store['action'] = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.uint8)
  mem.add_count = cap + 500
  mem.invalid_range = np.array([(500 - HORIZON + i) % cap for i in range(4 + HORIZON)])
  return rng


def _prioritized_shard(seed, cap, unit):
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  mem = prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, BATCH, update_horizon=HORIZON, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  rng = _fill(mem, seed, cap)
  prios = (np.ones(cap) if unit else np.sqrt(np.abs(rng.randn(cap)) + 1e-10))
  mem.set_priority(np.arange(cap, dtype=np.int32), prios.astype(np.float32))
  return mem


def _uniform_shard(seed, cap):
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  mem = crb.OutOfGraphReplayBuffer(
      (84, 84), 4, cap, BATCH, update_horizon=HORIZON, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  _fill(mem, seed, cap)
  return mem


def _learner(kind, rank, data_seed, graph, exchange=None, cap=CAP):
  """Rank `rank` of a learner of `kind`; its shard holds the transitions of
  data_seed + rank."""
  from dopamine_b200.agents.dqn import learner as dqn_learner
  from dopamine_b200.agents.implicit_quantile import learner as iqn_learner
  from dopamine_b200.agents.rainbow import agent
  seed = data_seed + rank
  common = dict(batch_size=BATCH, replay_capacity=cap, seed=3, exchange=exchange,
                cuda_graph=graph)
  if kind == 'dqn':
    return dqn_learner.ShardedDQNLearner(ACTIONS, memory=_uniform_shard(seed, cap),
                                         update_horizon=HORIZON, **common)
  if kind == 'iqn':
    return iqn_learner.ShardedIQNLearner(
        ACTIONS, memory=_prioritized_shard(seed, cap, True), num_tau_samples=8,
        num_tau_prime_samples=8, num_quantile_samples=8, **common)
  return agent.ShardedRainbowLearner(ACTIONS, memory=_prioritized_shard(seed, cap, False),
                                     replay_scheme=kind.split('-')[1], **common)


def _learners(kind, world, data_seed, graph=False, cap=CAP):
  from dopamine_b200.replay_memory import sharded_replay
  xs = sharded_replay.PeerExchange.emulated(world)
  return [_learner(kind, g, data_seed, graph, xs[g], cap) for g in range(world)]


def _publish(learners):
  if learners[0].__class__.__name__ == 'ShardedDQNLearner':
    for phase in (0, 1):  # both publish-ahead rounds of the uniform sampler
      for l in learners:
        l.sharded.publish(l.batch_size, phase)
  else:
    for l in learners:
      l.exchange.publish(l.memory)


def _apply(learner, out):
  if learner.__class__.__name__ == 'ShardedRainbowLearner':
    learner.apply(out)
  else:
    learner.apply()


def _bits(t):
  return t.detach().cpu().contiguous().numpy().tobytes()


def _record(learners, outs):
  """Every rank's loss, slots, indices and per-row output (priorities or losses)."""
  rec = []
  for l, out in zip(learners, outs):
    slots, count, batch = l._sample[:3]
    n = int(count.item())
    rec.append(dict(loss=_bits(l.loss), slots=_bits(slots[:n]), indices=_bits(batch[7][:n]),
                    out=_bits(out[:n])))
  return rec


def _update(torch, learners):
  """One update of every emulated rank, phase by phase; the all-reduce is a sum."""
  _publish(learners)
  for l in learners:
    l.sample()
  outs = [l.loss_backward() for l in learners]
  total = torch.stack([l._flat for l in learners]).sum(0)
  for l, out in zip(learners, outs):
    l._flat.copy_(total)
    _apply(l, out)
  torch.cuda.synchronize()
  return _record(learners, outs)


def _snapshot(learners):
  """Everything a restore writes, per rank, as bytes and ints."""
  snap = []
  for l in learners:
    m = l.memory
    opt = l.optimizer.state_dict()
    s = dict(
        params=[_bits(t) for t in list(l.online.state_dict().values()) +
                list(l.target.state_dict().values())],
        optimizer=[_bits(t) for _, st in sorted(opt['state'].items())
                   for _, t in sorted(st.items())] + [opt.get('step')],
        columns={name: hashlib.sha256(m._read_column(name).tobytes()).hexdigest()
                 for name in m._columns},
        add_count=int(m.add_count), invalid=m.invalid_range.tolist(),
        sampler=m.sampler_state(), exchange=l.exchange.state(),
        counters=(l.training_steps, l.updates))
    if hasattr(m, 'sum_tree'):
      s['tree'] = [a.view(np.uint64).tobytes() for a in m.sum_tree.nodes]
      s['max_recorded'] = m.sum_tree.max_recorded_priority
    if getattr(l, '_generator', None) is not None:
      s['taus'] = _bits(l._generator.get_state())
    snap.append(s)
  return snap


def _assert_same(a, b):
  assert len(a) == len(b)
  for g, (x, y) in enumerate(zip(a, b)):
    assert sorted(x) == sorted(y), g
    for key in x:
      assert x[key] == y[key], (g, key)


@pytest.mark.gpu
@pytest.mark.parametrize('graph', [False, True])
@pytest.mark.parametrize('world', [2, 3])
@pytest.mark.parametrize('kind', KINDS)
def test_restore_continues_bit_for_bit(tmp_path, kind, world, graph):
  """K updates, save, M more recorded; fresh learners over other transitions restore and
  run the same M updates: every rank's losses, slots, indices and priorities (or row
  losses), then every parameter, optimizer tensor, sum-tree node (as uint64 bits), store
  column and counter are identical.  Right after the restore every rank already holds
  exactly the state saved, exchange step number and draw counters included."""
  import torch
  from dopamine_b200.agents import sharded_learner
  _deterministic_convs(torch)
  path = str(tmp_path)
  learners = _learners(kind, world, 100, graph)
  for _ in range(K_UPDATES):
    _update(torch, learners)
  sharded_learner.ShardedLearner.save_ranks(learners, path, 1)
  at_save = _snapshot(learners)
  want = [_update(torch, learners) for _ in range(M_UPDATES)]
  want_end = _snapshot(learners)
  del learners

  fresh = _learners(kind, world, 500, graph)
  _update(torch, fresh)  # (a fresh run that has moved: nothing may survive the restore)
  sharded_learner.ShardedLearner.restore_ranks(fresh, path, 1)
  _assert_same(_snapshot(fresh), at_save)
  got = [_update(torch, fresh) for _ in range(M_UPDATES)]
  for u, (a, b) in enumerate(zip(got, want)):
    for g in range(world):
      for key in a[g]:
        assert a[g][key] == b[g][key], (u, g, key)
  _assert_same(_snapshot(fresh), want_end)
  for l in fresh:
    l.check()


def _capture(torch, learner):
  """The update of one emulated rank as three CUDA graphs: the sampler, loss + backward,
  and the optimizer (+ write-back).  The emulated ranks' samplers must all run before the
  first loss (the sharded C51 loss reads every rank's minimum probability), and the
  all-reduce between the last two stays the caller's."""
  graphs = [torch.cuda.CUDAGraph() for _ in range(3)]
  if getattr(learner, '_generator', None) is not None:
    graphs[0].register_generator_state(learner._generator)
  torch.cuda.synchronize()
  with torch.cuda.graph(graphs[0]):
    learner.sample()
  with torch.cuda.graph(graphs[1]):
    out = learner.loss_backward()
  with torch.cuda.graph(graphs[2]):
    _apply(learner, out)
  torch.cuda.synchronize()
  return graphs, out


def _graph_update(torch, learners, captured):
  _publish(learners)
  for l, (graphs, _) in zip(learners, captured):
    l._flush_replay()
    graphs[0].replay()
  for graphs, _ in captured:
    graphs[1].replay()
  total = torch.stack([l._flat for l in learners]).sum(0)
  for l, (graphs, _) in zip(learners, captured):
    l._flat.copy_(total)
    graphs[2].replay()
  torch.cuda.synchronize()
  return _record(learners, [out for _, out in captured])


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['rainbow-prioritized', 'iqn', 'dqn'])
def test_graphs_captured_before_the_restore_continue_the_run(tmp_path, kind):
  """Learners that captured their update as CUDA graphs BEFORE the restore replay them
  after it: the restore copies into the tensors the graphs read (parameters, optimizer
  state and step count, tau generator, replay, counters), so the replays equal the
  uninterrupted run's updates bit for bit."""
  import torch
  from dopamine_b200.agents import sharded_learner
  _deterministic_convs(torch)
  path = str(tmp_path)
  learners = _learners(kind, 2, 100, graph=True)
  for _ in range(K_UPDATES):
    _update(torch, learners)
  sharded_learner.ShardedLearner.save_ranks(learners, path, 1)
  want = [_update(torch, learners) for _ in range(M_UPDATES)]
  want_end = _snapshot(learners)
  del learners

  fresh = _learners(kind, 2, 500, graph=True)
  for _ in range(K_UPDATES + 1):
    _update(torch, fresh)
  graphs = [_capture(torch, l) for l in fresh]
  sharded_learner.ShardedLearner.restore_ranks(fresh, path, 1)
  got = [_graph_update(torch, fresh, graphs) for _ in range(M_UPDATES)]
  for u, (a, b) in enumerate(zip(got, want)):
    for g in range(2):
      for key in a[g]:
        assert a[g][key] == b[g][key], (u, g, key)
  end = _snapshot(fresh)
  for s in end + want_end:
    s.pop('counters')  # (a replay is not counted by the emulated phases)
  _assert_same(end, want_end)
  for l in fresh:
    l.check()


@pytest.mark.gpu
def test_every_rank_directory_is_a_plain_replay_checkpoint(tmp_path):
  """gzip + np.load read every rank's store files; a fresh buffer's `load` reads the rank
  directory (host path for the sum tree); so does the reference's own prioritized
  buffer where it is importable."""
  import torch
  from oracle import refshim
  from dopamine_b200.agents import sharded_learner
  _deterministic_convs(torch)
  path = str(tmp_path)
  learners = _learners('rainbow-prioritized', 2, 100)
  _update(torch, learners)
  sharded_learner.ShardedLearner.save_ranks(learners, path, 4)
  for g, l in enumerate(learners):
    rank_dir = os.path.join(path, 'rank_{}'.format(g))
    columns = {name: l.memory._read_column(name) for name in l.memory._columns}
    for name, col in columns.items():
      with gzip.open(os.path.join(rank_dir, '{}{}_ckpt.4.gz'.format(STORE, name))) as f:
        assert np.load(f, allow_pickle=False).tobytes() == col.tobytes(), (g, name)
    back = _prioritized_shard(900 + g, CAP, False)
    back.load(rank_dir, 4)
    for name, col in columns.items():
      assert back._read_column(name).tobytes() == col.tobytes(), (g, name)
    for a, b in zip(back.sum_tree.nodes, l.memory.sum_tree.nodes):
      assert a.view(np.uint64).tobytes() == b.view(np.uint64).tobytes()
    if refshim.reference_available():
      _, _, ref_prb = refshim.load_reference()
      ref = ref_prb.OutOfGraphPrioritizedReplayBuffer((84, 84), 4, CAP, 8,
                                                      update_horizon=HORIZON)
      ref.load(rank_dir, '4')
      for name, col in columns.items():
        assert ref._store[name].tobytes() == col.tobytes(), (g, name)
      assert int(ref.add_count) == int(l.memory.add_count)


def _corrupt(path):
  """Flips bytes in the middle of rank 1's observation file (CRC-32 no longer matches)."""
  name = os.path.join(path, 'rank_1', '{}observation_ckpt.1.gz'.format(STORE))
  with open(name, 'r+b') as f:
    f.seek(os.path.getsize(name) // 2)
    chunk = bytearray(f.read(16))
    f.seek(os.path.getsize(name) // 2)
    f.write(bytes(b ^ 0x5a for b in chunk))


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['missing_rank', 'no_sentinel', 'world', 'capacity',
                                  'kind', 'corrupt_shard'])
def test_a_refused_restore_changes_nothing(tmp_path, case):
  """Each refusal raises before any rank is written: columns, sum trees, parameters,
  optimizer state and counters of every target rank are as they were.  A corrupted shard
  file on rank 1 is found by the device verify pass while rank 0's shard is fine."""
  import torch
  from dopamine_b200.agents import sharded_learner
  _deterministic_convs(torch)
  path = str(tmp_path)
  saved = _learners('rainbow-prioritized', 2, 100)
  _update(torch, saved)
  sharded_learner.ShardedLearner.save_ranks(saved, path, 1)
  del saved
  files = sharded_learner._Files(path, 1)
  world, cap, kind = 2, CAP, 'rainbow-prioritized'
  if case == 'missing_rank':
    shutil.rmtree(files.rank_dir(1))
  elif case == 'no_sentinel':
    os.remove(files.sentinel)
  elif case == 'world':
    world = 3
  elif case == 'capacity':
    cap = CAP // 2
  elif case == 'kind':
    kind = 'rainbow-uniform'
  else:
    _corrupt(path)
  targets = _learners(kind, world, 500, cap=cap)
  _update(torch, targets)
  before = _snapshot(targets)
  with pytest.raises((sharded_learner.CheckpointError, gzip.BadGzipFile)):
    sharded_learner.ShardedLearner.restore_ranks(targets, path, 1)
  _assert_same(_snapshot(targets), before)
  _update(torch, targets)  # (the exchange still works)
  for l in targets:
    l.check()


# -- GPU: single-GPU agent -------------------------------------------------------------
def _constant_memory(cap):
  """Every transition alike: a batch does not depend on which rows are drawn, so two
  agents' updates differ only through their networks and optimizers."""
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  mem = prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, 32, update_horizon=1, gamma=0.99, output='torch', rng='device',
      seed=0, reuse_outputs=True)
  frame = np.random.RandomState(1).randint(0, 256, size=(84, 84)).astype(np.uint8)
  mem._store['observation'] = np.broadcast_to(frame, (cap, 84, 84)).copy()
  mem._store['action'] = np.full(cap, 2, np.int32)
  mem._store['reward'] = np.full(cap, 0.5, np.float32)
  mem._store['terminal'] = np.zeros(cap, np.uint8)
  mem.add_count = cap + 10
  mem.invalid_range = np.array([(10 - 1 + i) % cap for i in range(5)])
  mem.set_priority(np.arange(cap, dtype=np.int32), np.ones(cap, np.float32))
  return mem


@pytest.mark.gpu
@pytest.mark.parametrize('graph', [False, True])
def test_unbundled_rainbow_agent_resumes_adam(tmp_path, graph):
  """A single-GPU RainbowAgent bundled after K updates and unbundled into a fresh agent
  continues with the uninterrupted agent's parameters over M updates: Adam's bias
  correction resumes at t = K + 1, not at t = 1."""
  import torch
  from dopamine_b200.agents.rainbow import agent
  _deterministic_convs(torch)
  make = lambda: agent.RainbowAgent(
      num_actions=ACTIONS, replay_scheme='uniform', replay_capacity=500, batch_size=32,
      memory=_constant_memory(500), seed=2, cuda_graph=graph)
  first = make()
  for _ in range(K_UPDATES + 3):
    first.train_step()
  bundle = first.bundle_and_checkpoint(str(tmp_path), 1)
  for _ in range(M_UPDATES):
    first.train_step()
  second = make()
  if graph:  # captured before the unbundle, which then copies into what it reads
    second.train_step()
  assert second.unbundle(str(tmp_path), 1, bundle)
  for _ in range(M_UPDATES):
    second.train_step()
  torch.cuda.synchronize()
  for p, q in zip(first.online.parameters(), second.online.parameters()):
    assert _bits(p) == _bits(q)


# -- GPU: real processes -----------------------------------------------------------------
def _free_port():
  with socket.socket() as s:
    s.bind(('127.0.0.1', 0))
    return s.getsockname()[1]


def _process_worker(rank, world, port, out_dir, phase):
  """phase 'save': K updates, save, M updates recorded; phase 'restore': a fresh learner
  over other transitions restores and runs M updates recorded."""
  import pickle
  import torch
  import torch.distributed as dist
  from dopamine_b200.agents.rainbow import agent
  torch.cuda.set_device(rank)
  _deterministic_convs(torch)
  os.environ['MASTER_ADDR'] = '127.0.0.1'
  os.environ['MASTER_PORT'] = str(port)
  dist.init_process_group('nccl', rank=rank, world_size=world,
                          device_id=torch.device('cuda', rank))
  try:
    data_seed = 100 if phase == 'save' else 500
    learner = agent.ShardedRainbowLearner(
        ACTIONS, batch_size=BATCH, memory=_prioritized_shard(data_seed + rank, CAP, False),
        replay_capacity=CAP, seed=3)
    if phase == 'save':
      for _ in range(K_UPDATES):
        learner.train_step()
      learner.save(os.path.join(out_dir, 'ckpt'), 1)
    else:
      learner.train_step()
      learner.restore(os.path.join(out_dir, 'ckpt'), 1)
    records = []
    for _ in range(M_UPDATES):
      learner.train_step()
      torch.cuda.synchronize()
      slots, count, batch, _ = learner._sample
      n = int(count.item())
      records.append(dict(loss=_bits(learner.loss), slots=_bits(slots[:n]),
                          indices=_bits(batch[7][:n])))
    learner.check()
    with open(os.path.join(out_dir, '{}{}.pkl'.format(phase, rank)), 'wb') as f:
      pickle.dump(dict(records=records, params=[_bits(p) for p in learner.online.parameters()]),
                  f)
    dist.barrier()
  finally:
    dist.destroy_process_group()


def _run_processes(world, args, timeout=900):
  import torch.multiprocessing as mp
  ctx = mp.get_context('spawn')
  procs = [ctx.Process(target=_process_worker, args=(r, world) + args) for r in range(world)]
  for p in procs:
    p.start()
  for p in procs:
    p.join(timeout=timeout)
  alive = [p for p in procs if p.is_alive()]
  for p in alive:
    p.terminate()
    p.join(timeout=60)
  assert not alive, 'a rank did not finish'
  assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]


@pytest.mark.gpu
def test_two_processes_save_and_restore_like_the_emulated_ranks(tmp_path):
  """Two processes save after K updates and run M more; two NEW processes over other
  transitions restore and run the same M: their records and parameters equal the first
  pair's and those of the same ranks emulated on one device (saved and restored the same
  way)."""
  import pickle
  import torch
  from dopamine_b200.agents import sharded_learner
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs')
  out = str(tmp_path)
  os.makedirs(os.path.join(out, 'ckpt'))
  _run_processes(2, (_free_port(), out, 'save'))
  _run_processes(2, (_free_port(), out, 'restore'))
  load = lambda name: pickle.load(open(os.path.join(out, name), 'rb'))
  _deterministic_convs(torch)
  learners = _learners('rainbow-prioritized', 2, 100)
  for _ in range(K_UPDATES):
    _update(torch, learners)
  sharded_learner.ShardedLearner.save_ranks(learners, os.path.join(out, 'emulated'), 1)
  want = [_update(torch, learners) for _ in range(M_UPDATES)]
  for g in range(2):
    saved, restored = load('save{}.pkl'.format(g)), load('restore{}.pkl'.format(g))
    assert saved['params'] == restored['params'], g
    for u in range(M_UPDATES):
      a, b = saved['records'][u], restored['records'][u]
      assert a == b, (g, u)
      assert a['slots'] == want[u][g]['slots'] and a['indices'] == want[u][g]['indices']
      np.testing.assert_allclose(np.frombuffer(a['loss'], np.float32),
                                 np.frombuffer(want[u][g]['loss'], np.float32), rtol=1e-5)
