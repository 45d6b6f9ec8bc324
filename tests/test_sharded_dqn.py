"""The data-parallel DQN learner on a sharded global uniform batch (ShardedDQNLearner,
b2r_sample_transition_batch_uniform_sharded_device, b2r_dqn_loss_sharded).  CPU tests
check the host-side validation, the oracle's rule and a numpy model of the sampler's
second round; the GPU tests (`pytest -m gpu`) check that the ranks' rows are the oracle's
global batch, that a shard's loss and gradients are the global batch's, with ranks
emulated on one device, in one real process (eager against graph) and with two real
processes."""
import ctypes
import os
import re
import socket

import numpy as np
import pytest

from dopamine_b200 import _native
from oracle import dqn_port
from oracle import philox_port
from oracle import replay_port
from oracle import sharded_uniform_port

FRAME = 84 * 84
ACTIONS = 18
CAP = 4000
FILLS = (4000, 3000, 2000, 3500)  # transitions per shard: spans off the even split
STACK, HORIZON = 4, 3
GAMMA_N = 0.99 ** HORIZON
SEED = 5
ATTEMPTS = 1000  # the reference's max_sample_attempts
LIST_WORDS = 1024  # the rejection list a shard can publish


# -- CPU: validation before any device work ------------------------------------------
def test_sharded_dqn_loss_refuses_bad_arguments_without_a_device():
  lib = _native.lib()
  args = _native.DqnArgs()
  args.batch, args.num_actions = 32, ACTIONS
  status = lib.b2r_dqn_loss_sharded(None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'args' in _native.last_error()
  status = lib.b2r_dqn_loss_sharded(ctypes.byref(args), 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'batch_count' in _native.last_error()
  count = np.zeros(1, dtype=np.int32)
  args.batch_count = count.ctypes.data
  status = lib.b2r_dqn_loss_sharded(ctypes.byref(args), 0, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'global_batch' in _native.last_error()
  # then the checks of b2r_dqn_loss, still before any device work
  status = lib.b2r_dqn_loss_sharded(ctypes.byref(args), 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'pointer' in _native.last_error()


def test_uniform_sharded_sampler_refuses_bad_arguments_without_a_device():
  lib = _native.lib()
  fn = lib.b2r_sample_transition_batch_uniform_sharded_device
  # stand-ins for a buffer and an exchange: none of these refusals looks at them
  fake_buf, fake_x = np.zeros(64, np.uint8), np.zeros(64, np.uint8)
  buf, x = fake_buf.ctypes.data, fake_x.ctypes.data
  indices, slots, count = (np.zeros(4, np.int32), np.zeros(4, np.int32),
                           np.zeros(1, np.int32))
  out = _native.Batch()
  out.indices = indices.ctypes.data
  ok = dict(b=buf, x=x, global_batch=64, out=ctypes.byref(out), slots=slots.ctypes.data,
            count=count.ctypes.data, max_rows=0)
  cases = [(dict(b=None), 'buffer'), (dict(x=None), 'exchange'), (dict(out=None), 'out'),
           (dict(slots=None), 'out_slots'), (dict(count=None), 'out_count'),
           (dict(max_rows=-1), 'max_rows'), (dict(global_batch=0), 'global_batch')]
  for change, word in cases:
    a = dict(ok, **change)
    status = fn(a['b'], a['x'], a['global_batch'], SEED, 0, a['out'], a['slots'],
                a['count'], a['max_rows'], None)
    assert status == _native.ERR_INVALID_ARGUMENT, (change, status)
    assert word in _native.last_error(), (change, _native.last_error())
  empty = _native.Batch()
  status = fn(buf, x, 64, SEED, 0, ctypes.byref(empty), slots.ctypes.data,
              count.ctypes.data, 0, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'indices' in _native.last_error()
  publish = lib.b2r_exchange_publish_uniform_device
  assert publish(None, buf, 64, SEED, 0, 0, None) == _native.ERR_INVALID_ARGUMENT
  assert 'exchange' in _native.last_error()
  assert publish(x, None, 64, SEED, 0, 0, None) == _native.ERR_INVALID_ARGUMENT
  assert 'buffer' in _native.last_error()
  assert publish(x, buf, 0, SEED, 0, 0, None) == _native.ERR_INVALID_ARGUMENT
  assert 'global_batch' in _native.last_error()


def test_sharded_dqn_learner_refuses_ddp_and_a_missing_process_group():
  import torch.distributed as dist
  from dopamine_b200.agents.dqn import learner
  with pytest.raises(ValueError, match='ddp=False'):
    learner.ShardedDQNLearner(ACTIONS, ddp=True)
  assert not (dist.is_available() and dist.is_initialized())
  with pytest.raises(RuntimeError, match='torch.distributed'):
    learner.ShardedDQNLearner(ACTIONS)


# -- CPU: the rule --------------------------------------------------------------------
def _port_shard(terminal, fill, capacity=CAP, max_attempts=ATTEMPTS):
  """A PortReplay shard whose validity is that of `fill` transitions with these
  terminals (frames are irrelevant to the index rule)."""
  port = replay_port.PortReplay((1, 1), STACK, capacity, 32, update_horizon=HORIZON,
                                max_sample_attempts=max_attempts)
  port.store['terminal'][:] = terminal
  if fill < capacity:
    port.add_count = np.array(fill)
    port.invalid_range = replay_port.cursor_window(fill, capacity, STACK, HORIZON)
  else:
    port.add_count = np.array(capacity + 1000)
    port.invalid_range = replay_port.cursor_window(1000, capacity, STACK, HORIZON)
  return port


class _Candidates(object):
  """np.random stand-in: randint(lo, hi) gives lo + the device's offset of uniform j."""

  def __init__(self, uniforms):
    self.uniforms, self.j = uniforms, 0

  def randint(self, lo, hi):
    u = self.uniforms[self.j]
    self.j += 1
    return lo + min(int(np.float64(u) * np.float64(hi - lo)), hi - lo - 1)


@pytest.mark.parametrize('fill,density,attempts', [(CAP, 0.01, ATTEMPTS),
                                                   (2500, 0.01, ATTEMPTS), (CAP, 0.6, 20),
                                                   (300, 0.3, 50)])
def test_oracle_rule_with_one_shard_is_the_reference_sampler(fill, density, attempts):
  """G = 1: the sharded rule is the reference's uniform sample_index_batch fed the same
  candidates, including a run that exhausts its attempts."""
  rng = np.random.RandomState(fill)
  terminal = (rng.rand(CAP) < density).astype(np.uint8)
  uniforms = [philox_port.uniform53(SEED, 3, j) for j in range(256 + attempts)]
  port = _port_shard(terminal, fill, max_attempts=attempts)
  port.np_rng = _Candidates(uniforms)
  try:
    want = port.sample_index_batch(256)
  except RuntimeError as e:
    with pytest.raises(RuntimeError, match='Max sample attempts') as got:
      sharded_uniform_port.sharded_uniform_sample([port], uniforms, 256,
                                                  attempts)
    assert str(got.value) == str(e)
    return
  rows = sharded_uniform_port.sharded_uniform_sample([port], uniforms, 256,
                                                     attempts)
  assert rows[0][0] == list(range(256))
  assert [int(i) for i in rows[0][1]] == [int(i) for i in want]


def _sequential(owner, valid, batch, attempts, world):
  """The reference's loop over draws with known owners and validity: per rank its
  (global rows, draw numbers), and the number accepted."""
  rows = [([], []) for _ in range(world)]
  accepted = rejected = j = 0
  while accepted < batch and rejected < attempts:
    if valid[j]:
      rows[owner[j]][0].append(accepted)
      rows[owner[j]][1].append(j)
      accepted += 1
    else:
      rejected += 1
    j += 1
  return rows, accepted


def _two_rounds(owner, valid, batch, attempts, world):
  """What the sampling kernel does: every rank walks its own draws of the window
  [0, batch + attempts), stopping at `batch` valid or `attempts` invalid ones, and
  publishes the first `attempts` ordinals of its invalid draws; then each rank keeps
  its valid draws j with j - rejects_before(j) < batch and rejects_before(j) <
  attempts, rejects_before by binary search over the G lists."""
  window = batch + attempts
  lists, mine = [], []
  for g in range(world):
    rej, ok = [], []
    for j in range(window):
      if len(rej) >= attempts or len(ok) >= batch:
        break
      if owner[j] == g:
        (ok if valid[j] else rej).append(j)
    lists.append(np.array(rej[:attempts], dtype=np.int64))
    mine.append(ok[:batch])
  before = lambda j: sum(int(np.searchsorted(l, j, side='left')) for l in lists)
  rows = []
  for g in range(world):
    got = ([], [])
    for j in mine[g]:
      rb = before(j)
      if j - rb < batch and rb < attempts:
        got[0].append(j - rb)
        got[1].append(j)
      else:
        break  # (a prefix: both quantities only grow with j)
    rows.append(got)
  accepted = batch
  if sum(len(l) for l in lists) >= attempts:
    lo, hi = 0, window
    while lo < hi:
      mid = (lo + hi) // 2
      if before(mid) >= attempts:
        hi = mid
      else:
        lo = mid + 1
    if before(lo) >= attempts:
      accepted = min(accepted, lo - attempts)
  return rows, accepted


def test_two_round_model_matches_the_sequential_loop():
  """Thousands of random validity patterns and spans — zero spans, exhausted attempts,
  lists truncated exactly at the cutoff: each rank's rows and the accepted count of the
  two-round protocol equal the plain loop's."""
  rng = np.random.RandomState(0)
  exhausted = at_cutoff = zero_span = 0
  for trial in range(3000):
    world = int(rng.randint(1, 6))
    batch = int(rng.randint(1, 40))
    attempts = int(rng.randint(0, 12))
    spans = rng.randint(0, 4, size=world)
    if spans.sum() == 0:
      spans[rng.randint(world)] = 1
    zero_span += int((spans == 0).any())
    window = batch + attempts
    owner = rng.choice(world, size=window, p=spans / spans.sum())
    valid = rng.rand(window) >= rng.choice([0.0, 0.05, 0.3, 0.7, 1.0])
    if trial % 7 == 0 and attempts:
      # the attempts-th rejection is the last draw before the batch would be full (odd
      # trials) or the draw after it fills (even): exhausted by one row, or not at all
      last = batch + attempts - (2 if trial % 2 else 1)
      valid[:] = True
      valid[rng.choice(last, size=attempts - 1, replace=False)] = False
      valid[last] = False
    want, accepted = _sequential(owner, valid, batch, attempts, world)
    got, got_accepted = _two_rounds(owner, valid, batch, attempts, world)
    assert got_accepted == accepted, trial
    for g in range(world):
      assert got[g][0] == want[g][0] and got[g][1] == want[g][1], (trial, g)
    exhausted += int(accepted < batch)
    at_cutoff += int(accepted < batch and int((~valid).sum()) == attempts)
  assert exhausted > 100 and at_cutoff > 10 and zero_span > 100


# -- GPU ------------------------------------------------------------------------------
def _shard_data(seed, fill, density=0.01):
  rng = np.random.RandomState(seed)
  pattern = rng.randint(0, 256, size=(257, FRAME)).astype(np.uint8)
  return dict(
      observation=pattern[np.arange(CAP) % 257].reshape(CAP, 84, 84),
      action=rng.randint(0, ACTIONS, size=CAP).astype(np.int32),
      reward=np.clip(rng.randn(CAP), -1, 1).astype(np.float32),
      terminal=(rng.rand(CAP) < density).astype(np.uint8), fill=fill)


def _device_shard(data, batch, max_attempts=ATTEMPTS):
  """A uniform shard (DQN's replay) holding the seeded transitions of `data`."""
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  mem = crb.OutOfGraphReplayBuffer(
      (84, 84), STACK, CAP, batch, update_horizon=HORIZON, gamma=0.99,
      max_sample_attempts=max_attempts, output='torch', rng='device', seed=1,
      reuse_outputs=True)
  for name in ('observation', 'action', 'reward', 'terminal'):
    mem._store[name] = data[name]
  fill = data['fill']
  if fill < CAP:
    mem.add_count = fill
    mem.invalid_range = crb.invalid_range(fill, CAP, STACK, HORIZON)
  else:
    mem.add_count = CAP + 1000
    mem.invalid_range = crb.invalid_range(1000, CAP, STACK, HORIZON)
  return mem


def _uniform_shards(world, global_batch, fills, density=0.01, max_attempts=ATTEMPTS):
  from dopamine_b200.replay_memory import sharded_replay
  xs = sharded_replay.PeerExchange.emulated(world)
  data = [_shard_data(100 + g, fills[g], density) for g in range(world)]
  mems = [_device_shard(d, global_batch, max_attempts) for d in data]
  ports = [_port_shard(d['terminal'], d['fill'], max_attempts=max_attempts) for d in data]
  shards = [sharded_replay.ShardedUniformReplay(m, g, world, SEED, xs[g])
            for g, m in enumerate(mems)]
  return xs, mems, ports, shards


def _emulated_sample(torch, shards, global_batch):
  """Publish-ahead of both rounds on every rank (a launch cannot wait for a rank
  emulated after it), then every rank's sampler."""
  for phase in (0, 1):
    for s in shards:
      s.publish(global_batch, phase)
  outs = [s.sample_transition_batch_sharded(global_batch) for s in shards]
  torch.cuda.synchronize()
  return outs


def _oracle(ports, step, global_batch, max_attempts=ATTEMPTS):
  uniforms = [philox_port.uniform53(SEED, step, j)
              for j in range(global_batch + max_attempts)]
  return sharded_uniform_port.sharded_uniform_sample(ports, uniforms, global_batch,
                                                     max_attempts)


@pytest.mark.gpu
@pytest.mark.parametrize('global_batch', [64, 512])
@pytest.mark.parametrize('world', [2, 4])
def test_emulated_ranks_sample_the_oracle_batch(world, global_batch):
  """Two consecutive steps over shards of different fill levels (1 % terminals, so a
  few per cent of the draws are rejected): each rank's slots and indices are the
  oracle's bit for bit, the slots partition range(global_batch), and the gathered
  columns are the buffer's own gather of those indices."""
  import torch
  _, mems, ports, shards = _uniform_shards(world, global_batch, FILLS)
  for step in (1, 2):
    outs = _emulated_sample(torch, shards, global_batch)
    want = _oracle(ports, step, global_batch)
    counts = [int(o[1].item()) for o in outs]
    assert sum(counts) == global_batch
    assert counts != [global_batch // world] * world, 'the shares should be uneven'
    slots = []
    for g, ((s, count, batch), (w_slots, w_idx)) in enumerate(zip(outs, want)):
      n = counts[g]
      got = [t[:n].clone() for t in batch]
      slots.append(s[:n].cpu().numpy())
      assert slots[g].tolist() == w_slots, (step, g)
      assert got[7].cpu().numpy().tolist() == [int(i) for i in w_idx], (step, g)
      ref = mems[g].sample_transition_batch(batch_size=n, indices=got[7].cpu().numpy())
      for k in range(8):
        assert torch.equal(got[k], ref[k]), (step, g, k)
    assert np.array_equal(np.sort(np.concatenate(slots)), np.arange(global_batch))
  for s in shards:
    s.check()


@pytest.mark.gpu
def test_a_shard_with_span_zero_owns_no_draw():
  import torch
  _, _, ports, shards = _uniform_shards(2, 64, (CAP, 5))  # 5 < stack + horizon + 1
  outs = _emulated_sample(torch, shards, 64)
  want = _oracle(ports, 1, 64)
  assert int(outs[1][1].item()) == 0 and want[1] == ([], [])
  assert outs[0][0][:64].cpu().numpy().tolist() == list(range(64))
  assert outs[0][2][7][:64].cpu().numpy().tolist() == [int(i) for i in want[0][1]]
  for s in shards:
    s.check()


@pytest.mark.gpu
def test_too_few_transitions_everywhere_is_latched_on_every_rank():
  import torch
  _, _, ports, shards = _uniform_shards(2, 64, (5, 6))
  outs = _emulated_sample(torch, shards, 64)
  with pytest.raises(RuntimeError, match='Cannot sample'):
    _oracle(ports, 1, 64)
  for s, o in zip(shards, outs):
    assert int(o[1].item()) == 0
    with pytest.raises(_native.NativeError) as e:
      s.check()
    assert e.value.code == _native.ERR_TOO_FEW_TRANSITIONS


@pytest.mark.gpu
def test_exhausted_attempts_are_latched_on_every_rank_alike():
  """Dense terminals and max_sample_attempts 20: the oracle raises, and every rank
  latches B2R_ERR_SAMPLE_ATTEMPTS with the oracle's accepted count."""
  import torch
  _, _, ports, shards = _uniform_shards(3, 64, (CAP, 3000, 2000), density=0.5,
                                        max_attempts=20)
  _emulated_sample(torch, shards, 64)
  with pytest.raises(RuntimeError, match='Max sample attempts') as want:
    _oracle(ports, 1, 64, max_attempts=20)
  accepted = re.search(r'only sampled (\d+)', str(want.value)).group(1)
  for s in shards:
    with pytest.raises(_native.NativeError) as e:
      s.check()
    assert e.value.code == _native.ERR_SAMPLE_ATTEMPTS
    assert re.search(r'only sampled (\d+)', str(e.value)).group(1) == accepted


@pytest.mark.gpu
def test_a_peer_that_never_publishes_is_latched():
  import torch
  xs, _, _, shards = _uniform_shards(2, 64, (CAP, CAP))
  _native.check(_native.lib().b2r_exchange_set_timeout(xs[0]._h, 0.05))
  shards[0].sample_transition_batch_sharded(64)  # rank 1 never runs
  torch.cuda.synchronize()
  with pytest.raises(_native.NativeError) as e:
    shards[0].check()
  assert e.value.code == _native.ERR_EXCHANGE


@pytest.mark.gpu
def test_refusals_that_need_a_buffer_come_before_any_device_work():
  """max_sample_attempts above the 1024 ordinals a rank can publish, and an exchange with
  early publish on, are refused by the sampler and the publish-ahead before a launch."""
  import torch
  lib = _native.lib()
  xs, mems, _, shards = _uniform_shards(2, 64, (CAP, CAP), max_attempts=LIST_WORDS + 1)
  torch.cuda.synchronize()
  before = lib.b2r_launch_count()
  with pytest.raises(_native.NativeError, match='max_sample_attempts') as e:
    shards[0].sample_transition_batch_sharded(64)
  assert e.value.code == _native.ERR_UNSUPPORTED
  with pytest.raises(_native.NativeError, match='max_sample_attempts'):
    shards[0].publish(64, 0)
  assert lib.b2r_launch_count() == before
  _, mems, _, shards = _uniform_shards(2, 64, (CAP, CAP))
  shards[0].exchange.set_early_publish(True)
  torch.cuda.synchronize()
  before = lib.b2r_launch_count()
  with pytest.raises(_native.NativeError, match='early publish') as e:
    shards[0].sample_transition_batch_sharded(64)
  assert e.value.code == _native.ERR_INVALID_ARGUMENT
  with pytest.raises(_native.NativeError, match='early publish'):
    shards[0].publish(64, 1)
  assert lib.b2r_launch_count() == before


def _deterministic_convs(torch):
  """fp32 convolutions with a fixed algorithm: the comparisons below are between
  networks run on different row counts."""
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False


def _learner(global_batch, rank, **kwargs):
  from dopamine_b200.agents.dqn import learner
  memory = _device_shard(_shard_data(100 + rank, FILLS[rank]), global_batch)
  return learner.ShardedDQNLearner(
      ACTIONS, batch_size=global_batch, memory=memory, replay_capacity=CAP,
      update_horizon=HORIZON, gamma=0.99, seed=3, **kwargs)


def _emulated_learners(world, global_batch, graph=False):
  from dopamine_b200.replay_memory import sharded_replay
  xs = sharded_replay.PeerExchange.emulated(world)
  return xs, [_learner(global_batch, g, exchange=xs[g], cuda_graph=graph)
              for g in range(world)]


def _emulated_learner_sample(learners):
  for phase in (0, 1):
    for l in learners:
      l.sharded.publish(l.batch_size, phase)
  return [l.sample() for l in learners]


def _emulated_update(torch, learners):
  """One update of every emulated rank, phase by phase; the all-reduce is a sum."""
  _emulated_learner_sample(learners)
  for l in learners:
    l.loss_backward()
  total = torch.stack([l._flat for l in learners]).sum(0)
  for l in learners:
    l._flat.copy_(total)
    l.apply()
  torch.cuda.synchronize()


def _bits(x):
  return x.cpu().numpy().view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize('global_batch', [64, 512])
@pytest.mark.parametrize('world', [2, 4])
def test_shards_compute_the_global_batch_update(world, global_batch):
  """Every emulated rank samples its share, then computes its loss.  Ordering the ranks'
  rows by slot gives the global batch; the unsharded DQN loss on it with the same network
  outputs is the reference: per-row loss, target and gradient rows are bit-identical,
  padded gradient rows (NaN beforehand) are exact zeros, and the partial means sum to the
  global mean and to the oracle's within 1e-6.  The ranks' parameter gradients sum to the
  unsharded backward's; poisoning padded frames changes no gradient."""
  import torch
  from dopamine_b200.agents.dqn import dqn_agent
  _deterministic_convs(torch)
  _, learners = _emulated_learners(world, global_batch)
  online_net, target_net = learners[0].online, learners[0].target
  for l in learners[1:]:
    for p, q in zip(l.online.parameters(), online_net.parameters()):
      assert torch.equal(p, q)
  samples = _emulated_learner_sample(learners)
  torch.cuda.synchronize()
  counts = [int(s[1].item()) for s in samples]
  slots = [s[0][:n].cpu().numpy() for s, n in zip(samples, counts)]
  assert sum(counts) == global_batch
  assert np.array_equal(np.sort(np.concatenate(slots)), np.arange(global_batch))
  max_rows = learners[0].max_rows
  assert max(counts) <= max_rows

  cols = {}
  order = torch.as_tensor(np.argsort(np.concatenate(slots)), device='cuda')
  for k, name in ((0, 'state'), (1, 'action'), (2, 'reward'), (3, 'next_state'),
                  (6, 'terminal')):
    whole = torch.cat([s[2][k][:n] for s, n in zip(samples, counts)])
    cols[name] = whole[order].contiguous()
  with torch.no_grad():
    online = online_net(cols['state'])
    target = target_net(cols['next_state'])
  ref = dqn_agent.dqn_loss(online, target, cols['action'], cols['reward'],
                           cols['terminal'], GAMMA_N, want_target=True, want_grad=True)
  host = lambda x: x.cpu().numpy()
  oracle = dqn_port.dqn_update(host(cols['reward']), host(cols['terminal']),
                               host(cols['action']), host(online), host(target),
                               gamma=0.99, update_horizon=HORIZON)

  mean_sum = 0.
  rng = np.random.RandomState(0)
  for g, (s, n) in enumerate(zip(samples, counts)):
    slot_idx = torch.as_tensor(slots[g].astype(np.int64), device='cuda')
    local = {}
    for name, whole in (('online', online), ('target', target)):
      t = torch.as_tensor(rng.randn(max_rows, ACTIONS).astype(np.float32), device='cuda')
      t[:n] = whole[slot_idx]
      local[name] = t
    out = dict(loss=torch.full((max_rows,), np.nan, device='cuda'),
               mean_loss=torch.empty((), device='cuda'),
               target=torch.full((max_rows,), np.nan, device='cuda'),
               grad_q=torch.full((max_rows, ACTIONS), np.nan, device='cuda'))
    batch = s[2]
    dqn_agent.dqn_loss(local['online'], local['target'], batch[1], batch[2], batch[6],
                       GAMMA_N, out=out, sharded=(global_batch, s[1]))
    torch.cuda.synchronize()
    mean_sum += float(out['mean_loss'])
    assert np.array_equal(_bits(out['loss'][:n]), _bits(ref['loss'][slot_idx])), g
    assert np.array_equal(_bits(out['target'][:n]), _bits(ref['target'][slot_idx])), g
    assert np.array_equal(_bits(out['grad_q'][:n]), _bits(ref['grad_q'][slot_idx])), g
    assert np.array_equal(_bits(out['loss'][n:]), np.zeros(max_rows - n, np.uint32))
    assert np.array_equal(_bits(out['grad_q'][n:]),
                          np.zeros((max_rows - n, ACTIONS), np.uint32)), g
    np.testing.assert_allclose(host(out['loss'][:n]), oracle['loss'][slots[g]],
                               rtol=1e-6, atol=1e-7)
  np.testing.assert_allclose(mean_sum, float(ref['mean_loss']), rtol=1e-6)
  np.testing.assert_allclose(mean_sum, float(oracle['mean_loss']), rtol=1e-6)

  # parameter gradients through the learner's phases
  partial = []
  for l in learners:
    l.loss_backward()
    partial.append(l._flat.clone())
  torch.cuda.synchronize()
  total = torch.stack(partial).sum(0)
  learners[0]._flat.zero_()
  mean, _ = dqn_agent.DQNLoss.apply(online_net(cols['state']), target, cols['action'],
                                    cols['reward'], cols['terminal'], GAMMA_N)
  mean.backward()
  want = learners[0]._flat[:-1]
  scale = float(want.abs().max())
  # (the batch-size dependent reduction order of cuDNN / cuBLAS backward and the
  # G-way sum: fp32 reassociation over <= 512 rows and 3136-wide layers)
  torch.testing.assert_close(total[:-1], want, rtol=1e-4, atol=1e-5 * scale)
  np.testing.assert_allclose(float(total[-1]), float(ref['mean_loss']), rtol=1e-6)

  # poisoned padded rows change no gradient
  for g, (l, s, n) in enumerate(zip(learners, samples, counts)):
    if n == max_rows:
      continue
    s[2][0][n:] = 255
    s[2][3][n:] = 0
    l.loss_backward()
    torch.cuda.synchronize()
    assert torch.equal(l._flat, partial[g]), g
  for l in learners:
    l.check()


def _free_port():
  with socket.socket() as s:
    s.bind(('127.0.0.1', 0))
    return s.getsockname()[1]


K_UPDATES = 3
WARMUP = 3  # the eager updates a graph-mode learner runs before its capture


def _record(learner):
  slots, count, batch = learner._sample
  n = int(count.item())
  return dict(slots=slots[:n].cpu().numpy(), indices=batch[7][:n].cpu().numpy(),
              loss=float(learner.loss.item()))


def _init_process_group(rank, world, port):
  import torch
  import torch.distributed as dist
  torch.cuda.set_device(rank)
  _deterministic_convs(torch)
  os.environ['MASTER_ADDR'] = '127.0.0.1'
  os.environ['MASTER_PORT'] = str(port)
  dist.init_process_group('nccl', rank=rank, world_size=world,
                          device_id=torch.device('cuda', rank))


def _single_process_worker(rank, port, out_dir):
  import torch
  import torch.distributed as dist
  _init_process_group(rank, 1, port)
  try:
    records = {}
    for graph in (False, True):
      learner = _learner(64, 0, cuda_graph=graph)
      records[graph] = []
      for _ in range(K_UPDATES + (0 if graph else WARMUP)):
        learner.train_step()
        torch.cuda.synchronize()
        records[graph].append(_record(learner))
      learner.check()
      learner.sync_target()
    np.save(os.path.join(out_dir, 'records.npy'), np.array([records], dtype=object),
            allow_pickle=True)
  finally:
    dist.destroy_process_group()


def _run_processes(target, world, args, timeout=900):
  import torch.multiprocessing as mp
  ctx = mp.get_context('spawn')
  procs = [ctx.Process(target=target, args=(r,) + args) for r in range(world)]
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
def test_one_process_graph_replays_the_eager_update(tmp_path):
  """A world-size-1 NCCL group: K updates replayed as a CUDA graph sample the same
  slots and indices as the eager updates after the graph's warm-up, losses within 1e-5;
  consecutive replays draw different batches, and nothing is latched."""
  _run_processes(_single_process_worker, 1, (_free_port(), str(tmp_path)))
  records = np.load(os.path.join(tmp_path, 'records.npy'), allow_pickle=True)[0]
  eager, graph = records[False][WARMUP:], records[True]
  for u, (a, b) in enumerate(zip(graph, eager)):
    assert np.array_equal(a['slots'], b['slots']), u
    assert np.array_equal(a['indices'], b['indices']), u
    np.testing.assert_allclose(a['loss'], b['loss'], rtol=1e-5)
  for a, b in zip(graph, graph[1:]):
    assert not np.array_equal(a['indices'], b['indices'])


def _two_process_worker(rank, world, port, out_dir, graph):
  import torch
  import torch.distributed as dist
  _init_process_group(rank, world, port)
  try:
    learner = _learner(64, rank, cuda_graph=graph)
    records = []
    for _ in range(K_UPDATES):
      learner.train_step()
      torch.cuda.synchronize()
      records.append(_record(learner))
    learner.sync_target()  # (checks the latched status)
    flat = torch.cat([p.detach().reshape(-1) for p in learner.online.parameters()])
    np.save(os.path.join(out_dir, 'params{}.npy'.format(rank)), flat.cpu().numpy())
    np.save(os.path.join(out_dir, 'records{}.npy'.format(rank)),
            np.array(records, dtype=object), allow_pickle=True)
    dist.barrier()
  finally:
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize('graph', [False, True])
def test_two_processes_match_the_emulated_ranks(tmp_path, graph):
  """Two real processes (NCCL all-reduce, CUDA-IPC mailboxes) run K updates, eagerly
  or replayed as a CUDA graph: their parameters are bit-identical, and every update's
  slots and indices equal those of the same ranks emulated on one device (losses within
  1e-5)."""
  import torch
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs')
  _run_processes(_two_process_worker, 2, (2, _free_port(), str(tmp_path), graph))
  params = [np.load(os.path.join(tmp_path, 'params{}.npy'.format(r))) for r in range(2)]
  assert np.array_equal(params[0].view(np.uint32), params[1].view(np.uint32))
  got = [list(np.load(os.path.join(tmp_path, 'records{}.npy'.format(r)),
                      allow_pickle=True)) for r in range(2)]

  _deterministic_convs(torch)
  _, learners = _emulated_learners(2, 64, graph=graph)
  runs = K_UPDATES + (WARMUP if graph else 0)
  want = [[], []]
  for _ in range(runs):
    _emulated_update(torch, learners)
    for r in range(2):
      want[r].append(_record(learners[r]))
  for r in range(2):
    for u, (a, b) in enumerate(zip(got[r], want[r][-K_UPDATES:])):
      assert np.array_equal(a['slots'], b['slots']), (r, u)
      assert np.array_equal(a['indices'], b['indices']), (r, u)
      np.testing.assert_allclose(a['loss'], b['loss'], rtol=1e-5)
