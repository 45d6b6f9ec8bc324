"""The data-parallel IQN learner on the sharded global batch (ShardedIQNLearner,
b2r_iqn_loss_sharded).  CPU tests check the host-side validation; the GPU tests
(`pytest -m gpu`) check that a shard's loss, next actions and gradients are the global
batch's, with ranks emulated on one device, in one real process (eager against graph)
and with two real processes."""
import ctypes
import os
import socket

import numpy as np
import pytest

from dopamine_b200 import _native
from oracle import iqn_port

FRAME = 84 * 84
# IQN shapes of test_iqn.py's first case: the paper's N = N' = 64, K = 32, 18 actions
ACTIONS, N, N_PRIME, K = 18, 64, 64, 32
CAP = 4000
FILLS = (4000, 3000, 2000, 3500)  # transitions per shard: shares off the even split
GAMMA_N = 0.99 ** 3


# -- CPU: validation before any device work ------------------------------------------
def test_sharded_iqn_loss_refuses_bad_arguments_without_a_device():
  lib = _native.lib()
  args = _native.IqnArgs()
  args.batch, args.num_actions = 32, ACTIONS
  status = lib.b2r_iqn_loss_sharded(None, None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'args' in _native.last_error()
  status = lib.b2r_iqn_loss_sharded(ctypes.byref(args), None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'count' in _native.last_error()
  count = np.zeros(1, dtype=np.int32)
  status = lib.b2r_iqn_loss_sharded(ctypes.byref(args), count.ctypes.data, 0, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'global_batch' in _native.last_error()
  # then the checks of b2r_iqn_loss, still before any device work
  status = lib.b2r_iqn_loss_sharded(ctypes.byref(args), count.ctypes.data, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'shape' in _native.last_error()


def test_sharded_iqn_learner_refuses_ddp_and_a_missing_exchange():
  import torch.distributed as dist
  from dopamine_b200.agents.implicit_quantile import learner
  with pytest.raises(ValueError, match='ddp=False'):
    learner.ShardedIQNLearner(ACTIONS, ddp=True)
  assert not (dist.is_available() and dist.is_initialized())
  with pytest.raises(RuntimeError, match='torch.distributed'):
    learner.ShardedIQNLearner(ACTIONS)


# -- GPU ------------------------------------------------------------------------------
def _shard_memory(seed, batch, fill):
  """A unit-priority shard (IQN's replay) holding `fill` seeded transitions."""
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  rng = np.random.RandomState(seed)
  mem = prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, CAP, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  pattern = rng.randint(0, 256, size=(257, FRAME)).astype(np.uint8)
  mem._store['observation'] = pattern[np.arange(CAP) % 257].reshape(CAP, 84, 84)
  mem._store['action'] = rng.randint(0, ACTIONS, size=CAP).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(CAP), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(CAP) < 0.01).astype(np.uint8)
  if fill < CAP:
    mem.add_count = fill
    mem.invalid_range = crb.invalid_range(fill, CAP, 4, 3)
  else:
    mem.add_count = CAP + 1000
    mem.invalid_range = crb.invalid_range(1000, CAP, 4, 3)
  mem.set_priority(np.arange(fill, dtype=np.int32), np.ones(fill, dtype=np.float32))
  return mem


def _deterministic_convs(torch):
  """fp32 convolutions with a fixed algorithm: the comparisons below are between
  networks run on different row counts."""
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False


def _learner(global_batch, rank, double_dqn=False, **kwargs):
  from dopamine_b200.agents.implicit_quantile import learner
  return learner.ShardedIQNLearner(
      ACTIONS, batch_size=global_batch, memory=_shard_memory(100 + rank, global_batch,
                                                             FILLS[rank]),
      replay_capacity=CAP, seed=3, num_tau_samples=N, num_tau_prime_samples=N_PRIME,
      num_quantile_samples=K, double_dqn=double_dqn, **kwargs)


def _emulated_learners(world, global_batch, double_dqn=False, graph=False):
  from dopamine_b200.replay_memory import sharded_replay
  xs = sharded_replay.PeerExchange.emulated(world)
  return xs, [_learner(global_batch, g, double_dqn, exchange=xs[g], cuda_graph=graph)
              for g in range(world)]


def _emulated_update(torch, xs, learners):
  """One update of every emulated rank, phase by phase; the all-reduce is a sum."""
  for x, l in zip(xs, learners):
    x.publish(l.memory)  # (a launch cannot wait for a rank emulated after it)
  for l in learners:
    l.sample()
  for l in learners:
    l.loss_backward()
  total = torch.stack([l._flat for l in learners]).sum(0)
  for l in learners:
    l._flat.copy_(total)
    l.apply()
  torch.cuda.synchronize()


def _scatter(torch, whole, samples, global_batch, max_rows, slot_idx, rng):
  """(samples * global_batch, C) sample-major rows -> a rank's (samples * max_rows, C):
  row s * max_rows + r is global row s * global_batch + slot r; padding is noise."""
  cols = whole.shape[1]
  out = torch.as_tensor(rng.randn(samples, max_rows, cols).astype(np.float32),
                        device='cuda')
  out[:, :len(slot_idx)] = whole.view(samples, global_batch, cols)[:, slot_idx]
  return out.view(samples * max_rows, cols)


def _bits(x):
  return x.cpu().numpy().view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize('double_dqn', [False, True])
@pytest.mark.parametrize('global_batch', [64, 512])
@pytest.mark.parametrize('world', [2, 4])
def test_shards_compute_the_global_batch_update(world, global_batch, double_dqn):
  """Every emulated rank samples from a unit-priority shard of its own fill level, then
  every rank computes its loss.  Ordering the ranks' rows by stratum gives the global
  batch; the unsharded IQN loss on it with the same network outputs and taus is the
  reference.  Per-row loss, next action and gradient rows are bit-identical (one kernel
  variant), and within rtol 2e-6 / atol 1e-7 of the oracle.  The ranks' partial means
  and parameter gradients sum to the global ones; padded rows get zero gradients, so
  poisoning their frames changes no gradient."""
  import torch
  from dopamine_b200.agents.implicit_quantile import implicit_quantile_agent as iq
  _deterministic_convs(torch)
  xs, learners = _emulated_learners(world, global_batch, double_dqn)
  online_net, target_net = learners[0].online, learners[0].target
  for l in learners[1:]:
    for p, q in zip(l.online.parameters(), online_net.parameters()):
      assert torch.equal(p, q)
  for x, l in zip(xs, learners):
    x.publish(l.memory)
  samples = [l.sample() for l in learners]
  torch.cuda.synchronize()
  counts = [int(s[1].item()) for s in samples]
  slots = [s[0][:n].cpu().numpy() for s, n in zip(samples, counts)]
  assert sum(counts) == global_batch
  assert np.array_equal(np.sort(np.concatenate(slots)), np.arange(global_batch))
  max_rows = learners[0].max_rows
  assert max(counts) <= max_rows
  assert counts != [global_batch // world] * world, 'the shares should be uneven'

  # the global batch, rows ordered by stratum, and taus for it
  cols = {}
  order = torch.as_tensor(np.argsort(np.concatenate(slots)), device='cuda')
  for k, name in ((0, 'state'), (1, 'action'), (2, 'reward'), (3, 'next_state'),
                  (6, 'terminal')):
    whole = torch.cat([s[2][k][:n] for s, n in zip(samples, counts)])
    cols[name] = whole[order].contiguous()
  gen = torch.Generator(device='cuda').manual_seed(7)
  taus = {name: torch.rand(m * global_batch, 1, device='cuda', generator=gen)
          for name, m in (('online', N), ('target', N_PRIME), ('action', K))}
  picker = online_net if double_dqn else target_net
  with torch.no_grad():
    online, _ = online_net(cols['state'], N, taus['online'])
    target, _ = target_net(cols['next_state'], N_PRIME, taus['target'])
    action, _ = picker(cols['next_state'], K, taus['action'])
  ref = iq.quantile_huber_loss(online, taus['online'], target, action, cols['action'],
                               cols['reward'], cols['terminal'], GAMMA_N, want_grad=True)
  host = lambda x: x.cpu().numpy()
  oracle = iqn_port.iqn_update(
      host(cols['reward']), host(cols['terminal']), host(cols['action']), host(online),
      host(taus['online']), host(target), host(action), N, N_PRIME, K, gamma=0.99,
      update_horizon=3)

  mean_sum = 0.
  rng = np.random.RandomState(0)
  local_taus = []
  for g, (x, s, n) in enumerate(zip(xs, samples, counts)):
    slot_idx = torch.as_tensor(slots[g].astype(np.int64), device='cuda')
    scatter = lambda whole, m: _scatter(  # pylint: disable=cell-var-from-loop
        torch, whole, m, global_batch, max_rows, slot_idx, rng)
    local = dict(online=scatter(online, N), target=scatter(target, N_PRIME),
                 action=scatter(action, K))
    local_taus.append({name: scatter(taus[name], m).contiguous() for name, m in
                       (('online', N), ('target', N_PRIME), ('action', K))})
    batch = s[2]
    out = iq.quantile_huber_loss(local['online'], local_taus[g]['online'], local['target'],
                                 local['action'], batch[1], batch[2], batch[6], GAMMA_N,
                                 want_grad=True, sharded=(global_batch, s[1]))
    torch.cuda.synchronize()
    mean_sum += float(out['mean_loss'])
    assert np.array_equal(_bits(out['loss'][:n]), _bits(ref['loss'][slot_idx])), g
    assert not out['loss'][n:].cpu().numpy().any(), g
    assert np.array_equal(host(out['next_action'][:n]), host(ref['next_action'][slot_idx]))
    np.testing.assert_allclose(host(out['loss'][:n]), oracle['loss'][slots[g]],
                               rtol=2e-6, atol=1e-7)
    assert np.array_equal(host(out['next_action'][:n]), oracle['next_action'][slots[g]])
    grad = out['grad'].view(N, max_rows, ACTIONS)
    want = ref['grad'].view(N, global_batch, ACTIONS)[:, slot_idx]
    assert np.array_equal(_bits(grad[:, :n]), _bits(want)), g
    np.testing.assert_allclose(
        host(grad[:, :n]), oracle['grad'].reshape(N, global_batch, ACTIONS)[:, slots[g]],
        rtol=2e-6, atol=1e-7)
    assert not grad[:, n:].cpu().numpy().any(), 'padded rows must get exact zero gradients'
  # (f64 sums rounded once per rank: the G-way f32 sum differs in the last bits)
  np.testing.assert_allclose(mean_sum, float(ref['mean_loss']), rtol=1e-6)

  # parameter gradients through the learner's phases, the taus injected
  partial = []
  for l, lt in zip(learners, local_taus):
    l.online_taus.copy_(lt['online'])
    l.target_taus.copy_(lt['target'])
    l.action_taus.copy_(lt['action'])
    l.loss_backward()
    partial.append(l._flat.clone())
  torch.cuda.synchronize()
  total = torch.stack(partial).sum(0)
  learners[0]._flat.zero_()
  online_values, _ = online_net(cols['state'], N, taus['online'])
  mean, _ = iq.QuantileHuberLoss.apply(online_values, taus['online'], target, action,
                                       cols['action'], cols['reward'], cols['terminal'],
                                       GAMMA_N)
  mean.backward()
  want = learners[0]._flat[:-1]
  scale = float(want.abs().max())
  # (the batch-size dependent reduction order of cuDNN / cuBLAS backward and the
  # G-way sum: fp32 reassociation over <= 512 * N rows and 3136-wide layers)
  torch.testing.assert_close(total[:-1], want, rtol=1e-4, atol=1e-5 * scale)
  np.testing.assert_allclose(float(total[-1]), float(ref['mean_loss']), rtol=4e-5)

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


@pytest.mark.gpu
def test_sharded_loss_refuses_a_bad_count():
  import torch
  from dopamine_b200.agents.implicit_quantile import implicit_quantile_agent as iq
  rng = np.random.RandomState(0)
  dev = lambda *shape: torch.as_tensor(rng.randn(*shape).astype(np.float32), device='cuda')
  b = 4
  args = (dev(2 * b, 3), torch.rand(2 * b, 1, device='cuda'), dev(2 * b, 3), dev(2 * b, 3),
          torch.zeros(b, dtype=torch.int32, device='cuda'), dev(b),
          torch.zeros(b, dtype=torch.uint8, device='cuda'), GAMMA_N)
  for count in (torch.zeros(1, dtype=torch.int64, device='cuda'),
                torch.zeros(1, dtype=torch.int32), torch.zeros(2, dtype=torch.int32,
                                                               device='cuda')):
    with pytest.raises(ValueError, match='count'):
      iq.quantile_huber_loss(*args, sharded=(8, count))
  with pytest.raises(ValueError, match='global_batch'):
    iq.quantile_huber_loss(*args, sharded=(0, torch.zeros(1, dtype=torch.int32,
                                                          device='cuda')))


def _free_port():
  with socket.socket() as s:
    s.bind(('127.0.0.1', 0))
    return s.getsockname()[1]


K_UPDATES = 3
WARMUP = 3  # the eager updates a graph-mode learner runs before its capture


def _record(learner):
  slots, count, batch, _ = learner._sample
  n = int(count.item())
  return dict(slots=slots[:n].cpu().numpy(), indices=batch[7][:n].cpu().numpy(),
              loss=float(learner.loss.item()),
              taus=learner.online_taus.cpu().numpy().copy())


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
  slots and indices, and draw the same taus, as the eager updates after the graph's
  warm-up; losses within 1e-5 (a replayed graph applies Adam's step size computed on the
  device).  Consecutive replays draw different taus, and nothing is latched."""
  _run_processes(_single_process_worker, 1, (_free_port(), str(tmp_path)))
  records = np.load(os.path.join(tmp_path, 'records.npy'), allow_pickle=True)[0]
  eager, graph = records[False][WARMUP:], records[True]
  for u, (a, b) in enumerate(zip(graph, eager)):
    assert np.array_equal(a['slots'], b['slots']), u
    assert np.array_equal(a['indices'], b['indices']), u
    assert np.array_equal(a['taus'], b['taus']), u
    np.testing.assert_allclose(a['loss'], b['loss'], rtol=1e-5)
  for a, b in zip(graph, graph[1:]):
    assert not np.array_equal(a['taus'], b['taus'])


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
  slots, indices and taus equal those of the same ranks emulated on one device (losses
  within 1e-5)."""
  import torch
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs')
  _run_processes(_two_process_worker, 2, (2, _free_port(), str(tmp_path), graph))
  params = [np.load(os.path.join(tmp_path, 'params{}.npy'.format(r))) for r in range(2)]
  assert np.array_equal(params[0].view(np.uint32), params[1].view(np.uint32))
  got = [list(np.load(os.path.join(tmp_path, 'records{}.npy'.format(r)),
                      allow_pickle=True)) for r in range(2)]

  _deterministic_convs(torch)
  xs, learners = _emulated_learners(2, 64, graph=graph)
  runs = K_UPDATES + (WARMUP if graph else 0)
  want = [[], []]
  for _ in range(runs):
    _emulated_update(torch, xs, learners)
    for r in range(2):
      want[r].append(_record(learners[r]))
  for r in range(2):
    for u, (a, b) in enumerate(zip(got[r], want[r][-K_UPDATES:])):
      assert np.array_equal(a['slots'], b['slots']), (r, u)
      assert np.array_equal(a['indices'], b['indices']), (r, u)
      assert np.array_equal(a['taus'], b['taus']), (r, u)
      np.testing.assert_allclose(a['loss'], b['loss'], rtol=1e-5)
