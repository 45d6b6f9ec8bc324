"""The data-parallel Rainbow learner on the sharded global prioritized batch
(ShardedRainbowLearner, b2r_sample_transition_batch_sharded_device,
b2r_c51_loss_sharded).  CPU tests check the host-side validation; the GPU tests
(`pytest -m gpu`) check that a shard's loss, weights and gradients are the global
batch's, with ranks emulated on one device and with two real processes."""
import ctypes
import os
import socket

import numpy as np
import pytest

from dopamine_b200 import _native
from oracle import c51_port

FRAME = 84 * 84
ACTIONS, ATOMS = 6, 51


# -- CPU: validation before any device work ------------------------------------------
def _bad_call(fn, *args):
  status = fn(*args)
  return status, _native.last_error()


def test_sharded_loss_refuses_bad_arguments_without_a_device():
  lib = _native.lib()
  args = _native.C51Args()
  args.batch, args.num_actions, args.num_atoms = 32, ACTIONS, ATOMS
  status, msg = _bad_call(lib.b2r_c51_loss_sharded, None, None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'args' in msg
  status, msg = _bad_call(lib.b2r_c51_loss_sharded, ctypes.byref(args), None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'batch_count' in msg
  count = np.zeros(1, dtype=np.int32)
  args.batch_count = count.ctypes.data
  status, msg = _bad_call(lib.b2r_c51_loss_sharded, ctypes.byref(args), None, 0, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'global_batch' in msg
  probs = np.ones(32, dtype=np.float32)
  args.sampling_probabilities = probs.ctypes.data
  status, msg = _bad_call(lib.b2r_c51_loss_sharded, ctypes.byref(args), None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'min_probability' in msg
  args.min_probability = probs.ctypes.data
  status, msg = _bad_call(lib.b2r_c51_loss_sharded, ctypes.byref(args), None, 64, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'exchange' in msg


def test_sharded_sample_refuses_bad_arguments_without_a_device():
  lib = _native.lib()
  batch = _native.Batch()
  fn = lib.b2r_sample_transition_batch_sharded_device
  status, msg = _bad_call(fn, None, None, 0, 0, 0, ctypes.byref(batch), None, None, 0,
                          None, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'global_batch' in msg
  status, msg = _bad_call(fn, None, None, 64, 0, 0, ctypes.byref(batch), None, None, -1,
                          None, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'max_rows' in msg
  status, msg = _bad_call(fn, None, None, 64, 0, 0, ctypes.byref(batch), None, None, 0,
                          None, None)
  assert status == _native.ERR_INVALID_ARGUMENT and 'required' in msg


# -- GPU ------------------------------------------------------------------------------
def _shard_memory(cap, seed, batch):
  """A full, wrapped prioritized shard with seeded columns and priorities."""
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  rng = np.random.RandomState(seed)
  mem = prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  pattern = rng.randint(0, 256, size=(257, FRAME)).astype(np.uint8)
  obs = pattern[np.arange(cap) % 257]
  mem._store['observation'] = obs.reshape(cap, 84, 84)
  mem._store['action'] = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.uint8)
  mem.add_count = cap + 1000
  mem.invalid_range = np.array([(1000 - 3 + i) % cap for i in range(7)])
  mem.set_priority(np.arange(cap, dtype=np.int32),
                   np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(np.float32))
  return mem


def _deterministic_convs(torch):
  """fp32 convolutions with a fixed algorithm: the comparisons below are between
  networks run on different row counts."""
  torch.backends.cudnn.allow_tf32 = False
  torch.backends.cuda.matmul.allow_tf32 = False
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False


def _emulated_learners(world, global_batch, scheme, cap=4000, graph=False):
  from dopamine_b200.agents.rainbow import agent
  from dopamine_b200.replay_memory import sharded_replay
  xs = sharded_replay.PeerExchange.emulated(world)
  learners = []
  for g in range(world):
    mem = _shard_memory(cap, 100 + g, global_batch)
    learners.append(agent.ShardedRainbowLearner(
        ACTIONS, batch_size=global_batch, exchange=xs[g], memory=mem,
        replay_scheme=scheme, replay_capacity=cap, seed=3, cuda_graph=graph))
  return xs, learners


def _emulated_update(torch, xs, learners):
  """One update of every emulated rank, phase by phase; the all-reduce is a sum."""
  for x, l in zip(xs, learners):
    x.publish(l.memory)  # (a launch cannot wait for a rank emulated after it)
  for l in learners:
    l.sample()
  prios = [l.loss_backward() for l in learners]
  total = torch.stack([l._flat for l in learners]).sum(0)
  for l in learners:
    l._flat.copy_(total)
  for l, p in zip(learners, prios):
    l.apply(p)
  torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize('scheme', ['prioritized', 'uniform'])
@pytest.mark.parametrize('global_batch', [64, 512])
@pytest.mark.parametrize('world', [2, 4])
def test_shards_compute_the_global_batch_update(world, global_batch, scheme):
  """Every emulated rank samples, then every rank computes its loss.  Ordering the
  ranks' rows by stratum gives the global batch; the unsharded C51 loss on it with the
  same network is the reference.  Per-row loss, priority, weight and gradient row are
  bit-identical where both launches take the same kernel variant (one CTA per row below
  128 rows, one warp per row from 128), and always within rtol 1e-6 / atol 1e-7 of the
  oracle.  The ranks' partial means and parameter gradients sum to the global ones;
  padded rows get zero gradients, so poisoning their frames changes no gradient."""
  import torch
  from dopamine_b200.agents.rainbow import rainbow_agent as ra
  _deterministic_convs(torch)
  xs, learners = _emulated_learners(world, global_batch, scheme)
  ref_net, tgt_net = learners[0].online, learners[0].target
  for l in learners[1:]:
    for p, q in zip(l.online.parameters(), ref_net.parameters()):
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

  # the global batch, rows ordered by stratum
  cols = {}
  for k, name in ((0, 'state'), (1, 'action'), (2, 'reward'), (3, 'next_state'),
                  (6, 'terminal'), (8, 'probs')):
    parts = [s[2][k][:n] for s, n in zip(samples, counts)]
    whole = torch.cat(parts)
    order = torch.as_tensor(np.argsort(np.concatenate(slots)), device='cuda')
    cols[name] = whole[order].contiguous()
  probs = cols['probs'] if scheme == 'prioritized' else None
  support, gamma_n = learners[0].support, learners[0].cumulative_gamma
  with torch.no_grad():
    online = ref_net(cols['state']).contiguous()
    target = tgt_net(cols['next_state']).contiguous()
  ref = ra.c51_loss(online, target, cols['action'], cols['reward'], cols['terminal'],
                    probs, support, gamma_n, want_grad=True)
  oracle = c51_port.rainbow_update(
      cols['reward'].cpu().numpy(), cols['terminal'].cpu().numpy(),
      cols['action'].cpu().numpy(),
      (cols['probs'] if probs is not None else torch.ones_like(cols['reward'])).cpu().numpy(),
      online.cpu().numpy(), target.cpu().numpy())
  same_variant = (global_batch >= 128) == (max_rows >= 128)

  mean_sum = 0.
  rng = np.random.RandomState(0)
  for g, (x, s, n) in enumerate(zip(xs, samples, counts)):
    slot_idx = torch.as_tensor(slots[g].astype(np.int64), device='cuda')
    local_on = torch.as_tensor(rng.randn(max_rows, ACTIONS, ATOMS).astype(np.float32),
                               device='cuda')
    local_tg = torch.as_tensor(rng.randn(max_rows, ACTIONS, ATOMS).astype(np.float32),
                               device='cuda')
    local_on[:n] = online[slot_idx]
    local_tg[:n] = target[slot_idx]
    batch = s[2]
    out = ra.c51_loss(local_on, local_tg, batch[1], batch[2], batch[6],
                      batch[8] if probs is not None else None, support, gamma_n,
                      want_grad=True, sharded=(x, global_batch, s[1], s[3]))
    torch.cuda.synchronize()
    mean_sum += float(out['mean_weighted_loss'])
    for key in ('loss', 'priorities', 'weights'):
      got = out[key][:n].cpu().numpy()
      want = ref[key][slot_idx].cpu().numpy()
      if same_variant:
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (g, key)
      if key != 'weights' or probs is not None:
        np.testing.assert_allclose(got, oracle[key][slots[g]], rtol=1e-6, atol=1e-7)
    if probs is None:
      assert (out['weights'][:n].cpu().numpy() == 1.).all()
    grad = out['grad_logits'].cpu().numpy()
    if same_variant:
      want = ref['grad_logits'][slot_idx].cpu().numpy()
      assert np.array_equal(grad[:n].view(np.uint32), want.view(np.uint32)), g
    assert not grad[n:].any(), 'padded rows must get exact zero gradients'
  # (G partial sums, each over a rank's rows, against one sum over all rows: f32
  # reassociation of at most 512 positive terms, relative error below 512 * 2^-24)
  np.testing.assert_allclose(mean_sum, float(ref['mean_weighted_loss']), rtol=4e-5)

  # parameter gradients: the ranks' partial gradients summed vs the global batch's
  partial = []
  for l in learners:
    l.loss_backward()
    partial.append(l._flat.clone())
  torch.cuda.synchronize()
  total = torch.stack(partial).sum(0)
  learners[0]._flat.zero_()
  mean, _, _, _ = ra.C51Loss.apply(ref_net(cols['state']), target, cols['action'],
                                   cols['reward'], cols['terminal'], probs, support,
                                   gamma_n)
  mean.backward()
  want = learners[0]._flat[:-1]
  scale = float(want.abs().max())
  # (the batch-size dependent reduction order of cuDNN / cuBLAS backward and the
  # G-way sum: fp32 reassociation over <= 512 rows and 7744-wide layers)
  torch.testing.assert_close(total[:-1], want, rtol=1e-4, atol=1e-5 * scale)
  np.testing.assert_allclose(float(total[-1]), float(ref['mean_weighted_loss']),
                             rtol=4e-5)

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


def _record(learner):
  slots, count, batch, _ = learner._sample
  n = int(count.item())
  return dict(slots=slots[:n].cpu().numpy(), indices=batch[7][:n].cpu().numpy(),
              loss=float(learner.loss.item()))


def _process_worker(rank, world, port, out_dir, graph):
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
    cap, global_batch = 4000, 64
    mem = _shard_memory(cap, 100 + rank, global_batch)
    learner = agent.ShardedRainbowLearner(
        ACTIONS, batch_size=global_batch, memory=mem, replay_capacity=cap, seed=3,
        cuda_graph=graph)
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
  1e-5: a replayed graph applies Adam's step size computed on the device)."""
  import torch
  import torch.multiprocessing as mp
  if torch.cuda.device_count() < 2:
    pytest.skip('needs 2 GPUs')
  ctx = mp.get_context('spawn')
  port = _free_port()
  procs = [ctx.Process(target=_process_worker, args=(r, 2, port, str(tmp_path), graph))
           for r in range(2)]
  for p in procs:
    p.start()
  for p in procs:
    p.join(timeout=900)
  alive = [p for p in procs if p.is_alive()]
  for p in alive:
    p.terminate()
    p.join(timeout=60)
  assert not alive, 'a rank did not finish'
  assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
  params = [np.load(os.path.join(tmp_path, 'params{}.npy'.format(r))) for r in range(2)]
  assert np.array_equal(params[0].view(np.uint32), params[1].view(np.uint32))
  got = [list(np.load(os.path.join(tmp_path, 'records{}.npy'.format(r)),
                      allow_pickle=True)) for r in range(2)]

  _deterministic_convs(torch)
  xs, learners = _emulated_learners(2, 64, 'prioritized', graph=graph)
  # a graph-mode learner runs three eager warm-up updates before its first replay
  runs = K_UPDATES + (3 if graph else 0)
  want = [[], []]
  for _ in range(runs):
    _emulated_update(torch, xs, learners)
    for r in range(2):
      want[r].append(_record(learners[r]))
  for r in range(2):
    for u, (a, b) in enumerate(zip(got[r], want[r][-K_UPDATES:])):
      assert np.array_equal(a['slots'], b['slots']), (r, u)
      assert np.array_equal(a['indices'], b['indices']), (r, u)
      np.testing.assert_allclose(a['loss'], b['loss'], rtol=1e-5)
