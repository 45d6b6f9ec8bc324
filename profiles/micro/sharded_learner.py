"""ms per update and transitions/s of ShardedRainbowLearner (`--agent rainbow`),
ShardedIQNLearner (`--agent iqn`) or ShardedDQNLearner (`--agent dqn`) at 1/2/4/8 GPUs: a
global batch of 32 rows per GPU, a
replay shard of 1M transitions per GPU, eager and replayed as a CUDA graph.  Also reports
the rows the networks computed (max_rows per rank, the padding that keeps the shapes
static) next to the useful rows (the global batch), and the card's name and power limit
read in the same run.  With `--agent iqn` the shards have unit priorities (IQN's replay),
the tau counts are IQNLearner's defaults (N = N' = K = 32), and the run also times plain
IQNLearner.train_step() at batch 32 on one GPU, the N = 1 baseline.  With `--agent dqn`
the shards are uniform OutOfGraphReplayBuffers (DQN's replay), the eager runs also time
`sample()` alone (the sharded uniform sampler and the frame copies), and the baseline is
plain DQNLearner.train_step() at batch 32.

  python profiles/micro/sharded_learner.py [--agent rainbow|iqn|dqn] [--gpus 1,2,4,8]
      [--steps 200] [--out F]

Each configuration runs in fresh processes (one per GPU, NCCL); rank 0 times `--steps`
updates between CUDA events after `--warmup` updates.  The frames of the shards are
left as allocated (only the scalar columns and the priorities are written): the
timing does not depend on pixel values.
"""
import argparse
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

PER_GPU_BATCH = 32
CAPACITY = 1000000
ACTIONS = 18


def _shard(cap, seed, batch, unit_priorities=False):
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  rng = np.random.RandomState(seed)
  mem = prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  mem._store['action'] = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.uint8)
  mem.add_count = cap + 1000
  mem.invalid_range = np.array([(1000 - 3 + i) % cap for i in range(7)])
  priorities = (np.ones(cap, dtype=np.float32) if unit_priorities else
                np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(np.float32))
  mem.set_priority(np.arange(cap, dtype=np.int32), priorities)
  return mem


def _uniform_shard(cap, seed, batch):
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  rng = np.random.RandomState(seed)
  mem = crb.OutOfGraphReplayBuffer(
      (84, 84), 4, cap, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed, reuse_outputs=True)
  mem._store['action'] = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.uint8)
  mem.add_count = cap + 1000
  mem.invalid_range = np.array([(1000 - 3 + i) % cap for i in range(7)])
  return mem


def _make_learner(agent_name, global_batch, rank, graph):
  if agent_name == 'dqn':
    from dopamine_b200.agents.dqn import learner
    return learner.ShardedDQNLearner(
        ACTIONS, batch_size=global_batch,
        memory=_uniform_shard(CAPACITY, 10 + rank, global_batch),
        replay_capacity=CAPACITY, update_horizon=3, seed=1, cuda_graph=graph)
  if agent_name == 'iqn':
    from dopamine_b200.agents.implicit_quantile import learner
    return learner.ShardedIQNLearner(
        ACTIONS, batch_size=global_batch,
        memory=_shard(CAPACITY, 10 + rank, global_batch, unit_priorities=True),
        replay_capacity=CAPACITY, seed=1, cuda_graph=graph)
  from dopamine_b200.agents.rainbow import agent
  return agent.ShardedRainbowLearner(
      ACTIONS, batch_size=global_batch, memory=_shard(CAPACITY, 10 + rank, global_batch),
      replay_capacity=CAPACITY, seed=1, cuda_graph=graph)


def _time_updates(torch, learner, steps):
  start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  start.record()
  for _ in range(steps):
    learner.train_step()
  end.record()
  torch.cuda.synchronize()
  return start.elapsed_time(end) / steps


def _iqn_settings(learner):
  return dict(num_tau_samples=learner.num_tau_samples,
              num_tau_prime_samples=learner.num_tau_prime_samples,
              num_quantile_samples=learner.num_quantile_samples)


def _baseline_worker(rank, agent_name, steps, warmup, out_path):
  """Plain IQNLearner / DQNLearner .train_step() at batch 32 on one GPU: the N = 1
  baseline."""
  import torch
  torch.cuda.set_device(rank)
  if agent_name == 'dqn':
    from dopamine_b200.agents.dqn import learner as dqn_learner
    learner = dqn_learner.DQNLearner(
        ACTIONS, batch_size=PER_GPU_BATCH, replay_capacity=CAPACITY, update_horizon=3,
        seed=1, memory=_uniform_shard(CAPACITY, 10, PER_GPU_BATCH))
  else:
    from dopamine_b200.agents.implicit_quantile import learner as iqn_learner
    learner = iqn_learner.IQNLearner(
        ACTIONS, batch_size=PER_GPU_BATCH, replay_capacity=CAPACITY, seed=1,
        memory=_shard(CAPACITY, 10, PER_GPU_BATCH, unit_priorities=True))
  for _ in range(warmup):
    learner.train_step()
  torch.cuda.synchronize()
  ms = _time_updates(torch, learner, steps)
  result = dict(agent=agent_name, learner=type(learner).__name__, gpus=1, mode='eager',
                steps=steps, ms_per_update=round(ms, 4),
                transitions_per_s=round(PER_GPU_BATCH / ms * 1e3, 1),
                useful_rows=PER_GPU_BATCH, network_rows=PER_GPU_BATCH,
                capacity_per_gpu=CAPACITY)
  if agent_name == 'iqn':
    result.update(_iqn_settings(learner))
  with open(out_path, 'w') as f:
    json.dump(result, f)


def _worker(rank, world, port, agent_name, graph, steps, warmup, out_path):
  import torch
  import torch.distributed as dist
  torch.cuda.set_device(rank)
  os.environ['MASTER_ADDR'] = '127.0.0.1'
  os.environ['MASTER_PORT'] = str(port)
  dist.init_process_group('nccl', rank=rank, world_size=world,
                          device_id=torch.device('cuda', rank))
  try:
    global_batch = PER_GPU_BATCH * world
    learner = _make_learner(agent_name, global_batch, rank, graph)
    for _ in range(warmup):
      learner.train_step()
    torch.cuda.synchronize()
    dist.barrier()
    ms = _time_updates(torch, learner, steps)
    sample_ms = None
    if agent_name == 'dqn' and not graph:  # the sampler and the frame copies alone
      start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      dist.barrier()
      start.record()
      for _ in range(steps):
        learner.sample()
      end.record()
      torch.cuda.synchronize()
      sample_ms = start.elapsed_time(end) / steps
    learner.check()
    if rank == 0:
      result = dict(agent=agent_name, learner=type(learner).__name__, gpus=world,
                    mode='graph' if graph else 'eager', steps=steps,
                    ms_per_update=round(ms, 4),
                    transitions_per_s=round(global_batch / ms * 1e3, 1),
                    useful_rows=global_batch, max_rows_per_rank=learner.max_rows,
                    network_rows=learner.max_rows * world, capacity_per_gpu=CAPACITY,
                    loss=float(learner.loss.item()))
      if agent_name == 'iqn':
        result.update(_iqn_settings(learner))
      if sample_ms is not None:
        result['sample_ms'] = round(sample_ms, 4)
      with open(out_path, 'w') as f:
        json.dump(result, f)
    dist.barrier()
  finally:
    dist.destroy_process_group()


def _free_port():
  with socket.socket() as s:
    s.bind(('127.0.0.1', 0))
    return s.getsockname()[1]


def main():
  import torch
  import torch.multiprocessing as mp
  p = argparse.ArgumentParser()
  p.add_argument('--agent', choices=('rainbow', 'iqn', 'dqn'), default='rainbow')
  p.add_argument('--gpus', default='1,2,4,8')
  p.add_argument('--steps', type=int, default=200)
  p.add_argument('--warmup', type=int, default=20)
  p.add_argument('--out', default=None)
  a = p.parse_args()
  if not torch.cuda.is_available():
    sys.exit('needs CUDA devices')
  card = subprocess.check_output(
      ['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader']
  ).decode().strip().splitlines()
  lines = [json.dumps(dict(cards=card))]
  print(lines[0], flush=True)
  tmp = os.environ.get('TMPDIR', '/tmp')
  ctx = mp.get_context('spawn')

  def run(target, world, args, desc):
    procs = [ctx.Process(target=target, args=(r,) + args) for r in range(world)]
    for q in procs:
      q.start()
    for q in procs:
      q.join(timeout=1200)
    for q in procs:
      if q.is_alive():
        q.terminate()
        q.join(timeout=60)
    codes = [q.exitcode for q in procs]
    if any(c != 0 for c in codes):
      lines.append(json.dumps(dict(desc, failed=codes)))
    else:
      with open(args[-1]) as f:
        lines.append(f.read())
    print(lines[-1], flush=True)

  if a.agent in ('iqn', 'dqn'):
    run(_baseline_worker, 1,
        (a.agent, a.steps, a.warmup, os.path.join(tmp, a.agent + '_baseline.json')),
        dict(agent=a.agent, gpus=1, mode='eager'))
  for n in [int(x) for x in a.gpus.split(',')]:
    if n > torch.cuda.device_count():
      lines.append(json.dumps(dict(agent=a.agent, gpus=n, skipped='only {} devices'
                                   .format(torch.cuda.device_count()))))
      print(lines[-1], flush=True)
      continue
    for graph in (False, True):
      out_path = os.path.join(tmp, 'sharded_learner_{}_{}_{}.json'.format(
          a.agent, n, int(graph)))
      run(_worker, n, (n, _free_port(), a.agent, graph, a.steps, a.warmup, out_path),
          dict(agent=a.agent, gpus=n, mode='graph' if graph else 'eager'))
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
      f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
  main()
