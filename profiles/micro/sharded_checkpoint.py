"""Save and restore of a data-parallel learner (ShardedLearner.save / restore) at full
shard size, under torchrun, one GPU per rank:

  torchrun --nproc_per_node N profiles/micro/sharded_checkpoint.py [--kind rainbow]
      [--capacity 1000000] [--batch 256] [--updates-before-save 20]
      [--updates-after-save 10] [--checkpoint-dir DIR]

Every rank fills a shard of `capacity` Atari-shaped transitions (frames generated on the
device), trains K updates, saves, trains M more (--updates-before-save,
--updates-after-save) and records every loss; then it builds a
fresh learner over other transitions in the same process, restores, trains the same M
updates and asserts that the losses and the parameters are identical to the first run's.
Prints one JSON line per rank: save and restore wall time (each ends in a device
synchronise and a barrier of all ranks), the bytes the rank wrote, the card's name and
power limit.  `--checkpoint-dir` defaults to a temporary directory, removed at the end.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card(device):
  out = subprocess.check_output(
      ['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
       str(device)]).decode().strip()
  return [x.strip() for x in out.split(',')]


def fill(mem, seed, torch, native):
  """Frames generated on the device, seeded scalar columns, full ring, priorities."""
  lib = native.lib()
  cap = mem._replay_capacity  # pylint: disable=protected-access
  gen = torch.Generator(device='cuda')
  gen.manual_seed(seed)
  stream = native.current_stream()
  chunk = 65536
  for lo in range(0, cap, chunk):
    n = min(chunk, cap - lo)
    frames = torch.randint(0, 256, (n, 84, 84), dtype=torch.uint8, device='cuda',
                           generator=gen)
    native.check(lib.b2r_store_write(mem._h, 0, lo, n, frames.data_ptr(), stream))  # pylint: disable=protected-access
  rng = np.random.RandomState(seed)
  mem._store['action'] = rng.randint(0, 6, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.uint8)
  mem.add_count = cap + 1000
  mem.invalid_range = np.array([(1000 - 3 + i) % cap for i in range(7)])
  if hasattr(mem, 'sum_tree'):
    mem.set_priority(np.arange(cap, dtype=np.int32),
                     np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(np.float32))


def make_learner(kind, args, rank, seed, torch, native):
  from dopamine_b200.agents.dqn import learner as dqn_learner
  from dopamine_b200.agents.implicit_quantile import learner as iqn_learner
  from dopamine_b200.agents.rainbow import agent
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  buffer_class = (crb.OutOfGraphReplayBuffer if kind == 'dqn'
                  else prb.OutOfGraphPrioritizedReplayBuffer)
  mem = buffer_class((84, 84), 4, args.capacity, args.batch, update_horizon=3, gamma=0.99,
                     output='torch', rng='device', seed=seed, reuse_outputs=True)
  fill(mem, seed + rank, torch, native)
  common = dict(batch_size=args.batch, memory=mem, replay_capacity=args.capacity, seed=3,
                cuda_graph=args.graph)
  if kind == 'dqn':
    return dqn_learner.ShardedDQNLearner(6, update_horizon=3, **common)
  if kind == 'iqn':
    return iqn_learner.ShardedIQNLearner(6, **common)
  return agent.ShardedRainbowLearner(6, **common)


def main():
  parser = argparse.ArgumentParser()
  parser.add_argument('--kind', choices=['rainbow', 'iqn', 'dqn'], default='rainbow')
  parser.add_argument('--capacity', type=int, default=1000000)
  parser.add_argument('--batch', type=int, default=256)
  parser.add_argument('--updates-before-save', type=int, default=20)
  parser.add_argument('--updates-after-save', type=int, default=10)
  parser.add_argument('--graph', action='store_true')
  parser.add_argument('--checkpoint-dir', default=None)
  args = parser.parse_args()

  import torch
  import torch.distributed as dist
  from dopamine_b200 import _native
  rank, local = int(os.environ['RANK']), int(os.environ.get('LOCAL_RANK', 0))
  torch.cuda.set_device(local)
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False
  dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  world = dist.get_world_size()
  made = None
  if args.checkpoint_dir is None:
    box = [tempfile.mkdtemp(prefix='sharded_ckpt_') if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    made = path = box[0]
  else:
    path = args.checkpoint_dir
  try:
    def timed(fn):
      torch.cuda.synchronize()
      dist.barrier()
      t0 = time.perf_counter()
      fn()
      torch.cuda.synchronize()
      dist.barrier()
      return time.perf_counter() - t0

    def run(learner, n):
      losses = []
      for _ in range(n):
        loss = learner.train_step()
        losses.append(float(loss.item()))
      return losses

    first = make_learner(args.kind, args, rank, 100, torch, _native)
    run(first, args.updates_before_save)
    save_s = timed(lambda: first.save(path, 1))
    want = run(first, args.updates_after_save)
    want_params = [p.detach().clone() for p in first.online.parameters()]
    first.check()
    del first
    torch.cuda.empty_cache()

    second = make_learner(args.kind, args, rank, 500, torch, _native)
    run(second, 1)
    restore_s = timed(lambda: second.restore(path, 1))
    got = run(second, args.updates_after_save)
    second.check()
    assert got == want, (rank, got, want)
    for p, q in zip(second.online.parameters(), want_params):
      assert torch.equal(p, q), rank
    rank_dir = os.path.join(path, 'rank_{}'.format(rank))
    written = sum(os.path.getsize(os.path.join(rank_dir, f)) for f in os.listdir(rank_dir))
    name, limit = card(local)
    print(json.dumps(dict(kind=args.kind, world=world, rank=rank, capacity=args.capacity,
                          batch=args.batch, graph=args.graph, save_s=round(save_s, 3),
                          restore_s=round(restore_s, 3), rank_bytes=written,
                          identical=True, gpu=name, power_limit=limit)), flush=True)
    dist.barrier()
  finally:
    if made is not None and rank == 0:
      shutil.rmtree(made, ignore_errors=True)
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
