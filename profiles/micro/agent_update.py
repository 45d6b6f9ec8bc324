"""ms per update of the single-GPU DQNLearner and IQNLearner, eager and replayed as one
CUDA graph (`cuda_graph=True`), at batch 32 over a replay of 1M transitions.

  python profiles/micro/agent_update.py [--steps 200] [--warmup 20] [--runs 3] [--out F]

Each of the four learners (dqn / iqn x eager / graph) is built once and warmed up
(`--warmup` updates, the graph's capture included); then `--runs` rounds time
`--steps` updates of each learner in turn between CUDA events, so that the
configurations alternate and share whatever else the machine runs.  The time between
the events covers the whole update as the device sees it, host launch gaps included
(the eager update is bound by them).  One JSON line per learner: the median and the
spread (min, max) over the rounds, and the card's name and power limit read in the same
run.  The frames of the replay are left as allocated (only the scalar columns, validity
state and, for IQN, the unit priorities are written): the timing does not depend on
pixel values.  IQN runs with IQNLearner's defaults (N = N' = K = 32).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

BATCH = 32
CAPACITY = 1000000
ACTIONS = 18


def _fill(mem, rng):
  mem._store['action'] = rng.randint(0, ACTIONS, size=CAPACITY).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(CAPACITY), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(CAPACITY) < 0.01).astype(np.uint8)
  mem.add_count = CAPACITY + 1000
  mem.invalid_range = np.array([(1000 - 3 + i) % CAPACITY for i in range(7)])
  return mem


def _make(agent, graph):
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  rng = np.random.RandomState(10)
  if agent == 'dqn':
    from dopamine_b200.agents.dqn import learner
    mem = _fill(crb.OutOfGraphReplayBuffer(
        (84, 84), 4, CAPACITY, BATCH, update_horizon=1, gamma=0.99, output='torch',
        rng='device', seed=1, reuse_outputs=True), rng)
    return learner.DQNLearner(ACTIONS, replay_capacity=CAPACITY, batch_size=BATCH,
                              seed=1, memory=mem, cuda_graph=graph)
  from dopamine_b200.agents.implicit_quantile import learner
  mem = _fill(prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, CAPACITY, BATCH, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=1, reuse_outputs=True), rng)
  mem.set_priority(np.arange(CAPACITY, dtype=np.int32), np.ones(CAPACITY, np.float32))
  return learner.IQNLearner(ACTIONS, replay_capacity=CAPACITY, batch_size=BATCH, seed=1,
                            memory=mem, cuda_graph=graph)


def main():
  import torch
  p = argparse.ArgumentParser()
  p.add_argument('--steps', type=int, default=200)
  p.add_argument('--warmup', type=int, default=20)
  p.add_argument('--runs', type=int, default=3)
  p.add_argument('--out', default=None)
  a = p.parse_args()
  if not torch.cuda.is_available():
    sys.exit('needs a CUDA device')
  card = subprocess.check_output(
      ['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit', '--format=csv,noheader']
  ).decode().strip()
  configs = [(agent, graph) for agent in ('dqn', 'iqn') for graph in (False, True)]
  learners = {}
  for config in configs:
    learners[config] = _make(*config)
    for _ in range(a.warmup):
      learners[config].train_step()
    torch.cuda.synchronize()
  times = {config: [] for config in configs}
  start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for _ in range(a.runs):
    for config in configs:
      learner = learners[config]
      torch.cuda.synchronize()
      start.record()
      for _ in range(a.steps):
        learner.train_step()
      end.record()
      torch.cuda.synchronize()
      times[config].append(start.elapsed_time(end) / a.steps)
  lines = []
  for (agent, graph), ms in times.items():
    lines.append(json.dumps(dict(
        learner=type(learners[(agent, graph)]).__name__,
        mode='graph' if graph else 'eager', batch=BATCH, capacity=CAPACITY,
        steps=a.steps, runs=a.runs, ms_per_update_median=round(float(np.median(ms)), 4),
        ms_per_update_min=round(min(ms), 4), ms_per_update_max=round(max(ms), 4),
        card=card)))
  for line in lines:
    print(line)
  if a.out:
    with open(a.out, 'w') as f:
      f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
  main()
