"""The fused step with the loss in ONE kernel (more than 64 atoms) at 256 and 1024 rows.

That loss cannot run in two halves (c51_can_split), so nothing signals the early
write-back and the step's write-back is the plain tree_update_kernel launch (kFull) on
the caller's stream.  This script times b2r_train_step_device there with CUDA events and
dumps every tree level after a few seeded steps, so that two builds can be compared for
time and for bits:

  python profiles/r5/unsplit_writeback.py --out DIR

writes DIR/times.json and DIR/tree_<rows>.npy (all levels, as uint64 bit patterns) and
DIR/loss_<rows>.npy.  The buffer is test_gpu_step.py's: a full 200 000-slot ring with
Atari-sized frames and random priorities, high-priority slots in the invalid window.
"""
import argparse
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.test_gpu_step import ACTIONS, _filled  # noqa: E402


def main():
  p = argparse.ArgumentParser()
  p.add_argument('--atoms', type=int, default=101)
  p.add_argument('--rows', type=int, nargs='+', default=[256, 1024])
  p.add_argument('--cap', type=int, default=200000)
  p.add_argument('--warmup', type=int, default=20)
  p.add_argument('--steps', type=int, default=200)
  p.add_argument('--check-steps', type=int, default=5)
  p.add_argument('--out', required=True)
  a = p.parse_args()
  import torch
  assert torch.cuda.is_available(), 'needs a CUDA device'
  from dopamine_b200.agents.rainbow import rainbow_agent as ra
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  gpu = types.SimpleNamespace(prb=prb)
  os.makedirs(a.out, exist_ok=True)
  support = ra.make_support(10., a.atoms)
  result = {'atoms': a.atoms, 'cap': a.cap, 'steps': a.steps,
            'card': torch.cuda.get_device_name(0), 'rows': {}}
  for rows in a.rows:
    rng = np.random.RandomState(rows)
    shape = (rows, ACTIONS, a.atoms)

    def logits():
      return (torch.as_tensor(rng.randn(*shape).astype(np.float32), device='cuda'),
              torch.as_tensor(rng.randn(*shape).astype(np.float32), device='cuda'))

    # same bits: a fresh buffer, seeded logits, a few steps, then every tree level
    mem, _, _ = _filled(gpu, a.cap, rows, seed=3)
    out = None
    for _ in range(a.check_steps):
      online, target = logits()
      _, out = ra.train_step(mem, online, target, support, 0.99 ** 3, out=out)
    torch.cuda.synchronize()
    levels = mem.sum_tree.nodes
    np.save(os.path.join(a.out, 'tree_%d.npy' % rows),
            np.concatenate([l.view(np.uint64) for l in levels]))
    np.save(os.path.join(a.out, 'loss_%d.npy' % rows), out['loss'].cpu().numpy())
    # time: fixed logits, steady state; eager calls, then 10 steps per CUDA graph (no
    # host cost between the steps)
    online, target = logits()
    mem._reuse_outputs = True
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(side):
      for _ in range(a.warmup):
        ra.train_step(mem, online, target, support, 0.99 ** 3, out=out)
      side.synchronize()
      t0.record(side)
      for _ in range(a.steps):
        ra.train_step(mem, online, target, support, 0.99 ** 3, out=out)
      t1.record(side)
      t1.synchronize()
      eager = t0.elapsed_time(t1) * 1e3 / a.steps
      graph = torch.cuda.CUDAGraph()
      with torch.cuda.graph(graph, stream=side):
        for _ in range(10):
          ra.train_step(mem, online, target, support, 0.99 ** 3, out=out)
      for _ in range(max(1, a.warmup // 10)):
        graph.replay()
      side.synchronize()
      t0.record(side)
      for _ in range(a.steps // 10):
        graph.replay()
      t1.record(side)
      t1.synchronize()
      graphed = t0.elapsed_time(t1) * 1e3 / (a.steps // 10 * 10)
    torch.cuda.current_stream().wait_stream(side)
    result['rows'][str(rows)] = {'eager_us_per_step': round(eager, 3),
                                 'graph_us_per_step': round(graphed, 3)}
    print('rows %d atoms %d: %.3f us per step eager, %.3f in a graph' %
          (rows, a.atoms, eager, graphed), flush=True)
    del graph, mem
  with open(os.path.join(a.out, 'times.json'), 'w') as f:
    json.dump(result, f, indent=1)


if __name__ == '__main__':
  main()
