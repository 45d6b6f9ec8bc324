"""Kernel launch lists of the library's host paths, for comparing two builds.

  python profiles/launch_list.py --libs OLD.so,NEW.so [--out DIR]

Runs every scenario below once per library (each in its own process, the library
chosen through B2R_LIB) under torch.profiler with CUDA activities and with
b2r_launch_count().  Every scenario runs once unprofiled first, so that one-time set-up
(scratch growth, shared-memory opt-ins) is outside the list.  A kernel is listed by
name, grid, block, shared memory and stream (numbered in order of first use), in the
order of the launches (correlation ids).  Prints one JSON line per scenario saying
whether the two builds launched the same kernels in the same order with the same
configurations and counted the same launches; exits non-zero otherwise.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
ACTIONS = 18


def kernels(prof):
  """[(name, grid, block, shared memory, stream index)] in launch order."""
  with tempfile.TemporaryDirectory() as tmp:
    path = os.path.join(tmp, 'trace.json')
    prof.export_chrome_trace(path)
    with open(path) as f:
      events = json.load(f)['traceEvents']
  rows = [e for e in events if e.get('cat') == 'kernel']
  rows.sort(key=lambda e: e['args'].get('correlation', 0))
  streams = {}
  out = []
  for e in rows:
    a = e['args']
    s = streams.setdefault(a.get('stream'), len(streams))
    out.append([e['name'], a.get('grid'), a.get('block'), a.get('shared memory'), s])
  return out


def scenarios():
  """[(name, call)]: each call runs once unprofiled, then once profiled."""
  import bench  # noqa: E402
  import torch
  from dopamine_b200 import _native
  from dopamine_b200.agents.rainbow import agent
  from dopamine_b200.agents.rainbow import rainbow_agent
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb
  from dopamine_b200.replay_memory import sharded_replay

  wl = bench.GpuWorkload(200000, 4096, 0)
  mem = wl.mem
  out = []
  for batch in (32, 256, 1024, 4096):  # 32: the one-stream order
    out.append(('fused_step_%d' % batch, lambda b=batch: wl.step(b)))

  rng = np.random.RandomState(3)
  frames = rng.randint(0, 256, size=(64, 84, 84)).astype(np.uint8)
  online = wl.online[:32].cpu().pin_memory()
  target = wl.target[:32].cpu().pin_memory()
  for depth in (0, 2):
    trainer = rainbow_agent.ReplayTrainer(mem, bench.NUM_ACTIONS, bench.NUM_ATOMS, bench.VMAX,
                                          batch_size=32, pipeline_depth=depth, seed=wl.seed)

    def train(trainer=trainer, k=[0]):
      for _ in range(4):
        mem.add(frames[k[0] & 63], k[0] % bench.NUM_ACTIONS, 0.5, 0,
                prb.MAX_RECORDED_PRIORITY)
        k[0] += 1
      trainer.step_pointers(online.data_ptr(), target.data_ptr(),
                            _native.current_stream())
      trainer.drain()
    out.append(('trainer_depth_%d' % depth, train))

  def add_flush():
    for k in range(40):
      mem.add(frames[k & 63], k % bench.NUM_ACTIONS, 0.5, 0, prb.MAX_RECORDED_PRIORITY)
    mem.sample_transition_batch(32)
  out.append(('add_flush_40', add_flush))

  for n in (32, 200, 5000):
    idx = rng.randint(0, 200000 - 10, size=n).astype(np.int32)
    pr = rng.rand(n).astype(np.float32) + 0.1
    out.append(('set_priority_host_%d' % n, lambda i=idx, p=pr: mem.set_priority(i, p)))

  for kind in ('reference', 'device'):
    for cls in (crb.OutOfGraphReplayBuffer, prb.OutOfGraphPrioritizedReplayBuffer):
      small = cls((84, 84), 4, 1000, 32, update_horizon=3, output='torch', rng=kind, seed=5)
      prio = (prb.MAX_RECORDED_PRIORITY,) if cls is not crb.OutOfGraphReplayBuffer else ()
      for k in range(300):
        small.add(frames[k & 63], k % bench.NUM_ACTIONS, 0.5, int(k % 97 == 96), *prio)
      out.append(('sample_transition_batch_%s_%s' % (cls.__name__, kind),
                  lambda m=small: m.sample_transition_batch(32)))

  # two ranks emulated on one device: publish, sampler, loss and write-back of each
  torch.backends.cudnn.deterministic = True
  torch.backends.cudnn.benchmark = False
  xs = sharded_replay.PeerExchange.emulated(2)
  learners = []
  for g in range(2):
    shard = prb.OutOfGraphPrioritizedReplayBuffer(
        (84, 84), 4, 4000, 64, update_horizon=3, gamma=0.99, output='torch',
        rng='device', seed=100 + g, reuse_outputs=True)
    for k in range(600):
      shard.add(frames[(k + g) & 63], k % ACTIONS, 0.5, int(k % 211 == 210),
                prb.MAX_RECORDED_PRIORITY)
    learners.append(agent.ShardedRainbowLearner(
        ACTIONS, batch_size=64, exchange=xs[g], memory=shard, replay_scheme='prioritized',
        replay_capacity=4000, seed=3))

  def sharded_step():
    for x, l in zip(xs, learners):
      x.publish(l.memory)
    for l in learners:
      l.sample()
    prios = [l.loss_backward() for l in learners]
    total = sum(l._flat for l in learners)  # pylint: disable=protected-access
    for l in learners:
      l._flat.copy_(total)  # pylint: disable=protected-access
    for l, p in zip(learners, prios):
      l.apply(p)
  out.append(('sharded_step_2_ranks', sharded_step))
  return out


def record(path):
  import torch
  from torch.profiler import ProfilerActivity, profile
  from dopamine_b200 import _native
  lib = _native.lib()
  random.seed(1)  # the reference-RNG buffers draw their queries from `random`
  result = {}
  for name, call in scenarios():
    call()
    torch.cuda.synchronize()
    n0 = lib.b2r_launch_count()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
      call()
      torch.cuda.synchronize()
    result[name] = {'launches': lib.b2r_launch_count() - n0, 'kernels': kernels(prof)}
  with open(path, 'w') as f:
    json.dump(result, f)


def main():
  p = argparse.ArgumentParser()
  p.add_argument('--libs', help='two library paths, comma-separated')
  p.add_argument('--out', help='where the two lists go (default: a new temporary directory)')
  p.add_argument('--record', help=argparse.SUPPRESS)
  a = p.parse_args()
  if a.record:
    record(a.record)
    return 0
  libs = a.libs.split(',')
  a.out = a.out or tempfile.mkdtemp(prefix='launch_list_')
  os.makedirs(a.out, exist_ok=True)
  runs = []
  for i, lib in enumerate(libs):
    path = os.path.join(a.out, 'launch_list_%d.json' % i)
    subprocess.check_call([sys.executable, os.path.abspath(__file__), '--record', path],
                          env=dict(os.environ, B2R_LIB=os.path.abspath(lib)))
    with open(path) as f:
      runs.append(json.load(f))
  same = True
  for name in runs[0]:
    x, y = runs[0][name], runs[1].get(name)
    ok = y is not None and x == y
    same &= ok
    b2r = sum('b2r::' in k[0] for k in x['kernels'])
    print(json.dumps({'scenario': name, 'identical': ok, 'kernels': len(x['kernels']),
                      'library_kernels': b2r, 'launch_count': x['launches'],
                      'launch_count_other': y and y['launches']}), flush=True)
    if not ok and y is not None:
      for i, (kx, ky) in enumerate(zip(x['kernels'], y['kernels'])):
        if kx != ky:
          print('  first difference at %d: %s | %s' % (i, kx, ky))
          break
  return 0 if same else 1


if __name__ == '__main__':
  sys.exit(main())
