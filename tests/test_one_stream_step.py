"""The fused step at the agent's batch on ONE stream (csrc/replay.cuh: StageGate::rows;
csrc/step.cu: train_step): sampler -> first half of the loss -> frame copies -> tail +
write-back, each launched programmatically behind the one before, so that every kernel of
a captured step has one parent and the next step's sampler keeps its early launch.

The CPU part models the hand-overs under the edges the hardware gives: a kernel launches
once its predecessor has let its dependents start, and passes its griddepcontrol.wait
once its predecessor has ended.  The copies and the tail learn that the rows are final
from the sampler's count (launch numbers from tickets), not from their predecessor.  The
model checks that no copy or tail reads the rows of another step, that no first half
rewrites a scratch half a tail still reads, and that every launch ends, also when a gate
gives up; and that without the waits at the end of the kernels, or with a sampler that
lets its dependents start before its own wait, some schedule breaks one of these.

The GPU part checks that the one-stream step leaves what the separate calls leave, on a
buffer whose steps alternate with the other paths of the fused step, and that a kernel
queued right behind the call sees this step's frames."""
import os
import random

import numpy as np
import pytest

FRAME = 84 * 84
ACTIONS, ATOMS = 18, 51


class Broken(AssertionError):
  pass


class OneStreamModel:
  """Steps k = 0 .. steps-1 of sampler S, first half P, copies C (c CTAs), tail T (t CTAs).

  end_waits=False: P, C and T end without waiting for their predecessor.
  early_release=True: S lets its dependents start before its own wait.
  timeouts=True: a gate may give up at any poll (then the CTA waits for its predecessor)."""

  def __init__(self, steps, c, t, rng, end_waits=True, early_release=False, timeouts=False):
    self.steps, self.rng = steps, rng
    self.ctas = {'C': c, 'T': t}
    self.end_waits, self.early_release, self.timeouts = end_waits, early_release, timeouts
    self.rows_done = 0
    self.tickets = {'C': 0, 'T': 0}
    self.indices = None      # step whose rows the shared outputs hold
    self.half = [None, None]  # step whose first half last wrote each scratch half
    n = steps
    self.s = [set() for _ in range(n)]  # launched, waited, released, wrote, ended
    self.p = [set() for _ in range(n)]  # launched, signalled, ended
    # per consumer and step: CTAs not started, [launch] at the gate, reading, ended
    self.to_start = {w: [self.ctas[w]] * n for w in 'CT'}
    self.gate = {w: [[] for _ in range(n)] for w in 'CT'}
    self.fallback = {w: [0] * n for w in 'CT'}
    self.reading = {w: [0] * n for w in 'CT'}
    self.ended = {w: [0] * n for w in 'CT'}

  # ---- the edges
  def released(self, who, k):
    if k < 0:
      return True
    if who == 'S':
      return 'released' in self.s[k]
    if who == 'P':
      return 'launched' in self.p[k]  # (lets its dependents start at its first instruction)
    return self.to_start[who][k] == 0

  def done(self, who, k):
    if k < 0:
      return True
    if who == 'S':
      return 'ended' in self.s[k]
    if who == 'P':
      return 'ended' in self.p[k]
    return self.ended[who][k] == self.ctas[who]

  def enabled(self):
    ev = []
    for k in range(self.steps):
      s, p = self.s[k], self.p[k]
      if 'launched' not in s and self.released('T', k - 1):
        ev.append(('s_launch', k))
      if 'launched' in s and 'waited' not in s and self.done('T', k - 1):
        ev.append(('s_wait', k))
      if 'launched' in s and 'released' not in s and (self.early_release or 'waited' in s):
        ev.append(('s_release', k))
      if 'waited' in s and 'wrote' not in s:
        ev.append(('s_write', k))
      if 'wrote' in s and 'ended' not in s and 'signalled' in p:
        ev.append(('s_close', k))  # (PreSync: after the first half's signal)
      if 'launched' not in p and self.released('S', k):
        ev.append(('p_launch', k))
      if 'launched' in p and 'signalled' not in p:
        ev.append(('p_signal', k))
      if 'signalled' in p and 'ended' not in p and (not self.end_waits or self.done('S', k)):
        ev.append(('p_end', k))
      for w, before in (('C', 'P'), ('T', 'C')):
        if self.to_start[w][k] > 0 and self.released(before, k):
          ev.append(('start', w, k))
        if self.gate[w][k]:
          ev.append(('poll', w, k))
          if self.timeouts:
            ev.append(('give_up', w, k))
        if self.fallback[w][k] and self.done(before, k):
          ev.append(('late_read', w, k))
        if self.reading[w][k] and (not self.end_waits or self.done(before, k)):
          ev.append(('end', w, k))
    return ev

  def read(self, w, k):
    if self.indices != k or 'wrote' not in self.s[k]:
      raise Broken('%s of step %d reads the rows of step %s' % (w, k, self.indices))
    if w == 'T' and (self.half[k % 2] != k or 'signalled' not in self.p[k]):
      raise Broken('tail %d reads the scratch of step %s' % (k, self.half[k % 2]))
    self.reading[w][k] += 1

  def run(self):
    while True:
      ev = self.enabled()
      if not ev:
        break
      e = self.rng.choice(ev)
      what, k = e[0], e[-1]
      if what == 's_launch':
        self.s[k].add('launched')
      elif what == 's_wait':
        self.s[k].add('waited')
      elif what == 's_release':
        self.s[k].add('released')
      elif what == 's_write':
        for w in 'CT':  # the rows of step k - 1 are overwritten now
          if k > 0 and self.reading[w][k - 1]:
            raise Broken('sampler %d overwrites rows %s %d still reads' % (k, w, k - 1))
        self.indices = k
        self.s[k].add('wrote')
      elif what == 's_close':
        self.rows_done += 1
        self.s[k].add('ended')
      elif what == 'p_launch':
        for j in range(self.steps):
          if j % 2 == k % 2 and j != k and self.reading['T'][j]:
            raise Broken('first half %d rewrites the half tail %d reads' % (k, j))
        self.half[k % 2] = k
        self.p[k].add('launched')
      elif what == 'p_signal':
        self.p[k].add('signalled')
      elif what == 'p_end':
        self.p[k].add('ended')
      elif what == 'start':
        w = e[1]
        launch = self.tickets[w] // self.ctas[w]
        if launch != k:
          raise Broken('the tickets of %s launches %d and %d interleave' % (w, launch, k))
        self.tickets[w] += 1
        self.to_start[w][k] -= 1
        self.gate[w][k].append(launch)
      elif what == 'poll':
        w = e[1]
        if self.rows_done >= self.gate[w][k][0] + 1:
          self.gate[w][k].pop(0)
          self.read(w, k)
      elif what == 'give_up':
        w = e[1]
        self.gate[w][k].pop(0)
        self.fallback[w][k] += 1
      elif what == 'late_read':
        w = e[1]
        self.fallback[w][k] -= 1
        self.read(w, k)
      elif what == 'end':
        w = e[1]
        self.reading[w][k] -= 1
        self.ended[w][k] += 1
    for k in range(self.steps):
      assert self.done('T', k) and self.done('C', k) and self.done('S', k), 'step %d hangs' % k
    assert self.rows_done == self.steps
    return self


def _breaks(**kw):
  for seed in range(400):
    try:
      OneStreamModel(steps=5, c=2, t=2, rng=random.Random(seed), **kw).run()
    except Broken:
      return True
  return False


@pytest.mark.parametrize('timeouts', [False, True])
@pytest.mark.parametrize('ctas', [(1, 1), (3, 2)])
def test_one_stream_hand_overs_are_safe(timeouts, ctas):
  for seed in range(300):
    OneStreamModel(steps=6, c=ctas[0], t=ctas[1], timeouts=timeouts,
                   rng=random.Random(seed * 17 + ctas[0] + 5 * timeouts)).run()


def test_without_the_waits_at_the_end_some_schedule_breaks():
  assert _breaks(end_waits=False)


def test_a_sampler_releasing_before_its_wait_lets_some_schedule_break():
  assert _breaks(early_release=True)


# ---------------------------------------------------------------------------- GPU


@pytest.fixture(scope='module')
def gpu():
  import torch
  if not torch.cuda.is_available():
    pytest.fail('-m gpu tests need a CUDA device (no CPU fallback exists)')
  from dopamine_b200 import _native
  from dopamine_b200.agents.rainbow import rainbow_agent
  from dopamine_b200.replay_memory import prioritized_replay_buffer as prb

  class Mods(object):
    pass

  m = Mods()
  m.torch, m.prb, m.ra, m.native = torch, prb, rainbow_agent, _native
  return m


def _filled(gpu, cap, batch, seed, term_p=0.2):
  """A full prioritized buffer with many terminal transitions."""
  rng = np.random.RandomState(seed)
  mem = gpu.prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed)
  mem._store['observation'] = rng.randint(0, 256, size=(cap, 84, 84)).astype(np.uint8)
  mem._store['action'] = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < term_p).astype(np.uint8)
  mem.add_count = cap + 77
  mem.invalid_range = np.array([(77 - 3 + i) % cap for i in range(7)])
  ids = np.arange(cap, dtype=np.int32)
  mem.set_priority(ids, np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(np.float32))
  return mem


def _same(a, b, what):
  assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes(), what


def _check_step(gpu, mirror, batch, cols, out, online, target, support, what):
  """cols: the step's batch (state, action, reward, next_state, ..., indices, probs).
  Frames equal a gather of its indices, the loss columns equal c51_loss over its scalars;
  the mirror buffer takes the same write-back through set_priority."""
  gpu.torch.cuda.synchronize()
  want = mirror.sample_transition_batch(batch, indices=cols[7].cpu().numpy())
  for k in (0, 1, 2, 3, 6):
    _same(cols[k], want[k], '%s: column %d' % (what, k))
  ref = gpu.ra.c51_loss(online, target, cols[1], cols[2], cols[6], cols[8], support,
                        0.99 ** 3, want_mean=False)
  for key in ('loss', 'priorities', 'weights'):
    _same(out[key], ref[key], '%s: %s' % (what, key))
  mirror.set_priority(cols[7], out['priorities'])


def _trainer_cols(tr):
  return [tr[k] for k in ('state', 'action', 'reward', 'next_state', 'next_action',
                          'next_reward', 'terminal', 'indices', 'sampling_probabilities')]


@pytest.mark.gpu
@pytest.mark.parametrize('batch', [1, 5, 31, 32])
def test_one_stream_steps_between_the_other_paths(gpu, batch):
  """One buffer: one-stream steps alternate with deferred-copy steps and with the trainer
  (eager copy path, direct I/O, graph mode).  Every step's frames, scalars, losses,
  priorities and weights equal the separate calls over its batch, and the tree equals a
  twin that took every write-back through set_priority.  The frames of a one-stream step
  are cloned by a kernel queued right behind the call on the same stream."""
  torch, native = gpu.torch, gpu.native
  lib = native.lib()
  cap = 20000
  mem = _filled(gpu, cap, batch, seed=40 + batch)
  mirror = _filled(gpu, cap, batch, seed=40 + batch)
  rng = np.random.RandomState(batch)
  support = gpu.ra.make_support(10., ATOMS)
  trainers = {}
  for name, direct, graph in (('copy', '0', False), ('direct', '1', False),
                              ('graph', '0', True)):
    os.environ['B2R_TRAINER_DIRECT'] = direct
    try:
      trainers[name] = gpu.ra.ReplayTrainer(mem, ACTIONS, ATOMS, 10., pipeline_depth=0,
                                            seed=7, use_graph=graph)
    finally:
      os.environ.pop('B2R_TRAINER_DIRECT', None)
  modes = ['one', 'deferred', 'one', 'copy', 'one', 'direct', 'one', 'graph', 'one',
           'graph', 'one', 'graph', 'one', 'deferred', 'one']
  terminal_rows = 0
  for step, mode in enumerate(modes):
    what = '%s step %d' % (mode, step)
    logits = [rng.randn(batch, ACTIONS, ATOMS).astype(np.float32) * 3 for _ in range(2)]
    online, target = (torch.as_tensor(x, device='cuda') for x in logits)
    if mode in ('one', 'deferred'):
      stream = native.current_stream()
      if mode == 'deferred':
        native.check(lib.b2r_set_deferred_frames(mem._h, 1))
      got, out = gpu.ra.train_step(mem, online, target, support, 0.99 ** 3)
      if mode == 'deferred':
        native.check(lib.b2r_join_frames(mem._h, stream))
        native.check(lib.b2r_set_deferred_frames(mem._h, 0))
      cols = [c.clone() for c in got]  # (same stream, right behind the call)
      _check_step(gpu, mirror, batch, cols, out, online, target, support, what)
      terminal_rows += int(cols[6].sum())
    else:
      pin = [torch.from_numpy(x).pin_memory() for x in logits]
      loss, done = trainers[mode].step(pin[0], pin[1])
      assert done >= 0
      torch.cuda.synchronize()
      tr, out = trainers[mode].views()
      _check_step(gpu, mirror, batch, _trainer_cols(tr), out, online, target, support, what)
      assert loss.tobytes() == out['loss'].cpu().numpy().tobytes(), what
  assert batch < 5 or terminal_rows > 0
  torch.cuda.synchronize()
  for la, lb in zip(mem.sum_tree.nodes, mirror.sum_tree.nodes):
    assert np.array_equal(la.view(np.uint64), lb.view(np.uint64))
  native.check(lib.b2r_check(mem._h, native.current_stream()))


@pytest.mark.gpu
def test_one_stream_graph_frames_seen_by_the_next_kernel(gpu):
  """Ten one-stream steps in ONE captured graph, each followed on the same stream by a
  kernel that clones its batch: every clone holds that step's frames and scalars, and the
  losses equal c51_loss over them."""
  torch = gpu.torch
  batch, cap = 32, 20000
  mem = _filled(gpu, cap, batch, seed=21)
  mirror = _filled(gpu, cap, batch, seed=21)
  mem._reuse_outputs = True
  rng = np.random.RandomState(22)
  support = gpu.ra.make_support(10., ATOMS)
  logits = [tuple(torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32) * 3,
                                  device='cuda') for _ in range(2)) for _ in range(11)]
  outs = [{k: torch.empty(batch, device='cuda') for k in ('loss', 'priorities', 'weights')}
          for _ in range(11)]
  clones = [None] * 11
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    got, _ = gpu.ra.train_step(mem, logits[0][0], logits[0][1], support, 0.99 ** 3,
                               out=outs[0])
    clones[0] = [c.clone() for c in got]
    side.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
      for k in range(1, 11):
        got, _ = gpu.ra.train_step(mem, logits[k][0], logits[k][1], support, 0.99 ** 3,
                                   out=outs[k])
        clones[k] = [c.clone() for c in got]
    graph.replay()
    side.synchronize()
  torch.cuda.current_stream().wait_stream(side)
  for k in range(11):
    _check_step(gpu, mirror, batch, clones[k], outs[k], logits[k][0], logits[k][1],
                support, 'graph step %d' % k)
  for la, lb in zip(mem.sum_tree.nodes, mirror.sum_tree.nodes):
    assert np.array_equal(la.view(np.uint64), lb.view(np.uint64))
