"""The loss tail of the fused step at the agent's batch stages its inputs from the first
half of the loss while the sampler is still running (csrc/replay.cuh: StageGate::first_half;
csrc/c51.cu: c51_post_tree_kernel<true>).

The CPU part models the hand-shake.  The first half of step k runs on a side stream and
counts itself in `done` when its last CTA leaves; the tail of step k is resident long
before that and reads the scratch half k % 2, which every step rewrites.  Every CTA of a
tail takes a ticket before it lets its dependents start (so ticket // ctas numbers the
launches) and stages once done >= its launch's number + 1.  The model drives random
interleavings under the ordering the hardware gives — first halves in stream order, each
behind the tail that last read its half (the caller's stream, or the trainer's
first_half_after event two steps back), programmatic launch edges on the chain — and
checks that no tail reads a first half other than its own step's, that no first half
overwrites a half a tail is still reading, and that every launch ends.

The GPU part checks that the staged tail leaves the bits the separate calls leave."""
import os
import random

import numpy as np
import pytest

FRAME = 84 * 84
ACTIONS, ATOMS = 18, 51


class GateModel:
  """direct=False: the first half of step k is forked from the caller's stream behind the
  tail of step k - 1.  direct=True (the trainer's direct I/O): it waits only for the
  tail of step k - 2 (and for the first half of step k - 1: same stream)."""

  def __init__(self, steps, ctas, direct, rng, boolean=False):
    self.steps, self.ctas, self.direct, self.rng = steps, ctas, direct, rng
    self.boolean = boolean  # a done flag instead of a launch number (the stale variant)
    self.done = 0
    self.tickets = 0
    self.half = [None, None]      # step whose first half last completed each half
    self.writing = [None, None]   # step whose first half is writing each half now
    self.pre_state = ['wait'] * steps  # wait -> running -> done
    self.sampler_released = [False] * steps
    self.sampler_ended = [False] * steps
    self.to_start = [ctas] * steps     # tail CTAs not yet resident
    self.waiting = [[] for _ in range(steps)]  # launch numbers of CTAs at the gate
    self.staged = [0] * steps          # CTAs that have staged (and released)
    self.left = [0] * steps
    self.stale = False

  def tail_ended(self, k):
    return k < 0 or self.left[k] == self.ctas

  def tail_released(self, k):
    return k < 0 or (self.to_start[k] == 0 and not self.waiting[k])

  def enabled(self):
    ev = []
    for k in range(self.steps):
      behind = k - 2 if self.direct else k - 1
      prev_pre_done = k == 0 or self.pre_state[k - 1] == 'done'
      if self.pre_state[k] == 'wait' and prev_pre_done and self.tail_ended(behind):
        ev.append(('pre_starts', k))
      if self.pre_state[k] == 'running':
        ev.append(('pre_ends', k))
      # the sampler of step k follows the tail of step k - 1 programmatically: resident
      # once that tail has released, ended only after it has ended
      if not self.sampler_released[k] and self.tail_released(k - 1):
        ev.append(('sampler_releases', k))
      if (self.sampler_released[k] and not self.sampler_ended[k] and
          self.tail_ended(k - 1) and self.pre_state[k] == 'done'):
        ev.append(('sampler_ends', k))  # (PreSync: it waits for the first half too)
      if self.to_start[k] > 0 and self.sampler_released[k]:
        ev.append(('cta_starts', k))
      if self.waiting[k]:
        ev.append(('cta_polls', k))
      if self.staged[k] > self.left[k] and self.sampler_ended[k]:
        ev.append(('cta_leaves', k))
    return ev

  def run(self):
    while True:
      ev = self.enabled()
      if not ev:
        break
      what, k = self.rng.choice(ev)
      p = k % 2
      if what == 'pre_starts':
        # nobody may still be reading the half this first half rewrites
        for j in range(self.steps):
          if j % 2 == p and j != k and self.staged[j] > self.left[j]:
            raise AssertionError('first half %d overwrites a half tail %d reads' % (k, j))
        self.pre_state[k] = 'running'
        self.writing[p] = k
      elif what == 'pre_ends':
        self.pre_state[k] = 'done'
        self.writing[p] = None
        self.half[p] = k
        self.done += 1
      elif what == 'sampler_releases':
        self.sampler_released[k] = True
      elif what == 'sampler_ends':
        self.sampler_ended[k] = True
      elif what == 'cta_starts':
        self.to_start[k] -= 1
        self.waiting[k].append(self.tickets // self.ctas)
        self.tickets += 1
      elif what == 'cta_polls':
        launch = self.waiting[k][0]
        assert launch == k, 'tickets number the launches'
        go = self.done >= 1 if self.boolean else self.done >= launch + 1
        if go:
          if self.half[p] != k or self.writing[p] is not None:
            if self.boolean:
              self.stale = True
            else:
              raise AssertionError('tail %d staged the rows of step %s' % (k, self.half[p]))
          self.waiting[k].pop(0)
          self.staged[k] += 1
      elif what == 'cta_leaves':
        self.left[k] += 1
    assert all(self.tail_ended(k) for k in range(self.steps)), 'every launch ran to its end'
    assert self.done == self.steps and self.tickets == self.steps * self.ctas
    return self


@pytest.mark.parametrize('direct', [False, True])
@pytest.mark.parametrize('ctas', [1, 8])
def test_no_tail_stages_a_stale_first_half(direct, ctas):
  for seed in range(300):
    GateModel(steps=7, ctas=ctas, direct=direct,
              rng=random.Random(seed * 131 + ctas * 7 + direct)).run()


def test_a_done_flag_would_be_read_stale():
  """The same interleavings with "some first half has ended" in place of the launch
  number: some schedule lets a tail stage rows of another step."""
  assert any(GateModel(steps=6, ctas=2, direct=True, rng=random.Random(s),
                       boolean=True).run().stale for s in range(300))


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


def _filled(gpu, cap, batch, seed, term_p=0.2, bad_actions=False):
  """A full prioritized buffer with many terminal transitions (and, with bad_actions,
  every third stored action outside [0, ACTIONS))."""
  rng = np.random.RandomState(seed)
  mem = gpu.prb.OutOfGraphPrioritizedReplayBuffer(
      (84, 84), 4, cap, batch, update_horizon=3, gamma=0.99, output='torch',
      rng='device', seed=seed)
  obs = rng.randint(0, 256, size=(cap, FRAME)).astype(np.uint8)
  action = rng.randint(0, ACTIONS, size=cap).astype(np.int32)
  if bad_actions:
    action[::3] = np.where(np.arange(cap)[::3] % 2 == 0, ACTIONS, -1)
  mem._store['observation'] = obs.reshape(cap, 84, 84)
  mem._store['action'] = action
  mem._store['reward'] = np.clip(rng.randn(cap), -1, 1).astype(np.float32)
  mem._store['terminal'] = (rng.rand(cap) < term_p).astype(np.uint8)
  mem.add_count = cap + 77
  mem.invalid_range = np.array([(77 - 3 + i) % cap for i in range(7)])
  ids = np.arange(cap, dtype=np.int32)
  mem.set_priority(ids, np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(np.float32))
  return mem


def _separate(gpu, mem, batch, online, target, support):
  got = mem.sample_transition_batch(batch)
  out = gpu.ra.c51_loss(online, target, got[1], got[2], got[6], got[8], support, 0.99 ** 3,
                        want_mean=False)
  mem.set_priority(got[7], out['priorities'])
  return got, out


def _same(a, b, what):
  assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes(), what


def _same_tree(mem_a, mem_b):
  for la, lb in zip(mem_a.sum_tree.nodes, mem_b.sum_tree.nodes):
    assert np.array_equal(la.view(np.uint64), lb.view(np.uint64))


@pytest.mark.gpu
@pytest.mark.parametrize('batch', [1, 5, 31, 32])
def test_staged_tail_equals_separate_calls(gpu, batch):
  """Twin buffers, same seed, fresh logits every step (a tail that staged the previous
  step's first half would show), terminal rows in most batches: 12 fused steps in a row
  leave the bits of sample -> c51_loss -> set_priority, step by step."""
  torch = gpu.torch
  cap = 20000
  mem_a = _filled(gpu, cap, batch, seed=31 + batch)
  mem_b = _filled(gpu, cap, batch, seed=31 + batch)
  rng = np.random.RandomState(batch)
  support = gpu.ra.make_support(10., ATOMS)
  terminal_rows = 0
  for step in range(12):
    online = torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32) * 3,
                             device='cuda')
    target = torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32) * 3,
                             device='cuda')
    got_a, out_a = gpu.ra.train_step(mem_a, online, target, support, 0.99 ** 3)
    got_b, out_b = _separate(gpu, mem_b, batch, online, target, support)
    torch.cuda.synchronize()
    for k, (a, b) in enumerate(zip(got_a, got_b)):
      _same(a, b, 'column %d, step %d' % (k, step))
    for key in ('loss', 'priorities', 'weights'):
      _same(out_a[key], out_b[key], '%s, step %d' % (key, step))
    terminal_rows += int(got_a[6].sum())
  assert batch < 5 or terminal_rows > 0
  _same_tree(mem_a, mem_b)
  gpu.native.check(gpu.native.lib().b2r_check(mem_a._h, gpu.native.current_stream()))


@pytest.mark.gpu
def test_staged_tail_out_of_range_action(gpu):
  """A sampled action outside [0, A): the row is evaluated for action 0 with a zero loss,
  as the one-kernel loss does, and the fused step latches B2R_ERR_INDEX_RANGE."""
  torch, native = gpu.torch, gpu.native
  batch, cap = 32, 20000
  mem_a = _filled(gpu, cap, batch, seed=5, bad_actions=True)
  mem_b = _filled(gpu, cap, batch, seed=5, bad_actions=True)
  rng = np.random.RandomState(6)
  support = gpu.ra.make_support(10., ATOMS)
  online = torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32), device='cuda')
  target = torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32), device='cuda')
  got_a, out_a = gpu.ra.train_step(mem_a, online, target, support, 0.99 ** 3)
  got_b, out_b = _separate(gpu, mem_b, batch, online, target, support)
  torch.cuda.synchronize()
  act = got_a[1].cpu().numpy()
  bad = (act < 0) | (act >= ACTIONS)
  assert bad.any() and not bad.all()
  assert (out_a['loss'].cpu().numpy()[bad] == 0).all()
  for key in ('loss', 'priorities', 'weights'):
    _same(out_a[key], out_b[key], key)
  _same_tree(mem_a, mem_b)
  status = native.lib().b2r_check(mem_a._h, native.current_stream())
  assert status == native.ERR_INDEX_RANGE, (status, native.last_error())


@pytest.mark.gpu
def test_staged_tail_in_one_graph_of_ten_steps(gpu):
  """Ten fused steps captured in ONE graph, each on its own logits, replayed once: every
  step's losses, priorities and weights, the last batch and the tree equal ten eager
  steps on a twin buffer."""
  torch = gpu.torch
  batch, cap = 32, 20000
  mem_a = _filled(gpu, cap, batch, seed=8)
  mem_b = _filled(gpu, cap, batch, seed=8)
  mem_a._reuse_outputs = mem_b._reuse_outputs = True
  rng = np.random.RandomState(10)
  support = gpu.ra.make_support(10., ATOMS)
  logits = [tuple(torch.as_tensor(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32),
                                  device='cuda') for _ in range(2)) for _ in range(11)]
  outs = [{k: torch.empty(batch, device='cuda') for k in ('loss', 'priorities', 'weights')}
          for _ in range(11)]
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    gpu.ra.train_step(mem_a, logits[0][0], logits[0][1], support, 0.99 ** 3, out=outs[0])
    side.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
      for k in range(1, 11):
        got_a, _ = gpu.ra.train_step(mem_a, logits[k][0], logits[k][1], support,
                                     0.99 ** 3, out=outs[k])
    graph.replay()
    side.synchronize()
  torch.cuda.current_stream().wait_stream(side)
  for k in range(11):
    got_b, out_b = gpu.ra.train_step(mem_b, logits[k][0], logits[k][1], support, 0.99 ** 3)
    torch.cuda.synchronize()
    for key in ('loss', 'priorities', 'weights'):
      _same(outs[k][key], out_b[key], '%s, step %d' % (key, k))
  for a, b in zip(got_a, got_b):
    _same(a, b, 'last batch')
  _same_tree(mem_a, mem_b)


@pytest.mark.gpu
def test_staged_tail_under_the_trainers_direct_io(gpu):
  """The synchronous trainer with page-locked logits: the first half reads them in place
  (and leaves the device copy), the staged tail writes the losses into the result ring.
  Every step equals c51_loss over the batch the trainer sampled, bit for bit."""
  torch = gpu.torch
  batch, cap = 32, 20000
  os.environ['B2R_TRAINER_DIRECT'] = '1'
  try:
    mem = _filled(gpu, cap, batch, seed=12)
    trainer = gpu.ra.ReplayTrainer(mem, ACTIONS, ATOMS, 10., pipeline_depth=0, seed=12)
    support = gpu.ra.make_support(10., ATOMS)
    rng = np.random.RandomState(13)
    pin = [(torch.empty(batch, ACTIONS, ATOMS).pin_memory(),
            torch.empty(batch, ACTIONS, ATOMS).pin_memory()) for _ in range(8)]
    for step in range(8):
      for x in pin[step]:
        x.copy_(torch.from_numpy(rng.randn(batch, ACTIONS, ATOMS).astype(np.float32)))
      loss, done = trainer.step(pin[step][0], pin[step][1])
      assert done == step
      torch.cuda.synchronize()
      tr, out = trainer.views()
      ref = gpu.ra.c51_loss(pin[step][0].cuda(), pin[step][1].cuda(), tr['action'],
                            tr['reward'], tr['terminal'], tr['sampling_probabilities'],
                            support, 0.99 ** 3, want_mean=False)
      torch.cuda.synchronize()
      assert loss.tobytes() == ref['loss'].cpu().numpy().tobytes(), step
      for key in ('loss', 'priorities', 'weights'):
        _same(out[key], ref[key], '%s, step %d' % (key, step))
  finally:
    os.environ.pop('B2R_TRAINER_DIRECT', None)
