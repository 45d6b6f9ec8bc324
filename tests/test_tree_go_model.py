"""CPU model of the "indices are final" hand-shake between the loss tail and the early tree
write-back (csrc/tree.cuh: TreeGo, tree_go_signal, the words TreeSync::go and ::completed;
csrc/tree.cu: tree_update_early_kernel, whose tickets come from launch_ticket).

The write-back of step k is RESIDENT while the sampler and the loss tail of step k still
run — and, one programmatic launch further, so may be the write-back of step k + 1 while
step k's has not finished.  A boolean "go" flag would be read stale by the later launch.
The protocol instead:
  * every CTA of an early write-back takes a ticket from a counter that only grows, BEFORE
    it lets its dependents start — so all CTAs of launch k hold tickets
    [k * ctas, (k + 1) * ctas) and ticket // ctas is the launch's number;
  * the last CTA of a launch to leave counts it in `completed`;
  * the loss tail of step k runs its signal after the sampler of step k has ended, i.e.
    after write-back k - 1 has ended and before write-back k can have: it stores
    completed + 1 (= k + 1) in `go`;
  * a CTA proceeds only when go == its launch's number + 1.
This file drives random interleavings of those events under exactly the ordering
constraints the hardware gives (stream order and programmatic launch edges) and checks
that no CTA ever proceeds before ITS step's signal, and that every CTA does proceed."""
import random

import pytest


class Model:
  def __init__(self, steps, ctas, rng):
    self.steps, self.ctas, self.rng = steps, ctas, rng
    self.tickets = 0
    self.completed = 0
    self.go = 0
    self.sampler_done = [False] * steps
    self.signalled = [False] * steps
    # per step: CTAs not yet started / waiting (with their launch number) / working / left
    self.to_start = [ctas] * steps
    self.waiting = [[] for _ in range(steps)]
    self.working = [0] * steps
    self.left = [0] * steps
    self.tree_done = [False] * steps

  def enabled(self):
    ev = []
    for k in range(self.steps):
      prev_tree_done = k == 0 or self.tree_done[k - 1]
      # the sampler of step k ends only after write-back k - 1 has (stream order)
      if not self.sampler_done[k] and prev_tree_done:
        ev.append(('sampler_ends', k))
      # the loss tail's signal: behind its wait for the sampler
      if self.sampler_done[k] and not self.signalled[k]:
        ev.append(('signal', k))
      # a CTA of write-back k may become resident as soon as every CTA of write-back
      # k - 1 has let its dependents start (which it does only after its ticket AND its
      # go — tree.cu releases behind the wait): i.e. once none of them is unstarted/waiting
      prev_released = k == 0 or (self.to_start[k - 1] == 0 and not self.waiting[k - 1])
      if self.to_start[k] > 0 and prev_released:
        ev.append(('cta_starts', k))
      if self.waiting[k]:
        ev.append(('cta_polls', k))
      if self.working[k] > 0 and self.signalled[k]:
        ev.append(('cta_leaves', k))
    return ev

  def run(self):
    while True:
      ev = self.enabled()
      if not ev:
        break
      what, k = self.rng.choice(ev)
      if what == 'sampler_ends':
        self.sampler_done[k] = True
      elif what == 'signal':
        self.go = self.completed + 1
        self.signalled[k] = True
      elif what == 'cta_starts':
        ticket = self.tickets
        self.tickets += 1
        self.to_start[k] -= 1
        self.waiting[k].append(ticket // self.ctas)
      elif what == 'cta_polls':
        launch = self.waiting[k][0]
        assert launch == k, 'tickets number the launches'
        if self.go == launch + 1:
          assert self.signalled[k], 'a CTA went ahead of its step\'s signal'
          self.waiting[k].pop(0)
          self.working[k] += 1
      elif what == 'cta_leaves':
        self.working[k] -= 1
        self.left[k] += 1
        if self.left[k] == self.ctas:
          self.completed += 1
          self.tree_done[k] = True
    assert all(self.tree_done), 'every launch ran to its end'
    assert self.completed == self.steps and self.tickets == self.steps * self.ctas


@pytest.mark.parametrize('ctas', [1, 2, 21])
def test_no_cta_goes_ahead_of_its_signal(ctas):
  for seed in range(200):
    Model(steps=6, ctas=ctas, rng=random.Random(seed * 31 + ctas)).run()


def test_a_boolean_flag_would_be_read_stale():
  """The same interleavings with go = 1 / reset-by-the-last-leaver instead of launch
  numbers: some schedule lets a CTA of step k + 1 see step k's flag."""
  class Boolean(Model):
    def run_boolean(self):
      stale = False
      while True:
        ev = self.enabled()
        if not ev:
          break
        what, k = self.rng.choice(ev)
        if what == 'sampler_ends':
          self.sampler_done[k] = True
        elif what == 'signal':
          self.go = 1
          self.signalled[k] = True
        elif what == 'cta_starts':
          self.to_start[k] -= 1
          self.waiting[k].append(k)
        elif what == 'cta_polls':
          if self.go == 1:
            stale = stale or not self.signalled[k]
            self.waiting[k].pop(0)
            self.working[k] += 1
        elif what == 'cta_leaves':
          self.working[k] -= 1
          self.left[k] += 1
          if self.left[k] == self.ctas:
            self.go = 0
            self.completed += 1
            self.tree_done[k] = True
      return stale
  assert any(Boolean(steps=6, ctas=3, rng=random.Random(s)).run_boolean()
             for s in range(300))
