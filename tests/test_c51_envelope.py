"""The C51 loss kernels across their shape and value envelope, against a float64
evaluation of the reference formulas.

Every kernel instance (chosen by batch size, atom count, action count and entry point:
`c51_instances` below restates the choice) is run at the shapes where its layout
changes — one row, a warp of rows, 128 / 256 / 2048 rows, more than 32 actions, 2 and
128 atoms — and at the values where the arithmetic changes branch: gamma^n from 0 to 1
(the tail's five-term window holds from 2/3 up), returns inside, at and beyond the
support, integer supports where Bellman atoms land exactly on atoms or exactly dz away,
sharp, flat, offset and underflowing logits, exact Q ties, and extreme sampling
probabilities.

Pass rule, per case: with E(x) = max |x - f64| / (|f64| + 1e-6) over the rows (over
the elements for the projected target), a kernel passes when E(kernel) <= max(2 E(port),
1e-6) for loss, priorities and target, where `port` is the f32 numpy restatement
(oracle/c51_port.py) — the port's own distance from float64 calibrates what rounding
alone explains at each edge; its weights are within 1e-6 relative of float64; and, where
the older tests' domain applies (at least 5 atoms, logits of scale <= 3), it is within
rtol 1e-6 / atol 1e-7 of the port.  `-m "not gpu"` runs the reference's own check, the
dispatch map's coverage and the projection reference.
"""
import itertools
import math
import os
import re
import zlib

import numpy as np
import pytest

from oracle import c51_port
from oracle import fast

F32 = np.float32
F64 = np.float64


# ----------------------------------------------------------- float64 reference ----
def project_f64(supports, weights, z):
  """Dense clip / hat projection (rainbow_agent.py:381-494) in float64, chunked over
  rows: out[b, i] = sum_j clip(1 - |clip(s_bj, z0, zlast) - z_i| / dz, 0, 1) w_bj."""
  s = np.asarray(supports, F64)
  w = np.asarray(weights, F64)
  z = np.asarray(z, F64)
  dz = z[1] - z[0]
  out = np.empty(s.shape, F64)
  step = max(1, (1 << 22) // (z.size * z.size))
  for lo in range(0, s.shape[0], step):
    c = np.clip(s[lo:lo + step], z[0], z[-1])[:, None, :]
    hat = np.clip(1.0 - np.abs(c - z[None, :, None]) / dz, 0.0, 1.0)
    out[lo:lo + step] = (hat * w[lo:lo + step, None, :]).sum(axis=2)
  return out


def c51_f64(rewards, terminals, actions, probs, online, target, support, gamma_n):
  """rainbow_agent.py:200-293 in float64 from the same f32 inputs: the f32 support,
  float32(gamma^n), softmax, Q and FIRST argmax, Bellman atoms, dense projection,
  log-softmax, cross entropy, sqrt(ce + 1e-10), IS weights 1/sqrt(p + 1e-10) / max."""
  z = np.asarray(support, F32).astype(F64)
  g = F64(F32(gamma_n))
  rows = np.arange(len(actions))
  t = np.asarray(target, F64)
  t = t - t.max(axis=-1, keepdims=True)
  p = np.exp(t)
  p /= p.sum(axis=-1, keepdims=True)
  q = (p * z).sum(axis=2)
  best = np.argmax(q, axis=1)
  live = 1.0 - np.asarray(terminals).astype(F64)
  s = np.asarray(rewards, F64)[:, None] + (g * live)[:, None] * z[None, :]
  tgt = project_f64(s, p[rows, best], z)
  x = np.asarray(online, F64)[rows, np.asarray(actions)]
  x = x - x.max(axis=-1, keepdims=True)
  logp = x - np.log(np.exp(x).sum(axis=-1, keepdims=True))
  ce = -(tgt * logp).sum(axis=1)
  if probs is None:
    w = np.ones(len(actions), F64)
  else:
    w = 1.0 / np.sqrt(np.asarray(probs, F64) + 1e-10)
    w /= w.max()
  return dict(target=tgt, loss=ce, priorities=np.sqrt(ce + 1e-10), weights=w, q=q,
              argmax=best)


def c51_port_case(rewards, terminals, actions, probs, online, target, support, gamma_n):
  """The f32 port on the same inputs (gamma^n handed in as one factor)."""
  tgt, best = c51_port.target_distribution(rewards, terminals, target, support,
                                           float(F32(gamma_n)), 1)
  p = np.ones(len(actions), F32) if probs is None else probs
  ce, prio, w, _ = c51_port.loss_and_priorities(tgt, online, actions, p)
  return dict(target=tgt, loss=ce, priorities=prio, weights=w, argmax=best)


def rel_err(x, ref):
  """E(x): worst |x - f64| / (|f64| + 1e-6)."""
  x = np.asarray(x, F64)
  return float((np.abs(x - ref) / (np.abs(ref) + 1e-6)).max())


def near_ties(q, vmax):
  """Rows whose two largest float64 Q values are within 1e-5 relative, relative to the
  larger of |Q| and vmax: the f32 rounding of Q = sum z p scales with the support, so a
  gap below that can order the two actions either way in f32."""
  if q.shape[1] < 2:
    return np.zeros(q.shape[0], bool)
  top = np.sort(q, axis=1)[:, -2:]
  gap = top[:, 1] - top[:, 0]
  return gap <= 1e-5 * np.maximum(np.abs(top).max(axis=1), vmax)


# ------------------------------------------------------------------ value cases ----
# Defaults: vmax 10, gamma^n 0.97, returns inside the support, 10 % terminal rows,
# unit-scale logits, sampling probabilities sqrt(|randn|).
VALUE_CASES = {
    'gamma0': dict(gamma_n=0.0),
    'gamma1e-6': dict(gamma_n=1e-6),
    'gamma1e-3': dict(gamma_n=1e-3),
    'gamma0.3': dict(gamma_n=0.3),
    'gamma0.5': dict(gamma_n=0.5),
    'gamma0.66': dict(gamma_n=0.66),
    'gamma0.67': dict(gamma_n=0.67),
    'gamma0.97': dict(gamma_n=0.97),
    'gamma1': dict(gamma_n=1.0),
    'returns_at_vmax': dict(returns='at'),
    'returns_beyond': dict(returns='beyond'),
    'returns_beyond_gamma0.5': dict(returns='beyond', gamma_n=0.5),
    'vmax1': dict(vmax=1.),
    'vmax100': dict(vmax=100.),
    'vmax100_beyond': dict(vmax=100., returns='beyond'),
    'integer_gamma1': dict(vmax='integer', gamma_n=1.0, returns='integer'),
    'integer_gamma0.5': dict(vmax='integer', gamma_n=0.5, returns='integer'),
    'scale0.1': dict(scale=0.1),
    'scale8': dict(scale=8.),
    'scale30': dict(scale=30.),
    'offset1e4': dict(offset=1e4),
    'one_hot': dict(one_hot=True),
    'probs_equal': dict(probs='equal'),
    'probs_spread': dict(probs='spread'),
    'probs_zeros': dict(probs='zeros'),
    'probs_uniform_scheme': dict(probs=None),
}


def case_vmax(cfg, atoms):
  vmax = cfg.get('vmax', 10.)
  return (atoms - 1) / 2. if vmax == 'integer' else float(vmax)


def _returns(rng, n, vmax, kind):
  if kind == 'inside':
    return rng.uniform(-0.8, 0.8, n) * vmax
  if kind == 'at':
    return rng.choice([-vmax, vmax], n)
  if kind == 'beyond':  # every atom or most of them clip, either side
    return rng.choice([-1., 1.], n) * rng.uniform(1.0, 3.0, n) * vmax
  if kind == 'integer':
    k = int(math.ceil(vmax)) + 3
    return rng.randint(-k, k + 1, n).astype(F64)
  raise ValueError(kind)


def _probs(rng, n, kind):
  if kind is None:
    return None
  if kind == 'equal':
    return np.full(n, 0.37, F32)
  if kind == 'spread':
    return (10.0 ** rng.uniform(-12, 6, n)).astype(F32)
  if kind == 'zeros':
    p = np.sqrt(np.abs(rng.randn(n)) + 1e-10)
    p[rng.rand(n) < 0.3] = 0.
    return p.astype(F32)
  assert kind == 'random'
  return np.sqrt(np.abs(rng.randn(n)) + 1e-10).astype(F32)


def logits(rng, shape, cfg):
  """Random logits of the case's kind: scale * randn + offset, or one-hot rows (one
  atom at +100 and the rest at -100: the f32 exponentials underflow to exact zeros)."""
  if cfg.get('one_hot'):
    x = np.full(shape, -100., F32)
    hot = rng.randint(0, shape[-1], size=shape[:-1])
    np.put_along_axis(x, hot[..., None], F32(100.), axis=-1)
    return x
  return (cfg.get('scale', 1.) * rng.randn(*shape) + cfg.get('offset', 0.)).astype(F32)


def untied_target(rng, shape, cfg, support, vmax):
  """Target logits with no row whose two best float64 Q values are within 1e-5
  relative (the f32 and f64 argmax then agree): such rows are drawn again."""
  x = logits(rng, shape, cfg)
  z = np.asarray(support, F64)
  for _ in range(200):
    t = x.astype(F64)
    p = np.exp(t - t.max(axis=-1, keepdims=True))
    p /= p.sum(axis=-1, keepdims=True)
    bad = np.nonzero(near_ties((p * z).sum(axis=2), vmax))[0]
    if bad.size == 0:
      return x
    x[bad] = logits(rng, (bad.size,) + shape[1:], cfg)
  raise AssertionError('could not draw untied target logits')


def make_case(seed, batch, actions, atoms, cfg):
  """Inputs of one c51_loss call for a value case."""
  rng = np.random.RandomState(seed)
  vmax = case_vmax(cfg, atoms)
  support = c51_port.make_support(vmax, atoms)
  online = logits(rng, (batch, actions, atoms), cfg)
  target = untied_target(rng, (batch, actions, atoms), cfg, support, vmax)
  return dict(
      online=online, target=target, support=support, vmax=vmax,
      gamma_n=float(F32(cfg.get('gamma_n', 0.97))),
      actions=rng.randint(0, actions, size=batch).astype(np.int32),
      rewards=_returns(rng, batch, vmax, cfg.get('returns', 'inside')).astype(F32),
      terminals=(rng.rand(batch) < 0.1).astype(np.uint8),
      probs=_probs(rng, batch, cfg.get('probs', 'random')),
      in_port_domain=atoms >= 5 and not cfg.get('one_hot') and cfg.get('scale', 1.) <= 3)


def references(c):
  args = (c['rewards'], c['terminals'], c['actions'], c['probs'], c['online'],
          c['target'], c['support'], c['gamma_n'])
  return c51_f64(*args), c51_port_case(*args)


def judge(label, got, ref, port, in_port_domain, keys=('loss', 'priorities', 'target')):
  """The pass rule of the module docstring; returns {key: (E(kernel), E(port))}."""
  errs = {}
  for k in keys:
    e_kernel, e_port = rel_err(got[k], ref[k]), rel_err(port[k], ref[k])
    errs[k] = (e_kernel, e_port)
    assert e_kernel <= max(2 * e_port, 1e-6), (label, k, e_kernel, e_port)
  np.testing.assert_allclose(got['weights'], ref['weights'], rtol=1e-6, atol=0,
                             err_msg='%s weights' % label)
  if in_port_domain:
    for k in keys:
      atol = 1e-6 if k == 'target' else 1e-7
      np.testing.assert_allclose(got[k], port[k], rtol=1e-6, atol=atol,
                                 err_msg='%s %s vs port' % (label, k))
  print('E %s %s' % (label, ' '.join('%s=%.2g/%.2g' % (k, a, b)
                                     for k, (a, b) in errs.items())))
  return errs


# --------------------------------------------------------------- dispatch map ----
def c51_instances(entry, batch, actions, atoms):
  """The C51 kernels one call launches (c51.cu: launch_loss, c51_can_split,
  c51_pre_launch, c51_post_takes_tree, c51_tail_can_stage; step.cu: split_loss,
  staged), or None where the call is refused.  entry: 'loss' (b2r_c51_loss) or 'step'
  (b2r_train_step_device on a prioritized buffer whose tree is at most 31 levels deep;
  the trainer takes the same path)."""
  if entry == 'loss':
    if atoms > 128:
      return None
    if batch >= 128 and atoms <= 64:
      return ['c51_loss_rows_kernel<8,%d>' % (51 if atoms == 51 else 0)]
    return ['c51_loss_kernel<%d>' % (2 if atoms <= 64 else 4)]
  assert entry == 'step', entry
  if not (batch <= 2048 and 2 <= atoms <= 64):
    return c51_instances('loss', batch, actions, atoms)
  if batch >= 128:
    pre = 'c51_pre_rows_kernel<8,%d>' % (51 if atoms == 51 else 0)
  else:
    pre = 'c51_pre_kernel<2>'
  if batch <= 32:
    post = 'c51_post_tree_kernel<%s>' % ('true' if actions <= 32 else 'false')
  else:
    post = 'c51_post_kernel'
  return [pre, post]


def features(entry, batch, actions, atoms):
  """The kernel instances of a call, with the conditions under which an instance
  takes a different layout (more than 32 actions, a third of the warps above 256
  rows, a staged row stride other than the benchmark's)."""
  out = set()
  for k in c51_instances(entry, batch, actions, atoms) or ():
    out.add(k)
    if actions > 32:
      out.add(k + ' A>32')
    if k == 'c51_loss_kernel<4>':
      out.add(k + (' B>256' if batch > 256 else ' B<=256'))
    if k == 'c51_post_tree_kernel<true>' and (actions, atoms) != (18, 51):
      out.add(k + ' not 18x51')
  return out


REQUIRED_FEATURES = {
    'c51_loss_kernel<2>', 'c51_loss_kernel<2> A>32',
    'c51_loss_kernel<4> B<=256', 'c51_loss_kernel<4> B>256',
    'c51_loss_rows_kernel<8,51>', 'c51_loss_rows_kernel<8,0>',
    'c51_pre_kernel<2>', 'c51_pre_kernel<2> A>32',
    'c51_pre_rows_kernel<8,51>', 'c51_pre_rows_kernel<8,0>',
    'c51_post_kernel', 'c51_post_tree_kernel<false> A>32',
    'c51_post_tree_kernel<true>', 'c51_post_tree_kernel<true> not 18x51',
}


# ------------------------------------------------------------------- shapes ----
def pairwise(*axes):
  """A deterministic greedy cover of every pair of values of the axes."""
  want = set()
  for (a, xs), (b, ys) in itertools.combinations(enumerate(axes), 2):
    want.update((a, x, b, y) for x in xs for y in ys)
  out = []
  cands = list(itertools.product(*axes))
  while want:
    def gain(c):
      return sum((a, c[a], b, c[b]) in want
                 for a, b in itertools.combinations(range(len(c)), 2))
    best = max(cands, key=gain)
    out.append(best)
    want -= {(a, best[a], b, best[b]) for a, b in itertools.combinations(range(len(best)), 2)}
  return out


LOSS_SHAPES = pairwise((1, 31, 32, 33, 127, 128, 129, 131, 257, 2049),
                       (1, 2, 31, 32, 33, 64),
                       (2, 3, 21, 32, 33, 51, 63, 64, 65, 101, 128))
# one shape per instance of the loss entry, for the value cases
VALUE_SHAPES = [(31, 40, 64), (33, 18, 101), (300, 6, 101), (128, 18, 51), (129, 33, 64)]
# exact Q ties: integer supports with -1, 0, +1 among the atoms
TIE_SHAPES = [(31, 40, 21), (130, 40, 21), (33, 40, 65), (257, 40, 65), (5, 40, 3)]
# b2r_train_step_device: cluster tail (staged up to 32 actions), CTA-per-row first half,
# warp-per-row first half, unsplit
STEP_BATCHES = (1, 5, 32, 33, 127, 128, 129, 2048, 2049)
STEP_ACTIONS_ATOMS = ((18, 51), (33, 21), (32, 64), (40, 64), (6, 2), (18, 101))
STEP_TIE_BATCHES = (5, 33, 129)
# one buffer, shapes changing between steps: small, the largest staged row stride,
# the rows first half, more than 32 actions, back to small
STEP_SEQUENCE = [(5, 6, 2), (32, 32, 64), (129, 18, 51), (2048, 40, 64), (32, 18, 51),
                 (5, 33, 21), (1, 32, 64), (127, 40, 64)]
TRAINER_CASE = dict(batch=64, actions=40, atoms=21, vmax=100., gamma=0.5, horizon=3)


def all_calls():
  calls = [('loss',) + s for s in LOSS_SHAPES + VALUE_SHAPES + TIE_SHAPES]
  calls += [('step', b, a, n) for b in STEP_BATCHES for a, n in STEP_ACTIONS_ATOMS]
  calls += [('step', b, 40, 21) for b in STEP_TIE_BATCHES]
  calls += [('step',) + s for s in STEP_SEQUENCE]
  calls.append(('step', TRAINER_CASE['batch'], TRAINER_CASE['actions'],
                TRAINER_CASE['atoms']))
  return calls


# ============================================================= CPU tests ====
def test_dispatch_map_covers_every_instance():
  """The union of this file's parametrisations launches every C51 kernel instance,
  in each layout it has."""
  covered = set()
  for call in all_calls():
    covered |= features(*call)
  assert REQUIRED_FEATURES <= covered, sorted(REQUIRED_FEATURES - covered)
  assert c51_instances('loss', 32, 18, 129) is None


def test_pairwise_cover_is_complete():
  axes = ((1, 31, 32, 33, 127, 128, 129, 131, 257, 2049), (1, 2, 31, 32, 33, 64),
          (2, 3, 21, 32, 33, 51, 63, 64, 65, 101, 128))
  for (a, xs), (b, ys) in itertools.combinations(enumerate(axes), 2):
    for x in xs:
      for y in ys:
        assert any(s[a] == x and s[b] == y for s in LOSS_SHAPES), (a, x, b, y)


@pytest.mark.parametrize('name', sorted(VALUE_CASES))
@pytest.mark.parametrize('atoms', [2, 21, 51, 64, 101])
def test_port_meets_the_rule_against_float64(name, atoms):
  """The f32 port against c51_f64 on every value case, before the kernels are judged by
  the two: same argmax, weights within 1e-6 relative, every projected atom within 4e-6
  (the f32 Bellman atoms alone move a hat by ulp(vmax) / dz), and inside the older
  tests' domain loss and priorities within 1e-6 relative and atoms within 1e-6.  (Outside
  it the port's distance grows — 1e-3 on the loss at 2 atoms and logits of scale 30 —
  and is what the kernels are allowed twice of.)  The f64 projection conserves mass up
  to the uneven spacing of the f32 support."""
  cfg = VALUE_CASES[name]
  c = make_case(1000 + atoms, 64, 2 if atoms == 2 else 6, atoms, cfg)
  ref, port = references(c)
  assert np.array_equal(port['argmax'], ref['argmax'])
  np.testing.assert_allclose(port['weights'], ref['weights'], rtol=1e-6, atol=0)
  target_err = np.abs(port['target'] - ref['target']).max()
  assert target_err <= 4e-6, target_err
  if c['in_port_domain']:
    assert target_err <= 1e-6, target_err
    for k in ('loss', 'priorities'):
      assert rel_err(port[k], ref[k]) <= 1e-6, (k, rel_err(port[k], ref[k]))
  np.testing.assert_allclose(ref['target'].sum(axis=1), 1.0, rtol=1e-5)


def test_float64_reference_takes_the_first_maximum():
  """Exact ties: the f64 reference (and the port) pick the first tied action."""
  c = tie_case(0, 8, 40, 21)
  ref, port = references(c)
  assert np.array_equal(ref['argmax'], c['winner'])
  assert np.array_equal(port['argmax'], c['winner'])


def test_short_last_spacing_of_f32_supports():
  """The supports on which the projection's clipped terms reach the second-to-last
  atom: the f32 support's last spacing is shorter than z[1] - z[0]."""
  def short(vmax, n):
    z = c51_port.make_support(vmax, n)
    return z[-1] - z[-2] < z[1] - z[0]
  assert short(10., 64) and short(10., 101)
  assert not short(10., 51)
  # and there, clipped mass does reach atom N - 2 with a nonzero hat in the dense form
  z = c51_port.make_support(10., 64)
  proj = c51_port.project_distribution(np.full((1, 64), 50., F32),
                                       np.full((1, 64), 1. / 64, F32), z)
  assert 0 < proj[0, -2] < 1e-5


def _projection_case(seed, batch, atoms):
  rng = np.random.RandomState(seed)
  vmax = 10.
  z = c51_port.make_support(vmax, atoms)
  s = rng.uniform(-1.5 * vmax, 1.5 * vmax, size=(batch, atoms)).astype(F32)
  w = rng.rand(batch, atoms).astype(F32)
  return s, w, z


def _projection_tolerance(s, w, z):
  """1e-6 of the weight that can reach each atom (the terms a rounding of the hat or of
  the f32 sum may move): |clip(s_j) - z_i| < dz (1 + 1e-5)."""
  z64 = z.astype(F64)
  dz = z64[1] - z64[0]
  c = np.clip(s.astype(F64), z64[0], z64[-1])[:, None, :]
  reach = np.abs(c - z64[None, :, None]) < dz * (1 + 1e-5)
  return 1e-6 * (reach * np.abs(w.astype(F64))[:, None, :]).sum(axis=2) + 1e-12


@pytest.mark.parametrize('atoms', [2, 51, 300])
def test_projection_reference_matches_port(atoms):
  """project_f64 is the port's dense form evaluated in float64."""
  s, w, z = _projection_case(atoms, 16, atoms)
  ref = project_f64(s, w, z)
  port = c51_port.project_distribution(s, w, z)
  assert np.all(np.abs(port - ref) <= _projection_tolerance(s, w, z))
  np.testing.assert_allclose(ref.sum(axis=1), w.astype(F64).sum(axis=1), rtol=1e-5)


# ============================================================= GPU tests ====
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


def _dev(gpu, x):
  return gpu.torch.as_tensor(x, device='cuda')


def run_loss(gpu, c, want_target=True, want_grad=True):
  support = gpu.ra.make_support(c['vmax'], c['support'].size)
  assert support.cpu().numpy().tobytes() == c['support'].tobytes()
  probs = None if c['probs'] is None else _dev(gpu, c['probs'])
  out = gpu.ra.c51_loss(_dev(gpu, c['online']), _dev(gpu, c['target']),
                        _dev(gpu, c['actions']), _dev(gpu, c['rewards']),
                        _dev(gpu, c['terminals']), probs, support, c['gamma_n'],
                        want_target=want_target, want_grad=want_grad)
  gpu.torch.cuda.synchronize()
  return {k: v.cpu().numpy() for k, v in out.items()}


def check_loss(gpu, label, c):
  """One c51_loss call judged by the rule, plus its mean and its gradient (against
  float64 torch autograd of mean(w * ce) with the port's target and weights)."""
  torch = gpu.torch
  got = run_loss(gpu, c)
  ref, port = references(c)
  judge(label, got, ref, port, c['in_port_domain'])
  np.testing.assert_allclose(got['mean_weighted_loss'],
                             (ref['weights'] * ref['loss']).mean(), rtol=1e-5, atol=1e-7)
  batch = len(c['actions'])
  x = torch.tensor(c['online'], dtype=torch.float64, requires_grad=True)
  chosen = x[torch.arange(batch), torch.as_tensor(c['actions']).long()]
  t = torch.tensor(port['target'], dtype=torch.float64)
  w = torch.tensor(port['weights'], dtype=torch.float64)
  (w * -(t * torch.log_softmax(chosen, dim=1)).sum(1)).mean().backward()
  np.testing.assert_allclose(got['grad_logits'], x.grad.numpy(), rtol=1e-4, atol=1e-7,
                             err_msg=label + ' grad')


@pytest.mark.gpu
@pytest.mark.parametrize('batch,actions,atoms', LOSS_SHAPES)
def test_c51_loss_shapes(gpu, batch, actions, atoms):
  c = make_case(batch * 10007 + actions * 101 + atoms, batch, actions, atoms, {})
  check_loss(gpu, 'loss %dx%dx%d' % (batch, actions, atoms), c)


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(VALUE_CASES))
@pytest.mark.parametrize('batch,actions,atoms', VALUE_SHAPES)
def test_c51_loss_values(gpu, name, batch, actions, atoms):
  c = make_case(zlib.crc32(name.encode()) % 1000 + batch, batch, actions, atoms, VALUE_CASES[name])
  check_loss(gpu, 'loss %dx%dx%d %s' % (batch, actions, atoms, name), c)


@pytest.mark.gpu
def test_c51_loss_refuses_129_atoms(gpu):
  c = make_case(0, 4, 3, 129, {})
  with pytest.raises(gpu.native.NativeError) as e:
    run_loss(gpu, c)
  assert e.value.code == gpu.native.ERR_UNSUPPORTED


TIE_SETS = [(3, 35), (5, 35, 38), (1, 9), (2, 5), (0, 39), (9, 12, 33)]


def tie_case(seed, batch, actions, atoms):
  """Exact Q ties on an integer support (vmax = (N - 1) / 2, step 1): target logits
  -1000 (exp is an exact 0 in f32 and f64) except on chosen atoms, so probabilities
  are exactly 1 or 0.5 / 0.5 and Q is exact in any summation order.  In every row the
  actions of one tie set have Q = 0 — half the mass at -1 and +1, or all of it at 0 —
  the first of them with the other form than the rest, so the loss tells which one
  won; every other action has Q = -1."""
  rng = np.random.RandomState(seed)
  vmax = (atoms - 1) / 2.
  support = c51_port.make_support(vmax, atoms)
  zero = atoms // 2
  assert support[zero] == 0 and support[zero - 1] == -1 and support[zero + 1] == 1
  target = np.full((batch, actions, atoms), -1000., F32)
  target[:, :, zero - 1] = 0.
  winner = np.empty(batch, np.int64)
  for b in range(batch):
    ties = [a % actions for a in TIE_SETS[b % len(TIE_SETS)]]
    spread_first = b % 2 == 0
    for k, a in enumerate(sorted(set(ties))):
      target[b, a] = -1000.
      if (k == 0) == spread_first:
        target[b, a, zero - 1] = target[b, a, zero + 1] = 0.
      else:
        target[b, a, zero] = 0.
    winner[b] = min(ties)
  return dict(
      online=rng.randn(batch, actions, atoms).astype(F32), target=target,
      support=support, vmax=vmax, gamma_n=float(F32(0.97)),
      actions=rng.randint(0, actions, size=batch).astype(np.int32),
      rewards=rng.randint(-3, 4, size=batch).astype(F32),
      terminals=np.zeros(batch, np.uint8), probs=_probs(rng, batch, 'random'),
      in_port_domain=atoms >= 5, winner=winner)


@pytest.mark.gpu
@pytest.mark.parametrize('batch,actions,atoms', TIE_SHAPES)
def test_c51_loss_exact_ties_take_the_first_action(gpu, batch, actions, atoms):
  c = tie_case(batch + atoms, batch, actions, atoms)
  got = run_loss(gpu, c)
  ref, port = references(c)
  assert np.array_equal(ref['argmax'], c['winner'])
  judge('ties %dx%dx%d' % (batch, actions, atoms), got, ref, port, c['in_port_domain'])


# ----------------------------------------------------------------- projection ----
@pytest.mark.gpu
@pytest.mark.parametrize('batch', [1, 5, 4096])
@pytest.mark.parametrize('atoms', [2, 51, 1536])
def test_project_distribution_against_float64(gpu, batch, atoms):
  """Unsorted Bellman supports, clipped on both sides; at most 1536 atoms (the
  kernel's shared memory).  Large cases are checked on a sample of rows."""
  s, w, z = _projection_case(batch * 7 + atoms, batch, atoms)
  got = gpu.ra.project_distribution(s, w, z)
  rows = np.arange(batch)
  if batch * atoms * atoms > (1 << 26):
    rows = np.random.RandomState(0).choice(batch, 64, replace=False)
  ref = project_f64(s[rows], w[rows], z)
  tol = _projection_tolerance(s[rows], w[rows], z)
  bad = np.abs(got[rows] - ref) > tol
  assert not bad.any(), (np.abs(got[rows] - ref)[bad].max(), tol[bad].min())


@pytest.mark.gpu
def test_project_distribution_refuses_1537_atoms(gpu):
  s, w, z = _projection_case(0, 2, 1537)
  with pytest.raises(gpu.native.NativeError) as e:
    gpu.ra.project_distribution(s, w, z)
  assert e.value.code == gpu.native.ERR_UNSUPPORTED


# ------------------------------------------------------------- the fused step ----
def prioritized_buffer(gpu, cap, batch, seed, actions, vmax, horizon=1, gamma=0.99):
  """A full, wrapped prioritized buffer of 8 x 8 frames whose action column spans
  [0, actions) and whose stored rewards give returns inside, exactly at and beyond
  +-vmax (horizon 1: the return is the stored reward); with a float64 mirror of its
  tree."""
  rng = np.random.RandomState(seed)
  mem = gpu.prb.OutOfGraphPrioritizedReplayBuffer(
      (8, 8), 4, cap, batch, update_horizon=horizon, gamma=gamma, output='torch',
      rng='device', seed=seed)
  mem._store['observation'] = rng.randint(0, 256, size=(cap, 8, 8)).astype(np.uint8)
  action = rng.randint(0, actions, size=cap).astype(np.int32)
  action[:actions] = np.arange(actions)
  mem._store['action'] = action
  kind = rng.choice(['inside', 'at', 'beyond'], size=cap, p=[0.4, 0.1, 0.5])
  reward = np.empty(cap)
  for k in ('inside', 'at', 'beyond'):
    reward[kind == k] = _returns(rng, int((kind == k).sum()), vmax, k)
  mem._store['reward'] = reward.astype(F32)
  mem._store['terminal'] = (rng.rand(cap) < 0.1).astype(np.uint8)
  mem.add_count = cap + 4242
  mem.invalid_range = np.array([(4242 - horizon + i) % cap for i in range(4 + horizon)])
  tree = fast.FastTree(cap)
  ids = np.arange(cap, dtype=np.int32)
  pr = np.sqrt(np.abs(rng.randn(cap)) + 1e-10).astype(F32)
  mem.set_priority(ids, pr)
  tree.set_seq(ids, pr.astype(F64))
  return mem, tree


def check_step(label, transition, out, tree, online, target, support, gamma_n, scale):
  """One fused step on the batch it returned: sampling probabilities are the tree's
  leaves, loss / priorities / weights by the rule; applies the write-back to `tree`."""
  idx = transition['indices']
  probs = transition['sampling_probabilities']
  assert probs.tobytes() == tree.level(tree.depth)[idx].astype(F32).tobytes(), label
  args = (transition['reward'], transition['terminal'], transition['action'], probs,
          online, target, support, gamma_n)
  ref, port = c51_f64(*args), c51_port_case(*args)
  got = {k: out[k] for k in ('loss', 'priorities', 'weights')}
  judge(label, got, ref, port, support.size >= 5 and scale <= 3,
        keys=('loss', 'priorities'))
  tree.set_seq(idx, out['priorities'].astype(F64))


def assert_tree(mem, tree):
  for l, level in enumerate(mem.sum_tree.nodes):
    assert np.array_equal(level.view(np.uint64), tree.level(l).view(np.uint64)), l


# per step: gamma^n (0.97: the tail's five-term window; 0.5: its loop) and logit scale.
# (Sharper logits are the loss entry's value cases: over 2048 rows, logits of scale 3
# already give rows with a cross entropy near 0.01, where one ulp of the log-sum-exp is
# 1.7e-5 of the loss, the kernel's expf and numpy's exp differ by that, and the port's
# worst row against float64 is not the kernel's.)
STEP_VALUES = [(0.97, 1.), (0.5, 1.), (1.0, 0.1)]


def fused_step(gpu, mem, batch, actions, atoms, vmax, gamma_n, rng, scale, out=None,
               target=None):
  torch = gpu.torch
  support = c51_port.make_support(vmax, atoms)
  online = logits(rng, (batch, actions, atoms), dict(scale=scale))
  if target is None:
    target = untied_target(rng, (batch, actions, atoms), dict(scale=scale), support, vmax)
  got, out = gpu.ra.train_step(mem, _dev(gpu, online), _dev(gpu, target),
                               gpu.ra.make_support(vmax, atoms), gamma_n, out=out)
  torch.cuda.synchronize()
  names = ('state', 'action', 'reward', 'next_state', 'next_action', 'next_reward',
           'terminal', 'indices', 'sampling_probabilities')
  transition = {k: v.cpu().numpy() for k, v in zip(names, got)}
  return transition, {k: v.cpu().numpy() for k, v in out.items()}, out, online, target, support


@pytest.mark.gpu
@pytest.mark.parametrize('actions,atoms', STEP_ACTIONS_ATOMS)
@pytest.mark.parametrize('batch', STEP_BATCHES)
def test_fused_step_shapes(gpu, batch, actions, atoms):
  """train_step over three steps (gamma^n and logit scale change between them): loss,
  priorities and weights by the rule, the tree bit-exact after the write-backs."""
  vmax = 10.
  cap = 8192
  mem, tree = prioritized_buffer(gpu, cap, batch, batch + actions * 7 + atoms, actions, vmax)
  rng = np.random.RandomState(batch * 3 + atoms)
  out = None
  for step, (gamma_n, scale) in enumerate(STEP_VALUES):
    gamma_n = float(F32(gamma_n))
    t, host, out, online, target, support = fused_step(
        gpu, mem, batch, actions, atoms, vmax, gamma_n, rng, scale, out=out)
    assert t['action'].max() < actions
    check_step('step %dx%dx%d #%d' % (batch, actions, atoms, step), t, host, tree,
               online, target, support, gamma_n, scale)
  gpu.native.check(gpu.native.lib().b2r_check(mem._h, gpu.native.current_stream()))
  assert_tree(mem, tree)


@pytest.mark.gpu
@pytest.mark.parametrize('batch', STEP_TIE_BATCHES)
def test_fused_step_exact_ties_take_the_first_action(gpu, batch):
  """The split first half's tie rule (CTA per row with more than 32 actions, warp per
  row) on exact ties, through the tail that follows it."""
  actions, atoms = 40, 21
  c = tie_case(batch, batch, actions, atoms)
  mem, tree = prioritized_buffer(gpu, 8192, batch, batch, actions, c['vmax'])
  rng = np.random.RandomState(batch)
  t, host, _, online, target, support = fused_step(
      gpu, mem, batch, actions, atoms, c['vmax'], c['gamma_n'], rng, 1., target=c['target'])
  ref = c51_f64(t['reward'], t['terminal'], t['action'], t['sampling_probabilities'],
                online, target, support, c['gamma_n'])
  assert np.array_equal(ref['argmax'], c['winner'])
  check_step('step ties %d' % batch, t, host, tree, online, target, support,
             c['gamma_n'], 1.)
  assert_tree(mem, tree)


@pytest.mark.gpu
def test_fused_step_shape_changes_on_one_buffer(gpu):
  """(batch, actions, atoms) change between steps on one buffer: the first half's
  scratch and the staged tail's log-probability buffer are reallocated as they grow and
  reused as they shrink; every step stays right."""
  vmax, cap = 10., 8192
  amax = max(a for _, a, _ in STEP_SEQUENCE)
  mem, tree = prioritized_buffer(gpu, cap, 32, 77, amax, vmax)
  column = mem._store['action'].copy()
  rng = np.random.RandomState(78)
  for step, (batch, actions, atoms) in enumerate(STEP_SEQUENCE):
    mem._store['action'] = (column % actions).astype(np.int32)
    gamma_n = float(F32(STEP_VALUES[step % len(STEP_VALUES)][0]))
    t, host, _, online, target, support = fused_step(
        gpu, mem, batch, actions, atoms, vmax, gamma_n, rng, 1.)
    check_step('sequence #%d %dx%dx%d' % (step, batch, actions, atoms), t, host, tree,
               online, target, support, gamma_n, 1.)
  assert_tree(mem, tree)


@pytest.mark.gpu
@pytest.mark.parametrize('direct', [False, True])
def test_trainer_wide_support(gpu, direct):
  """The host-facing trainer away from the defaults: 40 actions, 21 atoms, vmax 100,
  buffer gamma 0.5 over 3 steps (gamma^n 0.125: the tail's loop), batch 64; its own
  support and cumulative gamma, and (direct) the first half's copy of pinned logits."""
  torch = gpu.torch
  k = TRAINER_CASE
  if direct:
    os.environ['B2R_TRAINER_DIRECT'] = '1'
  else:
    os.environ.pop('B2R_TRAINER_DIRECT', None)
  try:
    cap = 8192
    mem, tree = prioritized_buffer(gpu, cap, k['batch'], 31, k['actions'], k['vmax'],
                                   horizon=k['horizon'], gamma=k['gamma'])
    trainer = gpu.ra.ReplayTrainer(mem, k['actions'], k['atoms'], k['vmax'],
                                   pipeline_depth=1, seed=31)
    gamma_n = float(F32(math.pow(k['gamma'], k['horizon'])))
    support = c51_port.make_support(k['vmax'], k['atoms'])
    rng = np.random.RandomState(32)
    shape = (k['batch'], k['actions'], k['atoms'])
    pin = [(torch.empty(shape, dtype=torch.float32).pin_memory(),
            torch.empty(shape, dtype=torch.float32).pin_memory()) for _ in range(4)]
    device_losses, handed = {}, {}
    for step in range(4):
      online = logits(rng, shape, {})
      target = untied_target(rng, shape, {}, support, k['vmax'])
      if direct:
        pin[step][0].copy_(torch.from_numpy(online))
        pin[step][1].copy_(torch.from_numpy(target))
        loss, done = trainer.step(pin[step][0], pin[step][1])
      else:
        loss, done = trainer.step(online, target)
      if done >= 0:
        handed[done] = loss
      torch.cuda.synchronize()
      transition, out = trainer.views()
      t = {name: v.cpu().numpy() for name, v in transition.items()}
      host = {name: v.cpu().numpy() for name, v in out.items()}
      device_losses[step] = host['loss'].copy()
      check_step('trainer direct=%d #%d' % (direct, step), t, host, tree, online, target,
                 support, gamma_n, 1.)
    loss, done = trainer.drain()
    handed[done] = loss
    for step, loss in handed.items():
      assert loss.tobytes() == device_losses[step].tobytes(), step
    assert_tree(mem, tree)
  finally:
    os.environ.pop('B2R_TRAINER_DIRECT', None)


# ----------------------------------------------------------- dispatch on device ----
def _kernel_names(torch, fn):
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    fn()
    torch.cuda.synchronize()
  return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _c51_kernels(names):
  out = set()
  for n in names:
    m = re.search(r'(c51_\w+_kernel)(<[^>(]*>)?', n)
    if m:
      out.add(m.group(1) + (m.group(2) or '').replace(' ', ''))
  return out


@pytest.mark.gpu
def test_dispatch_map_matches_launched_kernels(gpu):
  """One representative call per instance under torch.profiler: the C51 kernels it
  launches are the ones c51_instances names."""
  torch = gpu.torch
  x = torch.ones(1 << 16, device='cuda')
  if not _kernel_names(torch, lambda: x.mul_(2)):
    pytest.skip('torch.profiler records no CUDA kernels on this machine')
  calls = [('loss', 31, 40, 64), ('loss', 33, 18, 101), ('loss', 300, 6, 101),
           ('loss', 128, 18, 51), ('loss', 129, 33, 64),
           ('step', 5, 40, 21), ('step', 32, 32, 64), ('step', 33, 18, 51),
           ('step', 129, 18, 51), ('step', 128, 33, 21), ('step', 2049, 18, 51),
           ('step', 32, 18, 51)]
  seen = set()
  for entry, batch, actions, atoms in calls:
    want = set(c51_instances(entry, batch, actions, atoms))
    if entry == 'loss':
      c = make_case(batch, batch, actions, atoms, {})
      names = _kernel_names(torch, lambda: run_loss(gpu, c))
    else:
      mem, _ = prioritized_buffer(gpu, 8192, batch, batch, actions, 10.)
      rng = np.random.RandomState(0)
      fused_step(gpu, mem, batch, actions, atoms, 10., 0.97, rng, 1.)  # (warm-up)
      names = _kernel_names(
          torch, lambda: fused_step(gpu, mem, batch, actions, atoms, 10., 0.97, rng, 1.))
    got = _c51_kernels(names)
    assert got == want, (entry, batch, actions, atoms, sorted(got), sorted(want))
    seen |= got
  assert seen == {k.split(' ')[0] for k in REQUIRED_FEATURES}
