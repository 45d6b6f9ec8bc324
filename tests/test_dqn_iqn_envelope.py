"""The DQN and IQN loss kernels across their shape and value envelope, against a
float64 evaluation of the reference formulas.

Kernels: dqn_loss_kernel (256-thread blocks, one thread per row), dqn_mean_kernel (one
1024-thread CTA, f32 fixed-order sum), dqn_mean_sharded_kernel (one 256-thread CTA, f64
sum) and iqn_loss_kernel (one CTA per row; its mean is summed by the last CTA to take a
ticket).  They are run at the shapes where their layout changes (rows across 256-thread
blocks and the 1024-thread mean; 1, 32, 33, 64, 65 and 257 actions; 1 to 256 tau
samples, and the refusal at 257; 1 to 200 action samples, across IQN's 4 warps), at the
values where the arithmetic changes branch (Bellman errors exactly 0, at the Huber
threshold and one ulp either side of it; tau exactly 0 and 1; kappa 1, 0.5, 3, 1e-3 and
100 — every kappa but 1 takes the division; gamma^n 0 and 1; terminal rows; scales from
1e-3 to 1e4; rewards far from the quantiles; exact and near ties of the greedy action;
target maxima of 1e30 and -inf entries), through every entry point and mode (gradient
and mean off, strided inputs, the DQN mean without per-row losses, the sharded entry
points at every `count` edge), and over launch sequences and a CUDA graph that
exercise IQN's mean ticket and the DQN mean kernels.

Pass rules, per case, with E(x) = max over the rows of |x - f64| / (|f64| + 1e-6):
- DQN target, loss and gradient rows are bit-identical to the f32 port
  (oracle/dqn_port.py): both apply the same single-rounded f32 operations in the same
  order.
- DQN mean, IQN loss and IQN mean: E(kernel) <= max(2 E(port), 1e-6), where `port` is
  the f32 numpy restatement; its own distance from float64 calibrates what rounding
  alone explains at each edge.
- IQN gradient, per element: |kernel - f64| <= max(2 |port - f64|, 4 * 2^-23 * S) with
  S = sum_t' |w dh| / (kappa N' B): the sum over t' cancels towards 0 near a fitted
  quantile, so the bound is absolute, a few f32 ulps of the terms it sums.
- IQN greedy action: always in [0, A); the first action on exact f64 ties; any action
  whose f64 mean is within the f32 rounding of the K-sum and the division of the best;
  otherwise the f64 argmax.
Rows whose action means are all -inf (action 0) or all NaN (some action in [0, A)) are
run against the fixed kernel only: before the fix, the greedy reduction kept its
sentinel 0x7fffffff there and gathered the target network at that column.

Not tested: IQN Bellman errors beyond about 1.8e19.  There the port's op-by-op Huber
form squares the error to inf and multiplies it by the 0 of the other case (NaN), while
the kernel selects one branch; values here keep |error| <= 1e18.

`-m "not gpu"` runs the port against float64 on every value case, the float64 IQN
reference against the looped closed form, the shape cover, the ABI refusals that come
before any device work, and a numpy model of IQN's greedy reduction.
"""
import ctypes
import itertools
import zlib

import numpy as np
import pytest

from oracle import dqn_port
from oracle import iqn_port

F32 = np.float32
F64 = np.float64
NO_ACTION = 0x7fffffff
ULP = 2.0 ** -23


# ----------------------------------------------------------- float64 references ----
def dqn_f64(rewards, terminals, actions, online_q, target_q, gamma_n):
  """dqn_agent.py:283-322 in float64 from the same f32 inputs and float32(gamma^n)."""
  g = F64(F32(gamma_n))
  rows = np.arange(len(actions))
  best = np.asarray(target_q, F64).max(axis=1)
  live = 1.0 - np.asarray(terminals).astype(F64)
  target = np.asarray(rewards, F64) + g * best * live
  err = np.asarray(online_q, F64)[rows, np.asarray(actions)] - target
  quad = np.minimum(np.abs(err), 1.0)
  loss = 0.5 * quad * quad + (np.abs(err) - quad)
  return dict(target=target, loss=loss, mean_loss=loss.mean())


def dqn_port_case(c):
  return dqn_port.dqn_update(c['rewards'], c['terminals'], c['actions'], c['online_q'],
                             c['target_q'], float(F32(c['gamma_n'])), 1)


def iqn_means_f64(action_values, batch, k):
  """The action network's mean over its K samples, in float64: (B, A)."""
  a = np.asarray(action_values, F64)
  return a.reshape(k, batch, a.shape[1]).mean(axis=0)


def iqn_f64(rewards, terminals, actions, online, quantiles, target_net, action_net, n,
            n_prime, k, kappa, gamma_n, next_action=None):
  """implicit_quantile_agent.py:176-315 in float64 from the same f32 inputs: the first
  maximum of the f64 mean over K (unless `next_action` is given), the target quantiles,
  the quantile-Huber loss per row and its mean, and d mean / d online on the chosen
  column, -sum_t' w dh / (kappa N' B); also S = sum_t' |w dh| / (kappa N' B)."""
  batch = len(rewards)
  num_actions = np.asarray(online).shape[1]
  kappa = F64(F32(kappa))
  g = F64(F32(gamma_n))
  if next_action is None:
    next_action = np.argmax(iqn_means_f64(action_net, batch, k), axis=1)
  b = np.arange(batch)
  z = np.asarray(target_net, F64).reshape(n_prime, batch, num_actions)[:, b, next_action]
  live = 1.0 - np.asarray(terminals).astype(F64)
  target = np.asarray(rewards, F64)[:, None] + (g * live)[:, None] * z.T  # B x N'
  chosen = np.asarray(online, F64).reshape(n, batch, num_actions)[:, b, actions].T  # B x N
  taus = np.asarray(quantiles, F64).reshape(n, batch).T
  loss = np.empty(batch)
  g_sum = np.empty((batch, n))
  g_abs = np.empty((batch, n))
  step = max(1, (1 << 22) // (n * n_prime))
  for lo in range(0, batch, step):
    s = slice(lo, lo + step)
    err = target[s, :, None] - chosen[s, None, :]  # B x N' x N
    abs_err = np.abs(err)
    small = abs_err <= kappa
    huber = np.where(small, 0.5 * err * err, kappa * (abs_err - 0.5 * kappa))
    w = np.abs(taus[s, None, :] - (err < 0))
    loss[lo:lo + step] = (w * huber / kappa).sum(axis=2).mean(axis=1)
    wdh = w * np.where(small, err, kappa * np.sign(err))
    g_sum[s] = wdh.sum(axis=1)
    g_abs[s] = np.abs(wdh).sum(axis=1)
  scale = kappa * n_prime * batch
  grad = np.zeros((n, batch, num_actions))
  grad[:, b, actions] = (-g_sum / scale).T
  bound = np.zeros((n, batch, num_actions))
  bound[:, b, actions] = (g_abs / scale).T
  return dict(next_action=np.asarray(next_action), target=target, loss=loss,
              mean_loss=loss.mean(), grad=grad.reshape(n * batch, num_actions),
              grad_terms=bound.reshape(n * batch, num_actions))


def iqn_args(c):
  return (c['rewards'], c['terminals'], c['actions'], c['online'], c['quantiles'],
          c['target'], c['action'], c['n'], c['n_prime'], c['k'], c['kappa'],
          c['gamma_n'])


def iqn_port_case(c, next_action=None):
  """The f32 port on the same inputs; with `next_action`, the port's loss at that
  greedy action (the port picks its own otherwise)."""
  action = c['action']
  if next_action is not None:  # one sample whose row maximum is the given action
    action = np.zeros((1, len(c['rewards']), c['target'].shape[1]), F32)
    action[0, np.arange(len(c['rewards'])), next_action] = 1.
    action = action.reshape(len(c['rewards']), -1)
  return iqn_port.iqn_update(
      c['rewards'], c['terminals'], c['actions'], c['online'], c['quantiles'],
      c['target'], action, c['n'], c['n_prime'], 1 if next_action is not None else c['k'],
      kappa=c['kappa'], gamma=float(F32(c['gamma_n'])), update_horizon=1)


def rel_err(x, ref):
  """E(x): worst |x - f64| / (|f64| + 1e-6)."""
  x = np.asarray(x, F64)
  ref = np.asarray(ref, F64)
  return float((np.abs(x - ref) / (np.abs(ref) + 1e-6)).max()) if ref.size else 0.


def check_rule(label, got, ref, port):
  e_kernel, e_port = rel_err(got, ref), rel_err(port, ref)
  assert e_kernel <= max(2 * e_port, 1e-6), (label, e_kernel, e_port)
  return e_kernel, e_port


def greedy_allowed(action_values, batch, k):
  """(first f64 argmax, boolean (B, A) of the actions the rule accepts)."""
  a = np.asarray(action_values, F64).reshape(k, batch, -1)
  q = a.mean(axis=0)
  first = np.argmax(q, axis=1)
  best = q[np.arange(batch), first]
  # f32 rounding of the K-sum and of the division, and the f64 sum's own rounding
  tol = 2 * ULP * np.abs(best) + 4 * 2.0 ** -52 * np.abs(a).sum(axis=0).max(axis=1) / k
  allowed = q >= (best - tol)[:, None]
  # where every accepted action ties exactly with the best, only the first is right
  only_exact = np.array([np.all(q[r, allowed[r]] == best[r]) for r in range(batch)])
  allowed[only_exact] = False
  allowed[only_exact, first[only_exact]] = True
  return first, allowed


def check_greedy(label, got, action_values, batch, k):
  got = np.asarray(got, np.int64)
  num_actions = np.asarray(action_values).shape[1]
  assert ((got >= 0) & (got < num_actions)).all(), (label, got.min(), got.max())
  first, allowed = greedy_allowed(action_values, batch, k)
  bad = ~allowed[np.arange(batch), got]
  assert not bad.any(), (label, np.nonzero(bad)[0][:8], got[bad][:8], first[bad][:8])


# ------------------------------------------------ the greedy reduction, modelled ----
def greedy_model(action_values, batch, k, b, fixed):
  """iqn_loss_kernel's greedy action for row b, step by step: warp w sums the samples
  k = w (mod 4) in f64 for 32 actions at a time (lane = action mod 32), warp 0 adds the
  four partials in warp order, rounds to f32 and divides by K, each lane keeps its
  running best, and five xor shuffles reduce the 32 lanes.  fixed=False is the parent's
  rule (strict > from -inf, sentinel 0x7fffffff), fixed=True the guarded one."""
  x = np.asarray(action_values, F32).reshape(k, batch, -1)[:, b, :]
  num_actions = x.shape[1]
  best_q = [F32(-np.inf)] * 32
  best_a = [NO_ACTION] * 32
  for base in range(0, num_actions, 32):
    for lane in range(32):
      act = base + lane
      if act >= num_actions:
        continue
      partial = [0.0] * 4
      for w in range(4):
        for s in range(w, k, 4):
          partial[w] += float(x[s, act])
      total = partial[0]
      for w in range(1, 4):
        total += partial[w]
      with np.errstate(over='ignore', invalid='ignore'):
        q = F32(F32(total) / F32(k))
      if (fixed and best_a[lane] == NO_ACTION) or q > best_q[lane]:
        best_q[lane], best_a[lane] = q, act
  for o in (16, 8, 4, 2, 1):
    q_old, a_old = list(best_q), list(best_a)
    for lane in range(32):
      q2, a2 = q_old[lane ^ o], a_old[lane ^ o]
      q1, a1 = q_old[lane], a_old[lane]
      if fixed:
        take = a2 != NO_ACTION and (a1 == NO_ACTION or q2 > q1 or (q2 == q1 and a2 < a1))
      else:
        take = q2 > q1 or (q2 == q1 and a2 < a1)
      if take:
        best_q[lane], best_a[lane] = q2, a2
  return best_a[0]


def tied_action_values(k, num_actions, ties, rng):
  """(K, 1, A) action samples whose means tie exactly on `ties` (each a permutation of
  the same small integers, so every summation order gives the same f64 and f32 sum)
  above every other action."""
  x = rng.randint(-20, 0, size=(k, num_actions)).astype(F32)
  top = rng.randint(1, 9, size=k).astype(F32)
  for a in ties:
    x[:, a] = rng.permutation(top)
  return x.reshape(k, num_actions)


# ------------------------------------------------------------------ value cases ----
# Defaults: kappa 1, gamma^n 0.99^3, quantile values randn * 1.5, rewards in [-1, 1],
# 20 % terminal rows, taus uniform in [0, 1).
IQN_VALUE_CASES = {
    'default': dict(),
    'kappa0.5': dict(kappa=0.5),
    'kappa3': dict(kappa=3.),
    'kappa1e-3': dict(kappa=1e-3),
    'kappa100': dict(kappa=100.),
    'gamma0': dict(gamma_n=0.),
    'gamma1': dict(gamma_n=1.),
    'all_terminal': dict(terminal_p=1.),
    'boundary_kappa1': dict(boundary=True),
    'boundary_kappa3': dict(boundary=True, kappa=3.),
    'boundary_kappa0.5': dict(boundary=True, kappa=0.5),
    'boundary_kappa1e-3': dict(boundary=True, kappa=1e-3),
    'tau_edges': dict(taus='edges'),
    'tau_edges_boundary': dict(taus='edges', boundary=True),
    'scale1e-3': dict(scale=1e-3),
    'scale1e-3_kappa1e-3': dict(scale=1e-3, kappa=1e-3),
    'scale1e4': dict(scale=1e4),
    'scale1e4_kappa100': dict(scale=1e4, kappa=100.),
    'rewards_far': dict(rewards='far'),
    'rewards_very_far': dict(rewards='very_far'),
    'ties_exact': dict(ties='exact'),
    'ties_near': dict(ties='near'),
}
# against the fixed kernel only (the parent reads out of bounds on these rows)
IQN_NONFINITE_CASES = {
    'means_all_-inf': dict(nonfinite='-inf'),
    'means_all_nan': dict(nonfinite='nan'),
    'means_overflow_to_-inf': dict(nonfinite='overflow'),
}


def _boundary_values(rng, shape, kappa):
  """Values v for which an error of exactly v forms: 0, +-kappa, +-kappa one ulp
  either side, and a few ordinary ones."""
  kp = F32(kappa)
  pool = np.array([0., kp, -kp, np.nextafter(kp, F32(0)), -np.nextafter(kp, F32(0)),
                   np.nextafter(kp, F32(np.inf)), -np.nextafter(kp, F32(np.inf)),
                   F32(0.5) * kp, F32(2) * kp], F32)
  return rng.choice(pool, size=shape)


def _taus(rng, shape, kind):
  t = rng.rand(*shape).astype(F32)
  if kind == 'edges':
    pick = rng.rand(*shape)
    t[pick < 0.4] = 0.
    t[pick > 0.6] = 1.
  return t


def make_iqn_case(seed, batch, num_actions, n, n_prime, k, cfg):
  """Inputs of one b2r_iqn_loss call for a value case."""
  rng = np.random.RandomState(seed)
  kappa = float(F32(cfg.get('kappa', 1.)))
  gamma_n = float(F32(cfg.get('gamma_n', 0.99 ** 3)))
  scale = cfg.get('scale', 1.5)
  online = (scale * rng.randn(n * batch, num_actions)).astype(F32)
  target = (scale * rng.randn(n_prime * batch, num_actions)).astype(F32)
  action = (scale * rng.randn(k * batch, num_actions)).astype(F32)
  rewards = (scale * rng.uniform(-1, 1, batch)).astype(F32)
  terminals = (rng.rand(batch) < cfg.get('terminal_p', 0.2)).astype(np.uint8)
  actions = rng.randint(0, num_actions, size=batch).astype(np.int32)
  if cfg.get('rewards') == 'far':
    rewards = (rng.choice([-1., 1.], batch) * 10.0 ** rng.uniform(3, 6, batch)).astype(F32)
  elif cfg.get('rewards') == 'very_far':
    rewards = (rng.choice([-1., 1.], batch) * 10.0 ** rng.uniform(15, 18, batch)).astype(F32)
  if cfg.get('boundary'):
    # rewards 0, gamma^n 1, no terminals and the chosen online values 0: the Bellman
    # error is the target quantile value, exactly, in f32 and in f64
    gamma_n, rewards[:] = 1., 0.
    terminals[:] = 0
    online.reshape(n, batch, num_actions)[:, np.arange(batch), actions] = 0.
    target = _boundary_values(rng, target.shape, kappa)
  quantiles = _taus(rng, (n * batch, 1), cfg.get('taus'))
  ties = cfg.get('ties')
  if ties:
    kk = action.reshape(k, batch, num_actions)
    for b in range(batch):
      picks = rng.choice(num_actions, size=min(num_actions, 3), replace=False)
      kk[:, b] = tied_action_values(k, num_actions, picks, rng)
      if ties == 'near' and len(picks) > 1:
        # one ulp of the mean apart: within the f32 rounding, either may win
        kk[0, b, picks[1]] = np.nextafter(kk[0, b, picks[1]], F32(np.inf))
  nonfinite = cfg.get('nonfinite')
  if nonfinite:
    kk = action.reshape(k, batch, num_actions)
    rows = np.arange(batch) % 2 == 0  # every other row; the rest stay finite
    if nonfinite == '-inf':
      kk[:, rows] = -np.inf
    elif nonfinite == 'nan':
      kk[:, rows] = np.nan
    else:  # the f64 K-sum exceeds f32's range: the cast gives -inf before the division
      assert k >= 2
      kk[:, rows] = -3e38
  return dict(online=online, target=target, action=action, rewards=rewards,
              terminals=terminals, actions=actions, quantiles=quantiles, n=n,
              n_prime=n_prime, k=k, kappa=kappa, gamma_n=gamma_n, nonfinite=nonfinite)


DQN_VALUE_CASES = {
    'default': dict(),
    'huber_boundary': dict(boundary=True),
    'gamma0': dict(gamma_n=0.),
    'gamma1': dict(gamma_n=1.),
    'all_terminal': dict(terminal_p=1.),
    'target_max_1e30': dict(huge=True),
    'equal_maxima': dict(equal_max=True),
    'neg_inf_entries': dict(neg_inf=True),
    'scale1e-3': dict(scale=1e-3),
    'scale1e4': dict(scale=1e4),
}


def make_dqn_case(seed, batch, num_actions, cfg):
  rng = np.random.RandomState(seed)
  scale = cfg.get('scale', 3.)
  online = (scale * rng.randn(batch, num_actions)).astype(F32)
  target = (scale * rng.randn(batch, num_actions)).astype(F32)
  actions = rng.randint(0, num_actions, size=batch).astype(np.int32)
  rewards = rng.uniform(-1, 1, batch).astype(F32)
  terminals = (rng.rand(batch) < cfg.get('terminal_p', 0.2)).astype(np.uint8)
  gamma_n = float(F32(cfg.get('gamma_n', 0.99 ** 3)))
  rows = np.arange(batch)
  if cfg.get('boundary'):
    # terminal rows with reward 0: the error is the chosen online value, exactly
    terminals[:] = 1
    rewards[:] = 0.
    pool = np.array([0., 1., -1., np.nextafter(F32(1), F32(0)), np.nextafter(F32(1), F32(2)),
                     -np.nextafter(F32(1), F32(0)), -np.nextafter(F32(1), F32(2)), 0.5, 2.],
                    F32)
    online[rows, actions] = rng.choice(pool, batch)
  if cfg.get('huge'):
    pick = rng.rand(batch) < 0.5
    target[pick, rng.randint(0, num_actions, batch)[pick]] = (
        rng.choice([1e30, 1e34], pick.sum())).astype(F32)
  if cfg.get('equal_max'):
    target[:] = np.round(target)  # integers: maxima tie often
    target[rows, (actions + 1) % num_actions] = target.max(axis=1)
  if cfg.get('neg_inf'):
    hole = rng.rand(batch, num_actions) < 0.5
    hole[rows, rng.randint(0, num_actions, batch)] = False  # a finite maximum per row
    target[hole] = -np.inf
  return dict(online_q=online, target_q=target, actions=actions, rewards=rewards,
              terminals=terminals, gamma_n=gamma_n)


# ------------------------------------------------------------------- shapes ----
def pairwise(*axes, cost=None):
  """A deterministic greedy cover of every pair of values of the axes; among the
  candidates that cover as many new pairs, the cheapest (by `cost`)."""
  want = set()
  for (a, xs), (b, ys) in itertools.combinations(enumerate(axes), 2):
    want.update((a, x, b, y) for x in xs for y in ys)
  out = []
  cands = list(itertools.product(*axes))
  pairs = list(itertools.combinations(range(len(axes)), 2))
  while want:
    def key(c):
      gain = sum((a, c[a], b, c[b]) in want for a, b in pairs)
      return (gain, -(cost(c) if cost else 0))
    best = max(cands, key=key)
    out.append(best)
    want -= {(a, best[a], b, best[b]) for a, b in pairs}
  return out


IQN_AXES = ((1, 7, 32, 33, 256, 4096),      # batch
            (1, 2, 31, 32, 33, 64, 65, 257),  # actions
            (1, 3, 32, 33, 64, 255, 256),   # N
            (1, 3, 4, 5, 64, 256),          # N'
            (1, 3, 4, 5, 32, 200))          # K


def _iqn_cost(s):
  batch, actions, n, n_prime, k = s
  return batch * (n * n_prime + (n + n_prime + k) * actions)


IQN_SHAPES = pairwise(*IQN_AXES, cost=_iqn_cost)
IQN_VALUE_SHAPES = [(33, 18, 64, 64, 32), (7, 65, 33, 5, 3)]
DQN_SHAPES = [(b, a) for b in (1, 255, 256, 257, 1023, 1024, 1025, 4096, 4097, 70000)
              for a in (1, 2, 18, 257)]
DQN_VALUE_SHAPES = [(1025, 18), (257, 2)]


# ============================================================= CPU tests ====
def test_pairwise_cover_is_complete():
  for (a, xs), (b, ys) in itertools.combinations(enumerate(IQN_AXES), 2):
    for x in xs:
      for y in ys:
        assert any(s[a] == x and s[b] == y for s in IQN_SHAPES), (a, x, b, y)


@pytest.mark.parametrize('name', sorted(DQN_VALUE_CASES))
def test_dqn_port_meets_the_rule_against_float64(name):
  """The port's rows are what the kernel must reproduce bit for bit; here they are
  within an f32 rounding of float64 (target and loss to 1e-6 relative, plus one ulp
  of the reward-scale terms the target sums), and the port's mean meets the rule."""
  c = make_dqn_case(1, 513, 18, DQN_VALUE_CASES[name])
  port = dqn_port_case(c)
  ref = dqn_f64(c['rewards'], c['terminals'], c['actions'], c['online_q'],
                c['target_q'], c['gamma_n'])
  assert np.isfinite(port['loss']).all() and np.isfinite(ref['loss']).all()
  scale = (np.abs(c['rewards']).astype(F64) +
           np.abs(np.asarray(c['target_q'], F64).max(axis=1)))
  assert (np.abs(port['target'] - ref['target']) <= 2 * ULP * scale + 1e-30).all()
  # the loss follows the error: |e| rounds with the target's ulp
  chosen = np.abs(c['online_q'][np.arange(513), c['actions']]).astype(F64)
  assert (np.abs(port['loss'] - ref['loss']) <=
          4 * ULP * (scale + chosen + np.abs(ref['loss'])) + 1e-30).all()
  assert rel_err(port['mean_loss'], ref['mean_loss']) <= 1e-6
  if name == 'huber_boundary':  # errors exact: the port is float64 rounded once
    assert (port['loss'] == ref['loss'].astype(F32)).all()


@pytest.mark.parametrize('name', sorted(IQN_VALUE_CASES))
def test_iqn_port_meets_the_rule_against_float64(name):
  """The port against iqn_f64 on every value case, before the kernel is judged by the
  two: its greedy action meets the rule, and at the f64 greedy action its loss and
  mean are within 1e-6 relative (2e-7 is the worst seen: every term is formed in f32
  from the same f32 inputs), so the kernel's loss is held to 1e-6 throughout."""
  c = make_iqn_case(2, 33, 18, 16, 8, 5, IQN_VALUE_CASES[name])
  ref = iqn_f64(*iqn_args(c))
  port = iqn_port_case(c)
  check_greedy(name, port['next_action'], c['action'], 33, 5)
  port = iqn_port_case(c, ref['next_action'])
  assert rel_err(port['loss'], ref['loss']) <= 1e-6, rel_err(port['loss'], ref['loss'])
  assert rel_err(port['mean_loss'], ref['mean_loss']) <= 1e-6


@pytest.mark.parametrize('batch,actions,n,n_prime,k,kappa', [
    (5, 3, 4, 6, 2, 1.0), (8, 4, 16, 8, 4, 0.5), (3, 2, 7, 5, 3, 3.0), (4, 33, 3, 4, 5, 1e-3)])
def test_iqn_f64_matches_looped_closed_form(batch, actions, n, n_prime, k, kappa):
  """iqn_f64 (vectorised) against iqn_port.closed_form_f64 (plain loops) at small
  shapes, and its gradient against central differences of the closed form."""
  c = make_iqn_case(batch * 3 + n, batch, actions, n, n_prime, k, dict(kappa=kappa))
  ref = iqn_f64(*iqn_args(c))
  want = iqn_port.closed_form_f64(
      c['rewards'], c['terminals'], c['actions'], c['online'], c['quantiles'],
      c['target'], ref['next_action'], n, n_prime, kappa=c['kappa'],
      gamma=c['gamma_n'], update_horizon=1)
  np.testing.assert_allclose(ref['loss'], want, rtol=1e-12, atol=1e-300)
  assert np.array_equal(ref['next_action'],
                        np.argmax(iqn_means_f64(c['action'], batch, k), axis=1))
  eps = 1e-6
  for b in range(batch):
    row = (b % n) * batch + b
    col = c['actions'][b]
    x = c['online'].astype(F64)
    f = []
    for d in (eps, -eps):
      y = x.copy()
      y[row, col] += d
      f.append(iqn_port.closed_form_f64(
          c['rewards'], c['terminals'], c['actions'], y, c['quantiles'], c['target'],
          ref['next_action'], n, n_prime, kappa=c['kappa'], gamma=c['gamma_n'],
          update_horizon=1).mean())
    fd = (f[0] - f[1]) / (2 * eps)
    assert abs(ref['grad'][row, col] - fd) <= 1e-5 * max(1., abs(fd)), (b, fd)


def test_greedy_model_parent_rule_keeps_the_sentinel_on_all_neg_inf():
  """An all -inf row: under the parent's rule no lane ever takes an action and the
  reduction returns 0x7fffffff (the kernel then gathered the target network at that
  column); under the fixed rule, action 0, as argmax gives."""
  x = np.full((4, 1, 40), -np.inf, F32).reshape(4, 40)
  assert greedy_model(x, 1, 4, 0, fixed=False) == NO_ACTION
  assert greedy_model(x, 1, 4, 0, fixed=True) == 0
  assert np.argmax(x.mean(axis=0)) == 0
  # the same through an f64 K-sum beyond f32's range: the cast gives -inf
  x = np.full((3, 40), -3e38, F32)
  assert greedy_model(x, 1, 3, 0, fixed=False) == NO_ACTION
  assert greedy_model(x, 1, 3, 0, fixed=True) == 0
  # all NaN: some action in range under the fixed rule
  x = np.full((2, 70), np.nan, F32)
  assert greedy_model(x, 1, 2, 0, fixed=False) == NO_ACTION
  assert 0 <= greedy_model(x, 1, 2, 0, fixed=True) < 70


@pytest.mark.parametrize('ties', [(3, 17), (9, 12, 31), (5, 37), (1, 33, 65), (40, 8),
                                  (0, 64)])
@pytest.mark.parametrize('k', [1, 4, 5, 7])
def test_greedy_model_takes_the_first_of_exact_ties(ties, k):
  """Exact ties across lanes, across 32-action blocks (the same lane) and, with K > 4,
  across the warps' K-slices (each tied action's samples are a permutation of the
  others'): both rules take the first tied action, and so does the f64 reference."""
  num_actions = 70
  x = tied_action_values(k, num_actions, ties, np.random.RandomState(k + sum(ties)))
  assert greedy_model(x, 1, k, 0, fixed=True) == min(ties)
  assert greedy_model(x, 1, k, 0, fixed=False) == min(ties)
  first, allowed = greedy_allowed(x, 1, k)
  assert first[0] == min(ties) and allowed[0].sum() == 1


def test_greedy_model_rules_agree_on_finite_rows():
  """For finite means the guard changes nothing: both rules pick the same action, the
  first f32 maximum, at action counts around the 32-action blocks."""
  rng = np.random.RandomState(7)
  for num_actions in (1, 2, 31, 32, 33, 64, 65, 100):
    for k in (1, 3, 5):
      x = (rng.randn(k * 3, num_actions) * 2).astype(F32)
      for b in range(3):
        a = greedy_model(x, 3, k, b, fixed=True)
        assert a == greedy_model(x, 3, k, b, fixed=False)
        q = x.reshape(k, 3, num_actions)[:, b].astype(F64).sum(axis=0).astype(F32) / F32(k)
        assert a == int(np.argmax(q))


# ------------------------------------------------------------------ ABI refusals ----
def _lib():
  from dopamine_b200 import _native
  return _native, _native.lib()


def _iqn_struct(native, **kw):
  args = native.IqnArgs()
  args.batch, args.num_actions = 4, 3
  args.num_tau_samples, args.num_tau_prime_samples, args.num_quantile_samples = 8, 8, 2
  args.cumulative_gamma, args.kappa = 0.99, 1.0
  for name in ('action_quantile_values', 'target_quantile_values',
               'online_quantile_values', 'quantiles', 'actions', 'rewards', 'terminals',
               'loss'):
    setattr(args, name, 0x1000)  # never dereferenced: the checks come first
  for name, value in kw.items():
    setattr(args, name, value)
  return args


IQN_REFUSALS = [
    (dict(num_tau_samples=257), 'UNSUPPORTED'),
    (dict(num_tau_prime_samples=257), 'UNSUPPORTED'),
    (dict(kappa=0.), 'INVALID_ARGUMENT'),
    (dict(kappa=-1.), 'INVALID_ARGUMENT'),
    (dict(kappa=float('nan')), 'INVALID_ARGUMENT'),
    (dict(batch=0), 'INVALID_ARGUMENT'),
    (dict(num_actions=0), 'INVALID_ARGUMENT'),
    (dict(num_quantile_samples=0), 'INVALID_ARGUMENT'),
] + [(dict([(p, None)]), 'INVALID_ARGUMENT') for p in (
    'action_quantile_values', 'target_quantile_values', 'online_quantile_values',
    'quantiles', 'actions', 'rewards', 'terminals', 'loss')]


@pytest.mark.parametrize('sharded', [False, True])
@pytest.mark.parametrize('kw,code', IQN_REFUSALS,
                         ids=['%s=%s' % next(iter(kw.items())) for kw, _ in IQN_REFUSALS])
def test_iqn_abi_refusals(kw, code, sharded):
  native, lib = _lib()
  args = _iqn_struct(native, **kw)
  count = np.array([4], np.int32)
  if sharded:
    status = lib.b2r_iqn_loss_sharded(ctypes.byref(args), count.ctypes.data, 8, None)
  else:
    status = lib.b2r_iqn_loss(ctypes.byref(args), None)
  assert status == getattr(native, 'ERR_' + code), (status, native.last_error())


def _dqn_struct(native, **kw):
  args = native.DqnArgs()
  args.batch, args.num_actions, args.cumulative_gamma = 4, 3, 0.99
  for name in ('target_q', 'online_q', 'actions', 'rewards', 'terminals'):
    setattr(args, name, 0x1000)  # never dereferenced: the checks come first
  for name, value in kw.items():
    setattr(args, name, value)
  return args


DQN_REFUSALS = [dict(batch=0), dict(batch=-1), dict(num_actions=0)] + [
    dict([(p, None)]) for p in ('target_q', 'online_q', 'actions', 'rewards', 'terminals')]


@pytest.mark.parametrize('sharded', [False, True])
@pytest.mark.parametrize('kw', DQN_REFUSALS,
                         ids=['%s=%s' % next(iter(kw.items())) for kw in DQN_REFUSALS])
def test_dqn_abi_refusals(kw, sharded):
  native, lib = _lib()
  args = _dqn_struct(native, **kw)
  count = np.array([4], np.int32)
  if sharded:
    args.batch_count = count.ctypes.data
    status = lib.b2r_dqn_loss_sharded(ctypes.byref(args), 8, None)
  else:
    status = lib.b2r_dqn_loss(ctypes.byref(args), None)
  assert status == native.ERR_INVALID_ARGUMENT, (status, native.last_error())


# ============================================================= GPU tests ====
@pytest.fixture(scope='module')
def gpu():
  import torch
  if not torch.cuda.is_available():
    pytest.fail('-m gpu tests need a CUDA device (no CPU fallback exists)')
  from dopamine_b200 import _native
  from dopamine_b200.agents.dqn import dqn_agent
  from dopamine_b200.agents.implicit_quantile import implicit_quantile_agent

  class Mods(object):
    pass

  m = Mods()
  m.torch, m.native = torch, _native
  m.dqn, m.iqn = dqn_agent, implicit_quantile_agent
  return m


def _dev(gpu, x):
  return gpu.torch.as_tensor(np.ascontiguousarray(x), device='cuda')


def _host(out):
  return {k: v.cpu().numpy() for k, v in out.items()}


def _bits(x):
  x = np.ascontiguousarray(x, F32)
  return x.view(np.uint32)


# ---------------------------------------------------------------------- DQN ----
def run_dqn(gpu, c, strided=False, **kw):
  d = {k: _dev(gpu, c[k]) for k in ('online_q', 'target_q', 'actions', 'rewards',
                                     'terminals')}
  if strided:  # column slices of wider tensors
    torch = gpu.torch
    for k in d:
      v = d[k]
      wide = torch.zeros((v.shape[0], 3) + tuple(v.shape[1:]), dtype=v.dtype,
                         device='cuda')
      wide[:, 1] = v
      d[k] = wide[:, 1] if v.dim() == 1 else wide.reshape(v.shape[0], -1)[
          :, v.shape[1]:2 * v.shape[1]]
      assert not d[k].is_contiguous()
      assert gpu.torch.equal(d[k], v)
  kw.setdefault('want_target', True)
  kw.setdefault('want_grad', True)
  out = gpu.dqn.dqn_loss(d['online_q'], d['target_q'], d['actions'], d['rewards'],
                         d['terminals'], c['gamma_n'], **kw)
  gpu.torch.cuda.synchronize()
  return _host(out)


def check_dqn(label, got, c):
  port = dqn_port_case(c)
  for key in ('target', 'loss', 'grad_q'):
    if key in got:
      g, p = _bits(got[key]), _bits(port[key])
      bad = g != p
      assert not bad.any(), (label, key, np.nonzero(bad)[0][:5], got[key][bad][:5],
                             port[key][bad][:5])
  if 'mean_loss' in got:
    ref = dqn_f64(c['rewards'], c['terminals'], c['actions'], c['online_q'],
                  c['target_q'], c['gamma_n'])
    check_rule(label + ' mean', got['mean_loss'], ref['mean_loss'], port['mean_loss'])


@pytest.mark.gpu
@pytest.mark.parametrize('batch,actions', DQN_SHAPES)
def test_dqn_loss_shapes(gpu, batch, actions):
  c = make_dqn_case(batch * 31 + actions, batch, actions, {})
  check_dqn('dqn %dx%d' % (batch, actions), run_dqn(gpu, c), c)


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(DQN_VALUE_CASES))
@pytest.mark.parametrize('batch,actions', DQN_VALUE_SHAPES)
def test_dqn_loss_values(gpu, name, batch, actions):
  c = make_dqn_case(zlib.crc32(name.encode()) % 1000 + batch, batch, actions,
                    DQN_VALUE_CASES[name])
  check_dqn('dqn %dx%d %s' % (batch, actions, name), run_dqn(gpu, c), c)


@pytest.mark.gpu
def test_dqn_loss_modes(gpu):
  """Target, gradient and mean off; strided inputs: the same bits as the full call."""
  c = make_dqn_case(5, 1025, 18, {})
  full = run_dqn(gpu, c)
  check_dqn('dqn full', full, c)
  bare = run_dqn(gpu, c, want_target=False, want_grad=False, want_mean=False)
  assert set(bare) == {'loss'}
  assert bare['loss'].tobytes() == full['loss'].tobytes()
  strided = run_dqn(gpu, c, strided=True)
  for key in full:
    assert strided[key].tobytes() == full[key].tobytes(), key


def _dqn_abi(gpu, c, dev, mean, loss=None, count=None, global_batch=None):
  """b2r_dqn_loss(_sharded) through the ctypes struct, loss and target unset unless
  given (the mean then sums the library's scratch array)."""
  native = gpu.native
  a = native.DqnArgs()
  a.batch, a.num_actions = c['online_q'].shape
  a.cumulative_gamma = float(F32(c['gamma_n']))
  a.target_q, a.online_q = dev['target_q'].data_ptr(), dev['online_q'].data_ptr()
  a.actions, a.rewards = dev['actions'].data_ptr(), dev['rewards'].data_ptr()
  a.terminals = dev['terminals'].data_ptr()
  a.loss = loss.data_ptr() if loss is not None else None
  a.mean_loss = mean.data_ptr()
  stream = native.current_stream()
  if count is None:
    native.check(native.lib().b2r_dqn_loss(ctypes.byref(a), stream))
  else:
    a.batch_count = count.data_ptr()
    native.check(native.lib().b2r_dqn_loss_sharded(ctypes.byref(a), global_batch, stream))


@pytest.mark.gpu
def test_dqn_mean_without_row_losses(gpu):
  """The mean with no per-row loss output: the library sums a scratch array it grows
  on demand (4096, then 8192 rows here) and reuses when the batch shrinks."""
  torch = gpu.torch
  for batch in (1, 4096, 4097, 32):
    c = make_dqn_case(batch, batch, 18, {})
    dev = {k: _dev(gpu, v) for k, v in c.items() if k != 'gamma_n'}
    mean = torch.full((), float('nan'), device='cuda')
    _dqn_abi(gpu, c, dev, mean)
    torch.cuda.synchronize()
    got = dict(mean_loss=mean.cpu().numpy())
    check_dqn('dqn no rows %d' % batch, got, c)
    # and the sharded mean over the same scratch, all rows valid
    count = torch.tensor([batch], dtype=torch.int32, device='cuda')
    mean.fill_(float('nan'))
    _dqn_abi(gpu, c, dev, mean, count=count, global_batch=batch)
    torch.cuda.synchronize()
    check_dqn('dqn no rows sharded %d' % batch, dict(mean_loss=mean.cpu().numpy()), c)


def _counts(rows):
  return [0, 1, rows - 1, rows, rows + 5, -1]


def _rank_slices(rows):
  """Rank r's valid rows [lo, lo + n) of the global batch for each count of _counts:
  the global batch is the sum of the valid rows."""
  out, lo = [], 0
  for count in _counts(rows):
    n = min(max(count, 0), rows)
    out.append((count, lo, n))
    lo += n
  return out, lo


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [1, 256, 257, 1500])
def test_dqn_sharded_counts(gpu, rows):
  """Six ranks of `rows` rows each, with count 0, 1, rows - 1, rows, rows + 5 and -1,
  over one global batch: every computed row has the bits of the unsharded launch on
  the whole global batch, padded rows loss 0 and zero gradient, and the partial means
  add up to the global mean by the rule."""
  torch = gpu.torch
  slices, global_batch = _rank_slices(rows)
  actions = 18
  g = make_dqn_case(rows + 3, global_batch, actions, {})
  whole = run_dqn(gpu, g)
  check_dqn('dqn global %d' % global_batch, whole, g)
  partial = 0.
  for count, lo, n in slices:
    c = make_dqn_case(rows * 7 + count, rows, actions, {})  # garbage in the padded rows
    for key in ('online_q', 'target_q', 'actions', 'rewards', 'terminals'):
      c[key][:n] = g[key][lo:lo + n]
    out = {'loss': torch.full((rows,), 7., device='cuda'),
           'target': torch.full((rows,), 7., device='cuda'),
           'mean_loss': torch.full((), float('nan'), device='cuda'),
           'grad_q': torch.full((rows, actions), 7., device='cuda')}
    cnt = torch.tensor([count], dtype=torch.int32, device='cuda')
    d = {k: _dev(gpu, c[k]) for k in ('online_q', 'target_q', 'actions', 'rewards',
                                       'terminals')}
    gpu.dqn.dqn_loss(d['online_q'], d['target_q'], d['actions'], d['rewards'],
                     d['terminals'], g['gamma_n'], out=out, sharded=(global_batch, cnt))
    got = _host(out)
    label = 'dqn rank rows %d count %d' % (rows, count)
    for key in ('loss', 'target', 'grad_q'):
      assert got[key][:n].tobytes() == whole[key][lo:lo + n].tobytes(), (label, key)
    assert (got['loss'][n:] == 0).all() and (got['grad_q'][n:] == 0).all(), label
    assert (got['target'][n:] == 7.).all(), label  # padded rows: no target written
    partial += float(got['mean_loss'])
  ref = dqn_f64(g['rewards'], g['terminals'], g['actions'], g['online_q'], g['target_q'],
                g['gamma_n'])
  check_rule('dqn partial means %d' % rows, partial, ref['mean_loss'],
             dqn_port_case(g)['mean_loss'])


# ---------------------------------------------------------------------- IQN ----
def run_iqn(gpu, c, want_grad=True, want_mean=True, flat_taus=False, strided=False):
  d = {k: _dev(gpu, c[k]) for k in ('online', 'quantiles', 'target', 'action',
                                     'actions', 'rewards', 'terminals')}
  if flat_taus:
    d['quantiles'] = d['quantiles'].reshape(-1)
  if strided:
    torch = gpu.torch
    for k in ('online', 'target', 'action', 'quantiles'):
      v = d[k]
      v2 = v.reshape(v.shape[0], -1)
      wide = torch.zeros(v2.shape[0], 2 * v2.shape[1] + 1, device='cuda')
      wide[:, 1:1 + v2.shape[1]] = v2
      d[k] = wide[:, 1:1 + v2.shape[1]].reshape(v.shape)
    for k in ('actions', 'rewards', 'terminals'):
      v = d[k]
      wide = torch.zeros(v.shape[0], 2, dtype=v.dtype, device='cuda')
      wide[:, 1] = v
      d[k] = wide[:, 1]
      assert not d[k].is_contiguous()
  out = gpu.iqn.quantile_huber_loss(
      d['online'], d['quantiles'], d['target'], d['action'], d['actions'], d['rewards'],
      d['terminals'], c['gamma_n'], c['kappa'], want_grad=want_grad, want_mean=want_mean)
  gpu.torch.cuda.synchronize()
  return _host(out)


def sample_rows(batch, n, n_prime):
  """The rows the float64 reference is evaluated on: all of them up to 2^22 error
  terms, else a fixed sample that keeps the first and last rows."""
  if batch * n * n_prime <= (1 << 22):
    return np.arange(batch)
  rng = np.random.RandomState(batch + n + n_prime)
  keep = max(2, (1 << 22) // (n * n_prime))
  return np.unique(np.concatenate([[0, batch - 1], rng.choice(batch, keep, replace=False)]))


def _iqn_rows(c, rows):
  """The case restricted to `rows` (the layout keeps sample-major rows)."""
  batch = len(c['rewards'])
  out = dict(c)
  for key, s in (('online', c['n']), ('target', c['n_prime']), ('action', c['k']),
                 ('quantiles', c['n'])):
    x = c[key].reshape(s, batch, -1)[:, rows]
    out[key] = x.reshape(s * len(rows), x.shape[-1])
  for key in ('rewards', 'terminals', 'actions'):
    out[key] = c[key][rows]
  return out


def check_iqn(label, got, c):
  """The rule of the module docstring on one call's outputs."""
  batch = len(c['rewards'])
  num_actions = c['online'].shape[1]
  n, k = c['n'], c['k']
  assert ((got['next_action'] >= 0) & (got['next_action'] < num_actions)).all(), label
  rows = sample_rows(batch, n, c['n_prime'])
  sub = _iqn_rows(c, rows)
  finite = np.isfinite(iqn_means_f64(sub['action'], len(rows), k)).all(axis=1)
  if c.get('nonfinite'):
    nf_rows = ~finite
    if c['nonfinite'] in ('-inf', 'overflow'):
      assert (got['next_action'][rows][nf_rows] == 0).all(), label
    sub_f = _iqn_rows(sub, np.nonzero(finite)[0])
    check_greedy(label, got['next_action'][rows][finite], sub_f['action'],
                 int(finite.sum()), k)
  else:
    assert finite.all()
    check_greedy(label, got['next_action'][rows], sub['action'], len(rows), k)
  # loss and gradient at the kernel's own greedy action (the near-tie rows may take
  # either; the choice is judged above)
  chosen = got['next_action'][rows].astype(np.int64)
  args = list(iqn_args(sub))
  ref = iqn_f64(*args, next_action=chosen)
  port = iqn_port_case(sub, chosen)
  # the scale of the loss: the gradient's divisor is the whole batch
  ref_grad = ref['grad'] * len(rows) / batch
  ref_terms = ref['grad_terms'] * len(rows) / batch
  port_grad = port['grad'].astype(F64) * len(rows) / batch
  e = check_rule(label + ' loss', got['loss'][rows], ref['loss'], port['loss'])
  if 'grad' in got:
    g = got['grad'].reshape(n, batch, num_actions)[:, rows].reshape(n * len(rows), -1)
    err = np.abs(g.astype(F64) - ref_grad)
    bound = np.maximum(2 * np.abs(port_grad - ref_grad), 4 * ULP * ref_terms)
    bad = err > bound
    assert not bad.any(), (label, 'grad', err[bad][:4], bound[bad][:4])
  if 'mean_loss' in got:
    if len(rows) == batch:
      check_rule(label + ' mean', got['mean_loss'], ref['mean_loss'], port['mean_loss'])
    else:  # sampled rows: the mean of the kernel's own rows, summed in f64
      want = got['loss'].astype(F64).mean()
      assert abs(float(got['mean_loss']) - want) <= 1e-6 * abs(want) + 1e-30, label
  print('E %s loss=%.2g/%.2g' % (label, e[0], e[1]))


@pytest.mark.gpu
@pytest.mark.parametrize('batch,actions,n,n_prime,k', IQN_SHAPES)
def test_iqn_loss_shapes(gpu, batch, actions, n, n_prime, k):
  c = make_iqn_case(batch * 7 + actions * 3 + n + n_prime + k, batch, actions, n,
                    n_prime, k, {})
  check_iqn('iqn %dx%dx%dx%dx%d' % (batch, actions, n, n_prime, k), run_iqn(gpu, c), c)


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(IQN_VALUE_CASES) + sorted(IQN_NONFINITE_CASES))
@pytest.mark.parametrize('batch,actions,n,n_prime,k', IQN_VALUE_SHAPES)
def test_iqn_loss_values(gpu, name, batch, actions, n, n_prime, k):
  cfg = dict(IQN_VALUE_CASES, **IQN_NONFINITE_CASES)[name]
  c = make_iqn_case(zlib.crc32(name.encode()) % 1000 + batch, batch, actions, n,
                    n_prime, k, cfg)
  check_iqn('iqn %dx%dx%dx%dx%d %s' % (batch, actions, n, n_prime, k, name),
            run_iqn(gpu, c), c)


@pytest.mark.gpu
def test_iqn_loss_modes(gpu):
  """Gradient and mean off, taus shaped (N B,) and (N B, 1), strided inputs: the
  same bits as the full call."""
  c = make_iqn_case(11, 33, 18, 32, 16, 8, {})
  full = run_iqn(gpu, c)
  check_iqn('iqn full', full, c)
  for kw in (dict(want_grad=False), dict(want_mean=False), dict(flat_taus=True),
             dict(strided=True)):
    got = run_iqn(gpu, c, **kw)
    for key in got:
      assert got[key].tobytes() == full[key].tobytes(), (kw, key)
    assert ('grad' in got) == kw.get('want_grad', True), kw
    assert ('mean_loss' in got) == kw.get('want_mean', True), kw


@pytest.mark.gpu
def test_iqn_refusals(gpu):
  """257 tau samples either side: B2R_ERR_UNSUPPORTED; batch 0 and kappa <= 0 or NaN:
  ValueError from the wrapper, before any launch."""
  for n, n_prime in ((257, 4), (4, 257)):
    c = make_iqn_case(0, 3, 4, n, n_prime, 2, {})
    with pytest.raises(gpu.native.NativeError) as e:
      run_iqn(gpu, c)
    assert e.value.code == gpu.native.ERR_UNSUPPORTED
  c = make_iqn_case(0, 3, 4, 4, 4, 2, {})
  empty = _iqn_rows(c, np.arange(0))
  with pytest.raises(ValueError, match='batch'):
    run_iqn(gpu, empty)
  for kappa in (0., -1., float('nan')):
    with pytest.raises(ValueError, match='kappa'):
      run_iqn(gpu, dict(c, kappa=kappa))


def _iqn_slice(c, lo, n, rows, filler):
  """Rank rows: the global rows [lo, lo + n) first, then `filler`'s rows as padding;
  kappa and gamma^n are the global batch's."""
  out = dict(filler, kappa=c['kappa'], gamma_n=c['gamma_n'])
  batch = len(c['rewards'])
  for key, s in (('online', c['n']), ('target', c['n_prime']), ('action', c['k']),
                 ('quantiles', c['n'])):
    x = filler[key].reshape(s, rows, -1).copy()
    x[:, :n] = c[key].reshape(s, batch, -1)[:, lo:lo + n]
    out[key] = x.reshape(s * rows, -1)
  for key in ('rewards', 'terminals', 'actions'):
    x = filler[key].copy()
    x[:n] = c[key][lo:lo + n]
    out[key] = x
  return out


def _iqn_call(gpu, c, out, sharded=None):
  d = {k: _dev(gpu, c[k]) for k in ('online', 'quantiles', 'target', 'action',
                                     'actions', 'rewards', 'terminals')}
  gpu.iqn.quantile_huber_loss(
      d['online'], d['quantiles'], d['target'], d['action'], d['actions'], d['rewards'],
      d['terminals'], c['gamma_n'], c['kappa'], out=out, sharded=sharded)
  return d


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [1, 33])
def test_iqn_sharded_counts(gpu, rows):
  """As test_dqn_sharded_counts for b2r_iqn_loss_sharded; padded rows also keep the
  next_action they had (pre-filled with a sentinel)."""
  torch = gpu.torch
  slices, global_batch = _rank_slices(rows)
  n, n_prime, k, actions = 16, 8, 5, 18
  g = make_iqn_case(rows, global_batch, actions, n, n_prime, k, dict(kappa=0.5))
  whole = run_iqn(gpu, g)
  check_iqn('iqn global %d' % global_batch, whole, g)
  partial = 0.
  for count, lo, m in slices:
    filler = make_iqn_case(rows * 7 + count + 1, rows, actions, n, n_prime, k, {})
    c = _iqn_slice(g, lo, m, rows, filler)
    out = {'loss': torch.full((rows,), 7., device='cuda'),
           'next_action': torch.full((rows,), -5, dtype=torch.int32, device='cuda'),
           'mean_loss': torch.full((), float('nan'), device='cuda'),
           'grad': torch.full((n * rows, actions), 7., device='cuda')}
    cnt = torch.tensor([count], dtype=torch.int32, device='cuda')
    _iqn_call(gpu, c, out, sharded=(global_batch, cnt))
    torch.cuda.synchronize()
    got = _host(out)
    label = 'iqn rank rows %d count %d' % (rows, count)
    assert got['loss'][:m].tobytes() == whole['loss'][lo:lo + m].tobytes(), label
    assert got['next_action'][:m].tobytes() == whole['next_action'][lo:lo + m].tobytes()
    gg = got['grad'].reshape(n, rows, actions)
    gw = whole['grad'].reshape(n, global_batch, actions)
    assert gg[:, :m].tobytes() == gw[:, lo:lo + m].tobytes(), label
    assert (got['loss'][m:] == 0).all() and (gg[:, m:] == 0).all(), label
    assert (got['next_action'][m:] == -5).all(), label
    partial += float(got['mean_loss'])
  ref = iqn_f64(*iqn_args(g))
  check_rule('iqn partial means %d' % rows, partial, ref['mean_loss'],
             iqn_port_case(g)['mean_loss'])


# ------------------------------------------------------------- the mean's ticket ----
TICKET_SEQUENCE = [  # (batch, mean, sharded)
    (1, True, False), (4096, True, True), (7, False, False), (4096, True, False),
    (1, True, True), (4096, False, True), (7, True, True), (4096, True, False),
    (7, True, False), (1, False, False)]


def _ticket_calls(gpu, entry):
  """The sequence's inputs and preallocated outputs (means pre-filled with NaN)."""
  torch = gpu.torch
  calls = []
  for i, (batch, mean, sharded) in enumerate(TICKET_SEQUENCE):
    if entry == 'iqn':
      c = make_iqn_case(100 + i, batch, 6, 4, 4, 2, {})
      out = {'loss': torch.empty(batch, device='cuda'),
             'next_action': torch.empty(batch, dtype=torch.int32, device='cuda')}
    else:
      c = make_dqn_case(100 + i, batch, 6, {})
      out = {'loss': torch.empty(batch, device='cuda')}
    if mean:
      out['mean_loss'] = torch.full((), float('nan'), device='cuda')
    count = None
    if sharded:  # a rank with all but 2 of its rows valid (one row: all valid)
      count = torch.tensor([max(batch - 2, 1)], dtype=torch.int32, device='cuda')
    calls.append(dict(c=c, out=out, count=count, global_batch=batch + 3,
                      dev=None))
  return calls


def _launch(gpu, entry, call):
  c, out = call['c'], call['out']
  sharded = None if call['count'] is None else (call['global_batch'], call['count'])
  if call['dev'] is None:
    call['dev'] = (
        {k: _dev(gpu, c[k]) for k in ('online', 'quantiles', 'target', 'action',
                                       'actions', 'rewards', 'terminals')}
        if entry == 'iqn' else
        {k: _dev(gpu, c[k]) for k in ('online_q', 'target_q', 'actions', 'rewards',
                                       'terminals')})
  d = call['dev']
  if entry == 'iqn':
    gpu.iqn.quantile_huber_loss(
        d['online'], d['quantiles'], d['target'], d['action'], d['actions'],
        d['rewards'], d['terminals'], c['gamma_n'], c['kappa'], out=out,
        sharded=sharded)
  else:
    gpu.dqn.dqn_loss(d['online_q'], d['target_q'], d['actions'], d['rewards'],
                     d['terminals'], c['gamma_n'], out=out, sharded=sharded)


def _check_means(gpu, entry, calls, label):
  for i, call in enumerate(calls):
    if 'mean_loss' not in call['out']:
      continue
    c = call['c']
    got = float(call['out']['mean_loss'])
    rows = len(c['rewards']) if call['count'] is None else int(call['count'])
    if entry == 'iqn':
      ref = iqn_f64(*iqn_args(_iqn_rows(c, np.arange(rows))))['loss']
      port = iqn_port_case(_iqn_rows(c, np.arange(rows)))['loss']
    else:
      sub = {k: (v[:rows] if isinstance(v, np.ndarray) else v) for k, v in c.items()}
      ref = dqn_f64(sub['rewards'], sub['terminals'], sub['actions'], sub['online_q'],
                    sub['target_q'], sub['gamma_n'])['loss']
      port = dqn_port_case(sub)['loss']
    div = len(c['rewards']) if call['count'] is None else call['global_batch']
    assert np.isfinite(got), (label, i)
    check_rule('%s #%d' % (label, i), got, ref.sum() / div,
               F32(port.astype(F64).sum() / div))


@pytest.mark.gpu
@pytest.mark.parametrize('entry', ['iqn', 'dqn'])
def test_mean_over_changing_launches(gpu, entry):
  """One stream, grid sizes 1, 4096, 7, 4096, ..., the mean on and off, sharded and
  unsharded launches in turn: every mean is right, so the IQN ticket is back at 0
  after each launch that took it; then the same ten launches captured in one CUDA
  graph and replayed twice."""
  torch = gpu.torch
  calls = _ticket_calls(gpu, entry)
  for call in calls:
    _launch(gpu, entry, call)
  torch.cuda.synchronize()
  _check_means(gpu, entry, calls, entry + ' eager')
  stream = torch.cuda.Stream()
  stream.wait_stream(torch.cuda.current_stream())
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.stream(stream):
    for call in calls:  # warm-up on the capture stream
      _launch(gpu, entry, call)
    stream.synchronize()
    with torch.cuda.graph(graph, stream=stream):
      for call in calls:
        _launch(gpu, entry, call)
  torch.cuda.synchronize()
  for replay in range(2):
    for call in calls:
      if 'mean_loss' in call['out']:
        call['out']['mean_loss'].fill_(float('nan'))
    graph.replay()
    torch.cuda.synchronize()
    _check_means(gpu, entry, calls, '%s graph replay %d' % (entry, replay))
