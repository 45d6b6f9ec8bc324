"""IQN's target and quantile-Huber loss as one fused CUDA kernel.

Drop-in for the loss side of `ImplicitQuantileAgent`
(dopamine/agents/implicit_quantile/implicit_quantile_agent.py): the greedy next action
from the action network's quantile samples (:176-188), `_build_target_quantile_values_op`
(:190-231) and the loss of `_build_train_op` (:233-315), over torch CUDA tensors that
keep the reference's layout — every network output is a (samples * batch, num_actions)
f32 matrix whose rows are sample-major (row = sample * batch + b), `quantiles` is the
(num_tau_samples * batch, 1) tau column of the online pass.  SURVEY.md section 8f,
row 4: an additional fused epilogue behind the same replay batch.
"""
import ctypes
import math

import numpy as np

from dopamine_b200 import _native


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


def cumulative_gamma(gamma, update_horizon):
  """dqn_agent.py:175."""
  return math.pow(gamma, update_horizon)


def quantile_huber_loss(online_quantile_values, quantiles, target_quantile_values,
                        action_quantile_values, actions, rewards, terminals,
                        cumulative_gamma, kappa=1.0, want_grad=False,  # pylint: disable=redefined-outer-name
                        want_mean=True, out=None, sharded=None):
  """Per-row IQN loss for one replay batch, on the device.

  Args:
    online_quantile_values: (N * B, A) f32 CUDA, online network on `state`.
    quantiles: (N * B, 1) or (N * B,) f32 CUDA, the taus of those rows.
    target_quantile_values: (N' * B, A) f32 CUDA, target network on `next_state`.
    action_quantile_values: (K * B, A) f32 CUDA, the network that picks the next
      action (target net; online net with double_dqn).
    actions: (B,) int32; rewards: (B,) f32; terminals: (B,) uint8.
    cumulative_gamma: gamma ** update_horizon; kappa: Huber threshold (> 0).
  Returns:
    dict with 'loss' (B,), 'next_action' (B,) int32, optionally 'mean_loss'
    (scalar) and 'grad' (N * B, A) = d mean(loss) / d online_quantile_values.
    sharded: (global_batch, count) — the B rows are one rank's share of a global batch
    of `global_batch` strata, as `ShardedPrioritizedReplay.sample_transition_batch_sharded`
    returns it (b2r_iqn_loss_sharded): the first `count` rows ((1,) int32 CUDA tensor)
    are valid, the mean and its gradient are this rank's part of the global batch's
    (divisor global_batch), rows past the count get loss 0 and zero gradients and keep
    their old next_action.
  """
  torch = _torch()
  if not kappa > 0:
    raise ValueError('kappa must be positive, got {}'.format(kappa))
  batch = actions.shape[0]
  if batch < 1:
    raise ValueError('batch must be >= 1, got {}'.format(batch))
  num_actions = online_quantile_values.shape[1]
  for name, x in (('online_quantile_values', online_quantile_values),
                  ('target_quantile_values', target_quantile_values),
                  ('action_quantile_values', action_quantile_values),
                  ('quantiles', quantiles), ('rewards', rewards)):
    if x.dtype != torch.float32 or not x.is_cuda:
      raise ValueError('{} must be a float32 CUDA tensor'.format(name))
  if actions.dtype != torch.int32 or terminals.dtype != torch.uint8:
    raise ValueError('actions must be int32 and terminals uint8')
  sizes = []
  for name, x in (('online_quantile_values', online_quantile_values),
                  ('target_quantile_values', target_quantile_values),
                  ('action_quantile_values', action_quantile_values)):
    if x.dim() != 2 or x.shape[1] != num_actions or x.shape[0] % batch:
      raise ValueError('{} must be (samples * batch, num_actions), got {}'.format(
          name, tuple(x.shape)))
    sizes.append(x.shape[0] // batch)
  n, n_prime, k = sizes
  if quantiles.numel() != n * batch:
    raise ValueError('quantiles must hold one tau per online row')
  if sharded is not None:
    global_batch, count = sharded
    if (not isinstance(count, torch.Tensor) or count.dtype != torch.int32 or
        not count.is_cuda or tuple(count.shape) != (1,)):
      raise ValueError('count must be a (1,) int32 CUDA tensor')
    if int(global_batch) < 1:
      raise ValueError('global_batch must be >= 1, got {}'.format(global_batch))
  dev = online_quantile_values.device
  if out is None:
    out = {'loss': torch.empty(batch, dtype=torch.float32, device=dev),
           'next_action': torch.empty(batch, dtype=torch.int32, device=dev)}
    if want_mean:
      out['mean_loss'] = torch.empty((), dtype=torch.float32, device=dev)
    if want_grad:
      out['grad'] = torch.empty(n * batch, num_actions, dtype=torch.float32, device=dev)
  keep = [online_quantile_values.contiguous(), target_quantile_values.contiguous(),
          action_quantile_values.contiguous(), quantiles.contiguous(),
          actions.contiguous(), rewards.contiguous(), terminals.contiguous()]
  args = _native.IqnArgs()
  args.batch, args.num_actions = batch, num_actions
  args.num_tau_samples, args.num_tau_prime_samples = n, n_prime
  args.num_quantile_samples = k
  args.cumulative_gamma = float(np.float32(cumulative_gamma))
  args.kappa = float(np.float32(kappa))
  args.online_quantile_values = keep[0].data_ptr()
  args.target_quantile_values = keep[1].data_ptr()
  args.action_quantile_values = keep[2].data_ptr()
  args.quantiles = keep[3].data_ptr()
  args.actions = keep[4].data_ptr()
  args.rewards = keep[5].data_ptr()
  args.terminals = keep[6].data_ptr()
  args.loss = out['loss'].data_ptr()
  args.next_action = out['next_action'].data_ptr() if 'next_action' in out else None
  args.mean_loss = out['mean_loss'].data_ptr() if 'mean_loss' in out else None
  args.grad_quantile_values = out['grad'].data_ptr() if 'grad' in out else None
  if sharded is None:
    _native.check(_native.lib().b2r_iqn_loss(ctypes.byref(args),
                                             _native.current_stream()))
    return out
  _native.check(_native.lib().b2r_iqn_loss_sharded(
      ctypes.byref(args), count.data_ptr(), int(global_batch), _native.current_stream()))
  return out


class QuantileHuberLoss(object):
  """Differentiable wrapper: `mean_loss, loss = QuantileHuberLoss.apply(...)`; the
  gradient flows to `online_quantile_values` only (the target side is behind
  tf.stop_gradient in the reference, :240-241)."""

  _fn = None

  @classmethod
  def _function(cls):
    if cls._fn is None:
      torch = _torch()

      class _Fn(torch.autograd.Function):

        @staticmethod
        def forward(ctx, online, taus, target, action_net, actions, rewards,  # pylint: disable=redefined-outer-name
                    terminals, gamma_n, kappa, sharded):  # pylint: disable=redefined-outer-name
          out = quantile_huber_loss(online.detach(), taus.detach(), target.detach(),
                                    action_net.detach(), actions, rewards, terminals,
                                    gamma_n, kappa, want_grad=True, sharded=sharded)
          ctx.save_for_backward(out['grad'])
          ctx.mark_non_differentiable(out['loss'])
          return out['mean_loss'], out['loss']

        @staticmethod
        def backward(ctx, grad_mean, *unused):
          (grad,) = ctx.saved_tensors
          return (grad * grad_mean,) + (None,) * 9

      cls._fn = _Fn
    return cls._fn

  @classmethod
  def apply(cls, online_quantile_values, quantiles, target_quantile_values,
            action_quantile_values, actions, rewards, terminals, gamma_n, kappa=1.0):
    return cls._function().apply(online_quantile_values, quantiles,
                                 target_quantile_values, action_quantile_values, actions,
                                 rewards, terminals, gamma_n, kappa, None)


class ShardedQuantileHuberLoss(QuantileHuberLoss):
  """`QuantileHuberLoss` over one rank's share of a sharded global batch
  (b2r_iqn_loss_sharded): `mean, loss = ShardedQuantileHuberLoss.apply(..., kappa,
  sharded)` with `sharded` = (global_batch, count) as in `quantile_huber_loss`.  `mean`
  is this rank's partial mean (its rows' losses over the global batch size) and backward
  gives its gradient; summed over the ranks both are the global batch's."""

  @classmethod
  def apply(cls, online_quantile_values, quantiles, target_quantile_values,
            action_quantile_values, actions, rewards, terminals, gamma_n, kappa,
            sharded):
    return cls._function().apply(online_quantile_values, quantiles,
                                 target_quantile_values, action_quantile_values, actions,
                                 rewards, terminals, gamma_n, kappa, tuple(sharded))
