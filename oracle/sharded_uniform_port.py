"""CPU statement of the sharded UNIFORM sampling rule.  TEST INFRASTRUCTURE ONLY.

The reference is single-process and has no notion of shards, so the cross-shard rule is
DEFINED here as the natural extension of circular_replay_buffer.py:462-470 to a virtual
buffer whose index range is the concatenation of the shards' ranges: the result is
uniform over the union of the shards' valid transitions.  Each shard is a
`replay_port.PortReplay`; the uniforms are those of `philox_port`.
"""
import numpy as np


def uniform_span(shard):
  """(min_id, span) of a PortReplay shard: circular_replay_buffer.py:449-460, with a
  shard that has too few transitions spanning nothing."""
  try:
    lo, hi = shard.uniform_bounds()
  except RuntimeError:
    return 0, 0
  return lo, max(0, hi - lo)


def sharded_uniform_sample(shards, uniforms, global_batch, max_attempts):
  """ONE uniform batch (circular_replay_buffer.py:462-470) over the concatenation of the
  shards' index ranges.  shards: list of PortReplay; uniforms[j]: the uniform in [0, 1)
  of draw j (philox_port.uniform53(seed, offset + step, j) for the device sampler).

  Draw j picks offset o = min(int(u_j * N), N - 1) into the N = sum of the spans; its
  owner is the shard the rank-order scan `o < n_g ? g : o -= n_g` stops at, the candidate
  (min_id_owner + o) % capacity.  Draws are processed in order while accepted <
  global_batch and rejected < max_attempts; a draw is accepted iff it is a valid
  transition of its owner, the k-th accepted draw is global row k.  Returns per shard
  (slots, indices): its accepted draws' global rows and indices, in row order.  Raises
  as the reference does for too few transitions and for exhausted attempts."""
  bounds = [uniform_span(s) for s in shards]
  total = sum(span for _, span in bounds)
  if total == 0:
    raise RuntimeError('Cannot sample a batch: no shard holds more than stack size + '
                       'update_horizon transitions.')
  rows = [([], []) for _ in shards]
  accepted = rejected = j = 0
  while accepted < global_batch and rejected < max_attempts:
    o = min(int(np.float64(uniforms[j]) * np.float64(total)), total - 1)
    j += 1
    g = 0
    while not o < bounds[g][1]:
      o -= bounds[g][1]
      g += 1
    candidate = (bounds[g][0] + o) % shards[g].capacity
    if shards[g].is_valid_transition(candidate):
      rows[g][0].append(accepted)
      rows[g][1].append(candidate)
      accepted += 1
    else:
      rejected += 1
  if accepted != global_batch:
    raise RuntimeError(
        'Max sample attempts: Tried {} times but only sampled {}'
        ' valid indices. Batch size is {}'.format(max_attempts, accepted, global_batch))
  return rows
