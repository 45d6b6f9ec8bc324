"""Prioritized replay on the GPU behind the reference's API.

Drop-in for `dopamine/replay_memory/prioritized_replay_buffer.py`
(OutOfGraphPrioritizedReplayBuffer, prioritized_replay_buffer.py:36;
WrappedPrioritizedReplayBuffer, :257): `add(..., priority)`,
`sample_index_batch`, `sample_transition_batch` (with the trailing
`sampling_probabilities`), `set_priority`, `get_priority`, and the `sum_tree`
attribute the Rainbow agent reads `max_recorded_priority` from.

Stratified sampling, the validity test, the in-order retry of invalid slots with a
shared attempt budget, the frame-stack gather and the batched, order-preserving
priority write-back are CUDA kernels (`include/b200_replay.h`).  With
rng='reference' the uniforms are drawn from Python's `random` exactly as the
reference does, so identical seeds give identical indices.
"""
import ctypes
import pickle
import random

import numpy as np

from dopamine_b200 import _native
from dopamine_b200.replay_memory import circular_replay_buffer
from dopamine_b200.replay_memory import sum_tree
from dopamine_b200.replay_memory.circular_replay_buffer import ReplayElement


class _MaxRecordedPriority(object):
  """Sentinel for add(): use sum_tree.max_recorded_priority as of that add,
  resolved on the device (what RainbowAgent._store_transition passes,
  rainbow_agent.py:330-334) without reading it back to the host."""

  def __repr__(self):
    return 'MAX_RECORDED_PRIORITY'


MAX_RECORDED_PRIORITY = _MaxRecordedPriority()


# -- checkpoint compatibility with the reference --------------------------------
# The reference pickles `memory.sum_tree`, a dopamine.replay_memory.sum_tree.SumTree
# instance whose state is {'nodes': [level arrays], 'max_recorded_priority': x}
# (sum_tree.py:79-89, written by circular_replay_buffer.py:641).  The tree lives in
# HBM here, so the same pickle is produced / consumed from its level arrays without
# the reference being importable.
_REFERENCE_TREE_CLASS = ('dopamine.replay_memory.sum_tree', 'SumTree')


class SumTreeState(object):
  """What a pickled reference SumTree unpickles to when the reference package is
  absent: a plain holder of `nodes` and `max_recorded_priority`."""


class _TreeUnpickler(pickle.Unpickler):

  def find_class(self, module, name):
    if (module, name) == _REFERENCE_TREE_CLASS or (
        module.endswith('replay_memory.sum_tree') and name == 'SumTree'):
      return SumTreeState
    return super(_TreeUnpickler, self).find_class(module, name)


def dump_reference_sum_tree(nodes, max_recorded_priority, outfile):
  """Writes the pickle the reference's save() writes for its SumTree: protocol-2
  `SumTree.__new__()` + `__dict__.update(state)`; loads back into the reference
  class when it is importable, into SumTreeState otherwise."""
  state = {'nodes': [np.asarray(level, dtype=np.float64) for level in nodes],
           'max_recorded_priority': max_recorded_priority}
  body = pickle.dumps(state, protocol=2)
  assert body[:2] == b'\x80\x02' and body[-1:] == b'.'
  module, name = _REFERENCE_TREE_CLASS
  outfile.write(b'\x80\x02' +                       # PROTO 2
                b'c' + module.encode() + b'\n' + name.encode() + b'\n' +  # GLOBAL
                b')\x81' +                           # EMPTY_TUPLE, NEWOBJ
                body[2:-1] +                         # the state dict
                b'b.')                               # BUILD, STOP


def _is_cuda_tensor(x):
  return hasattr(x, 'is_cuda') and x.is_cuda


class OutOfGraphPrioritizedReplayBuffer(
    circular_replay_buffer.OutOfGraphReplayBuffer):
  """Replay buffer with proportional prioritization (Schaul et al., 2015)."""

  _PRIORITIZED = 1

  def __init__(self,
               observation_shape,
               stack_size,
               replay_capacity,
               batch_size,
               update_horizon=1,
               gamma=0.99,
               max_sample_attempts=1000,
               extra_storage_types=None,
               observation_dtype=np.uint8,
               terminal_dtype=np.uint8,
               action_shape=(),
               action_dtype=np.int32,
               reward_shape=(),
               reward_dtype=np.float32,
               output='numpy',
               rng='reference',
               seed=0,
               reuse_outputs=False):
    super(OutOfGraphPrioritizedReplayBuffer, self).__init__(
        observation_shape=observation_shape,
        stack_size=stack_size,
        replay_capacity=replay_capacity,
        batch_size=batch_size,
        update_horizon=update_horizon,
        gamma=gamma,
        max_sample_attempts=max_sample_attempts,
        extra_storage_types=extra_storage_types,
        observation_dtype=observation_dtype,
        terminal_dtype=terminal_dtype,
        action_shape=action_shape,
        action_dtype=action_dtype,
        reward_shape=reward_shape,
        reward_dtype=reward_dtype,
        output=output,
        rng=rng,
        seed=seed,
        reuse_outputs=reuse_outputs)
    tree_handle = ctypes.c_void_p(self._lib.b2r_buffer_tree(self._h))
    # Reads of the tree must see every staged add (PRB:139-140 sets the priority
    # inside add), hence the flush hook.
    self.sum_tree = sum_tree.SumTree(
        replay_capacity, _handle=tree_handle, _before_read=self._flush)

  def get_add_args_signature(self):
    parent_add_signature = super(OutOfGraphPrioritizedReplayBuffer,
                                 self).get_add_args_signature()
    return parent_add_signature + [ReplayElement('priority', (), np.float32)]

  def add(self, observation, action, reward, terminal, *args):
    """add(observation, action, reward, terminal, *extras, priority)."""
    if len(args) == 1:
      last = args[0]
      if last is MAX_RECORDED_PRIORITY:
        if self._try_fast_add(observation, action, reward, terminal, 0.0,
                              _native.PRIORITY_MAX_RECORDED):
          return
      elif type(last) in circular_replay_buffer._PLAIN_SCALARS:  # pylint: disable=protected-access
        if self._try_fast_add(observation, action, reward, terminal, last,
                              _native.PRIORITY_EXPLICIT):
          return
    if args and args[-1] is MAX_RECORDED_PRIORITY:
      self._check_add_types(observation, action, reward, terminal,
                            *(args[:-1] + (0.0,)))
      priority, mode = 0.0, _native.PRIORITY_MAX_RECORDED
    else:
      self._check_add_types(observation, action, reward, terminal, *args)
      priority, mode = float(args[-1]), _native.PRIORITY_EXPLICIT
    self._native_add((observation, action, reward, terminal) + tuple(args[:-1]),
                     priority, mode)

  # -- sampling (PRB:142-201) ---------------------------------------------------
  def _native_sample(self, batch_size, queries, retries):
    out = np.zeros(batch_size, dtype=np.int32)
    used, fail_slot = ctypes.c_int32(0), ctypes.c_int32(0)
    status = self._lib.b2r_sample_indices_prioritized(
        self._h, batch_size, _native.ptr(queries), len(retries),
        _native.ptr(retries) if len(retries) else None, _native.ptr(out),
        ctypes.byref(used), ctypes.byref(fail_slot), self._stream())
    return status, out, used.value, fail_slot.value

  def add_batch(self, observations, actions, rewards, terminals, *args):
    """add_batch(observations, actions, rewards, terminals, *extras, priorities): n
    consecutive `add`s in one native call.  `priorities` is an array of n values or
    MAX_RECORDED_PRIORITY (every row takes sum_tree.max_recorded_priority as it stands
    when the row is applied, RA:330-334)."""
    if not args:
      raise ValueError('add_batch expects the priorities as its last argument')
    last = args[-1]
    if last is MAX_RECORDED_PRIORITY:
      self._native_add_batch((observations, actions, rewards, terminals) + tuple(args[:-1]),
                             None, _native.PRIORITY_MAX_RECORDED)
    else:
      self._native_add_batch((observations, actions, rewards, terminals) + tuple(args[:-1]),
                             last, _native.PRIORITY_EXPLICIT)

  def sample_index_batch(self, batch_size):
    """Stratified prioritized indices with in-order retries (PRB:142-171).

    rng='reference': list of ints, consuming `random` like the reference.
    rng='device': int32 CUDA tensor, no host round trip.
    """
    if self._rng == 'device':
      import torch  # pylint: disable=g-import-not-at-top
      out = torch.empty(batch_size, dtype=torch.int32, device='cuda')
      _native.check(self._lib.b2r_sample_indices_device(
          self._h, batch_size, self._seed, self._next_offset(), out.data_ptr(),
          self._stream()))
      return out
    start_state = random.getstate()
    bounds = np.linspace(0., 1., batch_size + 1)
    queries = np.array([random.uniform(bounds[i], bounds[i + 1])
                        for i in range(batch_size)], dtype=np.float64)
    # First pass without retry draws: succeeds iff every stratified pick is valid,
    # which is the common case, and then no extra uniforms are consumed.
    status, out, used, fail_slot = self._native_sample(
        batch_size, queries, np.zeros(0, dtype=np.float64))
    if status == _native.ERR_SAMPLE_ATTEMPTS and self._max_sample_attempts > 0:
      after_strata = random.getstate()
      retries = np.array([random.random()
                          for _ in range(self._max_sample_attempts)],
                         dtype=np.float64)
      status, out, used, fail_slot = self._native_sample(
          batch_size, queries, retries)
      random.setstate(after_strata)
      for _ in range(used):  # advance by what the reference would have drawn
        random.random()
    if status == _native.ERR_EMPTY_TREE:
      random.setstate(start_state)  # the reference raises before drawing
      raise Exception('Cannot sample from an empty sum tree.')
    if status == _native.ERR_SAMPLE_ATTEMPTS:
      raise RuntimeError(
          'Max sample attempts: Tried {} times but only sampled {}'
          ' valid indices. Batch size is {}'.
          format(self._max_sample_attempts, fail_slot, batch_size))
    _native.check(status)
    return [int(i) for i in out]

  # sample_transition_batch: the parent's, whose gather kernel also fills
  # `sampling_probabilities` with f32(leaf) (PRB:193-200) since
  # get_transition_elements lists it.

  def get_transition_elements(self, batch_size=None):
    parent_transition_type = (
        super(OutOfGraphPrioritizedReplayBuffer,
              self).get_transition_elements(batch_size))
    batch_size = self._batch_size if batch_size is None else batch_size
    probablilities_type = [
        ReplayElement('sampling_probabilities', (batch_size,), np.float32)
    ]
    return parent_transition_type + probablilities_type

  # -- priorities (PRB:203-235) ----------------------------------------------------
  def set_priority(self, indices, priorities):
    """Sets priorities in array order (later duplicates win, PRB:213-214).

    numpy inputs follow the reference contract (int32 indices); CUDA tensors
    (int32 indices, float32 priorities — e.g. straight from the loss kernel) are
    applied without leaving the device.
    """
    if _is_cuda_tensor(indices) or _is_cuda_tensor(priorities):
      import torch  # pylint: disable=g-import-not-at-top
      assert indices.dtype == torch.int32, (
          'Indices must be integers, given: {}'.format(indices.dtype))
      priorities = priorities.to(dtype=torch.float32).contiguous()
      indices = indices.contiguous()
      _native.check(self._lib.b2r_set_priority_device(
          self._h, indices.numel(), indices.data_ptr(), priorities.data_ptr(),
          self._stream()))
      return
    assert indices.dtype == np.int32, ('Indices must be integers, '
                                       'given: {}'.format(indices.dtype))
    n = min(len(indices), len(priorities))  # zip() semantics
    idx = np.ascontiguousarray(indices[:n], dtype=np.int32)
    values = np.ascontiguousarray(np.asarray(priorities)[:n], dtype=np.float64)
    bad = ctypes.c_int64(-1)
    status = self._lib.b2r_set_priority(
        self._h, n, _native.ptr(idx), _native.ptr(values), ctypes.byref(bad),
        self._stream())
    if status == _native.ERR_NEGATIVE_PRIORITY:
      raise ValueError('Sum tree values should be nonnegative. Got {}'.
                       format(priorities[bad.value]))
    if status == _native.ERR_INDEX_RANGE:
      raise IndexError(_native.last_error())
    _native.check(status)

  def get_priority(self, indices):
    """float32 leaf priorities for a batch of indices (0 for unused slots)."""
    if _is_cuda_tensor(indices):
      import torch  # pylint: disable=g-import-not-at-top
      assert indices.dtype == torch.int32, (
          'Indices must be int32s, given: {}'.format(indices.dtype))
      out = torch.empty(indices.numel(), dtype=torch.float32, device='cuda')
      _native.check(self._lib.b2r_get_priority_device(
          self._h, indices.numel(), indices.contiguous().data_ptr(),
          out.data_ptr(), self._stream()))
      return out
    assert indices.shape, 'Indices must be an array.'
    assert indices.dtype == np.int32, ('Indices must be int32s, '
                                       'given: {}'.format(indices.dtype))
    idx = np.ascontiguousarray(indices)
    out = np.empty(len(idx), dtype=np.float32)
    status = self._lib.b2r_get_priority(self._h, len(idx), _native.ptr(idx),
                                        _native.ptr(out), self._stream())
    if status == _native.ERR_INDEX_RANGE:
      raise IndexError(_native.last_error())
    _native.check(status)
    return out

  # -- checkpointing: the tree is saved as its level arrays ---------------------------
  def _pickle_attribute(self, attr, value, outfile):
    if attr == 'sum_tree':  # byte-compatible with the reference's pickled SumTree
      dump_reference_sum_tree(value.nodes, value.max_recorded_priority, outfile)
      return
    super(OutOfGraphPrioritizedReplayBuffer, self)._pickle_attribute(
        attr, value, outfile)

  def _unpickle_attribute(self, attr, infile):
    if attr == 'sum_tree':
      return _TreeUnpickler(infile).load()
    return super(OutOfGraphPrioritizedReplayBuffer, self)._unpickle_attribute(
        attr, infile)

  def _restore_attribute(self, attr, value):
    if attr == 'sum_tree':
      nodes = value['nodes'] if isinstance(value, dict) else value.nodes
      max_recorded = (value['max_recorded_priority'] if isinstance(value, dict)
                      else value.max_recorded_priority)
      if len(nodes) != len(self.sum_tree.nodes):
        raise ValueError('checkpointed sum tree has {} levels, this buffer {}'.
                         format(len(nodes), len(self.sum_tree.nodes)))
      for level, array in enumerate(nodes):
        array = np.ascontiguousarray(array, dtype=np.float64)
        _native.check(self._lib.b2r_tree_write_level(
            self.sum_tree._h, level, _native.ptr(array), self._stream()))  # pylint: disable=protected-access
      self.sum_tree.max_recorded_priority = float(max_recorded)
      return
    super(OutOfGraphPrioritizedReplayBuffer, self)._restore_attribute(attr, value)


class WrappedPrioritizedReplayBuffer(
    circular_replay_buffer.WrappedReplayBuffer):
  """The reference's graph-side wrapper (PRB:257-365) without TensorFlow.

  `tf_set_priority` / `tf_get_priority` take and return device tensors; like the
  reference (PRB:316-320) only extra_storage_types and observation_dtype are
  forwarded to the inner memory.
  """

  def __init__(self,
               observation_shape,
               stack_size,
               use_staging=True,
               replay_capacity=1000000,
               batch_size=32,
               update_horizon=1,
               gamma=0.99,
               max_sample_attempts=1000,
               extra_storage_types=None,
               observation_dtype=np.uint8,
               terminal_dtype=np.uint8,
               action_shape=(),
               action_dtype=np.int32,
               reward_shape=(),
               reward_dtype=np.float32,
               rng='reference',
               seed=0,
               reuse_outputs=False):
    memory = OutOfGraphPrioritizedReplayBuffer(
        observation_shape, stack_size, replay_capacity, batch_size,
        update_horizon, gamma, max_sample_attempts,
        extra_storage_types=extra_storage_types,
        observation_dtype=observation_dtype, output='torch', rng=rng, seed=seed,
        reuse_outputs=reuse_outputs)
    super(WrappedPrioritizedReplayBuffer, self).__init__(
        observation_shape,
        stack_size,
        use_staging,
        replay_capacity,
        batch_size,
        update_horizon,
        gamma,
        wrapped_memory=memory,
        extra_storage_types=extra_storage_types,
        observation_dtype=observation_dtype,
        terminal_dtype=terminal_dtype,
        action_shape=action_shape,
        action_dtype=action_dtype,
        reward_shape=reward_shape,
        reward_dtype=reward_dtype)

  def tf_set_priority(self, indices, priorities):
    """Device-side priority write-back (the reference's py_func, PRB:338-350)."""
    return self.memory.set_priority(indices, priorities)

  def tf_get_priority(self, indices):
    """Device-side priority read (PRB:352-365)."""
    return self.memory.get_priority(indices)
