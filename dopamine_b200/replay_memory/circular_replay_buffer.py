"""HBM-resident replay buffer behind the reference's OutOfGraphReplayBuffer API.

Drop-in for `dopamine/replay_memory/circular_replay_buffer.py`
(OutOfGraphReplayBuffer, circular_replay_buffer.py:80; WrappedReplayBuffer,
circular_replay_buffer.py:692): same constructor arguments and defaults, same
methods, same tuple order of `sample_transition_batch`, same exception types and
messages.  Storage, validity checks, index sampling and batch assembly run as CUDA
kernels on one B200 through the C ABI in `include/b200_replay.h`; this module only
validates arguments, draws the random numbers the reference would draw
(np.random, so a seeded run picks the same indices) and allocates outputs.

What is different on purpose:
  * `sample_transition_batch` can return device tensors (`output='torch'`) so the
    batch never leaves HBM; `output='numpy'` (default, reference behaviour) copies
    it to host arrays.
  * `rng='device'` draws indices on the GPU (Philox) without host round trips; it
    follows the same sampling rules but not numpy's random stream.
  * vector-valued rewards are not supported (the reference's np.sum over them only
    broadcasts by accident).
"""
import collections
import ctypes
import gzip
import io
import math
import os
import pickle
import struct
import sys
import zlib

import numpy as np

from dopamine_b200 import _native

# Same names as the reference module (circular_replay_buffer.py:43-50).
ReplayElement = (
    collections.namedtuple('shape_type', ['name', 'shape', 'type']))
STORE_FILENAME_PREFIX = '$store$_'
CHECKPOINT_DURATION = 4


def invalid_range(cursor, replay_capacity, stack_size, update_horizon):
  """Indices around the cursor that cannot start a transition (CRB:53-77)."""
  assert cursor < replay_capacity
  return np.array(
      [(cursor - update_horizon + i) % replay_capacity
       for i in range(stack_size + update_horizon)])


# Blocked gzip store files: every member starts with this header (FLG = FEXTRA, MTIME 0,
# XFL 0, OS 255, one 'BC' subfield of 2 bytes) followed by BSIZE = member size - 1.
_BGZF_PREFIX = b'\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00'
BGZF_HEADER_BYTES = len(_BGZF_PREFIX) + 2


def npy_header(shape, dtype):
  """The bytes `np.save(f, a, allow_pickle=False)` writes before the data of a
  C-contiguous array `a` of this shape and dtype (format 1.0, or 2.0 when the header
  does not fit 1.0, as np.save chooses)."""
  fmt = np.lib.format
  d = {'descr': fmt.dtype_to_descr(np.dtype(dtype)), 'fortran_order': False,
       'shape': tuple(int(s) for s in shape)}
  buf = io.BytesIO()
  try:
    fmt.write_array_header_1_0(buf, d)
  except ValueError:
    buf = io.BytesIO()
    fmt.write_array_header_2_0(buf, d)
  return buf.getvalue()


def bgzf_member(payload):
  """`payload` as one blocked-gzip member with a single stored block."""
  body = (b'\x01' + struct.pack('<HH', len(payload), len(payload) ^ 0xFFFF) +
          bytes(payload))
  size = BGZF_HEADER_BYTES + len(body) + 8
  return (_BGZF_PREFIX + struct.pack('<H', size - 1) + body +
          struct.pack('<II', zlib.crc32(payload), len(payload)))


def _write_all(fd, data):
  view = memoryview(data)
  while view:
    view = view[os.write(fd, view):]


def _torch():
  import torch  # pylint: disable=g-import-not-at-top
  return torch


_TORCH_DTYPES = None
# Scalars whose int() / float() conversion equals numpy's assignment cast.
_PLAIN_SCALARS = frozenset([int, float, bool, np.int32, np.int64, np.uint8,
                            np.float32, np.float64, np.bool_])


def _torch_dtype(np_dtype):
  global _TORCH_DTYPES
  torch = _torch()
  if _TORCH_DTYPES is None:
    _TORCH_DTYPES = {
        np.dtype(np.uint8): torch.uint8, np.dtype(np.int8): torch.int8,
        np.dtype(np.int16): torch.int16, np.dtype(np.int32): torch.int32,
        np.dtype(np.int64): torch.int64, np.dtype(np.float16): torch.float16,
        np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64,
        np.dtype(np.bool_): torch.bool,
    }
  return _TORCH_DTYPES.get(np.dtype(np_dtype))


class _StoreView(object):
  """`memory._store[name]`: host copies of the HBM-resident storage arrays."""

  def __init__(self, owner):
    self._owner = owner

  def keys(self):
    return [e.name for e in self._owner.get_storage_signature()]

  def __contains__(self, name):
    return name in self.keys()

  def __iter__(self):
    return iter(self.keys())

  def items(self):
    return [(k, self[k]) for k in self.keys()]

  def __getitem__(self, name):
    return self._owner._read_column(name)  # pylint: disable=protected-access

  def __setitem__(self, name, array):
    self._owner._write_column(name, array)  # pylint: disable=protected-access


class OutOfGraphReplayBuffer(object):
  """Circular replay buffer whose storage and sampling live on the GPU.

  Attributes:
    add_count: np.array (0-d), transitions added so far incl. padding ones.
    invalid_range: np.array, indices around the cursor that cannot be sampled.
  """

  _PRIORITIZED = 0

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
    assert isinstance(observation_shape, tuple)
    if replay_capacity < update_horizon + stack_size:
      raise ValueError('There is not enough capacity to cover '
                       'update_horizon and stack_size.')
    if output not in ('numpy', 'torch'):
      raise ValueError("output must be 'numpy' or 'torch'")
    if rng not in ('reference', 'device'):
      raise ValueError("rng must be 'reference' or 'device'")
    if tuple(reward_shape) != ():
      raise NotImplementedError('only scalar rewards are supported')
    if np.dtype(reward_dtype) not in (np.dtype(np.float32),
                                      np.dtype(np.float64)):
      raise NotImplementedError('reward_dtype must be float32 or float64')
    if np.dtype(terminal_dtype).kind not in 'iub':
      raise NotImplementedError('terminal_dtype must be an integer type')

    self._action_shape = action_shape
    self._action_dtype = action_dtype
    self._reward_shape = reward_shape
    self._reward_dtype = reward_dtype
    self._observation_shape = observation_shape
    self._stack_size = stack_size
    self._state_shape = self._observation_shape + (self._stack_size,)
    self._replay_capacity = replay_capacity
    self._batch_size = batch_size
    self._update_horizon = update_horizon
    self._gamma = gamma
    self._observation_dtype = observation_dtype
    self._terminal_dtype = terminal_dtype
    self._max_sample_attempts = max_sample_attempts
    if extra_storage_types:
      self._extra_storage_types = extra_storage_types
    else:
      self._extra_storage_types = []
    self._output = output
    self._rng = rng
    self._seed = int(seed)
    self._draw_counter = 0
    # The reference returns fresh arrays on every call (its StagingArea keeps
    # pointers, CRB:419-421).  reuse_outputs=True hands back the same buffers per
    # batch size instead: no allocation on the sampling path.
    self._reuse_outputs = bool(reuse_outputs)
    self._output_cache = {}
    self._slab_pool = {}   # (batch, bytes) -> page-locked numpy slabs (output='numpy')
    self._slab_plans = {}
    self._slab_at = _native.Batch()
    self._slab_needed = ctypes.c_size_t(0)
    self._lib = _native.lib()
    # add() fast path: Atari layout and plain scalars -> one native call.
    self._fast_add = (
        tuple(action_shape) == () and np.dtype(action_dtype) == np.int32 and
        np.dtype(reward_dtype) == np.float32 and
        np.dtype(terminal_dtype) == np.uint8 and not self._extra_storage_types)
    self._fast_obs = (tuple(observation_shape), np.dtype(observation_dtype))
    self._create_storage()
    # circular_replay_buffer.py:181-183
    self._cumulative_discount_vector = np.array(
        [math.pow(self._gamma, n) for n in range(update_horizon)],
        dtype=np.float32)

  # -- storage ------------------------------------------------------------------
  def _create_storage(self):
    """Allocates the HBM arrays (the reference's numpy `_store`, CRB:185-192)."""
    cfg = _native.Config()
    cfg.capacity = self._replay_capacity
    cfg.stack_size = self._stack_size
    cfg.update_horizon = self._update_horizon
    cfg.gamma = self._gamma
    cfg.max_sample_attempts = self._max_sample_attempts
    cfg.prioritized = self._PRIORITIZED
    obs_dtype = np.dtype(self._observation_dtype)
    cfg.obs_bytes = int(np.prod(self._observation_shape, dtype=np.int64) *
                        obs_dtype.itemsize)
    cfg.obs_itemsize = obs_dtype.itemsize
    cfg.action_bytes = int(np.prod(self._action_shape, dtype=np.int64) *
                           np.dtype(self._action_dtype).itemsize)
    cfg.reward_itemsize = np.dtype(self._reward_dtype).itemsize
    cfg.terminal_itemsize = np.dtype(self._terminal_dtype).itemsize
    if len(self._extra_storage_types) > _native.MAX_EXTRAS:
      raise NotImplementedError('at most {} extra storage types'.format(
          _native.MAX_EXTRAS))
    cfg.num_extras = len(self._extra_storage_types)
    for k, e in enumerate(self._extra_storage_types):
      cfg.extra_bytes[k] = int(np.prod(tuple(e.shape), dtype=np.int64) *
                               np.dtype(e.type).itemsize)
    cfg.add_queue_rows = 0
    handle = ctypes.c_void_p()
    status = self._lib.b2r_create(ctypes.byref(cfg), ctypes.byref(handle))
    if status == _native.ERR_UNSUPPORTED:
      raise NotImplementedError(_native.last_error())
    _native.check(status)
    self._h = handle
    self._store = _StoreView(self)
    self._columns = {e.name: k
                     for k, e in enumerate(self.get_storage_signature())}

  def __del__(self):
    if getattr(self, '_h', None):
      self._lib.b2r_destroy(self._h)
      self._h = None

  @staticmethod
  def _stream():
    return _native.current_stream()

  def _read_column(self, name, row0=0, nrows=None):
    element = self.get_storage_signature()[self._columns[name]]
    nrows = self._replay_capacity - row0 if nrows is None else nrows
    out = np.empty([nrows] + list(element.shape), dtype=element.type)
    _native.check(self._lib.b2r_store_read(
        self._h, self._columns[name], row0, nrows, _native.ptr(out),
        self._stream()))
    return out

  def _write_column(self, name, array):
    element = self.get_storage_signature()[self._columns[name]]
    array = np.ascontiguousarray(array, dtype=element.type)
    want = (self._replay_capacity,) + tuple(element.shape)
    if array.shape != want:
      raise ValueError('store {} has shape {}, expected {}'.format(
          name, array.shape, want))
    _native.check(self._lib.b2r_store_write(
        self._h, self._columns[name], 0, self._replay_capacity,
        _native.ptr(array), self._stream()))

  # -- signatures (CRB:194-223, 560-591) -------------------------------------------
  def get_add_args_signature(self):
    return self.get_storage_signature()

  def get_storage_signature(self):
    cached = self.__dict__.get('_storage_signature_cache')
    if cached is not None:
      return list(cached)
    storage_elements = [
        ReplayElement('observation', self._observation_shape,
                      self._observation_dtype),
        ReplayElement('action', self._action_shape, self._action_dtype),
        ReplayElement('reward', self._reward_shape, self._reward_dtype),
        ReplayElement('terminal', (), self._terminal_dtype)
    ]
    for extra_replay_element in self._extra_storage_types:
      storage_elements.append(extra_replay_element)
    self._storage_signature_cache = tuple(storage_elements)
    return storage_elements

  def get_transition_elements(self, batch_size=None):
    batch_size = self._batch_size if batch_size is None else batch_size
    transition_elements = [
        ReplayElement('state', (batch_size,) + self._state_shape,
                      self._observation_dtype),
        ReplayElement('action', (batch_size,) + self._action_shape,
                      self._action_dtype),
        ReplayElement('reward', (batch_size,) + self._reward_shape,
                      self._reward_dtype),
        ReplayElement('next_state', (batch_size,) + self._state_shape,
                      self._observation_dtype),
        ReplayElement('next_action', (batch_size,) + self._action_shape,
                      self._action_dtype),
        ReplayElement('next_reward', (batch_size,) + self._reward_shape,
                      self._reward_dtype),
        ReplayElement('terminal', (batch_size,), self._terminal_dtype),
        ReplayElement('indices', (batch_size,), np.int32)
    ]
    for element in self._extra_storage_types:
      transition_elements.append(
          ReplayElement(element.name, (batch_size,) + tuple(element.shape),
                        element.type))
    return transition_elements

  # -- bookkeeping attributes -------------------------------------------------------
  @property
  def add_count(self):
    return np.array(self._lib.b2r_add_count(self._h))

  @add_count.setter
  def add_count(self, value):
    self._set_state(int(value), self.invalid_range)

  @property
  def invalid_range(self):
    out = np.zeros(128, dtype=np.int64)
    n = ctypes.c_int32()
    _native.check(self._lib.b2r_get_invalid_range(self._h, _native.ptr(out),
                                                  ctypes.byref(n)))
    return out[:n.value].copy()

  @invalid_range.setter
  def invalid_range(self, value):
    self._set_state(int(self.add_count), value)

  def _flush(self):
    """Applies the staged adds (and with them the validity context in HBM)."""
    _native.check(self._lib.b2r_flush(self._h, self._stream()))

  def _set_state(self, add_count, invalid):
    invalid = np.ascontiguousarray(np.asarray(invalid).astype(np.int64))
    self._flush()
    _native.check(self._lib.b2r_set_state(self._h, add_count,
                                          _native.ptr(invalid), len(invalid)))

  def is_empty(self):
    return self.add_count == 0

  def is_full(self):
    return self.add_count >= self._replay_capacity

  def cursor(self):
    return np.int64(self._lib.b2r_cursor(self._h))

  # -- add (CRB:234-324) ---------------------------------------------------------------
  def _check_args_length(self, *args):
    if len(args) != len(self.get_add_args_signature()):
      raise ValueError('Add expects {} elements, received {}'.format(
          len(self.get_add_args_signature()), len(args)))

  def _check_add_types(self, *args):
    self._check_args_length(*args)
    for arg_element, store_element in zip(args, self.get_add_args_signature()):
      if isinstance(arg_element, np.ndarray):
        arg_shape = arg_element.shape
      elif isinstance(arg_element, (tuple, list)):
        arg_shape = np.array(arg_element).shape
      else:
        arg_shape = tuple()
      store_element_shape = tuple(store_element.shape)
      if arg_shape != store_element_shape:
        raise ValueError('arg has shape {}, expected {}'.format(
            arg_shape, store_element_shape))

  def add(self, observation, action, reward, terminal, *args):
    """Adds a transition; pads episode starts with stack_size-1 zero transitions.

    Values are cast to the storage dtypes with numpy assignment semantics
    (CRB:280-282) and staged; one kernel writes them to HBM at the next read.
    """
    if not args and self._try_fast_add(observation, action, reward, terminal, 0.0,
                                       _native.PRIORITY_EXPLICIT):
      return
    self._check_add_types(observation, action, reward, terminal, *args)
    self._native_add((observation, action, reward, terminal) + tuple(args), 0.0,
                     _native.PRIORITY_EXPLICIT)

  def add_batch(self, observations, actions, rewards, terminals, *args):
    """n consecutive `add`s of one trajectory stream in ONE native call (b2r_add_batch).

    Every argument is an array whose leading axis counts the steps; values are cast to
    the storage dtypes as `add` casts them (CRB:280-282).  Same buffer state afterwards
    as the loop `for k: add(observations[k], ...)` — zero padding after terminals,
    invalid_range — with the rows staged together.  (No counterpart in the reference,
    whose agents add one step at a time: DQ:444-458, RA:307-337.)"""
    self._native_add_batch((observations, actions, rewards, terminals) + tuple(args),
                           None, _native.PRIORITY_EXPLICIT)

  def _native_add_batch(self, columns, priorities, priority_mode):
    signature = self.get_storage_signature()
    if len(columns) != len(signature):
      raise ValueError('Add expects {} elements, received {}'.format(
          len(signature), len(columns)))
    n = len(columns[0])
    arrays = []
    for values, element in zip(columns, signature):
      array = np.ascontiguousarray(values, dtype=element.type)
      if array.shape != (n,) + tuple(element.shape):
        raise ValueError('arg {} has shape {}, expected {}'.format(
            element.name, array.shape, (n,) + tuple(element.shape)))
      arrays.append(array)
    extras = (ctypes.c_void_p * _native.MAX_EXTRAS)()
    for k, array in enumerate(arrays[4:]):
      extras[k] = array.ctypes.data
    prio_ptr = None
    if priorities is not None:
      priorities = np.ascontiguousarray(priorities, dtype=np.float64)
      if priorities.shape != (n,):
        raise ValueError('priorities has shape {}, expected {}'.format(
            priorities.shape, (n,)))
      prio_ptr = priorities.ctypes.data
    added = ctypes.c_int64(0)
    status = self._lib.b2r_add_batch(
        self._h, n, arrays[0].ctypes.data, arrays[1].ctypes.data, arrays[2].ctypes.data,
        arrays[3].ctypes.data, extras, prio_ptr, priority_mode, ctypes.byref(added),
        self._stream())
    if status == _native.ERR_NEGATIVE_PRIORITY:
      raise ValueError(_native.last_error())
    _native.check(status)

  def _try_fast_add(self, observation, action, reward, terminal, priority, mode):
    """One native call when the arguments are what an Atari agent passes: a
    C-contiguous observation of the storage dtype and plain scalars (whose
    int()/float() conversion equals numpy's assignment cast, CRB:280-282).
    Returns False when the general path (and its shape errors) must run."""
    if not self._fast_add:
      return False
    if (type(observation) is not np.ndarray or
        observation.shape != self._fast_obs[0] or
        observation.dtype != self._fast_obs[1] or
        not observation.flags.c_contiguous):
      return False
    if (type(action) not in _PLAIN_SCALARS or type(reward) not in _PLAIN_SCALARS
        or type(terminal) not in _PLAIN_SCALARS):
      return False
    terminal = int(terminal)
    if terminal < 0 or terminal > 255 or not -2147483648 <= action <= 2147483647:
      return False
    # No stream look-up per add: the call never launches; when the staging queue
    # is full it says so, and the flush (which launches) gets the current stream.
    # The call goes through the CPython shim (csrc/fastcall.c): b2r_add_atari with
    # the observation taken through the buffer protocol.
    add_atari = self.__dict__.get('_fast_add_fn')
    if add_atari is None:
      add_atari = self._fast_add_fn = _native.fast().add_atari
      self._h_int = self._h.value
      self._obs_bytes = int(np.prod(self._fast_obs[0], dtype=np.int64))
    action = int(action)
    status = add_atari(self._h_int, self._obs_bytes, observation, action, reward,
                       terminal, priority, mode, -1)
    if status == _native.QUEUE_FULL:
      _native.check(self._lib.b2r_flush(self._h, self._stream()))
      status = add_atari(self._h_int, self._obs_bytes, observation, action, reward,
                         terminal, priority, mode, -1)
    if status == -1:
      return False
    if status == _native.ERR_NEGATIVE_PRIORITY:
      raise ValueError(_native.last_error())
    if status:
      _native.check(status)
    return True

  def _native_add(self, values, priority, priority_mode):
    # One preallocated, correctly typed row buffer per storage element: numpy
    # assignment performs the reference's cast (CRB:280-282) without allocating.
    rows = self.__dict__.get('_row_buffers')
    if rows is None:
      rows = [np.zeros(tuple(e.shape), dtype=e.type)
              for e in self.get_storage_signature()]
      self._row_buffers = rows
      self._row_pointers = [r.ctypes.data for r in rows]
      self._extra_pointers = (ctypes.c_void_p * _native.MAX_EXTRAS)()
      for k, r in enumerate(rows[4:]):
        self._extra_pointers[k] = r.ctypes.data
    ptrs = list(self._row_pointers)
    obs = values[0]
    if (isinstance(obs, np.ndarray) and obs.dtype == rows[0].dtype and
        obs.flags['C_CONTIGUOUS']):
      ptrs[0] = obs.ctypes.data  # staged by the library before add() returns
    else:
      rows[0][...] = obs
    for k in range(1, len(rows)):
      rows[k][...] = values[k]
    status = self._lib.b2r_add(
        self._h, ptrs[0], ptrs[1], ptrs[2], ptrs[3], self._extra_pointers,
        priority, priority_mode, self._stream())
    if status == _native.ERR_NEGATIVE_PRIORITY:
      raise ValueError(_native.last_error())
    _native.check(status)

  # -- reads (CRB:338-414) -----------------------------------------------------------------
  def _assert_range(self, start_index, end_index):
    assert end_index > start_index, 'end_index must be larger than start_index'
    assert end_index >= 0
    assert start_index < self._replay_capacity
    if not self.is_full():
      assert end_index <= self.cursor(), (
          'Index {} has not been added.'.format(start_index))

  def get_range(self, array, start_index, end_index):
    """Rows [start_index, end_index) of a host array, wrapping around (CRB:338-366)."""
    self._assert_range(start_index, end_index)
    if start_index % self._replay_capacity < end_index % self._replay_capacity:
      return_array = array[start_index:end_index, ...]
    else:
      indices = [(start_index + i) % self._replay_capacity
                 for i in range(end_index - start_index)]
      return_array = array[indices, ...]
    return return_array

  def get_observation_stack(self, index):
    """(obs..., stack) stack ending at `index`, built by the gather kernel."""
    self._assert_range(index - self._stack_size + 1, index + 1)
    out = np.empty((1,) + self._state_shape, dtype=self._observation_dtype)
    batch = _native.Batch()
    batch.state = out.ctypes.data
    idx = np.array([index % self._replay_capacity], dtype=np.int32)
    _native.check(self._lib.b2r_gather(self._h, 1, _native.ptr(idx),
                                       ctypes.byref(batch), self._stream()))
    return out[0]

  def get_terminal_stack(self, index):
    start, end = index - self._stack_size + 1, index + 1
    self._assert_range(start, end)
    rows = [(start + i) % self._replay_capacity for i in range(end - start)]
    return np.array([self._read_column('terminal', r, 1)[0] for r in rows],
                    dtype=self._terminal_dtype)

  def is_valid_transition(self, index):
    """is_valid_transition (CRB:381-414), evaluated by the device routine that
    the sampling kernels use."""
    idx = np.array([index], dtype=np.int64)
    out = np.zeros(1, dtype=np.uint8)
    _native.check(self._lib.b2r_valid_mask(self._h, 1, _native.ptr(idx),
                                           _native.ptr(out), self._stream()))
    return bool(out[0])

  # -- sampling (CRB:436-558) ------------------------------------------------------------------
  def _next_offset(self):
    self._draw_counter += 1
    return self._draw_counter

  def sample_index_batch(self, batch_size):
    """Valid indices sampled uniformly (CRB:436-477).

    rng='reference': consumes np.random.randint draws exactly like the reference
    and returns a list of ints.  rng='device': returns an int32 CUDA tensor.
    """
    lo, hi = ctypes.c_int64(), ctypes.c_int64()
    status = self._lib.b2r_uniform_bounds(self._h, ctypes.byref(lo),
                                          ctypes.byref(hi))
    if status == _native.ERR_TOO_FEW_TRANSITIONS:
      raise RuntimeError('Cannot sample a batch with fewer than stack size '
                         '({}) + update_horizon ({}) transitions.'.
                         format(self._stack_size, self._update_horizon))
    _native.check(status)
    if self._rng == 'device':
      torch = _torch()
      out = torch.empty(batch_size, dtype=torch.int32, device='cuda')
      _native.check(self._lib.b2r_sample_indices_device(
          self._h, batch_size, self._seed, self._next_offset(), out.data_ptr(),
          self._stream()))
      return out
    min_id, max_id = lo.value, hi.value
    out = np.zeros(batch_size, dtype=np.int32)
    accepted, rejected, used = (ctypes.c_int32(0), ctypes.c_int32(0),
                                ctypes.c_int32(0))
    while (accepted.value < batch_size and
           rejected.value < self._max_sample_attempts):
      window = max(64, 2 * (batch_size - accepted.value))
      state = np.random.get_state()
      candidates = np.ascontiguousarray(
          np.random.randint(min_id, max_id, size=window), dtype=np.int64)
      _native.check(self._lib.b2r_sample_indices_uniform(
          self._h, batch_size, window, _native.ptr(candidates),
          _native.ptr(out), ctypes.byref(accepted), ctypes.byref(rejected),
          ctypes.byref(used), self._stream()))
      if used.value < window:
        # The reference stopped mid-window: rewind and consume what it consumed.
        np.random.set_state(state)
        if used.value:
          np.random.randint(min_id, max_id, size=used.value)
    if accepted.value != batch_size:
      raise RuntimeError(
          'Max sample attempts: Tried {} times but only sampled {}'
          ' valid indices. Batch size is {}'.
          format(self._max_sample_attempts, accepted.value, batch_size))
    return [int(i) for i in out]

  def _alloc_outputs(self, batch_size, on_device):
    if self._reuse_outputs and (batch_size, on_device) in self._output_cache:
      return self._output_cache[(batch_size, on_device)]
    elements = self.get_transition_elements(batch_size)
    if on_device:
      torch = _torch()
      arrays = []
      for e in elements:
        dtype = _torch_dtype(e.type)
        if dtype is None:
          raise NotImplementedError(
              'no torch dtype for {}; use output="numpy"'.format(e.type))
        arrays.append(torch.empty(tuple(e.shape), dtype=dtype, device='cuda'))
      pointers = [a.data_ptr() for a in arrays]
    else:
      arrays = [np.empty(e.shape, dtype=e.type) for e in elements]
      pointers = [a.ctypes.data for a in arrays]
    batch = _native.Batch()
    extra = 0
    for e, p in zip(elements, pointers):
      if e.name in ('state', 'action', 'reward', 'next_state', 'next_action',
                    'next_reward', 'terminal', 'indices',
                    'sampling_probabilities'):
        setattr(batch, e.name, p)
      else:
        batch.extras[extra] = p
        extra += 1
    if self._reuse_outputs:
      self._output_cache[(batch_size, on_device)] = (elements, arrays, batch)
    return elements, arrays, batch

  def _check_explicit_indices(self, indices):
    """The get_range assertions an explicit index would trip (CRB:351-356)."""
    full = bool(self.is_full())
    cursor = int(self.cursor())
    for i in indices:
      i = int(i)
      if i < 0 or i >= self._replay_capacity:
        raise IndexError('index {} is out of bounds for capacity {}'.format(
            i, self._replay_capacity))
      if not full:
        assert i + 1 <= cursor, 'Index {} has not been added.'.format(
            i - self._stack_size + 1)

  def _pinned_slab(self, batch_size, nbytes):
    """A page-locked slab of `nbytes` that no array handed out earlier still views.

    The reference returns FRESH arrays on every call (CRB:416-434, 516): a caller may
    keep as many batches as it likes.  The slabs of a pool are therefore reused only
    once every numpy view over them has been dropped (their reference count says so);
    while views are alive the pool grows.  Page-locked memory is what lets the whole
    batch travel in ONE copy at PCIe speed; allocating it is slow, hence the pool."""
    pool = self._slab_pool.setdefault((batch_size, nbytes), [])
    for slab in pool:
      if sys.getrefcount(slab) == 3:  # the pool's list, `slab`, getrefcount's argument
        return slab
    torch = _torch()
    keep = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    slab = keep.numpy()  # (holds `keep` alive as its base)
    pool.append(slab)
    return slab

  def _host_batch_plan(self, batch_size):
    """Per batch size, once: which columns are wanted, how large the slab is and where
    each returned array sits in it."""
    plan = self._slab_plans.get(batch_size)
    if plan is not None:
      return plan
    elements = self.get_transition_elements(batch_size)
    want = _native.Batch()
    fields = []
    extra = 0
    for e in elements:
      if hasattr(want, e.name) and e.name != 'extras':
        setattr(want, e.name, 1)
        fields.append(e.name)
      else:
        want.extras[extra] = 1
        fields.append(extra)
        extra += 1
    needed = ctypes.c_size_t(0)
    at = _native.Batch()  # with a NULL slab the pointers come back as offsets
    _native.check(self._lib.b2r_gather_slab(
        self._h, batch_size, None, 0, ctypes.byref(want), None, 0, ctypes.byref(at),
        ctypes.byref(needed), self._stream()))
    views = []
    for e, f in zip(elements, fields):
      offset = int((at.extras[f] if isinstance(f, int) else getattr(at, f)) or 0)
      count = int(np.prod(e.shape, dtype=np.int64)) * np.dtype(e.type).itemsize
      views.append((offset, offset + count, np.dtype(e.type), tuple(e.shape)))
    plan = (want, int(needed.value), views)
    self._slab_plans[batch_size] = plan
    return plan

  def _gather_to_host(self, batch_size, indices, device_indices):
    """output='numpy': the batch as host arrays (the reference's return convention),
    built on the device and shipped in one copy into a page-locked slab; the arrays are
    views over it (b2r_gather_slab)."""
    want, nbytes, views = self._host_batch_plan(batch_size)
    slab = self._pinned_slab(batch_size, nbytes)
    if device_indices is not None:
      idx_ptr, on_device = device_indices.data_ptr(), 1
    else:
      host_idx = np.ascontiguousarray(indices, dtype=np.int32)
      idx_ptr, on_device = host_idx.ctypes.data, 0
    _native.check(self._lib.b2r_gather_slab(
        self._h, batch_size, idx_ptr, on_device, ctypes.byref(want), slab.ctypes.data,
        nbytes, ctypes.byref(self._slab_at), ctypes.byref(self._slab_needed),
        self._stream()))
    return tuple(slab[lo:hi].view(dtype).reshape(shape)
                 for lo, hi, dtype, shape in views)

  def sample_transition_batch(self, batch_size=None, indices=None):
    """Batch of transitions in get_transition_elements() order (CRB:479-558).

    One fused kernel builds stacks, n-step returns, terminals and next_* for the
    whole batch.  With output='torch' the result stays in HBM.
    """
    if batch_size is None:
      batch_size = self._batch_size
    on_device = self._output == 'torch'
    torch_indices = None
    if indices is None:
      indices = self.sample_index_batch(batch_size)
      if self._rng == 'device':
        torch_indices = indices
    else:
      self._check_explicit_indices(indices)
    assert len(indices) == batch_size
    if on_device:
      _, arrays, batch = self._alloc_outputs(batch_size, on_device)
      torch = _torch()
      if torch_indices is None:
        torch_indices = torch.as_tensor(
            np.asarray(indices, dtype=np.int32), device='cuda')
      _native.check(self._lib.b2r_gather_device(
          self._h, batch_size, torch_indices.data_ptr(), ctypes.byref(batch),
          self._stream()))
    else:
      return self._gather_to_host(batch_size, indices, torch_indices)
    return tuple(arrays)

  # -- checkpointing (CRB:593-687) -----------------------------------------------------------
  def _generate_filename(self, checkpoint_dir, name, suffix):
    return os.path.join(checkpoint_dir, '{}_ckpt.{}.gz'.format(name, suffix))

  def _return_checkpointable_elements(self):
    """Public attributes + every `_store` array, keyed like the reference."""
    checkpointable_elements = {}
    for name in self._store.keys():
      checkpointable_elements[STORE_FILENAME_PREFIX + name] = None
    checkpointable_elements['add_count'] = None
    checkpointable_elements['invalid_range'] = None
    for member_name in self.__dict__:
      if not member_name.startswith('_'):
        checkpointable_elements[member_name] = None
    return checkpointable_elements

  def save(self, checkpoint_dir, iteration_number):
    """Writes one gzip file per attribute / store array, reference layout.

    Store arrays are compressed on the device into blocked gzip (see
    `_save_store_column`); any gzip reader, the reference's `load` included, reads them
    as the `np.save` stream of the array."""
    if not os.path.exists(checkpoint_dir):
      return
    for attr in self._return_checkpointable_elements():
      filename = self._generate_filename(checkpoint_dir, attr, iteration_number)
      if attr.startswith(STORE_FILENAME_PREFIX):
        self._save_store_column(attr[len(STORE_FILENAME_PREFIX):], filename)
      else:
        value = getattr(self, attr)
        with open(filename, 'wb') as f:
          with gzip.GzipFile(fileobj=f) as outfile:
            if isinstance(value, np.ndarray):
              np.save(outfile, value, allow_pickle=False)
            else:
              self._pickle_attribute(attr, value, outfile)
      stale_iteration_number = iteration_number - CHECKPOINT_DURATION
      if stale_iteration_number >= 0:
        stale_filename = self._generate_filename(checkpoint_dir, attr,
                                                 stale_iteration_number)
        try:
          os.remove(stale_filename)
        except FileNotFoundError:
          pass

  def load(self, checkpoint_dir, suffix):
    """Restores from files written by `save` (or by the reference's save).

    A store file in the blocked layout `save` writes, whose .npy header matches the
    buffer's storage shape and dtype, is inflated on the device; any other gzip file
    takes the host path.  Every file is read (blocked ones: inflated and checked on the
    device without writing) before any state changes, so a load that raises leaves
    the buffer as it was."""
    self._load_apply(self._load_prepare(checkpoint_dir, suffix))

  def _load_prepare(self, checkpoint_dir, suffix):
    """The reading half of `load`: every file read, blocked store files verified on the
    device, nothing changed.  Returns what `_load_apply` writes.  A caller restoring
    several buffers as one checkpoint prepares all of them before applying any."""
    save_elements = self._return_checkpointable_elements()
    for attr in save_elements:
      filename = self._generate_filename(checkpoint_dir, attr, suffix)
      if not os.path.exists(filename):
        raise FileNotFoundError('Missing file: {}'.format(filename))
    loaded = {}
    blocked = {}
    for attr in save_elements:
      filename = self._generate_filename(checkpoint_dir, attr, suffix)
      if attr.startswith(STORE_FILENAME_PREFIX):
        name = attr[len(STORE_FILENAME_PREFIX):]
        offset = self._blocked_data_offset(name, filename)
        if offset is not None:
          self._load_store_column(name, filename, offset, verify_only=True)
          blocked[name] = (filename, offset)
          continue
      with open(filename, 'rb') as f:
        with gzip.GzipFile(fileobj=f) as infile:
          current = getattr(self, attr) if not attr.startswith(
              STORE_FILENAME_PREFIX) else None
          if attr.startswith(STORE_FILENAME_PREFIX) or isinstance(
              current, np.ndarray):
            loaded[attr] = np.load(infile, allow_pickle=False)
          else:
            loaded[attr] = self._unpickle_attribute(attr, infile)
    return loaded, blocked

  def _load_apply(self, prepared):
    """The writing half of `load`, on what `_load_prepare` returned."""
    loaded, blocked = prepared
    for attr, value in loaded.items():
      if attr.startswith(STORE_FILENAME_PREFIX):
        self._store[attr[len(STORE_FILENAME_PREFIX):]] = value
    for name, (filename, offset) in blocked.items():
      self._load_store_column(name, filename, offset, verify_only=False)
    self._set_state(int(loaded['add_count']), loaded['invalid_range'])
    for attr, value in loaded.items():
      if attr.startswith(STORE_FILENAME_PREFIX) or attr in ('add_count',
                                                            'invalid_range'):
        continue
      self._restore_attribute(attr, value)

  # -- sampler state (b2r_sampler_state_get / _set) ------------------------------------------
  def sampler_state(self):
    """What decides the next draws besides the stored transitions: the device's draw
    counters (Philox samplers, sharded prioritized sampler) and the host's draw counter
    of rng='device' sampling.  A dict of plain ints; `set_sampler_state` takes it back."""
    words = np.zeros(_native.SAMPLER_STATE_WORDS, dtype=np.uint64)
    _native.check(self._lib.b2r_sampler_state_get(
        self._h, _native.SAMPLER_STATE_VERSION, _native.ptr(words), len(words),
        self._stream()))
    _torch().cuda.current_stream().synchronize()
    return {'version': _native.SAMPLER_STATE_VERSION,
            'words': [int(w) for w in words], 'draw_counter': int(self._draw_counter)}

  def set_sampler_state(self, state):
    """Restores what `sampler_state` returned (stream-ordered on the device)."""
    words = np.ascontiguousarray(state['words'], dtype=np.uint64)
    _native.check(self._lib.b2r_sampler_state_set(
        self._h, int(state['version']), _native.ptr(words), len(words), self._stream()))
    self._draw_counter = int(state['draw_counter'])

  # -- blocked gzip store files (csrc/ckpt.cu) ----------------------------------------------
  def _npy_header(self, name):
    """The bytes `np.save(f, _store[name], allow_pickle=False)` writes before the data."""
    element = self.get_storage_signature()[self._columns[name]]
    return npy_header((self._replay_capacity,) + tuple(element.shape), element.type)

  def _save_store_column(self, name, filename):
    """Member 0 (the .npy header) from the host, members 1.. from the device."""
    fd = os.open(filename, os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o666)
    try:
      _write_all(fd, bgzf_member(self._npy_header(name)))
      written = ctypes.c_int64(0)
      _native.check(self._lib.b2r_ckpt_save_column(
          self._h, self._columns[name], fd, 0, ctypes.byref(written), self._stream()))
    finally:
      os.close(fd)

  def _blocked_data_offset(self, name, filename):
    """Where member 1 starts when `filename` is a blocked file of store `name` (member 0
    a BGZF member holding exactly this buffer's .npy header for it), else None."""
    with open(filename, 'rb') as f:
      head = f.read(BGZF_HEADER_BYTES)
      if (len(head) < BGZF_HEADER_BYTES or
          head[:BGZF_HEADER_BYTES - 2] != _BGZF_PREFIX[:BGZF_HEADER_BYTES - 2]):
        return None
      size = struct.unpack('<H', head[-2:])[0] + 1
      rest = f.read(size - BGZF_HEADER_BYTES)
    if size < BGZF_HEADER_BYTES + 8 or len(rest) != size - BGZF_HEADER_BYTES:
      return None
    inflater = zlib.decompressobj(-15)
    try:
      payload = inflater.decompress(rest[:-8])
    except zlib.error:
      return None
    crc, isize = struct.unpack('<II', rest[-8:])
    if (not inflater.eof or inflater.unused_data or crc != zlib.crc32(payload) or
        isize != len(payload) or payload != self._npy_header(name)):
      return None
    return size

  def _load_store_column(self, name, filename, offset, verify_only):
    fd = os.open(filename, os.O_RDONLY)
    try:
      status = self._lib.b2r_ckpt_load_column(self._h, self._columns[name], fd, offset,
                                              1 if verify_only else 0, self._stream())
    finally:
      os.close(fd)
    if status == _native.ERR_INVALID_ARGUMENT:
      raise gzip.BadGzipFile('{}: {}'.format(filename, _native.last_error()))
    _native.check(status)

  def _restore_attribute(self, attr, value):
    setattr(self, attr, value)

  def _pickle_attribute(self, attr, value, outfile):
    del attr
    pickle.dump(value, outfile)

  def _unpickle_attribute(self, attr, infile):
    del attr
    return pickle.load(infile)


class WrappedReplayBuffer(object):
  """The reference's graph-side wrapper (CRB:692-915) without TensorFlow.

  Where the reference exposes tf.py_func tensors, this exposes device tensors:
  every call to `sample()` refreshes `.transition` (an OrderedDict keyed like the
  reference's) and the `.states/.actions/...` attributes with a batch that never
  left HBM.
  """

  def __init__(self,
               observation_shape,
               stack_size,
               use_staging=True,
               replay_capacity=1000000,
               batch_size=32,
               update_horizon=1,
               gamma=0.99,
               wrapped_memory=None,
               max_sample_attempts=1000,
               extra_storage_types=None,
               observation_dtype=np.uint8,
               terminal_dtype=np.uint8,
               action_shape=(),
               action_dtype=np.int32,
               reward_shape=(),
               reward_dtype=np.float32):
    if replay_capacity < update_horizon + 1:
      raise ValueError(
          'Update horizon ({}) should be significantly smaller '
          'than replay capacity ({}).'.format(update_horizon, replay_capacity))
    if not update_horizon >= 1:
      raise ValueError('Update horizon must be positive.')
    if not 0.0 <= gamma <= 1.0:
      raise ValueError('Discount factor (gamma) must be in [0, 1].')
    self.batch_size = batch_size
    del use_staging  # the batch is produced on the device; nothing to prefetch
    if wrapped_memory is not None:
      self.memory = wrapped_memory
    else:
      self.memory = OutOfGraphReplayBuffer(
          observation_shape, stack_size, replay_capacity, batch_size,
          update_horizon, gamma, max_sample_attempts,
          observation_dtype=observation_dtype, terminal_dtype=terminal_dtype,
          extra_storage_types=extra_storage_types, action_shape=action_shape,
          action_dtype=action_dtype, reward_shape=reward_shape,
          reward_dtype=reward_dtype, output='torch')
    self.transition = None

  def add(self, observation, action, reward, terminal, *args):
    self.memory.add(observation, action, reward, terminal, *args)

  def sample(self):
    """Samples a fresh batch (what a sess.run on `.transition` did, CRB:814-827)."""
    tensors = self.memory.sample_transition_batch()
    self.unpack_transition(tensors, self.memory.get_transition_elements())
    return self.transition

  def unpack_transition(self, transition_tensors, transition_type):
    self.transition = collections.OrderedDict()
    for element, element_type in zip(transition_tensors, transition_type):
      self.transition[element_type.name] = element
    self.states = self.transition['state']
    self.actions = self.transition['action']
    self.rewards = self.transition['reward']
    self.next_states = self.transition['next_state']
    self.next_actions = self.transition['next_action']
    self.next_rewards = self.transition['next_reward']
    self.terminals = self.transition['terminal']
    self.indices = self.transition['indices']

  def save(self, checkpoint_dir, iteration_number):
    self.memory.save(checkpoint_dir, iteration_number)

  def load(self, checkpoint_dir, suffix):
    self.memory.load(checkpoint_dir, suffix)
