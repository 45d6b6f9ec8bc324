"""ctypes binding of libb200replay.so (the C ABI declared in include/b200_replay.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if
there is no CUDA device every create call raises.
"""
import ctypes
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
# B2R_LIB lets the profiling scripts load an instrumented build of the same library.
LIB_PATH = os.environ.get('B2R_LIB') or os.path.join(_PKG, 'libb200replay.so')

MAX_EXTRAS = 8
OK = 0
ERR_INVALID_ARGUMENT = 1
ERR_CUDA = 2
ERR_NEGATIVE_PRIORITY = 3
ERR_EMPTY_TREE = 4
ERR_SAMPLE_ATTEMPTS = 5
ERR_TOO_FEW_TRANSITIONS = 6
ERR_INDEX_RANGE = 7
ERR_UNSUPPORTED = 8
ERR_EXCHANGE = 9
ERR_STALE_TOTAL = 11
QUEUE_FULL = 10
STREAM_NONE = ctypes.c_void_p(-1)
IPC_HANDLE_BYTES = 64
SAMPLER_STATE_VERSION, SAMPLER_STATE_WORDS = 1, 2
EXCHANGE_STATE_VERSION, EXCHANGE_STATE_WORDS = 1, 1

PRIORITY_EXPLICIT = 0
PRIORITY_MAX_RECORDED = 1

COL_OBSERVATION, COL_ACTION, COL_REWARD, COL_TERMINAL, COL_EXTRA0 = 0, 1, 2, 3, 4

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_int32 = ctypes.c_int32
c_int64 = ctypes.c_int64
c_uint64 = ctypes.c_uint64
c_double = ctypes.c_double
c_float = ctypes.c_float


class Config(ctypes.Structure):
  _fields_ = [
      ('capacity', c_int64),
      ('stack_size', c_int32),
      ('update_horizon', c_int32),
      ('gamma', c_double),
      ('max_sample_attempts', c_int32),
      ('prioritized', c_int32),
      ('obs_bytes', c_int64),
      ('obs_itemsize', c_int32),
      ('action_bytes', c_int32),
      ('reward_itemsize', c_int32),
      ('terminal_itemsize', c_int32),
      ('num_extras', c_int32),
      ('extra_bytes', c_int32 * MAX_EXTRAS),
      ('add_queue_rows', c_int32),
  ]


class Batch(ctypes.Structure):
  _fields_ = [
      ('state', c_void_p),
      ('action', c_void_p),
      ('reward', c_void_p),
      ('next_state', c_void_p),
      ('next_action', c_void_p),
      ('next_reward', c_void_p),
      ('terminal', c_void_p),
      ('indices', c_void_p),
      ('extras', c_void_p * MAX_EXTRAS),
      ('sampling_probabilities', c_void_p),
  ]


class C51Args(ctypes.Structure):
  _fields_ = [
      ('batch', c_int32),
      ('num_actions', c_int32),
      ('num_atoms', c_int32),
      ('cumulative_gamma', c_float),
      ('support', c_void_p),
      ('target_logits', c_void_p),
      ('online_logits', c_void_p),
      ('actions', c_void_p),
      ('rewards', c_void_p),
      ('terminals', c_void_p),
      ('sampling_probabilities', c_void_p),
      ('target', c_void_p),
      ('loss', c_void_p),
      ('priorities', c_void_p),
      ('weights', c_void_p),
      ('mean_weighted_loss', c_void_p),
      ('grad_logits', c_void_p),
      ('batch_count', c_void_p),
      ('min_probability', c_void_p),
  ]


class DqnArgs(ctypes.Structure):
  _fields_ = [
      ('batch', c_int32),
      ('num_actions', c_int32),
      ('cumulative_gamma', c_float),
      ('target_q', c_void_p),
      ('online_q', c_void_p),
      ('actions', c_void_p),
      ('rewards', c_void_p),
      ('terminals', c_void_p),
      ('loss', c_void_p),
      ('target', c_void_p),
      ('mean_loss', c_void_p),
      ('grad_q', c_void_p),
      ('batch_count', c_void_p),
  ]


class TrainerConfig(ctypes.Structure):
  _fields_ = [
      ('batch', c_int32),
      ('num_actions', c_int32),
      ('num_atoms', c_int32),
      ('vmax', c_float),
      ('cumulative_gamma', c_float),
      ('seed', c_uint64),
      ('pipeline_depth', c_int32),
      ('use_graph', c_int32),
      ('logit_rows', c_int32),
  ]


P = ctypes.POINTER
c_size_t = ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol of include/b200_replay.h.
class IqnArgs(ctypes.Structure):
  """b2r_iqn_args."""
  _fields_ = [
      ('batch', c_int32), ('num_actions', c_int32), ('num_tau_samples', c_int32),
      ('num_tau_prime_samples', c_int32), ('num_quantile_samples', c_int32),
      ('cumulative_gamma', ctypes.c_float), ('kappa', ctypes.c_float),
      ('reserved', c_int32),
      ('action_quantile_values', c_void_p), ('target_quantile_values', c_void_p),
      ('online_quantile_values', c_void_p), ('quantiles', c_void_p),
      ('actions', c_void_p), ('rewards', c_void_p), ('terminals', c_void_p),
      ('loss', c_void_p), ('mean_loss', c_void_p),
      ('grad_quantile_values', c_void_p), ('next_action', c_void_p),
  ]


SIGNATURES = {
    'b2r_last_error': (ctypes.c_char_p, []),
    'b2r_abi_version': (c_int, []),
    'b2r_launch_count': (c_int64, []),
    'b2r_tree_create': (c_int, [c_int64, P(c_void_p)]),
    'b2r_tree_destroy': (c_int, [c_void_p]),
    'b2r_tree_depth': (c_int, [c_void_p]),
    'b2r_tree_set': (c_int, [c_void_p, c_int64, c_void_p, c_void_p, P(c_int64),
                             c_void_p]),
    'b2r_tree_set_device': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                    c_void_p]),
    'b2r_tree_check': (c_int, [c_void_p, c_void_p]),
    'b2r_tree_get': (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    'b2r_tree_total': (c_int, [c_void_p, P(c_double), c_void_p]),
    'b2r_tree_max_recorded': (c_int, [c_void_p, P(c_double), c_void_p]),
    'b2r_tree_set_max_recorded': (c_int, [c_void_p, c_double, c_void_p]),
    'b2r_tree_sample': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                c_void_p]),
    'b2r_tree_read_level': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'b2r_tree_write_level': (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    'b2r_create': (c_int, [P(Config), P(c_void_p)]),
    'b2r_destroy': (c_int, [c_void_p]),
    'b2r_buffer_tree': (c_void_p, [c_void_p]),
    'b2r_add': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                        P(c_void_p), c_double, c_int, c_void_p]),
    'b2r_add_atari': (c_int, [c_void_p, c_void_p, c_int32, c_float,
                              ctypes.c_uint8, c_double, c_int, c_void_p]),
    'b2r_flush': (c_int, [c_void_p, c_void_p]),
    'b2r_add_count': (c_int64, [c_void_p]),
    'b2r_cursor': (c_int64, [c_void_p]),
    'b2r_get_invalid_range': (c_int, [c_void_p, c_void_p, P(c_int32)]),
    'b2r_set_state': (c_int, [c_void_p, c_int64, c_void_p, c_int32]),
    'b2r_valid_mask': (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    'b2r_uniform_bounds': (c_int, [c_void_p, P(c_int64), P(c_int64)]),
    'b2r_sample_indices_uniform': (c_int, [
        c_void_p, c_int32, c_int32, c_void_p, c_void_p, P(c_int32), P(c_int32),
        P(c_int32), c_void_p]),
    'b2r_sample_indices_prioritized': (c_int, [
        c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_void_p, P(c_int32),
        P(c_int32), c_void_p]),
    'b2r_sample_indices_device': (c_int, [c_void_p, c_int32, c_uint64, c_uint64,
                                          c_void_p, c_void_p]),
    'b2r_check': (c_int, [c_void_p, c_void_p]),
    'b2r_gather_device': (c_int, [c_void_p, c_int32, c_void_p, P(Batch),
                                  c_void_p]),
    'b2r_gather': (c_int, [c_void_p, c_int32, c_void_p, P(Batch), c_void_p]),
    'b2r_sample_transition_batch_device': (c_int, [
        c_void_p, c_int32, c_uint64, c_uint64, P(Batch), c_void_p]),
    'b2r_set_priority': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                 P(c_int64), c_void_p]),
    'b2r_set_priority_device': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                        c_void_p]),
    'b2r_get_priority': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                 c_void_p]),
    'b2r_get_priority_device': (c_int, [c_void_p, c_int64, c_void_p, c_void_p,
                                        c_void_p]),
    'b2r_store_read': (c_int, [c_void_p, c_int32, c_int64, c_int64, c_void_p,
                               c_void_p]),
    'b2r_store_write': (c_int, [c_void_p, c_int32, c_int64, c_int64, c_void_p,
                                c_void_p]),
    'b2r_store_device_ptr': (c_void_p, [c_void_p, c_int32]),
    'b2r_ckpt_save_column': (c_int, [c_void_p, c_int32, c_int32, c_int32, P(c_int64),
                                     c_void_p]),
    'b2r_ckpt_load_column': (c_int, [c_void_p, c_int32, c_int32, c_int64, c_int32,
                                     c_void_p]),
    'b2r_sampler_state_get': (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'b2r_sampler_state_set': (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'b2r_exchange_state_get': (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'b2r_exchange_state_set': (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    'b2r_sample_indices_sharded_device': (c_int, [
        c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32,
        c_void_p, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'b2r_gather_device_counted': (c_int, [c_void_p, c_int32, c_void_p, c_void_p,
                                          P(Batch), c_void_p]),
    'b2r_set_priority_device_counted': (c_int, [c_void_p, c_int64, c_void_p,
                                                c_void_p, c_void_p, c_void_p]),
    'b2r_copy_total_device': (c_int, [c_void_p, c_void_p, c_void_p]),
    'b2r_total_device_ptr': (c_void_p, [c_void_p]),
    'b2r_c51_project': (c_int, [c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    'b2r_c51_loss': (c_int, [P(C51Args), c_void_p]),
    'b2r_c51_loss_sharded': (c_int, [P(C51Args), c_void_p, c_int32, c_void_p]),
    'b2r_sample_transition_batch_sharded_device': (c_int, [
        c_void_p, c_void_p, c_int32, c_uint64, c_uint64, P(Batch), c_void_p, c_void_p,
        c_int32, c_void_p, c_void_p]),
    'b2r_dqn_loss': (c_int, [P(DqnArgs), c_void_p]),
    'b2r_dqn_loss_sharded': (c_int, [P(DqnArgs), c_int32, c_void_p]),
    'b2r_sample_transition_batch_uniform_sharded_device': (c_int, [
        c_void_p, c_void_p, c_int32, c_uint64, c_uint64, P(Batch), c_void_p, c_void_p,
        c_int32, c_void_p]),
    'b2r_exchange_publish_uniform_device': (c_int, [c_void_p, c_void_p, c_int32, c_uint64,
                                                     c_uint64, c_int32, c_void_p]),
    'b2r_train_step_device': (c_int, [c_void_p, c_int32, c_uint64, c_uint64,
                                      P(Batch), P(C51Args), c_void_p]),
    'b2r_stack_to_planes_device': (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int32,
                                           c_int32, c_void_p]),
    'b2r_add_batch': (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                              P(c_void_p), c_void_p, c_int, P(c_int64), c_void_p]),
    'b2r_gather_variant': (c_int32, [c_void_p, c_int32]),
    'b2r_gather_slab': (c_int, [c_void_p, c_int32, c_void_p, c_int32, P(Batch), c_void_p,
                                c_size_t, P(Batch), P(c_size_t), c_void_p]),
    'b2r_set_deferred_frames': (c_int, [c_void_p, c_int32]),
    'b2r_join_frames': (c_int, [c_void_p, c_void_p]),
    'b2r_train_step_sharded_device': (c_int, [
        c_void_p, c_void_p, c_int32, c_uint64, c_uint64, P(Batch), P(C51Args),
        c_void_p, c_void_p, c_int32, c_void_p]),
    'b2r_exchange_set_early_publish': (c_int, [c_void_p, c_int32]),
    'b2r_exchange_create': (c_int, [c_int32, c_int32, P(c_void_p)]),
    'b2r_exchange_destroy': (c_int, [c_void_p]),
    'b2r_exchange_local_handle': (c_int, [c_void_p, c_void_p]),
    'b2r_exchange_connect': (c_int, [c_void_p, c_void_p]),
    'b2r_exchange_connect_pointers': (c_int, [c_void_p, P(c_void_p)]),
    'b2r_exchange_mailbox': (c_void_p, [c_void_p]),
    'b2r_exchange_set_timeout': (c_int, [c_void_p, c_double]),
    'b2r_exchange_publish_device': (c_int, [c_void_p, c_void_p, c_void_p]),
    'b2r_sample_indices_sharded_p2p_device': (c_int, [
        c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p, c_uint64,
        c_uint64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'b2r_trainer_create': (c_int, [c_void_p, P(TrainerConfig), P(c_void_p)]),
    'b2r_trainer_destroy': (c_int, [c_void_p]),
    'b2r_trainer_step_host': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p,
                                      P(c_int64), c_void_p]),
    'b2r_trainer_set_exchange': (c_int, [c_void_p, c_void_p]),
    'b2r_trainer_last_rows': (c_int32, [c_void_p]),
    'b2r_trainer_drain': (c_int, [c_void_p, c_void_p, P(c_int64), c_void_p]),
    'b2r_trainer_views': (c_int, [c_void_p, P(Batch), P(C51Args)]),
    'b2r_iqn_loss': (c_int, [P(IqnArgs), c_void_p]),
    'b2r_iqn_loss_sharded': (c_int, [P(IqnArgs), c_void_p, c_int32, c_void_p]),
    'b2r_actor_create': (c_int, [c_int64, c_int32, c_int32, c_int32, P(c_void_p)]),
    'b2r_actor_destroy': (c_int, [c_void_p]),
    'b2r_actor_reset': (c_int, [c_void_p, c_void_p, c_void_p]),
    'b2r_actor_record': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None
# The version of include/b200_replay.h this table of signatures (and the ctypes mirrors of
# b2r_config, b2r_batch, b2r_c51_args, ...) was written against; b2r_abi_version() of the
# loaded binary must agree, so that a stale libb200replay.so is an error at load time and
# not a silent layout mismatch.  Bump both together.
ABI_VERSION = 3


class NativeError(RuntimeError):
  """A libb200replay call failed; `.code` is the b2r_status."""

  def __init__(self, code, message):
    super().__init__(message)
    self.code = code


def build():
  from dopamine_b200.csrc import build as _build  # pylint: disable=g-import-not-at-top
  return _build.build()


def lib():
  """Loads (building first if needed) the shared library. Never falls back."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      build()
    handle = ctypes.CDLL(LIB_PATH)
    handle.b2r_abi_version.restype = c_int
    found = handle.b2r_abi_version()
    if found != ABI_VERSION and os.environ.get('B2R_LIB') is None:
      # a binary built from older sources: rebuild once, then insist
      build()
      handle = ctypes.CDLL(LIB_PATH)
      handle.b2r_abi_version.restype = c_int
      found = handle.b2r_abi_version()
    if found != ABI_VERSION:
      raise NativeError(ERR_INVALID_ARGUMENT,
                        '{} implements ABI version {}, this package needs {}: rebuild it '
                        '(python -m dopamine_b200.csrc.build --force)'.format(
                            LIB_PATH, found, ABI_VERSION))
    for name, (restype, argtypes) in SIGNATURES.items():
      fn = getattr(handle, name)  # AttributeError if the ABI is incomplete
      fn.restype = restype
      fn.argtypes = argtypes
    _lib = handle
  return _lib


_fast = None


def fast():
  """The CPython fast-call shims (dopamine_b200/csrc/fastcall.c), bound to the same
  library; built on first use like the library itself."""
  global _fast
  if _fast is None:
    lib()
    from dopamine_b200.csrc import build as _build  # pylint: disable=g-import-not-at-top
    path = _build.fast_module_path()
    if not os.path.exists(path):
      _build.build_fast()
    import importlib.util  # pylint: disable=g-import-not-at-top
    spec = importlib.util.spec_from_file_location('_b2rfast', path)
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    module.bind(LIB_PATH)
    _fast = module
  return _fast


def last_error():
  return lib().b2r_last_error().decode('utf-8', 'replace')


def check(status):
  """Raises NativeError for a non-zero status."""
  if status != OK:
    raise NativeError(status, last_error())


def ptr(array):
  """Address of a C-contiguous numpy array."""
  assert array.flags['C_CONTIGUOUS']
  return array.ctypes.data


def current_stream():
  """torch's current CUDA stream as an integer handle (plumbing only)."""
  import torch  # pylint: disable=g-import-not-at-top
  return torch.cuda.current_stream().cuda_stream


def as_i64(values):
  return np.ascontiguousarray(values, dtype=np.int64)
