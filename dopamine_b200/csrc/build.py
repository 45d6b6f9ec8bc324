"""Builds libb200replay.so in-tree with nvcc for sm_100a (no JIT cache)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.dirname(HERE)
ROOT = os.path.dirname(PKG)
LIB = os.path.join(PKG, 'libb200replay.so')
SOURCES = ['common.cu', 'tree.cu', 'replay.cu', 'sample.cu', 'gather.cu',
           'c51.cu', 'dqn.cu', 'step.cu', 'exchange.cu', 'actor.cu', 'iqn.cu', 'ckpt.cu']
HEADERS = ['common.cuh', 'tree.cuh', 'replay.cuh', 'gather.cuh',
           os.path.join(ROOT, 'include', 'b200_replay.h')]

NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17',
    '-lineinfo', '-Xcompiler', '-fPIC',
    '-I', os.path.join(ROOT, 'include'), '-I', HERE,
]


def _nvcc():
  for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
    if cand and (os.path.isabs(cand) and os.path.exists(cand) or
                 not os.path.isabs(cand)):
      return cand
  raise RuntimeError('nvcc not found')


def _stale(target, deps):
  if not os.path.exists(target):
    return True
  t = os.path.getmtime(target)
  return any(os.path.getmtime(d) > t for d in deps)


TRACE_LIB = os.path.join(ROOT, 'profiles', 'micro', 'libb200replay_trace.so')
FAST_SRC = os.path.join(HERE, 'fastcall.c')


def fast_module_path():
  import sysconfig
  return os.path.join(PKG, '_b2rfast' + (sysconfig.get_config_var('EXT_SUFFIX') or '.so'))


def build_fast(force=False, verbose=False):
  """Compiles the CPython fast-call shims (gcc; no CUDA, no link to the library)."""
  import sysconfig
  target = fast_module_path()
  if not force and not _stale(target, [FAST_SRC, __file__]):
    return target
  cmd = ['gcc', '-O2', '-shared', '-fPIC', '-I', sysconfig.get_paths()['include'],
         FAST_SRC, '-o', target, '-ldl']
  if verbose:
    print(' '.join(cmd), file=sys.stderr)
  subprocess.check_call(cmd)
  return target


def build(force=False, verbose=False, extra_flags=(), trace=False):
  """Compiles every .cu for sm_100a and links the C-ABI shared library.

  trace=True builds the instrumented copy (-DB2R_TRACE: clock64 phase marks) used
  by profiles/micro/trace_step.py; it is never the library the package loads."""
  nvcc = _nvcc()
  obj_dir = os.path.join(HERE, '_obj_trace' if trace else '_obj')
  lib_path = TRACE_LIB if trace else LIB
  if trace:
    # clock64 phase marks; B2R_TRACE_GT=1 in the environment: %globaltimer marks
    # (one timeline for all kernels of the step)
    extra_flags = tuple(extra_flags) + ('-DB2R_TRACE',)
    if os.environ.get('B2R_TRACE_GT'):
      extra_flags += ('-DB2R_TRACE_GT',)
  os.makedirs(obj_dir, exist_ok=True)
  headers = [h if os.path.isabs(h) else os.path.join(HERE, h) for h in HEADERS]
  objects = []
  for src in SOURCES:
    src_path = os.path.join(HERE, src)
    obj = os.path.join(obj_dir, src.replace('.cu', '.o'))
    objects.append(obj)
    if force or _stale(obj, [src_path] + headers + [__file__]):
      cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ['-c', src_path, '-o', obj]
      if verbose:
        print(' '.join(cmd), file=sys.stderr)
      subprocess.check_call(cmd)
  if force or _stale(lib_path, objects):
    cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a',
           '-o', lib_path] + objects + ['-lcudart_static', '-lpthread', '-ldl',
                                        '-lrt']
    if verbose:
      print(' '.join(cmd), file=sys.stderr)
    subprocess.check_call(cmd)
  if not trace:
    build_fast(force=force, verbose=verbose)
  return lib_path


if __name__ == '__main__':
  print(build(force='--force' in sys.argv, verbose=True,
              extra_flags=('-Xptxas', '-v') if '--ptxas' in sys.argv else (),
              trace='--trace' in sys.argv))
