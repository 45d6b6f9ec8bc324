"""One timeline of the fused step: %globaltimer marks of all its kernels.

  B2R_TRACE_GT=1 python -m dopamine_b200.csrc.build --trace --force
  B2R_LIB=profiles/micro/libb200replay_trace.so python profiles/micro/timeline.py 1024

Prints the marks of the LAST replayed step in microseconds since the sampler started."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

NAMES = {
    'sample': {10: 'S start (CTA 0)', 11: 'S acquired', 12: 'S prologue loads in',
               13: 'S draw + owner', 14: 'S descent done', 15: 'S validity done',
               16: 'S rows written (CTA 0)', 17: 'S last CTA: alone', 18: 'S invalid list',
               19: 'S fix-ups done', 20: 'S END'},
    'gather': {0: 'G start (CTA 0)', 1: 'G acquired', 5: 'G CTA 0 stored', 6: 'G END'},
    'c51': {0: 'L-pre start', 1: 'L-pre acquired', 3: 'L softmaxes', 5: 'L projection',
            8: 'L-pre END', 10: 'L-tail start', 11: 'L-tail acquired', 12: 'L-tail loss END',
            9: 'L-tail tree END', 13: 'L-tail row scalars in', 14: 'L-tail log-softmax done',
            15: 'L-tail staged'},
    'tree': {30: 'T tiny start', 7: 'T tiny / one-CTA END',
             0: 'T one-CTA start', 1: 'T one-CTA acquired', 5: 'T one-CTA leaf level done',
             12: 'P presort start',
             14: 'P presort END', 13: 'T apply start', 10: 'T leaf deltas published',
             11: 'T levels released', 15: 'T apply END'},
}


# the level-per-CTA write-back (more than 32 sets): marks by the CTA of a given level
TREE_BIG = {12: 'P presort start', 14: 'P presort END', 13: 'T apply start',
            16: 'T leaf: level taken', 17: 'T leaf: values staged', 18: 'T leaf: deltas computed',
            19: 'T leaf: deltas written', 10: 'T leaf: deltas published',
            0: 'T root: level taken', 29: 'T root: values staged', 1: 'T root: at the flag',
            2: 'T root: released', 3: 'T root: deltas in group order', 4: 'T root: chains done',
            22: 'T deepest: level taken', 23: 'T deepest: values staged',
            24: 'T deepest: at the flag', 25: 'T deepest: released',
            26: 'T deepest: deltas in group order', 27: 'T deepest: chains done',
            20: 'T level 1: deltas in group order', 21: 'T level 1: chains done',
            11: 'T levels released (last)', 15: 'T apply END'}


def main():
  batch = int(sys.argv[1]) if len(sys.argv) > 1 else 32
  capacity = int(sys.argv[2]) if len(sys.argv) > 2 else 1000000
  if batch > 32:
    NAMES['tree'] = TREE_BIG
  import torch
  from dopamine_b200 import _native
  defer = len(sys.argv) > 3 and sys.argv[3] == 'defer'
  wl = bench.GpuWorkload(capacity, batch, 0)
  lib = _native.lib()
  g = torch.cuda.CUDAGraph()
  s = torch.cuda.Stream()
  with torch.cuda.stream(s):
    if defer:  # the copies of step n beside the chain of step n + 1, joined per graph
      wl.set_deferred(True)
    for _ in range(5):
      wl.step(batch)
    if defer:
      wl.join()
    s.synchronize()
    with torch.cuda.graph(g, stream=s):
      for _ in range(4 if defer else 1):
        wl.step(batch)
      if defer:
        wl.join()
    for _ in range(300):
      g.replay()
    s.synchronize()
  events = []
  for name in ('sample', 'gather', 'c51', 'tree'):
    out = (ctypes.c_longlong * 32)()
    fn = getattr(lib, 'b2r_debug_trace_' + name)
    fn.argtypes = [ctypes.c_void_p]
    fn(out)
    for i, v in enumerate(out):
      if v and i in NAMES[name]:
        events.append((int(v), NAMES[name][i]))
  t0 = dict((n, t) for t, n in events).get('S start (CTA 0)', min(t for t, _ in events))
  recent = [(t, n) for t, n in events if t >= t0 - 1000]
  for t, n in sorted(recent):
    print('%9.2f us  %s' % ((t - t0) / 1e3, n))
  stale = [n for t, n in events if t < t0 - 1000]
  if stale:
    print('(not in the last step: %s)' % ', '.join(stale))
  if batch > 32 and hasattr(lib, 'b2r_debug_trace_tree_levels'):
    lv = (ctypes.c_longlong * 128)()
    lib.b2r_debug_trace_tree_levels.argtypes = [ctypes.c_void_p]
    lib.b2r_debug_trace_tree_levels(lv)
    if hasattr(lib, 'b2r_debug_trace_tree_counts'):
      cnt = (ctypes.c_ulonglong * 8)()
      lib.b2r_debug_trace_tree_counts.argtypes = [ctypes.c_void_p]
      lib.b2r_debug_trace_tree_counts(cnt)
      print('early write-backs: %d launched, %d with own lists, %d without a hand-over '
            'behind the values' % (cnt[0], cnt[1], cnt[2]))
    if hasattr(lib, 'b2r_debug_trace_tree_phases'):
      ph = (ctypes.c_longlong * 32)()
      lib.b2r_debug_trace_tree_phases.argtypes = [ctypes.c_void_p]
      lib.b2r_debug_trace_tree_phases(ph)
      names = ['start', 'indices in', 'analysed', 'grouped by leaf', 'duplicates counted',
               'list made', 'grouped by node', 'nodes fetched', 'leaves landed',
               'said so', 'before the wait', 'parent ended']
      for who, label in ((0, 'leaf CTA'), (1, 'CTA of level 10')):
        print('  %s: %s' % (label, ', '.join(
            '%s %.2f' % (names[i], (ph[who * 16 + i] - t0) / 1e3)
            for i in range(len(names)) if ph[who * 16 + i])))
    print('write-back per level (us): grouped | parent ended | released | done')
    for level in range(32):
      row = [lv[w * 32 + level] for w in range(4)]
      if any(row):
        print('  level %2d: %s' % (level, '  '.join(
            '%7.2f' % ((t - t0) / 1e3) if t else '      -' for t in row)))


if __name__ == '__main__':
  main()
