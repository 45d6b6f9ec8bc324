"""Checkpoint I/O of the replay's store columns: the host path the reference uses
(every column copied to host memory and written with np.save into gzip.GzipFile at
level 9; load: gzip + np.load + a copy back) against the device path of save() / load()
(blocked gzip compressed and inflated by csrc/ckpt.cu), on one Atari-shaped ring.

Two fills: random bytes (what bench.py fills the ring with; incompressible, so the device
writes stored blocks) and crude Atari-like frames (flat background, a moving sprite, a
noisy score band).  The two paths alternate on the same ring.  Per path and fill: wall
time of save and of load of the store columns, the kernels' device time (torch.profiler,
CUDA activity, in a pass of its own), the compressed size and GB/s of column bytes over
wall time.  One JSON line per measurement, the card's name and power limit in each.

  python profiles/micro/checkpoint_io.py [--capacity 1000000] [--out FILE]
"""
import argparse
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
  out = subprocess.check_output(
      ['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
       os.environ.get('CUDA_VISIBLE_DEVICES', '0').split(',')[0]]).decode().strip()
  name, limit = [x.strip() for x in out.split(',')]
  return name, limit


def fill(mem, kind, torch, lib, native):
  cap = mem._replay_capacity  # pylint: disable=protected-access
  gen = torch.Generator(device='cuda')
  gen.manual_seed(3)
  stream = native.current_stream()
  chunk = 65536
  for lo in range(0, cap, chunk):
    n = min(chunk, cap - lo)
    if kind == 'random':
      frames = torch.randint(0, 256, (n, 84, 84), dtype=torch.uint8, device='cuda',
                             generator=gen)
    else:
      i = torch.arange(lo, lo + n, device='cuda')
      x, y = (i * 3) % 70, (i * 7) % 70
      r = torch.arange(84, device='cuda')
      rows = (r[None, :] >= y[:, None]) & (r[None, :] < y[:, None] + 8)
      cols = (r[None, :] >= x[:, None]) & (r[None, :] < x[:, None] + 6)
      frames = torch.full((n, 84, 84), 30, dtype=torch.uint8, device='cuda')
      frames[rows[:, :, None] & cols[:, None, :]] = 200
      frames[:, 0:6, :] = (torch.randint(0, 4, (n, 6, 84), device='cuda', generator=gen) *
                           60).to(torch.uint8)
    native.check(lib.b2r_store_write(mem._h, 0, lo, n, frames.data_ptr(), stream))  # pylint: disable=protected-access
  actions = torch.randint(0, 18, (cap,), dtype=torch.int32, device='cuda', generator=gen)
  rewards = torch.randn(cap, device='cuda', generator=gen).clamp_(-1, 1)
  terms = (torch.rand(cap, device='cuda', generator=gen) < 1e-3).to(torch.uint8)
  for col, t in ((1, actions), (2, rewards), (3, terms)):
    native.check(lib.b2r_store_write(mem._h, col, 0, cap, t.data_ptr(), stream))  # pylint: disable=protected-access
  mem.add_count = cap + 500
  mem.invalid_range = [(500 - 1 + i) % cap for i in range(4 + 1)]


def host_save(mem, d, it, crb):
  for name in mem._store.keys():  # pylint: disable=protected-access
    path = os.path.join(d, '{}{}_ckpt.{}.gz'.format(crb.STORE_FILENAME_PREFIX, name, it))
    with open(path, 'wb') as f:
      with gzip.GzipFile(fileobj=f) as g:
        np.save(g, mem._store[name], allow_pickle=False)  # pylint: disable=protected-access


def host_load(mem, d, it, crb):
  for name in mem._store.keys():  # pylint: disable=protected-access
    path = os.path.join(d, '{}{}_ckpt.{}.gz'.format(crb.STORE_FILENAME_PREFIX, name, it))
    with open(path, 'rb') as f:
      with gzip.GzipFile(fileobj=f) as g:
        mem._store[name] = np.load(g, allow_pickle=False)  # pylint: disable=protected-access


def device_save(mem, d, it, crb):
  for name in mem._store.keys():  # pylint: disable=protected-access
    mem._save_store_column(  # pylint: disable=protected-access
        name, os.path.join(d, '{}{}_ckpt.{}.gz'.format(crb.STORE_FILENAME_PREFIX, name, it)))


def device_load(mem, d, it, crb):
  # what load() does for blocked files: verify every member, then inflate for real
  for verify in (True, False):
    for name in mem._store.keys():  # pylint: disable=protected-access
      path = os.path.join(d, '{}{}_ckpt.{}.gz'.format(crb.STORE_FILENAME_PREFIX, name, it))
      offset = mem._blocked_data_offset(name, path)  # pylint: disable=protected-access
      assert offset is not None, path
      mem._load_store_column(name, path, offset, verify_only=verify)  # pylint: disable=protected-access


def dir_bytes(d):
  return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def kernel_ms(fn, torch):
  from torch.profiler import profile, ProfilerActivity
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    fn()
    torch.cuda.synchronize()
  out = {}
  for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA and 'ckpt_' in e.name:
      key = e.name.split('ckpt_')[1].split('_kernel')[0]
      out[key] = out.get(key, 0.0) + e.device_time_total / 1e3
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--capacity', type=int, default=1000000)
  ap.add_argument('--fills', default='random,frames')
  ap.add_argument('--out', default=None)
  args = ap.parse_args()
  import torch
  assert torch.cuda.is_available(), 'checkpoint_io.py measures on a CUDA device'
  from dopamine_b200 import _native
  from dopamine_b200.replay_memory import circular_replay_buffer as crb
  lib = _native.lib()
  name, limit = card()
  mem = crb.OutOfGraphReplayBuffer((84, 84), 4, args.capacity, 32, output='torch')
  column_bytes = args.capacity * sum(int(np.prod(e.shape, dtype=np.int64)) * np.dtype(e.type).itemsize
                                     for e in mem.get_storage_signature())
  lines = []
  root = tempfile.mkdtemp(prefix='ckpt_io_')
  try:
    for kind in args.fills.split(','):
      fill(mem, kind, torch, lib, _native)
      torch.cuda.synchronize()
      want = {n: mem._store[n] for n in mem._store.keys()}  # pylint: disable=protected-access
      paths = (('host', host_save, host_load), ('device', device_save, device_load))
      for path, save, load in paths:  # alternating on the same ring
        d = os.path.join(root, path)
        os.makedirs(d)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        save(mem, d, 0, crb)
        torch.cuda.synchronize()
        t_save = time.perf_counter() - t0
        size = dir_bytes(d)
        t0 = time.perf_counter()
        load(mem, d, 0, crb)
        torch.cuda.synchronize()
        t_load = time.perf_counter() - t0
        same = all(np.array_equal(mem._store[n], want[n]) for n in want)  # pylint: disable=protected-access
        rec = dict(fill=kind, path=path, capacity=args.capacity, column_bytes=column_bytes,
                   compressed_bytes=size, ratio=round(column_bytes / size, 2),
                   save_s=round(t_save, 3), load_s=round(t_load, 3),
                   save_GBps=round(column_bytes / t_save / 1e9, 3),
                   load_GBps=round(column_bytes / t_load / 1e9, 3),
                   round_trip_identical=same, gpu=name, power_limit=limit)
        if path == 'device':
          d2 = os.path.join(root, 'profiled')
          os.makedirs(d2)
          rec['save_kernel_ms'] = kernel_ms(lambda: device_save(mem, d2, 0, crb), torch)
          rec['load_kernel_ms'] = kernel_ms(lambda: device_load(mem, d2, 0, crb), torch)
          shutil.rmtree(d2)
        shutil.rmtree(d)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
  finally:
    shutil.rmtree(root, ignore_errors=True)
  if args.out:
    with open(args.out, 'w') as f:
      for rec in lines:
        f.write(json.dumps(rec) + '\n')


if __name__ == '__main__':
  main()
