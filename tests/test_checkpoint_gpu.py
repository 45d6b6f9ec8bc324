"""Store columns checkpointed as blocked gzip, compressed and inflated on the device
(csrc/ckpt.cu): the files are what np.save writes, member by member readable by any
gzip reader; they load back bit for bit; malformed files are refused on the host with
the buffer untouched.  Python's zlib is the reference encoder and decoder throughout.
"""
import gzip
import io
import os
import random
import shutil
import struct
import zlib

import numpy as np
import pytest

from dopamine_b200.replay_memory import circular_replay_buffer as crb

SLICE = 65280
STORE = crb.STORE_FILENAME_PREFIX


def _npy(array):
  buf = io.BytesIO()
  np.save(buf, array, allow_pickle=False)
  return buf.getvalue()


def _members(raw):
  """The BGZF members of a file, found from the headers alone."""
  out, q = [], 0
  while q < len(raw):
    assert raw[q:q + 16] == b'\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00BC\x02\x00', q
    size = struct.unpack('<H', raw[q + 16:q + 18])[0] + 1
    assert q + size <= len(raw)
    out.append(raw[q:q + size])
    q += size
  return out


def _block_type(member):
  """BTYPE of the first deflate block of a member (the device writes one block)."""
  first = member[18]
  assert first & 1, 'the first block is not the final one'
  return (first >> 1) & 3


def _frames(n, seed=0):
  """Crude Atari-like screens: flat background, a moving sprite, a noisy score band."""
  rng = np.random.RandomState(seed)
  f = np.full((n, 84, 84), 30, np.uint8)
  for i in range(n):
    x, y = (i * 3) % 70, (i * 7) % 70
    f[i, y:y + 8, x:x + 6] = 200
    f[i, 0:6, :] = rng.randint(0, 4, size=(6, 84)) * 60
  return f


# -------------------------------------------------------------- fixed Huffman in Python --
_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67,
             83, 99, 115, 131, 163, 195, 227, 258]
_LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
_DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513,
              769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577]
_DIST_EXTRA = [0, 0, 0, 0] + [k for k in range(1, 14) for _ in (0, 1)]


class _Bits(object):
  def __init__(self):
    self.bits = []

  def put(self, value, n):  # LSB first
    self.bits.extend((value >> i) & 1 for i in range(n))

  def code(self, value, n):  # Huffman codes go MSB first
    self.bits.extend((value >> (n - 1 - i)) & 1 for i in range(n))

  def symbol(self, s):
    if s < 144:
      self.code(0x30 + s, 8)
    elif s < 256:
      self.code(0x190 + s - 144, 9)
    elif s < 280:
      self.code(s - 256, 7)
    else:
      self.code(0xC0 + s - 280, 8)

  def tobytes(self):
    return np.packbits(np.array(self.bits, np.uint8), bitorder='little').tobytes()


def _fixed_deflate(tokens):
  """One final fixed-Huffman block; a token is a literal byte or (length, distance)."""
  b = _Bits()
  b.put(1, 1)
  b.put(1, 2)
  for t in tokens:
    if isinstance(t, tuple):
      length, dist = t
      k = max(i for i in range(29) if _LEN_BASE[i] <= length)
      b.symbol(257 + k)
      b.put(length - _LEN_BASE[k], _LEN_EXTRA[k])
      d = max(i for i in range(30) if _DIST_BASE[i] <= dist)
      b.code(d, 5)
      b.put(dist - _DIST_BASE[d], _DIST_EXTRA[d])
    else:
      b.symbol(t)
  b.symbol(256)
  return b.tobytes()


def _member(body, data):
  size = 18 + len(body) + 8
  return (b'\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\x00BC\x02\x00' + struct.pack('<H', size - 1)
          + body + struct.pack('<II', zlib.crc32(data), len(data)))


def _zlib_member(data, strategy=zlib.Z_FIXED):
  c = zlib.compressobj(9, zlib.DEFLATED, -15, 9, strategy)
  return _member(c.compress(data) + c.flush(), data)


# ------------------------------------------------------------------------- CPU side ----
@pytest.mark.parametrize('shape,dtype', [
    ((100, 84, 84), np.uint8), ((10,), np.int32), ((7,), np.float32), ((5, 5, 3), np.float64),
    ((3, 2), np.int64), ((1000000, 84, 84), np.uint8), ((4,), np.bool_), ((0,), np.uint8)])
def test_npy_header_is_the_one_np_save_writes(shape, dtype):
  class Stop(Exception):
    pass

  class FirstWrite(object):  # np.save writes the whole header in its first write
    def write(self, data):
      self.data = bytes(data)
      raise Stop()

  first = FirstWrite()
  view = np.lib.stride_tricks.as_strided(np.zeros(1, dtype), shape, (0,) * len(shape))
  with pytest.raises(Stop):
    np.save(first, view, allow_pickle=False)
  header = crb.npy_header(shape, dtype)
  assert header == first.data
  if np.prod(shape) <= 10**5:
    want = _npy(np.zeros(shape, dtype))
    assert want[:len(header)] == header
    assert len(want) == len(header) + int(np.prod(shape)) * np.dtype(dtype).itemsize


def test_header_member_is_ordinary_gzip():
  payload = crb.npy_header((12, 84, 84), np.uint8)
  member = crb.bgzf_member(payload)
  assert zlib.decompress(member, 31) == payload
  assert gzip.decompress(member + member) == payload + payload
  assert _members(member) == [member]


def test_python_fixed_encoder_is_read_by_zlib():
  data = bytes(range(256)) * 3
  tokens = list(data[:256]) + [(258, 256), (254, 256)]
  assert zlib.decompress(_fixed_deflate(tokens), -15) == data


# ------------------------------------------------------------------------- GPU side ----
@pytest.fixture(scope='module')
def prb():
  import torch
  if not torch.cuda.is_available():
    pytest.fail('-m gpu tests need a CUDA device (no CPU fallback exists)')
  from dopamine_b200.replay_memory import prioritized_replay_buffer
  return prioritized_replay_buffer


def _columns(mem):
  return {name: mem._store[name].copy() for name in mem._store.keys()}


def _check_files(mem, ckpt, suffix):
  """Payload: every store file inflates to np.save of the column; every member is a
  well-formed BGZF member that zlib inflates alone.  Returns {name: [BTYPE per data
  member]}."""
  types = {}
  for name, column in _columns(mem).items():
    path = os.path.join(ckpt, '{}{}_ckpt.{}.gz'.format(STORE, name, suffix))
    raw = open(path, 'rb').read()
    want = _npy(column)
    with gzip.GzipFile(path) as g:
      assert g.read() == want, name
    with gzip.GzipFile(path) as g:
      back = np.load(g, allow_pickle=False)
    assert back.dtype == column.dtype and back.shape == column.shape
    members = _members(raw)
    header = crb.npy_header(column.shape, column.dtype)
    data = column.tobytes()
    assert len(members) == 1 + -(-len(data) // SLICE), name
    assert zlib.decompress(members[0], 31) == header
    types[name] = []
    for k, m in enumerate(members[1:]):
      piece = data[k * SLICE:(k + 1) * SLICE]
      assert zlib.decompress(m, 31) == piece, (name, k)
      crc, isize = struct.unpack('<II', m[-8:])
      assert crc == zlib.crc32(piece) and isize == len(piece), (name, k)
      assert len(m) <= 65536
      types[name].append(_block_type(m))
      assert types[name][-1] in (0, 1)
  return types


def _uniform(shape=(84, 84), cap=100, **kw):
  return crb.OutOfGraphReplayBuffer(shape, 4, cap, 8, **kw)


def _fill(mem, obs, seed=0):
  rng = np.random.RandomState(seed)
  cap = mem._replay_capacity
  mem._store['observation'] = obs
  mem._store['action'] = rng.randint(0, 18, size=cap).astype(np.int32)
  mem._store['reward'] = rng.randn(cap).astype(mem._reward_dtype)
  mem._store['terminal'] = (rng.rand(cap) < 0.05).astype(mem._terminal_dtype)
  mem.add_count = cap + 7
  mem.invalid_range = crb.invalid_range(7, cap, mem._stack_size, mem._update_horizon)


@pytest.mark.gpu
def test_saved_members_are_np_save_bytes_and_stream_alone(prb, tmp_path):
  mem = _uniform(cap=300)
  _fill(mem, _frames(300))
  mem.save(str(tmp_path), 3)
  types = _check_files(mem, str(tmp_path), 3)
  assert set(types['observation']) == {1}  # structured frames compress
  obs = os.path.getsize(os.path.join(str(tmp_path), STORE + 'observation_ckpt.3.gz'))
  assert obs * 8 < 300 * 84 * 84


@pytest.mark.gpu
def test_device_verify_only_compress_matches_the_file(prb, tmp_path):
  import ctypes
  from dopamine_b200 import _native
  mem = _uniform(cap=300)
  _fill(mem, _frames(300, seed=2))
  mem.save(str(tmp_path), 0)
  for name, col in mem._columns.items():
    size = ctypes.c_int64(-1)
    _native.check(mem._lib.b2r_ckpt_save_column(mem._h, col, -1, 1, ctypes.byref(size),
                                                _native.current_stream()))
    path = os.path.join(str(tmp_path), '{}{}_ckpt.0.gz'.format(STORE, name))
    head = len(crb.bgzf_member(mem._npy_header(name)))
    assert size.value == os.path.getsize(path) - head, name


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['uniform', 'prioritized'])
def test_round_trip_is_bit_identical(prb, tmp_path, kind):
  rng = np.random.RandomState(5)
  if kind == 'uniform':
    make = lambda: _uniform(cap=500, update_horizon=3)
  else:
    make = lambda: prb.OutOfGraphPrioritizedReplayBuffer((84, 84), 4, 500, 8,
                                                         update_horizon=3)
  mem = make()
  frames = _frames(40, seed=1)
  for i in range(700):
    obs = frames[i % 40] if i % 3 else rng.randint(0, 256, (84, 84)).astype(np.uint8)
    row = (obs, rng.randint(18), np.float32(rng.randn()), int(rng.rand() < 0.03))
    if kind == 'uniform':
      mem.add(*row)
    else:
      mem.add(*row, float(rng.rand() + 0.1))
  mem.save(str(tmp_path), 2)
  _check_files(mem, str(tmp_path), 2)
  back = make()
  back.load(str(tmp_path), 2)
  for name, col in _columns(mem).items():
    assert back._store[name].tobytes() == col.tobytes(), name
  assert int(back.add_count) == int(mem.add_count)
  assert back.invalid_range.tolist() == mem.invalid_range.tolist()
  if kind == 'prioritized':
    for a, b in zip(mem.sum_tree.nodes, back.sum_tree.nodes):
      assert np.array_equal(a.view(np.uint64), b.view(np.uint64))
    assert mem.sum_tree.max_recorded_priority == back.sum_tree.max_recorded_priority
  np.random.seed(9)
  random.seed(9)
  want = mem.sample_transition_batch()
  np.random.seed(9)
  random.seed(9)
  got = back.sample_transition_batch()
  for w, g in zip(want, got):
    assert np.asarray(w).tobytes() == np.asarray(g).tobytes()


@pytest.mark.gpu
def test_device_files_load_through_the_host_path(prb, tmp_path):
  """gzip + np.load read every store file; the reference's own load reads the
  directory where the reference is importable; a reference-written checkpoint takes the
  host path."""
  from oracle import refshim
  mem = _uniform(cap=200)
  _fill(mem, _frames(200, seed=4))
  mem.save(str(tmp_path), 1)
  for name, col in _columns(mem).items():
    path = os.path.join(str(tmp_path), '{}{}_ckpt.1.gz'.format(STORE, name))
    with open(path, 'rb') as f:
      with gzip.GzipFile(fileobj=f) as g:
        assert np.load(g, allow_pickle=False).tobytes() == col.tobytes()
  if refshim.reference_available():
    _, ref_crb, _ = refshim.load_reference()
    ref = ref_crb.OutOfGraphReplayBuffer((84, 84), 4, 200, 8)
    ref.load(str(tmp_path), '1')
    for name, col in _columns(mem).items():
      assert ref._store[name].tobytes() == col.tobytes(), name
  golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ckpt_ref')
  for f in os.listdir(golden):
    if f.startswith(STORE):
      name = f[len(STORE):].split('_ckpt')[0]
      assert mem._blocked_data_offset(name, os.path.join(golden, f)) is None


@pytest.mark.gpu
@pytest.mark.parametrize('fill', ['zeros', 'random', 'frames'])
@pytest.mark.parametrize('cap', [10, 100, 1000])
def test_envelope_against_zlib(prb, tmp_path, fill, cap):
  """All-zero, random and structured columns; capacity 10 (every column smaller than a
  member), sizes that are not multiples of 65280."""
  mem = _uniform(cap=cap)
  if fill == 'zeros':
    obs = np.zeros((cap, 84, 84), np.uint8)
  elif fill == 'random':
    obs = np.random.RandomState(cap).randint(0, 256, (cap, 84, 84)).astype(np.uint8)
  else:
    obs = _frames(cap, seed=cap)
  _fill(mem, obs)
  mem.save(str(tmp_path), 4)
  types = _check_files(mem, str(tmp_path), 4)
  if fill == 'random':
    assert set(types['observation']) == {0}
  else:
    assert set(types['observation']) == {1}
  back = _uniform(cap=cap)
  back.load(str(tmp_path), 4)
  for name, col in _columns(mem).items():
    assert back._store[name].tobytes() == col.tobytes(), name


@pytest.mark.gpu
def test_non_atari_shapes_and_dtypes(prb, tmp_path):
  extras = [crb.ReplayElement('extra1', (2,), np.float32),
            crb.ReplayElement('extra2', (3, 2), np.int16)]
  make = lambda: crb.OutOfGraphReplayBuffer(
      (5, 3), 2, 30000, 8, observation_dtype=np.float64, terminal_dtype=np.int64,
      extra_storage_types=extras, action_shape=(2,), action_dtype=np.int64,
      reward_dtype=np.float64)
  mem = make()
  rng = np.random.RandomState(3)
  cap = 30000
  mem._store['observation'] = np.round(rng.randn(cap, 5, 3), 1)
  mem._store['action'] = rng.randint(0, 5, (cap, 2))
  mem._store['reward'] = rng.randn(cap)
  mem._store['terminal'] = (rng.rand(cap) < 0.01).astype(np.int64)
  mem._store['extra1'] = rng.rand(cap, 2).astype(np.float32)
  mem._store['extra2'] = rng.randint(-3, 3, (cap, 3, 2)).astype(np.int16)
  mem.add_count = 12345
  mem.invalid_range = crb.invalid_range(12345 % cap, cap, 2, 1)
  mem.save(str(tmp_path), 0)
  _check_files(mem, str(tmp_path), 0)
  back = make()
  back.load(str(tmp_path), 0)
  for name, col in _columns(mem).items():
    assert back._store[name].tobytes() == col.tobytes(), name
  for i in range(0, cap, 997):  # the terminal mirror followed the inflated column
    assert back.is_valid_transition(i) == mem.is_valid_transition(i)


@pytest.mark.gpu
def test_device_inflates_zlib_members_with_long_and_far_matches(prb, tmp_path):
  """Members encoded outside this library: zlib's fixed-Huffman members and a member of
  258-byte matches at distance exactly 32768 (zlib itself never reaches that far)."""
  cap = 140  # two full data members and a short one
  mem = crb.OutOfGraphReplayBuffer((1024,), 4, cap, 8)
  rng = np.random.RandomState(8)
  head = rng.randint(0, 256, 32768).astype(np.uint8).tobytes()
  far = (head * 2)[:SLICE]
  tokens = list(head)
  left = SLICE - 32768
  while left:
    n = min(258, left) if left - min(258, left) >= 3 or left <= 258 else left - 3
    tokens.append((n, 32768))
    left -= n
  body = _fixed_deflate(tokens)
  assert zlib.decompress(body, -15) == far
  second = _frames(20).tobytes()[:SLICE]
  rest = rng.randint(0, 4, cap * 1024 - 2 * SLICE).astype(np.uint8).tobytes()
  column = np.frombuffer(far + second + rest, np.uint8).reshape(cap, 1024)
  _fill(mem, column)
  mem.save(str(tmp_path), 6)
  path = os.path.join(str(tmp_path), STORE + 'observation_ckpt.6.gz')
  with open(path, 'wb') as f:
    f.write(crb.bgzf_member(crb.npy_header(column.shape, column.dtype)))
    f.write(_member(body, far))
    f.write(_zlib_member(second))
    f.write(_zlib_member(rest))
  back = crb.OutOfGraphReplayBuffer((1024,), 4, cap, 8)
  assert back._blocked_data_offset('observation', path) is not None
  back.load(str(tmp_path), 6)
  assert back._store['observation'].tobytes() == column.tobytes()


def _corrupt_variants(raw):
  members = _members(raw)
  m1 = bytearray(members[1])
  out = {}
  flipped = bytearray(m1)
  flipped[len(flipped) // 2] ^= 0x5A
  out['flipped_byte'] = [flipped]
  bad_crc = bytearray(m1)
  bad_crc[-8] ^= 1
  out['wrong_crc'] = [bad_crc]
  out['truncated'] = None  # handled below
  bad_bsize = bytearray(members[-1])
  bad_bsize[16:18] = struct.pack('<H', 0xFFFF)
  out['bsize_past_end'] = ('last', bad_bsize)
  data = zlib.decompress(bytes(m1), 31)
  out['dynamic_huffman'] = [_zlib_member(data, zlib.Z_DEFAULT_STRATEGY)]
  files = {}
  for kind, v in out.items():
    if kind == 'truncated':
      files[kind] = raw[:-100]
    elif kind == 'bsize_past_end':
      files[kind] = b''.join(members[:-1]) + bytes(v[1])
    else:
      files[kind] = members[0] + bytes(v[0]) + b''.join(members[2:])
  return files


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['flipped_byte', 'wrong_crc', 'truncated',
                                  'bsize_past_end', 'dynamic_huffman'])
def test_malformed_files_are_refused_and_change_nothing(prb, tmp_path, kind):
  from dopamine_b200 import _native
  src = str(tmp_path / 'good')
  os.makedirs(src)
  mem = _uniform(cap=100)
  _fill(mem, _frames(100, seed=6))
  mem.save(src, 1)
  obs_name = STORE + 'observation_ckpt.1.gz'
  raw = open(os.path.join(src, obs_name), 'rb').read()
  bad = _corrupt_variants(raw)[kind]
  dst = str(tmp_path / kind)
  shutil.copytree(src, dst)
  with open(os.path.join(dst, obs_name), 'wb') as f:
    f.write(bad)
  if kind == 'dynamic_huffman':
    with gzip.GzipFile(os.path.join(dst, obs_name)) as g:  # a valid gzip file all the same
      assert g.read() == _npy(mem._store['observation'])
  target = _uniform(cap=100)
  _fill(target, np.random.RandomState(1).randint(0, 256, (100, 84, 84)).astype(np.uint8),
        seed=11)
  before = _columns(target)
  count, invalid = int(target.add_count), target.invalid_range.tolist()
  with pytest.raises(gzip.BadGzipFile):
    target.load(dst, 1)
  assert _native.lib().b2r_check(target._h, _native.current_stream()) == 0
  import torch
  torch.cuda.synchronize()
  for name, col in _columns(target).items():
    assert col.tobytes() == before[name].tobytes(), name
  assert int(target.add_count) == count and target.invalid_range.tolist() == invalid
  target.load(src, 1)  # and the device path still works
  assert target._store['observation'].tobytes() == mem._store['observation'].tobytes()
