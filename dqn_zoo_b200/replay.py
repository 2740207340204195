"""HBM-resident replay with the reference's `dqn_zoo/replay.py` surface.

Same class names, constructor arguments, return types/dtypes and exceptions as the
reference (cited per method), so agents and tests written for `dqn_zoo.replay`
run unchanged, with two stated differences: a (snappy) encoder/decoder pair is applied as a
host round trip at insert time instead of at rest, and the accumulators return lists, not
generators.  What else differs is where things live:

  * transition storage (`OrderedDict` in the reference, `replay.py:140,688`) is a
    transition-major uint8 array in device memory: row = id % capacity holds
    s_tm1 | s_t back to back (DESIGN.md §3); with `frame_capacity=F` the row holds frame
    slot numbers instead and every distinct (H, W) frame of the stacks is stored once
    (`_FrameStore`), with byte-identical results;
  * the float64 sum tree (`replay.py:246-426`) is a device array traversed by a
    warp-cooperative CUDA kernel (csrc/dz_replay.cu);
  * O(1) integer bookkeeping per add (free-slot stack, swap-remove lists,
    id<->index maps; `replay.py:52-74,475-534`) stays on the host exactly as in the
    reference, and is mirrored to the device as (position, value) patches so that
    sampling needs no host lookups;
  * the host `np.random.RandomState` is consumed in the reference's order
    (`replay.py:551-567`), its draws are shipped to the device, and index selection,
    probabilities, importance weights and the gather run in CUDA.

No CPU fallback: every numeric result returned by `sample()` is computed on the GPU.
"""

from __future__ import annotations

import collections
import ctypes as C
from typing import Any, Callable, Iterable, List, Mapping, NamedTuple, Optional, Sequence, Tuple

import numpy as np
import torch

from dqn_zoo_b200 import _lib

_POOL_FULL_MESSAGE = ('frame pool is full: frame_capacity is too small for the frames the live transitions reference '
                      '(the transitions added since are not stored)')
_FLAG_NAMES = {1: 'value must be finite and positive', 2: 'index out of range', 4: 'Require 0 <= target < total sum.',
               8: 'sum-tree root is zero in the fused path', 16: 'Weights are not finite'}


class Transition(NamedTuple):
  """`replay.py:36-41`."""
  s_tm1: Any
  a_tm1: Any
  r_t: Any
  discount_t: Any
  s_t: Any


def _device():
  if not torch.cuda.is_available():
    raise RuntimeError('dqn_zoo_b200.replay needs a CUDA device (there is no CPU fallback)')
  return torch.device('cuda', torch.cuda.current_device())


def _stream():
  return torch.cuda.current_stream().cuda_stream


def _ptr(t):
  return 0 if t is None else t.data_ptr()


def _power(base, exponent):
  """`replay.py:203-208` for the HOST-side add path (float64 scalar per add, as the
  reference evaluates it at `replay.py:507`).  The float32 `update_priorities` path is
  evaluated on the device instead (csrc/dz_replay.cu:exponentiate_f32)."""
  b = np.asarray(base, dtype=np.float64)
  return np.where(b == 0.0, 0.0, b ** exponent)


def importance_sampling_weights(probabilities, uniform_probability, exponent, normalize):
  """`replay.py:211-243`, evaluated on the device (float64)."""
  if not 0.0 <= exponent <= 1.0:
    raise ValueError('Require 0 <= exponent <= 1.')
  if not 0.0 <= uniform_probability <= 1.0:
    raise ValueError('Expected 0 <= uniform_probability <= 1.')
  p = torch.as_tensor(np.asarray(probabilities, dtype=np.float64), device=_device())
  w = (uniform_probability / p) ** exponent
  if normalize:
    w = w / w.max()
  w = w.cpu().numpy()
  if not np.isfinite(w).all():
    raise ValueError('Weights are not finite: %s.' % w)
  return w


# ------------------------------------------------------------------------------------------------
# R1: SumTree
# ------------------------------------------------------------------------------------------------


class SumTree:
  """Device-resident float64 sum tree with the interface of `replay.py:246-426`."""

  def __init__(self):
    self._size = 0
    self._first_leaf = 0
    self._nodes = torch.zeros(0, dtype=torch.float64, device=_device())
    self._flags = torch.zeros(1, dtype=torch.int32, device=_device())

  # -- helpers ---------------------------------------------------------------------------------
  def _rebuild(self, n_valid):
    if self._first_leaf:
      _lib.call('dz_sumtree_rebuild', _ptr(self._nodes), self._first_leaf, n_valid, _stream())

  def _raise_flags(self):
    f = int(self._flags.item())
    if f:
      self._flags.zero_()
      if f & _lib.DZ_FLAG_FRAME_POOL_FULL:
        raise RuntimeError(_POOL_FULL_MESSAGE)
      if f & _lib.DZ_FLAG_BAD_INDEX:
        raise IndexError('index out of range, expect 0 <= index < %s' % self._size)
      raise ValueError(_FLAG_NAMES.get(f & -f, 'device flag %d' % f))

  def _initialize(self, size, values):
    """`replay.py:361-392`."""
    assert size >= 0
    assert values is None or len(values) == size
    fl = self._first_leaf
    if size < self._size:
      self._size = size
      if values is not None:
        self._nodes[fl:fl + size] = values
      self._rebuild(size)
    elif size <= fl:
      self._size = size
      if values is not None:
        self._nodes[fl:fl + size] = values
        self._rebuild(size)
    else:
      cap = 1
      while cap < size:
        cap *= 2
      new = torch.empty(2 * cap, dtype=torch.float64, device=self._nodes.device)
      if values is None:
        keep = self._size
        new[cap:cap + keep] = self._nodes[fl:fl + keep]
      else:
        keep = size
        new[cap:cap + keep] = values
      self._nodes, self._first_leaf, self._size = new, cap, size
      self._rebuild(keep)

  @staticmethod
  def _validated(values, msg):
    v = np.asarray(values, dtype=np.float64)
    if not np.isfinite(v).all() or (v < 0.0).any():
      raise ValueError(msg)
    return v

  # -- reference surface -------------------------------------------------------------------------
  def resize(self, size: int) -> None:
    """`replay.py:267-269`."""
    self._initialize(size, None)

  def get(self, indices) -> np.ndarray:
    """`replay.py:271-276`."""
    idx = np.asarray(indices, dtype=np.int64)
    if idx.size and not ((0 <= idx) & (idx < self._size)).all():
      raise IndexError('index out of range, expect 0 <= index < %s' % self._size)
    if idx.size == 0:
      return np.zeros(idx.shape, dtype=np.float64)
    d_idx = torch.as_tensor(idx.reshape(-1), device=self._nodes.device)
    out = torch.empty(idx.size, dtype=torch.float64, device=self._nodes.device)
    _lib.call('dz_sumtree_get', _ptr(self._nodes), self._first_leaf, self._size, _ptr(d_idx), idx.size, _ptr(out),
              _ptr(self._flags), _stream())
    return out.cpu().numpy().reshape(idx.shape)

  def set(self, indices, values) -> None:
    """`replay.py:278-290`."""
    v = self._validated(values, 'value must be finite and positive.').reshape(-1)
    idx = np.asarray(indices, dtype=np.int64).reshape(-1)
    if idx.size == 0:
      return
    if not ((0 <= idx) & (idx < self._size)).all():
      raise IndexError('index out of range')
    self.set_device(torch.as_tensor(idx, device=self._nodes.device), torch.as_tensor(v, device=self._nodes.device))

  def set_device(self, d_idx: torch.Tensor, d_values: torch.Tensor) -> None:
    """`set` with device-resident int64 indices / float64 values (no host round trip)."""
    _lib.call('dz_sumtree_set', _ptr(self._nodes), self._first_leaf, self._size, _ptr(d_idx), _ptr(d_values),
              d_idx.numel(), _ptr(self._flags), _stream())

  def set_all(self, values) -> None:
    """`replay.py:292-297`."""
    v = self._validated(values, 'Values must be finite positive numbers.')
    self._initialize(len(v), torch.as_tensor(v, device=self._nodes.device))

  def query(self, targets) -> List[int]:
    """`replay.py:299-313`: ValueError unless 0 <= target < root for every target."""
    t = np.asarray(targets, dtype=np.float64).reshape(-1)
    root = self.root()
    if t.size and not ((0.0 <= t) & (t < root)).all():
      raise ValueError('Require 0 <= target < total sum.')
    if t.size == 0:
      return []
    d_t = torch.as_tensor(t, device=self._nodes.device)
    out = torch.empty(t.size, dtype=torch.int64, device=self._nodes.device)
    _lib.call('dz_sumtree_query', _ptr(self._nodes), self._first_leaf, _ptr(d_t), t.size, _ptr(out), _ptr(self._flags),
              _stream())
    return out.cpu().tolist()

  def root(self) -> float:
    """`replay.py:315-317`."""
    return float(self._nodes[1].item()) if self._size > 0 else np.nan

  @property
  def values(self) -> np.ndarray:
    """`replay.py:319-322` (a host COPY here; the reference returns a view)."""
    return self._nodes[self._first_leaf:self._first_leaf + self._size].cpu().numpy()

  @property
  def size(self) -> int:
    return self._size

  @property
  def capacity(self) -> int:
    return self._first_leaf

  @property
  def device_nodes(self) -> torch.Tensor:
    return self._nodes

  def get_state(self) -> Mapping[str, Any]:
    """`replay.py:334-340`: same keys; `storage` is a host float64 array."""
    return {'size': self._size, 'storage': self._nodes.cpu().numpy(), 'first_leaf': self._first_leaf}

  def set_state(self, state: Mapping[str, Any]) -> None:
    """`replay.py:342-346`."""
    self._size = int(state['size'])
    self._first_leaf = int(state['first_leaf'])
    self._nodes = torch.as_tensor(np.array(state['storage'], dtype=np.float64), device=self._nodes.device)

  def check_valid(self) -> Tuple[bool, str]:
    """`replay.py:348-359` (consistency is verified on a host copy)."""
    nodes = self._nodes.cpu().numpy()
    fl = self._first_leaf
    if len(nodes) != 2 * fl:
      return False, 'first_leaf should be half the size of storage.'
    if not 0 <= self._size <= fl:
      return False, 'Require 0 <= self.size <= self.capacity.'
    if fl > 1:
      sums = nodes[2:2 * fl:2] + nodes[3:2 * fl:2]
      bad = np.nonzero(nodes[1:fl] != sums)[0]
      if bad.size:
        return False, 'Non-leaf node %d should be sum of child nodes.' % (bad[0] + 1)
    return True, ''


# ------------------------------------------------------------------------------------------------
# Device mirrors of the dense host lists
# ------------------------------------------------------------------------------------------------


class _DeviceList:
  """int64 device array that mirrors a host list through (position, value) patches."""

  def __init__(self, n=0):
    self.t = torch.zeros(max(n, 1), dtype=torch.int64, device=_device())

  def ensure(self, n):
    if n > self.t.numel():
      new = torch.zeros(max(n, 2 * self.t.numel()), dtype=torch.int64, device=self.t.device)
      new[:self.t.numel()] = self.t
      self.t = new

  def upload(self, values):
    v = np.asarray(values, dtype=np.int64)
    self.ensure(len(v))
    if len(v):
      self.t[:len(v)] = torch.as_tensor(v, device=self.t.device)


def _apply_index_record(view, patches, tree_index=-1, leaf_value=0.0, evict_index=-1, size_after=0, slot=0,
                        action=0, reward=0.0, discount=0.0, h_s_tm1=None, h_s_t=None, d_priority=None, alpha=1.0,
                        item_id=0, oldest_live=0):
  """One dz_replay_add call: <=4 list patches + optional evict/set on the tree (+ optional row write)."""
  rec = _lib.AddRecord()
  rec.item_id, rec.oldest_live = item_id, oldest_live
  rec.slot, rec.action, rec.reward, rec.discount = slot, action, reward, discount
  rec.n_patches = len(patches)
  for k, (target, pos, val) in enumerate(patches):
    rec.patch_target[k], rec.patch_pos[k], rec.patch_val[k] = target, pos, val
  rec.tree_index, rec.leaf_value, rec.evict_index, rec.size_after = tree_index, leaf_value, evict_index, size_after
  rec.d_priority = None if d_priority is None else d_priority.data_ptr()
  rec.alpha = alpha
  def addr(x):
    if x is None:
      return None
    return x.data_ptr() if isinstance(x, torch.Tensor) else x.ctypes.data
  _lib.call('dz_replay_add', C.byref(view), C.byref(rec), addr(h_s_tm1), addr(h_s_t), _stream())


# ------------------------------------------------------------------------------------------------
# R6: UniformDistribution
# ------------------------------------------------------------------------------------------------


class UniformDistribution:
  """`replay.py:44-117`.  Host swap-remove list + device mirror for in-kernel lookups."""

  def __init__(self, random_state: np.random.RandomState):
    self._random_state = random_state
    self._ids: List[int] = []
    self._id_to_index = {}
    self._mirror = _DeviceList()
    self._pending = []  # (target=2, position, value) patches not yet on the device

  def add(self, ids: Sequence[int]) -> None:
    """`replay.py:52-61`."""
    for i in ids:
      if i in self._id_to_index:
        raise IndexError('Cannot add ID %d, it already exists.' % i)
    for i in ids:
      self._id_to_index[i] = len(self._ids)
      self._pending.append((2, len(self._ids), i))
      self._ids.append(i)

  def remove(self, ids: Sequence[int]) -> None:
    """`replay.py:63-74`."""
    for i in ids:
      if i not in self._id_to_index:
        raise IndexError('Cannot remove ID %d, it does not exist.' % i)
    for i in ids:
      hole = self._id_to_index.pop(i)
      tail = self._ids.pop()
      if tail != i:
        self._ids[hole] = tail
        self._id_to_index[tail] = hole
        self._pending.append((2, hole, tail))

  def take_patches(self):
    p, self._pending = self._pending, []
    self._mirror.ensure(len(self._ids))
    return p

  def flush(self, view=None):
    """Pushes pending patches to the device mirror."""
    patches = self.take_patches()
    if not patches:
      return
    if len(patches) > 16:
      self._mirror.upload(self._ids)
      return
    v = view if view is not None else self.device_view()
    for k in range(0, len(patches), 4):
      _apply_index_record(v, patches[k:k + 4])

  def device_view(self):
    v = _lib.ReplayView()
    v.capacity = 1
    v.d_ids = _ptr(self._mirror.t)
    # dz_replay_add also writes the row scalars; give it a scratch row.
    if not hasattr(self, '_scratch'):
      self._scratch = torch.zeros(8, dtype=torch.float64, device=self._mirror.t.device)
    v.d_action, v.d_reward, v.d_discount, v.d_obs = (_ptr(self._scratch),) * 4
    return v

  def sample(self, size: int) -> np.ndarray:
    """`replay.py:76-82`: host randint draw, device lookup (uniform_sample_kernel)."""
    picks = self._random_state.randint(self.size, size=size).astype(np.int64)
    self.flush()
    dev = self._mirror.t.device
    d_pos = torch.as_tensor(picks, device=dev)
    out_i = torch.empty(2 * size, dtype=torch.int64, device=dev)
    sin = _lib.SampleInputs(_ptr(d_pos), None, None, None)
    sout = _lib.SampleOutputs(out_i.data_ptr(), None, out_i.data_ptr() + 8 * size, None, None)
    v = self.device_view()
    _lib.call('dz_replay_sample', C.byref(v), 0, C.byref(sin), C.byref(sout), size, _stream())
    return out_i[:size].cpu().numpy()

  def ids(self) -> Iterable[int]:
    return self._id_to_index.keys()

  @property
  def size(self) -> int:
    return len(self._ids)

  @property
  def device_ids(self):
    return self._mirror.t

  def get_state(self) -> Mapping[str, Any]:
    """`replay.py:93-98`."""
    return {'ids': self._ids, 'id_to_index': self._id_to_index}

  def set_state(self, state: Mapping[str, Any]) -> None:
    """`replay.py:100-103`."""
    self._ids = state['ids']
    self._id_to_index = state['id_to_index']
    self._pending = []
    self._mirror.upload(self._ids)

  def check_valid(self) -> Tuple[bool, str]:
    """`replay.py:105-117` plus: the device mirror equals the host list."""
    if len(self._ids) != len(self._id_to_index):
      return False, 'ids and id_to_index should be the same size.'
    if len(set(self._ids)) != len(self._ids):
      return False, 'IDs should be unique.'
    for pos, i in enumerate(self._ids):
      if self._id_to_index.get(i) != pos:
        return False, 'ID %d should map to itself.' % i
    self.flush()
    if self._ids and self._mirror.t[:len(self._ids)].cpu().tolist() != list(self._ids):
      return False, 'device mirror of ids is stale.'
    return True, ''


# ------------------------------------------------------------------------------------------------
# R2: PrioritizedDistribution
# ------------------------------------------------------------------------------------------------


class PrioritizedDistribution:
  """`replay.py:429-651`: host id/index bookkeeping, device sum tree and sampling."""

  def __init__(self, priority_exponent: float, uniform_sample_probability: float,
               random_state: np.random.RandomState, min_capacity: int = 0, max_capacity: Optional[int] = None):
    if priority_exponent < 0.0:
      raise ValueError('Require priority_exponent >= 0.')
    if not 0.0 <= uniform_sample_probability <= 1.0:
      raise ValueError('Require 0 <= uniform_sample_probability <= 1.')
    if max_capacity is not None and max_capacity < min_capacity:
      raise ValueError('Require max_capacity >= min_capacity.')
    if min_capacity < 0:
      raise ValueError('Require min_capacity >= 0.')
    self._priority_exponent = priority_exponent
    self._uniform_sample_probability = uniform_sample_probability
    self._max_capacity = max_capacity
    self._random_state = random_state
    self._sum_tree = SumTree()
    self._sum_tree.resize(min_capacity)
    self._id_to_index = {}
    self._index_to_id = {}
    self._inactive_indices = list(range(min_capacity))
    self._active_indices: List[int] = []
    self._active_indices_location = {}
    self._live_dev = _DeviceList(min_capacity)     # mirror of _active_indices
    self._id_at_dev = _DeviceList(min_capacity)    # mirror of _index_to_id (dense by tree index)
    self._pending = []                             # (target, position, value): 0 = live, 1 = id_at
    self._stage = None

  # -- capacity ----------------------------------------------------------------------------------
  def ensure_capacity(self, capacity: int) -> None:
    """`replay.py:463-473`."""
    if self._max_capacity is not None and capacity > self._max_capacity:
      raise ValueError('capacity %d cannot exceed max_capacity %d' % (capacity, self._max_capacity))
    if capacity <= self._sum_tree.size:
      return
    self._inactive_indices.extend(range(self._sum_tree.size, capacity))
    self._sum_tree.resize(capacity)
    self._live_dev.ensure(capacity)
    self._id_at_dev.ensure(capacity)

  # -- host bookkeeping (no device work) -----------------------------------------------------------
  def _host_add(self, ids):
    for i in ids:
      if i in self._id_to_index:
        raise IndexError('ID %d already exists.' % i)
    new_size = self.size + len(ids)
    if self._max_capacity is not None and new_size > self._max_capacity:
      raise ValueError('Cannot add IDs as max capacity would be exceeded.')
    if new_size > self.capacity:
      grown = max(new_size, 2 * self.capacity)
      if self._max_capacity is not None:
        grown = min(self._max_capacity, grown)
      self.ensure_capacity(grown)
    got = []
    for i in ids:
      idx = self._inactive_indices.pop()          # allocation pops from the END (`replay.py:499`)
      pos = len(self._active_indices)
      self._active_indices_location[idx] = pos
      self._active_indices.append(idx)
      self._id_to_index[i] = idx
      self._index_to_id[idx] = i
      self._pending.append((0, pos, idx))
      self._pending.append((1, idx, i))
      got.append(idx)
    return got

  def _host_remove(self, ids):
    gone = [self._id_to_index[i] for i in ids]
    for i, idx in zip(ids, gone):
      del self._id_to_index[i]
      del self._index_to_id[idx]
      hole = self._active_indices_location.pop(idx)
      tail = self._active_indices.pop()
      if tail != idx:                             # swap-remove (`replay.py:519-531`)
        self._active_indices[hole] = tail
        self._active_indices_location[tail] = hole
        self._pending.append((0, hole, tail))
    self._inactive_indices.extend(gone)
    return gone

  def take_patches(self):
    p, self._pending = self._pending, []
    return p

  def device_view(self):
    v = _lib.ReplayView()
    v.capacity = 1
    v.d_tree = _ptr(self._sum_tree.device_nodes)
    v.first_leaf = self._sum_tree.capacity
    v.d_live = _ptr(self._live_dev.t)
    v.d_id_at = _ptr(self._id_at_dev.t)
    v.d_flags = _ptr(self._sum_tree._flags)
    if not hasattr(self, '_scratch'):
      self._scratch = torch.zeros(8, dtype=torch.float64, device=self._live_dev.t.device)
    v.d_action, v.d_reward, v.d_discount, v.d_obs = (_ptr(self._scratch),) * 4
    return v

  def flush(self):
    patches = self.take_patches()
    if not patches:
      return
    if len(patches) > 32:
      self._live_dev.upload(self._active_indices)
      dense = np.zeros(max(self._sum_tree.size, 1), dtype=np.int64)
      if self._index_to_id:
        k = np.fromiter(self._index_to_id.keys(), dtype=np.int64, count=len(self._index_to_id))
        dense[k] = np.fromiter(self._index_to_id.values(), dtype=np.int64, count=len(self._index_to_id))
      self._id_at_dev.upload(dense)
      return
    v = self.device_view()
    for k in range(0, len(patches), 4):
      _apply_index_record(v, patches[k:k + 4])

  # -- reference surface ---------------------------------------------------------------------------
  def add_priorities(self, ids: Sequence[int], priorities: Sequence[float]) -> None:
    """`replay.py:475-507`."""
    got = self._host_add(ids)
    self.flush()
    self._sum_tree.set(got, _power(priorities, self._priority_exponent))

  def remove_priorities(self, ids: Sequence[int]) -> None:
    """`replay.py:509-534`."""
    gone = self._host_remove(ids)
    self.flush()
    self._sum_tree.set(gone, np.zeros((len(gone),), dtype=np.float64))

  def update_priorities(self, ids: Sequence[int], priorities: Sequence[float]) -> None:
    """`replay.py:536-545`.  float32 priorities (what comes back from the learner) are
    exponentiated on the device in float32 as the reference's numpy does; other dtypes take the
    reference's float64 host `_power` and only the tree update runs on the device."""
    where = []
    for i in ids:
      if i not in self._id_to_index:
        raise IndexError('ID %d does not exist.' % i)
      where.append(self._id_to_index[i])
    pri = np.asarray(priorities)
    if pri.dtype == np.float32:
      if not np.isfinite(pri).all() or (pri < 0.0).any():
        raise ValueError('value must be finite and positive.')
      dev = self._live_dev.t.device
      self.update_priorities_device(torch.as_tensor(np.asarray(where, dtype=np.int64), device=dev),
                                    torch.as_tensor(pri.reshape(-1), device=dev))
    else:
      self._sum_tree.set(where, _power(pri, self._priority_exponent))

  def update_priorities_device(self, d_indices: torch.Tensor, d_priorities: torch.Tensor) -> None:
    """Priority write-back with device-resident tree indices (int64) and float32 priorities."""
    v = self.device_view()
    _lib.call('dz_replay_update_priorities', C.byref(v), _ptr(d_indices), _ptr(d_priorities), d_indices.numel(),
              float(self._priority_exponent), self._sum_tree.size, _stream())

  def _draw(self, size):
    """The three host draws of `replay.py:551-567`, in order; needs root (one 8-byte D2H)."""
    pos = self._random_state.randint(self.size, size=size).astype(np.int64)
    root = self._sum_tree.root()
    u_tree = self._random_state.uniform(size=size) if root != 0.0 else np.zeros(size)
    u_mix = self._random_state.uniform(size=size)
    return pos, u_tree, u_mix

  def sample_device(self, size, beta=1.0, normalize=False, capacity_for_slots=1):
    """Runs the sampling kernel; returns device tensors (ids, indices, slots, probs, weights)."""
    if self.size == 0:
      raise RuntimeError('No IDs to sample.')
    self.flush()
    pos, u_tree, u_mix = self._draw(size)
    dev = self._live_dev.t.device
    out_i = torch.empty(3 * size, dtype=torch.int64, device=dev)
    out_f = torch.empty(2 * size, dtype=torch.float64, device=dev)
    v = self.device_view()
    v.capacity = capacity_for_slots
    chunk = 1024  # the kernel normalises over one block; larger requests run in chunks, normalised below
    big = size > chunk
    for lo in range(0, size, chunk):
      n = min(chunk, size - lo)
      host = np.concatenate([u_tree[lo:lo + n], u_mix[lo:lo + n],
                             [float(self.size), float(beta), float(self._uniform_sample_probability),
                              1.0 if (normalize and not big) else 0.0]])
      d_f = torch.as_tensor(host, device=dev)
      d_pos = torch.as_tensor(pos[lo:lo + n], device=dev)
      sin = _lib.SampleInputs(_ptr(d_pos), d_f.data_ptr(), d_f.data_ptr() + 8 * n, d_f.data_ptr() + 16 * n)
      ip, fp = out_i.data_ptr() + 8 * lo, out_f.data_ptr() + 8 * lo
      sout = _lib.SampleOutputs(ip, ip + 8 * size, ip + 16 * size, fp, fp + 8 * size)
      _lib.call('dz_replay_sample', C.byref(v), 1, C.byref(sin), C.byref(sout), n, _stream())
    if big and normalize:
      out_f[size:] /= out_f[size:].max()
    return out_i[:size], out_i[size:2 * size], out_i[2 * size:], out_f[:size], out_f[size:]

  def sample(self, size: int) -> Tuple[np.ndarray, np.ndarray]:
    """`replay.py:547-583`."""
    ids, _, _, probs, _ = self.sample_device(size)
    self._sum_tree._raise_flags()
    return ids.cpu().numpy(), probs.cpu().numpy()

  def get_exponentiated_priorities(self, ids: Sequence[int]) -> Sequence[float]:
    """`replay.py:585-590`."""
    return self._sum_tree.get(np.fromiter((self._id_to_index[i] for i in ids), dtype=np.int64, count=len(ids)))

  def ids(self) -> Iterable[int]:
    return self._id_to_index.keys()

  @property
  def capacity(self) -> int:
    return self._sum_tree.size

  @property
  def size(self) -> int:
    return len(self._id_to_index)

  def get_state(self) -> Mapping[str, Any]:
    """`replay.py:606-615` (same keys)."""
    return {
        'sum_tree': self._sum_tree.get_state(),
        'id_to_index': self._id_to_index,
        'index_to_id': self._index_to_id,
        'inactive_indices': self._inactive_indices,
        'active_indices': self._active_indices,
        'active_indices_location': self._active_indices_location,
    }

  def set_state(self, state: Mapping[str, Any]) -> None:
    """`replay.py:617-624`."""
    self._sum_tree.set_state(state['sum_tree'])
    self._id_to_index = state['id_to_index']
    self._index_to_id = state['index_to_id']
    self._inactive_indices = state['inactive_indices']
    self._active_indices = state['active_indices']
    self._active_indices_location = state['active_indices_location']
    self._live_dev.ensure(self._sum_tree.size)
    self._id_at_dev.ensure(self._sum_tree.size)
    self._pending = [(0, 0, 0)] * 64  # forces a full re-upload of both mirrors
    self.flush()

  def check_valid(self) -> Tuple[bool, str]:
    """`replay.py:626-651`, plus the device mirrors agree with the host lists."""
    if len(self._id_to_index) != len(self._index_to_id):
      return False, 'ID to index maps are not the same size.'
    for i, idx in self._id_to_index.items():
      if self._index_to_id.get(idx) != i:
        return False, 'ID %d should map to itself.' % i
    if len(set(self._inactive_indices)) != len(self._inactive_indices):
      return False, 'Inactive indices should be unique.'
    if len(set(self._active_indices)) != len(self._active_indices):
      return False, 'Active indices should be unique.'
    if set(self._active_indices) != set(self._index_to_id.keys()):
      return False, 'Active indices should match index to ID mapping keys.'
    if sorted(self._inactive_indices + self._active_indices) != list(range(self._sum_tree.size)):
      return False, 'Inactive and active indices should partition all indices.'
    for pos, idx in enumerate(self._active_indices):
      if self._active_indices_location.get(idx) != pos:
        return False, 'Active index location %d not correct for index %d.' % (pos, idx)
    self.flush()
    n = len(self._active_indices)
    if n and self._live_dev.t[:n].cpu().tolist() != list(self._active_indices):
      return False, 'device mirror of active indices is stale.'
    if n:
      id_at = self._id_at_dev.t.cpu().numpy()
      for idx, i in self._index_to_id.items():
        if id_at[idx] != i:
          return False, 'device mirror of index_to_id is stale at %d.' % idx
    return self._sum_tree.check_valid()


# ------------------------------------------------------------------------------------------------
# Transition storage in HBM
# ------------------------------------------------------------------------------------------------


class _TransitionStore:
  """Row = id % capacity; each row holds s_tm1 | s_t (uint8, stride padded to 16 B)."""

  def __init__(self, capacity):
    self.capacity = capacity
    self.obs = None
    self.obs_shape = None
    self.obs_dtype = None
    dev = _device()
    n = max(capacity, 1)
    self.action = torch.zeros(n, dtype=torch.int32, device=dev)
    self.reward = torch.zeros(n, dtype=torch.float64, device=dev)
    self.discount = torch.zeros(n, dtype=torch.float64, device=dev)
    self.flags = torch.zeros(1, dtype=torch.int32, device=dev)
    self.obs_bytes = 0
    self.obs_stride = 0

  def allocate(self, obs_shape, obs_dtype=np.uint8):
    if self.obs is not None:
      return
    self.obs_shape, self.obs_dtype = tuple(obs_shape), np.dtype(obs_dtype)
    self.obs_bytes = int(np.prod(obs_shape)) * self.obs_dtype.itemsize
    self.obs_stride = (self.obs_bytes + 15) // 16 * 16
    self.obs = torch.empty((max(self.capacity, 1), 2, self.obs_stride), dtype=torch.uint8, device=self.action.device)

  def fill_view(self, v):
    v.d_obs, v.d_action, v.d_reward, v.d_discount = _ptr(self.obs), _ptr(self.action), _ptr(self.reward), _ptr(self.discount)
    v.capacity, v.obs_bytes, v.obs_stride = self.capacity, self.obs_bytes, self.obs_stride
    v.d_flags = _ptr(self.flags)
    return v

  def reserve_batch(self, batch_size):
    """Staging for the fused learner's batch (the frame store assembles stacks there); rows are read in place here."""

  def check_flags(self, flags):
    """Raises if the storage could not keep an added transition (the frame store's pool overflow)."""

  def reset(self):
    """Forgets the insert history before set_state() rewrites the rows."""

  @property
  def device_bytes(self):
    """Bytes of device memory this store holds."""
    return sum(t.numel() * t.element_size() for t in vars(self).values() if isinstance(t, torch.Tensor))

  def gather(self, d_slots, size):
    """`np.stack` of `get(ids)` (`replay.py:718-722`) on the device; returns device tensors."""
    dev = self.action.device
    s_tm1 = torch.empty((size, self.obs_bytes), dtype=torch.uint8, device=dev)
    s_t = torch.empty((size, self.obs_bytes), dtype=torch.uint8, device=dev)
    a = torch.empty(size, dtype=torch.int64, device=dev)
    r = torch.empty(size, dtype=torch.float64, device=dev)
    d = torch.empty(size, dtype=torch.float64, device=dev)
    v = self.fill_view(_lib.ReplayView())
    _lib.call('dz_replay_gather', C.byref(v), _ptr(d_slots), size, _ptr(s_tm1), _ptr(s_t), _ptr(a), _ptr(r), _ptr(d),
              _stream())
    return s_tm1, a, r, d, s_t

  def get_rows(self, structure, slots, chunk=4096):
    """`[storage[i] for i in ids]` (`replay.py:153-156`): rows are gathered on the device and copied to the host in
    chunks, so the staging memory is bounded (2 * chunk * obs_bytes) whatever the number of rows — `get_state()` of a
    full 1M-capacity replay goes through here."""
    out = []
    dev = self.action.device
    for lo in range(0, len(slots), chunk):
      part = np.ascontiguousarray(slots[lo:lo + chunk])
      tr = self.to_host_transition(structure, self.gather(torch.as_tensor(part, device=dev), len(part)))
      out.extend(type(structure)(*[f[k] for f in tr]) for k in range(len(part)))
    return out

  def to_host_transition(self, structure, tensors):
    s_tm1, a, r, d, s_t = [t.cpu().numpy() for t in tensors]
    shape = (len(a),) + self.obs_shape
    return type(structure)(s_tm1.view(self.obs_dtype).reshape(shape), a, r, d, s_t.view(self.obs_dtype).reshape(shape))


class _FrameStore(_TransitionStore):
  """Frame-deduplicated storage (DESIGN.md §3): observations are uint8 (H, W, S) stacks, every distinct (H, W) frame is
  kept once in a ring of `frame_capacity` slots, and row = id % capacity holds the 2S frame slots of s_tm1 | s_t.  The
  insert rule (include/dqn_zoo_b200.h, dz_frame_store) runs on the device in dz_replay_add; `gather` assembles the stacks
  on the device, so everything returned is byte-identical to `_TransitionStore` after the same adds."""

  def __init__(self, capacity, frame_capacity):
    if int(frame_capacity) < 1:
      raise ValueError('frame_capacity must be a positive integer, got %r' % (frame_capacity,))
    super().__init__(capacity)
    self.frame_capacity = int(frame_capacity)
    self.batch_capacity = 0
    self.batch_stage = None
    self.state = None

  def allocate(self, obs_shape, obs_dtype=np.uint8):
    if self.obs_shape is not None:
      return
    shape, dtype = tuple(obs_shape), np.dtype(obs_dtype)
    if len(shape) != 3 or dtype != np.uint8 or min(shape) < 1 or shape[2] > _lib.DZ_FRAME_MAX_STACK:
      raise ValueError('frame store needs uint8 observations of shape (H, W, S) with S <= %d: %s %s'
                       % (_lib.DZ_FRAME_MAX_STACK, shape, dtype))
    if 2 * shape[2] * ((shape[0] * shape[1] + 15) // 16 * 16) > _lib.DZ_FRAME_MAX_STAGE_BYTES:
      raise ValueError('frame store needs 2 * S * (H * W rounded up to 16) <= %d bytes: %s %s'
                       % (_lib.DZ_FRAME_MAX_STAGE_BYTES, shape, dtype))
    self.obs_shape, self.obs_dtype = shape, dtype
    self.obs_bytes = int(np.prod(shape))
    self.obs_stride = (self.obs_bytes + 15) // 16 * 16
    h, w, self.stack = shape
    self.frame_bytes = h * w
    self.frame_stride = (self.frame_bytes + 15) // 16 * 16
    dev, F, P = self.action.device, self.frame_capacity, 2 * self.stack
    self.frames = torch.empty((F + 1, self.frame_stride), dtype=torch.uint8, device=dev)
    self.frames[0].zero_()                              # slot 0: the zero frame of the padded stacks
    self.row_frames = torch.zeros((max(self.capacity, 1), P), dtype=torch.int32, device=dev)
    self.frame_hash = torch.zeros(F + 1, dtype=torch.int64, device=dev)   # uint64 bit patterns
    self.frame_born = torch.full((F + 1,), -1, dtype=torch.int64, device=dev)
    self.frame_last_ref = torch.full((F + 1,), -1, dtype=torch.int64, device=dev)
    self.state = torch.empty(2 + _lib.DZ_FRAME_WINDOW * (1 + P), dtype=torch.int64, device=dev)
    self.add_stage = torch.zeros((2, self.obs_stride), dtype=torch.uint8, device=dev)
    self.reset()
    self._allocate_batch_stage()

  def _allocate_batch_stage(self):
    if self.obs_shape is not None and self.batch_capacity:
      self.batch_stage = torch.zeros((2, self.batch_capacity, self.obs_stride), dtype=torch.uint8,
                                     device=self.action.device)

  def reserve_batch(self, batch_size):
    """The fused learner assembles each sampled batch into [2][batch_capacity][obs_stride] staging rows; the address
    stays fixed once reserved, so captured CUDA graphs remain valid."""
    if batch_size > self.batch_capacity:
      self.batch_capacity = int(batch_size)
      self._allocate_batch_stage()

  def reset(self):
    if self.state is not None:
      self.state.fill_(-1)
      self.state[:2] = 0

  def check_flags(self, flags):
    f = int(flags.item())
    if f & _lib.DZ_FLAG_FRAME_POOL_FULL:
      flags.fill_(f & ~_lib.DZ_FLAG_FRAME_POOL_FULL)
      raise RuntimeError(_POOL_FULL_MESSAGE)

  def fill_view(self, v):
    super().fill_view(v)
    if self.obs_shape is None:
      return v
    fs = v.frames
    fs.d_frames, fs.d_row_frames = _ptr(self.frames), _ptr(self.row_frames)
    fs.d_frame_hash, fs.d_frame_born, fs.d_frame_last_ref = (_ptr(self.frame_hash), _ptr(self.frame_born),
                                                              _ptr(self.frame_last_ref))
    fs.d_state, fs.d_add_stage, fs.d_batch_stage = _ptr(self.state), _ptr(self.add_stage), _ptr(self.batch_stage)
    fs.num_frames, fs.frame_bytes, fs.frame_stride = self.frame_capacity, self.frame_bytes, self.frame_stride
    fs.stack, fs.batch_capacity = self.stack, self.batch_capacity
    return v

  def fill_synthetic(self, n, seed, num_actions, discount, episode_length):
    v = self.fill_view(_lib.ReplayView())
    _lib.call('dz_replay_fill_synthetic_frames', C.byref(v), n, int(episode_length), int(seed), int(num_actions),
              float(discount), _stream())


def _make_store(capacity, frame_capacity):
  return _TransitionStore(capacity) if frame_capacity is None else _FrameStore(capacity, frame_capacity)


def _host_obs(x, store):
  """Flat uint8 view of an observation to be written into a replay row.  Host arrays are copied H2D by
  dz_replay_add; CUDA tensors (e.g. the frame stack of `processors.atari(device_observations=True)`) are copied
  device-to-device on the same stream — the device-resident insert path, no host round trip."""
  if isinstance(x, torch.Tensor) and x.is_cuda:
    t = x.contiguous()
    dtype = np.dtype(str(t.dtype).replace('torch.', ''))
    store.allocate(tuple(t.shape), dtype)
    if tuple(t.shape) != store.obs_shape or dtype != store.obs_dtype:
      raise ValueError('observation shape/dtype changed: %s %s' % (tuple(t.shape), dtype))
    return t.view(torch.uint8).reshape(-1)
  arr = np.ascontiguousarray(x)
  store.allocate(arr.shape, arr.dtype)
  if arr.shape != store.obs_shape or arr.dtype != store.obs_dtype:
    raise ValueError('observation shape/dtype changed: %s %s' % (arr.shape, arr.dtype))
  return arr.view(np.uint8).reshape(-1)


def _check_codec(encoder, decoder):
  """The reference stores `encoder(item)` and returns `decoder(stored)` (`replay.py:148,155`; every run_atari.py passes
  the snappy pair of `replay.py:895-904` so that 1M x 56 KB fits in host RAM).  HBM holds raw observations, so a codec
  pair is accepted and applied as the round trip `decoder(encoder(item))` on the host at insert time — the identity
  for a lossless codec such as snappy — and both must be given together."""
  if (encoder is None) != (decoder is None):
    raise ValueError('encoder and decoder must be given together')
  if encoder is None:
    return None
  return lambda item: decoder(encoder(item))


# ------------------------------------------------------------------------------------------------
# R6: TransitionReplay
# ------------------------------------------------------------------------------------------------


class TransitionReplay:
  """Uniform replay with oldest-out eviction (`replay.py:120-200`), storage in HBM."""

  def __init__(self, capacity: int, structure, random_state: np.random.RandomState, encoder=None, decoder=None, *,
               frame_capacity: Optional[int] = None):
    """`frame_capacity=F` stores every distinct frame of the (H, W, S) uint8 observation stacks once, in F slots
    (`_FrameStore`); None keeps two full stacks per transition."""
    self._codec = _check_codec(encoder, decoder)
    self._capacity = capacity
    self._structure = structure
    self._random_state = random_state
    self._distribution = UniformDistribution(random_state=random_state)
    self._distribution._mirror.ensure(capacity)   # fixed address: captured CUDA graphs keep pointing at it
    self._store = _make_store(capacity, frame_capacity)
    self._live_ids = collections.deque()   # ids currently stored, oldest first (keys of the OrderedDict)
    self._t = 0

  def device_view(self):
    v = self._store.fill_view(_lib.ReplayView())
    v.d_ids = _ptr(self._distribution.device_ids)
    return v

  def add(self, item) -> None:
    """`replay.py:142-151`."""
    if self._codec is not None:
      item = self._codec(item)
    s_tm1 = _host_obs(item[0], self._store)
    s_t = _host_obs(item[4], self._store)
    if self.size == self._capacity:
      self._distribution.remove([self._live_ids.popleft()])
    item_id = self._t
    self._distribution.add([item_id])
    patches = self._distribution.take_patches()
    v = self.device_view()
    first = patches[:4]
    _apply_index_record(v, first, slot=item_id % self._capacity, action=int(item[1]), reward=float(item[2]),
                        discount=float(item[3]), h_s_tm1=s_tm1, h_s_t=s_t, item_id=item_id,
                        oldest_live=self._live_ids[0] if self._live_ids else item_id)
    assert len(patches) <= 4
    self._live_ids.append(item_id)
    self._t += 1

  def get(self, ids: Sequence[int]):
    """`replay.py:153-156`."""
    ids = [int(i) for i in ids]
    for i in ids:
      if not self._live_ids or not (self._live_ids[0] <= i <= self._live_ids[-1]):
        raise KeyError(i)
    self._store.check_flags(self._store.flags)
    return self._store.get_rows(self._structure, np.asarray(ids, dtype=np.int64) % self._capacity)

  def sample_device(self, size: int):
    """Host randint draw (`replay.py:78`), device id lookup + gather; returns device tensors."""
    picks = self._random_state.randint(self.size, size=size).astype(np.int64)
    dev = self._store.action.device
    d_pos = torch.as_tensor(picks, device=dev)
    out_i = torch.empty(2 * size, dtype=torch.int64, device=dev)
    sin = _lib.SampleInputs(_ptr(d_pos), None, None, None)
    sout = _lib.SampleOutputs(out_i.data_ptr(), None, out_i.data_ptr() + 8 * size, None, None)
    v = self.device_view()
    _lib.call('dz_replay_sample', C.byref(v), 0, C.byref(sin), C.byref(sout), size, _stream())
    return out_i[:size], out_i[size:], self._store.gather(out_i[size:], size)

  def sample(self, size: int):
    """`replay.py:158-165`."""
    _, _, tensors = self.sample_device(size)
    self._store.check_flags(self._store.flags)
    return self._store.to_host_transition(self._structure, tensors)

  def ids(self) -> Iterable[int]:
    return list(self._live_ids)

  @property
  def size(self) -> int:
    return len(self._live_ids)

  @property
  def capacity(self) -> int:
    return self._capacity

  def reserve_batch(self, batch_size: int) -> None:
    """Reserves the storage's staging for fused learner batches of up to `batch_size` (the agent calls it)."""
    self._store.reserve_batch(batch_size)

  def get_state(self) -> Mapping[str, Any]:
    """`replay.py:179-187`: same keys; `storage` is a list of (id, Transition) with host arrays."""
    ids = list(self._live_ids)
    return {'storage': list(zip(ids, self.get(ids))) if ids else [], 't': self._t,
            'distribution': self._distribution.get_state()}

  def _flags(self):
    return self._store.flags

  def set_state(self, state: Mapping[str, Any]) -> None:
    """`replay.py:189-193`."""
    _restore_rows(self, state['storage'])
    self._t = state['t']
    self._distribution.set_state(state['distribution'])

  def check_valid(self) -> Tuple[bool, str]:
    """`replay.py:195-200`."""
    self._store.check_flags(self._flags())
    if self._t < self.size:
      return False, 't should be >= storage size.'
    if set(self._live_ids) != set(self._distribution.ids()):
      return False, 'IDs in storage and distribution do not match.'
    return self._distribution.check_valid()


def _restore_rows(rep, storage):
  """Rewrites device rows from a `storage` list of (id, item) (set_state)."""
  rep._live_ids = collections.deque(int(i) for i, _ in storage)
  rep._store.reset()
  v = None
  for i, item in storage:
    s_tm1 = _host_obs(item[0], rep._store)
    s_t = _host_obs(item[4], rep._store)
    if v is None:
      v = rep.device_view()
    _apply_index_record(v, [], slot=int(i) % rep._capacity, action=int(item[1]), reward=float(item[2]),
                        discount=float(item[3]), h_s_tm1=s_tm1, h_s_t=s_t, item_id=int(i), oldest_live=rep._live_ids[0])


# ------------------------------------------------------------------------------------------------
# R5: PrioritizedTransitionReplay
# ------------------------------------------------------------------------------------------------


class PrioritizedTransitionReplay:
  """Proportional prioritized replay (`replay.py:654-768`), storage + sum tree in HBM."""

  def __init__(self, capacity: int, structure, priority_exponent: float,
               importance_sampling_exponent: Callable[[int], float], uniform_sample_probability: float,
               normalize_weights: bool, random_state: np.random.RandomState, encoder=None, decoder=None, *,
               frame_capacity: Optional[int] = None):
    """`frame_capacity`: as for `TransitionReplay`."""
    self._codec = _check_codec(encoder, decoder)
    self._capacity = capacity
    self._structure = structure
    self._random_state = random_state
    self._distribution = PrioritizedDistribution(
        min_capacity=capacity, max_capacity=capacity, priority_exponent=priority_exponent,
        uniform_sample_probability=uniform_sample_probability, random_state=random_state)
    self._importance_sampling_exponent = importance_sampling_exponent
    self._normalize_weights = normalize_weights
    self._store = _make_store(capacity, frame_capacity)
    self._live_ids = collections.deque()
    self._t = 0

  def device_view(self):
    v = self._distribution.device_view()
    self._store.fill_view(v)
    v.d_flags = _ptr(self._distribution._sum_tree._flags)
    return v

  def add(self, item, priority: float) -> None:
    """`replay.py:690-699`: one device call carries the row, the list patches, the evicted
    leaf's zeroing and the new leaf (= priority**alpha evaluated in float64 on the host, as
    `replay.py:507` does)."""
    if self._codec is not None:
      item = self._codec(item)
    s_tm1 = _host_obs(item[0], self._store)
    s_t = _host_obs(item[4], self._store)
    dist = self._distribution
    alpha = dist._priority_exponent
    d_priority = None
    if isinstance(priority, torch.Tensor):
      # priority kept on the device by the agent (max_seen_priority); exact for alpha in {0.5, 1}
      if alpha in (0.5, 1.0):
        d_priority, priority = priority, 1.0
      else:
        priority = float(priority.item())
    leaf = np.asarray(_power([priority], alpha))
    if not np.isfinite(leaf).all() or (leaf < 0.0).any():
      raise ValueError('value must be finite and positive.')
    evicted = -1
    if self.size == self._capacity:
      (evicted,) = dist._host_remove([self._live_ids.popleft()])
    item_id = self._t
    (idx,) = dist._host_add([item_id])
    patches = dist.take_patches()
    v = self.device_view()
    _apply_index_record(v, patches[:4], tree_index=idx, leaf_value=float(leaf[0]), evict_index=evicted,
                        size_after=dist._sum_tree.size, slot=item_id % self._capacity, action=int(item[1]),
                        reward=float(item[2]), discount=float(item[3]), h_s_tm1=s_tm1, h_s_t=s_t,
                        d_priority=d_priority, alpha=float(alpha), item_id=item_id,
                        oldest_live=self._live_ids[0] if self._live_ids else item_id)
    assert len(patches) <= 4
    self._live_ids.append(item_id)
    self._t += 1

  def get(self, ids: Sequence[int]):
    ids = [int(i) for i in ids]
    for i in ids:
      if i not in self._distribution._id_to_index:
        raise KeyError(i)
    self._store.check_flags(self._flags())
    return self._store.get_rows(self._structure, np.asarray(ids, dtype=np.int64) % self._capacity)

  def sample_device(self, size: int):
    """Sampling + gather, everything left on the device: (ids, indices, slots, probs, weights, batch)."""
    beta = self.importance_sampling_exponent
    if not 0.0 <= beta <= 1.0:
      raise ValueError('Require 0 <= exponent <= 1.')
    ids, indices, slots, probs, weights = self._distribution.sample_device(
        size, beta=beta, normalize=self._normalize_weights, capacity_for_slots=self._capacity)
    return ids, indices, slots, probs, weights, self._store.gather(slots, size)

  def sample(self, size: int):
    """`replay.py:701-723`: (Transition of stacked arrays, ids int64, weights float64)."""
    ids, _, _, _, weights, tensors = self.sample_device(size)
    tr = self._store.to_host_transition(self._structure, tensors)
    w = weights.cpu().numpy()
    self._store.check_flags(self._flags())
    self._distribution._sum_tree._raise_flags()
    if not np.isfinite(w).all():
      raise ValueError('Weights are not finite: %s.' % w)
    return tr, ids.cpu().numpy(), w

  def update_priorities(self, ids: Sequence[int], priorities: Sequence[float]) -> None:
    """`replay.py:725-730`."""
    self._distribution.update_priorities(ids, np.asarray(priorities))

  @property
  def size(self) -> int:
    return len(self._live_ids)

  @property
  def capacity(self) -> int:
    return self._capacity

  def reserve_batch(self, batch_size: int) -> None:
    """Reserves the storage's staging for fused learner batches of up to `batch_size` (the agent calls it)."""
    self._store.reserve_batch(batch_size)

  def _flags(self):
    return self._distribution._sum_tree._flags

  @property
  def importance_sampling_exponent(self):
    """`replay.py:742-745`."""
    return self._importance_sampling_exponent(self._t)

  def get_state(self) -> Mapping[str, Any]:
    """`replay.py:747-754`."""
    ids = list(self._live_ids)
    return {'storage': list(zip(ids, self.get(ids))) if ids else [], 't': self._t,
            'distribution': self._distribution.get_state()}

  def set_state(self, state: Mapping[str, Any]) -> None:
    """`replay.py:756-760`."""
    _restore_rows(self, state['storage'])
    self._t = state['t']
    self._distribution.set_state(state['distribution'])

  def check_valid(self) -> Tuple[bool, str]:
    """`replay.py:762-768`."""
    self._store.check_flags(self._flags())
    if self._t < self.size:
      return False, 't should be >= storage size.'
    if set(self._live_ids) != set(self._distribution.ids()):
      return False, 'IDs in storage and distribution do not match.'
    return self._distribution.check_valid()


def bulk_fill_synthetic(rep, obs_shape, seed, num_actions, discount=0.99, priority=1.0, episode_length=1000):
  """Benchmark/test helper: brings `rep` (uniform or prioritized, empty) to the exact state it
  has after `capacity` sequential `add()`s of synthetic transitions (ids 0..C-1, priority
  `priority` each) without C host->device copies: contents are generated on the device
  (dz_replay_fill_synthetic, byte-identical to oracle/replay_oracle.py:synthetic_rows) and the
  host bookkeeping is written in closed form (allocation order of replay.py:457,499: id i gets
  tree index C-1-i).

  A frame store gets synthetic EPISODES instead (dz_replay_fill_synthetic_frames): `episode_length` 1-step transitions
  each, a new iid frame per timestep, stacks zero-padded at episode start as processors.atari() pads them; the device
  state equals that of the same sequential adds (oracle/frame_store_oracle.py:synthetic_fill)."""
  assert rep._t == 0 and rep.size == 0
  cap = rep._capacity
  rep._store.allocate(obs_shape, np.uint8)
  if isinstance(rep._store, _FrameStore):
    rep._store.fill_synthetic(cap, seed, num_actions, discount, episode_length)
  else:
    v = rep._store.fill_view(_lib.ReplayView())
    _lib.call('dz_replay_fill_synthetic', C.byref(v), 0, cap, int(seed), int(num_actions), float(discount), _stream())
  rep._live_ids = collections.deque(range(cap))
  rep._t = cap
  dist = rep._distribution
  if isinstance(dist, UniformDistribution):
    dist._ids = list(range(cap))
    dist._id_to_index = {i: i for i in range(cap)}
    dist._pending = []
    dist._mirror.upload(dist._ids)
    return
  idx = np.arange(cap - 1, -1, -1, dtype=np.int64)          # id i -> index C-1-i
  dist._id_to_index = dict(zip(range(cap), idx.tolist()))
  dist._index_to_id = dict(zip(idx.tolist(), range(cap)))
  dist._inactive_indices = []
  dist._active_indices = idx.tolist()
  dist._active_indices_location = dict(zip(idx.tolist(), range(cap)))
  dist._pending = []
  dist._live_dev.upload(idx)
  dist._id_at_dev.upload(idx)                                  # id_at[index] = C-1-index
  leaf = float(_power([priority], dist._priority_exponent)[0])
  dist._sum_tree.set_all(np.full(cap, leaf, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# R7: accumulators (host, insert time)
# ------------------------------------------------------------------------------------------------


def _fold_n_steps(window):
  """`replay.py:808-824`: discounted return and discount product in python floats (f64)."""
  ret, disc = 0.0, 1.0
  for tr in window:
    ret += disc * tr.r_t
    disc *= tr.discount_t
  return Transition(s_tm1=window[0].s_tm1, a_tm1=window[0].a_tm1, r_t=ret, discount_t=disc, s_t=window[-1].s_t)


class NStepTransitionAccumulator:
  """`replay.py:827-892`."""

  def __init__(self, n):
    self._transitions = collections.deque(maxlen=n)
    self.reset()

  def step(self, timestep_t, a_t) -> Iterable[Transition]:
    if timestep_t.first():
      self.reset()
    if self._timestep_tm1 is None:
      if not timestep_t.first():
        raise ValueError('Expected FIRST timestep, got %s.' % str(timestep_t))
      self._timestep_tm1, self._a_tm1 = timestep_t, a_t
      return []
    self._transitions.append(Transition(s_tm1=self._timestep_tm1.observation, a_tm1=self._a_tm1,
                                        r_t=timestep_t.reward, discount_t=timestep_t.discount,
                                        s_t=timestep_t.observation))
    self._timestep_tm1, self._a_tm1 = timestep_t, a_t
    out = []
    if timestep_t.last():
      while self._transitions:
        out.append(_fold_n_steps(list(self._transitions)))
        self._transitions.popleft()
    elif len(self._transitions) == self._transitions.maxlen:
      out.append(_fold_n_steps(list(self._transitions)))
    return out

  def reset(self) -> None:
    self._transitions.clear()
    self._timestep_tm1 = None
    self._a_tm1 = None


class TransitionAccumulator(NStepTransitionAccumulator):
  """`replay.py:771-805` (the n = 1 case; equivalence pinned by `replay_test.py:264-280`)."""

  def __init__(self):
    super().__init__(1)
