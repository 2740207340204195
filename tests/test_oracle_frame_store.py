"""CPU: the numpy restatement of the frame-deduplicated replay storage (oracle/frame_store_oracle.py) — round trips,
frame counts on Atari-like streams, ring reclaim and overflow, the closed-form synthetic fill — and the host-compiled
frame hash of csrc/dz_frames.cu against the numpy hash."""

import ctypes as C

import numpy as np

from oracle import frame_store_oracle as fo
from oracle import processors_oracle as po
from oracle import replay_oracle as ro
from oracle import scenarios


def _iid_stacks(n, shape, seed):
  rs = np.random.RandomState(seed)
  return [(rs.randint(1, 256, size=shape).astype(np.uint8), rs.randint(1, 256, size=shape).astype(np.uint8))
          for _ in range(n)]


def atari_stream(n_step, episodes=3, max_len=40, seed=0, shape=(12, 10), stack=4):
  """(s_tm1, s_t) of the transitions an agent adds: random RGB frames -> the processors.atari() oracle (pool, luma,
  resize, zero-padded stack) -> the n-step accumulator.  Returns the transitions and the distinct non-zero frames."""
  rs = np.random.RandomState(seed)
  proc = po.AtariPreprocessor(resize_shape=shape, num_stacked_frames=stack)
  acc = ro.NStepTransitionAccumulator(n_step)
  out, frames = [], set()
  for _ in range(episodes):
    proc.reset()
    acc.reset()
    length = int(rs.randint(max_len // 2, max_len))
    for t in range(length + 1):
      st = po.FIRST if t == 0 else (po.LAST if t == length else po.MID)
      rgb = rs.randint(0, 256, size=(2 * shape[0], 2 * shape[1], 3)).astype(np.uint8)
      ts = proc(st, None if t == 0 else 1.0, None if t == 0 else 1.0, (rgb, 3))
      if ts is None:
        continue
      obs = ts[3]
      for c in range(stack):
        if obs[:, :, c].any():
          frames.add(obs[:, :, c].tobytes())
      for tr in acc.step(scenarios._TS(ts[0], ts[1], ts[2], obs), 0):
        out.append((tr.s_tm1, tr.s_t))
  return out, frames


def _feed(store, transitions, capacity):
  live = []
  for i, (a, b) in enumerate(transitions):
    live.append(i)
    if len(live) > capacity:
      live.pop(0)
    store.add(i, live[0], a, b)
  return live


def _assert_round_trip(store, transitions, live):
  for i in live:
    a, b = store.get(i)
    np.testing.assert_array_equal(a, transitions[i][0])
    np.testing.assert_array_equal(b, transitions[i][1])


def test_round_trip_iid_stacks_appends_every_plane():
  shape = (6, 4, 4)
  tr = _iid_stacks(50, shape, 1)
  st = fo.FrameStore(20, 20 * 8, shape)
  live = _feed(st, tr, 20)
  _assert_round_trip(st, tr, live)
  assert st.appends == 50 * 8
  assert not st.pool_full


def test_round_trip_and_frame_counts_on_atari_like_streams():
  for n_step in (1, 3):
    tr, frames = atari_stream(n_step, seed=n_step)
    shape = tr[0][0].shape
    st = fo.FrameStore(len(tr), 4 * len(tr), shape)
    appends_per_add = []
    for i, (a, b) in enumerate(tr):
      before = st.appends
      st.add(i, 0, a, b)
      appends_per_add.append(st.appends - before)
      for p, row in zip(fo.planes(a) + fo.planes(b), st.row_frames[i]):
        assert (row == 0) == (not p.any())          # zero planes, and only they, map to slot 0
    _assert_round_trip(st, tr, range(len(tr)))
    assert st.appends == len(frames)
    # steady state inside an episode: exactly one new frame per add
    assert appends_per_add.count(1) >= len(tr) // 2
    assert max(appends_per_add) <= n_step + 1      # the first add of an episode appends s_t's n + 1 frames


def test_slot_is_reclaimed_exactly_when_its_last_reference_is_evicted():
  shape = (4, 4, 2)
  tr = _iid_stacks(12, shape, 2)
  cap = 3
  F = cap * 4
  st = fo.FrameStore(cap, F, shape)
  live = _feed(st, tr[:cap], cap)
  assert st.appends == F and not st.pool_full
  # the ring is full: the next append reuses slot 1, whose last reference is id 0 -> allowed once id 0 is evicted
  assert st.last_ref[1] == 0
  st.add(cap, 0, *tr[cap])                        # id 0 still live: overflow
  assert st.pool_full and st.full_ids == [cap] and (st.row_frames[cap % cap] == -1).all()
  st2 = fo.FrameStore(cap, F, shape)
  live = _feed(st2, tr, cap)
  assert not st2.pool_full
  _assert_round_trip(st2, tr, live)


def test_overflow_is_predicted_at_the_smallest_frame_capacity():
  tr, _ = atari_stream(3, episodes=2, max_len=24, seed=5)
  cap = 10
  shape = tr[0][0].shape
  F = fo.min_frame_capacity(cap, shape, tr)
  ok = fo.FrameStore(cap, F, shape)
  live = _feed(ok, tr, cap)
  assert not ok.pool_full
  _assert_round_trip(ok, tr, live)
  bad = fo.FrameStore(cap, F - 1, shape)
  _feed(bad, tr, cap)
  assert bad.pool_full
  first = bad.full_ids[0]
  # rows stored before the first overflow are intact
  for i in range(max(0, first - cap + 1), first):
    a, b = bad.get(i)
    np.testing.assert_array_equal(a, tr[i][0])
    np.testing.assert_array_equal(b, tr[i][1])


def test_closed_form_synthetic_fill_equals_sequential_adds():
  shape = (4, 6, 4)
  for n, L in ((37, 9), (40, 40), (25, 3), (16, 100)):
    tr = fo.synthetic_transitions(n, L, 11, shape)
    seq = fo.FrameStore(n, 2 * n, shape)
    _feed(seq, tr, n)
    cf = fo.synthetic_fill(n, 2 * n, shape, n, L, 11)
    assert cf.appends == seq.appends
    np.testing.assert_array_equal(cf.row_frames, seq.row_frames)
    np.testing.assert_array_equal(cf.born, seq.born)
    np.testing.assert_array_equal(cf.last_ref, seq.last_ref)
    np.testing.assert_array_equal(cf.window, seq.window)
    for s, f in cf.frames.items():
      np.testing.assert_array_equal(f, seq.frames[s])
      if s:
        assert cf.hash[s] == int(seq.hash[s])


def test_host_compiled_frame_hash_equals_numpy():
  from dqn_zoo_b200 import _lib
  rs = np.random.RandomState(3)
  for n in (0, 1, 7, 8, 9, 24, 7056, 7057):
    data = rs.randint(0, 256, size=n).astype(np.uint8)
    out = C.c_uint64()
    _lib.call('dz_test_frame_hash', data.ctypes.data, n, C.byref(out))
    assert out.value == fo.frame_hash(data), n
