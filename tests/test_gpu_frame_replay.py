"""GPU: the frame-deduplicated replay (`frame_capacity=F`) against the raw store and the numpy oracle
(oracle/frame_store_oracle.py): identical samples / get / get_state, the reference contract and golden scenarios, device
frame slots and counters bit-exact after every add, bit-identical fused learner steps, the device-resident insert path,
pool overflow, the 1M-row store, and state moving between store kinds."""

import collections
import types

import numpy as np
import pytest
import torch

from oracle import frame_store_oracle as fo
from oracle import replay_oracle as ro
from oracle import scenarios
import replay_contract as rc
import test_oracle_frame_store as tof

pytestmark = pytest.mark.gpu

T = None  # Transition structure, set by the fixture


@pytest.fixture(scope='module')
def dev():
  from dqn_zoo_b200 import replay
  global T
  T = replay.Transition(None, None, None, None, None)
  return replay


def _frame_lib(dev):
  """The replay module with both replay classes building frame stores (F = 4 * capacity + 64 fits iid stacks)."""
  lib = types.SimpleNamespace(**{k: getattr(dev, k) for k in dir(dev) if not k.startswith('__')})
  lib.TransitionReplay = lambda capacity, *a, **k: dev.TransitionReplay(capacity, *a, frame_capacity=4 * capacity + 64,
                                                                         **k)
  lib.PrioritizedTransitionReplay = lambda capacity, *a, **k: dev.PrioritizedTransitionReplay(
      capacity, *a, frame_capacity=4 * capacity + 64, **k)
  return lib


@pytest.mark.parametrize('name', list(scenarios.ALL))
def test_frame_store_reproduces_reference_golden(dev, name):
  rc.check_scenario(_frame_lib(dev), name, 'device')


@pytest.mark.parametrize('fn', rc.CONTRACT, ids=lambda f: f.__name__)
def test_frame_store_contract(dev, fn):
  fn(_frame_lib(dev))


def _make(dev, prioritized, cap, seed, frame_capacity=None):
  if prioritized:
    return dev.PrioritizedTransitionReplay(cap, T, 0.5, lambda t: 0.6, 1e-2, True, np.random.RandomState(seed),
                                           frame_capacity=frame_capacity)
  return dev.TransitionReplay(cap, T, np.random.RandomState(seed), frame_capacity=frame_capacity)


def _stream(n_step=3, seed=4, episodes=4, max_len=30):
  tr, _ = tof.atari_stream(n_step, episodes=episodes, max_len=max_len, seed=seed)
  rs = np.random.RandomState(seed)
  return [dict(s_tm1=a, s_t=b, a=int(rs.randint(6)), r=float(rs.randint(-1, 2)), d=float(rs.uniform()),
               p=float(rs.uniform(0.1, 2.0))) for a, b in tr]


def _add(rep, k, x, prioritized, device_source):
  s_tm1, s_t = x['s_tm1'], x['s_t']
  if device_source:
    s_tm1, s_t = torch.as_tensor(s_tm1, device='cuda'), torch.as_tensor(s_t, device='cuda')
  item = T._replace(s_tm1=s_tm1, a_tm1=x['a'], r_t=x['r'], discount_t=x['d'], s_t=s_t)
  if prioritized:
    rep.add(item, priority=x['p'])
  else:
    rep.add(item)


def _assert_same_transition(a, b):
  for x, y in zip(a, b):
    x, y = np.asarray(x), np.asarray(y)
    assert x.dtype == y.dtype and x.shape == y.shape
    np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize('prioritized', [False, True])
def test_same_results_as_raw_store(dev, prioritized):
  stream = _stream()
  cap = 24                                           # the stream wraps the ring several times
  raw, frm = _make(dev, prioritized, cap, 5), _make(dev, prioritized, cap, 5, frame_capacity=4 * cap + 64)
  for k, x in enumerate(stream):
    for rep in (raw, frm):
      _add(rep, k, x, prioritized, device_source=k % 3 == 1)
    if k % 7 == 6:
      out_r, out_f = raw.sample(8), frm.sample(8)
      if prioritized:
        _assert_same_transition(out_r[0], out_f[0])
        np.testing.assert_array_equal(out_r[1], out_f[1])
        np.testing.assert_array_equal(out_r[2], out_f[2])
        ids = out_r[1]
        pri = np.linspace(0.5, 1.5, 8).astype(np.float32)
        raw.update_priorities(ids, pri)
        frm.update_priorities(ids, pri)
      else:
        _assert_same_transition(out_r, out_f)
  live = list(raw._live_ids)
  for a, b in zip(raw.get(live), frm.get(live)):
    _assert_same_transition(a, b)
  sr, sf = raw.get_state(), frm.get_state()
  assert [i for i, _ in sr['storage']] == [i for i, _ in sf['storage']]
  for (_, a), (_, b) in zip(sr['storage'], sf['storage']):
    _assert_same_transition(a, b)
  assert frm.check_valid()[0]


def _device_state(store):
  n = store.frame_capacity + 1
  return dict(row_frames=store.row_frames.cpu().numpy(), born=store.frame_born.cpu().numpy()[:n],
              last_ref=store.frame_last_ref.cpu().numpy()[:n], hash=store.frame_hash.cpu().numpy().view(np.uint64),
              state=store.state.cpu().numpy(), frames=store.frames.cpu().numpy()[:, :store.frame_bytes])


def test_device_matches_oracle_after_every_add(dev):
  """Episode starts (zero-padded stacks), n-step transitions, iid stacks and ring wrap with reclaim."""
  atari = _stream(n_step=3, seed=9, episodes=10, max_len=80)
  rs = np.random.RandomState(2)
  iid = [dict(s_tm1=rs.randint(0, 256, size=atari[0]['s_tm1'].shape).astype(np.uint8),
              s_t=rs.randint(0, 256, size=atari[0]['s_t'].shape).astype(np.uint8), a=1, r=0.0, d=1.0, p=1.0)
         for _ in range(10)]
  stream = atari[:30] + iid[:5] + atari[30:]
  cap, F = 6, 64
  rep = _make(dev, False, cap, 1, frame_capacity=F)
  ora = fo.FrameStore(cap, F, atari[0]['s_tm1'].shape)
  live = collections.deque()
  for k, x in enumerate(stream):
    live.append(k)
    if len(live) > cap:
      live.popleft()
    _add(rep, k, x, False, device_source=k % 2 == 1)
    ora.add(k, live[0], x['s_tm1'], x['s_t'])
    got = _device_state(rep._store)
    np.testing.assert_array_equal(got['row_frames'], ora.row_frames, err_msg='row_frames after add %d' % k)
    np.testing.assert_array_equal(got['born'], ora.born, err_msg='born after add %d' % k)
    np.testing.assert_array_equal(got['last_ref'], ora.last_ref, err_msg='last_ref after add %d' % k)
    np.testing.assert_array_equal(got['state'], ora.state_vector(), err_msg='state after add %d' % k)
    written = np.flatnonzero(ora.born >= 0)
    np.testing.assert_array_equal(got['hash'][written], ora.hash[written])
    np.testing.assert_array_equal(got['frames'][written], ora.frames[written])
  assert not ora.pool_full and ora.appends > F       # the ring wrapped and reclaimed slots
  assert rep.check_valid()[0]


def test_pool_overflow_raises_at_the_predicted_add(dev):
  rs = np.random.RandomState(8)
  shape = (6, 4, 2)
  tr = [(rs.randint(1, 256, size=shape).astype(np.uint8), rs.randint(1, 256, size=shape).astype(np.uint8))
        for _ in range(30)]
  cap = 5
  F = fo.min_frame_capacity(cap, shape, tr) - 1
  ora = fo.FrameStore(cap, F, shape)
  tof._feed(ora, tr, cap)
  first = ora.full_ids[0]
  rep = _make(dev, False, cap, 3, frame_capacity=F)
  for k in range(first):
    rep.add(T._replace(s_tm1=tr[k][0], a_tm1=0, r_t=0.0, discount_t=1.0, s_t=tr[k][1]))
  assert rep.check_valid()[0]
  rep.add(T._replace(s_tm1=tr[first][0], a_tm1=0, r_t=0.0, discount_t=1.0, s_t=tr[first][1]))
  with pytest.raises(RuntimeError, match='frame pool is full'):
    rep.sample(4)
  before = [i for i in rep.ids() if i < first]
  for i, got in zip(before, rep.get(before)):
    np.testing.assert_array_equal(got.s_tm1, tr[i][0])
    np.testing.assert_array_equal(got.s_t, tr[i][1])
  # a prioritized replay raises on its flag word too
  per = _make(dev, True, cap, 3, frame_capacity=F)
  for k in range(first + 1):
    per.add(T._replace(s_tm1=tr[k][0], a_tm1=0, r_t=0.0, discount_t=1.0, s_t=tr[k][1]), priority=1.0)
  with pytest.raises(RuntimeError, match='frame pool is full'):
    per.check_valid()


def test_bad_observation_format_is_rejected_at_the_first_add(dev):
  rep = _make(dev, False, 4, 1, frame_capacity=16)
  with pytest.raises(ValueError, match='frame store needs uint8 observations'):
    rep.add(T._replace(s_tm1=np.zeros((4, 4), np.uint8), a_tm1=0, r_t=0.0, discount_t=1.0, s_t=np.zeros((4, 4), np.uint8)))
  rep = _make(dev, False, 4, 1, frame_capacity=16)
  with pytest.raises(ValueError, match='frame store needs uint8 observations'):
    rep.add(T._replace(s_tm1=np.zeros((4, 4, 2), np.float32), a_tm1=0, r_t=0.0, discount_t=1.0,
                       s_t=np.zeros((4, 4, 2), np.float32)))


def test_oversize_frame_geometry_is_rejected_before_anything_changes(dev):
  """The insert stages both stacks in shared memory: (210, 160, 4) stacks need 268,800 B > DZ_FRAME_MAX_STAGE_BYTES.
  The first add raises ValueError with the replay untouched, and dz_replay_add itself rejects such a view before it
  enqueues the add's copies, index patches or tree update."""
  import ctypes as C
  from dqn_zoo_b200 import _lib
  big = np.zeros((210, 160, 4), np.uint8)
  for prioritized in (False, True):
    rep = _make(dev, prioritized, 4, 1, frame_capacity=16)
    with pytest.raises(ValueError, match='frame store needs 2 \\* S'):
      _add(rep, 0, dict(s_tm1=big, s_t=big, a=3, r=1.0, d=1.0, p=1.0), prioritized, False)
    assert rep.size == 0 and rep._t == 0
  rep = _make(dev, True, 4, 1, frame_capacity=16)
  x = np.ones((6, 4, 2), np.uint8)
  rep.add(T._replace(s_tm1=x, a_tm1=1, r_t=0.0, discount_t=1.0, s_t=x), priority=1.0)
  v = rep.device_view()
  v.obs_bytes, v.frames.frame_bytes, v.frames.frame_stride, v.frames.stack = 210 * 160 * 4, 210 * 160, 33600, 4
  rec = _lib.AddRecord()
  rec.slot, rec.action, rec.n_patches, rec.tree_index, rec.leaf_value = 1, 5, 0, 1, 7.0
  rec.evict_index, rec.size_after, rec.alpha, rec.item_id, rec.oldest_live = -1, 4, 1.0, 1, 0
  with pytest.raises(ValueError, match='DZ_FRAME_MAX_STAGE_BYTES'):
    _lib.call('dz_replay_add', C.byref(v), C.byref(rec), big.ctypes.data, big.ctypes.data,
              torch.cuda.current_stream().cuda_stream)
  torch.cuda.synchronize()
  assert int(rep._store.action[1].item()) == 0                       # no scalar write
  assert rep._distribution._sum_tree.root() == 1.0                    # no tree update
  assert rep.check_valid()[0]


@pytest.mark.parametrize('prioritized', [False, True])
def test_state_moves_between_store_kinds(dev, prioritized):
  stream = _stream(n_step=1, seed=12)[:40]
  cap = 16
  src_raw, src_frm = _make(dev, prioritized, cap, 6), _make(dev, prioritized, cap, 6, frame_capacity=200)
  for k, x in enumerate(stream[:30]):
    _add(src_raw, k, x, prioritized, False)
    _add(src_frm, k, x, prioritized, False)
  for src, dst in ((src_frm, _make(dev, prioritized, cap, 99)), (src_raw, _make(dev, prioritized, cap, 99, 200))):
    import copy
    dst.set_state(copy.deepcopy(src.get_state()))
    rc._rebind_rng(src, np.random.RandomState(4))
    rc._rebind_rng(dst, np.random.RandomState(4))
    for k, x in enumerate(stream[30:]):
      _add(src, 30 + k, x, prioritized, False)
      _add(dst, 30 + k, x, prioritized, False)
      a, b = src.sample(6), dst.sample(6)
      if prioritized:
        _assert_same_transition(a[0], b[0])
        np.testing.assert_array_equal(a[1], b[1])
        np.testing.assert_array_equal(a[2], b[2])
      else:
        _assert_same_transition(a, b)
    assert dst.check_valid()[0]


def test_bulk_fill_equals_sequential_adds_at_small_capacity(dev):
  shape, cap, L, seed = (8, 6, 4), 50, 7, 5
  bulk = _make(dev, True, cap, 1, frame_capacity=80)
  dev.bulk_fill_synthetic(bulk, shape, seed, 6, discount=0.9, episode_length=L)
  seq = _make(dev, True, cap, 1, frame_capacity=80)
  tr = fo.synthetic_transitions(cap, L, seed, shape)
  _, a, r, d = ro.synthetic_rows(seed, np.arange(cap), 8, 6, discount=0.9)
  for i, (s0, s1) in enumerate(tr):
    seq.add(T._replace(s_tm1=s0, a_tm1=int(a[i]), r_t=float(r[i]), discount_t=float(d[i]), s_t=s1), priority=1.0)
  gb, gs = _device_state(bulk._store), _device_state(seq._store)
  appended = np.arange(1, gb['state'][0] + 1)
  for k in ('row_frames', 'state'):
    np.testing.assert_array_equal(gb[k], gs[k], err_msg=k)
  for k in ('born', 'last_ref', 'hash', 'frames'):
    np.testing.assert_array_equal(gb[k][appended], gs[k][appended], err_msg=k)
  for (i0, t0), (i1, t1) in zip(bulk.get_state()['storage'], seq.get_state()['storage']):
    assert i0 == i1
    _assert_same_transition(t0, t1)
  cf = fo.synthetic_fill(cap, 80, shape, cap, L, seed)
  np.testing.assert_array_equal(gb['row_frames'], cf.row_frames)
  np.testing.assert_array_equal(gb['state'], cf.state_vector())


def test_full_size_store(dev):
  """1M transitions of 84x84x4 in a 1.25M-frame store: the bytes it allocates, and gathers at frame byte offsets above
  2^32 and around the row wrap against the oracle."""
  cap, F, shape, L, seed = 1_000_000, 1_250_000, (84, 84, 4), 1000, 3
  rep = _make(dev, False, cap, 2, frame_capacity=F)
  dev.bulk_fill_synthetic(rep, shape, seed, 6, episode_length=L)
  st = rep._store
  want = (F + 1) * 7056 + cap * 8 * 4 + 3 * (F + 1) * 8 + (2 + 16 * 9) * 8 + 2 * 28224 + cap * (4 + 8 + 8) + 4
  assert st.device_bytes == want and want < 10e9
  rows = [0, 1, 999, 1000, 608_000, 650_000, 999_998, 999_999]
  cf = fo.synthetic_fill(cap, F, shape, cap, L, seed, rows=rows)
  assert int(cf.row_frames[rows].max()) * 7056 > 2 ** 32
  for i, got in zip(rows, rep.get(rows)):
    want0, want1 = cf.get(i)
    np.testing.assert_array_equal(got.s_tm1, want0)
    np.testing.assert_array_equal(got.s_t, want1)
  # two more adds wrap the row ring (ids 1M, 1M+1 land in rows 0, 1)
  rs = np.random.RandomState(1)
  extra = [rs.randint(0, 256, size=shape).astype(np.uint8) for _ in range(3)]
  rep.add(T._replace(s_tm1=extra[0], a_tm1=1, r_t=0.0, discount_t=1.0, s_t=extra[1]))
  rep.add(T._replace(s_tm1=extra[1], a_tm1=2, r_t=0.0, discount_t=1.0, s_t=extra[2]))
  got = rep.get([cap - 1, cap, cap + 1])
  np.testing.assert_array_equal(got[0].s_tm1, cf.get(cap - 1)[0])
  np.testing.assert_array_equal(got[1].s_t, extra[1])
  np.testing.assert_array_equal(got[2].s_tm1, extra[1])
  np.testing.assert_array_equal(got[2].s_t, extra[2])
  assert rep.check_valid()[0]


# ---- fused learner ---------------------------------------------------------------------------------------------------


def _agent(kind, rep, use_graph):
  from dqn_zoo_b200 import agent as agent_lib
  from dqn_zoo_b200 import learner as learner_lib
  common = dict(preprocessor=lambda ts: ts, sample_network_input=np.zeros((84, 84, 4), np.uint8),
                network=learner_lib.NetworkSpec(kind, 6), optimizer=None,
                transition_accumulator=dev_replay().NStepTransitionAccumulator(1), replay=rep, batch_size=32,
                min_replay_capacity_fraction=0.0, learn_period=1, target_network_update_period=1000, rng_key=[0, 5],
                use_cuda_graph=use_graph)
  if kind == 'rainbow':
    return agent_lib.Rainbow(support=np.linspace(-10, 10, 51), **common)
  if kind == 'iqn':
    return agent_lib.Iqn(exploration_epsilon=lambda t: 0.01, huber_param=1.0, tau_samples_policy=64,
                         tau_samples_s_tm1=64, tau_samples_s_t=64, **common)
  return agent_lib.Dqn(exploration_epsilon=lambda t: 0.01, grad_error_bound=1.0 / 32, **common)


def dev_replay():
  from dqn_zoo_b200 import replay
  return replay


@pytest.fixture(scope='module')
def atari_transitions():
  tr = fo.synthetic_transitions(300, 37, 17, (84, 84, 4))
  rs = np.random.RandomState(3)
  return [(a, b, int(rs.randint(6)), float(rs.randint(-1, 2)), 0.99) for a, b in tr]


@pytest.mark.parametrize('use_graph', [False, True], ids=['eager', 'graph'])
@pytest.mark.parametrize('kind', ['rainbow', 'dqn', 'iqn'])
def test_fused_learn_is_bit_identical(dev, atari_transitions, kind, use_graph):
  prioritized = kind == 'rainbow'
  outs = []
  for frame_capacity in (None, 600):
    rep = _make(dev, prioritized, 256, 11, frame_capacity=frame_capacity)
    ag = _agent(kind, rep, use_graph)
    L = ag.learner
    steps = []
    for k, (a, b, act, r, d) in enumerate(atari_transitions):
      ag._add(T._replace(s_tm1=a if k % 2 else torch.as_tensor(a, device='cuda'), a_tm1=act, r_t=r, discount_t=d,
                         s_t=b if k % 2 else torch.as_tensor(b, device='cuda')))
      if k >= 64 and k % 40 == 0:
        for _ in range(3):
          ag.learn()
          torch.cuda.synchronize()
          steps.append([t.detach().cpu().numpy().copy() for t in (L.loss, L.per_example, L.priorities, L.grad_norm,
                                                                  L.sampled_ids)])
    ag.check_device_flags()
    outs.append((steps, L.online.detach().cpu().numpy().copy()))
  (s_raw, p_raw), (s_frm, p_frm) = outs
  assert len(s_raw) == len(s_frm) >= 15
  for a, b in zip(s_raw, s_frm):
    for x, y in zip(a, b):
      np.testing.assert_array_equal(x, y)
  np.testing.assert_array_equal(p_raw, p_frm)


def test_learn_rejects_batches_beyond_the_reserved_staging(dev, atari_transitions):
  rep = _make(dev, False, 256, 1, frame_capacity=600)
  ag = _agent('dqn', rep, False)
  for a, b, act, r, d in atari_transitions[:64]:
    ag._add(T._replace(s_tm1=a, a_tm1=act, r_t=r, discount_t=d, s_t=b))
  rep._store.batch_capacity = 16                    # as if a smaller batch had been reserved
  with pytest.raises(ValueError, match='batch staging'):
    ag.learn()


def test_agent_with_device_resident_frames_and_frame_store_equals_raw_store(dev):
  """Raw RGB frames -> processors.atari(device_observations=True) -> rainbow with a frame store: the actions and the
  replay contents equal those of the raw store fed the same way."""
  import test_gpu_processors as tgp
  from dqn_zoo_b200 import agent as ag
  from dqn_zoo_b200 import learner as dl
  from dqn_zoo_b200 import processors
  rs = np.random.RandomState(21)
  episodes = [tgp.random_episode(rs, n, (210, 160, 3), life_loss_at=loss) for n, loss in [(23, 9), (14, None), (31, 17)]]

  def run(frame_capacity):
    rep = dev.PrioritizedTransitionReplay(16, T, 0.5, lambda t: 0.5, 1e-3, True, np.random.RandomState(3),
                                          frame_capacity=frame_capacity)
    agent = ag.Rainbow(preprocessor=processors.atari(device_observations=True),
                       sample_network_input=np.zeros((84, 84, 4), np.uint8), network=dl.NetworkSpec('rainbow', 6),
                       support=np.linspace(-10, 10, 51), optimizer=None,
                       transition_accumulator=dev.NStepTransitionAccumulator(3), replay=rep, batch_size=4,
                       min_replay_capacity_fraction=0.5, learn_period=4, target_network_update_period=16, rng_key=[0, 7],
                       use_cuda_graph=False)
    actions = []
    for ep in episodes:
      agent.reset()
      for st, r, d, f, lives in ep:
        actions.append(agent.step(tgp.ts(st, r, d, f, lives)))
    torch.cuda.synchronize()
    return actions, rep.get_state(), agent.learner.online.cpu().numpy()

  a_raw, s_raw, p_raw = run(None)
  a_frm, s_frm, p_frm = run(128)
  assert a_raw == a_frm
  assert len(s_raw['storage']) == len(s_frm['storage']) > 5
  for (i0, t0), (i1, t1) in zip(s_raw['storage'], s_frm['storage']):
    assert i0 == i1
    _assert_same_transition(t0, t1)
  np.testing.assert_array_equal(p_raw, p_frm)
