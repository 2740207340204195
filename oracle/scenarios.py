"""Deterministic replay op-scripts shared by the golden generator and the tests.

TEST INFRASTRUCTURE ONLY (see oracle/replay_oracle.py header).

Each scenario takes a namespace `lib` exposing the reference's replay API
(`SumTree`, `PrioritizedDistribution`, `TransitionReplay`,
`PrioritizedTransitionReplay`, `NStepTransitionAccumulator`,
`TransitionAccumulator`, `Transition`) and returns a dict of numpy arrays.
`oracle/gen_golden.py` runs them against the REFERENCE's own `replay.py` and
stores the result under tests/golden/; the tests run them against the oracle
(CPU) and against the CUDA-backed `dqn_zoo_b200.replay` and demand equality.
"""

from __future__ import annotations

import collections

import numpy as np

OBS_SHAPE = (6, 4, 2)  # 48 bytes, small so fixtures stay tiny


class _Schedule:
  """`parts.py:414-430` LinearSchedule restated (tiny; pinned by tests/test_parts.py)."""

  def __init__(self, begin_value, end_value, begin_t, decay_steps):
    self.b, self.e, self.t0, self.n = begin_value, end_value, begin_t, decay_steps

  def __call__(self, t):
    frac = min(max(t - self.t0, 0), self.n) / self.n
    return (1 - frac) * self.b + frac * self.e


def _item(lib, rs, k):
  obs_a = rs.randint(0, 256, size=OBS_SHAPE).astype(np.uint8)
  obs_b = rs.randint(0, 256, size=OBS_SHAPE).astype(np.uint8)
  return lib.Transition(s_tm1=obs_a, a_tm1=int(rs.randint(0, 6)), r_t=float(rs.randint(-1, 2)),
                        discount_t=float(0.99 ** int(rs.randint(0, 4))), s_t=obs_b)


def sum_tree_ops(lib, seed=3):
  """Random resize/set/set_all/query mix (after `replay_test.py:1120-1137`)."""
  rs = np.random.RandomState(seed)
  tree = lib.SumTree()
  out = collections.OrderedDict()
  q_all, r_all = [], []
  for step in range(60):
    op = rs.randint(4)
    if op == 0 or tree.size == 0:
      n = int(rs.randint(1, 70))
      vals = np.abs(rs.standard_cauchy(n))
      vals[rs.uniform(size=n) < 0.2] = 0.0
      tree.set_all(vals)
    elif op == 1:
      tree.resize(int(rs.randint(1, 90)))
    elif op == 2:
      k = int(rs.randint(1, 12))
      idx = rs.randint(tree.size, size=k)
      vals = np.abs(rs.standard_cauchy(k))
      tree.set(idx, vals)
    if tree.size and tree.root() > 0:
      targets = rs.uniform(size=5) * tree.root()
      q_all.append(np.asarray(tree.query(targets), dtype=np.int64))
      r_all.append(tree.root())
  out['queries'] = np.concatenate(q_all)
  out['roots'] = np.asarray(r_all, dtype=np.float64)
  st = tree.get_state()
  out['final_storage'] = np.array(st['storage'], dtype=np.float64)[: 2 * st['first_leaf']]
  out['final_size'] = np.asarray(st['size'])
  out['final_first_leaf'] = np.asarray(st['first_leaf'])
  return out


def prioritized_replay_script(lib, capacity=48, alpha=0.5, usp=0.25, normalize=True,
                              batch=16, rounds=40, seed=7):
  """add / sample / update_priorities interleaved on a small PER, wrapping the
  ring several times.  Records every sampled id and weight plus the final tree."""
  rs_replay = np.random.RandomState(seed)       # consumed by the replay itself
  rs_script = np.random.RandomState(seed + 100)  # contents and priorities
  sched = _Schedule(0.4, 1.0, begin_t=capacity // 2, decay_steps=4 * capacity)
  structure = lib.Transition(None, None, None, None, None)
  rep = lib.PrioritizedTransitionReplay(capacity, structure, alpha, sched, usp, normalize, rs_replay)
  ids_all, w_all, s_sum, a_all, r_all, d_all = [], [], [], [], [], []
  max_seen = 1.0
  for rnd in range(rounds):
    for _ in range(int(rs_script.randint(1, 9))):
      # zero priority sometimes: those items must never be sampled by the tree branch
      pr = 0.0 if rs_script.uniform() < 0.1 else max_seen
      rep.add(_item(lib, rs_script, 0), pr)
    if rep.size < 4:
      continue
    tr, ids, w = rep.sample(batch)
    ids_all.append(np.asarray(ids, dtype=np.int64))
    w_all.append(np.asarray(w, dtype=np.float64))
    s_sum.append(tr.s_tm1.astype(np.int64).sum(axis=(1, 2, 3)) * 1000 + tr.s_t.astype(np.int64).sum(axis=(1, 2, 3)))
    a_all.append(np.asarray(tr.a_tm1, dtype=np.int64))
    r_all.append(np.asarray(tr.r_t, dtype=np.float64))
    d_all.append(np.asarray(tr.discount_t, dtype=np.float64))
    # float32 priorities, as they come back from the device (`rainbow/agent.py:194-195`)
    pri = np.clip(np.abs(rs_script.standard_cauchy(batch)), 0.0, 100.0).astype(np.float32)
    pri[rs_script.uniform(size=batch) < 0.05] = 0.0
    max_seen = float(np.max([max_seen, pri.max()]))
    rep.update_priorities(ids, pri)
  st = rep.get_state()
  tree = st['distribution']['sum_tree']
  out = collections.OrderedDict()
  out['ids'] = np.stack(ids_all)
  out['weights'] = np.stack(w_all)
  out['obs_checksum'] = np.stack(s_sum)
  out['a'] = np.stack(a_all)
  out['r'] = np.stack(r_all)
  out['d'] = np.stack(d_all)
  out['tree_storage'] = np.array(tree['storage'], dtype=np.float64)
  out['active_indices'] = np.asarray(list(st['distribution']['active_indices']), dtype=np.int64)
  out['t'] = np.asarray(st['t'])
  out['storage_ids'] = np.asarray([k for k, _ in st['storage']], dtype=np.int64)
  return out


def uniform_replay_script(lib, capacity=37, batch=16, rounds=30, seed=11):
  """Uniform replay wrapped several times; pins the swap-remove id permutation."""
  rs_replay = np.random.RandomState(seed)
  rs_script = np.random.RandomState(seed + 100)
  structure = lib.Transition(None, None, None, None, None)
  rep = lib.TransitionReplay(capacity, structure, rs_replay)
  ids_like, a_all, s_sum = [], [], []
  for rnd in range(rounds):
    for _ in range(int(rs_script.randint(1, 12))):
      rep.add(_item(lib, rs_script, 0))
    tr = rep.sample(batch)
    s_sum.append(tr.s_tm1.astype(np.int64).sum(axis=(1, 2, 3)) * 1000 + tr.s_t.astype(np.int64).sum(axis=(1, 2, 3)))
    a_all.append(np.asarray(tr.a_tm1, dtype=np.int64))
  st = rep.get_state()
  out = collections.OrderedDict()
  out['obs_checksum'] = np.stack(s_sum)
  out['a'] = np.stack(a_all)
  out['dist_ids'] = np.asarray(list(st['distribution']['ids']), dtype=np.int64)
  out['storage_ids'] = np.asarray([k for k, _ in st['storage']], dtype=np.int64)
  out['t'] = np.asarray(st['t'])
  return out


def distribution_growth_script(lib, seed=5):
  """`PrioritizedDistribution` with growing capacity, arbitrary ids, removals."""
  rs = np.random.RandomState(seed)
  rs_script = np.random.RandomState(seed + 100)
  dist = lib.PrioritizedDistribution(priority_exponent=0.7, uniform_sample_probability=0.2,
                                     random_state=rs, min_capacity=0, max_capacity=None)
  next_id = 100
  live = []
  ids_all, p_all = [], []
  for rnd in range(30):
    k = int(rs_script.randint(1, 6))
    new = list(range(next_id, next_id + k))
    next_id += k + int(rs_script.randint(0, 3))
    dist.add_priorities(new, np.abs(rs_script.standard_cauchy(k)))  # float64 path
    live.extend(new)
    if len(live) > 6 and rs_script.uniform() < 0.5:
      drop = [live.pop(int(rs_script.randint(len(live)))) for _ in range(2)]
      dist.remove_priorities(drop)
    if rs_script.uniform() < 0.5:
      upd = [live[int(j)] for j in rs_script.randint(len(live), size=3)]
      dist.update_priorities(upd, np.abs(rs_script.standard_cauchy(3)))
    ids, probs = dist.sample(8)
    ids_all.append(np.asarray(ids, dtype=np.int64))
    p_all.append(np.asarray(probs, dtype=np.float64))
  out = collections.OrderedDict()
  out['ids'] = np.stack(ids_all)
  out['probs'] = np.stack(p_all)
  out['all_ids'] = np.asarray(list(dist.ids()), dtype=np.int64)
  out['capacity'] = np.asarray(dist.capacity)
  st = dist.get_state()
  out['active_indices'] = np.asarray(list(st['active_indices']), dtype=np.int64)
  out['inactive_indices'] = np.asarray(list(st['inactive_indices']), dtype=np.int64)
  return out


class _TS:
  """Minimal dm_env.TimeStep stand-in: FIRST=0, MID=1, LAST=2."""

  def __init__(self, step_type, reward, discount, observation):
    self.step_type, self.reward, self.discount, self.observation = step_type, reward, discount, observation

  def first(self):
    return self.step_type == 0

  def mid(self):
    return self.step_type == 1

  def last(self):
    return self.step_type == 2


def n_step_script(lib, n=3, seed=13):
  """Episodes of random length (incl. shorter than n) through the n-step accumulator."""
  rs = np.random.RandomState(seed)
  acc = lib.NStepTransitionAccumulator(n)
  rows = []
  obs_id = 0
  for ep in range(12):
    length = int(rs.randint(1, 9))
    acc.reset()
    for t in range(length + 1):
      st = 0 if t == 0 else (2 if t == length else 1)
      reward = None if t == 0 else float(rs.randint(-3, 4)) * 0.37
      disc = None if t == 0 else (0.0 if (st == 2 and rs.uniform() < 0.5) else float(rs.uniform(0.5, 1.0)))
      ts = _TS(st, reward, disc, obs_id)
      a = int(rs.randint(0, 6))
      for tr in acc.step(ts, a):
        rows.append([float(tr.s_tm1), float(tr.a_tm1), tr.r_t, tr.discount_t, float(tr.s_t)])
      obs_id += 1
  return collections.OrderedDict(rows=np.asarray(rows, dtype=np.float64))


ALL = collections.OrderedDict([
    ('replay_sumtree', lambda lib: sum_tree_ops(lib)),
    ('replay_per_sqrt', lambda lib: prioritized_replay_script(lib, alpha=0.5, usp=0.25, normalize=True)),
    ('replay_per_usp_small', lambda lib: prioritized_replay_script(lib, capacity=64, alpha=0.5, usp=1e-3,
                                                                   normalize=True, batch=32, seed=21)),
    ('replay_per_pow06', lambda lib: prioritized_replay_script(lib, alpha=0.6, usp=0.1, normalize=False, seed=9)),
    ('replay_uniform', lambda lib: uniform_replay_script(lib)),
    ('replay_distribution_growth', lambda lib: distribution_growth_script(lib)),
    ('replay_nstep3', lambda lib: n_step_script(lib, n=3)),
    ('replay_nstep1', lambda lib: n_step_script(lib, n=1, seed=17)),
])

# a longer PER run (wraps a 257-slot ring ~7 times), compared with the reference's result in replay_per_long_random.npz
LONG_PER_RUN = dict(capacity=257, alpha=0.5, usp=1e-3, normalize=True, batch=32, rounds=400, seed=31)
