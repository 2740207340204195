"""CPU timing of the reference algorithm for the hot path (TEST/BENCH INFRASTRUCTURE ONLY).

Used by bench.py's `cpu_baseline` leg and by `bench.py --impl reference`.  JAX/haiku/rlax/optax
and the reference tree itself are unavailable on the GPU box, so this times the oracle PORT:
  half A  replay sample + update_priorities  -> oracle/replay_oracle.py (python/numpy, one
          thread: the reference's replay is single-threaded python by construction, README.md:93-95)
  half B  jit(update)                        -> oracle/learner_oracle.py in float32 on all host
          cores through torch's CPU kernels (stand-in for XLA:CPU; NOT JAX — labelled "port")
executed serially per learner step as `_learn()` does (rainbow/agent.py:181-198).
"""

import collections
import time

import numpy as np
import torch

from oracle import learner_oracle as lo
from oracle import replay_oracle as ro

POOL = 512  # distinct synthetic frames shared by all transitions (host RAM; BASELINE.md §3)


def build_replay(kind, capacity, batch, seed, obs_shape=(84, 84, 4), num_actions=6):
  """Oracle replay in the state it has after `capacity` adds with priority 1 (closed form for the
  id/index bookkeeping, exactly what dqn_zoo_b200.replay.bulk_fill_synthetic writes)."""
  rs = np.random.RandomState(seed)
  obs_bytes = int(np.prod(obs_shape))
  pool_obs, _, _, _ = ro.synthetic_rows(seed, np.arange(POOL), obs_bytes, num_actions)
  pool_obs = pool_obs.reshape(POOL, 2, *obs_shape)
  _, a, r, d = ro.synthetic_rows(seed, np.arange(8), 8, num_actions)  # warm the hash path
  rows = np.arange(capacity)
  # scalars for every row without generating 56 GB of observations
  _, a, r, d = _scalars(seed, rows, num_actions)
  structure = ro.Transition(None, None, None, None, None)
  prioritized = kind in ('rainbow', 'prioritized')
  if prioritized:
    alpha = 0.5 if kind == 'rainbow' else 0.6
    rep = ro.PrioritizedTransitionReplay(capacity, structure, alpha, lambda t: 0.4, 1e-3, True, rs)
    dist = rep._distribution
    idx = list(range(capacity - 1, -1, -1))
    dist._idx_of = dict(zip(range(capacity), idx))
    dist._id_at = dict(zip(idx, range(capacity)))
    dist._free = []
    dist._live = idx
    dist._live_pos = dict(zip(idx, range(capacity)))
    dist._tree.set_all(np.ones(capacity))
  else:
    rep = ro.TransitionReplay(capacity, structure, rs)
    rep._distribution._slots = list(range(capacity))
    rep._distribution._where = {i: i for i in range(capacity)}
  items = collections.OrderedDict()
  for i in range(capacity):
    p = i % POOL
    items[i] = ro.Transition(pool_obs[p, 0], int(a[i]), float(r[i]), float(d[i]), pool_obs[p, 1])
  rep._items = items
  rep._t = capacity
  return rep, prioritized


def _scalars(seed, rows, num_actions):
  obs, a, r, d = ro.synthetic_rows(seed, rows[:1], 8, num_actions)
  # synthetic_rows computes scalars independently of obs_bytes; call it with a tiny obs size
  out_a, out_r, out_d = [], [], []
  for lo_ in range(0, len(rows), 1 << 18):
    _, a, r, d = ro.synthetic_rows(seed, rows[lo_:lo_ + (1 << 18)], 8, num_actions)
    out_a.append(a); out_r.append(r); out_d.append(d)
  return None, np.concatenate(out_a), np.concatenate(out_r), np.concatenate(out_d)


def cgroup_cpu_limit():
  """CPUs this process may actually use: min(affinity mask, cgroup v2 / v1 CPU quota)."""
  import math
  import os
  try:
    n = len(os.sched_getaffinity(0))
  except Exception:
    n = os.cpu_count() or 1
  try:
    with open('/sys/fs/cgroup/cpu.max') as f:
      quota, period = f.read().split()
    if quota != 'max':
      n = min(n, max(1, int(math.ceil(int(quota) / int(period)))))
  except Exception:
    try:
      with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
        q = int(f.read())
      with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
        per = int(f.read())
      if q > 0:
        n = min(n, max(1, int(math.ceil(q / per))))
    except Exception:
      pass
  return n


def pick_threads(learner, make_inputs, limit):
  """The batch-32 learner does not scale to every core (64 OpenMP threads were 3-4x SLOWER than 8 on the GPU box's host, and
  the reference arm's throughput varied 8 -> 36 steps/s between runs): time two updates per candidate thread count and keep
  the fastest, so the CPU baseline is the strongest and most repeatable one this host can give."""
  best, best_t = None, None
  for t in [c for c in (4, 8, 16, 32, 64, 128) if c <= limit] or [limit]:
    torch.set_num_threads(t)
    learner.update(*make_inputs())           # warm the thread pool
    t0 = time.perf_counter()
    for _ in range(2):
      learner.update(*make_inputs())
    dt = time.perf_counter() - t0
    if best_t is None or dt < best_t:
      best, best_t = t, dt
    if dt > 4.0 * best_t:                    # far past the optimum: larger counts only get worse
      break
  torch.set_num_threads(best)
  return best


def run(kind='rainbow', capacity=1000000, batch=32, steps=20, warmup=3, seed=1, threads=None, budget_s=60.0, prewarm=0):
  """Returns dict(steps_per_s, replay_ms, learner_ms, steps, cores).  threads: an int, None (torch default) or 'auto'
  (calibrated thread count within the CPUs this process may use).  budget_s: wall-clock seconds after which the timed
  steps stop early; None runs all `steps`."""
  t_start = time.perf_counter()
  if threads and threads != 'auto':
    torch.set_num_threads(threads)
  rep, prioritized = build_replay(kind, capacity, batch, seed)
  spec = lo.NetSpec(kind, 6)
  learner = lo.Learner(spec, lo.init_params(spec, seed), dtype=torch.float32)
  gen = torch.Generator().manual_seed(seed)
  if threads == 'auto':
    def make_inputs():
      if prioritized:
        tr, ids, w = rep.sample(batch)
        weights = torch.as_tensor(w)
      else:
        tr, weights = rep.sample(batch), None
      b = lo.batch_from_numpy(tr.s_tm1, tr.a_tm1, tr.r_t, tr.discount_t, tr.s_t)
      taus = [torch.rand(batch, 64, generator=gen) for _ in range(3)] if kind == 'iqn' else None
      noise = None
      if kind == 'rainbow':
        noise = []
        for _ in range(3):
          one = {}
          for name, n in lo.noise_shapes(spec):
            x = torch.randn(n, generator=gen).clamp(-2, 2)
            one[name] = torch.sign(x) * torch.sqrt(torch.abs(x))
          noise.append(one)
      return b, weights, taus, noise
    pick_threads(learner, make_inputs, cgroup_cpu_limit())
  cores = torch.get_num_threads()
  t_replay = t_learn = 0.0
  done = 0
  t_begin = None
  warmup = warmup + prewarm   # pre-warm steps are untimed like the warm-up, but not part of the reported warm-up count
  for it in range(warmup + steps):
    if it == warmup:
      t_replay = t_learn = 0.0
      t_begin = time.perf_counter()
    t0 = time.perf_counter()
    if prioritized:
      tr, ids, w = rep.sample(batch)
      weights = torch.as_tensor(w)
    else:
      tr = rep.sample(batch)
      ids, weights = None, None
    t1 = time.perf_counter()
    b = lo.batch_from_numpy(tr.s_tm1, tr.a_tm1, tr.r_t, tr.discount_t, tr.s_t)
    taus = [torch.rand(batch, 64, generator=gen) for _ in range(3)] if kind == 'iqn' else None
    noise = None
    if kind == 'rainbow':
      noise = []
      for _ in range(3):
        one = {}
        for name, n in lo.noise_shapes(spec):
          x = torch.randn(n, generator=gen).clamp(-2, 2)
          one[name] = torch.sign(x) * torch.sqrt(torch.abs(x))
        noise.append(one)
    aux = learner.update(b, weights, taus, noise)
    t2 = time.perf_counter()
    if prioritized:
      rep.update_priorities(ids, aux['priorities'].numpy())
    t3 = time.perf_counter()
    t_replay += (t1 - t0) + (t3 - t2)
    t_learn += t2 - t1
    if it >= warmup:
      done += 1
      if budget_s is not None and time.perf_counter() - t_begin > budget_s:
        break
    elif budget_s is not None and time.perf_counter() - t_start > 2.0 * budget_s and it + 1 < warmup:
      warmup = it + 1          # a pathologically slow host: stop warming up, time what the budget allows
  wall = time.perf_counter() - t_begin
  return {'steps_per_s': done / wall, 'replay_ms': 1e3 * t_replay / done, 'learner_ms': 1e3 * t_learn / done,
          'steps': done, 'cores': cores, 'wall_s': wall}
