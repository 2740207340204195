#!/usr/bin/env python
"""Benchmark of the dqn_zoo hot path (replay sample -> learner update -> priority write-back).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--agent rainbow|dqn|c51|iqn|...]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
      bench.py --gpus N --steps K --warmup W

Prints ONE JSON line (rank 0).  Metric = BASELINE.json's: learner grad-steps/s (sampled
transitions/s = x batch) on a synthetic 84x84x4 uint8 replay of 1M transitions, batch 32.
`value`  : inputs resident in HBM (pre-uploaded RandomState draws), CUDA-graph step, CUDA events.
`e2e`    : the public agent.learn() call: host RandomState draws -> pinned -> H2D every step and an
           asynchronous D2H of the step's loss every step.
`roofline`: the dominant kernel of the step, timed with CUDA events on its stream (dz_profile_*).
`cpu_baseline` / `--impl reference`: the oracle PORT of the reference algorithm on the host cores
(JAX is not installable here or on the GPU box; see oracle/cpu_reference.py).
`--dump-outputs DIR`: after the timed steps, the results of the last timed step as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments, hence the same inputs, can be compared output for output.
"""

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

AGENT_SETUP = {
    # kind: (prioritized, priority_exponent, n_step, target_period_in_learner_steps)
    'dqn': (False, 0.0, 1, 40000 // 16), 'double_q': (False, 0.0, 1, 120000 // 16),
    'prioritized': (True, 0.6, 1, 120000 // 16), 'c51': (False, 0.0, 1, 40000 // 16),
    'qrdqn': (False, 0.0, 1, 40000 // 16), 'rainbow': (True, 0.5, 3, 32000 // 16), 'iqn': (False, 0.0, 1, 40000 // 16),
}
# learner FLOPs per step, B*F_fwd*(n_fwd+2), SURVEY §8(a) (A = 6)
GFLOP_PER_STEP = {'dqn': 2.39, 'double_q': 2.99, 'prioritized': 2.99, 'c51': 2.43, 'qrdqn': 2.55, 'rainbow': 4.65, 'iqn': 39.5}


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=2000)
  ap.add_argument('--warmup', type=int, default=200)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--agent', default='rainbow', choices=sorted(AGENT_SETUP))
  ap.add_argument('--capacity', type=int, default=1000000)
  ap.add_argument('--batch', type=int, default=32)
  ap.add_argument('--seed', type=int, default=1)
  ap.add_argument('--no-graph', action='store_true')
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--cpu-steps', type=int, default=40)
  ap.add_argument('--dump-outputs', metavar='DIR', default=None)
  args = ap.parse_args()
  if args.dump_outputs and args.impl != 'ours':
    ap.error('--dump-outputs writes the results of the CUDA path (--impl ours)')
  return args


def workload_name(args):
  pri, alpha, n, _ = AGENT_SETUP[args.agent]
  rep = 'per_alpha%g' % alpha if pri else 'uniform'
  return '%s_%s_nstep%d_cap%d_b%d_84x84x4' % (args.agent, rep, n, args.capacity, args.batch)


def config_of(args, target_period):
  """The workload description; identical for `--impl ours` and `--impl reference` (the driver compares them)."""
  return {'workload': workload_name(args), 'agent': args.agent, 'replay_capacity': args.capacity, 'batch': args.batch,
          'replay_bytes_per_gpu': int(args.capacity) * 2 * 84 * 84 * 4, 'obs': '84x84x4 uint8',
          'target_sync_period_steps': target_period,
          'l2': 'inputs larger than L2: 56.4 GB replay store sampled at random rows; parameters+optimizer state as in '
                'steady-state training',
          'multi_gpu': 'independent replay+learner shard per rank; the target refresh is an NCCL broadcast of the online blob',
          'seed': args.seed}


class ClockSampler:
  """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

  def __init__(self, index):
    self.rows, self.proc, self.index = [], None, index

  def start(self):
    q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '100',
                                    '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._pump, daemon=True)
      self.thread.start()
    except Exception:
      self.proc = None

  def _pump(self):
    for line in self.proc.stdout:
      self.rows.append(line.strip().split(', '))

  def stop(self):
    if self.proc is None:
      return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
    time.sleep(0.15)
    self.proc.terminate()
    sm, mx, reasons = [], [], set()
    for r in self.rows:
      try:
        sm.append(float(r[1])); mx.append(float(r[2]))
        for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
          if v.strip().lower().startswith('active'):
            reasons.add(name)
      except Exception:
        pass
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as f:
      p = json.load(f)
    return p.get('hbm_gbs', 6650.0), p.get('bf16_tflops', 1590.0), 'measured (MEASURED_PEAKS.json)'
  return 6650.0, 1590.0, 'fallback (B200_PROFILING.md)'


def host_cores():
  try:
    return len(os.sched_getaffinity(0))
  except Exception:
    return os.cpu_count() or 1


def reference_arm(args, rank, world):
  """The oracle PORT of the reference algorithm on the host cores (rank 0 only; the other ranks exit without work).
  torchrun exports OMP_NUM_THREADS=1, so the thread count is set explicitly: calibrated over {4, 8, ..., CPUs this process
  may use} (the batch-32 learner is 3-4x slower on 64 OpenMP threads than on 8) and reported.  Ten untimed pre-warm steps
  (thread pools, allocator) come before the W warm-up + K timed steps."""
  if rank != 0:
    return
  from oracle import cpu_reference
  steps, warmup = max(1, args.steps), max(0, args.warmup)
  res = cpu_reference.run(args.agent, capacity=args.capacity, batch=args.batch, steps=steps, warmup=warmup, seed=args.seed,
                          threads='auto', prewarm=10, budget_s=None)
  value = res['steps_per_s']
  sample = ('%d learner steps (replay.sample + update + update_priorities) of %s after %d warm-up (+10 pre-warm) steps; replay '
            '%.2f ms + learner %.2f ms per step; observations reference a pool of 512 synthetic frames'
            % (res['steps'], workload_name(args), warmup, res['replay_ms'], res['learner_ms']))
  line = {
      'impl': 'reference', 'metric': 'learner_grad_steps_per_sec', 'value': value, 'unit': 'grad-steps/s',
      'sampled_transitions_per_sec': value * args.batch, 'n_gpus': args.gpus, 'steps': res['steps'],
      'warmup': warmup, 'ms_per_step': 1e3 / value, 'higher_is_better': True, 'scaling': 'weak',
      'vs_baseline': None, 'dtype': 'f32 (f64 sum tree)', 'data': 'synthetic',
      'config': config_of(args, AGENT_SETUP[args.agent][3]),
      'impl_note': 'oracle port (numpy replay, one thread as the reference; torch-CPU float32 learner on all host cores); the '
                   'JAX CPU path is not installable here or on the GPU box',
      'cpu_baseline': {'value': value, 'unit': 'grad-steps/s', 'cores': res['cores'], 'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': 'grad-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
      'gpu_launches': 0,
  }
  emit(line)


def build_agent(args, rank, device):
  from dqn_zoo_b200 import agent as agent_lib
  from dqn_zoo_b200 import learner as learner_lib
  from dqn_zoo_b200 import parts
  from dqn_zoo_b200 import replay as replay_lib
  pri, alpha, n_step, _ = AGENT_SETUP[args.agent]
  kind = args.agent
  from dqn_zoo_b200 import distributed as dz_dist
  seed = dz_dist.shard_seed(args.seed, rank)
  rs = np.random.RandomState(seed)
  structure = replay_lib.Transition(None, None, None, None, None)
  if pri:
    sched = parts.LinearSchedule(begin_t=int(0.02 * args.capacity), end_t=200 * 250000, begin_value=0.4, end_value=1.0)
    rep = replay_lib.PrioritizedTransitionReplay(args.capacity, structure, alpha, sched, 1e-3, True, rs)
  else:
    rep = replay_lib.TransitionReplay(args.capacity, structure, rs)
  replay_lib.bulk_fill_synthetic(rep, (84, 84, 4), seed, 6, discount=0.99 ** n_step)
  net = learner_lib.NetworkSpec(kind, 6)
  acc = replay_lib.NStepTransitionAccumulator(n_step)
  common = dict(preprocessor=lambda ts: ts, sample_network_input=np.zeros((84, 84, 4), np.uint8), network=net,
                optimizer=None, transition_accumulator=acc, replay=rep, batch_size=args.batch,
                min_replay_capacity_fraction=0.02, learn_period=16, target_network_update_period=32000, rng_key=[0, seed],
                use_cuda_graph=not args.no_graph)
  eps = lambda t: 0.01
  if kind == 'rainbow':
    ag = agent_lib.Rainbow(support=np.linspace(-10, 10, 51), **common)
  elif kind == 'c51':
    ag = agent_lib.C51(support=np.linspace(-10, 10, 51), exploration_epsilon=eps, **common)
  elif kind == 'qrdqn':
    ag = agent_lib.QrDqn(quantiles=(np.arange(201) + 0.5) / 201, exploration_epsilon=eps, huber_param=1.0, **common)
  elif kind == 'iqn':
    ag = agent_lib.Iqn(exploration_epsilon=eps, huber_param=1.0, tau_samples_policy=64, tau_samples_s_tm1=64,
                       tau_samples_s_t=64, **common)
  else:
    ag = agent_lib.AGENTS[kind](exploration_epsilon=eps, grad_error_bound=1.0 / 32, **common)
  return ag, rep


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, ag, L, prioritized):
  """Writes what the last learner step returned to its caller, as float32 / float64 .npy files: the loss, the per-example
  loss, the new priorities, the global gradient norm, the sampled ids (as float64, exact below 2^53) and importance
  weights, the updated online parameters and, with prioritized replay, the sum-tree leaves of the sampled transitions after
  the priority write-back, the tree's root and the running max priority."""
  arrays = {'loss': L.loss, 'per_example_loss': L.per_example, 'priorities': L.priorities, 'grad_norm': L.grad_norm,
            'sampled_ids': L.sampled_ids.double(), 'importance_weights': L.sampled_weights, 'online_params': L.online}
  if prioritized:
    tree = ag._replay._distribution._sum_tree
    arrays['sum_tree_leaves_sampled'] = tree._nodes[tree._first_leaf + L.sampled_indices]
    arrays['sum_tree_root'] = tree._nodes[1:2]
    arrays['max_seen_priority'] = L.max_seen_priority
  arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
  total = sum(a.nbytes for a in arrays.values())
  assert total <= DUMP_LIMIT_BYTES, 'outputs of %d bytes exceed the dump limit' % total
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    assert a.dtype in (np.float32, np.float64), (name, a.dtype)
    np.save(os.path.join(out_dir, name + '.npy'), a)


_REAL_STDOUT = None


def guard_stdout():
  """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on rank 0),
  so file descriptor 1 is pointed at stderr for the whole run and the JSON line goes to the saved descriptor."""
  global _REAL_STDOUT
  if _REAL_STDOUT is None:
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
    os.dup2(2, 1)


def emit(line):
  out = _REAL_STDOUT or sys.stdout
  out.write(json.dumps(line) + '\n')
  out.flush()


def main():
  args = parse()
  guard_stdout()
  rank = int(os.environ.get('RANK', '0'))
  local_rank = int(os.environ.get('LOCAL_RANK', '0'))
  world = int(os.environ.get('WORLD_SIZE', '1'))
  if args.impl == 'reference':
    reference_arm(args, rank, world)
    return
  if not torch.cuda.is_available():
    raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
  torch.cuda.set_device(local_rank)
  device = torch.device('cuda', local_rank)
  dist = None
  if world > 1:
    import torch.distributed as dist
    dist.init_process_group('nccl', device_id=device)
  from dqn_zoo_b200 import _lib

  ag, rep = build_agent(args, rank, device)
  L = ag.learner
  K, W, B = args.steps, max(args.warmup, 3), args.batch
  target_period = AGENT_SETUP[args.agent][3]

  from dqn_zoo_b200 import distributed as dz_dist

  def sync_target():
    # BASELINE configs[4]: periodic online->target parameter broadcast over NCCL/NVLink.  Root 0's
    # online net becomes every shard's target (shared-target reading, DESIGN.md §6); at N=1 it is the
    # reference's plain target <- online copy.
    dz_dist.broadcast_target(L.online, L.target, dist, src=0)

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()

  # ---- (1) value: draws resident in HBM ---------------------------------------------------------
  draws = np.stack([ag.host_draws() for _ in range(W + K)])
  d_draws = torch.as_tensor(draws, device=device)
  for i in range(W):
    ag.learn_from_device_draws(d_draws[i])
  sync_target()   # warm-up of the refresh path too (the first NCCL broadcast pays communicator set-up: 1.6 ms measured at N = 2)
  barrier()
  launches_before = _lib.lib.dz_launch_count()
  clocks = ClockSampler(local_rank)
  clocks.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  # The target refresh (an NCCL broadcast at N > 1) must be inside every timed region, however short: it runs every
  # `sync_every` = min(target period, K) steps, i.e. at least once (the reference's cadence is `target_period`).
  sync_every = max(1, min(target_period, K))
  coll_events = []
  barrier()
  e0.record()
  for i in range(K):
    ag.learn_from_device_draws(d_draws[W + i])
    if (i + 1) % sync_every == 0:
      c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      c0.record()
      sync_target()
      c1.record()
      coll_events.append((c0, c1))
  e1.record()
  barrier()
  clk = clocks.stop()
  ms = e0.elapsed_time(e1)
  if args.dump_outputs and rank == 0:
    ag.check_device_flags()   # a step that set an error flag leaves no outputs behind that look valid
    dump_outputs(args.dump_outputs, ag, L, AGENT_SETUP[args.agent][0])
  collective_us = 1e3 * float(np.mean([a.elapsed_time(b) for a, b in coll_events])) if coll_events else None
  t = torch.tensor([ms], dtype=torch.float64, device=device)
  if dist is not None:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  ms_max = float(t.item())
  value = world * K / (ms_max / 1e3)
  ag.check_device_flags()

  # ---- (2) e2e: public learn() with host draws + H2D + D2H of the loss every step ---------------
  loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()
  for i in range(3):
    ag.learn()
  barrier()
  e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t_host0 = time.perf_counter()
  e2.record()
  for i in range(K):
    ag.learn()
    loss_host[i:i + 1].copy_(L.loss, non_blocking=True)
    if (i + 1) % sync_every == 0:
      sync_target()
  e3.record()
  barrier()
  t_host = time.perf_counter() - t_host0
  ms_e2e = max(e2.elapsed_time(e3), 1e3 * t_host)
  t = torch.tensor([ms_e2e], dtype=torch.float64, device=device)
  if dist is not None:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
  e2e_value = world * K / (float(t.item()) / 1e3)
  assert np.isfinite(loss_host.numpy()).all(), 'non-finite loss in the e2e run'
  ag.check_device_flags()

  # ---- (3) launches per step + per-kernel timing (outside every timed region) --------------------
  ag._use_graph = False
  c0 = _lib.lib.dz_launch_count()
  ag.learn()
  torch.cuda.synchronize()
  launches_per_step = int(_lib.lib.dz_launch_count() - c0)
  prof_steps = 50
  _lib.call('dz_profile_begin')
  for i in range(prof_steps):
    ag.learn()
  buf = C.create_string_buffer(1 << 16)
  _lib.call('dz_profile_end', buf, len(buf))
  prof = json.loads(buf.value.decode())
  total_ms = sum(v[1] for v in prof.values())
  top = max(prof.items(), key=lambda kv: kv[1][1])
  per_launch_us = {k: 1e3 * v[1] / v[0] for k, v in prof.items()}
  share = {k: round(v[1] / total_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])[:8]}

  # ---- (3b) device timeline of the CUDA-graph step: every kernel stamps %globaltimer when its dependencies have completed
  # (dz_debug_timeline); a kernel's time = its start to the next start in the step (the last one: to the step's end).
  # Eager per-launch events above include the host's launch latency whenever the host is the bottleneck (they read 52 us
  # for a 37 us optimizer launch), so the roofline below uses the graph timeline and reports the event figure beside it.
  graph_us, graph_share, graph_step_us = {}, {}, None
  if not args.no_graph:
    ag._use_graph = True
    for i in range(5):
      ag.learn()
    torch.cuda.synchronize()
    tl_steps = 40
    tl = torch.zeros(2 + 2 * 4000, dtype=torch.int64, device=device)
    _lib.call('dz_debug_timeline', tl.data_ptr())
    for i in range(tl_steps):
      ag.learn_from_device_draws(d_draws[i % (W + K)])
    torch.cuda.synchronize()
    _lib.call('dz_debug_timeline', 0)
    t = tl.cpu().numpy()
    n = int(t[0] & 0xffffffff)
    per = n // tl_steps
    if per * tl_steps == n and per > 0 and n <= 4000:
      ts = t[2:2 + 2 * n:2].astype(np.int64)
      sg = t[3:3 + 2 * n:2].astype(np.int64)
      order = np.argsort(ts, kind='stable')
      ts, sg = ts[order].reshape(tl_steps, per)[2:], sg[order].reshape(tl_steps, per)[2:]
      graph_step_us = float(np.median(np.diff(ts[:, 0])) / 1e3)   # median: steps whose replay the host submitted late drop out
      nxt = np.concatenate([ts[:, 1:], ts[:, :1] + int(round(graph_step_us * 1e3))], axis=1)
      dur = np.median(nxt - ts, axis=0) / 1e3
      by_geo = {}
      for k, v in prof.items():
        by_geo.setdefault((int(v[2]), int(v[3]), int(v[4])), []).append(k)
      for j in range(per):
        g = int(sg[-1, j])
        names = by_geo.get((g >> 32, (g >> 16) & 0xffff, g & 0xffff), ['?'])
        key = '/'.join(names)
        graph_us[key] = graph_us.get(key, 0.0) + float(dur[j])
      graph_share = {k: round(v / graph_step_us, 4) for k, v in sorted(graph_us.items(), key=lambda kv: -kv[1])[:8]}
    ag._use_graph = False

  hbm_peak, tf_peak, peak_src = measured_peaks()
  # Dominant-kernel roofline.  Algorithmic bytes per launch of each candidate (DESIGN.md §5):
  P = L.plan.param_count
  alg_bytes = {
      # noisy fc1 (rainbow): 2 streams x (mu.w + sigma.w) x {online, target} weights read once + 3 x feat reads
      'noisy1_fwd': 2 * 2 * 2 * 3136 * 512 * 4 + 3 * B * 3136 * 4,
      'noisy1_wgrad': 2 * 2 * 3136 * 512 * 4 + B * (3136 + 1024) * 4,
      'noisy1_dgrad': 2 * 2 * 3136 * 512 * 4 + B * (3136 + 1024) * 4 * 2,
      'fc1_fwd': 2 * 3136 * 512 * 4 + 3 * B * 3136 * 4,
      'fc1_wgrad': 3136 * 512 * 4 + B * (3136 + 512) * 4,
      'fc1_dgrad': 3136 * 512 * 4 + B * (3136 + 512) * 4,
      'optimizer_kernel': 7 * 4 * P,
      'grad_norm_kernel': 4 * P,
      'conv1_fwd': (3 if args.agent in ('rainbow', 'double_q', 'prioritized') else 2) * B * (28224 + 20 * 20 * 32 * 4),
  }
  name = top[0]
  dur_s = 1e-3 * top[1][1] / top[1][0]
  event_us = 1e6 * dur_s
  timing_source = 'cuda events around each eager launch (dz_profile)'
  single = {k: v for k, v in graph_us.items() if '/' not in k and k in prof}
  if single:
    # stable choice: the kernel with the largest share of the graph-replayed step; per-launch time = its share / launches
    name = max(single.items(), key=lambda kv: kv[1])[0]
    launches_in_step = max(1, int(round(prof[name][0] / prof_steps)))
    dur_s = 1e-6 * single[name] / launches_in_step
    event_us = 1e3 * prof[name][1] / prof[name][0]
    timing_source = 'device %globaltimer stamps inside the CUDA-graph step (dz_debug_timeline)'
  traffic, ncu_facts = None, {}
  try:
    with open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')) as f:
      ncu_facts = json.load(f).get(args.agent, {})
    traffic = ncu_facts.get('dram_bytes', {}).get(name)
  except Exception:
    traffic = None
  # dense-contraction kernels: algorithmic FLOPs per launch (2*M*N*K per problem, SURVEY §2.1 shapes)
  npass = 3 if args.agent in ('rainbow', 'double_q', 'prioritized') else 2
  nq = 64
  alg_flops = {
      'conv1_fwd': npass * B * 400 * 256 * 32 * 2, 'conv2_fwd': npass * B * 81 * 512 * 64 * 2, 'conv3_fwd': npass * B * 49 * 576 * 64 * 2,
      'conv1_wgrad': B * 400 * 256 * 32 * 2, 'conv2_wgrad': B * 81 * 512 * 64 * 2, 'conv3_wgrad': B * 49 * 576 * 64 * 2,
      'conv2_dgrad': B * 81 * 512 * 64 * 2, 'conv3_dgrad': B * 49 * 576 * 64 * 2,
      'iqn_fc1_fwd': 3 * B * nq * 3136 * 512 * 2, 'iqn_fc1_wgrad': B * nq * 3136 * 512 * 2, 'iqn_fc1_dgrad': B * nq * 3136 * 512 * 2,
      'iqn_embed_fwd': 3 * B * nq * 64 * 3136 * 2, 'iqn_embed_wgrad': B * nq * 64 * 3136 * 2,
  }
  if name in alg_bytes and name not in alg_flops:
    achieved = alg_bytes[name] / dur_s / 1e9
    roofline = {'kernel': name, 'bound': 'hbm', 'achieved': achieved, 'peak': hbm_peak, 'unit': 'GB/s',
                'frac': achieved / hbm_peak, 'traffic': traffic, 'alg_bytes_per_launch': alg_bytes[name],
                'avg_launch_us': 1e6 * dur_s, 'peak_source': peak_src}
  elif name in alg_flops:
    achieved = alg_flops[name] / dur_s / 1e12
    roofline = {'kernel': name, 'bound': 'tensor', 'achieved': achieved, 'peak': tf_peak, 'unit': 'TFLOP/s',
                'frac': achieved / tf_peak, 'traffic': traffic, 'alg_flops_per_launch': alg_flops[name],
                'avg_launch_us': 1e6 * dur_s, 'peak_source': peak_src,
                'note': ('tcgen05 kernel (csrc/dz_tcp.cuh): error-compensated 3xTF32, i.e. three kind::tf32 MMAs per fp32 product '
                         'to hold the 1e-5 parity bar; `achieved` counts the algorithmic 2*M*N*K only, the peak is the measured '
                         'dense bf16 tensor throughput')
                        if name.startswith('iqn_') and os.environ.get('DZ_PK_IQN', '1') != '0' else
                        ('fp32 FMA kernel today (exact-fp32 products for the 1e-5 parity bar); the peak is the measured dense bf16 '
                         'tensor throughput, i.e. the fraction states how far this contraction is from the tensor-core roofline')}
  else:
    flops = GFLOP_PER_STEP[args.agent] * 1e9
    achieved = flops / (1e-3 * total_ms / prof_steps) / 1e12
    roofline = {'kernel': name, 'bound': 'tensor', 'achieved': achieved, 'peak': tf_peak, 'unit': 'TFLOP/s',
                'frac': achieved / tf_peak, 'traffic': traffic, 'avg_launch_us': 1e6 * dur_s, 'peak_source': peak_src,
                'note': 'whole-step algorithmic FLOPs over summed kernel time'}
  roofline['kernel_time_share'] = graph_share or share
  roofline['timing_source'] = timing_source
  roofline['event_us_eager'] = event_us
  # north-star fields: HBM GB/s on sample + gather, tensor-pipe % on the conv stack, whole-step HBM fraction
  gather_bytes = 2 * B * 28224 + 12 * B + (20480 if AGENT_SETUP[args.agent][0] else 0)
  sampler = 'per_sample_kernel' if AGENT_SETUP[args.agent][0] else 'uniform_sample_kernel'
  sg_us = (graph_us.get(sampler, per_launch_us.get(sampler, float('nan'))) +
           graph_us.get('conv1_fwd', per_launch_us.get('conv1_fwd', float('nan'))))
  roofline['sample_gather_gbs'] = gather_bytes / (sg_us * 1e-6) / 1e9
  roofline['sample_gather'] = {
      'alg_bytes_per_step': gather_bytes, 'us': sg_us, 'frac_of_hbm_peak': gather_bytes / (sg_us * 1e-6) / 1e9 / hbm_peak,
      'note': 'sampler kernel + conv1_fwd (the gather of the sampled rows IS conv1_fwd\'s bulk-copy operand load): '
              'latency-bound at batch 32 (1.8 MB per step)'}
  step_bytes = sum(alg_bytes[k] * max(1, int(round(prof[k][0] / prof_steps))) for k in alg_bytes if k in prof)
  step_s = (graph_step_us * 1e-6) if graph_step_us else (ms_max / K / 1e3)
  roofline['step_hbm_frac'] = step_bytes / step_s / 1e9 / hbm_peak
  roofline['step_alg_bytes'] = step_bytes
  roofline['conv_tensor_pipe_pct'] = ncu_facts.get('tensor_pipe_pct')   # ncu sm__pipe_tensor_cycles_active of this build (profiles/)

  # ---- (4) CPU baseline (rank 0, N = 1 only) ---------------------------------------------------------
  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    from oracle import cpu_reference
    res = cpu_reference.run(args.agent, capacity=args.capacity, batch=B, steps=args.cpu_steps, warmup=2, seed=args.seed,
                            threads='auto', budget_s=25.0)
    cpu = {'value': res['steps_per_s'], 'unit': 'grad-steps/s', 'cores': res['cores'], 'kind': 'port',
           'sample': '%d learner steps of the same workload: numpy replay %.2f ms + torch-CPU f32 learner %.2f ms per step'
                     % (res['steps'], res['replay_ms'], res['learner_ms'])}

  if rank == 0:
    stage_bytes = (3 * B + 4) * 8
    line = {
        'metric': 'learner_grad_steps_per_sec', 'value': value, 'unit': 'grad-steps/s',
        'sampled_transitions_per_sec': value * B, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms_max / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32 (f64 sum tree)', 'data': 'synthetic',
        'config': config_of(args, target_period),
        'run': {'cuda_graph': not args.no_graph, 'replay_bytes_allocated': int(rep._store.obs.numel()),
                'optimizer_state_mb': 7 * 4 * P / 1e6, 'target_sync_every_steps_in_timed_region': sync_every,
                'target_syncs_in_timed_region': len(coll_events), 'collective_us': collective_us,
                'collective': ('ncclBroadcast of the %.1f MB online blob into every rank\'s target' % (4 * P / 1e6)) if world > 1
                              else 'device-to-device copy online -> target (one rank)'},
        'collective_us': collective_us,
        'clocks': clk,
        'e2e': {'value': e2e_value, 'unit': 'grad-steps/s', 'h2d_bytes_per_step': stage_bytes, 'd2h_bytes_per_step': 4,
                'note': 'agent.learn(): host RandomState draws -> pinned -> H2D; async D2H of the loss each step'},
        'gpu_launches': launches_per_step * K,
        'gpu_launches_per_step': launches_per_step,
        'roofline': roofline,
        'kernel_avg_us': {k: round(v, 2) for k, v in per_launch_us.items()},
        'kernel_graph_us': {k: round(v, 2) for k, v in graph_us.items()},
        'graph_step_us': graph_step_us,
        'learner_gflop_per_step': GFLOP_PER_STEP[args.agent],
        'learner_tflops_achieved': GFLOP_PER_STEP[args.agent] * value / world / 1e3,
        'cpu_baseline': cpu,
    }
    emit(line)
  if dist is not None:
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
