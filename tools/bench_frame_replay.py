"""Raw store vs frame-deduplicated store (replay `frame_capacity`), one JSON line per measurement:
  * grad-steps/s of the fused learner step (bench.build_agent's agents, CUDA graph) for rainbow (PER, n = 3) and dqn
    (uniform) at C = 1M, batch 32, the two stores alternated with the same seeds;
  * the frame_assemble_kernel's share of the step, from the in-graph timeline (dz_debug_timeline: its start to the next
    kernel's start) and from eager per-launch CUDA events;
  * the device bytes each store holds;
  * add() latency from host and from device observations;
  * K learners on one GPU, each with a 1M frame store (K = 1, 2, 4, 8): aggregate grad-steps/s, device memory in use.
  python tools/bench_frame_replay.py [--steps 400] [--warmup 50] [--out profiles/frame_replay.jsonl]"""

import argparse
import ctypes as C
import functools
import gc
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from dqn_zoo_b200 import _lib  # noqa: E402
from dqn_zoo_b200 import replay as replay_lib  # noqa: E402

OUT = []


def emit(line, path):
  OUT.append(line)
  print(json.dumps(line), flush=True)
  if path:
    with open(path, 'a') as f:
      f.write(json.dumps(line) + '\n')


def card():
  q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                     text=True).stdout.strip().splitlines()
  return q[0] if q else 'unknown'


def build(agent, capacity, frame_capacity, seed=1):
  """bench.build_agent with the replay classes building a frame store when frame_capacity is set."""
  args = argparse.Namespace(agent=agent, capacity=capacity, batch=32, seed=seed, no_graph=False)
  orig = replay_lib.TransitionReplay, replay_lib.PrioritizedTransitionReplay
  if frame_capacity:
    replay_lib.TransitionReplay = functools.partial(orig[0], frame_capacity=frame_capacity)
    replay_lib.PrioritizedTransitionReplay = functools.partial(orig[1], frame_capacity=frame_capacity)
  try:
    return bench.build_agent(args, 0, torch.device('cuda', 0))
  finally:
    replay_lib.TransitionReplay, replay_lib.PrioritizedTransitionReplay = orig


def steps_per_s(ags, steps, warmup):
  for _ in range(warmup):
    for ag in ags:
      ag.learn()
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for _ in range(steps):
    for ag in ags:
      ag.learn()
  torch.cuda.synchronize()
  return steps * len(ags) / (time.perf_counter() - t0)


def assemble_times(ag, steps=40):
  """(eager CUDA-event ms of frame_assemble_kernel per step, in-graph start-to-next-start us, graph step period us)."""
  ag._use_graph = False
  ag.learn()
  _lib.call('dz_profile_begin')
  ag.learn()
  buf = C.create_string_buffer(1 << 16)
  _lib.call('dz_profile_end', buf, len(buf))
  prof = json.loads(buf.value.decode())
  ev = prof.get('frame_assemble_kernel')
  ag._use_graph = True
  for _ in range(5):
    ag.learn()
  torch.cuda.synchronize()
  tl = torch.zeros(2 + 2 * 4000, dtype=torch.int64, device='cuda')
  _lib.call('dz_debug_timeline', tl.data_ptr())
  for _ in range(steps):
    ag.learn()
  torch.cuda.synchronize()
  _lib.call('dz_debug_timeline', 0)
  t = tl.cpu().numpy()
  n = int(t[0] & 0xffffffff)
  ts, sig = t[2:2 + 2 * n:2], t[3:3 + 2 * n:2].astype(np.uint64)
  order = np.argsort(ts, kind='stable')
  ts, sig = ts[order], sig[order]
  want = (ev[2] << 32) | (ev[3] << 16) | ev[4] if ev else None
  gaps = [ts[i + 1] - ts[i] for i in range(n - 1) if int(sig[i]) == want]
  per = n // steps
  period = float(np.diff(ts[::per]).mean() / 1e3) if per else float('nan')
  return (ev[1] / ev[0] if ev else None), (float(np.median(gaps)) / 1e3 if gaps else None), period


def add_latency(frame_capacity, device_source, n=300):
  rep = replay_lib.TransitionReplay(4096, replay_lib.Transition(None, None, None, None, None), np.random.RandomState(0),
                                    frame_capacity=frame_capacity)
  rs = np.random.RandomState(1)
  frames = [rs.randint(0, 256, size=(84, 84), dtype=np.uint8) for _ in range(n + 4)]
  stacks = [np.stack(frames[i:i + 4], axis=-1) for i in range(n + 1)]
  if device_source:
    stacks = [torch.as_tensor(s, device='cuda') for s in stacks]
  T = replay_lib.Transition(None, None, None, None, None)
  for i in range(20):
    rep.add(T._replace(s_tm1=stacks[i], a_tm1=0, r_t=0.0, discount_t=1.0, s_t=stacks[i + 1]))
  torch.cuda.synchronize()
  t0 = time.perf_counter()
  for i in range(20, n):
    rep.add(T._replace(s_tm1=stacks[i], a_tm1=0, r_t=0.0, discount_t=1.0, s_t=stacks[i + 1]))
  torch.cuda.synchronize()
  return (time.perf_counter() - t0) / (n - 20) * 1e6


def release():
  gc.collect()
  torch.cuda.empty_cache()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--steps', type=int, default=400)
  ap.add_argument('--warmup', type=int, default=50)
  ap.add_argument('--capacity', type=int, default=1_000_000)
  ap.add_argument('--frame-capacity', type=int, default=1_250_000)
  ap.add_argument('--repeats', type=int, default=2)
  ap.add_argument('--learners', default='1,2,4,8')
  ap.add_argument('--out', default='')
  a = ap.parse_args()
  torch.cuda.set_device(0)
  gpu = card()
  base = {'gpu': gpu, 'capacity': a.capacity, 'frame_capacity': a.frame_capacity, 'batch': 32}
  for agent in ('rainbow', 'dqn'):
    for rep_i in range(a.repeats):
      for store, fc in (('raw', None), ('frames', a.frame_capacity)):
        ag, rep = build(agent, a.capacity, fc)
        rate = steps_per_s([ag], a.steps, a.warmup)
        line = dict(base, kind='step_rate', agent=agent, store=store, repeat=rep_i, grad_steps_per_s=round(rate, 1),
                    store_device_bytes=rep._store.device_bytes)
        if fc and rep_i == 0:
          ev_ms, gap_us, period = assemble_times(ag)
          line.update(assemble_event_ms=ev_ms, assemble_in_graph_us=gap_us, graph_step_period_us=period)
        emit(line, a.out)
        del ag, rep
        release()
  for store, fc in (('raw', None), ('frames', 8192)):
    for src in ('host', 'device'):
      emit(dict(base, kind='add_latency', store=store, source=src, us_per_add=round(add_latency(fc, src == 'device'), 2)),
           a.out)
  for k in [int(x) for x in a.learners.split(',')]:
    ags = []
    try:
      for i in range(k):
        ags.append(build('rainbow', a.capacity, a.frame_capacity, seed=1 + i))
      rate = steps_per_s([g for g, _ in ags], a.steps // 2, a.warmup)
      emit(dict(base, kind='learners_per_gpu', agent='rainbow', store='frames', learners=k,
                aggregate_grad_steps_per_s=round(rate, 1), memory_allocated_gb=round(torch.cuda.memory_allocated() / 1e9, 2)),
           a.out)
    except torch.cuda.OutOfMemoryError as e:   # reported, not hidden: the row says how far K went
      emit(dict(base, kind='learners_per_gpu', store='frames', learners=k, error='out of memory: %s' % str(e)[:120]), a.out)
    del ags
    release()


if __name__ == '__main__':
  main()
