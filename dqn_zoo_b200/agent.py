"""The seven dqn_zoo agents behind the reference's `parts.Agent` surface, running on the
CUDA replay + learner.

Each class keeps the reference constructor's argument names and the `step / reset /
get_state / set_state / statistics` behaviour (dqn/agent.py:133-229, rainbow/agent.py:135-245,
iqn/agent.py:245-340 ...).  Two arguments necessarily change type (SURVEY §8(b)):
  * `network`   is a `learner.NetworkSpec`   instead of an `hk.Transformed`,
  * `optimizer` is a `learner.OptimizerSpec` instead of an `optax.GradientTransformation`,
and `rng_key` seeds a host `np.random.RandomState` (epsilon-greedy) and the device Philox
stream (IQN taus, noisy-net noise) instead of the JAX threefry stream.

`_learn()` is ONE enqueue: host RandomState draws (reference order) -> pinned staging -> H2D ->
[sample -> gather-in-place -> forward x2/3 -> loss -> backward -> optimizer -> priority
write-back], optionally replayed as a CUDA graph.  Nothing is read back per learner step
(the reference's `jax.device_get(priorities)` sync, rainbow/agent.py:195, is gone):
`max_seen_priority` lives on the device and new transitions take their priority from there.
"""

from __future__ import annotations

import ctypes as C
from typing import Any, Callable, Mapping, Optional

import numpy as np
import torch

from dqn_zoo_b200 import _lib
from dqn_zoo_b200 import jax_prng
from dqn_zoo_b200 import learner as learner_lib
from dqn_zoo_b200 import parts
from dqn_zoo_b200 import replay as replay_lib

NetworkSpec = learner_lib.NetworkSpec
OptimizerSpec = learner_lib.OptimizerSpec


def _seed_of(rng_key) -> int:
  arr = np.asarray(rng_key).astype(np.uint64).reshape(-1)
  seed = 0
  for v in arr:
    seed = (seed * 0x9E3779B97F4A7C15 + int(v)) % (1 << 63)
  return seed


class _DeviceAgent(parts.Agent):
  """Shared machinery; subclasses set KIND / PRIORITIZED and mirror the reference constructors."""

  KIND = 'dqn'
  PRIORITIZED = False
  GREEDY = False

  def _setup(self, preprocessor, sample_network_input, network: NetworkSpec, optimizer: Optional[OptimizerSpec],
             transition_accumulator, replay, batch_size, exploration_epsilon, min_replay_capacity_fraction,
             learn_period, target_network_update_period, rng_key, grad_error_bound=1.0 / 32, huber_param=1.0,
             use_cuda_graph=True):
    if network.kind != self.KIND:
      raise ValueError('network spec kind %r does not match agent %r' % (network.kind, self.KIND))
    if sample_network_input is not None and tuple(np.asarray(sample_network_input).shape) != tuple(network.obs_shape):
      raise ValueError('sample_network_input shape %s != network obs_shape %s'
                       % (np.asarray(sample_network_input).shape, network.obs_shape))
    self._preprocessor = preprocessor
    self._replay = replay
    replay.reserve_batch(batch_size)          # before the first view: the staging address is part of a captured graph
    self._transition_accumulator = transition_accumulator
    self._batch_size = batch_size
    self._exploration_epsilon = exploration_epsilon
    self._min_replay_capacity = min_replay_capacity_fraction * replay.capacity
    self._learn_period = learn_period
    self._target_network_update_period = target_network_update_period
    self._seed = _seed_of(rng_key)
    self._host_rng = np.random.RandomState(self._seed % (1 << 32))
    self._learner = learner_lib.Learner(network, batch_size=batch_size, optimizer=optimizer,
                                        grad_error_bound=grad_error_bound, huber_param=huber_param)
    self._learner.init_params(seed=self._seed % (1 << 31))      # network.init + target = online
    self._action = None
    self._frame_t = -1
    self._statistics = {'state_value': np.nan}
    self._use_graph = use_cuda_graph
    self._graph = None
    self._graph_key = None
    self._io = None
    self._obs_dev = torch.zeros(int(np.prod(network.obs_shape)), dtype=torch.uint8, device=self._learner.device)
    B = batch_size
    self._stage_words = 3 * B + 4
    self._stage_dev = torch.zeros(self._stage_words, dtype=torch.float64, device=self._learner.device)
    self._ring = [torch.zeros(self._stage_words, dtype=torch.float64).pin_memory() for _ in range(8)]
    self._ring_events = [None] * len(self._ring)
    self._ring_pos = 0
    self._learn_steps = 0

  # -- parts.Agent -----------------------------------------------------------------------------------
  def step(self, timestep) -> parts.Action:
    """dqn/agent.py:133-158 (identical control flow for every agent)."""
    self._frame_t += 1
    timestep = self._preprocessor(timestep)
    if timestep is None:  # repeat action
      if self._action is None:
        raise RuntimeError('Cannot repeat if action has never been selected.')
      action = self._action
    else:
      action = self._action = self._act(timestep)
      for transition in self._transition_accumulator.step(timestep, action):
        self._add(transition)
    if self._replay.size < self._min_replay_capacity:
      return action
    if self._frame_t % self._learn_period == 0:
      self._learn()
    if self._frame_t % self._target_network_update_period == 0:
      self._learner.sync_target()
      # The fused step only RECORDS bad priorities / non-finite weights as sticky device flags (no per-step D2H sync);
      # read them on the target-update cadence so a diverged run stops with the reference's exceptions
      # (replay.py:281-282 'value must be finite and positive', :240-241 'Weights are not finite') instead of
      # training on with stale priorities.
      self.check_device_flags()
    return action

  def reset(self) -> None:
    """dqn/agent.py:160-167."""
    self._transition_accumulator.reset()
    if hasattr(self._preprocessor, 'reset'):
      self._preprocessor.reset()
    self._action = None

  @property
  def statistics(self) -> Mapping[str, float]:
    return self._statistics

  @property
  def online_params(self):
    """hk.Params-shaped nested dict of host arrays."""
    return self._learner.haiku_params('online')

  @property
  def exploration_epsilon(self) -> float:
    return 0.0 if self._exploration_epsilon is None else self._exploration_epsilon(self._frame_t)

  @property
  def learner(self) -> learner_lib.Learner:
    return self._learner

  def get_state(self) -> Mapping[str, Any]:
    """dqn/agent.py:210-220 / rainbow/agent.py:224-235: same keys."""
    state = {
        'rng_key': {'host': self._host_rng.get_state(), 'seed': self._seed,
                    'device_counter': int(self._learner.counters[1].item())},
        'frame_t': self._frame_t,
        'opt_state': self._learner.get_opt_state(),
        'online_params': self._learner.get_params('online'),
        'target_params': self._learner.get_params('target'),
        'replay': self._replay.get_state(),
    }
    if self.PRIORITIZED:
      state['max_seen_priority'] = self.max_seen_priority
    if getattr(self, '_jax_key', None) is not None:
      state['rng_key']['jax'] = self._jax_key.copy()
    return state

  def set_state(self, state: Mapping[str, Any]) -> None:
    """dqn/agent.py:222-229 / rainbow/agent.py:237-245."""
    self._host_rng.set_state(state['rng_key']['host'])
    self._seed = state['rng_key']['seed']
    self._learner.counters[1] = int(state['rng_key']['device_counter'])
    if getattr(self, '_jax_key', None) is not None:
      self._jax_key = np.asarray(state['rng_key']['jax'], dtype=np.uint32).copy()
    self._frame_t = state['frame_t']
    self._learner.set_opt_state(state['opt_state'])
    self._learner.set_params(state['online_params'], blob='online')
    self._learner.set_params(state['target_params'], blob='target')
    self._replay.set_state(state['replay'])
    if self.PRIORITIZED:
      self._learner.max_seen_priority.fill_(float(state['max_seen_priority']))
    self._graph = None  # device pointers of the replay may have changed

  # -- acting (dqn/agent.py:121-131,169-177) --------------------------------------------------------------
  def _act(self, timestep) -> parts.Action:
    obs = timestep.observation
    if isinstance(obs, torch.Tensor):        # device-resident frame stack (processors.atari(device_observations=True))
      self._obs_dev.copy_(obs.reshape(-1))
    else:
      self._obs_dev.copy_(torch.from_numpy(np.ascontiguousarray(obs).reshape(-1)))
    L = self._learner
    taus = noise = None
    if getattr(self, '_jax_key', None) is not None:
      # iqn/agent.py:220-222: rng_key, sample_key, apply_key, policy_key = split(rng_key, 4); tau_t = uniform(sample_key)
      self._jax_key, sample = jax_prng.iqn_act_keys(self._jax_key)
      self._jax_act.set_keys(sample)
      self._jax_act.launch(L.taus)
      taus = L.taus
    elif self.KIND in ('iqn', 'rainbow'):
      L.generate_randomness(self._seed)
      taus = L.taus if self.KIND == 'iqn' else None
      noise = L.noise if self.KIND == 'rainbow' else None
    q = L.q_values(self._obs_dev, taus=taus, noise=noise).cpu().numpy()   # D2H sync, as jax.device_get
    eps = 0.0 if self.GREEDY else self.exploration_epsilon
    if eps > 0.0 and self._host_rng.uniform() < eps:
      a_t = int(self._host_rng.randint(len(q)))
    else:
      a_t = int(np.argmax(q))
    self._statistics['state_value'] = float(q.max())
    return parts.Action(a_t)

  # -- insert --------------------------------------------------------------------------------------
  def _add(self, transition) -> None:
    if self.PRIORITIZED:
      # rainbow/agent.py:148-149: priority = max_seen_priority (kept on the device)
      self._replay.add(transition, priority=self._learner.max_seen_priority)
    else:
      self._replay.add(transition)

  # -- learn -----------------------------------------------------------------------------------------
  def _draws(self):
    """Host RandomState draws in the reference's order (replay.py:551-567 / :78)."""
    rs = self._replay._random_state
    B = self._batch_size
    size = self._replay.size
    slot = self._ring[self._ring_pos]
    ev = self._ring_events[self._ring_pos]
    if ev is not None:
      ev.synchronize()
    host = slot.numpy()
    host[:B].view(np.int64)[:] = rs.randint(size, size=B)
    if self.PRIORITIZED:
      # Scaled by the root on the device.  KNOWN DIVERGENCE: the reference skips this draw when the root is 0
      # (replay.py:556-560); the root lives on the device here and is not read back per step, so the draw is always
      # consumed and the kernel raises DZ_FLAG_ROOT_ZERO instead (surfaced by check_device_flags on the target-update
      # cadence).  A zero root needs every stored priority to be 0, which the agents' priority rule never produces.
      host[B:2 * B] = rs.uniform(size=B)
      host[2 * B:3 * B] = rs.uniform(size=B)
      dist = self._replay._distribution
      host[3 * B:] = (float(size), float(self._replay.importance_sampling_exponent),
                      float(dist._uniform_sample_probability), 1.0 if self._replay._normalize_weights else 0.0)
    else:
      host[3 * B:] = (float(size), 1.0, 0.0, 0.0)
    return slot

  def _learn(self) -> None:
    """rainbow/agent.py:181-198 as one enqueue."""
    slot = self._draws()
    if getattr(self, '_jax_key', None) is not None:
      # iqn/agent.py:207 + 182: the agent key advances once per update; three sample keys feed the tau draws
      self._jax_key, sample = jax_prng.iqn_update_keys(self._jax_key)
      self._jax_learn.set_keys(sample)
    self._stage_dev.copy_(slot, non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    self._ring_events[self._ring_pos] = ev
    self._ring_pos = (self._ring_pos + 1) % len(self._ring)
    self._launch()

  def learn(self) -> None:
    """Public alias of one learner step (`_learn`): host RNG draws -> H2D -> fused device step."""
    self._learn()

  def learn_from_device_draws(self, draws: torch.Tensor) -> None:
    """One learner step whose sampling draws are already in device memory (`draws` = float64
    [3B+4] in the staging layout).  Used by bench.py for the inputs-resident-in-HBM number."""
    self._stage_dev.copy_(draws, non_blocking=True)
    self._launch()

  def host_draws(self) -> np.ndarray:
    """The staging record for the next learner step (consumes the replay's RandomState)."""
    return self._draws().numpy().copy()

  def _launch(self) -> None:
    L = self._learner
    if self.PRIORITIZED:
      self._replay._distribution.flush()
    self._view = self._replay.device_view()
    key = bytes(self._view)
    if self._graph is not None and key != self._graph_key:
      self._graph = None                     # a device array moved (growth / set_state): recapture
    self._graph_key = key
    if self._io is None:
      alpha = self._replay._distribution._priority_exponent if self.PRIORITIZED else 1.0
      self._io = L.make_learn_io(self._stage_dev, self.PRIORITIZED, alpha)
    if self._use_graph:
      if self._graph is None:
        self._enqueue()                      # first step runs eagerly (also the warm-up for capture)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
          self._enqueue()
        self._graph = g                      # capture does not execute: nothing was applied twice
      else:
        self._graph.replay()
    else:
      self._enqueue()
    self._learn_steps += 1

  def _enqueue(self):
    L = self._learner
    if getattr(self, '_jax_key', None) is not None:
      self._jax_learn.launch(L.taus)            # jax.random.uniform draws from the keys staged by _learn()
    elif self.KIND in ('iqn', 'rainbow'):
      L.generate_randomness(self._seed, beside_sampler=True)
    L.learn(self._view, self.PRIORITIZED, self._io)

  def check_device_flags(self):
    """Raises if a kernel set a sticky error flag (bad priority, root == 0 in the fused path...)."""
    flags = self._replay._distribution._sum_tree._flags if self.PRIORITIZED else self._replay._store.flags
    f = int(flags.item())
    if f:
      flags.zero_()
      if f & _lib.DZ_FLAG_FRAME_POOL_FULL:
        raise RuntimeError('frame pool is full: frame_capacity is too small for the frames the live transitions '
                           'reference (device flags %d).' % f)
      if f & (_lib.DZ_FLAG_BAD_VALUE | _lib.DZ_FLAG_BAD_INDEX):
        raise ValueError('value must be finite and positive, index in range (device flags %d).' % f)
      if f & _lib.DZ_FLAG_NONFINITE_WEIGHT:
        raise ValueError('Weights are not finite (device flags %d).' % f)
      raise RuntimeError('device error flags: %d (bad sum-tree target / empty tree in the fused sampler)' % f)


class Dqn(_DeviceAgent):
  """dqn/agent.py:40-229."""
  KIND = 'dqn'

  def __init__(self, preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay,
               batch_size, exploration_epsilon, min_replay_capacity_fraction, learn_period,
               target_network_update_period, grad_error_bound, rng_key, use_cuda_graph=True):
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                exploration_epsilon, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                grad_error_bound=grad_error_bound, use_cuda_graph=use_cuda_graph)


class DoubleQ(Dqn):
  """double_q/agent.py:40-233."""
  KIND = 'double_q'


class PrioritizedDqn(_DeviceAgent):
  """prioritized/agent.py:40-258."""
  KIND = 'prioritized'
  PRIORITIZED = True

  def __init__(self, preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay,
               batch_size, exploration_epsilon, min_replay_capacity_fraction, learn_period,
               target_network_update_period, grad_error_bound, rng_key, use_cuda_graph=True):
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                exploration_epsilon, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                grad_error_bound=grad_error_bound, use_cuda_graph=use_cuda_graph)

  @property
  def importance_sampling_exponent(self) -> float:
    return self._replay.importance_sampling_exponent

  @property
  def max_seen_priority(self) -> float:
    return float(self._learner.max_seen_priority.item())


class C51(_DeviceAgent):
  """c51/agent.py:42-229.  `support` must be linspace(-vmax, vmax, atoms) (c51/run_atari.py:135)."""
  KIND = 'c51'

  def __init__(self, preprocessor, sample_network_input, network, support, optimizer, transition_accumulator,
               replay, batch_size, exploration_epsilon, min_replay_capacity_fraction, learn_period,
               target_network_update_period, rng_key, use_cuda_graph=True):
    _check_support(support, network)
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                exploration_epsilon, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                use_cuda_graph=use_cuda_graph)


class QrDqn(_DeviceAgent):
  """qrdqn/agent.py:42-232.  `quantiles` must be (arange(n)+0.5)/n (qrdqn/run_atari.py:137)."""
  KIND = 'qrdqn'

  def __init__(self, preprocessor, sample_network_input, network, quantiles, optimizer, transition_accumulator,
               replay, batch_size, exploration_epsilon, min_replay_capacity_fraction, learn_period,
               target_network_update_period, huber_param, rng_key, use_cuda_graph=True):
    q = np.asarray(quantiles, dtype=np.float64)
    n = network.num_quantiles
    if len(q) != n or not np.allclose(q, (np.arange(n) + 0.5) / n, rtol=0, atol=1e-6):
      raise ValueError('quantiles must be the %d midpoints (i + 0.5) / n' % n)
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                exploration_epsilon, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                huber_param=huber_param, use_cuda_graph=use_cuda_graph)


class Rainbow(_DeviceAgent):
  """rainbow/agent.py:41-245: greedy acting on the noisy network, PER, n-step, C51 double-Q."""
  KIND = 'rainbow'
  PRIORITIZED = True
  GREEDY = True

  def __init__(self, preprocessor, sample_network_input, network, support, optimizer, transition_accumulator,
               replay, batch_size, min_replay_capacity_fraction, learn_period, target_network_update_period,
               rng_key, use_cuda_graph=True):
    _check_support(support, network)
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                None, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                use_cuda_graph=use_cuda_graph)

  @property
  def importance_sampling_exponent(self) -> float:
    return self._replay.importance_sampling_exponent

  @property
  def max_seen_priority(self) -> float:
    return float(self._learner.max_seen_priority.item())


class Iqn(_DeviceAgent):
  """iqn/agent.py:133-340."""
  KIND = 'iqn'

  def __init__(self, preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay,
               batch_size, exploration_epsilon, min_replay_capacity_fraction, learn_period,
               target_network_update_period, huber_param, tau_samples_policy, tau_samples_s_tm1, tau_samples_s_t,
               rng_key, use_cuda_graph=True, jax_prng_taus=False):
    """`jax_prng_taus=True`: `rng_key` is treated as a jax PRNG key (`jax.random.PRNGKey(seed)` = [0, seed]) and the tau
    samples of every update and every action selection follow the reference's key chain bit for bit
    (iqn/agent.py:182-190, 207, 220-222; threefry2x32 + jax.random.split/uniform, csrc/dz_jaxprng.cu).  The default keeps
    the device Philox stream.  Epsilon-greedy exploration uses a host RandomState either way."""
    if (network.tau_samples_policy, network.tau_samples_s_tm1, network.tau_samples_s_t) != (
        tau_samples_policy, tau_samples_s_tm1, tau_samples_s_t):
      raise ValueError('tau sample counts must match the NetworkSpec')
    self._setup(preprocessor, sample_network_input, network, optimizer, transition_accumulator, replay, batch_size,
                exploration_epsilon, min_replay_capacity_fraction, learn_period, target_network_update_period, rng_key,
                huber_param=huber_param, use_cuda_graph=use_cuda_graph)
    if jax_prng_taus:
      key = np.asarray(rng_key, dtype=np.uint32).reshape(-1)
      if key.size != 2:
        raise ValueError('jax_prng_taus needs a jax-style rng_key of two uint32 words')
      self._jax_key = key.copy()
      dev = self._learner.device
      self._jax_learn = jax_prng.DeviceUniform([batch_size * tau_samples_s_tm1, batch_size * tau_samples_policy,
                                                batch_size * tau_samples_s_t], dev)
      self._jax_act = jax_prng.DeviceUniform([tau_samples_policy], dev)


def _check_support(support, network):
  s = np.asarray(support, dtype=np.float64)
  want = np.linspace(-network.vmax, network.vmax, network.num_atoms)
  if s.shape != want.shape or not np.allclose(s, want, rtol=0, atol=1e-5):
    raise ValueError('support must be linspace(-vmax, vmax, num_atoms) of the NetworkSpec')


class EpsilonGreedyActor(parts.Agent):
  """Acts epsilon-greedily with externally supplied network parameters (parts.py:336-411): the evaluation agent of
  the run drivers (`eval_agent.network_params = train_agent.online_params`, dqn/run_atari.py:260).

  `network_params` accepts what `agent.online_params` returns (haiku-shaped nested dict of host arrays), a flat
  `{canonical_name: array}` dict, or — the device-resident shortcut — the training learner itself
  (`eval_agent.network_params = train_agent.learner`: one D2D copy of the parameter blob).  The epsilon draw uses a
  host RandomState seeded from `rng_key` (the reference uses the JAX PRNG; action-sequence parity with it is SURVEY
  §8(f) #2)."""

  def __init__(self, preprocessor, network: NetworkSpec, exploration_epsilon: float, rng_key, device=None):
    self._preprocessor = preprocessor
    self._net = network
    self._epsilon = float(exploration_epsilon)
    self._learner = learner_lib.Learner(network, batch_size=1, device=device)
    self._rng = np.random.RandomState(int(np.asarray(rng_key).reshape(-1)[-1]) & 0x7FFFFFFF)
    self._seed = int(np.asarray(rng_key).reshape(-1)[-1]) & 0x7FFFFFFF
    self._obs_dev = torch.zeros(int(np.prod(network.obs_shape)), dtype=torch.uint8, device=self._learner.device)
    self._action = None
    self._has_params = False

  @property
  def network_params(self):
    return self._learner.haiku_params('online') if self._has_params else None

  @network_params.setter
  def network_params(self, params) -> None:
    if params is None:
      self._has_params = False
      return
    if isinstance(params, learner_lib.Learner):
      self._learner.online.copy_(params.online)
    else:
      flat = {}
      for key, value in params.items():
        if isinstance(value, Mapping):            # haiku-shaped {module: {leaf: array}}
          for leaf, arr in value.items():
            flat[self._canonical(key, leaf)] = arr
        else:
          flat[key] = value
      self._learner.set_params(flat)
    self._has_params = True

  def _canonical(self, module, leaf):
    for name in self._learner.tensors:
      if learner_lib.haiku_name(name, self._learner.kind) == (module, leaf):
        return name
    raise KeyError('unknown parameter %s/%s' % (module, leaf))

  def step(self, timestep) -> parts.Action:
    timestep = self._preprocessor(timestep)
    if timestep is None:
      if self._action is None:
        raise RuntimeError('Cannot repeat if action has never been selected.')
      return self._action
    if not self._has_params:
      raise RuntimeError('network_params have not been set.')
    obs = timestep.observation
    if isinstance(obs, torch.Tensor):
      self._obs_dev.copy_(obs.reshape(-1))
    else:
      self._obs_dev.copy_(torch.from_numpy(np.ascontiguousarray(obs).reshape(-1)))
    L = self._learner
    taus = noise = None
    if L.kind in ('iqn', 'rainbow'):
      self._seed += 1
      L.generate_randomness(self._seed)
      taus = L.taus if L.kind == 'iqn' else None
      noise = L.noise if L.kind == 'rainbow' else None
    q = L.q_values(self._obs_dev, taus=taus, noise=noise).cpu().numpy()
    if self._epsilon > 0.0 and self._rng.uniform() < self._epsilon:
      self._action = parts.Action(int(self._rng.randint(len(q))))
    else:
      self._action = parts.Action(int(np.argmax(q)))
    return self._action

  def reset(self) -> None:
    if hasattr(self._preprocessor, 'reset'):
      self._preprocessor.reset()
    self._action = None

  def get_state(self) -> Mapping[str, Any]:
    return {'rng_key': (self._rng.get_state(), self._seed),
            'network_params': self._learner.get_params('online') if self._has_params else None}

  def set_state(self, state: Mapping[str, Any]) -> None:
    rng_state, self._seed = state['rng_key']
    self._rng.set_state(rng_state)
    self.network_params = state['network_params']

  @property
  def statistics(self) -> Mapping[str, float]:
    return {}


AGENTS = {'dqn': Dqn, 'double_q': DoubleQ, 'prioritized': PrioritizedDqn, 'c51': C51, 'qrdqn': QrDqn,
          'rainbow': Rainbow, 'iqn': Iqn}


class BatchedEpsilonGreedyActor:
  """E independent actor streams served by ONE network evaluation per tick (the many-actors shape of
  parts.py:342-411 with dqn/agent.py:121-131 acting): observations of all streams -> `Learner.act_batch` (online forward,
  q-values and the epsilon-greedy choice on the device) -> one device-to-host copy of E actions.

  `learner` is the training agent's `Learner` (shared parameters, as the reference's actors read the learner's online
  params) or any `Learner` whose batch size is >= E.  Exploration uniforms come from a host RandomState seeded from
  `rng_key` (2E floats per tick; the reference draws with the JAX PRNG per actor).  Rainbow: one noise sample per tick is
  shared by the E streams; IQN: every stream gets its own tau samples."""

  def __init__(self, learner: learner_lib.Learner, num_streams: int, exploration_epsilon, rng_key):
    if num_streams < 1 or num_streams > learner.batch_size:
      raise ValueError('num_streams must be in [1, learner.batch_size]')
    self._learner = learner
    self._E = int(num_streams)
    self._epsilon = exploration_epsilon
    seed = int(np.asarray(rng_key).reshape(-1)[-1]) & 0x7FFFFFFF
    self._rng = np.random.RandomState(seed)
    self._seed = seed
    self._t = 0
    self._explore_host = torch.zeros((2, self._E), dtype=torch.float32).pin_memory()
    self._explore_dev = torch.zeros((2, self._E), dtype=torch.float32, device=learner.device)
    self._actions_host = torch.zeros(self._E, dtype=torch.int32).pin_memory()
    self.q_values = None

  def step(self, observations) -> np.ndarray:
    """observations: [E, H, W, C] uint8 (device tensor, e.g. the stacks of processors.BatchedAtariPreprocessor, or host
    array).  Returns the E actions as a host int32 array."""
    L = self._learner
    eps = self._epsilon(self._t) if callable(self._epsilon) else float(self._epsilon)
    explore = None
    if eps > 0.0:
      self._explore_host.copy_(torch.from_numpy(self._rng.uniform(size=(2, self._E)).astype(np.float32)))
      self._explore_dev.copy_(self._explore_host, non_blocking=True)
      explore = self._explore_dev
    taus = noise = None
    kind = L.net.kind
    if kind in ('iqn', 'rainbow'):
      L.generate_randomness(self._seed)
      if kind == 'iqn':
        taus = L.taus[:self._E * L.net.tau_samples_policy] if hasattr(L.net, 'tau_samples_policy') else L.taus
      else:
        noise = L.noise
    actions, self.q_values = L.act_batch(observations, epsilon=eps, explore=explore, taus=taus, noise=noise)
    self._actions_host.copy_(actions, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    self._t += 1
    return self._actions_host.numpy().copy()

