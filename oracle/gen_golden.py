"""Generates the replay fixtures under tests/golden/ by running the REFERENCE's own
replay.py (imported by oracle/ref_import.py from a checkout of the original dqn_zoo):

  replay_*.npz                    oracle/scenarios.py's scripts (ALL and LONG_PER_RUN)
  replay_contract_reference.xz    every answer the reference gave to the checks of
                                  tests/replay_contract.py (oracle/call_log.py)

  DQN_ZOO_REFERENCE=<checkout of dqn_zoo> python -m oracle.gen_golden

TEST INFRASTRUCTURE ONLY.  The fixtures are committed; this script is committed
so they can be regenerated and audited.

One documented deviation: for scenarios with priority_exponent != 0.5 the
reference's `_power` is evaluated through the canonical float32 definition
round_f32(pow_f64(x, (double)(float)alpha)) (SURVEY §8(a) R3) because numpy's
float32 SIMD `powf` is library/version dependent (differs by 1 ulp on ~20 % of
inputs between the pinned numpy 1.21.5 and this image's 2.3.5).  alpha = 0.5
(every BASELINE.json PER config) needs no such pin: `**0.5` is a correctly
rounded sqrt everywhere.
"""

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), 'tests'))

from oracle import call_log, ref_import, replay_oracle, scenarios  # noqa: E402
import replay_contract  # noqa: E402


def main():
  ref = ref_import.load_reference_replay()
  out_dir = os.path.join(os.path.dirname(HERE), 'tests', 'golden')
  os.makedirs(out_dir, exist_ok=True)
  stock_power = ref._power
  runs = dict(scenarios.ALL)
  runs['replay_per_long_random'] = lambda lib: scenarios.prioritized_replay_script(lib, **scenarios.LONG_PER_RUN)
  for name, fn in runs.items():
    ref._power = replay_oracle.power_keep_zero if 'pow06' in name else stock_power
    res = fn(ref)
    np.savez_compressed(os.path.join(out_dir, name + '.npz'), **res)
    print(name, {k: tuple(v.shape) for k, v in res.items()})
  ref._power = stock_power
  logs = {}
  for check in replay_contract.CONTRACT:
    rec = call_log.Recorder(ref)
    check(rec)
    logs[check.__name__] = rec.log
  path = os.path.join(out_dir, 'replay_contract_reference.xz')
  call_log.save(path, logs)
  print('replay_contract_reference', {k: len(v) for k, v in logs.items()}, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
  main()
