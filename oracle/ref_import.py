"""Import the REFERENCE's own `dqn_zoo/replay.py` from a checkout of the original dqn_zoo (DQN_ZOO_REFERENCE).

TEST INFRASTRUCTURE ONLY.  Used by `oracle/gen_golden.py` alone, to generate
the fixtures under tests/golden/; the tests, smoke() and bench.py read those
fixtures and never need the reference itself.

`replay.py` only needs numpy + stdlib for its arithmetic; its three imports
that are missing from this image are stubbed in `sys.modules`:
  dm_env          -> StepType / TimeStep stand-ins (only `.first()/.last()` used)
  snappy          -> empty module (compress_state is never enabled here)
  dqn_zoo.parts   -> `Action = int` (only used in annotations)
"""

import importlib.util
import os
import sys
import types

REFERENCE_ROOT = os.environ.get('DQN_ZOO_REFERENCE', '')


def available():
  return os.path.exists(os.path.join(REFERENCE_ROOT, 'dqn_zoo', 'replay.py'))


def load_reference_replay():
  """Returns the reference `dqn_zoo.replay` module object, unmodified."""
  if not available():
    raise RuntimeError('no dqn_zoo/replay.py under DQN_ZOO_REFERENCE=%r' % REFERENCE_ROOT)
  saved = {k: sys.modules.get(k) for k in ('dm_env', 'snappy', 'dqn_zoo', 'dqn_zoo.parts')}
  try:
    dm_env = types.ModuleType('dm_env')
    dm_env.TimeStep = object
    dm_env.StepType = object
    sys.modules['dm_env'] = dm_env
    sys.modules['snappy'] = types.ModuleType('snappy')
    pkg = types.ModuleType('dqn_zoo')
    pkg.__path__ = []
    parts = types.ModuleType('dqn_zoo.parts')
    parts.Action = int
    pkg.parts = parts
    sys.modules['dqn_zoo'] = pkg
    sys.modules['dqn_zoo.parts'] = parts
    spec = importlib.util.spec_from_file_location(
        '_reference_dqn_zoo_replay', os.path.join(REFERENCE_ROOT, 'dqn_zoo', 'replay.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
  finally:
    for k, v in saved.items():
      if v is None:
        sys.modules.pop(k, None)
      else:
        sys.modules[k] = v
