"""Records every answer a replay library gives to a script, and plays the answers back later.

TEST INFRASTRUCTURE ONLY.  `oracle/gen_golden.py` runs each contract check of
`tests/replay_contract.py` against the REFERENCE's own `replay.py` through a
`Recorder` and stores the log under tests/golden/.  `Playback` then stands in
for the reference: it hands the script the reference's recorded answers (return
values, attribute values, raised exception types, yielded items) in order, so the
contract's assertions are checked against what the reference did without the
reference being present.  Every call is matched on its name and on a snapshot of
its arguments: a script that asks anything other than what the reference was
asked, or in another order, fails.
"""

import builtins
import collections
import inspect
import lzma
import pickle

import numpy as np

MISMATCH = 'script differs from the recording, regenerate with oracle.gen_golden'


def _encode(x):
  """A snapshot of `x` in builtins + numpy only (the reference hands out live views and namedtuples of its own).
  Functions are recorded by type only; other plain objects (a time step, say) by a snapshot of their attributes."""
  if isinstance(x, np.ndarray):
    return np.array(x, copy=True)
  if isinstance(x, tuple) and hasattr(x, '_fields'):
    return {'__namedtuple__': type(x).__name__, 'fields': list(x._fields), 'values': [_encode(v) for v in x]}
  if isinstance(x, (list, tuple)):
    return type(x)(_encode(v) for v in x)
  if isinstance(x, dict):
    return {k: _encode(v) for k, v in x.items()}
  if isinstance(x, (collections.abc.KeysView, collections.abc.ValuesView)):
    return [_encode(v) for v in x]
  if isinstance(x, np.random.RandomState):
    return {'__random_state__': _encode(list(x.get_state()))}
  if x is None or isinstance(x, (bool, int, float, str, np.generic, set, frozenset)):
    return x
  if callable(x):
    return {'__callable__': type(x).__name__}
  if hasattr(x, '__dict__') and not isinstance(x, (_RecordedObject, _PlaybackObject)):
    return {'__object__': type(x).__name__, 'attrs': _encode(vars(x))}
  raise TypeError('cannot record a %s' % type(x).__name__)


_NAMEDTUPLES = {}


def _decode(x):
  if isinstance(x, dict) and '__namedtuple__' in x:
    key = (x['__namedtuple__'], tuple(x['fields']))
    if key not in _NAMEDTUPLES:
      _NAMEDTUPLES[key] = collections.namedtuple(*key)
    return _NAMEDTUPLES[key](*[_decode(v) for v in x['values']])
  if isinstance(x, dict) and '__random_state__' in x:
    rs = np.random.RandomState()
    rs.set_state(tuple(x['__random_state__']))
    return rs
  if isinstance(x, dict):
    return {k: _decode(v) for k, v in x.items()}
  if isinstance(x, (list, tuple)):
    return type(x)(_decode(v) for v in x)
  return x


def _same(a, b):
  """Equality of two snapshots: same container types and keys, arrays and numpy scalars equal bit for bit."""
  if type(a) is not type(b):
    return False
  if isinstance(a, (np.ndarray, np.generic)):
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()
  if isinstance(a, dict):
    return a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
  if isinstance(a, (list, tuple)):
    return len(a) == len(b) and all(_same(u, v) for u, v in zip(a, b))
  if isinstance(a, float):
    return a == b or (a != a and b != b)
  return a == b


def _builtin_exception(e):
  """The first builtin class of `e` (messages are not recorded: they can hold object addresses)."""
  return next(c for c in type(e).__mro__ if getattr(builtins, c.__name__, None) is c).__name__


def _raise(exc_name):
  raise getattr(builtins, exc_name)('%s raised by the reference (recorded)' % exc_name)


def _replay_items(items, exc_name):
  for v in items:
    yield v
  if exc_name is not None:
    _raise(exc_name)


def save(path, logs):
  """`logs`: {script name: Recorder.log}."""
  with lzma.open(path, 'wb') as f:
    pickle.dump(logs, f, protocol=4)


def load(path):
  with lzma.open(path, 'rb') as f:
    return pickle.load(f)


class Recorder:
  """Wraps a replay module; `log` collects (op, name, snapshot of the arguments, outcome) for every constructor call,
  method call, attribute read and attribute write the script makes on it or on the objects it returns."""

  def __init__(self, lib):
    self._lib, self.log = lib, []

  def __getattr__(self, name):
    return self._callable(getattr(self._lib, name), 'new', name)

  def _is_object(self, v):
    return type(v).__module__ == self._lib.__name__ and not isinstance(v, tuple)

  def _outcome(self, v):
    if self._is_object(v):
      return ('obj',), _RecordedObject(self, v)
    if inspect.isgenerator(v):
      items, exc = [], None
      try:
        for item in v:
          items.append(item)
      except Exception as e:  # noqa: BLE001  (replayed at the same point of the iteration)
        exc = _builtin_exception(e)
      return ('gen', [_encode(i) for i in items], exc), _replay_items(items, exc)
    return ('val', _encode(v)), v

  def _callable(self, fn, op, name):
    def call(*args, **kwargs):
      snapshot = _encode((args, kwargs))      # before the call: the callee may change its arguments
      try:
        v = fn(*args, **kwargs)
      except Exception as e:
        self.log.append((op, name, snapshot, ('raise', _builtin_exception(e))))
        raise
      rec, v = self._outcome(v)
      self.log.append((op, name, snapshot, rec))
      return v
    return call


class _RecordedObject:

  def __init__(self, rec, obj):
    object.__setattr__(self, '_rec', rec)
    object.__setattr__(self, '_obj', obj)

  def __getattr__(self, name):
    rec = self._rec
    try:
      v = getattr(self._obj, name)
    except AttributeError as e:
      rec.log.append(('get', name, None, ('raise', _builtin_exception(e))))
      raise
    if callable(v) and not rec._is_object(v):
      # logged at lookup and at call: Python looks a method up before it evaluates the arguments
      rec.log.append(('get', name, None, ('method',)))
      return rec._callable(v, 'call', name)
    out, v = rec._outcome(v)
    rec.log.append(('get', name, None, out))
    return v

  def __setattr__(self, name, value):
    self._rec.log.append(('set', name, _encode(value), None))
    setattr(self._obj, name, value)


class Playback:
  """Stands in for the recorded module: answers from a `Recorder.log`, in order."""

  def __init__(self, log):
    self._log, self._pos = log, 0

  def _next(self, op, name, args=None):
    assert self._pos < len(self._log), '%s: the script goes on after the recorded run ended (%s %s)' % (MISMATCH, op,
                                                                                                         name)
    want_op, want_name, want_args, out = self._log[self._pos]
    assert (op, name) == (want_op, want_name), '%s: recorded %s %s here, the script does %s %s' % (
        MISMATCH, want_op, want_name, op, name)
    assert _same(_encode(args), want_args), '%s: %s %s with other arguments' % (MISMATCH, op, name)
    self._pos += 1
    return out

  def _answer(self, out, name=None):
    if out[0] == 'raise':
      _raise(out[1])
    if out[0] == 'obj':
      return _PlaybackObject(self)
    if out[0] == 'method':
      return lambda *args, **kwargs: self._answer(self._next('call', name, (args, kwargs)))
    if out[0] == 'gen':
      return _replay_items([_decode(v) for v in out[1]], out[2])
    return _decode(out[1])

  def finished(self):
    return self._pos == len(self._log)

  def __getattr__(self, name):
    return lambda *args, **kwargs: self._answer(self._next('new', name, (args, kwargs)))


class _PlaybackObject:

  def __init__(self, player):
    object.__setattr__(self, '_player', player)

  def __getattr__(self, name):
    return self._player._answer(self._player._next('get', name), name)

  def __setattr__(self, name, value):
    self._player._next('set', name, value)
