"""CPU: the oracle restatement vs (1) golden vectors made from the reference's replay.py,
(2) the reference's known-answer tables, (3) the reference's recorded answers to the contract."""

import os

import numpy as np
import pytest

from oracle import call_log, replay_oracle, scenarios
import replay_contract as rc


@pytest.mark.parametrize('name', list(scenarios.ALL))
def test_oracle_reproduces_reference_golden(name):
  rc.check_scenario(replay_oracle, name, 'oracle')


@pytest.mark.parametrize('fn', rc.CONTRACT, ids=lambda f: f.__name__)
def test_oracle_contract(fn):
  fn(replay_oracle)


@pytest.fixture(scope='module')
def reference_answers():
  return call_log.load(os.path.join(rc.GOLDEN, 'replay_contract_reference.xz'))


@pytest.mark.parametrize('fn', rc.CONTRACT, ids=lambda f: f.__name__)
def test_contract_holds_for_the_reference_itself(fn, reference_answers):
  """The contract file must describe the reference: run it on the answers the reference's own classes gave to the same
  calls (recorded by oracle/gen_golden.py)."""
  ref = call_log.Playback(reference_answers[fn.__name__])
  fn(ref)
  assert ref.finished(), 'the contract asks the reference fewer questions than were recorded'


def test_playback_rejects_calls_with_other_arguments(reference_answers):
  """A check whose inputs change while its asserted answers stay must fail on the recording: sumtree_get_set with
  set_all([1, 1, 1, 1]) in place of set_all([4, 5, 3, 9]) gets no answer."""
  ref = call_log.Playback(reference_answers['sumtree_get_set'])
  t = ref.SumTree()
  t.resize(3)
  for bad in (-1, 3):
    with pytest.raises(IndexError):
      t.get([bad])
  t = ref.SumTree()
  with pytest.raises(AssertionError, match='regenerate with oracle.gen_golden'):
    t.set_all([1.0, 1.0, 1.0, 1.0])
  ref = call_log.Playback(reference_answers['sumtree_get_set'])
  with pytest.raises(AssertionError, match='regenerate with oracle.gen_golden'):
    ref.SumTree().resize(4)


def test_oracle_matches_reference_on_long_random_per_run():
  want = np.load(os.path.join(rc.GOLDEN, 'replay_per_long_random.npz'))
  got = scenarios.prioritized_replay_script(replay_oracle, **scenarios.LONG_PER_RUN)
  assert set(got) == set(want.files)
  for k in want.files:
    np.testing.assert_array_equal(want[k], got[k], err_msg=k)


def test_synthetic_rows_are_deterministic_and_in_range():
  obs, a, r, d = replay_oracle.synthetic_rows(1, np.arange(100), 64, 6)
  obs2, a2, r2, d2 = replay_oracle.synthetic_rows(1, np.arange(100), 64, 6)
  np.testing.assert_array_equal(obs, obs2)
  assert obs.shape == (100, 2, 64) and obs.dtype == np.uint8
  assert a.min() >= 0 and a.max() < 6
  assert set(np.unique(r)).issubset({-1.0, 0.0, 1.0}) and set(np.unique(d)).issubset({0.0, 0.99})
  obs3, *_ = replay_oracle.synthetic_rows(2, np.arange(100), 64, 6)
  assert (obs3 != obs).mean() > 0.9
