"""CPU: the oracle restatement reproduces every golden vector generated from the
unmodified reference (tests/golden/*.npz, generator oracle/make_golden.py) bit-for-bit."""
import pytest

from oracle import cases
from helpers import KEYS, assert_equal_records, load_golden, oracle_case


@pytest.mark.parametrize('name', sorted(cases.CASES))
def test_oracle_matches_golden(name):
    kind = cases.CASES[name][0]
    want = load_golden(name)
    got = oracle_case(name, golden=want)
    keys = list(KEYS[kind])
    if kind == 'dynaq':
        keys += ['test_states', 'test_actions', 'test_trial_steps', 'test_trial_reward', 'draws_after_test']
    if 'modes' in want:          # SFMA dynamic mode: the per-trial replay modes and the TD accumulator
        keys += ['modes', 'td']
    # PMA's SR = inv(I - gamma T) comes from LAPACK on both sides, whose kernels (and last bits) depend on the host
    # CPU: SR within the norm-wise bound of tests/test_pma_gpu.py, everything else (trajectory, replay, Q, T) bit-equal
    assert_equal_records(got, want, keys, rtol={'SR': 1e-12}, what=name)
