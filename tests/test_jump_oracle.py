"""CPU checks of tests/jump_oracle.py, the exact per-branch jump-count law the posterior-draw tests
compare against: its marginal over k is expm(tQ), and its mean count given both end states is the
closed-form expected number of transitions of oracle/np_oracle.py."""
import numpy as np
import pytest
import scipy.linalg

from jump_oracle import jump_count_distribution
from oracle import np_oracle
from raoteh_b200 import synth


def _random_nonreversible(S, seed):
    rng = np.random.default_rng(seed)
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    return Q


@pytest.mark.parametrize('which,t', [('hky', 0.7), ('random3', 1.3), ('hky', 0.05)])
def test_summed_over_counts_is_the_transition_matrix(which, t):
    Q = synth.hky85()[0] if which == 'hky' else _random_nonreversible(3, 7)
    p = jump_count_distribution(Q, t, 60)
    assert np.all(p >= -1e-15)
    np.testing.assert_allclose(p.sum(axis=0), scipy.linalg.expm(t * Q), rtol=0, atol=1e-12)


@pytest.mark.parametrize('which,t', [('hky', 0.6), ('random3', 0.9)])
def test_mean_count_matches_closed_form_expectation(which, t):
    """Sum_k k p[k, a, b] / P[a, b] = E[number of transitions | X_0 = a, X_t = b]: the closed form of
    np_oracle.expected_history_statistics on a one-branch tree with both ends observed."""
    Q = synth.hky85()[0] if which == 'hky' else _random_nonreversible(3, 11)
    S = Q.shape[0]
    p = jump_count_distribution(Q, t, 80)
    P = scipy.linalg.expm(t * Q)
    parent, length = np.array([-1, 0]), np.array([0.0, t])
    Pe = np_oracle.expm_edges(Q, length)
    for a in range(S):
        for b in range(S):
            mask = np.array([[1 << a], [1 << b]], dtype=np.uint64)
            o = np_oracle.expected_history_statistics(parent, length, Q, Pe,
                                                      np_oracle.Obs('mask', S, 1, mask=mask), None)
            mean = (np.arange(81)[:, None, None] * p).sum(axis=0)[a, b] / P[a, b]
            np.testing.assert_allclose(mean, o['trans'].sum(), rtol=1e-10)
