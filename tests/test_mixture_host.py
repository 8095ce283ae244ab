"""Host side of site-class mixtures: discrete-gamma rates (Yang 1994), the mixture reference
(mixture_oracle) against the single-class reference, and the argument checks of SiteMixtureMJP,
which run before anything touches a device."""
import numpy as np
import pytest
from scipy import integrate, stats

from oracle import np_oracle
import mixture_oracle
from raoteh_b200 import synth
from raoteh_b200.lowering import TreeSchedule
from raoteh_b200.mixture import SiteMixtureMJP, discrete_gamma_rates


@pytest.mark.parametrize('alpha', [0.05, 0.5, 1.0, 3.7, 50.0])
@pytest.mark.parametrize('K', [2, 4, 8])
def test_discrete_gamma_means(alpha, K):
    r = discrete_gamma_rates(alpha, K)
    assert r.shape == (K,) and (np.diff(r) > 0).all()
    assert abs(r.mean() - 1.0) < 1e-12
    g = stats.gamma(alpha, scale=1.0 / alpha)
    cuts = g.ppf(np.arange(K + 1) / K)
    for k in range(K):
        lo, hi = cuts[k], cuts[k + 1]
        if np.isinf(hi):
            # the upper tail: K * (mean - integral below the last cut)
            below, _ = integrate.quad(lambda x: x * g.pdf(x), 0, lo, epsabs=1e-14, epsrel=1e-13, limit=200)
            ref = K * (1.0 - below)
        else:
            ref, _ = integrate.quad(lambda x: x * g.pdf(x), lo, hi, epsabs=1e-14, epsrel=1e-13, limit=200)
            ref *= K
        assert abs(r[k] - ref) <= 1e-10 * max(1.0, abs(ref)), (k, r[k], ref)


@pytest.mark.parametrize('alpha', [0.3, 2.0])
def test_discrete_gamma_medians(alpha):
    r = discrete_gamma_rates(alpha, 4, median=True)
    assert abs(r.mean() - 1.0) < 1e-12 and (np.diff(r) > 0).all()
    med = stats.gamma(alpha, scale=1.0 / alpha).ppf((2 * np.arange(4) + 1) / 8.0)
    np.testing.assert_allclose(r, med * 4 / med.sum(), rtol=1e-12)


def test_discrete_gamma_one_category():
    assert discrete_gamma_rates(0.7, 1).tolist() == [1.0]
    assert discrete_gamma_rates(0.7, 1, median=True).tolist() == [1.0]
    for bad in (0.0, -1.0, np.inf, np.nan):
        with pytest.raises(ValueError):
            discrete_gamma_rates(bad, 4)
    with pytest.raises(ValueError):
        discrete_gamma_rates(1.0, 0)


def _case(seed=7, n_leaves=6, N=40):
    rng = np.random.default_rng(seed)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.2, rng)
    Q, pi = synth.hky85()
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, N, rng, 0.1)
    return parent, length, Q, pi, np_oracle.Obs('codes', 4, N, leaf_nodes=leaves, codes=codes)


def test_oracle_one_class_is_np_oracle():
    parent, length, Q, pi, obs = _case()
    got = mixture_oracle.mixture(parent, length, [Q], [1.0], [1.0], obs, pi)
    P = np_oracle.expm_edges(Q, length)
    ref = np_oracle.expected_history_statistics(parent, length, Q, P, obs, pi)
    np.testing.assert_allclose(got['loglik'], ref['loglik'], rtol=1e-12)
    np.testing.assert_allclose(got['class_post'], 1.0, rtol=0, atol=0)
    for k in ('dwell', 'trans'):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(got['root_post_sum'], ref['root_post'].sum(axis=0), rtol=1e-12)


def test_oracle_identical_classes():
    parent, length, Q, pi, obs = _case(seed=11)
    one = mixture_oracle.mixture(parent, length, [Q], [1.0], [1.0], obs, pi)
    w = np.array([0.3, 0.7])
    two = mixture_oracle.mixture(parent, length, [Q, Q], [1.0, 1.0], w, obs, pi)
    np.testing.assert_allclose(two['class_post'], np.repeat(w[:, None], obs.N, axis=1), rtol=1e-12)
    np.testing.assert_allclose(two['loglik'], one['loglik'], rtol=1e-12)
    for k in ('dwell', 'trans', 'root_post_sum'):
        np.testing.assert_allclose(two[k], one[k], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(two['class_post_sum'], w * obs.N, rtol=1e-12)


def test_mixture_rejects_bad_arguments():
    parent, length, _ = synth.random_binary_tree(4, 0.1, np.random.default_rng(0))
    sched = TreeSchedule(parent, length)
    Q, pi = synth.hky85()
    bad = [dict(Q=np.stack([Q, Q]), rates=[1.0, 1.0, 1.0]),             # K mismatch
           dict(Q=Q, rates=[1.0, -0.5]),                                 # negative rate
           dict(Q=Q, rates=[1.0, np.inf]),                               # non-finite rate
           dict(Q=Q, rates=[1.0, np.nan]),
           dict(Q=Q, rates=[1.0, 1.0], weights=[0.5, 0.6]),              # does not sum to 1
           dict(Q=Q, rates=[1.0, 1.0], weights=[1.0, 0.0]),              # zero weight
           dict(Q=Q, rates=[1.0, 1.0], weights=[0.5]),                   # weight count
           dict(Q=np.zeros((1, 1))),                                     # S < 2
           dict(Q=np.zeros((65, 65))),                                   # S > 64
           dict(Q=Q, q_index=np.zeros(sched.n, dtype=np.int32))]         # per-edge matrices
    for kw in bad:
        with pytest.raises(ValueError):
            SiteMixtureMJP(sched, root_distn=pi, **kw)
