"""The log-space reference (range_oracle) against np_oracle on ordinary inputs and against 50-digit
mpmath arithmetic on inputs where a product of partials underflows in double precision."""
import mpmath
import numpy as np
import pytest

from oracle import np_oracle
import range_oracle
from raoteh_b200 import synth


def _star(n_leaves, t):
    parent = np.concatenate([[-1], np.zeros(n_leaves, dtype=np.int64)]).astype(np.int32)
    length = np.concatenate([[0.0], np.full(n_leaves, t)])
    return parent, length, np.arange(1, n_leaves + 1, dtype=np.int32)


def _random_Q(S, rng):
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    return Q, rng.dirichlet(np.ones(S))


def _mp_site(parent, P, rows, pi, prec=50):
    """(log-likelihood, root posterior) of one site in `prec`-digit arithmetic; rows[v] is the
    emission row of node v (None = unobserved)."""
    with mpmath.workdps(prec):
        n, S = len(parent), P.shape[-1]
        Pm = [None] + [[[mpmath.mpf(float(P[b, x, y])) for y in range(S)] for x in range(S)]
                       for b in range(1, n)]
        L = [[mpmath.mpf(1)] * S for _ in range(n)]
        for v in range(n - 1, -1, -1):
            if rows[v] is not None:
                L[v] = [L[v][a] * mpmath.mpf(float(rows[v][a])) for a in range(S)]
            if v > 0:
                p = parent[v]
                L[p] = [L[p][a] * mpmath.fsum(Pm[v][a][y] * L[v][y] for y in range(S)) for a in range(S)]
        w = [mpmath.mpf(float(pi[a])) * L[0][a] for a in range(S)]
        tot = mpmath.fsum(w)
        return float(mpmath.log(tot)), np.array([float(x / tot) for x in w])


def _site_rows(obs, n, i):
    rows = []
    for v in range(n):
        e = obs.emission(v, i, i + 1)
        rows.append(None if e is None else e[0])
    return rows


@pytest.mark.parametrize('kind', ['codes', 'mask', 'dense'])
def test_agrees_with_np_oracle_on_ordinary_inputs(kind):
    rng = np.random.default_rng(11)
    S, N = 4, 97
    parent, length, leaves = synth.random_binary_tree(12, 0.2, rng)
    n = len(parent)
    Q, pi = _random_Q(S, rng)
    P = np_oracle.expm_edges(Q, length)
    if kind == 'codes':
        codes = rng.integers(0, S, size=(len(leaves), N)).astype(np.uint8)
        codes[rng.random(codes.shape) < 0.1] = np_oracle.MISSING
        obs = np_oracle.Obs('codes', S, N, leaf_nodes=leaves, codes=codes)
    elif kind == 'mask':
        bits = rng.random((n, N, S)) < 0.6
        bits[..., 0] |= ~bits.any(axis=2)
        mask = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)).sum(axis=2).astype(np.uint64)
        obs = np_oracle.Obs('mask', S, N, mask=mask)
    else:
        has = np.zeros(n, dtype=bool)
        has[leaves] = True
        has[0] = True
        obs = np_oracle.Obs('dense', S, N, lik=rng.random((n, N, S)) ** 2, has=has)
    ref = np_oracle.expected_history_statistics(parent, length, Q, P, obs, pi)
    ll, st = np_oracle.log_likelihood(parent, P, obs, pi)
    got = range_oracle.posterior(parent, length, Q, P, obs, pi)
    assert (got['status'] == st).all()
    assert (st == 0).all()          # np_oracle's site sums are only defined on feasible sites
    np.testing.assert_allclose(got['loglik'], ll, rtol=1e-12)
    np.testing.assert_allclose(got['dwell'], ref['dwell'], rtol=1e-12)
    np.testing.assert_allclose(got['trans'], ref['trans'], rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(got['root_post'], ref['root_post'], rtol=1e-12, atol=1e-15)


def test_agrees_with_mpmath_on_a_wide_star():
    # a 300-leaf star: the product of 300 child messages underflows in double precision
    rng = np.random.default_rng(5)
    Q, pi = synth.hky85()
    parent, length, leaves = _star(300, 0.1)
    P = np_oracle.expm_edges(Q, length)
    N = 4
    codes = rng.integers(0, 4, size=(300, N)).astype(np.uint8)
    obs = np_oracle.Obs('codes', 4, N, leaf_nodes=leaves, codes=codes)
    got = range_oracle.posterior(parent, length, Q, P, obs, pi)
    assert (got['status'] == 0).all()
    for i in range(N):
        ll, rp = _mp_site(parent, P, _site_rows(obs, len(parent), i), pi)
        assert ll < -708.4          # exp(ll) is below the smallest normal double
        np.testing.assert_allclose(got['loglik'][i], ll, rtol=1e-12)
        np.testing.assert_allclose(got['root_post'][i], rp, rtol=1e-12, atol=1e-15)


def test_agrees_with_mpmath_on_tiny_emissions():
    # cherries of leaves whose emission rows are of order 1e-200: the pair product is 1e-400
    rng = np.random.default_rng(6)
    S, N = 4, 5
    parent, length, leaves, _ = synth.tree_from_nested(((0, 1), ((2, 3), (4, 5))), 0.3)
    parent = np.asarray(parent, dtype=np.int32)
    length = np.asarray(length, dtype=float)
    n = len(parent)
    Q, pi = _random_Q(S, rng)
    P = np_oracle.expm_edges(Q, length)
    lik = rng.random((n, N, S)) * 10.0 ** rng.uniform(-210, -190, size=(n, N, 1))
    has = np.zeros(n, dtype=bool)
    has[np.asarray(leaves)] = True
    obs = np_oracle.Obs('dense', S, N, lik=lik, has=has)
    got = range_oracle.posterior(parent, length, Q, P, obs, pi)
    assert (got['status'] == 0).all()
    for i in range(N):
        ll, rp = _mp_site(parent, P, _site_rows(obs, n, i), pi)
        np.testing.assert_allclose(got['loglik'][i], ll, rtol=1e-12)
        np.testing.assert_allclose(got['root_post'][i], rp, rtol=1e-12, atol=1e-15)
