"""Exact posterior draws of (class, history) under site-class mixtures (SiteMixtureMJP.history_draws,
rt_posterior_draw_mixture) on the GPU: a one-class mixture is the single-class draw bit for bit,
every history respects the tree and the data, class frequencies, per-class statistics and node
states match the mixture's closed forms (tests/mixture_oracle.py, SiteMixtureMJP), draws are
counter-based, and the failure paths.  z-score bounds are stated per test."""
import ctypes

import numpy as np
import pytest

from oracle import np_oracle
import mixture_oracle

pytestmark = pytest.mark.gpu


def _random_q(S, rng):
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    return Q / np.abs(np.diag(Q)).mean()


def _setup(S, n_leaves, n_sites, seed, missing=0.0, masks=False, scale=0.25, Q=None):
    """Random binary tree and leaf data simulated from Q (HKY85 at S = 4 unless given); masks=True:
    every leaf gets a random allowed-state mask containing its simulated state (as in
    test_gpu_posterior_draw)."""
    from raoteh_b200 import synth, engine
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(seed)
    parent, length, leaves = synth.random_binary_tree(n_leaves, scale, rng)
    if Q is None:
        Q = synth.hky85()[0] if S == 4 else _random_q(S, rng)
    pi = synth.hky85()[1] if S == 4 else rng.dirichlet(np.ones(S) * 3)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, missing)
    sched = TreeSchedule(parent, length)
    if masks:
        full = (1 << S) - 1
        mask = np.full((sched.n, n_sites), full, dtype=np.uint64)
        for i, leaf in enumerate(leaves):
            for s in range(n_sites):
                extra = int(rng.integers(0, full + 1)) & int(rng.integers(0, full + 1))
                code = int(codes[i, s])
                mask[leaf, s] = full if code == 255 else (1 << code) | extra
        obs = engine.Observations.from_masks(sched, mask)
        data = np_oracle.Obs('mask', S, n_sites, mask=mask)
    else:
        mask = None
        obs = engine.Observations.from_leaf_codes(sched, codes, leaves)
        data = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    return dict(parent=parent, length=length, leaves=leaves, Q=Q, pi=pi, codes=codes, mask=mask,
                sched=sched, obs=obs, data=data, rng=rng)


def _check_history(dr, t, d, site):
    """The invariants of test_gpu_posterior_draw._check_history."""
    parent, length = d['parent'], d['length']
    ns, edges = dr.trajectory(t)
    assert len(edges) == d['sched'].n - 1
    for c, (times, states) in edges.items():
        assert states[0] == ns[parent[c]] and states[-1] == ns[c]
        assert len(states) == len(times) + 1
        assert len(times) < 2 or np.all(np.diff(times) > 0)
        assert np.all(times > 0) and np.all(times < length[c])
        assert np.all(states[1:] != states[:-1])
    if d['mask'] is None:
        for i, leaf in enumerate(d['leaves']):
            if d['codes'][i, site] != 255:
                assert ns[leaf] == d['codes'][i, site]
    else:
        for v in range(d['sched'].n):
            assert (int(d['mask'][v, site]) >> int(ns[v])) & 1


def _z_check(groups, want):
    """|mean - want| < 5 standard errors of the mean over the independent groups (rows); a zero
    expectation must come out exactly zero."""
    mean = groups.mean(axis=0)
    se = groups.std(axis=0, ddof=1) / np.sqrt(groups.shape[0])
    for m, s, w in zip(mean, se, want):
        if w == 0:
            assert m == 0
        else:
            assert abs(m - w) < 5 * s + 1e-9, (m, w, s)


def _gamma_i(n_gamma=4, alpha=0.5, p_inv=0.2):
    from raoteh_b200.mixture import discrete_gamma_rates
    rates = np.concatenate([[0.0], discrete_gamma_rates(alpha, n_gamma)])
    weights = np.concatenate([[p_inv], np.full(n_gamma, (1 - p_inv) / n_gamma)])
    return rates, weights


@pytest.mark.parametrize('S,kind,time_dtype', [(4, 'codes', 'float32'), (8, 'masks', 'float64'),
                                               (7, 'codes', 'float32')])
def test_one_class_equals_single_class_draw(S, kind, time_dtype):
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP
    from raoteh_b200.raoteh import RaoTehChains
    d = _setup(S, 12, 7, 60 + S, missing=0.1, masks=(kind == 'masks'))
    ch = RaoTehChains(d['sched'], d['Q'], d['obs'], n_chains=33, root_distn=d['pi'], seed=11,
                      time_dtype=time_dtype)
    mix = SiteMixtureMJP(d['sched'], d['Q'], root_distn=d['pi'])
    dr = mix.history_draws(d['obs'], n_chains=33, seed=11, time_dtype=time_dtype)
    for k in range(2):
        ch.reset_statistics()
        dr.reset_statistics()
        ch.draw_posterior()
        dr.draw()
        assert dr.draws_done == k + 1
        for name in ('node_state', 'ev_count', 'ev_total', 'ev_time', 'ev_sb', 'status'):
            assert torch.equal(getattr(dr, name), getattr(ch, name)), name
        assert int(dr.site_class.max()) == 0
        assert torch.equal(dr.trans_class[0], ch.trans_sum)
        np.testing.assert_allclose(dr.dwell_class[0].cpu().numpy(), ch.dwell_sum.cpu().numpy(),
                                   rtol=1e-12)


STRUCTURE_CASES = [('hky_g4_i', 'float32'), ('hky_g4_i', 'float64'), ('s3_masks_two_q', 'float32'),
                   ('s7_codes', 'float32'), ('s8_two', 'float64')]


def _structure_case(name):
    if name == 'hky_g4_i':
        d = _setup(4, 12, 9, 71, missing=0.1)
        rates, weights = _gamma_i()
        return d, d['Q'], rates, weights
    if name == 's3_masks_two_q':
        d = _setup(3, 10, 9, 72, masks=True)
        Qs = np.stack([d['Q'], _random_q(3, d['rng'])])
        return d, Qs, np.array([0.5, 2.0]), np.array([0.4, 0.6])
    if name == 's7_codes':
        d = _setup(7, 10, 9, 73, missing=0.1)
        return d, d['Q'], np.array([0.0, 0.6, 1.4]), np.array([0.2, 0.4, 0.4])
    assert name == 's8_two'
    d = _setup(8, 10, 9, 74, missing=0.1)
    Qs = np.stack([d['Q'], _random_q(8, d['rng'])])
    return d, Qs, np.array([0.5, 1.5]), np.array([0.5, 0.5])


@pytest.mark.parametrize('name,time_dtype', STRUCTURE_CASES)
def test_drawn_histories_respect_structure(name, time_dtype):
    from raoteh_b200.mixture import SiteMixtureMJP
    d, Q, rates, weights = _structure_case(name)
    n_sites = d['obs'].n_sites
    mix = SiteMixtureMJP(d['sched'], Q, root_distn=d['pi'], rates=rates, weights=weights)
    dr = mix.history_draws(d['obs'], n_chains=40, seed=5, time_dtype=time_dtype)
    cp = dr.class_post.cpu().numpy()
    for _ in range(2):
        dr.draw()
        cls = dr.site_class.cpu().numpy().astype(int)
        total = dr.ev_total.cpu().numpy()
        ns = dr.node_state.cpu().numpy()
        assert len(set(cls.tolist())) > 1
        for t in range(dr.n_traj):
            site = t % n_sites
            _check_history(dr, t, d, site)
            assert cp[cls[t], site] > 0
            if rates[cls[t]] == 0:                       # +I: no jumps, one state everywhere
                assert total[t] == 0 and np.all(ns[:, t] == ns[0, t])


def test_class_frequencies_match_class_posterior():
    """Per site and class, the frequency of the drawn class over 32768 chains against class_post:
    binomial |z| < 5 (variance floored at 1/n)."""
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP
    d = _setup(4, 10, 12, 81, missing=0.1)
    rates, weights = _gamma_i()
    mix = SiteMixtureMJP(d['sched'], d['Q'], root_distn=d['pi'], rates=rates, weights=weights)
    n_chains = 32768
    dr = mix.history_draws(d['obs'], n_chains=n_chains, seed=17)
    dr.draw(stats=False)
    cls = dr.site_class.long().view(n_chains, -1)
    freq = torch.nn.functional.one_hot(cls, mix.K).double().mean(dim=0).T.cpu().numpy()   # [K, N]
    want = dr.class_post.cpu().numpy()
    se = np.sqrt((want * (1 - want) + 1.0 / n_chains) / n_chains)
    assert np.all(np.abs(freq - want) < 5 * se), (freq, want)
    assert np.all(freq[want == 0] == 0)


def test_per_class_statistics_match_closed_form():
    """HKY+G4+I (alpha = 1) on a 6-leaf tree, 3 sites: means of dwell_class and trans_class over 32
    groups (one draw of 262144 chains each) within |z| < 5 of mixture_oracle; +I transitions exactly
    zero; the dwell of every draw summed over classes is tree length x sites.  The slowest gamma
    class makes the rarest transitions: its rarest nonzero count is expected ~3e-4 per chain, so
    it is seen ~2600 times in all (asserted below from the oracle), enough for the normal
    approximation.  With alpha = 0.5 and shorter branches it would be seen about once."""
    from raoteh_b200.mixture import SiteMixtureMJP
    d = _setup(4, 6, 3, 92, scale=0.5)
    rates, weights = _gamma_i(alpha=1.0)
    Qs = [d['Q']] * len(rates)
    ref = mixture_oracle.mixture(d['parent'], d['length'], Qs, rates, weights, d['data'], d['pi'])
    mix = SiteMixtureMJP(d['sched'], d['Q'], root_distn=d['pi'], rates=rates, weights=weights)
    n_chains, groups, n_sites = 262144, 32, 3
    rare = ref['trans_class'][ref['trans_class'] > 0].min()
    assert rare * n_chains * groups > 100
    dr = mix.history_draws(d['obs'], n_chains=n_chains, seed=23)
    K, S = mix.K, mix.S
    dwell = np.zeros((groups, K, S))
    trans = np.zeros((groups, K, S, S))
    for g in range(groups):
        dr.reset_statistics()
        dr.draw()
        dwell[g] = dr.dwell_class.cpu().numpy() / n_chains
        trans[g] = dr.trans_class.cpu().numpy() / n_chains
    np.testing.assert_allclose(dwell.sum(axis=(1, 2)), d['length'].sum() * n_sites, rtol=1e-5)
    assert np.all(trans[:, 0] == 0)
    _z_check(dwell.reshape(groups, -1), ref['dwell_class'].reshape(-1))
    _z_check(trans.reshape(groups, -1), ref['trans_class'].reshape(-1))


def test_node_state_frequencies_match_mixture_marginals():
    """Per-node state frequencies of 16384 draws per site against the mixture node marginals of
    expected_history_statistics(want_node_distn=True): binomial |z| < 5 (variance floored at 1/n)."""
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP
    n_sites, n_chains = 4, 16384
    d = _setup(4, 10, n_sites, 31, missing=0.1)
    rates, weights = _gamma_i()
    mix = SiteMixtureMJP(d['sched'], d['Q'], root_distn=d['pi'], rates=rates, weights=weights)
    marg = mix.expected_history_statistics(d['obs'], want_node_distn=True)['node_distn']
    marg = marg[:, :, :n_sites].cpu().numpy()
    dr = mix.history_draws(d['obs'], n_chains=n_chains, seed=5)
    dr.draw(stats=False)
    sched = d['sched']
    ns = dr.node_state.long().view(sched.n, n_chains, n_sites)
    for v in sched.internal:
        freq = torch.nn.functional.one_hot(ns[v], 4).double().mean(dim=0).cpu().numpy()
        want = marg[sched.store_index[v]].T
        np.testing.assert_allclose(want.sum(axis=1), 1.0, rtol=1e-10)
        se = np.sqrt((want * (1 - want) + 1.0 / n_chains) / n_chains)
        assert np.all(np.abs(freq - want) < 5 * se), (v, freq, want)


def test_draws_are_counter_based():
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP
    d = _setup(4, 10, 6, 5, missing=0.1)
    rates, weights = _gamma_i()
    mix = SiteMixtureMJP(d['sched'], d['Q'], root_distn=d['pi'], rates=rates, weights=weights)
    names = ('node_state', 'ev_count', 'ev_total', 'ev_time', 'ev_sb', 'site_class')
    full = mix.history_draws(d['obs'], n_chains=400, seed=9)
    full.draw()
    lo = mix.history_draws(d['obs'], n_chains=400, seed=9, traj0=0, n_traj=1001)
    hi = mix.history_draws(d['obs'], n_chains=400, seed=9, traj0=1001, n_traj=2400 - 1001)
    for part in (lo, hi):
        part.draw()
    for name in names:
        dim = 1 if name in ('node_state', 'ev_count') else 0
        assert torch.equal(torch.cat([getattr(lo, name), getattr(hi, name)], dim=dim), getattr(full, name))
    np.testing.assert_allclose((lo.trans_class + hi.trans_class).cpu().numpy(), full.trans_class.cpu().numpy())
    again = mix.history_draws(d['obs'], n_chains=400, seed=9)
    again.draw()
    for name in names:
        assert torch.equal(getattr(again, name), getattr(full, name))
    first = full.node_state.clone(), full.site_class.clone()
    full.draw()
    assert full.draws_done == 2
    assert not torch.equal(full.node_state, first[0]) and not torch.equal(full.site_class, first[1])


def test_failure_paths():
    from raoteh_b200 import engine, _native
    from raoteh_b200.engine import _stream
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.mixture import SiteMixtureMJP
    sched = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, 1.0]))
    # S = 9, dense observations
    Q9 = np.ones((9, 9)) - 9 * np.eye(9)
    obs9 = engine.Observations.from_masks(sched, np.array([[511], [511]], dtype=np.uint64))
    with pytest.raises(ValueError):
        SiteMixtureMJP(sched, Q9, rates=[0.5, 1.5]).history_draws(obs9)
    Q4 = np.ones((4, 4)) - 4 * np.eye(4)
    dense = engine.Observations.from_dense(sched, np.ones((1, 4, 3)), np.array([1]))
    with pytest.raises(ValueError):
        SiteMixtureMJP(sched, Q4, rates=[0.5, 1.5]).history_draws(dense)
    # a class whose branch is too long; the same tree without that class draws fine
    long = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, 2.0]))
    Q2 = np.array([[-1.0, 1.0], [1.0, -1.0]])
    obs2 = engine.Observations.from_masks(long, np.array([[3], [3]], dtype=np.uint64))
    with pytest.raises(ValueError, match='class 1 .rate 200.*subdivide_long_branches'):
        SiteMixtureMJP(long, Q2, rates=[1.0, 200.0], weights=[0.5, 0.5]).history_draws(obs2)
    SiteMixtureMJP(long, Q2, rates=[1.0]).history_draws(obs2, n_chains=4, cap=64).draw()
    # a site infeasible in every class: 0 -> 1 -> 2 absorbing, observed 2 at the root and 0 below
    Qa = np.array([[-1.0, 1.0, 0.0], [0.0, -1.0, 1.0], [0.0, 0.0, 0.0]])
    obs3 = engine.Observations.from_masks(sched, np.array([[1 << 2], [1 << 0]], dtype=np.uint64))
    dr = SiteMixtureMJP(sched, Qa, rates=[0.5, 2.0]).history_draws(obs3, n_chains=3)
    with pytest.raises(_native.NativeError, match='no feasible history'):
        dr.draw()
    assert bool((dr.status == 1).all())
    # a tiny cap
    Qjc = np.array([[-3.0, 1.0, 1.0, 1.0], [1.0, -3.0, 1.0, 1.0], [1.0, 1.0, -3.0, 1.0], [1.0, 1.0, 1.0, -3.0]])
    sched2 = TreeSchedule(np.array([-1, 0, 0], dtype=np.int32), np.array([0.0, 2.0, 2.0]))
    obs4 = engine.Observations.from_masks(sched2, np.array([[15], [15], [15]], dtype=np.uint64))
    tiny = SiteMixtureMJP(sched2, Qjc, rates=[0.5, 1.5]).history_draws(obs4, n_chains=64, seed=2, cap=2)
    with pytest.raises(_native.NativeError, match='cap=2'):
        tiny.draw()
    assert bool((tiny.status == 4).any())
    # the C ABI: K = 0 and a null class_post are argument errors
    ok = SiteMixtureMJP(sched2, Qjc, rates=[0.5, 1.5]).history_draws(obs4, n_chains=2)
    lib = _native.lib()
    A = ok._args(True)
    A.K = 0
    assert lib.rt_posterior_draw_mixture(ctypes.byref(A), _stream()) == 1
    A = ok._args(True)
    A.class_post = None
    assert lib.rt_posterior_draw_mixture(ctypes.byref(A), _stream()) == 1
    A = ok._args(True)
    assert lib.rt_posterior_draw_mixture(ctypes.byref(A), _stream()) == 0
