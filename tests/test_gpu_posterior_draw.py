"""Exact posterior draws of whole histories (RaoTehChains.draw_posterior, rt_posterior_draw) on the
GPU: the invariants every sampled history must respect, the exact per-branch law of the number of
real jumps (tests/jump_oracle.py), agreement of iid draws with the closed-form posterior
expectations and node marginals, chains started from a draw with no burn-in, counter-based
reproducibility, and the failure paths.  z-score bounds are stated per test."""
import numpy as np
import pytest

from jump_oracle import jump_count_distribution
from oracle import np_oracle

pytestmark = pytest.mark.gpu


def _random_q(S, rng):
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    return Q / np.abs(np.diag(Q)).mean()


def _setup(S, n_leaves, n_sites, seed, missing=0.0, masks=False, scale=0.25):
    """Random binary tree and leaf data simulated from the model; masks=True: every node gets a
    random allowed-state mask that contains its simulated state (leaves) or all states."""
    from raoteh_b200 import synth, engine
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(seed)
    parent, length, leaves = synth.random_binary_tree(n_leaves, scale, rng)
    if S == 4:
        Q, pi = synth.hky85()
    else:
        Q = _random_q(S, rng)
        pi = rng.dirichlet(np.ones(S) * 3)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, missing)
    sched = TreeSchedule(parent, length)
    if masks:
        full = (1 << S) - 1
        mask = np.full((sched.n, n_sites), full, dtype=np.uint64)
        for i, leaf in enumerate(leaves):
            for s in range(n_sites):
                extra = int(rng.integers(0, full + 1)) & int(rng.integers(0, full + 1))
                code = int(codes[i, s])
                mask[leaf, s] = full if code == 255 else (1 << code) | extra     # 255: missing
        obs = engine.Observations.from_masks(sched, mask)
        data = np_oracle.Obs('mask', S, n_sites, mask=mask)
    else:
        mask = None
        obs = engine.Observations.from_leaf_codes(sched, codes, leaves)
        data = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    return dict(parent=parent, length=length, leaves=leaves, Q=Q, pi=pi, codes=codes, mask=mask,
                sched=sched, obs=obs, data=data)


def _check_history(ch, t, d, site):
    parent, length = d['parent'], d['length']
    ns, edges = ch.trajectory(t)
    assert len(edges) == d['sched'].n - 1
    for c, (times, states) in edges.items():
        assert states[0] == ns[parent[c]] and states[-1] == ns[c]     # consistent at the nodes
        assert len(states) == len(times) + 1
        assert len(times) < 2 or np.all(np.diff(times) > 0)          # strictly increasing
        assert np.all(times > 0) and np.all(times < length[c])        # inside the branch
        assert np.all(states[1:] != states[:-1])                      # no self-transitions
    if d['mask'] is None:
        for i, leaf in enumerate(d['leaves']):                        # observed leaves respected
            if d['codes'][i, site] != 255:
                assert ns[leaf] == d['codes'][i, site]
    else:
        for v in range(d['sched'].n):
            assert (int(d['mask'][v, site]) >> int(ns[v])) & 1


def _z_check(groups, want):
    """|mean - want| < 5 standard errors of the mean over the independent groups (rows)."""
    mean = groups.mean(axis=0)
    se = groups.std(axis=0, ddof=1) / np.sqrt(groups.shape[0])
    for m, s, w in zip(mean, se, want):
        if w == 0:
            assert m == 0
        else:
            assert abs(m - w) < 5 * s + 1e-9, (m, w, s)


@pytest.mark.parametrize('S,kind,time_dtype', [
    (4, 'codes', 'float32'), (4, 'codes', 'float64'), (3, 'masks', 'float32'), (3, 'masks', 'float64'),
    (7, 'codes', 'float32'), (8, 'codes', 'float32'), (8, 'masks', 'float64')])
def test_drawn_histories_respect_structure(S, kind, time_dtype):
    """Every drawn history: segment states consistent at the nodes, times strictly increasing and
    inside the branch, no self-transitions, observed leaves (codes with 10 % missing) or allowed
    states (masks) respected.  Two consecutive draws, each checked."""
    from raoteh_b200.raoteh import RaoTehChains
    n_sites = 5
    d = _setup(S, 12, n_sites, 40 + S, missing=0.1, masks=(kind == 'masks'))
    ch = RaoTehChains(d['sched'], d['Q'], d['obs'], n_chains=9, root_distn=d['pi'], seed=3,
                      time_dtype=time_dtype)
    for k in range(2):
        ch.draw_posterior()
        assert ch.sweeps_done == k + 1 and ch.initialized
        if ch.sweep_count is not None:
            assert bool((ch.sweep_count == k + 1).all())
        for t in range(ch.n_traj):
            _check_history(ch, t, d, t % n_sites)
    ch.sweep(3)                      # the sweeps continue from the draw
    for t in range(0, ch.n_traj, 4):
        _check_history(ch, t, d, t % n_sites)


@pytest.mark.parametrize('which', ['jc4', 'random3'])
def test_one_branch_jump_counts_and_dwell_match_exact_law(which):
    """Two-node tree, both ends fixed by masks, 16 draws x 8192 trajectories: the histogram of real
    jumps (k = 0..4 and the tail) against jump_count_distribution / P[a, b], per-bin binomial |z| < 5;
    the mean dwell per state against the closed form, |z| < 5 over the 16 draws."""
    import scipy.linalg
    from raoteh_b200 import engine
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    if which == 'jc4':
        S, t, a, b = 4, 0.5, 0, 2
        Q = (np.ones((S, S)) - np.eye(S)) / (S - 1)
        Q -= np.diag(Q.sum(axis=1))
    else:
        S, t, a, b = 3, 0.8, 0, 1
        Q = _random_q(3, np.random.default_rng(17))
    parent, length = np.array([-1, 0], dtype=np.int32), np.array([0.0, t])
    sched = TreeSchedule(parent, length)
    mask = np.array([[1 << a], [1 << b]], dtype=np.uint64)
    obs = engine.Observations.from_masks(sched, mask)
    n_chains, draws = 8192, 16
    ch = RaoTehChains(sched, Q, obs, n_chains=n_chains, seed=21, time_dtype='float64')
    hist = np.zeros(6)
    dwell = np.zeros((draws, S))
    for g in range(draws):
        ch.reset_statistics()
        ch.draw_posterior()
        k = ch.ev_total.cpu().numpy()
        assert bool((ch.node_state[0] == a).all()) and bool((ch.node_state[1] == b).all())
        hist += np.bincount(np.minimum(k, 5), minlength=6)
        dwell[g] = ch.dwell_sum.cpu().numpy() / n_chains
    n = n_chains * draws
    p = jump_count_distribution(Q, t, 60)[:, a, b] / scipy.linalg.expm(t * Q)[a, b]
    want = np.concatenate([p[:5], [1.0 - p[:5].sum()]])
    for got, w in zip(hist, want):
        if w < 1e-15:
            assert got == 0
        else:
            se = np.sqrt(n * w * (1 - w))
            assert abs(got - n * w) < 5 * se, (got, n * w, se)
    np.testing.assert_allclose(dwell.sum(axis=1), t, rtol=1e-12)
    o = np_oracle.expected_history_statistics(parent, length, Q, np_oracle.expm_edges(Q, length),
                                              np_oracle.Obs('mask', S, 1, mask=mask), None)
    _z_check(dwell, o['dwell'])


@pytest.mark.parametrize('S', [3, 4, 6, 8])
def test_iid_draws_match_closed_form(S):
    """Repeated draw_posterior() with no burn-in is an iid sampler: mean dwell times and transition
    counts over 32 groups (one draw of 262144 chains x 3 sites each) within |z| < 5 of the closed
    form; the total dwell of every draw is the tree length.  The draws are cheap, so every group is
    large: the rarest transition count (expected ~2e-5 per chain at S = 8) is then seen ~190 times
    in total, enough for the normal approximation of the z-score."""
    from raoteh_b200.raoteh import RaoTehChains
    n_sites, n_chains, groups = 3, 262144, 32
    d = _setup(S, 6, n_sites, 200 + S)
    o = np_oracle.expected_history_statistics(d['parent'], d['length'], d['Q'],
                                              np_oracle.expm_edges(d['Q'], d['length']), d['data'], d['pi'])
    ch = RaoTehChains(d['sched'], d['Q'], d['obs'], n_chains=n_chains, root_distn=d['pi'], seed=77)
    dwell = np.zeros((groups, S))
    trans = np.zeros((groups, S, S))
    for g in range(groups):
        ch.reset_statistics()
        ch.draw_posterior()
        dwell[g] = ch.dwell_sum.cpu().numpy() / n_chains
        trans[g] = ch.trans_sum.cpu().numpy() / n_chains
    np.testing.assert_allclose(dwell.sum(axis=1), d['length'].sum() * n_sites, rtol=1e-5)
    _z_check(dwell, o['dwell'])
    _z_check(trans.reshape(groups, -1), o['trans'].reshape(-1))


def test_node_state_frequencies_match_posterior_marginals():
    """Per-node state frequencies of 16384 draws per site, root and internal nodes, against the exact
    marginals of TreeMJP.posterior: binomial |z| < 5 (variance floored at 1/n for rare states)."""
    import torch
    from raoteh_b200 import engine
    from raoteh_b200.raoteh import RaoTehChains
    n_sites, n_chains = 3, 16384
    d = _setup(4, 10, n_sites, 31, missing=0.1)
    sched = d['sched']
    mjp = engine.TreeMJP(sched, d['Q'], root_distn=d['pi'])
    post = mjp.posterior(d['obs'], want_node_distn=True)
    marg = post['node_distn'][:, :, :n_sites].cpu().numpy()           # [n_store, S, n_sites]
    ch = RaoTehChains(sched, d['Q'], d['obs'], n_chains=n_chains, root_distn=d['pi'], seed=5)
    ch.draw_posterior(stats=False)
    ns = ch.node_state.long().view(sched.n, n_chains, n_sites)          # trajectory = chain * n_sites + site
    for v in sched.internal:
        freq = torch.nn.functional.one_hot(ns[v], 4).double().mean(dim=0).cpu().numpy()   # [n_sites, S]
        want = marg[sched.store_index[v]].T
        np.testing.assert_allclose(want.sum(axis=1), 1.0, rtol=1e-12)
        se = np.sqrt((want * (1 - want) + 1.0 / n_chains) / n_chains)
        assert np.all(np.abs(freq - want) < 5 * se), (v, freq, want)


@pytest.mark.parametrize('time_dtype', ['float32', 'float64'])
def test_c4_shape_draw_then_sweeps_need_no_burn_in(time_dtype):
    """BASELINE configs[3], the 127-node tree: chains started by draw_posterior() and swept 200 times
    with NO burn-in sweeps match the closed form, |z| < 5 over 16 groups of 512 chains (chains
    started by initialize() need 1000 burn-in sweeps here)."""
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    n_sites = 3
    cfg = synth.config_c4(n_sites=n_sites)
    assert len(cfg['parent']) == 127
    parent, length, leaves, Q, pi, codes = (cfg[k] for k in ('parent', 'length', 'leaves', 'Q', 'pi', 'codes'))
    sched = TreeSchedule(parent, length)
    obs = engine.Observations.from_leaf_codes(sched, codes, leaves)
    o = np_oracle.expected_history_statistics(
        parent, length, Q, np_oracle.expm_edges(Q, length),
        np_oracle.Obs('codes', 4, n_sites, leaf_nodes=leaves, codes=codes), pi)
    groups, n_chains, n_sweeps = 16, 512, 200
    dwell = np.zeros((groups, 4))
    trans = np.zeros((groups, 4, 4))
    d = dict(parent=parent, length=length, leaves=leaves, codes=codes, mask=None, sched=sched)
    for g in range(groups):
        ch = RaoTehChains(sched, Q, obs, n_chains=n_chains, root_distn=pi, seed=7000 + g, cap=112,
                          time_dtype=time_dtype)
        ch.draw_posterior(stats=False)
        ch.sweep(n_sweeps)
        assert bool((ch.sweep_count == 1 + n_sweeps).all())
        dwell[g] = ch.dwell_sum.cpu().numpy() / (n_chains * n_sweeps)
        trans[g] = ch.trans_sum.cpu().numpy() / (n_chains * n_sweeps)
        if g == 0:
            for t in range(0, ch.n_traj, 97):
                _check_history(ch, t, d, t % n_sites)
    np.testing.assert_allclose(dwell.sum(axis=1), length.sum() * n_sites,
                               rtol=1e-5 if time_dtype == 'float32' else 1e-12)
    _z_check(dwell, o['dwell'])
    _z_check(trans.reshape(groups, -1), o['trans'].reshape(-1))


def test_draws_are_counter_based():
    """Two shards (traj0 / n_traj) reproduce the unsharded draw bit for bit; the same seed and index
    give the same draw; consecutive draws differ; float32 and float64 times give the same discrete
    history for more than 99.9 % of trajectories."""
    import torch
    from raoteh_b200.raoteh import RaoTehChains
    d = _setup(4, 10, 6, 5, missing=0.1)
    args = (d['sched'], d['Q'], d['obs'])
    kw = dict(n_chains=400, root_distn=d['pi'], seed=9)
    full = RaoTehChains(*args, **kw)
    full.draw_posterior()
    lo = RaoTehChains(*args, traj0=0, n_traj=1001, **kw)
    hi = RaoTehChains(*args, traj0=1001, n_traj=2400 - 1001, **kw)
    for part in (lo, hi):
        part.draw_posterior()
    for name in ('node_state', 'ev_count'):
        assert torch.equal(torch.cat([getattr(lo, name), getattr(hi, name)], dim=1), getattr(full, name))
    for name in ('ev_total', 'ev_time', 'ev_sb', 'sweep_count'):
        assert torch.equal(torch.cat([getattr(lo, name), getattr(hi, name)]), getattr(full, name))
    np.testing.assert_allclose((lo.trans_sum + hi.trans_sum).cpu().numpy(), full.trans_sum.cpu().numpy())
    again = RaoTehChains(*args, **kw)
    again.draw_posterior()
    for name in RaoTehChains._STATE:
        assert torch.equal(getattr(again, name), getattr(full, name))
    first = full.node_state.clone(), full.ev_total.clone()
    full.draw_posterior()
    assert full.sweeps_done == 2
    assert not torch.equal(full.node_state, first[0]) and not torch.equal(full.ev_total, first[1])
    f64 = RaoTehChains(*args, time_dtype='float64', **kw)
    f64.draw_posterior()
    same = ((again.node_state == f64.node_state).all(dim=0) & (again.ev_count == f64.ev_count).all(dim=0) &
            (again.ev_sb == f64.ev_sb).all(dim=1) & (again.ev_total == f64.ev_total))
    assert float(same.double().mean()) > 0.999
    close = torch.isclose(again.ev_time.double(), f64.ev_time, rtol=1e-6, atol=0)
    assert float(close.double().mean()) > 0.999


def test_failure_paths():
    """Infeasible site -> status 1 and NativeError; a tiny cap -> status 4 and NativeError; a branch
    too long for the power table -> ValueError with the subdivision advice; chain_matrix chains and
    S = 9 -> ValueError."""
    from raoteh_b200 import engine, _native
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    sched = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, 1.0]))
    Q = np.array([[-1.0, 1.0, 0.0], [0.0, -1.0, 1.0], [0.0, 0.0, 0.0]])   # 0 -> 1 -> 2, absorbing
    obs = engine.Observations.from_masks(sched, np.array([[1 << 2], [1 << 0]], dtype=np.uint64))
    ch = RaoTehChains(sched, Q, obs, n_chains=3, seed=1)
    with pytest.raises(_native.NativeError, match='no feasible history'):
        ch.draw_posterior()
    assert bool((ch.status == 1).all())

    Qjc = np.array([[-3.0, 1.0, 1.0, 1.0], [1.0, -3.0, 1.0, 1.0], [1.0, 1.0, -3.0, 1.0], [1.0, 1.0, 1.0, -3.0]])
    sched2 = TreeSchedule(np.array([-1, 0, 0], dtype=np.int32), np.array([0.0, 2.0, 2.0]))
    full = np.array([[15], [15], [15]], dtype=np.uint64)
    obs2 = engine.Observations.from_masks(sched2, full)
    tiny = RaoTehChains(sched2, Qjc, obs2, n_chains=64, seed=2, cap=2)
    with pytest.raises(_native.NativeError, match='cap=2'):
        tiny.draw_posterior()
    assert bool((tiny.status == 4).any())

    long = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, 2.0]))
    obs3 = engine.Observations.from_masks(long, np.array([[3], [3]], dtype=np.uint64))
    ch3 = RaoTehChains(long, np.array([[-200.0, 200.0], [200.0, -200.0]]), obs3, n_chains=2, cap=4000)
    with pytest.raises(ValueError, match='subdivide_long_branches'):
        ch3.draw_posterior()

    obs4 = engine.Observations.from_masks(sched, np.array([[7], [7]], dtype=np.uint64))
    cm = RaoTehChains(sched, None, obs4, n_chains=1, chain_matrix=np.full((3, 3), 1 / 3.0))
    with pytest.raises(ValueError):
        cm.draw_posterior()
    Q9 = np.ones((9, 9)) - 9 * np.eye(9)
    obs9 = engine.Observations.from_masks(sched, np.array([[511], [511]], dtype=np.uint64))
    with pytest.raises(ValueError):
        RaoTehChains(sched, Q9, obs9, n_chains=1).draw_posterior()
