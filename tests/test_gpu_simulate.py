"""Forward (prior) simulation on the GPU (rt_forward_simulate: simulate.simulate_sites,
simulate.ForwardHistories, SiteMixtureMJP.simulate): the exact law of the leaf patterns and node
states, the structure and law of simulated histories, their layout as read by the Rao-Teh kernels,
the joint-distribution test of the sweeps (Geweke 2004), mixtures, and counter-based
reproducibility.  z-score bounds are stated per test."""
import ctypes

import numpy as np
import pytest
import scipy.linalg

from jump_oracle import jump_count_distribution
from oracle import np_oracle

pytestmark = pytest.mark.gpu


def _random_q(S, rng):
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    return Q / np.abs(np.diag(Q)).mean()


def _model(S, rng):
    from raoteh_b200 import synth
    if S == 4:
        return synth.hky85()
    if S == 61:
        Q, pi, _ = synth.mg94()
        return Q, pi
    return _random_q(S, rng), rng.dirichlet(np.ones(S) * 3)


def _tree(n_leaves, seed, scale=0.25):
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    parent, length, leaves = synth.random_binary_tree(n_leaves, scale, np.random.default_rng(seed))
    return parent, length, leaves, TreeSchedule(parent, length)


def _path_matrices(parent, length, Q, nodes):
    """P_path[v] = product of expm(t_b Q) along the path root -> v."""
    S = Q.shape[0]
    out = {}
    for v in nodes:
        M, u = np.eye(S), int(v)
        while u > 0:
            M = scipy.linalg.expm(length[u] * Q) @ M
            u = int(parent[u])
        out[int(v)] = M
    return out


def _pair_joint(parent, length, Q, p0, i, j):
    """Joint law of the states of nodes i and j: sum_m d_m P_{m->i}[m, x] P_{m->j}[m, y], with m their
    most recent common ancestor and d = p0 P_path(m) its marginal (m = the root: the textbook
    sum_a pi_a P_i[a, x] P_j[a, y])."""
    def up(v):
        out = [int(v)]
        while out[-1] > 0:
            out.append(int(parent[out[-1]]))
        return out
    ai = up(i)
    m = next(u for u in up(j) if u in ai)

    def down(v):
        M = np.eye(Q.shape[0])
        while v != m:
            M = scipy.linalg.expm(length[v] * Q) @ M
            v = int(parent[v])
        return M
    d = p0 @ _path_matrices(parent, length, Q, [m])[m]
    return (d[:, None, None] * down(int(i))[:, :, None] * down(int(j))[:, None, :]).sum(0)


def _counts_match(got, want, n, floor=20):
    """Binomial |z| < 5 for every cell with expectation >= floor; the cells below it pooled into one
    (a one-degree-of-freedom chi-square, as a z-score)."""
    got = np.asarray(got, dtype=float)
    e = n * np.asarray(want, dtype=float)
    big = e >= floor
    z = (got[big] - e[big]) / np.sqrt(e[big] * (1 - want[big]))
    assert np.all(np.abs(z) < 5), (np.abs(z).max(), np.nonzero(big)[0][np.argmax(np.abs(z))])
    rest_o, rest_e = got[~big].sum(), e[~big].sum()
    assert abs(rest_o - rest_e) < 5 * np.sqrt(rest_e + 1), (rest_o, rest_e)


def _z_check(groups, want, n_indep=None):
    """|mean - want| < 5 standard errors of the mean over the independent groups (rows).  n_indep:
    the number of independent sites behind all groups; the standard error is then floored at the
    Poisson one, sqrt(want / n_indep), so that a rare count seen in no group is not a failure."""
    mean = groups.mean(axis=0)
    se = groups.std(axis=0, ddof=1) / np.sqrt(groups.shape[0])
    if n_indep is not None:
        se = np.maximum(se, np.sqrt(np.abs(np.asarray(want)) / n_indep))
    for m, s, w in zip(mean, se, want):
        if w == 0:
            assert m == 0
        else:
            assert abs(m - w) < 5 * s + 1e-12, (m, w, s)


def _prior_stats(parent, length, Q, pi, leaves):
    """Prior expectations of dwell / trans per site: the closed form with every leaf missing."""
    S = Q.shape[0]
    obs = np_oracle.Obs('codes', S, 1, leaf_nodes=leaves, codes=np.full((len(leaves), 1), 255, np.uint8))
    pi = np.full(S, 1.0 / S) if pi is None else pi
    o = np_oracle.expected_history_statistics(parent, length, Q, np_oracle.expm_edges(Q, length), obs, pi)
    return o['dwell'], o['trans']


def _patterns(codes, S):
    idx = np.zeros(codes.shape[1], dtype=np.int64)
    for i in range(codes.shape[0]):
        idx = idx * S + codes[i].astype(np.int64)
    return np.bincount(idx, minlength=S ** codes.shape[0])


def _all_patterns(n_leaves, S):
    grid = np.stack(np.meshgrid(*[np.arange(S)] * n_leaves, indexing='ij'), 0).reshape(n_leaves, -1)
    return np.ascontiguousarray(grid.astype(np.uint8))


@pytest.mark.parametrize('with_root', [True, False])
def test_leaf_pattern_law_four_leaves(with_root):
    """S = 4, 4 leaves, 2^20 sites: every one of the 256 leaf patterns against
    n exp(TreeMJP.log_likelihood(pattern)); None root = uniform."""
    from raoteh_b200 import engine, simulate
    parent, length, leaves, sched = _tree(4, 3, 0.4)
    Q, pi = _model(4, None)
    n = 1 << 20
    obs = simulate.simulate_sites(sched, Q, n, root_distn=pi if with_root else None, seed=11)
    assert obs.kind == engine.OBS_CODES and obs.n_sites == n and tuple(obs.data.shape) == (4, n)
    got = _patterns(obs.data.cpu().numpy(), 4)
    pats = _all_patterns(4, 4)
    mjp = engine.TreeMJP(sched, Q, root_distn=pi if with_root else np.full(4, 0.25))
    want = np.exp(mjp.log_likelihood(engine.Observations.from_leaf_codes(sched, pats, leaves))['loglik'].cpu().numpy())
    np.testing.assert_allclose(want.sum(), 1.0, rtol=1e-12)
    _counts_match(got, want, n)


@pytest.mark.parametrize('S,with_root', [(20, True), (20, False), (61, True), (61, False)])
def test_leaf_pair_tables_and_node_marginals(S, with_root):
    """5-leaf tree, 2^18 sites: every leaf pair's joint table against the law from scipy's expm
    (_pair_joint), and every node's state frequencies against pi P_path (binomial |z| < 5 with the
    variance floored at one count)."""
    from raoteh_b200 import simulate
    rng = np.random.default_rng(100 + S)
    parent, length, leaves, sched = _tree(5, S, 0.3)
    Q, pi = _model(S, rng)
    n = 1 << 18
    obs, ns = simulate.simulate_sites(sched, Q, n, root_distn=pi if with_root else None, seed=5 + S,
                                      keep_node_states=True)
    codes = obs.data.cpu().numpy()
    ns = ns.cpu().numpy()
    assert np.array_equal(codes, ns[leaves])
    p0 = pi if with_root else np.full(S, 1.0 / S)
    Pp = _path_matrices(parent, length, Q, range(sched.n))
    for i in range(len(leaves)):
        for j in range(i + 1, len(leaves)):
            want = _pair_joint(parent, length, Q, p0, leaves[i], leaves[j])
            np.testing.assert_allclose(want.sum(), 1.0, rtol=1e-9)
            got = np.bincount(codes[i].astype(np.int64) * S + codes[j], minlength=S * S).reshape(S, S)
            e = n * want
            assert np.all(np.abs(got - e) < 5 * np.sqrt(e * (1 - want) + 1)), (i, j)
    for v in range(sched.n):
        want = p0 @ Pp[v]
        got = np.bincount(ns[v], minlength=S)
        e = n * want
        assert np.all(np.abs(got - e) < 5 * np.sqrt(e * (1 - want) + 1)), v


def _structure(fh, parent, length, leaves, ts):
    ns_all = fh.node_state.cpu().numpy()
    codes = fh.codes.cpu().numpy()
    assert np.array_equal(codes, ns_all[leaves])                       # leaves = the written codes
    cnt = fh.ev_count.cpu().numpy().astype(np.int64)
    assert np.array_equal(cnt[1:].sum(axis=0), fh.ev_total.cpu().numpy())
    for t in ts:
        ns, edges = fh.trajectory(t)
        assert len(edges) == len(parent) - 1
        for c, (times, states) in edges.items():
            assert states[0] == ns[parent[c]] and states[-1] == ns[c]
            assert len(states) == len(times) + 1
            assert len(times) < 2 or np.all(np.diff(times) > 0)
            assert np.all(times > 0) and np.all(times < length[c])
            assert np.all(states[1:] != states[:-1])


@pytest.mark.parametrize('S,time_dtype', [
    (3, 'float32'), (3, 'float64'), (4, 'float32'), (4, 'float64'), (7, 'float32'), (8, 'float32'),
    (8, 'float64'), (20, 'float32'), (61, 'float32')])
def test_histories_respect_structure(S, time_dtype):
    """Every history: segment states consistent at the nodes, times strictly increasing inside the
    branch in the stored precision, no self-transitions, per-branch counts summing to ev_total, and
    the leaf codes equal to the leaf states."""
    from raoteh_b200.simulate import ForwardHistories
    rng = np.random.default_rng(S)
    parent, length, leaves, sched = _tree(12, 40 + S, 0.3)
    Q, pi = _model(S, rng)
    fh = ForwardHistories(sched, Q, 4096, root_distn=pi, seed=3, cap=160, time_dtype=time_dtype)
    for _ in range(2):
        fh.draw()
        assert bool((fh.status == 0).all())
        _structure(fh, parent, length, leaves, range(0, 4096, 37))


@pytest.mark.parametrize('which', ['jc4', 'random3'])
def test_one_branch_jump_count_law(which):
    """Two-node tree, start state fixed by the root distribution, 2^20 histories: the histogram of
    jumps (k = 0..5 and the tail) against jump_count_distribution summed over end states, binomial
    |z| < 5; the dwell total is the branch length per history."""
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.simulate import ForwardHistories
    if which == 'jc4':
        S, t, a = 4, 0.7, 1
        Q = (np.ones((S, S)) - np.eye(S)) / (S - 1)
        Q -= np.diag(Q.sum(axis=1))
    else:
        S, t, a = 3, 1.3, 0
        Q = _random_q(3, np.random.default_rng(17))
    sched = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, t]))
    n = 1 << 20
    fh = ForwardHistories(sched, Q, n, root_distn=np.eye(S)[a], seed=21, cap=64, time_dtype='float64')
    fh.draw()
    assert bool((fh.node_state[0] == a).all())
    got = np.bincount(np.minimum(fh.ev_total.cpu().numpy(), 6), minlength=7)
    p = jump_count_distribution(Q, t, 60)[:, a, :].sum(axis=1)
    want = np.concatenate([p[:6], [1.0 - p[:6].sum()]])
    _counts_match(got, want, n, floor=0)
    np.testing.assert_allclose(fh.dwell_sum.sum().item(), t * n, rtol=1e-12)


@pytest.mark.parametrize('S,time_dtype', [(4, 'float64'), (4, 'float32'), (20, 'float32'), (61, 'float32')])
def test_history_statistics_match_prior_expectations(S, time_dtype):
    """Mean dwell and transition counts per history over 16 draws against the closed form with
    every leaf missing (|z| < 5); the dwell total of every draw is the tree length per history."""
    from raoteh_b200.simulate import ForwardHistories
    rng = np.random.default_rng(300 + S)
    parent, length, leaves, sched = _tree(8, 300 + S, 0.2)
    Q, pi = _model(S, rng)
    dwell_w, trans_w = _prior_stats(parent, length, Q, pi, leaves)
    n, groups = 1 << 16, 16
    fh = ForwardHistories(sched, Q, n, root_distn=pi, seed=9, cap=128, time_dtype=time_dtype)
    dwell = np.zeros((groups, S))
    trans = np.zeros((groups, S, S))
    for g in range(groups):
        fh.reset_statistics()
        fh.draw()
        dwell[g] = fh.dwell_sum.cpu().numpy() / n
        trans[g] = fh.trans_sum.cpu().numpy() / n
    np.testing.assert_allclose(dwell.sum(axis=1), length.sum(), rtol=1e-9 if time_dtype == 'float64' else 1e-6)
    _z_check(dwell, dwell_w)
    _z_check(trans.reshape(groups, -1), trans_w.reshape(-1), n * groups)


@pytest.mark.parametrize('S', [4, 20])
def test_layout_is_read_by_the_rao_teh_kernels(S):
    """Simulated float32 histories loaded into RaoTehChains: the device trajectory log-likelihood
    equals the host _mjp.get_trajectory_log_likelihood of trajectory(t) built from the same stored
    times (relative 1e-6)."""
    import networkx as nx
    from raoteh_b200.raoteh import RaoTehChains
    from raoteh_b200.sampler import _mjp, _sampler
    from raoteh_b200.simulate import ForwardHistories
    rng = np.random.default_rng(S)
    parent, length, leaves, sched = _tree(6, 60 + S, 0.3)
    Q, pi = _model(S, rng)
    T = 256
    fh = ForwardHistories(sched, Q, T, root_distn=pi, seed=4, cap=96)
    fh.draw(stats=False)
    ch = RaoTehChains(sched, Q, fh.leaf_observations(), n_chains=1, root_distn=pi, cap=96)
    ch.load_trajectories(fh.node_state, fh.ev_count, fh.ev_total, fh.ev_time, fh.ev_sb)
    assert ch.initialized
    dev = ch.trajectory_log_likelihood().cpu().numpy()
    Qg = nx.DiGraph()
    for a in range(S):
        for b in range(S):
            if a != b and Q[a, b] > 0:
                Qg.add_edge(a, b, weight=float(Q[a, b]))
    distn = dict((s, float(pi[s])) for s in range(S))
    for t in range(0, T, 17):
        ns, edges = ch.trajectory(t)
        G = _sampler._trajectory_to_graph(sched, list(range(S)), ns, edges, sched.n)
        host = _mjp.get_trajectory_log_likelihood(G, 0, distn, Qg)
        np.testing.assert_allclose(dev[t], host, rtol=1e-6)


def test_sweeps_run_from_loaded_fp64_histories():
    """S = 4 fp64 histories loaded into RaoTehChains with a larger cap sweep without error and keep
    the observed leaves."""
    from raoteh_b200.raoteh import RaoTehChains
    from raoteh_b200.simulate import ForwardHistories
    parent, length, leaves, sched = _tree(10, 8)
    Q, pi = _model(4, None)
    fh = ForwardHistories(sched, Q, 2048, root_distn=pi, seed=8, cap=64, time_dtype='float64')
    fh.draw()
    ch = RaoTehChains(sched, Q, fh.leaf_observations(), root_distn=pi, cap=128, time_dtype='float64', seed=2)
    ch.load_trajectories(fh.node_state, fh.ev_count, fh.ev_total, fh.ev_time, fh.ev_sb)
    assert bool((ch.sweep_count == 0).all())
    ch.sweep(5)
    assert bool((ch.sweep_count == 5).all())
    assert bool((ch.node_state[leaves] == fh.codes).all())


@pytest.mark.parametrize('S,n_traj', [(4, 4096), (11, 1024), (61, 512)])
def test_joint_distribution_no_burn_in(S, n_traj):
    """Geweke's joint-distribution test: (H, D) from the prior, Rao-Teh chains on D started at H and
    swept 100 times with no burn-in; the means over sites, sweeps and 16 groups equal the prior
    expectations (|z| < 5).  S = 4 runs the thread kernel, S = 11 and 61 the warp kernel."""
    from raoteh_b200.raoteh import RaoTehChains
    from raoteh_b200.simulate import ForwardHistories
    rng = np.random.default_rng(500 + S)
    parent, length, leaves, sched = _tree(6, 500 + S, 0.2)
    Q, pi = _model(S, rng)
    dwell_w, trans_w = _prior_stats(parent, length, Q, pi, leaves)
    groups, n_sweeps = 16, 100
    dwell = np.zeros((groups, S))
    trans = np.zeros((groups, S, S))
    for g in range(groups):
        fh = ForwardHistories(sched, Q, n_traj, root_distn=pi, seed=1000 + g, cap=128)
        fh.draw(stats=False)
        ch = RaoTehChains(sched, Q, fh.leaf_observations(), root_distn=pi, seed=2000 + g, cap=128)
        ch.load_trajectories(fh.node_state, fh.ev_count, fh.ev_total, fh.ev_time, fh.ev_sb)
        ch.sweep(n_sweeps)
        dwell[g] = ch.dwell_sum.cpu().numpy() / (n_traj * n_sweeps)
        trans[g] = ch.trans_sum.cpu().numpy() / (n_traj * n_sweeps)
    np.testing.assert_allclose(dwell.sum(axis=1), length.sum(), rtol=1e-5)
    _z_check(dwell, dwell_w)
    _z_check(trans.reshape(groups, -1), trans_w.reshape(-1), n_traj * groups)


def _hky_g4_i(sched):
    from raoteh_b200 import synth
    from raoteh_b200.mixture import SiteMixtureMJP, discrete_gamma_rates
    Q, pi = synth.hky85()
    rates = np.concatenate([discrete_gamma_rates(0.5, 4) / 0.8, [0.0]])
    weights = np.array([0.2, 0.2, 0.2, 0.2, 0.2])
    return SiteMixtureMJP(sched, Q, root_distn=pi, rates=rates, weights=weights), Q, pi


def test_mixture_hky_gamma_invariant():
    """HKY+G4+I, 4 leaves, 2^20 sites: class frequencies against the weights (multinomial |z| < 5),
    every +I site constant over the tree, and per class the 256 leaf-pattern counts against
    exp(that class's log-likelihood)."""
    from raoteh_b200 import engine
    parent, length, leaves, sched = _tree(4, 12, 0.5)
    mix, Q, pi = _hky_g4_i(sched)
    n = 1 << 20
    obs, cls, ns = mix.simulate(n, seed=3, keep_node_states=True)
    cls = cls.cpu().numpy()
    ns = ns.cpu().numpy()
    counts = np.bincount(cls, minlength=5)
    _counts_match(counts, mix.weights, n)
    inv = cls == 4
    assert np.all(ns[:, inv] == ns[0, inv][None, :])
    codes = obs.data.cpu().numpy()
    pats = engine.Observations.from_leaf_codes(sched, _all_patterns(4, 4), leaves)
    for k in range(5):
        want = np.exp(mix.classes[k].log_likelihood(pats)['loglik'].cpu().numpy())
        _counts_match(_patterns(codes[:, cls == k], 4), want, int(counts[k]))


def test_mixture_mg94_omega_classes():
    """Three MG94 omega classes (M2a-like), 5 leaves, 2^17 sites: class frequencies, and per class
    two leaf pairs' joint tables against that class's P (|z| < 5, variance floored at one count)."""
    from raoteh_b200 import synth
    from raoteh_b200.mixture import SiteMixtureMJP
    parent, length, leaves, sched = _tree(5, 13, 0.2)
    Qs, pi = [], None
    for om in (0.1, 1.0, 3.0):
        Q, pi, _ = synth.mg94(omega=om)
        Qs.append(Q)
    weights = np.array([0.6, 0.3, 0.1])
    mix = SiteMixtureMJP(sched, np.stack(Qs), root_distn=pi, weights=weights)
    n = 1 << 17
    obs, cls = mix.simulate(n, seed=4)
    cls = cls.cpu().numpy()
    counts = np.bincount(cls, minlength=3)
    _counts_match(counts, weights, n)
    codes = obs.data.cpu().numpy()
    for k in range(3):
        sel = codes[:, cls == k]
        for i, j in ((0, 1), (2, 4)):
            want = _pair_joint(parent, length, Qs[k], pi, leaves[i], leaves[j])
            got = np.bincount(sel[i].astype(np.int64) * 61 + sel[j], minlength=61 * 61).reshape(61, 61)
            e = counts[k] * want
            assert np.all(np.abs(got - e) < 5 * np.sqrt(e * (1 - want) + 1)), (k, i, j)


def test_mixture_with_one_class_is_the_single_class_call():
    from raoteh_b200 import simulate
    from raoteh_b200.mixture import SiteMixtureMJP
    parent, length, leaves, sched = _tree(9, 14)
    Q, pi = _model(4, None)
    a = simulate.simulate_sites(sched, Q, 100003, root_distn=pi, seed=6, k=2)
    b, cls = SiteMixtureMJP(sched, Q, root_distn=pi).simulate(100003, seed=6, k=2)
    assert bool((cls == 0).all())
    assert np.array_equal(a.data.cpu().numpy(), b.data.cpu().numpy())


def _history_abi(sched, Qk, weights, pi, n, seed, cap=128):
    """rt_forward_simulate, RT_SIM_HISTORY with K classes, straight through the C ABI."""
    import torch
    from raoteh_b200 import _native
    from raoteh_b200.engine import _ptr, _stream
    K, S = Qk.shape[0], Qk.shape[-1]
    dev = 'cuda'
    ops, _ = sched.up_program()
    ops = torch.from_numpy(ops).to(dev)
    T = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    parent, length = T(sched.parent, np.int32), T(sched.length, np.float64)
    Qd, w, p = T(Qk, np.float64), T(weights, np.float64), T(pi, np.float64)
    out = dict(node_state=torch.zeros((sched.n, n), dtype=torch.uint8, device=dev),
               ev_count=torch.zeros((sched.n, n), dtype=torch.uint8, device=dev),
               ev_total=torch.zeros(n, dtype=torch.int32, device=dev),
               ev_time=torch.zeros((n, cap), dtype=torch.float32, device=dev),
               ev_sb=torch.zeros((n, cap), dtype=torch.uint8, device=dev),
               status=torch.zeros(n, dtype=torch.int8, device=dev),
               site_class=torch.zeros(n, dtype=torch.uint8, device=dev),
               dwell=torch.zeros((K, S), dtype=torch.float64, device=dev),
               trans=torch.zeros((K, S, S), dtype=torch.float64, device=dev))
    A = _native.ForwardArgs()
    A.S, A.n_nodes, A.n_ops, A.K, A.mode, A.cap = S, sched.n, len(ops), K, _native.SIM_HISTORY, cap
    A.n_traj, A.traj_stride, A.seed = n, n, seed
    A.program, A.parent, A.length = _ptr(ops), _ptr(parent), _ptr(length)
    A.class_weight, A.Q, A.root_distn = _ptr(w), _ptr(Qd), _ptr(p)
    for f in ('node_state', 'ev_count', 'ev_total', 'ev_time', 'ev_sb', 'status', 'site_class'):
        setattr(A, f, _ptr(out[f]))
    A.dwell_sum, A.trans_sum = _ptr(out['dwell']), _ptr(out['trans'])
    _native.check(_native.lib().rt_forward_simulate(ctypes.byref(A), _stream()), 'rt_forward_simulate')
    return out


def test_mixture_histories_per_class():
    """HKY+G4+I histories through the C ABI, 2^18 sites: +I sites have no jump, every class's mean
    dwell and transition counts per site match that class's prior expectations (|z| < 5 over 16
    interleaved groups of sites; the statistics come from the trajectories)."""
    from raoteh_b200 import synth
    from raoteh_b200.mixture import discrete_gamma_rates
    parent, length, leaves, sched = _tree(8, 15, 0.2)
    Q, pi = synth.hky85()
    rates = np.concatenate([discrete_gamma_rates(0.5, 4) / 0.8, [0.0]])
    Qk = rates[:, None, None] * Q[None]
    n = 1 << 18
    out = _history_abi(sched, Qk, np.full(5, 0.2), pi, n, seed=31)
    assert bool((out['status'] == 0).all())
    cls = out['site_class'].cpu().numpy()
    tot = out['ev_total'].cpu().numpy()
    assert np.all(tot[cls == 4] == 0)
    _counts_match(np.bincount(cls, minlength=5), np.full(5, 0.2), n)
    # per-class totals from the accumulators against the closed form times the class counts
    counts = np.bincount(cls, minlength=5)
    dw = out['dwell'].cpu().numpy()
    np.testing.assert_allclose(dw.sum(axis=1), counts * length.sum(), rtol=1e-6)
    cnt = out['ev_count'].cpu().numpy()
    for k in range(4):
        _, trans_w = _prior_stats(parent, length, Qk[k], pi, leaves)
        per_site = tot[cls == k].astype(float)
        groups = per_site[: len(per_site) // 16 * 16].reshape(16, -1).mean(axis=1)
        _z_check(groups[:, None], [trans_w.sum()])
        np.testing.assert_allclose(out['trans'][k].sum().item(), per_site.sum())
    assert cnt[:, cls == 4].sum() == 0


def test_shards_repeats_and_replicates():
    """Two shards concatenate to the unsharded output bit for bit (codes, node states, histories),
    a repeated call reproduces it, and replicate k + 1 differs from k."""
    import torch
    from raoteh_b200 import simulate
    parent, length, leaves, sched = _tree(10, 16)
    Q, pi = _model(4, None)
    n = 50001
    full, ns = simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=7, k=3, keep_node_states=True)
    a, nsa = simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=7, k=3, keep_node_states=True, n_traj=20000)
    b, nsb = simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=7, k=3, keep_node_states=True, traj0=20000)
    assert torch.equal(torch.cat([a.data, b.data], dim=1), full.data)
    assert torch.equal(torch.cat([nsa, nsb], dim=1), ns)
    again = simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=7, k=3)
    assert torch.equal(again.data, full.data)
    other = simulate.simulate_sites(sched, Q, n, root_distn=pi, seed=7, k=4)
    assert float((other.data != full.data).float().mean()) > 0.3
    hf = simulate.ForwardHistories(sched, Q, n, root_distn=pi, seed=7)
    h1 = simulate.ForwardHistories(sched, Q, 20000, root_distn=pi, seed=7)
    h2 = simulate.ForwardHistories(sched, Q, n - 20000, root_distn=pi, seed=7, traj0=20000)
    for h in (hf, h1, h2):
        h.draw()
    for f in ('node_state', 'ev_count', 'codes'):
        assert torch.equal(torch.cat([getattr(h1, f), getattr(h2, f)], dim=1), getattr(hf, f)), f
    for f in ('ev_total', 'ev_time', 'ev_sb'):
        assert torch.equal(torch.cat([getattr(h1, f), getattr(h2, f)], dim=0), getattr(hf, f)), f
    nodes0 = hf.node_state.clone()
    hf.draw()                                      # the next draw is replicate k = 1
    assert float((hf.node_state != nodes0).float().mean()) > 0.3


def test_missing_cells_follow_the_template():
    """missing_like: every cell missing in the template (site i % N) is missing in the output, every
    other cell is the code drawn without a template."""
    import torch
    from raoteh_b200 import engine, simulate
    parent, length, leaves, sched = _tree(7, 18)
    Q, pi = _model(4, None)
    N, B = 3001, 5
    rng = np.random.default_rng(2)
    real = rng.integers(0, 4, size=(len(leaves), N)).astype(np.uint8)
    real[rng.random(real.shape) < 0.2] = 255
    tmpl = engine.Observations.from_leaf_codes(sched, real, leaves)
    plain = simulate.simulate_sites(sched, Q, N * B, root_distn=pi, seed=1)
    gapped = simulate.simulate_sites(sched, Q, N * B, root_distn=pi, seed=1, missing_like=tmpl)
    assert np.array_equal(gapped.obs_slot, tmpl.obs_slot)
    want = np.where(np.tile(real, B) == 255, 255, plain.data.cpu().numpy())
    assert np.array_equal(gapped.data.cpu().numpy(), want)
    fh = simulate.ForwardHistories(sched, Q, N * B, root_distn=pi, seed=1)
    fh.draw(stats=False)
    lo = fh.leaf_observations(missing_like=tmpl).data.cpu().numpy()
    assert np.array_equal(lo, np.where(np.tile(real, B) == 255, 255, fh.codes.cpu().numpy()))
    # the simulated alignment feeds the likelihood as it is
    mjp = engine.TreeMJP(sched, Q, root_distn=pi)
    r = mjp.log_likelihood(gapped)
    assert bool(torch.isfinite(r['loglik']).all())


def test_capacity_and_long_branch_errors():
    """A tiny cap gives status 4 and a branch with ~400 expected jumps status 3; ForwardHistories
    raises NativeError with the advice."""
    from raoteh_b200 import _native
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.simulate import ForwardHistories
    parent, length, leaves, sched = _tree(10, 19)
    Q, pi = _model(4, None)
    fh = ForwardHistories(sched, Q, 1000, root_distn=pi, seed=1, cap=2)
    with pytest.raises(_native.NativeError, match='larger cap'):
        fh.draw()
    assert bool((fh.status == 4).any()) and bool((fh.ev_total[fh.status == 4] == 0).all())
    long = TreeSchedule(np.array([-1, 0], dtype=np.int32), np.array([0.0, 400.0]))
    fh = ForwardHistories(long, Q, 64, root_distn=pi, seed=1, cap=2048)
    with pytest.raises(_native.NativeError, match='subdivide'):
        fh.draw()
    assert bool((fh.status == 3).all())
    with pytest.raises(ValueError):
        ForwardHistories(sched, _random_q(7, np.random.default_rng(0)), 10, time_dtype='float64')
