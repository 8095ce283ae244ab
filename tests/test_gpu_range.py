"""The tree kernels at the edges of their range, against the log-space reference (range_oracle):
S <= 8 on trees on both sides of the size where the down walk's per-node tables stop fitting in
shared memory and the level-synchronous kernels take over.  Every output must be finite and match
the reference to the suite's tolerances."""
import numpy as np
import pytest

from oracle import np_oracle
import range_oracle
from raoteh_b200 import synth

pytestmark = pytest.mark.gpu

RTOL = 1e-10        # log-likelihoods
RTOL_E = 1e-9       # expectations


@pytest.fixture(scope='module')
def rt():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import raoteh_b200.engine as engine
    return engine


def _np(x):
    return x.cpu().numpy() if hasattr(x, 'cpu') else np.asarray(x)


def _model(S, rng):
    if S == 4:
        return synth.hky85()
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    Q /= np.abs(np.diag(Q)).mean()
    return Q, rng.dirichlet(np.ones(S) * 2)


def walk_smem(sched, S, obs_slot, branch=False):
    """Shared memory of the S <= 8 down walk (launch_walk in rt_posterior_small.cu); above
    100 KB the level-synchronous kernels run instead."""
    ops, n_slots = sched.up_program(obs_slot)
    NS = 2
    return (24 * len(ops) + 8 * (2 * S + sched.n * ((3 if branch else 2) * S * S + S * (S + 1))) +
            8 * n_slots * NS * S * 128)


def _check_stats(got, ref, N=None):
    ll = _np(got['loglik'])[:N]
    st = _np(got['status'])[:N]
    assert (st == ref['status']).all(), np.flatnonzero(st != ref['status'])[:10]
    ok = ref['status'] == 0
    assert np.isfinite(ll[ok]).all()
    np.testing.assert_allclose(ll[ok], ref['loglik'][ok], rtol=RTOL)
    np.testing.assert_allclose(float(got['loglik_sum']), ref['loglik_sum'], rtol=RTOL)
    for k in ('dwell', 'trans', 'root_post_sum'):
        g = _np(got[k])
        assert np.isfinite(g).all(), k
        scale = max(np.abs(ref[k]).max(), 1e-300)
        np.testing.assert_allclose(g / scale, ref[k] / scale, rtol=0, atol=RTOL_E, err_msg=k)


def _check_W(W, ref):
    W = _np(W)
    assert np.isfinite(W).all()
    for b in range(1, len(W)):
        scale = max(np.abs(ref['W'][b]).max(), 1e-300)
        np.testing.assert_allclose(W[b] / scale, ref['W'][b] / scale, rtol=0, atol=RTOL_E)


def _observations(rt, kind, sched, S, leaves, N, rng, codes):
    """(engine observations, np_oracle observations) of one encoding."""
    n = sched.n
    if kind in ('codes', 'codes4'):
        make = rt.Observations.from_leaf_codes if kind == 'codes' else rt.Observations.from_leaf_codes4
        return (make(sched, codes, leaves),
                np_oracle.Obs('codes', S, N, leaf_nodes=leaves, codes=codes))
    if kind == 'mask':
        full = np.uint64((1 << S) - 1)
        mask = np.full((n, N), full, dtype=np.uint64)
        c = codes.astype(np.uint64)
        mask[leaves] = np.where(codes == 255, full, np.uint64(1) << c)
        # observed internal nodes: a random allowed set (with the simulated state) at some cells
        internal = sched.internal[1:]
        bits = rng.random((len(internal), N, S)) < 0.7
        bits[..., 0] = True
        sets = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)).sum(axis=2).astype(np.uint64)
        sel = rng.random((len(internal), N)) < 0.3
        mask[internal] = np.where(sel, sets, full)
        return rt.Observations.from_masks(sched, mask), np_oracle.Obs('mask', S, N, mask=mask)
    assert kind == 'dense'
    nodes = np.concatenate([leaves, sched.internal[1:3]])
    lik = 0.05 + rng.random((len(nodes), S, N)) ** 2
    lik[:len(leaves)] += 2.0 * (np.arange(S)[None, :, None] == np.where(codes == 255, 0, codes)[:, None, :])
    lik_all = np.zeros((n, N, S))
    lik_all[nodes] = lik.transpose(0, 2, 1)
    has = np.zeros(n, dtype=bool)
    has[nodes] = True
    return (rt.Observations.from_dense(sched, lik, nodes),
            np_oracle.Obs('dense', S, N, lik=lik_all, has=has))


@pytest.mark.parametrize('kind', ['codes', 'codes4', 'mask', 'dense'])
# `walk`: whether the down walk runs (else the level-synchronous kernels) for every encoding, with
# and without per-branch output
@pytest.mark.parametrize('S,n_leaves,walk', [(2, 120, True), (2, 300, False), (4, 48, True),
                                             (4, 120, False), (5, 32, True), (5, 80, False),
                                             (8, 12, True), (8, 32, False)])
def test_large_tree_small_S(rt, S, n_leaves, walk, kind):
    import torch
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(1000 * S + n_leaves)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    Q, pi = _model(S, rng)
    N = 1000                                   # not a multiple of 128
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, N, rng, 0.05)
    sched = TreeSchedule(parent, length)
    P = np_oracle.expm_edges(Q, length)
    obs, oobs = _observations(rt, kind, sched, S, leaves, N, rng, codes)
    for branch in (False, True):
        assert (walk_smem(sched, S, obs.obs_slot, branch) <= 100 * 1024) == walk
    K = range_oracle.transition_kernels(Q, length)
    ref = range_oracle.posterior(parent, length, Q, P, oobs, pi, K=K)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi, P=P)

    _check_stats(mjp.expected_history_statistics(obs), ref)

    post = mjp.posterior(obs, want_node_distn=True)
    _check_W(post['W'], ref)
    nd = _np(post['node_distn'])
    assert np.isfinite(nd[:, :, :N]).all()
    for v in sched.internal:
        np.testing.assert_allclose(nd[sched.store_index[v], :, :N].T, ref['node_distn'][v],
                                   rtol=0, atol=RTOL_E)
    post = mjp.posterior(obs, want_node_distn=False)
    _check_W(post['W'], ref)
    post = mjp.posterior(obs, want_node_distn=False, overlap_chunks=3)
    _check_W(post['W'], ref)

    br = mjp.branch_expectations(obs, K=torch.from_numpy(K).cuda())
    got = _np(br['branch'])
    assert np.isfinite(got).all()
    np.testing.assert_allclose(got, ref['branch'], rtol=0,
                               atol=RTOL_E * max(1.0, np.abs(ref['branch']).max()))

    if kind in ('codes', 'codes4'):
        host = codes if kind == 'codes' else rt.pack_codes4(codes)
        pinned = torch.from_numpy(np.ascontiguousarray(host)).pin_memory()
        out_ll = torch.empty(N, dtype=torch.float64).pin_memory()
        out_st = torch.empty(N, dtype=torch.int8).pin_memory()
        r = mjp.expected_history_statistics_from_host(pinned, leaves, out_ll, out_st, n_chunks=3,
                                                      packed=kind == 'codes4')
        torch.cuda.synchronize()
        r.update(loglik=out_ll, status=out_st)
        _check_stats(r, ref)


@pytest.mark.parametrize('kind', ['codes4', 'dense'])
def test_level_kernels_over_several_workspace_chunks(rt, kind):
    """Without a node-marginal buffer the level kernels take the sites in workspace chunks of 65536:
    70001 sites (an odd remainder of 4465 after the first chunk) made of 7 copies of 10001 distinct
    sites, so a chunk offset that is off by any amount pairs a site with the wrong data."""
    import torch
    from raoteh_b200.lowering import TreeSchedule
    S, n_leaves, base, reps = 8, 32, 10001, 7
    rng = np.random.default_rng(8032)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    Q, pi = _model(S, rng)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, base, rng, 0.05)
    sched = TreeSchedule(parent, length)
    P = np_oracle.expm_edges(Q, length)
    obs1, oobs = _observations(rt, kind, sched, S, leaves, base, rng, codes)
    N = base * reps
    if kind == 'codes4':
        obs = rt.Observations.from_leaf_codes4(sched, np.tile(codes, reps), leaves)
    else:
        lik = _np(obs1.data)[:, :, :base]
        obs = rt.Observations.from_dense(sched, np.tile(lik, reps), np.argsort(obs1.obs_slot)[-lik.shape[0]:])
    assert walk_smem(sched, S, obs.obs_slot) > 100 * 1024
    K = range_oracle.transition_kernels(Q, length)
    one = range_oracle.posterior(parent, length, Q, P, oobs, pi, K=K)
    ref = dict(status=np.tile(one['status'], reps), loglik=np.tile(one['loglik'], reps),
               loglik_sum=reps * one['loglik_sum'], W=reps * one['W'],
               branch=np.tile(one['branch'], (1, reps)))
    for k in ('dwell', 'trans', 'root_post_sum'):
        ref[k] = reps * one[k]
    mjp = rt.TreeMJP(sched, Q, root_distn=pi, P=P)
    r = mjp.expected_history_statistics(obs)
    _check_stats(r, ref)
    _check_W(r['W'], ref)
    br = mjp.branch_expectations(obs, K=torch.from_numpy(K).cuda())
    got = _np(br['branch'])
    assert got.shape == (sched.n, N) and np.isfinite(got).all()
    np.testing.assert_allclose(got, ref['branch'], rtol=0,
                               atol=RTOL_E * max(1.0, np.abs(ref['branch']).max()))
