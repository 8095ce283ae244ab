"""The 4-state down walk keeps every state vector of a lane in a lane-dependent XOR order (its
frame), so that the warp reduction of the edge statistics needs no selects.  These tests run
S = 4 through the walk for every observation encoding and output, with data that puts every code
and a missing code at every lane and in both site slots of a thread, and check that W, node
marginals, per-branch expectations and root_post_sum come back in natural state order, against
the NumPy oracle."""
import numpy as np
import pytest

from oracle import np_oracle
import range_oracle
from raoteh_b200 import synth

pytestmark = pytest.mark.gpu

S = 4
N = 2 * 5 * 256 + 77           # not a multiple of the 256 sites of a walk tile
TOL = 1e-10


@pytest.fixture(scope='module')
def rt():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import raoteh_b200.engine as engine
    return engine


def walk_smem(sched, obs_slot, branch):
    """Shared memory of the S <= 8 down walk (launch_walk in rt_posterior_small.cu); above 100 KB
    the level-synchronous kernels run instead."""
    ops, n_slots = sched.up_program(obs_slot)
    NS = 2
    return (24 * len(ops) + 8 * (2 * S + sched.n * ((3 if branch else 2) * S * S + S * (S + 1))) +
            8 * n_slots * NS * S * 128)


def _problem(kind):
    """Tree, P with structural zeros, engine and oracle observations.  Leaf j of site s has code
    (s // 32 + s + j) % 5, 4 = missing: every code at every lane (s % 32) and slot of a thread.
    Column 3 of P is zero on one leaf edge, so the sites where that leaf shows state 3 are
    infeasible; one entry of an internal edge's P is zero as well."""
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(4004)
    parent, length, leaves = synth.random_binary_tree(12, 0.15, rng)
    Q, pi = synth.hky85()
    sched = TreeSchedule(parent, length)
    P = np_oracle.expm_edges(Q, length)
    b0 = leaves[0]
    P[b0][:, 3] = 0.0
    b1 = sched.internal[1]
    P[b1][1, 2] = 0.0
    s = np.arange(N)
    c = (s[None, :] // 32 + s[None, :] + np.arange(len(leaves))[:, None]) % 5
    codes = np.where(c == 4, 255, c).astype(np.uint8)
    n = sched.n
    if kind in ('codes', 'codes4'):
        oobs = np_oracle.Obs('codes', S, N, leaf_nodes=leaves, codes=codes)
        return parent, length, sched, P, Q, pi, (kind, codes, leaves), oobs
    if kind == 'mask':
        full = np.uint64((1 << S) - 1)
        mask = np.full((n, N), full, dtype=np.uint64)
        mask[leaves] = np.where(codes == 255, full, np.uint64(1) << codes.astype(np.uint64))
        # an observed internal node: a random allowed set at some sites
        bits = rng.random((N, S)) < 0.6
        bits[:, 0] = True
        sets = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)).sum(axis=1).astype(np.uint64)
        mask[sched.internal[2]] = np.where(rng.random(N) < 0.4, sets, full)
        return parent, length, sched, P, Q, pi, (kind, mask), np_oracle.Obs('mask', S, N, mask=mask)
    # dense: the leaf codes as soft emission rows (exact one-hot on leaf b0), plus one internal node
    onehot = (np.arange(S)[None, :, None] == codes[:, None, :]).astype(float)
    lik = np.where(codes[:, None, :] == 255, 1.0, onehot + 0.1 * rng.random(onehot.shape))
    lik[0] = np.where(codes[0][None, :] == 255, 1.0, onehot[0])
    nodes = np.concatenate([leaves, [sched.internal[2]]])
    lik = np.concatenate([lik, 0.2 + rng.random((1, S, N))])
    full = np.ones((n, N, S))
    has = np.zeros(n, dtype=bool)
    has[nodes] = True
    full[nodes] = lik.transpose(0, 2, 1)
    return parent, length, sched, P, Q, pi, (kind, lik, nodes), np_oracle.Obs('dense', S, N, lik=full, has=has)


def _engine_obs(rt, sched, spec):
    kind = spec[0]
    if kind == 'codes':
        return rt.Observations.from_leaf_codes(sched, spec[1], spec[2])
    if kind == 'codes4':
        return rt.Observations.from_leaf_codes4(sched, spec[1], spec[2])
    if kind == 'mask':
        return rt.Observations.from_masks(sched, spec[1])
    return rt.Observations.from_dense(sched, spec[1], spec[2])


def _reference(parent, P, oobs, pi, weight, K):
    """Oracle log-lik, status, W, node marginals, root_post_sum and per-branch expectations."""
    L, ls = np_oracle.prune(parent, P, oobs)
    with np.errstate(divide='ignore'):
        ll = np.log(L[0] @ pi) + ls[0]
    ok = np.isfinite(ll)
    Lk = L[:, ok]
    D, G = np_oracle.node_distn(parent, P, Lk, pi)
    w = weight[ok][None, :, None]
    D, G = D * w, G * w
    n = len(parent)
    nd = np.zeros((n, N, S))
    nd[:, ok] = D
    branch = np.zeros((n, N))
    for b in range(1, n):
        branch[b, ok] = np.einsum('sa,sa->s', G[b], Lk[b] @ K[b].T)
    return dict(ok=ok, loglik=ll, W=np_oracle.edge_weight_matrices(parent, P, Lk, G),
                node_distn=nd, root_post_sum=D[0].sum(axis=0), branch=branch)


def _close(got, want, what):
    scale = max(np.abs(want).max(), 1e-300)
    np.testing.assert_allclose(got / scale, want / scale, rtol=0, atol=TOL, err_msg=what)


@pytest.mark.parametrize('kind', ['codes', 'codes4', 'mask', 'dense'])
@pytest.mark.parametrize('mode', ['stats', 'node_distn', 'weighted', 'branch'])
def test_walk_frames_s4(rt, kind, mode):
    import torch
    parent, length, sched, P, Q, pi, spec, oobs = _problem(kind)
    obs = _engine_obs(rt, sched, spec)
    assert walk_smem(sched, obs.obs_slot, mode == 'branch') <= 100 * 1024
    K = range_oracle.transition_kernels(Q, length)
    rng = np.random.default_rng(7)
    weight = rng.random(N) * 2.0 if mode == 'weighted' else np.ones(N)
    ref = _reference(parent, P, oobs, pi, weight, K)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi, P=P)
    ok = ref['ok']
    assert 0 < (~ok).sum() < N // 2

    if mode == 'branch':
        r = mjp.branch_expectations(obs, K=torch.from_numpy(K).cuda())
        got = r['branch'].cpu().numpy()
        assert np.isfinite(got).all()
        _close(got, ref['branch'], 'branch')
    else:
        sw = torch.from_numpy(weight).cuda() if mode == 'weighted' else None
        r = mjp.posterior(obs, want_node_distn=mode == 'node_distn', site_weight=sw)
        W = r['W'].cpu().numpy()
        assert np.isfinite(W).all()
        for b in range(1, sched.n):
            _close(W[b], ref['W'][b], 'W[%d]' % b)
        _close(r['root_post_sum'].cpu().numpy(), ref['root_post_sum'], 'root_post_sum')
        if mode == 'node_distn':
            nd = r['node_distn'].cpu().numpy()
            for v in sched.internal:
                _close(nd[sched.store_index[v], :, :N].T, ref['node_distn'][v], 'node_distn[%d]' % v)
    st = r['status'].cpu().numpy()
    assert ((st == 0) == ok).all()
    np.testing.assert_allclose(r['loglik'].cpu().numpy()[ok], ref['loglik'][ok], rtol=TOL)
