"""Parity of the CUDA path (through the C ABI) against the pinned oracle and the
committed golden fixtures.  Tolerance: relative 1e-10 on log-likelihoods and
expectations in fp64 (BASELINE.json north_star)."""
import numpy as np
import pytest
import scipy.linalg

from oracle import np_oracle
from helpers import load_golden, case_sched_mask, oracle_obs_from_mask

pytestmark = pytest.mark.gpu

RTOL = 1e-10


@pytest.fixture(scope='module')
def rt():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import raoteh_b200.engine as engine
    return engine


def _engine_case(rt, case):
    T, root, sched, mask = case_sched_mask(case)
    S = case['nstates']
    Q = np.array(case['Q'])
    pi = None if case.get('root_distn') is None else np.array(case['root_distn'])
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    obs = rt.Observations.from_masks(sched, mask[:, None])
    return sched, Q, pi, mjp, obs, mask


@pytest.mark.parametrize('S', [2, 3, 4, 6, 20, 48, 61, 64])
def test_expm_matches_scipy(rt, S):
    # t in 2^[-5,5] as raoteh/sampler/tests/test_expm.py:48-82
    import torch
    rng = np.random.default_rng(1234 + S)
    Q = rng.exponential(1.0, size=(3, S, S))
    Q[1] *= rng.random((S, S)) < 0.3
    for q in Q:
        np.fill_diagonal(q, 0)
        q -= np.diag(q.sum(axis=1))
    t = 2.0 ** rng.uniform(-5, 5, size=24)
    q_index = rng.integers(0, 3, size=24).astype(np.int32)
    dev = torch.device('cuda')
    P = torch.empty((24, S, S), dtype=torch.float64, device=dev)
    from raoteh_b200 import _native
    Qd, qd, td = (torch.from_numpy(Q).to(dev), torch.from_numpy(q_index).to(dev),
                  torch.from_numpy(t).to(dev))   # keep the device tensors alive
    rc = _native.lib().rt_expm_batched(Qd.data_ptr(), qd.data_ptr(), td.data_ptr(), 24, S,
                                       P.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, 'rt_expm_batched')
    P = P.cpu().numpy()
    for m in range(24):
        ref = scipy.linalg.expm(Q[q_index[m]] * t[m])
        np.testing.assert_allclose(P[m], ref, rtol=0, atol=2e-13)
        np.testing.assert_allclose(P[m].sum(axis=1), 1.0, rtol=0, atol=1e-12)


@pytest.mark.parametrize('S', [2, 4, 6, 20, 48, 61])
def test_frechet_contract_matches_scipy(rt, S):
    import torch
    from raoteh_b200 import _native
    rng = np.random.default_rng(99 + S)
    Q = rng.exponential(1.0, size=(1, S, S))
    np.fill_diagonal(Q[0], 0)
    Q[0] -= np.diag(Q[0].sum(axis=1))
    Q[0] /= np.abs(np.diag(Q[0])).mean()
    n = 12
    t = 2.0 ** rng.uniform(-5, 3, size=n)
    W = rng.exponential(1.0, size=(n, S, S)) * (rng.random((n, S, S)) < 0.5)
    W[3] = 0.0
    dev = torch.device('cuda')
    M = torch.empty((n, S, S), dtype=torch.float64, device=dev)
    Qd, td, Wd = (torch.from_numpy(Q).to(dev), torch.from_numpy(t).to(dev),
                  torch.from_numpy(W).to(dev))   # keep the device tensors alive
    rc = _native.lib().rt_frechet_contract(Qd.data_ptr(), None, td.data_ptr(), Wd.data_ptr(), n, S,
                                           M.data_ptr(), torch.cuda.current_stream().cuda_stream)
    _native.check(rc, 'rt_frechet_contract')
    M = M.cpu().numpy()
    for m in range(n):
        ref = np_oracle.frechet_contract(Q[0], t[m], W[m])
        scale = max(np.abs(ref).max(), 1e-300)
        np.testing.assert_allclose(M[m] / scale, ref / scale, rtol=0, atol=1e-12)


def test_golden_code2x3(rt):
    g = load_golden('code2x3.json')
    for call in g['calls']:
        sched, Q, pi, mjp, obs, mask = _engine_case(rt, call)
        if call['kind'] == 'likelihood':
            r = mjp.log_likelihood(obs)
            assert int(r['status'][0]) == 0
            np.testing.assert_allclose(np.exp(float(r['loglik'][0])), call['out'], rtol=RTOL)
        else:
            E = np.ones_like(Q) - np.eye(len(Q)) if call['E'] is None else np.array(call['E'])
            r = mjp.expected_history_statistics(obs)
            per_edge = (E[None] * Q[None] * r['M_edges'].cpu().numpy()).sum(axis=(1, 2))
            for a, b, v in call['out']:
                np.testing.assert_allclose(per_edge[sched.node_index[b]], v, rtol=1e-9, atol=1e-12)


def test_golden_random_cases(rt):
    g = load_golden('mjp_random.json')
    for case in g['cases']:
        sched, Q, pi, mjp, obs, mask = _engine_case(rt, case)
        S = case['nstates']
        r = mjp.expected_history_statistics(obs, want_node_distn=True)
        if 'raises' in case:
            assert int(r['status'][0]) == 1
            continue
        assert int(r['status'][0]) == 0
        np.testing.assert_allclose(np.exp(float(r['loglik'][0])), case['likelihood'], rtol=RTOL)
        np.testing.assert_allclose(r['dwell'].cpu().numpy(), case['dwell'], rtol=1e-9, atol=1e-12)
        ref_trans = np.array(case['trans'])
        np.fill_diagonal(ref_trans, 0.0)   # dense-reference quirk, see np_oracle._finish_ehs
        np.testing.assert_allclose(r['trans'].cpu().numpy(), ref_trans, rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(r['root_post_sum'].cpu().numpy(), case['root_post'],
                                   rtol=1e-10, atol=1e-14)
        nd = r['node_distn'].cpu().numpy()
        for v, d in case['node_distn'].items():
            i = sched.node_index[int(v)]
            if sched.store_index[i] >= 0:
                np.testing.assert_allclose(nd[sched.store_index[i], :, 0], d, rtol=1e-10, atol=1e-14)


def _synthetic(name, n_sites, seed, n_leaves, S):
    from raoteh_b200 import synth
    rng = np.random.default_rng(seed)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1 if S == 4 else 0.05, rng)
    if S == 4:
        Q, pi = synth.hky85()
    else:
        Q, pi, _ = synth.mg94()
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.01)
    return parent, length, leaves, Q, pi, codes


@pytest.mark.parametrize('S,n_leaves,n_sites', [(4, 32, 3001), (61, 16, 300), (61, 128, 515)])
def test_loglik_codes_matches_oracle(rt, S, n_leaves, n_sites):
    from raoteh_b200.lowering import TreeSchedule
    parent, length, leaves, Q, pi, codes = _synthetic('x', n_sites, 7 + S, n_leaves, S)
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    r = mjp.log_likelihood(obs, keep_partials=True, want_exponents=True)
    P_gpu = mjp.transition_matrices().cpu().numpy()
    P = np_oracle.expm_edges(Q, length)
    np.testing.assert_allclose(P_gpu[1:], P[1:], rtol=0, atol=1e-13)
    oobs = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    ll, st = np_oracle.log_likelihood(parent, P, oobs, pi)
    assert (r['status'].cpu().numpy() == st).all()
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), ll, rtol=RTOL)
    # stored partials: true value = partial * 2^exponent
    L, ls = np_oracle.prune(parent, P, oobs)
    part = r['partials'].cpu().numpy()
    expo = r['exponents'].cpu().numpy()
    for v in sched.internal[:: max(1, len(sched.internal) // 7)]:
        k = sched.store_index[v]
        mine = np.log(part[k].T) + expo[k][:, None] * np.log(2.0)
        with np.errstate(divide='ignore'):
            ref = np.log(L[v]) + ls[v][:, None]
        ok = np.isfinite(ref)
        np.testing.assert_allclose(mine[ok], ref[ok], rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize('S,n_leaves,n_sites', [(4, 32, 2000), (5, 9, 700), (61, 24, 260)])
def test_loglik_mask_and_dense_match_oracle(rt, S, n_leaves, n_sites):
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(31 + S)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    if S == 61:
        Q, pi, _ = synth.mg94()
    else:
        Q = rng.exponential(1.0, size=(S, S))
        np.fill_diagonal(Q, 0)
        Q -= np.diag(Q.sum(axis=1))
        pi = rng.dirichlet(np.ones(S))
    n = len(parent)
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    P = np_oracle.expm_edges(Q, length)
    # y-type: random allowed sets at every node (internal nodes mostly unrestricted)
    bits = rng.random((n, n_sites, S)) < 0.5
    bits[np.arange(n)[:, None], np.arange(n_sites)[None, :], rng.integers(0, S, size=(n, n_sites))] = True
    unrestricted = rng.random((n, n_sites)) < 0.6
    unrestricted[leaves] = rng.random((len(leaves), n_sites)) < 0.1
    bits[unrestricted] = True
    mask = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, None, :]).sum(axis=2).astype(np.uint64)
    obs = rt.Observations.from_masks(sched, mask)
    r = mjp.log_likelihood(obs)
    ll, st = np_oracle.log_likelihood(parent, P, np_oracle.Obs('mask', S, n_sites, mask=mask), pi)
    assert (r['status'].cpu().numpy() == st).all()
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), ll, rtol=RTOL)
    # z-type: emission likelihoods at the leaves and at two internal nodes
    nodes = np.concatenate([leaves, sched.internal[:2]])
    lik = rng.random((len(nodes), S, n_sites)) ** 3
    obs = rt.Observations.from_dense(sched, lik, nodes)
    r = mjp.log_likelihood(obs)
    full = np.ones((n, n_sites, S))
    has = np.zeros(n, dtype=bool)
    has[nodes] = True
    full[nodes] = lik.transpose(0, 2, 1)
    ll, st = np_oracle.log_likelihood(parent, P, np_oracle.Obs('dense', S, n_sites, lik=full, has=has), pi)
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), ll, rtol=RTOL)


@pytest.mark.parametrize('S,n_leaves,n_sites', [(4, 32, 5000), (3, 6, 100), (20, 9, 300), (61, 12, 333)])
def test_expectations_match_oracle(rt, S, n_leaves, n_sites):
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(5 + S)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    if S == 61:
        Q, pi, _ = synth.mg94()            # sparse codon matrix: structural zeros in P for short branches
    else:
        Q = rng.exponential(1.0, size=(S, S))
        np.fill_diagonal(Q, 0)
        Q -= np.diag(Q.sum(axis=1))
        Q /= np.abs(np.diag(Q)).mean()
        pi = rng.dirichlet(np.ones(S))
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.02)
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    r = mjp.expected_history_statistics(obs)
    P = np_oracle.expm_edges(Q, length)
    o = np_oracle.expected_history_statistics(
        parent, length, Q, P, np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes), pi)
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), o['loglik'], rtol=RTOL)
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(r['root_post_sum'].cpu().numpy(), o['root_post'].sum(axis=0), rtol=RTOL)
    # total expected dwell time = tree length per site
    np.testing.assert_allclose(float(r['dwell'].sum()), length.sum() * n_sites, rtol=1e-10)


@pytest.mark.parametrize('S,n_leaves,n_sites,kind', [(20, 9, 2500, 'codes'), (61, 10, 2112, 'codes'),     # 2112 = 16 * 132: vector code loads of the leaf scatter
                                                     (13, 8, 4133, 'codes'),     # odd row stride: scalar loads of the leaf scatter
                                                     (20, 7, 1300, 'mask'), (11, 6, 1100, 'dense')])
def test_large_state_down_pass_tiles_and_observation_kinds(rt, S, n_leaves, n_sites, kind):
    """The DMMA down pass (9 <= S <= 64) across several CTAs of the site axis (1024 sites each: the
    next tile's rows are prefetched across tile ends and past the last site), with 30 % unobserved
    leaf cells, and with mask / dense observations (contracted, not gathered), against the oracle
    (_mjp_dense.py:410-539).  Coded leaf edges go through down_leaf_scatter_kernel (2048 sites per
    CTA, groups of 16 sites, 256-bit loads when the row stride allows): the site counts cover
    several CTAs, a ragged last group, both load paths and the unobserved-site spread."""
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(77 + S)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.15, rng)
    if S == 61:
        Q, pi, _ = synth.mg94()
    else:
        Q = rng.exponential(1.0, size=(S, S))
        np.fill_diagonal(Q, 0)
        Q -= np.diag(Q.sum(axis=1))
        Q /= np.abs(np.diag(Q)).mean()
        pi = rng.dirichlet(np.ones(S))
    n = len(parent)
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    P = np_oracle.expm_edges(Q, length)
    if kind == 'codes':
        codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.3)
        obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
        oobs = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    elif kind == 'mask':
        bits = rng.random((n, n_sites, S)) < 0.4
        bits[np.arange(n)[:, None], np.arange(n_sites)[None, :], rng.integers(0, S, size=(n, n_sites))] = True
        unrestricted = rng.random((n, n_sites)) < 0.7
        unrestricted[leaves] = rng.random((len(leaves), n_sites)) < 0.1
        bits[unrestricted] = True
        mask = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, None, :]).sum(axis=2).astype(np.uint64)
        obs = rt.Observations.from_masks(sched, mask)
        oobs = np_oracle.Obs('mask', S, n_sites, mask=mask)
    else:
        lik = rng.random((len(leaves), S, n_sites)) ** 3
        obs = rt.Observations.from_dense(sched, lik, leaves)
        full = np.ones((n, n_sites, S))
        has = np.zeros(n, dtype=bool)
        has[leaves] = True
        full[leaves] = lik.transpose(0, 2, 1)
        oobs = np_oracle.Obs('dense', S, n_sites, lik=full, has=has)
    r = mjp.expected_history_statistics(obs)
    o = np_oracle.expected_history_statistics(parent, length, Q, P, oobs, pi)
    ok = np.isfinite(o['loglik'])
    assert ok.sum() > n_sites // 2
    np.testing.assert_allclose(r['loglik'].cpu().numpy()[ok], o['loglik'][ok], rtol=RTOL)
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(float(r['dwell'].sum()), length.sum() * ok.sum(), rtol=1e-10)


def test_support_sets_match_oracle(rt):
    import torch
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(77)
    S, n_sites = 7, 400
    parent, length, leaves = synth.random_binary_tree(10, 0.3, rng)
    n = len(parent)
    Q = np.triu(rng.exponential(1.0, size=(S, S)), 1)
    Q -= np.diag(Q.sum(axis=1))
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q)
    P = np_oracle.expm_edges(Q, length)
    bits = rng.random((n, n_sites, S)) < 0.4
    bits[np.arange(n)[:, None], np.arange(n_sites)[None, :], rng.integers(0, S, size=(n, n_sites))] = True
    mask = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, None, :]).sum(axis=2).astype(np.uint64)
    ref = np_oracle.support_masks(parent, P, bits)
    ref_mask = (ref.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, None, :]).sum(axis=2)
    dev_mask = torch.from_numpy(mask.view(np.int64).copy()).cuda()
    mjp.support_sets(dev_mask)
    got = dev_mask.cpu().numpy().view(np.uint64)
    assert (got == ref_mask).all()


def test_c2_full_size_properties(rt):
    """Full C2 size: size-independent properties (the oracle is too slow here)."""
    import torch
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    cfg = synth.config_c2(n_sites=1_000_000)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    mjp = rt.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'])
    obs = rt.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    s = torch.zeros(1, dtype=torch.float64, device='cuda')
    r = mjp.log_likelihood(obs, loglik_sum=s)
    ll = r['loglik']
    assert bool((r['status'] == 0).all()) and bool(torch.isfinite(ll).all())
    np.testing.assert_allclose(float(s[0]), float(ll.sum()), rtol=1e-12)
    # identical columns give identical log-likelihoods; check against the oracle on a slice
    sl = slice(123_456, 123_456 + 512)
    P = np_oracle.expm_edges(cfg['Q'], cfg['length'])
    ref, _ = np_oracle.log_likelihood(
        cfg['parent'], P, np_oracle.Obs('codes', 4, 512, leaf_nodes=cfg['leaves'],
                                         codes=cfg['codes'][:, sl]), cfg['pi'])
    np.testing.assert_allclose(ll[sl].cpu().numpy(), ref, rtol=RTOL)
    # expectations: total expected dwell = tree length * sites; transitions >= 0
    e = mjp.expected_history_statistics(obs)
    np.testing.assert_allclose(float(e['dwell'].sum()), cfg['length'].sum() * 1_000_000, rtol=1e-10)
    np.testing.assert_allclose(float(e['root_post_sum'].sum()), 1_000_000, rtol=1e-12)
    assert bool((e['trans'] >= 0).all())


def test_host_buffer_pipeline_matches_resident_path(rt):
    """The chunked host-buffer entry point (e2e path of bench.py) gives the same numbers, and so
    does the same site-chunk pipeline on device-resident observations of every encoding
    (expected_history_statistics(overlap_chunks=k)), for a site count that is not a multiple of
    the 128-site chunk granule."""
    import torch
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule, MISSING
    cfg = synth.config_c2(n_sites=10_007, n_leaves=16)
    keys = ('loglik', 'status', 'dwell', 'trans', 'root_post_sum')
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    mjp = rt.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'])
    obs = rt.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    ref = mjp.expected_history_statistics(obs)
    ref = {k: ref[k].clone() for k in keys}
    codes_pinned = torch.from_numpy(cfg['codes']).pin_memory()
    out_ll = torch.empty(10_007, dtype=torch.float64).pin_memory()
    out_st = torch.empty(10_007, dtype=torch.int8).pin_memory()
    r = mjp.expected_history_statistics_from_host(codes_pinned, cfg['leaves'], out_ll, out_st, n_chunks=3)
    torch.cuda.synchronize()
    np.testing.assert_allclose(out_ll.numpy(), ref['loglik'].cpu().numpy(), rtol=1e-14)
    assert (out_st.numpy() == ref['status'].cpu().numpy()).all()
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), ref['dwell'].cpu().numpy(), rtol=1e-12)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), ref['trans'].cpu().numpy(), rtol=1e-12)
    np.testing.assert_allclose(float(r['loglik_sum']), float(ref['loglik'].sum()), rtol=1e-12)

    S, codes, leaves = cfg['S'], cfg['codes'], cfg['leaves']
    assert (codes == MISSING).any()
    allowed = (codes[:, None, :] == np.arange(S)[None, :, None]) | (codes == MISSING)[:, None, :]
    mask = np.full((sched.n, codes.shape[1]), (1 << S) - 1, dtype=np.uint64)
    mask[leaves] = (allowed.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, :, None]).sum(axis=1)
    for obs in (obs, rt.Observations.from_leaf_codes4(sched, codes, leaves),
                rt.Observations.from_masks(sched, mask),
                rt.Observations.from_dense(sched, allowed.astype(np.float64), leaves)):
        ref = mjp.expected_history_statistics(obs)
        ref = {k: ref[k].clone() for k in keys}
        for k in (3, 8):
            r = mjp.expected_history_statistics(obs, overlap_chunks=k)
            assert torch.equal(r['loglik'], ref['loglik']) and torch.equal(r['status'], ref['status'])
            for key in ('dwell', 'trans', 'root_post_sum'):
                np.testing.assert_allclose(r[key].cpu().numpy(), ref[key].cpu().numpy(), rtol=1e-12)
            np.testing.assert_allclose(float(r['loglik_sum']), float(ref['loglik'].sum()), rtol=1e-12)


@pytest.mark.parametrize('S,n_leaves,n_sites', [(4, 9, 70), (6, 6, 33), (20, 5, 37), (61, 6, 150)])
def test_branch_expectations_per_site(S, n_leaves, n_sites):
    """rt_posterior_branch_stats: expected number of E-type transitions per site and branch vs
    the oracle evaluated one site at a time (examples/code2x3/extras.py:19-132), relative 1e-9."""
    from raoteh_b200 import synth, engine
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(40 + S)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.2, rng)
    if S == 61:
        Q, pi, _ = synth.mg94()
    else:
        Q = rng.exponential(1.0, size=(S, S))
        np.fill_diagonal(Q, 0)
        Q -= np.diag(Q.sum(axis=1))
        Q /= np.abs(np.diag(Q)).mean()
        pi = rng.dirichlet(np.ones(S) * 3)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.05)
    E = (rng.random((S, S)) < 0.5).astype(float)
    np.fill_diagonal(E, 0.0)        # a transition-type mask: pairs of distinct states
    sched = TreeSchedule(parent, length)
    mjp = engine.TreeMJP(sched, Q, root_distn=pi)
    obs = engine.Observations.from_leaf_codes(sched, codes, leaves)
    got = mjp.branch_expectations(obs, E)['branch'].cpu().numpy()
    P = np_oracle.expm_edges(Q, length)
    oobs = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    n_check = min(n_sites, 12 if S > 8 else n_sites)
    for i in list(range(n_check - 1)) + [n_sites - 1]:
        r = np_oracle._ehs_chunk(parent, length, Q, P, oobs, pi, None, i, i + 1)
        want = np_oracle.edge_expected_ntransitions(Q, r['M_edges'], E)
        np.testing.assert_allclose(got[:, i], want, rtol=1e-9, atol=1e-13)
    # summed over sites and branches with E = all pairs it is the total expected transition count
    tot = mjp.branch_expectations(obs)['branch'].sum()
    ehs = mjp.expected_history_statistics(obs)
    np.testing.assert_allclose(float(tot), float(ehs['trans'].sum()), rtol=1e-9)


def _tree(kind):
    if kind == 'star':         # one polytomy: root with 7 leaves
        return np.array([-1, 0, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    if kind == 'path':         # a chain of degree-2 nodes ending in one leaf
        return np.array([-1, 0, 1, 2, 3, 4], dtype=np.int32)
    if kind == 'edge':         # a single branch
        return np.array([-1, 0], dtype=np.int32)
    if kind == 'mixed':        # polytomy + degree-2 nodes + zero-length branch
        return np.array([-1, 0, 1, 1, 1, 0, 5, 6, 6, 0], dtype=np.int32)
    raise ValueError(kind)


@pytest.mark.parametrize('kind', ['star', 'path', 'edge', 'mixed'])
@pytest.mark.parametrize('S', [2, 4, 7, 13, 64])
def test_unusual_trees_and_extreme_state_counts(kind, S):
    """Edge cases the reference's tests cover with hand-made trees (tests/test_mc.py:244-467,
    test_mjp.py:52-89): polytomies, chains of degree-2 nodes, a single branch, a zero-length
    branch, observed internal nodes, all-missing sites, 1 site, S = 2 and S = 64.
    Log-likelihood and expectations vs the oracle, relative 1e-10."""
    from raoteh_b200 import engine
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(S * 7 + len(kind))
    parent = _tree(kind)
    n = len(parent)
    length = rng.uniform(0.05, 0.6, size=n)
    length[0] = 0.0
    if kind == 'mixed':
        length[3] = 0.0
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    Q /= np.abs(np.diag(Q)).mean()
    pi = rng.dirichlet(np.ones(S) * 2)
    for n_sites in (1, 37):
        full = np.uint64((1 << S) - 1) if S < 64 else np.uint64(0xFFFFFFFFFFFFFFFF)
        mask = np.full((n, n_sites), full, dtype=np.uint64)
        # a true history per site keeps every site feasible (also across the zero-length branch)
        Pt = np_oracle.expm_edges(Q, length)
        truth = np.zeros((n, n_sites), dtype=int)
        truth[0] = rng.choice(S, size=n_sites, p=pi)
        for v in range(1, n):
            for i in range(n_sites):
                p = np.maximum(Pt[v][truth[parent[v], i]], 0)
                truth[v, i] = rng.choice(S, p=p / p.sum())
        for v in range(n):
            for i in range(n_sites):
                r = rng.random()
                if r < 0.5:                                  # a hard observation, also at internal nodes
                    mask[v, i] = np.uint64(1) << np.uint64(truth[v, i])
                elif r < 0.7:                                # a set of allowed states
                    m = 1 << int(truth[v, i])
                    for s in rng.choice(S, size=min(S, 3), replace=False):
                        m |= 1 << int(s)
                    mask[v, i] = np.uint64(m)
        mask[:, 0] = full                                    # site 0: nothing observed anywhere
        sched = TreeSchedule(parent, length)
        mjp = engine.TreeMJP(sched, Q, root_distn=pi)
        obs = engine.Observations.from_masks(sched, mask)
        r = mjp.expected_history_statistics(obs)
        P = np_oracle.expm_edges(Q, length)
        o = np_oracle.expected_history_statistics(parent, length, Q, P, np_oracle.Obs('mask', S, n_sites, mask=mask), pi)
        ll = r['loglik'].cpu().numpy()
        np.testing.assert_allclose(ll, o['loglik'], rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(ll[0], 0.0, atol=1e-12)   # no data: likelihood 1
        np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(float(r['dwell'].sum()), length.sum() * n_sites, rtol=1e-10)


@pytest.mark.parametrize('S,n_sites', [(4, 3001), (8, 515), (2, 64)])
def test_packed_codes4_are_bit_identical_to_uint8_codes(S, n_sites):
    """RT_OBS_CODES4 (two leaf codes per byte) is only another encoding of the same observations:
    log-likelihoods, statuses and statistics must be bit-identical, also through the pipelined
    host-buffer entry point (odd site counts, missing cells)."""
    import torch
    from raoteh_b200 import synth, engine
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng(S + n_sites)
    parent, length, leaves = synth.random_binary_tree(12, 0.15, rng)
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    pi = rng.dirichlet(np.ones(S) * 3)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.07)
    sched = TreeSchedule(parent, length)
    mjp = engine.TreeMJP(sched, Q, root_distn=pi)
    a = mjp.expected_history_statistics(engine.Observations.from_leaf_codes(sched, codes, leaves))
    a = dict((k, a[k].clone()) for k in ('loglik', 'status', 'dwell', 'trans', 'root_post_sum'))
    b = mjp.expected_history_statistics(engine.Observations.from_leaf_codes4(sched, codes, leaves))
    assert torch.equal(a['loglik'], b['loglik']) and torch.equal(a['status'], b['status'])
    for k in ('dwell', 'trans', 'root_post_sum'):
        np.testing.assert_allclose(b[k].cpu().numpy(), a[k].cpu().numpy(), rtol=1e-13)
    packed = torch.from_numpy(engine.pack_codes4(codes)).pin_memory()
    out_ll = torch.empty(n_sites, dtype=torch.float64).pin_memory()
    out_st = torch.empty(n_sites, dtype=torch.int8).pin_memory()
    r = mjp.expected_history_statistics_from_host(packed, leaves, out_ll, out_st, n_chunks=3, packed=True)
    torch.cuda.synchronize()
    assert torch.equal(out_ll, a['loglik'].cpu()) and torch.equal(out_st, a['status'].cpu())
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), a['dwell'].cpu().numpy(), rtol=1e-12)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), a['trans'].cpu().numpy(), rtol=1e-12)


@pytest.mark.parametrize('S,n_leaves,n_sites,kind', [(4, 32, 3001, 'codes'), (4, 32, 777, 'codes4'), (3, 9, 515, 'codes'),
                                                     (2, 6, 300, 'mask'), (4, 11, 1300, 'mask'), (4, 7, 600, 'dense')])
def test_small_state_expectations_match_oracle(rt, S, n_leaves, n_sites, kind):
    """The S <= 4 expectation pass (rt_prune_loglik, then rt_posterior_stats: root combine, down
    walk and W accumulation) against the oracle, for every observation encoding, ragged site counts,
    missing cells and a reducible rate matrix with infeasible sites (_mjp_dense.py:410-539)."""
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(900 + S + n_leaves)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    if S == 4:
        Q, pi = synth.hky85()
    else:
        Q = rng.exponential(1.0, size=(S, S))
        np.fill_diagonal(Q, 0)
        if S == 3:
            Q[2, :] = 0.0                 # absorbing state: structural zeros in P, infeasible sites
        Q -= np.diag(Q.sum(axis=1))
        pi = rng.dirichlet(np.ones(S))
    n = len(parent)
    sched = TreeSchedule(parent, length)
    P = np_oracle.expm_edges(Q, length)
    if kind in ('codes', 'codes4'):
        codes = synth.simulate_leaf_codes(parent, length, leaves, Q if S != 3 else Q + 0.3 * (1 - np.eye(3)) - 0.6 * np.eye(3),
                                          pi, n_sites, rng, 0.05)
        obs = (rt.Observations.from_leaf_codes4 if kind == 'codes4' else rt.Observations.from_leaf_codes)(
            sched, codes, leaves)
        oobs = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    elif kind == 'mask':
        bits = rng.random((n, n_sites, S)) < 0.5
        bits[np.arange(n)[:, None], np.arange(n_sites)[None, :], rng.integers(0, S, size=(n, n_sites))] = True
        unrestricted = rng.random((n, n_sites)) < 0.6
        unrestricted[leaves] = rng.random((len(leaves), n_sites)) < 0.1
        bits[unrestricted] = True
        mask = (bits.astype(np.uint64) << np.arange(S, dtype=np.uint64)[None, None, :]).sum(axis=2).astype(np.uint64)
        obs = rt.Observations.from_masks(sched, mask)
        oobs = np_oracle.Obs('mask', S, n_sites, mask=mask)
    else:
        nodes = np.concatenate([leaves, sched.internal[1:3]])
        lik = rng.random((len(nodes), S, n_sites)) ** 3
        obs = rt.Observations.from_dense(sched, lik, nodes)
        full = np.ones((n, n_sites, S))
        has = np.zeros(n, dtype=bool)
        has[nodes] = True
        full[nodes] = lik.transpose(0, 2, 1)
        oobs = np_oracle.Obs('dense', S, n_sites, lik=full, has=has)
    o = np_oracle.expected_history_statistics(parent, length, Q, P, oobs, pi)
    r = rt.TreeMJP(sched, Q, root_distn=pi).expected_history_statistics(obs)
    ok = np.isfinite(o['loglik'])
    assert ((r['status'].cpu().numpy() == 0) == ok).all()
    # atol: an unrestricted site has likelihood 1, log-lik 0 up to one rounding
    np.testing.assert_allclose(r['loglik'].cpu().numpy()[ok], o['loglik'][ok], rtol=RTOL, atol=1e-13)
    np.testing.assert_allclose(float(r['loglik_sum']), o['loglik'][ok].sum(), rtol=1e-10)
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(r['root_post_sum'].cpu().numpy(), o['root_post'].sum(axis=0), rtol=RTOL)


@pytest.mark.parametrize('shape', ['star', 'caterpillar', 'many_tiles', 'polytomy'])
def test_dmma_pruning_walk_edge_cases(rt, shape):
    """The persistent per-warp walk of the DMMA pruning kernel: a star tree (no contraction at all:
    the TMA ring is never armed), a caterpillar (every internal node has one internal and one leaf
    child: the longest chain of fresh hand-offs), more tiles than SMs (every CTA loops over tiles and
    the ring runs on across tile boundaries; ragged last tile), and polytomies with observed internal
    nodes -- log-lik, stored partials' consistency (through the expectations) and expectations
    against the oracle."""
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    rng = np.random.default_rng({'star': 1, 'caterpillar': 2, 'many_tiles': 3, 'polytomy': 4}[shape])
    S = {'star': 20, 'caterpillar': 61, 'many_tiles': 11, 'polytomy': 33}[shape]
    if shape == 'star':
        parent = np.array([-1] + [0] * 9, dtype=np.int32)
        n_sites = 300
    elif shape == 'caterpillar':
        # spine 0-2-4-6-8-10, a leaf hanging off every spine node, two leaves at the end
        parent = np.array([-1, 0, 0, 2, 2, 4, 4, 6, 6, 8, 8, 10, 10], dtype=np.int32)
        n_sites = 700
    elif shape == 'many_tiles':
        parent, _, _ = synth.random_binary_tree(6, 0.1, rng)
        n_sites = 148 * 128 * 2 + 77
    else:
        parent = np.array([-1, 0, 0, 0, 0, 4, 4, 4, 4, 8, 8, 8], dtype=np.int32)
        n_sites = 515
    n = len(parent)
    length = rng.exponential(0.15, size=n)
    length[0] = 0.0
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    Q /= np.abs(np.diag(Q)).mean()
    pi = rng.dirichlet(np.ones(S))
    sched = TreeSchedule(parent, length)
    leaves = sched.leaves
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, n_sites, rng, 0.05)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    P = np_oracle.expm_edges(Q, length)
    if shape == 'polytomy':
        # observations as masks at every node (an observed internal node: OP_APPLY_OBS)
        full = (1 << S) - 1
        mask = np.full((n, n_sites), full, dtype=np.uint64)
        for i, v in enumerate(leaves):
            c = codes[i].astype(np.uint64)
            mask[v] = np.where(codes[i] == 255, np.uint64(full), np.uint64(1) << c)
        mask[4] = np.where(rng.random(n_sites) < 0.5, np.uint64(full), np.uint64(full) ^ np.uint64(5))
        obs = rt.Observations.from_masks(sched, mask)
        oobs = np_oracle.Obs('mask', S, n_sites, mask=mask)
    else:
        obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
        oobs = np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes)
    r = mjp.log_likelihood(obs)
    ll, st = np_oracle.log_likelihood(parent, P, oobs, pi)
    assert (r['status'].cpu().numpy() == st).all()
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), ll, rtol=RTOL)
    if n_sites <= 1000:
        e = mjp.expected_history_statistics(obs)
        o = np_oracle.expected_history_statistics(parent, length, Q, P, oobs, pi)
        np.testing.assert_allclose(e['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
        np.testing.assert_allclose(e['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)


@pytest.mark.parametrize('S,n_leaves,n_sites', [(12, 5, 3000), (61, 6, 2304)])      # 2304 % 16 == 0: the leaf scatter's vector path, which does not read the status row
def test_large_state_expectations_skip_infeasible_sites(rt, S, n_leaves, n_sites):
    """A reducible rate matrix (two closed classes) and uniformly random leaf codes: most sites have
    probability zero (StructuralZeroProb in the reference, _mjp_dense.py:186-190) and must contribute
    nothing to the expectations -- in the DMMA kernel their rows are zero, in down_leaf_scatter_kernel
    they go to the pad column of the W tile.  Feasible sites against the oracle."""
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200 import synth
    rng = np.random.default_rng(4242 + S)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.3, rng)
    h = S // 2
    Q = np.zeros((S, S))
    Q[:h, :h] = rng.exponential(1.0, size=(h, h))
    Q[h:, h:] = rng.exponential(1.0, size=(S - h, S - h))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    pi = rng.dirichlet(np.ones(S))
    # leaves drawn from one class with probability 0.8 per site, anywhere otherwise
    cls = rng.integers(0, 2, size=n_sites)
    codes = np.where(cls[None, :] == 0, rng.integers(0, h, size=(len(leaves), n_sites)),
                     rng.integers(h, S, size=(len(leaves), n_sites)))
    stray = rng.random((len(leaves), n_sites)) < 0.08
    codes = np.where(stray, rng.integers(0, S, size=codes.shape), codes).astype(np.uint8)
    codes[rng.random(codes.shape) < 0.05] = 255          # some unobserved cells as well
    sched = TreeSchedule(parent, length)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    r = mjp.expected_history_statistics(obs)
    P = np_oracle.expm_edges(Q, length)
    o = np_oracle.expected_history_statistics(
        parent, length, Q, P, np_oracle.Obs('codes', S, n_sites, leaf_nodes=leaves, codes=codes), pi)
    ok = np.isfinite(o['loglik'])
    assert 0.2 * n_sites < ok.sum() < 0.95 * n_sites
    np.testing.assert_array_equal(r['status'].cpu().numpy() == 0, ok)
    np.testing.assert_allclose(r['loglik'].cpu().numpy()[ok], o['loglik'][ok], rtol=RTOL)
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(float(r['dwell'].sum()), length.sum() * ok.sum(), rtol=1e-10)
