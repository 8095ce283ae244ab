"""Per-site weights of the down pass (TreeMJP(..., site_weight=)) and site-class mixtures
(raoteh_b200.mixture.SiteMixtureMJP) on the GPU: weights against duplicated columns on every
down-pass path (S <= 8 walk, level-synchronous kernels, S > 8 DMMA) and encoding, mixtures against
the per-class reference combined site by site (mixture_oracle)."""
import numpy as np
import pytest

from oracle import np_oracle
import mixture_oracle
from test_gpu_range import walk_smem
from raoteh_b200 import synth
from raoteh_b200.lowering import TreeSchedule, MISSING

pytestmark = pytest.mark.gpu

RTOL = 1e-10        # log-likelihoods, class posteriors, summed statistics
RTOL_E = 1e-9       # node marginals, branch expectations


@pytest.fixture(scope='module')
def rt():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    import raoteh_b200.engine as engine
    return engine


def _np(x):
    return x.cpu().numpy() if hasattr(x, 'cpu') else np.asarray(x)


def _random_Q(S, rng):
    Q = rng.exponential(1.0, size=(S, S))
    np.fill_diagonal(Q, 0)
    Q -= np.diag(Q.sum(axis=1))
    Q /= np.abs(np.diag(Q)).mean()
    return Q


class Data(object):
    """Host observations of N sites in every encoding; `engine(kind, cols)` / `oracle(kind, cols)`
    give the observations of the columns `cols` (repeats allowed)."""

    def __init__(self, sched, S, leaves, codes, rng):
        self.sched, self.S, self.leaves, self.codes = sched, S, leaves, codes
        n, N = sched.n, codes.shape[1]
        full = np.uint64((1 << S) - 1)
        self.mask = np.full((n, N), full, dtype=np.uint64)
        c = codes.astype(np.uint64)
        amb = np.uint64(1) << ((c + np.uint64(1)) % np.uint64(S))     # a second allowed state
        one = np.uint64(1) << np.where(codes == MISSING, 0, c)
        self.mask[leaves] = np.where(codes == MISSING, full,
                                     np.where(rng.random(codes.shape) < 0.2, one | amb, one))
        self.nodes = np.concatenate([leaves, sched.internal[1:2]])
        lik = 0.05 + rng.random((len(self.nodes), S, N)) ** 2
        hard = np.where(codes == MISSING, 0, codes)
        lik[:len(leaves)] += 2.0 * (np.arange(S)[None, :, None] == hard[:, None, :])
        self.lik = lik

    def engine(self, rt, kind, cols):
        if kind in ('codes', 'codes4'):
            make = rt.Observations.from_leaf_codes if kind == 'codes' else rt.Observations.from_leaf_codes4
            return make(self.sched, np.ascontiguousarray(self.codes[:, cols]), self.leaves)
        if kind == 'mask':
            return rt.Observations.from_masks(self.sched, np.ascontiguousarray(self.mask[:, cols]))
        return rt.Observations.from_dense(self.sched, self.lik[:, :, cols], self.nodes)

    def oracle(self, kind, cols):
        S, N = self.S, len(cols)
        if kind in ('codes', 'codes4'):
            return np_oracle.Obs('codes', S, N, leaf_nodes=self.leaves, codes=self.codes[:, cols])
        if kind == 'mask':
            return np_oracle.Obs('mask', S, N, mask=self.mask[:, cols])
        lik_all = np.zeros((self.sched.n, N, S))
        lik_all[self.nodes] = self.lik[:, :, cols].transpose(0, 2, 1)
        has = np.zeros(self.sched.n, dtype=bool)
        has[self.nodes] = True
        return np_oracle.Obs('dense', S, N, lik=lik_all, has=has)


def _rel(got, ref, tol, what):
    got, ref = _np(got), np.asarray(ref)
    assert np.isfinite(got).all(), what
    scale = max(np.abs(ref).max(), 1e-300)
    np.testing.assert_allclose(got / scale, ref / scale, rtol=0, atol=tol, err_msg=what)


# ---- 1. site weights on TreeMJP --------------------------------------------------------------

WEIGHT_CASES = [(4, 20, 'walk'), (8, 40, 'levels'), (20, 12, 'dmma')]


@pytest.mark.parametrize('kind', ['codes', 'codes4', 'mask', 'dense'])
@pytest.mark.parametrize('S,n_leaves,path', WEIGHT_CASES)
def test_site_weights_equal_duplicated_columns(rt, S, n_leaves, path, kind):
    import torch
    if kind == 'codes4' and S > 8:
        pytest.skip('4-bit codes hold S <= 8')
    rng = np.random.default_rng(100 * S + n_leaves)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.15, rng)
    Q = synth.hky85()[0] if S == 4 else _random_Q(S, rng)
    pi = rng.dirichlet(np.ones(S) * 3)
    N0 = 401
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, N0, rng, 0.05)
    sched = TreeSchedule(parent, length)
    data = Data(sched, S, leaves, codes, rng)
    cols = np.arange(N0)
    obs = data.engine(rt, kind, cols)
    if S <= 8:
        assert (walk_smem(sched, S, obs.obs_slot) <= 100 * 1024) == (path == 'walk')
    w = rng.integers(0, 4, size=N0)
    dup = data.engine(rt, kind, np.repeat(cols, w))
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    ref = {k: _np(v).copy() for k, v in mjp.expected_history_statistics(dup).items()
           if k in ('W', 'dwell', 'trans', 'root_post_sum', 'loglik_sum')}
    wt = torch.from_numpy(w.astype(np.float64)).cuda()
    chunks = (0, 3) if S <= 8 else (0,)
    for oc in chunks:
        got = mjp.expected_history_statistics(obs, site_weight=wt, overlap_chunks=oc)
        for k in ('W', 'dwell', 'trans', 'root_post_sum'):
            _rel(got[k], ref[k], 1e-12, '%s overlap_chunks=%d' % (k, oc))
        np.testing.assert_allclose(float(got['loglik_sum']), float(ref['loglik_sum']), rtol=1e-12)
    # all-ones weights: the unweighted result
    plain = {k: _np(v).copy() for k, v in mjp.expected_history_statistics(obs).items()
             if k in ('W', 'dwell', 'trans', 'root_post_sum', 'loglik_sum', 'loglik')}
    ones = mjp.expected_history_statistics(obs, site_weight=torch.ones(N0, dtype=torch.float64,
                                                                      device='cuda'))
    for k in ('W', 'dwell', 'trans', 'root_post_sum'):
        _rel(ones[k], plain[k], 1e-14, k)
    np.testing.assert_allclose(float(ones['loglik_sum']), float(plain['loglik_sum']), rtol=1e-14)
    assert (_np(ones['loglik']) == plain['loglik']).all()
    # node marginals carry the weight
    nd_plain = _np(mjp.posterior(obs, want_node_distn=True)['node_distn'])[:, :, :N0].copy()
    nd = _np(mjp.posterior(obs, want_node_distn=True, site_weight=wt)['node_distn'])[:, :, :N0]
    _rel(nd, nd_plain * w[None, None, :], 1e-14, 'node_distn')


def test_site_weight_argument_checks(rt):
    import torch
    rng = np.random.default_rng(3)
    parent, length, leaves = synth.random_binary_tree(5, 0.1, rng)
    Q, pi = synth.hky85()
    sched = TreeSchedule(parent, length)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, 10, rng)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    for bad in (torch.ones(10, dtype=torch.float32, device='cuda'), torch.ones(10, dtype=torch.float64),
                torch.ones(11, dtype=torch.float64, device='cuda'),
                torch.ones(20, dtype=torch.float64, device='cuda')[::2]):
        with pytest.raises(ValueError):
            mjp.posterior(obs, site_weight=bad)
    with pytest.raises(TypeError):
        mjp.posterior(obs, site_weight=np.ones(10))


def test_site_weights_over_several_workspace_chunks(rt):
    """70001 sites (7 copies of 10001) with random weights on the level-synchronous path, whose root
    kernel takes the sites in workspace chunks of 65536: a weight offset that is off by any amount
    pairs a site with another site's weight."""
    import torch
    S, n_leaves, base, reps = 8, 32, 10001, 7
    rng = np.random.default_rng(8033)
    parent, length, leaves = synth.random_binary_tree(n_leaves, 0.1, rng)
    Q, pi = _random_Q(S, rng), rng.dirichlet(np.ones(S) * 2)
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, base, rng, 0.05)
    sched = TreeSchedule(parent, length)
    obs1 = rt.Observations.from_leaf_codes(sched, codes, leaves)
    assert walk_smem(sched, S, obs1.obs_slot) > 100 * 1024
    obs = rt.Observations.from_leaf_codes(sched, np.tile(codes, reps), leaves)
    w = torch.from_numpy(rng.random(base * reps)).cuda()
    mjp = rt.TreeMJP(sched, Q, root_distn=pi)
    keys = ('W', 'dwell', 'trans', 'root_post_sum', 'loglik_sum')
    ref = {k: 0.0 for k in keys}
    for r in range(reps):
        one = mjp.expected_history_statistics(obs1, site_weight=w[r * base:(r + 1) * base].contiguous())
        for k in keys:
            ref[k] = ref[k] + _np(one[k]).copy()
    got = mjp.expected_history_statistics(obs, site_weight=w)
    for k in keys:
        _rel(got[k], ref[k], 1e-12, k)


# ---- 2. mixtures against the reference -----------------------------------------------------

def _simulate(parent, length, leaves, Qs, rates, weights, pi, N, rng):
    """Leaf codes of N sites, each from a class drawn with `weights`, 5 % missing cells."""
    cls = rng.choice(len(rates), size=N, p=weights)
    codes = np.empty((len(leaves), N), dtype=np.uint8)
    for k in range(len(rates)):
        idx = np.flatnonzero(cls == k)
        if len(idx):
            codes[:, idx] = synth.simulate_leaf_codes(parent, rates[k] * length, leaves, Qs[k], pi,
                                                      len(idx), rng, 0.05)
    return codes


def _mixture_case(name, rng):
    from raoteh_b200.mixture import discrete_gamma_rates
    if name == 'hky_g4_i':
        parent, length, leaves = synth.random_binary_tree(20, 0.1, rng)
        Q, pi = synth.hky85()
        rates = np.concatenate([[0.0], discrete_gamma_rates(0.5, 4)])
        weights = np.array([0.2, 0.2, 0.2, 0.2, 0.2])
        return parent, length, leaves, [Q] * 5, rates, weights, pi, 400
    if name == 's8_levels':
        parent, length, leaves = synth.random_binary_tree(40, 0.1, rng)
        Qs = [_random_Q(8, rng) for _ in range(2)]
        return parent, length, leaves, Qs, np.array([0.4, 1.6]), np.array([0.6, 0.4]), \
            rng.dirichlet(np.ones(8) * 3), 300
    if name == 's20_three':
        parent, length, leaves = synth.random_binary_tree(8, 0.15, rng)
        Qs = [_random_Q(20, rng) for _ in range(3)]
        return parent, length, leaves, Qs, np.array([0.5, 1.0, 2.0]), np.array([0.5, 0.3, 0.2]), \
            rng.dirichlet(np.ones(20) * 3), 300
    assert name == 'mg94_three'
    parent, length, leaves = synth.random_binary_tree(6, 0.2, rng)
    Qs, pis = zip(*[synth.mg94(omega=om)[:2] for om in (0.1, 1.0, 2.5)])
    return parent, length, leaves, list(Qs), np.ones(3), np.array([0.6, 0.3, 0.1]), pis[0], 300


MIXTURE_CASES = [('hky_g4_i', 'codes'), ('hky_g4_i', 'codes4'), ('hky_g4_i', 'mask'),
                 ('hky_g4_i', 'dense'), ('s8_levels', 'codes'), ('s8_levels', 'mask'),
                 ('s20_three', 'codes'), ('s20_three', 'dense'), ('mg94_three', 'codes')]


@pytest.mark.parametrize('name,kind', MIXTURE_CASES)
def test_mixture_matches_reference(rt, name, kind):
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP
    rng = np.random.default_rng(sum(map(ord, name)))
    parent, length, leaves, Qs, rates, weights, pi, N = _mixture_case(name, rng)
    S = Qs[0].shape[0]
    codes = _simulate(parent, length, leaves, Qs, rates, weights, pi, N, rng)
    sched = TreeSchedule(parent, length)
    data = Data(sched, S, leaves, codes, rng)
    cols = np.arange(N)
    obs, oobs = data.engine(rt, kind, cols), data.oracle(kind, cols)
    if name == 's8_levels':
        assert walk_smem(sched, S, obs.obs_slot) > 100 * 1024
    sw = rng.random(N) + 0.5
    ref = mixture_oracle.mixture(parent, length, Qs, rates, weights, oobs, pi, site_weight=sw,
                                 node_distn=True)
    mix = SiteMixtureMJP(sched, np.stack(Qs), root_distn=pi, rates=rates, weights=weights)
    got = mix.expected_history_statistics(obs, want_node_distn=True,
                                          site_weight=torch.from_numpy(sw).cuda())
    st = _np(got['status'])
    assert (st == ref['status']).all()
    ok = ref['status'] == 0
    np.testing.assert_allclose(_np(got['loglik'])[ok], ref['loglik'][ok], rtol=RTOL)
    np.testing.assert_allclose(_np(got['class_post']), ref['class_post'], rtol=0, atol=RTOL)
    np.testing.assert_allclose(float(got['loglik_sum']), ref['loglik_sum'], rtol=RTOL)
    for k in ('dwell', 'trans', 'root_post_sum', 'class_post_sum', 'dwell_class', 'trans_class'):
        _rel(got[k], ref[k], RTOL, k)
    nd = _np(got['node_distn'])
    for v in sched.internal:
        np.testing.assert_allclose(nd[sched.store_index[v], :, :N].T, ref['node_distn'][v],
                                   rtol=0, atol=RTOL_E * sw.max())
    br = _np(mix.branch_expectations(obs)['branch'])
    np.testing.assert_allclose(br, ref['branch'], rtol=0,
                               atol=RTOL_E * max(1.0, np.abs(ref['branch']).max()))


# ---- 3. identities at the C2 shape ----------------------------------------------------------

def test_mixture_identities_c2_shape(rt):
    import torch
    from raoteh_b200.mixture import SiteMixtureMJP, discrete_gamma_rates
    rng = np.random.default_rng(20260201)
    parent, length, leaves = synth.random_binary_tree(32, 0.1, rng)
    Q, pi = synth.hky85()
    rates = np.concatenate([[0.0], discrete_gamma_rates(0.5, 4)])
    weights = np.array([0.1, 0.225, 0.225, 0.225, 0.225])
    N = 100_000
    codes = _simulate(parent, length, leaves, [Q] * 5, rates, weights, pi, N, rng)
    sched = TreeSchedule(parent, length)
    mix = SiteMixtureMJP(sched, Q, root_distn=pi, rates=rates, weights=weights)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    r = mix.expected_history_statistics(obs)
    n_ok = int((_np(r['status']) == 0).sum())
    assert n_ok == N
    tree_length = length[1:].sum()
    np.testing.assert_allclose(float(r['dwell'].sum()), tree_length * n_ok, rtol=1e-10)
    np.testing.assert_allclose(_np(r['class_post'].sum(dim=0)), 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(float(r['class_post_sum'].sum()), n_ok, rtol=1e-12)
    keys = ('dwell', 'trans', 'root_post_sum', 'class_post_sum', 'loglik_sum')
    whole = {k: _np(r[k]).copy() for k in keys}
    half = N // 2
    parts = [mix.expected_history_statistics(rt.Observations.from_leaf_codes(
        sched, np.ascontiguousarray(codes[:, a:b]), leaves)) for a, b in ((0, half), (half, N))]
    for k in keys:
        _rel(_np(parts[0][k]) + _np(parts[1][k]), whole[k], 1e-12, k)


# ---- 4. edge cases --------------------------------------------------------------------------

def test_invariant_class_and_infeasible_sites(rt):
    from raoteh_b200.mixture import SiteMixtureMJP
    rng = np.random.default_rng(5)
    parent, length, leaves = synth.random_binary_tree(6, 0.2, rng)
    sched = TreeSchedule(parent, length)
    Q, pi = synth.hky85()
    codes = np.zeros((len(leaves), 4), dtype=np.uint8)
    codes[:, 1] = 2                        # constant
    codes[0, 2] = 1                        # variable
    codes[:, 3] = MISSING
    codes[1, 3] = 3                        # constant with missing cells
    mix = SiteMixtureMJP(sched, Q, root_distn=pi, rates=[0.0, 1.0], weights=[0.3, 0.7])
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    r = mix.expected_history_statistics(obs)
    cp, st = _np(r['class_post']), _np(r['status'])
    assert (st == 0).all()
    assert cp[0, 2] == 0.0 and (cp[0, [0, 1, 3]] > 0).all()
    assert np.isfinite(_np(r['loglik'])).all()
    # a reducible rate matrix: {0, 1} and {2, 3} do not communicate, so a site with leaves in both
    # blocks is infeasible in every class
    Qr = np.zeros((4, 4))
    Qr[0, 1] = Qr[1, 0] = Qr[2, 3] = Qr[3, 2] = 1.0
    Qr -= np.diag(Qr.sum(axis=1))
    codes = np.zeros((len(leaves), 3), dtype=np.uint8)
    codes[0, 1] = 2
    codes[:, 2] = 1
    mix = SiteMixtureMJP(sched, Qr, root_distn=np.full(4, 0.25), rates=[0.5, 2.0])
    r = mix.expected_history_statistics(rt.Observations.from_leaf_codes(sched, codes, leaves))
    st, ll, cp = _np(r['status']), _np(r['loglik']), _np(r['class_post'])
    assert st.tolist() == [0, 1, 0]
    assert ll[1] == -np.inf and np.isfinite(ll[[0, 2]]).all()
    assert (cp[:, 1] == 0).all()
    np.testing.assert_allclose(float(r['loglik_sum']), ll[0] + ll[2], rtol=1e-14)
    np.testing.assert_allclose(float(r['class_post_sum'].sum()), 2.0, rtol=1e-14)


@pytest.mark.parametrize('S', [4, 61])
def test_one_class_is_tree_mjp(rt, S):
    from raoteh_b200.mixture import SiteMixtureMJP
    rng = np.random.default_rng(S)
    parent, length, leaves = synth.random_binary_tree(10, 0.1, rng)
    Q, pi = synth.hky85() if S == 4 else synth.mg94()[:2]
    codes = synth.simulate_leaf_codes(parent, length, leaves, Q, pi, 777, rng, 0.05)
    sched = TreeSchedule(parent, length)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    ref = {k: _np(v).copy() for k, v in rt.TreeMJP(sched, Q, root_distn=pi)
           .expected_history_statistics(obs).items()
           if k in ('loglik', 'dwell', 'trans', 'root_post_sum', 'loglik_sum')}
    got = SiteMixtureMJP(sched, Q, root_distn=pi).expected_history_statistics(obs)
    assert (_np(got['loglik']) == ref['loglik']).all()
    for k in ('dwell', 'trans', 'root_post_sum'):
        _rel(got[k], ref[k], 1e-14, k)
    np.testing.assert_allclose(float(got['loglik_sum']), float(ref['loglik_sum']), rtol=1e-14)
