"""Parity at the shapes BASELINE.json names (synth.config_c2 .. config_c5), through the C ABI:

C3  61-state codon model, 128-leaf tree: log-lik AND expected dwell / transition counts against the
    oracle on a slice of the sites (relative 1e-10), plus the size-independent identities at the
    larger batch (sum of expected dwell = tree length x sites, root posterior sums to sites).
C4  4-state HKY on the 64-leaf tree: Rao-Teh sweeps, every history checked structurally and the
    mean dwell times / transition counts against the closed-form posterior expectations (|z| < 5),
    in float32 and in fp64 event-time mode.
C5  25-taxon p53 tree, 61 codons x 20 tolerance classes: log-lik of a site slice against the
    oracle (1e-10); the blocked Gibbs sampler at the full model size, every history checked for
    compatibility (class of the primary state on throughout, disease data, leaf codons).
Sharded samplers: a REAL 2-process run (gloo on one GPU, NCCL when two GPUs are visible) of
RaoTehChains and ToleranceChains against the unsharded run.
"""
import os
import socket

import numpy as np
import pytest

from oracle import np_oracle

pytestmark = pytest.mark.gpu
RTOL = 1e-10


@pytest.fixture(scope='module')
def rt():
    import torch
    assert torch.cuda.is_available()
    from raoteh_b200 import engine
    return engine


def test_c3_shape_loglik_and_expectations_match_oracle(rt):
    """BASELINE configs[2]: the 255-node tree, DMMA up pass + down pass + Frechet contraction."""
    import torch
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    n_sites, n_slice = 2304, 320            # 18 DMMA tiles of 128 sites; the oracle takes the first 320
    cfg = synth.config_c3(n_sites=n_sites)
    assert len(cfg['parent']) == 255 and cfg['S'] == 61
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    mjp = rt.TreeMJP(sched, cfg['Q'], root_distn=cfg['pi'])
    P = np_oracle.expm_edges(cfg['Q'], cfg['length'])
    np.testing.assert_allclose(mjp.transition_matrices().cpu().numpy()[1:], P[1:], rtol=0, atol=2e-13)
    # the slice alone: site-summed expectations are comparable only on the same sites
    obs = rt.Observations.from_leaf_codes(sched, np.ascontiguousarray(cfg['codes'][:, :n_slice]), cfg['leaves'])
    r = mjp.expected_history_statistics(obs)
    o = np_oracle.expected_history_statistics(
        cfg['parent'], cfg['length'], cfg['Q'], P,
        np_oracle.Obs('codes', 61, n_slice, leaf_nodes=cfg['leaves'], codes=cfg['codes'][:, :n_slice]), cfg['pi'])
    assert (r['status'].cpu().numpy() == 0).all()
    np.testing.assert_allclose(r['loglik'].cpu().numpy(), o['loglik'], rtol=RTOL)
    np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
    np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)
    np.testing.assert_allclose(r['root_post_sum'].cpu().numpy(), o['root_post'].sum(axis=0), rtol=RTOL)
    # the larger batch: per-site log-lik of the slice unchanged, identities over all sites
    obs = rt.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    r = mjp.expected_history_statistics(obs)
    np.testing.assert_allclose(r['loglik'].cpu().numpy()[:n_slice], o['loglik'], rtol=RTOL)
    np.testing.assert_allclose(float(r['dwell'].sum()), cfg['length'].sum() * n_sites, rtol=1e-10)
    np.testing.assert_allclose(float(r['root_post_sum'].sum()), n_sites, rtol=1e-10)
    q = -np.diag(cfg['Q'])
    # expected number of transitions out of s = q_s x expected dwell in s, summed over the tree, only
    # in expectation over data -- not an identity per data set; what IS one: no negative counts and
    # zero counts exactly where the rate is zero
    tr = r['trans'].cpu().numpy()
    assert (tr >= 0).all() and (tr[cfg['Q'] == 0] == 0).all() and q.min() > 0


def test_c5_shape_loglik_matches_oracle(rt):
    """BASELINE configs[4]: 25-taxon p53 topology, primary proposal model, site slice vs oracle."""
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    n_sites = 1500
    cfg = synth.config_c5(n_sites=n_sites)
    assert len(cfg['parent']) == 49
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    for Q in (cfg['Q_proposal'], cfg['Q']):
        mjp = rt.TreeMJP(sched, Q, root_distn=cfg['pi'])
        obs = rt.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
        r = mjp.expected_history_statistics(obs)
        P = np_oracle.expm_edges(Q, cfg['length'])
        o = np_oracle.expected_history_statistics(
            cfg['parent'], cfg['length'], Q, P,
            np_oracle.Obs('codes', 61, n_sites, leaf_nodes=cfg['leaves'], codes=cfg['codes']), cfg['pi'])
        np.testing.assert_allclose(r['loglik'].cpu().numpy(), o['loglik'], rtol=RTOL)
        np.testing.assert_allclose(r['dwell'].cpu().numpy(), o['dwell'], rtol=RTOL)
        np.testing.assert_allclose(r['trans'].cpu().numpy(), o['trans'], rtol=RTOL, atol=1e-12)


def _check_history(ch, t, sched, parent, length, leaves, codes, site):
    ns, edges = ch.trajectory(t)
    assert len(edges) == sched.n - 1
    for c, (times, states) in edges.items():
        assert states[0] == ns[parent[c]] and states[-1] == ns[c]
        assert len(states) == len(times) + 1
        assert len(times) < 2 or np.all(np.diff(times) > 0)
        assert np.all(times > 0) and np.all(times < length[c])
        assert np.all(states[1:] != states[:-1])
    for i, leaf in enumerate(leaves):
        if codes[i, site] != 255:
            assert ns[leaf] == codes[i, site]


@pytest.mark.parametrize('time_dtype', ['float32', 'float64'])
def test_c4_shape_sweeps_match_closed_form(rt, time_dtype):
    """BASELINE configs[3]: the 127-node tree.  Mean dwell times / transition counts of the sampled
    histories against _mjp.get_expected_history_statistics (closed form, oracle), |z| < 5 with the
    standard error from 16 independent groups of chains; both event-time precisions.
    Burn-in: on this tree the sampler needs several hundred sweeps to forget the initial history
    (one event in the middle of every branch) -- at 60 sweeps of burn-in a transition count sits
    5-10 standard errors off (relative 1e-3 .. 2e-2), at 1000 every statistic is inside 3.5
    (tools/diag_c4_bias.py, run on the B200; float32 and fp64 times give the same z-scores)."""
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    n_sites = 3
    cfg = synth.config_c4(n_sites=n_sites)
    assert len(cfg['parent']) == 127
    parent, length, leaves, Q, pi, codes = (cfg[k] for k in ('parent', 'length', 'leaves', 'Q', 'pi', 'codes'))
    sched = TreeSchedule(parent, length)
    obs = rt.Observations.from_leaf_codes(sched, codes, leaves)
    P = np_oracle.expm_edges(Q, length)
    o = np_oracle.expected_history_statistics(
        parent, length, Q, P, np_oracle.Obs('codes', 4, n_sites, leaf_nodes=leaves, codes=codes), pi)
    groups, n_chains, burn, n_sweeps = 16, 512, 1000, 200
    dwell = np.zeros((groups, 4))
    trans = np.zeros((groups, 4, 4))
    for g in range(groups):
        ch = RaoTehChains(sched, Q, obs, n_chains=n_chains, root_distn=pi, seed=5000 + g, cap=112,
                          time_dtype=time_dtype)
        ch.sweep(burn, stats=False)
        ch.sweep(n_sweeps)
        ch.check()
        assert bool((ch.sweep_count == 1 + burn + n_sweeps).all())
        dwell[g] = ch.dwell_sum.cpu().numpy() / (n_chains * n_sweeps)
        trans[g] = ch.trans_sum.cpu().numpy() / (n_chains * n_sweeps)
        if g == 0:
            for t in range(0, ch.n_traj, 97):
                _check_history(ch, t, sched, parent, length, leaves, codes, t % n_sites)
    # total dwell per sweep is the tree length: to float32 rounding, or to fp64 rounding
    np.testing.assert_allclose(dwell.sum(axis=1), length.sum() * n_sites,
                               rtol=1e-5 if time_dtype == 'float32' else 1e-12)
    for got, want in ((dwell, o['dwell']), (trans.reshape(groups, -1), o['trans'].reshape(-1))):
        mean = got.mean(axis=0)
        se = got.std(axis=0, ddof=1) / np.sqrt(groups)
        for m, s, w in zip(mean, se, want):
            if w == 0:
                assert m == 0
            else:
                assert abs(m - w) < 5 * s + 1e-9, (m, w, s)


def test_float32_and_float64_event_times_agree():
    """The two event-time precisions consume the same Philox words in the same order, so for the
    same seed they sample the SAME discrete history (root state, jump counts, states) except where a
    float32 rounding flips a comparison; their dwell-time totals then agree to float32 resolution.
    This bounds what the 4-byte times can move: no statistic beyond ~1e-6 relative per history."""
    import torch
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    cfg = synth.config_c4(n_sites=50)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    out = {}
    for td in ('float32', 'float64'):
        ch = RaoTehChains(sched, cfg['Q'], obs, n_chains=40, root_distn=cfg['pi'], seed=77, cap=112,
                          time_dtype=td)
        ch.sweep(1)          # one sweep from the (identical, deterministic) initial history
        out[td] = (ch.node_state.clone(), ch.ev_total.clone(), ch.dwell_sum.clone(), ch.trans_sum.clone())
    same = (out['float32'][0] == out['float64'][0]).all(dim=0) & (out['float32'][1] == out['float64'][1])
    assert float(same.double().mean()) > 0.999          # a rounding flip is a ~1e-6 event per comparison
    if bool(same.all()):
        np.testing.assert_allclose(out['float32'][2].cpu().numpy(), out['float64'][2].cpu().numpy(), rtol=2e-6)
        assert torch.equal(out['float32'][3], out['float64'][3])


def test_c5_shape_gibbs_histories_are_compatible(rt):
    """BASELINE configs[4] at the full model size (61 codons x 20 classes, 49 nodes): after blocked
    Gibbs sweeps every compound history has the class of the primary state ON throughout, respects
    the disease data at the first leaf and the observed leaf codons."""
    import torch
    from raoteh_b200 import synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.tmjp import ToleranceChains
    n_sites = 64
    cfg = synth.config_c5(n_sites=n_sites)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = rt.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    ch = ToleranceChains(sched, cfg['Q'], cfg['pi'], dict(enumerate(cfg['part'])), cfg['rate_on'],
                         cfg['rate_off'], obs, n_chains=2, tol_obs=cfg['tol_obs'],
                         tol_obs_nodes=cfg['tol_obs_nodes'], cap_p=96, cap_t=48, seed=3)
    ch.sweep(6)
    ch.check()
    part = np.asarray(cfg['part'])
    p_node = ch.p_node.cpu().numpy()
    t_node = ch.t_node.cpu().numpy()
    leaf0 = int(cfg['tol_obs_nodes'][0])
    for t in range(ch.n_traj):
        site = t % n_sites
        for i, leaf in enumerate(cfg['leaves']):
            assert p_node[t, leaf] == cfg['codes'][i, site]
        # the class of the primary state is on at every node
        for v in range(sched.n):
            assert (int(t_node[t, v]) >> int(part[p_node[t, v]])) & 1
        # disease data: bit0 = off allowed, bit1 = on allowed
        for c in range(cfg['n_parts']):
            on = (int(t_node[t, leaf0]) >> c) & 1
            assert (int(cfg['tol_obs'][0, c, site]) >> on) & 1
    # the statistics of the sampled primary histories: total dwell = tree length per history
    np.testing.assert_allclose(float(ch.prim_dwell.sum()), cfg['length'].sum() * ch.n_traj * 6, rtol=1e-5)


# ---------------------------------------------------------------------------------------
# sharded samplers, two real processes
# ---------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _shard_worker(rank, world_size, port, backend, q):
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dev = torch.device('cuda', rank if backend == 'nccl' else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world_size)
    from raoteh_b200 import dist as rdist
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    from raoteh_b200.tmjp import ToleranceChains
    res = {}
    # Rao-Teh chains on the C4 tree
    cfg = synth.config_c4(n_sites=37)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'], device=dev)
    traj0, n_traj = rdist.shard_trajectories(5, 37)
    ch = RaoTehChains(sched, cfg['Q'], obs, n_chains=5, root_distn=cfg['pi'], seed=11, cap=112,
                      device=dev, traj0=traj0, n_traj=n_traj)
    ch.sweep(4, stats=False)
    ch.sweep(6)
    red = rdist.allreduce_sampler_stats(ch)
    res['raoteh'] = (traj0, n_traj, red['dwell'].cpu().numpy(), red['trans'].cpu().numpy(),
                     ch.node_state.cpu().numpy(), ch.ev_total.cpu().numpy())
    # tolerance chains on the C5 model
    cfg = synth.config_c5(n_sites=21)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'], device=dev)
    traj0, n_traj = rdist.shard_trajectories(3, 21)
    tc = ToleranceChains(sched, cfg['Q'], cfg['pi'], dict(enumerate(cfg['part'])), cfg['rate_on'],
                         cfg['rate_off'], obs, n_chains=3, tol_obs=cfg['tol_obs'],
                         tol_obs_nodes=cfg['tol_obs_nodes'], cap_p=96, cap_t=48, seed=13, device=dev,
                         traj0=traj0, n_traj=n_traj)
    tc.sweep(3)
    red = rdist.allreduce_sampler_stats(tc)
    res['tmjp'] = (traj0, n_traj, red['dwell'].cpu().numpy(), red['trans'].cpu().numpy(),
                   red['tol_stats'].cpu().numpy(), tc.p_node.cpu().numpy(), tc.t_node.cpu().numpy())
    q.put((rank, res))
    dist.destroy_process_group()


def _run_sharded(backend):
    import torch
    import torch.multiprocessing as mp
    from raoteh_b200 import engine, synth
    from raoteh_b200.lowering import TreeSchedule
    from raoteh_b200.raoteh import RaoTehChains
    from raoteh_b200.tmjp import ToleranceChains
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, backend, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    # the unsharded runs
    cfg = synth.config_c4(n_sites=37)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    ch = RaoTehChains(sched, cfg['Q'], obs, n_chains=5, root_distn=cfg['pi'], seed=11, cap=112)
    ch.sweep(4, stats=False)
    ch.sweep(6)
    a, b = res[0]['raoteh'], res[1]['raoteh']
    assert (a[0], a[1], b[0], b[1]) == (0, 93, 93, 92)
    for r in (a, b):       # both ranks hold the reduced statistics of the whole run
        np.testing.assert_allclose(r[2], ch.dwell_sum.cpu().numpy(), rtol=1e-12)
        np.testing.assert_array_equal(r[3], ch.trans_sum.cpu().numpy())
    np.testing.assert_array_equal(np.concatenate([a[4], b[4]], axis=1), ch.node_state.cpu().numpy())
    np.testing.assert_array_equal(np.concatenate([a[5], b[5]]), ch.ev_total.cpu().numpy())
    cfg = synth.config_c5(n_sites=21)
    sched = TreeSchedule(cfg['parent'], cfg['length'])
    obs = engine.Observations.from_leaf_codes(sched, cfg['codes'], cfg['leaves'])
    tc = ToleranceChains(sched, cfg['Q'], cfg['pi'], dict(enumerate(cfg['part'])), cfg['rate_on'],
                         cfg['rate_off'], obs, n_chains=3, tol_obs=cfg['tol_obs'],
                         tol_obs_nodes=cfg['tol_obs_nodes'], cap_p=96, cap_t=48, seed=13)
    tc.sweep(3)
    a, b = res[0]['tmjp'], res[1]['tmjp']
    assert (a[0], a[1], b[0], b[1]) == (0, 32, 32, 31)
    for r in (a, b):
        np.testing.assert_allclose(r[2], tc.prim_dwell.cpu().numpy(), rtol=1e-12)
        np.testing.assert_array_equal(r[3], tc.prim_trans.cpu().numpy())
        np.testing.assert_allclose(r[4], tc.tol_stats.cpu().numpy(), rtol=1e-12)
    np.testing.assert_array_equal(np.concatenate([a[5], b[5]], axis=0), tc.p_node.cpu().numpy())
    np.testing.assert_array_equal(np.concatenate([a[6], b[6]], axis=0), tc.t_node.cpu().numpy())


def test_sharded_samplers_two_processes_one_gpu_gloo():
    """Two processes sharing cuda:0, gloo allreduce of the CUDA statistic tensors: the sharded
    RaoTehChains / ToleranceChains reproduce the unsharded histories and reduced statistics."""
    _run_sharded('gloo')


def test_sharded_samplers_two_ranks_nccl():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    _run_sharded('nccl')
