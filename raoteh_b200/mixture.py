"""
Site-class mixtures of tree MJPs: among-site rate variation (discrete gamma, +G, Yang 1994), an
invariant-sites class (+I, rate 0) and classes with their own rate matrix (codon models with
several omega classes, the M1a/M2a/M8 family).

Every site evolves under one of K classes, class k with prior weight w_k, rate matrix Q_k and
branch lengths r_k t; the classes share the tree and the root distribution.  Per site

    loglik = logsumexp_k(log w_k + loglik_k),    class_post[k] = exp(log w_k + loglik_k - loglik),

and the expected statistics under the mixture are sum_s class_post[k](s) E_k[stat | s].  Each
class is one TreeMJP on the schedule with lengths r_k t, so P, both tree passes and the Frechet
contraction are the single-class ones; the class posterior enters the down pass as a per-site
weight of the root marginal (rt_posterior_weighted_stats).  The classes share one workspace, so
the device memory is that of one single-class evaluation plus [K, n_sites] per-site arrays.
"""
from __future__ import annotations

import math

import numpy as np
import torch
from scipy import special

from .engine import TreeMJP
from .lowering import TreeSchedule


def discrete_gamma_rates(alpha, K, median=False):
    """Rates of the K equal-probability categories of Gamma(alpha, rate alpha) (mean 1), Yang
    (1994): the category boundaries are the quantiles k/K; the rate of a category is its mean
    (K times the integral of x g(x) over the category), or with `median` its median, rescaled so
    that the K rates have mean 1."""
    alpha = float(alpha)
    if not (math.isfinite(alpha) and alpha > 0):
        raise ValueError('alpha must be positive and finite')
    if int(K) != K or K < 1:
        raise ValueError('K must be a positive integer')
    K = int(K)
    if median:
        r = special.gammaincinv(alpha, (2.0 * np.arange(K) + 1.0) / (2.0 * K)) / alpha
        return r * (K / r.sum())
    # boundaries in units of the rate-1 gamma: alpha * b_k, with b_0 = 0 and b_K = inf
    cut = np.concatenate([[0.0], special.gammaincinv(alpha, np.arange(1, K) / K), [np.inf]])
    # int_a^b x g(x) dx = P(alpha + 1, alpha b) - P(alpha + 1, alpha a), P the regularised gamma
    return K * np.diff(special.gammainc(alpha + 1.0, cut))


class SiteMixtureMJP(object):
    """K site classes on one tree.

    Q: one rate matrix [S, S] shared by the K = len(rates) classes, or K matrices [K, S, S].
    rates: per-class multipliers of the branch lengths (default all 1); rate 0 is the +I class.
    weights: prior class probabilities (default uniform), positive, summing to 1.
    root_distn: the root distribution of every class (None: weights of 1, as TreeMJP).
    Per-edge rate matrices inside a class (TreeMJP's q_index) are not supported."""

    def __init__(self, sched, Q, root_distn=None, rates=None, weights=None, q_index=None,
                 device='cuda'):
        if q_index is not None:
            raise ValueError('per-edge rate matrices (q_index) are not supported inside mixture classes')
        Q = np.asarray(Q, dtype=np.float64)
        if Q.ndim == 2:
            K = 1 if rates is None else len(rates)
            Qs = np.broadcast_to(Q, (K,) + Q.shape)
        elif Q.ndim == 3:
            K = Q.shape[0]
            Qs = Q
        else:
            raise ValueError('Q must be [S, S] or [K, S, S]')
        S = Q.shape[-1]
        if Q.shape[-2] != S or not 2 <= S <= 64:
            raise ValueError('rate matrices must be square with 2..64 states')
        rates = np.ones(K) if rates is None else np.asarray(rates, dtype=np.float64).ravel()
        weights = np.full(K, 1.0 / K) if weights is None else np.asarray(weights, dtype=np.float64).ravel()
        if len(rates) != K or len(weights) != K:
            raise ValueError('rates and weights need one entry per class (K = %d)' % K)
        if not (np.isfinite(rates).all() and (rates >= 0).all()):
            raise ValueError('class rates must be finite and non-negative')
        if not (np.isfinite(weights).all() and (weights > 0).all() and abs(weights.sum() - 1.0) <= 1e-9):
            raise ValueError('class weights must be positive and sum to 1')
        self.K, self.S, self.sched = K, S, sched
        self.rates, self.weights = rates, weights
        self.device = torch.device(device)
        self.length = torch.from_numpy(np.asarray(sched.length, dtype=np.float64).copy()).to(self.device)
        self.tree_length = float(np.asarray(sched.length, dtype=np.float64)[1:].sum())
        self.classes = []
        for k in range(K):
            s = TreeSchedule(sched.parent, rates[k] * sched.length, sched.nodes)
            m = TreeMJP(s, Qs[k], root_distn=root_distn, device=device)
            if self.classes:
                # the classes run one after the other on one stream and have the same topology:
                # one set of workspaces (partials, W, node marginals) and of programs serves all
                m._ws = self.classes[0]._ws
                m._prog_cache = self.classes[0]._prog_cache
            self.classes.append(m)
        self.log_weights = torch.from_numpy(np.log(weights)).to(self.device)

    def log_likelihood(self, obs):
        """Per-site mixture log-likelihood.  Returns dict(loglik [N], status [N], class_post [K, N],
        loglik_class [K, N], loglik_sum).  status is 0 where some class has status 0, else 2 where
        some class has 2, else 1; infeasible sites have loglik -inf and class_post 0 and are left
        out of loglik_sum."""
        K, N, dev = self.K, obs.n_sites, self.device
        ll_class = torch.empty((K, N), dtype=torch.float64, device=dev)
        st_class = torch.empty((K, N), dtype=torch.int8, device=dev)
        for k, m in enumerate(self.classes):
            m.log_likelihood(obs, out=(ll_class[k], st_class[k]))
        ok_class = st_class == 0
        lw = torch.where(ok_class, self.log_weights[:, None] + ll_class,
                         torch.full_like(ll_class, -math.inf))
        loglik = torch.logsumexp(lw, dim=0)
        ok = ok_class.any(dim=0)
        loglik = torch.where(ok, loglik, torch.full_like(loglik, -math.inf))
        class_post = torch.where(ok[None, :], torch.exp(lw - torch.where(ok, loglik, 0.0)[None, :]),
                                 torch.zeros_like(lw))
        two = (st_class == 2).any(dim=0)
        status = torch.where(ok, 0, torch.where(two, 2, 1)).to(torch.int8)
        loglik_sum = torch.where(ok, loglik, torch.zeros_like(loglik)).sum()
        return dict(loglik=loglik, status=status, class_post=class_post, loglik_class=ll_class,
                    loglik_sum=loglik_sum)

    def expected_history_statistics(self, obs, want_node_distn=False, site_weight=None):
        """Expected statistics under the mixture, summed over sites (each site weighted by
        site_weight, default 1).  Returns the keys of TreeMJP's result that dist.pack_stats
        reads -- loglik_sum (sum of w_s loglik_s over feasible sites), dwell [S], trans [S, S],
        root_post_sum [S] -- and the per-site loglik, status, class_post; per class dwell_class
        [K, S], trans_class [K, S, S], M_edges_class [K, n, S, S] and class_post_sum [K] (the EM
        update of the class weights, times the total site weight); with want_node_distn the
        mixture node marginals [n_store, S, stride].  Dwell times are in tree time (the class's
        contraction runs on lengths r_k t and is divided by r_k; a rate-0 class dwells
        sum_b t_b per unit of root posterior and makes no transitions)."""
        N, S, K, n = obs.n_sites, self.S, self.K, self.sched.n
        if site_weight is not None:
            self.classes[0]._check_site_weight(site_weight, N)
        mix = self.log_likelihood(obs)
        cp = mix['class_post']
        w = cp if site_weight is None else cp * site_weight[None, :]
        dev = self.device
        dwell = torch.empty((K, S), dtype=torch.float64, device=dev)
        trans = torch.empty((K, S, S), dtype=torch.float64, device=dev)
        M_class = torch.empty((K, n, S, S), dtype=torch.float64, device=dev)
        rps = torch.empty((K, S), dtype=torch.float64, device=dev)
        node_distn = None
        for k, m in enumerate(self.classes):
            post = m.posterior(obs, want_node_distn=want_node_distn, site_weight=w[k])
            rps[k] = post['root_post_sum']
            r = float(self.rates[k])
            if r > 0:
                M, d, t = m.history_statistics(post['W'])
                M_class[k] = M / r
                dwell[k] = d / r
                trans[k] = t
            else:
                # P = I: W_b is diagonal and L(r t Q^T, r t W) / r -> t W as r -> 0
                M_class[k] = self.length[:, None, None] * post['W']
                dwell[k] = self.tree_length * post['root_post_sum']
                trans[k].zero_()
            if want_node_distn:
                nd = post['node_distn']
                node_distn = nd.clone() if node_distn is None else node_distn.add_(nd)
        loglik_sum = (mix['loglik_sum'] if site_weight is None else
                      TreeMJP._weighted_loglik_sum(mix['loglik'], mix['status'], site_weight))
        return dict(loglik=mix['loglik'], status=mix['status'], class_post=cp,
                    loglik_class=mix['loglik_class'], loglik_sum=loglik_sum,
                    dwell=dwell.sum(dim=0), trans=trans.sum(dim=0), root_post_sum=rps.sum(dim=0),
                    dwell_class=dwell, trans_class=trans, M_edges_class=M_class,
                    class_post_sum=w.sum(dim=1), node_distn=node_distn)

    def branch_expectations(self, obs, E=None):
        """Per site and branch posterior expectation of the number of E-type transitions under
        the mixture: sum_k class_post[k] * (class k's TreeMJP.branch_expectations, with K_b built
        on the class's lengths r_k t).  Returns dict(branch [n, N], loglik, status, class_post)."""
        mix = self.log_likelihood(obs)
        cp = mix['class_post']
        branch = None
        for k, m in enumerate(self.classes):
            b = m.branch_expectations(obs, E=E)['branch'] * cp[k][None, :]
            branch = b if branch is None else branch.add_(b)
        return dict(branch=branch, loglik=mix['loglik'], status=mix['status'], class_post=cp)

    def simulate(self, n_sites, seed=0, k=0, leaf_nodes=None, missing_like=None, keep_node_states=False,
                 traj0=0, n_traj=None):
        """Leaf codes of n_sites sites simulated from the mixture (rt_forward_simulate, RT_SIM_NODES):
        each site draws its class from the weights, then its node states from that class's P (on
        lengths r_k t; the +I class keeps the root state everywhere).  The root distribution is the
        mixture's (None: uniform).  Arguments as simulate.simulate_sites.  Returns (Observations,
        site_class uint8 [n_traj]), plus the node states [n_nodes, n_traj] with keep_node_states.
        With K = 1 the codes are bit for bit those of simulate_sites."""
        from .simulate import _simulate_nodes
        P = torch.stack([m.transition_matrices() for m in self.classes])
        w = torch.from_numpy(self.weights.copy()).to(self.device)
        obs, ns, cls = _simulate_nodes(self.sched, P, w, self.classes[0].root_distn_host, n_sites, seed, k,
                                       leaf_nodes, missing_like, keep_node_states, traj0, n_traj, self.device)
        if cls is None:
            cls = torch.zeros(obs.n_sites, dtype=torch.uint8, device=self.device)
        return (obs, cls, ns) if keep_node_states else (obs, cls)

    def history_draws(self, obs, n_chains=1, seed=0, cap=96, time_dtype='float32', traj0=0,
                      n_traj=None):
        """Exact posterior draws of (class, history) per site under the mixture (stochastic mapping
        under +G, +I or omega classes): see MixtureHistoryDraws.  2..8 states, hard codes or
        allowed-state masks."""
        return MixtureHistoryDraws(self, obs, n_chains=n_chains, seed=seed, cap=cap,
                                   time_dtype=time_dtype, traj0=traj0, n_traj=n_traj)


class MixtureHistoryDraws(object):
    """n_chains x n_sites iid exact draws from p(class, history | data) of a SiteMixtureMJP
    (rt_posterior_draw_mixture): each trajectory draws its site's class from the class posterior,
    then the whole history from that class's P, pruning partials and uniformization (the
    single-class draw of RaoTehChains.draw_posterior).  A fast site gets the jumps of its rate class
    and a site drawn into the +I class none.

    Trajectory arrays as RaoTehChains (trajectory t = chain * n_sites + site; this object may own
    the shard [traj0, traj0 + n_traj)): node_state, ev_count, ev_total, ev_time, ev_sb, status,
    plus site_class [n_traj] (uint8); draw(stats=True) accumulates dwell_class [K, S] (tree time)
    and trans_class [K, S, S].  Draw k is keyed by (seed; traj0 + t, k), so shards and repeats
    reproduce it bit for bit.

    There is no sweep(): the draws are iid, so Rao-Teh sweeps are not needed, and a sweep under a
    mixture would have to update the class inside the sweep, which is not implemented.

    Memory: every class's up-pass partials are kept, K x n_store x S x 8 bytes per site (about
    100 MB for K = 5 at 4 states, 63 stored nodes and 1e4 sites; about 10 GB at 1e6 sites), plus
    the class P and the per-site class posteriors."""

    def __init__(self, mix, obs, n_chains=1, seed=0, cap=96, time_dtype='float32', traj0=0,
                 n_traj=None):
        from . import raoteh
        from .engine import OBS_CODES, OBS_MASK
        S, K = mix.S, mix.K
        if not 2 <= S <= 8:
            raise ValueError('exact history draws support 2..8 states')
        if obs.kind not in (OBS_CODES, OBS_MASK):
            raise ValueError('exact history draws take hard codes or allowed-state masks')
        if time_dtype not in ('float32', 'float64'):
            raise ValueError("time_dtype must be 'float32' or 'float64'")
        if time_dtype == 'float64' and S == 7:
            raise ValueError('fp64 event times are implemented for 2, 3, 4, 5, 6 or 8 states')
        length = np.asarray(mix.sched.length, dtype=np.float64)
        gens = [float(mix.rates[k]) * mix.classes[k].Q_host[0] for k in range(K)]
        for k, G in enumerate(gens):
            n_pow = raoteh.draw_power_table_length(G, length)
            if n_pow > raoteh.DRAW_MAX_POW:
                raise ValueError(
                    'class %d (rate %g) has a branch too long for the exact draw: max_s q_s * rate * '
                    'length = %.0f needs B^n up to n = %d, more than %d; subdivide long branches '
                    'with degree-two nodes (lowering.subdivide_long_branches)'
                    % (k, mix.rates[k], float(-np.diag(G).min()) * float(length.max()), n_pow,
                       raoteh.DRAW_MAX_POW))
        self.mix, self.obs, self.S, self.K = mix, obs, S, K
        self.sched, self.device = mix.sched, mix.device
        dev = self.device
        self.n_sites, self.n_chains = obs.n_sites, int(n_chains)
        self.traj0 = int(traj0)
        self.n_traj = T = self.n_chains * self.n_sites if n_traj is None else int(n_traj)
        self.cap, self.seed, self.time_dtype = int(cap), int(seed), time_dtype
        self._tt = torch.float64 if time_dtype == 'float64' else torch.float32
        self._max_rate_length = max(float(-np.diag(G).min()) for G in gens) * float(length.max())
        # inputs, built once: class generators r_k Q_k, class P on lengths r_k t, every class's
        # up-pass partials in its own slice (the classes share one workspace), class posteriors
        self.Q = torch.from_numpy(np.ascontiguousarray(np.stack(gens))).to(dev)
        n, ns, stride = self.sched.n, self.sched.n_store, obs.stride
        self.P = torch.empty((K, n, S, S), dtype=torch.float64, device=dev)
        self.partials = torch.empty((K, ns, S, stride), dtype=torch.float64, device=dev)
        lik = mix.log_likelihood(obs)
        self.class_post = lik['class_post'].contiguous()
        self.site_status = lik['status'].contiguous()
        for k, m in enumerate(mix.classes):
            self.P[k].copy_(m.transition_matrices())
            self.partials[k].copy_(m.log_likelihood(obs, keep_partials=True)['partials'])
        ops, _ = self.sched.up_program(obs.obs_slot)
        self.ops, self.n_ops = torch.from_numpy(ops).to(dev), len(ops)
        self.parent = torch.from_numpy(self.sched.parent.copy()).to(dev)
        self.stride = T
        self.node_state = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_count = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_total = torch.zeros(T, dtype=torch.int32, device=dev)
        self.ev_time = torch.zeros((T, self.cap), dtype=self._tt, device=dev)
        self.ev_sb = torch.zeros((T, self.cap), dtype=torch.uint8, device=dev)
        self.status = torch.zeros(T, dtype=torch.int8, device=dev)
        self.site_class = torch.zeros(T, dtype=torch.uint8, device=dev)
        self.dwell_class = torch.zeros((K, S), dtype=torch.float64, device=dev)
        self.trans_class = torch.zeros((K, S, S), dtype=torch.float64, device=dev)
        self.draws_done = 0

    def _args(self, stats):
        from . import _native
        from .engine import _ptr
        A = _native.PosteriorDrawMixtureArgs()
        B = A.base
        B.S, B.n_nodes, B.n_ops, B.cap = self.S, self.sched.n, self.n_ops, self.cap
        B.obs_kind, B.time_f64 = self.obs.kind, 1 if self.time_dtype == 'float64' else 0
        B.n_traj, B.traj_stride, B.n_sites, B.traj0 = self.n_traj, self.stride, self.n_sites, self.traj0
        B.obs_stride, B.site_stride = self.obs.stride, self.obs.stride
        B.seed, B.k = self.seed, self.draws_done
        B.program, B.parent, B.length = _ptr(self.ops), _ptr(self.parent), _ptr(self.mix.length)
        B.Q, B.P, B.root_distn = _ptr(self.Q), _ptr(self.P), _ptr(self.mix.classes[0].root_distn)
        B.obs, B.partials, B.site_status = _ptr(self.obs.data), _ptr(self.partials), _ptr(self.site_status)
        B.node_state, B.ev_time, B.ev_sb = _ptr(self.node_state), _ptr(self.ev_time), _ptr(self.ev_sb)
        B.ev_count, B.ev_total, B.sweep_count = _ptr(self.ev_count), _ptr(self.ev_total), None
        B.dwell_sum = _ptr(self.dwell_class) if stats else None
        B.trans_sum = _ptr(self.trans_class) if stats else None
        B.status = _ptr(self.status)
        A.K = self.K
        A.partials_class_stride = self.partials[0].numel()
        A.class_post_stride = self.class_post.shape[1]
        A.class_post, A.site_class = _ptr(self.class_post), _ptr(self.site_class)
        return A

    def draw(self, stats=True):
        """Replace every trajectory with a new iid draw (index k = draws_done); stats=True adds the
        drawn histories' statistics to dwell_class / trans_class."""
        import ctypes
        from . import _native
        from .engine import _stream
        self.status.zero_()
        A = self._args(stats)
        rc = _native.lib().rt_posterior_draw_mixture(ctypes.byref(A), _stream())
        _native.check(rc, 'rt_posterior_draw_mixture')
        self.draws_done += 1
        self.check()

    def trajectory(self, t):
        """Trajectory t as (node states, dict child node -> (times, segment states)), as
        RaoTehChains.trajectory."""
        from .raoteh import trajectory_edges
        return trajectory_edges(self.ops, self.node_state, self.ev_count, self.ev_total, self.ev_time,
                                self.ev_sb, self.cap, t)

    def check(self):
        from .raoteh import check_status
        check_status(self.status, self.cap, self._max_rate_length)

    def reset_statistics(self):
        self.dwell_class.zero_()
        self.trans_class.zero_()
