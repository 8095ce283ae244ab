"""
Forward (prior) simulation of tree MJP sites on the device (K10, csrc/rt_simulate.cu).

  simulate_sites      leaf codes of n_sites sites drawn node by node from P = expm(t Q)
                      (the law of synth.simulate_leaf_codes), returned as Observations that
                      TreeMJP / RaoTehChains / SiteMixtureMJP take without a copy;
  ForwardHistories    whole histories, jump by jump on every branch as the reference's
                      _sampler.get_forward_sample (raoteh/sampler/_sampler.py:67-235), in the
                      trajectory layout of RaoTehChains.

Uses: predictive checks of mapped statistics (simulate replicates under the fitted model with the
real alignment's gaps and compare their expectations with the real data's, Nielsen 2002), data
under a fitted mixture (SiteMixtureMJP.simulate), and the joint-distribution test of the samplers
(Geweke 2004): a history H and leaf data D drawn together from the prior make H an exact posterior
draw given D, so a Rao-Teh chain on D started at H (RaoTehChains.load_trajectories) is stationary
from its first sweep.

Randomness: Philox4x32-10 keyed by (seed; global site index, k) on a substream of its own, so the
output does not depend on how sites are split over calls (traj0 / n_traj) and replicate k + 1 is
independent of replicate k.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _native
from .engine import OBS_CODES, Observations, TreeMJP, _obs_slot, _ptr, _stream


def _root_tensor(root_distn, S, device):
    if root_distn is None:
        return None
    pi = np.asarray(root_distn, dtype=np.float64).ravel()
    if pi.shape != (S,) or not np.isfinite(pi).all() or (pi < 0).any() or not pi.sum() > 0:
        raise ValueError('root_distn must be %d non-negative finite weights with a positive sum' % S)
    return torch.from_numpy(pi.copy()).to(device)


def _leaf_layout(sched, leaf_nodes, missing_like):
    """(obs_slot, observed nodes in row order) of the simulated codes; with missing_like, the rows
    of the template."""
    if missing_like is not None:
        if missing_like.kind != OBS_CODES:
            raise ValueError('missing_like must hold hard codes (Observations.from_leaf_codes)')
        slot = np.asarray(missing_like.obs_slot, dtype=np.int32)
        if len(slot) != sched.n:
            raise ValueError('missing_like belongs to another tree')
        nodes = np.full(int(slot.max()) + 1, -1, dtype=np.int32)
        nodes[slot[slot >= 0]] = np.nonzero(slot >= 0)[0]
        if leaf_nodes is not None and not np.array_equal(np.asarray(leaf_nodes), nodes):
            raise ValueError('leaf_nodes differ from the observed nodes of missing_like')
        return slot, nodes
    nodes = sched.leaves if leaf_nodes is None else np.asarray(leaf_nodes, dtype=np.int32)
    return _obs_slot(sched, nodes), nodes


def _shard(n_sites, traj0, n_traj):
    n_sites, traj0 = int(n_sites), int(traj0)
    n_traj = n_sites - traj0 if n_traj is None else int(n_traj)
    if n_sites < 0 or traj0 < 0 or n_traj < 0 or traj0 + n_traj > n_sites:
        raise ValueError('the shard [traj0, traj0 + n_traj) must lie inside [0, n_sites)')
    return traj0, n_traj


def _call(A):
    _native.check(_native.lib().rt_forward_simulate(ctypes.byref(A), _stream()), 'rt_forward_simulate')


def _nodes_call(sched, P, class_weight, root_distn, n_sites, seed, k, leaf_nodes, missing_like,
                keep_node_states, traj0, n_traj, device):
    """Arguments of one RT_SIM_NODES call on the class transition matrices P [K, n, S, S], with its
    output tensors and the inputs it points to: (args, (Observations, node states or None, site
    classes or None), inputs).  The args hold raw device addresses, so the caller keeps the rest."""
    K, n, S = int(P.shape[0]), sched.n, int(P.shape[-1])
    traj0, T = _shard(n_sites, traj0, n_traj)
    if int(k) < 0:
        raise ValueError('the replicate index k must be non-negative')
    dev = torch.device(device)
    slot, nodes = _leaf_layout(sched, leaf_nodes, missing_like)
    ops, _ = sched.up_program(slot)
    ops = torch.from_numpy(ops).to(dev)
    parent = torch.from_numpy(sched.parent.copy()).to(dev)
    slot_d = torch.from_numpy(slot.copy()).to(dev)
    codes = torch.empty((len(nodes), T), dtype=torch.uint8, device=dev)
    node_state = torch.empty((n, T), dtype=torch.uint8, device=dev) if keep_node_states else None
    site_class = torch.empty(T, dtype=torch.uint8, device=dev) if K > 1 else None
    pi = _root_tensor(root_distn, S, dev)
    A = _native.ForwardArgs()
    A.S, A.n_nodes, A.n_ops, A.K, A.mode = S, n, len(ops), K, _native.SIM_NODES
    A.n_traj, A.traj_stride, A.traj0, A.obs_stride = T, T, traj0, T
    A.seed, A.k = int(seed), int(k)
    A.program, A.parent, A.obs_slot = _ptr(ops), _ptr(parent), _ptr(slot_d)
    A.class_weight, A.P, A.root_distn = _ptr(class_weight), _ptr(P), _ptr(pi)
    if missing_like is not None:
        A.tmpl, A.tmpl_stride, A.tmpl_n_sites = _ptr(missing_like.data), missing_like.stride, missing_like.n_sites
    A.obs, A.site_class, A.node_state = _ptr(codes), _ptr(site_class), _ptr(node_state)
    return A, (Observations(OBS_CODES, codes, slot, T), node_state, site_class), (ops, parent, slot_d, pi)


def _simulate_nodes(*args):
    """One RT_SIM_NODES call (arguments of _nodes_call): (Observations, node states or None, site
    classes or None)."""
    A, out, keep = _nodes_call(*args)
    _call(A)
    return out


def simulate_sites(sched, Q, n_sites, root_distn=None, seed=0, k=0, leaf_nodes=None, missing_like=None,
                   keep_node_states=False, traj0=0, n_traj=None, device='cuda'):
    """Leaf codes of n_sites sites simulated from the prior of the MJP Q [S, S] (2..64 states):
    x_root ~ root_distn (None: uniform), x_c ~ P_c[x_a, :] with P = TreeMJP.transition_matrices().

    Returns Observations (RT_OBS_CODES, rows = leaf_nodes, default the leaves) of the sites
    [traj0, traj0 + n_traj) (default all); with keep_node_states also the states of every node,
    uint8 [n_nodes, n_traj].  missing_like: the Observations of a real alignment (hard codes, N
    sites); the rows and obs_slot are taken from it, and site i is missing wherever site i % N is
    there (B replicates of the alignment: n_sites = B N).  k: the replicate index of the draw."""
    mjp = TreeMJP(sched, Q, device=device)
    if mjp.Q_host.shape[0] != 1:
        raise ValueError('Q must be one rate matrix [S, S]; SiteMixtureMJP.simulate takes classes')
    P = mjp.transition_matrices()[None]
    obs, ns, _ = _simulate_nodes(sched, P, None, root_distn, n_sites, seed, k, leaf_nodes, missing_like,
                                 keep_node_states, traj0, n_traj, mjp.device)
    return (obs, ns) if keep_node_states else obs


class ForwardHistories(object):
    """n_traj whole histories of the MJP Q [S, S] (2..64 states) simulated from the prior, jump by
    jump (rt_forward_simulate, RT_SIM_HISTORY), in the trajectory arrays of RaoTehChains:
    node_state / ev_count [n_nodes, n_traj] uint8, ev_total [n_traj] int32, ev_time [n_traj, cap]
    (float32, or float64 for 2, 3, 4, 5, 6 or 8 states), ev_sb [n_traj, cap] uint8, status.

    Trajectory t is the global site traj0 + t; draw() number k (k = 0, 1, ... counted by draws_done)
    is keyed by (seed; traj0 + t, k).  Each draw also writes the leaf codes; leaf_observations()
    returns them as Observations (one site per trajectory), to build a TreeMJP or RaoTehChains on,
    and RaoTehChains.load_trajectories() takes the histories."""

    def __init__(self, sched, Q, n_traj, root_distn=None, seed=0, cap=96, time_dtype='float32', traj0=0,
                 leaf_nodes=None, device='cuda'):
        if not torch.cuda.is_available():
            raise _native.NativeError('raoteh_b200 needs a CUDA device; there is no CPU fallback')
        Q = np.asarray(Q, dtype=np.float64)
        if Q.ndim != 2 or Q.shape[0] != Q.shape[1] or not 2 <= Q.shape[0] <= 64:
            raise ValueError('Q must be one square rate matrix with 2..64 states')
        self.S = S = Q.shape[0]
        if time_dtype not in ('float32', 'float64'):
            raise ValueError("time_dtype must be 'float32' or 'float64'")
        if time_dtype == 'float64' and (S > 8 or S == 7):
            raise ValueError('fp64 event times are implemented for 2, 3, 4, 5, 6 or 8 states '
                             '(the Rao-Teh kernels that read them)')
        if int(cap) <= 0:
            raise ValueError('cap must be positive')
        self.sched = sched
        self.device = dev = torch.device(device)
        self.n_traj = T = int(n_traj)
        self.traj0 = int(traj0)
        if T < 0 or self.traj0 < 0:
            raise ValueError('n_traj and traj0 must be non-negative')
        self.cap, self.seed, self.time_dtype = int(cap), int(seed), time_dtype
        self.Q_host = Q
        self.Q = torch.from_numpy(Q.copy()).to(dev)
        self.root_distn = _root_tensor(root_distn, S, dev)
        self.leaf_slot, self.leaf_nodes = _leaf_layout(sched, leaf_nodes, None)
        ops, _ = sched.up_program(self.leaf_slot)
        self.ops, self.n_ops = torch.from_numpy(ops).to(dev), len(ops)
        self.parent = torch.from_numpy(sched.parent.copy()).to(dev)
        self.length = torch.from_numpy(sched.length.copy()).to(dev)
        self._slot = torch.from_numpy(self.leaf_slot.copy()).to(dev)
        n = sched.n
        tt = torch.float64 if time_dtype == 'float64' else torch.float32
        self.node_state = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_count = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_total = torch.zeros(T, dtype=torch.int32, device=dev)
        self.ev_time = torch.zeros((T, self.cap), dtype=tt, device=dev)
        self.ev_sb = torch.zeros((T, self.cap), dtype=torch.uint8, device=dev)
        self.status = torch.zeros(T, dtype=torch.int8, device=dev)
        self.codes = torch.zeros((len(self.leaf_nodes), T), dtype=torch.uint8, device=dev)
        self.dwell_sum = torch.zeros(S, dtype=torch.float64, device=dev)
        self.trans_sum = torch.zeros((S, S), dtype=torch.float64, device=dev)
        self.draws_done = 0
        self._max_rate_length = float((-np.diag(Q)).max()) * float(np.max(sched.length))

    def draw(self, stats=True):
        """Replace every trajectory with a new history from the prior (and the leaf codes with its
        leaves); stats=True adds its dwell times and transition counts to dwell_sum / trans_sum."""
        A = _native.ForwardArgs()
        A.S, A.n_nodes, A.n_ops, A.K, A.mode = self.S, self.sched.n, self.n_ops, 1, _native.SIM_HISTORY
        A.cap, A.time_f64 = self.cap, 1 if self.time_dtype == 'float64' else 0
        A.n_traj, A.traj_stride, A.traj0, A.obs_stride = self.n_traj, self.n_traj, self.traj0, self.n_traj
        A.seed, A.k = self.seed, self.draws_done
        A.program, A.parent, A.length, A.obs_slot = _ptr(self.ops), _ptr(self.parent), _ptr(self.length), _ptr(self._slot)
        A.Q, A.root_distn = _ptr(self.Q), _ptr(self.root_distn)
        A.obs, A.node_state = _ptr(self.codes), _ptr(self.node_state)
        A.ev_time, A.ev_sb, A.ev_count, A.ev_total = (_ptr(self.ev_time), _ptr(self.ev_sb), _ptr(self.ev_count),
                                                      _ptr(self.ev_total))
        A.dwell_sum = _ptr(self.dwell_sum) if stats else None
        A.trans_sum = _ptr(self.trans_sum) if stats else None
        A.status = _ptr(self.status)
        _call(A)
        self.draws_done += 1
        self.check()

    def check(self):
        """Raise NativeError if a history could not be stored (status 3 or 4)."""
        over = int((self.status == 4).sum())
        long_branch = int((self.status == 3).sum())
        if long_branch:
            raise _native.NativeError(
                '%d simulated histories have more than 255 jumps on one branch (the per-branch counts '
                'are uint8; expected jumps per branch up to max_s q_s * length = %.0f): subdivide long '
                'branches with degree-two nodes (lowering.subdivide_long_branches)'
                % (long_branch, self._max_rate_length))
        if over:
            raise _native.NativeError('%d simulated histories have more than cap=%d jumps; create '
                                      'ForwardHistories with a larger cap' % (over, self.cap))

    def reset_statistics(self):
        self.dwell_sum.zero_()
        self.trans_sum.zero_()

    def trajectory(self, t):
        """Trajectory t as (node states, dict child node -> (times from the parent end, ascending;
        states of the segments, parent side first)), as RaoTehChains.trajectory."""
        from .raoteh import trajectory_edges
        return trajectory_edges(self.ops, self.node_state, self.ev_count, self.ev_total, self.ev_time,
                                self.ev_sb, self.cap, t)

    def leaf_observations(self, missing_like=None):
        """The leaf codes of the last draw as Observations with one site per trajectory (no copy).
        missing_like (Observations of hard codes on the same leaf rows, N sites): a copy in which
        trajectory t is missing wherever site (traj0 + t) % N is missing there."""
        obs = Observations(OBS_CODES, self.codes, self.leaf_slot, self.n_traj)
        if missing_like is None:
            return obs
        if missing_like.kind != OBS_CODES or not np.array_equal(missing_like.obs_slot, self.leaf_slot):
            raise ValueError('missing_like must hold hard codes on the same leaf rows')
        cols = (torch.arange(self.n_traj, device=self.device) + self.traj0) % missing_like.n_sites
        gaps = missing_like.data[:, :missing_like.n_sites][:, cols] == 255
        return Observations(OBS_CODES, torch.where(gaps, 255, self.codes).to(torch.uint8).contiguous(),
                            self.leaf_slot, self.n_traj)
