"""
Batched Rao-Teh sampler: many independent (chain, site) trajectories on device.

Host side of K6 (csrc/rt_raoteh.cu).  Mirrors the generator loop of the
reference, raoteh/sampler/_sampler.py:300-390 (gen_restricted_histories):
uniformization constants (:346-355), initial feasible history (:362 -> :563),
then sweeps (:366-390); statistics as _mjp.get_history_statistics
(raoteh/sampler/_mjp.py:150).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native
from .engine import OBS_CODES, OBS_MASK, _ptr, _stream


# longest table of powers B^0..B^n of rt_posterior_draw (csrc/rt_posterior_draw.cu, kMaxPow)
DRAW_MAX_POW = 320


def draw_power_table_length(Q, length, eps=1e-17):
    """n such that the Poisson tail beyond n at mu * max_b t_b (mu = max_s q_s) is below eps: the
    length of the table of powers B^n the exact draw needs (the kernel's own rule, before its cap)."""
    import math
    Q = np.asarray(Q, dtype=np.float64)
    mu = float((-np.diag(Q)).max())
    if not mu > 0:
        mu = 1.0
    lam = mu * float(np.max(length[1:])) if len(length) > 1 else 0.0
    n = int(math.ceil(lam))
    while n < 4 * DRAW_MAX_POW:
        r = lam / (n + 1)
        logp = (-lam + n * math.log(lam) - math.lgamma(n + 1.0)) if lam > 0 else (0.0 if n == 0 else -math.inf)
        if r < 1.0 and math.exp(logp) * r / (1.0 - r) < eps:
            break
        n += 1
    return max(n, 2 * Q.shape[0] + 8)


def check_status(status, cap, max_rate_length):
    """Raise NativeError for trajectories with status != 0 (1: no feasible history, 4: more than
    `cap` real jumps, else out of event capacity); max_rate_length = the largest expected number of
    events on one branch, for the message."""
    bad = int((status != 0).sum())
    if bad and int((status == 1).sum()):
        raise _native.NativeError('no feasible history (structural zero) for %d trajectories'
                                  % int((status == 1).sum()))
    if bad and int((status == 4).sum()):
        raise _native.NativeError('initial history has more than cap=%d real jumps' % cap)
    if bad:
        raise _native.NativeError(
            '%d trajectories exceeded the event capacity in one sweep (status 3): more than '
            'cap=%d candidate events in the trajectory, or more than 255 on one branch '
            '(expected per branch: omega * length, here up to %.0f); re-create the sampler '
            'with a larger cap, or subdivide long branches with degree-two nodes'
            % (bad, cap, max_rate_length))


def trajectory_edges(ops, node_state, ev_count, ev_total, ev_time, ev_sb, cap, t):
    """Trajectory t of the trajectory arrays as per-edge arrays: (node states, dict child node ->
    (times from the parent end, ascending; states of the k+1 segments, parent side first))."""
    cnt = ev_count[:, t].cpu().numpy().astype(int)
    tot = int(ev_total[t])
    times = ev_time[t, cap - tot:].cpu().numpy()
    sbs = ev_sb[t, cap - tot:].cpu().numpy().astype(int)
    ns = node_state[:, t].cpu().numpy().astype(int)
    out = {}
    pos = 0
    for code, c, a, b in ops.cpu().numpy():
        if (code & 0xff) > 2:
            continue
        k = cnt[c]
        tt = times[pos:pos + k][::-1]          # stored child end first
        sb = sbs[pos:pos + k][::-1]
        pos += k
        states = np.concatenate([sb, [ns[c]]]) if k else np.array([ns[c]])
        out[int(c)] = (tt.astype(float), states)
    return ns, out


class RaoTehChains(object):
    """n_chains x n_sites trajectories of one MJP on one tree.

    trajectory t = chain * n_sites + site; observations are per site.
    """

    def __init__(self, sched, Q, obs, n_chains=1, root_distn=None, uniformization_factor=2.0,
                 cap=96, seed=0, device='cuda', traj0=0, n_traj=None, chain_matrix=None,
                 time_dtype='float32'):
        """time_dtype: 'float32' (default: 4-byte jump lists) or 'float64' (every event time,
        branch position and Poisson hazard in the reference's fp64 arithmetic; S <= 8).
        chain_matrix: instead of a rate matrix, a transition matrix B applied at every
        candidate event, with no virtual events (Poisson rates 0): the discrete-time chain
        samplers of raoteh/sampler/_sample_mcy.py / _sample_mcx.py are this special case."""
        if not torch.cuda.is_available():
            raise _native.NativeError('raoteh_b200 needs a CUDA device; there is no CPU fallback')
        if uniformization_factor <= 1:
            raise ValueError('the uniformization factor must be greater than 1')
        if chain_matrix is not None:
            Bc = np.asarray(chain_matrix, dtype=np.float64)
            Q = Bc - np.eye(Bc.shape[0])          # placeholder generator with the same pattern
        Q = np.asarray(Q, dtype=np.float64)
        self.S = S = Q.shape[0]
        if not 2 <= S <= 64:
            raise ValueError('the Rao-Teh kernels support 2..64 states')
        if obs.kind not in (OBS_CODES, OBS_MASK):
            raise ValueError('Rao-Teh sampling takes hard codes or allowed-state masks')
        self.sched = sched
        self.obs = obs
        self.device = dev = torch.device(device)
        self.n_sites = obs.n_sites
        self.n_chains = int(n_chains)
        # this object may own a contiguous shard [traj0, traj0 + n_traj) of the global
        # (chain, site) index space (site sharding across GPUs)
        self.traj0 = int(traj0)
        self.n_traj = int(n_chains) * self.n_sites if n_traj is None else int(n_traj)
        self.cap = int(cap)
        self.seed = int(seed)
        if time_dtype not in ('float32', 'float64'):
            raise ValueError("time_dtype must be 'float32' or 'float64'")
        if time_dtype == 'float64' and (S > 8 or S == 7):
            raise ValueError('fp64 event times are implemented by the thread-per-trajectory kernel '
                             '(2, 3, 4, 5, 6 or 8 states)')
        self.time_dtype = time_dtype
        self._tt = torch.float64 if time_dtype == 'float64' else torch.float32
        # uniformization: omega = f * max_s q_s; B = I + Q/omega; rates omega - q_s
        q = -np.diag(Q)
        self.omega = float(uniformization_factor * q.max())
        if not self.omega > 0:
            if chain_matrix is None:
                raise ValueError('the rate matrix is empty')
            self.omega = 1.0
        B = np.eye(S) + Q / self.omega
        rate = self.omega - q
        if chain_matrix is not None:
            B, rate, self.omega = Bc, np.zeros(S), 1.0
        self.Q_host = Q
        self._chain_matrix = chain_matrix is not None
        self._root_distn_host = None if root_distn is None else np.asarray(root_distn, dtype=np.float64)
        self._draw_inputs = None       # (TreeMJP, P, partials, site status) of draw_posterior
        self.B = torch.from_numpy(np.ascontiguousarray(B)).to(dev)
        self.rate = torch.from_numpy(np.ascontiguousarray(rate)).to(dev)
        self.root_distn = None if root_distn is None else torch.from_numpy(
            np.asarray(root_distn, dtype=np.float64).copy()).to(dev)
        ops, n_slots = sched.up_program(obs.obs_slot)
        self.ops = torch.from_numpy(ops).to(dev)
        self.n_ops, self.n_slots = len(ops), n_slots
        self.parent = torch.from_numpy(sched.parent.copy()).to(dev)
        self.length = torch.from_numpy(sched.length.copy()).to(dev)
        T, n = self.n_traj, sched.n
        self.stride = T
        self.node_state = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_count = torch.zeros((n, T), dtype=torch.uint8, device=dev)
        self.ev_total = torch.zeros(T, dtype=torch.int32, device=dev)
        self.ev_time = torch.zeros((T, self.cap), dtype=self._tt, device=dev)
        # sweeps completed per trajectory (thread-per-trajectory kernel): lets a trajectory that
        # ran out of event capacity resume at its own sweep index after grow()
        self.sweep_count = (torch.zeros(T, dtype=torch.int32, device=dev)
                            if (S <= 8 and S != 7) else None)
        self.ev_sb = torch.zeros((T, self.cap), dtype=torch.uint8, device=dev)
        self.status = torch.zeros(T, dtype=torch.int8, device=dev)
        self.dwell_sum = torch.zeros(S, dtype=torch.float64, device=dev)
        self.trans_sum = torch.zeros((S, S), dtype=torch.float64, device=dev)
        self.sweeps_done = 0
        self.initialized = False

    def _call(self, n_sweeps, init_k, stats):
        import ctypes
        A = _native.RaotehArgs()
        A.S, A.n_nodes, A.n_ops, A.n_slots = self.S, self.sched.n, self.n_ops, self.n_slots
        A.obs_kind, A.cap, A.n_sweeps, A.init_k = self.obs.kind, self.cap, int(n_sweeps), int(init_k)
        A.time_f64 = 1 if self.time_dtype == 'float64' else 0
        A.n_traj, A.traj_stride, A.n_sites, A.traj0 = self.n_traj, self.stride, self.n_sites, self.traj0
        A.obs_stride, A.sweep0, A.seed = self.obs.stride, self.sweeps_done, self.seed
        A.program, A.parent, A.length = _ptr(self.ops), _ptr(self.parent), _ptr(self.length)
        A.B, A.rate, A.root_distn = _ptr(self.B), _ptr(self.rate), _ptr(self.root_distn)
        A.obs = _ptr(self.obs.data)
        A.node_state, A.ev_time, A.ev_sb = _ptr(self.node_state), _ptr(self.ev_time), _ptr(self.ev_sb)
        A.ev_count, A.ev_total = _ptr(self.ev_count), _ptr(self.ev_total)
        A.sweep_count = _ptr(self.sweep_count)
        A.dwell_sum = _ptr(self.dwell_sum) if stats else None
        A.trans_sum = _ptr(self.trans_sum) if stats else None
        A.status = _ptr(self.status)
        rc = _native.lib().rt_raoteh_run(ctypes.byref(A), _stream())
        _native.check(rc, 'rt_raoteh_run')

    def initialize(self):
        """Initial feasible history: 0, 1, 3, 7, ... equally spaced events per edge
        until FFBS under B succeeds (raoteh/sampler/_sampler.py:612-643)."""
        DONE = 5
        k, j = 0, 0
        self.status.zero_()
        while True:
            if k > self.S:
                raise RuntimeError('failed to find a feasible history')
            self._call(1, k, False)
            failed = self.status == 1
            self.status[self.status == 0] = DONE
            if not bool(failed.any()):
                break
            self.status[failed] = 0
            k += 2 ** j
            j += 1
        self.status[self.status == DONE] = 0
        self.check()
        if self.sweep_count is not None:
            self.sweep_count.fill_(1)
        self.sweeps_done = 1      # sweep index 0 was the initial history
        self.initialized = True
        return k

    def sweep(self, n_sweeps=1, stats=True, auto_grow=False):
        """n_sweeps Rao-Teh sweeps of every trajectory; raises if any trajectory needed
        more than `cap` candidate events in one sweep."""
        if not self.initialized:
            self.initialize()
        self._call(int(n_sweeps), -1, stats)
        if auto_grow and self.sweep_count is not None:
            # a trajectory that ran out of event capacity stopped at its last completed sweep
            # (a valid history) and its own sweep counter: double the pools and repeat the SAME
            # call -- trajectories already at the target do nothing, the stopped ones resume at
            # their own sweep index, so every (trajectory, sweep) enters the statistics once
            tries = 0
            while bool((self.status == 3).any()) and self.omega * float(self.sched.length.max()) < 200 \
                    and tries < 4:
                self.grow(2 * self.cap)
                self._call(int(n_sweeps), -1, stats)
                tries += 1
        self.sweeps_done += int(n_sweeps)
        self.check()

    def draw_posterior(self, stats=True):
        """Replace every trajectory with an independent exact draw from the posterior over histories
        given its site's observations (rt_posterior_draw: node states top-down from the pruning
        partials, then a path on every branch given its end states by uniformization).  The draw
        takes sweep index k = sweeps_done, as a sweep would, so

          - called instead of initialize(), the chains start at stationarity: no burn-in is needed
            before the sweeps' statistics are unbiased;
          - called repeatedly, it is an iid Monte Carlo sampler whose statistics accumulate in
            dwell_sum / trans_sum (stats=True) exactly like those of sweeps.

        Thread-per-trajectory kernel: 2..8 states; not for chain_matrix chains (no rate matrix)."""
        import ctypes
        from .engine import TreeMJP
        if self._chain_matrix:
            raise ValueError('draw_posterior needs a rate matrix; chain_matrix chains have none')
        if self.S > 8:
            raise ValueError('draw_posterior supports 2..8 states')
        n_pow = draw_power_table_length(self.Q_host, self.sched.length)
        if n_pow > DRAW_MAX_POW:
            raise ValueError(
                'a branch is too long for the exact draw: max_s q_s * length = %.0f needs B^n up to '
                'n = %d, more than %d; subdivide long branches with degree-two nodes '
                '(lowering.subdivide_long_branches)'
                % (float(-np.diag(self.Q_host).min()) * float(self.sched.length.max()), n_pow, DRAW_MAX_POW))
        if self._draw_inputs is None:
            # P and the pruning partials depend on Q and the observations only, both fixed here
            mjp = TreeMJP(self.sched, self.Q_host, root_distn=self._root_distn_host, device=self.device)
            P = mjp.transition_matrices()
            up = mjp.log_likelihood(self.obs, keep_partials=True)
            self._draw_inputs = (mjp, P, up['partials'], up['status'])
        mjp, P, partials, site_status = self._draw_inputs
        self.status.zero_()
        A = _native.PosteriorDrawArgs()
        A.S, A.n_nodes, A.n_ops, A.cap = self.S, self.sched.n, self.n_ops, self.cap
        A.obs_kind, A.time_f64 = self.obs.kind, 1 if self.time_dtype == 'float64' else 0
        A.n_traj, A.traj_stride, A.n_sites, A.traj0 = self.n_traj, self.stride, self.n_sites, self.traj0
        A.obs_stride, A.site_stride = self.obs.stride, self.obs.stride
        A.seed, A.k = self.seed, self.sweeps_done
        A.program, A.parent, A.length = _ptr(self.ops), _ptr(self.parent), _ptr(self.length)
        A.Q, A.P, A.root_distn = _ptr(mjp.Q), _ptr(P), _ptr(self.root_distn)
        A.obs, A.partials, A.site_status = _ptr(self.obs.data), _ptr(partials), _ptr(site_status)
        A.node_state, A.ev_time, A.ev_sb = _ptr(self.node_state), _ptr(self.ev_time), _ptr(self.ev_sb)
        A.ev_count, A.ev_total, A.sweep_count = _ptr(self.ev_count), _ptr(self.ev_total), _ptr(self.sweep_count)
        A.dwell_sum = _ptr(self.dwell_sum) if stats else None
        A.trans_sum = _ptr(self.trans_sum) if stats else None
        A.status = _ptr(self.status)
        _native.check(_native.lib().rt_posterior_draw(ctypes.byref(A), _stream()), 'rt_posterior_draw')
        self.sweeps_done += 1
        self.initialized = True
        self.check()

    def grow(self, cap):
        """Re-allocate the jump pools with a larger capacity (contents stay right-aligned) and
        clear the capacity flags; flagged trajectories continue from their last completed sweep."""
        cap = int(cap)
        if cap <= self.cap:
            return
        T, dev = self.n_traj, self.device
        for name, dt in (('ev_time', self._tt), ('ev_sb', torch.uint8)):
            new = torch.zeros((T, cap), dtype=dt, device=dev)
            new[:, cap - self.cap:] = getattr(self, name)
            setattr(self, name, new)
        self.cap = cap
        self.status[self.status == 3] = 0

    def check(self):
        check_status(self.status, self.cap, self.omega * float(self.sched.length.max()))

    def reset_statistics(self):
        self.dwell_sum.zero_()
        self.trans_sum.zero_()

    def trajectory_log_likelihood(self, stats=False):
        """log-likelihood of every trajectory under this MJP (_mjp.get_trajectory_log_likelihood,
        raoteh/sampler/_mjp.py:186-250) -> fp64 [n_traj], computed on the device.  stats=True also
        adds the sufficient statistics of the CURRENT histories to dwell_sum / trans_sum."""
        import ctypes
        A = _native.TmjpArgs()
        A.S, A.n_parts, A.n_nodes = self.S, 0, self.sched.n
        A.n_ops, A.n_slots, A.cap_p, A.cap_t = self.n_ops, self.n_slots, self.cap, 1
        A.obs_kind = self.obs.kind
        A.program, A.parent, A.length = _ptr(self.ops), _ptr(self.parent), _ptr(self.length)
        A.B, A.rate_p, A.pi_p = _ptr(self.B), _ptr(self.rate), _ptr(self.root_distn)
        A.omega_p = self.omega
        A.obs, A.obs_stride = _ptr(self.obs.data), self.obs.stride
        A.n_traj, A.n_sites, A.traj0 = self.n_traj, self.n_sites, self.traj0
        A.p_node, A.p_cnt = _ptr(self.node_state), _ptr(self.ev_count)
        A.pn_traj_stride, A.pn_node_stride = 1, self.stride
        A.p_total, A.p_time, A.p_sb = _ptr(self.ev_total), _ptr(self.ev_time), _ptr(self.ev_sb)
        A.status = _ptr(self.status)
        A.mode = 4
        if stats:
            A.flags = 1
            A.prim_dwell, A.prim_trans = _ptr(self.dwell_sum), _ptr(self.trans_sum)
        out = torch.empty(self.n_traj, dtype=torch.float64, device=self.device)
        A.traj_loglik = _ptr(out)
        _native.check(_native.lib().rt_tmjp_run(ctypes.byref(A), _stream()), 'rt_tmjp_run')
        return out

    def load_events(self, edge_times):
        """Install the same candidate events on every trajectory: edge_times[child node] = event
        times from the parent end.  The next sweep runs FFBS over exactly these events (plus
        virtual ones if the Poisson rates are positive)."""
        n = self.sched.n
        ops = self.ops.cpu().numpy()
        order = [int(c) for code, c, a, b in ops if (code & 0xff) <= 2]
        cnt = np.zeros(n, dtype=np.uint8)
        tt = []
        for c in order:
            ts = sorted(float(x) for x in edge_times.get(c, ()))
            if len(ts) > 255:
                raise ValueError('more than 255 events on the branch above node %d: the per-branch '
                                 'event counts of the kernels are uint8; subdivide the branch with '
                                 'degree-two nodes (lowering.subdivide_long_branches)' % c)
            cnt[c] = len(ts)
            tt.extend(ts[::-1])                # child end first
        k = len(tt)
        if k > self.cap:
            raise ValueError('more events than cap')
        row = np.zeros(self.cap, dtype=np.float64 if self.time_dtype == 'float64' else np.float32)
        if k:
            row[self.cap - k:] = tt
        dev = self.device
        self.ev_time.copy_(torch.from_numpy(row).to(dev)[None, :].expand(self.n_traj, -1))
        self.ev_sb.zero_()
        self.ev_count.copy_(torch.from_numpy(cnt).to(dev)[:, None].expand(-1, self.n_traj))
        self.ev_total.fill_(k)
        self.node_state.zero_()
        self.status.zero_()
        if self.sweep_count is not None:
            self.sweep_count.fill_(self.sweeps_done)
        self.initialized = True

    def load_trajectories(self, node_state, ev_count, ev_total, ev_time, ev_sb):
        """Copy in a whole trajectory state in this object's layout (for instance the histories of
        simulate.ForwardHistories, whose leaves are these observations): node_state / ev_count
        [n_nodes, n_traj], ev_total [n_traj], ev_time / ev_sb [n_traj, c] with c <= cap (jumps
        right-aligned; ev_time of this object's time dtype).  The chains are then initialized and
        the next sweep takes index sweeps_done (sweep_count is set to it where the kernel keeps one)."""
        n, T = self.sched.n, self.n_traj
        c = int(ev_time.shape[-1])
        if tuple(node_state.shape) != (n, T) or tuple(ev_count.shape) != (n, T) or \
                tuple(ev_total.shape) != (T,) or tuple(ev_time.shape) != (T, c) or tuple(ev_sb.shape) != (T, c):
            raise ValueError('trajectory arrays must be [n_nodes, n_traj] / [n_traj] / [n_traj, c]')
        if c > self.cap:
            raise ValueError('the jump lists hold %d entries, more than cap=%d' % (c, self.cap))
        if ev_time.dtype != self._tt:
            raise ValueError('ev_time must be %s like this object (time_dtype)' % self._tt)
        self.node_state.copy_(node_state)
        self.ev_count.copy_(ev_count)
        self.ev_total.copy_(ev_total)
        self.ev_time[:, self.cap - c:].copy_(ev_time)
        self.ev_sb[:, self.cap - c:].copy_(ev_sb)
        self.status.zero_()
        if self.sweep_count is not None:
            self.sweep_count.fill_(self.sweeps_done)
        self.initialized = True

    _STATE = ('node_state', 'ev_count', 'ev_total', 'ev_time', 'ev_sb')

    def snapshot(self):
        """Copy of the trajectory state (for Metropolis-Hastings rejection)."""
        return dict((k, getattr(self, k).clone()) for k in self._STATE)

    def restore(self, snap, reject=None):
        """Put back the snapshot; with `reject` (bool [n_traj]) only those trajectories."""
        for k in self._STATE:
            cur = getattr(self, k)
            if reject is None:
                cur.copy_(snap[k])
            elif k in ('node_state', 'ev_count'):          # [n_nodes, n_traj]
                torch.where(reject[None, :], snap[k], cur, out=cur)
            elif k == 'ev_total':
                torch.where(reject, snap[k], cur, out=cur)
            else:                                          # [n_traj, cap]
                torch.where(reject[:, None], snap[k], cur, out=cur)

    # -- host-side views --------------------------------------------------------
    def trajectory(self, t):
        """Trajectory t as per-edge arrays: dict child node -> (times from the parent
        end, ascending; states of the k+1 segments, parent side first)."""
        return trajectory_edges(self.ops, self.node_state, self.ev_count, self.ev_total, self.ev_time,
                                self.ev_sb, self.cap, t)
