"""
Batched tree-MJP engine: the host side of the hot path.

Lowers (tree, Q, observations) to device tensors (PyTorch owns memory and
streams), then calls the CUDA kernels through the C ABI (include/rt_b200.h).
One `TreeMJP` = one (tree, rate matrices, root prior); its methods take a
whole batch of sites.  The scalar, reference-shaped functions in
raoteh_b200.sampler are thin wrappers over batch size 1.

Reference call stacks replaced (SURVEY.md section 3):
  _mjp_dense.get_likelihood                  raoteh/sampler/_mjp_dense.py:362-407
  _mjp_dense.get_expected_history_statistics raoteh/sampler/_mjp_dense.py:410-539
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native
from .lowering import TreeSchedule, MISSING

OBS_CODES, OBS_MASK, OBS_DENSE, OBS_CODES4 = 0, 1, 2, 3

# compute streams of the site-chunk pipeline (TreeMJP._chunked); chunks take turns: the kernels of
# consecutive chunks are independent, so the tail wave of one chunk's kernel (a chunk is only
# ~1.3-1.7 waves of CTAs) is filled with CTAs of the next chunks' kernels
E2E_STREAMS = 3


def _ptr(t, lo=0):
    """Device address of `t` (None: NULL), or of its site `lo` when the last axis is the site axis."""
    return None if t is None else t.data_ptr() + lo * t.element_size()


def _stream(s=None):
    return (torch.cuda.current_stream() if s is None else s).cuda_stream


def _obs_slot(sched, nodes):
    """Row of the observations per tree node (-1 = unobserved) for observations of `nodes`, in
    order (None: the leaves)."""
    nodes = sched.leaves if nodes is None else np.asarray(nodes)
    obs_slot = np.full(sched.n, -1, dtype=np.int32)
    obs_slot[nodes] = np.arange(len(nodes), dtype=np.int32)
    return obs_slot


def pack_codes4(codes):
    """uint8 codes [n_obs, n_sites] (255 = unobserved) -> RT_OBS_CODES4: two codes per byte, site i in
    nibble i & 1 of byte i >> 1, 15 = unobserved.  For state spaces of at most 8 states (nucleotides):
    halves the bytes that cross PCIe."""
    c = np.ascontiguousarray(codes, dtype=np.uint8)
    if ((c > 14) & (c != MISSING)).any():
        raise ValueError('4-bit codes hold states 0..14')
    c = np.where(c == MISSING, 15, c).astype(np.uint8)
    if c.shape[1] % 2:
        c = np.concatenate([c, np.full((c.shape[0], 1), 15, dtype=np.uint8)], axis=1)
    return np.ascontiguousarray(c[:, 0::2] | (c[:, 1::2] << 4))


def _round_up(x, m):
    return (x + m - 1) // m * m


class Observations(object):
    """Device-resident observations for a batch of sites.

    kind OBS_CODES: data uint8  [n_obs, stride]      (255 = unobserved)
    kind OBS_MASK : data int64  [n_obs, stride]      (bit s set = state s allowed)
    kind OBS_DENSE: data float64[n_obs, S, stride]   (emission likelihoods)
    obs_slot[n_nodes]: row of `data` per tree node, -1 = unobserved node.
    """

    def __init__(self, kind, data, obs_slot, n_sites):
        self.kind = kind
        self.data = data
        self.obs_slot = np.asarray(obs_slot, dtype=np.int32)
        self.n_sites = int(n_sites)
        # site stride of the per-site arrays that go with these observations
        self.stride = int(data.shape[-1]) * (2 if kind == OBS_CODES4 else 1)

    def site_ptr(self, lo):
        """Device address of site `lo` in `data` (every encoding is site-minor; OBS_CODES4 holds
        two sites per byte, so `lo` must be even there)."""
        return self.data.data_ptr() + lo // 2 if self.kind == OBS_CODES4 else _ptr(self.data, lo)

    @classmethod
    def from_leaf_codes(cls, sched, codes, leaf_nodes=None, device='cuda'):
        """codes: uint8 [n_leaves, n_sites] host array (numpy) or device tensor."""
        if isinstance(codes, np.ndarray):
            host = torch.from_numpy(np.ascontiguousarray(codes, dtype=np.uint8))
            data = host.to(device, non_blocking=False)
        else:
            data = codes.to(device=device, dtype=torch.uint8).contiguous()
        return cls(OBS_CODES, data, _obs_slot(sched, leaf_nodes), data.shape[1])

    @classmethod
    def from_leaf_codes4(cls, sched, codes, leaf_nodes=None, device='cuda'):
        """Hard leaf codes stored two per byte (RT_OBS_CODES4, S <= 8)."""
        data = torch.from_numpy(pack_codes4(codes)).to(device)
        return cls(OBS_CODES4, data, _obs_slot(sched, leaf_nodes), codes.shape[1])

    @classmethod
    def from_masks(cls, sched, mask, device='cuda'):
        """mask: uint64 [n_nodes, n_sites]; full-mask rows may be dropped by the caller."""
        mask = np.ascontiguousarray(mask).view(np.int64)
        obs_slot = np.arange(sched.n, dtype=np.int32)
        data = torch.from_numpy(mask).to(device)
        return cls(OBS_MASK, data, obs_slot, data.shape[1])

    @classmethod
    def from_dense(cls, sched, lik, nodes, device='cuda'):
        """lik: float64 [len(nodes), S, n_sites] emission likelihoods of `nodes`."""
        data = torch.from_numpy(np.ascontiguousarray(lik, dtype=np.float64)).to(device)
        return cls(OBS_DENSE, data, _obs_slot(sched, nodes), data.shape[2])


class TreeMJP(object):
    """Markov jump process on a rooted tree, evaluated for batches of sites."""
    _n_made = 0

    def __init__(self, sched, Q, root_distn=None, q_index=None, device='cuda', P=None):
        if not torch.cuda.is_available():
            raise _native.NativeError('raoteh_b200 needs a CUDA device; there is no CPU fallback')
        _native.lib()
        self.sched = sched
        self.device = torch.device(device)
        Q = np.asarray(Q, dtype=np.float64)
        self.Q_host = Q if Q.ndim == 3 else Q[None]
        self.S = int(self.Q_host.shape[-1])
        if self.S < 2 or self.S > 64:
            raise ValueError('number of states must be in 2..64')
        self.q_index_host = None if q_index is None else np.asarray(q_index, dtype=np.int32)
        self.Q = torch.from_numpy(np.ascontiguousarray(self.Q_host)).to(self.device)
        self.q_index = (None if self.q_index_host is None
                        else torch.from_numpy(self.q_index_host).to(self.device))
        self.length = torch.from_numpy(sched.length.copy()).to(self.device)
        self.root_distn_host = None if root_distn is None else np.asarray(root_distn, np.float64)
        self.root_distn = (None if root_distn is None
                           else torch.from_numpy(self.root_distn_host.copy()).to(self.device))
        self.parent = torch.from_numpy(sched.parent.copy()).to(self.device)
        self._P = None
        self._P_valid = False
        if P is not None:   # caller-supplied per-edge transition matrices [n,S,S]
            self._P = torch.from_numpy(np.ascontiguousarray(P, dtype=np.float64)).to(self.device)
            self._P_valid = True
        self._prog_cache = {}
        self._ws = {}
        TreeMJP._n_made += 1
        self._serial = TreeMJP._n_made
        self._Q_stage = None
        self._spectral_D = None     # stationary weights of use_spectral, None = Pade
        self._spectral_dec = None   # (A, lam, B) behind the spectral P
        self._rev_cache = None      # (hash of Q, (A, lam, B) or None): _reversible_decomposition
        self._streams = None        # copy-in, copy-out and E2E_STREAMS compute streams of _chunked
        self._graph_refused = False
        self.events = None     # optional dict: name -> [(start, end) CUDA events]

    def _buf(self, name, shape, dtype, zero=False):
        """Reusable device workspace (avoids per-call allocation)."""
        key = (name, tuple(shape), dtype)
        t = self._ws.get(key)
        if t is None:
            t = torch.empty(shape, dtype=dtype, device=self.device)
            self._ws[key] = t
        if zero:
            t.zero_()
        return t

    def _mark(self, name):
        if self.events is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.events.setdefault(name, []).append(e)
        return e

    def set_rate_matrix(self, Q):
        """New rate matrix/matrices for the same tree (e.g. inside an optimiser
        loop): one small pinned, non-blocking H2D copy; P is recomputed lazily."""
        Q = np.asarray(Q, dtype=np.float64)
        Q = Q if Q.ndim == 3 else Q[None]
        if Q.shape != tuple(self.Q.shape):
            raise ValueError('rate matrix shape changed')
        if self._Q_stage is None:
            self._Q_stage = torch.empty(self.Q.shape, dtype=torch.float64).pin_memory()
        self._Q_stage.copy_(torch.from_numpy(Q))
        self.Q.copy_(self._Q_stage, non_blocking=True)
        self.Q_host = Q
        self._P_valid = False

    def use_spectral(self, D):
        """Switch P(t) to the spectral scheme of examples/p53/qtop.py:76-85 for a time-reversible
        rate matrix with stationary weights `D` (one shared rate matrix only): the symmetric
        eigenproblem is solved on the host whenever the rate matrix changes, the reconstruction
        for all branches is one `rt_expm_spectral` call.  `D=None` goes back to Pade."""
        if D is not None and (self.q_index is not None or self.Q.shape[0] != 1):
            raise ValueError('the spectral scheme needs one shared rate matrix')
        self._spectral_D = None if D is None else np.asarray(D, dtype=np.float64)
        self._P_valid = False

    def _decompose(self, D, rtol):
        """(A, lam, B) on the device, Q = A diag(lam) B (examples/p53/qtop.py:126-148), for the one
        rate matrix; ValueError unless it is time-reversible with respect to the weights `D`."""
        from . import qtop
        S = self.S
        A, lam, B = qtop.decompose_spectral_v2(qtop.symmetric_factor(self.Q_host[0], D, rtol=rtol), D)
        dec = torch.from_numpy(np.concatenate([A.ravel(), lam, B.ravel()])).to(self.device)
        return dec[:S * S].view(S, S), dec[S * S:S * S + S], dec[S * S + S:].view(S, S)

    def _spectral_matrices(self):
        D = self._spectral_D
        self._spectral_dec = A, lam, B = self._decompose(D, rtol=1e-9)
        off = torch.from_numpy((D == 0).astype(np.uint8)).to(self.device)
        rc = _native.lib().rt_expm_spectral(_ptr(A), _ptr(lam), _ptr(B), _ptr(self.length), _ptr(off),
                                            self.sched.n, self.S, _ptr(self._P), _stream())
        _native.check(rc, 'rt_expm_spectral')

    # ---- K1 ---------------------------------------------------------------
    def transition_matrices(self):
        """P[b] = expm(Q_b t_b) for every node b (slot 0 = identity); cached."""
        if not self._P_valid:
            n, S = self.sched.n, self.S
            if self._P is None:
                self._P = torch.empty((n, S, S), dtype=torch.float64, device=self.device)
            if self._spectral_D is not None:
                self._spectral_matrices()
            else:
                rc = _native.lib().rt_expm_batched(_ptr(self.Q), _ptr(self.q_index), _ptr(self.length),
                                                   n, S, _ptr(self._P), _stream())
                _native.check(rc, 'rt_expm_batched')
            self._P_valid = True
        return self._P

    def _programs(self, obs):
        key = obs.obs_slot.tobytes()
        hit = self._prog_cache.get(key)
        if hit is None:
            ops, n_slots = self.sched.up_program(obs.obs_slot)
            edges, level_ptr = self.sched.down_program(obs.obs_slot)
            hit = dict(ops=torch.from_numpy(ops).to(self.device), n_ops=len(ops), n_slots=n_slots,
                       edges=torch.from_numpy(edges).to(self.device),
                       level_ptr=np.ascontiguousarray(level_ptr, dtype=np.int32))
            self._prog_cache[key] = hit
        return hit

    # ---- A4 ---------------------------------------------------------------
    def support_sets(self, mask, passes=3):
        """In-place structural-support pruning of int64 bitmasks [n_nodes, stride];
        passes=1 backward only ("pset"), 3 backward + forward ("set")."""
        P = self.transition_matrices()
        n_sites = mask.shape[1]
        rc = _native.lib().rt_support_sets(self.S, self.sched.n, n_sites, mask.shape[1], passes,
                                           _ptr(self.parent), _ptr(P), _ptr(mask), _stream())
        _native.check(rc, 'rt_support_sets')
        return mask

    # ---- K2 / K3 ------------------------------------------------------------
    def _up(self, obs, prog, lo, hi, stream, loglik, status, partials=None, exponents=None,
            loglik_sum=None):
        """rt_prune_loglik for the sites [lo, hi) of `obs` on `stream` (None: the current one).
        Every per-site array is site-minor, so each pointer is its base + lo * element size.
        P comes from transition_matrices(): a caller that forks streams computes it first."""
        rc = _native.lib().rt_prune_loglik(
            self.S, self.sched.n, hi - lo, obs.stride, _ptr(prog['ops']), prog['n_ops'], prog['n_slots'],
            _ptr(self.transition_matrices()), _ptr(self.root_distn), obs.kind, obs.site_ptr(lo),
            _ptr(partials, lo), _ptr(exponents, lo), _ptr(loglik, lo), _ptr(status, lo),
            _ptr(loglik_sum), _stream(stream))
        _native.check(rc, 'rt_prune_loglik')

    def _down(self, obs, prog, lo, hi, stream, partials, status, node_distn, W, root_post_sum,
              K=None, branch=None, site_weight=None):
        """rt_posterior_stats for the sites [lo, hi) of `obs` on `stream`, addressed as in _up;
        rt_posterior_branch_stats when a per-edge kernel K is given (per-site output `branch`),
        rt_posterior_weighted_stats when per-site weights are given."""
        lp = prog['level_ptr']
        args = (self.S, self.sched.n, hi - lo, obs.stride, _ptr(prog['ops']), prog['n_ops'],
                prog['n_slots'], _ptr(prog['edges']), lp.ctypes.data, len(lp) - 1,
                _ptr(self.transition_matrices()), _ptr(self.root_distn), obs.kind, obs.site_ptr(lo),
                _ptr(partials, lo), _ptr(status, lo), _ptr(node_distn, lo), _ptr(W),
                _ptr(root_post_sum))
        if K is not None:
            name = 'rt_posterior_branch_stats'
            rc = _native.lib().rt_posterior_branch_stats(*args, _ptr(K), _ptr(branch, lo), _stream(stream))
        elif site_weight is not None:
            name = 'rt_posterior_weighted_stats'
            rc = _native.lib().rt_posterior_weighted_stats(*args, _ptr(site_weight, lo), _stream(stream))
        else:
            name = 'rt_posterior_stats'
            rc = _native.lib().rt_posterior_stats(*args, _stream(stream))
        _native.check(rc, name)

    def _check_site_weight(self, site_weight, n_sites):
        """Shape, dtype and device of per-site weights, on the host (no device sync)."""
        if not isinstance(site_weight, torch.Tensor):
            raise TypeError('site_weight must be a torch tensor')
        if site_weight.dtype != torch.float64:
            raise ValueError('site_weight must be float64')
        dev = self.device
        if dev.type == 'cuda' and dev.index is None:
            dev = torch.device('cuda', torch.cuda.current_device())
        if site_weight.device != dev:
            raise ValueError('site_weight must be on %s' % dev)
        if tuple(site_weight.shape) != (n_sites,) or not site_weight.is_contiguous():
            raise ValueError('site_weight must be a contiguous [n_sites] = [%d] tensor' % n_sites)

    @staticmethod
    def _weighted_loglik_sum(loglik, status, site_weight):
        """sum_s w_s * loglik_s over the feasible sites."""
        return (torch.where(status == 0, loglik, torch.zeros_like(loglik)) * site_weight).sum()

    def log_likelihood(self, obs, keep_partials=False, want_exponents=False, out=None,
                       loglik_sum=None):
        """Per-site log-likelihood.  Returns dict(loglik, status[, partials, exponents])."""
        self.transition_matrices()          # before the 'up' event: P is not part of the up pass
        prog = self._programs(obs)
        N, stride = obs.n_sites, obs.stride
        dev = self.device
        if out is None:
            loglik = torch.empty(N, dtype=torch.float64, device=dev)
            status = torch.empty(N, dtype=torch.int8, device=dev)
        else:
            loglik, status = out
        partials = exponents = None
        if keep_partials:
            partials = self._buf('partials', (self.sched.n_store, self.S, stride), torch.float64)
            if want_exponents:
                exponents = self._buf('exponents', (self.sched.n_store, stride), torch.int32)
        self._mark('up')
        self._up(obs, prog, 0, N, None, loglik, status, partials, exponents, loglik_sum)
        self._mark('up')
        res = dict(loglik=loglik, status=status)
        if keep_partials:
            res['partials'] = partials
            res['exponents'] = exponents
        return res

    # ---- K4 / K5 ------------------------------------------------------------
    def _chunked(self, obs, n_chunks, codes_host=None, out_loglik=None, out_status=None,
                 site_weight=None):
        """Up + down pass with the site axis cut into `n_chunks` chunks (multiples of 128 sites) that
        take turns on E2E_STREAMS compute streams.  codes_host: pinned codes in the layout of
        obs.data; the H2D copies of all chunks are enqueued first on the copy-in stream, one event
        per chunk, so chunk k+1 arrives under the kernels of chunk k.  out_loglik / out_status:
        pinned arrays the chunk's log-likelihoods and status go to on the copy-out stream as soon as
        its kernels are done; the caller joins that stream.  Sites are independent and W only
        accumulates, so the chunks need no order among themselves.  Returns the dict of
        `posterior`, without node marginals and exponents."""
        S, n, N = self.S, self.sched.n, obs.n_sites
        prog = self._programs(obs)
        self.transition_matrices()          # on the current stream, before the fork
        loglik = self._buf('h_loglik', (N,), torch.float64)
        status = self._buf('h_status', (N,), torch.int8)
        partials = self._buf('partials', (self.sched.n_store, S, obs.stride), torch.float64)
        W = self._buf('W', (n, S, S), torch.float64, zero=True)
        rps = self._buf('root_post_sum', (S,), torch.float64, zero=True)
        llsum = self._buf('h_llsum', (1,), torch.float64, zero=True)
        cur = torch.cuda.current_stream()
        if self._streams is None:
            self._streams = [torch.cuda.Stream(device=self.device) for _ in range(2 + E2E_STREAMS)]
        s_in, s_out, *compute = self._streams
        for s in self._streams:
            s.wait_stream(cur)
        chunk = _round_up((N + n_chunks - 1) // n_chunks, 128)
        bounds = [(lo, min(N, lo + chunk)) for lo in range(0, N, chunk)]
        ev_in = []
        if codes_host is not None:
            base, (L, row) = obs.data.data_ptr(), obs.data.shape     # uint8 rows of `row` bytes
            for lo, hi in bounds:
                off = obs.site_ptr(lo) - base
                end = obs.site_ptr(hi) - base if hi < N else row     # with an odd last site's byte
                rc = _native.lib().rt_copy2d_async(base + off, row, codes_host.data_ptr() + off, row,
                                                   end - off, L, 1, s_in.cuda_stream)
                _native.check(rc, 'rt_copy2d_async')
                e = torch.cuda.Event()
                e.record(s_in)
                ev_in.append(e)
        for k, (lo, hi) in enumerate(bounds):
            cs = compute[k % E2E_STREAMS]
            if ev_in:
                cs.wait_event(ev_in[k])
            self._up(obs, prog, lo, hi, cs, loglik, status, partials, loglik_sum=llsum)
            self._down(obs, prog, lo, hi, cs, partials, status, None, W, rps, site_weight=site_weight)
            if out_loglik is not None:
                done = torch.cuda.Event()
                done.record(cs)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(done)
                    out_loglik[lo:hi].copy_(loglik[lo:hi], non_blocking=True)
                    out_status[lo:hi].copy_(status[lo:hi], non_blocking=True)
        for cs in compute:
            cur.wait_stream(cs)
        if site_weight is not None:
            llsum = self._weighted_loglik_sum(loglik, status, site_weight).reshape(1)
        return dict(loglik=loglik, status=status, loglik_sum=llsum[0], partials=partials,
                    exponents=None, node_distn=None, W=W, root_post_sum=rps,
                    n_levels=len(prog['level_ptr']) - 1)

    def posterior(self, obs, want_exponents=False, want_node_distn=True, overlap_chunks=0,
                  site_weight=None):
        """Up + down pass.  Returns loglik, status, loglik_sum, partials, node_distn (internal
        nodes, by store index), W[n,S,S] (site-summed J/P weights), root_post_sum[S].
        overlap_chunks > 1 (S <= 8, no node marginals / exponents wanted): the site chunks of the
        host-buffer pipeline, without its copies, see _chunked.
        site_weight: fp64 device tensor [n_sites] of non-negative, finite weights, or None (all
        1).  Site s then counts w_s times in W, root_post_sum and node_distn, and loglik_sum is
        sum_s w_s loglik_s over the feasible sites; per-site loglik and status do not change.
        Integer weights are site-pattern compression (w = columns with the pattern); class
        posteriors give the E-step of a site-class mixture (raoteh_b200.mixture)."""
        if site_weight is not None:
            self._check_site_weight(site_weight, obs.n_sites)
        if overlap_chunks > 1 and self.S <= 8 and not want_node_distn and not want_exponents:
            return self._chunked(obs, int(overlap_chunks), site_weight=site_weight)
        llsum = self._buf('loglik_sum', (1,), torch.float64, zero=True)
        up = self.log_likelihood(obs, keep_partials=True, want_exponents=want_exponents,
                                 loglik_sum=llsum)
        up['loglik_sum'] = llsum[0]      # sum of the finite log-likelihoods, reduced by the kernel
        if site_weight is not None:
            up['loglik_sum'] = self._weighted_loglik_sum(up['loglik'], up['status'], site_weight)
        prog = self._programs(obs)
        node_distn = None
        if want_node_distn or self.S > 8:
            node_distn = self._buf('node_distn', (self.sched.n_store, self.S, obs.stride), torch.float64)
        W = self._buf('W', (self.sched.n, self.S, self.S), torch.float64, zero=True)
        root_post_sum = self._buf('root_post_sum', (self.S,), torch.float64, zero=True)
        self._mark('down')
        self._down(obs, prog, 0, obs.n_sites, None, up['partials'], up['status'], node_distn, W,
                   root_post_sum, site_weight=site_weight)
        self._mark('down')
        up.update(node_distn=node_distn, W=W, root_post_sum=root_post_sum,
                  n_levels=len(prog['level_ptr']) - 1)
        return up

    def _edge_rates(self):
        """Q_b for every node b: [n, S, S]."""
        n, S = self.sched.n, self.S
        return self.Q[0].expand(n, S, S) if self.q_index is None else self.Q[self.q_index.long()]

    def _frechet(self, Q, W, M):
        """M[b] = L(t_b Q_b^T, t_b W[b]) for every node b, Q_b = Q[q_index[b]]."""
        rc = _native.lib().rt_frechet_contract(_ptr(Q), _ptr(self.q_index), _ptr(self.length), _ptr(W),
                                               self.sched.n, self.S, _ptr(M), _stream())
        _native.check(rc, 'rt_frechet_contract')
        return M

    def transition_kernels(self, E=None):
        """K_b = L(t_b Q_b, t_b (E o Q_b)) for every edge: K_b[a, c] = expected number of E-type
        transitions on the branch jointly with the end state c, from the start state a
        (the Frechet-derivative form of examples/code2x3/extras.py:108-129)."""
        n, S = self.sched.n, self.S
        off = 1.0 - torch.eye(S, dtype=torch.float64, device=self.device)
        if E is None:
            Et = off
        else:
            Et = torch.as_tensor(np.asarray(E, dtype=np.float64), device=self.device) * off
        C = (self._edge_rates() * Et).contiguous()
        K = torch.empty((n, S, S), dtype=torch.float64, device=self.device)
        self._frechet(self.Q.transpose(1, 2).contiguous(), C, K)
        K[0].zero_()
        return K

    def branch_expectations(self, obs, E=None, K=None):
        """Per SITE and BRANCH posterior expectation of the number of E-type transitions
        (E: S x S 0/1 or weight mask, default all off-diagonal pairs) -> dict with
        'branch' [n_nodes, n_sites] (row of the child node; root row zero), 'loglik', 'status'.
        Batched form of examples/code2x3/extras.py:19-132 and of the per-branch tables of
        examples/p53/liwen-branch-expectation.py:176-356."""
        if K is None:
            K = self.transition_kernels(E)
        up = self.log_likelihood(obs, keep_partials=True)
        prog = self._programs(obs)
        N, stride = obs.n_sites, obs.stride
        node_distn = None
        if self.S > 8:
            node_distn = self._buf('node_distn', (self.sched.n_store, self.S, stride), torch.float64)
        W = self._buf('W', (self.sched.n, self.S, self.S), torch.float64, zero=True)
        rps = self._buf('root_post_sum', (self.S,), torch.float64, zero=True)
        branch = torch.zeros((self.sched.n, stride), dtype=torch.float64, device=self.device)
        self._down(obs, prog, 0, N, None, up['partials'], up['status'], node_distn, W, rps, K, branch)
        return dict(branch=branch[:, :N], loglik=up['loglik'], status=up['status'], W=W,
                    root_post_sum=rps, K=K)

    def posterior_given_partials(self, obs, partials, status=None):
        """Downward pass for caller-supplied partials of the internal nodes
        ([n_store, S, stride]; leaves come from `obs`): the batched form of
        _mc0_dense.get_node_to_distn (raoteh/sampler/_mc0_dense.py:400), whose input
        is a node_to_pmap rather than observations."""
        prog = self._programs(obs)
        N, stride = obs.n_sites, obs.stride
        if status is None:
            status = torch.zeros(N, dtype=torch.int8, device=self.device)
        node_distn = self._buf('node_distn', (self.sched.n_store, self.S, stride), torch.float64)
        W = self._buf('W', (self.sched.n, self.S, self.S), torch.float64, zero=True)
        root_post_sum = self._buf('root_post_sum', (self.S,), torch.float64, zero=True)
        self._down(obs, prog, 0, N, None, partials, status, node_distn, W, root_post_sum)
        return dict(partials=partials, status=status, node_distn=node_distn, W=W,
                    root_post_sum=root_post_sum)

    def joint_distn(self, obs, post):
        """Materialised joints J[n, N, S, S] and marginals of every node D[n, N, S]
        (row 0 of D = root posterior) from the result of `posterior`."""
        prog = self._programs(obs)
        n, S, N = self.sched.n, self.S, obs.n_sites
        J = torch.zeros((n, N, S, S), dtype=torch.float64, device=self.device)
        D = torch.zeros((n, N, S), dtype=torch.float64, device=self.device)
        rc = _native.lib().rt_joint_distn(
            S, n, N, obs.stride, _ptr(prog['edges']), n - 1, _ptr(self.transition_matrices()),
            obs.kind, _ptr(obs.data), _ptr(post['partials']), _ptr(post['node_distn']),
            _ptr(post['status']), _ptr(J), _ptr(D), _stream())
        _native.check(rc, 'rt_joint_distn')
        D[0] = post['node_distn'][0, :, :N].T
        return J, D

    # ---- host-buffer entry point (pipelined) ----------------------------------------
    def expected_history_statistics_from_host(self, codes_pinned, leaf_nodes, out_loglik,
                                              out_status, n_chunks=4, packed=False):
        """The C2 evaluation from HOST buffers: uint8 leaf codes [n_leaves, n_sites] in
        pinned memory in, per-site log-likelihoods / status into pinned `out_*`, summed
        statistics returned.  The site axis is cut into `n_chunks` chunks; the H2D copy
        of chunk k+1 and the D2H copy of chunk k-1 run on their own streams under the
        kernels of chunk k (sites are independent, W only accumulates; see _chunked)."""
        # packed=True: codes_pinned is RT_OBS_CODES4 (pack_codes4), N = len(out_loglik) sites
        N = int(out_loglik.shape[0]) if packed else codes_pinned.shape[1]
        codes_dev = self._buf('h_codes', tuple(codes_pinned.shape), torch.uint8)
        obs = Observations(OBS_CODES4 if packed else OBS_CODES, codes_dev,
                           _obs_slot(self.sched, leaf_nodes), N)
        r = self._chunked(obs, n_chunks, codes_pinned, out_loglik, out_status)
        M, dwell, trans = self.history_statistics(r['W'])
        torch.cuda.current_stream().wait_stream(self._streams[1])    # the D2H copies
        return dict(loglik_sum=r['loglik_sum'], dwell=dwell, trans=trans,
                    root_post_sum=r['root_post_sum'], M_edges=M)

    def history_statistics(self, W):
        """(M_edges, dwell, trans) from the per-edge weights W: one Frechet contraction per edge
        and the accumulation over edges, one library call (rt_history_statistics;
        raoteh/sampler/_mjp_dense.py:497-533), or the same contraction in an eigenbasis of the
        rate matrix where _eigenbasis gives one."""
        dec = self._eigenbasis()
        if dec is not None:
            return self._history_statistics_spectral(W, dec)
        n, S = self.sched.n, self.S
        M = self._buf('M', (n, S, S), torch.float64)
        dwell = torch.empty(S, dtype=torch.float64, device=self.device)
        trans = torch.empty((S, S), dtype=torch.float64, device=self.device)
        rc = _native.lib().rt_history_statistics(_ptr(self.Q), _ptr(self.q_index), _ptr(self.length),
                                                 _ptr(W), n, 1, S, _ptr(M), _ptr(dwell), _ptr(trans),
                                                 _stream())
        _native.check(rc, 'rt_history_statistics')
        return M, dwell, trans

    def _eigenbasis(self):
        """(A, lam, B) for history_statistics, or None (Pade): the use_spectral decomposition when
        no state has zero weight; otherwise, for S > 16, the decomposition of a rate matrix that is
        time-reversible w.r.t. the root distribution, so that the edge weights are contracted in
        its eigenbasis instead of exponentiating a 2S x 2S block per edge."""
        D = self._spectral_D
        if D is not None and self._P_valid and not (D == 0).any():
            return self._spectral_dec
        if self.S > 16:
            return self._reversible_decomposition()
        return None

    def _reversible_decomposition(self):
        """(A, lam, B) on the device if the (single) rate matrix is time-reversible with respect to
        the root distribution and every state has positive weight, else None; cached per rate
        matrix.  Used for the Frechet contraction of large state spaces (codon models are
        reversible): the check is S^2 host work, the symmetric eigenproblem ~0.5 ms at S = 61."""
        key = hash(self.Q_host.tobytes())
        if self._rev_cache is None or self._rev_cache[0] != key:
            dec = None
            D = self.root_distn_host
            if D is not None and self.q_index is None and self.Q_host.shape[0] == 1 and (D > 0).all():
                try:
                    dec = self._decompose(D, rtol=1e-10)
                except ValueError:
                    pass
            self._rev_cache = (key, dec)
        return self._rev_cache[1]

    def _history_statistics_spectral(self, W, dec):
        """The same contraction in the eigenbasis of a time-reversible rate matrix (spectral scheme,
        use_spectral): with Q = A diag(lam) B, B = A^-1 (examples/p53/qtop.py:140-148),
            L(t Q^T, t W) = B^T [Phi(t) o (A^T (t W) B^T)] A^T,
            Phi_ij(t) = (e^{t lam_i} - e^{t lam_j}) / (t (lam_i - lam_j))   (e^{t lam_i} on the diagonal),
        four batched S x S products per edge (plain library GEMMs) instead of the Pade exponential
        of a 2S x 2S block matrix per edge: 0.3 ms instead of 4.0 ms for the 254 edges of C3."""
        A, lam, B = dec
        t = self.length[:, None, None]
        x = lam[None, :, None] * t                 # t lam_i
        y = lam[None, None, :] * t                 # t lam_j
        d = x - y
        small = d.abs() < 1e-9
        # (e^x - e^y) / (x - y) = e^y expm1(x - y) / (x - y); -> e^y (1 + d/2) where x ~ y
        phi = torch.where(small, torch.exp(y) * (1.0 + 0.5 * d),
                          torch.exp(y) * torch.expm1(d) / torch.where(small, torch.ones_like(d), d))
        At, Bt = A.T.contiguous(), B.T.contiguous()
        inner = torch.matmul(torch.matmul(At, W * t), Bt)
        M = torch.matmul(torch.matmul(Bt, phi * inner), At)
        M[0].zero_()
        Ms = M[1:].sum(dim=0)
        dwell = torch.diagonal(Ms).clone()
        Q0 = self.Q[0]
        trans = Q0 * Ms
        trans.fill_diagonal_(0.0)
        return M, dwell, trans

    def frechet_contract(self, W):
        """M[b] = L(t_b Q_b^T, t_b W[b]) for every node b (slot 0 -> 0)."""
        return self._frechet(self.Q, W, self._buf('M', (self.sched.n, self.S, self.S), torch.float64))

    def expected_history_statistics_graphed(self, obs):
        """expected_history_statistics for a NEW rate matrix (set_rate_matrix) replayed as one
        CUDA graph: batched expm, up pass, down walk, Frechet contraction and the packing of the
        statistics are ~13 small launches, and for a few hundred thousand sites per GPU (strong
        scaling, optimiser loops) the host cannot issue them as fast as the GPU runs them.
        Captured once per (engine, observations) -- the graph lives on the Observations object --
        and replayed afterwards; the H2D copy of the rate matrix stays
        outside (stream ordered before the replay).  Returns the same dict (static tensors, valid
        until the next call) plus 'stats' = the packed [1 + S + S*S + S] vector for the allreduce.
        Falls back to the eager path if the capture is refused."""
        cache = obs.__dict__.setdefault('_rt_graphs', {})
        prog = self._programs(obs)
        key = ('ehs', self._serial, obs.kind, obs.data.data_ptr(), obs.n_sites, obs.stride,
               _ptr(self.root_distn), prog['ops'].data_ptr())
        entry = cache.get(key)
        if entry is None:
            if self._graph_refused:
                return self._ehs_with_stats(obs)
            self._P_valid = False
            self._ehs_with_stats(obs)                 # eager once: workspaces, pool growth
            torch.cuda.synchronize()
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._P_valid = False
                    out = self._ehs_with_stats(obs)
                entry = (g, out)
                cache[key] = entry
            except Exception:
                self._graph_refused = True
                torch.cuda.synchronize()
                self._P_valid = False
                return self._ehs_with_stats(obs)
        g, out = entry
        g.replay()
        self._P_valid = True
        return out

    def _ehs_with_stats(self, obs):
        r = self.expected_history_statistics(obs)
        r['stats'] = torch.cat([r['loglik_sum'].reshape(1), r['dwell'].reshape(-1), r['trans'].reshape(-1),
                                r['root_post_sum'].reshape(-1)])
        return r

    def expected_history_statistics(self, obs, want_node_distn=False, overlap_chunks=0,
                                    site_weight=None):
        """Site-summed expected dwell[S], transition counts[S,S], root posterior sum[S],
        per-site loglik, per-edge contraction matrices M_edges[n,S,S].

        dwell[c] = sum_b M_b[c,c]; trans[c,d] = Q_b[c,d] * M_b[c,d] summed over
        edges (raoteh/sampler/_mjp_dense.py:497-533 with one Frechet derivative per
        edge, the form of examples/code2x3/extras.py:108-129).
        site_weight: per-site weights of the sums, as in `posterior`."""
        post = self.posterior(obs, want_node_distn=want_node_distn, overlap_chunks=overlap_chunks,
                              site_weight=site_weight)
        M, dwell, trans = self.history_statistics(post['W'])
        post.update(dwell=dwell, trans=trans, M_edges=M, Q_edges=self._edge_rates())
        return post
