"""TEST INFRASTRUCTURE -- log-space reference of the tree passes, for inputs at the edges of the
kernels' range: wide polytomies, badly scaled emission rows, near-zero transition probabilities.
numpy/scipy only; the product never imports it.

np_oracle.prune multiplies all of a node's child messages into one accumulator and rescales once
per node, the same structure as the kernels, so it underflows where they do.  Here the upward pass
runs in log space,
    log L_v[a] = log obs_v[a] + sum_c logsumexp_b(log P_c[a, b] + log L_c[b]),
which forms no product that can underflow.  The per-node partials, normalised to a maximum of 1,
then go to np_oracle's scale-invariant down pass and edge weights (node_distn,
edge_weight_matrices, _finish_ehs), which divide in IEEE arithmetic.

Conventions as np_oracle: nodes 0..n-1 in preorder, per-edge matrices indexed by the child node,
observations an np_oracle.Obs (codes, mask or dense; observed internal nodes allowed)."""
import numpy as np
import scipy.linalg
from scipy.special import logsumexp

from oracle import np_oracle


def _log(x):
    with np.errstate(divide='ignore'):
        return np.log(x)


def log_partials(parent, P, obs):
    """logL[n, N, S]: log of the true (unscaled) partial likelihoods of every node."""
    n = len(parent)
    N, S = obs.N, P.shape[-1]
    logP = _log(P)
    logL = np.zeros((n, N, S))
    for a in range(n - 1, -1, -1):
        e = obs.emission(a)
        if e is not None:
            logL[a] += _log(np.asarray(e, dtype=float))
        if a > 0:
            # msg[i, x] = logsumexp_y(logP[x, y] + logL_a[i, y]); all -inf gives -inf
            with np.errstate(invalid='ignore'):
                msg = logsumexp(logP[a][None, :, :] + logL[a][:, None, :], axis=2)
            logL[parent[a]] += msg
    return logL


def normalized(logL):
    """Partials scaled to a maximum of 1 per node and site (all-zero rows stay zero)."""
    mx = logL.max(axis=-1, keepdims=True)
    with np.errstate(invalid='ignore'):
        L = np.exp(logL - np.where(np.isfinite(mx), mx, 0.0))
    return np.where(np.isfinite(mx), L, 0.0)


def log_likelihood(parent, P, obs, root_distn=None):
    """(loglik[N], status[N], logL): status 1 (loglik -inf) where the likelihood is exactly 0."""
    S = P.shape[-1]
    logL = log_partials(parent, P, obs)
    pi = np.ones(S) if root_distn is None else np.asarray(root_distn, float)
    ll = logsumexp(logL[0] + _log(pi)[None, :], axis=1)
    status = (~np.isfinite(ll)).astype(np.int8)
    ll[status == 1] = -np.inf
    return ll, status, logL


def transition_kernels(Q, lengths, E=None, q_index=None):
    """K_b = L(t_b Q_b, t_b (E o Q_b)) per edge (slot 0 zero), as TreeMJP.transition_kernels."""
    Q = np.asarray(Q, float)
    n = len(lengths)
    S = Q.shape[-1]
    off = np.ones((S, S)) - np.eye(S)
    E = off if E is None else np.asarray(E, float) * off
    K = np.zeros((n, S, S))
    for b in range(1, n):
        Qb = Q if Q.ndim == 2 else Q[q_index[b]]
        K[b] = scipy.linalg.expm_frechet(lengths[b] * Qb, lengths[b] * (E * Qb), compute_expm=False)
    return K


def posterior(parent, lengths, Q, P, obs, root_distn=None, q_index=None, K=None):
    """Everything the kernels report for a batch of sites, computed through log space.

    Returns dict(loglik[N], status[N], loglik_sum, dwell[S], trans[S,S], root_post[N,S] (0 on
    infeasible sites), root_post_sum[S], M_edges[n,S,S], W[n,S,S], node_distn[n,N,S]) and, when
    per-edge kernels K are given, branch[n,N] = sum_ac G_b[a] K_b[a,c] L_b[c] (posterior expectation
    of the statistic of K on each branch and site; 0 on infeasible sites and the root row)."""
    n = len(parent)
    S = P.shape[-1]
    N = obs.N
    ll, status, logL = log_likelihood(parent, P, obs, root_distn)
    ok = status == 0
    L = normalized(logL[:, ok])
    D, G = np_oracle.node_distn(parent, P, L, root_distn)
    W = np_oracle.edge_weight_matrices(parent, P, L, G)
    r = np_oracle._finish_ehs(parent, lengths, np.asarray(Q, float), q_index, W, D[0], ll[ok])
    root_post = np.zeros((N, S))
    root_post[ok] = D[0]
    node_distn = np.zeros((n, N, S))
    node_distn[:, ok] = D
    out = dict(loglik=ll, status=status, loglik_sum=float(ll[ok].sum()), dwell=r['dwell'],
               trans=r['trans'], root_post=root_post, root_post_sum=D[0].sum(axis=0),
               M_edges=r['M_edges'], W=W, node_distn=node_distn, logL=logL)
    if K is not None:
        branch = np.zeros((n, N))
        for b in range(1, n):
            branch[b, ok] = np.einsum('ia,ac,ic->i', G[b], K[b], L[b])
        out['branch'] = branch
    return out
