"""TEST INFRASTRUCTURE -- reference of site-class mixtures (raoteh_b200.mixture), numpy/scipy only.

Per class k (rate matrix Q_k, rate r_k, prior weight w_k) the single-class references run on the
branch lengths r_k t: range_oracle.log_likelihood for the per-site log-likelihood and
np_oracle.expected_history_statistics(..., per_site=True) for the per-site statistics.  Those are
then combined site by site with the class posteriors
    class_post[k](s) = w_k L_k(s) / sum_j w_j L_j(s),
so no weight ever enters a down pass here.  Dwell times of class k are divided by r_k (tree time);
a rate-0 class dwells sum_b t_b per unit of root posterior and makes no transitions."""
import numpy as np
from scipy.special import logsumexp

from oracle import np_oracle
import range_oracle


def subset(obs, idx):
    """The np_oracle.Obs of the sites `idx` of `obs`."""
    if obs.kind == 'codes':
        return np_oracle.Obs('codes', obs.S, len(idx), leaf_nodes=obs.leaf_nodes, codes=obs.codes[:, idx])
    if obs.kind == 'mask':
        return np_oracle.Obs('mask', obs.S, len(idx), mask=obs.mask[:, idx])
    return np_oracle.Obs('dense', obs.S, len(idx), lik=obs.lik[:, idx], has=obs.has)


def mixture(parent, lengths, Qs, rates, weights, obs, root_distn, site_weight=None, E=None,
            node_distn=False):
    """dict(loglik[N], status[N] (0 feasible in some class, else 1), loglik_class[K,N],
    class_post[K,N], loglik_sum, dwell[S], trans[S,S], root_post_sum[S], dwell_class[K,S],
    trans_class[K,S,S], class_post_sum[K]) and, with node_distn, the mixture node marginals
    node_distn[n,N,S] and branch[n,N] (expected E-type transitions per branch and site)."""
    K, N = len(rates), obs.N
    lengths = np.asarray(lengths, float)
    sw = np.ones(N) if site_weight is None else np.asarray(site_weight, float)
    ll = np.full((K, N), -np.inf)
    per = []
    for k in range(K):
        tk = rates[k] * lengths
        Pk = np_oracle.expm_edges(Qs[k], tk)
        ll_k, st_k, _ = range_oracle.log_likelihood(parent, Pk, obs, root_distn)
        ok = np.flatnonzero(st_k == 0)
        ll[k, ok] = ll_k[ok]
        per.append((tk, Pk, ok))
    lw = np.log(np.asarray(weights, float))[:, None] + ll
    feasible = np.isfinite(lw).any(axis=0)
    loglik = np.full(N, -np.inf)
    loglik[feasible] = logsumexp(lw[:, feasible], axis=0)
    cp = np.zeros((K, N))
    cp[:, feasible] = np.exp(lw[:, feasible] - loglik[feasible])
    S = Qs[0].shape[0]
    n = len(parent)
    dwell_c, trans_c, rps_c = np.zeros((K, S)), np.zeros((K, S, S)), np.zeros((K, S))
    nd = np.zeros((n, N, S)) if node_distn else None
    branch = np.zeros((n, N)) if node_distn else None
    for k, (tk, Pk, ok) in enumerate(per):
        if not len(ok):
            continue
        r = np_oracle.expected_history_statistics(parent, tk, Qs[k], Pk, subset(obs, ok), root_distn,
                                                  per_site=True)
        c = cp[k, ok] * sw[ok]
        rps_c[k] = c @ r['root_post']
        if rates[k] > 0:
            dwell_c[k] = c @ r['dwell'] / rates[k]
            trans_c[k] = np.einsum('s,scd->cd', c, r['trans'])
        else:
            dwell_c[k] = lengths[1:].sum() * rps_c[k]
        if node_distn:
            Kb = range_oracle.transition_kernels(Qs[k], tk, E)
            p = range_oracle.posterior(parent, tk, Qs[k], Pk, obs, root_distn, K=Kb)
            nd += (cp[k] * sw)[None, :, None] * p['node_distn']
            branch += cp[k][None, :] * p['branch']
    status = np.where(feasible, 0, 1).astype(np.int8)
    out = dict(loglik=loglik, status=status, loglik_class=ll, class_post=cp,
               loglik_sum=float((sw * np.where(feasible, loglik, 0.0)).sum()),
               dwell=dwell_c.sum(axis=0), trans=trans_c.sum(axis=0), root_post_sum=rps_c.sum(axis=0),
               dwell_class=dwell_c, trans_class=trans_c, class_post_sum=(cp * sw).sum(axis=1))
    if node_distn:
        out.update(node_distn=nd, branch=branch)
    return out
