"""TEST INFRASTRUCTURE -- exact law of the number of real jumps on one branch, for the tests of the
exact posterior draws (rt_posterior_draw).  numpy/scipy only; the product never imports it."""
import numpy as np
import scipy.linalg


def jump_count_distribution(Q, t, K):
    """p[k, a, b] = Pr(k real jumps on (0, t), X_t = b | X_0 = a) for k = 0..K.

    One matrix exponential of the (K+1)S x (K+1)S block-bidiagonal generator that counts jumps:
    diagonal blocks diag(Q) (holding in a state), super-diagonal blocks Q - diag(Q) (a jump moves
    the count up by one); block (0, k) of expm(t G) is p[k].  Exact for every k <= K: the count
    only increases, so truncating above K does not change the blocks below it."""
    Q = np.asarray(Q, dtype=np.float64)
    S = Q.shape[0]
    D = np.diag(np.diag(Q))
    J = Q - D
    G = np.zeros(((K + 1) * S, (K + 1) * S))
    for k in range(K + 1):
        G[k * S:(k + 1) * S, k * S:(k + 1) * S] = D
        if k < K:
            G[k * S:(k + 1) * S, (k + 1) * S:(k + 2) * S] = J
    E = scipy.linalg.expm(t * G)
    return np.stack([E[:S, k * S:(k + 1) * S] for k in range(K + 1)])
