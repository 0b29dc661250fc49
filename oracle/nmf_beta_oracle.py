"""CPU oracle for β-divergence NMF by multiplicative updates (fit and transform).  TEST INFRASTRUCTURE ONLY.

A numpy restatement of what scikit-learn 1.9.0 executes for `NMF(solver="mu", beta_loss=beta)` with beta != 2 and no
regularisation, dense X (sklearn/decomposition/_nmf.py: _beta_divergence, _multiplicative_update_w,
_multiplicative_update_h, _fit_multiplicative_update), with update_H on (fit) or off (transform, W starting at
sqrt(X.mean() / k)).  tests/test_nmf_beta_oracle.py pins it against sklearn bit for bit in float64.
"""
import numpy as np

EPSILON = np.finfo(np.float32).eps  # sklearn's EPSILON
_NAMES = {"frobenius": 2, "kullback-leibler": 1, "itakura-saito": 0}


def beta_to_float(beta):
    return float(_NAMES[beta]) if isinstance(beta, str) else float(beta)


def gamma_of(beta):
    """The exponent of the Maximization-Minimization update (Fevotte & Idier 2011)."""
    if beta < 1:
        return 1.0 / (2.0 - beta)
    if beta > 2:
        return 1.0 / (beta - 1.0)
    return 1.0


def beta_divergence(X, W, H, beta):
    """_beta_divergence(X, W, H, beta, square_root=True), dense X, beta != 2."""
    WH = np.dot(W, H)
    WH_data = WH.ravel()
    X_data = X.ravel()
    keep = X_data > EPSILON  # the X terms drop X <= EPSILON, zeros included
    WH_data = WH_data[keep]
    X_data = X_data[keep]
    WH_data[WH_data < EPSILON] = EPSILON
    if beta == 1:
        sum_WH = np.dot(np.sum(W, axis=0), np.sum(H, axis=1))
        div = X_data / WH_data
        res = np.dot(X_data, np.log(div))
        res += sum_WH - X_data.sum()
    elif beta == 0:
        div = X_data / WH_data
        res = np.sum(div) - np.prod(X.shape) - np.sum(np.log(div))
    else:
        sum_WH_beta = np.sum(WH**beta)
        sum_X_WH = np.dot(X_data, WH_data ** (beta - 1))
        res = (X_data**beta).sum() - beta * sum_X_WH
        res += sum_WH_beta * (beta - 1)
        res /= beta * (beta - 1)
    res = max(res, 0)
    return np.sqrt(2 * res)


def _ratio_terms(X, W, H, beta):
    """X * WHs^(beta - 2) and the denominator's WHd^(beta - 1) (None for KL), as the W and H steps form them."""
    WH_safe_X = np.dot(W, H)
    WH = WH_safe_X.copy()
    if beta - 1.0 < 0:
        WH[WH < EPSILON] = EPSILON
    if beta - 2.0 < 0:
        WH_safe_X[WH_safe_X < EPSILON] = EPSILON
    if beta == 1:
        np.divide(X, WH_safe_X, out=WH_safe_X)
    elif beta == 0:
        WH_safe_X **= -1
        WH_safe_X **= 2
        WH_safe_X *= X
    else:
        WH_safe_X **= beta - 2
        WH_safe_X *= X
    if beta == 1:
        return WH_safe_X, None
    WH **= beta - 1
    return WH_safe_X, WH


def update_w(X, W, H, beta, gamma, H_sum=None):
    """_multiplicative_update_w (beta != 2); returns (W, H_sum)."""
    F, G = _ratio_terms(X, W, H, beta)
    numerator = np.dot(F, H.T)
    if beta == 1:
        if H_sum is None:
            H_sum = np.sum(H, axis=1)
        denominator = H_sum[np.newaxis, :]
    else:
        denominator = np.dot(G, H.T)
    denominator[denominator == 0] = EPSILON
    numerator /= denominator
    delta_W = numerator
    if gamma != 1:
        delta_W **= gamma
    W *= delta_W
    return W, H_sum


def update_h(X, W, H, beta, gamma):
    """_multiplicative_update_h (beta != 2)."""
    F, G = _ratio_terms(X, W, H, beta)
    numerator = np.dot(W.T, F)
    if beta == 1:
        W_sum = np.sum(W, axis=0)
        W_sum[W_sum == 0] = 1.0
        denominator = W_sum[:, np.newaxis]
    else:
        denominator = np.dot(W.T, G)
    denominator[denominator == 0] = EPSILON
    delta_H = numerator
    delta_H /= denominator
    if gamma != 1:
        delta_H **= gamma
    H *= delta_H
    return H


def fit(X, W, H, beta_loss, max_iter=200, tol=1e-4, update_H=True):
    """_fit_multiplicative_update from (W, H), beta_loss != 2; returns (W, H, n_iter).  update_H=False is the
    transform loop (pass W = sqrt(X.mean() / k) everywhere, as sklearn starts it)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.array(W, dtype=np.float64)
    H = np.array(H, dtype=np.float64)
    beta = beta_to_float(beta_loss)
    gamma = gamma_of(beta)
    error_at_init = beta_divergence(X, W, H, beta)
    previous_error = error_at_init
    H_sum = None
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        W, H_sum = update_w(X, W, H, beta, gamma, H_sum)
        if beta < 1:
            W[W < np.finfo(np.float64).eps] = 0.0
        if update_H:
            H = update_h(X, W, H, beta, gamma)
            H_sum = None
            if beta <= 1:
                H[H < np.finfo(np.float64).eps] = 0.0
        if tol > 0 and n_iter % 10 == 0:
            error = beta_divergence(X, W, H, beta)
            with np.errstate(invalid="ignore", divide="ignore"):
                if (previous_error - error) / error_at_init < tol:
                    break
            previous_error = error
    return W, H, n_iter


def transform(X, H, beta_loss, max_iter=200, tol=1e-4):
    """sklearn's NMF(solver="mu", beta_loss=...).transform: returns (W, n_iter)."""
    X = np.asarray(X, dtype=np.float64)
    W0 = np.full((X.shape[0], H.shape[0]), np.sqrt(X.mean() / H.shape[0]))
    W, _, n_iter = fit(X, W0, H, beta_loss, max_iter, tol, update_H=False)
    return W, n_iter
