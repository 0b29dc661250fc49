"""CPU oracle for the NMF coordinate-descent and NNDSVD EXTENSION stage.  TEST INFRASTRUCTURE ONLY.

Beside oracle/nmf_oracle.py (the MU solver), a numpy restatement of what scikit-learn executes for its default
solver="cd" with shuffle=False and no regularisation (sklearn/decomposition/_nmf.py: _fit_coordinate_descent,
_update_coordinate_descent; _cdnmf_fast.pyx: _update_cdnmf_fast), which tests/test_nmf_cd_oracle.py pins against
sklearn bit for bit in float64, and of _initialize_nmf(init="nndsvd" / "nndsvda") on an exact SVD
(np.linalg.svd) instead of sklearn's randomized one - the device computes exact singular triplets too.
"""
import numpy as np


def _sweep(X, W, Ht):
    """_update_coordinate_descent(X, W, Ht): one cyclic pass over the columns of W, in place; returns the violation.

    The Cython loop is t-outer, i-inner, and row i's gradient only reads row i of W, so each column t is updated for
    all rows at once with the same products in the same order; the violation is accumulated sequentially (cumsum)."""
    HHt = np.dot(Ht.T, Ht)
    XHt = X @ Ht
    violation = 0.0
    for t in range(W.shape[1]):
        grad = -XHt[:, t]
        for r in range(W.shape[1]):
            grad = grad + HHt[t, r] * W[:, r]
        pg = np.where(W[:, t] == 0, np.minimum(0.0, grad), grad)
        violation = np.cumsum(np.concatenate([[violation], np.abs(pg)]))[-1]
        hess = HHt[t, t]
        if hess != 0:
            W[:, t] = np.maximum(W[:, t] - grad / hess, 0.0)
    return violation


def cd(X, W, H, max_iter=200, tol=1e-4):
    """Returns (W, H, n_iter) after sklearn's coordinate-descent loop (float64)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.ascontiguousarray(W, dtype=np.float64).copy()
    Ht = np.ascontiguousarray(np.asarray(H, dtype=np.float64).T).copy()
    violation_init = 0.0
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        violation = 0.0
        violation += _sweep(X, W, Ht)
        violation += _sweep(X.T, Ht, W)
        if n_iter == 1:
            violation_init = violation
        if violation_init == 0:
            break
        if violation / violation_init <= tol:
            break
    return W, Ht.T, n_iter


def nndsvd_exact(X, k, variant="nndsvda", eps=1e-6):
    """_initialize_nmf(X, k, init=variant) with the singular triplets of an exact SVD."""
    X = np.asarray(X, dtype=np.float64)
    U, S, Vt = np.linalg.svd(X, full_matrices=False)
    U, S, V = U[:, :k], S[:k], Vt[:k]
    W = np.zeros((X.shape[0], k))
    H = np.zeros((k, X.shape[1]))
    W[:, 0] = np.sqrt(S[0]) * np.abs(U[:, 0])
    H[0, :] = np.sqrt(S[0]) * np.abs(V[0, :])
    for j in range(1, k):
        x, y = U[:, j], V[j, :]
        x_p, y_p = np.maximum(x, 0), np.maximum(y, 0)
        x_n, y_n = np.abs(np.minimum(x, 0)), np.abs(np.minimum(y, 0))
        x_p_nrm, y_p_nrm = np.linalg.norm(x_p), np.linalg.norm(y_p)
        x_n_nrm, y_n_nrm = np.linalg.norm(x_n), np.linalg.norm(y_n)
        m_p, m_n = x_p_nrm * y_p_nrm, x_n_nrm * y_n_nrm
        if m_p > m_n:
            u, v, sigma = x_p / x_p_nrm, y_p / y_p_nrm, m_p
        else:
            u, v, sigma = x_n / x_n_nrm, y_n / y_n_nrm, m_n
        lbd = np.sqrt(S[j] * sigma)
        W[:, j] = lbd * u
        H[j, :] = lbd * v
    W[W < eps] = 0
    H[H < eps] = 0
    if variant == "nndsvda":
        avg = X.mean()
        W[W == 0] = avg
        H[H == 0] = avg
    elif variant != "nndsvd":
        raise ValueError(variant)
    return W, H
