"""CPU oracle for NMF.transform (activations fitted to fixed synergies).  TEST INFRASTRUCTURE ONLY.

A numpy restatement of what scikit-learn 1.9.0 executes for `NMF.transform(X)`, i.e.
`_fit_transform(X, H=components_, update_H=False)` (sklearn/decomposition/_nmf.py), with no regularisation:
solver="cd" (_fit_coordinate_descent with W = 0; the sweep is oracle/nmf_cd_oracle.py's) and solver="mu"
(_fit_multiplicative_update, beta_loss=2, W = sqrt(X.mean() / k)).  tests/test_nmf_transform_oracle.py pins both
against sklearn bit for bit in float64.
"""
import numpy as np

from .nmf_cd_oracle import _sweep

EPSILON = np.finfo(np.float32).eps  # sklearn's EPSILON


def transform_cd(X, H, max_iter=200, tol=1e-4):
    """Returns (W, n_iter)."""
    X = np.asarray(X, dtype=np.float64)
    W = np.zeros((X.shape[0], H.shape[0]))
    Ht = np.ascontiguousarray(np.asarray(H, dtype=np.float64).T)
    violation_init = 0.0
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        violation = 0.0
        violation += _sweep(X, W, Ht)
        if n_iter == 1:
            violation_init = violation
        if violation_init == 0:
            break
        if violation / violation_init <= tol:
            break
    return W, n_iter


def frobenius(X, W, H):
    """_beta_divergence(X, W, H, 2, square_root=True)."""
    R = (X - np.dot(W, H)).ravel()
    return np.sqrt(np.dot(R, R) / 2.0 * 2)


def transform_mu(X, H, max_iter=200, tol=1e-4):
    """Returns (W, n_iter)."""
    X = np.asarray(X, dtype=np.float64)
    H = np.asarray(H, dtype=np.float64)
    W = np.full((X.shape[0], H.shape[0]), np.sqrt(X.mean() / H.shape[0]))
    error_at_init = frobenius(X, W, H)
    previous_error = error_at_init
    XHt = X @ H.T
    HHt = np.dot(H, H.T)
    n_iter = 0
    for n_iter in range(1, max_iter + 1):
        numerator = XHt.copy()
        denominator = np.dot(W, HHt)
        denominator[denominator == 0] = EPSILON
        numerator /= denominator
        W *= numerator
        if tol > 0 and n_iter % 10 == 0:
            error = frobenius(X, W, H)
            with np.errstate(invalid="ignore", divide="ignore"):
                if (previous_error - error) / error_at_init < tol:
                    break
            previous_error = error
    return W, n_iter


def transform(X, H, solver="cd", max_iter=200, tol=1e-4):
    return (transform_cd if solver == "cd" else transform_mu)(X, H, max_iter, tol)
