"""Pins oracle/nmf_transform_oracle.py (numpy restatement of sklearn's NMF.transform for solver "cd" and "mu") against
scikit-learn itself bit for bit, and checks the argument errors of NMFModel.transform and nmf_transform_batched - all
without a GPU."""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_transform_oracle as to
from test_nmf_oracle import envelopes


def synergies(k, m=16, seed=0):
    return np.random.default_rng(100 + seed).uniform(0, 1, (k, m))


def sk_transform(X, H, solver, max_iter, tol):
    """sklearn's transform path, _fit_transform(update_H=False), with its iteration count."""
    from sklearn.decomposition import NMF

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        W, _, n_iter = NMF(n_components=H.shape[0], solver=solver, max_iter=max_iter, tol=tol)._fit_transform(
            X, H=H, update_H=False)
    return W, n_iter


@pytest.mark.parametrize("solver", ["cd", "mu"])
@pytest.mark.parametrize("tol", [0.0, 1e-4, 1e-6])
@pytest.mark.parametrize("k", [1, 2, 5, 8])
def test_transform_restatement_equals_sklearn_bit_for_bit(solver, tol, k):
    X = envelopes(k)
    H = synergies(k, seed=k)
    W_ref, n_ref = sk_transform(X, H, solver, 400, tol)
    W, n_iter = to.transform(X, H, solver, 400, tol)
    assert n_iter == n_ref
    assert np.array_equal(W, W_ref)


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_transform_restatement_edge_cases(solver):
    H = synergies(3)
    H[1] = 0.0  # a synergy that is zero everywhere
    X = envelopes(1)
    for Xc in (X, np.zeros_like(X)):
        W_ref, n_ref = sk_transform(Xc, H, solver, 50, 1e-4)
        W, n_iter = to.transform(Xc, H, solver, 50, 1e-4)
        assert n_iter == n_ref and np.array_equal(W, W_ref)
    # an all-zero X: cd stops at once, mu never meets its test (0 / 0)
    assert to.transform(np.zeros_like(X), H, solver, 50, 1e-4)[1] == (1 if solver == "cd" else 50)


def model(k=3, m=8, solver="cd"):
    from muscle_synergies_b200.analysis import NMFModel

    return NMFModel(k, synergies(k, m), 10, 0.1, m, None, solver=solver, init="nndsvda")


def test_transform_argument_errors_need_no_device():
    X = envelopes(0, m=8)
    mdl = model()
    assert mdl.max_iter == 100_000 and mdl.tol == 1e-6  # the reference's find_synergies defaults
    for bad, msg in [(-X, "Negative values in data passed to X in NMF."), (X * np.nan, "Input X contains NaN"),
                     (X * np.inf, "Input X contains infinity"), (X[:, :5], "X has 5 features, but NMF is expecting 8")]:
        with pytest.raises(ValueError, match=msg.replace(".", r"\.")):
            mdl.transform(bad)
        with pytest.raises(ValueError, match=msg.replace(".", r"\.")):
            mdl.transform(pd.DataFrame(bad))
    W = np.abs(np.random.default_rng(0).standard_normal((5, 3)))
    assert np.array_equal(mdl.inverse_transform(W), W @ mdl.components_)


def test_transform_batched_argument_errors_need_no_device():
    from muscle_synergies_b200.analysis import nmf_transform_batched

    X = envelopes(0, m=8)
    H = [synergies(2, 8)]
    for kw, msg in [({"X": -X}, "Negative"), ({"X": X * np.nan}, "NaN"), ({"solver": "lbfgs"}, "solver"),
                    ({"regime": "auto"}, "regime"), ({"H": [synergies(2, 7)]}, "features"),
                    ({"H": [synergies(17, 8)]}, "1 <= k <= 16"), ({"H": [synergies(2, 8), synergies(3, 9)]}, "H\\[1\\]"),
                    ({"H": [-synergies(2, 8)]}, "non-negative"), ({"x_index": [1]}, "x_index"),
                    ({"x_index": [0, 0]}, "x_index"), ({"max_iter": -1}, "max_iter"), ({"H": []}, "one")]:
        args = dict(X=X, H=H)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            nmf_transform_batched(**args)
    with pytest.raises(ValueError, match="m <= 64"):
        nmf_transform_batched(np.zeros((3, 50, 65)), [np.ones((1, 65))])  # m > 64 is refused by name
