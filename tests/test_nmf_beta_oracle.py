"""Pins oracle/nmf_beta_oracle.py (numpy restatement of scikit-learn's multiplicative updates for the β-divergence, fit
and transform) against scikit-learn itself bit for bit, and checks the argument errors of nmf_beta_batched,
nmf_transform_batched, NMFModel.transform and find_synergies(engine="gpu") for beta_loss != 2 - all without a GPU."""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_beta_oracle as bo
from test_nmf_oracle import envelopes

BETAS = [1, 0, 0.5, 1.5, 3, "kullback-leibler", "itakura-saito"]


def sk_init(X, k):
    """sklearn's own nndsvda init (the start of the fixed-iteration comparisons)."""
    from sklearn.decomposition._nmf import _initialize_nmf

    return _initialize_nmf(X, k, init="nndsvda", random_state=0)  # a fixed seed for sklearn's randomized SVD


def sk_factorize(X, W, H, beta_loss, max_iter, tol, update_H=True):
    """non_negative_factorization(solver="mu", init="custom"): (W, H, n_iter)."""
    from sklearn.decomposition import non_negative_factorization

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return non_negative_factorization(X, W=W.copy() if update_H else None, H=H.copy(), n_components=H.shape[0],
                                          init="custom", solver="mu", beta_loss=beta_loss, max_iter=max_iter, tol=tol,
                                          update_H=update_H)


def awkward_x(seed, n=200, m=16):
    """An envelope with exact zeros and entries below EPSILON (dropped from the divergence's X terms)."""
    X = envelopes(seed, n=n, m=m)
    X[::17, 3] = 0.0
    X[5::23, 7] = 0.5 * bo.EPSILON
    X[9::29, 11] = bo.EPSILON  # not above EPSILON: dropped too
    return X


@pytest.mark.parametrize("beta", BETAS)
@pytest.mark.parametrize("tol", [0.0, 1e-4])
@pytest.mark.parametrize("k", [1, 4, 8])
def test_fit_restatement_equals_sklearn_bit_for_bit(beta, tol, k):
    X = envelopes(k + 3) if bo.beta_to_float(beta) <= 0 else awkward_x(k + 3)
    W0, H0 = sk_init(X, k)
    W_ref, H_ref, n_ref = sk_factorize(X, W0, H0, beta, 120, tol)
    W, H, n_iter = bo.fit(X, W0, H0, beta, 120, tol)
    assert n_iter == n_ref
    assert np.array_equal(W, W_ref) and np.array_equal(H, H_ref)


@pytest.mark.parametrize("beta", BETAS)
@pytest.mark.parametrize("tol", [0.0, 1e-4])
def test_transform_restatement_equals_sklearn_bit_for_bit(beta, tol):
    X = envelopes(2) if bo.beta_to_float(beta) <= 0 else awkward_x(2)
    H = np.random.default_rng(5).uniform(0, 1, (5, 16))
    W_ref, _, n_ref = sk_factorize(X, None, H, beta, 150, tol, update_H=False)
    W, n_iter = bo.transform(X, H, beta, 150, tol)
    assert n_iter == n_ref and np.array_equal(W, W_ref)


@pytest.mark.parametrize("beta", [1, 0, 0.5, 3])
def test_divergence_restatement_equals_sklearn(beta):
    from sklearn.decomposition._nmf import _beta_divergence

    X = envelopes(1) if beta <= 0 else awkward_x(1)
    W, H = sk_init(X, 3)
    assert bo.beta_divergence(X, W, H, beta) == _beta_divergence(X, W, H, beta, square_root=True)


def test_converged_stop_iteration_matches_sklearn():
    X = envelopes(4)
    for beta in ("kullback-leibler", "itakura-saito"):
        W0, H0 = sk_init(X, 3)
        _, _, n_ref = sk_factorize(X, W0, H0, beta, 5000, 1e-4)
        assert bo.fit(X, W0, H0, beta, 5000, 1e-4)[2] == n_ref < 5000


ZEROS = "When beta_loss <= 0 and X contains zeros"


def test_beta_argument_errors_need_no_device():
    from muscle_synergies_b200.analysis import NMFModel, find_synergies, nmf_beta_batched, nmf_transform_batched

    X = envelopes(0, m=8)
    Xz = X.copy()
    Xz[3, 2] = 0.0
    for kw, msg in [({"X": -X}, "Negative values in data passed to NMF"), ({"X": Xz, "beta_loss": 0}, ZEROS),
                    ({"X": Xz, "beta_loss": "itakura-saito"}, ZEROS), ({"X": Xz, "beta_loss": -0.5}, ZEROS),
                    ({"beta_loss": "frobenius"}, "Frobenius"), ({"beta_loss": 2}, "Frobenius"),
                    ({"beta_loss": "kl"}, "beta_loss must be"), ({"init": "custom"}, "init must be"),
                    ({"ranks": [17]}, "1..16"), ({"init": "random"}, "seed"), ({"regime": "auto"}, "regime"),
                    ({"x_index": [1]}, "x_index"), ({"max_iter": -1}, "max_iter"),
                    ({"init": [(np.ones((5, 2)), np.ones((2, 8)))]}, "shapes"),
                    ({"init": [(np.ones((200, 2)), -np.ones((2, 8)))]}, "Negative values in data passed to NMF \\(input H\\)"),
                    ({"init": [(np.zeros((200, 2)), np.ones((2, 8)))]}, "Array passed to NMF \\(input W\\) is full of zeros"),
                    ({"init": [(np.ones((200, 2)), np.full((2, 8), np.nan))]}, "NaN")]:
        args = dict(X=X, ranks=[2], beta_loss="kullback-leibler")
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            nmf_beta_batched(**args)
    # a zero is fine for beta_loss > 0
    H = [np.ones((2, 8))]
    with pytest.raises(ValueError, match="Invalid beta_loss parameter: solver 'cd' does not handle beta_loss = "
                                         "'kullback-leibler'"):
        nmf_transform_batched(X, H, solver="cd", beta_loss="kullback-leibler")
    with pytest.raises(ValueError, match=ZEROS):
        nmf_transform_batched(Xz, H, solver="mu", beta_loss="itakura-saito")
    model = NMFModel(2, H[0], 10, 0.1, 8, None, solver="mu", beta_loss=0.0, init="nndsvda")
    with pytest.raises(ValueError, match=ZEROS):
        model.transform(Xz)
    with pytest.raises(ValueError, match="Negative values in data passed to X in NMF"):
        model.transform(-X)
    df = pd.DataFrame(Xz, columns=list("abcdefgh"))
    with pytest.raises(ValueError, match="Invalid beta_loss parameter: solver 'cd' does not handle beta_loss = 1"):
        find_synergies(df, 2, engine="gpu", beta_loss=1)
    with pytest.raises(ValueError, match="Invalid beta_loss parameter: solver 'cd' does not handle beta_loss = "
                                         "'itakura-saito'"):
        find_synergies(df, 2, engine="gpu", solver="cd", beta_loss="itakura-saito")
    # sklearn's order: the nndsvd warning of _check_params, then the zeros
    with pytest.warns(UserWarning, match="The multiplicative update \\('mu'\\) solver cannot update zeros"):
        with pytest.raises(ValueError, match=ZEROS):
            find_synergies(df, 2, engine="gpu", solver="mu", init="nndsvd", beta_loss="itakura-saito")
    with pytest.raises(NotImplementedError, match="beta_loss='kl'"):
        find_synergies(df, 2, engine="gpu", solver="mu", beta_loss="kl")


def test_sklearn_raises_the_same_errors():
    """The texts above are scikit-learn's own."""
    from sklearn.decomposition import NMF

    X = envelopes(0, m=8)
    X[3, 2] = 0.0
    with pytest.raises(ValueError, match=ZEROS):
        NMF(2, solver="mu", beta_loss="itakura-saito").fit(X)
    with pytest.raises(ValueError, match="Invalid beta_loss parameter: solver 'cd' does not handle beta_loss = 1"):
        NMF(2, beta_loss=1).fit(X)
    with pytest.warns(UserWarning, match="The multiplicative update \\('mu'\\) solver cannot update zeros"):
        NMF(2, solver="mu", init="nndsvd", beta_loss=1, max_iter=5).fit(X + 0.1)
    from sklearn.decomposition import non_negative_factorization

    for W0, H0, msg in [(np.ones((200, 2)), -np.ones((2, 8)), "Negative values in data passed to NMF \\(input H\\)"),
                        (np.zeros((200, 2)), np.ones((2, 8)), "Array passed to NMF \\(input W\\) is full of zeros")]:
        with pytest.raises(ValueError, match=msg):
            non_negative_factorization(X + 0.1, W0, H0, n_components=2, init="custom", solver="mu", beta_loss=1)
