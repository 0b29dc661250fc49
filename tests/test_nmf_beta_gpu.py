"""β-divergence NMF by multiplicative updates (nmf_beta_batched, find_synergies(solver="mu", beta_loss=...),
nmf_transform_batched(beta_loss=...), NMFModel.transform; csrc/ms_nmf_beta.cu) against scikit-learn in fp64.

Tolerances: from sklearn's own init at the same iteration count (tol 0): |W H - W_sk H_sk|_max <= 1e-9 (X scaled to
max 1), |VAF| <= 1e-9 and err (sklearn's reconstruction_err_) to 1e-9 relative; converged: |VAF| <= 1e-8, n_iter within
one check (10).  Streaming and resident sum the H-step terms in different orders: they agree to 1e-10.
"""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_beta_oracle as bo
from oracle import nmf_oracle as no
from test_nmf_beta_oracle import BETAS, awkward_x, sk_factorize, sk_init
from test_nmf_oracle import envelopes

pytestmark = pytest.mark.gpu

TIGHT = 1e-9
CONVERGED_VAF = 1e-8


@pytest.fixture(scope="module")
def analysis():
    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import analysis

    return analysis


def x_for(beta, seed, n=200):
    """X scaled to max 1; with exact zeros and sub-EPSILON entries where beta_loss > 0 allows them."""
    return envelopes(seed, n=n) if bo.beta_to_float(beta) <= 0 else awkward_x(seed, n=n)


def check_same(res, p, X, W_sk, H_sk, beta):
    from sklearn.decomposition._nmf import _beta_divergence

    want_all, want_cols = no.vaf(X, W_sk, H_sk)
    assert np.abs(res.W[p] @ res.H[p] - W_sk @ H_sk).max() <= TIGHT, p
    assert abs(res.vaf[p, 0] - want_all) <= TIGHT and np.abs(res.vaf[p, 1:] - want_cols).max() <= TIGHT, p
    want_err = _beta_divergence(X, W_sk, H_sk, beta, square_root=True)
    assert abs(res.err[p] - want_err) <= TIGHT * want_err, (p, res.err[p], want_err)


@pytest.mark.parametrize("beta", BETAS)
def test_fixed_iterations_match_sklearn(analysis, beta):
    X = x_for(beta, 3)
    ranks = list(range(1, 9)) + [16]
    init = [sk_init(X, k) for k in ranks]
    res = analysis.nmf_beta_batched(X, ranks, beta, init=init, max_iter=300, tol=0.0)
    assert (res.n_iter == 300).all() and res.W[0].dtype == np.float64
    for p, k in enumerate(ranks):
        W_sk, H_sk, n_sk = sk_factorize(X, *init[p], beta, 300, 0.0)
        check_same(res, p, X, W_sk, H_sk, beta)


@pytest.mark.parametrize("beta", ["kullback-leibler", "itakura-saito"])
def test_converged_matches_sklearn(analysis, beta):
    X = envelopes(1)
    for ranks, max_iter, tol in ((list(range(1, 9)), 200, 1e-4), ([2, 4], 100_000, 1e-6)):
        init = [sk_init(X, k) for k in ranks]
        res = analysis.nmf_beta_batched(X, ranks, beta, init=init, max_iter=max_iter, tol=tol)
        for p, k in enumerate(ranks):
            W_sk, H_sk, n_sk = sk_factorize(X, *init[p], beta, max_iter, tol)
            want_all, want_cols = no.vaf(X, W_sk, H_sk)
            assert abs(int(res.n_iter[p]) - n_sk) <= 10, (k, tol, res.n_iter[p], n_sk)
            assert abs(res.vaf[p, 0] - want_all) <= CONVERGED_VAF, (k, tol)
            assert np.abs(res.vaf[p, 1:] - want_cols).max() <= CONVERGED_VAF, (k, tol)


@pytest.mark.parametrize("beta", ["kullback-leibler", "itakura-saito", 1.5, 0.5])
def test_streaming_agrees_with_resident_and_repeats_bit_for_bit(analysis, beta):
    X = x_for(beta, 4, n=300)
    ranks = list(range(1, 9)) + [16]
    init = [sk_init(X, k) for k in ranks]
    for max_iter in (1, 45, 300):
        a = analysis.nmf_beta_batched(X, ranks, beta, init=init, max_iter=max_iter, tol=0.0, regime="resident")
        b = analysis.nmf_beta_batched(X, ranks, beta, init=init, max_iter=max_iter, tol=0.0, regime="stream")
        assert (a.n_iter == max_iter).all() and (b.n_iter == max_iter).all()
        for p in range(len(ranks)):
            assert np.abs(a.W[p] - b.W[p]).max() <= 1e-10 and np.abs(a.H[p] - b.H[p]).max() <= 1e-10, (max_iter, p)
        assert np.abs(a.vaf - b.vaf).max() <= 1e-10 and np.abs(a.err - b.err).max() <= 1e-10 * a.err.max()
    # converged: the stop test of the streaming regime rides along with the next pass and still stops where sklearn does
    for regime in ("resident", "stream"):
        kw = dict(init=init, max_iter=3000, tol=1e-4, regime=regime)
        a = analysis.nmf_beta_batched(X, ranks, beta, **kw)
        b = analysis.nmf_beta_batched(X, ranks, beta, **kw)
        c = analysis.nmf_beta_batched(X, ranks, beta, defer=True, **kw).result()
        for r in (b, c):
            assert np.array_equal(a.n_iter, r.n_iter) and np.array_equal(a.err, r.err) and np.array_equal(a.vaf, r.vaf)
            assert all(np.array_equal(a.W[p], r.W[p]) and np.array_equal(a.H[p], r.H[p]) for p in range(len(ranks)))
        for p, k in enumerate(ranks):
            W_sk, H_sk, n_sk = sk_factorize(X, *init[p], beta, 3000, 1e-4)
            assert abs(int(a.n_iter[p]) - n_sk) <= 10, (regime, k, a.n_iter[p], n_sk)
            assert abs(a.vaf[p, 0] - no.vaf(X, W_sk, H_sk)[0]) <= CONVERGED_VAF, (regime, k)


def test_streaming_long_signal_matches_sklearn(analysis):
    X = awkward_x(5, n=40_000)
    ranks = [1, 3, 8]
    init = [sk_init(X, k) for k in ranks]
    for beta in ("kullback-leibler", 3):
        res = analysis.nmf_beta_batched(X, ranks, beta, init=init, max_iter=30, tol=0.0)  # by size: streaming
        for p in range(len(ranks)):
            W_sk, H_sk, _ = sk_factorize(X, *init[p], beta, 30, 0.0)
            check_same(res, p, X, W_sk, H_sk, beta)


@pytest.mark.parametrize("regime", ["resident", "stream"])
def test_strided_input_and_stacks(analysis, regime):
    import torch

    X = envelopes(6, n=200)
    ranks = [1, 3, 8]
    env = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()  # channel-major (muscles, samples)
    view = env.T
    assert not view.is_contiguous()
    # explicit pairs and sklearn's random draws: the device NNDSVD init sums X^T X with atomics, so its last bits may
    # differ from call to call whatever the layout
    for init in ([sk_init(X, k) for k in ranks], "random"):
        seeds = [0, 1, 2] if init == "random" else None
        kw = dict(init=init, seeds=seeds, max_iter=500, tol=1e-4, regime=regime)
        a = analysis.nmf_beta_batched(view, ranks, "kullback-leibler", **kw)
        b = analysis.nmf_beta_batched(view.contiguous(), ranks, "kullback-leibler", **kw)
        assert np.array_equal(a.n_iter, b.n_iter) and np.array_equal(a.err, b.err) and np.array_equal(a.vaf, b.vaf)
        assert all(np.array_equal(a.W[p], b.W[p]) and np.array_equal(a.H[p], b.H[p]) for p in range(len(ranks)))
    # a (B, n, m) stack with x_index: each problem as if run alone
    stack = np.stack([envelopes(s) for s in (7, 8, 9)])
    ranks, xi = [2, 3, 4, 2], [0, 1, 2, 2]
    init = [sk_init(stack[b], k) for k, b in zip(ranks, xi)]
    res = analysis.nmf_beta_batched(stack, ranks, "itakura-saito", init=init, x_index=xi, max_iter=400, tol=1e-4,
                                    regime=regime)
    for p, (k, b) in enumerate(zip(ranks, xi)):
        one = analysis.nmf_beta_batched(stack[b], [k], "itakura-saito", init=[init[p]], max_iter=400, tol=1e-4,
                                        regime=regime)
        assert one.n_iter[0] == res.n_iter[p] and np.array_equal(one.W[0], res.W[p]) and np.array_equal(one.H[0], res.H[p])


def sk_beta_transform(X, H, beta, max_iter, tol):
    from sklearn.decomposition import NMF

    sk = NMF(H.shape[0], solver="mu", beta_loss=beta, max_iter=max_iter, tol=tol)
    sk.components_ = H
    sk.n_components_ = H.shape[0]
    sk.n_features_in_ = H.shape[1]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return sk.transform(X)


@pytest.mark.parametrize("regime", ["resident", "stream"])
def test_transform_matches_sklearn(analysis, regime):
    X = envelopes(2)
    ranks = [1, 2, 4, 8]
    H = [sk_factorize(envelopes(12), *sk_init(envelopes(12), k), "kullback-leibler", 500, 1e-4)[1] for k in ranks]
    for beta in ("kullback-leibler", "itakura-saito", 0.5):
        res = analysis.nmf_transform_batched(X, H, solver="mu", max_iter=300, tol=0.0, regime=regime, beta_loss=beta)
        assert (res.n_iter == 300).all()
        for p in range(len(ranks)):
            assert np.array_equal(res.H[p], H[p])
            W_sk = sk_beta_transform(X, H[p], beta, 300, 0.0)
            assert np.abs(res.W[p] @ H[p] - W_sk @ H[p]).max() <= TIGHT, (beta, p)
            assert abs(res.vaf[p, 0] - no.vaf(X, W_sk, H[p])[0]) <= TIGHT, (beta, p)
        conv = analysis.nmf_transform_batched(X, H, solver="mu", max_iter=100_000, tol=1e-6, regime=regime,
                                              beta_loss=beta)
        for p in range(len(ranks)):
            W_sk, n_sk = bo.transform(X, H[p], beta, 100_000, 1e-6)
            assert abs(int(conv.n_iter[p]) - n_sk) <= 10, (beta, p, conv.n_iter[p], n_sk)
            assert abs(conv.vaf[p, 0] - no.vaf(X, W_sk, H[p])[0]) <= CONVERGED_VAF, (beta, p)


def test_find_synergies_kl_matches_sklearn(analysis):
    """Both sides start from sklearn's random init for the same random_state (the device draws sklearn's numbers and
    scales them by sklearn's own X.mean()), so the comparison is deterministic.  The default nndsvda init is compared
    only for what does not depend on its last bits: the device's comes from an exact SVD whose X^T X is summed with
    atomics, sklearn's from a randomized SVD."""
    from sklearn.exceptions import ConvergenceWarning

    X = envelopes(3)
    df = pd.DataFrame(X, columns=[f"m{j}" for j in range(16)])
    for max_iter, tol in ((300, 0.0), (5000, 1e-4)):
        kw = dict(solver="mu", beta_loss="kullback-leibler", init="random", random_state=0, max_iter=max_iter, tol=tol)
        gpu = analysis.find_synergies(df, 1, 8, engine="gpu", **kw)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = analysis.find_synergies(df, 1, 8, engine="sklearn", **kw)
        for k in range(1, 9):
            model, sk = gpu.model[k], ref.model[k]
            assert model.beta_loss == "kullback-leibler" and model.solver == "mu" and model.random_state == 0
            dvaf = np.abs(gpu.vaf_values.loc[k].to_numpy() - ref.vaf_values.loc[k].to_numpy()).max()
            if tol == 0:
                assert model.n_iter_ == sk.n_iter_ == 300
                assert np.abs(gpu.transformed[k] @ model.components_ - ref.transformed[k] @ sk.components_).max() <= TIGHT
                assert dvaf <= TIGHT and abs(model.reconstruction_err_ - sk.reconstruction_err_) <= TIGHT * sk.reconstruction_err_
            else:
                assert abs(model.n_iter_ - sk.n_iter_) <= 10, (k, model.n_iter_, sk.n_iter_)
                assert dvaf <= CONVERGED_VAF, (k, dvaf)
                # the model's transform runs the same divergence on the GPU
                W = model.transform(df)
                W_sk = sk_beta_transform(X, model.components_, "kullback-leibler", model.max_iter, model.tol)
                assert abs(no.vaf(X, W, model.components_)[0] - no.vaf(X, W_sk, model.components_)[0]) <= CONVERGED_VAF, k
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        default = analysis.find_synergies(df, 1, 8, engine="gpu", solver="mu", beta_loss="kullback-leibler", max_iter=200)
    assert all(default.model[k].init == "nndsvda" and default.model[k].beta_loss == "kullback-leibler" for k in range(1, 9))
    kw = dict(solver="mu", beta_loss="kullback-leibler", max_iter=5000, tol=1e-4)
    # restarts: the smallest divergence wins
    res = analysis.find_synergies(df, 3, engine="gpu", init="random", random_state=0, n_restarts=4, **kw)
    table = res.model.restarts
    assert len(table) == 4 and res.model.reconstruction_err_ == table["reconstruction_err"].min()
    assert res.model.random_state == int(table["random_state"][table["reconstruction_err"].idxmin()])
    with pytest.warns(ConvergenceWarning, match="Maximum number of iterations 20 reached"):
        analysis.find_synergies(df, 2, engine="gpu", solver="mu", beta_loss=0.5, max_iter=20, tol=1e-4)
    with pytest.warns(UserWarning, match="cannot update zeros"):
        analysis.find_synergies(df, 2, engine="gpu", solver="mu", init="nndsvd", beta_loss=1, max_iter=50, tol=0.0)


def test_device_input_errors(analysis):
    import torch

    X = envelopes(2)
    Xz = X.copy()
    Xz[4, 4] = 0.0
    for bad, beta, msg in [(-X, 1, "Negative values in data passed to NMF"),
                           (Xz, "itakura-saito", "When beta_loss <= 0 and X contains zeros")]:
        d = torch.from_numpy(bad).cuda()
        with pytest.raises(ValueError, match=msg):
            analysis.nmf_beta_batched(d, [2], beta)
        pending = analysis.nmf_beta_batched(d, [2], beta, init="random", seeds=[0], defer=True)
        with pytest.raises(ValueError, match=msg):
            pending.result()
    with pytest.raises(ValueError, match="When beta_loss <= 0 and X contains zeros"):
        analysis.nmf_transform_batched(torch.from_numpy(Xz).cuda(), [np.ones((2, 16))], solver="mu", beta_loss=0)
    # a zero is fine for beta_loss > 0, and an all-zero synergy stays zero
    H = np.random.default_rng(0).uniform(0, 1, (3, 16))
    H[1] = 0.0
    res = analysis.nmf_transform_batched(Xz, [H], solver="mu", max_iter=200, tol=0.0, beta_loss=1)
    W_sk = sk_beta_transform(Xz, H, 1, 200, 0.0)
    assert np.abs(res.W[0] @ H - W_sk @ H).max() <= TIGHT
