"""NMF by coordinate descent (fp64) and the device NNDSVD init against scikit-learn's NMF(solver="cd") in fp64.

Tolerances (fp64 CD is insensitive to init perturbations of 1e-13: same n_iter_, error moved by <= 2e-16 ||X||):
  same init, same iteration count:  |W H - W_sk H_sk|_max, |VAF| (overall, per muscle) <= 1e-9, |err| <= 1e-9 ||X||
  converged (tol 1e-6, max_iter 100 000), device NNDSVD vs sklearn's:  |VAF| <= 1e-8, |n_iter| within max(3, 0.5 %)
"""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_cd_oracle as co
from oracle import nmf_oracle as no
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


def sk_cd(X, k, max_iter, tol, init, W0=None, H0=None, solver="cd"):
    from sklearn.decomposition import NMF

    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = NMF(n_components=k, solver=solver, init=init, max_iter=max_iter, tol=tol, random_state=0)
        W = model.fit_transform(X, W=W0, H=H0) if init == "custom" else model.fit_transform(X)
    return W, model.components_, model


def iter_ok(got, want):
    return abs(int(got) - int(want)) <= max(3, 0.005 * want)


def check_same(res, p, X, W, H, err):
    want_all, want_cols = no.vaf(X, W, H)
    assert np.abs(res.W[p] @ res.H[p] - W @ H).max() <= TIGHT, p
    assert abs(res.vaf[p, 0] - want_all) <= TIGHT and np.abs(res.vaf[p, 1:] - want_cols).max() <= TIGHT, p
    assert abs(res.err[p] - err) <= TIGHT * np.linalg.norm(X), p


def test_same_init_fixed_iterations_matches_sklearn(analysis):
    for seed in (1, 2, 3):
        X = envelopes(seed)
        ranks = list(range(1, 9))
        inits = [no.random_init(X, k, 10 * seed + k) for k in ranks]
        res = analysis.nmf_cd_batched(X, ranks, init=inits, max_iter=300, tol=0.0)
        assert (res.n_iter == 300).all() and res.W[0].dtype == np.float64
        for p, k in enumerate(ranks):
            W, H, model = sk_cd(X, k, 300, 0.0, "custom", inits[p][0].copy(), inits[p][1].copy())
            check_same(res, p, X, W, H, model.reconstruction_err_)
    # sklearn's init="random" drawn by the batch itself
    X = envelopes(4)
    res = analysis.nmf_cd_batched(X, [2, 5], init="random", seeds=[3, 7], max_iter=300, tol=0.0)
    for p, (k, s) in enumerate([(2, 3), (5, 7)]):
        from sklearn.decomposition import NMF

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            model = NMF(n_components=k, init="random", random_state=s, max_iter=300, tol=0.0)
            W = model.fit_transform(X)
        check_same(res, p, X, W, model.components_, model.reconstruction_err_)


def test_converged_reference_defaults_match_sklearn(analysis):
    for seed in (1, 2):
        X = envelopes(seed)
        ranks = list(range(1, 9))
        res = analysis.nmf_cd_batched(X, ranks, init="nndsvda", max_iter=100_000, tol=1e-6)
        assert res.n_iter[0] == 100_000  # k = 1 never meets tol 1e-6, as in sklearn
        for p, k in enumerate(ranks):
            W, H, model = sk_cd(X, k, 100_000, 1e-6, "nndsvda")
            want_all, want_cols = no.vaf(X, W, H)
            assert iter_ok(res.n_iter[p], model.n_iter_), (seed, k, res.n_iter[p], model.n_iter_)
            assert abs(res.vaf[p, 0] - want_all) <= CONVERGED_VAF, (seed, k)
            assert np.abs(res.vaf[p, 1:] - want_cols).max() <= CONVERGED_VAF, (seed, k)


@pytest.mark.parametrize("variant", ["nndsvd", "nndsvda"])
def test_device_nndsvd_init(analysis, variant):
    from sklearn.decomposition._nmf import _initialize_nmf

    for seed in (1, 2, 4):
        X = envelopes(seed)
        ranks = list(range(1, 17))
        res = analysis.nmf_cd_batched(X, ranks, init=variant, max_iter=0, tol=0.0)
        for p, k in enumerate(ranks):
            W, H = co.nndsvd_exact(X, k, variant)
            assert np.abs(res.W[p] - W).max() <= TIGHT * np.abs(W).max(), (seed, k)
            assert np.abs(res.H[p] - H).max() <= TIGHT * np.abs(H).max(), (seed, k)
            if k <= 4:
                Ws, Hs = _initialize_nmf(X, k, init=variant, random_state=0)
                assert np.abs(res.W[p] - Ws).max() <= 1e-8 * np.abs(Ws).max()
                assert np.abs(res.H[p] - Hs).max() <= 1e-8 * np.abs(Hs).max()


def test_nndsvd_that_would_divide_by_zero_raises(analysis):
    rng = np.random.default_rng(0)
    X = np.outer(rng.uniform(0.1, 1, 50), rng.uniform(0.1, 1, 6))  # rank 1: the second singular value is zero
    with pytest.raises(ValueError, match="NNDSVD"):
        analysis.nmf_cd_batched(X, [2], init="nndsvd")
    with pytest.raises(ValueError, match="NNDSVD"):
        analysis.nmf_cd_batched(X, [1, 2], init="nndsvda", defer=True).result()
    assert analysis.nmf_cd_batched(X, [1], init="nndsvda").vaf[0, 0] > 1 - 1e-12
    with pytest.raises(ValueError, match="Negative"):
        analysis.nmf_cd_batched(-X, [1])


def tutorial_df():
    rng = np.random.default_rng(0)
    t = np.linspace(0, 1, 200)[:, None]
    basis = np.abs(np.sin(np.pi * (rng.uniform(0.5, 3, (1, 3)) * t + rng.uniform(0, 1, (1, 3))))) ** 2
    X = basis @ rng.uniform(0, 1, (3, 8)) + 0.02 * rng.uniform(0, 1, (200, 8))
    return pd.DataFrame(X / X.max(axis=0), columns=[f"m{i}" for i in range(8)], index=np.arange(200) * 2)


def test_find_synergies_tutorial_call_on_the_gpu(analysis):
    df = tutorial_df()
    res = analysis.find_synergies(df, 2, 3, max_iter=50_000, engine="gpu")
    assert list(res.vaf_values.index) == [2, 3]
    assert list(res.vaf_values.columns) == ["All signals"] + list(df.columns)
    X = df.to_numpy()
    for k in (2, 3):
        W, H, model = sk_cd(X, k, 50_000, 1e-6, None)
        ref = analysis.vaf(df, transformed_signal=W, components=H)
        assert np.abs(res.vaf_values.loc[k].to_numpy() - ref.iloc[0].to_numpy()).max() <= CONVERGED_VAF
        assert iter_ok(res.model[k].n_iter_, model.n_iter_)
        assert res.model[k].solver == "cd" and res.model[k].init == "nndsvda" and res.model[k].random_state is None
        assert list(res.components[k].columns) == list(df.columns) and res.components[k].shape == (k, 8)
        assert res.transformed[k].shape == (200, k)


def test_convergence_warning_when_max_iter_is_hit(analysis):
    from sklearn.exceptions import ConvergenceWarning

    df = tutorial_df()
    with pytest.warns(ConvergenceWarning, match="Maximum number of iterations 20 reached"):
        res = analysis.find_synergies(df, 2, max_iter=20, engine="gpu")
    assert res.model.n_iter_ == 20
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        analysis.find_synergies(df, 2, max_iter=20, tol=0.0, engine="gpu")  # tol = 0: no warning, as in sklearn


def test_mu_from_device_nndsvda(analysis):
    df = tutorial_df()
    res = analysis.find_synergies(df, 2, 4, max_iter=300, tol=0.0, solver="mu", init="nndsvda", engine="gpu")
    for k in (2, 3, 4):
        W, H, _ = sk_cd(df.to_numpy(), k, 300, 0.0, "nndsvda", solver="mu")
        ref = analysis.vaf(df, transformed_signal=W, components=H)
        assert np.abs(res.vaf_values.loc[k].to_numpy() - ref.iloc[0].to_numpy()).max() <= 1e-4
        assert res.model[k].solver == "mu" and res.model[k].init == "nndsvda"


@pytest.mark.parametrize("n", [700, 5000, 60001])
def test_streaming_regime(analysis, n):
    X = envelopes(5, n=n)
    ranks = [1, 3, 8]
    inits = [no.random_init(X, k, k) for k in ranks]
    res = analysis.nmf_cd_batched(X, ranks, init=inits, max_iter=30, tol=0.0, regime="stream")
    assert (res.n_iter == 30).all()
    for p, k in enumerate(ranks):
        W, H, model = sk_cd(X, k, 30, 0.0, "custom", inits[p][0].copy(), inits[p][1].copy())
        check_same(res, p, X, W, H, model.reconstruction_err_)
    if n <= 1000:
        same = analysis.nmf_cd_batched(X, ranks, init="nndsvda", max_iter=2000, tol=1e-6, regime="resident")
        stream = analysis.nmf_cd_batched(X, ranks, init="nndsvda", max_iter=2000, tol=1e-6, regime="stream")
        assert np.abs(same.vaf - stream.vaf).max() <= TIGHT
        assert all(iter_ok(a, b) for a, b in zip(stream.n_iter, same.n_iter))


def test_trial_synergies_cd_on_the_synthetic_trial(analysis):
    import muscle_synergies_b200 as ms
    from muscle_synergies_b200.pipeline import trial_synergies
    from tools.synth_vicon import synth_layout

    data = ms.load_vicon_bytes(synth_layout("D", seed=0), name="D")
    trial = trial_synergies(data, 1, 4, max_iter=500, tol=1e-4, window_size=0.05, solver="cd", keep_batch=True)
    env = trial.envelopes.cpu().numpy()
    assert env.shape[0] == 8 and len(trial.cycles) == 8 and trial.batch.W[0].dtype == np.float64
    for ci, cyc in enumerate(trial.cycles):
        for ki, k in enumerate((1, 2, 3, 4)):
            W, H, model = sk_cd(env[ci], k, 500, 1e-4, "nndsvda")
            want_all, want_cols = no.vaf(env[ci], W, H)
            assert iter_ok(cyc.n_iter[k], model.n_iter_), (ci, k, cyc.n_iter[k], model.n_iter_)
            assert abs(cyc._vaf[ki][0] - want_all) <= CONVERGED_VAF and np.abs(cyc._vaf[ki][1:] - want_cols).max() <= CONVERGED_VAF
    with pytest.raises(ValueError):
        trial_synergies(data, 1, 2, n_restarts=3, solver="cd")
