"""NMF with fixed synergies (NMFModel.transform, nmf_transform_batched; csrc/ms_nmf_fixed.cu) against scikit-learn's
NMF.transform in fp64, for solver "cd" and "mu".

Tolerances: same iteration count (tol 0): |W H - W_sk H|_max, |VAF| <= 1e-9; converged (tol 1e-6, max_iter 100 000):
|VAF| <= 1e-8, n_iter within max(3, 0.5 %) for cd and within one check (10) for mu.
"""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_oracle as no
from test_nmf_oracle import envelopes
from test_nmf_transform_oracle import sk_transform, synergies

pytestmark = pytest.mark.gpu

TIGHT = 1e-9
CONVERGED_VAF = 1e-8


@pytest.fixture(scope="module")
def analysis():
    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import analysis

    return analysis


def iter_ok(solver, got, want):
    return abs(int(got) - int(want)) <= (max(3, 0.005 * want) if solver == "cd" else 10)


def check_same(res, p, X, H, W_sk, tight=TIGHT):
    want_all, want_cols = no.vaf(X, W_sk, H)
    assert np.abs(res.W[p] @ H - W_sk @ H).max() <= tight, p
    assert abs(res.vaf[p, 0] - want_all) <= tight and np.abs(res.vaf[p, 1:] - want_cols).max() <= tight, p
    assert abs(res.err[p] - np.linalg.norm(X - res.W[p] @ H)) <= TIGHT * np.linalg.norm(X), p


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_resident_fixed_iterations_match_sklearn(analysis, solver):
    X = envelopes(3)
    ranks = list(range(1, 9)) + [16]
    H = [synergies(k, seed=k) for k in ranks]
    res = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=300, tol=0.0, regime="resident")
    assert (res.n_iter == 300).all() and res.W[0].dtype == np.float64 and (res.seeds == -1).all()
    for p in range(len(ranks)):
        assert np.array_equal(res.H[p], H[p])
        check_same(res, p, X, H[p], sk_transform(X, H[p], solver, 300, 0.0)[0])


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_converged_matches_sklearn(analysis, solver):
    from sklearn.decomposition import NMF

    for seed in (1, 2):
        X = envelopes(seed)
        ranks = list(range(1, 9))
        # synergies fitted to another recording, as in cross-cycle generalisation
        H = [NMF(k, init="nndsvda", max_iter=2000).fit(envelopes(seed + 10)).components_ for k in ranks]
        res = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=100_000, tol=1e-6)
        for p, k in enumerate(ranks):
            W, n_iter = sk_transform(X, H[p], solver, 100_000, 1e-6)
            want_all, want_cols = no.vaf(X, W, H[p])
            assert iter_ok(solver, res.n_iter[p], n_iter), (seed, k, res.n_iter[p], n_iter)
            assert abs(res.vaf[p, 0] - want_all) <= CONVERGED_VAF, (seed, k)
            assert np.abs(res.vaf[p, 1:] - want_cols).max() <= CONVERGED_VAF, (seed, k)


def sk_model_transform(X, model):
    from sklearn.decomposition import NMF

    sk = NMF(model.n_components, solver=model.solver, max_iter=model.max_iter, tol=model.tol)
    sk.components_ = model.components_
    sk.n_components_ = model.n_components
    sk.n_features_in_ = model.n_features_in_
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return sk.transform(X)


def test_models_of_gpu_fits_transform_like_sklearn(analysis):
    from test_nmf_cd_gpu import tutorial_df

    df = tutorial_df()
    new = pd.DataFrame(envelopes(7, m=8), columns=df.columns)
    fits = {"cd": analysis.find_synergies(df, 2, 3, max_iter=50_000, engine="gpu"),
            "mu": analysis.find_synergies(df, 2, 3, solver="mu", init="random", random_state=0, max_iter=3000)}
    for solver, res in fits.items():
        for k in (2, 3):
            model = res.model[k]
            assert model.solver == solver and model.max_iter == (50_000 if solver == "cd" else 3000) and model.tol == 1e-6
            W = model.transform(new)
            W_sk = sk_model_transform(new.to_numpy(), model)
            assert W.shape == (len(new), k)
            want = no.vaf(new.to_numpy(), W_sk, model.components_)[0]
            assert abs(no.vaf(new.to_numpy(), W, model.components_)[0] - want) <= CONVERGED_VAF, (solver, k)
            assert np.array_equal(model.inverse_transform(W), W @ model.components_)
            # the training data itself: transform reproduces the fit's activations' quality
            assert analysis.vaf(df, transformed_signal=model.transform(df), components=model.components_).shape == (1, 9)
    import torch

    model = fits["cd"].model[2]
    Wd = model.transform(torch.from_numpy(new.to_numpy()).cuda())
    assert Wd.is_cuda and np.array_equal(Wd.cpu().numpy(), model.transform(new))
    assert np.allclose(model.inverse_transform(Wd).cpu().numpy(), model.inverse_transform(Wd.cpu().numpy()), atol=1e-12)


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_streaming_is_bit_identical_to_resident_at_tol_zero(analysis, solver):
    X = envelopes(4, n=300)
    ranks = list(range(1, 9)) + [16]
    H = [synergies(k, seed=k) for k in ranks]
    for max_iter in (1, 45, 300):
        a = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=max_iter, tol=0.0, regime="resident")
        b = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=max_iter, tol=0.0, regime="stream")
        assert (a.n_iter == max_iter).all() and (b.n_iter == max_iter).all()
        for p in range(len(ranks)):
            assert np.array_equal(a.W[p], b.W[p]), (max_iter, p)
        assert np.abs(a.vaf - b.vaf).max() <= 1e-12


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_streaming_long_signal_matches_sklearn(analysis, solver):
    X = envelopes(5, n=300_000)
    ranks = list(range(1, 9))
    H = [synergies(k, seed=k) for k in ranks]
    res = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=50, tol=0.0)  # by size: streaming
    for p in range(len(ranks)):
        check_same(res, p, X, H[p], sk_transform(X, H[p], solver, 50, 0.0)[0])


@pytest.mark.parametrize("solver", ["cd", "mu"])
def test_streaming_converged_and_strided_input(analysis, solver):
    import torch

    X = envelopes(6, n=5000)
    ranks = [1, 3, 8]
    H = [synergies(k, seed=k) for k in ranks]
    res = analysis.nmf_transform_batched(X, H, solver=solver, max_iter=100_000, tol=1e-6, regime="stream")
    for p, k in enumerate(ranks):
        W, n_iter = sk_transform(X, H[p], solver, 100_000, 1e-6)
        assert iter_ok(solver, res.n_iter[p], n_iter), (k, res.n_iter[p], n_iter)
        assert abs(res.vaf[p, 0] - no.vaf(X, W, H[p])[0]) <= CONVERGED_VAF
    # a channel-major (muscles, samples) envelope, passed as its transposed view, reads in place
    env = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    for regime in ("stream", "resident"):
        view = env[:, :600].T if regime == "resident" else env.T
        assert not view.is_contiguous()
        a = analysis.nmf_transform_batched(view, H, solver=solver, max_iter=500, tol=1e-6, regime=regime)
        b = analysis.nmf_transform_batched(view.contiguous(), H, solver=solver, max_iter=500, tol=1e-6, regime=regime)
        assert np.array_equal(a.n_iter, b.n_iter) and np.array_equal(a.err, b.err) and np.array_equal(a.vaf, b.vaf)
        assert all(np.array_equal(a.W[p], b.W[p]) for p in range(len(ranks)))


@pytest.mark.parametrize("regime", ["resident", "stream"])
def test_edge_cases(analysis, regime):
    from sklearn.exceptions import ConvergenceWarning
    from muscle_synergies_b200.analysis import NMFModel

    X = envelopes(2)
    H = synergies(3)
    H[1] = 0.0
    for solver in ("cd", "mu"):
        # an H with an all-zero synergy
        res = analysis.nmf_transform_batched(X, [H], solver=solver, max_iter=300, tol=0.0, regime=regime)
        check_same(res, 0, X, H, sk_transform(X, H, solver, 300, 0.0)[0])
        assert (res.W[0][:, 1] == 0).all()
        # an all-zero X: cd stops at iteration 1, mu runs to max_iter (its test is 0 / 0) and warns
        zero = analysis.nmf_transform_batched(np.zeros_like(X), [H, H[:1]], solver=solver, max_iter=40, tol=1e-4,
                                              regime=regime)
        assert (zero.n_iter == (1 if solver == "cd" else 40)).all() and (zero.W[0] == 0).all()
        model = NMFModel(3, H, 1, 0.0, 16, None, solver=solver, max_iter=40, tol=1e-4)
        if solver == "mu":
            with pytest.warns(ConvergenceWarning, match="Maximum number of iterations 40 reached"):
                model.transform(np.zeros_like(X))
        # defer=True, and two identical calls: bit-identical
        args = (X, [H, synergies(5)])
        kw = dict(solver=solver, max_iter=2000, tol=1e-6, regime=regime)
        a = analysis.nmf_transform_batched(*args, **kw)
        b = analysis.nmf_transform_batched(*args, **kw)
        c = analysis.nmf_transform_batched(*args, defer=True, **kw).result()
        for r in (b, c):
            assert np.array_equal(a.n_iter, r.n_iter) and np.array_equal(a.err, r.err) and np.array_equal(a.vaf, r.vaf)
            assert all(np.array_equal(a.W[p], r.W[p]) for p in range(2))
    import torch

    bad = torch.from_numpy(-X).cuda()
    with pytest.raises(ValueError, match="Negative values in data passed to X in NMF"):
        analysis.nmf_transform_batched(bad, [H])
    pending = analysis.nmf_transform_batched(bad, [H], defer=True, regime=regime)
    with pytest.raises(ValueError, match="Negative values in data passed to X in NMF"):
        pending.result()


def test_cross_cycle_vaf_on_the_synthetic_trial(analysis):
    import muscle_synergies_b200 as ms
    from muscle_synergies_b200.pipeline import cross_cycle_vaf, trial_synergies
    from tools.synth_vicon import synth_layout

    data = ms.load_vicon_bytes(synth_layout("D", seed=0), name="D")
    trial = trial_synergies(data, 1, 8, max_iter=500, tol=1e-4, window_size=0.05, solver="cd")
    table = cross_cycle_vaf(trial)
    env = trial.envelopes.cpu().numpy()
    assert table.shape == (64, 8) and list(table.index.names) == ["n_components", "trecho", "cycle"]
    for k in range(1, 9):
        for si, src in enumerate(trial.cycles):
            H = src.components[k].to_numpy()
            for ti, tgt in enumerate(trial.cycles):
                W, _ = sk_transform(env[ti], H, "cd", 100_000, 1e-6)
                want = no.vaf(env[ti], W, H)[0]
                got = table.loc[(k, src.trecho.value, src.cycle.value), (tgt.trecho.value, tgt.cycle.value)]
                assert abs(got - want) <= CONVERGED_VAF, (k, si, ti)
