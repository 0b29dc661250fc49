"""Pins oracle/nmf_cd_oracle.py (numpy restatement of sklearn's coordinate-descent solver and NNDSVD init) against
scikit-learn itself, and checks the argument errors of find_synergies(engine="gpu") - all without a GPU."""
import warnings

import numpy as np
import pandas as pd
import pytest

from oracle import nmf_cd_oracle as co
from oracle import nmf_oracle as no
from test_nmf_oracle import envelopes


@pytest.mark.parametrize("k,seed,tol", [(1, 0, 1e-5), (2, 3, 1e-5), (3, 4, 1e-6), (5, 7, 1e-5), (8, 11, 0.0)])
def test_cd_restatement_equals_sklearn_bit_for_bit(k, seed, tol):
    from sklearn.decomposition import NMF

    X = envelopes(seed)
    W0, H0 = no.random_init(X, k, seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = NMF(n_components=k, solver="cd", init="custom", max_iter=300, tol=tol)
        W_ref = model.fit_transform(X, W=W0.copy(), H=H0.copy())
    W, H, n_iter = co.cd(X, W0, H0, max_iter=300, tol=tol)
    assert n_iter == model.n_iter_
    assert np.array_equal(W, W_ref) and np.array_equal(H, model.components_)


@pytest.mark.parametrize("variant", ["nndsvd", "nndsvda"])
@pytest.mark.parametrize("seed", [1, 2, 4])
def test_exact_nndsvd_matches_sklearn_init(variant, seed):
    from sklearn.decomposition._nmf import _initialize_nmf

    X = envelopes(seed)
    for k in range(1, 5):
        W_ref, H_ref = _initialize_nmf(X, k, init=variant, random_state=0)
        W, H = co.nndsvd_exact(X, k, variant)
        assert np.abs(W - W_ref).max() <= 1e-9 * np.abs(W_ref).max()
        assert np.abs(H - H_ref).max() <= 1e-9 * np.abs(H_ref).max()


def test_engine_gpu_argument_errors_need_no_device():
    from muscle_synergies_b200.analysis import find_synergies

    df = pd.DataFrame(envelopes(0, m=8), columns=[f"m{i}" for i in range(8)])
    with pytest.raises(ValueError, match="engine"):
        find_synergies(df, 2, engine="cuda")
    for kw, name in [({"alpha_W": 0.1}, "alpha_W"), ({"shuffle": True}, "shuffle"), ({"init": "nndsvdar"}, "nndsvdar"),
                     ({"solver": "lbfgs"}, "lbfgs"), ({"beta_loss": "kullback-leibler"}, "kullback-leibler"),
                     ({"l1_ratio": 0.5}, "l1_ratio")]:
        with pytest.raises(NotImplementedError, match=name):
            find_synergies(df, 2, 3, engine="gpu", **kw)
    with pytest.raises(ValueError, match="n_restarts"):
        find_synergies(df, 2, engine="gpu", n_restarts=4)  # init None resolves to nndsvda: deterministic
    with pytest.raises(ValueError, match="n_restarts"):
        find_synergies(df, 2, engine="gpu", n_restarts=2, init="nndsvd")
    with pytest.raises(ValueError):
        find_synergies(df, 0, engine="gpu")


def test_trial_synergies_argument_errors_need_no_device():
    from muscle_synergies_b200.pipeline import _deterministic

    assert _deterministic("cd", None) and _deterministic("cd", "nndsvd") and not _deterministic("cd", "random")
    assert not _deterministic("mu", None)
    for solver, init in [("mu", "nndsvda"), ("cd", "nndsvdar"), ("lbfgs", None)]:
        with pytest.raises(ValueError):
            _deterministic(solver, init)


def test_sharded_cd_runs_one_seed_per_file():
    """A deterministic init has no restarts to split: every rank gets one seed per file (or nothing)."""
    from muscle_synergies_b200.pipeline import synergies_for_files_sharded

    calls = []

    def analyse(paths, seeds, **kw):
        calls.append((list(paths), list(seeds), kw))
        return iter(())

    for rank in range(4):
        synergies_for_files_sharded(["a", "b"], rank=rank, world=4, analyse=analyse, gather=False, solver="cd")
    assert calls == [(["a", "b"], [0], {"solver": "cd"})]
    calls.clear()
    for rank in range(2):
        synergies_for_files_sharded(["a", "b", "c"], rank=rank, world=2, analyse=analyse, gather=False, solver="cd",
                                    init="nndsvd", random_state=5)
    assert sorted(p for c in calls for p in c[0]) == ["a", "b", "c"] and all(c[1] == [5] for c in calls)
