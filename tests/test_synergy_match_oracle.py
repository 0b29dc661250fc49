"""Pins oracle/synergy_match_oracle.py (unit-length synergies, scipy's linear_sum_assignment) against a search over
every permutation, checks its zero-norm rule, and checks every argument error of match_synergies_batched and the
host-side argument checks of ms_synergy_match - all without a GPU."""
import ctypes

import numpy as np
import pytest

from oracle import synergy_match_oracle as so


def random_sets(k, m=16, seed=0):
    rng = np.random.default_rng(seed)
    return rng.uniform(0, 1, (k, m)), rng.uniform(0, 1, (k, m))


def tie_heavy_sets(k, m=16, seed=0):
    """Identical sets, sets with duplicated rows, and a permuted copy with duplicated rows: many optimal pairings."""
    rng = np.random.default_rng(seed)
    A = rng.uniform(0, 1, (k, m))
    dup = A.copy()
    dup[k // 2:] = A[0]
    yield A, A.copy()
    yield dup, dup.copy()
    yield dup, dup[rng.permutation(k)]
    yield np.ones((k, m)), np.ones((k, m))


@pytest.mark.parametrize("k", range(1, 8))
def test_oracle_total_equals_brute_force(k):
    for seed in range(5):
        A, B = random_sets(k, seed=seed)
        mean, sim, perm = so.match(A, B)
        assert sorted(perm.tolist()) == list(range(k))
        assert abs(sim.sum() - so.brute_force(so.similarity(A, B))) <= 1e-12
        assert abs(mean * k - sim.sum()) <= 1e-12
    for A, B in tie_heavy_sets(k, seed=k):
        mean, sim, perm = so.match(A, B)
        assert sorted(perm.tolist()) == list(range(k))
        assert abs(sim.sum() - so.brute_force(so.similarity(A, B))) <= 1e-12


def test_identical_sets_match_with_similarity_one():
    A, _ = random_sets(6, seed=3)
    mean, sim, perm = so.match(A, A[::-1])
    assert np.abs(sim - 1).max() <= 1e-12 and abs(mean - 1) <= 1e-12
    assert perm.tolist() == list(range(5, -1, -1))


def test_zero_norm_rule():
    A, B = random_sets(4, seed=1)
    A[2] = 0.0
    B[0] = 0.0
    S = so.similarity(A, B)
    assert np.isfinite(S).all()
    assert (S[2] == 0).all() and (S[:, 0] == 0).all()
    mean, sim, perm = so.match(A, B)
    assert np.isfinite(sim).all() and sorted(perm.tolist()) == [0, 1, 2, 3]
    assert abs(sim.sum() - so.brute_force(S)) <= 1e-12
    zero = np.zeros((3, 5))
    assert so.match(zero, zero)[0] == 0.0


def test_match_argument_errors_need_no_device():
    from muscle_synergies_b200.analysis import match_synergies_batched

    A, B = random_sets(3, m=8)
    good = [A, B, A[:2]]
    nan = A.copy()
    nan[1, 2] = np.nan
    inf = A.copy()
    inf[0, 0] = np.inf
    for args, kw, msg in [
        (([A, B, A[:2]], [[0, 2]]), {}, r"pair 0 compares H\[0\] \(rank 3\) with H\[2\] \(rank 2\)"),
        (([A, B, A[:2]],), {}, "mixes ranks"),
        (([A, np.ones((17, 8))],), {}, r"H\[1\] has rank k = 17"),
        ((np.ones((2, 17, 8)),), {}, r"H\[0\] has rank k = 17"),
        (([np.ones((2, 65)), np.ones((2, 65))],), {}, "m = 65 muscles"),
        ((np.ones((2, 3, 65)),), {}, "m = 65 muscles"),
        (([A, B[:, :7]],), {}, r"H\[1\] has m = 7 muscles, H\[0\] has 8"),
        (([A, nan],), {}, r"H\[1\] contains a non-finite entry"),
        (([inf, B],), {}, r"H\[0\] contains a non-finite entry"),
        ((good, [[0, 3]]), {}, r"pair 0 = \(0, 3\) names a set H does not have"),
        ((good, [[-1, 0]]), {}, "names a set H does not have"),
        ((good, [0, 1]), {}, r"\(P, 2\) integer array"),
        ((good, [[0.0, 1.0]]), {}, r"\(P, 2\) integer array"),
        (([A, np.ones(8)],), {}, r"H\[1\] must be a \(k, m\) synergy set"),
        (([],), {}, "no synergy set"),
        ((np.ones((3, 8)),), {}, r"\(S, k, m\) stack"),
        (([np.ones((0, 8)), np.ones((0, 8))],), {}, r"H\[0\] has rank k = 0"),
    ]:
        with pytest.raises(ValueError, match=msg):
            match_synergies_batched(*args, **kw)


def test_native_entry_checks_its_scalar_arguments_without_a_device():
    """ms_synergy_match refuses m and kmax outside 1..64 / 1..16 before any CUDA call; no pairs is a no-op."""
    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import _native

    lib = _native.lib()
    dummy = ctypes.c_void_p(64)
    wb = int(lib.ms_synergy_match_workspace_bytes(4))
    assert wb >= 4 * 16 * 8
    call = lambda m, kmax, n_pairs=1, work=wb: lib.ms_synergy_match(dummy, m, dummy, 4, kmax, dummy, n_pairs, None,  # noqa: E731
                                                                   None, dummy, dummy, work, None)
    for m, kmax in [(0, 4), (65, 4), (16, 0), (16, 17)]:
        assert call(m, kmax) == -1, (m, kmax)
    assert call(16, 4, n_pairs=-1) == -1
    assert call(16, 4, work=wb - 1) == -3  # MS_E_WORKSPACE
    assert call(16, 4, n_pairs=0) == 0
    # no pair list: every pair a < b of the 4 sets, so n_pairs must be 6
    no_list = lambda n_pairs: lib.ms_synergy_match(dummy, 16, dummy, 4, 4, None, n_pairs, None, None, dummy,  # noqa: E731
                                                   dummy, wb, None)
    assert no_list(5) == -1 and no_list(7) == -1
