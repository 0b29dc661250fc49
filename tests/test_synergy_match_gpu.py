"""Matched cosine similarity of synergy sets (match_synergies_batched, pipeline.synergy_similarity;
csrc/ms_synmatch.cu) against oracle/synergy_match_oracle.py (numpy unit rows + scipy's linear_sum_assignment).

Tolerances: mean and per-synergy similarity within 1e-12 of the oracle; the pairing equal to scipy's where the optimum
is unique (continuous random sets), and otherwise a permutation that reaches the oracle's total to 1e-12.
"""
import numpy as np
import pytest

from oracle import synergy_match_oracle as so

pytestmark = pytest.mark.gpu

TOL = 1e-12


@pytest.fixture(scope="module")
def analysis():
    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import analysis

    return analysis


def check_against_oracle(res, sets, pairs, unique=True):
    """res: a SynergyMatch with sim and perm, as numpy."""
    for p, (a, b) in enumerate(pairs):
        k = sets[a].shape[0]
        mean, sim, perm = so.match(sets[a], sets[b])
        got_perm = res.perm[p, :k].astype(np.int64)
        assert abs(res.mean[p] - mean) <= TOL, (p, res.mean[p], mean)
        assert sorted(got_perm.tolist()) == list(range(k)), (p, got_perm)
        S = so.similarity(sets[a], sets[b])
        assert np.abs(res.sim[p, :k] - S[np.arange(k), got_perm]).max() <= TOL, p
        assert abs(res.sim[p, :k].sum() - sim.sum()) <= TOL * k, p
        if unique:
            assert np.array_equal(got_perm, perm), (p, got_perm, perm)
            assert np.abs(res.sim[p, :k] - sim).max() <= TOL, p
        assert (res.perm[p, k:] == -1).all() and np.isnan(res.sim[p, k:]).all()


@pytest.mark.parametrize("m", [1, 8, 16, 64])
def test_random_sets_match_scipy(analysis, m):
    rng = np.random.default_rng(m)
    for k in range(1, 17):
        sets = rng.uniform(0, 1, (6, k, m))
        res = analysis.match_synergies_batched(sets, similarities=True, permutations=True)
        pairs = list(zip(*np.triu_indices(6, 1)))
        assert res.mean.shape == (15,) and res.sim.shape == (15, k) and res.perm.shape == (15, k)
        assert res.perm.dtype == np.int8
        # m = 1: every unit vector is (1,), S is all ones and every pairing is optimal
        check_against_oracle(res, sets, pairs, unique=m > 1 or k == 1)


def tie_sets(k, m, seed):
    rng = np.random.default_rng(seed)
    A = rng.uniform(0, 1, (k, m))
    dup = A.copy()
    dup[k // 2:] = A[0]
    zero = A.copy()
    zero[::3] = 0.0
    return [A, A.copy(), A[rng.permutation(k)], dup, dup[rng.permutation(k)], zero, zero[rng.permutation(k)],
            np.zeros((k, m))]


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 13, 16])
def test_tie_cases_reach_the_optimum(analysis, k):
    sets = tie_sets(k, 16, k)
    pairs = [(0, 1), (0, 2), (3, 3), (3, 4), (5, 6), (5, 5), (7, 7), (0, 7), (4, 7)]
    res = analysis.match_synergies_batched(sets, pairs, similarities=True, permutations=True)
    check_against_oracle(res, sets, pairs, unique=False)
    for p in (0, 1, 2, 3):  # identical sets, in any row order, duplicated rows included
        assert np.abs(res.sim[p] - 1).max() <= TOL and abs(res.mean[p] - 1) <= TOL, p
    assert res.mean[6] == 0.0 and res.mean[7] == 0.0  # zero rows: similarity 0, never NaN
    assert np.isfinite(res.sim).all()


def test_mixed_ranks_one_launch_and_cuda_input(analysis):
    import torch

    rng = np.random.default_rng(7)
    sets = [rng.uniform(0, 1, (k, 16)) for k in range(1, 17) for _ in range(3)]
    pairs = [(3 * (k - 1) + i, 3 * (k - 1) + j) for k in range(1, 17) for i in range(3) for j in range(3)]
    host = analysis.match_synergies_batched(sets, pairs, similarities=True, permutations=True)
    assert host.sim.shape == (len(pairs), 16)
    check_against_oracle(host, sets, pairs, unique=False)
    off = [p for p, (a, b) in enumerate(pairs) if a != b]
    oracle_perm = [so.match(sets[pairs[p][0]], sets[pairs[p][1]])[2] for p in off]
    assert all(np.array_equal(host.perm[p, :len(q)], q) for p, q in zip(off, oracle_perm))
    # a list of CUDA tensors and CUDA pairs: results stay on the device, bit for bit the host input's
    dev = analysis.match_synergies_batched([torch.from_numpy(s).cuda() for s in sets], torch.tensor(pairs).cuda(),
                                           similarities=True, permutations=True)
    assert dev.mean.is_cuda and dev.sim.is_cuda and dev.perm.is_cuda
    assert np.array_equal(dev.mean.cpu().numpy().view(np.uint64), host.mean.view(np.uint64))
    assert np.array_equal(dev.sim.cpu().numpy(), host.sim, equal_nan=True)
    assert np.array_equal(dev.perm.cpu().numpy(), host.perm)
    # a strided CUDA stack (a transposed view) and float32 input are read as they are given
    stack = rng.uniform(0, 1, (10, 16, 6))  # (S, m, k)
    view = torch.from_numpy(stack).cuda().transpose(1, 2)
    assert not view.is_contiguous()
    a = analysis.match_synergies_batched(view, similarities=True, permutations=True)
    b = analysis.match_synergies_batched(np.ascontiguousarray(stack.transpose(0, 2, 1)), similarities=True,
                                         permutations=True)
    assert np.array_equal(a.mean.cpu().numpy(), b.mean) and np.array_equal(a.perm.cpu().numpy(), b.perm)
    check_against_oracle(b, list(stack.transpose(0, 2, 1)), list(zip(*np.triu_indices(10, 1))))
    f32 = analysis.match_synergies_batched(view.float())
    want = analysis.match_synergies_batched(view.float().double())
    assert torch.equal(f32.mean, want.mean)


def test_repeats_and_optional_outputs_are_bit_identical(analysis):
    rng = np.random.default_rng(11)
    sets = rng.uniform(0, 1, (40, 8, 16))
    full = analysis.match_synergies_batched(sets, similarities=True, permutations=True)
    for kw in ({}, {"similarities": True}, {"permutations": True}, {"similarities": True, "permutations": True}):
        again = analysis.match_synergies_batched(sets, **kw)
        assert np.array_equal(again.mean.view(np.uint64), full.mean.view(np.uint64)), kw
        if kw.get("similarities"):
            assert np.array_equal(again.sim.view(np.uint64), full.sim.view(np.uint64))
        else:
            assert again.sim is None
        if kw.get("permutations"):
            assert np.array_equal(again.perm, full.perm)
        else:
            assert again.perm is None


def test_large_all_pairs_run(analysis):
    import torch

    S, k, m = 2000, 8, 16
    sets = np.random.default_rng(5).uniform(0, 1, (S, k, m))
    res = analysis.match_synergies_batched(torch.from_numpy(sets).cuda())
    P = S * (S - 1) // 2
    assert res.mean.shape == (P,) and res.sim is None and res.perm is None
    mean = res.mean.cpu().numpy()
    a, b = np.triu_indices(S, 1)
    for p in np.random.default_rng(6).choice(P, 2000, replace=False):
        assert abs(mean[p] - so.match(sets[a[p]], sets[b[p]])[0]) <= TOL, p
    # the kernel's own all-pairs order is np.triu_indices's: the same means as the explicit pair list
    head = torch.from_numpy(sets[:300]).cuda()
    implicit = analysis.match_synergies_batched(head, permutations=True)
    explicit = analysis.match_synergies_batched(head, np.stack(np.triu_indices(300, 1), axis=1), permutations=True)
    assert torch.equal(implicit.mean, explicit.mean) and torch.equal(implicit.perm, explicit.perm)


def test_huge_finite_entries_give_the_oracle_s_similarity(analysis):
    """Rows whose squared norm overflows have similarity 0 (the oracle's unit rows are then 0), and rows whose norm
    is finite but large are compared exactly: no inf or NaN reaches the matching."""
    rng = np.random.default_rng(13)
    big = np.full((2, 4), 1e200)
    huge = np.full((3, 4), 1e308)
    mixed = rng.uniform(0, 1, (3, 4))
    mixed[1] = 1e300
    scaled = rng.uniform(0, 1, (3, 4)) * 1e10
    large = rng.uniform(0.5, 1, (3, 4)) * 1e153  # squared norm ~1e306: finite
    small = rng.uniform(0, 1, (3, 4))
    sets = [big, big.copy(), huge, huge.copy(), mixed, scaled, large, small, large[::-1].copy()]
    pairs = [(0, 1), (2, 3), (4, 5), (5, 4), (6, 7), (6, 8), (4, 7)]
    res = analysis.match_synergies_batched(sets, pairs, similarities=True, permutations=True)
    check_against_oracle(res, sets, pairs, unique=False)
    assert res.mean[0] == 0.0 and res.mean[1] == 0.0
    assert res.sim[2, 1] == 0.0  # the 1e300 row of `mixed` matches at 0
    assert np.isfinite(res.sim[0, :2]).all() and np.isfinite(res.sim[1:]).all() and abs(res.mean[5] - 1) <= TOL


def test_native_entry_refuses_bad_device_tables(analysis):
    """Ranks and pairs live on the device: the entry finds an unequal-rank pair, a pair index outside the table and a
    rank above kmax there and returns MS_E_INVALID, with NaN for the pairs it refused."""
    import torch

    from muscle_synergies_b200 import _native as nat

    lib = nat.lib()
    H = torch.rand(7 * 16, dtype=torch.float64, device="cuda")
    table = torch.tensor([[0, 3], [48, 3], [96, 1]], dtype=torch.int64, device="cuda")
    work = torch.empty(int(lib.ms_synergy_match_workspace_bytes(3)), dtype=torch.uint8, device="cuda")
    mean = torch.empty(3, dtype=torch.float64, device="cuda")

    def call(pairs, tab=table, kmax=3):
        p = torch.tensor(pairs, dtype=torch.int32, device="cuda")
        rc = lib.ms_synergy_match(H.data_ptr(), 16, tab.data_ptr(), 3, kmax, p.data_ptr(), len(pairs), None, None,
                                  mean.data_ptr(), work.data_ptr(), work.numel(), None)
        torch.cuda.synchronize()
        return rc

    assert call([[0, 1], [2, 2], [1, 0]]) == 0 and torch.isfinite(mean).all()
    assert call([[0, 1], [0, 2], [1, 1]]) == -1
    assert torch.isnan(mean[1]) and torch.isfinite(mean[[0, 2]]).all()
    assert call([[0, 1], [0, 3], [1, 1]]) == -1
    assert call([[0, 1]], tab=torch.tensor([[0, 3], [48, 3], [96, 17]], dtype=torch.int64, device="cuda")) == -1
    assert call([[0, 1]], kmax=2) == -1
    assert call([[0, 1], [2, 2]]) == 0  # and the next call is clean again


def test_synergy_similarity_on_the_synthetic_trial(analysis):
    import muscle_synergies_b200 as ms
    from muscle_synergies_b200.pipeline import synergy_similarity, trial_synergies
    from tools.synth_vicon import synth_layout

    data = ms.load_vicon_bytes(synth_layout("D", seed=0), name="D")
    trial = trial_synergies(data, 1, 8, max_iter=500, tol=1e-4, window_size=0.05, solver="cd")
    table = synergy_similarity(trial)
    assert table.shape == (64, 8) and list(table.index.names) == ["n_components", "trecho", "cycle"]
    assert list(table.columns.names) == ["trecho", "cycle"]
    values = table.to_numpy().reshape(8, 8, 8)
    assert np.array_equal(values, values.transpose(0, 2, 1))  # exactly symmetric, rank by rank
    for k in range(1, 9):
        for src in trial.cycles:
            A = src.components[k].to_numpy()
            for tgt in trial.cycles:
                want = so.match(A, tgt.components[k].to_numpy())[0]
                got = table.loc[(k, src.trecho.value, src.cycle.value), (tgt.trecho.value, tgt.cycle.value)]
                assert abs(got - want) <= TOL, (k, src.trecho, src.cycle, tgt.trecho, tgt.cycle)
