"""Every NMF kernel family across its supported shapes: 1..64 muscles, every rank 1..16, both regimes, and both sides of
the shared-memory limit of the resident kernels.

Each launch holds the 16 ranks 1..16 on one X (kmax = 16), so every K instance of a family's kernels runs once per
launch; a launch of ranks [16, 1, 9, 2] and launches of one rank alone (kmax = k) check that a problem's result does not
depend on its neighbours.  Every problem starts from explicit factors drawn like sklearn's random init (no.random_init)
and runs a fixed number of iterations (tol = 0), so kernel and numpy fp64 oracle follow the same trajectory; the oracles
are pinned to scikit-learn by the *_oracle test files.

Tolerances are those of each family's own test file:
  fp64 (cd, fixed-H, β):  |W H - W_ref H_ref|_max, |VAF| (overall and per muscle) <= TIGHT = 1e-9; err to TIGHT ||X||
                          (Frobenius) or TIGHT err_ref (β-divergence)
  fp32 (mu):              |VAF| <= VAF_TOL = 1e-4, |err| <= ERR_TOL = 1e-3 ||X||, |W H - W_ref H_ref|_max <= 5e-3
  stream vs resident:     mu 2e-5 in VAF, cd TIGHT, fixed-H bit-identical W, β 1e-10
"""
import numpy as np
import pytest

from oracle import nmf_beta_oracle as bo
from oracle import nmf_cd_oracle as co
from oracle import nmf_oracle as no
from oracle import nmf_transform_oracle as to
from test_nmf_beta_oracle import awkward_x
from test_nmf_oracle import envelopes

pytestmark = pytest.mark.gpu

TIGHT = 1e-9                       # test_nmf_cd_gpu, test_nmf_transform_gpu, test_nmf_beta_gpu
VAF_TOL, ERR_TOL, WH_MU = 1e-4, 1e-3, 5e-3  # test_nmf_gpu: fp32 against the fp64 trajectory
MU_FUSED = 2e-5                    # test_nmf_gpu: the fp32 kernel's VAF against a recomputation from its W and H
MU_STREAM = 2e-5                   # test_nmf_gpu: streaming against resident, VAF
BT_STREAM = 1e-10                  # test_nmf_beta_gpu: streaming against resident
FX_STREAM_VAF = 1e-12              # test_nmf_transform_gpu: streaming against resident, VAF (W is bit-identical)

MUSCLES = [1, 3, 4, 5, 31, 32, 33, 63, 64]
RANKS = list(range(1, 17))
MIXED = [16, 1, 9, 2]
ITERS = 30
FX_ITERS = 45                      # fixed-H streams chunks of FX_CHUNK = 32 iterations: one whole chunk, one partial
RESIDENT_N = [1, 2, 37, 200]       # plus max_rows; those above max_rows are left out
STREAM_N = [1, 37, 3 * 256 + 1]    # plus max_rows + 1; 769 rows is not a whole number of 256-row tiles
SOLO_N = 37                        # where the mixed-rank and one-rank launches run


class Family:
    def __init__(self, name, limit, kind, beta=None, solver=None):
        self.name, self.limit, self.kind, self.beta, self.solver = name, limit, kind, beta, solver
        self.iters = FX_ITERS if kind == "fixed" else ITERS
        self.zero_violation_stops = kind == "cd" or solver == "cd"
        # the streaming kernels of fixed-H and β sum in a fixed order (no floating-point atomics): repeats bit-identical
        self.stream_deterministic = kind in ("fixed", "beta", "beta-transform")

    def __repr__(self):
        return self.name


FAMILIES = [Family("mu", "ms_nmf_resident_max_rows", "mu"),
            Family("cd", "ms_nmf_cd_resident_max_rows", "cd"),
            Family("fixed-cd", "ms_nmf_fixed_h_resident_max_rows", "fixed", solver="cd"),
            Family("fixed-mu", "ms_nmf_fixed_h_resident_max_rows", "fixed", solver="mu")]
for _beta in ("kullback-leibler", "itakura-saito", 0.5):
    FAMILIES.append(Family(f"beta-{_beta}", "ms_nmf_beta_resident_max_rows", "beta", beta=_beta))
    FAMILIES.append(Family(f"beta-transform-{_beta}", "ms_nmf_beta_resident_max_rows", "beta-transform", beta=_beta))


@pytest.fixture(scope="module")
def analysis():
    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import analysis

    return analysis


def max_rows(fam, m, kmax=16):
    from muscle_synergies_b200 import _native

    return int(getattr(_native.lib(), fam.limit)(m, kmax))


def awkward(seed, n, m):
    """awkward_x of test_nmf_beta_oracle (exact zeros and entries at or below EPSILON in columns 3, 7 and 11) for any
    width: the columns taken modulo m."""
    if m >= 12:
        return awkward_x(seed, n=n, m=m)
    X = envelopes(seed, n=n, m=m)
    X[::17, 3 % m] = 0.0
    X[5::23, 7 % m] = 0.5 * bo.EPSILON
    X[9::29, 11 % m] = bo.EPSILON
    return X


def x_for(fam, n, m, seed=1):
    """Structured non-negative X; with exact zeros and sub-EPSILON entries where beta_loss > 0 allows them.  One row:
    the second row of a two-row envelope (a single row scaled to its column maxima would be all ones)."""
    if n == 1:
        return envelopes(seed, n=2, m=m)[1:]
    if fam.beta is not None and bo.beta_to_float(fam.beta) > 0:
        return awkward(seed, n, m)
    return envelopes(seed, n=n, m=m)


def starts(X, ranks):
    """(W0, H0) of rank k drawn like sklearn's init="random" with seed k: the same start for a rank in every launch."""
    return [no.random_init(X, k, k) for k in ranks]


def run(analysis, fam, X, ranks, init, regime):
    if fam.kind == "mu":
        return analysis.nmf_mu_batched(X, ranks, [0] * len(ranks), max_iter=fam.iters, tol=0.0, init=init, regime=regime)
    if fam.kind == "cd":
        return analysis.nmf_cd_batched(X, ranks, init=init, max_iter=fam.iters, tol=0.0, regime=regime)
    if fam.kind == "beta":
        return analysis.nmf_beta_batched(X, ranks, fam.beta, init=init, max_iter=fam.iters, tol=0.0, regime=regime)
    H = [h for _, h in init]
    if fam.kind == "fixed":
        return analysis.nmf_transform_batched(X, H, solver=fam.solver, max_iter=fam.iters, tol=0.0, regime=regime)
    return analysis.nmf_transform_batched(X, H, solver="mu", max_iter=fam.iters, tol=0.0, regime=regime,
                                          beta_loss=fam.beta)


def reference(fam, X, W0, H0):
    """(W, H, n_iter) of the numpy fp64 oracle from the same start."""
    if fam.kind == "mu":
        return no.mu(X, W0, H0, max_iter=fam.iters, tol=0.0)
    if fam.kind == "cd":
        return co.cd(X, W0, H0, max_iter=fam.iters, tol=0.0)
    if fam.kind == "beta":
        return bo.fit(X, W0, H0, fam.beta, fam.iters, 0.0)
    if fam.kind == "fixed":
        W, n_iter = to.transform(X, H0, fam.solver, fam.iters, 0.0)
    else:
        W, n_iter = bo.transform(X, H0, fam.beta, fam.iters, 0.0)
    return W, H0, n_iter


def divergence(fam, X, W, H):
    """What the family reports as err: ||X - W H||_F, or sklearn's sqrt(2 D_beta)."""
    if fam.beta is None:
        return np.linalg.norm(X - np.asarray(W, np.float64) @ np.asarray(H, np.float64))
    return bo.beta_divergence(X, W, H, bo.beta_to_float(fam.beta))


def divergence_rounding(fam, X, W, H):
    """A bound on the rounding of D_beta = err^2 / 2 summed in another order: n m eps times the sum of the absolute
    values of its terms (the kernel sums them element by element, sklearn as separate sums).  Where W H fits X to
    rounding, D is only that noise, and err = sqrt(2 D) turns it into ~1e-8."""
    beta = bo.beta_to_float(fam.beta)
    WH = W @ H
    keep = X > bo.EPSILON
    x, wh = X[keep], np.maximum(WH[keep], bo.EPSILON)
    if beta == 1:
        terms = WH.sum() + np.sum(x * np.abs(np.log(x / wh)) + x)
    elif beta == 0:
        terms = np.sum(x / wh + np.abs(np.log(x / wh))) + X.size
    else:
        terms = abs(beta - 1) * np.sum(WH**beta) + np.sum(x**beta + abs(beta) * x * wh ** (beta - 1))
        terms /= abs(beta * (beta - 1))
    return X.size * np.finfo(np.float64).eps * terms


def err_close(fam, got, want, X, W, H):
    """err within TIGHT of the reference: relative for a β-divergence (or, at a fit exact to rounding, D within its
    rounding), against ||X|| for the Frobenius norm."""
    if fam.beta is None:
        return abs(got - want) <= TIGHT * np.linalg.norm(X)
    return abs(got - want) <= TIGHT * want or abs(got**2 - want**2) / 2 <= divergence_rounding(fam, X, W, H)


def check_invariants(fam, res, X, ranks):
    n, m = X.shape
    # tol = 0: coordinate descent stops early only where its violation is exactly zero (sklearn does too)
    assert (res.n_iter == fam.iters).all() or (fam.zero_violation_stops and (res.n_iter <= fam.iters).all()), res.n_iter
    for p, k in enumerate(ranks):
        W, H = res.W[p], res.H[p]
        assert W.shape == (n, k) and H.shape == (k, m), (p, W.shape, H.shape)
        assert np.isfinite(W).all() and np.isfinite(H).all() and (W >= 0).all() and (H >= 0).all(), p
        # the fused VAF and err equal a recomputation from the returned factors
        got_all, got_cols = no.vaf(X, W, H)
        fused = MU_FUSED if fam.kind == "mu" else TIGHT
        assert abs(res.vaf[p, 0] - got_all) <= fused and np.abs(res.vaf[p, 1:] - got_cols).max() <= fused, p
        want = divergence(fam, X, W, H)
        if fam.kind == "mu":  # test_nmf_gpu: the fp32 kernel's err against a recomputation
            assert abs(res.err[p] - want) <= 1e-5 * np.linalg.norm(X), (p, res.err[p], want)
        else:
            assert err_close(fam, res.err[p], want, X, W, H), (p, res.err[p], want)


def check_oracle(fam, res, p, X, ref):
    W_ref, H_ref, n_ref = ref
    if n_ref < fam.iters:
        # coordinate descent at tol = 0 stops where every projected gradient is exactly zero - in sklearn's (and the
        # oracle's) rounding, a product and then a sum.  The kernels form each gradient with fused multiply-adds, which
        # keep the last bits of that difference, so they run on to max_iter from the same fixed point: each further
        # sweep moves W by the rounding of a zero gradient, and W H still agrees to TIGHT below.
        assert fam.zero_violation_stops and res.n_iter[p] in (n_ref, fam.iters), (res.n_iter[p], n_ref)
    else:
        assert res.n_iter[p] == n_ref, (res.n_iter[p], n_ref)
    want_all, want_cols = no.vaf(X, W_ref, H_ref)
    WH = np.asarray(res.W[p], np.float64) @ np.asarray(res.H[p], np.float64)
    dwh = np.abs(WH - W_ref @ H_ref).max()
    dvaf = max(abs(res.vaf[p, 0] - want_all), np.abs(res.vaf[p, 1:] - want_cols).max())
    want = divergence(fam, X, W_ref, H_ref)
    if fam.kind == "mu":
        ok = dwh <= WH_MU and dvaf <= VAF_TOL and abs(res.err[p] - want) <= ERR_TOL * np.linalg.norm(X)
    else:
        ok = dwh <= TIGHT and dvaf <= TIGHT and err_close(fam, res.err[p], want, X, W_ref, H_ref)
    assert ok, (fam, X.shape, int(res.ranks[p]), dwh, dvaf, res.err[p], want)


def bits_equal(a, b, p, q=None):
    q = p if q is None else q
    return (np.array_equal(a.W[p], b.W[q]) and np.array_equal(a.H[p], b.H[q]) and a.n_iter[p] == b.n_iter[q]
            and np.array_equal(a.err[p], b.err[q]) and np.array_equal(a.vaf[p], b.vaf[q]))


def check_same_problem(fam, regime, a, p, b, q):
    """Problem p of launch a against problem q of launch b (the same X, rank and start), other neighbours or kmax."""
    if regime == "resident":
        assert bits_equal(a, b, p, q), (fam, regime, p, q)
        return
    if fam.kind == "mu":  # W^T W, W^T X summed with atomics over a grid sized by the batch
        assert a.n_iter[p] == b.n_iter[q] and np.abs(a.vaf[p] - b.vaf[q]).max() <= MU_STREAM, (p, q)
    elif fam.kind == "cd":  # the same, in fp64
        assert a.n_iter[p] == b.n_iter[q]
        assert np.abs(a.W[p] @ a.H[p] - b.W[q] @ b.H[q]).max() <= TIGHT and np.abs(a.vaf[p] - b.vaf[q]).max() <= TIGHT
    elif fam.kind == "fixed":  # rows independent, W bit-identical; the VAF's CTA partials follow the grid
        assert a.n_iter[p] == b.n_iter[q] and np.array_equal(a.W[p], b.W[q]), (p, q)
        assert np.abs(a.vaf[p] - b.vaf[q]).max() <= FX_STREAM_VAF, (p, q)
    else:  # β: the H-step partials follow the tile height (kmax) and the grid
        assert a.n_iter[p] == b.n_iter[q]
        assert np.abs(a.W[p] - b.W[q]).max() <= BT_STREAM and np.abs(a.H[p] - b.H[q]).max() <= BT_STREAM, (p, q)
        assert np.abs(a.vaf[p] - b.vaf[q]).max() <= BT_STREAM and abs(a.err[p] - b.err[q]) <= BT_STREAM * a.err[p]


@pytest.mark.parametrize("m", MUSCLES)
@pytest.mark.parametrize("fam", FAMILIES, ids=repr)
def test_every_rank_both_regimes_and_the_shared_memory_limit(analysis, fam, m):
    from muscle_synergies_b200._native import NativeError

    limit = max_rows(fam, m)
    assert limit > SOLO_N
    resident = sorted({n for n in RESIDENT_N if n <= limit} | {limit})
    stream = sorted(set(STREAM_N) | {limit + 1})
    for n in sorted(set(resident) | set(stream)):
        X = x_for(fam, n, m)
        init = starts(X, RANKS)
        refs = [reference(fam, X, *init[p]) for p in range(len(RANKS))]
        for regime in ("resident", "stream"):
            if n not in (resident if regime == "resident" else stream):
                continue
            res = run(analysis, fam, X, RANKS, init, regime)
            check_invariants(fam, res, X, RANKS)
            for p in range(len(RANKS)):
                check_oracle(fam, res, p, X, refs[p])
            deterministic = regime == "resident" or fam.stream_deterministic
            if deterministic and n in (limit, limit + 1):  # no floating-point atomics: a repeat is bit-identical
                again = run(analysis, fam, X, RANKS, init, regime)
                assert all(bits_equal(res, again, p) for p in range(len(RANKS))), (fam, m, n, regime)
            if n == limit:  # by size, the largest resident n stays resident ...
                auto = run(analysis, fam, X, RANKS, init, None)
                assert all(bits_equal(res, auto, p) for p in range(len(RANKS))), (fam, m, n)
            if n == limit + 1:  # ... and one row more streams; the resident kernel refuses it
                auto = run(analysis, fam, X, RANKS, init, None)
                for p in range(len(RANKS)):
                    if deterministic:
                        assert bits_equal(res, auto, p), (fam, m, n, p)
                    else:
                        check_same_problem(fam, regime, res, p, auto, p)
                with pytest.raises(NativeError):
                    run(analysis, fam, X, RANKS, init, "resident")
            if n == SOLO_N:
                # neighbours: ranks [16, 1, 9, 2] in one launch, and every rank alone (kmax = k)
                mixed = run(analysis, fam, X, MIXED, [init[k - 1] for k in MIXED], regime)
                check_invariants(fam, mixed, X, MIXED)
                for q, k in enumerate(MIXED):
                    check_same_problem(fam, regime, res, k - 1, mixed, q)
                for k in RANKS:
                    alone = run(analysis, fam, X, [k], [init[k - 1]], regime)
                    check_same_problem(fam, regime, res, k - 1, alone, 0)


def gram_tolerance(X, k):
    """How far two exact fp64 NNDSVDs may differ: the device takes V from a Jacobi eigen-solve of X^T X, the oracle from
    LAPACK's SVD of X.  An eigenvector of X^T X is determined to about eps lambda_1 / gap, gap = the distance from its
    eigenvalue to the nearest other (Davis-Kahan); 32 >= sqrt(769) covers the rounding of Gram sums over up to 769 rows,
    which grows like a random walk.  Where that is below TIGHT, TIGHT stands."""
    lam = np.sort(np.linalg.eigvalsh(X.T @ X))[::-1]
    gap = min(min(lam[j - 1] - lam[j] if j > 0 else np.inf, lam[j] - lam[j + 1] if j + 1 < len(lam) else np.inf)
              for j in range(k))
    return max(TIGHT, 32 * np.finfo(np.float64).eps * lam[0] / gap)


@pytest.mark.parametrize("m", [2, 5, 33, 64])
@pytest.mark.parametrize("n", [37, 3 * 256 + 1])
def test_device_nndsvd_at_every_width(analysis, m, n):
    """The exact SVD behind init="nndsvd"/"nndsvda" (X^T X over 256-row tiles, Jacobi on the m x m Gram matrix) against
    nndsvd_exact, for every rank up to min(n, m, 16)."""
    X = envelopes(2, n=n, m=m)
    ranks = list(range(1, min(n, m, 16) + 1))
    for variant in ("nndsvd", "nndsvda"):
        res = analysis.nmf_cd_batched(X, ranks, init=variant, max_iter=0, tol=0.0)
        for p, k in enumerate(ranks):
            W, H = co.nndsvd_exact(X, k, variant)
            tol = gram_tolerance(X, k)
            assert np.abs(res.W[p] - W).max() <= tol * np.abs(W).max(), (variant, m, n, k)
            assert np.abs(res.H[p] - H).max() <= tol * np.abs(H).max(), (variant, m, n, k)
