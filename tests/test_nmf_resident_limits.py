"""The resident row limits of the NMF kernels (ms_*_resident_max_rows, pure host code: no GPU needed).  They route
regime=None between each family's resident kernel, which holds a problem in one CTA's shared memory, and its streaming
kernels."""
import numpy as np


def _pad4(v):
    return (v + 3) & ~3


def _mu_stride(padded):
    return padded if (padded >> 2) & 1 else padded + 4


def _odd(v):
    return v | 1


# dynamic shared memory of each resident launch of n rows, restated from the launch code in bytes
RESIDENT_SMEM = {
    # ms_nmf.cu: sX [n][stride(MP)], sW [n][stride(KP)], sHt [MP][KP], sH [kmax][MP], sHHt [kmax][KP], sWtW [KP][KP],
    # sWtX [KP][MP], sPart [256 * 16], s_red [32] floats
    "ms_nmf_resident_max_rows": lambda n, m, k: 4 * (
        n * (_mu_stride(_pad4(m)) + _mu_stride(_pad4(k))) + _pad4(m) * _pad4(k) + k * _pad4(m) + k * _pad4(k)
        + _pad4(k) * _pad4(k) + _pad4(k) * _pad4(m) + 256 * 16 + 32),
    # ms_nmf_cd.cu: sX [n][odd(m)], sW [n][odd(kmax)], sH, sWtX [kmax][m], sHHt, sWtW [kmax][kmax],
    # sPart [max(256, kmax^2 + kmax m)], s_red [64] doubles
    "ms_nmf_cd_resident_max_rows": lambda n, m, k: 8 * (
        n * (_odd(m) + _odd(k)) + 2 * k * m + 2 * k * k + max(256, k * k + k * m) + 64),
    # ms_nmf_fixed.cu: sX [n][odd(m)], sW and sXHt [n][odd(kmax)], sXX [n], sH [kmax][m], sHHt [kmax][kmax],
    # sPart [2][64], s_red [32] doubles
    "ms_nmf_fixed_h_resident_max_rows": lambda n, m, k: 8 * (
        n * (_odd(m) + 2 * _odd(k) + 1) + k * m + k * k + 2 * 64 + 32),
    # ms_nmf_beta.cu: sX, sF, sG [n][odd(m)], sW [n][odd(kmax)], sH [kmax][m], sHs [kmax], sPart [2][64], s_red [32] doubles
    "ms_nmf_beta_resident_max_rows": lambda n, m, k: 8 * (n * (3 * _odd(m) + _odd(k)) + k * m + k + 2 * 64 + 32),
}


def test_nmf_resident_row_limits_fit_shared_memory():
    """0 outside m in 1..64, kmax in 1..16; inside, positive, never larger for more muscles or a larger rank, and the
    largest n whose launch fits the 226 KiB budget, so the request stays within the 227 KiB a B200 block may opt into."""
    from muscle_synergies_b200 import _native

    lib = _native.lib()
    for name, smem in RESIDENT_SMEM.items():
        limit = getattr(lib, name)
        for m, k in [(0, 4), (-1, 4), (65, 4), (1000, 4), (16, 0), (16, -3), (16, 17), (0, 0), (65, 17)]:
            assert limit(m, k) == 0, (name, m, k)
        rows = np.array([[limit(m, k) for k in range(1, 17)] for m in range(1, 65)])
        assert (rows > 0).all(), name
        assert (np.diff(rows, axis=0) <= 0).all() and (np.diff(rows, axis=1) <= 0).all(), name
        for m in range(1, 65):
            for k in range(1, 17):
                n = int(rows[m - 1, k - 1])
                assert smem(n, m, k) <= 226 * 1024 < smem(n + 1, m, k), (name, m, k, n)


