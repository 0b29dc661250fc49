"""Argument checks shared by the four NMF entries (nmf_mu_batched, nmf_cd_batched, nmf_beta_batched,
nmf_transform_batched) and by the C ABI's host-side table builder: bad arguments are refused before any device work."""
import ctypes

import numpy as np
import pytest

from test_nmf_oracle import envelopes

FAMILIES = ("mu", "cd", "beta", "transform")
# (case, arguments, message, the entries that take the argument)
SHARED_ERRORS = [("regime", {"regime": "auto"}, "regime", FAMILIES), ("max_iter", {"max_iter": -1}, "max_iter", FAMILIES),
                 ("x_index", {"x_index": [1]}, "x_index", FAMILIES),
                 ("rank17", {"ranks": [17]}, "1..16", ("mu", "cd", "beta")),
                 ("rank17", {"ranks": [17]}, "1 <= k <= 16", ("transform",)),
                 ("init_shape", {"init": [(np.ones((5, 2)), np.ones((2, 8)))]}, "shapes", ("mu", "cd", "beta")),
                 ("init_name", {"init": "custom"}, "init must be", ("cd", "beta"))]


def call_entry(family, X, ranks=(2,), **kw):
    """One NMF entry point on X with the given ranks (the transform's synergies have those ranks)."""
    from muscle_synergies_b200 import analysis

    ranks = list(ranks)
    if family == "mu":
        return analysis.nmf_mu_batched(X, ranks, [0] * len(ranks), **kw)
    if family == "cd":
        return analysis.nmf_cd_batched(X, ranks, **kw)
    if family == "beta":
        return analysis.nmf_beta_batched(X, ranks, "kullback-leibler", **kw)
    return analysis.nmf_transform_batched(X, [np.ones((k, X.shape[1])) for k in ranks], **kw)


@pytest.mark.parametrize("family,kw,msg", [pytest.param(f, kw, msg, id=f"{f}-{case}")
                                           for case, kw, msg, families in SHARED_ERRORS for f in families])
def test_nmf_argument_errors_need_no_device(family, kw, msg):
    """Every NMF entry refuses a bad argument with a ValueError before it asks for a device."""
    with pytest.raises(ValueError, match=msg):
        call_entry(family, envelopes(0, m=8), **kw)


def test_mu_stream_refuses_a_negative_matrix_index_before_any_cuda_call():
    """ms_nmf_mu_stream builds its problem table on the host before it copies anything: a negative x_index is
    MS_E_INVALID, and the device pointers (placeholders here) are never used."""
    from muscle_synergies_b200 import _native

    lib = ctypes.CDLL(_native.LIB_PATH)
    vp, i32, i32p = ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)
    lib.ms_nmf_mu_stream.restype = ctypes.c_int
    lib.ms_nmf_mu_stream.argtypes = [vp, ctypes.c_int64, i32, i32p, i32p, i32, vp, vp, i32, ctypes.c_float, i32, vp, vp,
                                     vp, vp, vp]
    ranks = np.array([2, 3], dtype=np.int32)
    xi = np.array([0, -1], dtype=np.int32)
    fake = vp(256)  # never dereferenced on this path
    rc = lib.ms_nmf_mu_stream(fake, 200, 16, ranks.ctypes.data_as(i32p), xi.ctypes.data_as(i32p), 2, fake, fake, 10,
                              0.0, 10, fake, fake, fake, fake, None)
    assert rc == -1  # MS_E_INVALID
