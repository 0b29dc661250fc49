"""Pins oracle/emg_oracle.py against the reference preprocessing functions: live where a reference checkout is present,
and against their stored outputs (tests/golden/emg_pinning.npz) everywhere."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import emg_oracle as eo
from oracle import make_golden as mg
from oracle.refstub import reference_available


def golden():
    with np.load(os.path.join(GOLDEN, "emg_pinning.npz")) as z:
        return {k: z[k] for k in z.files}


def assert_matches_golden(outputs, gold):
    """The stored rows of every output.  1e-12 relative: the stored values come from another numpy / scipy build,
    whose vectorised sums (np.convolve's dot products) may add in another order."""
    assert sorted(outputs) == sorted(k for k in gold if k not in ("input", "source"))
    for name, a in outputs.items():
        want = gold[name]
        got = a[mg.emg_golden_rows(len(a))]
        assert got.shape == want.shape, name
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max(), err_msg=name)


def test_oracle_equals_reference_golden():
    gold = golden()
    x = mg.emg_pinning_input()
    assert np.array_equal(x[mg.emg_golden_rows(len(x))], gold["input"])  # the seeded input is the one recorded
    assert_matches_golden(mg.emg_oracle_outputs(x), gold)


@pytest.mark.reference
@pytest.mark.skipif(not reference_available(), reason="reference checkout not present")
def test_oracle_equals_reference_functions():
    from oracle.refstub import import_reference

    ms, _ = import_reference()
    x = mg.emg_pinning_input()
    want = mg.emg_reference_outputs(ms, x)
    got = mg.emg_oracle_outputs(x)
    assert sorted(got) == sorted(want)
    for name in want:  # the oracle makes the reference's numpy / scipy calls
        assert np.array_equal(want[name], got[name]), name
    assert_matches_golden(want, golden())


def test_same_convolution_window_alignment():
    x = np.zeros((50, 1))
    x[20, 0] = 3.0
    out = eo.rms(x, 10)[:, 0]
    # np.convolve "same" with an even window: sample 20 contributes to outputs 16..25
    assert np.flatnonzero(out).tolist() == list(range(16, 26))
