"""Pins oracle/segment_oracle.py against the reference Segmenter: its stored output (golden) everywhere, and live
where a reference checkout is present."""
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import make_golden as mg
from oracle import segment_oracle as so
from oracle import vicon_oracle_fast as vof
from oracle.refstub import reference_available
from tools.synth_vicon import synth_layout


@pytest.fixture(scope="module")
def d_arrays():
    return vof.parse(synth_layout("D", seed=0))


def test_transitions_and_windows_match_reference(d_arrays):
    gold = json.load(open(os.path.join(GOLDEN, "segment_D.json")))
    dev, _traj = d_arrays
    left, right = dev[:, 2], dev[:, 11]  # Fz of plate 1 and plate 2
    t = so.transition_indices(left, right)
    assert t == gold["transitions"]
    got = so.organize(t, left, right, 20)
    assert len(got) == len(gold["windows"]) == 32
    names = {0: "FIRST", 1: "SECOND", 2: "THIRD", 3: "FOURTH"}
    for g, w in zip(got, gold["windows"]):
        assert names[g["trecho"]] == w["trecho"] and names[g["cycle"]] == w["cycle"]
        assert g["phase"] == w["phase"] and g["order"] == w["order"]
        assert list(g["start"]) == w["start"] and list(g["stop"]) == w["stop"]
        a, b = so.window_rows(1, g["start"], g["stop"], 20)
        assert [b - a, 8] == w["emg_shape"]
        a, b = so.window_rows(2, g["start"], g["stop"], 20)
        assert [b - a, 3] == w["traj0_shape"]


def test_transition_search_matches_reference_golden():
    """Runs shorter than min_phase_size, fewer alternations than asked for: the stored results of the transition
    search on seeded on/off signals."""
    gold = json.load(open(os.path.join(GOLDEN, "segment_pinning.json")))["cases"]
    cases = list(mg.segment_pinning_cases())
    assert len(cases) == len(gold)
    for (left, right, k), want in zip(cases, gold):
        assert (len(left), k) == (want["n"], want["k"])
        assert so.transition_indices(left, right, 10, k) == want["transitions"]


@pytest.mark.reference
@pytest.mark.skipif(not reference_available(), reason="reference checkout not present")
def test_oracle_equals_live_reference_on_random_signals():
    import pandas as pd

    from oracle.refstub import import_reference

    _ms, seg = import_reference()
    gold = json.load(open(os.path.join(GOLDEN, "segment_pinning.json")))["cases"]
    for (left, right, k), want in zip(mg.segment_pinning_cases(), gold):
        ref = [int(x) for x in seg._transition_indices(pd.Series(left), pd.Series(right), 10, k)]
        assert ref == so.transition_indices(left, right, 10, k)
        assert ref == want["transitions"]
