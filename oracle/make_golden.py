"""Generates tests/golden/* by running the UNMODIFIED reference in the build container.

    python oracle/make_golden.py

Needs /root/reference (see oracle/refstub.py); the GPU box does not have it, which is why the
outputs are committed.  Everything here is deterministic: re-running must not change a byte.

Outputs
  abridged_data.csv            the reference's own sample file (data fixture of its tests,
                               sample_data/abridged_data.csv), copied verbatim
  abridged_expected.npz/.json  arrays (uint64 views) and metadata the reference loads from it
  variants/*.csv + variants.json   malformed / unusual inputs derived from the sample and what
                               the reference does with each (arrays or exception text)
  synth_small_*.npz            reference arrays for small synthetic trials (LF and CRLF)
  synth_D_digest.json          sha256 of every reference array for the 41.6 MB D-layout trial
  segment_D.json               reference Segmenter output (40 transitions, 32 slices) on it
  float_table.json             CPython float() known answers (Appendix B of SURVEY.md)
  emg_pinning.npz              EMG preprocessing outputs on a seeded signal (seeded sample of rows)
  segment_pinning.json         transition search results on seeded on/off force-plate signals
"""
import hashlib
import json
import os
import shutil
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle.refstub import REFERENCE_ROOT, import_reference  # noqa: E402
from tools.synth_vicon import synth_layout, synth_vicon  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def devices_of(data):
    return list(data.forcepl) + [data.emg] + list(data.traj)


def describe(data):
    meta = {"devices": []}
    arrays = {}
    for i, dev in enumerate(devices_of(data)):
        meta["devices"].append(
            {
                "name": dev.name,
                "dev_type": dev.dev_type.name,
                "units": list(dev.units),
                "coords": [str(c) for c in dev.df.columns],
                "sampling_frequency": dev.sampling_frequency,
                "shape": list(dev.df.shape),
            }
        )
        arrays[f"dev{i}"] = np.ascontiguousarray(dev.df.to_numpy(dtype=np.float64)).view(np.uint64)
    meta["num_frames"] = devices_of(data)[0]._frame_tracker.num_frames
    return meta, arrays


def outcome(ms, path, shown_name):
    """What the reference does with the file at `path` (arrays or exception)."""
    try:
        data = ms.load_vicon_file(path)
    except Exception as exc:  # noqa: BLE001
        cause = exc.__cause__
        return {
            "raises": type(exc).__name__,
            "message": str(exc).replace(path, shown_name),
            "cause": type(cause).__name__ if cause is not None else None,
        }, None
    meta, arrays = describe(data)
    return {"raises": None, "meta": meta}, arrays


def make_variants(sample: bytes):
    text = sample.decode()
    lines = text.split("\n")
    assert lines[-1] == ""
    lines = lines[:-1]
    L = lambda ls: ("\n".join(ls) + "\n").encode()  # noqa: E731
    v = {}
    v["crlf"] = text.replace("\n", "\r\n").encode()
    v["cr_only"] = text.replace("\n", "\r").encode()
    v["no_final_newline"] = text[:-1].encode()
    v["trailing_blank_row"] = L(lines + ["," * 13])
    v["two_trailing_blank_rows"] = L(lines + ["," * 13, ""])
    v["trailing_empty_line"] = L(lines + [""])
    v["bom"] = b"\xef\xbb\xbf" + sample
    def sub(line_no, old, new, count=1):
        ls = list(lines)
        assert old in ls[line_no - 1], (line_no, old)
        ls[line_no - 1] = ls[line_no - 1].replace(old, new, count)
        return L(ls)
    v["padded_field"] = sub(6, "0.0037236", " 0.0037236 ")
    v["space_field"] = sub(7, "0.00463913", " ")
    v["nan_field"] = sub(7, "0.00463913", "nan")
    v["neg_inf_field"] = sub(7, "0.00463913", "-inf")
    v["underscore_field"] = sub(7, "0.00463913", "1_0.5")
    v["bad_underscore"] = sub(7, "0.00463913", "1__0")
    v["garbage_field"] = sub(8, "0.00448654", "abc")
    v["garbage_frame_col"] = sub(9, "2,0,", "x,0,")
    v["garbage_traj_field"] = sub(19, "209.475", "20x.475")
    v["extra_fields_beyond_num_cols"] = sub(6, ",,,,,,,,,,", ",,,,junk,,,,,,")
    v["exponent_forms"] = sub(10, "0.00204514", "+2.04514E-03")
    v["long_mantissa"] = sub(10, "0.00204514", "0.002045140000000000000000000000000000001")
    v["halfway"] = sub(10, "0.00204514", "9007199254740993")
    v["huge"] = sub(10, "0.00204514", "1e400")
    v["tiny"] = sub(10, "0.00204514", "2.4703282292062328e-324")
    v["neg_zero"] = sub(10, "0.00204514", "-0.0")
    v["tab_padded"] = sub(10, "0.00204514", "\t0.00204514\t")
    v["fs_char_field"] = sub(10, "0.00204514", "\x1c0.00204514")
    # short row: cut the EMG columns of one data row
    ls = list(lines)
    ls[7] = ",".join(ls[7].split(",")[:22])
    v["short_row"] = L(ls)
    ls = list(lines)
    del ls[8]
    v["one_devices_row_deleted"] = L(ls)
    ls = list(lines)
    ls.insert(8, "," * 121)
    v["blank_row_inside_devices"] = L(ls)
    ls = list(lines)
    ls.insert(8, " , ,\t,")
    v["whitespace_blank_row_inside_devices"] = L(ls)
    v["only_devices_section"] = L(lines[:11])
    v["only_devices_section_with_separator"] = L(lines[:12])
    v["truncated_in_header"] = L(lines[:3])
    v["wrong_first_word"] = sub(1, "Devices", "Device")
    v["trajectories_first"] = L(lines[12:] + [lines[11]] + lines[:11])
    v["freq_not_int"] = sub(2, "300", "300.5")
    v["freq_extra_col"] = sub(2, "300,", "300,1")
    v["device_header_misplaced"] = sub(3, ",,Imported", ",Imported,")
    v["force_plate_name_without_dash"] = sub(3, "Plate #1 - Force", "Plate #1 Force")
    v["second_section_wrong_word"] = sub(13, "Trajectories", "Trajectory")
    v["row_after_end"] = L(lines + ["," * 13, "Devices"])
    v["quoted_number"] = sub(7, "0.00463913", '"0.00463913"')
    v["empty_file"] = b""
    v["single_newline"] = b"\n"
    return v


def sha(arr: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


# ---- inputs and outputs that pin oracle/emg_oracle.py and oracle/segment_oracle.py to the reference ----------
EMG_ENVELOPES = (dict(order=4), dict(order=2, zero_lag=False), dict(order=3, filter_type="cheby1", cheby_param=1.0),
                 dict(order=4, filter_type="cheby2", cheby_param=30.0))
EMG_GOLDEN_ROWS = 400  # a seeded sample of the 5000 rows keeps emg_pinning.npz small


def emg_pinning_input():
    """The seeded (5000, 6) EMG-like signal the preprocessing functions are compared on."""
    return np.random.default_rng(0).normal(0.001, 0.01, (5000, 6))


def emg_reference_outputs(ms, x):
    """name -> (rows, channels) output of each reference call; emg_oracle_outputs makes the same calls."""
    import pandas as pd

    df = pd.DataFrame(x, columns=list("abcdef"))
    out = {"zero_center": ms.zero_center(df), "rms": ms.rms(df, 0.5, sampling_frequency=2000),
           "normalize": ms.normalize(df), "time_normalize": ms.time_normalize(df, 200)}
    for i, kw in enumerate(EMG_ENVELOPES):
        out[f"linear_envelope_{i}"] = ms.analysis.linear_envelope(df, 6.0, 2000, **kw)
    out["digital_filter_bandpass"] = ms.analysis.digital_filter(df, (20.0, 450.0), 2000, 4, band_type="bandpass")
    out["linear_envelope_no_zero_center"] = ms.analysis.linear_envelope(df, 6.0, 2000, 4, zero_center_=False)
    return {k: v.to_numpy() for k, v in out.items()}


def emg_oracle_outputs(x):
    from oracle import emg_oracle as eo

    out = {"zero_center": eo.zero_center(x), "rms": eo.rms(x, 1000), "normalize": eo.normalize(x),
           "time_normalize": eo.time_normalize(x, 200)}
    for i, kw in enumerate(EMG_ENVELOPES):
        out[f"linear_envelope_{i}"] = eo.linear_envelope(x, 6.0, 2000, **kw)
    out["digital_filter_bandpass"] = eo.digital_filter(x, (20.0, 450.0), 2000, 4, band_type="bandpass")
    out["linear_envelope_no_zero_center"] = eo.linear_envelope(x, 6.0, 2000, 4, zero_center_=False)
    return out


def emg_golden_rows(n_rows):
    if n_rows <= EMG_GOLDEN_ROWS:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(1).choice(n_rows, EMG_GOLDEN_ROWS, replace=False))


def segment_pinning_signals():
    """Six seeded on/off force-plate signal pairs (runs of 1 to 120 samples) for the transition search."""
    rnd = np.random.default_rng(3)
    for _ in range(6):
        n = int(rnd.integers(300, 5000))
        left, right = np.zeros(n), np.zeros(n)
        i = 0
        while i < n:
            run = int(rnd.choice([1, 3, 9, 10, 11, 30, 120]))
            state = rnd.integers(0, 4)
            left[i : i + run] = 1.0 if state & 1 else 0.0
            right[i : i + run] = 1.0 if state & 2 else 0.0
            i += run
        yield left, right


def segment_pinning_cases():
    """(left, right, k) per signal pair that has alternations: k = min(alternations found, 12) transitions asked for."""
    from oracle import segment_oracle as so

    for left, right in segment_pinning_signals():
        k = min(len(so.transition_indices(left, right, 10, 0)), 12)
        if k:
            yield left, right, k


def write_pinning_golden(emg_outputs, segment_transitions, source):
    """tests/golden/emg_pinning.npz (sampled rows of every EMG output) and segment_pinning.json (transitions)."""
    x = emg_pinning_input()
    arrays = {"input": x[emg_golden_rows(len(x))], "source": np.array(source)}
    for name, a in emg_outputs.items():
        arrays[name] = np.ascontiguousarray(a[emg_golden_rows(len(a))], dtype=np.float64)
    np.savez(os.path.join(GOLD, "emg_pinning.npz"), **arrays)
    cases = [{"n": len(left), "k": k, "transitions": [int(t) for t in segment_transitions(left, right, k)]}
             for left, right, k in segment_pinning_cases()]
    json.dump({"source": source, "cases": cases}, open(os.path.join(GOLD, "segment_pinning.json"), "w"), indent=1)


def main():
    ms, seg = import_reference()
    os.makedirs(os.path.join(GOLD, "variants"), exist_ok=True)

    # 1. the sample file
    sample_src = os.path.join(REFERENCE_ROOT, "sample_data", "abridged_data.csv")
    sample_dst = os.path.join(GOLD, "abridged_data.csv")
    shutil.copyfile(sample_src, sample_dst)
    info, arrays = outcome(ms, sample_dst, "abridged_data.csv")
    np.savez_compressed(os.path.join(GOLD, "abridged_expected.npz"), **arrays)
    json.dump(info, open(os.path.join(GOLD, "abridged_expected.json"), "w"), indent=1, sort_keys=True)

    # 2. variants
    sample = open(sample_src, "rb").read()
    table = {}
    for name, blob in sorted(make_variants(sample).items()):
        path = os.path.join(GOLD, "variants", name + ".csv")
        open(path, "wb").write(blob)
        info, arrays = outcome(ms, path, name + ".csv")
        if arrays is not None:
            info["sha256"] = {k: sha(a) for k, a in arrays.items()}
            np.savez_compressed(os.path.join(GOLD, "variants", name + ".npz"), **arrays)
        table[name] = info
    json.dump(table, open(os.path.join(GOLD, "variants.json"), "w"), indent=1, sort_keys=True)

    # 3. small synthetic trials, full arrays
    for tag, kw in {
        "lf": dict(seed=11, seconds=0.5, n_emg=16, n_markers=40, crlf=False),
        "crlf": dict(seed=12, seconds=0.73, n_emg=8, n_markers=40, crlf=True, trailing_blank=True),
        "narrow": dict(seed=13, seconds=0.4, n_emg=3, n_markers=2, crlf=True),
    }.items():
        blob = synth_vicon(**kw)
        path = f"/tmp/ms_golden_{tag}.csv"
        blob.tofile(path)
        info, arrays = outcome(ms, path, f"synth_small_{tag}.csv")
        assert info["raises"] is None, info
        info["generator"] = kw
        info["csv_sha256"] = hashlib.sha256(blob.tobytes()).hexdigest()
        np.savez_compressed(os.path.join(GOLD, f"synth_small_{tag}.npz"), **arrays)
        json.dump(info, open(os.path.join(GOLD, f"synth_small_{tag}.json"), "w"), indent=1, sort_keys=True)

    # 4. the D-layout trial (dynamic_trial.csv shape): digests + segmenter output
    blob = synth_layout("D", seed=0)
    path = "/tmp/ms_golden_D.csv"
    blob.tofile(path)
    data = ms.load_vicon_file(path)
    meta, arrays = describe(data)
    digest = {
        "generator": {"layout": "D", "seed": 0},
        "csv_sha256": hashlib.sha256(blob.tobytes()).hexdigest(),
        "csv_bytes": int(blob.nbytes),
        "meta": meta,
        "sha256": {k: sha(a) for k, a in arrays.items()},
    }
    json.dump(digest, open(os.path.join(GOLD, "synth_D_digest.json"), "w"), indent=1, sort_keys=True)

    transitions = [int(t) for t in seg._transition_indices(*seg.reactions(data))]
    segmenter = seg.Segmenter(data)
    windows = []
    for trecho in seg.Trecho:
        for cycle in seg.Cycle:
            for i in range(1, 5):
                phase = segmenter.ith_phase(trecho, i)
                sl = segmenter.get_times_of(trecho, cycle, phase)
                emg_rows = data.emg[sl]
                traj_rows = data.traj[0][sl]
                windows.append(
                    {
                        "trecho": trecho.name, "cycle": cycle.name, "phase": phase.name, "order": i,
                        "start": [int(x) for x in sl.start], "stop": [int(x) for x in sl.stop],
                        "emg_shape": list(emg_rows.shape), "emg_sha256": sha(emg_rows.to_numpy().view(np.uint64)),
                        "traj0_shape": list(traj_rows.shape),
                        "traj0_sha256": sha(traj_rows.to_numpy().view(np.uint64)),
                    }
                )
    cyc = segmenter.get_times_of(seg.Trecho.SECOND, seg.Cycle.SECOND)
    tre = segmenter.get_times_of(seg.Trecho.THIRD)
    json.dump(
        {
            "generator": {"layout": "D", "seed": 0},
            "transitions": transitions,
            "windows": windows,
            "cycle_2_2": {"start": [int(x) for x in cyc.start], "stop": [int(x) for x in cyc.stop]},
            "trecho_3": {"start": [int(x) for x in tre.start], "stop": [int(x) for x in tre.stop]},
        },
        open(os.path.join(GOLD, "segment_D.json"), "w"), indent=1, sort_keys=True,
    )

    # 5. float() known answers
    texts = [
        "-0", "-0.0", "0", "nan", "NaN", "+nan", "-nan", "inf", "iNf", "1e400", "1.7976931348623159e308",
        "-Infinity", "-1e400", "1e-400", "2.4703282292062327e-324", "4.9e-324", "2.4703282292062328e-324",
        "9007199254740993", "9007199254740992.5", "1.7976931348623157e308", "123456789012345678901234567890",
        "0.1", ".", "1e", "1e+", "1__0", "_1", "1_", "1d5", "1,5", "0x10", "0x1p3", "abc", " ", "  .5  ", "1.",
        "+.5e-3", "1_0", "1_0.5", "0.000001E5", "-3.56E-05", "5.20E-05", "0.0037236", "209.331", "1e23",
        "2.2250738585072011e-308", "2.2250738585072014e-308", "1e1_0", "1_e5", "infinity", "infinit", "\x1c1",
        "1\x0b", "0e99999999999999999999", "1e99999999999999999999", "1e-99999999999999999999",
    ]
    table = {}
    for t in texts:
        try:
            table[t] = "0x%016x" % struct.unpack("<Q", struct.pack("<d", float(t)))[0]
        except ValueError:
            table[t] = "ValueError"
    json.dump(table, open(os.path.join(GOLD, "float_table.json"), "w"), indent=1, sort_keys=True)

    # 6. the preprocessing functions and the transition search on seeded inputs
    import pandas as pd

    write_pinning_golden(
        emg_reference_outputs(ms, emg_pinning_input()),
        lambda left, right, k: seg._transition_indices(pd.Series(left), pd.Series(right), 10, k),
        "the reference (elvis-sik/muscle_synergies), by oracle/make_golden.py")
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
