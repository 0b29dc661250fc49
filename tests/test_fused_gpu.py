"""The single-pass loader kernel (ms_load_fused: one launch from CSV bytes to both sections' blocks) against the CPU
oracles, bit for bit, at tile sizes that move every tile boundary around; and that it declines - so that the two-pass
path answers, with the reference's behaviour - exactly the files it is not meant for."""
import ctypes
import os
import random

import numpy as np
import pytest

from conftest import GOLDEN, bits

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as g

    g.build()
    import muscle_synergies_b200 as ms
    from muscle_synergies_b200.vicon_data import loader as loader_mod

    return ms, loader_mod


@pytest.fixture(autouse=True)
def _always_try_single_pass(env):
    _ms, loader_mod = env
    old = loader_mod.FORCE_PATH, loader_mod.FORCE_TILE
    loader_mod.FORCE_PATH = "fused"
    yield
    loader_mod.FORCE_PATH, loader_mod.FORCE_TILE = old


def section_arrays(data):
    import torch

    dev = torch.cat([d.tensor for d in data.forcepl] + [data.emg.tensor]).cpu().numpy().T
    traj = torch.cat([d.tensor for d in data.traj]).cpu().numpy().T
    return np.ascontiguousarray(dev), np.ascontiguousarray(traj)


def load_single_pass(env, blob, tile=None, fresh=True):
    """Loads through a loader of its own (no size history unless fresh=False) and insists the single-pass kernel answered."""
    ms, loader_mod = env
    loader_mod.FORCE_TILE = tile
    loader = ms.ViconLoader()
    data = loader.load_bytes(blob, name="t.csv")
    assert loader.stats["fused"] == 1 and loader.stats["two_pass"] == 0, loader.stats
    return loader, data


TILES = [4096, 4112, 5008, 8192, 20000, 43872, 49152]


@pytest.mark.parametrize("kw", [
    dict(seed=51, seconds=1.3, n_emg=16, n_markers=40, crlf=True),
    dict(seed=52, seconds=0.9, n_emg=16, n_markers=40, crlf=False),
    dict(seed=53, seconds=0.7, n_emg=1, n_markers=1, crlf=True),
    dict(seed=54, seconds=1.1, n_emg=5, n_markers=100, crlf=False, trailing_blank=True),
    dict(seed=55, seconds=0.02, n_emg=16, n_markers=40, crlf=True),
    dict(seed=56, seconds=1.0, n_emg=16, n_markers=40, crlf=True, blank_marker_frac=0.9),
])
def test_bit_exact_at_every_tile_size(env, kw):
    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    blob = synth_vicon(**kw)
    want_dev, want_traj = vof.parse(blob)
    for tile in TILES:
        _loader, data = load_single_pass(env, blob, tile)
        got_dev, got_traj = section_arrays(data)
        assert got_dev.shape == want_dev.shape and got_traj.shape == want_traj.shape, tile
        assert (bits(got_dev) == bits(want_dev)).all(), tile
        assert (bits(got_traj) == bits(want_traj)).all(), tile


def test_line_ends_and_eof_shapes(env, tmp_path):
    """LF, CRLF and lone CR files; with and without a final line end; with and without the trailing blank row."""
    from oracle import vicon_oracle as vo

    rnd = random.Random(3)
    for eol in ("\n", "\r\n", "\r"):
        for final_eol in (True, False):
            for trailing_blank in (True, False):
                emg, mark = 3, 2
                lines = ["Devices", "1000", ",,P #1 - Force,,,P #1 - Moment,,,P #1 - CoP,,,EMG - V",
                         "Frame,Sub Frame," + ",".join(f"c{i}" for i in range(9 + emg)), ",," + ",".join("u" * (9 + emg))]
                for r in range(700):
                    lines.append(",".join([str(r // 10 + 1), str(r % 10)] + ["%.6g" % rnd.uniform(-9, 9) for _ in range(9 + emg)]))
                lines.append("," * (10 + emg))
                lines += ["Trajectories", "100", ",," + ",,,".join(f"S:M{i}" for i in range(mark)),
                          "Frame,Sub Frame," + ",".join("XYZ"[i % 3] for i in range(3 * mark)), ",," + ",".join(["mm"] * (3 * mark))]
                for r in range(70):
                    lines.append(",".join([str(r + 1), "0"] + ["%.6g" % rnd.uniform(-900, 900) for _ in range(3 * mark)]))
                if trailing_blank:
                    lines.append("," * (1 + 3 * mark))
                blob = (eol.join(lines) + (eol if final_eol else "")).encode()
                path = tmp_path / "eof_case.csv"
                with open(path, "wb") as f:
                    f.write(blob)
                want = vo.load_vicon_file_oracle(path)
                for tile in (4096, 4160, 49152):
                    _loader, data = load_single_pass(env, np.frombuffer(blob, dtype=np.uint8), tile)
                    devs = list(data.forcepl) + [data.emg] + list(data.traj)
                    for dev, odev in zip(devs, want.all_devices()):
                        got, exp = bits(dev.df.to_numpy()), bits(vo.device_array(odev))
                        assert got.shape == exp.shape and (got == exp).all(), (eol, final_eol, trailing_blank, tile, dev.name)
                os.unlink(path)


def test_tile_boundary_sweep(env):
    """Grow a header name byte by byte: every row start and line end crosses a tile edge at some padding."""
    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    base = synth_vicon(seed=57, seconds=0.25, n_emg=16, n_markers=40, crlf=True).tobytes()
    marker = b"EMG2000 - Voltage"
    want = None
    for pad in list(range(0, 36)) + [347, 348, 349]:
        blob = np.frombuffer(base.replace(marker, b"EMG2000" + b"x" * pad + b" - Voltage", 1), dtype=np.uint8)
        if want is None:
            want = vof.parse(blob)
        _loader, data = load_single_pass(env, blob, 4096)
        got = section_arrays(data)
        assert (bits(got[0]) == bits(want[0])).all(), pad
        assert (bits(got[1]) == bits(want[1])).all(), pad
        assert data.emg.name == "EMG2000" + "x" * pad + " - Voltage"


def test_second_file_uses_the_first_files_shapes(env):
    """The size guess for a file comes from the previous one: same loader, three trials of different lengths."""
    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    ms, loader_mod = env
    loader_mod.FORCE_TILE = None
    loader = ms.ViconLoader()
    for seed, seconds in ((61, 1.0), (62, 1.6), (63, 0.4), (64, 3.0)):
        blob = synth_vicon(seed=seed, seconds=seconds, n_emg=16, n_markers=40, crlf=True)
        want = vof.parse(blob)
        got = section_arrays(loader.load_bytes(blob))
        assert (bits(got[0]) == bits(want[0])).all() and (bits(got[1]) == bits(want[1])).all(), seed
    # a much longer file than the guess allows is declined once (MS_LOAD_OVERFLOW) and parsed by the two-pass path
    assert loader.stats["fused"] + loader.stats["two_pass"] == 4 and loader.stats["fused"] >= 3, loader.stats


def test_declines_what_it_is_not_meant_for(env, variants_table):
    """Every golden variant loads (or raises) exactly as through the two-pass path; the single-pass kernel may only
    have answered for files the reference loads without complaint."""
    ms, loader_mod = env
    loader_mod.FORCE_TILE = None
    for name, info in sorted(variants_table.items()):
        path = os.path.join(GOLDEN, "variants", name + ".csv")
        loader = ms.ViconLoader()
        try:
            loader.load_file(path)
            raised = None
        except Exception as exc:  # noqa: BLE001
            raised = exc
        assert (raised is None) == (info["raises"] is None), (name, raised)
        if info["raises"] is not None:
            assert loader.stats["fused"] == 0, (name, loader.stats)


def test_c_abi_direct(env):
    """ms_load_fused through ctypes alone: result struct, header peeks, blocks in the arena."""
    import torch

    from muscle_synergies_b200 import _native as nat
    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    blob = synth_vicon(seed=58, seconds=0.8, n_emg=16, n_markers=40, crlf=True)
    want_dev, want_traj = vof.parse(blob)
    n = int(blob.nbytes)
    lib = nat.lib()
    d_bytes = torch.zeros((n + 15) // 16 * 16 + 16, dtype=torch.uint8, device="cuda")
    d_bytes[:n] = torch.from_numpy(blob.copy()).cuda()
    arena = torch.full((want_dev.size + want_traj.size + 200_000,), -1.0, dtype=torch.float64, device="cuda")
    ws = torch.empty(int(lib.ms_load_workspace_bytes(n, 0)), dtype=torch.uint8, device="cuda")
    d_res = torch.empty(ctypes.sizeof(nat.LoadResult), dtype=torch.uint8, device="cuda")
    d_peek = torch.empty(2 * nat.MS_LOAD_PEEK, dtype=torch.uint8, device="cuda")
    plan = nat.LoadPlan(arena.data_ptr(), arena.numel(), (ctypes.c_int64 * 2)(want_dev.shape[0] + 10, 0), 0, 0)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    nat.check(lib.ms_load_fused(d_bytes.data_ptr(), n, ctypes.byref(plan), ws.data_ptr(), ws.numel(), d_res.data_ptr(),
                                d_peek.data_ptr(), stream), "ms_load_fused")
    torch.cuda.synchronize()
    res = nat.LoadResult.from_buffer_copy(d_res.cpu().numpy().tobytes())
    assert res.flags == 0 and res.status == nat.MS_ERR_NONE
    assert list(res.data_rows) == [want_dev.shape[0], want_traj.shape[0]]
    assert list(res.num_cols) == [want_dev.shape[1] + 2, want_traj.shape[1] + 2]
    assert res.header_offset[0] == 0 and bytes(d_peek[:7].cpu().numpy()) == b"Devices"
    off2 = int(res.header_offset[1])
    assert blob[off2 : off2 + 12].tobytes() == b"Trajectories" == bytes(d_peek[nat.MS_LOAD_PEEK : nat.MS_LOAD_PEEK + 12].cpu().numpy())
    for s, want in ((0, want_dev), (1, want_traj)):
        keep, stride, off = int(res.n_keep[s]), int(res.stride[s]), int(res.out_offset[s])
        got = arena[off : off + keep * stride].view(keep, stride)[:, : want.shape[0]].cpu().numpy().T
        assert (bits(np.ascontiguousarray(got)) == bits(want)).all()


def test_results_kept_across_a_batch_stay_valid(env):
    """load_many with to_host: every result's host arrays still hold ITS file after the whole batch was consumed
    (the pinned buffers are on loan to the results, not a ring that the next files overwrite)."""
    import torch

    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    ms, loader_mod = env
    loader_mod.FORCE_TILE = None
    blobs = [synth_vicon(seed=70 + i, seconds=0.5, n_emg=16, n_markers=40, crlf=True) for i in range(5)]
    loader = ms.ViconLoader()
    kept = list(loader.load_many([torch.from_numpy(b.copy()).pin_memory() for b in blobs], to_host=True))
    for blob, data in zip(blobs, kept):
        want_dev, _ = vof.parse(blob)
        got = np.concatenate([d.df.to_numpy() for d in list(data.forcepl) + [data.emg]], axis=1)
        assert (bits(np.ascontiguousarray(got)) == bits(want_dev)).all()
    del kept, data
    import gc

    gc.collect()
    assert len(loader._host_pool) >= 2  # the buffers came back


def test_stream_of_device_resident_trials(env):
    """load_device_many: several trials in flight on the loader's pipeline streams, the caller's work on a stream of
    its own - every trial's arrays bit-exact against the C oracle, transitions equal to a one-at-a-time load's, a trial
    the single-pass kernel declines (a quoted field) answered by the two-pass path in its place, results kept across
    the whole batch still valid."""
    import torch

    from muscle_synergies_b200.segment import Segmenter
    from oracle import vicon_oracle_fast as vof
    from tools.synth_vicon import synth_vicon

    ms, loader_mod = env
    loader_mod.FORCE_TILE = None
    loader_mod.FORCE_PATH = None
    blobs = [synth_vicon(seed=90 + i, seconds=4.0 + 0.5 * i, n_emg=16, n_markers=40, crlf=bool(i & 1)) for i in range(6)]
    # trial 3: one quoted number in a data row - not for the single-pass kernel, same arrays from the two-pass path
    text = blobs[3].tobytes()
    cut = text.index(b",", text.index(b"\n", len(text) // 3) + 1) + 1  # start of the second field of a Devices row
    end = text.index(b",", cut)
    quoted = text[:cut] + b'"' + text[cut:end] + b'"' + text[end:]
    blobs[3] = np.frombuffer(quoted, dtype=np.uint8)

    def on_device(blob):
        d = torch.empty(ms.ViconLoader.padded_size(blob.nbytes), dtype=torch.uint8, device="cuda")
        d[: blob.nbytes].copy_(torch.from_numpy(np.ascontiguousarray(blob)))
        return d, int(blob.nbytes)

    sources = [on_device(b) for b in blobs]
    loader = ms.ViconLoader()
    work = loader.work_stream
    kept, transitions = [], []
    for data in loader.load_device_many(iter(sources), depth=3, stream=work):
        with torch.cuda.stream(work):
            # odd trials through the deferred constructor (search queued, finished a moment later)
            seg = Segmenter.begin(data).finish() if len(kept) & 1 else Segmenter(data)
            transitions.append(list(seg.transitions))
        kept.append(data)
    torch.cuda.current_stream().wait_stream(work)
    assert len(kept) == len(blobs)
    assert loader.stats["fused"] >= 4 and loader.stats["two_pass"] >= 1, loader.stats
    for i, (blob, data) in enumerate(zip(blobs, kept)):
        want = vof.parse(blobs[i] if i != 3 else np.frombuffer(text, dtype=np.uint8))
        got = section_arrays(data)
        assert (bits(got[0]) == bits(want[0])).all() and (bits(got[1]) == bits(want[1])).all(), i
        one = ms.ViconLoader().load_device(*sources[i])
        assert list(Segmenter(one).transitions) == transitions[i]
