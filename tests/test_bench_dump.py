"""bench.py --dump-outputs: what it writes for one step, on host tensors large enough to be sampled."""
import os
import types

import numpy as np

import bench


def _step_outputs(rng):
    import torch

    def block(n_ch, n_rows, stride):
        t = torch.from_numpy(rng.normal(size=(n_ch, stride)))
        return types.SimpleNamespace(tensor=t, n_rows=n_rows)

    data = types.SimpleNamespace(blocks=[block(34, 100_000, 100_064), block(120, 20_001, 20_065)])
    traj = data.blocks[1].tensor.numpy()
    traj[rng.random(traj.shape) < 0.05] = np.nan  # blank marker fields
    traj[0, :3], traj[1, :3] = np.inf, -np.inf
    emg = torch.from_numpy(rng.normal(size=(16, 200_000)))
    bounds = np.linspace(0, 180_000, 33).astype(int)
    windows = [emg[:, a:b] for a, b in zip(bounds[:-1], bounds[1:])]
    seg = types.SimpleNamespace(transitions=list(range(100, 4100, 100)))
    return data, seg, windows


def test_dump_is_finite_bounded_and_reproducible(tmp_path):
    rng = np.random.default_rng(0)
    outputs = _step_outputs(rng)
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), *outputs)
    bench.dump_outputs(str(b), *outputs)
    names = sorted(os.listdir(a))
    sampled = [f"{n}{part}" for n in ("devices", "trajectories", "emg_phase_windows") for part in ("", "_rows", "_nonfinite")]
    assert names == sorted(os.listdir(b)) == sorted(f"{n}.npy" for n in sampled + ["transitions", "emg_phase_window_bounds"])
    assert sum(os.path.getsize(a / n) for n in names) <= 64e6
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == (np.float32 if n.endswith("_nonfinite.npy") else np.float64), n
        assert np.isfinite(x).all() and np.array_equal(x, y), n

    data, seg, windows = outputs
    dev, rows = np.load(a / "devices.npy"), np.load(a / "devices_rows.npy").astype(np.int64)
    assert dev.shape == (34, rows.size) and (np.diff(rows) > 0).all() and rows[-1] < data.blocks[0].n_rows
    assert np.array_equal(dev, data.blocks[0].tensor.numpy()[:, rows])
    assert not np.load(a / "devices_nonfinite.npy").any()
    traj, codes = np.load(a / "trajectories.npy"), np.load(a / "trajectories_nonfinite.npy")
    want = data.blocks[1].tensor.numpy()[:, np.load(a / "trajectories_rows.npy").astype(np.int64)]
    nan, pinf, ninf = (codes == bench.NONFINITE_CODES[k] for k in ("nan", "+inf", "-inf"))
    assert nan.any() and pinf.any() and ninf.any()
    assert np.array_equal(nan, np.isnan(want)) and np.array_equal(pinf, np.isposinf(want))
    assert np.array_equal(ninf, np.isneginf(want))
    assert np.array_equal(traj[codes == 0], want[codes == 0]) and (traj[codes != 0] == 0).all()
    assert np.load(a / "transitions.npy").tolist() == seg.transitions
    bounds = np.load(a / "emg_phase_window_bounds.npy")
    assert bounds.tolist() == np.cumsum([0] + [w.shape[1] for w in windows]).tolist()
    win, wrows = np.load(a / "emg_phase_windows.npy"), np.load(a / "emg_phase_windows_rows.npy").astype(np.int64)
    assert np.array_equal(win, np.concatenate([w.numpy() for w in windows], axis=1)[:, wrows])


def test_small_arrays_are_written_whole():
    assert bench.sample_rows(34, 1000, 0).tolist() == list(range(1000))
    assert bench.sample_rows(120, 20_001, 1).size == bench.DUMP_ELEMENTS // 120
