#!/usr/bin/env python
"""Headline benchmark: Vicon CSV loader throughput (GB of CSV per second, output bit-exact) on synthetic 10-minute
trials of the dynamic_trial.csv layout (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One step = one pass of the hot path over one trial per GPU: the single-pass loader kernel (ms_load_fused: every data
row of both sections -> channel-major float64 in HBM) + Segmenter (40 transitions) + gather of the 32 phase windows
of the EMG device.  `value` times it with the CSV bytes already resident in HBM; `e2e` times the public batch call
`ViconLoader.load_many` from pinned HOST bytes to HOST arrays (H2D of every CSV byte and D2H of every parsed double
inside the timed region, overlapped across consecutive trials on three streams) and is set against what the box's
PCIe links deliver with all ranks copying at once (`pcie`).  Multi-GPU: one process per GPU, trials sharded by file,
no collective on the data path (weak scaling); NCCL carries only the barrier, the max-over-ranks time and the one
host-side gather of result tables.  Besides the T10 step every rank also runs its shard of `configs[2]` (files in
tmpfs -> host arrays) and `configs[4]` (files -> synergies).

`--impl reference` times the UNMODIFIED reference (baseline/_ref, installed by oracle/install_ref.py):
muscle_synergies.load_vicon_file + project/segment.py Segmenter + the 32 EMG phase windows per trial in a persistent
multiprocessing.Pool over all host cores, on a bounded sample of the same layout; and scikit-learn's NMF(mu) over
the same cores.

`--dump-outputs DIR` writes, after the timed steps, what the last streamed step handed its caller (rank 0): the two
section blocks, the 40 transitions and the 32 EMG phase windows, as DIR/<name>.npy (float64; seeded samples of rows
where a block is larger than DUMP_ELEMENTS; NaN and infinities written as 0 and marked in a float32 code array), so
that two builds can be compared output for output.  The benchmark reads the library that `__graft_entry__.build()`
left in the tree (with a warning if it is older than the CUDA sources) and writes nothing there.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "vicon_csv_loader_throughput"
UNIT = "GB/s"
WORKLOAD = "T10: synthetic 10-min Vicon trial, 2 force plates + 16 EMG @2 kHz, 40 markers @100 Hz, load + segment"
SAMPLE_SECONDS = 6.0  # length of the trials of the CPU sample (T10 column layout, ~5 MB each)


def shm_dir(need_bytes):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need_bytes else None
    return base


# ---- CPU arm: the reference itself ------------------------------------------------------------------------------
def _ref_init():
    global _REF
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
    from oracle import refstub

    _REF = refstub.import_reference()


def _ref_trial(path):
    """What one step does to one trial, by the reference: load_csv.py:96-135, project/segment.py:124-298,
    user_data.py:727-731 (dev[slice] for the 32 phase windows of the EMG device)."""
    ms_ref, seg_mod = _REF
    data = ms_ref.load_vicon_file(path)
    seg = seg_mod.Segmenter(data)
    rows = 0
    for trecho in seg_mod.Trecho:
        for cycle in seg_mod.Cycle:
            for phase in seg_mod.Phase:
                rows += len(data.emg[seg.get_times_of(trecho, cycle, phase)])
    return os.path.getsize(path), rows


def _port_init():
    pass


def _port_trial(path):
    from oracle.vicon_oracle import load_vicon_file_oracle

    res = load_vicon_file_oracle(path)
    return os.path.getsize(path), res.num_frames


def _nmf_task(args):
    import warnings

    from sklearn.decomposition import NMF

    X, k, seed, iters = args
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = NMF(n_components=k, solver="mu", init="random", random_state=seed, max_iter=iters, tol=0.0)
        m.fit_transform(X)
    return int(m.n_iter_)


class CpuArm:
    """The reference's CPU implementation of the step over a persistent pool of all host cores."""

    def __init__(self, cores=None):
        import multiprocessing as mp

        from oracle import refstub
        from tools.synth_vicon import synth_vicon

        self.cores = cores or len(os.sched_getaffinity(0))
        self.kind = "reference" if refstub.reference_available() else "port"
        n_files = max(16, self.cores)
        self.tmp = tempfile.mkdtemp(prefix="ms_b200_cpu_", dir=shm_dir(n_files * (8 << 20)))
        self.paths, self.bytes = [], 0
        for i in range(n_files):
            blob = synth_vicon(seed=5000 + i, seconds=SAMPLE_SECONDS, n_emg=16, n_markers=40)
            path = os.path.join(self.tmp, f"sample{i}.csv")
            blob.tofile(path)
            self.paths.append(path)
            self.bytes += int(blob.nbytes)
        ctx = mp.get_context("fork")
        init, self.task = (_ref_init, _ref_trial) if self.kind == "reference" else (_port_init, _port_trial)
        self.pool = ctx.Pool(self.cores, initializer=init)
        what = ("unmodified reference: load_vicon_file + Segmenter + 32 EMG phase windows" if self.kind == "reference"
                else "python port of load_vicon_file (load only; baseline/_ref is missing)")
        self.sample = (f"{n_files} distinct {SAMPLE_SECONDS:g} s T10-layout trials ({self.bytes / n_files / 1e6:.1f} MB each) "
                       f"per step over a persistent Pool({self.cores}); {what}")

    def step(self):
        t = time.perf_counter()
        done = self.pool.map(self.task, self.paths, chunksize=1)
        wall = time.perf_counter() - t
        assert sum(b for b, _ in done) == self.bytes
        return wall

    def nmf(self, iters=200):
        """sklearn NMF(mu) over the same pool: the (k, restart) grid of configs[3] on a 200 x 16 envelope matrix."""
        X = nmf_envelopes()
        grid = [(X, k, s, iters) for k in range(1, 9) for s in range(20)]
        self.pool.map(_nmf_task, grid[: self.cores], chunksize=1)  # warm-up: imports
        t = time.perf_counter()
        n_iter = sum(self.pool.map(_nmf_task, grid, chunksize=1))
        wall = time.perf_counter() - t
        return {"iterations_per_s": n_iter / wall, "processes": self.cores, "problems": len(grid), "iterations_per_problem": iters,
                "solver": "sklearn.decomposition.NMF(solver='mu', init='random', tol=0), float64"}

    def close(self):
        self.pool.close()
        self.pool.join()
        shutil.rmtree(self.tmp, ignore_errors=True)


def cpu_baseline(target_wall=15.0):
    """Bounded run of the CPU arm for the `cpu_baseline` object of our own line."""
    arm = CpuArm()
    try:
        arm.step()  # warm-up: imports, page cache
        walls = [arm.step()]
        while sum(walls) < target_wall and len(walls) < 20:
            walls.append(arm.step())
        gbs = arm.bytes * len(walls) / sum(walls) / 1e9
        return {"value": gbs, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                "sample": f"{len(walls)} steps of: {arm.sample}"}
    finally:
        arm.close()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm()
    try:
        for _ in range(max(1, args.warmup)):
            arm.step()
        steps = max(1, args.steps)
        walls = []
        budget = time.perf_counter() + 240.0  # the whole run ends within a few minutes whatever --steps says
        for _ in range(steps):
            walls.append(arm.step())
            if time.perf_counter() > budget:
                break
        t_total = sum(walls)
        value = arm.bytes * len(walls) / t_total / 1e9
        try:
            nmf = arm.nmf()
        except Exception as exc:  # noqa: BLE001
            nmf = {"error": f"{type(exc).__name__}: {exc}"}
        note = "" if len(walls) == steps else f"; stopped after {len(walls)} of {steps} steps (time budget)"
        line = {
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(walls), "warmup": max(1, args.warmup), "ms_per_step": 1e3 * t_total / len(walls),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "note": "the reference's own CPU implementation on a bounded sample per step" + note},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "nmf": nmf,
            "gpu_launches": 0,
        }
        print(json.dumps(line))
    finally:
        arm.close()


# ---- clocks ---------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._thread = None

    def _run(self):
        # NVML in-process (a sample every 10 ms: the timed region of a short run is tens of milliseconds);
        # nvidia-smi, one process per sample, only when the binding is missing
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu_index)
            smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self._stop.is_set():
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    why = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001 - older bindings
                    why = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                flags = ["Active" if why & b else "Not Active" for b in (0x8, 0x40, 0x20, 0x4)]
                self.samples.append(["", str(sm), str(smax), "", ""] + flags)
                self._stop.wait(0.01)
            return
        except Exception:  # noqa: BLE001
            pass
        while not self._stop.is_set():
            try:
                out = subprocess.run(
                    ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-i", str(self.gpu_index)],
                    capture_output=True, text=True, timeout=5,
                ).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        sm, reasons, smax = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                smax = float(s[2])
                for name, val in zip(names, s[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- NMF-MU extension -------------------------------------------------------------------------------------
def nmf_envelopes(seed=1, n=200, m=16, k_true=4):
    import numpy as np

    rng = np.random.default_rng(seed)
    t = np.linspace(0, 1, n)[:, None]
    basis = np.abs(np.sin(np.pi * (rng.uniform(0.5, 3, (1, k_true)) * t + rng.uniform(0, 1, (1, k_true))))) ** 2
    X = basis @ rng.uniform(0, 1, (k_true, m)) + 0.02 * rng.uniform(0, 1, (n, m))
    return X / X.max(axis=0)


def bench_nmf(dev, iters=2000):
    """160 problems (k=1..8 x 20 restarts) x `iters` MU iterations in one launch (configs[3]); and the long-signal
    regime where X and W stream from HBM every iteration."""
    import ctypes

    import torch

    from muscle_synergies_b200 import _native as nat
    from muscle_synergies_b200 import analysis

    X = nmf_envelopes()
    ranks = [k for k in range(1, 9) for _ in range(20)]
    seeds = [r for _ in range(1, 9) for r in range(20)]
    analysis.nmf_mu_batched(X, ranks, seeds, max_iter=50, tol=0.0)  # warm-up
    torch.cuda.synchronize()
    t = time.perf_counter()
    res = analysis.nmf_mu_batched(X, ranks, seeds, max_iter=iters, tol=0.0)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t
    t = time.perf_counter()
    analysis.nmf_mu_batched(X, ranks, seeds, max_iter=1, tol=0.0)
    torch.cuda.synchronize()
    overhead = time.perf_counter() - t
    kernel_s = max(wall - overhead, 1e-6)
    total_iters = int(res.n_iter.sum())
    out = {"problems": len(ranks), "shape": [200, 16], "iterations_per_problem": iters,
           "iterations_per_s": total_iters / kernel_s, "kernel_s": kernel_s, "host_overhead_s": overhead,
           "regime": "shared-memory resident (no HBM traffic between iterations): bound by SM issue, not HBM"}
    try:
        n_long, m, k, P = 2_000_000, 16, 8, 4
        lib = nat.lib()
        Xl = torch.rand((n_long, m), device=dev, dtype=torch.float32)
        W0 = torch.rand((P, n_long, k), device=dev, dtype=torch.float32)
        H0 = torch.rand((P, k, m), device=dev, dtype=torch.float32)
        work = torch.empty(int(lib.ms_nmf_stream_workspace_bytes(m, P)), dtype=torch.uint8, device=dev)
        d_iter = torch.empty(P, dtype=torch.int32, device=dev)
        d_err = torch.empty(P, dtype=torch.float32, device=dev)
        d_vaf = torch.empty((P, m + 1), dtype=torch.float32, device=dev)
        ranks_c = (ctypes.c_int32 * P)(*([k] * P))
        stream = torch.cuda.current_stream(dev)
        sptr = ctypes.c_void_p(stream.cuda_stream)

        def run(n_it):
            W, H = W0.clone(), H0.clone()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            nat.check(lib.ms_nmf_mu_stream(Xl.data_ptr(), n_long, m, ranks_c, None, P, W.data_ptr(), H.data_ptr(), n_it,
                                           ctypes.c_float(0.0), 10, work.data_ptr(), d_iter.data_ptr(), d_err.data_ptr(),
                                           d_vaf.data_ptr(), sptr), "ms_nmf_mu_stream")
            e1.record(stream)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e-3

        run(3)
        its = 40
        t_small = min(run(5) for _ in range(2))
        t_big = min(run(5 + its) for _ in range(2))
        per_iter = max(t_big - t_small, 1e-6) / its
        shared_x = 4 * n_long * m + P * 8 * n_long * k  # X read once for all problems, W read + written per problem
        out["long_signal"] = {"shape": [n_long, m], "rank": k, "problems": P, "iterations_per_s": P / per_iter,
                              "ms_per_iteration_all_problems": per_iter * 1e3,
                              "algorithmic_gbs": shared_x / per_iter / 1e9,
                              "note": "algorithmic bytes per iteration = 4nm (X once for all problems of the launch) + P x 8nk; CUDA events"}
        del Xl, W0, H0
    except Exception as exc:  # noqa: BLE001
        out["long_signal"] = {"error": f"{type(exc).__name__}: {exc}"}
    return out


# ---- outputs of the timed path ------------------------------------------------------------------------------
DUMP_ELEMENTS = 1 << 20  # per sampled array: 8 MiB of float64 + 4 MiB of float32 codes, three such pairs under 64 MB
# codes of `<name>_nonfinite.npy`: what stood where `<name>.npy` holds 0 (a blank CSV field is NaN, as in the reference)
NONFINITE_CODES = {"nan": 1.0, "+inf": 2.0, "-inf": 3.0}


def sample_rows(n_ch, n_rows, seed):
    """Ascending row indices of a fixed, seeded sample: every row if all of them fit DUMP_ELEMENTS, else as many
    whole rows (all channels) as fit."""
    import numpy as np

    keep = max(1, DUMP_ELEMENTS // max(1, n_ch))
    if keep >= n_rows:
        return np.arange(n_rows, dtype=np.int64)
    return np.sort(np.random.default_rng(seed).choice(n_rows, keep, replace=False))


def split_nonfinite(a):
    """(a with every NaN / infinity replaced by 0, float32 array of NONFINITE_CODES, 0 where a is finite)."""
    import numpy as np

    codes = np.zeros(a.shape, dtype=np.float32)
    codes[np.isnan(a)] = NONFINITE_CODES["nan"]
    codes[np.isposinf(a)] = NONFINITE_CODES["+inf"]
    codes[np.isneginf(a)] = NONFINITE_CODES["-inf"]
    return np.where(codes == 0, a, 0.0), codes


def dump_outputs(out_dir, data, seg, windows):
    """Writes what one step hands its caller - the trial's section blocks, the Segmenter's transitions and the 32
    phase windows of the EMG device - as .npy files of finite floats.  A channel-major (channels, rows) array larger
    than DUMP_ELEMENTS is sampled by rows (`<name>_rows.npy` holds the row indices); its non-finite entries are
    written as 0 and told apart in `<name>_nonfinite.npy` (NONFINITE_CODES)."""
    import numpy as np
    import torch

    def put(name, a, dtype=np.float64):
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=dtype))

    def put_sampled(name, t, seed):
        rows = sample_rows(int(t.shape[0]), int(t.shape[1]), seed)
        values, codes = split_nonfinite(t.index_select(1, torch.from_numpy(rows).to(t.device)).cpu().numpy())
        put(name, values)
        put(f"{name}_nonfinite", codes, np.float32)
        put(f"{name}_rows", rows)

    os.makedirs(out_dir, exist_ok=True)
    for seed, (name, blk) in enumerate(zip(("devices", "trajectories"), data.blocks)):
        put_sampled(name, blk.tensor[:, : blk.n_rows], seed)
    put("transitions", np.asarray(seg.transitions))
    put_sampled("emg_phase_windows", torch.cat(list(windows), dim=1), 2)
    put("emg_phase_window_bounds", np.cumsum([0] + [int(w.shape[1]) for w in windows]))


# ---- our arm ------------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    # staging buffers and the threads that fill them next to the GPU (restored before the CPU baseline)
    from muscle_synergies_b200.sharding import bind_to_gpu_numa, gather_results, shard

    all_cpus = os.sched_getaffinity(0)
    numa_cpus = bind_to_gpu_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)

    import muscle_synergies_b200 as ms
    from muscle_synergies_b200 import _native
    from muscle_synergies_b200.csrc import build as cuda_build

    if rank == 0 and cuda_build.stale():
        print(f"bench.py: warning: {cuda_build.OUT} is missing or older than its CUDA sources; "
              "run __graft_entry__.build() to time the current code", file=sys.stderr)
    from muscle_synergies_b200.segment import Segmenter
    from muscle_synergies_b200.vicon_data import loader as loader_mod
    from tools.synth_vicon import synth_layout

    layout = args.layout
    blobs = [synth_layout(layout, seed=1000 + 2 * rank + i) for i in range(2)]  # two distinct trials per rank
    blob = blobs[0]
    n = int(blob.nbytes)
    loader = ms.ViconLoader(dev)
    pinned_in = []
    for b in blobs:
        p = torch.empty(loader.padded_size(int(b.nbytes)), dtype=torch.uint8, pin_memory=True)
        p.numpy()[: b.nbytes] = b
        pinned_in.append(p[: int(b.nbytes)])
    d_bytes = torch.empty(loader.padded_size(n), dtype=torch.uint8, device=dev)
    d_bytes[:n].copy_(pinned_in[0])
    torch.cuda.synchronize()

    def step_resident():
        # one submission per stage: the single-pass loader kernel, then transition search + window plan + gather of
        # the 32 EMG phase windows queued back to back
        data = loader.load_device(d_bytes, n=n, name=layout, defer_check=True)
        seg = Segmenter(data, cut_phases_of=(data.emg,))
        cuts = seg.phase_cuts(data.emg)
        return data, cuts

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        barrier()
        return ms_total

    # shapes for the algorithmic byte count (SURVEY.md section 8d): B_alg = B_csv + 8 * N_kept
    data, cuts = step_resident()
    n_kept = sum(int(d.tensor.numel()) for d in list(data.forcepl) + [data.emg] + list(data.traj))
    b_alg = n + 8 * n_kept
    def steps_streamed(k):
        # the same K steps as a stream of trials (what a 1000-trial job is): load_device_many keeps the loader kernel of
        # the next two trials queued on its own stream while the host finishes trial i's objects and runs Segmenter + the
        # window gather on it - every step still ends with the 40 transitions and the 32 windows of ITS trial on the host.
        # Returns (data, Segmenter, windows) of the last step.
        out, begun = None, None
        work = loader.work_stream  # high priority: the small kernels of a step run beside the next trial's loader kernel
        for data in loader.load_device_many(((d_bytes, n) for _ in range(k)), depth=args.depth, stream=work):
            with torch.cuda.stream(work):
                pending = Segmenter.begin(data, cut_phases_of=(data.emg,))  # search + gather queued, no wait
            if begun is not None:  # the trial before: its transitions and windows are on the host by now
                out = begun[0].finish().phase_cuts(begun[1].emg)
            begun = (pending, data)
        data, seg = None, None
        if begun is not None:
            seg, data = begun[0].finish(), begun[1]
            out = seg.phase_cuts(data.emg)
        torch.cuda.current_stream().wait_stream(work)  # the closing event is recorded after the last step's kernels
        return data, seg, out

    for _ in range(max(3, args.warmup)):
        step_resident()
    ms_serial = timed(step_resident, args.steps)  # one trial at a time, the host's work between the kernels exposed
    # warm-up of the streamed loop: the caching allocator keeps a pool per stream, and the pipeline streams' pools hold
    # the four or five 0.4 GB arenas a stream of trials cycles through only after a dozen steps (before that every step
    # pays a cudaMalloc)
    steps_streamed(max(12, args.warmup))
    path_used = dict(loader.stats)
    launches0 = _native.launch_count()
    last = []
    with ClockSampler(local_rank) as clocks:
        ms_total = timed(lambda: last.append(steps_streamed(args.steps)), 1)
    launches = _native.launch_count() - launches0
    value = world * n * args.steps / (ms_total * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last[0])
    del last

    # ---- kernel-only timings on the launching stream (roofline of the loader: ONE kernel reads the CSV and writes the arrays)
    stream = torch.cuda.current_stream()
    sptr = ctypes.c_void_p(stream.cuda_stream)
    lib = _native.lib()

    def time_kernel(call, reps=10):
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            a.record(stream)
            call()
            b.record(stream)
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / reps

    rows = [b.n_rows for b in data.blocks]
    keep = [int(b.tensor.shape[0]) for b in data.blocks]
    arena = torch.empty(keep[0] * (rows[0] + 64) + 2 + keep[1] * (rows[1] + 64), dtype=torch.float64, device=dev)
    ws_bytes = int(lib.ms_load_workspace_bytes(n, 0))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    d_res = torch.empty(256 + 2 * _native.MS_LOAD_PEEK, dtype=torch.uint8, device=dev)
    plan = _native.LoadPlan(arena.data_ptr(), arena.numel(), (ctypes.c_int64 * 2)(rows[0] + 64, rows[1] + 64), *getattr(loader, "last_plan", (0, 0)))  # tile, overhang: as the step's loads
    t_fused = time_kernel(lambda: _native.check(lib.ms_load_fused(d_bytes.data_ptr(), n, ctypes.byref(plan), ws.data_ptr(), ws_bytes,
                                                                   d_res.data_ptr(), d_res.data_ptr() + 256, sptr), "ms_load_fused"))
    fres = _native.LoadResult.from_buffer_copy(d_res[: ctypes.sizeof(_native.LoadResult)].cpu().numpy().tobytes())
    assert fres.flags == 0 and fres.status == _native.MS_ERR_NONE, "the single-pass kernel declined the benchmark input"
    # the two-pass path (what answers for files the single-pass kernel declines), for comparison
    src = loader_mod._Source(d_bytes, n, None)
    summary, ws2 = loader._scan(src)
    plan2 = loader_mod._plan(src, summary, layout)
    sections = (_native.Section * _native.MS_MAX_SECTIONS)()
    keepalive = []
    k = 0
    for lay, (r0, r1) in zip(plan2.layouts, plan2.data_rows):
        blk = torch.empty((lay.n_keep, r1 - r0), dtype=torch.float64, device=dev)
        keepalive.append(blk)
        s = sections[k]
        s.row_begin, s.row_end, s.num_cols, s.n_keep, s.d_out, s.stride = r0, r1, lay.num_cols, lay.n_keep, blk.data_ptr(), r1 - r0
        k += 1
    d_status = torch.empty(1, dtype=torch.int64, device=dev)
    d_summary = torch.empty(ctypes.sizeof(_native.ScanSummary), dtype=torch.uint8, device=dev)
    t_parse = time_kernel(lambda: lib.ms_parse(d_bytes.data_ptr(), n, ws2.data_ptr(), sections, k, d_status.data_ptr(), sptr))
    t_scan = time_kernel(lambda: lib.ms_scan(d_bytes.data_ptr(), n, ws2.data_ptr(), ws2.numel(), d_summary.data_ptr(), sptr))
    del keepalive, ws2, arena

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = b_alg / (t_fused * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_load_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")

    # ---- what the PCIe links deliver with every rank copying both ways at once (the ceiling of `e2e`)
    def pcie_probe(mb=256, reps=8):
        h_in = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)
        h_out = torch.empty(mb << 20, dtype=torch.uint8, pin_memory=True)
        d_in = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
        d_out = torch.empty(mb << 20, dtype=torch.uint8, device=dev)
        s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        out = {}
        for name, up, down in (("h2d_alone", True, False), ("d2h_alone", False, True), ("both", True, True)):
            barrier()
            t = time.perf_counter()
            for _ in range(reps):
                if up:
                    with torch.cuda.stream(s1):
                        d_in.copy_(h_in, non_blocking=True)
                if down:
                    with torch.cuda.stream(s2):
                        h_out.copy_(d_out, non_blocking=True)
            torch.cuda.synchronize()
            wall = max_over_ranks(time.perf_counter() - t)
            out[name] = world * reps * (mb << 20) / wall / 1e9  # aggregate GB/s per direction
        return out

    pcie = pcie_probe()

    # ---- end to end from host memory: the public batch API, H2D / compute / D2H overlapped
    def run_e2e(steps):
        """`steps` trials through the public pipelined API: pinned host CSV -> host arrays."""
        last = None
        srcs = [pinned_in[i % 2] for i in range(steps)]
        for d in loader.load_many(srcs, names=[layout] * steps, to_host=True):
            last = d
        for blk in last.blocks:
            blk.host()
        return last

    e2e_steps = max(4, min(args.steps, 8))
    # warm-up, as long as the timed pass: the pinned result buffers (0.38 GB each, ~0.1 s to allocate) and the per-stream
    # device pools of the pipeline reach their steady-state count only after several trials; one allocated inside the
    # timed pass costs it a quarter of its throughput (seen as 35 GB/s instead of 45 with a three-trial warm-up)
    run_e2e(e2e_steps)
    barrier()
    t_e2e = time.perf_counter()
    run_e2e(e2e_steps)
    torch.cuda.synchronize()
    ms_e2e = max_over_ranks((time.perf_counter() - t_e2e) * 1e3)
    e2e_value = world * n * e2e_steps / (ms_e2e * 1e-3) / 1e9
    d2h = int(8 * n_kept)
    # per trial the links carry n bytes up and d2h bytes down at the same time
    ceiling = n / max(n / (pcie["both"] / world * 1e9), d2h / (pcie["both"] / world * 1e9)) * world / 1e9

    # ---- configs[2] and configs[4]: distinct trial files in tmpfs, sharded by file over the ranks
    files_leg, pipeline_leg = None, None
    try:
        per_rank = 8
        n_files = per_rank * world
        base = shm_dir((n_files + 2) * (110 << 20))
        tmp_root = os.path.join(base or tempfile.gettempdir(), f"ms_b200_bench_{os.environ.get('MASTER_PORT', 'single')}")
        os.makedirs(tmp_root, exist_ok=True)
        paths = [os.path.join(tmp_root, f"trial{i:03d}.csv") for i in range(n_files)]
        sizes = []
        for i in range(rank, n_files, world):  # every rank writes its share of the files; all ranks see the directory
            synth_layout("T127", seed=2000 + i).tofile(paths[i])
        barrier()
        sizes = [os.path.getsize(p) for p in paths]
        mine = shard(paths, rank, world, sizes)
        my_bytes = sum(os.path.getsize(p) for p in mine)

        def run_files():
            last = None
            for _name, d in loader.load_files(mine, to_host=True):
                if isinstance(d, Exception):
                    raise d
                last = d
            for blk in last.blocks:
                blk.host()
            torch.cuda.synchronize()

        # what the HOST delivers with every rank reading at once: the same files copied out of the page cache into a
        # pinned buffer by the loader's reader pool, nothing else running (the ceiling of this leg and of configs[4])
        def read_only():
            buf = torch.empty(loader.padded_size(max(os.path.getsize(p) for p in mine)), dtype=torch.uint8, pin_memory=True)
            for p in mine:
                loader_mod.read_file_into(p, buf.numpy(), os.path.getsize(p))

        read_only()
        barrier()
        t = time.perf_counter()
        read_only()
        read_wall = max_over_ranks(time.perf_counter() - t)
        read_ceiling = sum(sizes) / read_wall / 1e9

        run_files()
        barrier()
        t = time.perf_counter()
        run_files()
        wall = max_over_ranks(time.perf_counter() - t)
        files_leg = {"value": sum(sizes) / wall / 1e9, "unit": UNIT, "files": n_files, "files_per_rank": len(mine),
                     "host_read_ceiling": read_ceiling, "frac_of_host_read_ceiling": sum(sizes) / wall / 1e9 / read_ceiling,
                     "host_read_note": "page cache -> pinned memory by the reader pools of all ranks at once, no GPU work",
                     "reader_threads_per_rank": loader_mod._read_pool._max_workers if loader_mod._read_pool is not None else None,
                     "mb_per_file": sizes[0] / 1e6, "ms_per_file_per_rank": wall / max(1, len(mine)) * 1e3,
                     "where": "tmpfs" if base else "temp directory", "bytes_this_rank": my_bytes,
                     "api": "ViconLoader.load_files (reader thread -> pinned ring -> H2D / parse / D2H) -> host arrays; "
                            "distinct T127 trials sharded by size over the ranks; wall clock, max over ranks"}

        from muscle_synergies_b200.pipeline import synergies_for_files_sharded

        kw = dict(min_components=1, max_components=8, n_restarts=20, random_state=0, max_iter=200, tol=0.0)
        # warm-up: one full pass.  The pipeline is one trial deep and every file has its own size, so the pinned result
        # buffers, the read ring and the allocator's blocks reach their steady state only after a pass over the list
        # (a cold pass costs 2-5x: cudaMalloc / cudaHostAlloc and their implicit synchronisations); the timed pass is
        # the steady state a 1000-trial job runs in
        synergies_for_files_sharded(paths, loader=loader, **kw)
        barrier()
        t = time.perf_counter()
        table = synergies_for_files_sharded(paths, loader=loader, **kw)  # includes the host-side gather of the tables
        wall = max_over_ranks(time.perf_counter() - t)
        ok_rows = [r for r in table if "error" not in r]
        n_cycles = len({(r["file"], r["trecho"], r["cycle"]) for r in ok_rows})
        pipeline_leg = {"workload": "configs[4]: per trial load + segment + 8 gait cycles x (RMS envelope, time-normalise 200) + NMF "
                                    "k=1..8 x 20 restarts x 200 it; best-of-restarts VAF tables gathered on the host",
                        "trials": n_files, "cycles": n_cycles, "cycles_per_s": n_cycles / wall, "ms_per_trial_per_rank": wall / per_rank * 1e3,
                        "table_rows": len(table), "failed_files": len(table) - len(ok_rows),
                        "csv_gbs": sum(sizes) / wall / 1e9, "frac_of_host_read_ceiling": sum(sizes) / wall / 1e9 / read_ceiling,
                        "timing": "wall clock, max over ranks, files in tmpfs; second pass over the file list (allocator and pinned pools warm)"}
        barrier()
        if rank == 0:
            shutil.rmtree(tmp_root, ignore_errors=True)
    except Exception as exc:  # noqa: BLE001
        files_leg = files_leg or {"error": f"{type(exc).__name__}: {exc}"}
        pipeline_leg = pipeline_leg or {"error": f"{type(exc).__name__}: {exc}"}

    # ---- NMF-MU extension: rank sweep k=1..8 x 20 restarts on 200 x 16 envelopes (configs[3])
    nmf = bench_nmf(dev) if rank == 0 else None

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, all_cpus)
        try:
            cpu = cpu_baseline()
        except Exception as exc:  # noqa: BLE001
            cpu = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "ms_per_step_serial": ms_serial / args.steps,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {
                "workload": WORKLOAD if layout == "T10" else layout, "csv_bytes_per_gpu": n, "kept_doubles_per_gpu": n_kept,
                "l2": "input (CSV) and output are each larger than the 126 MB L2; no explicit flush",
                "parallelism": f"{world} ranks, trials sharded by file, no data-path collective",
                "host_cpus_bound": len(numa_cpus) if numa_cpus else None,
                "loader_path": path_used,
                "step": f"load + Segmenter + 32 EMG windows per trial; K trials streamed through ViconLoader.load_device_many "
                        f"(depth {args.depth}: the next trials' loader kernels queued while the host works on this one); "
                        "ms_per_step_serial = the same step one trial at a time",
            },
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps,
                    "pcie_ceiling": ceiling, "frac_of_pcie_ceiling": e2e_value / ceiling,
                    "api": "ViconLoader.load_many(pinned host CSV) -> host arrays, 3-stream pipeline, wall clock, two distinct trials alternating"},
            "pcie": dict(pcie, unit="GB/s aggregate per direction, all ranks copying at once (256 MB pinned buffers)"),
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "ms_load_kernel (the whole loader: CSV bytes -> float64 blocks)", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": b_alg, "kernel_ms": t_fused},
            "kernels_ms": {"ms_load_fused": t_fused, "two_pass": {"ms_parse": t_parse, "ms_scan+resolve": t_scan}},
            "nmf": nmf,
            "files": files_leg,
            "pipeline": pipeline_leg,
            "cpu_baseline": cpu,
            "clocks": clocks.summary(),
        }
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=50,
                    help="timed steps of the headline (streamed) and serial legs; the e2e leg times min(max(K, 4), 8) "
                         "trials and reports its own count")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--layout", default="T10", help="synthetic layout (tools/synth_vicon.py LAYOUTS)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--depth", type=int, default=2, help="trials in flight in the streamed headline loop (load_device_many)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (finite floats, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
