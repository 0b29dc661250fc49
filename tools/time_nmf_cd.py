"""Times the coordinate-descent NMF kernels (CUDA events around each native entry point) and scikit-learn's
NMF(solver="cd") on the same box:

  1. the tutorial sweep on 200 x 16 envelopes: k = 1..8, tol 1e-6, max_iter 100 000, init nndsvda, run to convergence
  2. one trial's 64 cycle x rank problems (8 envelopes x k = 1..8) in one launch, same settings
  3. the streaming regime on 1.2 M x 16 at fixed iterations, in GB/s of algorithmic bytes (8 n m + P 16 n k per
     iteration) against the HBM bandwidth a device-to-device copy reaches on the same card

    python tools/time_nmf_cd.py [--sklearn-cycles C] [--out DIR]

sklearn runs the trial's cycles 0..C-1 only (default 2; each cycle costs about 10 s of one core) and the total is
reported for those cycles.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


class EntryTimer:
    """Wraps native entry points: CUDA events around every call, kept per name."""

    def __init__(self, torch, lib, names):
        self.torch, self.lib, self.real, self.times = torch, lib, {}, {n: [] for n in names}
        for name in names:
            real = getattr(lib, name)
            self.real[name] = real

            def timed(*a, _real=real, _name=name):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                rc = _real(*a)
                e1.record()
                self.times[_name].append((e0, e1))
                return rc

            setattr(lib, name, timed)

    def take(self, name):
        self.torch.cuda.synchronize()
        out = [a.elapsed_time(b) for a, b in self.times[name]]
        self.times[name] = []
        return out

    def restore(self):
        for name, real in self.real.items():
            setattr(self.lib, name, real)


def sklearn_cd(X, k, max_iter, tol):
    from sklearn.decomposition import NMF

    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = NMF(n_components=k, init="nndsvda", max_iter=max_iter, tol=tol)
        model.fit_transform(X)
    return time.perf_counter() - t0, model.n_iter_


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sklearn-cycles", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import _native as nat
    from muscle_synergies_b200 import analysis
    from test_nmf_oracle import envelopes

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "cpu_threads": os.cpu_count()}
    print("device:", report["gpu"])
    lib = nat.lib()
    timer = EntryTimer(torch, lib, ["ms_nmf_cd_batched_planned", "ms_nmf_cd_stream", "ms_nndsvd_init"])
    ranks = list(range(1, 9))

    # 1. tutorial sweep
    X = envelopes(1)
    Xd = torch.from_numpy(X).cuda()
    analysis.nmf_cd_batched(Xd, ranks, max_iter=100, tol=1e-6)  # warm-up
    timer.take("ms_nmf_cd_batched_planned"), timer.take("ms_nndsvd_init")
    res = analysis.nmf_cd_batched(Xd, ranks, max_iter=100_000, tol=1e-6)
    kern = timer.take("ms_nmf_cd_batched_planned")[0]
    init = timer.take("ms_nndsvd_init")[0]
    sk = [sklearn_cd(X, k, 100_000, 1e-6) for k in ranks]
    sweep = {"n_iter": res.n_iter.tolist(), "kernel_ms": kern, "nndsvd_ms": init,
             "us_per_iteration_longest": kern * 1e3 / int(res.n_iter.max()),
             "sklearn_s": [t for t, _ in sk], "sklearn_n_iter": [it for _, it in sk], "sklearn_total_s": sum(t for t, _ in sk)}
    report["tutorial_sweep_200x16"] = sweep
    print(f"tutorial sweep 200x16 k=1..8: kernel {kern:.1f} ms + nndsvd {init:.3f} ms; n_iter {res.n_iter.tolist()}; "
          f"{sweep['us_per_iteration_longest']:.2f} us/iteration (longest problem); sklearn {sweep['sklearn_total_s']:.2f} s "
          f"(n_iter {sweep['sklearn_n_iter']})")

    # 2. one trial: 8 cycles x k = 1..8
    Xs = np.stack([envelopes(c + 1) for c in range(8)])
    Xsd = torch.from_numpy(Xs).cuda()
    tr = [k for _ in range(8) for k in ranks]
    xi = [c for c in range(8) for _ in ranks]
    analysis.nmf_cd_batched(Xsd, tr, x_index=xi, max_iter=100, tol=1e-6)
    timer.take("ms_nmf_cd_batched_planned"), timer.take("ms_nndsvd_init")
    res = analysis.nmf_cd_batched(Xsd, tr, x_index=xi, max_iter=100_000, tol=1e-6)
    kern = timer.take("ms_nmf_cd_batched_planned")[0]
    init = timer.take("ms_nndsvd_init")[0]
    C = max(0, min(8, args.sklearn_cycles))
    sk = [sklearn_cd(Xs[c], k, 100_000, 1e-6)[0] for c in range(C) for k in ranks]
    trial = {"problems": len(tr), "kernel_ms": kern, "nndsvd_ms": init, "n_iter_max": int(res.n_iter.max()),
             "n_iter_sum": int(res.n_iter.sum()), "sklearn_cycles": C, "sklearn_s_for_those_cycles": sum(sk)}
    report["trial_64_problems"] = trial
    print(f"trial 64 problems: kernel {kern:.1f} ms + nndsvd {init:.3f} ms; longest {trial['n_iter_max']} it, "
          f"total {trial['n_iter_sum']} it; sklearn {sum(sk):.2f} s for {C} of 8 cycles")

    # 3. streaming regime on 1.2 M x 16, fixed iterations
    copy_src = torch.empty(1 << 28, dtype=torch.float64, device="cuda")  # 2 GiB: far beyond L2
    copy_dst = torch.empty_like(copy_src)
    copy_dst.copy_(copy_src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        copy_dst.copy_(copy_src)
    e1.record()
    torch.cuda.synchronize()
    hbm = 10 * 2 * copy_src.numel() * 8 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del copy_src, copy_dst
    n, m = 1_200_000, 16
    Xl = torch.from_numpy(envelopes(7, n=n)).cuda()
    stream = {"hbm_copy_GBps": hbm}
    for label, rk in (("P=1 k=8", [8]), ("P=8 k=1..8", ranks)):
        analysis.nmf_cd_batched(Xl, rk, max_iter=2, tol=0.0, regime="stream")
        timer.take("ms_nmf_cd_stream"), timer.take("ms_nndsvd_init")
        t = {}
        for iters in (10, 60):
            analysis.nmf_cd_batched(Xl, rk, max_iter=iters, tol=0.0, regime="stream")
            t[iters] = timer.take("ms_nmf_cd_stream")[0]
        init = timer.take("ms_nndsvd_init")[-1]
        per_it = (t[60] - t[10]) / 50 * 1e-3
        nbytes = 8 * n * m + sum(16 * n * k for k in rk)
        stream[label] = {"ms_per_iteration": per_it * 1e3, "algorithmic_GB_per_iteration": nbytes / 1e9,
                         "GBps": nbytes / per_it / 1e9, "share_of_copy_bandwidth": nbytes / per_it / 1e9 / hbm,
                         "nndsvd_ms": init}
        print(f"stream 1.2M x 16 {label}: {per_it * 1e3:.3f} ms/iteration, {nbytes / per_it / 1e9:.0f} GB/s "
              f"({100 * nbytes / per_it / 1e9 / hbm:.0f} % of the {hbm:.0f} GB/s a D2D copy reaches); nndsvd {init:.2f} ms")
    secs = sklearn_cd(Xl.cpu().numpy(), 8, 10, 0.0)[0]  # includes sklearn's randomized-SVD init
    stream["sklearn_k8_10_iterations_s"] = secs
    print(f"sklearn 1.2M x 16 k=8, 10 iterations (with its init): {secs:.2f} s")
    report["stream_1p2M_x16"] = stream
    timer.restore()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_nmf_cd.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
