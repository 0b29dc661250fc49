"""Times β-divergence NMF (the native entry ms_nmf_beta, CUDA events around each call) and scikit-learn's
NMF(solver="mu", beta_loss=...) on one core of the same box, for beta_loss "kullback-leibler" and "itakura-saito":

  a. 200 x 16, k = 1..8 in one launch, run to convergence with the reference's defaults (tol 1e-6, max_iter 100 000)
     from the device's nndsvda init; sklearn fits each rank from its own nndsvda init
  b. a trial's 64 problems (8 cycle envelopes x k = 1..8, x_index) in one launch, same settings; cycle 0 is (a)'s
     envelope, so sklearn's time for it is (a)'s
  c. a T10-sized trial envelope, 1.2 M x 16 (channel-major, passed as its transposed view), k = 1..8 in one launch:
     time per iteration at fixed iterations (the difference of a 40- and a 20-iteration run), with the fp64
     operations, transcendental calls and HBM bytes of an iteration computed from shapes

    python tools/time_nmf_beta.py [--out DIR]
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

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def sklearn_fit(X, k, beta, max_iter, tol):
    from sklearn.decomposition import NMF

    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = NMF(k, solver="mu", beta_loss=beta, init="nndsvda", max_iter=max_iter, tol=tol)
        model.fit_transform(X)
    return time.perf_counter() - t0, model.n_iter_


def iteration_cost(n, m, ranks, beta):
    """One streaming iteration, summed over the problems.  Per element of X and problem: WH twice (2 k FMAs), the
    W-step numerator and denominator (2 k FMAs; KL: k), the H-step sums (2 k FMAs; KL: k FMAs + k adds); an FMA counts
    2 operations.  Transcendental-class calls per element: 2 divisions (KL, IS; IS also 4 multiplications), 4 pow for
    any other beta.  HBM: X read once per problem (X, 154 MB at 1.2 M x 16, exceeds the 126 MB L2) and W read and
    written once."""
    kl = beta == "kullback-leibler"
    flops = sum(n * m * (2 * (2 * k + (k if kl else 2 * k)) + (3 * k if kl else 4 * k)) for k in ranks)
    calls = sum(n * m * (2 if beta in ("kullback-leibler", "itakura-saito") else 4) for _ in ranks)
    nbytes = sum(n * m * 8 + 2 * n * k * 8 for k in ranks)
    return flops, calls, nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    from threadpoolctl import threadpool_limits

    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import _native as nat
    from muscle_synergies_b200 import analysis
    from test_nmf_oracle import envelopes
    from tools.time_nmf_cd import EntryTimer

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "sklearn_threads": 1}
    print("device:", report["gpu"])
    timer = EntryTimer(torch, nat.lib(), ["ms_nmf_beta"])
    ranks = list(range(1, 9))
    betas = ("kullback-leibler", "itakura-saito")

    # a. one gait cycle, k = 1..8
    X = envelopes(1)
    report["cycle_200x16_k1to8"] = {}
    for beta in betas:
        analysis.nmf_beta_batched(X, ranks, beta, max_iter=50, tol=0.0)  # warm-up
        timer.take("ms_nmf_beta")
        res = analysis.nmf_beta_batched(X, ranks, beta, max_iter=100_000, tol=1e-6)
        kern = timer.take("ms_nmf_beta")[0]
        with threadpool_limits(1):
            sk = [sklearn_fit(X, k, beta, 100_000, 1e-6) for k in ranks]
        row = {"kernel_ms": kern, "n_iter": res.n_iter.tolist(), "us_per_iteration_longest": kern * 1e3 / int(res.n_iter.max()),
               "sklearn_s": sum(t for t, _ in sk), "sklearn_n_iter": [int(it) for _, it in sk]}
        report["cycle_200x16_k1to8"][beta] = row
        print(f"200x16 k=1..8 {beta}: kernel {kern:.2f} ms, n_iter {row['n_iter']}; sklearn {row['sklearn_s']:.2f} s, "
              f"n_iter {row['sklearn_n_iter']}")

    # b. a trial's 64 problems
    env = torch.from_numpy(np.stack([envelopes(c + 1) for c in range(8)])).cuda()
    tr = [k for _ in range(8) for k in ranks]
    xi = [c for c in range(8) for _ in ranks]
    report["trial_64_problems"] = {}
    for beta in betas:
        analysis.nmf_beta_batched(env, tr, beta, x_index=xi, max_iter=50, tol=0.0)
        timer.take("ms_nmf_beta")
        res = analysis.nmf_beta_batched(env, tr, beta, x_index=xi, max_iter=100_000, tol=1e-6)
        kern = timer.take("ms_nmf_beta")[0]
        a = report["cycle_200x16_k1to8"][beta]  # cycle 0 is workload a's envelope: sklearn's time for it is a's
        row = {"kernel_ms": kern, "n_iter_max": int(res.n_iter.max()), "n_iter_sum": int(res.n_iter.sum()),
               "sklearn_cycle0_s": a["sklearn_s"], "sklearn_cycle0_n_iter_sum": int(sum(a["sklearn_n_iter"]))}
        report["trial_64_problems"][beta] = row
        print(f"trial 64 problems {beta}: kernel {kern:.1f} ms, longest {row['n_iter_max']} it, total "
              f"{row['n_iter_sum']} it; sklearn cycle 0 alone (8 of 64 problems) {row['sklearn_cycle0_s']:.2f} s")

    # c. a T10-sized envelope, channel-major on the device, passed as its transposed view
    n, m = 1_200_000, 16
    chan = torch.from_numpy(np.ascontiguousarray(envelopes(7, n=n).T)).cuda()
    Xl = chan.T
    report["trial_1p2M_x16_k1to8"] = {}
    for beta in betas:
        analysis.nmf_beta_batched(Xl, ranks, beta, max_iter=2, tol=0.0)
        timer.take("ms_nmf_beta")
        t = {}
        for iters in (20, 40):
            analysis.nmf_beta_batched(Xl, ranks, beta, max_iter=iters, tol=0.0)
            t[iters] = timer.take("ms_nmf_beta")[0]
        per_it = (t[40] - t[20]) / 20 * 1e-3
        flops, calls, nbytes = iteration_cost(n, m, ranks, beta)
        row = {"ms_20_iterations": t[20], "ms_40_iterations": t[40], "ms_per_iteration": per_it * 1e3,
               "fp64_GFLOP_per_iteration": flops / 1e9, "GFLOPps": flops / per_it / 1e9,
               "transcendental_calls_per_iteration": calls, "GB_per_iteration": nbytes / 1e9,
               "GBps": nbytes / per_it / 1e9, "hbm_bound_ms": nbytes / HBM_BYTES_PER_S * 1e3}
        report["trial_1p2M_x16_k1to8"][beta] = row
        print(f"1.2M x 16 k=1..8 {beta}: {per_it * 1e3:.3f} ms/iteration; {flops / 1e9:.2f} GFLOP fp64 "
              f"({flops / per_it / 1e9:.0f} GFLOP/s), {calls / 1e6:.0f} M divisions/pow; {nbytes / 1e9:.3f} GB HBM "
              f"({nbytes / per_it / 1e9:.0f} GB/s; at 7.7 TB/s {row['hbm_bound_ms']:.3f} ms)")
    timer.restore()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_nmf_beta.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
