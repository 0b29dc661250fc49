"""Times NMF with fixed synergies (the native entry ms_nmf_fixed_h, CUDA events around each call) and scikit-learn's
NMF.transform on one core of the same box:

  a. cross_cycle_vaf's batch: 8 ranks x 8 source cycles x 8 target envelopes = 512 problems of 200 x 16, run to
     convergence (tol 1e-6, max_iter 100 000), both solvers, one launch each
  b. a T10-sized trial envelope, 1.2 M x 16, k = 1..8 in one launch, both solvers: time per iteration at fixed
     iterations (the difference of a 96- and a 32-iteration run), with the fp64 operations and bytes of an iteration
     computed from shapes; then the converged run

    python tools/time_nmf_transform.py [--out DIR]

sklearn runs all 512 problems of (a) for cd and the first 64 for mu, and in (b) k = 8 alone for 32 iterations.
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


def sklearn_transform(X, H, solver, max_iter, tol):
    from sklearn.decomposition import NMF

    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _, _, n_iter = NMF(H.shape[0], solver=solver, max_iter=max_iter, tol=tol)._fit_transform(X, H=H, update_H=False)
    return time.perf_counter() - t0, n_iter


def iteration_cost(n, ranks, solver):
    """fp64 operations of one iteration (per row: K^2 FMAs and K divisions for cd; K^2 FMAs, K divisions and K
    multiplications for mu) and its HBM bytes: X is read once per launch, so an iteration moves only W and X H^T in
    and W and the chunk's saved W out once per chunk of 32 iterations (4 k doubles per row)."""
    flops = sum(n * (2 * k * k + (k if solver == "cd" else 2 * k)) for k in ranks)
    nbytes = sum(n * 8 * 4 * k for k in ranks) / 32
    return flops, nbytes


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
    timer = EntryTimer(torch, nat.lib(), ["ms_nmf_fixed_h"])
    ranks = list(range(1, 9))

    # a. cross_cycle_vaf's 512 problems: synergies of 8 cycles (device CD fits), every target envelope
    env = torch.from_numpy(np.stack([envelopes(c + 1) for c in range(8)])).cuda()
    fits = analysis.nmf_cd_batched(env, [k for _ in range(8) for k in ranks], x_index=[c for c in range(8) for _ in ranks],
                                   max_iter=2000, tol=1e-6)
    H = [fits.H[s * 8 + k - 1] for k in ranks for s in range(8) for _ in range(8)]
    xi = [t for _ in ranks for _ in range(8) for t in range(8)]
    Xh = env.cpu().numpy()
    report["cross_cycle_512x200x16"] = {}
    for solver in ("cd", "mu"):
        analysis.nmf_transform_batched(env, H, x_index=xi, solver=solver, max_iter=100, tol=1e-6)  # warm-up
        timer.take("ms_nmf_fixed_h")
        res = analysis.nmf_transform_batched(env, H, x_index=xi, solver=solver, max_iter=100_000, tol=1e-6)
        kern = timer.take("ms_nmf_fixed_h")[0]
        todo = range(len(H)) if solver == "cd" else range(64)
        with threadpool_limits(1):
            sk = [sklearn_transform(Xh[xi[p]], H[p], solver, 100_000, 1e-6) for p in todo]
        row = {"kernel_ms": kern, "n_iter_max": int(res.n_iter.max()), "n_iter_sum": int(res.n_iter.sum()),
               "us_per_iteration_longest": kern * 1e3 / int(res.n_iter.max()),
               "sklearn_problems": len(sk), "sklearn_s": sum(t for t, _ in sk),
               "sklearn_n_iter_sum": int(sum(it for _, it in sk)), "n_iter_sum_same_problems": int(res.n_iter[list(todo)].sum())}
        report["cross_cycle_512x200x16"][solver] = row
        print(f"cross-cycle 512 x 200x16 {solver}: kernel {kern:.2f} ms, longest {row['n_iter_max']} it, total "
              f"{row['n_iter_sum']} it; sklearn {row['sklearn_s']:.2f} s for {len(sk)} problems "
              f"({row['sklearn_n_iter_sum']} it; device {row['n_iter_sum_same_problems']} it on those)")

    # b. a T10-sized envelope, channel-major on the device as DeviceData keeps it, passed as its transposed view
    n, m = 1_200_000, 16
    chan = torch.from_numpy(np.ascontiguousarray(envelopes(7, n=n).T)).cuda()
    X = chan.T
    Hl = [fits.H[k - 1] for k in ranks]
    report["trial_1p2M_x16_k1to8"] = {}
    for solver in ("cd", "mu"):
        analysis.nmf_transform_batched(X, Hl, solver=solver, max_iter=2, tol=0.0)
        timer.take("ms_nmf_fixed_h")
        t = {}
        for iters in (32, 96):
            analysis.nmf_transform_batched(X, Hl, solver=solver, max_iter=iters, tol=0.0)
            t[iters] = timer.take("ms_nmf_fixed_h")[0]
        per_it = (t[96] - t[32]) / 64 * 1e-3
        flops, nbytes = iteration_cost(n, ranks, solver)
        res = analysis.nmf_transform_batched(X, Hl, solver=solver, max_iter=100_000, tol=1e-6)
        conv = timer.take("ms_nmf_fixed_h")[0]
        with threadpool_limits(1):
            sk_s, sk_it = sklearn_transform(np.ascontiguousarray(X.cpu().numpy()), Hl[-1], solver, 32, 0.0)
        row = {"ms_32_iterations": t[32], "ms_per_iteration": per_it * 1e3, "fp64_GFLOP_per_iteration": flops / 1e9,
               "GFLOPps": flops / per_it / 1e9, "GB_per_iteration": nbytes / 1e9, "GBps": nbytes / per_it / 1e9,
               "converged_ms": conv, "converged_n_iter": res.n_iter.tolist(),
               "sklearn_k8_32_iterations_s": sk_s}
        report["trial_1p2M_x16_k1to8"][solver] = row
        print(f"1.2M x 16 k=1..8 {solver}: {per_it * 1e3:.3f} ms/iteration, {flops / per_it / 1e9:.0f} GFLOP/s fp64 "
              f"({flops / 1e9:.3f} GFLOP), {nbytes / per_it / 1e9:.0f} GB/s ({nbytes / 1e9:.4f} GB); first 32 iterations "
              f"with the X pass {t[32]:.2f} ms; converged {conv:.1f} ms, n_iter {res.n_iter.tolist()}; "
              f"sklearn k=8 alone, 32 iterations {sk_s:.2f} s")
    timer.restore()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_nmf_transform.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
