"""Times matched cosine similarity of synergy sets (the native entry ms_synergy_match, CUDA events around each call)
and the numpy + scipy.optimize.linear_sum_assignment loop a user writes today, on one core of the same box:

  a. one trial: 8 cycles x ranks 1..8, every pair of cycles per rank (8 x 28 = 224 pairs), one launch, with
     similarities and pairings
  b. 8 000 sets of k = 8, m = 16 (a study of 1 000 trials' cycles at one rank), all 31 996 000 pairs, mean only
  c. the same at k = 16

The scipy loop is timed on a sample of pairs; its full-size figure is extrapolated (and labelled so).  The fp64
operations and bytes of a workload are computed from the shapes (`pair_cost`).

    python tools/time_synergy_match.py [--out DIR] [--cpu-sample N]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def pair_cost(k, m):
    """Per pair: 2 k^2 m fp64 operations for S (an FMA counts 2), plus k m multiplications that scale b's rows; the
    sets' rows, 2 k m doubles, come from L2 after the first pass (8 000 sets of k = 16, m = 16 are 16 MB); HBM moves
    only the pair's mean (all pairs: the kernel decodes the pair index, there is no pair list to read)."""
    return 2 * k * k * m + k * m, 8


def cpu_loop(sets, pairs):
    """The per-pair numpy + scipy loop; returns seconds per pair."""
    from oracle import synergy_match_oracle as so

    t0 = time.perf_counter()
    for a, b in pairs:
        so.match(sets[a], sets[b])
    return (time.perf_counter() - t0) / len(pairs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cpu-sample", type=int, default=4000)
    args = ap.parse_args()

    import numpy as np
    import torch
    from threadpoolctl import threadpool_limits

    import __graft_entry__ as g

    g.build()
    from muscle_synergies_b200 import _native as nat
    from muscle_synergies_b200 import analysis
    from tools.time_nmf_cd import EntryTimer

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    report = {"gpu": smi[0] if smi else torch.cuda.get_device_name(0), "cpu_threads": 1}
    print("device:", report["gpu"])
    timer = EntryTimer(torch, nat.lib(), ["ms_synergy_match"])
    rng = np.random.default_rng(0)

    # a. one trial
    m = 16
    sets = [rng.uniform(0, 1, (k, m)) for k in range(1, 9) for _ in range(8)]
    iu = np.stack(np.triu_indices(8, 1), axis=1)
    pairs = np.concatenate([iu + 8 * r for r in range(8)])
    for _ in range(3):
        analysis.match_synergies_batched(sets, pairs, similarities=True, permutations=True)
    timer.take("ms_synergy_match")
    reps = 50
    t0 = time.perf_counter()
    for _ in range(reps):
        analysis.match_synergies_batched(sets, pairs, similarities=True, permutations=True)
    host_ms = (time.perf_counter() - t0) / reps * 1e3
    kern = sorted(timer.take("ms_synergy_match"))
    with threadpool_limits(1):
        cpu = cpu_loop(sets, pairs)
    row = {"pairs": len(pairs), "entry_ms_median": kern[len(kern) // 2], "entry_ms_min": kern[0],
           "python_call_ms": host_ms, "scipy_loop_ms": cpu * len(pairs) * 1e3, "scipy_us_per_pair": cpu * 1e6}
    report["trial_8_ranks_x_28_pairs"] = row
    print(f"trial 224 pairs (k = 1..8): entry {row['entry_ms_median']:.3f} ms (median of {reps}; the entry includes "
          f"its status read-back), Python call {host_ms:.3f} ms; scipy loop {row['scipy_loop_ms']:.2f} ms "
          f"({row['scipy_us_per_pair']:.1f} us/pair)")

    # b, c. 8 000 sets, all pairs, mean only
    n_sets = 8000
    P = n_sets * (n_sets - 1) // 2
    for k in (8, 16):
        host = rng.uniform(0, 1, (n_sets, k, m))
        dev = torch.from_numpy(host).cuda()
        res = analysis.match_synergies_batched(dev)  # warm-up
        timer.take("ms_synergy_match")
        times = []
        for _ in range(3):
            res = analysis.match_synergies_batched(dev)
            times.append(timer.take("ms_synergy_match")[0])
        kern = min(times)
        checksum = float(res.mean.sum())
        sample = rng.choice(P, args.cpu_sample, replace=False)
        a, b = np.triu_indices(n_sets, 1)
        sample_pairs = list(zip(a[sample], b[sample]))
        means = res.mean.cpu().numpy()
        from oracle import synergy_match_oracle as so

        worst = max(abs(means[p] - so.match(host[a[p]], host[b[p]])[0]) for p in sample[:500])
        with threadpool_limits(1):
            cpu = cpu_loop(host, sample_pairs)
        flops, nbytes = pair_cost(k, m)
        row = {"sets": n_sets, "k": k, "m": m, "pairs": P, "kernel_ms_min": kern, "kernel_ms_all": times,
               "pairs_per_s": P / (kern * 1e-3), "S_fp64_GFLOP": flops * P / 1e9,
               "S_fp64_TFLOPps": flops * P / (kern * 1e-3) / 1e12, "hbm_GB": nbytes * P / 1e9,
               "hbm_bound_ms": nbytes * P / HBM_BYTES_PER_S * 1e3, "mean_checksum": checksum,
               "max_abs_diff_vs_oracle_500_pairs": worst, "scipy_us_per_pair": cpu * 1e6,
               "scipy_sample_pairs": len(sample_pairs), "scipy_extrapolated_s": cpu * P}
        report[f"sets8000_k{k}_all_pairs"] = row
        print(f"8000 sets k = {k}: {P} pairs in {kern:.1f} ms ({row['pairs_per_s'] / 1e9:.2f} G pairs/s); S is "
              f"{row['S_fp64_GFLOP']:.0f} GFLOP fp64 ({row['S_fp64_TFLOPps']:.2f} TFLOP/s); HBM {row['hbm_GB']:.2f} GB "
              f"(at 7.7 TB/s {row['hbm_bound_ms']:.3f} ms); max |diff| vs oracle on 500 pairs {worst:.1e}; scipy loop "
              f"{row['scipy_us_per_pair']:.1f} us/pair on {len(sample_pairs)} sampled pairs -> "
              f"{row['scipy_extrapolated_s']:.0f} s for all pairs (extrapolated)")
        del dev, res
        torch.cuda.empty_cache()
    timer.restore()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_synergy_match.json"), "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
