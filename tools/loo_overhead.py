"""Cost of the pointwise log-likelihood (PSIS-LOO / WAIC): ms per sweep without and with the log-likelihood table at
BASELINE configs 2, 3 and 5, the two arms alternated inside one process, then the time of bnr_loo_summary on a pooled
table of N = 64 x 20 000 draws x n = 1000 observations, next to the card's name and power limit.

    python tools/loo_overhead.py [--sweeps 40] [--reps 5] [--configs c2,c3,c5] [--draws 1280000] [--obs 1000]

Each arm is its own handle on the config's inputs (bench.synth) and chain count, warmed up with a few sweeps; every
repetition times each arm over --sweeps sweeps with CUDA events (bnr_last_run_ms) and the median is reported.  The
summary is timed on a table of normal draws (10 GB at the defaults, generated on the device) with CUDA events around
the whole call (select, pass, tail kernels and the copy of the [5][n] results), median of --reps calls after one warm-up.
"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=40)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="c2,c3,c5")
    ap.add_argument("--draws", type=int, default=64 * 20000)
    ap.add_argument("--obs", type=int, default=1000)
    args = ap.parse_args()
    import torch
    import bench
    from __graft_entry__ import load_package
    bnr = load_package()
    from bnr_b200.engine import loo_summary
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    for cfg in args.configs.split(","):
        X, y, info = bench.synth(cfg)
        C = bench.CONFIGS[cfg]["chains"]
        arms = [("off", False), ("log-likelihood", True)]
        engines = []
        for name, on in arms:
            eng = bnr.Engine(X, y, info["R"], num_chains=C, seed=3)
            if on:
                eng.set_loglik(args.sweeps + 8)
            eng.init_state()
            eng.run(6)
            engines.append(eng)
        times = [[] for _ in arms]
        for _ in range(args.reps):
            for i, eng in enumerate(engines):
                eng.trace_row = 0
                eng.run(args.sweeps)
                times[i].append(eng.last_run_ms() / args.sweeps)
        base = float(np.median(times[0]))
        for i, (name, _) in enumerate(arms):
            t = float(np.median(times[i]))
            print("%s n=%d C=%d %-16s %.4f ms/sweep (spread %.4f-%.4f)  %+.2f %%" %
                  (cfg, X.shape[0], C, name, t, min(times[i]), max(times[i]), 100.0 * (t / base - 1.0)))
        for eng in engines:
            eng.close()
    N, n = args.draws, args.obs
    g = torch.Generator(device="cuda:0").manual_seed(7)
    tab = -1.0 + 0.5 * torch.randn(N, n, dtype=torch.float64, device="cuda:0", generator=g)
    loo_summary(0, tab.data_ptr(), N, n)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ts = []
    for _ in range(args.reps):
        ev0.record()
        out = loo_summary(0, tab.data_ptr(), N, n)
        ev1.record()
        ev1.synchronize()
        ts.append(ev0.elapsed_time(ev1))
    print("bnr_loo_summary N=%d n=%d (%.2f GB): %.2f ms (spread %.2f-%.2f); max pareto k %.3f" %
          (N, n, 8.0 * N * n / 1e9, float(np.median(ts)), min(ts), max(ts), float(np.max(out["pareto_k"]))))


if __name__ == "__main__":
    main()
