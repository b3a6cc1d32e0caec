"""Cost of the predictions for new networks: ms per sweep without and with predictors (m new networks, mean and
predictive mode) at BASELINE configs 2, 3 and 5, the arms alternated inside one process, then the pooled select against
k_summary_select on the same buffer (tools/lab/pred_select_lab, built as its header says), next to the card's name and
power limit.

    python tools/predict_overhead.py [--sweeps 40] [--reps 5] [--configs c2,c3,c5] [--ms 100,1000]

Each arm is its own handle on the config's inputs (bench.synth) and chain count, warmed up with a few sweeps; every
repetition times each arm over --sweeps sweeps with CUDA events (bnr_last_run_ms) and the median is reported.
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
    ap.add_argument("--ms", default="100,1000")
    args = ap.parse_args()
    import bench
    from __graft_entry__ import load_package
    bnr = load_package()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    ms = [int(x) for x in args.ms.split(",")]
    for cfg in args.configs.split(","):
        X, y, info = bench.synth(cfg)
        C = bench.CONFIGS[cfg]["chains"]
        rng = np.random.default_rng(5)
        arms = [("off", None, False)]
        for m in ms:
            Xn = X[rng.integers(0, X.shape[0], size=m)]          # new networks drawn like the fitted ones
            arms += [("m=%d mean" % m, Xn, False), ("m=%d predictive" % m, Xn, True)]
        engines = []
        for name, Xn, pred in arms:
            eng = bnr.Engine(X, y, info["R"], num_chains=C, seed=3)
            if Xn is not None:
                eng.set_predictors(Xn, args.sweeps + 8, predictive=pred)
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
        for i, (name, _, _) in enumerate(arms):
            t = float(np.median(times[i]))
            print("%s %-30s %.4f ms/sweep (spread %.4f-%.4f)  %+.2f %%" %
                  (cfg, name, t, min(times[i]), max(times[i]), 100.0 * (t / base - 1.0)))
        for eng in engines:
            eng.close()
    lab = os.path.join(ROOT, "tools", "lab", "pred_select_lab")
    if os.path.exists(lab):
        print(subprocess.run([lab], capture_output=True, text=True).stdout.strip())
    else:
        print("pooled select: %s not built" % lab)


if __name__ == "__main__":
    main()
