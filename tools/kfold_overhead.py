"""What K-fold cross-validation costs, and what running its folds together gains: at BASELINE configs 2, 3 and 5 and
K = 5, 10, the wall time of
  (a) bnr_fit_kfold: all K fold handles advanced by one control loop, every fold's sweeps launched before any is
      waited for;
  (b) the same K fits one after another: each fold's handle with its held-out table (bnr_set_heldout) driven through
      the operations bnr_fit issues (bnr_fit_plan, replayed by `replay`), then its bnr_lpd_summary;
  (c) one bnr_fit of K x C chains on the full data: the throughput reference,
then the per-sweep cost of a held-out table of n / K observations against a handle without it, next to the card's name
and power limit.

    python tools/kfold_overhead.py [--configs c2,c3,c5] [--ks 5,10] [--nburn 60] [--nsamples 60] [--reps 5]

The schedule is fixed (psrf_cutoff 1e9: one R-hat check, no extension), so every arm runs the same sweeps.  Chains per
fold: 16 at config 2, 8 at config 3, 32 at config 5.  Each arm runs once untimed, then the three arms alternate --reps
times; the host clock brackets each call (every call ends synchronised) and the median is reported.
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

from kfold_util import fit_params, plan, replay, split  # noqa: E402

_DP = C.POINTER(C.c_double)
CHAINS = {"c2": 16, "c3": 8, "c5": 32}


def kfold(bnr, p, X, y, K, folds):
    """bnr_fit_kfold: (pointwise elpd_kfold, info)."""
    from bnr_b200 import capi
    L = bnr.lib()
    Xf = np.asfortranarray(X, dtype=np.float64)
    yv = np.ascontiguousarray(y, dtype=np.float64)
    fv = np.ascontiguousarray(folds, dtype=np.int32)
    res = C.c_void_p()
    capi.check_fit(L.bnr_fit_kfold(C.byref(p), Xf.ctypes.data_as(_DP), yv.ctypes.data_as(_DP), K,
                                   fv.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(res)))
    try:
        info = capi.FitInfo()
        capi.check_fit(L.bnr_fit_get_info(res, C.byref(info)))
        pw = np.empty(X.shape[0])
        capi.check_fit(L.bnr_fit_kfold_pointwise(res, pw.ctypes.data_as(_DP)))
        return pw, info
    finally:
        L.bnr_fit_free(res)


def sequential(bnr, p, X, y, K, folds):
    """Arm (b): the folds one after another, each a standalone handle with its held-out table: pointwise elpd_kfold."""
    import torch
    from bnr_b200.engine import lpd_summary
    out = np.empty(X.shape[0])
    for f in range(1, K + 1):
        Xt, yt, Xh, yh = split(X, y, folds, f)
        pf = fit_params(bnr, Xt.shape[0], p.base.V, p.base.R, p.base.num_chains, p.base.seed,
                        p.base.chain_offset + (f - 1) * p.base.num_chains, nburn=p.nburn, nsamples=p.nsamples,
                        psrf_cutoff=p.psrf_cutoff, return_state=p.return_state)
        with replay(bnr, pf, plan(bnr, pf, (0.0,)), Xt, yt, Xh, yh) as eng:
            N = p.base.num_chains * p.nsamples
            buf = torch.empty(N * Xh.shape[0], dtype=torch.float64, device="cuda:%d" % p.base.device)
            eng.export_predictions(p.nburn, p.nsamples, buf.data_ptr())
            out[folds == f] = lpd_summary(p.base.device, buf.data_ptr(), N, Xh.shape[0])
    return out


def full_fit(bnr, p, X, y):
    """Arm (c): one bnr_fit of the same total chains on the full data."""
    from bnr_b200 import capi
    L = bnr.lib()
    Xf = np.asfortranarray(X, dtype=np.float64)
    yv = np.ascontiguousarray(y, dtype=np.float64)
    res = C.c_void_p()
    capi.check_fit(L.bnr_fit(C.byref(p), Xf.ctypes.data_as(_DP), yv.ctypes.data_as(_DP), C.byref(res)))
    L.bnr_fit_free(res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3,c5")
    ap.add_argument("--ks", default="5,10")
    ap.add_argument("--nburn", type=int, default=60)
    ap.add_argument("--nsamples", type=int, default=60)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=40, help="sweeps per repetition of the held-out table cost")
    args = ap.parse_args()
    import bench
    from __graft_entry__ import load_package
    bnr = load_package()
    from bnr_b200.capi import STATE
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    print("schedule: nburn %d, nsamples %d, psrf_cutoff 1e9 (fixed); wall ms, median of %d alternated runs"
          % (args.nburn, args.nsamples, args.reps))
    for cfg in args.configs.split(","):
        X, y, info = bench.synth(cfg)
        n, R, V = X.shape[0], info["R"], bench.CONFIGS[cfg]["V"]
        C_ = CHAINS[cfg]
        for K in (int(k) for k in args.ks.split(",")):
            folds = bnr.kfold_split(n, K, 11)
            sched = dict(nburn=args.nburn, nsamples=args.nsamples, psrf_cutoff=1e9, return_state=STATE["none"])
            pk = fit_params(bnr, n, V, R, C_, 5, **sched)
            pc = fit_params(bnr, n, V, R, K * C_, 5, **sched)
            arms = [("a kfold", lambda: kfold(bnr, pk, X, y, K, folds)[0]),
                    ("b sequential", lambda: sequential(bnr, pk, X, y, K, folds)),
                    ("c full K*C", lambda: full_fit(bnr, pc, X, y))]
            res = [fn() for _, fn in arms]           # warm-up, and the two pointwise arrays to compare
            same = np.array_equal(res[0], res[1])
            times = [[] for _ in arms]
            for _ in range(args.reps):
                for i, (_, fn) in enumerate(arms):
                    t0 = time.perf_counter()
                    fn()
                    times[i].append(1e3 * (time.perf_counter() - t0))
            med = [float(np.median(t)) for t in times]
            sweeps = args.nburn + args.nsamples - 1
            for i, (name, _) in enumerate(arms):
                print("%s n=%d K=%2d C/fold=%3d %-13s %9.1f ms (spread %.1f-%.1f)  %.2f k chain-sweeps/s  a/this %.2f"
                      % (cfg, n, K, C_, name, med[i], min(times[i]), max(times[i]),
                         K * C_ * sweeps / med[i], med[0] / med[i]))
            print("%s K=%d: elpd_kfold of (a) and (b) bit-identical: %s; elpd_kfold = %.2f"
                  % (cfg, K, same, float(res[0].sum())))
        # per-sweep cost of a held-out table of n / K observations (K = the first of --ks) on one handle of C chains
        K = int(args.ks.split(",")[0])
        Xt, yt, Xh, yh = split(X, y, bnr.kfold_split(n, K, 11), 1)
        engines = []
        for on in (False, True):
            eng = bnr.Engine(Xt, yt, R, num_chains=C_, seed=3)
            if on:
                eng.set_heldout(Xh, yh, args.sweeps + 8)
            eng.init_state()
            eng.run(6)
            engines.append(eng)
        t = [[], []]
        for _ in range(args.reps):
            for i, eng in enumerate(engines):
                eng.trace_row = 0
                eng.run(args.sweeps)
                t[i].append(eng.last_run_ms() / args.sweeps)
        base = float(np.median(t[0]))
        for i, name in enumerate(("no table", "held-out table")):
            m = float(np.median(t[i]))
            print("%s n_train=%d m=%d C=%d %-15s %.4f ms/sweep (spread %.4f-%.4f)  %+.2f %%"
                  % (cfg, Xt.shape[0], Xh.shape[0], C_, name, m, min(t[i]), max(t[i]), 100.0 * (m / base - 1.0)))
        for eng in engines:
            eng.close()


if __name__ == "__main__":
    main()
