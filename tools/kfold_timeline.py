#!/usr/bin/env python
"""Kernel timeline of K-fold cross-validation: bnr_fit_kfold (a) against the same folds run one after another (b), at one
config, K and chain count per fold (development tool, not part of the product; tools/kfold_overhead.py times the arms).

CUPTI (through torch.profiler) records every kernel of one warmed-up call of each arm.  Printed per arm: the wall time
of the call, the GPU-busy time (the union of all kernel intervals), the summed kernel time and their ratio (the mean
number of kernels running at once), and per kernel name the launches, summed and mean duration.  When (a) runs the same
kernels as (b) but each takes longer, the folds slow each other down on the device; when the busy time of (a) falls short
of its wall time, the host or the launches hold it back.

    python tools/kfold_timeline.py [--config c5] [--k 10] [--chains 32] [--nburn 60] [--nsamples 60] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True


def kernels(fn):
    """(wall ms of fn(), kernel events sorted by start) with CUDA activities recorded around one call."""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        wall = 1e3 * (time.perf_counter() - t0)
    path = os.path.join(tempfile.mkdtemp(), "trace.json")
    prof.export_chrome_trace(path)
    ev = [e for e in json.load(open(path))["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    return wall, ev


def describe(name, wall, ev, out, top=8):
    busy, end = 0.0, -1e30
    for e in ev:                                   # union of [ts, ts + dur)
        s, t = e["ts"], e["ts"] + e["dur"]
        if s > end:
            busy += t - s
            end = t
        elif t > end:
            busy += t - end
            end = t
    tot = sum(e["dur"] for e in ev)
    span = (max(e["ts"] + e["dur"] for e in ev) - ev[0]["ts"]) / 1e3
    print("%s: wall %.1f ms, kernel span %.1f ms, GPU busy %.1f ms, summed kernel time %.1f ms, mean kernels at once "
          "%.2f, %d kernels" % (name, wall, span, busy / 1e3, tot / 1e3, tot / busy, len(ev)), file=out)
    per = {}
    for e in ev:
        nm = e["name"].split("(")[0].replace("bnr::", "").replace("void ", "")
        c, d = per.get(nm, (0, 0.0))
        per[nm] = (c + 1, d + e["dur"])
    for nm, (c, d) in sorted(per.items(), key=lambda kv: -kv[1][1])[:top]:
        print("    %-28s %6d launches  %9.1f ms  mean %8.1f us" % (nm, c, d / 1e3, d / c), file=out)
    return per


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c5")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--chains", type=int, default=32)
    ap.add_argument("--nburn", type=int, default=60)
    ap.add_argument("--nsamples", type=int, default=60)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import bench
    import kfold_overhead as KO
    from __graft_entry__ import load_package
    bnr = load_package()
    from bnr_b200.capi import STATE
    out = open(args.out, "w") if args.out else sys.stdout
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    X, y, info = bench.synth(args.config)
    n, R, V = X.shape[0], info["R"], bench.CONFIGS[args.config]["V"]
    folds = bnr.kfold_split(n, args.k, 11)
    p = KO.fit_params(bnr, n, V, R, args.chains, 5, nburn=args.nburn, nsamples=args.nsamples, psrf_cutoff=1e9,
                      return_state=STATE["none"])
    print("# card: %s; %s n=%d K=%d C/fold=%d, %d + %d rows, one warmed-up call per arm" %
          (card, args.config, n, args.k, args.chains, args.nburn, args.nsamples), file=out)
    arms = [("(a) bnr_fit_kfold", lambda: KO.kfold(bnr, p, X, y, args.k, folds)),
            ("(b) sequential", lambda: KO.sequential(bnr, p, X, y, args.k, folds))]
    for _, fn in arms:
        fn()
    per = []
    for name, fn in arms:
        wall, ev = kernels(fn)
        per.append(describe(name, wall, ev, out))
    print("# mean kernel duration (a) / (b), kernels with the most time in (b):", file=out)
    for nm, (c, d) in sorted(per[1].items(), key=lambda kv: -kv[1][1])[:8]:
        if nm in per[0]:
            ca, da = per[0][nm]
            print("    %-28s %.2f" % (nm, (da / ca) / (d / c)), file=out)


if __name__ == "__main__":
    main()
