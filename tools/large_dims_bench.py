"""Sweep and back-solve times around and above the former 8192 limit of the factored dimension N.

    python tools/large_dims_bench.py [--sweeps 3] [--profiles 3] [--points all|quick]

For each point (V, n, chains), all in the n-form (AUTO would pick the q-form at these shapes):
  * sweep_ms: event-timed graph sweeps (bnr_last_run_ms / sweeps) after two warm-up sweeps;
  * solve_ms, chol_ms: the back solve and the Cholesky of bnr_profile_sweep (eager sweeps, median of --profiles);
  * solve_GBps: the factor bytes the back solve reads (T(T+1)/2 blocks of 128 x 128 doubles per chain, the diagonal
    ones as their inverses) over solve_ms.
n = 8191 (N = 8192) runs the one-CTA back solve (k_bwd_stream), n = 8192 (N = 8320) the cluster back solve
(k_bwd_cluster) on almost the same factor, so the two show the gain per byte.  Prints one JSON line, with the card's
name, power limit and maximum SM clock read in the same run.  Writes nothing."""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from __graft_entry__ import load_package  # noqa: E402

POINTS = [(50, 8191, 1), (50, 8192, 1), (50, 16383, 1), (50, 8191, 4), (50, 8192, 4), (50, 16383, 4), (12, 32767, 1)]
QUICK = [(50, 8191, 1), (50, 8192, 1)]


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power, clock = [s.strip() for s in out.split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def factor_bytes(N):
    T = N // 128
    return T * (T + 1) // 2 * 128 * 128 * 8


def run_point(bnr, V, n, C, sweeps, profiles):
    q = V * (V + 1) // 2
    rng = np.random.default_rng(V * 100003 + n)
    X = (rng.random((n, q)) < 0.3) * (0.13 + rng.gamma(1.2, 0.2, size=(n, q)))
    y = 3.0 + X[:, :5].sum(axis=1) + rng.normal(size=n)
    N = -(-(n + 1) // 128) * 128
    with bnr.Engine(X, y, 3, num_chains=C, seed=1, gamma_mode="nform") as eng:
        assert eng.gamma_mode == "nform"
        eng.init_state()
        eng.run(2)
        eng.run(sweeps)
        sweep_ms = eng.last_run_ms() / sweeps
        prof = [eng.profile_sweep() for _ in range(profiles)]
        status = int(np.bitwise_or.reduce(eng.status()))
    solve_ms = statistics.median(p["solves"] for p in prof)
    chol_ms = statistics.median(p["cholesky"] for p in prof)
    return dict(V=V, n=n, N=N, chains=C, back_solve="k_bwd_stream" if N <= 8192 else "k_bwd_cluster",
                sweep_ms=round(sweep_ms, 3), chol_ms=round(chol_ms, 3), solve_ms=round(solve_ms, 4),
                factor_GB_per_chain=round(factor_bytes(N) / 1e9, 4),
                solve_GBps=round(C * factor_bytes(N) / (solve_ms * 1e-3) / 1e9, 1), status_or=status)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--sweeps", type=int, default=3)
    ap.add_argument("--profiles", type=int, default=3)
    ap.add_argument("--points", choices=("all", "quick"), default="all")
    a = ap.parse_args()
    bnr = load_package()
    info = card()
    rows = [run_point(bnr, V, n, C, a.sweeps, a.profiles) for V, n, C in (POINTS if a.points == "all" else QUICK)]
    print(json.dumps(dict(tool="large_dims_bench", card=info, gamma_mode="nform", sweeps=a.sweeps,
                          profiles=a.profiles, points=rows)))


if __name__ == "__main__":
    main()
