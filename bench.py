#!/usr/bin/env python
"""Benchmark of the Gibbs hot path (BASELINE.json metric: Gibbs iterations/s summed over all chains; gamma ESS/s).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine (libbnr.so through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host CPU cores

A "step" is one Gibbs sweep (all ten full conditionals) of EVERY chain held by a GPU.  Workload at any N:
BASELINE config 3 -- synthetic networks with V=100 nodes (q = V(V+1)/2 = 5050 edge coefficients, the reference's
HEAD convention), n=1000 samples, R=7, 64 chains per GPU (weak scaling: N GPUs advance 64*N independent chains,
global chain ids key the RNG; the only exchange is an NCCL all-gather of split-half moments for R-hat).
Inputs are larger than L2 by construction (the per-sweep working set is 64 x 8 MB Gram matrices = 512 MB >> 126 MB),
so no explicit L2 flush is needed between timed iterations.

Legs of the default run (every number in the JSON line is measured in this run unless its key says otherwise):
  value          K timed sweeps, inputs resident in HBM, CUDA events on the handle's stream, max over ranks
  roofline       the dominant kernel (Gram SYRK) timed alone with CUDA events; FP64 peak = cuBLAS DGEMM in this run
  e2e            Fit(X, y, R; ...) + Summary through the public API with HOST buffers (H2D / D2H inside the timed region)
  strong_scaling BASELINE config 3 as written: 64 chains IN TOTAL split over the N GPUs (= value at N = 1)
  gamma_ess_per_sec  a separate leg: burn-in sweeps, then retained draws of every chain, device-side multi-chain Geyer
                 ESS of every gamma_j, divided by the device time of burn-in + draws
  other_configs  BASELINE configs 2, 4, 5 on one GPU (N = 1 only): ms/sweep, chain-iterations/s, roofline fraction
  cpu_baseline   the reference's algorithm (NumPy/OpenBLAS port, Julia is absent) on the host cores (N = 1 only)

--dump-outputs DIR writes what the K timed sweeps computed as DIR/<name>.npy.  Inputs and seeds are fixed, so two builds
run with the same arguments can be compared output for output.
"""
import os
import sys

if "--impl" in sys.argv and "reference" in sys.argv:
    # the CPU arm runs one single-threaded chain per process (src/gibbs.jl:946-948): pin every BLAS / OpenMP pool
    # BEFORE NumPy is imported (the timing itself additionally runs in a child interpreter, oracle/cpu_baseline.py)
    for _v in ("OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "OMP_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_v] = "1"

import argparse
import json
import math
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # bench.py writes nothing into the tree: no __pycache__ for what it imports from it

CONFIGS = {
    # name: V, n, R, chains per GPU
    "c2": dict(V=30, n=500, R=7, chains=16),
    "c3": dict(V=100, n=1000, R=7, chains=64),
    "c4": dict(V=200, n=400, R=9, chains=8),
    "c5": dict(V=50, n=500, R=5, chains=128),
}
CFG_ID = {"c2": 2, "c3": 3, "c4": 4, "c5": 5}


def synth(cfg_name, dense=False):
    """SURVEY 8(d) generator: sparse weighted networks with a low-rank-ish truth; seeded, identical on every rank."""
    cfg = CONFIGS[cfg_name]
    V, n = cfg["V"], cfg["n"]
    rng = np.random.Generator(np.random.Philox(key=20241000 + CFG_ID[cfg_name]))
    q = V * (V + 1) // 2
    xi_true = rng.random(V) < 2.0 / 3.0
    il, ik = np.tril_indices(V)
    # column-major lower triangle incl. diagonal: column k, rows l = k..V-1
    order = np.lexsort((il, ik))
    il, ik = il[order], ik[order]
    B = np.where(xi_true[il] & xi_true[ik] & (il != ik), rng.normal(1.5, 0.9, size=q), 0.0)
    if dense:
        X = rng.normal(size=(n, q))
    else:
        present = rng.random((n, V)) < 0.73
        both = present[:, il] & present[:, ik] & (il != ik)[None, :]
        on = rng.random((n, q)) < 0.9
        X = np.where(both & on, 0.13 + rng.gamma(1.2, 0.2, size=(n, q)), 0.0)
    y = 55.0 + X @ B + rng.normal(0.0, 10.0, size=n)
    return np.asfortranarray(X), y, dict(V=V, n=n, q=q, R=cfg["R"])


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of one GPU, sampled through NVML every `period` seconds (falls back to the
    B200_PROFILING.md nvidia-smi query when NVML cannot be loaded).  `mark()` / `unmark()` bracket the timed region so
    that the record says how many samples fell INSIDE it."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index, uuid=None, period=0.01):
        super().__init__(daemon=True)
        self.index, self.uuid, self.period = index, uuid, period
        self.rows, self._stop_evt, self._in = [], threading.Event(), False
        self.nv = self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                for cand in (uuid, "GPU-" + uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand if isinstance(cand, bytes) else cand.encode())
                        break
                    except Exception:
                        try:
                            h = pynvml.nvmlDeviceGetHandleByUUID(cand)
                            break
                        except Exception:
                            h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.nv, self.h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def mark(self):
        self._in = True

    def unmark(self):
        self._in = False

    def _reasons(self):
        nv = self.nv
        for fn in ("nvmlDeviceGetCurrentClocksEventReasons", "nvmlDeviceGetCurrentClocksThrottleReasons"):
            if hasattr(nv, fn):
                try:
                    return int(getattr(nv, fn)(self.h))
                except Exception:
                    continue
        return 0

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nv is not None:
                    sm = float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    mask = self._reasons()
                    self.rows.append((sm, self.max_mhz, [n for n, b in self.BITS if mask & b], self._in))
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    r = [t.strip() for t in out.strip().split(",")]
                    names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
                    self.rows.append((float(r[0]), float(r[1]),
                                      [n for n, v in zip(names, r[3:7]) if v.lower().startswith("active")], self._in))
            except Exception:
                pass
            self._stop_evt.wait(self.period if self.nv is not None else 0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        inside = [r for r in self.rows if r[3]]
        use = inside if len(inside) >= 5 else self.rows
        sm = [r[0] for r in use]
        reasons = sorted({n for r in use for n in r[2]})
        return dict(sm_mhz=float(np.median(sm)) if sm else None,
                    sm_min_mhz=float(np.min(sm)) if sm else None,
                    sm_max_mhz=max([r[1] for r in self.rows], default=None), reasons=reasons,
                    samples=len(use), samples_in_timed_region=len(inside),
                    window="timed region" if use is inside else "warm-up + timed region (timed region too short for 5 samples)",
                    source="nvml" if self.nv is not None else "nvidia-smi")


def fp64_peak_tflops(torch, dev):
    """Measured FP64 GEMM rate (cuBLAS DGEMM through torch.matmul, best of 5 at 4096^3 and 8192x8192x4096):
    the roofline denominator for the DMMA kernels; MEASURED_PEAKS.json only holds HBM and bf16 numbers."""
    best = 0.0
    for (m, n, k) in ((4096, 4096, 4096), (8192, 8192, 4096)):
        a = torch.randn(m, k, dtype=torch.float64, device=dev)
        b = torch.randn(k, n, dtype=torch.float64, device=dev)
        for _ in range(2):
            (a @ b)
        torch.cuda.synchronize(dev)
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); c = a @ b; e1.record(); torch.cuda.synchronize(dev)
            best = max(best, 2.0 * m * n * k / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        del a, b, c
    torch.cuda.empty_cache()
    return best


def cpu_port_sample(X, y, R, chains, sweeps, warm):
    """The reference's algorithm on the host cores: one single-threaded chain per process, min(chains, cores) of them
    at once (oracle/cpu_baseline.py).  Returns the cpu_baseline object and the raw timing record."""
    from oracle import cpu_baseline as B
    r = B.time_port(np.ascontiguousarray(X), y, R, chains, sweeps, warm=warm)
    cpu = {"value": r["value"], "unit": "chain-iterations/s", "cores": r["nproc"], "kind": "port",
           "threads_per_proc": r["threads_per_proc"], "chains": r["nproc"], "sweeps": r["sweeps"],
           "per_core": r["value"] / r["nproc"], "timed_s": r["timed_s"],
           "sample": "%d chains x %d sweeps (+%d warm-up) of the same workload, one single-threaded chain per process "
                     "(BLAS pools pinned to 1 thread before NumPy loads, asserted in every worker), barrier-timed %.1f s; "
                     "NumPy/OpenBLAS port of gibbs_sample!'s dense formulation (Julia is absent)"
                     % (r["nproc"], r["sweeps"], r["warm"], r["timed_s"])}
    return cpu, r


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU path (port) on all host cores, same config / metric / unit.
    One step = one sweep of the min(64, cores) chains that run concurrently (the bounded sample of the 64-chain
    workload); exactly `steps` timed sweeps (main() refuses more than --ref-max-sweeps) are run and reported, after
    min(warmup, 3), at least 1, untimed ones."""
    if rank != 0:
        return
    X, y, dims = synth(args.config, args.dense)
    chains = CONFIGS[args.config]["chains"]
    sweeps = args.steps
    warm = max(1, min(args.warmup, 3))
    cpu, r = cpu_port_sample(X, y, dims["R"], chains, sweeps, warm)
    val = cpu["value"]
    line = {
        "impl": "reference", "metric": "gibbs_iters_per_sec_all_chains", "value": val, "unit": "chain-iterations/s",
        "n_gpus": args.gpus, "steps": sweeps, "warmup": warm, "ms_per_step": 1e3 * r["timed_s"] / sweeps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, dims, chains),
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": "chain-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": r["wall_s"],
    }
    print(json.dumps(line), flush=True)


def _finite(o):
    """JSON has no NaN / Infinity: non-finite floats become null."""
    if isinstance(o, float):
        return o if math.isfinite(o) else None
    if isinstance(o, dict):
        return {k: _finite(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_finite(v) for v in o]
    return o


def workload_config(args, dims, chains):
    return {"workload": "BASELINE config 3-style synthetic network regression" if args.config == "c3" else args.config,
            "name": args.config, "V": dims["V"], "q": dims["q"], "n": dims["n"], "R": dims["R"],
            "chains_per_gpu": chains, "q_convention": "V(V+1)/2 (reference HEAD, diagonal included)",
            "X": "dense N(0,1)" if args.dense else "sparse weighted networks (SURVEY 8d)",
            "l2": "inputs larger than L2 (per-sweep working set %d MB)" % (chains * (math.ceil(dims["n"] / 128) * 128) ** 2 * 8 // 2 ** 20),
            "parallelism": "chains sharded over GPUs, %d per GPU" % chains}


def algo_flops(n, q):
    """SURVEY 8(d): min of the n-form (n^2 q + n^3/3 + 2 n^2 + 10 n q) and the q-form (q^3/3 + 4 q^2 + 6 n q)."""
    return min(n * n * q + n ** 3 / 3.0 + 2.0 * n * n + 10.0 * n * q, q ** 3 / 3.0 + 4.0 * q * q + 6.0 * n * q)


def dominant_kernel(eng, phases, n, q, chains):
    """(name, ms per launch, algorithmic flops per launch) of the kernel that bounds the sweep."""
    if eng.gamma_mode == "nform":
        # G = X D X' + I.  SURVEY 8(d): n^2 q flops per chain-iteration (lower half, mul + add)
        return ("k_gram_syrk (X diag(S) X' + I, DMMA m8n8k4, TMA ring)", phases["syrk"], chains * float(n) * n * q)
    # q-form: the batched blocked Cholesky of the q x q precision dominates; q^3/3 flops per chain-iteration
    return ("blocked Cholesky of P = (X'X + D^-1)/tau2 (k_chol_panel + k_chol_update)", phases["cholesky"],
            chains * float(q) ** 3 / 3.0)


def time_sweeps(eng, K):
    """K sweeps timed with CUDA events on the handle's stream (bnr_last_run_ms)."""
    eng.run(K, sync=True)
    return eng.last_run_ms()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, eng, var_names, rank, world, chain_offset, rx, rg, status):
    """--dump-outputs: what the timed sweeps hand to a caller -- every chain's state after the last sweep (Engine.get_state,
    stacked over chains), the per-chain status bits and the split R-hat of the timed draws -- as float64 <name>.npy.
    Beyond DUMP_BYTES in all, a fixed seeded sample of the chains is written; chain_ids.npy names the global chains kept.
    With several ranks every rank writes its own chains under <name>_rank<r>.npy."""
    per_chain = 8 * (2 + sum(int(np.prod(eng.var_shape(k))) for k in var_names))    # + status and chain id
    room = DUMP_BYTES // world - 8 * (rx.size + rg.size) - (1 << 16)                  # 64 KB for the .npy headers
    keep = max(1, min(eng.C, room // per_chain))
    chains = np.arange(eng.C)
    if keep < eng.C:
        chains = np.sort(np.random.default_rng(0).choice(eng.C, keep, replace=False))
    out = {"chain_ids": chain_offset + chains, "status": status[chains], "rhat_xi": rx, "rhat_gamma": rg}
    for k in var_names:
        out[k] = np.stack([eng.get_state(int(c), k) for c in chains])
    os.makedirs(out_dir, exist_ok=True)
    suffix = "_rank%d" % rank if world > 1 else ""
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + suffix + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (default: the config's)")
    ap.add_argument("--total-chains", type=int, default=0,
                    help="strong scaling as the headline: this many chains in total, split evenly over the GPUs; default "
                         "is weak scaling with the config's chains per GPU (the strong-scaling figure of BASELINE config 3, "
                         "64 chains in total, is always reported beside it in `strong_scaling`)")
    ap.add_argument("--chain-groups", type=int, default=0, help="independent stream/graph groups per GPU (0 = library default)")
    ap.add_argument("--gamma-mode", default="auto", choices=["auto", "nform", "qform"])
    ap.add_argument("--dense", action="store_true", help="dense Gaussian X instead of sparse networks")
    ap.add_argument("--ref-max-sweeps", type=int, default=200, help="reference arm: largest --steps it accepts")
    ap.add_argument("--cpu-sweeps", type=int, default=10, help="cpu_baseline leg of our arm: timed sweeps per chain")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-sweeps", type=int, default=5)
    ap.add_argument("--ess-burn", type=int, default=1000, help="ESS leg: burn-in sweeps (0 with --ess-draws 0 skips the leg)")
    ap.add_argument("--ess-draws", type=int, default=1000, help="ESS leg: retained draws per chain")
    ap.add_argument("--ess-max-lag", type=int, default=255)
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the timed sweeps computed (chain states after the last one, status, R-hat) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference" and args.steps > args.ref_max_sweeps:
        ap.error("--impl reference times exactly --steps sweeps: %d is above --ref-max-sweeps %d"
                 % (args.steps, args.ref_max_sweeps))

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from __graft_entry__ import load_package
    bnr = load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))

    X, y, dims = synth(args.config, args.dense)
    chains = args.chains or CONFIGS[args.config]["chains"]
    scaling = "weak"
    if args.total_chains:
        if args.total_chains % world:
            raise SystemExit("--total-chains must be a multiple of the GPU count")
        chains, scaling = args.total_chains // world, "strong"
    V, q, n, R = dims["V"], dims["q"], dims["n"], dims["R"]
    K, Wm = args.steps, max(args.warmup, 3)

    peak = fp64_peak_tflops(torch, dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather_stats(eng, nrows, lag):
        """ESS of (xi, gamma) over the chains of all ranks from this rank's accumulated statistics."""
        (pa, na), (pm, nm), lag = eng.ess_device()
        if world == 1:
            return eng.ess_from_stats(pa, 1, pm, eng.C, nrows, lag, with_lags=True)
        a_mine = torch.empty(na, dtype=torch.float64, device=dev)
        m_mine = torch.empty(nm, dtype=torch.float64, device=dev)
        eng.export_ess(a_mine.data_ptr(), m_mine.data_ptr())
        a_all = torch.empty(na * world, dtype=torch.float64, device=dev)
        m_all = torch.empty(nm * world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(a_all, a_mine)
        dist.all_gather_into_tensor(m_all, m_mine)
        torch.cuda.synchronize(dev)
        return eng.ess_from_stats(a_all.data_ptr(), world, m_all.data_ptr(), eng.C * world, nrows, lag, with_lags=True)

    # ---------------- device-resident timing: `value` ----------------
    try:
        uuid = str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local_rank, uuid)
    sampler.start()
    eng = bnr.Engine(X, y, R, num_chains=chains, seed=20241018, chain_offset=rank * chains, device=local_rank,
                     trace_rows=0, chain_groups=args.chain_groups, gamma_mode=args.gamma_mode)
    eng.init_state()
    eng.run(Wm)
    eng.set_moment_window(Wm + 1, K)
    launches0 = eng.launch_count()
    iter0 = eng.iteration
    barrier()
    sampler.mark()
    t0 = time.perf_counter()
    eng.run(K, sync=True)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    sampler.unmark()
    dev_ms = eng.last_run_ms()
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    assert eng.iteration - iter0 == K, "the timed run advanced %d sweeps, not --steps %d" % (eng.iteration - iter0, K)
    total_ms = max_over_ranks(dev_ms)          # collective: every rank calls it exactly once, here
    step_ms = total_ms / K
    value = world * chains * K / (total_ms * 1e-3)

    # R-hat over all chains of all ranks: NCCL all-gather of split-half moments, reduced identically on every rank
    if K // 2 < 2:
        rx, rg = np.full(V, np.nan), np.full(q, np.nan)        # too few timed draws for a split R-hat
    elif world > 1:
        ptr, cnt = eng.moments_device()
        mine = torch.empty(cnt, dtype=torch.float64, device=dev)
        eng.export_moments(mine.data_ptr())
        allm = torch.empty(cnt * world, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allm, mine)
        torch.cuda.synchronize(dev)
        rx, rg = eng.rhat_from_moments(allm.data_ptr(), chains * world, K // 2)
    else:
        rx, rg = eng.rhat()
    status = eng.status()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, bnr.VAR, rank, world, rank * chains, rx, rg, status)

    # ---------------- per-phase CUDA-event profile of eager sweeps (roofline numerator) ----------------
    phases = {}
    for _ in range(max(1, args.profile_sweeps)):
        for k, v in eng.profile_sweep().items():
            phases.setdefault(k, []).append(v)
    phases = {k: float(np.mean(v)) for k, v in phases.items()}
    gmode = eng.gamma_mode
    chain_groups = eng.chain_groups
    dom_kernel, dom_ms, dom_flops = dominant_kernel(eng, phases, n, q, chains)
    achieved = dom_flops / (dom_ms * 1e-3) / 1e12
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "syrk_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(args.config)
        except Exception:
            traffic = None
    eng.close()

    # ---------------- end to end through the public API with HOST buffers: `e2e` ----------------
    # The call a user makes: Fit(X, y, R; nburn, nsamples, num_chains, seed) -> Results, then Summary(Results).
    # Inside the timed region: handle creation, H2D of X and y, prior init, K sweeps of every chain, streamed R-hat,
    # Summary reduced on the device, D2H of chain 1's gamma / xi table, the R-hat vectors and the Summary statistics.
    nsamp_e = min(max(2, K // 2), K)
    nburn_e = K + 1 - nsamp_e                      # nburn + nsamples rows = prior row + K sweeps
    # one untimed Fit first: the steady state of the API is what is measured, not the first call's lazy loading of the
    # Fit-only kernels (Summary select, R-hat), across ranks NCCL's first all-gather, and the device allocator (a Fit of
    # the same shape leaves every buffer of the timed one in libbnr's cache; a cudaMalloc of a new size was seen to take
    # anything from 0.1 to 30 ms).  Same shape up to 256 sweeps, an 8-sweep one beyond.
    wb, wn = (nburn_e, nsamp_e) if K <= 256 else (5, 4)
    bnr.Fit(X, y, R, nburn=wb, nsamples=wn, num_chains=chains, seed=7, x_transform=False, filename=None,
            psrf_cutoff=float("inf"), device=local_rank, return_state="gamma_xi")
    barrier()
    t0 = time.perf_counter()
    res = bnr.Fit(X, y, R, nburn=nburn_e, nsamples=nsamp_e, num_chains=chains, seed=7, x_transform=False,
                  filename=None, psrf_cutoff=float("inf"), device=local_rank, return_state="gamma_xi")
    summ = bnr.Summary(res) if nsamp_e >= 40 else None     # the reference's Summary needs >= 20 draws per tail index
    torch.cuda.synchronize(dev)
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_val = world * chains * K / e2e_s
    h2d = (X.nbytes + y.nbytes) / K
    d2h = (res.state["gamma"].nbytes + res.state["xi"].nbytes + 8 * (V + q) + 8 * (3 * q + V)) / K
    assert (summ is None or len(summ.edge_coef["estimate"]) == q) and res.extra["tot_generated"] == K + 1

    # ---------------- strong scaling: BASELINE config 3 as written, 64 chains IN TOTAL over the N GPUs ----------------
    strong = None
    total64 = CONFIGS[args.config]["chains"]
    if not args.no_strong and not args.total_chains and total64 % world == 0:
        cs = total64 // world
        if world == 1 and cs == chains:
            strong = {"total_chains": total64, "chains_per_gpu": cs, "value": value, "ms_per_step": step_ms,
                      "chain_groups": chain_groups, "note": "identical to the headline run at N = 1"}
        else:
            e2 = bnr.Engine(X, y, R, num_chains=cs, seed=20241018, chain_offset=rank * cs, device=local_rank,
                            trace_rows=0, chain_groups=args.chain_groups, gamma_mode=args.gamma_mode)
            e2.init_state()
            e2.run(Wm)
            barrier()
            ms2 = max_over_ranks(time_sweeps(e2, K))
            strong = {"total_chains": total64, "chains_per_gpu": cs, "value": total64 * K / (ms2 * 1e-3),
                      "ms_per_step": ms2 / K, "chain_groups": e2.chain_groups}
            e2.close()

    # ---------------- gamma ESS/s: burn-in, then retained draws of every chain, Geyer ESS on the device ----------------
    ess = None
    if args.ess_draws >= 8:
        Bn, Dn = max(0, args.ess_burn), args.ess_draws
        e3 = bnr.Engine(X, y, R, num_chains=chains, seed=20241019, chain_offset=rank * chains, device=local_rank,
                        trace_rows=0, chain_groups=args.chain_groups, gamma_mode=args.gamma_mode)
        e3.init_state()
        barrier()
        ms_burn = time_sweeps(e3, Bn) if Bn else 0.0
        e3.ess_stream_begin(args.ess_max_lag, Dn)
        ms_draw = time_sweeps(e3, Dn)
        e3.ess_stream_finish()
        ess_ms = max_over_ranks(ms_burn + ms_draw)
        ex, eg, lag_x, lag_g = gather_stats(e3, Dn, args.ess_max_lag)
        lag = e3.ess_device()[2]
        e3.close()
        fin = np.isfinite(eg)
        ess = {"median": float(np.nanmedian(eg)) / (ess_ms * 1e-3) if fin.any() else None,
               "min": float(np.nanmin(eg)) / (ess_ms * 1e-3) if fin.any() else None,
               "mean": float(np.nanmean(eg)) / (ess_ms * 1e-3) if fin.any() else None,
               "unit": "effective gamma draws per second (per edge coefficient; pooled over all chains)",
               "ess_median": float(np.nanmedian(eg)) if fin.any() else None,
               "ess_min": float(np.nanmin(eg)) if fin.any() else None,
               "edges": int(q), "burn_in": Bn, "draws_per_chain": Dn, "chains": chains * world, "max_lag": int(lag),
               "geyer_terminated_frac": float(np.mean(lag_g <= lag - 1)),
               "seconds": ess_ms * 1e-3, "iters_per_sec_in_leg": world * chains * (Bn + Dn) / (ess_ms * 1e-3),
               "estimator": "multi-chain Geyer initial monotone sequence on per-chain-centred autocovariances "
                            "(streamed lagged products, no all-chain trace), seconds = device time of burn-in + draws"}

    # ---------------- the other BASELINE configs on one GPU ----------------
    others = None
    if rank == 0 and world == 1 and not args.no_other_configs and args.config == "c3":
        others = {}
        for name in ("c2", "c4", "c5"):
            Xo, yo, do = synth(name)
            co = CONFIGS[name]["chains"]
            eo = bnr.Engine(Xo, yo, do["R"], num_chains=co, seed=20241018, device=local_rank, trace_rows=0)
            eo.init_state()
            eo.run(10)
            l0 = eo.launch_count()
            Ko = 200
            ms = time_sweeps(eo, Ko)
            lo = eo.launch_count() - l0
            ph = {}
            for _ in range(3):
                for k, v in eo.profile_sweep().items():
                    ph.setdefault(k, []).append(v)
            ph = {k: float(np.mean(v)) for k, v in ph.items()}
            dk, dms, dfl = dominant_kernel(eo, ph, do["n"], do["q"], co)
            its = co * Ko / (ms * 1e-3)
            others[name] = {"V": do["V"], "q": do["q"], "n": do["n"], "R": do["R"], "chains": co,
                            "ms_per_sweep": ms / Ko, "value": its, "unit": "chain-iterations/s",
                            "gamma_mode": eo.gamma_mode, "chain_groups": eo.chain_groups,
                            "launches_per_sweep": lo / Ko,
                            "algorithmic_tflops": its * algo_flops(do["n"], do["q"]) / 1e12,
                            "frac_of_fp64_peak_whole_sweep": its * algo_flops(do["n"], do["q"]) / 1e12 / peak,
                            "dominant_kernel": dk, "dominant_ms": dms,
                            "dominant_frac_of_peak": dfl / (dms * 1e-3) / 1e12 / peak,
                            "phases_ms": ph, "status_or": int(np.bitwise_or.reduce(eo.status()))}
            eo.close()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _ = cpu_port_sample(X, y, R, chains, max(2, args.cpu_sweeps), 2)

    if rank == 0:
        af = algo_flops(n, q)
        line = {
            "metric": "gibbs_iters_per_sec_all_chains", "value": value, "unit": "chain-iterations/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, dims, chains),
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "chain-iterations/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "includes": "Fit(X, y, R; ...) + Summary through the public API (one bnr_fit call): handle creation "
                    "(device buffers come from libbnr's cache, warmed by one untimed Fit of the same shape), H2D of X,y from host memory, "
                    "graph capture, prior init, K sweeps, streamed R-hat (NCCL all-gather of the moments across ranks), "
                    "device Summary, D2H of chain-1 gamma/xi table, handle teardown"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": dom_kernel,
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": "offline: dram__bytes_read.sum + dram__bytes_write.sum of one launch from the ncu "
                                           "--set full capture committed under profiles/ (not measured in this run)",
                         "ms_per_launch": dom_ms, "flops_per_launch": dom_flops,
                         "peak_source": "cuBLAS DGEMM measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                         "peak_theoretical": 128 * 148 * 1.965e9 / 1e12,
                         "frac_of_theoretical": achieved / (128 * 148 * 1.965e9 / 1e12),
                         "whole_sweep_frac": value / world * af / 1e12 / peak,
                         "note": "theoretical = 128 FP64 flop/clk/SM (DMMA and DFMA alike) x 148 SMs x 1.965 GHz; "
                                 "whole_sweep_frac = algorithmic flops of the whole sweep / step time / peak"},
            "cpu_baseline": cpu,
            "gamma_ess_per_sec": ess,
            "strong_scaling": strong,
            "other_configs": others,
            "gamma_mode": gmode,
            "chain_groups": chain_groups,
            "algorithmic_tflops": value * af / 1e12,
            "phases_ms": phases,
            "wall_ms_per_step": wall_ms / K,
            "rhat": {"max_gamma": float(np.nanmax(rg)) if np.isfinite(rg).any() else None, "max_xi": float(np.nanmax(rx[np.isfinite(rx)])) if np.isfinite(rx).any() else None,
                     "chains": chains * world},
            "status_or": int(np.bitwise_or.reduce(status)),
        }
        print(json.dumps(_finite(line)), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
