"""Host side of `Fit!` / `Summary` (src/gibbs.jl:725-751, 897-1020, 1051-1198, 1214-1250).

Only argument handling lives here: keyword names, parameters.log, X vectorisation (setup_X!), wrapping the returned
buffers as Results and the Summary tables.  The chain generation -- every Gibbs iteration, the row bookkeeping of run!
(purge_burn ring), both PSRF-driven control loops, the R-hat reduction and the Summary statistics -- is ONE call into
libbnr (bnr_fit, csrc/bnr_fit.cu), so a Julia `ccall` wrapper is equally thin (julia/BNRB200.jl).
"""
import ctypes as C
import datetime
import math
import random
import warnings

import numpy as np

from .capi import lib, check, check_fit, FitParams, FitInfo, ALLGATHER_FN, STATE, VAR, GAMMA_MODE, PRED_MEAN, \
    PRED_PREDICTIVE
from .engine import LOO_FIELDS

_DP = C.POINTER(C.c_double)

_UNI = {"tau2": "τ²", "u": "u", "xi": "ξ", "gamma": "γ", "S": "S", "theta": "θ", "Delta": "Δ", "M": "M",
        "mu": "μ", "lam": "λ", "pi": "πᵥ"}
_ASCII = {v: k for k, v in _UNI.items()}
_ASCII.update({"lambda": "lam", "pi_v": "pi", "tau²": "tau2"})


class Table(dict):
    """Column container standing in for TypedTables.Table: columns by reference name (state["γ"], state.γ)
    or ASCII alias (state.gamma); each column is a Fortran-ordered (rows, d1, d2) Float64 array."""

    def _key(self, name):
        return _ASCII.get(name, name)

    def __getitem__(self, name):
        return dict.__getitem__(self, self._key(name))

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError:
            raise AttributeError(name)

    def __len__(self):
        for v in self.values():
            return v.shape[0]
        return 0


class Results:
    """src/gibbs.jl:23-29: state table of the first chain, PSRF tables, burn_in, sampled."""

    def __init__(self, state, rhat_xi, rhat_gamma, burn_in, sampled, extra=None):
        self.state = state
        self.rhatξ = Table(xi=np.asarray(rhat_xi))
        self.rhatγ = Table(gamma=np.asarray(rhat_gamma))
        self.burn_in = int(burn_in)
        self.sampled = int(sampled)
        self.extra = extra or {}

    rhat_xi = property(lambda self: self.rhatξ)
    rhat_gamma = property(lambda self: self.rhatγ)

    def __repr__(self):
        return repr(Summary(self))


class BNRSummary:
    """src/gibbs.jl:39-43.  edge_coef / prob_nodes are dicts of columns (DataFrame stand-ins)."""

    def __init__(self, edge_coef, prob_nodes, ci_level):
        self.edge_coef = edge_coef
        self.prob_nodes = prob_nodes
        self.ci_level = ci_level

    def __repr__(self):
        e = self.edge_coef
        lines = ["", "Edge Coefficient Estimates (%d%% credible intervals)" % self.ci_level,
                 " node1 node2  estimate  lower_bound  upper_bound"]
        n = len(e["node1"])
        show = list(range(n)) if n <= 20 else list(range(10)) + [None] + list(range(n - 10, n))
        for i in show:
            if i is None:
                lines.append("   ...")
            else:
                lines.append(" %5d %5d  %8.3f  %11.3f  %11.3f" % (e["node1"][i], e["node2"][i], e["estimate"][i],
                                                                e["lower_bound"][i], e["upper_bound"][i]))
        lines.append("Node Probabilities")
        lines.extend(" %4d  %.3f" % (i + 1, p) for i, p in enumerate(self.prob_nodes["probability"]))
        return "\n".join(lines)


class BNRPrediction:
    """Predict's table: per new network (1-based `sample`) the posterior mean of the prediction and the order-statistic
    bounds of its interval (a dict of columns, like BNRSummary.edge_coef)."""

    def __init__(self, table, ci_level, predictive):
        self.table = table
        self.ci_level = ci_level
        self.predictive = predictive

    def __repr__(self):
        t = self.table
        kind = "posterior predictive" if self.predictive else "credible"
        lines = ["", "Predicted Responses (%d%% %s intervals)" % (self.ci_level, kind),
                 " sample  estimate  lower_bound  upper_bound"]
        n = len(t["sample"])
        show = list(range(n)) if n <= 20 else list(range(10)) + [None] + list(range(n - 10, n))
        for i in show:
            if i is None:
                lines.append("   ...")
            else:
                lines.append(" %6d  %8.3f  %11.3f  %11.3f" % (t["sample"][i], t["estimate"][i], t["lower_bound"][i],
                                                             t["upper_bound"][i]))
        return "\n".join(lines)


# -- index maps (src/utils.jl:17-57) -------------------------------------------------------------------
def lower_triangle(matrix):
    m = np.asarray(matrix)
    if m.ndim != 2 or m.shape[0] != m.shape[1]:
        raise ValueError("matrix must be square")
    V = m.shape[0]
    return np.concatenate([m[k:, k] for k in range(V)])


def create_lower_tri(vector, V):
    v = np.asarray(vector)
    mat = np.zeros((V, V), dtype=v.dtype)
    i = 0
    for k in range(V):
        mat[k:, k] = v[i:i + V - k]
        i += V - k
    return mat


def setup_X(X, x_transform=True):
    """setup_X! (src/gibbs.jl:239-247) -> n x q Float64 matrix."""
    if x_transform:
        return np.stack([lower_triangle(np.asarray(x, dtype=np.float64)) for x in X])
    return np.asarray(X, dtype=np.float64)


def _jround(x):
    """Julia round(): half to even."""
    return int(np.rint(x))


def _citation():
    return ("If you use BayesianNetworkRegression.jl, please cite:\n@article{Ozminkowski2022,\n"
            "author = {Ozminkowski, S. and Sol\\'{i}s-Lemus, C.},\nyear = {2022},\n"
            "title = {{Identifying microbial drivers in biological phenotypes with a Bayesian Network Regression model}},\n"
            "journal = {In preparation}\n}")


def _dist_world():
    """(rank, world) of an initialised torch.distributed process group, else (0, 1).  One process per GPU: every rank
    calls Fit with its own share of the chains (the reference spreads chains over Distributed.jl workers,
    src/gibbs.jl:946-948)."""
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    return 0, 1


def _torch_allgather(ctx, device, send, recv, count):
    """bnr_allgather_fn for a torch.distributed job: the per-rank moments ([chain][half][param][mean, M2], 32 (V+q)
    bytes per chain -- the only data that crosses NVLink) are all-gathered over NCCL (or on the host with gloo, for the
    CPU-side rendezvous of the tests); every rank then reduces them in the same order inside libbnr."""
    try:
        import torch
        import torch.distributed as dist
        L = lib()
        dev = torch.device("cuda", device)
        world = dist.get_world_size()
        mine = torch.empty(count, dtype=torch.float64, device=dev)
        check(L.bnr_device_copy(device, C.c_void_p(mine.data_ptr()), C.c_void_p(send), count * 8))
        if dist.get_backend() == "nccl":
            allm = torch.empty(count * world, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(allm, mine)
        else:
            host = torch.empty(count * world, dtype=torch.float64)
            dist.all_gather_into_tensor(host, mine.cpu())
            allm = host.to(dev)
        torch.cuda.synchronize(dev)
        check(L.bnr_device_copy(device, C.c_void_p(recv), C.c_void_p(allm.data_ptr()), count * world * 8))
        return 0
    except Exception:                                   # an exception must not unwind through the C frames
        import traceback
        traceback.print_exc()
        return 1


_ALLGATHER = ALLGATHER_FN(_torch_allgather)


def _native_fit(Xn, y, R, *, eta, zeta, iota, a_delta, b_delta, nu, nburn=0, nsamp=0, mingen=0, maxgen=0,
                psrf_cutoff=1.01, purge_burn=None, num_chains=2, seed=0, device=0, return_state="full", verbose=False,
                chain_offset=0, n_devices=1, ess_max_lag=0, interval=95, gamma_mode="auto", chain_groups=0, X_new=None,
                predictive=False, loo=False):
    """One bnr_fit call (include/bnr.h): chain generation, purge ring, PSRF loop, R-hat, Summary statistics on the GPU.
    With X_new (m x q, already vectorised) the call is bnr_fit_predict, which also pools the predictions; with loo=True
    it is bnr_fit_loo, which also scores the fit by PSIS-LOO and WAIC."""
    L = lib()
    Xf = np.asfortranarray(Xn, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    n, q = Xf.shape
    V = int(round((-1 + math.sqrt(1 + 8 * q)) / 2))
    if V * (V + 1) // 2 != q:
        raise ValueError("q = %d is not V(V+1)/2 for an integer V" % q)
    p = FitParams()
    L.bnr_fit_default_params(C.byref(p))
    b = p.base
    b.n, b.V, b.R, b.num_chains, b.chain_offset, b.device = n, V, int(R), int(num_chains), int(chain_offset), int(device)
    b.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    b.eta, b.zeta, b.iota, b.a_delta, b.b_delta, b.nu = eta, zeta, iota, a_delta, b_delta, float(nu)
    b.gamma_mode = GAMMA_MODE[gamma_mode] if isinstance(gamma_mode, str) else int(gamma_mode)
    b.chain_groups = int(chain_groups)
    p.nburn, p.nsamples, p.mingen, p.maxgen = int(nburn), int(nsamp), int(mingen), int(maxgen)
    p.psrf_cutoff = float(psrf_cutoff)
    p.purge_burn = int(purge_burn) if purge_burn else 0
    p.return_state = STATE[return_state]
    p.n_devices, p.interval, p.ess_max_lag, p.verbose = int(n_devices), int(interval), int(ess_max_lag), 1 if verbose else 0
    rank, world = _dist_world()
    if world > 1:
        p.ext_world, p.ext_rank, p.allgather = world, rank, _ALLGATHER
    res = C.c_void_p()
    if X_new is not None:
        Xp = np.asfortranarray(X_new, dtype=np.float64)
        if Xp.ndim != 2 or Xp.shape[1] != q:
            raise ValueError("X_new must hold networks like X (%d edge columns after setup_X)" % q)
    if loo:
        m, xp = (0, None) if X_new is None else (Xp.shape[0], Xp.ctypes.data_as(_DP))
        check_fit(L.bnr_fit_loo(C.byref(p), Xf.ctypes.data_as(_DP), y.ctypes.data_as(_DP), m, xp,
                                PRED_PREDICTIVE if predictive else PRED_MEAN, C.byref(res)))
    elif X_new is None:
        check_fit(L.bnr_fit(C.byref(p), Xf.ctypes.data_as(_DP), y.ctypes.data_as(_DP), C.byref(res)))
    else:
        check_fit(L.bnr_fit_predict(C.byref(p), Xf.ctypes.data_as(_DP), y.ctypes.data_as(_DP), Xp.shape[0],
                                    Xp.ctypes.data_as(_DP), PRED_PREDICTIVE if predictive else PRED_MEAN,
                                    C.byref(res)))
    try:
        info = FitInfo()
        check_fit(L.bnr_fit_get_info(res, C.byref(info)))
        rx, rg = np.empty(V), np.empty(q)
        check_fit(L.bnr_fit_rhat(res, rx.ctypes.data_as(_DP), rg.ctypes.data_as(_DP)))
        dev_summary = None
        if info.summary_ok:
            gm, gl, gh, xm = np.empty(q), np.empty(q), np.empty(q), np.empty(V)
            check_fit(L.bnr_fit_summary(res, *(a.ctypes.data_as(_DP) for a in (gm, gl, gh, xm))))
            dev_summary = dict(interval=interval, mean=gm, lower=gl, upper=gh, xi_mean=xm, V=V, q=q)
        ess = None
        if info.ess_ok:
            ex, eg = np.empty(V), np.empty(q)
            check_fit(L.bnr_fit_ess(res, ex.ctypes.data_as(_DP), eg.ctypes.data_as(_DP)))
            ess = dict(xi=ex, gamma=eg, max_lag=ess_max_lag)
        prediction = None
        if X_new is not None:
            m = Xp.shape[0]
            pm, pl, ph = np.empty(m), np.empty(m), np.empty(m)
            rc = L.bnr_fit_prediction(res, *(a.ctypes.data_as(_DP) for a in (pm, pl, ph)))
            if rc == -4:                      # BNR_ESTATE: too few pooled draws for the interval's ranks
                pm = pl = ph = None
            else:
                check_fit(rc)
            prediction = dict(interval=interval, mean=pm, lower=pl, upper=ph, predictive=bool(predictive), m=m,
                              draws=int(info.total_chains) * int(info.sampled))
        loo_out = None
        if loo:
            pw = [np.empty(n) for _ in LOO_FIELDS]
            rc = L.bnr_fit_loo_pointwise(res, *(a.ctypes.data_as(_DP) for a in pw))
            if rc == -4:                      # BNR_ESTATE: fewer than 2 pooled draws
                pw = None
            else:
                check_fit(rc)
            loo_out = dict(pointwise=None if pw is None else dict(zip(LOO_FIELDS, pw)),
                           draws=int(info.total_chains) * int(info.sampled), y=y.copy())
        st = Table()
        rows = int(info.rows)
        shapes = {"tau2": (1, 1), "u": (R, V), "xi": (V, 1), "gamma": (q, 1), "S": (q, 1), "theta": (1, 1),
                  "Delta": (1, 1), "M": (R, R), "mu": (1, 1), "lam": (R, 1), "pi": (R, 3)}
        names = list(_UNI) if return_state == "full" else (["xi", "gamma"] if return_state == "gamma_xi" else [])
        for k in names:
            shp = shapes[k]
            out = np.empty(rows * shp[0] * shp[1])
            check_fit(L.bnr_fit_state(res, VAR[k], out.ctypes.data_as(_DP)))
            st[k] = out.reshape((rows,) + shp, order="F")
        status = []
        for d in range(info.n_devices):
            h = C.c_void_p()
            check_fit(L.bnr_fit_handle(res, d, C.byref(h)))
            s_ = np.zeros(num_chains, dtype=np.int32)
            check(L.bnr_status(h, s_.ctypes.data_as(C.POINTER(C.c_int32))))
            status.append(s_)
        extra = dict(status=np.concatenate(status), tot_generated=int(info.tot_generated), seed=seed,
                     gamma_mode={1: "nform", 2: "qform"}[int(info.gamma_mode)], device_summary=dev_summary,
                     rhat_streamed=bool(info.streamed), n_psrf=int(info.n_psrf), total_chains=int(info.total_chains),
                     n_devices=int(info.n_devices), exchange={0: "none", 1: "nccl", 2: "peer-copy"}[int(info.exchange)],
                     ess=ess)
        if prediction is not None:
            extra["prediction"] = prediction
        if loo_out is not None:
            extra["loo"] = loo_out
        return Results(st, rx, rg, int(info.burn_in), int(info.sampled), extra)
    finally:
        L.bnr_fit_free(res)


def Fit(X, y, R, *, η=None, V=30, ζ=None, ι=None, aΔ=None, bΔ=None, ν=None, nburn=30000, nsamples=20000,
        mingen=0, maxgen=0, psrf_cutoff=1.01, x_transform=True, suppress_timer=False, num_chains=2, seed=None,
        purge_burn=None, filename="parameters.log", eta=None, zeta=None, iota=None, a_delta=None, b_delta=None,
        nu=None, device=0, return_state="full", verbose=False, chain_offset=0, n_devices=1, ess_max_lag=0,
        gamma_mode="auto", chain_groups=0, X_new=None, predictive=False, loo=False):
    """Drop-in for `Fit!(X, y, R; ...)` (src/gibbs.jl:725-751).  Greek keyword names are accepted as in the
    reference; ASCII aliases (eta, zeta, iota, a_delta, b_delta, nu) are equivalent.  Engine-only keywords: device,
    n_devices (GPUs of this process to shard the chains over; num_chains is the count PER GPU), return_state
    ("full" | "gamma_xi" | "none": how much of chain 1's table is copied back), ess_max_lag (> 0: gamma / xi ESS of the
    retained draws in res.extra["ess"]), chain_offset (global id of the first chain), gamma_mode, chain_groups.
    Inside a torch.distributed job every rank calls Fit with its own share of the chains; the R-hat tables then cover
    the chains of all ranks.
    X_new (new networks, in the form of X; vectorised by setup_X with the same x_transform): every chain also records
    mu + X_new gamma at every sweep (plus sqrt(tau2) N(0,1) noise with predictive=True, the posterior predictive), and
    the retained draws of all chains are pooled on the GPU into res.extra["prediction"] (see Predict).
    loo=True: every chain also records the pointwise log-likelihood log N(y_i | mu + (X gamma)_i, tau2) at every sweep,
    and PSIS-LOO and WAIC of the retained draws of all chains are computed on the GPU into res.extra["loo"] (see Loo
    and Compare)."""
    def pick(greek, ascii_, default):
        return default if (greek is None and ascii_ is None) else (greek if greek is not None else ascii_)

    eta = pick(η, eta, 1.01)
    zeta = pick(ζ, zeta, 1.0)
    iota = pick(ι, iota, 1.0)
    a_delta = pick(aΔ, a_delta, 1.0)
    b_delta = pick(bΔ, b_delta, 1.0)
    nu = pick(ν, nu, 10)
    if seed is None:
        seed = random.randint(1, 55555)
    rank, world = _dist_world()
    if world > 1 and rank != 0:
        filename = None                  # one parameters.log per job
    if filename:
        with open(filename, "w") as fh:
            fh.write("BayesianNetworkRegression.jl Fit! function\n")
            fh.write(datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S.%f")[:-3] + "\n")
            fh.write(_citation())
            fh.write("\n\nParameters:\n")
            fh.write("R=%s, η=%s, ζ=%s, ι=%s, aΔ=%s, bΔ=%s, ν=%s, nburn=%s, nsamples=%s, \n" %
                     (R, eta, zeta, iota, a_delta, b_delta, nu, nburn, nsamples))
            fh.write("mingen=%s, maxgen=%s, psrf_cutoff=%s, \n" % (mingen, maxgen, psrf_cutoff))
            fh.write("x_transform=%s, suppress_timer=%s, num_chains=%s, purge_burn=%s \n" %
                     (str(x_transform).lower(), str(suppress_timer).lower(), num_chains, purge_burn))
            fh.write("seed=%s" % seed)
    kw = dict(eta=eta, zeta=zeta, iota=iota, a_delta=a_delta, b_delta=b_delta, nu=nu,
              psrf_cutoff=psrf_cutoff, x_transform=x_transform, num_chains=num_chains, seed=seed,
              purge_burn=purge_burn, device=device, return_state=return_state, verbose=verbose,
              chain_offset=chain_offset, n_devices=n_devices, ess_max_lag=ess_max_lag, gamma_mode=gamma_mode,
              chain_groups=chain_groups, X_new=X_new, predictive=predictive, loo=loo)
    if mingen > 0 and maxgen > 0:
        return generate_samples_dbl(X, y, R, mingen=mingen, maxgen=maxgen, **kw)
    return generate_samples(X, y, R, nburn=nburn, nsamp=nsamples, **kw)


def _prepare_new(X_new, x_transform):
    return None if X_new is None else setup_X(X_new, x_transform)


def _prepare(X, y, R, nu, x_transform):
    if nu < R:
        # the reference builds this ArgumentError without throwing it (src/gibbs.jl:901-902); the
        # InverseWishart draw is undefined for nu <= R-1, so the engine refuses instead of continuing.
        raise ValueError("ν value (%s) must be greater than R value (%s)" % (nu, R))
    if nu == R:
        print("Warning: ν==R may give poor accuracy. Consider increasing ν")
    Xn = setup_X(X, x_transform)
    y = np.asarray(y, dtype=np.float64).ravel()
    return Xn, y


def generate_samples(X, y, R, *, eta=1.01, zeta=1.0, iota=1.0, a_delta=1.0, b_delta=1.0, nu=10, nburn=30000,
                     nsamp=20000, psrf_cutoff=1.2, x_transform=True, num_chains=2, seed=None, purge_burn=None, **kw):
    """The "traditional" scheme (generate_samples!, src/gibbs.jl:897-1020; maxburn = nburn + nsamp as Fit! passes it):
    the control loop runs inside libbnr (bnr_fit)."""
    Xn, y = _prepare(X, y, R, nu, x_transform)
    kw["X_new"] = _prepare_new(kw.get("X_new"), x_transform)
    seed = random.randint(1, 55555) if seed is None else seed
    return _native_fit(Xn, y, R, eta=eta, zeta=zeta, iota=iota, a_delta=a_delta, b_delta=b_delta, nu=nu, nburn=nburn,
                       nsamp=nsamp, psrf_cutoff=psrf_cutoff, purge_burn=purge_burn, num_chains=num_chains, seed=seed, **kw)


def generate_samples_dbl(X, y, R, *, eta=1.01, zeta=1.0, iota=1.0, a_delta=1.0, b_delta=1.0, nu=10, mingen=10000,
                         maxgen=100000, psrf_cutoff=1.01, x_transform=True, num_chains=2, seed=None,
                         purge_burn=None, **kw):
    """The "doubling generation" scheme (generate_samples_dbl!, src/gibbs.jl:1051-1198), inside libbnr (bnr_fit)."""
    Xn, y = _prepare(X, y, R, nu, x_transform)
    kw["X_new"] = _prepare_new(kw.get("X_new"), x_transform)
    seed = random.randint(1, 55555) if seed is None else seed
    return _native_fit(Xn, y, R, eta=eta, zeta=zeta, iota=iota, a_delta=a_delta, b_delta=b_delta, nu=nu, mingen=mingen,
                       maxgen=maxgen, psrf_cutoff=psrf_cutoff, purge_burn=purge_burn, num_chains=num_chains, seed=seed,
                       **kw)


def _summary_ranks(nsamp, interval):
    """lw / hi of src/gibbs.jl:1221-1223 (Julia round = ties to even, 1-based indices)."""
    lower = (100 - interval) / 200.0
    return _jround(nsamp * lower), _jround(nsamp * (1.0 - lower))


def Summary(results, interval=95, digits=3):
    """src/gibbs.jl:1214-1250: per-edge posterior mean and order-statistic credible bounds, per-node mean xi."""
    nburn, nsamp = results.burn_in, results.sampled
    total = nburn + nsamp
    lw, hi = _summary_ranks(nsamp, interval)
    if lw < 1 or hi > nsamp:
        raise IndexError("BoundsError: nsamp=%d too small for a %d%% interval" % (nsamp, interval))
    dev = (getattr(results, "extra", None) or {}).get("device_summary")
    if dev is not None and dev["interval"] == interval:
        # statistics were reduced on the GPU at the end of Fit (bnr_summary): only rounding and the tables remain
        mean, lo, up, xm, V = dev["mean"], dev["lower"], dev["upper"], dev["xi_mean"], dev["V"]
    else:
        # a different interval than the one reduced on the device: order statistics of chain 1's returned table
        if "gamma" not in results.state:
            raise ValueError("Summary(interval=%s) needs the gamma/xi table: call Fit with return_state='gamma_xi' "
                             "or 'full' (the device-side summary was computed for interval=%s only)"
                             % (interval, dev["interval"] if dev else None))
        g = np.asarray(results.state["gamma"])[nburn:total, :, 0]
        x = np.asarray(results.state["xi"])[nburn:total, :, 0]
        gs = np.sort(g, axis=0)
        mean, lo, up, xm = g.mean(axis=0), gs[lw - 1], gs[hi - 1], x.mean(axis=0)
        V = int((-1 + math.sqrt(1 + 8 * g.shape[1])) / 2)
    node1 = np.concatenate([np.full(V - k, k + 1, dtype=np.int64) for k in range(V)])
    node2 = np.concatenate([np.arange(k + 1, V + 1, dtype=np.int64) for k in range(V)])
    edge = dict(node1=node1, node2=node2, estimate=np.round(mean, digits),
                lower_bound=np.round(lo, digits), upper_bound=np.round(up, digits))
    nodes = dict(probability=np.round(xm, digits))
    return BNRSummary(edge, nodes, interval)


def Predict(results, interval=95, digits=3):
    """Predicted responses for the networks passed to Fit as X_new: per network the posterior mean of the prediction
    and the exact order statistics lw, hi of the draws of ALL chains (on every GPU and rank), lw / hi the Julia-rounded
    ranks of Summary applied to the pooled count.  The statistics are reduced on the GPU at the end of Fit for the
    95 % interval; only the rounding happens here."""
    pred = (getattr(results, "extra", None) or {}).get("prediction")
    if pred is None:
        raise ValueError("Predict needs a fit with new networks: call Fit(..., X_new=...)")
    if pred["interval"] != interval:
        raise ValueError("the prediction interval was reduced on the GPU for interval=%s only, not %s"
                         % (pred["interval"], interval))
    if pred["mean"] is None:
        raise IndexError("BoundsError: %d pooled draws are too few for a %d%% interval" % (pred["draws"], interval))
    m = int(pred["m"])
    table = dict(sample=np.arange(1, m + 1, dtype=np.int64), estimate=np.round(pred["mean"], digits),
                 lower_bound=np.round(pred["lower"], digits), upper_bound=np.round(pred["upper"], digits))
    return BNRPrediction(table, interval, bool(pred["predictive"]))


# -- out-of-sample scoring (the R package loo: print.loo, loo_compare) ----------------------------------------------
def _loo_pointwise(results):
    lo = (getattr(results, "extra", None) or {}).get("loo")
    if lo is None:
        raise ValueError("Loo needs a fit scored out of sample: call Fit(..., loo=True)")
    if lo["pointwise"] is None:
        raise ValueError("PSIS-LOO needs at least 2 retained draws, the fit kept %d" % lo["draws"])
    return lo


def _estimate(x):
    x = np.asarray(x, dtype=np.float64)
    return float(x.sum()), float(math.sqrt(x.size * x.var(ddof=1))) if x.size > 1 else float("nan")


class BNRLoo:
    """Loo's result: `estimates` maps elpd_loo, p_loo, looic, elpd_waic, p_waic, waic to (estimate, SE) with
    SE = sqrt(n var(pointwise)); `pointwise` holds the [n] arrays (looic / waic are -2 elpd); `n_high_k` counts the
    observations whose Pareto k exceeds `k_threshold` = min(1 - 1 / log10(S), 0.7) for S pooled draws."""

    NAMES = ("elpd_loo", "p_loo", "looic", "elpd_waic", "p_waic", "waic")

    def __init__(self, pointwise, draws):
        pw = {k: np.asarray(v, dtype=np.float64) for k, v in pointwise.items()}
        pw["looic"] = -2.0 * pw["elpd_loo"]
        pw["waic"] = -2.0 * pw["elpd_waic"]
        self.pointwise = pw
        self.draws = int(draws)
        self.n = int(pw["elpd_loo"].size)
        self.estimates = {k: _estimate(pw[k]) for k in self.NAMES}
        self.k_threshold = min(1.0 - 1.0 / math.log10(self.draws), 0.7)
        self.n_high_k = int(np.sum(pw["pareto_k"] > self.k_threshold))

    def __repr__(self):
        lines = ["", "Computed from %d by %d log-likelihood matrix." % (self.draws, self.n), "",
                 "           Estimate      SE"]
        for k in self.NAMES:
            e, se = self.estimates[k]
            lines.append("%-9s %9.1f %7.1f" % (k, e, se))
        if self.n_high_k:
            lines.append("")
            lines.append("Warning: %d of %d Pareto k diagnostic values are above %.2f: PSIS-LOO is unreliable for "
                         "these observations." % (self.n_high_k, self.n, self.k_threshold))
        else:
            lines.append("")
            lines.append("All Pareto k estimates are good (k <= %.2f)." % self.k_threshold)
        return "\n".join(lines)


def Loo(results):
    """PSIS-LOO and WAIC of a fit run with Fit(..., loo=True): estimates with standard errors, the pointwise arrays and
    the Pareto k diagnostic.  The pointwise values were computed on the GPU from the retained draws of ALL chains;
    only the sums happen here.  Warns (like loo's print method) when some Pareto k are too high."""
    lo = _loo_pointwise(results)
    out = BNRLoo(lo["pointwise"], lo["draws"])
    if out.n_high_k:
        warnings.warn("%d of %d Pareto k diagnostic values are above %.2f: PSIS-LOO is unreliable for these "
                      "observations" % (out.n_high_k, out.n, out.k_threshold), stacklevel=2)
    return out


class BNRCompare:
    """Compare's table: one row per fit, best first (a dict of columns like BNRSummary.edge_coef)."""

    COLUMNS = ("elpd_diff", "se_diff", "elpd_loo", "se_elpd_loo", "p_loo", "se_p_loo", "looic", "se_looic")

    def __init__(self, table):
        self.table = table

    def __repr__(self):
        t = self.table
        lines = ["", "%-10s" % "model" + "".join("%12s" % c for c in self.COLUMNS)]
        for i, name in enumerate(t["model"]):
            lines.append("%-10s" % name + "".join("%12.1f" % t[c][i] for c in self.COLUMNS))
        return "\n".join(lines)


def Compare(*results, names=None):
    """loo_compare: the fits ranked by elpd_loo (best first); elpd_diff = elpd_loo - elpd_loo(best) and
    se_diff = sqrt(n) sd(pointwise elpd_loo differences to the best), both 0 for the best.  The fits must have been
    run on the same responses y."""
    if len(results) < 2:
        raise ValueError("Compare needs at least two fits")
    names = list(names) if names is not None else ["model%d" % (i + 1) for i in range(len(results))]
    if len(names) != len(results):
        raise ValueError("one name per fit")
    los = [_loo_pointwise(r) for r in results]
    y0 = los[0]["y"]
    for lo in los[1:]:
        if lo["y"].shape != y0.shape or not np.array_equal(lo["y"], y0):
            raise ValueError("Compare needs fits of the same responses y")
    loos = [BNRLoo(lo["pointwise"], lo["draws"]) for lo in los]
    elpd = np.array([lo.estimates["elpd_loo"][0] for lo in loos])
    order = sorted(range(len(loos)), key=lambda i: -elpd[i])
    best = loos[order[0]].pointwise["elpd_loo"]
    n = best.size
    table = {c: [] for c in ("model",) + BNRCompare.COLUMNS}
    for i in order:
        lo = loos[i]
        d = lo.pointwise["elpd_loo"] - best
        table["model"].append(names[i])
        table["elpd_diff"].append(float(d.sum()))
        table["se_diff"].append(float(math.sqrt(n) * d.std(ddof=1)) if n > 1 else 0.0)
        for k in ("elpd_loo", "p_loo", "looic"):
            e, se = lo.estimates[k]
            table[k].append(e)
            table["se_" + k].append(se)
    for c in BNRCompare.COLUMNS:
        table[c] = np.asarray(table[c])
    return BNRCompare(table)
