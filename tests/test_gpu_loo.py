"""Pointwise log-likelihood and pooled PSIS-LOO / WAIC on the device (bnr_set_loglik, bnr_loo_summary, bnr_fit_loo):
every recorded row holds log N(y_i | mu + (X gamma)_i, tau2) of that row's own state, nothing of the sampler changes
when the table is on, the pooled estimates equal the NumPy restatement (oracle/loo.py) applied to the retained rows of
all chains, and PSIS-LOO agrees with brute-force leave-one-out refits."""
import ctypes as C
import os
import socket
import warnings

import numpy as np
import pytest

from oracle import loo as OL
from oracle import psrf_loops as PL

pytestmark = pytest.mark.gpu

_DP = C.POINTER(C.c_double)
FIELDS = ("elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic")


def _toy(seed, V=6, n=40):
    rng = np.random.default_rng(seed)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.7)
    y = 1.0 + X[:, :5].sum(axis=1) + rng.normal(0, 1.5, size=n)
    return X, y


# (V, n, gamma form): the q-form, and an n-form with qp >= 1024 (the INT8 Gram path)
FORMS = [(6, 40, "qform"), (45, 40, "nform")]


def _want(eng, X, y, c, rows):
    tau2 = eng.get_trace(c, "tau2", 0, rows)[:, 0, 0]
    mu = eng.get_trace(c, "mu", 0, rows)[:, 0, 0]
    G = eng.get_trace(c, "gamma", 0, rows)[:, :, 0]
    xg = G @ X.T
    want = OL.loglik(y[None, :], mu[:, None], xg, tau2[:, None])
    r = np.abs(y[None, :] - mu[:, None] - xg)
    scale = np.abs(want) + r * (np.abs(G) @ np.abs(X).T + np.abs(mu)[:, None] + np.abs(y)[None, :]) / tau2[:, None]
    return want, scale


@pytest.mark.parametrize("V,n,form", FORMS)
def test_every_row_is_the_log_density_of_its_own_state(bnr, V, n, form):
    X, y = _toy(1, V, n)
    C_, sweeps, cap = 5, 7, 10
    with bnr.Engine(X, y, 3, num_chains=C_, seed=4, trace_rows=cap, trace_full_chains=C_, gamma_mode=form) as eng:
        eng.set_loglik(cap)
        eng.init_state()
        eng.run(sweeps)
        # one more sweep conditional by conditional (bnr_step / bnr_finish_sweep)
        for cond in ("tau2", "u_xi", "gamma", "D", "theta", "Delta", "M", "mu", "lam", "pi"):
            eng.step(cond)
        eng.finish_sweep()
        rows = sweeps + 2
        for c in range(C_):
            got = eng.loglik_trace(c, 0, cap)
            want, scale = _want(eng, X, y, c, rows)
            assert np.all(np.abs(got[:rows] - want) <= 1e-12 * scale), "chain %d" % c
            assert np.isnan(got[rows:]).all()                # rows never written


def _sampler_outputs(eng, C_, rows):
    out = [eng.get_state_dict(c) for c in range(C_)]
    tr = [eng.get_trace(c, "gamma", 0, rows) for c in range(C_)]
    rx, rg = eng.rhat()
    summ = eng.summary(0, rows // 2, rows - rows // 2, 1, rows - rows // 2)
    ess = eng.ess(rows // 2, rows - rows // 2, 7)
    return out, tr, (rx, rg), summ, ess


def _same(a, b):
    if isinstance(a, dict):
        assert a.keys() == b.keys()
        for k in a:
            _same(a[k], b[k])
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            _same(x, y)
    else:
        np.testing.assert_array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.parametrize("V,n,form", FORMS)
def test_the_table_changes_nothing_in_the_sampler(bnr, V, n, form):
    X, y = _toy(2, V, n)
    Xn = np.random.default_rng(2).normal(size=(9, X.shape[1]))
    C_, sweeps = 7, 16
    got, counts = [], []
    for on in (False, True):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=8, trace_rows=sweeps + 1, trace_full_chains=1,
                        gamma_mode=form, chain_groups=2) as eng:
            eng.set_predictors(Xn, sweeps + 1)
            if on:
                eng.set_loglik(sweeps + 1)
            eng.set_moment_window(1, sweeps)
            eng.init_state()
            eng.run(sweeps)
            got.append(_sampler_outputs(eng, C_, sweeps + 1) +
                       ([eng.prediction_trace(c, 0, sweeps + 1) for c in range(C_)],))
            counts.append((eng.launch_count(), eng.chain_groups))
    _same(got[0], got[1])
    (off, g), (on_, g2) = counts
    assert g == g2 and on_ - off == sweeps * g          # one k_loglik_record per sweep and chain group


def _fit(bnr, fn, X, y, R, num_chains=3, seed=21, n_devices=1, **kw):
    """bnr_fit_loo / bnr_fit_predict through ctypes: info, pointwise LOO (or None), R-hat, Summary and every chain's
    retained log-likelihood rows read back per handle and chain."""
    from bnr_b200 import capi
    L = bnr.lib()
    Xf = np.asfortranarray(X, dtype=np.float64)
    yv = np.ascontiguousarray(y, dtype=np.float64)
    n, q = Xf.shape
    V = int(round((-1 + np.sqrt(1 + 8 * q)) / 2))
    p = capi.FitParams()
    L.bnr_fit_default_params(C.byref(p))
    p.base.n, p.base.V, p.base.R, p.base.num_chains, p.base.seed = n, V, R, num_chains, seed
    p.nburn, p.nsamples = kw.get("nburn", 0), kw.get("nsamples", 0)
    p.mingen, p.maxgen = kw.get("mingen", 0), kw.get("maxgen", 0)
    p.purge_burn = kw.get("purge_burn", 0) or 0
    p.psrf_cutoff = kw["cutoff"]
    p.return_state, p.n_devices = capi.STATE["full"], n_devices
    res = C.c_void_p()
    rc = getattr(L, fn)(C.byref(p), Xf.ctypes.data_as(_DP), yv.ctypes.data_as(_DP), 0, None, 0, C.byref(res))
    if rc != 0:
        raise capi.BnrError(rc, L.bnr_fit_last_error().decode())
    try:
        info = capi.FitInfo()
        capi.check_fit(L.bnr_fit_get_info(res, C.byref(info)))
        rx, rg = np.empty(V), np.empty(q)
        capi.check_fit(L.bnr_fit_rhat(res, rx.ctypes.data_as(_DP), rg.ctypes.data_as(_DP)))
        summ = None
        if info.summary_ok:
            summ = [np.empty(q), np.empty(q), np.empty(q), np.empty(V)]
            capi.check_fit(L.bnr_fit_summary(res, *(a.ctypes.data_as(_DP) for a in summ)))
        gam = np.empty(int(info.rows) * q)
        capi.check_fit(L.bnr_fit_state(res, capi.VAR["gamma"], gam.ctypes.data_as(_DP)))
        pw, draws = None, []
        if fn == "bnr_fit_loo":
            out = [np.empty(n) for _ in FIELDS]
            rc = L.bnr_fit_loo_pointwise(res, *(a.ctypes.data_as(_DP) for a in out))
            if rc == 0:
                pw = dict(zip(FIELDS, out))
            else:
                assert rc == -4
            b, s = int(info.burn_in), int(info.sampled)
            for d in range(info.n_devices):
                h = C.c_void_p()
                capi.check_fit(L.bnr_fit_handle(res, d, C.byref(h)))
                for c in range(num_chains):
                    o = np.empty(s * n)
                    capi.check(L.bnr_get_loglik_trace(h, c, b, b + s, o.ctypes.data_as(_DP)))
                    draws.append(o.reshape((s, n), order="F"))
        other = (int(info.burn_in), int(info.sampled), int(info.tot_generated), rx, rg, summ, gam)
        return info, pw, draws, other
    finally:
        L.bnr_fit_free(res)


def _close(got, want):
    for k in ("elpd_loo", "p_loo", "elpd_waic", "p_waic"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-10, atol=1e-12, err_msg=k)
    kg, kw = got["pareto_k"], want["pareto_k"]
    assert np.array_equal(np.isinf(kg), np.isinf(kw))
    fin = np.isfinite(kw)
    np.testing.assert_allclose(kg[fin], kw[fin], rtol=0, atol=1e-9)


CASES = [dict(nburn=40, nsamples=30, purge_burn=10, cutoff=1.02), dict(nburn=24, nsamples=8, purge_burn=4, cutoff=1.02),
         dict(nburn=30, nsamples=21, purge_burn=5, cutoff=1e9), dict(mingen=40, maxgen=200, cutoff=1.02),
         dict(mingen=14, maxgen=60, purge_burn=3, cutoff=1.02)]


@pytest.mark.parametrize("kw", CASES)
def test_fit_loo_pools_the_retained_rows_of_all_chains(bnr, kw):
    X, y = _toy(5)
    C_, R, seed, smax = 3, 3, 21, 420
    with bnr.Engine(X, y, R, num_chains=C_, seed=seed, trace_rows=smax + 1, trace_full_chains=C_) as eng:
        eng.init_state()
        eng.run(smax)
        Xi = np.stack([eng.get_trace(c, "xi", 0, smax + 1)[:, :, 0] for c in range(C_)])
        G = np.stack([eng.get_trace(c, "gamma", 0, smax + 1)[:, :, 0] for c in range(C_)])
        want_rows = [_want(eng, X, y, c, smax + 1) for c in range(C_)]
    draw = lambda c, s: (Xi[c, s], G[c, s])           # noqa: E731
    try:
        if "mingen" in kw:
            plan = PL.generate_samples_dbl(draw, C_, kw["mingen"], kw["maxgen"], kw["cutoff"], kw.get("purge_burn"))
        else:
            plan = PL.generate_samples(draw, C_, kw["nburn"], kw["nsamples"], kw["nburn"] + kw["nsamples"],
                                       kw["cutoff"], kw.get("purge_burn"))
    except IndexError:
        with pytest.raises(bnr.BnrError, match="BoundsError"):
            _fit(bnr, "bnr_fit_loo", X, y, R, num_chains=C_, seed=seed, **kw)
        return
    info, pw, draws, other = _fit(bnr, "bnr_fit_loo", X, y, R, num_chains=C_, seed=seed, **kw)
    b, s = int(info.burn_in), int(info.sampled)
    assert (b, s) == (plan["burn_in"], plan["sampled"])
    for c in range(C_):
        sw = plan["rows"][c][b:b + s]
        want, scale = want_rows[c]
        assert np.all(np.abs(draws[c] - want[sw]) <= 1e-12 * scale[sw]), "chain %d" % c
    pooled = np.concatenate(draws)
    if pooled.shape[0] < 2:
        assert pw is None
    else:
        _close(pw, OL.loo_pointwise(pooled))
    _, _, _, plain = _fit(bnr, "bnr_fit_predict", X, y, R, num_chains=C_, seed=seed, **kw)
    _same(list(other), list(plain))


def _upload(a):
    import torch
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda:0")


def _tables():
    rng = np.random.default_rng(11)
    out = {}
    out["gaussian"] = rng.normal(-1.0, 0.5, size=(4000, 16))
    heavy = -np.log1p(rng.pareto(0.9, size=(4000, 5)))        # importance ratios with a Pareto(0.9) tail: k ~ 1.1
    out["heavy"] = heavy
    const = rng.normal(size=(3000, 4))
    const[:, 2] = -1.25
    out["constant"] = const
    out["ties"] = np.round(rng.normal(size=(5000, 9)), 1)     # many copies of the boundary value
    out["small"] = rng.normal(size=(12, 6))
    out["odd_n"] = rng.normal(size=(777, 13)) * rng.uniform(0.1, 3.0, 13)
    out["many_blocks"] = rng.standard_t(5, size=(200_000, 3))
    return out


def test_loo_summary_matches_the_oracle(bnr):
    from bnr_b200.engine import loo_summary
    for name, tab in _tables().items():
        t = _upload(tab)
        got = loo_summary(0, t.data_ptr(), tab.shape[0], tab.shape[1])
        want = OL.loo_pointwise(tab)
        try:
            _close(got, want)
        except AssertionError as e:
            raise AssertionError("%s: %s" % (name, e))
        again = loo_summary(0, t.data_ptr(), tab.shape[0], tab.shape[1])
        _same(got, again)
        if name == "heavy":
            assert (got["pareto_k"] > 0.7).all()
        if name == "constant":
            assert np.isinf(got["pareto_k"][2])
        if name == "small":
            assert np.isinf(got["pareto_k"]).all()
    # a tail that does not fit one block's shared memory is refused with the limit in the message
    with pytest.raises(bnr.BnrError, match="shared memory") as ei:
        loo_summary(0, t.data_ptr(), 10**9, 1)
    assert ei.value.code == -1


def _mr_data():
    return _toy(3, V=7, n=50)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from conftest import load_package
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    bnr = load_package()
    X, y = _mr_data()
    res = bnr.Fit(X, y, 3, nburn=60, nsamples=40, num_chains=3, seed=17, x_transform=False, filename=None,
                  psrf_cutoff=1e9, device=0, return_state="none", loo=True)
    q.put((rank, {k: np.asarray(v) for k, v in res.extra["loo"]["pointwise"].items()}))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_equal_one_handle(bnr):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        r, pw = q.get(timeout=300)
        got[r] = pw
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    X, y = _mr_data()
    one = bnr.Fit(X, y, 3, nburn=60, nsamples=40, num_chains=6, seed=17, x_transform=False, filename=None,
                  psrf_cutoff=1e9, return_state="none", loo=True)
    _same(got[0], got[1])
    _same(got[0], one.extra["loo"]["pointwise"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")              # 240 draws of a short fit: many k above 1 - 1/log10(240)
        lo = bnr.Loo(one)
    assert lo.draws == 6 * 40 and lo.n == 50


def test_two_devices_equal_one_device(bnr):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    X, y = _toy(8)
    for kw in (dict(nburn=60, nsamples=40, cutoff=1e9), dict(mingen=40, maxgen=120, cutoff=0.0)):
        two = _fit(bnr, "bnr_fit_loo", X, y, 3, num_chains=3, n_devices=2, seed=17, **kw)
        one = _fit(bnr, "bnr_fit_loo", X, y, 3, num_chains=6, n_devices=1, seed=17, **kw)
        assert two[0].n_devices == 2 and two[0].total_chains == 6
        _same(two[1], one[1])
        _same(two[2], one[2])


def test_psis_loo_agrees_with_brute_force_refits(bnr):
    """Level 2: for three observations, log p(y_i | y_-i) from a refit without i (the pooled draws of all chains)
    agrees with PSIS-LOO's elpd_i of the full fit within 4 Monte Carlo standard errors (from per-chain estimates)."""
    from scipy.special import logsumexp
    from bnr_b200.engine import loo_summary
    X, y = _toy(9, V=5, n=40)
    R, C_, burn, S = 3, 32, 300, 400
    rows = burn + S + 1
    with bnr.Engine(X, y, R, num_chains=C_, seed=5) as eng:
        eng.set_loglik(rows)
        eng.init_state()
        eng.run(burn + S)
        ll = np.stack([eng.loglik_trace(c, burn + 1, rows) for c in range(C_)])      # [C][S][n]
    full = loo_summary(0, _upload(ll.reshape(-1, ll.shape[2])).data_ptr(), C_ * S, ll.shape[2])
    groups = 8
    part = [OL.loo_pointwise(g.reshape(-1, ll.shape[2]))["elpd_loo"] for g in np.split(ll, groups)]
    se_psis = np.std(part, axis=0, ddof=1) / np.sqrt(groups)
    for i in (0, 1, 2):
        keep = np.arange(X.shape[0]) != i
        with bnr.Engine(X[keep], y[keep], R, num_chains=C_, seed=6, trace_rows=rows, trace_full_chains=C_) as eng:
            eng.init_state()
            eng.run(burn + S)
            lli = np.stack([OL.loglik(y[i], eng.get_trace(c, "mu", burn + 1, rows)[:, 0, 0],
                                      eng.get_trace(c, "gamma", burn + 1, rows)[:, :, 0] @ X[i],
                                      eng.get_trace(c, "tau2", burn + 1, rows)[:, 0, 0]) for c in range(C_)])
        brute = logsumexp(lli) - np.log(lli.size)
        per_chain = logsumexp(lli, axis=1) - np.log(S)
        se_brute = np.std(per_chain, ddof=1) / np.sqrt(C_)
        se = np.hypot(se_brute, se_psis[i])
        assert abs(full["elpd_loo"][i] - brute) < 4 * se + 1e-3, (i, full["elpd_loo"][i], brute, se)
