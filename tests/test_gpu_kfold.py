"""K-fold cross-validation on the device (bnr_set_heldout, bnr_lpd_summary, bnr_fit_kfold): every held-out row is the log
density of its observation under that row's own state, the table changes nothing in the sampler, the pooled
log-mean-exp is exact and repeatable, every fold is bit for bit the standalone fit of its training rows, the pooling
puts each observation's log-mean-exp in its place, and K = n agrees with PSIS-LOO."""
import ctypes as C
import warnings

import numpy as np
import pytest

import kfold_util as KU
from oracle import loo as OL

pytestmark = pytest.mark.gpu

_DP = C.POINTER(C.c_double)


def _toy(seed, V=6, n=40):
    rng = np.random.default_rng(seed)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.7)
    y = 1.0 + X[:, :5].sum(axis=1) + rng.normal(0, 1.5, size=n)
    return X, y


# (V, n, gamma form): the q-form, and an n-form with qp >= 1024 (the INT8 Gram path)
FORMS = [(6, 40, "qform"), (45, 40, "nform")]


def _want(eng, Xh, yh, c, rows):
    tau2 = eng.get_trace(c, "tau2", 0, rows)[:, 0, 0]
    mu = eng.get_trace(c, "mu", 0, rows)[:, 0, 0]
    G = eng.get_trace(c, "gamma", 0, rows)[:, :, 0]
    xg = G @ Xh.T
    want = OL.loglik(yh[None, :], mu[:, None], xg, tau2[:, None])
    r = np.abs(yh[None, :] - mu[:, None] - xg)
    scale = np.abs(want) + r * (np.abs(G) @ np.abs(Xh).T + np.abs(mu)[:, None] + np.abs(yh)[None, :]) / tau2[:, None]
    return want, scale


@pytest.mark.parametrize("V,n,form", FORMS)
def test_every_heldout_row_is_the_log_density_of_its_own_state(bnr, V, n, form):
    X, y = _toy(1, V, n)
    Xh, yh = _toy(2, V, 13)
    C_, sweeps, cap = 5, 7, 10
    with bnr.Engine(X, y, 3, num_chains=C_, seed=4, trace_rows=cap, trace_full_chains=C_, gamma_mode=form) as eng:
        eng.set_heldout(Xh, yh, cap)
        eng.init_state()
        eng.run(sweeps)
        for cond in ("tau2", "u_xi", "gamma", "D", "theta", "Delta", "M", "mu", "lam", "pi"):
            eng.step(cond)
        eng.finish_sweep()
        rows = sweeps + 2
        for c in range(C_):
            got = eng.heldout_trace(c, 0, cap)
            want, scale = _want(eng, Xh, yh, c, rows)
            assert np.all(np.abs(got[:rows] - want) <= 1e-12 * scale), "chain %d" % c
            assert np.isnan(got[rows:]).all()                # rows never written


def _outputs(eng, C_, rows):
    st = [eng.get_state_dict(c) for c in range(C_)]
    tr = [eng.get_trace(c, "gamma", 0, rows) for c in range(C_)]
    return st, tr, eng.rhat(), eng.summary(0, rows // 2, rows - rows // 2, 1, rows - rows // 2), \
        eng.ess(rows // 2, rows - rows // 2, 7)


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
def test_the_heldout_table_changes_nothing_in_the_sampler(bnr, V, n, form):
    X, y = _toy(3, V, n)
    Xh, yh = _toy(4, V, 9)
    C_, sweeps = 7, 16
    got, counts = [], []
    for arm in ("off", "predictors", "heldout"):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=8, trace_rows=sweeps + 1, trace_full_chains=1,
                        gamma_mode=form, chain_groups=2) as eng:
            if arm == "predictors":
                eng.set_predictors(Xh, sweeps + 1)
            if arm == "heldout":
                eng.set_heldout(Xh, yh, sweeps + 1)
            eng.set_moment_window(1, sweeps)
            eng.init_state()
            eng.run(sweeps)
            got.append(_outputs(eng, C_, sweeps + 1))
            counts.append(eng.launch_count())
    _same(got[0], got[1])
    _same(got[0], got[2])
    assert counts[2] == counts[1] > counts[0]


def test_lpd_summary_is_exact_and_repeatable(bnr):
    import torch
    from scipy.special import logsumexp
    from bnr_b200.engine import lpd_summary
    rng = np.random.default_rng(5)
    for N, m in ((200_000, 5), (3000, 37), (1, 4), (50_000, 1)):
        tab = rng.normal(-1.0, 2.0, size=(N, m)) * rng.uniform(0.1, 3.0, m)
        t = torch.tensor(tab, dtype=torch.float64, device="cuda:0")
        got = lpd_summary(0, t.data_ptr(), N, m)
        want = logsumexp(tab, axis=0) - np.log(N)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
        _same(got, lpd_summary(0, t.data_ptr(), N, m))


def _states(bnr, h, C_, R, V, q):
    from bnr_b200 import capi
    from bnr_b200.engine import var_shape
    L = bnr.lib()
    out = []
    for c in range(C_):
        d = {}
        for k, v in capi.VAR.items():
            shp = var_shape(k, R, V, q)
            a = np.empty(shp[0] * shp[1])
            capi.check(L.bnr_get_state(h, c, v, a.ctypes.data_as(_DP)))
            d[k] = a
        out.append(d)
    return out


def _heldout_rows(bnr, h, C_, first, last, m):
    from bnr_b200 import capi
    rows = []
    for c in range(C_):
        a = np.empty((last - first) * m)
        capi.check(bnr.lib().bnr_get_prediction_trace(h, c, first, last, a.ctypes.data_as(_DP)))
        rows.append(a.reshape((last - first, m), order="F"))
    return rows


def _kfold(bnr, p, X, y, K, folds):
    """bnr_fit_kfold: info, pointwise, per fold (R-hat xi, gamma, states, every chain's retained held-out rows)."""
    from bnr_b200 import capi
    L = bnr.lib()
    R, V, C_ = p.base.R, p.base.V, p.base.num_chains
    q = V * (V + 1) // 2
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
        b, s = int(info.burn_in), int(info.sampled)
        per = []
        for f in range(K):
            rx, rg = np.empty(V), np.empty(q)
            capi.check_fit(L.bnr_fit_kfold_rhat(res, f, rx.ctypes.data_as(_DP), rg.ctypes.data_as(_DP)))
            h = C.c_void_p()
            capi.check_fit(L.bnr_fit_handle(res, f, C.byref(h)))
            per.append(dict(rhat=(rx, rg), states=_states(bnr, h, C_, R, V, q),
                            rows=_heldout_rows(bnr, h, C_, b, b + s, int((folds == f + 1).sum()))))
        allr = (np.empty(V), np.empty(q))
        capi.check_fit(L.bnr_fit_rhat(res, *(a.ctypes.data_as(_DP) for a in allr)))
        for fn in ("bnr_fit_summary", "bnr_fit_ess", "bnr_fit_prediction", "bnr_fit_loo_pointwise"):
            assert getattr(L, fn)(res, *([None] * {"bnr_fit_summary": 4, "bnr_fit_ess": 2, "bnr_fit_prediction": 3,
                                                    "bnr_fit_loo_pointwise": 5}[fn])) == -4, fn
        assert L.bnr_fit_state(res, 0, np.empty(1).ctypes.data_as(_DP)) == -4
        return info, pw, per, allr
    finally:
        L.bnr_fit_free(res)


def _fit(bnr, p, X, y):
    """bnr_fit: info, R-hat, every chain's state."""
    from bnr_b200 import capi
    L = bnr.lib()
    V, C_ = p.base.V, p.base.num_chains
    q = V * (V + 1) // 2
    Xf = np.asfortranarray(X, dtype=np.float64)
    yv = np.ascontiguousarray(y, dtype=np.float64)
    res = C.c_void_p()
    capi.check_fit(L.bnr_fit(C.byref(p), Xf.ctypes.data_as(_DP), yv.ctypes.data_as(_DP), C.byref(res)))
    try:
        info = capi.FitInfo()
        capi.check_fit(L.bnr_fit_get_info(res, C.byref(info)))
        rx, rg = np.empty(V), np.empty(q)
        capi.check_fit(L.bnr_fit_rhat(res, rx.ctypes.data_as(_DP), rg.ctypes.data_as(_DP)))
        h = C.c_void_p()
        capi.check_fit(L.bnr_fit_handle(res, 0, C.byref(h)))
        return info, (rx, rg), _states(bnr, h, C_, p.base.R, V, q)
    finally:
        L.bnr_fit_free(res)


SCHEMES = [dict(nburn=30, nsamples=20, psrf_cutoff=1e9), dict(mingen=16, maxgen=48, psrf_cutoff=0.0)]


@pytest.mark.parametrize("sched", SCHEMES, ids=["traditional", "doubling"])
@pytest.mark.parametrize("V,n,form", FORMS)
def test_every_fold_is_the_standalone_fit_of_its_training_rows(bnr, sched, V, n, form):
    from bnr_b200 import capi
    from scipy.special import logsumexp
    X, y = _toy(6, V, n)
    K, C_, R, off = 4, 3, 3, 5
    folds = bnr.kfold_split(n, K, 2)
    gm = capi.GAMMA_MODE[form]
    p = KU.fit_params(bnr, n, V, R, C_, 13, off, **sched)
    p.base.gamma_mode = gm
    info, pw, per, allr = _kfold(bnr, p, X, y, K, folds)
    assert info.total_chains == K * C_ and info.n_devices == 1
    b, s = int(info.burn_in), int(info.sampled)
    for f in range(K):
        Xt, yt, Xh, yh = KU.split(X, y, folds, f + 1)
        pf = KU.fit_params(bnr, Xt.shape[0], V, R, C_, 13, off + f * C_, **sched)
        pf.base.gamma_mode = gm
        finfo, frhat, fstates = _fit(bnr, pf, Xt, yt)
        assert (finfo.tot_generated, finfo.burn_in, finfo.sampled) == (info.tot_generated, b, s)
        _same(per[f]["states"], fstates)
        _same(per[f]["rhat"], frhat)
        # the held-out rows of the same handle driven alone through bnr_fit's operations
        with KU.replay(bnr, pf, KU.plan(bnr, pf), Xt, yt, Xh, yh) as eng:
            _same(per[f]["rows"], [eng.heldout_trace(c, b, b + s) for c in range(C_)])
            _same(per[f]["states"], [{k: eng.get_state(c, k).ravel(order="F") for k in capi.VAR} for c in range(C_)])
        # the pooling: log-mean-exp of every chain's retained rows, in the original observation order
        pooled = np.concatenate(per[f]["rows"])
        np.testing.assert_allclose(pw[folds == f + 1], logsumexp(pooled, axis=0) - np.log(pooled.shape[0]),
                                   rtol=1e-12, atol=0)
    # bnr_fit_rhat: the element-wise maximum over the folds
    for i in range(2):
        stack = np.stack([per[f]["rhat"][i] for f in range(K)])
        np.testing.assert_array_equal(allr[i], np.max(stack, axis=0))


def test_k_equal_n_is_exact_loo(bnr):
    """elpd_kfold_i with K = n (brute-force refits, all folds together) agrees with the PSIS elpd_loo_i of the full fit
    within 4 Monte Carlo standard errors wherever Pareto k <= 0.7."""
    import torch
    from bnr_b200.engine import loo_summary
    X, y = _toy(9, V=5, n=40)
    n = X.shape[0]
    R, C_, burn, S = 3, 32, 300, 400
    rows = burn + S + 1
    with bnr.Engine(X, y, R, num_chains=C_, seed=5) as eng:
        eng.set_loglik(rows)
        eng.init_state()
        eng.run(burn + S)
        ll = np.stack([eng.loglik_trace(c, burn + 1, rows) for c in range(C_)])      # [C][S][n]
    t = torch.tensor(ll.reshape(-1, n), dtype=torch.float64, device="cuda:0")
    full = loo_summary(0, t.data_ptr(), C_ * S, n)
    groups = 8
    part = [OL.loo_pointwise(g.reshape(-1, n))["elpd_loo"] for g in np.split(ll, groups)]
    se_psis = np.std(part, axis=0, ddof=1) / np.sqrt(groups)
    folds = np.arange(1, n + 1)
    p = KU.fit_params(bnr, n, 5, R, C_, 6, 0, nburn=burn + 1, nsamples=S, psrf_cutoff=1e9)
    info, pw, per, _ = _kfold(bnr, p, X, y, n, folds)
    assert (int(info.burn_in), int(info.sampled)) == (burn + 1, S)
    from scipy.special import logsumexp
    ok = full["pareto_k"] <= 0.7
    assert ok.sum() >= n // 2
    for i in np.flatnonzero(ok):
        per_chain = np.array([logsumexp(r[:, 0]) - np.log(S) for r in per[i]["rows"]])
        se = np.hypot(np.std(per_chain, ddof=1) / np.sqrt(C_), se_psis[i])
        assert abs(full["elpd_loo"][i] - pw[i]) < 4 * se + 1e-3, (i, full["elpd_loo"][i], pw[i], se)


def test_two_devices_equal_one_device(bnr):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    X, y = _toy(8)
    folds = bnr.kfold_split(X.shape[0], 5, 1)
    for sched in SCHEMES:
        out = []
        for nd in (1, 2):
            p = KU.fit_params(bnr, X.shape[0], 6, 3, 3, 17, 0, n_devices=nd, **sched)
            out.append(_kfold(bnr, p, X, y, 5, folds))
        assert out[0][0].n_devices == 1 and out[1][0].n_devices == 2
        _same(out[0][1], out[1][1])
        # every fold's R-hat, chain states and retained held-out rows
        _same(out[0][2], out[1][2])
        _same(out[0][3], out[1][3])


def test_kfold_and_compare_end_to_end(bnr):
    X, y = _toy(10, V=6, n=40)
    res = {}
    for R in (3, 5):
        res[R] = bnr.KFold(X, y, R, K=5, nburn=40, nsamples=30, num_chains=4, seed=3, fold_seed=7, x_transform=False,
                           psrf_cutoff=1e9)
        r = res[R]
        assert isinstance(r, bnr.BNRKFold) and r.K == 5 and r.draws == 4 * 30
        assert np.isfinite(r.pointwise["elpd_kfold"]).all() and r.rhat_max.shape == (5,)
        assert r.status & bnr.STATUS_BITS["nan"] == 0
        np.testing.assert_array_equal(r.folds, bnr.kfold_split(40, 5, 7))
        assert "5-fold" in repr(r)
    cmp = bnr.Compare(res[3], res[5], names=["R3", "R5"])
    assert sorted(cmp.table["model"]) == ["R3", "R5"] and cmp.table["elpd_diff"][0] == 0.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fit = bnr.Fit(X, y, 3, nburn=40, nsamples=30, num_chains=4, seed=3, x_transform=False, filename=None,
                      psrf_cutoff=1e9, loo=True)
    with pytest.raises(ValueError, match="cannot mix"):
        bnr.Compare(res[3], fit)
