"""Predictions for new networks (bnr_set_predictors / bnr_fit_predict): every recorded row of every chain holds
mu + X_new gamma (+ sqrt(tau2) z) of that row's own state, the rows follow the trace bookkeeping (purge ring, extension
rounds, doubling rounds), the pooled summary is the exact order statistics of all retained draws of all chains, and
nothing of the sampler changes when predictions are on."""
import ctypes as C

import numpy as np
import pytest

from oracle import psrf_loops as PL

pytestmark = pytest.mark.gpu

_DP = C.POINTER(C.c_double)


def _toy(seed, V=6, n=40):
    rng = np.random.default_rng(seed)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.7)
    y = 1.0 + X[:, :5].sum(axis=1) + rng.normal(0, 1.5, size=n)
    return X, y


def _new(seed, m, q):
    rng = np.random.default_rng(1000 + seed)
    return rng.normal(size=(m, q)) * (rng.random((m, q)) < 0.7)


# (V, n, gamma form): the q-form, and an n-form with qp >= 1024 (the INT8 Gram path)
FORMS = [(6, 40, "qform"), (45, 40, "nform")]


def _trace(eng, c, var, rows):
    return eng.get_trace(c, var, 0, rows)


@pytest.mark.parametrize("V,n,form", FORMS)
@pytest.mark.parametrize("m", [1, 37, 300])
def test_every_row_is_mu_plus_xnew_gamma_of_its_own_state(bnr, V, n, form, m):
    X, y = _toy(1, V, n)
    q = X.shape[1]
    Xn = _new(1, m, q)
    C_, sweeps, cap = 5, 7, 10
    with bnr.Engine(X, y, 3, num_chains=C_, seed=4, trace_rows=cap, trace_full_chains=C_, gamma_mode=form) as eng:
        eng.set_predictors(Xn, cap)
        eng.init_state()
        eng.run(sweeps)
        for c in range(C_):
            P = eng.prediction_trace(c, 0, cap)
            G = _trace(eng, c, "gamma", sweeps + 1)[:, :, 0]
            mu = _trace(eng, c, "mu", sweeps + 1)[:, 0, 0]
            want = mu[:, None] + G @ Xn.T
            scale = np.abs(G) @ np.abs(Xn).T + np.abs(mu)[:, None]
            assert np.all(np.abs(P[:sweeps + 1] - want) <= 1e-12 * scale), "chain %d" % c
            assert np.isnan(P[sweeps + 1:]).all()        # rows never written


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
@pytest.mark.parametrize("predictive", [False, True])
def test_predictions_change_nothing_in_the_sampler(bnr, V, n, form, predictive):
    X, y = _toy(2, V, n)
    Xn = _new(2, 37, X.shape[1])
    C_, sweeps = 7, 16
    got, counts = [], []
    for on in (False, True):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=8, trace_rows=sweeps + 1, trace_full_chains=1,
                        gamma_mode=form) as eng:
            if on:
                eng.set_predictors(Xn, sweeps + 1, predictive=predictive)
            eng.set_moment_window(1, sweeps)
            eng.init_state()
            eng.run(sweeps)
            got.append(_sampler_outputs(eng, C_, sweeps + 1))
            counts.append((eng.launch_count(), eng.chain_groups))
    _same(got[0], got[1])
    # two kernels per sweep and chain group (k_xmma of X_new gamma, k_pred_record), nothing else
    (off, g), (on_, g2) = counts
    assert g == g2 and on_ - off == 2 * sweeps * g


@pytest.mark.parametrize("V,n,form", FORMS)
def test_predictions_do_not_depend_on_grouping_or_graphs(bnr, V, n, form):
    X, y = _toy(3, V, n)
    Xn = _new(3, 37, X.shape[1])
    C_, cap = 7, 14
    ref = None
    for groups, runs in ((1, [13]), (2, [1, 12]), (3, [2, 1, 4, 3, 3]), (2, [1] * 13)):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=9, chain_groups=groups, gamma_mode=form) as eng:
            eng.set_predictors(Xn, cap, predictive=True)
            eng.init_state()
            for r in runs:
                eng.run(r)
            P = np.stack([eng.prediction_trace(c, 0, cap) for c in range(C_)])
        if ref is None:
            ref = P
        else:
            np.testing.assert_array_equal(P, ref, err_msg="groups %d runs %s" % (groups, runs))


def test_predictive_noise_is_standard_normal_and_reproducible(bnr):
    from scipy import stats
    X, y = _toy(4)
    Xn = _new(4, 50, X.shape[1])
    C_, sweeps = 6, 60
    P = {}
    for mode in ("mean", "pred", "pred"):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=12, trace_rows=sweeps + 1, trace_full_chains=C_) as eng:
            eng.set_predictors(Xn, sweeps + 1, predictive=mode == "pred")
            eng.init_state()
            eng.run(sweeps)
            Pm = np.stack([eng.prediction_trace(c, 0, sweeps + 1) for c in range(C_)])
            tau2 = np.stack([eng.get_trace(c, "tau2", 0, sweeps + 1)[:, 0, 0] for c in range(C_)])
        if mode in P:
            np.testing.assert_array_equal(Pm, P[mode])        # run to run
        P[mode] = Pm
    z = ((P["pred"] - P["mean"]) / np.sqrt(tau2)[:, :, None]).ravel()
    assert stats.kstest(z, "norm").pvalue > 1e-3


def _fit_predict(bnr, X, y, R, Xn, mode=0, num_chains=3, seed=21, n_devices=1, **kw):
    """bnr_fit_predict through ctypes, returning the result's info, its prediction summary and every chain's retained
    prediction rows (read back per handle and chain)."""
    from bnr_b200 import capi
    L = bnr.lib()
    Xf = np.asfortranarray(X, dtype=np.float64)
    yv = np.ascontiguousarray(y, dtype=np.float64)
    Xp = np.asfortranarray(Xn, dtype=np.float64)
    n, q = Xf.shape
    V = int(round((-1 + np.sqrt(1 + 8 * q)) / 2))
    p = capi.FitParams()
    L.bnr_fit_default_params(C.byref(p))
    p.base.n, p.base.V, p.base.R, p.base.num_chains, p.base.seed = n, V, R, num_chains, seed
    p.nburn, p.nsamples = kw.get("nburn", 0), kw.get("nsamples", 0)
    p.mingen, p.maxgen = kw.get("mingen", 0), kw.get("maxgen", 0)
    p.purge_burn = kw.get("purge_burn", 0) or 0
    p.psrf_cutoff = kw["cutoff"]
    p.return_state, p.n_devices = capi.STATE["none"], n_devices
    res = C.c_void_p()
    rc = L.bnr_fit_predict(C.byref(p), Xf.ctypes.data_as(_DP), yv.ctypes.data_as(_DP), Xp.shape[0],
                           Xp.ctypes.data_as(_DP), mode, C.byref(res))
    if rc != 0:
        raise capi.BnrError(rc, L.bnr_fit_last_error().decode())
    try:
        info = capi.FitInfo()
        capi.check_fit(L.bnr_fit_get_info(res, C.byref(info)))
        m = Xp.shape[0]
        mean, lo, hi = np.empty(m), np.empty(m), np.empty(m)
        rc = L.bnr_fit_prediction(res, mean.ctypes.data_as(_DP), lo.ctypes.data_as(_DP), hi.ctypes.data_as(_DP))
        if rc == -4:                                  # too few pooled draws for the ranks of the interval
            mean = lo = hi = None
        else:
            capi.check_fit(rc)
        draws = []
        b, s = int(info.burn_in), int(info.sampled)
        for d in range(info.n_devices):
            h = C.c_void_p()
            capi.check_fit(L.bnr_fit_handle(res, d, C.byref(h)))
            for c in range(num_chains):
                out = np.empty(s * m)
                capi.check(L.bnr_get_prediction_trace(h, c, b, b + s, out.ctypes.data_as(_DP)))
                draws.append(out.reshape((s, m), order="F"))
        return info, (mean, lo, hi), draws
    finally:
        L.bnr_fit_free(res)


CASES = [
    dict(nburn=40, nsamples=30), dict(nburn=40, nsamples=30, purge_burn=10), dict(nburn=20, nsamples=30),
    dict(nburn=24, nsamples=8, purge_burn=4), dict(nburn=30, nsamples=21, purge_burn=5), dict(nburn=12, nsamples=50, purge_burn=4),
    dict(mingen=40, maxgen=200), dict(mingen=10, maxgen=45), dict(mingen=14, maxgen=60, purge_burn=3),
]


@pytest.mark.parametrize("kw", CASES)
@pytest.mark.parametrize("cutoff", [1.02, 1e9])
def test_pooled_predictions_follow_the_row_bookkeeping(bnr, kw, cutoff):
    X, y = _toy(5)
    Xn = _new(5, 37, X.shape[1])
    C_, R, seed, smax = 3, 3, 21, 420
    with bnr.Engine(X, y, R, num_chains=C_, seed=seed, trace_rows=smax + 1, trace_full_chains=C_) as eng:
        eng.init_state()
        eng.run(smax)
        G = np.stack([eng.get_trace(c, "gamma", 0, smax + 1)[:, :, 0] for c in range(C_)])
        Xi = np.stack([eng.get_trace(c, "xi", 0, smax + 1)[:, :, 0] for c in range(C_)])
        Mu = np.stack([eng.get_trace(c, "mu", 0, smax + 1)[:, 0, 0] for c in range(C_)])

    def draw(c, s):
        return Xi[c, s], G[c, s]

    try:
        if "mingen" in kw:
            want = PL.generate_samples_dbl(draw, C_, kw["mingen"], kw["maxgen"], cutoff, kw.get("purge_burn"))
        else:
            want = PL.generate_samples(draw, C_, kw["nburn"], kw["nsamples"], kw["nburn"] + kw["nsamples"], cutoff,
                                       kw.get("purge_burn"))
    except IndexError:
        with pytest.raises(bnr.BnrError, match="BoundsError"):
            _fit_predict(bnr, X, y, R, Xn, num_chains=C_, seed=seed, cutoff=cutoff, **kw)
        return
    info, (mean, lo, hi), draws = _fit_predict(bnr, X, y, R, Xn, num_chains=C_, seed=seed, cutoff=cutoff, **kw)
    b, s = int(info.burn_in), int(info.sampled)
    assert (b, s) == (want["burn_in"], want["sampled"])
    expect = []
    for c in range(C_):
        sw = want["rows"][c][b:b + s]
        assert None not in sw
        expect.append(Mu[c, sw][:, None] + G[c, sw] @ Xn.T)
    expect = np.concatenate(expect)
    pooled = np.concatenate(draws)
    scale = np.abs(G).max() * np.abs(Xn).sum(axis=1).max() + np.abs(Mu).max()
    np.testing.assert_allclose(np.sort(pooled, axis=0), np.sort(expect, axis=0), rtol=0, atol=1e-12 * scale)
    N = pooled.shape[0]
    lw, up = int(np.rint(N * 0.025)), int(np.rint(N * 0.975))
    if lw < 1:
        assert mean is None
        return
    ps = np.sort(pooled, axis=0)
    np.testing.assert_array_equal(lo, ps[lw - 1])
    np.testing.assert_array_equal(hi, ps[up - 1])
    np.testing.assert_allclose(mean, pooled.mean(axis=0), rtol=1e-13, atol=1e-13 * scale)


def test_fit_keyword_and_predict_table(bnr):
    """Fit(..., X_new=) runs bnr_fit_predict on networks vectorised like X; Predict rounds what the GPU reduced."""
    rng = np.random.default_rng(6)
    V, n, m = 6, 40, 9
    nets = rng.normal(size=(n, V, V))
    nets = nets + nets.transpose(0, 2, 1)
    new = rng.normal(size=(m, V, V))
    new = new + new.transpose(0, 2, 1)
    y = rng.normal(size=n)
    kw = dict(nburn=40, nsamples=30, num_chains=3, seed=5, filename=None, psrf_cutoff=1e9)
    res = bnr.Fit(nets, y, 3, X_new=new, **kw)
    pr = res.extra["prediction"]
    assert pr["m"] == m and not pr["predictive"] and pr["interval"] == 95
    assert (pr["lower"] <= pr["mean"]).all() and (pr["mean"] <= pr["upper"]).all()
    t = bnr.Predict(res)
    np.testing.assert_array_equal(t.table["estimate"], np.round(pr["mean"], 3))
    np.testing.assert_array_equal(t.table["sample"], np.arange(1, m + 1))
    plain = bnr.Fit(nets, y, 3, **kw)
    np.testing.assert_array_equal(plain.rhatγ.γ, res.rhatγ.γ)
    np.testing.assert_array_equal(plain.state["gamma"], res.state["gamma"])
    assert "prediction" not in plain.extra
    wide = bnr.Fit(nets, y, 3, X_new=new, predictive=True, **kw)
    assert wide.extra["prediction"]["predictive"]
    np.testing.assert_array_equal(wide.state["gamma"], res.state["gamma"])
    assert np.mean(wide.extra["prediction"]["upper"] - wide.extra["prediction"]["lower"]) > np.mean(pr["upper"] - pr["lower"])


@pytest.mark.parametrize("exchange", ["nccl", "peer"])
def test_two_devices_equal_one_device(bnr, exchange, monkeypatch):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    if exchange == "peer":
        monkeypatch.setenv("BNR_EXCHANGE", "peer")
    X, y = _toy(8)
    Xn = _new(8, 37, X.shape[1])
    for kw in (dict(nburn=60, nsamples=40, cutoff=1e9), dict(mingen=40, maxgen=120, cutoff=0.0)):
        for mode in (0, 1):
            two = _fit_predict(bnr, X, y, 3, Xn, mode, num_chains=3, n_devices=2, seed=17, **kw)
            one = _fit_predict(bnr, X, y, 3, Xn, mode, num_chains=6, n_devices=1, seed=17, **kw)
            assert two[0].n_devices == 2 and two[0].total_chains == 6
            _same(two[1], one[1])
            _same(two[2], one[2])


def test_switching_predictions_off_and_impossible_tables(bnr):
    X, y = _toy(9)
    Xn = _new(9, 20, X.shape[1])
    C_ = 4
    states, counts = [], []
    for had in (False, True):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=30) as eng:
            if had:
                eng.set_predictors(Xn, 50)
            eng.init_state()
            eng.run(6)
            eng.set_predictors(None)
            c0 = eng.launch_count()
            eng.run(8)
            states.append([eng.get_state_dict(c) for c in range(C_)])
            counts.append(eng.launch_count() - c0)
            if had:
                with pytest.raises(bnr.BnrError):
                    eng.prediction_trace(0, 0, 1)
    _same(states[0], states[1])
    assert counts[0] == counts[1]
    # a fit whose prediction tables cannot exist is refused before its first sweep
    big = _new(10, 20000, X.shape[1])
    with pytest.raises(bnr.BnrError) as ei:
        _fit_predict(bnr, X, y, 3, big, nburn=2_000_000, nsamples=10, cutoff=1e9)
    assert ei.value.code == -3 and "bytes" in str(ei.value)
