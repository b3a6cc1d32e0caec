"""K-fold cross-validation without a GPU: the default folds, the host arithmetic of BNRKFold and Compare on K-fold
results, and the argument refusals of bnr_fit_kfold (all checked before any device call)."""
import ctypes as C

import numpy as np
import pytest

_DP = C.POINTER(C.c_double)


def test_default_folds_are_balanced_deterministic_and_one_based(bnr):
    for n, K in ((40, 10), (37, 5), (1000, 3), (7, 7)):
        f = bnr.kfold_split(n, K, 123)
        assert f.shape == (n,) and f.min() == 1 and f.max() == K
        sizes = np.bincount(f, minlength=K + 1)[1:]
        assert sizes.max() - sizes.min() <= 1
        np.testing.assert_array_equal(f, bnr.kfold_split(n, K, 123))
        perm = np.random.default_rng(123).permutation(n)
        want = np.empty(n, dtype=np.int64)
        want[perm] = np.arange(n) % K + 1
        np.testing.assert_array_equal(f, want)
    assert not np.array_equal(bnr.kfold_split(50, 5, 1), bnr.kfold_split(50, 5, 2))
    with pytest.raises(ValueError, match="2 <= K <= n"):
        bnr.kfold_split(5, 1, 0)
    with pytest.raises(ValueError, match="2 <= K <= n"):
        bnr.kfold_split(5, 6, 0)


def _kf(bnr, rng, n, folds, y, shift=0.0):
    return bnr.BNRKFold(rng.normal(-1.2 + shift, 0.4, size=n), folds, y, 800, np.full(folds.max(), 1.01), 50, 100)


def test_kfold_estimates_match_numpy(bnr):
    rng = np.random.default_rng(1)
    n = 60
    folds = bnr.kfold_split(n, 6, 9)
    r = _kf(bnr, rng, n, folds, np.zeros(n))
    e = r.pointwise["elpd_kfold"]
    assert r.estimates["elpd_kfold"][0] == pytest.approx(e.sum(), rel=1e-14)
    assert r.estimates["elpd_kfold"][1] == pytest.approx(np.sqrt(n * np.var(e, ddof=1)), rel=1e-14)
    assert r.estimates["kfoldic"][0] == pytest.approx(-2 * e.sum(), rel=1e-14)
    assert r.estimates["kfoldic"][1] == pytest.approx(2 * r.estimates["elpd_kfold"][1], rel=1e-14)
    np.testing.assert_array_equal(r.pointwise["kfoldic"], -2 * e)
    assert r.K == 6 and r.n == n and r.draws == 800
    text = repr(r)
    assert "Based on 6-fold cross-validation." in text and "elpd_kfold" in text and "kfoldic" in text


def test_compare_ranks_kfold_results_and_refuses_mixtures(bnr):
    rng = np.random.default_rng(2)
    n = 50
    y = rng.normal(size=n)
    folds = bnr.kfold_split(n, 5, 3)
    a, b, c = _kf(bnr, rng, n, folds, y, -0.2), _kf(bnr, rng, n, folds, y, 0.1), _kf(bnr, rng, n, folds, y, 0.0)
    cmp = bnr.Compare(a, b, c, names=["A", "B", "C"])
    t = cmp.table
    assert cmp.columns == ("elpd_diff", "se_diff", "elpd_kfold", "se_elpd_kfold", "kfoldic", "se_kfoldic")
    want = sorted(zip("ABC", (a, b, c)), key=lambda p: -p[1].estimates["elpd_kfold"][0])
    assert t["model"] == [w[0] for w in want]
    best = want[0][1].pointwise["elpd_kfold"]
    for i, (_, r) in enumerate(want):
        d = r.pointwise["elpd_kfold"] - best
        assert t["elpd_diff"][i] == pytest.approx(d.sum(), rel=1e-13, abs=1e-13)
        assert t["se_diff"][i] == pytest.approx(np.sqrt(n) * np.std(d, ddof=1), rel=1e-13, abs=1e-13)
        assert t["elpd_kfold"][i] == pytest.approx(r.pointwise["elpd_kfold"].sum(), rel=1e-14)
        assert t["se_elpd_kfold"][i] == pytest.approx(r.estimates["elpd_kfold"][1], rel=1e-14)
        assert t["kfoldic"][i] == pytest.approx(-2 * r.pointwise["elpd_kfold"].sum(), rel=1e-14)
        assert t["se_kfoldic"][i] == pytest.approx(2 * r.estimates["elpd_kfold"][1], rel=1e-14)
    assert t["elpd_diff"][0] == 0.0 and t["se_diff"][0] == 0.0
    assert "se_elpd_kfold" in repr(cmp)
    # a PSIS-LOO fit
    class R:
        pass
    lo = R()
    lo.extra = dict(loo=dict(pointwise=dict(elpd_loo=np.zeros(n), p_loo=np.zeros(n), pareto_k=np.zeros(n),
                                            elpd_waic=np.zeros(n), p_waic=np.zeros(n)), draws=800, y=y))
    with pytest.raises(ValueError, match="cannot mix"):
        bnr.Compare(a, lo)
    with pytest.raises(ValueError, match="same folds"):
        bnr.Compare(a, _kf(bnr, rng, n, bnr.kfold_split(n, 5, 4), y))
    with pytest.raises(ValueError, match="same responses"):
        bnr.Compare(a, _kf(bnr, rng, n, folds, y + 1.0))


def test_kfold_refuses_fit_only_keywords(bnr):
    X = np.random.default_rng(0).normal(size=(12, 10))
    y = np.zeros(12)
    for kw in (dict(X_new=X[:2]), dict(predictive=True), dict(loo=True), dict(ess_max_lag=5)):
        with pytest.raises(ValueError, match="KFold does not take"):
            bnr.KFold(X, y, 2, K=3, x_transform=False, **kw)
    with pytest.raises(TypeError, match="unexpected"):
        bnr.KFold(X, y, 2, K=3, x_transform=False, nsamplez=3)
    # an explicit K must agree with the folds given
    with pytest.raises(ValueError, match="K = 5 disagrees"):
        bnr.KFold(X, y, 2, K=5, folds=np.arange(12) % 4 + 1, x_transform=False)


def test_fit_kfold_refuses_bad_arguments(bnr):
    from bnr_b200 import capi
    L = bnr.lib()
    n, V = 12, 4
    q = V * (V + 1) // 2
    X = np.zeros(n * q)
    y = np.zeros(n)
    out = np.empty(q)

    def call(folds, K, **kw):
        p = capi.FitParams()
        L.bnr_fit_default_params(C.byref(p))
        p.base.n, p.base.V, p.base.R, p.base.num_chains = n, V, 2, 2
        p.nburn, p.nsamples = 4, 4
        for k, v in kw.items():
            setattr(p, k, v)
        f = np.ascontiguousarray(folds, dtype=np.int32)
        res = C.c_void_p()
        rc = L.bnr_fit_kfold(C.byref(p), X.ctypes.data_as(_DP), y.ctypes.data_as(_DP), K,
                             f.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(res))
        return rc, L.bnr_fit_last_error().decode()

    good = np.arange(n) % 3 + 1
    assert call(good, 1) == (-1, "K-fold cross-validation needs K >= 2 folds")
    bad = good.copy()
    bad[4] = 4
    rc, msg = call(bad, 3)
    assert rc == -1 and "fold label 4 of observation 5" in msg
    bad[4] = 0
    assert call(bad, 3)[0] == -1
    rc, msg = call(np.where(good == 2, 1, good), 3)
    assert rc == -1 and "fold 2 holds no observation" in msg
    rc, msg = call(good, 3, ext_world=2, ext_rank=0)
    assert rc == -1 and "ext_world" in msg
    rc, msg = call(good, 3, ess_max_lag=7)
    assert rc == -1 and "ess_max_lag" in msg
    # accessors on a missing result, and the handle entry points without a handle
    assert L.bnr_fit_kfold_pointwise(None, out.ctypes.data_as(_DP)) == -1
    assert L.bnr_fit_kfold_rhat(None, 0, out.ctypes.data_as(_DP), out.ctypes.data_as(_DP)) == -1
    assert L.bnr_set_heldout(None, 2, out.ctypes.data_as(_DP), out.ctypes.data_as(_DP), 4) == -1
    assert L.bnr_lpd_summary(0, None, 10, 3, out.ctypes.data_as(_DP)) == -1
    assert L.bnr_lpd_summary(0, C.c_void_p(256), 0, 3, out.ctypes.data_as(_DP)) == -1
