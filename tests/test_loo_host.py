"""PSIS-LOO and WAIC without a GPU: the NumPy restatement (oracle/loo.py) against known answers -- the GPD fit against
scipy's generalised Pareto, PSIS-LOO against the exact leave-one-out densities of a conjugate normal model, the Pareto k
of a high-leverage outlier, WAIC against its formula -- and the host arithmetic of Loo / Compare, and the argument
refusals of the new C entry points."""
import ctypes as C
import warnings

import numpy as np
import pytest
from scipy import stats
from scipy.special import logsumexp

from oracle import loo as OL

_DP = C.POINTER(C.c_double)


@pytest.mark.parametrize("c", [-0.3, 0.2, 0.6])
def test_gpdfit_recovers_the_shape(c):
    x = np.sort(stats.genpareto.rvs(c, scale=1.5, size=20000, random_state=np.random.default_rng(int(10 * c) + 7)))
    k, sigma = OL.gpdfit(x)
    assert abs(k - c) < 0.05
    assert abs(sigma / 1.5 - 1.0) < 0.1


def _conjugate(seed, n=60, p=3, sigma=1.0, tau0=2.0, S=4000, outlier=False):
    """y = X beta + N(0, sigma^2), beta ~ N(0, tau0^2 I), sigma known: exact posterior draws and exact LOO densities."""
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, p))
    y = X @ np.array([1.0, -0.5, 0.25]) + sigma * rng.normal(size=n)
    if outlier:
        X = np.vstack([X, np.full((1, p), 6.0)])
        y = np.append(y, -40.0)
        n += 1

    def post(Xs, ys):
        Vinv = Xs.T @ Xs / sigma ** 2 + np.eye(p) / tau0 ** 2
        V = np.linalg.inv(Vinv)
        return V @ Xs.T @ ys / sigma ** 2, V

    m, V = post(X, y)
    beta = rng.multivariate_normal(m, V, size=S)
    ll = OL.loglik(y[None, :], 0.0, beta @ X.T, sigma ** 2)
    exact = np.empty(n)
    for i in range(n):
        keep = np.arange(n) != i
        mi, Vi = post(X[keep], y[keep])
        exact[i] = stats.norm.logpdf(y[i], X[i] @ mi, np.sqrt(sigma ** 2 + X[i] @ Vi @ X[i]))
    return ll, exact


def test_psis_loo_matches_the_exact_leave_one_out_densities():
    ll, exact = _conjugate(1)
    got = OL.loo_pointwise(ll)
    assert np.all(got["pareto_k"] < 0.5)
    # Monte Carlo error of each elpd_i: the standard error of the self-normalised importance sampling estimate
    w = np.exp(ll.min(axis=0) - ll)
    r = np.exp(ll - ll.max(axis=0))
    mcse = np.sqrt(np.var(w * r, axis=0) / ll.shape[0]) / np.mean(w * r, axis=0) + np.std(w, axis=0) / np.mean(w, axis=0) / np.sqrt(ll.shape[0])
    assert np.all(np.abs(got["elpd_loo"] - exact) < 4 * mcse + 1e-3)
    assert abs(got["elpd_loo"].sum() - exact.sum()) < 0.1


def test_a_high_leverage_outlier_gets_a_large_pareto_k():
    ll, _ = _conjugate(2, outlier=True)
    k = OL.loo_pointwise(ll)["pareto_k"]
    assert k[-1] > 0.7
    assert np.median(k[:-1]) < 0.5


def test_waic_is_its_formula():
    rng = np.random.default_rng(3)
    ll = rng.normal(-1.0, 0.4, size=(500, 7)) + rng.normal(size=7)
    got = OL.loo_pointwise(ll)
    lpd = np.log(np.mean(np.exp(ll), axis=0))
    pw = np.sum((ll - ll.mean(axis=0)) ** 2, axis=0) / (ll.shape[0] - 1)
    np.testing.assert_allclose(got["p_waic"], pw, rtol=1e-12)
    np.testing.assert_allclose(got["elpd_waic"], lpd - pw, rtol=1e-12)
    np.testing.assert_allclose(got["p_loo"], lpd - got["elpd_loo"], rtol=1e-10, atol=1e-12)


def test_small_and_degenerate_columns():
    ll = np.random.default_rng(4).normal(size=(12, 2))
    ll[:, 1] = -0.7
    got = OL.loo_pointwise(ll)
    assert OL.tail_len(12) < 5 and np.isinf(got["pareto_k"]).all()
    # without smoothing the weights are the raw ratios: elpd_loo = -log mean exp(-ll)
    np.testing.assert_allclose(got["elpd_loo"], -(logsumexp(-ll, axis=0) - np.log(12)), rtol=1e-12)


def _fake(pointwise, draws, y):
    class R:
        pass
    r = R()
    r.extra = dict(loo=dict(pointwise=pointwise, draws=draws, y=np.asarray(y, dtype=np.float64)))
    return r


def _pw(rng, n, shift=0.0, k=None):
    e = rng.normal(-1.0 + shift, 0.3, size=n)
    p = np.abs(rng.normal(0.1, 0.05, size=n))
    return dict(elpd_loo=e, p_loo=p, pareto_k=rng.uniform(0, 0.4, n) if k is None else k,
                elpd_waic=e + 0.01, p_waic=p - 0.01)


def test_loo_estimates_and_warning(bnr):
    rng = np.random.default_rng(5)
    n, S = 40, 8000
    k = rng.uniform(0, 0.4, n)
    k[[3, 17]] = [0.75, np.inf]
    pw = _pw(rng, n, k=k)
    res = _fake(pw, S, np.zeros(n))
    with pytest.warns(UserWarning, match="2 of 40 Pareto k"):
        lo = bnr.Loo(res)
    for name, arr in (("elpd_loo", pw["elpd_loo"]), ("p_loo", pw["p_loo"]), ("elpd_waic", pw["elpd_waic"]),
                      ("p_waic", pw["p_waic"])):
        e, se = lo.estimates[name]
        assert e == pytest.approx(arr.sum(), rel=1e-14)
        assert se == pytest.approx(np.sqrt(n * np.var(arr, ddof=1)), rel=1e-14)
    assert lo.estimates["looic"][0] == pytest.approx(-2 * pw["elpd_loo"].sum(), rel=1e-14)
    assert lo.estimates["looic"][1] == pytest.approx(2 * lo.estimates["elpd_loo"][1], rel=1e-14)
    assert lo.estimates["waic"][0] == pytest.approx(-2 * pw["elpd_waic"].sum(), rel=1e-14)
    assert lo.k_threshold == pytest.approx(min(1 - 1 / np.log10(S), 0.7)) and lo.n_high_k == 2
    assert "Warning: 2 of 40" in repr(lo) and "elpd_loo" in repr(lo)
    # few draws: the threshold follows 1 - 1 / log10(S)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        small = bnr.Loo(_fake(pw, 100, np.zeros(n)))
    assert small.k_threshold == pytest.approx(0.5)
    with pytest.raises(ValueError, match="loo=True"):
        bnr.Loo(_fake(pw, S, np.zeros(n)).__class__())
    with pytest.raises(ValueError, match="at least 2"):
        bnr.Loo(_fake(None, 1, np.zeros(n)))


def test_compare_ranks_and_differences(bnr):
    rng = np.random.default_rng(6)
    n = 50
    y = rng.normal(size=n)
    a, b, c = _pw(rng, n, -0.2), _pw(rng, n, 0.1), _pw(rng, n, 0.0)
    t = bnr.Compare(_fake(a, 4000, y), _fake(b, 4000, y), _fake(c, 4000, y), names=["A", "B", "C"]).table
    assert t["model"] == ["B", "C", "A"]
    best = b["elpd_loo"]
    for i, pw in enumerate((b, c, a)):
        d = pw["elpd_loo"] - best
        assert t["elpd_diff"][i] == pytest.approx(d.sum(), rel=1e-13, abs=1e-13)
        assert t["se_diff"][i] == pytest.approx(np.sqrt(n) * np.std(d, ddof=1), rel=1e-13, abs=1e-13)
        assert t["elpd_loo"][i] == pytest.approx(pw["elpd_loo"].sum(), rel=1e-14)
        assert t["se_elpd_loo"][i] == pytest.approx(np.sqrt(n * np.var(pw["elpd_loo"], ddof=1)), rel=1e-14)
        assert t["looic"][i] == pytest.approx(-2 * pw["elpd_loo"].sum(), rel=1e-14)
    assert t["elpd_diff"][0] == 0.0 and t["se_diff"][0] == 0.0
    assert (np.diff(t["elpd_loo"]) <= 0).all()
    with pytest.raises(ValueError, match="same responses"):
        bnr.Compare(_fake(a, 4000, y), _fake(b, 4000, y + 1.0))
    with pytest.raises(ValueError, match="two fits"):
        bnr.Compare(_fake(a, 4000, y))


def test_loo_entry_points_refuse_bad_arguments(bnr):
    from bnr_b200 import capi
    L = bnr.lib()
    out = np.empty(3)
    assert L.bnr_loo_summary(0, None, 10, 3, *([out.ctypes.data_as(_DP)] * 5)) == -1
    assert L.bnr_loo_summary(0, C.c_void_p(256), 1, 3, *([out.ctypes.data_as(_DP)] * 5)) == -1
    assert L.bnr_set_loglik(None, 10) == -1
    assert L.bnr_get_loglik_trace(None, 0, 0, 1, out.ctypes.data_as(_DP)) == -1
    assert L.bnr_export_loglik(None, 0, 1, C.c_void_p(256)) == -1
    assert L.bnr_fit_loo_pointwise(None, *([out.ctypes.data_as(_DP)] * 5)) == -1
    p = capi.FitParams()
    L.bnr_fit_default_params(C.byref(p))
    res = C.c_void_p()
    assert L.bnr_fit_loo(C.byref(p), out.ctypes.data_as(_DP), out.ctypes.data_as(_DP), -1, None, 0, C.byref(res)) == -1
    assert L.bnr_fit_loo(C.byref(p), out.ctypes.data_as(_DP), out.ctypes.data_as(_DP), 2, None, 0, C.byref(res)) == -1
    assert L.bnr_fit_loo(C.byref(p), out.ctypes.data_as(_DP), out.ctypes.data_as(_DP), 0, None, 7, C.byref(res)) == -1
