"""Host side of the predictions for new networks: argument refusals of the C entry points (before any CUDA call), X_new
vectorised like X, the pooled rank rule and the Predict table."""
import ctypes as C

import numpy as np
import pytest

_DP = C.POINTER(C.c_double)
EINVAL, ESTATE, ENODEV = -1, -4, -5


def _fit_params(bnr):
    from bnr_b200 import capi
    p = capi.FitParams()
    bnr.lib().bnr_fit_default_params(C.byref(p))
    p.base.n, p.base.V, p.base.R, p.base.num_chains = 4, 4, 2, 2
    p.nburn, p.nsamples = 10, 10
    return p


def test_prediction_entry_points_refuse_bad_arguments(bnr):
    L = bnr.lib()
    x = np.zeros(40)
    out = np.zeros(40)
    fake = C.c_void_p(1)                   # never dereferenced: every call below fails on its arguments first
    assert L.bnr_set_predictors(None, 1, x.ctypes.data_as(_DP), 5, 0) == EINVAL
    assert L.bnr_get_prediction_trace(None, 0, 0, 1, out.ctypes.data_as(_DP)) == EINVAL
    assert L.bnr_export_predictions(None, 0, 1, fake) == EINVAL
    summ = lambda rows, count, m, lo, hi: L.bnr_prediction_summary(0, rows, count, m, lo, hi, None, None, None)
    assert summ(None, 10, 2, 1, 10) == EINVAL
    assert summ(fake, 0, 2, 1, 1) == EINVAL
    assert summ(fake, 10, 0, 1, 10) == EINVAL
    assert summ(fake, 10, 2, 0, 10) == EINVAL
    assert summ(fake, 10, 2, 1, 11) == EINVAL
    p = _fit_params(bnr)
    res = C.c_void_p()
    X, y = np.zeros(40), np.zeros(4)
    fp = lambda m, Xn, mode: L.bnr_fit_predict(C.byref(p), X.ctypes.data_as(_DP), y.ctypes.data_as(_DP), m, Xn, mode,
                                               C.byref(res))
    assert fp(-1, x.ctypes.data_as(_DP), 0) == EINVAL
    assert fp(3, None, 0) == EINVAL
    assert fp(3, x.ctypes.data_as(_DP), 2) == EINVAL
    assert L.bnr_fit_prediction(None, None, None, None) == EINVAL


def test_valid_prediction_calls_without_a_device_are_a_loud_error(bnr):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = bnr.lib()
    assert L.bnr_prediction_summary(0, C.c_void_p(1), 10, 2, 1, 10, None, None, None) == ENODEV
    p = _fit_params(bnr)
    res = C.c_void_p()
    X, y, Xn = np.zeros(40), np.zeros(4), np.zeros(30)
    assert L.bnr_fit_predict(C.byref(p), X.ctypes.data_as(_DP), y.ctypes.data_as(_DP), 3, Xn.ctypes.data_as(_DP), 1,
                             C.byref(res)) == ENODEV


@pytest.mark.parametrize("x_transform", [True, False])
def test_new_networks_are_vectorised_like_X(bnr, x_transform):
    from bnr_b200 import fit
    rng = np.random.default_rng(3)
    V = 5
    nets = rng.normal(size=(7, V, V))
    got = fit._prepare_new(nets if x_transform else bnr.setup_X(nets), x_transform)
    want = np.stack([np.concatenate([a[k:, k] for k in range(V)]) for a in nets])
    np.testing.assert_array_equal(got, want)
    assert fit._prepare_new(None, x_transform) is None


@pytest.mark.parametrize("N", [40, 90, 100, 120, 1000, 64 * 20000, 3 * 30])
@pytest.mark.parametrize("interval", [95, 90, 50])
def test_pooled_ranks_use_julia_rounding(bnr, N, interval):
    from bnr_b200 import fit
    lw, hi = fit._summary_ranks(N, interval)
    a = N * (100 - interval) / 200
    b = N * (1 - (100 - interval) / 200)

    def julia_round(x):                   # ties to even, written out
        f = np.floor(x)
        d = x - f
        return int(f + 1) if d > 0.5 or (d == 0.5 and int(f) % 2 == 1) else int(f)
    assert (lw, hi) == (julia_round(a), julia_round(b))


def _results(bnr, mean, lower, upper, interval=95, predictive=False):
    res = bnr.Results(bnr.Table(), np.zeros(3), np.zeros(6), 10, 10)
    res.extra["prediction"] = dict(interval=interval, mean=mean, lower=lower, upper=upper, predictive=predictive,
                                   m=None if mean is None else len(mean), draws=20)
    return res


def test_predict_table_and_refusals(bnr):
    mean = np.array([1.23456, -0.5, 7.0])
    lower, upper = mean - 1.0004, mean + 2.0006
    t = bnr.Predict(_results(bnr, mean, lower, upper, predictive=True))
    assert isinstance(t, bnr.BNRPrediction) and t.ci_level == 95 and t.predictive
    np.testing.assert_array_equal(t.table["sample"], [1, 2, 3])
    np.testing.assert_array_equal(t.table["estimate"], np.round(mean, 3))
    np.testing.assert_array_equal(t.table["lower_bound"], np.round(lower, 3))
    np.testing.assert_array_equal(t.table["upper_bound"], np.round(upper, 3))
    assert "posterior predictive" in repr(t)
    t2 = bnr.Predict(_results(bnr, mean, lower, upper), digits=1)
    np.testing.assert_array_equal(t2.table["estimate"], np.round(mean, 1))
    with pytest.raises(ValueError, match="X_new"):
        bnr.Predict(bnr.Results(bnr.Table(), np.zeros(3), np.zeros(6), 10, 10))
    with pytest.raises(ValueError, match="interval=95"):
        bnr.Predict(_results(bnr, mean, lower, upper), interval=90)
    with pytest.raises(IndexError, match="BoundsError"):
        bnr.Predict(_results(bnr, None, None, None))
