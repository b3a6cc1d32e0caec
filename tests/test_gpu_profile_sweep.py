"""bnr_profile_sweep runs the sweep that eager sweeps run (enqueue_sweep), with CUDA events between its phases: a
profiled sweep leaves every chain's state, trace row, prediction row and log-likelihood row bit-identical to an
ordinary eager sweep, and its eight phase times are finite and non-negative."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _toy(V, n):
    rng = np.random.default_rng(V + n)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.7)
    y = 1.0 + X[:, :5].sum(axis=1) + rng.normal(0, 1.5, size=n)
    Xn = rng.normal(size=(11, q)) * (rng.random((11, q)) < 0.7)
    return X, y, Xn


# (V, n, gamma form), three factored panels each: the q-form, the n-form on the FP64 SYRK, the n-form on the INT8 Gram
# path (qp >= 1024)
FORMS = [(24, 200, "qform"), (30, 300, "nform"), (45, 300, "nform")]


@pytest.mark.parametrize("V,n,form", FORMS)
def test_a_profiled_sweep_is_the_eager_sweep(bnr, V, n, form):
    from bnr_b200.capi import VAR
    X, y, Xn = _toy(V, n)
    C_, sweeps, profiled = 4, 4, 2
    rows = sweeps + 1
    got, phases = [], None
    for profile in (False, True):
        with bnr.Engine(X, y, 3, num_chains=C_, seed=6, trace_rows=rows, trace_full_chains=C_,
                        gamma_mode=form) as eng:
            assert eng.gamma_mode == form
            eng.set_predictors(Xn, rows, predictive=True)
            eng.set_loglik(rows)
            eng.init_state()
            for k in range(sweeps):
                if profile and k == profiled:
                    phases = eng.profile_sweep()
                else:
                    eng.run(1)
            assert eng.iteration == sweeps and eng.trace_row == rows
            out = []
            for c in range(C_):
                out.append(eng.get_state_dict(c))
                out.append({v: eng.get_trace(c, v, 0, rows) for v in VAR})
                out.append(eng.prediction_trace(c, 0, rows))
                out.append(eng.loglik_trace(c, 0, rows))
            got.append(out)
    for a, b in zip(*got):
        if isinstance(a, dict):
            assert a.keys() == b.keys()
            for k in a:
                np.testing.assert_array_equal(a[k], b[k], err_msg=k)
        else:
            assert np.isfinite(b).all()                  # every prediction / log-likelihood row was written
            np.testing.assert_array_equal(a, b)
    assert tuple(phases) == bnr.Engine.PHASES
    t = np.array(list(phases.values()))
    assert np.isfinite(t).all() and (t >= 0).all(), phases
