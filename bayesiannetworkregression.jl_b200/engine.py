"""Thin object wrapper over one libbnr handle (= the chain batch of one GPU)."""
import ctypes as C

import numpy as np

from .capi import lib, check, Params, VAR, COND, AUX, GAMMA_MODE, PRED_MEAN, PRED_PREDICTIVE

_DP = C.POINTER(C.c_double)


def _dp(a):
    return a.ctypes.data_as(_DP)


LOO_FIELDS = ("elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic")


def loo_summary(device, dev_ptr, N, n):
    """bnr_loo_summary on a device table of N draws x n observations: dict of the five pointwise [n] arrays."""
    out = [np.empty(int(n)) for _ in LOO_FIELDS]
    check(lib().bnr_loo_summary(int(device), C.c_void_p(dev_ptr), int(N), int(n), *(_dp(a) for a in out)))
    return dict(zip(LOO_FIELDS, out))


class Engine:
    """`Engine(X, y, R, num_chains=...)` uploads the n x q design matrix once and owns every chain's state on
    the device.  X may be C- or F-ordered; it is passed to the library column-major like the reference's
    Matrix{Float64} (src/gibbs.jl:917)."""

    def __init__(self, X, y, R, num_chains=2, seed=0, chain_offset=0, device=0, trace_rows=0,
                 trace_full_chains=1, trace_gamma_xi_all=True, eta=1.01, zeta=1.0, iota=1.0, a_delta=1.0,
                 b_delta=1.0, nu=10.0, gig_inject_len=64, gamma_mode="auto", chain_groups=0, trace_gamma_xi_chains=0):
        X = np.asarray(X, dtype=np.float64)
        y = np.ascontiguousarray(y, dtype=np.float64)
        if X.ndim != 2 or y.ndim != 1 or X.shape[0] != y.shape[0]:
            raise ValueError("X must be n x q and y of length n")
        n, q = X.shape
        V = int(round((-1 + np.sqrt(1 + 8 * q)) / 2))
        if V * (V + 1) // 2 != q:
            raise ValueError("q = %d is not V(V+1)/2 for an integer V" % q)
        self.n, self.q, self.V, self.R, self.C = n, q, V, int(R), int(num_chains)
        self._L = lib()
        p = Params()
        self._L.bnr_default_params(C.byref(p))
        p.n, p.V, p.R, p.num_chains = n, V, int(R), int(num_chains)
        p.chain_offset, p.device = int(chain_offset), int(device)
        p.trace_rows, p.trace_full_chains = int(trace_rows), int(trace_full_chains)
        p.trace_gamma_xi_all = 1 if trace_gamma_xi_all else 0
        p.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        p.eta, p.zeta, p.iota, p.a_delta, p.b_delta, p.nu = eta, zeta, iota, a_delta, b_delta, float(nu)
        p.gig_inject_len = int(gig_inject_len)
        p.gamma_mode = GAMMA_MODE[gamma_mode] if isinstance(gamma_mode, str) else int(gamma_mode)
        p.chain_groups = int(chain_groups)
        p.trace_gamma_xi_chains = int(trace_gamma_xi_chains)
        self.params = p
        self.pred_m = 0
        self.device = int(device)
        self.trace_rows = int(trace_rows)
        Xf = np.asfortranarray(X)
        h = C.c_void_p()
        check(self._L.bnr_create(C.byref(p), _dp(Xf), _dp(y), C.byref(h)))
        self._h = h

    # -- life cycle ------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.bnr_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    @property
    def chain_groups(self):
        v = C.c_int32()
        check(self._L.bnr_chain_groups(self._h, C.byref(v)))
        return int(v.value)

    @property
    def gamma_mode(self):
        """"nform" (the reference's n x n Bhattacharya draw) or "qform" (q x q precision Cholesky)."""
        v = C.c_int32()
        check(self._L.bnr_gamma_mode(self._h, C.byref(v)))
        return {1: "nform", 2: "qform"}[int(v.value)]

    # -- sampling --------------------------------------------------------------------------------------
    def init_state(self):
        check(self._L.bnr_init_state(self._h))

    def run(self, n_iters, sync=True):
        check(self._L.bnr_run(self._h, int(n_iters)))
        if sync:
            self.sync()

    def sync(self):
        check(self._L.bnr_sync(self._h))

    def last_run_ms(self):
        ms = C.c_float()
        check(self._L.bnr_last_run_ms(self._h, C.byref(ms)))
        return float(ms.value)

    @property
    def iteration(self):
        v = C.c_int64()
        check(self._L.bnr_iteration(self._h, C.byref(v)))
        return int(v.value)

    @property
    def trace_row(self):
        v = C.c_int64()
        check(self._L.bnr_get_trace_row(self._h, C.byref(v)))
        return int(v.value)

    @trace_row.setter
    def trace_row(self, row):
        check(self._L.bnr_set_trace_row(self._h, int(row)))

    def copy_trace_rows(self, dst, src, count=1):
        check(self._L.bnr_copy_trace_rows(self._h, int(dst), int(src), int(count)))

    # -- convergence -----------------------------------------------------------------------------------
    def set_moment_window(self, first_sweep, length):
        check(self._L.bnr_set_moment_window(self._h, int(first_sweep), int(length)))

    def set_moment_blocks(self, first_sweep, block_len, nblocks):
        check(self._L.bnr_set_moment_blocks(self._h, int(first_sweep), int(block_len), int(nblocks)))

    def moments_from_blocks(self, first_block, nblocks):
        check(self._L.bnr_moments_from_blocks(self._h, int(first_block), int(nblocks)))

    def moments_from_trace(self, first_row, nrows):
        check(self._L.bnr_moments_from_trace(self._h, int(first_row), int(nrows)))

    def moments_device(self):
        """(device pointer, number of doubles) of [chain][half][xi(V) then gamma(q)][mean, M2]."""
        p = C.c_void_p()
        n = C.c_int64()
        check(self._L.bnr_moments_device(self._h, C.byref(p), C.byref(n)))
        return p.value, int(n.value)

    def moment_half_len(self):
        v = C.c_int64()
        check(self._L.bnr_moment_half_len(self._h, C.byref(v)))
        return int(v.value)

    def rhat(self):
        rx = np.empty(self.V)
        rg = np.empty(self.q)
        check(self._L.bnr_rhat(self._h, _dp(rx), _dp(rg)))
        return rx, rg

    def rhat_from_moments(self, dev_ptr, total_chains, half_len):
        rx = np.empty(self.V)
        rg = np.empty(self.q)
        check(self._L.bnr_rhat_from_moments(self.device, C.c_void_p(dev_ptr), int(total_chains), self.V, self.q,
                                            int(half_len), _dp(rx), _dp(rg)))
        return rx, rg

    def summary(self, chain, first_row, nrows, rank_lo, rank_hi):
        """Device Summary statistics of one chain: (mean gamma, sort(gamma)[rank_lo], sort(gamma)[rank_hi], mean xi);
        ranks are 1-based like the reference's lw / hi (src/gibbs.jl:1221-1236)."""
        gm, gl, gh, xm = np.empty(self.q), np.empty(self.q), np.empty(self.q), np.empty(self.V)
        check(self._L.bnr_summary(self._h, int(chain), int(first_row), int(nrows), int(rank_lo), int(rank_hi),
                                  _dp(gm), _dp(gl), _dp(gh), _dp(xm)))
        return gm, gl, gh, xm

    def ess(self, first_row, nrows, max_lag=255):
        """(ESS of xi, ESS of gamma) over the rows of all local chains (multi-chain Geyer estimator)."""
        ex, eg = np.empty(self.V), np.empty(self.q)
        check(self._L.bnr_ess(self._h, int(first_row), int(nrows), int(max_lag), _dp(ex), _dp(eg)))
        return ex, eg

    def ess_accumulate(self, first_row, nrows, max_lag=255):
        check(self._L.bnr_ess_accumulate(self._h, int(first_row), int(nrows), int(max_lag)))

    def ess_device(self):
        """((acov ptr, count), (chain-mean ptr, count), max_lag) device buffers of the last ess_accumulate."""
        pa, pm = C.c_void_p(), C.c_void_p()
        na, nm = C.c_int64(), C.c_int64()
        lag = C.c_int32()
        check(self._L.bnr_ess_device(self._h, C.byref(pa), C.byref(na), C.byref(pm), C.byref(nm), C.byref(lag)))
        return (pa.value, int(na.value)), (pm.value, int(nm.value)), int(lag.value)

    def export_ess(self, acov_dev_ptr, means_dev_ptr):
        check(self._L.bnr_export_ess(self._h, C.c_void_p(acov_dev_ptr), C.c_void_p(means_dev_ptr)))

    def ess_from_stats(self, acov_ptr, nparts, means_ptr, total_chains, nrows, max_lag, with_lags=False):
        """(ESS xi, ESS gamma) from gathered statistics; with_lags also returns the lags each Geyer sequence consumed
        (max_lag + 1 = not terminated inside the lag budget)."""
        ex, eg = np.empty(self.V), np.empty(self.q)
        lx, lg = np.empty(self.V), np.empty(self.q)
        check(self._L.bnr_ess_from_stats_lags(self.device, C.c_void_p(acov_ptr), int(nparts), C.c_void_p(means_ptr),
                                              int(total_chains), self.V, self.q, int(nrows), int(max_lag),
                                              _dp(ex), _dp(eg), _dp(lx), _dp(lg)))
        return (ex, eg, lx, lg) if with_lags else (ex, eg)

    def ess_stream_begin(self, max_lag, ndraws):
        """Accumulate the ESS statistics of the next `ndraws` sweeps on the device while they run (no traces)."""
        check(self._L.bnr_ess_stream_begin(self._h, int(max_lag), int(ndraws)))
        self._last_ess_rows = int(ndraws)

    def ess_stream_finish(self):
        check(self._L.bnr_ess_stream_finish(self._h))

    def ess_streamed(self):
        """(ESS xi, ESS gamma) of this handle's chains from the streamed statistics (after ess_stream_finish)."""
        (pa, _), (pm, _), lag = self.ess_device()
        return self.ess_from_stats(pa, 1, pm, self.C, self._ess_rows(), lag)

    def _ess_rows(self):
        return self._last_ess_rows

    def export_moments(self, dev_ptr):
        check(self._L.bnr_export_moments(self._h, C.c_void_p(dev_ptr)))

    def launch_count(self):
        v = C.c_int64()
        check(self._L.bnr_launch_count(self._h, C.byref(v)))
        return int(v.value)

    PHASES = ("tau2", "u_xi", "gamma_prep", "syrk", "cholesky", "solves", "xt_gamma_gig", "xg_scalars_record")

    def profile_sweep(self):
        ms = (C.c_float * 8)()
        check(self._L.bnr_profile_sweep(self._h, ms))
        return dict(zip(self.PHASES, [float(x) for x in ms]))

    # -- predictions for new networks ------------------------------------------------------------------
    def set_predictors(self, X_new, rows=0, predictive=False):
        """Record mu + X_new gamma (+ sqrt(tau2) z with predictive=True) for the m rows of X_new (m x q, laid out like
        X) at every recorded row of every chain, in a table of `rows` (>= 1) rows per chain.  X_new=None switches it
        off (rows is then not needed)."""
        if X_new is None:
            check(self._L.bnr_set_predictors(self._h, 0, None, 0, PRED_MEAN))
            self.pred_m = 0
            return
        Xn = np.asfortranarray(X_new, dtype=np.float64)
        if Xn.ndim != 2 or Xn.shape[1] != self.q:
            raise ValueError("X_new must be m x q with q = %d" % self.q)
        check(self._L.bnr_set_predictors(self._h, Xn.shape[0], _dp(Xn), int(rows),
                                         PRED_PREDICTIVE if predictive else PRED_MEAN))
        self.pred_m = Xn.shape[0]

    def prediction_trace(self, chain, first, last):
        """Rows [first, last) of one chain's prediction table as an array of shape (last - first, m)."""
        rows = int(last) - int(first)
        out = np.empty(rows * self.pred_m)
        check(self._L.bnr_get_prediction_trace(self._h, int(chain), int(first), int(last), _dp(out)))
        return out.reshape((rows, self.pred_m), order="F")

    def export_predictions(self, first_row, nrows, dev_ptr):
        """Rows [first_row, first_row + nrows) of every chain into device memory at dev_ptr as [chain][row][m]."""
        check(self._L.bnr_export_predictions(self._h, int(first_row), int(nrows), C.c_void_p(dev_ptr)))

    def prediction_summary(self, dev_ptr, count, m, rank_lo, rank_hi):
        """(mean, sort[rank_lo], sort[rank_hi]) of each of the m columns of `count` rows at a device pointer; ranks are
        1-based."""
        mean, lo, hi = np.empty(m), np.empty(m), np.empty(m)
        check(self._L.bnr_prediction_summary(self.device, C.c_void_p(dev_ptr), int(count), int(m), int(rank_lo),
                                             int(rank_hi), _dp(mean), _dp(lo), _dp(hi)))
        return mean, lo, hi

    # -- pointwise log-likelihood (PSIS-LOO / WAIC) --------------------------------------------------------
    def set_loglik(self, rows):
        """Record log N(y_i | mu + (X gamma)_i, tau2) for every observation i at every recorded row of every chain, in
        a table of `rows` rows per chain (C x rows x n doubles on the device).  rows=0 switches it off."""
        check(self._L.bnr_set_loglik(self._h, int(rows)))

    def loglik_trace(self, chain, first, last):
        """Rows [first, last) of one chain's log-likelihood table as an array of shape (last - first, n)."""
        rows = int(last) - int(first)
        out = np.empty(rows * self.n)
        check(self._L.bnr_get_loglik_trace(self._h, int(chain), int(first), int(last), _dp(out)))
        return out.reshape((rows, self.n), order="F")

    def export_loglik(self, first_row, nrows, dev_ptr):
        """Rows [first_row, first_row + nrows) of every chain into device memory at dev_ptr as [chain][row][n]."""
        check(self._L.bnr_export_loglik(self._h, int(first_row), int(nrows), C.c_void_p(dev_ptr)))

    def loo_summary(self, dev_ptr, N, n):
        """PSIS-LOO and WAIC of N pooled draws x n observations at a device pointer (row-major): a dict of the
        pointwise arrays elpd_loo, p_loo, pareto_k, elpd_waic, p_waic."""
        return loo_summary(self.device, dev_ptr, N, n)

    # -- state / traces in reference layout ------------------------------------------------------------
    def var_shape(self, var):
        R, V, q = self.R, self.V, self.q
        return {"tau2": (1, 1), "u": (R, V), "xi": (V, 1), "gamma": (q, 1), "S": (q, 1), "theta": (1, 1),
                "Delta": (1, 1), "M": (R, R), "mu": (1, 1), "lam": (R, 1), "pi": (R, 3)}[var]

    def get_state(self, chain, var):
        shp = self.var_shape(var)
        out = np.empty(shp[0] * shp[1])
        check(self._L.bnr_get_state(self._h, int(chain), VAR[var], _dp(out)))
        return out.reshape(shp, order="F")

    def set_state(self, chain, var, value):
        shp = self.var_shape(var)
        a = np.asarray(value, dtype=np.float64).reshape(shp, order="F") if np.ndim(value) else \
            np.full(shp, float(value))
        a = np.asfortranarray(a)
        check(self._L.bnr_set_state(self._h, int(chain), VAR[var], _dp(a)))

    def get_state_dict(self, chain):
        d = {k: self.get_state(chain, k) for k in VAR}
        for k in ("tau2", "theta", "Delta", "mu"):
            d[k] = float(d[k][0, 0])
        for k in ("xi", "gamma", "S", "lam"):
            d[k] = d[k][:, 0]
        return d

    def set_state_dict(self, chain, st):
        for k in VAR:
            self.set_state(chain, k, st[k])

    def get_trace(self, chain, var, first, last):
        """Rows [first, last) as an array of shape (last-first, d1, d2), Fortran-ordered exactly like the
        reference's state.<var> (iteration is the fastest index)."""
        shp = self.var_shape(var)
        rows = int(last) - int(first)
        out = np.empty(rows * shp[0] * shp[1])
        check(self._L.bnr_get_trace(self._h, int(chain), VAR[var], int(first), int(last), _dp(out)))
        return out.reshape((rows,) + shp, order="F")

    def status(self):
        s = np.zeros(self.C, dtype=np.int32)
        check(self._L.bnr_status(self._h, s.ctypes.data_as(C.POINTER(C.c_int32))))
        return s

    # -- parity-test hooks -----------------------------------------------------------------------------
    def injection_size(self, for_init=False):
        v = C.c_int64()
        check(self._L.bnr_injection_size(self._h, 1 if for_init else 0, C.byref(v)))
        return int(v.value)

    def set_injection(self, inj):
        if inj is None:
            check(self._L.bnr_set_injection(self._h, None, 0))
            return
        a = np.ascontiguousarray(inj, dtype=np.float64)
        if a.ndim != 2 or a.shape[0] != self.C:
            raise ValueError("injection array must be (num_chains, per_chain)")
        check(self._L.bnr_set_injection(self._h, _dp(a), a.shape[1]))

    def step(self, cond):
        check(self._L.bnr_step(self._h, COND[cond]))

    def finish_sweep(self):
        check(self._L.bnr_finish_sweep(self._h))

    def enable_aux(self, on=True):
        check(self._L.bnr_enable_aux(self._h, 1 if on else 0))

    def get_aux(self, chain, name):
        R, V, q, n = self.R, self.V, self.q, self.n
        if self.gamma_mode == "qform":
            n = q          # G / G_chol are q x q (the precision P), rhs / a4 hold beta = gamma - W
        size = {"tau2_params": 2, "sigma_inv": V * R * R, "sigma_chol": V * R * R, "mu_t": V * R, "log_odds": V,
                "W": q, "G": n * n, "G_chol": n * n, "rhs": n, "a4": n, "chi": q, "theta_params": 2,
                "delta_params": 2, "m_params": 1 + 2 * R * R, "mu_params": 2, "lambda_logw": 3 * R,
                "lambda_weights": 3 * R, "pi_alpha": 3 * R, "gig_used": q}[name]
        out = np.empty(size)
        check(self._L.bnr_get_aux(self._h, int(chain), AUX[name], _dp(out), size))
        return out

    def test_chol_jitter(self, A):
        """(matrix that factored, lower factor, status bits) of the device's Cholesky-with-jitter ladder."""
        A = np.asfortranarray(A, dtype=np.float64)
        R = A.shape[0]
        used, L = np.empty(R * R), np.empty(R * R)
        st = C.c_int32()
        check(self._L.bnr_test_chol_jitter(self._h, R, _dp(A), _dp(used), _dp(L), C.byref(st)))
        return used.reshape((R, R), order="F"), L.reshape((R, R), order="F"), int(st.value)

    def rng_stream(self, chain, iteration, site, element, kind, count):
        out = np.empty(count)
        check(self._L.bnr_rng_stream(self._h, chain, iteration, site, element, {"uniform": 0, "normal": 1}[kind],
                                     count, _dp(out)))
        return out

    def rng_gamma(self, chain, iteration, site, element, shape, count):
        out = np.empty(count)
        check(self._L.bnr_rng_gamma(self._h, chain, iteration, site, element, float(shape), count, _dp(out)))
        return out
