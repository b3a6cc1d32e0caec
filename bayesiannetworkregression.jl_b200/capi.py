"""ctypes binding of include/bnr.h -- one prototype per exported symbol, nothing else."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIBBNR", os.path.join(_HERE, "libbnr.so"))   # LIBBNR: alternative build (debugging)


class BnrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libbnr error %d: %s" % (code, msg))
        self.code = code


class Params(C.Structure):
    """struct bnr_params (include/bnr.h)."""
    _fields_ = [("n", C.c_int32), ("V", C.c_int32), ("R", C.c_int32), ("num_chains", C.c_int32),
                ("chain_offset", C.c_int32), ("device", C.c_int32), ("trace_full_chains", C.c_int32),
                ("trace_gamma_xi_all", C.c_int32), ("trace_rows", C.c_int64), ("seed", C.c_uint64),
                ("eta", C.c_double), ("zeta", C.c_double), ("iota", C.c_double), ("a_delta", C.c_double),
                ("b_delta", C.c_double), ("nu", C.c_double), ("gig_inject_len", C.c_int32),
                ("gamma_mode", C.c_int32), ("chain_groups", C.c_int32), ("trace_gamma_xi_chains", C.c_int32)]


ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64)


class FitParams(C.Structure):
    """struct bnr_fit_params (include/bnr.h)."""
    _fields_ = [("base", Params), ("nburn", C.c_int64), ("nsamples", C.c_int64), ("mingen", C.c_int64),
                ("maxgen", C.c_int64), ("psrf_cutoff", C.c_double), ("purge_burn", C.c_int64),
                ("return_state", C.c_int32), ("n_devices", C.c_int32), ("interval", C.c_int32),
                ("ess_max_lag", C.c_int32), ("verbose", C.c_int32), ("ext_world", C.c_int32), ("ext_rank", C.c_int32),
                ("allgather", ALLGATHER_FN), ("allgather_ctx", C.c_void_p)]


class FitInfo(C.Structure):
    """struct bnr_fit_info (include/bnr.h)."""
    _fields_ = [("tot_generated", C.c_int64), ("burn_in", C.c_int64), ("sampled", C.c_int64), ("rows", C.c_int64),
                ("n_psrf", C.c_int64), ("streamed", C.c_int32), ("summary_ok", C.c_int32), ("ess_ok", C.c_int32),
                ("gamma_mode", C.c_int32), ("status_or", C.c_int32), ("total_chains", C.c_int32),
                ("n_devices", C.c_int32), ("exchange", C.c_int32)]


STATE = dict(none=0, gamma_xi=1, full=2)
VAR = dict(tau2=0, u=1, xi=2, gamma=3, S=4, theta=5, Delta=6, M=7, mu=8, lam=9, pi=10)
COND = dict(tau2=0, u_xi=1, gamma=2, D=3, theta=4, Delta=5, M=6, mu=7, lam=8, pi=9)
AUX = dict(tau2_params=0, sigma_inv=1, sigma_chol=2, mu_t=3, log_odds=4, W=5, G=6, G_chol=7, rhs=8, a4=9, chi=10,
           theta_params=11, delta_params=12, m_params=13, mu_params=14, lambda_logw=15, lambda_weights=16,
           pi_alpha=17, gig_used=18)
GAMMA_MODE = dict(auto=0, nform=1, qform=2)
PRED_MEAN, PRED_PREDICTIVE = 0, 1
STATUS_BITS = dict(jitter=1, sigma_notpd=2, g_notpd=4, gig_cap=8, inj_exhausted=16, nan=32, psi_notpd=64)

_H = C.c_void_p
_DP = C.POINTER(C.c_double)
_I64P = C.POINTER(C.c_int64)

# name -> (restype, argtypes): every symbol include/bnr.h declares
PROTOTYPES = {
    "bnr_version": (C.c_int, []),
    "bnr_last_error": (C.c_char_p, []),
    "bnr_default_params": (None, [C.POINTER(Params)]),
    "bnr_create": (C.c_int, [C.POINTER(Params), _DP, _DP, C.POINTER(_H)]),
    "bnr_destroy": (C.c_int, [_H]),
    "bnr_set_cache_limit": (C.c_int, [C.c_int64]),
    "bnr_trim_cache": (C.c_int, []),
    "bnr_init_state": (C.c_int, [_H]),
    "bnr_run": (C.c_int, [_H, C.c_int64]),
    "bnr_sync": (C.c_int, [_H]),
    "bnr_iteration": (C.c_int, [_H, _I64P]),
    "bnr_last_run_ms": (C.c_int, [_H, C.POINTER(C.c_float)]),
    "bnr_set_trace_row": (C.c_int, [_H, C.c_int64]),
    "bnr_get_trace_row": (C.c_int, [_H, _I64P]),
    "bnr_copy_trace_rows": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int64]),
    "bnr_set_moment_window": (C.c_int, [_H, C.c_int64, C.c_int64]),
    "bnr_set_moment_blocks": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int32]),
    "bnr_moments_from_blocks": (C.c_int, [_H, C.c_int32, C.c_int32]),
    "bnr_moments_device": (C.c_int, [_H, C.POINTER(C.c_void_p), _I64P]),
    "bnr_rhat_from_moments": (C.c_int, [C.c_int, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _DP, _DP]),
    "bnr_moments_from_trace": (C.c_int, [_H, C.c_int64, C.c_int64]),
    "bnr_moment_half_len": (C.c_int, [_H, _I64P]),
    "bnr_rhat": (C.c_int, [_H, _DP, _DP]),
    "bnr_get_state": (C.c_int, [_H, C.c_int32, C.c_int32, _DP]),
    "bnr_set_state": (C.c_int, [_H, C.c_int32, C.c_int32, _DP]),
    "bnr_var_size": (C.c_int, [_H, C.c_int32, _I64P]),
    "bnr_get_trace": (C.c_int, [_H, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _DP]),
    "bnr_status": (C.c_int, [_H, C.POINTER(C.c_int32)]),
    "bnr_export_moments": (C.c_int, [_H, C.c_void_p]),
    "bnr_summary": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _DP, _DP, _DP, _DP]),
    "bnr_ess": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int32, _DP, _DP]),
    "bnr_ess_accumulate": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_int32]),
    "bnr_ess_device": (C.c_int, [_H, C.POINTER(C.c_void_p), _I64P, C.POINTER(C.c_void_p), _I64P, C.POINTER(C.c_int32)]),
    "bnr_export_ess": (C.c_int, [_H, C.c_void_p, C.c_void_p]),
    "bnr_ess_from_stats": (C.c_int, [C.c_int, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_int64, C.c_int32, _DP, _DP]),
    "bnr_ess_from_stats_lags": (C.c_int, [C.c_int, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int64, C.c_int32, _DP, _DP, _DP, _DP]),
    "bnr_ess_stream_begin": (C.c_int, [_H, C.c_int32, C.c_int64]),
    "bnr_ess_stream_finish": (C.c_int, [_H]),
    "bnr_ess_stream_window": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int64]),
    "bnr_chain_groups": (C.c_int, [_H, C.POINTER(C.c_int32)]),
    "bnr_set_predictors": (C.c_int, [_H, C.c_int32, _DP, C.c_int64, C.c_int32]),
    "bnr_get_prediction_trace": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int64, _DP]),
    "bnr_export_predictions": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_void_p]),
    "bnr_prediction_summary": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _DP, _DP,
                                         _DP]),
    "bnr_set_loglik": (C.c_int, [_H, C.c_int64]),
    "bnr_get_loglik_trace": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int64, _DP]),
    "bnr_export_loglik": (C.c_int, [_H, C.c_int64, C.c_int64, C.c_void_p]),
    "bnr_loo_summary": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int32, _DP, _DP, _DP, _DP, _DP]),
    "bnr_device_copy": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]),
    "bnr_fit_default_params": (None, [C.POINTER(FitParams)]),
    "bnr_fit_last_error": (C.c_char_p, []),
    "bnr_fit": (C.c_int, [C.POINTER(FitParams), _DP, _DP, C.POINTER(_H)]),
    "bnr_fit_get_info": (C.c_int, [_H, C.POINTER(FitInfo)]),
    "bnr_fit_rhat": (C.c_int, [_H, _DP, _DP]),
    "bnr_fit_summary": (C.c_int, [_H, _DP, _DP, _DP, _DP]),
    "bnr_fit_ess": (C.c_int, [_H, _DP, _DP]),
    "bnr_fit_state": (C.c_int, [_H, C.c_int32, _DP]),
    "bnr_fit_handle": (C.c_int, [_H, C.c_int32, C.POINTER(_H)]),
    "bnr_fit_free": (C.c_int, [_H]),
    "bnr_fit_predict": (C.c_int, [C.POINTER(FitParams), _DP, _DP, C.c_int32, _DP, C.c_int32, C.POINTER(_H)]),
    "bnr_fit_prediction": (C.c_int, [_H, _DP, _DP, _DP]),
    "bnr_fit_loo": (C.c_int, [C.POINTER(FitParams), _DP, _DP, C.c_int32, _DP, C.c_int32, C.POINTER(_H)]),
    "bnr_fit_loo_pointwise": (C.c_int, [_H, _DP, _DP, _DP, _DP, _DP]),
    "bnr_fit_plan": (C.c_int, [C.POINTER(FitParams), _DP, C.c_int32, _I64P, C.c_int64, _I64P, C.POINTER(FitInfo)]),
    "bnr_gamma_mode": (C.c_int, [_H, C.POINTER(C.c_int32)]),
    "bnr_launch_count": (C.c_int, [_H, _I64P]),
    "bnr_profile_sweep": (C.c_int, [_H, C.POINTER(C.c_float)]),
    "bnr_set_injection": (C.c_int, [_H, _DP, C.c_int64]),
    "bnr_injection_size": (C.c_int, [_H, C.c_int32, _I64P]),
    "bnr_step": (C.c_int, [_H, C.c_int32]),
    "bnr_finish_sweep": (C.c_int, [_H]),
    "bnr_enable_aux": (C.c_int, [_H, C.c_int32]),
    "bnr_get_aux": (C.c_int, [_H, C.c_int32, C.c_int32, _DP, C.c_int64]),
    "bnr_test_chol_jitter": (C.c_int, [_H, C.c_int32, _DP, _DP, _DP, C.POINTER(C.c_int32)]),
    "bnr_rng_stream": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _DP]),
    "bnr_rng_gamma": (C.c_int, [_H, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_double, C.c_int32, _DP]),
}

_lib = None


def lib():
    """Load libbnr.so (built in-tree by `make` / __graft_entry__.build()).  Fails loudly when absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libbnr.so not found at %s: build it with `make` (there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code != 0:
        raise BnrError(code, lib().bnr_last_error().decode("utf8", "replace"))


def check_fit(code):
    if code != 0:
        msg = lib().bnr_fit_last_error().decode("utf8", "replace") or lib().bnr_last_error().decode("utf8", "replace")
        raise BnrError(code, msg)
