"""Helpers shared by the K-fold tests and tools/kfold_overhead.py: bnr_fit parameters, the operations bnr_fit issues
(bnr_fit_plan) and their replay on one standalone handle with a held-out table, and the rows of one fold."""
import ctypes as C

import numpy as np

_DP = C.POINTER(C.c_double)


def fit_params(bnr, n, V, R, C_, seed, chain_offset=0, **kw):
    """struct bnr_fit_params with the library defaults and the given fields (psrf_cutoff etc. as keywords)."""
    from bnr_b200 import capi
    p = capi.FitParams()
    bnr.lib().bnr_fit_default_params(C.byref(p))
    p.base.n, p.base.V, p.base.R, p.base.num_chains, p.base.seed = n, V, R, C_, seed
    p.base.chain_offset = chain_offset
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def plan(bnr, p, psrf_max=(1.0,) * 64):
    """The operations bnr_fit issues with parameters p when every R-hat check returns psrf_max[k]: [n_ops][4]."""
    from bnr_b200 import capi
    pm = np.asarray(psrf_max, dtype=np.float64)
    n_ops = C.c_int64()
    cap = 1 << 16
    ops = np.zeros((cap, 4), dtype=np.int64)
    capi.check_fit(bnr.lib().bnr_fit_plan(C.byref(p), pm.ctypes.data_as(_DP), len(pm),
                                          ops.ctypes.data_as(C.POINTER(C.c_int64)), cap, C.byref(n_ops), None))
    return ops[:n_ops.value]


def replay(bnr, p, ops, X, y, Xh, yh):
    """One handle on (X, y) with the held-out rows (Xh, yh), driven through `ops` as bnr_fit drives its device-0 handle
    (the same bnr_create parameters, row bookkeeping and moment windows); returns the open Engine."""
    b = p.base
    eng = None
    for op, a, bb, c in ops:
        if op == 0:
            eng = bnr.Engine(X, y, b.R, num_chains=b.num_chains, seed=b.seed, chain_offset=b.chain_offset,
                             device=b.device, trace_rows=int(a), trace_full_chains=int(c), trace_gamma_xi_all=bool(bb),
                             eta=b.eta, zeta=b.zeta, iota=b.iota, a_delta=b.a_delta, b_delta=b.b_delta, nu=b.nu,
                             gamma_mode=b.gamma_mode, chain_groups=b.chain_groups, trace_gamma_xi_chains=1)
            eng.set_heldout(Xh, yh, int(a))
        elif op == 1:
            eng.init_state()
        elif op == 2:
            eng.run(int(a))
        elif op == 3:
            eng.trace_row = int(a)
        elif op == 4:
            eng.copy_trace_rows(int(a), int(bb), int(c))
        elif op == 5:
            eng.set_moment_window(int(a), int(bb))
        elif op == 6:
            eng.set_moment_blocks(int(a), int(bb), int(c))
        elif op == 7:
            eng.moments_from_trace(int(a), int(bb))
            eng.rhat()
        elif op == 8:
            eng.rhat()
        elif op == 9:
            eng.moments_from_blocks(int(a), int(bb))
            eng.rhat()
        else:
            raise ValueError("operation %d is not replayed here" % op)
    return eng


def split(X, y, folds, f):
    """(training X, y, held-out X, y) of fold f (1-based), rows in their original order."""
    tr, ho = folds != f, folds == f
    return X[tr], y[tr], X[ho], y[ho]
