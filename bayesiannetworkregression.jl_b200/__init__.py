"""B200-native Gibbs engine for Bayesian Network Regression -- host-side mirror of the reference interface.

`Fit(X, y, R; ...) -> Results` and `Summary(results)` keep the names, keyword arguments, defaults and
return structure of the reference's public API (src/gibbs.jl:725-751, 1214-1250, 23-43); everything that
happens per Gibbs iteration runs inside libbnr.so (hand-written sm_100a CUDA, see csrc/ and include/bnr.h)
through `ctypes`.  There is NO CPU fallback: if the shared library or a CUDA device is missing, importing
`Engine`/`Fit` raises.

The package directory name contains a dot, so it is loaded by path (see tests/conftest.py:load_package or
__graft_entry__.load_package) and registered as module `bnr_b200`.
"""
from .capi import lib, BnrError, check, Params, VAR, COND, AUX, STATUS_BITS  # noqa: F401
from .engine import Engine  # noqa: F401
from .io import read_matrix_networks, read_adjacency_csvs, read_responses  # noqa: F401
from .fit import Fit, Summary, Predict, Loo, Compare, Results, BNRSummary, BNRPrediction, BNRLoo, BNRCompare, Table, \
    setup_X, lower_triangle, create_lower_tri  # noqa: F401

__all__ = ["Fit", "Summary", "Predict", "Loo", "Compare", "Results", "BNRSummary", "BNRPrediction", "BNRLoo",
           "BNRCompare", "Table", "Engine", "BnrError", "setup_X",
           "lower_triangle", "create_lower_tri", "lib", "read_matrix_networks", "read_adjacency_csvs", "read_responses"]
