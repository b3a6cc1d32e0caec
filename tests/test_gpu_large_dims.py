"""Factored dimensions above 8192, up to 32768: n <= 32767 in the n-form, V <= 255 in the q-form.

Above N = 8192 the back solve runs on a cluster of 8 CTAs per chain (k_bwd_cluster); at and below it on one CTA
(k_bwd_stream), so no shape accepted under the former limit changes.  AUTO keeps its former choice wherever that choice
fits 8192 and otherwise takes the cheaper of the forms that fit 32768.  The CPU tests restate that rule and a Woodbury
reference of the solve that needs no N x N matrix; the GPU tests hold the gamma draw at the new sizes to a float64
reference and a long-double backward error, and the new back solve to the determinism rules of the old one."""
import math
import os

import numpy as np
import pytest
import scipy.linalg as sla

from parity_util import EPS, solve_tol, assert_close_normwise, rel_err, note
from test_gpu_parity import make_problem, random_state, sweep_injection
from test_gpu_launch_lattice import (padded, selection, _gamma_reference, _backward_error, _cond_bound, _chain_states,
                                     _run_injected, TRACED)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OLD_MAX, NEW_MAX = 8192, 32768
BWC_K = 8


# ------------------------------------------------------------------------------------------------------------------
# the choice of form, restated (bnr_api.cu: create_impl), and the back solve each dimension selects
# ------------------------------------------------------------------------------------------------------------------
def _costs(V, n):
    q = V * (V + 1) // 2
    qd, nd = np.asarray(q, dtype=np.float64), np.asarray(n, dtype=np.float64)
    return qd * qd * qd / 3.0 + 4.0 * qd * qd, nd * nd * qd + nd * nd * nd / 3.0


def _dims(V, n):
    q = V * (V + 1) // 2
    return -(-(n + 1) // 128) * 128, -(-(q + 1) // 128) * 128          # np, qp128


def auto_rule_old(V, n):
    """(q-form?, accepted) under the 8192 limit."""
    cost_q, cost_n = _costs(V, n)
    np_, qp128 = _dims(V, n)
    qform = (cost_q < cost_n) & (qp128 <= OLD_MAX)
    return qform, np.where(qform, qp128, np_) <= OLD_MAX


def auto_rule(V, n):
    """(q-form?, accepted) now."""
    cost_q, cost_n = _costs(V, n)
    np_, qp128 = _dims(V, n)
    old_q, old_ok = auto_rule_old(V, n)
    q_fits, n_fits = qp128 <= NEW_MAX, np_ <= NEW_MAX
    new_q = q_fits & ((cost_q < cost_n) | np.logical_not(n_fits))
    qform = np.where(old_ok, old_q, new_q)
    return qform, np.where(qform, qp128, np_) <= NEW_MAX


def back_solve(N):
    """(kernel, CTAs per chain) of the back solve at factored dimension N."""
    return ("k_bwd_stream", 1) if N <= OLD_MAX else ("k_bwd_cluster", BWC_K)


def test_auto_rule_keeps_every_shape_accepted_under_the_old_limit():
    V = np.arange(2, 301)[:, None]
    n = np.arange(1, 40001)[None, :]
    V, n = np.broadcast_arrays(V, n)
    old_q, old_ok = auto_rule_old(V, n)
    new_q, new_ok = auto_rule(V, n)
    np_, qp128 = _dims(V, n)
    assert (new_q[old_ok] == old_q[old_ok]).all()
    assert (new_ok[old_ok]).all()
    # accepted exactly when the chosen dimension fits, and refused only when neither form fits
    gdim = np.where(new_q, qp128, np_)
    assert (new_ok == (gdim <= NEW_MAX)).all()
    assert (~new_ok == ((np_ > NEW_MAX) & (qp128 > NEW_MAX))).all()
    # the new ground is reached in both forms
    new = new_ok & ~old_ok
    assert new_q[new].any() and (~new_q[new]).any()
    # the points the GPU test checks against the library
    assert auto_rule(130, 6000) == (False, True)          # n-form although the q-form is cheaper: unchanged
    assert auto_rule(130, 9000) == (True, True)           # q-form above the old limit
    assert auto_rule(256, 32768)[1] == False and auto_rule(255, 40000) == (True, True)
    assert auto_rule(12, 32767) == (True, True)           # AUTO never needs n-form sizes this large ...
    assert _dims(12, 32767)[0] == NEW_MAX and _dims(12, 32768)[0] > NEW_MAX   # ... an explicit n-form reaches n = 32767


def test_back_solve_selection_by_dimension():
    """The cluster back solve starts right above N = 8192; K is a constant, so the summation order depends on N only."""
    assert back_solve(padded(12, 8191, "nform")[3]) == ("k_bwd_stream", 1)
    assert padded(12, 8192, "nform")[3] == 8320 and back_solve(8320) == ("k_bwd_cluster", BWC_K)
    assert padded(127, 60, "qform")[3] == 8192 and padded(128, 60, "qform")[3] == 8320
    assert padded(255, 60, "qform")[3] == NEW_MAX and padded(12, 32767, "nform")[3] == NEW_MAX
    # every rank of the cluster owns at least one block row
    assert all(N // 128 > BWC_K for N in range(8320, NEW_MAX + 1, 128))


def test_header_states_the_new_limit():
    with open(os.path.join(ROOT, "include", "bnr.h")) as fh:
        text = fh.read()
    assert "#define BNR_MAX_FACTOR_DIM 32768" in text
    assert "#define BNR_VERSION 200" in text


# ------------------------------------------------------------------------------------------------------------------
# a reference of the solve at any N without N x N matrices (Woodbury)
# ------------------------------------------------------------------------------------------------------------------
def woodbury_nform(X, S, r):
    """(X diag(S) X' + I)^-1 r = r - X (diag(1/S) + X'X)^-1 X' r: a q x q system (q << n)."""
    K = X.T @ X + np.diag(1.0 / S)
    return r - X @ sla.solve(K, X.T @ r, assume_a="pos")


def woodbury_qform(X, S, tau2, b):
    """((X'X + diag(1/S)) / tau2)^-1 b = tau2 (D b - D X' (I + X D X')^-1 X D b), D = diag(S): an n x n system (n << q)."""
    Db = S * b
    K = (X * S[None, :]) @ X.T + np.eye(X.shape[0])
    return tau2 * (Db - S * (X.T @ sla.solve(K, X @ Db, assume_a="pos")))


def test_woodbury_reference_matches_a_dense_solve():
    rng = np.random.default_rng(5)
    n, q = 300, 21
    X = rng.normal(size=(n, q))
    S = rng.gamma(1.0, size=q) + 1e-3
    r = rng.normal(size=n)
    G = (X * S[None, :]) @ X.T + np.eye(n)
    want = np.linalg.solve(G, r)
    np.testing.assert_allclose(woodbury_nform(X, S, r), want, rtol=0, atol=1e-12 * np.abs(want).max())
    n, q = 20, 210
    X = rng.normal(size=(n, q))
    S = rng.gamma(1.0, size=q) + 1e-3
    b = rng.normal(size=q)
    tau2 = 1.7
    P = (X.T @ X + np.diag(1.0 / S)) / tau2
    want = np.linalg.solve(P, b)
    np.testing.assert_allclose(woodbury_qform(X, S, tau2, b), want, rtol=0, atol=1e-10 * np.abs(want).max())


# ------------------------------------------------------------------------------------------------------------------
# GPU: limits and the choice of form in the library
# ------------------------------------------------------------------------------------------------------------------
def _raw_create(bnr, V, n, mode):
    """bnr_create with one-element X / y buffers: the dimension checks come before any read of X."""
    import ctypes as C
    L = bnr.lib()
    p = bnr.Params()
    L.bnr_default_params(C.byref(p))
    p.n, p.V, p.R, p.num_chains = n, V, 2, 1
    p.gamma_mode = dict(auto=0, nform=1, qform=2)[mode]
    one = (C.c_double * 1)(0.0)
    h = C.c_void_p()
    rc = L.bnr_create(C.byref(p), one, one, C.byref(h))
    if rc == 0:
        L.bnr_destroy(h)
    return rc, L.bnr_last_error().decode()


@pytest.mark.gpu
@pytest.mark.parametrize("V,n,mode", [(2, 32768, "nform"), (256, 10, "qform"), (256, 32768, "auto")])
def test_create_refuses_beyond_32768(bnr, V, n, mode):
    rc, msg = _raw_create(bnr, V, n, mode)
    assert rc == -1 and "32768" in msg, (rc, msg)


@pytest.mark.gpu
@pytest.mark.parametrize("V,n,want", [(130, 6000, "nform"), (130, 9000, "qform")])
def test_auto_choice_in_the_library(bnr, V, n, want):
    assert auto_rule(V, n) == (want == "qform", True)
    X, y = make_problem(V + n, V, 2, n, dense=False)
    with bnr.Engine(X, y, 2, num_chains=1, seed=1) as eng:
        assert eng.gamma_mode == want


# ------------------------------------------------------------------------------------------------------------------
# GPU: one injected gamma step against the float64 reference (and, at N = 32768, Woodbury only)
# ------------------------------------------------------------------------------------------------------------------
# (mode, V, n): N = 8320 on the FP64 SYRK and on the INT8 Gram path, 12032, 16384, 32768; q-form qp = 8320 and 11392
POINTS = [("nform", 12, 8192), ("nform", 50, 8192), ("nform", 12, 12000), ("nform", 12, 16383), ("nform", 12, 32767),
          ("qform", 128, 60), ("qform", 150, 100)]
DENSE_MAX = 16384          # the float64 reference builds N x N matrices up to here


def _ids(points):
    return ["%s-V%d-n%d" % p for p in points]


def _normA_nform(X, S, rows=2048):
    """|X diag(S) X' + I|_inf, one slab of rows at a time."""
    best = 0.0
    XS = X * S[None, :]
    for i0 in range(0, X.shape[0], rows):
        B = XS[i0:i0 + rows] @ X.T
        B[np.arange(B.shape[0]), np.arange(i0, i0 + B.shape[0])] += 1.0
        best = max(best, float(np.abs(B).sum(axis=1).max()))
    return best


@pytest.mark.gpu
@pytest.mark.parametrize("mode,V,n", POINTS, ids=_ids(POINTS))
def test_gamma_step_at_large_dimensions(bnr, mode, V, n):
    R, K = 3, 8
    q, _, _, N = padded(V, n, mode)
    assert N > OLD_MAX and auto_rule(V, n)[1]
    m = q if mode == "qform" else n
    X, y = make_problem(V + n, V, R, n)
    rng = np.random.default_rng(n + V)
    st = random_state(rng, V, R)
    inj, lay = sweep_injection(rng, n, V, R, K)
    o1, s1 = lay["gamma_z1"]
    o2, s2 = lay["gamma_z2"]
    if mode == "qform":
        inj[o1:o1 + s1] = 0.0
    z1, z2 = inj[o1:o1 + s1].copy(), inj[o2:o2 + s2].copy()
    dense = N <= DENSE_MAX
    with bnr.Engine(X, y, R, num_chains=1, seed=3, gig_inject_len=K, gamma_mode=mode) as eng:
        assert eng.gamma_mode == mode
        eng.enable_aux(True)
        eng.set_state_dict(0, st)
        eng.set_injection(inj[None, :])
        eng.step("gamma")
        assert not (eng.status() & ~1).any(), eng.status()
        a4 = eng.get_aux(0, "a4")
        W = eng.get_aux(0, "W")
        gamma = eng.get_state(0, "gamma")[:, 0]
        Lg = eng.get_aux(0, "G_chol").reshape(m, m).T if dense else None
    cond = _cond_bound(X, st["S"], st["tau2"], mode)
    tol = solve_tol(cond)
    if dense:
        ref = _gamma_reference(X, y, st, z1, z2, mode)
        e_chol = float(np.max(np.abs(Lg - ref["L"]))) / float(np.max(np.abs(ref["L"])))
        del Lg
        eta = _backward_error(X, y, st, z1, z2, mode, W, a4, ref["A"])
        a4_ref, gamma_ref = ref["a4"], ref["gamma"]
        del ref
        assert e_chol <= tol, (e_chol, cond)
    else:
        # n-form only: a4 = G^-1 r by Woodbury; |G|_inf by slabs (a 1 x 1 stand-in carries it into _backward_error).
        # gamma = d1 + tau2 S X' a4 / tau: X' a4 sums n terms that largely cancel, so at n = 32767 a forward error of a4
        # within cond eps grows by far more than cond in gamma.  gamma is held instead to the same formula applied to
        # the engine's own a4, with the rounding bound of an n-term dot product.
        tau = math.sqrt(st["tau2"])
        d1 = np.sqrt(st["tau2"] * st["S"]) * z1
        r = (y - X @ W - st["mu"]) / tau - (X @ d1 / tau + z2)
        a4_ref = woodbury_nform(X, st["S"], r)
        gamma_ref = d1 + st["tau2"] * st["S"] * (X.T @ a4) / tau + W
        bound = 2 * n * EPS * (st["tau2"] * st["S"] * (np.abs(X).T @ np.abs(a4)) / tau + np.abs(d1) + np.abs(W))
        assert (np.abs(gamma - gamma_ref) <= bound).all(), float(np.max(np.abs(gamma - gamma_ref) / bound))
        gamma_ref = gamma
        e_chol = float("nan")
        eta = _backward_error(X, y, st, z1, z2, mode, W, a4, np.array([[_normA_nform(X, st["S"])]]))
    note(test="large_dims", mode=mode, V=V, n=n, N=N, cond=cond, eta=eta, c_eta=eta / EPS,
         c_a4=rel_err(a4, a4_ref) / (cond * EPS), c_gamma=rel_err(gamma, gamma_ref) / (cond * EPS),
         c_chol=e_chol / (cond * EPS))
    assert_close_normwise(a4, a4_ref, tol, "a4")
    assert_close_normwise(gamma, gamma_ref, tol, "gamma")
    assert eta <= N * EPS, eta


# ------------------------------------------------------------------------------------------------------------------
# GPU: the cluster back solve keeps the chains apart, and its rounding does not depend on chain count or grouping
# ------------------------------------------------------------------------------------------------------------------
V0, N0 = 12, 8192          # N = 8320: the first dimension of the cluster back solve


@pytest.mark.gpu
def test_chains_do_not_mix_at_8320(bnr):
    R, K, C, mode = 3, 48, 3, "nform"
    sel = selection(V0, N0, mode, C)
    X, y = make_problem(V0 + N0, V0, R, N0)
    rng = np.random.default_rng(41)
    states = _chain_states(rng, V0, R, C)
    inj = np.stack([sweep_injection(rng, N0, V0, R, K)[0] for _ in range(C)])
    got, launches, status = _run_injected(bnr, X, y, R, K, mode, states, inj)
    assert launches == sel["sweep_launches"] + sel["refresh_launches"], (launches, sel)
    assert not (status & ~1).any(), status
    rev, _, status_r = _run_injected(bnr, X, y, R, K, mode, states[::-1], inj[::-1].copy())
    assert not (status_r & ~1).any(), status_r
    for c in range(C):
        for k in got[c]:
            np.testing.assert_array_equal(np.asarray(got[c][k]), np.asarray(rev[C - 1 - c][k]),
                                          err_msg="%s chain %d vs reversed handle" % (k, c))


@pytest.mark.gpu
@pytest.mark.parametrize("groups", [1, 2, 3])
def test_graph_sweeps_equal_eager_sweeps_at_8320(bnr, groups):
    R, C = 3, 3
    sel = selection(V0, N0, "nform", C)
    X, y = make_problem(V0 + N0 + C, V0, R, N0, dense=False)
    kw = dict(num_chains=C, seed=17, trace_rows=5, trace_full_chains=C, chain_groups=groups, gamma_mode="nform")
    with bnr.Engine(X, y, R, **kw) as a, bnr.Engine(X, y, R, **kw) as b:
        assert a.gamma_mode == "nform" and a.chain_groups == groups
        a.init_state()
        b.init_state()
        a.run(2)
        a.run(2)
        b.run(1)
        l0 = b.launch_count()
        b.run(1)
        assert b.launch_count() - l0 == sel["sweep_launches"]        # the back solve is still one launch
        b.run(1)
        b.run(1)
        assert a.iteration == b.iteration == 4
        assert not (a.status() & ~1).any() and not (b.status() & ~1).any()
        for c in range(C):
            for k in TRACED:
                np.testing.assert_array_equal(a.get_trace(c, k, 0, 5), b.get_trace(c, k, 0, 5),
                                              err_msg="trace of %s, chain %d, %d groups" % (k, c, groups))
            sa, sb = a.get_state_dict(c), b.get_state_dict(c)
            for k in sa:
                np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg="%s chain %d" % (k, c))


@pytest.mark.gpu
def test_runs_are_reproducible_at_8320(bnr):
    """Two handles, same seed, graph sweeps: bit-identical.  A race in the DSMEM / mbarrier hand-offs of the cluster
    back solve would show as a difference here."""
    R, C = 3, 4
    X, y = make_problem(V0 + N0 + 7, V0, R, N0, dense=False)
    out = []
    for _ in range(2):
        with bnr.Engine(X, y, R, num_chains=C, seed=23, gamma_mode="nform") as eng:
            assert eng.gamma_mode == "nform"
            eng.init_state()
            eng.run(3)
            assert not (eng.status() & ~1).any()
            out.append([eng.get_state_dict(c) for c in range(C)])
    for c in range(C):
        for k in out[0][c]:
            np.testing.assert_array_equal(np.asarray(out[0][c][k]), np.asarray(out[1][c][k]), err_msg="%s chain %d" % (k, c))


# ------------------------------------------------------------------------------------------------------------------
# GPU: Fit end to end above the old limit
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("V,n,mode", [(50, 9000, "nform"), (130, 9000, "auto")])
def test_fit_above_the_old_limit(bnr, V, n, mode):
    q = V * (V + 1) // 2
    X, y = make_problem(V * 3 + n, V, 3, n, dense=False)
    res = bnr.Fit(X, y, 3, nburn=20, nsamples=40, num_chains=2, seed=5, x_transform=False, filename=None,
                  gamma_mode=mode, psrf_cutoff=1e9)
    assert res.extra["gamma_mode"] == ("nform" if mode == "nform" else "qform")
    assert np.isfinite(res.rhatγ.γ).all() and np.isfinite(res.rhatξ.ξ).all()
    summ = bnr.Summary(res)
    assert len(summ.edge_coef["estimate"]) == q and np.isfinite(np.asarray(summ.edge_coef["estimate"], dtype=float)).all()
    assert not (np.asarray(res.extra["status"]) & ~1).any(), res.extra["status"]
