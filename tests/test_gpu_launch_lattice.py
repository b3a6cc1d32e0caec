"""The gamma draw at every chain count and size that picks a different launch.

The library chooses how to run the gamma draw from the handle's chain count and the padded dimension: the Cholesky
schedule (A or B), row strips per tile, the separate diagonal update Ud, the split-K of the Gram SYRK and of the X
products, the k_xmma chain tiles and the depth of the back-solve ring.  `selection` restates those rules
(bnr_linalg.cu: x_times_splits, syrk_splits, launch_cholesky, bwd_stages) so that the tests below know which variant
each point runs; the launch count of an eager sweep checks the restatement against the library.  Every point is then
held to the oracle, graph sweeps (chain groups) to eager sweeps bit for bit, the dimension edges to a float64 reference
and a long-double backward error, and the bordered factorisation to a right-hand side of 1e10."""
import math

import numpy as np
import pytest
import scipy.linalg as sla

from oracle import bnr_oracle as O
from parity_util import EPS, solve_tol, assert_close_normwise, rel_err, note
from test_gpu_parity import make_problem, random_state, sweep_injection, close

SMS = 148
TILE = 128


# ------------------------------------------------------------------------------------------------------------------
# the selection rules, restated
# ------------------------------------------------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def padded(V, n, mode):
    """(q, np, qp, factored dimension N) as bnr_create pads them."""
    q = V * (V + 1) // 2
    np_ = _cdiv(n + 1, TILE) * TILE
    qp = _cdiv(q + 1, TILE) * TILE if mode == "qform" else _cdiv(q, 16) * 16
    return q, np_, qp, (qp if mode == "qform" else np_)


def x_splits(M, K, C):
    tiles = _cdiv(M, 128) * _cdiv(C, 64)
    return max(1, min(_cdiv(2 * SMS, tiles), max(K // 64, 1), 64))


def syrk_splits(np_, qp, C):
    T = np_ // TILE
    tiles, nk = T * (T + 1) // 2, qp // 16
    if tiles * C >= SMS:
        return 1
    return max(1, min(_cdiv(4 * SMS, tiles * C), nk // 24, 8))


def bwd_stages(N):
    return min(6, (227 * 1024 - 8 * N - 512) // (8 * 32 * 128))


def selection(V, n, mode, C):
    """Everything (V, n, mode, C) selects for the eager sweep of a handle of C chains."""
    q, np_, qp, N = padded(V, n, mode)
    T = N // TILE
    syrk = syrk_splits(np_, qp, C) if mode == "nform" else 1
    latency = C * (T - 1) <= 128

    def strips(tiles):
        return 4 if C * tiles * 4 <= SMS else (2 if C * tiles * 2 <= SMS else 1)

    quiet = mode == "qform" or syrk > 1
    ud = (8 if C * 8 <= SMS else (4 if C * 4 <= SMS else 0)) if quiet else 0
    if latency:
        used_strips = {strips(r) for r in range(1, T - 1)} | ({strips(1)} if T > 1 and not ud else set())
        chol = T + (T - 1) * (2 if ud else 1) + 3 * max(T - 2, 0)
    else:
        used_strips, ud = set(), None
        chol = 4 * T - 4
    xs = (x_splits(np_, qp, C), x_splits(qp, np_, C))
    tiles = _cdiv(C, 64)
    # tau2, u/xi, edge prep, X products, rhs, SYRK or P, k_augment, back solve, GIG, finish, record: 13 + the rest
    sweep = 13 + chol + 2 * (xs[0] > 1) + (xs[1] > 1) + (syrk > 1)
    return dict(schedule="B" if latency else "A", strips=used_strips, ud=ud, syrk_split=syrk > 1, x_splits=xs,
                xmma_tiles=tiles, last_tile_chains=C - 64 * (tiles - 1), bwd_stages=bwd_stages(N),
                sweep_launches=sweep, refresh_launches=1 + (xs[0] > 1))


# (mode, V, n, chains).  n-form V=40 / n=1000 is T = 8: split and unsplit SYRK, Ud, 4 / 2 / 1 strips, B -> A at 19,
# 1 / 2 / 3 chain tiles with a one-chain last tile; q-form V=30 / n=500 is T = 4: Ud 8 -> 4 -> 0, B -> A at 43;
# n-form V=20 / n=200 is T = 2: strips 4 -> 2 -> 1 inside schedule B; V=10 leaves X v unsplit (K = 64).
LATTICE = ([("nform", 40, 1000, C) for C in (2, 4, 5, 6, 7, 12, 13, 18, 19, 65, 129)]
           + [("qform", 30, 500, C) for C in (18, 19, 37, 38, 42, 43)]
           + [("nform", 20, 200, C) for C in (37, 38, 74, 75, 128)]
           + [("nform", 10, 300, 3)])

# (mode, V, n): the bordering row on the matrix's last row (n = 127, q = 4095), the last dimensions with 6 and 5
# back-solve stages (N = 4352, 4480), and the largest factored dimension (N = 8192) in both forms
EDGES = [("qform", 90, 100), ("nform", 12, 4351), ("nform", 12, 4479), ("nform", 12, 8191), ("qform", 127, 60)]


def _ids(points):
    return ["%s-V%d-n%d" % p[:3] + ("-C%d" % p[3] if len(p) > 3 else "") for p in points]


def test_lattice_reaches_every_rule_value():
    """The points below run every value of every rule (else a change of the rules would quietly stop testing one)."""
    sel = [selection(V, n, mode, C) for mode, V, n, C in LATTICE] + [selection(V, n, mode, 1) for mode, V, n in EDGES]
    assert {s["schedule"] for s in sel} == {"A", "B"}
    assert set().union(*(s["strips"] for s in sel)) == {1, 2, 4}
    assert {s["ud"] for s in sel if s["schedule"] == "B"} == {0, 4, 8}
    assert {s["syrk_split"] for s in sel} == {False, True}
    assert {s["x_splits"][0] > 1 for s in sel} == {False, True}
    assert {s["xmma_tiles"] for s in sel} == {1, 2, 3}
    assert {2, 3} <= {s["xmma_tiles"] for s in sel if s["last_tile_chains"] == 1}
    assert {s["bwd_stages"] for s in sel} == {5, 6}
    # and the rule edges the lattice is built around
    assert selection(40, 1000, "nform", 18)["schedule"] == "B" and selection(40, 1000, "nform", 19)["schedule"] == "A"
    assert selection(30, 500, "qform", 42)["schedule"] == "B" and selection(30, 500, "qform", 43)["schedule"] == "A"
    assert [selection(30, 500, "qform", C)["ud"] for C in (18, 19, 37, 38)] == [8, 4, 4, 0]
    assert [selection(20, 200, "nform", C)["strips"] for C in (37, 38, 74, 75)] == [{4}, {2}, {2}, {1}]
    assert [bwd_stages(N) for N in (4352, 4480, 8192)] == [6, 5, 5]


# ------------------------------------------------------------------------------------------------------------------
# injected sweeps at natural chain counts: every chain its own state, the oracle on a subset, bits on the rest
# ------------------------------------------------------------------------------------------------------------------
def _chain_states(rng, V, R, C):
    """Neighbouring chains 100x apart in S: a chain that reads its neighbour's tile is off by O(1)."""
    states = []
    for c in range(C):
        st = random_state(rng, V, R)
        st["S"] = st["S"] * 10.0 ** (2 * (c % 4) - 2)
        states.append(st)
    return states


def _run_injected(bnr, X, y, R, K, mode, states, inj):
    C = len(states)
    eng = bnr.Engine(X, y, R, num_chains=C, seed=1, gig_inject_len=K, gamma_mode=mode)
    eng.init_state()
    for c, st in enumerate(states):
        eng.set_state_dict(c, st)
    eng.set_injection(inj)
    l0 = eng.launch_count()
    eng.run(1)
    launches = eng.launch_count() - l0
    got = [eng.get_state_dict(c) for c in range(C)]
    status = eng.status()
    eng.close()
    return got, launches, status


@pytest.mark.gpu
@pytest.mark.parametrize("mode,V,n,C", LATTICE, ids=_ids(LATTICE))
def test_injected_sweep_at_natural_chain_count(bnr, mode, V, n, C):
    R, K = 4, 48
    sel = selection(V, n, mode, C)
    X, y = make_problem(V * 7 + n, V, R, n)
    rng = np.random.default_rng(C * 1000 + V)
    states = _chain_states(rng, V, R, C)
    inj = np.stack([sweep_injection(rng, n, V, R, K)[0] for _ in range(C)])
    got, launches, status = _run_injected(bnr, X, y, R, K, mode, states, inj)
    # one eager sweep (+ X gamma for the state just set): the restated rules must count the kernels the library ran
    assert launches == sel["sweep_launches"] + sel["refresh_launches"], (launches, sel)
    assert not (status & ~1).any(), status
    if C > 20:
        # every chain: the same states in reverse chain order on a second handle give the same bits
        rev, _, _ = _run_injected(bnr, X, y, R, K, mode, states[::-1], inj[::-1].copy())
        for c in range(C):
            for k in got[c]:
                np.testing.assert_array_equal(np.asarray(got[c][k]), np.asarray(rev[C - 1 - c][k]),
                                              err_msg="%s chain %d vs reversed handle" % (k, c))
        pick = {c for c in (0, 63, 64, 127, 128) if c < C}
        pick |= set(np.random.default_rng(C).choice(C, 4, replace=False).tolist())
    else:
        pick = set(range(C))
    for c in sorted(pick):
        new, aux = O.gibbs_sweep(states[c], X, y, V, R, O.DEFAULT_HYPER, inj[c], K, literal=False,
                                 gamma_form="q" if mode == "qform" else "n")
        A = aux["gamma"]["P" if mode == "qform" else "G"]
        ev = np.linalg.eigvalsh(A)
        cond = float(ev[-1] / ev[0])
        tol = solve_tol(cond)
        for k in ("tau2", "xi", "lam"):
            close(got[c][k], new[k], rtol=1e-10, msg="%s chain %d" % (k, c))
        for k in ("u", "gamma", "S", "theta", "Delta", "M", "pi"):
            assert_close_normwise(got[c][k], new[k], tol, "%s chain %d" % (k, c))
        # mu = mean(y - X gamma) + sd z inherits the error of gamma through the column means of X, which the large
        # gammas of the S = 1e2, 1e4 chains make larger than tol |mu|
        mu_tol = tol * max(abs(new["mu"]), float(np.abs(X.mean(axis=0)) @ np.abs(new["gamma"])))
        assert abs(got[c]["mu"] - new["mu"]) <= mu_tol, ("mu chain %d" % c, got[c]["mu"], new["mu"], mu_tol)
        note(test="lattice", mode=mode, V=V, n=n, C=C, chain=c, cond=cond,
             c_gamma=rel_err(got[c]["gamma"], new["gamma"]) / (cond * EPS))


# ------------------------------------------------------------------------------------------------------------------
# graph sweeps (chain groups) == eager sweeps (whole handle), bit for bit
# ------------------------------------------------------------------------------------------------------------------
TRACED = ("tau2", "u", "xi", "gamma", "S", "theta", "Delta", "M", "mu", "lam", "pi")


@pytest.mark.gpu
@pytest.mark.parametrize("groups", [0, 1, 2, 4])
@pytest.mark.parametrize("V,R,n,C", [(60, 5, 500, 129), (100, 7, 1000, 193)], ids=["V60-n500-C129", "c3-C193"])
def test_graph_sweeps_equal_eager_sweeps(bnr, V, R, n, C, groups):
    """run(2), run(1), run(2), run(3) mixes both graph parities with eager sweeps; eight run(1) are eight eager sweeps.
    Every state variable and every trace row must agree: the chain grouping must not change any summation order."""
    X, y = make_problem(V + n + C, V, R, n, dense=False)
    kw = dict(num_chains=C, seed=17, trace_rows=9, trace_full_chains=C, chain_groups=groups)
    with bnr.Engine(X, y, R, **kw) as a, bnr.Engine(X, y, R, **kw) as b:
        assert a.gamma_mode == "nform"
        a.init_state()
        b.init_state()
        for k in (2, 1, 2, 3):
            a.run(k)
        for _ in range(8):
            b.run(1)
        assert a.iteration == b.iteration == 8
        assert not (a.status() & ~1).any() and not (b.status() & ~1).any()
        for c in range(C):
            for k in TRACED:
                np.testing.assert_array_equal(a.get_trace(c, k, 0, 9), b.get_trace(c, k, 0, 9),
                                              err_msg="trace of %s, chain %d, %d groups" % (k, c, a.chain_groups))
            sa, sb = a.get_state_dict(c), b.get_state_dict(c)
            for k in sa:
                np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg="%s chain %d" % (k, c))


# ------------------------------------------------------------------------------------------------------------------
# dimension edges: gamma, a4 and the factor against a float64 reference, and the long-double backward error
# ------------------------------------------------------------------------------------------------------------------
def _gamma_reference(X, y, st, z1, z2, mode):
    """O.update_gamma / O.update_gamma_qform with the solves done by Cholesky and triangular solves (LAPACK), which
    keeps the float64 reference affordable at N = 8192."""
    tau2, S, mu = st["tau2"], st["S"], st["mu"]
    W = O.W_of(st["u"], st["lam"])
    if mode == "qform":
        P = (X.T @ X + np.diag(1.0 / S)) / tau2
        L = sla.cholesky(P, lower=True)
        b = X.T @ ((y - mu - X @ W) / tau2)
        beta = sla.solve_triangular(L, sla.solve_triangular(L, b, lower=True) + z1, lower=True, trans="T")
        return dict(A=P, L=L, a4=beta, gamma=W + beta, W=W)
    tau = math.sqrt(tau2)
    d1 = np.sqrt(tau2 * S) * z1
    Xt = X / tau
    G = (Xt * (tau2 * S)[None, :]) @ Xt.T + np.eye(X.shape[0])
    L = sla.cholesky(G, lower=True)
    a4 = sla.cho_solve((L, True), (y - X @ W - mu) / tau - (Xt @ d1 + z2))
    return dict(A=G, L=L, a4=a4, gamma=d1 + (tau2 * S) * (Xt.T @ a4) + W, W=W)


def _cond_bound(X, S, tau2, mode):
    """cond(G) exactly from the small Gram matrix (n-form); an upper bound of cond(P) (q-form)."""
    n, q = X.shape
    if mode == "nform":
        B = X * np.sqrt(S)[None, :]
        lam = np.linalg.eigvalsh(B.T @ B if q <= n else B @ B.T)
        return (1.0 + lam[-1]) / (1.0 + (lam[0] if n <= q else 0.0))
    smax2 = np.linalg.eigvalsh(X @ X.T if n <= q else X.T @ X)[-1]
    return (smax2 + 1.0 / S.min()) * S.max()


def _backward_error(X, y, st, z1, z2, mode, W, a4, A):
    """|A a4 - r|_inf / (|A|_inf |a4|_inf) in long double, A a4 by products with X (r: the system's right-hand side
    from the engine's own W; the q-form runs with z = 0, so that P beta = b)."""
    ld = np.longdouble
    Xl, x = X.astype(ld), a4.astype(ld)
    S, tau2, mu = st["S"].astype(ld), ld(st["tau2"]), ld(st["mu"])
    if mode == "qform":
        Ax = (Xl.T @ (Xl @ x) + x / S) / tau2
        r = Xl.T @ ((y.astype(ld) - mu - Xl @ W.astype(ld)) / tau2)
    else:
        Ax = Xl @ (S * (Xl.T @ x)) + x
        v = W + np.sqrt(st["tau2"] * st["S"]) * z1
        r = (y.astype(ld) - mu - Xl @ v.astype(ld)) / np.sqrt(tau2) - z2.astype(ld)
    normA = float(np.abs(A).sum(axis=1).max())
    return float(np.max(np.abs(Ax - r))) / (normA * float(np.max(np.abs(a4))))


@pytest.mark.gpu
@pytest.mark.parametrize("mode,V,n", EDGES, ids=_ids(EDGES))
def test_dimension_edges_against_reference(bnr, mode, V, n):
    R, K = 3, 8
    q, _, _, N = padded(V, n, mode)
    m = q if mode == "qform" else n
    X, y = make_problem(V + n, V, R, n)
    rng = np.random.default_rng(n)
    st = random_state(rng, V, R)
    inj, lay = sweep_injection(rng, n, V, R, K)
    o1, s1 = lay["gamma_z1"]
    o2, s2 = lay["gamma_z2"]
    if mode == "qform":
        inj[o1:o1 + s1] = 0.0
    z1, z2 = inj[o1:o1 + s1].copy(), inj[o2:o2 + s2].copy()
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
        Lg = eng.get_aux(0, "G_chol").reshape(m, m).T
    ref = _gamma_reference(X, y, st, z1, z2, mode)
    cond = _cond_bound(X, st["S"], st["tau2"], mode)
    tol = solve_tol(cond)
    e_chol = float(np.max(np.abs(Lg - ref["L"]))) / float(np.max(np.abs(ref["L"])))
    del Lg
    eta = _backward_error(X, y, st, z1, z2, mode, W, a4, ref["A"])
    note(test="dimension_edge", mode=mode, V=V, n=n, N=N, stages=bwd_stages(N), cond=cond, eta=eta, c_eta=eta / EPS,
         c_a4=rel_err(a4, ref["a4"]) / (cond * EPS), c_gamma=rel_err(gamma, ref["gamma"]) / (cond * EPS),
         c_chol=e_chol / (cond * EPS))
    assert e_chol <= tol, (e_chol, cond)
    assert_close_normwise(a4, ref["a4"], tol, "a4")
    assert_close_normwise(gamma, ref["gamma"], tol, "gamma")
    assert eta <= N * EPS, eta


# ------------------------------------------------------------------------------------------------------------------
# the bordering corner at large right-hand sides
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("norm", [1e6, 1e8, 1e10])
def test_bordered_solve_at_large_right_hand_sides(bnr, norm):
    """y orthogonal to the range of X, u = 0, mu = 0, tau2 = 1, z = 0: G a4 = y has the exact answer a4 = y (X'y = 0)
    and gamma = S X' a4 = 0.  The last pivot of the bordered matrix is then 1 + |y|^2 - y'G^-1 y = 1, a difference of
    two terms of size |y|^2: the factorisation must not lose it (a non-positive pivot flags a positive-definite G)."""
    V, R, n, C, K = 10, 3, 300, 2, 8
    X, _ = make_problem(5, V, R, n)
    rng = np.random.default_rng(6)
    Q, _ = np.linalg.qr(X)
    z = rng.normal(size=n)
    y = z - Q @ (Q.T @ z)
    y *= norm / np.linalg.norm(y)
    with bnr.Engine(X, y, R, num_chains=C, seed=3, gig_inject_len=K, gamma_mode="nform") as eng:
        eng.enable_aux(True)
        states = []
        for c in range(C):
            st = random_state(rng, V, R)
            st.update(u=np.zeros((R, V)), mu=0.0, tau2=1.0)
            states.append(st)
            eng.set_state_dict(c, st)
        inj = np.stack([sweep_injection(rng, n, V, R, K)[0] for _ in range(C)])
        lay = O.draw_layout(n, V, R, K)
        for name in ("gamma_z1", "gamma_z2"):
            o, s = lay[name]
            inj[:, o:o + s] = 0.0
        eng.set_injection(inj)
        eng.step("gamma")
        status = eng.status()
        for c, st in enumerate(states):
            a4 = eng.get_aux(c, "a4")
            gamma = eng.get_state(c, "gamma")[:, 0]
            cond = _cond_bound(X, st["S"], 1.0, "nform")
            tol = solve_tol(cond)
            note(test="bordered_corner", norm=norm, chain=c, cond=cond, status=int(status[c]),
                 e_a4=rel_err(a4, y), gamma_max=float(np.max(np.abs(gamma))))
            assert_close_normwise(a4, y, tol, "a4, |y| = %g, chain %d" % (norm, c))
            # |X' a4| is rounding of a sum of n terms of size |X_ij| |y_i|
            bound = tol * float(np.max(st["S"])) * float(np.max(np.abs(X).T @ np.abs(y)))
            assert np.max(np.abs(gamma)) <= bound, (np.max(np.abs(gamma)), bound)
        assert not (status & ~1).any(), status
