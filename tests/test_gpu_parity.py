"""Level-1 parity of the CUDA path against the CPU oracle, through the C ABI (libbnr.so via ctypes).

Every conditional is run on the GPU from an identical state with injected standard-normal / uniform /
unit-gamma variates; conditional parameters, means, Cholesky factors and draws must match the oracle to
RTOL = 1e-10 relative (north_star's FP64 tolerance); quantities that pass through a linear solve (the R x R
system of a node, the n x n or q x q system of the gamma draw) are held to max(1e-10, 8 cond eps), the bound
backward stability allows, with the constant measured against a long-double arbiter (tests/parity_util.py).
"""
import math

import numpy as np
import pytest

from oracle import bnr_oracle as O
from parity_util import solve_tol, assert_close_normwise, rel_err, note

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def make_problem(seed, V, R, n, dense=True):
    rng = np.random.default_rng(seed)
    q = V * (V + 1) // 2
    if dense:
        X = rng.normal(size=(n, q))
    else:
        X = (rng.random((n, q)) < 0.3) * (0.13 + rng.gamma(1.2, 0.2, size=(n, q)))
    y = 3.0 + X[:, : min(q, 5)].sum(axis=1) + rng.normal(size=n)
    return X, y


def random_state(rng, V, R):
    q = V * (V + 1) // 2
    A = rng.normal(size=(R, R))
    st = dict(tau2=float(rng.gamma(3.0) + 0.2), u=rng.normal(size=(R, V)), xi=(rng.random(V) < 0.6).astype(float),
              gamma=rng.normal(size=q) * 2, S=rng.gamma(1.0, size=q) + 1e-3, theta=float(rng.gamma(2.0) + 0.1),
              Delta=float(rng.uniform(0.1, 0.9)), M=A @ A.T / R + np.eye(R), mu=float(rng.normal()),
              lam=rng.choice([0.0, 1.0, -1.0], size=R), pi=rng.dirichlet([1, 1, 1], size=R))
    st["u"] = st["u"] * st["xi"][None, :]
    return st


def sweep_injection(rng, n, V, R, K):
    lay = O.draw_layout(n, V, R, K)
    inj = rng.normal(size=lay["_total"])
    for name in ("tau2", "theta", "pi"):
        o, s = lay[name]
        inj[o:o + s] = rng.gamma(3.0, size=s)
    o, s = lay["Delta"]
    inj[o:o + s] = [rng.gamma(4.0), rng.gamma(2.0), rng.random()]
    o, s = lay["M"]
    inj[o:o + R] = rng.chisquare(10, size=R)
    for name in ("S", "lambda"):
        o, s = lay[name]
        inj[o:o + s] = rng.random(s)
    o, s = lay["uxi"]
    inj[o:o + s:R + 1] = rng.random(V)
    return inj, lay


def close(a, b, rtol=RTOL, atol=0.0, msg=""):
    np.testing.assert_allclose(np.asarray(a), np.asarray(b), rtol=rtol, atol=atol, err_msg=msg)


@pytest.fixture(scope="module")
def small(bnr):
    V, R, n, C, K = 7, 4, 23, 3, 64
    X, y = make_problem(11, V, R, n)
    eng = bnr.Engine(X, y, R, num_chains=C, seed=5, gig_inject_len=K, gamma_mode="nform")
    eng.enable_aux(True)
    rng = np.random.default_rng(2)
    states = [random_state(rng, V, R) for _ in range(C)]
    injs = [sweep_injection(rng, n, V, R, K) for _ in range(C)]
    yield dict(eng=eng, X=X, y=y, V=V, R=R, n=n, C=C, K=K, states=states,
               inj=np.stack([i[0] for i in injs]), lay=injs[0][1])
    eng.close()


def _load(p, states=None):
    eng = p["eng"]
    for c, st in enumerate(states or p["states"]):
        eng.set_state_dict(c, st)
    eng.set_injection(p["inj"])


def _seg(p, c, name):
    o, s = p["lay"][name]
    return p["inj"][c, o:o + s]


def test_abi_version_and_sizes(small, bnr):
    assert bnr.lib().bnr_version() == 200
    eng = small["eng"]
    assert eng.injection_size() == small["lay"]["_total"]
    assert eng.injection_size(for_init=True) == O.init_layout(small["V"], small["R"])["_total"]


def test_state_roundtrip(small):
    _load(small)
    eng = small["eng"]
    for c, st in enumerate(small["states"]):
        got = eng.get_state_dict(c)
        for k in st:
            np.testing.assert_array_equal(np.asarray(got[k]), np.asarray(st[k]), err_msg=k)


def test_tau2(small):
    p = small
    _load(p)
    p["eng"].step("tau2")
    for c, st in enumerate(p["states"]):
        want = O.update_tau2(p["X"], p["y"], p["V"], st["mu"], st["gamma"], st["u"], st["lam"], st["S"],
                             _seg(p, c, "tau2")[0])
        aux = p["eng"].get_aux(c, "tau2_params")
        close(aux, [want["shape"], want["scale"]])
        close(p["eng"].get_state(c, "tau2")[0, 0], want["tau2"])


def test_u_xi(small):
    p = small
    _load(p)
    eng, V, R = p["eng"], p["V"], p["R"]
    eng.step("u_xi")
    for c, st in enumerate(p["states"]):
        uz = _seg(p, c, "uxi").reshape(V, R + 1)
        want = O.update_u_xi(V, st["tau2"], st["u"], st["lam"], st["S"], st["gamma"], st["Delta"], st["M"],
                             uz[:, 0], uz[:, 1:], literal=True)
        sig = eng.get_aux(c, "sigma_inv").reshape(V, R, R)
        ch = eng.get_aux(c, "sigma_chol").reshape(V, R, R)
        mt = eng.get_aux(c, "mu_t").reshape(V, R)
        lo = eng.get_aux(c, "log_odds")
        worst = 1.0
        for k in range(V):
            nd = want["nodes"][k]
            tol = solve_tol(np.linalg.cond(nd["Sigma_inv"]))
            worst = max(worst, np.linalg.cond(nd["Sigma_inv"]))
            close(sig[k].T, nd["Sigma_inv"], atol=1e-13, msg="Sigma_inv")
            assert_close_normwise(ch[k].T, nd["chol"], tol, "chol")            # stored col-major
            assert_close_normwise(mt[k], nd["mu_t"], tol, "mu_t")
            note(test="u_xi", node=k, cond=float(np.linalg.cond(nd["Sigma_inv"])), e_chol=rel_err(ch[k].T, nd["chol"]),
                 e_mu=rel_err(mt[k], nd["mu_t"]), e_logodds=abs(lo[k] - nd["log_odds"]) / max(1.0, abs(nd["log_odds"])))
            # literal (V-1)-dim densities (a dense (V-1) x (V-1) factorisation) vs the R x R identity
            assert abs(lo[k] - nd["log_odds"]) <= 1e-10 * max(1.0, abs(nd["log_odds"])) * max(1.0, 1e-2 * worst)
        np.testing.assert_array_equal(eng.get_state(c, "xi")[:, 0], want["xi"])
        assert_close_normwise(eng.get_state(c, "u"), want["u"], solve_tol(worst), "u")
    assert not (eng.status() & 2).any()


def test_gamma(small):
    p = small
    _load(p)
    eng, n = p["eng"], p["n"]
    eng.step("gamma")
    for c, st in enumerate(p["states"]):
        want = O.update_gamma(p["X"], p["y"], st["tau2"], st["u"], st["lam"], st["S"], st["mu"],
                              _seg(p, c, "gamma_z1"), _seg(p, c, "gamma_z2"))
        cond = np.linalg.cond(want["G"])
        close(eng.get_aux(c, "W"), want["W"], atol=1e-14)
        G = eng.get_aux(c, "G").reshape(n, n).T
        close(G, want["G"], atol=1e-12 * np.abs(want["G"]).max(), msg="G")
        Lg = eng.get_aux(c, "G_chol").reshape(n, n).T
        tol = solve_tol(cond)
        assert_close_normwise(Lg, np.linalg.cholesky(want["G"]), tol, "chol(G)")
        assert_close_normwise(eng.get_aux(c, "a4"), want["a4"], tol, "a4")
        assert_close_normwise(eng.get_state(c, "gamma")[:, 0], want["gamma"], tol, "gamma")
        note(test="gamma", cond=float(cond), e_chol=rel_err(Lg, np.linalg.cholesky(want["G"])),
             e_a4=rel_err(eng.get_aux(c, "a4"), want["a4"]), e_gamma=rel_err(eng.get_state(c, "gamma")[:, 0], want["gamma"]))
    assert not (eng.status() & 4).any()


def test_gamma_qform(bnr):
    """q x q precision form (BASELINE north_star): P, chol(P), conditional mean and the draw given injected z."""
    V, R, n, C, K = 7, 4, 40, 3, 64
    q = V * (V + 1) // 2
    X, y = make_problem(21, V, R, n)
    rng = np.random.default_rng(8)
    states = [random_state(rng, V, R) for _ in range(C)]
    injs = [sweep_injection(rng, n, V, R, K) for _ in range(C)]
    inj, lay = np.stack([i[0] for i in injs]), injs[0][1]
    with bnr.Engine(X, y, R, num_chains=C, seed=5, gig_inject_len=K, gamma_mode="qform") as eng:
        assert eng.gamma_mode == "qform"
        eng.enable_aux(True)
        for c, st in enumerate(states):
            eng.set_state_dict(c, st)
        eng.set_injection(inj)
        eng.step("gamma")
        for c, st in enumerate(states):
            o, s = lay["gamma_z1"]
            want = O.update_gamma_qform(X, y, st["tau2"], st["u"], st["lam"], st["S"], st["mu"], inj[c, o:o + s])
            cond = np.linalg.cond(want["P"])
            P = eng.get_aux(c, "G").reshape(q, q).T
            close(P, want["P"], atol=1e-13 * np.abs(want["P"]).max(), msg="P")
            Lg = eng.get_aux(c, "G_chol").reshape(q, q).T
            close(Lg, want["L"], rtol=RTOL * cond, atol=1e-13 * cond, msg="chol(P)")
            close(eng.get_aux(c, "a4"), want["beta"], rtol=RTOL * cond, atol=1e-13 * cond, msg="beta")
            close(eng.get_state(c, "gamma")[:, 0], want["gamma"], rtol=RTOL * cond, atol=1e-13 * cond, msg="gamma")
        assert not (eng.status() & 4).any()
        # z = 0 gives the conditional mean, which is also the reference's Bhattacharya draw with z1 = z2 = 0
        inj0 = inj.copy()
        o, s = lay["gamma_z1"]; inj0[:, o:o + s] = 0.0
        for c, st in enumerate(states):
            eng.set_state_dict(c, st)
        eng.set_injection(inj0)
        eng.step("gamma")
        for c, st in enumerate(states):
            ref = O.update_gamma(X, y, st["tau2"], st["u"], st["lam"], st["S"], st["mu"], np.zeros(q), np.zeros(n))
            cond = np.linalg.cond(ref["G"])
            close(eng.get_state(c, "gamma")[:, 0], ref["gamma"], rtol=max(1e-9, RTOL * cond), atol=1e-12 * cond, msg="mean")


def test_gamma_mode_cost_model(bnr):
    """AUTO resolves by the SURVEY 8(d) flop model: q-form iff q^3/3 + 4q^2 < n^2 q + n^3/3."""
    for V, n, want in ((6, 40, "qform"), (6, 8, "nform"), (12, 30, "nform"), (12, 60, "qform")):
        q = V * (V + 1) // 2
        X, y = make_problem(1, V, 3, n)
        with bnr.Engine(X, y, 3, num_chains=1, seed=1) as eng:
            assert (q ** 3 / 3 + 4 * q * q < n * n * q + n ** 3 / 3) == (want == "qform")
            assert eng.gamma_mode == want, (V, n)


def test_D_gig(small):
    p = small
    # cover all three GIG branches: scale some residuals down / up
    states = [dict(s) for s in p["states"]]
    rng = np.random.default_rng(4)
    for st in states:
        W = O.W_of(st["u"], st["lam"])
        q = W.shape[0]
        scale = rng.choice([1e-3, 0.3, 6.0], size=q)
        st["gamma"] = W + scale * rng.normal(size=q) * math.sqrt(st["tau2"])
    _load(p, states)
    eng, K = p["eng"], p["K"]
    eng.step("D")
    seen = set()
    for c, st in enumerate(states):
        q = st["gamma"].shape[0]
        want = O.update_D(st["gamma"], st["u"], st["lam"], st["tau2"], st["theta"], _seg(p, c, "S").reshape(q, K))
        seen |= set(want["branch"])
        close(eng.get_aux(c, "chi"), want["chi"], atol=1e-300)
        np.testing.assert_array_equal(eng.get_aux(c, "gig_used"), want["used"])
        close(eng.get_state(c, "S")[:, 0], want["S"], rtol=1e-10)
        note(test="D_gig", e_S=float(np.max(np.abs(eng.get_state(c, "S")[:, 0] / want["S"] - 1.0))))
    assert {"concave", "noshift", "shift"} <= seen
    assert not (eng.status() & (8 | 16)).any()


def test_theta_Delta_M_mu(small):
    p = small
    eng, R = p["eng"], p["R"]
    for cond in ("theta", "Delta", "M", "mu"):
        _load(p)
        eng.step(cond)
        for c, st in enumerate(p["states"]):
            if cond == "theta":
                want = O.update_theta(st["S"], 1.0, 1.0, p["V"], _seg(p, c, "theta")[0])
                close(eng.get_aux(c, "theta_params"), [want["shape"], want["scale"]])
                close(eng.get_state(c, "theta")[0, 0], want["theta"])
            elif cond == "Delta":
                dd = _seg(p, c, "Delta")
                want = O.update_Delta(st["xi"], 1.0, 1.0, dd[0], dd[1], dd[2])
                close(eng.get_aux(c, "delta_params"), [want["a"], want["b"]])
                close(eng.get_state(c, "Delta")[0, 0], want["Delta"])
            elif cond == "M":
                mm = _seg(p, c, "M")
                want = O.update_M(st["u"], st["xi"], 10, mm[:R], mm[R:])
                aux = eng.get_aux(c, "m_params")
                assert aux[0] == want["df"]
                close(aux[1:1 + R * R].reshape(R, R).T, want["Psi"])
                close(aux[1 + R * R:].reshape(R, R).T, want["chol_Psi"], atol=1e-14)
                assert_close_normwise(eng.get_state(c, "M"), want["M"], solve_tol(np.linalg.cond(want["Psi"])), "M")
                note(test="M", cond=float(np.linalg.cond(want["Psi"])), e_M=rel_err(eng.get_state(c, "M"), want["M"]))
            else:
                want = O.update_mu(p["X"] @ st["gamma"], p["y"], st["tau2"], _seg(p, c, "mu")[0])
                close(eng.get_aux(c, "mu_params"), [want["mean"], want["sd"]], rtol=1e-10, atol=1e-13)
                close(eng.get_state(c, "mu")[0, 0], want["mu"], rtol=1e-10, atol=1e-13)


def test_lambda_pi(small):
    p = small
    eng, R = p["eng"], p["R"]
    _load(p)
    eng.step("lam")
    lam_new = []
    for c, st in enumerate(p["states"]):
        want = O.update_lambda(st["gamma"], st["u"], st["S"], st["tau2"], st["lam"], st["pi"], _seg(p, c, "lambda"))
        lw = eng.get_aux(c, "lambda_logw").reshape(3, R).T
        ref = want["loglik"] - want["loglik"].max(axis=1, keepdims=True)
        # the reference sums q log-densities (|loglik| ~ 1e2..1e4) and subtracts; the engine sums only the differences:
        # the absolute error of a log-weight is eps-relative to the magnitude of those sums, and a weight
        # pi * exp(logw) inherits it as a relative error
        mag = float(np.max(np.abs(want["loglik"])))
        tol_l = max(1e-10, 64 * mag * 2.2e-16)
        close(lw, ref, rtol=tol_l, atol=tol_l * max(1.0, mag * 1e-3), msg="loglik - max")
        w = eng.get_aux(c, "lambda_weights").reshape(3, R).T
        close(w, want["weights"], rtol=10 * tol_l * max(1.0, mag * 1e-3), atol=1e-300)
        note(test="lambda", mag=mag, e_logw=float(np.max(np.abs(lw - ref))),
             e_w=float(np.max(np.abs(w / np.where(want["weights"] > 0, want["weights"], 1.0) - 1.0))))
        np.testing.assert_array_equal(eng.get_state(c, "lam")[:, 0], want["lam"])
        lam_new.append(want["lam"])
    eng.step("pi")
    for c, st in enumerate(p["states"]):
        want = O.update_pi(lam_new[c], 1.01, _seg(p, c, "pi").reshape(R, 3))
        close(eng.get_aux(c, "pi_alpha").reshape(3, R).T, want["alpha"])
        close(eng.get_state(c, "pi"), want["pi"])


@pytest.mark.parametrize("V,R,n,dense,mode", [(7, 4, 23, True, "nform"), (12, 5, 150, False, "nform"),
                                              (20, 7, 300, True, "nform"), (7, 4, 23, True, "qform"),
                                              (18, 5, 150, False, "qform"), (22, 7, 300, True, "qform"),
                                              # edge cases: smallest network, single sample, n a multiple of 128
                                              # (extra padding block for the bordering row), R at its maximum
                                              (2, 1, 3, True, "nform"), (3, 2, 1, True, "nform"), (2, 1, 5, True, "qform"),
                                              (6, 3, 128, True, "nform"), (4, 16, 30, True, "qform"),
                                              # the bordering row on the last row of the matrix (n + 1 = 128, 1024)
                                              (6, 3, 127, True, "nform"), (6, 3, 1023, True, "nform")])
def test_full_sweeps_injected(bnr, V, R, n, dense, mode):
    """bnr_run (production schedule, fused kernels) == oracle gibbs_sweep for consecutive sweeps; the larger
    cases span several 128-row tiles and 64-column Cholesky panels."""
    C, K = 2, 64
    X, y = make_problem(V * 100 + n, V, R, n, dense)
    rng = np.random.default_rng(V)
    hyper = dict(O.DEFAULT_HYPER)
    if R > 9:
        hyper["nu"] = R + 4              # InverseWishart needs nu > R - 1
    with bnr.Engine(X, y, R, num_chains=C, seed=1, gig_inject_len=K, trace_rows=4, gamma_mode=mode,
                    nu=hyper["nu"]) as eng:
        init = np.stack([_init_injection(rng, V, R) for _ in range(C)])
        eng.set_injection(init)
        eng.init_state()
        sts = [O.initialize_state(V, R, hyper, init[c]) for c in range(C)]
        for c in range(C):
            got = eng.get_state_dict(c)
            for k in sts[c]:
                close(got[k], sts[c][k], rtol=1e-12, atol=1e-14, msg="init " + k)
        for sweep in range(2):
            inj = np.stack([sweep_injection(rng, n, V, R, K)[0] for _ in range(C)])
            eng.set_injection(inj)
            eng.run(1)
            for c in range(C):
                new, aux = O.gibbs_sweep(sts[c], X, y, V, R, hyper, inj[c], K, literal=False,
                                         gamma_form="q" if mode == "qform" else "n")
                cond = np.linalg.cond(aux["gamma"]["P" if mode == "qform" else "G"])
                got = eng.get_state_dict(c)
                # the second sweep starts from the first one's output: its inputs already differ by the first sweep's
                # tolerance, hence the factor 8 there
                tol = solve_tol(cond) * (8.0 if sweep else 1.0)
                for k in ("tau2", "xi", "lam"):
                    close(got[k], new[k], rtol=1e-10 * (8.0 if sweep else 1.0), msg=k)
                for k in ("u", "gamma", "S", "theta", "Delta", "M", "mu", "pi"):
                    assert_close_normwise(got[k], new[k], tol, "%s sweep %d" % (k, sweep))
                note(test="full_sweep", V=V, n=n, mode=mode, sweep=sweep, cond=float(cond),
                     worst=max(rel_err(got[k], new[k]) for k in ("u", "gamma", "S", "theta", "Delta", "M", "mu", "pi")))
                sts[c] = new
            assert eng.iteration == sweep + 1
        assert not eng.status().any()
        # trace rows: row 0 = init, rows 1..2 = the sweeps
        g = eng.get_trace(0, "gamma", 0, 3)
        close(g[2, :, 0], sts[0]["gamma"], rtol=1e-6)
        assert eng.get_trace(0, "pi", 1, 3).shape == (2, R, 3)


def _init_injection(rng, V, R):
    il = O.init_layout(V, R)
    inj = np.empty(il["_total"])
    o, s = il["S"]; inj[o:o + s] = rng.exponential(size=s)
    o, s = il["pi"]; inj[o:o + s] = rng.gamma(2.0, size=s)
    o, s = il["lambda"]; inj[o:o + s] = rng.random(s)
    o, s = il["xi"]; inj[o:o + s] = rng.random(s)
    o, s = il["M"]; inj[o:o + R] = rng.chisquare(10, size=R); inj[o + R:o + s] = rng.normal(size=s - R)
    o, s = il["u"]; inj[o:o + s] = rng.normal(size=s)
    o, s = il["gamma"]; inj[o:o + s] = rng.normal(size=s)
    return inj


def test_step_sequence_equals_run(bnr):
    """Ten bnr_step calls in gibbs_sample! order == one bnr_run sweep (same Philox draws)."""
    V, R, n, C = 9, 3, 40, 2
    X, y = make_problem(3, V, R, n)
    with bnr.Engine(X, y, R, num_chains=C, seed=77) as a, bnr.Engine(X, y, R, num_chains=C, seed=77) as b:
        a.init_state(); b.init_state()
        a.run(1)
        for cond in ("tau2", "u_xi", "gamma", "D", "theta", "Delta", "M", "mu", "lam", "pi"):
            b.step(cond)
        b.finish_sweep()
        for c in range(C):
            sa, sb = a.get_state_dict(c), b.get_state_dict(c)
            for k in sa:
                np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg=k)
        assert a.iteration == b.iteration == 1
