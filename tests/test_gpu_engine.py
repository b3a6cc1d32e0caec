"""Engine-level GPU tests: RNG streams, chain batching invariance, R-hat / traces on device, the Fit/Summary
drop-in surface, level-2 (posterior) agreement with the oracle chain and with the reference's golden run, and
size-independent properties at the benchmark's full size (V=100, n=1000)."""
import math

import numpy as np
import pytest
from scipy import stats

from oracle import bnr_oracle as O
from oracle import chain as OC

pytestmark = pytest.mark.gpu


def _toy(seed=0, V=6, R=3, n=30):
    rng = np.random.default_rng(seed)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q))
    y = 2.0 + X[:, 1] * 1.5 + rng.normal(size=n)
    return X, y


def test_rng_streams(bnr):
    X, y = _toy()
    with bnr.Engine(X, y, 3, num_chains=2, seed=123) as eng:
        u = eng.rng_stream(0, 5, 5, 17, "uniform", 20000)
        z = eng.rng_stream(1, 5, 3, 2, "normal", 20000)
        assert 0 < u.min() and u.max() < 1
        assert stats.kstest(u, "uniform").pvalue > 1e-3
        assert stats.kstest(z, "norm").pvalue > 1e-3
        for shape in (0.4, 1.0, 7.5, 2525.5):
            g = eng.rng_gamma(0, 9, 6, 0, shape, 20000)
            assert stats.kstest(g, "gamma", args=(shape,)).pvalue > 1e-3, shape
        # streams are keyed by (chain, iteration, site, element): all distinct, all reproducible
        a = eng.rng_stream(0, 5, 5, 17, "uniform", 8)
        np.testing.assert_array_equal(a, u[:8])
        for other in (eng.rng_stream(1, 5, 5, 17, "uniform", 8), eng.rng_stream(0, 6, 5, 17, "uniform", 8),
                      eng.rng_stream(0, 5, 4, 17, "uniform", 8), eng.rng_stream(0, 5, 5, 18, "uniform", 8)):
            assert not np.array_equal(a, other)


def test_philox_known_answer(bnr):
    """Philox4x32-10 KAT (Random123 kat_vectors: ctr = key = 0 -> 6627e8d5 e169c58d bc57ac4c 9b00dbd8): the first
    uniform of chain 0 / seed 0 / iteration 0 / site 0 / element 0 is built from words 0 and 1."""
    X, y = _toy()
    with bnr.Engine(X, y, 3, num_chains=1, seed=0) as eng:
        u = eng.rng_stream(0, 0, 0, 0, "uniform", 2)
    w = [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    want0 = (((w[1] << 32 | w[0]) >> 11) + 0.5) / 2 ** 53
    want1 = (((w[3] << 32 | w[2]) >> 11) + 0.5) / 2 ** 53
    assert u[0] == want0 and u[1] == want1


def test_chain_batching_invariance(bnr):
    """Chains are keyed by GLOBAL id: a handle holding chains 2..3 reproduces chains 2..3 of a 4-chain handle
    bit for bit (what makes 1/2/4/8-GPU sharding a pure partition)."""
    X, y = _toy(1, V=8, R=4, n=50)
    with bnr.Engine(X, y, 4, num_chains=4, seed=9) as a, \
            bnr.Engine(X, y, 4, num_chains=2, seed=9, chain_offset=2) as b:
        for e in (a, b):
            e.init_state()
            e.run(25)
        for c in range(2):
            sa, sb = a.get_state_dict(c + 2), b.get_state_dict(c)
            for k in sa:
                np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg=k)
        # and a run is reproducible / resumable: 25 = 10 + 15
        with bnr.Engine(X, y, 4, num_chains=4, seed=9) as c2:
            c2.init_state(); c2.run(10); c2.run(15)
            for k, v in a.get_state_dict(1).items():
                np.testing.assert_array_equal(np.asarray(v), np.asarray(c2.get_state_dict(1)[k]), err_msg=k)


def test_device_rhat_matches_oracle(bnr, golden):
    """On-device R-hat (streaming Welford moments AND two-pass from traces) == oracle rhat on the same traces
    to 1e-10; the oracle itself reproduces the reference's stored R-hat exactly (test_oracle_golden)."""
    X, y = golden["test1.X"], golden["test1.y"]
    C, nburn, nsamp = 4, 60, 101      # odd nsamp: the middle draw is dropped
    with bnr.Engine(X, y, 5, num_chains=C, seed=4, trace_rows=nburn + nsamp + 1) as eng:
        eng.init_state()
        eng.set_moment_window(nburn + 1, nsamp)
        eng.run(nburn + nsamp)
        rx_s, rg_s = eng.rhat()
        eng.moments_from_trace(nburn + 1, nsamp)
        rx_t, rg_t = eng.rhat()
        tg = np.stack([eng.get_trace(c, "gamma", nburn + 1, nburn + 1 + nsamp)[:, :, 0] for c in range(C)], axis=2)
        tx = np.stack([eng.get_trace(c, "xi", nburn + 1, nburn + 1 + nsamp)[:, :, 0] for c in range(C)], axis=2)
        assert not eng.status().any()
    want_g, want_x = O.rhat(tg), O.rhat(tx)
    for got_g, got_x in ((rg_s, rx_s), (rg_t, rx_t)):
        np.testing.assert_allclose(got_g, want_g, rtol=1e-10)
        fin = np.isfinite(want_x)
        np.testing.assert_allclose(got_x[fin], want_x[fin], rtol=1e-10)
        np.testing.assert_array_equal(np.isfinite(got_x), fin)


def test_fit_summary_dropin(bnr, tmp_path):
    """Fit!/Summary surface (src/gibbs.jl:725-751, 1214-1250): keyword names, Results fields, table shapes in
    reference layout, Summary == oracle summary of the returned traces."""
    rng = np.random.default_rng(1234)
    Xl = []
    for _ in range(10):
        A = (rng.random((4, 4)) < 0.5).astype(float)
        Xl.append(np.tril(A) + np.tril(A, -1).T)
    y = 12 + rng.normal(0, 2, size=10)
    log = tmp_path / "parameters.log"
    res = bnr.Fit(Xl, y, 5, η=1.01, ζ=1.0, ι=1.0, aΔ=1.0, bΔ=1.0, ν=10, nburn=300, nsamples=100,
                  psrf_cutoff=1e9, x_transform=True, num_chains=2, seed=1234, filename=str(log))
    assert res.burn_in == 300 and res.sampled == 100
    st = res.state
    assert st["γ"].shape == (400, 10, 1) and st["u"].shape == (400, 5, 4) and st["πᵥ"].shape == (400, 5, 3)
    assert st["M"].shape == (400, 5, 5) and st["τ²"].shape == (400, 1, 1) and st.xi.shape == (400, 4, 1)
    assert st["θ"][0, 0, 0] == 0.5 and st["μ"][0, 0, 0] == 1.0 and st["τ²"][0, 0, 0] == 1.0   # row 1 = prior init
    np.testing.assert_allclose(st["πᵥ"].sum(axis=2), 1.0, rtol=1e-12)
    assert set(np.unique(st["λ"])) <= {-1.0, 0.0, 1.0} and set(np.unique(st["ξ"])) <= {0.0, 1.0}
    assert res.rhatγ.γ.shape == (10,) and res.rhatξ.ξ.shape == (4,)
    assert "seed=1234" in log.read_text() and "nburn=300" in log.read_text()
    out = bnr.Summary(res)
    want = O.summary(st["γ"][300:400, :, 0], st["ξ"][300:400, :, 0])
    for k in ("node1", "node2", "estimate", "lower_bound", "upper_bound"):
        np.testing.assert_array_equal(out.edge_coef[k], want[k], err_msg=k)
    np.testing.assert_array_equal(out.prob_nodes["probability"], want["probability"])
    assert out.ci_level == 95
    assert res.extra["device_summary"] is not None and res.extra["gamma_mode"] in ("nform", "qform")
    # the same fit without copying any table back: Summary comes from the device reduction alone
    res0 = bnr.Fit(Xl, y, 5, nburn=300, nsamples=100, psrf_cutoff=1e9, num_chains=2, seed=1234, filename=None,
                   return_state="none")
    out0 = bnr.Summary(res0)
    assert len(res0.state) == 0
    for k in ("estimate", "lower_bound", "upper_bound"):
        np.testing.assert_array_equal(out0.edge_coef[k], out.edge_coef[k], err_msg=k)
    np.testing.assert_array_equal(out0.prob_nodes["probability"], out.prob_nodes["probability"])
    out90 = bnr.Summary(res, interval=90)        # not the interval reduced on the device: host order statistics
    want90 = O.summary(st["γ"][300:400, :, 0], st["ξ"][300:400, :, 0], interval=90)
    np.testing.assert_array_equal(out90.edge_coef["upper_bound"], want90["upper_bound"])
    with pytest.raises(ValueError):
        bnr.Summary(res0, interval=90)
    with pytest.raises(IndexError):
        bnr.Summary(bnr.Results(bnr.Table(gamma=st["γ"][:10], xi=st["ξ"][:10]), [], [], 0, 10))


def test_fit_purge_burn_and_extension(bnr):
    """purge_burn ring (src/gibbs.jl:857-860) keeps only nsamp + purge rows yet yields the same retained draws;
    the PSRF loop extends burn-in by nburn exactly once when it cannot converge (maxburn = nburn + nsamp)."""
    X, y = _toy(2, V=5, R=3, n=25)
    kw = dict(nburn=40, nsamples=30, num_chains=2, seed=3, x_transform=False, filename=None)
    a = bnr.Fit(X, y, 3, psrf_cutoff=1e9, **kw)
    b = bnr.Fit(X, y, 3, psrf_cutoff=1e9, purge_burn=10, **kw)
    assert len(a.state) == 70 and len(b.state) == 40 and b.burn_in == 10
    np.testing.assert_array_equal(a.state["γ"][40:70], b.state["γ"][10:40])
    np.testing.assert_array_equal(a.rhatγ.γ, b.rhatγ.γ)
    assert a.extra["rhat_streamed"] and b.extra["rhat_streamed"]
    # the streamed split-half moments give the R-hat of exactly rows nburn+1 .. nburn+nsamp of every chain
    with bnr.Engine(X, y, 3, num_chains=2, seed=3, trace_rows=70) as eng:
        eng.init_state()
        eng.run(69)
        eng.moments_from_trace(40, 30)
        rx, rg = eng.rhat()
    np.testing.assert_allclose(a.rhatγ.γ, rg, rtol=1e-9)
    fin = np.isfinite(rx)
    np.testing.assert_allclose(a.rhatξ.ξ[fin], rx[fin], rtol=1e-9)
    e = bnr.Fit(X, y, 3, psrf_cutoff=1e9, nburn=20, nsamples=30, num_chains=2, seed=3, x_transform=False, filename=None)
    assert not e.extra["rhat_streamed"] and len(e.state) == 50          # nburn < nsamp: trace-based R-hat
    c = bnr.Fit(X, y, 3, psrf_cutoff=0.0, **kw)       # never "converged"
    assert c.extra["tot_generated"] == 70 + 40 and len(c.state) == 70
    with bnr.Engine(X, y, 3, num_chains=2, seed=3, trace_rows=110) as eng:     # 69 + 40 sweeps, last 30 retained
        eng.init_state()
        eng.run(109)
        eng.moments_from_trace(80, 30)
        _, rg2 = eng.rhat()
    np.testing.assert_allclose(c.rhatγ.γ, rg2, rtol=1e-9)
    np.testing.assert_array_equal(c.state["γ"][:30], a.state["γ"][40:70])   # old samples moved to the front
    d = bnr.Fit(X, y, 3, mingen=40, maxgen=120, psrf_cutoff=0.0, num_chains=2, seed=3, x_transform=False,
                filename=None)
    assert d.extra["tot_generated"] == 120 and d.burn_in == 20 and d.sampled == 60 and len(d.state) == 80


def _batch_se(x, nb=10):
    m = len(x) // nb
    bm = x[: m * nb].reshape(nb, m, *x.shape[1:]).mean(axis=1)
    return bm.std(axis=0, ddof=1) / math.sqrt(nb)


def test_posterior_matches_oracle_chain(bnr, golden):
    """Level-2 parity: posterior summaries of the GPU sampler agree with the CPU oracle's own Gibbs run on the
    same data (reference test data test1.csv, R=5) within 4 Monte-Carlo standard errors (batch means)."""
    X, y = golden["test1.X"], golden["test1.y"]
    nburn, nsamp, C = 600, 1000, 8
    with bnr.Engine(X, y, 5, num_chains=C, seed=2024, trace_rows=nburn + nsamp + 1, trace_full_chains=C) as eng:
        eng.init_state()
        eng.run(nburn + nsamp)
        gp = {k: np.stack([eng.get_trace(c, k, nburn + 1, nburn + nsamp + 1) for c in range(C)])
              for k in ("gamma", "xi", "tau2", "mu", "theta", "Delta")}
        assert not (eng.status() & ~1).any()
    ora = []
    for s in range(3):
        tr, _ = OC.run_chain(X, y, 5, nburn + nsamp, seed=100 + s)
        ora.append({k: v[nburn + 1:] for k, v in tr.items()})
    failures = []
    for k in ("tau2", "mu", "theta", "Delta", "gamma", "xi"):
        g = np.concatenate([gp[k][c].reshape(nsamp, -1) for c in range(C)])
        o = np.concatenate([t[k].reshape(nsamp, -1) for t in ora])
        se = np.sqrt(_batch_se(g, 20) ** 2 + _batch_se(o, 15) ** 2)
        z = np.abs(g.mean(axis=0) - o.mean(axis=0)) / np.maximum(se, 1e-12)
        # 4 s.e. on every coordinate; allow the expected handful of batch-means underestimates in 190 edges
        frac = float(np.mean(z > 4.0))
        if frac > 0.03:
            failures.append((k, frac, float(z.max())))
    assert not failures, failures


def test_posterior_vs_reference_golden(bnr, golden):
    """The reference's own stored run (res2: seed 1234, ONE chain, 200 burn-in + 200 retained draws on
    test1.csv, test/test1-generate-samples-test.jl:10-12) is a real Julia sample of this run protocol.  The GPU
    sampler replays the same protocol on 96 independent chains; every summary of the Julia run must lie within
    4 standard deviations of the replicate distribution (chains this short have not converged, so the replicate
    spread -- not a within-chain s.e. -- is the honest yardstick)."""
    X, y = golden["test1.X"], golden["test1.y"]
    nburn, nsamp, C = 200, 200, 96
    with bnr.Engine(X, y, 5, num_chains=C, seed=7, trace_rows=nburn + nsamp, trace_full_chains=C,
                    trace_gamma_xi_all=False) as eng:
        eng.init_state()
        eng.run(nburn + nsamp - 1)          # rows 1..400 of the reference table = init + 399 sweeps
        rep = {k: np.stack([eng.get_trace(c, k, nburn, nburn + nsamp).reshape(nsamp, -1) for c in range(C)])
               for k in ("tau2", "mu", "theta", "Delta", "xi", "gamma", "S")}
        assert not (eng.status() & ~1).any()
    ref = {k: golden["res2." + k][nburn:nburn + nsamp].reshape(nsamp, -1) for k in rep}
    stats_ = {
        "mean tau2": lambda t: t["tau2"].mean(axis=-2)[..., 0],
        "mean mu": lambda t: t["mu"].mean(axis=-2)[..., 0],
        "mean theta": lambda t: t["theta"].mean(axis=-2)[..., 0],
        "mean Delta": lambda t: t["Delta"].mean(axis=-2)[..., 0],
        "mean xi": lambda t: t["xi"].mean(axis=(-2, -1)),
        "mean |gamma|": lambda t: np.abs(t["gamma"]).mean(axis=(-2, -1)),
        "mean log S": lambda t: np.log(t["S"]).mean(axis=(-2, -1)),
        "sd tau2": lambda t: t["tau2"].std(axis=-2)[..., 0],
    }
    bad = []
    for name, f in stats_.items():
        r = f(rep)
        z = (f(ref) - r.mean()) / r.std(ddof=1)
        if abs(z) > 4.0:
            bad.append((name, float(z), float(f(ref)), float(r.mean()), float(r.std(ddof=1))))
    assert not bad, bad


def test_full_size_properties(bnr):
    """BASELINE config 3 shape (V=100, q=5050, n=1000, R=7): size-independent properties of the gamma draw's
    linear algebra -- L L' = X D X' + I, G a4 = rhs -- and sane chain output after a few sweeps."""
    V, R, n, C = 100, 7, 1000, 2
    rng = np.random.default_rng(0)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q))
    y = 55 + X[:, :20].sum(axis=1) + rng.normal(0, 10, size=n)
    with bnr.Engine(X, y, R, num_chains=C, seed=1) as eng:
        eng.init_state()
        eng.run(2)
        eng.enable_aux(True)
        S_old = eng.get_state(0, "S")[:, 0].copy()
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        G = eng.get_aux(0, "G").reshape(n, n).T
        L = eng.get_aux(0, "G_chol").reshape(n, n).T
        a4 = eng.get_aux(0, "a4")
        want = (X * S_old[None, :]) @ X.T + np.eye(n)
        scale = np.abs(want).max()
        assert np.abs(G - want).max() <= 1e-12 * scale
        assert np.abs(G - G.T).max() == 0.0
        assert np.abs(L @ L.T - want).max() <= 1e-11 * scale
        assert np.all(np.diag(L) > 0) and np.all(np.triu(L, 1) == 0)
        assert np.isfinite(a4).all()
        for cond in ("D", "theta", "Delta", "M", "mu", "lam", "pi"):
            eng.step(cond)
        eng.finish_sweep()
        eng.enable_aux(False)
        eng.run(3)
        st = eng.get_state_dict(1)
        assert eng.iteration == 6 and not eng.status().any()
        assert np.isfinite(st["gamma"]).all() and (st["S"] > 0).all() and st["tau2"] > 0
        np.testing.assert_allclose(st["pi"].sum(axis=1), 1.0, rtol=1e-12)
        ev = np.linalg.eigvalsh(st["M"])
        assert ev.min() > 0


def test_qform_and_nform_sample_the_same_posterior(bnr, golden):
    """The q x q precision draw and the reference's n x n Bhattacharya draw are two samplers of one conditional:
    full Gibbs runs under either formulation must agree on every posterior mean within 4 Monte-Carlo s.e."""
    X, y = golden["test1.X"], golden["test1.y"]
    nburn, nsamp, C = 500, 800, 12
    out = {}
    for mode in ("nform", "qform"):
        with bnr.Engine(X, y, 5, num_chains=C, seed=31 if mode == "nform" else 32, trace_rows=nburn + nsamp + 1,
                        trace_full_chains=C, gamma_mode=mode) as eng:
            assert eng.gamma_mode == mode
            eng.init_state()
            eng.run(nburn + nsamp)
            out[mode] = {k: np.concatenate([eng.get_trace(c, k, nburn + 1, nburn + nsamp + 1).reshape(nsamp, -1)
                                            for c in range(C)]) for k in ("gamma", "xi", "tau2", "mu", "theta", "Delta")}
            assert not (eng.status() & ~1).any()
    failures = []
    for k in ("tau2", "mu", "theta", "Delta", "gamma", "xi"):
        a, b = out["nform"][k], out["qform"][k]
        se = np.sqrt(_batch_se(a, 24) ** 2 + _batch_se(b, 24) ** 2)
        z = np.abs(a.mean(axis=0) - b.mean(axis=0)) / np.maximum(se, 1e-12)
        frac = float(np.mean(z > 4.0))
        if frac > 0.03:
            failures.append((k, frac, float(z.max())))
    assert not failures, failures


def test_qform_full_size_properties(bnr):
    """BASELINE config 2 shape (V=30, q=465, n=500, R=7), where the cost model picks the q x q form:
    L L' = P = (X'X + D^-1)/tau2 and P beta = X'(y - mu - XW)/tau2 + L z at full size."""
    V, R, n, C = 30, 7, 500, 3
    rng = np.random.default_rng(1)
    q = V * (V + 1) // 2
    X = (rng.random((n, q)) < 0.5) * (0.13 + rng.gamma(1.2, 0.2, size=(n, q)))
    X[:, np.cumsum([0] + [V - k for k in range(V - 1)])] = 0.0        # zero diagonal columns, like the shipped example
    y = 55 + X[:, :20].sum(axis=1) + rng.normal(0, 10, size=n)
    with bnr.Engine(X, y, R, num_chains=C, seed=1) as eng:
        assert eng.gamma_mode == "qform"
        eng.init_state()
        eng.run(2)
        eng.enable_aux(True)
        S_old = eng.get_state(1, "S")[:, 0].copy()
        mu_old = float(eng.get_state(1, "mu")[0, 0])
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        tau2 = float(eng.get_state(1, "tau2")[0, 0])
        P = eng.get_aux(1, "G").reshape(q, q).T
        L = eng.get_aux(1, "G_chol").reshape(q, q).T
        beta = eng.get_aux(1, "a4")
        W = eng.get_aux(1, "W")
        want = (X.T @ X + np.diag(1.0 / S_old)) / tau2
        scale = np.abs(want).max()
        assert np.abs(P - want).max() <= 1e-13 * scale
        assert np.abs(L @ L.T - want).max() <= 1e-12 * scale
        b = X.T @ ((y - mu_old - X @ W) / tau2)
        zrec = np.linalg.solve(L, want @ beta - b)            # P beta - b = L z
        for j in (0, 17, q - 1):                              # site GAMMA_Z1 = 3 (bnr_rng.cuh), sweep 3
            z = eng.rng_stream(1, 3, 3, j, "normal", 1)[0]
            assert abs(zrec[j] - z) <= 1e-6, (j, zrec[j], z)
        np.testing.assert_allclose(eng.get_state(1, "gamma")[:, 0], W + beta, rtol=1e-14)
        for cond in ("D", "theta", "Delta", "M", "mu", "lam", "pi"):
            eng.step(cond)
        eng.finish_sweep()
        eng.enable_aux(False)
        eng.run(5)
        st = eng.get_state_dict(2)
        assert eng.iteration == 8 and not (eng.status() & ~1).any()
        assert np.isfinite(st["gamma"]).all() and (st["S"] > 0).all() and st["tau2"] > 0


def test_device_summary_and_ess_match_oracle(bnr, golden):
    """Device Summary (radix-select order statistics) == the oracle's sort-based Summary bit for bit on the bounds;
    device ESS == the oracle's Geyer estimator on the same traces."""
    X, y = golden["test1.X"], golden["test1.y"]
    nburn, nsamp, C = 150, 333, 5
    with bnr.Engine(X, y, 5, num_chains=C, seed=11, trace_rows=nburn + nsamp + 1, trace_full_chains=2) as eng:
        eng.init_state()
        eng.run(nburn + nsamp)
        lw, hi = O.julia_round(nsamp * 0.025), O.julia_round(nsamp * 0.975)
        for chain in (0, 3):                       # chain 0 is read from the full-state trace, chain 3 from the gamma/xi trace
            g = eng.get_trace(chain, "gamma", nburn + 1, nburn + nsamp + 1)[:, :, 0]
            x = eng.get_trace(chain, "xi", nburn + 1, nburn + nsamp + 1)[:, :, 0]
            gm, gl, gh, xm = eng.summary(chain, nburn + 1, nsamp, lw, hi)
            gs = np.sort(g, axis=0)
            np.testing.assert_array_equal(gl, gs[lw - 1])
            np.testing.assert_array_equal(gh, gs[hi - 1])
            np.testing.assert_allclose(gm, g.mean(axis=0), rtol=1e-12, atol=1e-14)
            np.testing.assert_allclose(xm, x.mean(axis=0), rtol=1e-12, atol=1e-14)
            want = O.summary(g, x)
            np.testing.assert_allclose(np.round(gm, 3), want["estimate"], atol=1.001e-3)
            np.testing.assert_array_equal(np.round(gl, 3), want["lower_bound"])
            np.testing.assert_array_equal(np.round(gh, 3), want["upper_bound"])
        # extreme ranks = min / max
        gm, gl, gh, xm = eng.summary(0, nburn + 1, nsamp, 1, nsamp)
        g = eng.get_trace(0, "gamma", nburn + 1, nburn + nsamp + 1)[:, :, 0]
        np.testing.assert_array_equal(gl, g.min(axis=0))
        np.testing.assert_array_equal(gh, g.max(axis=0))
        with pytest.raises(bnr.BnrError):
            eng.summary(0, nburn + 1, nsamp, 0, nsamp)
        # ESS
        L = 63
        ex, eg = eng.ess(nburn + 1, nsamp, L)
        G = np.stack([eng.get_trace(c, "gamma", nburn + 1, nburn + nsamp + 1)[:, :, 0] for c in range(C)], axis=2)
        Xi = np.stack([eng.get_trace(c, "xi", nburn + 1, nburn + nsamp + 1)[:, :, 0] for c in range(C)], axis=2)
        for j in list(range(0, G.shape[1], 7)):
            np.testing.assert_allclose(eg[j], O.ess_geyer(G[:, j, :], L), rtol=1e-8, err_msg="gamma %d" % j)
        for k in range(Xi.shape[1]):
            want = O.ess_geyer(Xi[:, k, :], L)
            if math.isnan(want):
                assert math.isnan(ex[k])
            else:
                np.testing.assert_allclose(ex[k], want, rtol=1e-8, err_msg="xi %d" % k)
        # gathered form: two "ranks" holding the same statistics = one handle with every chain counted twice
        (pa, na), (pm, nm), lag = eng.ess_device()
        assert lag == L and na == (L + 1) * (eng.V + eng.q) and nm == C * (eng.V + eng.q)
        ex1, eg1 = eng.ess_from_stats(pa, 1, pm, C, nsamp, lag)
        np.testing.assert_array_equal(eg1, eg)


@pytest.mark.parametrize("nsamp,L,groups", [(333, 63, 1), (100, 255, 2), (37, 15, 3), (64, 63, 2)])
def test_streamed_ess_equals_trace_ess(bnr, golden, nsamp, L, groups):
    """bnr_ess_stream_*: lagged products accumulated while the chains run (no traces) give the same statistics, hence
    the same ESS, as the two-pass kernels over the recorded traces of the same draws -- for window lengths that are
    and are not multiples of the 8-draw accumulation block, lag budgets above and below the window, odd chain groups."""
    X, y = golden["test1.X"], golden["test1.y"]
    nburn, C = 41, 5
    with bnr.Engine(X, y, 5, num_chains=C, seed=11, trace_rows=nburn + nsamp + 1, trace_full_chains=0,
                    chain_groups=groups) as eng:
        eng.init_state()
        eng.run(nburn)
        eng.ess_stream_begin(L, nsamp)
        eng.run(nsamp - 5)
        eng.run(5)                                   # a window may span several bnr_run calls (odd counts run eagerly)
        eng.ess_stream_finish()
        (pa, na), (pm, nm), lag = eng.ess_device()
        P = eng.V + eng.q
        want_lag = min(L, nsamp - 1)
        assert lag == (want_lag if want_lag % 2 else want_lag - 1)
        import torch
        acov_s = torch.empty(na, dtype=torch.float64, device="cuda")
        mean_s = torch.empty(nm, dtype=torch.float64, device="cuda")
        eng.export_ess(acov_s.data_ptr(), mean_s.data_ptr())
        exs, egs = eng.ess_from_stats(pa, 1, pm, C, nsamp, lag)
        # the same draws through the trace kernels
        ext, egt = eng.ess(nburn + 1, nsamp, L)
        acov_t = torch.empty(na, dtype=torch.float64, device="cuda")
        mean_t = torch.empty(nm, dtype=torch.float64, device="cuda")
        eng.export_ess(acov_t.data_ptr(), mean_t.data_ptr())
        a_s, a_t = acov_s.cpu().numpy().reshape(lag + 1, P), acov_t.cpu().numpy().reshape(lag + 1, P)
        scale = np.abs(a_t[0])[None, :] + 1e-300
        assert np.max(np.abs(a_s - a_t) / scale) < 1e-11
        np.testing.assert_allclose(mean_s.cpu().numpy(), mean_t.cpu().numpy(), rtol=1e-13, atol=1e-13)
        ok = np.isfinite(egt)
        np.testing.assert_allclose(egs[ok], egt[ok], rtol=1e-7)
        assert (np.isnan(exs) == np.isnan(ext)).all()
        okx = np.isfinite(ext)
        np.testing.assert_allclose(exs[okx], ext[okx], rtol=1e-7)
        # a second window on the same handle reuses the buffers
        eng.ess_stream_begin(L, 16)
        eng.run(16)
        eng.ess_stream_finish()
        assert np.isfinite(eng.ess_streamed()[1]).any()
        with pytest.raises(bnr.BnrError):
            eng.ess_stream_finish()


@pytest.mark.parametrize("shape", [(100, 7, 1000, 6, "nform"), (30, 7, 500, 6, "qform"), (40, 5, 384, 5, "nform")])
def test_full_size_runs_are_bitwise_reproducible_across_chain_groups(bnr, shape):
    """Full-size sweeps (TMA rings, mbarrier hand-shakes, bordered Cholesky, streamed solves) are deterministic:
    the same seed gives bit-identical states for 1, 2 and 3 chain groups and on a repeated run -- a race in any
    of the producer/consumer pipelines would show up here.  n = 384 exercises the extra padding block that carries
    the bordering row when n is a multiple of 128."""
    V, R, n, C, mode = shape
    rng = np.random.default_rng(V)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.6)
    y = 10 + X[:, :15].sum(axis=1) + rng.normal(0, 3, size=n)
    ref = None
    for groups in (1, 2, 3, 2):
        with bnr.Engine(X, y, R, num_chains=C, seed=99, gamma_mode=mode, chain_groups=groups) as eng:
            eng.init_state()
            eng.run(5)                      # two graph replays + one eager sweep
            st = [eng.get_state_dict(c) for c in range(C)]
            assert not (eng.status() & ~1).any()
        if ref is None:
            ref = st
            assert all(np.isfinite(s["gamma"]).all() for s in st)
        else:
            for c in range(C):
                for k in ref[c]:
                    np.testing.assert_array_equal(np.asarray(st[c][k]), np.asarray(ref[c][k]), err_msg="%s chain %d groups %d" % (k, c, groups))


def test_chains_are_reproducible_under_load(bnr):
    """Three chain groups of config-3-sized problems keep every SM busy, so the producer/consumer rings run under memory
    pressure: 24 chains x 40 sweeps, twice with the default grouping and once as a single group, must agree bit for bit.
    (This is the check that caught a ring stage released before its shared-memory loads had been consumed: 1 in ~400
    chain-sweeps was perturbed, invisible to the 5-sweep test above.)"""
    V, R, n, C, K = 100, 7, 1000, 24, 40
    rng = np.random.default_rng(31)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.6)
    y = 10 + X[:, :15].sum(axis=1) + rng.normal(0, 3, size=n)
    ref = None
    for groups in (0, 0, 1):
        with bnr.Engine(X, y, R, num_chains=C, seed=7, chain_groups=groups) as eng:
            eng.init_state()
            eng.run(K)
            st = np.stack([np.concatenate([np.ravel(eng.get_state(c, k)) for k in ("gamma", "S", "u", "tau2", "M", "lam")])
                           for c in range(C)])
            assert not (eng.status() & ~1).any()
        if ref is None:
            ref = st
        else:
            differ = [c for c in range(C) if not np.array_equal(ref[c], st[c])]
            assert not differ, "chains %s differ from the first run (chain_groups=%d)" % (differ, groups)


def test_config1_shipped_example(bnr, golden):
    """BASELINE config 1: Fit! on the shipped example (examples/matrix_networks.csv: n=100, V=30, q=465), R=5.
    The reference's own stored 50 000-iteration fit of this data (older diagonal-free model, R=7;
    test/data/R=7_mu=1.6_n_microbes=22_*.csv) and the simulation truth (examples/true_xi.csv, true_b.csv) are
    soft level-2 references: the influential-node calls must match, posterior edge means must track the stored
    ones, and the stored 95% intervals must cover our posterior means for nearly all edges."""
    X, y = golden["example.X"], golden["example.y"]
    res = bnr.Fit(X, y, 5, nburn=12000, nsamples=8000, num_chains=8, seed=2358, x_transform=False, filename=None,
                  psrf_cutoff=1e9, return_state="none")
    assert res.extra["gamma_mode"] == "nform" and not (res.extra["status"] & ~1).any()
    out = bnr.Summary(res)
    prob = out.prob_nodes["probability"]
    true_xi = golden["example.true_xi"]
    ref_prob = golden["example.ref_xi_posterior"]
    assert ((prob > 0.5) == (true_xi > 0.5)).mean() >= 0.9, prob
    assert ((prob > 0.5) == (ref_prob > 0.5)).mean() >= 0.9, prob
    # edges: our table has the diagonal (465 rows), the stored one does not (435 rows, same column-major order)
    offdiag = out.edge_coef["node1"] != out.edge_coef["node2"]
    est = out.edge_coef["estimate"][offdiag]
    ref_mean, lo, hi = golden["example.ref_edge_mean"], golden["example.ref_edge_lo"], golden["example.ref_edge_hi"]
    assert np.corrcoef(est, ref_mean)[0, 1] > 0.9
    assert np.corrcoef(est, golden["example.true_b"])[0, 1] > 0.6
    assert np.mean((est >= lo - 0.25) & (est <= hi + 0.25)) > 0.95
    # (the diagonal columns of X are all zero: those coefficients are draws from N(W_kk, tau2 S), W_kk = u_k' Lambda u_k,
    #  so they carry no data information and are left out of the comparison)
    sig = (out.edge_coef["lower_bound"] > 0) | (out.edge_coef["upper_bound"] < 0)
    # significant-edge calls: edges between truly influential nodes dominate the calls
    tb = golden["example.true_b"] != 0
    called = sig[offdiag]
    assert called.sum() > 20 and (called & tb).sum() / max(called.sum(), 1) > 0.8


def test_syrk_split_k_path(bnr):
    """Few chains x large q (BASELINE config 4's regime): the Gram SYRK splits its contraction over gridDim.z and adds
    the partial matrices in a fixed order.  G must still equal X D X' + I to rounding and the run stay reproducible."""
    V, R, n, C = 64, 3, 200, 2          # q = 2080 -> 130 k-steps -> 4 splits for 2 x 3 tiles
    rng = np.random.default_rng(3)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q))
    y = X[:, :10].sum(axis=1) + rng.normal(size=n)
    outs = []
    for rep in range(2):
        with bnr.Engine(X, y, R, num_chains=C, seed=5, chain_groups=1) as eng:
            assert eng.gamma_mode == "nform"
            eng.init_state()
            eng.run(2)
            eng.enable_aux(True)
            S_old = eng.get_state(1, "S")[:, 0].copy()
            eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
            G = eng.get_aux(1, "G").reshape(n, n).T
            want = (X * S_old[None, :]) @ X.T + np.eye(n)
            assert np.abs(G - want).max() <= 1e-12 * np.abs(want).max()
            L = eng.get_aux(1, "G_chol").reshape(n, n).T
            assert np.abs(L @ L.T - want).max() <= 1e-11 * np.abs(want).max()
            outs.append(eng.get_state(1, "gamma").copy())
            assert not (eng.status() & ~1).any()
    np.testing.assert_array_equal(outs[0], outs[1])


def test_config2_qform_matches_nform_and_oracle_chain():
    """BASELINE config 2 (V=30, n=500, R=7, 16 chains; the cost model runs the q x q form): node-inclusion
    probabilities of the GPU sampler in both gamma formulations and of the CPU oracle chain agree within Monte-Carlo
    error on the benchmark's own synthetic data."""
    import bench
    from __graft_entry__ import load_package
    bnr = load_package()
    X, y, dims = bench.synth("c2")
    X = np.ascontiguousarray(X)
    V, R = dims["V"], dims["R"]
    prob = {}
    for mode in ("auto", "nform"):
        with bnr.Engine(X, y, R, num_chains=16, seed=5, trace_rows=6001, trace_full_chains=0, gamma_mode=mode) as eng:
            assert eng.gamma_mode == ("qform" if mode == "auto" else "nform")
            eng.init_state()
            eng.run(6000)
            prob[mode] = np.mean([eng.get_trace(c, "xi", 3001, 6001)[:, :, 0].mean(axis=0) for c in range(16)], axis=0)
            assert not (eng.status() & ~1).any()
    ora = np.mean([OC.run_chain(X, y, R, 1600, seed=s_, record=("xi",))[0]["xi"][601:].reshape(-1, V).mean(axis=0)
                   for s_ in (1, 2)], axis=0)
    assert np.abs(prob["auto"] - prob["nform"]).max() < 0.03
    assert np.abs(prob["auto"] - ora).max() < 0.07


def test_device_memory_cache_is_transparent(bnr):
    """Handles created from recycled device buffers (the process-wide cache behind bnr_destroy) behave exactly like
    fresh ones; the cache can be switched off and trimmed."""
    X, y = _toy(5, V=8, R=3, n=40)
    L = bnr.lib()

    def run():
        with bnr.Engine(X, y, 3, num_chains=3, seed=21, trace_rows=8) as eng:
            eng.init_state()
            eng.run(7)
            return eng.get_state_dict(2), eng.get_trace(0, "gamma", 0, 8).copy()

    try:
        assert L.bnr_set_cache_limit(0) == 0            # no caching: every buffer is cudaMalloc'ed / cudaFree'd
        a = run()
        assert L.bnr_set_cache_limit(4 << 30) == 0
        b = run()                                      # fills the cache on destroy
        c = run()                                      # served from the cache (stale contents in non-zeroed buffers)
        assert L.bnr_trim_cache() == 0
        d = run()
    finally:
        L.bnr_set_cache_limit(4 << 30)
    for other in (b, c, d):
        for k in a[0]:
            np.testing.assert_array_equal(np.asarray(a[0][k]), np.asarray(other[0][k]), err_msg=k)
        np.testing.assert_array_equal(a[1], other[1])


def test_plain_c_client_runs_a_fit(bnr, tmp_path):
    """The plain-C client of include/bnr.h (tests/c/abi_smoke.c) creates a handle, runs sweeps, reads R-hat and a trace."""
    import subprocess
    from test_abi_and_host import _build_c_client
    exe = _build_c_client(tmp_path)
    r = subprocess.run([exe, "60", "10", "3", "6", "80"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "sweeps 80" in r.stdout


def test_plain_c_client_runs_bnr_fit(bnr, tmp_path):
    """tests/c/fit_client.c: a whole doubling-scheme Fit through bnr_fit from plain C; with two GPUs also the chains
    sharded over both inside the library (moments all-gathered with NCCL) against one GPU holding all chains."""
    import subprocess
    import torch
    from test_abi_and_host import _build_c_client
    exe = _build_c_client(tmp_path, "fit_client")
    ndev = 2 if torch.cuda.device_count() >= 2 else 1
    r = subprocess.run([exe, str(ndev)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "tot_generated 120 burn_in 20 sampled 60 rows 80" in r.stdout
    if ndev == 2:
        assert "two devices: 4 chains" in r.stdout


def test_block_moments_equal_trace_moments(bnr):
    """Per-block streaming moments merged over a window (what the doubling scheme uses instead of all-chain traces)
    give the same split R-hat as the two-pass reduction of the recorded rows, for every window made of whole blocks."""
    X, y = _toy(7, V=6, R=3, n=30)
    blk, nblocks = 10, 12
    with bnr.Engine(X, y, 3, num_chains=5, seed=8, trace_rows=blk * nblocks + 1) as eng:
        eng.set_moment_blocks(0, blk, nblocks)
        eng.init_state()
        eng.run(37)                       # windows keep working across several bnr_run calls (graph + eager sweeps)
        eng.run(blk * nblocks - 1 - 37)
        for first_block, nb in ((2, 2), (4, 4), (6, 6), (0, 12)):
            eng.moments_from_blocks(first_block, nb)
            assert eng.moment_half_len() == nb // 2 * blk
            rx_b, rg_b = eng.rhat()
            eng.moments_from_trace(first_block * blk, nb * blk)        # row r holds sweep r
            rx_t, rg_t = eng.rhat()
            np.testing.assert_allclose(rg_b, rg_t, rtol=1e-10)
            fin = np.isfinite(rx_t)
            np.testing.assert_array_equal(np.isfinite(rx_b), fin)
            np.testing.assert_allclose(rx_b[fin], rx_t[fin], rtol=1e-10)
        with pytest.raises(bnr.BnrError):
            eng.moments_from_blocks(0, 3)
    # the doubling scheme on top of it: blocked (mingen % 4 == 0) and trace-based runs see the same chains
    a = bnr.Fit(X, y, 3, mingen=40, maxgen=120, psrf_cutoff=0.0, num_chains=3, seed=3, x_transform=False, filename=None)
    assert a.extra["rhat_streamed"] and a.extra["tot_generated"] == 120 and a.sampled == 60
    with bnr.Engine(X, y, 3, num_chains=3, seed=3, trace_rows=120) as eng:
        eng.init_state()
        eng.run(119)
        eng.moments_from_trace(60, 60)   # the last 60 of the 120 generated rows
        _, rg = eng.rhat()
        last = eng.get_trace(0, "gamma", 119, 120)[0, :, 0]
    np.testing.assert_allclose(a.rhatγ.γ, rg, rtol=1e-9)
    np.testing.assert_array_equal(a.state["γ"][-1, :, 0], last)


@pytest.mark.parametrize("V,n,R,mode", [(40, 3000, 4, "nform"), (60, 2000, 5, "qform"), (300, 300, 9, "nform"),
                                        # beyond the 4096 limit of round 1: 34 panels (n-form), 40 panels (q-form)
                                        (12, 4250, 3, "nform"), (100, 150, 3, "qform")])
def test_unusual_shapes_factorisation_properties(bnr, V, n, R, mode):
    """Tall n-form (24 and 34 panels of 128), long q-form (15 and 40 panels) and a large network (q = 45150): the
    factored matrix satisfies L L' = G (resp. P) and G a4 = rhs-type residuals stay at rounding level; chains stay healthy."""
    rng = np.random.default_rng(V + n)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q)) * (rng.random((n, q)) < 0.4)
    y = 3 + X[:, :12].sum(axis=1) + rng.normal(size=n)
    with bnr.Engine(X, y, R, num_chains=2, seed=1, gamma_mode=mode) as eng:
        assert eng.gamma_mode == mode
        eng.init_state()
        eng.run(3)
        eng.enable_aux(True)
        S_old = eng.get_state(1, "S")[:, 0].copy()
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        tau2 = float(eng.get_state(1, "tau2")[0, 0])
        m = q if mode == "qform" else n
        G = eng.get_aux(1, "G").reshape(m, m).T
        L = eng.get_aux(1, "G_chol").reshape(m, m).T
        want = (X.T @ X + np.diag(1.0 / S_old)) / tau2 if mode == "qform" else (X * S_old[None, :]) @ X.T + np.eye(n)
        scale = np.abs(want).max()
        assert np.abs(G - want).max() <= 1e-12 * scale
        assert np.abs(L @ L.T - want).max() <= 1e-11 * scale
        for cond in ("D", "theta", "Delta", "M", "mu", "lam", "pi"):
            eng.step(cond)
        eng.finish_sweep()
        eng.enable_aux(False)
        eng.run(4)
        st = eng.get_state_dict(0)
        assert not (eng.status() & ~1).any()
        assert np.isfinite(st["gamma"]).all() and (st["S"] > 0).all() and st["tau2"] > 0
