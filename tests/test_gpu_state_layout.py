"""The per-chain layout of the state, the trace rows and the aux outputs, read back through every path that uses it.

For each chain grouping, the last trace row of every traced variable equals the state it was recorded from, bit for
bit, after graph replays and an eager sweep.  set_state / get_state round-trip every variable (pi included, whose
storage order differs from the reference's), and finish_sweep records exactly the state that was set.  Every aux
output has the size include/bnr.h documents.  The three shapes cover the arrays a handle may or may not have: the
q-form, the FP64 n-form with a split Gram SYRK (its partial-product workspace exists at 4 chains) and the INT8
n-form (digit planes and row scales)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CHAINS, R = 4, 3
SHAPES = {                        # name: V, n, gamma_mode
    "qform": (12, 150, "qform"),
    "nform_split_syrk": (40, 200, "nform"),   # qp = 832 < 1024: FP64 SYRK; 3 tiles x 4 chains -> 2 k-splits
    "nform_int8": (46, 200, "nform"),         # qp = 1088: INT8 Gram path
}
BNR_EINVAL = -1


def _doc_aux_sizes(V, q, n, qform):
    """The per-chain size of every aux output as include/bnr.h documents it."""
    m = q if qform else n
    return {"tau2_params": 2, "sigma_inv": V * R * R, "sigma_chol": V * R * R, "mu_t": V * R, "log_odds": V,
            "W": q, "G": m * m, "G_chol": m * m, "rhs": m, "a4": m, "chi": q, "theta_params": 2, "delta_params": 2,
            "m_params": 1 + 2 * R * R, "mu_params": 2, "lambda_logw": 3 * R, "lambda_weights": 3 * R,
            "pi_alpha": 3 * R, "gig_used": q}


@pytest.mark.parametrize("groups", [1, 2, 3])
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_state_trace_and_aux_layout(bnr, shape, groups):
    V, n, mode = SHAPES[shape]
    q = V * (V + 1) // 2
    rng = np.random.default_rng(V + n)
    X = rng.normal(size=(n, q))
    y = 2.0 + X[:, :3].sum(axis=1) + rng.normal(size=n)
    last = CHAINS - 1             # traced through the gamma/xi trace only
    with bnr.Engine(X, y, R, num_chains=CHAINS, seed=13, trace_rows=8, trace_full_chains=CHAINS - 1,
                    gamma_mode=mode, chain_groups=groups) as eng:
        assert eng.chain_groups == groups and eng.gamma_mode == mode

        def traced(c):
            return ("xi", "gamma") if c == last else tuple(bnr.VAR)

        # rows 0 (initial state) to 5: two two-sweep graph replays, then one eager sweep
        eng.init_state()
        eng.run(5)
        assert eng.iteration == 5 and eng.trace_row == 6
        for c in range(CHAINS):
            for v in traced(c):
                np.testing.assert_array_equal(eng.get_trace(c, v, 5, 6)[0], eng.get_state(c, v),
                                              err_msg="chain %d %s" % (c, v))
        with pytest.raises(bnr.BnrError):
            eng.get_trace(last, "u", 5, 6)

        # every aux output: the documented size fits, one element less is refused
        eng.enable_aux(True)
        for cond in bnr.COND:
            eng.step(cond)
        sizes = _doc_aux_sizes(V, q, n, mode == "qform")
        assert set(sizes) == set(bnr.AUX)
        lib = bnr.lib()
        for c in range(CHAINS):
            for name, size in sizes.items():
                assert eng.get_aux(c, name).shape == (size,)
                out = np.empty(size)
                rc = lib.bnr_get_aux(eng._h, c, bnr.AUX[name], out.ctypes.data_as(C.POINTER(C.c_double)), size - 1)
                assert rc == BNR_EINVAL, "chain %d %s" % (c, name)
        eng.enable_aux(False)

        # set_state / get_state round trip, then finish_sweep records exactly that state as row 6
        states = []
        for c in range(CHAINS):
            st = {v: rng.normal(size=eng.var_shape(v)) for v in bnr.VAR}
            st["pi"] = np.arange(3 * R, dtype=np.float64).reshape((R, 3), order="F") + 0.25 * c   # not symmetric
            for v, a in st.items():
                eng.set_state(c, v, a)
            states.append(st)
        for c in range(CHAINS):
            for v, a in states[c].items():
                np.testing.assert_array_equal(eng.get_state(c, v), a, err_msg="chain %d %s" % (c, v))
        eng.finish_sweep()
        assert eng.trace_row == 7
        for c in range(CHAINS):
            for v in traced(c):
                np.testing.assert_array_equal(eng.get_trace(c, v, 6, 7)[0], states[c][v],
                                              err_msg="recorded row, chain %d %s" % (c, v))
