"""The n-form Gram matrix G = X diag(S) X' + I on the INT8 tensor cores (bnr_linalg.cu: k_gram_slice, k_gram_i8).

Row i of A = X diag(sqrt(S)) is scaled by a power of two, rounded once to an integer below 2^55 and split into 7
balanced base-256 digits; G is recombined in FP64 from the int32 sums of the 28 digit products with digit sum <= 6.
The CPU tests restate that arithmetic in NumPy and check the selection rule and the int32 bound; the GPU tests hold
the device's G to a long-double X diag(S) X' + I, show the switch to the FP64 SYRK past the int32 limit, and require
graph sweeps to equal eager sweeps bit for bit on the new path."""
import os
import re

import numpy as np
import pytest

from parity_util import EPS, note
from test_gpu_launch_lattice import padded, selection

S_PLANES = 7
HERE = os.path.dirname(os.path.abspath(__file__))


def _kernel_constants():
    src = open(os.path.join(HERE, os.pardir, "bayesiannetworkregression.jl_b200", "csrc", "bnr_kernels.h")).read()
    return tuple(int(re.search(r"constexpr int %s = (\d+);" % k, src).group(1)) for k in ("GRAM_I8_QP_MIN", "GRAM_I8_QP_MAX"))


QP_MIN, QP_MAX = _kernel_constants()


def gram_i8(V, n, mode):
    """Does a handle of this shape compute G on the INT8 path?  (gram_i8_selected: the shape only, never the chains)"""
    q, np_, qp, N = padded(V, n, mode)
    return mode == "nform" and QP_MIN <= qp <= QP_MAX


# ------------------------------------------------------------------------------------------------------------------
# NumPy restatement of the two kernels
# ------------------------------------------------------------------------------------------------------------------
def slice_rows(A):
    """(digit planes [7][rows][k] int8, row scales 2^-p) as k_gram_slice computes them."""
    m = np.abs(A).max(axis=1)
    p = np.zeros(A.shape[0], dtype=np.int64)
    nz = m > 0
    p[nz] = 54 - (np.frexp(m[nz])[1] - 1)
    p[nz & (np.ldexp(m, p) > 126.0 * 2.0 ** 48)] -= 1
    N = np.rint(np.ldexp(A, p[:, None])).astype(np.int64)
    planes = np.zeros((S_PLANES,) + A.shape, dtype=np.int8)
    for s in range(S_PLANES - 1, 0, -1):
        dg = ((N + 128) & 255) - 128
        planes[s] = dg
        N = (N - dg) >> 8
    assert np.abs(N).max() <= 127
    planes[0] = N
    return planes, np.ldexp(1.0, -p)


def gram_from_planes(P, rs):
    """(C_g, G): C_g = sum_{s+t=g} D^(s) D^(t)' in exact integers, G = 2^96 rs_i rs_j sum_g 2^-8g C_g (Horner from g = 6)."""
    C = [sum(P[s].astype(np.int64) @ P[g - s].astype(np.int64).T for s in range(g + 1)) for g in range(S_PLANES)]
    v = C[-1].astype(np.float64)
    for g in range(S_PLANES - 2, -1, -1):
        v = C[g].astype(np.float64) + v * 2.0 ** -8
    return C, v * (rs[:, None] * 2.0 ** 96) * rs[None, :]


def _design(rng, n, q, dominant_rows=()):
    """X like bench.py's synthetic networks (48 % dense, X >= 0) with a few rows dominated by one entry, and S over
    1e-12 .. 1e6 inside one chain."""
    X = np.where(rng.random((n, q)) < 0.48, 0.13 + rng.gamma(1.2, 0.2, size=(n, q)), 0.0)
    for i in dominant_rows:
        X[i, rng.integers(q)] = 1e4
    S = np.exp(rng.uniform(np.log(1e-12), np.log(1e6), size=q))
    return X, S


def _delta(G, X, S, rows):
    """max over rows x all columns of |G_ij - G_exact,ij| / sqrt(G_ii G_jj), G_exact in long double, in units of eps."""
    Xl = X.astype(np.longdouble)
    want = (Xl[rows] * S.astype(np.longdouble)[None, :]) @ Xl.T
    diag = np.einsum("ij,ij->i", Xl * S.astype(np.longdouble)[None, :], Xl) + 1
    want[np.arange(len(rows)), rows] += 1
    d = np.sqrt(diag)
    return float((np.abs(G[rows].astype(np.longdouble) - want) / (d[rows][:, None] * d[None, :])).max() / EPS)


def _bound(q, int8):
    """delta bound in units of eps.  INT8 path: sqrt(q) 2^-56, the error of q terms each rounded to ~2^-56 of the row
    maxima with random signs (the first neglected digit).  FP64 SYRK (the shapes outside the INT8 rule, unchanged by it):
    the worst-case bound q u of a q-term FP64 dot product, u = 2^-53, with sum |x_ik S_k x_jk| <= sqrt(G_ii G_jj)."""
    return np.sqrt(q) / 8.0 if int8 else q / 2.0


def test_digits_spell_the_row_rounded_once():
    rng = np.random.default_rng(0)
    A = np.abs(rng.normal(size=(40, 300))) * np.exp(rng.uniform(-20, 20, size=(1, 300)))
    A[3, 7] = 1e9
    A[5] = 0.0                           # a padding row: no digits, any scale
    P, rs = slice_rows(A)
    assert P[0].min() >= -127 and P[0].max() <= 127
    N = sum(P[s].astype(np.int64) << (8 * (S_PLANES - 1 - s)) for s in range(S_PLANES))
    assert np.abs(N).max() < 2 ** 55
    err = np.abs(N.astype(np.float64) * rs[:, None] - A)
    assert (err <= 0.5 * rs[:, None]).all()                                  # one rounding to the nearest integer
    assert (err <= 2.0 ** -54 * np.abs(A).max(axis=1, keepdims=True)).all()
    assert (err[:, 7][A[:, 7] >= 2.0 ** -2 * np.abs(A).max(axis=1)] == 0).all()   # entries near the row max: exact


def test_gram_of_the_digits_against_long_double():
    rng = np.random.default_rng(1)
    X, S = _design(rng, 24, 600, dominant_rows=(2, 11))
    P, rs = slice_rows(X * np.sqrt(S)[None, :])
    C, G = gram_from_planes(P, rs)
    assert max(np.abs(c).max() for c in C) < 2 ** 31
    assert _delta(G + np.eye(24), X, S, np.arange(24)) <= 4.0


def test_selection_rule_and_int32_bound():
    # the largest digit-sum group adds 7 ordered products of at most 2^14 per k
    assert 7 * QP_MAX * 2 ** 14 < 2 ** 31 <= 7 * (QP_MAX + 1) * 2 ** 14
    assert gram_i8(100, 1000, "nform") and gram_i8(50, 500, "nform")         # BASELINE configs 3 and 5
    assert not gram_i8(200, 400, "nform")                                     # config 4: qp = 20112 > QP_MAX
    assert gram_i8(192, 200, "nform") and not gram_i8(193, 200, "nform")      # qp = 18528 and 18736
    # the launch-count lattice (q <= 820) stays on the FP64 SYRK
    for V in (10, 20, 40):
        assert not gram_i8(V, 1000, "nform")


# ------------------------------------------------------------------------------------------------------------------
# on the device
# ------------------------------------------------------------------------------------------------------------------
def _device_G(bnr, X, y, S_chains, **kw):
    n = X.shape[0]
    with bnr.Engine(X, y, 4, num_chains=len(S_chains), seed=3, **kw) as eng:
        assert eng.gamma_mode == "nform"
        eng.init_state()
        l0 = eng.launch_count()
        eng.run(1)                                   # one eager sweep: its launch count
        launches = eng.launch_count() - l0
        for c, S in enumerate(S_chains):
            eng.set_state(c, "S", S[:, None])
        eng.enable_aux(True)
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        G = [eng.get_aux(c, "G").reshape(n, n).T for c in range(min(2, len(S_chains)))]
        assert not (eng.status() & ~1).any()
    return G, launches


@pytest.mark.gpu
@pytest.mark.parametrize("V,n", [(100, 1000), (200, 400)], ids=["c3", "c4"])
def test_gram_against_long_double(bnr, V, n):
    """S over 1e-12 .. 1e6 inside a chain, the neighbouring chain's S 100x larger, rows dominated by one entry."""
    rng = np.random.default_rng(V)
    q = V * (V + 1) // 2
    X, S = _design(rng, n, q, dominant_rows=(0, 5, n - 1))
    y = rng.normal(size=n)
    G, _ = _device_G(bnr, X, y, [S, 100.0 * S])
    rows = np.concatenate([[0, 5, n - 1], rng.choice(n, 29, replace=False)])
    for c, Sc in enumerate((S, 100.0 * S)):
        d = _delta(G[c], X, Sc, rows)
        note(test="gram_i8", V=V, n=n, chain=c, path="int8" if gram_i8(V, n, "nform") else "fp64", delta_eps=d)
        assert d <= _bound(q, gram_i8(V, n, "nform")), (c, d)


@pytest.mark.gpu
def test_int32_limit(bnr):
    """qp = 18528 (V = 192, the last V below the int32 limit) runs the INT8 path, qp = 18736 (V = 193) the FP64 SYRK;
    both hold G to long double (_bound).  With 50 chains the FP64 SYRK is not split and every other launch rule picks the same
    for both shapes, so the INT8 path shows as exactly one more launch per eager sweep (k_gram_slice)."""
    n, C = 200, 50
    launches = {}
    for V in (192, 193):
        rng = np.random.default_rng(V)
        q = V * (V + 1) // 2
        X, S = _design(rng, n, q, dominant_rows=(1,))
        y = rng.normal(size=n)
        S_chains = [S * 10.0 ** (2 * (c % 4) - 2) for c in range(C)]
        G, launches[V] = _device_G(bnr, X, y, S_chains)
        rows = np.arange(0, n, 7)
        for c in range(2):
            d = _delta(G[c], X, S_chains[c], rows)
            note(test="gram_i8_limit", V=V, chain=c, path="int8" if gram_i8(V, n, "nform") else "fp64", delta_eps=d)
            assert d <= _bound(q, gram_i8(V, n, "nform")), (V, c, d)
    a, b = selection(192, n, "nform", C), selection(193, n, "nform", C)
    assert not a["syrk_split"] and not b["syrk_split"] and a["x_splits"] == b["x_splits"]
    assert gram_i8(192, n, "nform") and not gram_i8(193, n, "nform")
    assert launches[192] == launches[193] + 1, launches


@pytest.mark.gpu
@pytest.mark.parametrize("groups", [1, 2, 3])
def test_graph_sweeps_equal_eager_sweeps_int8(bnr, groups):
    """BASELINE config 3 shape with 12 chains: graph sweeps in 1, 2 or 3 chain groups equal eager sweeps bit for bit."""
    from test_gpu_parity import make_problem
    V, R, n, C = 100, 7, 1000, 12
    assert gram_i8(V, n, "nform")
    X, y = make_problem(V + n + groups, V, R, n, dense=False)
    kw = dict(num_chains=C, seed=29, trace_rows=6, trace_full_chains=C, chain_groups=groups)
    with bnr.Engine(X, y, R, **kw) as a, bnr.Engine(X, y, R, **kw) as b:
        a.init_state()
        b.init_state()
        for k in (2, 1, 3):
            a.run(k)
        for _ in range(6):
            b.run(1)
        assert a.iteration == b.iteration == 6 and a.chain_groups == groups
        assert not (a.status() & ~1).any() and not (b.status() & ~1).any()
        for c in range(C):
            sa, sb = a.get_state_dict(c), b.get_state_dict(c)
            for k in sa:
                np.testing.assert_array_equal(np.asarray(sa[k]), np.asarray(sb[k]), err_msg="%s chain %d" % (k, c))
