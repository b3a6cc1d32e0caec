"""The INT8 Gram path (k_gram_slice + k_gram_i8) at its arithmetic limits, held to the NumPy restatement bit for bit.

Its correctness rests on three claims: the int32 digit sums are exact while 7 qp 2^14 < 2^31, each entry of
A = X diag(sqrt(S)) is rounded once, and the error stays within _bound.  Random non-negative data never come near the
limits, so each construction here is built to reach one, and a CPU test checks that it does:
  * signed X, with rows whose largest entry is negative;
  * the digits that fill the int32 sums (|C_6| ~ 0.98 2^31 at qp = 18528, the largest qp on the path), both signs;
  * row scales 2^-p with p > 1000 (the split scale), p > 1074 (a subnormal row maximum) and p < 0;
  * rounding errors of one sign, and dropped digit products of one sign, against _bound;
  * the row-block edges of k_gram_i8 (a T = 1 matrix, a last block of padding only, 1 and 7 valid rows in it) and the
    lower end of the INT8 rule (V = 44 -> qp 992 on the FP64 SYRK, V = 45 -> qp 1040 on INT8);
  * NaN, infinite and negative S: both Gram paths must flag the chain (BNR_ST_G_NOTPD), as the reference throws.
Every expected value comes from the restatement (slice_rows, gram_from_planes) or a long-double product."""
import numpy as np
import pytest

from parity_util import assert_close_normwise, note, solve_tol
from test_gpu_gram_i8 import _bound, _delta, _design, _device_G, gram_from_planes, gram_i8, slice_rows
from test_gpu_gram_i8_exact import gram_from_planes_blas
from test_gpu_launch_lattice import _cond_bound, _gamma_reference, padded, selection
from test_gpu_parity import make_problem, random_state, sweep_injection

LOW = sum(2 ** (8 * s) for s in range(6))       # digits 1..6 all equal to 1


# ------------------------------------------------------------------------------------------------------------------
# the constructions (A = X diag(sqrt(S)); S = 1 keeps sqrt(S) exact, so X is A)
# ------------------------------------------------------------------------------------------------------------------
def worst_digits(n, q):
    """Rows of alternating sign whose digits fill the int32 sums: a row maximum of -126 2^48 (+126 2^48) integer units
    in column 0 and every other entry with the digits (-125, -128, ..., -128) ((125, 127, ..., 127, 124): a value in
    [2^54, 2^55) is a multiple of 4 in float64).  C_6 per k is 2 (-125)(-128) + 5 128^2 between two rows of the first
    kind and -125 124 - 5 128 127 - 128 125 between rows of both."""
    neg = np.full(q, -125 * 2 ** 48 - 128 * LOW, dtype=np.float64)
    pos = np.full(q, 125 * 2 ** 48 + 127 * (LOW - 1) + 124, dtype=np.float64)
    neg[0], pos[0] = -126 * 2.0 ** 48, 126 * 2.0 ** 48
    return np.ldexp(np.stack([neg if i % 2 == 0 else pos for i in range(n)]), -48)


def extreme_scales(rng, n, q):
    """Signed normal rows scaled by 2^-1010 (row 0: scale exponent 1000 < p <= 1074), 2^-1070 (row 1: a subnormal row
    maximum, p > 1074, so the row scale itself underflows to 0) and 2^400 (rows 2, 3: p < 0); the others O(1)."""
    X = rng.normal(size=(n, q))
    X[0] *= 2.0 ** -1010
    X[1] *= 2.0 ** -1070
    X[2:4] *= 2.0 ** 400
    return X


def scale_exponents(A):
    """p of every row as k_gram_slice picks it (slice_rows returns 2^-p, which is 0 for p > 1074)."""
    m = np.abs(A).max(axis=1)
    p = 54 - (np.frexp(m)[1] - 1)
    return p - (np.ldexp(m, p) > 126.0 * 2.0 ** 48)


def aligned_rounding(q):
    """Row 0: its maximum 63.02 2^48 integer units (the low end of the scale range) and every other entry just under a
    half unit, so that every rounding error has the same sign; row 1: ones.  Rows 2, 3: a maximum of 63.02 2^48 units
    and every other entry with the digits (0, -128, ..., -128), so that every dropped digit product (s + t > 6) of the
    two rows has the same sign."""
    A = np.zeros((4, q))
    A[0, 0] = 63.02 * 2.0 ** 48
    A[0, 1:] = 0.49999
    A[2:, 0] = 63.02 * 2.0 ** 48
    A[2:, 1:] = -128.0 * LOW
    A = np.ldexp(A, -40)
    A[1] = 1.0
    return A


# ------------------------------------------------------------------------------------------------------------------
# each construction reaches its limit (CPU)
# ------------------------------------------------------------------------------------------------------------------
def test_worst_case_digits_fill_the_int32_sums():
    q = 192 * 193 // 2                                  # qp = q: the largest qp on the INT8 path
    assert padded(192, 200, "nform")[2] == q and gram_i8(192, 200, "nform") and not gram_i8(193, 200, "nform")
    P, rs = slice_rows(worst_digits(4, q))
    assert list(P[:, 0, 1]) == [-125] + [-128] * 6 and list(P[:, 1, 1]) == [125] + [127] * 5 + [124]
    C, _ = gram_from_planes(P, rs)
    top = max(np.abs(c).max() for c in C)
    assert 0.95 * 2 ** 31 <= top < 2 ** 31, top / 2 ** 31
    assert C[6].max() >= 0.95 * 2 ** 31 and C[6].min() <= -0.95 * 2 ** 31, (C[6].max() / 2 ** 31, C[6].min() / 2 ** 31)


def test_extreme_row_scales_reach_every_exponent_range():
    X = extreme_scales(np.random.default_rng(3), 8, 1035)
    p = scale_exponents(X)
    assert 1000 < p[0] <= 1074 and p[1] > 1074 and (p[2:4] < 0).all(), p[:4]
    assert np.abs(X[1]).max() < np.finfo(np.float64).tiny
    _, rs = slice_rows(X)
    assert rs[1] == 0.0 and 0.0 < rs[0] < np.finfo(np.float64).tiny and (rs[2:4] > 1.0).all()


def test_aligned_errors_exceed_the_random_sign_estimate():
    """The rounding errors of one sign exceed sqrt(q) 2^-56 (sqrt(q) / 8 eps), the estimate for random signs; the dropped
    products of one sign exceed it ~700-fold and reach over half of _bound, whose q term is therefore needed."""
    q = 5050
    A = aligned_rounding(q)
    _, G = gram_from_planes(*slice_rows(A))
    G += np.eye(4)
    d_round = _delta(G, A, np.ones(q), np.array([0, 1]))
    d_drop = _delta(G, A, np.ones(q), np.array([2, 3]))
    assert np.sqrt(q) / 8 < d_round <= _bound(q, True), d_round
    assert 0.5 * _bound(q, True) < d_drop <= _bound(q, True), (d_drop, _bound(q, True))


# ------------------------------------------------------------------------------------------------------------------
# on the device: G bit for bit
# ------------------------------------------------------------------------------------------------------------------
def _device_grams(bnr, X, S_chains, clean=True):
    """G of every chain (the lower triangle of the n x n block is what k_gram_i8 stores) after tau2, u_xi, gamma."""
    n = X.shape[0]
    y = np.linspace(-1.0, 1.0, n)
    with bnr.Engine(X, y, 4, num_chains=len(S_chains), seed=3) as eng:
        assert eng.gamma_mode == "nform"
        eng.init_state()
        for c, S in enumerate(S_chains):
            eng.set_state(c, "S", S[:, None])
        eng.enable_aux(True)
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        if clean:
            assert not (eng.status() & ~1).any(), eng.status()
        return [eng.get_aux(c, "G").reshape(n, n).T for c in range(len(S_chains))]


def _assert_bits(G, X, S, msg):
    n = X.shape[0]
    want = gram_from_planes_blas(*slice_rows(X * np.sqrt(S)[None, :])) + np.eye(n)
    bad = np.argwhere((G != want) & np.tril(np.ones((n, n), dtype=bool)))
    assert len(bad) == 0, "%s: %d of %d entries differ, first (i, j) = %s" % (msg, len(bad), n * (n + 1) // 2,
                                                                           tuple(bad[0]))


@pytest.mark.gpu
def test_signed_x_bit_exact(bnr):
    """BASELINE config 5 shape, normal entries, 3 chains with their own S over 1e-12 .. 1e6."""
    V, n = 50, 500
    assert gram_i8(V, n, "nform")
    rng = np.random.default_rng(55)
    q = V * (V + 1) // 2
    X = rng.normal(size=(n, q))
    _, S = _design(rng, 1, q)
    S_chains = [S, 1e3 * rng.permutation(S), 1e-3 * S]
    for S in S_chains:
        A = X * np.sqrt(S)[None, :]
        assert (A[np.arange(n), np.abs(A).argmax(axis=1)] < 0).sum() > n // 4       # rows with a negative maximum
    G = _device_grams(bnr, X, S_chains)
    for c, S in enumerate(S_chains):
        _assert_bits(G[c], X, S, "chain %d" % c)


@pytest.mark.gpu
def test_worst_case_digits_bit_exact(bnr):
    """V = 192 (qp = 18528, the int32 limit), every entry with the digits that fill C_6, rows of both signs."""
    V, n = 192, 200
    q = V * (V + 1) // 2
    X = worst_digits(n, q)
    C, _ = gram_from_planes(*slice_rows(X[:2]))
    note(test="gram_i8_limits", case="worst_digits", c6_max=float(C[6].max() / 2 ** 31), c6_min=float(C[6].min() / 2 ** 31))
    S = np.ones(q)
    (G,) = _device_grams(bnr, X, [S], clean=False)
    _assert_bits(G, X, S, "worst-case digits")


@pytest.mark.gpu
def test_extreme_row_scales_bit_exact(bnr):
    """Row maxima near 2^-1000, a subnormal one and near 2^400 in one matrix: G bit for bit, and normwise within _bound
    of the long-double product (every entry is finite).  The factorisation of so ill-scaled a G may flag the chain;
    G is copied before it."""
    V, n = 45, 200
    q = V * (V + 1) // 2
    X = extreme_scales(np.random.default_rng(7), n, q)
    S = np.ones(q)
    (G,) = _device_grams(bnr, X, [S], clean=False)
    _assert_bits(G, X, S, "extreme row scales")
    assert np.isfinite(G[np.tril_indices(n)]).all()
    low = np.tril(G) + np.tril(G, -1).T
    d = _delta(low, X, S, np.arange(n))
    note(test="gram_i8_limits", case="extreme_scales", delta_eps=d)
    assert d <= _bound(q, True), d


@pytest.mark.gpu
def test_aligned_errors_within_the_worst_case_bound(bnr):
    """Rounding errors of one sign (rows 0, 1) and dropped digit products of one sign (rows 2, 3) at q = 5050: G bit
    for bit, and delta within _bound."""
    V, n = 100, 200
    q = V * (V + 1) // 2
    assert gram_i8(V, n, "nform")
    A = aligned_rounding(q)
    X = np.concatenate([A, np.tile(A[1], (n - 4, 1))])
    S = np.ones(q)
    (G,) = _device_grams(bnr, X, [S], clean=False)
    _assert_bits(G, X, S, "aligned errors")
    low = np.tril(G) + np.tril(G, -1).T
    for rows, case in (([0, 1], "aligned_rounding"), ([2, 3], "dropped_products")):
        d = _delta(low, X, S, np.array(rows))
        note(test="gram_i8_limits", case=case, q=q, delta_eps=d, bound=_bound(q, True))
        assert d <= _bound(q, True), (case, d)


# ------------------------------------------------------------------------------------------------------------------
# on the device: the shape edges, with the gamma step that reads the bordering row
# ------------------------------------------------------------------------------------------------------------------
EDGES = [(45, 127), (45, 384), (45, 385), (45, 391), (192, 384)]   # T = 1; last block padding only; 1, 7 valid rows


@pytest.mark.gpu
@pytest.mark.parametrize("V,n", EDGES, ids=["V%d-n%d" % e for e in EDGES])
def test_shape_edges_bit_exact_and_gamma(bnr, V, n):
    """G bit for bit, and one injected gamma step against the float64 reference: a store into row n, the bordering row
    that carries the forward solve, would not show in G's n x n block."""
    assert gram_i8(V, n, "nform")
    R, K = 3, 8
    X, y = make_problem(V + n, V, R, n)
    rng = np.random.default_rng(n + V)
    st = random_state(rng, V, R)
    inj, lay = sweep_injection(rng, n, V, R, K)
    (o1, s1), (o2, s2) = lay["gamma_z1"], lay["gamma_z2"]
    z1, z2 = inj[o1:o1 + s1].copy(), inj[o2:o2 + s2].copy()
    with bnr.Engine(X, y, R, num_chains=1, seed=3, gig_inject_len=K, gamma_mode="nform") as eng:
        eng.enable_aux(True)
        eng.set_state_dict(0, st)
        eng.set_injection(inj[None, :])
        eng.step("gamma")
        assert not (eng.status() & ~1).any(), eng.status()
        G = eng.get_aux(0, "G").reshape(n, n).T
        a4 = eng.get_aux(0, "a4")
        gamma = eng.get_state(0, "gamma")[:, 0]
    _assert_bits(G, X, st["S"], "V %d n %d" % (V, n))
    ref = _gamma_reference(X, y, st, z1, z2, "nform")
    tol = solve_tol(_cond_bound(X, st["S"], st["tau2"], "nform"))
    assert_close_normwise(a4, ref["a4"], tol, "a4")
    assert_close_normwise(gamma, ref["gamma"], tol, "gamma")


@pytest.mark.gpu
def test_lower_switch(bnr):
    """qp = 992 (V = 44) runs the FP64 SYRK, qp = 1040 (V = 45) the INT8 path.  With 449 chains the SYRK is not split
    and the X products split alike for both shapes, so the INT8 path shows as exactly one more launch per eager sweep
    (k_gram_slice); both hold G to long double."""
    n, C = 300, 449
    a, b = selection(44, n, "nform", C), selection(45, n, "nform", C)
    assert not a["syrk_split"] and not b["syrk_split"] and a["x_splits"] == b["x_splits"]
    assert not gram_i8(44, n, "nform") and gram_i8(45, n, "nform")
    launches = {}
    for V in (44, 45):
        rng = np.random.default_rng(V)
        q = V * (V + 1) // 2
        X, S = _design(rng, n, q, dominant_rows=(1,))
        y = rng.normal(size=n)
        G, launches[V] = _device_G(bnr, X, y, [S] * C)
        d = _delta(G[0], X, S, np.arange(0, n, 7))
        assert d <= _bound(q, gram_i8(V, n, "nform")), (V, d)
    assert launches[45] == launches[44] + 1, launches


# ------------------------------------------------------------------------------------------------------------------
# on the device: NaN, infinite and negative S are flagged on both Gram paths
# ------------------------------------------------------------------------------------------------------------------
def _bad_scales(S, case):
    S = S.copy()
    if case == "nan":
        S[7] = np.nan
    elif case == "negative":
        S[:] = -100.0
    else:
        S[7] = np.inf
    return S


def _positive_definite(G):
    full = np.tril(G) + np.tril(G, -1).T
    if not np.isfinite(full).all():
        return False
    try:
        np.linalg.cholesky(full)
        return True
    except np.linalg.LinAlgError:
        return False


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["nan", "negative", "inf"])
@pytest.mark.parametrize("V", [50, 44], ids=["int8", "fp64"])
def test_non_finite_scales_flag_the_chain(bnr, V, case):
    """The reference's cholesky(X D X' + I) throws PosDefException for these S; the engine sets BNR_ST_G_NOTPD on
    chain 0 only, and chains 1-2 are bit for bit those of a handle whose chain 0 is clean.  The right-hand side in the
    bordering row is NaN for these S as well, so the flag alone would not show a G that is wrongly positive definite:
    G itself must hold a NaN or be indefinite, on either Gram path."""
    n, R, K, C = 500, 3, 8, 3
    assert gram_i8(V, n, "nform") == (V == 50)
    X, y = make_problem(V + 1, V, R, n)
    rng = np.random.default_rng(V)
    states = [random_state(rng, V, R) for _ in range(C)]
    inj = np.stack([sweep_injection(rng, n, V, R, K)[0] for _ in range(C)])
    out = {}
    for bad in (True, False):
        with bnr.Engine(X, y, R, num_chains=C, seed=5, gig_inject_len=K, gamma_mode="nform") as eng:
            for c, st in enumerate(states):
                if bad and c == 0:
                    st = dict(st, S=_bad_scales(st["S"], case))
                eng.set_state_dict(c, st)
            eng.set_injection(inj)
            eng.enable_aux(True)
            eng.step("gamma")
            G0 = eng.get_aux(0, "G").reshape(n, n).T
            out[bad] = eng.status(), G0, [eng.get_state_dict(c) for c in range(1, C)]
    status, G0 = out[True][0], out[True][1]
    assert status[0] & 4, status                            # BNR_ST_G_NOTPD
    assert not (status[1:] & ~1).any() and not (out[False][0] & ~1).any(), (status, out[False][0])
    assert not _positive_definite(G0), "chain 0: G is finite and positive definite"
    assert _positive_definite(out[False][1])
    for c, (got, want) in enumerate(zip(out[True][2], out[False][2]), start=1):
        for k in want:
            np.testing.assert_array_equal(np.asarray(got[k]), np.asarray(want[k]), err_msg="%s chain %d" % (k, c))
