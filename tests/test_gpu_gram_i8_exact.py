"""The INT8 Gram path is exact up to its one rounding per entry of A = X diag(sqrt(S)): the device's G must equal the
NumPy restatement gram_from_planes(slice_rows(A)) + I bit for bit on every stored entry (the lower triangle of the
n x n block).  The int32 digit sums are exact and the FP64 recombination has a fixed order, so any re-tiling or
re-issuing of the integer products must leave every bit of G as it is; a wrong half of an operand, a missed k-block or
a mis-addressed accumulator shows here as entries that differ, where a tolerance test could let them through.

Shapes: BASELINE configs 3 and 5, n = 300 (the last 128-row block holds 44 rows), and qp = 1840, which is not a
multiple of the 64-byte k-block (the tail is read as zeros); 1, 3 and 64 chains, each with its own S."""
import numpy as np
import pytest

from test_gpu_gram_i8 import S_PLANES, _design, gram_from_planes, gram_i8, slice_rows


def gram_from_planes_blas(P, rs):
    """gram_from_planes with the digit products as float64 matrix products: every product and partial sum is an
    integer below 2^53 (|D| <= 128, k < 2^19), so the float64 sums are exact in any order and C_g is the same integer."""
    F = [p.astype(np.float64) for p in P]
    C = [sum(F[s] @ F[g - s].T for s in range(g + 1)) for g in range(S_PLANES)]
    v = C[-1]
    for g in range(S_PLANES - 2, -1, -1):
        v = C[g] + v * 2.0 ** -8
    return v * (rs[:, None] * 2.0 ** 96) * rs[None, :]


def test_blas_restatement_equals_integer_restatement():
    rng = np.random.default_rng(7)
    X, S = _design(rng, 40, 700, dominant_rows=(3, 17))
    P, rs = slice_rows(X * np.sqrt(S)[None, :])
    _, G = gram_from_planes(P, rs)
    np.testing.assert_array_equal(gram_from_planes_blas(P, rs), G)


CASES = [  # (V, n, chains, chains checked)
    (100, 1000, 64, (0, 37, 63)),      # BASELINE config 3
    (50, 500, 3, (0, 1, 2)),           # BASELINE config 5
    (50, 300, 1, (0,)),                # a short last row block
    (60, 500, 3, (0, 1, 2)),           # qp = 1840: a k-tail inside the last 64-byte k-block
]


@pytest.mark.gpu
@pytest.mark.parametrize("V,n,C,check", CASES, ids=["c3_64", "c5_3", "n300_1", "ktail_3"])
def test_gram_i8_bit_exact(bnr, V, n, C, check):
    assert gram_i8(V, n, "nform")
    rng = np.random.default_rng(V * 7 + n + C)
    q = V * (V + 1) // 2
    X, S = _design(rng, n, q, dominant_rows=(0, 5, n - 1))
    y = rng.normal(size=n)
    S_chains = [S * 10.0 ** (c % 5 - 2) if c % 2 == 0 else rng.permutation(S) for c in range(C)]
    with bnr.Engine(X, y, 4, num_chains=C, seed=3) as eng:
        assert eng.gamma_mode == "nform"
        eng.init_state()
        for c, Sc in enumerate(S_chains):
            eng.set_state(c, "S", Sc[:, None])
        eng.enable_aux(True)
        eng.step("tau2"); eng.step("u_xi"); eng.step("gamma")
        assert not (eng.status() & ~1).any()
        G = {c: eng.get_aux(c, "G").reshape(n, n).T for c in check}
    low = np.tril(np.ones((n, n), dtype=bool))
    for c in check:
        want = gram_from_planes_blas(*slice_rows(X * np.sqrt(S_chains[c])[None, :])) + np.eye(n)
        bad = np.argwhere((G[c] != want) & low)
        assert len(bad) == 0, "chain %d: %d of %d entries differ, first (i, j) = %s" % (
            c, len(bad), n * (n + 1) // 2, tuple(bad[0]))
