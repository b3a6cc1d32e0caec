"""k_gram_slice takes GS_CB chains per CTA (bnr_linalg.cu), so a launch whose chain count is not a multiple of GS_CB
ends in a partial chain block.  Every chain must still get the digits and row scales of the NumPy restatement
(slice_rows), bit for bit in G, whichever block and position in the block it falls on; and the chain groups, each a
launch of its own chain count, must not change a bit of a sweep."""
import os
import re

import numpy as np
import pytest

from test_gpu_gram_i8 import _design, gram_i8, slice_rows
from test_gpu_gram_i8_exact import gram_from_planes_blas

HERE = os.path.dirname(os.path.abspath(__file__))


def _chains_per_cta():
    src = open(os.path.join(HERE, os.pardir, "bayesiannetworkregression.jl_b200", "csrc", "bnr_linalg.cu")).read()
    return int(re.search(r"\bGS_CB = (\d+)", src).group(1))


CB = _chains_per_cta()


def _checked(C):
    """first and last chain of every chain block, and the chain before the last"""
    return sorted({c for b in range(0, C, CB) for c in (b, min(b + CB, C) - 1)} | {max(C - 2, 0)})


CASES = [  # (V, n, chains)
    (50, 500, 1),             # BASELINE config 5 shape, one chain: a block of one
    (50, 500, CB + 1),        # one full block and a block of one
    (50, 500, 2 * CB + 1),
    (60, 500, CB + 1),        # qp = 1840: the last 32-k block of a row ends past qp
]


@pytest.mark.gpu
@pytest.mark.parametrize("V,n,C", CASES, ids=["c5_1", "c5_cb+1", "c5_2cb+1", "ktail_cb+1"])
def test_gram_slice_partial_chain_blocks_bit_exact(bnr, V, n, C):
    assert gram_i8(V, n, "nform")
    rng = np.random.default_rng(V * 11 + C)
    q = V * (V + 1) // 2
    X, S = _design(rng, n, q, dominant_rows=(1, 6, n - 2))
    X[[4, 17]] = 0.0                                  # rows that are all zero: no digits, scale 1
    y = rng.normal(size=n)
    S_chains = [S * 10.0 ** (c % 7 - 3) if c % 2 == 0 else rng.permutation(S) for c in range(C)]
    check = _checked(C)
    with bnr.Engine(X, y, 4, num_chains=C, seed=5, chain_groups=1) as eng:
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
        assert len(bad) == 0, "chain %d of %d: %d entries differ, first (i, j) = %s" % (c, C, len(bad), tuple(bad[0]))


GROUP_CHAINS = 19   # groups of 19; 10 + 9; 7 + 6 + 6 chains: none a multiple of GS_CB = 4


@pytest.mark.gpu
@pytest.mark.parametrize("groups", [1, 2, 3])
def test_graph_sweeps_equal_eager_sweeps_partial_blocks(bnr, groups):
    """BASELINE config 5 shape with 19 chains: graph sweeps in 1, 2 or 3 chain groups equal eager sweeps bit for bit."""
    from test_gpu_parity import make_problem
    V, R, n, C = 50, 5, 500, GROUP_CHAINS
    assert gram_i8(V, n, "nform")
    X, y = make_problem(V + n + groups, V, R, n, dense=False)
    kw = dict(num_chains=C, seed=31, trace_rows=6, trace_full_chains=C, chain_groups=groups)
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
