"""The three streamed convergence statistics armed together on one handle -- the split-half R-hat window, the block
moments of the doubling scheme and an ESS window -- give bit-identical results for every chain grouping.  Each chain
group's sweep graph sees the statistics buffers through its own view, offset to the group's first chain, while the
eager sweep of an odd count sees the whole handle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

V, R, N, C = 7, 3, 60, 5
SWEEPS = 41                      # 20 two-sweep graph replays, then one eager sweep
BLK, NBLOCKS = 5, 8              # blocks cover sweeps 1 .. 40
L = 15


def _streams(bnr, groups):
    import torch
    rng = np.random.default_rng(21)
    q = V * (V + 1) // 2
    X = rng.normal(size=(N, q))
    y = 1.0 + X[:, :3].sum(axis=1) + rng.normal(size=N)
    with bnr.Engine(X, y, R, num_chains=C, seed=17, trace_full_chains=0, chain_groups=groups) as eng:
        assert eng.chain_groups == groups
        eng.init_state()
        eng.set_moment_window(1, SWEEPS)
        eng.set_moment_blocks(1, BLK, NBLOCKS)
        eng.ess_stream_begin(L, SWEEPS)
        eng.run(SWEEPS)
        P = eng.V + eng.q
        mom = torch.empty(C * 2 * P * 2, dtype=torch.float64, device="cuda")
        eng.export_moments(mom.data_ptr())
        window = mom.cpu().numpy()
        eng.moments_from_blocks(0, NBLOCKS)
        eng.export_moments(mom.data_ptr())
        merged = mom.cpu().numpy()
        eng.ess_stream_finish()
        (_, na), (_, nm), lag = eng.ess_device()
        assert lag == L
        acov = torch.empty(na, dtype=torch.float64, device="cuda")
        means = torch.empty(nm, dtype=torch.float64, device="cuda")
        eng.export_ess(acov.data_ptr(), means.data_ptr())
        return window, merged, acov.cpu().numpy(), means.cpu().numpy()


def test_stat_streams_are_identical_across_chain_groups(bnr):
    ref = _streams(bnr, 1)
    for a in ref:
        assert np.isfinite(a).all() and np.any(a != 0.0)
    names = ("split-half moments", "merged block moments", "ESS lagged sums", "ESS chain means")
    for groups in (2, 3):
        got = _streams(bnr, groups)
        for name, r, g in zip(names, ref, got):
            np.testing.assert_array_equal(g, r, err_msg="%s, %d chain groups" % (name, groups))
