"""NumPy restatement of pooled PSIS-LOO and WAIC as the R package loo 2.x computes them (psis(), gpdfit(),
r_eff = 1), written from the algorithm's definition.  Test infrastructure only: libbnr's k_loo_pass / k_loo_tail
compute the same quantities on the device (bnr_loo_summary)."""
import numpy as np
from scipy.special import logsumexp


def loglik(y, mu, xg, tau2):
    """Pointwise log density log N(y_i | mu + (X gamma)_i, tau2) of one draw."""
    r = y - mu - xg
    return -0.5 * np.log(6.283185307179586 * tau2) - r * r / (2.0 * tau2)


def tail_len(S):
    """M = ceil(min(0.2 S, 3 sqrt(S))): the Pareto tail of S draws (r_eff = 1)."""
    return int(np.ceil(min(0.2 * S, 3.0 * np.sqrt(S))))


def gpdfit(x):
    """Zhang & Stephens fit of the generalised Pareto distribution to x (sorted ascending): (k, sigma), k with the
    weakly informative prior of loo (M k + 5) / (M + 10); NaN -> inf."""
    M = x.size
    G = 30 + int(np.floor(np.sqrt(M)))
    xs = x[int(np.floor(M / 4.0 + 0.5)) - 1]
    j = np.arange(G, dtype=np.float64)
    theta = 1.0 / x[M - 1] + (1.0 - np.sqrt(G / (j + 0.5))) / (3.0 * xs)
    kt = np.array([np.mean(np.log1p(-t * x)) for t in theta])
    lt = M * (np.log(-theta / kt) - kt - 1.0)
    w = np.exp(lt - logsumexp(lt))
    th = np.sum(theta * w)
    k = np.mean(np.log1p(-th * x))
    sigma = -k / th
    k = (M * k + 5.0) / (M + 10.0)
    if np.isnan(k):
        k = np.inf
    return k, sigma


def psis(ll):
    """Smoothed, truncated log weights of one column of S log-likelihood draws and its Pareto k."""
    S = ll.size
    lw = -ll - np.max(-ll)
    M = tail_len(S)
    k = np.inf
    order = np.argsort(lw, kind="stable")
    tail_ids = order[S - M:]
    tail = lw[tail_ids]
    if M >= 5 and tail[0] != tail[-1]:
        cutoff = lw[order[S - M - 1]]
        ec = np.exp(cutoff)
        k, sigma = gpdfit(np.exp(tail) - ec)
        if np.isfinite(k):
            p = (np.arange(M, dtype=np.float64) + 0.5) / M
            q = -sigma * np.log1p(-p) if k == 0.0 else sigma * np.expm1(-k * np.log1p(-p)) / k
            lw = lw.copy()
            lw[tail_ids] = np.log(q + ec)
    lw = np.where(lw > 0.0, 0.0, lw)
    return lw, k


def loo_pointwise(ll):
    """ll: [S][n] pooled draws x observations.  dict of the [n] arrays elpd_loo, p_loo, pareto_k, elpd_waic, p_waic."""
    ll = np.asarray(ll, dtype=np.float64)
    S, n = ll.shape
    out = {k: np.empty(n) for k in ("elpd_loo", "p_loo", "pareto_k", "elpd_waic", "p_waic")}
    for i in range(n):
        c = ll[:, i]
        lw, k = psis(c)
        elpd = logsumexp(lw + c) - logsumexp(lw)
        lpd = logsumexp(c) - np.log(S)
        pw = np.var(c, ddof=1)
        out["elpd_loo"][i] = elpd
        out["p_loo"][i] = lpd - elpd
        out["pareto_k"][i] = k
        out["elpd_waic"][i] = lpd - pw
        out["p_waic"][i] = pw
    return out
