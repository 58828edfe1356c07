"""Cross-chain convergence diagnostics from the per-chain summaries the sampler streams on the device
(mean, population std, number of kept rows) — no raw chains needed, so they are available for
BASELINE config 3 (299 cells x 64 chains, whose raw chains would be 3.9 TB).

Not part of the reference (SURVEY.md 8f rank 4): `TranscriptionCycleMCMC.m` runs one chain per cell and
reports no diagnostic; with 'numChains' > 1 the extra variable `MCMCdiagnostics` is written next to
`MCMCresults` (the reference's layout is untouched).

Gelman-Rubin potential scale reduction (Gelman et al., BDA3 11.4, without chain splitting):
    W  = mean_c s_c^2                      within-chain variance (s_c^2 with n-1 normalisation)
    B  = n * var_c(mean_c)                 between-chain variance (m-1 normalisation)
    V+ = (n-1)/n * W + B/n
    Rhat = sqrt(V+ / W),   n_eff ~= m * n * V+ / B   (capped at m*n)
`n_eff` from summaries is the BETWEEN-CHAIN estimate: it is read off the scatter of the m chain means (m - 1 degrees of
freedom: the right order of magnitude, no more) and never looks at the autocorrelation inside a chain.  When the raw chains are kept
('saveChains') the proper quantities are computed from them: split-Rhat (every chain cut in halves: also detects a single
chain that is still drifting) and the effective sample size from the autocorrelation (Geyer's initial positive / monotone
sequence over the chain-averaged autocovariance, as in BDA3 11.5 / Stan).
"""
import numpy as np


def rhat_from_summaries(means, stds, n):
    """means, stds: [m chains x p parameters] per-chain mean and POPULATION std (what tc_mcmc_run returns);
    n: kept rows per chain.  Returns (Rhat[p], n_eff[p]); NaN where a parameter did not move in any chain."""
    means = np.asarray(means, dtype=np.float64); stds = np.asarray(stds, dtype=np.float64)
    m = means.shape[0]
    if m < 2 or n < 2:
        raise ValueError("diagnostics need at least 2 chains of at least 2 rows")
    W = (stds ** 2).mean(axis=0) * n / (n - 1.0)
    B = n * means.var(axis=0, ddof=1)
    Vp = (n - 1.0) / n * W + B / n
    with np.errstate(divide="ignore", invalid="ignore"):
        rhat = np.sqrt(Vp / W)
        neff = np.minimum(m * n * Vp / B, float(m * n))
    rhat[~(W > 0)] = np.nan
    neff[~(W > 0)] = np.nan
    return rhat, neff


def split_rhat(chains):
    """chains [m, n, p] -> split-Rhat [p]: every chain is cut in two halves (2m sequences of n//2 rows), then Gelman-Rubin.
    Works with m = 1 (the reference's one chain per cell): the two halves of the same chain must agree."""
    x = np.asarray(chains, dtype=np.float64)
    m, n, p = x.shape
    h = n // 2
    if h < 2:
        raise ValueError("split-Rhat needs at least 4 rows per chain")
    y = np.concatenate([x[:, :h], x[:, n - h:]], axis=0)               # [2m, h, p]
    W = y.var(axis=1, ddof=1).mean(axis=0)
    B = h * y.mean(axis=1).var(axis=0, ddof=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.sqrt(((h - 1.0) / h * W + B / h) / W)
    r[~(W > 0)] = np.nan
    return r


def ess(chains):
    """chains [m, n, p] -> effective sample size [p] of the pooled m*n draws, from the autocorrelation: rho_t = 1 -
    (W - mean_c acov_c(t)) / V+ (BDA3 11.5), summed over Geyer's initial positive, monotone sequence of pair sums.
    The draws are the rows given: for chains stored with 'thin' = k (every k-th row) it counts stored draws, at most m*n."""
    x = np.asarray(chains, dtype=np.float64)
    m, n, p = x.shape
    if n < 4:
        raise ValueError("ess needs at least 4 rows per chain")
    xc = x - x.mean(axis=1, keepdims=True)
    nfft = 1 << int(np.ceil(np.log2(2 * n)))
    f = np.fft.rfft(xc, nfft, axis=1)
    acov = np.fft.irfft(f * np.conj(f), nfft, axis=1)[:, :n] / n        # biased autocovariance per chain [m, n, p]
    W = (acov[:, 0] * n / (n - 1.0)).mean(axis=0)
    B_over_n = x.mean(axis=1).var(axis=0, ddof=1) if m > 1 else np.zeros(p)
    Vp = (n - 1.0) / n * W + B_over_n
    out = np.full(p, np.nan)
    mean_acov = acov.mean(axis=0)                                       # [n, p]
    for j in range(p):
        if not (W[j] > 0 and Vp[j] > 0):
            continue
        rho = 1.0 - (W[j] - mean_acov[:, j]) / Vp[j]
        rho[0] = 1.0
        npair = (n - 1) // 2
        pairs = rho[0:2 * npair:2] + rho[1:2 * npair:2]                 # Gamma_k = rho_2k + rho_2k+1
        neg = np.flatnonzero(pairs < 0)
        kmax = neg[0] if neg.size else npair
        g = np.minimum.accumulate(pairs[:kmax]) if kmax > 0 else np.zeros(0)
        tau = -1.0 + 2.0 * g.sum()
        out[j] = min(m * n / max(tau, 1.0 / np.log10(max(m * n, 10))), float(m * n))
    return out
