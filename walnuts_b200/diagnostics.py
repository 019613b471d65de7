"""Cross-chain convergence diagnostics: bulk ESS and R-hat (Vehtari, Gelman, Simpson, Carpenter,
Buerkner 2021), the quantities the reference's experiment scripts obtain from arviz
(`az.ess`, WALNUTSpy_examples/gaussian/mainGaussESS.py:17,50-55), and the posterior summary (`summary`: quantiles,
MCSEs, tail ESS, folded R-hat, nested R-hat).  arviz is not a dependency here.

Inputs are draws of ONE scalar quantity with shape (n_chains, n_draws), as numpy arrays or torch
tensors (the same code runs on the GPU for the many-chain case: 65 536 chains x tens of draws).
For multi-GPU runs `ess_from_stats` consumes per-rank sufficient statistics so that only O(lags)
numbers per coordinate cross NVLink (one all-reduce / all-gather at the end of sampling).
"""
import math

import numpy as np


def _xp(x):
    if type(x).__module__.startswith("torch"):
        import torch
        return torch
    return np


def rank_normalize(x):
    """z = Phi^-1((rank - 3/8) / (S + 1/4)) over all draws of all chains (average ranks for ties are
    replaced by ordinal ranks; ties have probability zero for continuous targets)."""
    xp = _xp(x)
    flat = x.reshape(-1)
    S = flat.shape[0]
    if xp is np:
        order = np.argsort(flat, kind="stable")
        ranks = np.empty(S, dtype=np.float64)
        ranks[order] = np.arange(1, S + 1, dtype=np.float64)
        p = (ranks - 0.375) / (S + 0.25)
        from scipy.special import ndtri
        return ndtri(p).reshape(x.shape)
    order = xp.argsort(flat, stable=True)
    ranks = xp.empty(S, dtype=xp.float64, device=flat.device)
    ranks[order] = xp.arange(1, S + 1, dtype=xp.float64, device=flat.device)
    p = (ranks - 0.375) / (S + 0.25)
    return (math.sqrt(2.0) * xp.erfinv(2.0 * p - 1.0)).reshape(x.shape)


def chain_stats(x, max_lag=None):
    """Per-rank sufficient statistics of (n_chains, n) draws:
    dict(m = n_chains, n, sum_mean, sum_mean2, sum_var, acov_sum[max_lag+1]) where acov_sum[t] is the
    sum over chains of the (biased, 1/n) lag-t autocovariance.  Additive across ranks."""
    xp = _xp(x)
    m, n = x.shape
    max_lag = n - 1 if max_lag is None else min(max_lag, n - 1)
    mean = x.mean(1, keepdims=True) if xp is np else x.mean(1, keepdim=True)
    xc = x - mean
    acov = []
    for t in range(max_lag + 1):
        acov.append(((xc[:, :n - t] * xc[:, t:]).sum() / n))
    acov = xp.stack(acov) if xp is not np else np.array(acov)
    var_c = (xc * xc).sum(1) / (n - 1)
    return dict(m=m, n=n, sum_mean=mean.sum(), sum_mean2=(mean * mean).sum(), sum_var=var_c.sum(),
                acov_sum=acov)


def ess_from_stats(st):
    """(ESS, R-hat) from (summed) chain_stats.  The estimator is the one arviz / Stan use (Geyer's
    initial positive + monotone sequence on the chain-averaged autocorrelations)."""
    m, n = int(st["m"]), int(st["n"])
    acov = np.asarray([float(a) for a in st["acov_sum"]], dtype=np.float64) / m   # mean over chains, 1/n form
    T = len(acov)
    if n < 4 or T < 2:
        return float("nan"), float("nan")
    mean_var = float(st["sum_var"]) / m                         # W
    mean_of_means = float(st["sum_mean"]) / m
    var_plus = mean_var * (n - 1.0) / n
    if m > 1:
        var_plus += (float(st["sum_mean2"]) - m * mean_of_means ** 2) / (m - 1)   # B / n
    if not (var_plus > 0):
        return float("nan"), float("nan")

    def rho(t):
        return 1.0 - (mean_var - acov[t]) / var_plus if t < T else 0.0

    rho_hat = np.zeros(n + 2)
    even = 1.0
    rho_hat[0] = even
    odd = rho(1)
    rho_hat[1] = odd
    t = 1
    while t < (n - 3) and (even + odd) > 0.0:
        even, odd = rho(t + 1), rho(t + 2)
        if (even + odd) >= 0:
            rho_hat[t + 1], rho_hat[t + 2] = even, odd
        t += 2
    max_t = t - 2
    if even > 0:
        rho_hat[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        if (rho_hat[t + 1] + rho_hat[t + 2]) > (rho_hat[t - 1] + rho_hat[t]):
            rho_hat[t + 1] = (rho_hat[t - 1] + rho_hat[t]) / 2.0
            rho_hat[t + 2] = rho_hat[t + 1]
        t += 2
    ess = m * n
    tau = -1.0 + 2.0 * np.sum(rho_hat[:max_t + 1]) + np.sum(rho_hat[max_t + 1:max_t + 2])
    tau = max(tau, 1.0 / math.log10(ess))
    rhat = math.sqrt(var_plus / mean_var) if mean_var > 0 else float("nan")
    return ess / tau, rhat


def ess_bulk(x, split=True, max_lag=None):
    """Bulk ESS (rank-normalised, split chains) and split-R-hat of draws x (n_chains, n_draws)."""
    z = rank_normalize(x)
    n = z.shape[1]
    if split and n >= 4:
        h = n // 2
        xp = _xp(z)
        z = xp.concatenate([z[:, :h], z[:, n - h:]], 0) if xp is np else xp.cat([z[:, :h], z[:, n - h:]], 0)
    return ess_from_stats(chain_stats(z, max_lag))


def _split_ess(y):
    """(ESS, R-hat) of y (n_chains, n) split into halves [0, h) and [n - h, n), h = n // 2, without rank
    normalisation."""
    n = y.shape[1]
    h = n // 2
    return ess_from_stats(chain_stats(np.concatenate([y[:, :h], y[:, n - h:]], 0)))


def summary(x, superchain_size=None):
    """Posterior summary of ONE quantity, draws x (n_chains, n_draws) with n_draws >= 4 (numpy; a torch tensor is
    copied to the host): a dict of floats keyed mean, sd, q05, q50, q95, mcse_mean, mcse_sd, ess_bulk, ess_tail, rhat,
    nested_rhat.  The host statement of what ChainBatch.summary / wn_summary compute on the device.

    With M chains of N draws, S = M N, and "split ESS of y" = ESS of y with every chain split into [0, N // 2) and
    [N - N // 2, N), without rank normalisation:
      mean, sd       over all S draws, sd with 1 / (S - 1)
      q05, q50, q95  np.quantile of the S draws (linear interpolation, numpy's default)
      mcse_mean      sd / sqrt(split ESS of x)
      mcse_sd        c = (x - mean)^2, E = mean(c), varvar = (mean(c^2) - E^2) / split ESS of c, sqrt(varvar / (4 E))
      ess_bulk       ess_bulk(x)[0]: rank-normalised split ESS
      ess_tail       min(split ESS of 1[x <= q05], split ESS of 1[x <= q95])
      rhat           max(ess_bulk(x)[1], ess_bulk(|x - q50|)[1]): bulk and folded split-R-hat
      nested_rhat    (superchain_size = s; chains k*s ... k*s + s - 1 form superchain k, K = M / s >= 2)
                     sqrt(1 + B / W), B = 1/(K-1) sum_k (xbar_k - xbar)^2 over the superchain means,
                     W = 1/K sum_k (Btilde_k + Wtilde_k), Btilde_k = 1/(s-1) sum_m (xbar_mk - xbar_k)^2 (0 if s = 1),
                     Wtilde_k = 1/s sum_m var_mk (within-chain variance, 1 / (N - 1)); raw draws, not ranks.
                     NaN without superchain_size (Margossian, Hoffman, Sountsov, Riou-Durand, Vehtari, Gelman 2024).
    Ranks are ordinal and taken over all S draws before the split (for odd N the middle draw is ranked but dropped); an
    ESS or R-hat of a series with zero variance is NaN, and so is every column computed from one (min / max are NaN
    when either argument is).  ValueError for fewer than 4 draws or a superchain size that does not give at least 2
    superchains."""
    if _xp(x) is not np:
        x = x.detach().cpu().numpy()
    x = np.asarray(x, dtype=np.float64)
    if x.ndim != 2 or x.shape[1] < 4:
        raise ValueError("summary: draws must be (n_chains, n_draws >= 4)")
    m, n = x.shape
    s = int(superchain_size or 0)
    if s < 0 or (s > 0 and (m % s != 0 or m // s < 2)):
        raise ValueError(f"summary: {m} chains do not form at least 2 superchains of {superchain_size}")
    S = x.size
    with np.errstate(divide="ignore", invalid="ignore"):
        mean = x.mean()
        sd = np.sqrt(((x - mean) ** 2).sum() / (S - 1))
        q05, q50, q95 = np.quantile(x.reshape(-1), [0.05, 0.5, 0.95])
        ess_b, rhat_b = (np.float64(v) for v in ess_bulk(x))
        rhat_f = np.float64(ess_bulk(np.abs(x - q50))[1])
        ess_05 = np.float64(_split_ess((x <= q05).astype(np.float64))[0])
        ess_95 = np.float64(_split_ess((x <= q95).astype(np.float64))[0])
        c = (x - mean) ** 2
        E = c.mean()
        varvar = ((c * c).mean() - E * E) / np.float64(_split_ess(c)[0])
        nested = np.float64("nan")
        if s > 0:
            xm = x.mean(1).reshape(-1, s)                      # chain means by superchain
            xv = x.var(1, ddof=1).reshape(-1, s)
            xk = xm.mean(1)
            bt = ((xm - xk[:, None]) ** 2).sum(1) / (s - 1) if s > 1 else np.zeros_like(xk)
            B = xk.var(ddof=1)
            W = (bt + xv.mean(1)).mean()
            nested = np.sqrt(1.0 + B / W)
        return dict(mean=float(mean), sd=float(sd), q05=float(q05), q50=float(q50), q95=float(q95),
                    mcse_mean=float(sd / np.sqrt(np.float64(_split_ess(x)[0]))), mcse_sd=float(np.sqrt(varvar / (4 * E))),
                    ess_bulk=float(ess_b), ess_tail=float(np.minimum(ess_05, ess_95)),
                    rhat=float(np.maximum(rhat_b, rhat_f)), nested_rhat=float(nested))


def min_ess(draws, split=True, max_lag=None):
    """min over coordinates of bulk ESS; draws (n_iter, n_chains, k) as produced by wn_run."""
    k = draws.shape[2]
    vals = []
    for j in range(k):
        xj = draws[:, :, j].T if _xp(draws) is np else draws[:, :, j].t()
        vals.append(ess_bulk(xj, split, max_lag)[0])
    return min(vals), vals
