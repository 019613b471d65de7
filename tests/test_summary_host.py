"""diagnostics.summary on the host: every column against a literal transcription of its definition, and the statistical
behaviour of the columns on draws with known answers (iid, AR(1), superchains with and without shifted means)."""
import math

import numpy as np
import pytest

from walnuts_b200 import diagnostics as dg


def ar1(m, n, rho, rng):
    x = np.empty((m, n))
    x[:, 0] = rng.standard_normal(m)
    for t in range(1, n):
        x[:, t] = rho * x[:, t - 1] + math.sqrt(1 - rho * rho) * rng.standard_normal(m)
    return x


# ---- the definitions, transcribed --------------------------------------------------------------------------------
def split_ess(y):
    """ESS of y with every chain split into [0, h) and [N - h, N), h = N // 2, without rank normalisation."""
    N = y.shape[1]
    h = N // 2
    halves = [y[c, :h] for c in range(y.shape[0])] + [y[c, N - h:] for c in range(y.shape[0])]
    return dg.ess_from_stats(dg.chain_stats(np.array(halves)))


def linear_quantile(x, p):
    s = np.sort(x.reshape(-1))
    v = (s.size - 1) * p
    i = int(math.floor(v))
    if i >= s.size - 1:
        return s[-1]
    return s[i] + (s[i + 1] - s[i]) * (v - i)


def nested_rhat(x, s):
    M, N = x.shape
    K = M // s
    cmean = [sum(x[c]) / N for c in range(M)]
    cvar = [sum((v - cmean[c]) ** 2 for v in x[c]) / (N - 1) for c in range(M)]
    xk = [sum(cmean[k * s + m] for m in range(s)) / s for k in range(K)]
    xbar = sum(xk) / K
    B = sum((v - xbar) ** 2 for v in xk) / (K - 1)
    W = 0.0
    for k in range(K):
        bt = sum((cmean[k * s + m] - xk[k]) ** 2 for m in range(s)) / (s - 1) if s > 1 else 0.0
        wt = sum(cvar[k * s + m] for m in range(s)) / s
        W += (bt + wt) / K
    return math.sqrt(1 + B / W)


def transcribed(x, s=None):
    S = x.size
    mean = x.sum() / S
    sd = math.sqrt(((x - mean) ** 2).sum() / (S - 1))
    q05, q50, q95 = (linear_quantile(x, p) for p in (0.05, 0.5, 0.95))
    c = (x - mean) ** 2
    E = c.mean()
    varvar = ((c ** 2).mean() - E ** 2) / split_ess(c)[0]
    return dict(mean=mean, sd=sd, q05=q05, q50=q50, q95=q95,
                mcse_mean=sd / math.sqrt(split_ess(x)[0]),
                mcse_sd=math.sqrt(varvar / (4 * E)),
                ess_bulk=split_ess(dg.rank_normalize(x))[0],
                ess_tail=min(split_ess((x <= q05).astype(float))[0], split_ess((x <= q95).astype(float))[0]),
                rhat=max(split_ess(dg.rank_normalize(x))[1], split_ess(dg.rank_normalize(np.abs(x - q50)))[1]),
                nested_rhat=nested_rhat(x, s) if s else float("nan"))


@pytest.mark.parametrize("m,n,s", [(1, 40, None), (8, 33, 4), (12, 50, 1), (16, 21, 16 // 2)])
def test_summary_matches_transcribed_definitions(m, n, s):
    rng = np.random.default_rng(m * 100 + n)
    x = 1.5 + ar1(m, n, 0.6, rng) * np.exp(rng.uniform(-0.5, 0.5, (m, 1)))     # chains of different scales
    got, want = dg.summary(x, s), transcribed(x, s)
    assert list(got) == list(want)
    for k in want:
        if math.isnan(want[k]):
            assert math.isnan(got[k]), k
        else:
            assert abs(got[k] - want[k]) <= 1e-12 * abs(want[k]), (k, got[k], want[k])


def test_summary_columns_are_the_c_abi_columns():
    from walnuts_b200 import _ffi
    assert tuple(dg.summary(np.random.default_rng(0).standard_normal((2, 8)))) == _ffi.SUMMARY_COLS


def test_iid_normal_ess_near_draw_count():
    x = np.random.default_rng(1).standard_normal((64, 200))
    r = dg.summary(x)
    S = x.size
    ess_mean = (r["sd"] / r["mcse_mean"]) ** 2
    for e in (r["ess_bulk"], r["ess_tail"], ess_mean):
        assert 0.8 * S < e < 1.25 * S, e
    assert abs(r["rhat"] - 1) < 0.01 and math.isnan(r["nested_rhat"])
    assert abs(r["q05"] + 1.645) < 0.05 and abs(r["q50"]) < 0.03 and abs(r["q95"] - 1.645) < 0.05
    assert abs(r["mcse_sd"] - 1 / math.sqrt(2 * S)) < 0.2 / math.sqrt(2 * S)       # var(sd) = sigma^2 / (2 S) for iid normals


def test_ar1_mean_ess():
    rho = 0.9
    x = ar1(64, 1000, rho, np.random.default_rng(2))
    r = dg.summary(x)
    expect = x.size * (1 - rho) / (1 + rho)
    ess_mean = (r["sd"] / r["mcse_mean"]) ** 2
    assert 0.85 * expect < ess_mean < 1.15 * expect, (ess_mean, expect)


def test_nested_rhat_detects_shifted_superchains():
    rng = np.random.default_rng(3)
    K, s, n = 16, 8, 20
    x = rng.standard_normal((K * s, n))
    assert abs(dg.summary(x, s)["nested_rhat"] - 1) < 0.05                          # exchangeable superchains
    shifted = x + np.repeat(rng.normal(0.0, 1.0, K), s)[:, None]                  # one offset per superchain
    assert dg.summary(shifted, s)["nested_rhat"] > 1.3
    # the same offsets spread over all chains of every superchain leave the superchain means alike
    mixed = x + np.tile(rng.normal(0.0, 1.0, s), K)[:, None]
    assert dg.summary(mixed, s)["nested_rhat"] < dg.summary(shifted, s)["nested_rhat"]


def test_folded_rhat_sees_scale_differences():
    rng = np.random.default_rng(4)
    x = rng.standard_normal((8, 400))
    x[:4] *= 3.0                                                                  # same location, different scale
    r = dg.summary(x)
    assert r["rhat"] > 1.1 and dg.ess_bulk(x)[1] < 1.02


def test_constant_draws_give_nan():
    r = dg.summary(np.full((4, 10), 2.5), 2)
    assert r["mean"] == 2.5 and r["sd"] == 0.0 and r["q05"] == r["q50"] == r["q95"] == 2.5
    for k in ("mcse_mean", "mcse_sd", "ess_tail", "nested_rhat"):
        assert math.isnan(r[k]), k


@pytest.mark.parametrize("m,s", [(8, 3), (8, 8), (8, -1), (1, 1)])
def test_bad_superchain_size_raises(m, s):
    with pytest.raises(ValueError):
        dg.summary(np.random.default_rng(5).standard_normal((m, 10)), s)


def test_too_few_draws_raise():
    with pytest.raises(ValueError):
        dg.summary(np.zeros((4, 3)))
