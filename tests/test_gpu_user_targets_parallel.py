"""User CUDA targets in the parallel protocol (cuda_target(..., parallel=True)): the threads of a chain evaluate the
density together, up to d = 4096, on the shapes the built-in targets run on (wn_user_plugin.cuh: UserParT).

Every case asserts the plan it ran on (ChainBatch.last_plan) and holds draws to 1e-10 (tests.helpers.close) with the
discrete diagnostics columns equal:
  - a diagonal Gaussian written in the parallel protocol against the built-in diag_gauss, every plan row and its
    boundaries, four integrators and package mode (more chains than resident slots);
  - a stationary Gaussian AR(1) prior, whose gradient reads the neighbours q[j-1] and q[j+1] (owned by other threads),
    per transition against the numpy oracle;
  - Neal's funnel with n = d - 1 (ctx.sum) and a logistic regression with rows split over the threads (ctx.scratch,
    ctx.sync), per transition against oracle.targets;
  - WALNUTS(tg, q0) with the reference's default adaptation, and a continuation against one call.
"""
import numpy as np
import pytest

from oracle import targets as ot
from oracle import walnutspy_oracle as wo
from tests.helpers import KIND, close
from walnuts_b200._ffi import FAMILIES

pytestmark = pytest.mark.gpu

EXACT = [0, 1, 4, 5, 6, 7, 8, 9, 12, 13, 19, 20, 21, 22]
EXT, PKG = FAMILIES["ext"], FAMILIES["pkg"]

DIAG_SRC = """
WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
  double lp = 0.0;
  for (int j = ctx.rank; j < WN_D; j += ctx.size) { g[j] = -q[j] * data[j]; lp += q[j] * g[j]; }
  return 0.5 * lp;
}"""

# lp = -1/2 (1 - phi^2) q0^2 - 1/2 sum_{j >= 1} (q_j - phi q_{j-1})^2, phi = data[0]
AR1_SRC = """
WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
  const double phi = data[0], c0 = 1.0 - phi * phi;
  double lp = 0.0;
  for (int j = ctx.rank; j < WN_D; j += ctx.size) {
    const double r = (j == 0) ? q[0] : q[j] - phi * q[j - 1];
    const double w = (j == 0) ? c0 : 1.0;
    lp -= 0.5 * w * r * r;
    const double up = (j + 1 < WN_D) ? phi * (q[j + 1] - phi * q[j]) : 0.0;
    g[j] = -(w * r) + up;
  }
  return lp;
}"""

FUNNEL_SRC = """
WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {   // oracle.targets.funnel10 with n = d - 1
  const double L2PI = 0.91893853320467274178, L3 = 1.09861228866810969140;
  const double n = (double)(WN_D - 1), q0 = q[0];
  double ss = 0.0;
  for (int j = ctx.rank; j < WN_D; j += ctx.size) if (j >= 1) ss += q[j] * q[j];
  ss = ctx.sum(ss);
  const double ex = exp(-q0), a = q0 / 3.0;
  for (int j = ctx.rank; j < WN_D; j += ctx.size)
    g[j] = (j == 0) ? -0.5 * n - q0 / 9.0 + 0.5 * ex * ss : -q[j] * ex;
  return (ctx.rank == 0) ? (-(a * a) / 2.0 - L2PI - L3) + (-0.5 * ex * ss - n * L2PI - n * 0.5 * q0) : 0.0;
}"""

# Bernoulli-logit likelihood, N(0, 1) prior; data = [X (N x d, row-major), y (N)].  Rows are split over the threads:
# each thread forms eta_n = x_n . q for its rows and stores y_n - sigmoid(eta_n) in the scratch, then (after the
# barrier) each thread forms the gradient entries it owns, X^T (y - sigmoid) - q.
LOGREG_SRC = """
WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
  const int N = n_data / (WN_D + 1);
  const double* X = data;
  const double* y = data + (size_t)N * WN_D;
  double* res = ctx.scratch;                       // N doubles: y - sigmoid(X q)
  double lp = 0.0;
  for (int n = ctx.rank; n < N; n += ctx.size) {
    const double* x = X + (size_t)n * WN_D;
    double eta = 0.0;
    for (int k = 0; k < WN_D; ++k) eta = fma(x[k], q[k], eta);
    lp += y[n] * eta - (fmax(eta, 0.0) + log1p(exp(-fabs(eta))));
    res[n] = y[n] - 0.5 * (1.0 + tanh(0.5 * eta));
  }
  ctx.sync();
  for (int j = ctx.rank; j < WN_D; j += ctx.size) {
    double s = 0.0;
    for (int n = 0; n < N; ++n) s = fma(X[(size_t)n * WN_D + j], res[n], s);
    g[j] = s - q[j];
    lp -= 0.5 * q[j] * q[j];
  }
  return lp;
}"""


def plan_of(d):
    for dmax, G, E2, NT in [(256, 32, 4, 128), (512, 32, 8, 128), (1024, 64, 8, 64), (2048, 256, 4, 256),
                            (4096, 512, 4, 512)]:
        if d <= dmax:
            return G, E2, NT


_PLUGINS = {}


@pytest.fixture(scope="module")
def plugin(cuda_lib):
    """cuda_target(src, d, parallel=True, scratch=...) -> target handle, compiled once per module."""
    import walnuts_b200 as wb

    def get(name, src, d, data=None, scratch=0):
        key = (name, d, scratch)
        if key not in _PLUGINS:
            _PLUGINS[key] = wb.targets.cuda_target(src, d, data=data, name=f"{name}{d}", parallel=True,
                                                   scratch=scratch)
        tg = _PLUGINS[key]
        if data is not None:   # the same plug-in with this call's data array
            tg = wb.targets.Target(tg.name, data={"data": np.ascontiguousarray(data, dtype=np.float64).ravel()},
                                   d=d, ref=tg.ref, plugin=tg.plugin)
        return tg
    return get


def run_batch(tg, q0, integrator, H0, delta, M, n_iter, seed, mode="walnutspy", inv_mass=None):
    import walnuts_b200 as wb
    from walnuts_b200 import ChainBatch
    n, d = q0.shape
    tid, data = wb.targets.resolve(tg, d)
    data = dict(data)
    if mode == "package":
        data["inv_mass"] = inv_mass
    with ChainBatch(tid, d, n, mode=mode, integrator=integrator, H0=H0, delta=delta, M=M, seed=seed,
                    data=data) as cb:
        cb.set_state(q0)
        out = cb.run(n_iter, draws=True, diag=(mode == "walnutspy"))
        out["plan"], out["slots"] = cb.last_plan(), cb.last_slots()
    return out


def per_transition(tg, lp, q0, integrator, H0, delta, M, n_iter, seed, plan):
    """Each transition from the oracle's previous state; returns the worst relative error of the draws."""
    from walnuts_b200 import ChainBatch
    import walnuts_b200 as wb
    n, d = q0.shape
    ref = np.empty((n_iter, n, d))
    refd = np.empty((n_iter, n, 24))
    for c in range(n):
        with np.errstate(all="ignore"):
            s, dg = wo.WALNUTS(lp, q0[c], integrator=KIND[integrator], H0=H0, delta0=delta, numIter=n_iter, M=M,
                               seed=seed, chain=c)
        ref[:, c], refd[:, c] = s[:, 1:].T, dg
    tid, data = wb.targets.resolve(tg, d)
    worst = 0.0
    with ChainBatch(tid, d, n, integrator=integrator, H0=H0, delta=delta, M=M, seed=seed, data=data) as cb:
        prev = q0
        for it in range(n_iter):
            cb.set_state(prev)
            out = cb.run(1, draws=True, diag=True)
            assert cb.last_plan() == plan, f"ran on plan {cb.last_plan()}, expected {plan}"
            ok, err = close(out["draws"][0], ref[it])
            worst = max(worst, err)
            assert ok, f"transition {it}: {err:.3e}"
            assert np.array_equal(out["diag"][0][:, EXACT], refd[it][:, EXACT]), f"transition {it}"
            prev = ref[it]
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# 1. the parallel diagonal Gaussian against the built-in diag_gauss
# ---------------------------------------------------------------------------------------------------------------------
SIZES = [100, 256, 257, 512, 513, 1024, 1025, 2048, 2049, 4096]
H_FOR = {"R2P": 1.4, "fixed": 1.0, "Yoshida": 1.4, "Flow": 1.4}
DELTA = {"R2P": 0.3, "fixed": 0.3, "Yoshida": 0.05, "Flow": 0.02}


@pytest.mark.parametrize("integrator", ["R2P", "fixed", "Yoshida", "Flow"])
@pytest.mark.parametrize("d", SIZES)
def test_diag_gauss_matches_builtin(plugin, d, integrator):
    import walnuts_b200 as wb
    rng = np.random.default_rng(d)
    sigma = np.exp(rng.uniform(-1.0, 1.0, d))
    q0 = rng.standard_normal((3, d)) * sigma
    tg = plugin("pdiag", DIAG_SRC, d, data=1.0 / sigma ** 2)
    H0 = sigma.min() * (d ** -0.5 if integrator == "fixed" else H_FOR[integrator] * d ** -0.25)
    args = (integrator, H0, DELTA[integrator], 6, 6, 21)
    a = run_batch(tg, q0, *args)
    b = run_batch(wb.targets.diag_gauss(sigma), q0, *args)
    assert a["plan"] == (EXT,) + plan_of(d), a["plan"]
    ok, err = close(a["draws"], b["draws"], scale=sigma)
    print(f"diag d={d} {integrator}: plan {a['plan']}, worst relative error {err:.2e}")
    assert ok, err
    assert np.array_equal(a["diag"][..., EXACT], b["diag"][..., EXACT])
    assert np.array_equal(a["nevalF"], b["nevalF"]) and np.array_equal(a["nevalB"], b["nevalB"])


# package mode, one size per plan row, with more chains than the kernel holds resident
PKG_CASES = [(256, 3500), (512, 1500), (1024, 1000), (2048, 600), (4096, 300)]


@pytest.mark.parametrize("d,n", PKG_CASES)
def test_diag_gauss_package_mode_matches_builtin(plugin, d, n):
    import walnuts_b200 as wb
    rng = np.random.default_rng(d + 1)
    sigma = np.exp(rng.uniform(-0.5, 0.5, d))
    q0 = rng.standard_normal((n, d)) * sigma
    inv_mass = np.exp(rng.uniform(-0.3, 0.3, d))
    tg = plugin("pdiag", DIAG_SRC, d, data=1.0 / sigma ** 2)
    args = ("fixed", 0.6 * sigma.min(), 0.3, 5, 3, 9)
    a = run_batch(tg, q0, *args, mode="package", inv_mass=inv_mass)
    b = run_batch(wb.targets.diag_gauss(sigma), q0, *args, mode="package", inv_mass=inv_mass)
    assert a["plan"] == (PKG,) + plan_of(d), a["plan"]
    assert a["slots"] < n, (a["slots"], n)
    ok, err = close(a["draws"], b["draws"], scale=sigma)
    print(f"package d={d}: plan {a['plan']}, {a['slots']} slots for {n} chains, worst relative error {err:.2e}")
    assert ok, err


# ---------------------------------------------------------------------------------------------------------------------
# 2. cross-coordinate reads: AR(1) prior
# ---------------------------------------------------------------------------------------------------------------------
def ar1_numpy(phi):
    """numpy restatement of AR1_SRC."""
    c0 = 1.0 - phi * phi

    def lp(q, hessian=False):
        r = np.empty_like(q)
        r[0] = q[0]
        r[1:] = q[1:] - phi * q[:-1]
        w = np.ones_like(q)
        w[0] = c0
        up = np.zeros_like(q)
        up[:-1] = phi * (q[1:] - phi * q[:-1])
        return [-0.5 * np.sum(w * r * r), -(w * r) + up]
    return lp


@pytest.mark.parametrize("integrator", ["R2P", "fixed"])
@pytest.mark.parametrize("d", [1025, 4096])
def test_ar1_cross_coordinate_reads(plugin, d, integrator):
    phi = 0.6
    tg = plugin("par1", AR1_SRC, d, data=np.array([phi]))
    q0 = np.random.default_rng(d).standard_normal((2, d))
    H0 = 0.25 if integrator == "fixed" else 0.5
    worst = per_transition(tg, ar1_numpy(phi), q0, integrator, H0, 0.3, 6, 4, 31, (EXT,) + plan_of(d))
    print(f"ar1 d={d} {integrator}: worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. ctx.sum: funnel with n = d - 1
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("integrator", ["fixed", "D", "R2P"])
@pytest.mark.parametrize("d", [513, 2049])
def test_funnel_ctx_sum(plugin, d, integrator):
    tg = plugin("pfunnel", FUNNEL_SRC, d)
    rng = np.random.default_rng(d)
    q0 = np.column_stack([np.array([0.3, -0.4]), 0.8 * rng.standard_normal((2, d - 1))])
    H0 = {"fixed": 0.05, "D": 0.2, "R2P": 0.2}[integrator]
    worst = per_transition(tg, ot.funnel10, q0, integrator, H0, 0.3, 6, 4, 17, (EXT,) + plan_of(d))
    print(f"funnel d={d} {integrator}: worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. ctx.scratch + ctx.sync: logistic regression, P = 1025, N = 2000, one saturated row
# ---------------------------------------------------------------------------------------------------------------------
def logreg_problem(P=1025, N=2000, seed=3):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, P)) / np.sqrt(P)
    beta = rng.standard_normal(P)
    y = (rng.uniform(size=N) < 1.0 / (1.0 + np.exp(-X @ beta))).astype(np.float64)
    X[0] = 400.0 / np.sqrt(P)        # |eta_0| ~ 400 |mean(q)| sqrt(P): the sigmoid saturates to 0 or 1
    y[0] = 1.0
    return X, y


@pytest.mark.parametrize("integrator", ["R2P", "fixed"])
def test_logreg_scratch_and_sync(plugin, integrator):
    P, N = 1025, 2000
    X, y = logreg_problem(P, N)
    tg = plugin("plogreg", LOGREG_SRC, P, data=np.concatenate([X.ravel(), y]), scratch=N)
    q0 = 0.3 * np.random.default_rng(5).standard_normal((2, P)) + 0.05
    assert np.all(np.abs(X[0] @ q0.T) > 20.0)     # the saturated row starts saturated
    H0 = 0.15 if integrator == "fixed" else 0.4
    worst = per_transition(tg, ot.make_logreg(X, y, 1.0), q0, integrator, H0, 0.3, 6, 3, 23, (EXT,) + plan_of(P))
    print(f"logreg P={P} N={N} {integrator}: worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 5. WALNUTS(tg, q0) with the reference's default adaptation; continuation
# ---------------------------------------------------------------------------------------------------------------------
def test_walnuts_default_adaptation_d2048(plugin):
    import walnuts_b200 as wb
    from walnuts_b200 import ChainBatch
    d, n, n_iter, warm = 2048, 2, 16, 12
    rng = np.random.default_rng(2048)
    sigma = np.exp(rng.uniform(-0.5, 0.5, d))
    q0 = rng.standard_normal((n, d)) * sigma
    tg = plugin("pdiag", DIAG_SRC, d, data=1.0 / sigma ** 2)
    s, dg = wb.WALNUTS(tg, q0, numIter=n_iter, warmupIter=warm, seed=41)
    worst = 0.0
    for c in range(n):
        with np.errstate(all="ignore"):
            so, do = wo.WALNUTS(ot.make_diag_gauss(sigma), q0[c], integrator=wo.FIXED, numIter=n_iter, M=10, seed=41,
                                chain=c, warmupIter=warm, adaptH=True, adaptDelta=True)
        # warm-up feeds each transition's energy error (a sum over d whose last bits depend on the summation order)
        # back into H and delta: held to 1e-6 with the discrete columns exact (DESIGN.md section 5)
        ok, err = close(s[c], so, rtol=1e-6, axis=-2)
        worst = max(worst, err)
        assert ok, err
        assert np.array_equal(dg[c][:, EXACT], do[:, EXACT])
    print(f"WALNUTS default adaptation d={d}: worst relative error {worst:.2e}")
    # continuation: 5 + 11 transitions in two calls equal 16 in one
    tid, data = wb.targets.resolve(tg, d)
    outs = []
    for split in ((n_iter,), (5, n_iter - 5)):
        with ChainBatch(tid, d, n, integrator="fixed", seed=41, data=data) as cb:
            cb.set_adapt(warm)
            cb.set_state(q0)
            parts = [cb.run(k, draws=True, diag=True) for k in split]
            assert cb.last_plan() == (EXT,) + plan_of(d)
        outs.append((np.concatenate([p["draws"] for p in parts]), np.concatenate([p["diag"] for p in parts])))
    assert np.array_equal(outs[0][0], outs[1][0])
    assert np.array_equal(outs[0][1], outs[1][1], equal_nan=True)
