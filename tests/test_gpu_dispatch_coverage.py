"""Parity of the kernel instantiations that the benchmarked shapes do not reach, and a check that the suite keeps up
with the dispatcher.

Every transition kernel comes from wn_dispatch.cuh: one template instantiation per (family, target, dimension range),
family = plain WALNUTSpy D / R2P ("wpy"), plain NUTS ("nuts"), package mode ("pkg"), the general kernels behind
Yoshida, warm-up adaptation and orbit statistics ("adapt") and Flow / Midpoint / Rescaled ("ext").  Each case below
names the (family, G, E2, NT) it must run on -- read back with ChainBatch.last_plan() -- and compares against the
oracle at the usual tolerances: draws to 1e-10 through helpers.close, the discrete diagnostics (EXACT_COLS, which
include the evaluation counts) exactly.  Shapes are tested at their capacity (2 G E2 coordinates, G * 4 time steps
for Stock-Watson) and one past it, where the last thread holds padding lanes.  Chaotic targets (funnels,
Stock-Watson) are compared per transition on identical inputs, as in test_funnel10.

test_every_dispatched_plan_has_a_parity_test walks every built-in target, every family trigger and every dimension
boundary of the dispatcher and requires each plan it sees to be covered by a case here or by an existing test named
in ALREADY_COVERED: a shape added to the dispatcher fails it until a parity case exists.
"""
import numpy as np
import pytest

from oracle import package_oracle as po
from oracle import targets as ot
from oracle import walnutspy_oracle as wo
from tests.helpers import KIND, close, close_diag, oracle_target, oracle_walnutspy
from tests.test_gpu_walnutspy_parity import EXACT_COLS, FLOAT_COLS, check, check_forced, q0_for, sw_q0
from walnuts_b200._ffi import FAMILIES

pytestmark = pytest.mark.gpu

FAMILY = FAMILIES      # WN_FAMILY_*
FAMILY_NAME = {v: k for k, v in FAMILY.items()}
DELTA = {"Yoshida": 0.05, "Flow": 0.02, "Midpoint": 0.05, "Rescaled": 0.3}
TAU = 0.5        # logistic-regression prior scale: 1 / tau^2 = 4 is not an identity


# ---------------------------------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------------------------------
def sw_series(T):
    """Stock-Watson observations of length T: the stored T = 252 series (tests/golden/sw_y.npy), extended
    deterministically by appending it reversed and then again forwards (y, y[::-1], y, ...), cut to T."""
    y = ot.load_sw_data()
    reps = [y if k % 2 == 0 else y[::-1] for k in range(-(-T // y.size))]
    return np.concatenate(reps)[:T].copy()


def logreg_data(N, P, seed=0):
    """Synthetic logistic regression (synth_logreg_data) with rows that take the numerically special paths of the
    likelihood.  Coordinate 0 is pinned near beta_0 ~ 2 (N // 6 rows e_0 with y = 1 against the N(0, TAU^2) prior), so
    that rows along e_0 have a predictable linear predictor eta = X_n beta:
      row 0       40 e_0, y = 1     eta ~ +70 (> 37): the sigmoid rounds to 1 (first row tile)
      row N // 2  all zero          eta = 0
      row N - 3   -40 e_0, y = 0    eta ~ -70: the sigmoid rounds to 0
      row N - 2   -800 e_0, y = 0   eta ~ -1400 (< -710): exp(|eta|) overflows, exp(-|eta|) underflows
    The last row N - 1 is an ordinary row (it ends the ragged last tile).  Returns X, y and the special rows."""
    X, y, _ = ot.synth_logreg_data(N=N, P=P, seed=seed)
    pin = np.arange(1, 1 + N // 6)
    X[pin] = 0.0
    X[pin, 0] = 1.0
    y[pin] = 1.0
    X[N // 2] = 0.0
    special = {"sat": [0, N - 3], "zero": [N // 2], "huge": [N - 2]}
    for r, (s, yy) in zip((0, N - 3, N - 2), ((40.0, 1.0), (-40.0, 0.0), (-800.0, 0.0))):
        X[r] = 0.0
        X[r, 0] = s
        y[r] = yy
    return X, y, special


def logreg_q0(n, P, seed=4):
    q0 = 0.2 * np.random.default_rng(seed).standard_normal((n, P))
    q0[:, 0] += 2.0
    return q0


def check_logreg_rows_hit(data, special, draws):
    """The special rows really take their paths at the oracle's states."""
    eta = np.asarray(draws).reshape(-1, data["X"].shape[1]) @ data["X"].T
    assert (np.abs(eta[:, special["sat"]]) > 37.0).all(), np.abs(eta[:, special["sat"]]).min()
    assert (eta[:, special["zero"]] == 0.0).all()
    assert (np.abs(eta[:, special["huge"]]) > 710.0).all(), np.abs(eta[:, special["huge"]]).min()


def funnel_q0(n, d, seed=3, scale=0.7):
    rng = np.random.default_rng(seed)
    q0 = np.empty((n, d))
    q0[:, 0] = scale * rng.standard_normal(n)
    q0[:, 1:] = np.exp(0.5 * q0[:, :1]) * rng.standard_normal((n, d - 1))
    return q0


def random_precision(d, seed, cond=20.0):
    rng = np.random.default_rng(seed)
    Qm, _ = np.linalg.qr(rng.standard_normal((d, d)))
    ev = np.exp(rng.uniform(-0.5 * np.log(cond), 0.5 * np.log(cond), d))
    P = (Qm * ev) @ Qm.T
    return 0.5 * (P + P.T)


def problem(target, d, n, seed=5, N=None):
    """(q0 [n, d], data, H0 scale) of a small well-posed problem of `target` at dimension d."""
    if target == "std_normal":
        return q0_for(n, d, seed=seed), {}, 1.0
    if target == "diag_gauss":
        sigma = np.exp(np.linspace(-1.0, 1.0, d))
        return q0_for(n, d, seed=seed) * sigma, {"inv_var": 1.0 / sigma ** 2}, sigma.min()
    if target in ("funnel", "funnel_pkg"):
        return funnel_q0(n, d, seed=seed), {}, 0.4
    if target == "logreg":
        X, y, _ = logreg_data(N or 257, d)
        return logreg_q0(n, d), {"X": X, "y": y, "tau": np.array([TAU])}, 0.3
    if target == "stock_watson":
        T = d // 3
        return sw_q0(n, T), {"y": sw_series(T)}, 0.1
    if target == "dense_gauss":
        P = random_precision(d, seed=d)
        L = np.linalg.cholesky(np.linalg.inv(P))
        return np.random.default_rng(seed).standard_normal((n, d)) @ L.T, {"precision": P}, \
            float(np.sqrt(1.0 / np.linalg.eigvalsh(P).max()))
    if target == "corr_gauss":
        return np.tile(np.array([1.0, 0.0]), (n, 1)), {}, 1.0
    raise KeyError(target)


def step_size(target, d, integrator, scale):
    if target == "stock_watson":
        return 0.002 if integrator == "fixed" else 0.1
    base = {"fixed": 0.5, "Yoshida": 1.2}.get(integrator, 0.9)
    return base * scale * min(1.0, (11.0 / d) ** 0.25) if target in ("funnel", "funnel_pkg", "logreg") \
        else base * scale * d ** -0.25


def pkg_lp(target, data):
    """Package-protocol (logp, grad) of a target."""
    if target == "std_normal":
        return ot.standard_normal_lpdf, ot.standard_normal_grad
    if target == "funnel_pkg":
        return ot.funnel_lpdf, ot.funnel_grad
    f = oracle_target(target, None, data)
    return (lambda q: f(q)[0]), (lambda q: f(q)[1])


# ---------------------------------------------------------------------------------------------------------------------
# runners
# ---------------------------------------------------------------------------------------------------------------------
def plan_of(family, shape):
    return (FAMILY[family],) + tuple(shape)


def run_walnutspy(target, d, integrator, family, shape, forced, n_iter, n_chains=3, N=None, M=None, seed=1234):
    """Plain WALNUTSpy-mode parity through check (free-running) or check_forced (per transition)."""
    q0, data, scale = problem(target, d, n_chains, N=N)
    H0 = step_size(target, d, integrator, scale)
    delta = DELTA.get(integrator, 0.3)
    minC = 3 if target == "stock_watson" and integrator != "fixed" else 0
    M = M or (5 if target == "stock_watson" and integrator != "fixed" else 6)
    plan = plan_of(family, shape)
    if forced:
        dg, worst = check_forced(target, q0, integrator, H0=H0, delta=delta, M=M, n_iter=n_iter, seed=seed, minC=minC,
                                 data=data, plan=plan)
    else:
        chains = [0, n_chains - 1]
        dg = check(target, q0, integrator, H0=H0, delta=delta, M=M, n_iter=n_iter, seed=seed, chains=chains,
                   minC=minC, data=data, float_rtol=1e-8, plan=plan)      # float diagnostics as in test_logreg
        worst = None
    print(f"{target} d={d} {integrator}: plan {family} {shape}" +
          (f", worst relative error per transition {worst:.2e}" if worst is not None else ""))
    if target == "logreg":        # the special rows take their paths at chain 0's states
        draws_o, _ = oracle_walnutspy(target, q0, integrator, H0, delta, M, n_iter, seed, [0], minC, 10, data)
        check_logreg_rows_hit(data, logreg_data(N or 257, d)[2], np.concatenate([q0[:1], draws_o[:, 0]]))
    return dg


def run_adapt(target, d, shape, warmup, orbit, n_iter, integrator="R2P", n_chains=3, N=None, seed=77):
    """The general ("adapt") kernels through warm-up adaptation and / or orbit statistics against wo.WALNUTS with
    warmupIter / recordOrbitStats, free-running (non-chaotic targets only)."""
    from walnuts_b200 import ChainBatch
    q0, data, scale = problem(target, d, n_chains, N=N)
    H0 = step_size(target, d, integrator, scale)
    delta, M = 0.3, 6
    with ChainBatch(target, d, n_chains, integrator=integrator, H0=H0, delta=delta, M=M, seed=seed, data=data) as cb:
        if warmup:
            cb.set_adapt(n_iter)
        cb.set_state(q0)
        out = cb.run(n_iter, draws=True, diag=True, orbit_stats=orbit)
        assert cb.last_plan() == plan_of("adapt", shape), cb.last_plan()
    lp = oracle_target(target, d, data)
    worst = 0.0
    for c in (0, n_chains - 1):
        with np.errstate(all="ignore"):
            res = wo.WALNUTS(lp, q0[c], integrator=KIND[integrator], H0=H0, delta0=delta, numIter=n_iter, M=M, seed=seed,
                             chain=c, warmupIter=n_iter if warmup else 0, adaptH=warmup, adaptDelta=warmup,
                             recordOrbitStats=orbit)
        so, do = res[0], res[1]
        dgc = out["diag"][:, c]
        assert np.array_equal(dgc[:, EXACT_COLS], do[:, EXACT_COLS]), f"chain {c}: discrete diagnostics differ"
        assert int(out["nevalF"][c]) == int(do[:, 6].sum()) and int(out["nevalB"][c]) == int(do[:, 7].sum())
        # Warm-up adaptation feeds every transition's energy error back into delta and H (WALNUTS.py:701-712), and
        # the next orbits run with that H.  The energy error is a difference of energies summed over d coordinates
        # (and N rows for logreg), so its last bits depend on the summation order.  Measured on B200 (1000 W): diag_gauss
        # 3e-10 / 8e-10 / 3e-7 relative at d = 300 / 513 / 2049 after 12 adapted transitions, logreg 1.3e-9 at P = 7
        # after 14, every discrete column identical.  Without warm-up the 1e-10 bound holds.
        rtol = 1e-6 if warmup else 1e-10
        scale_ = (1.0 / np.sqrt(data["inv_var"])) if target == "diag_gauss" else None
        ok, err = close(out["draws"][:, c], so[:, 1:].T, rtol=rtol, scale=scale_)
        worst = max(worst, err)
        assert ok, f"chain {c}: draws differ, max rel err {err:.3e}"
        ok, err = close_diag(dgc[:, FLOAT_COLS], do[:, FLOAT_COLS], rtol=max(rtol, 1e-8))   # incl. adapted H, delta
        assert ok, f"chain {c}: float diagnostics differ {err:.3e}"
        if orbit:
            for a, b in ((out["orbit_min"][:, c], res[2].T), (out["orbit_max"][:, c], res[3].T)):
                ok, err = close(a, b, rtol=rtol, scale=scale_)
                assert ok, f"chain {c}: orbit statistics differ {err:.3e}"
        if target == "logreg":
            check_logreg_rows_hit(data, logreg_data(N or 257, d)[2], so.T)
    if warmup:
        assert not np.allclose(out["diag"][-1, :, 15], H0), "the adaptation did not move H"
    print(f"{target} d={d} {integrator} warmup={warmup} orbit={orbit}: plan adapt {shape}, "
          f"worst relative error {worst:.2e}")


def run_package(target, d, shape, n_iter, n_chains=3, N=None, macro_step=None, depth=4, max_error=0.3, seed=31):
    """Package mode, one transition at a time on identical inputs: a fresh ChainBatch(first_iteration = it + 1) from
    the oracle's previous state (chains 0 and n_chains - 1; the middle chain continues from its own state)."""
    from walnuts_b200 import ChainBatch
    q0, data, scale = problem(target, d, n_chains, N=N)
    logp, grad = pkg_lp(target, data)
    inv_mass = np.linspace(0.8, 1.25, d)
    h = macro_step or (2.0 * scale * d ** -0.25 if target in ("std_normal", "diag_gauss", "dense_gauss") else 0.3 * scale)
    checked = [0, n_chains - 1]
    prev = q0.copy()
    worst = 0.0
    states = [q0]
    for it in range(n_iter):
        with ChainBatch(target, d, n_chains, mode="package", H0=h, delta=max_error, M=depth, seed=seed,
                        first_iteration=it + 1, data=dict(data, inv_mass=inv_mass)) as cb:
            cb.set_state(prev)
            out = cb.run(1, draws=True)["draws"][0]
            assert cb.last_plan() == plan_of("pkg", shape), cb.last_plan()
        nxt = out.copy()
        for c in checked:
            with np.errstate(all="ignore"):
                ref = po.walnuts(seed, c, prev[c], logp, grad, inv_mass, h, depth, max_error, 0, 1,
                                 first_iteration=it + 1)[0]
            ok, err = close(out[c], ref)
            worst = max(worst, err)
            assert ok, f"transition {it}, chain {c}: max rel err {err:.3e}"
            nxt[c] = ref
        prev = nxt
        states.append(prev[checked])
    assert any(not np.array_equal(a, b) for a, b in zip(states[1:], states[:-1])), "no checked chain moved"
    if target == "logreg":
        check_logreg_rows_hit(data, logreg_data(N or 257, d)[2], np.concatenate([s.reshape(-1, d) for s in states]))
    print(f"{target} d={d} package: plan pkg {shape}, worst relative error per transition {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# the case table: (id, target, family, shape, runner); the id is the test id
# ---------------------------------------------------------------------------------------------------------------------
S = {"1x2": (1, 2, 128), "1x6": (1, 6, 128), "8x1": (8, 1, 128), "16x1": (16, 1, 128), "32x2": (32, 2, 128), "32x8": (32, 8, 128),
     "64x8": (64, 8, 64), "256x4": (256, 4, 256), "512x4": (512, 4, 512), "warp256": (32, 2, 256),
     "sw64": (64, 7, 64), "sw128": (128, 7, 128), "corr": (1, 1, 128)}
INT_FAMILY = {"fixed": "nuts", "D": "wpy", "R2P": "wpy", "Yoshida": "adapt", "Flow": "ext", "Midpoint": "ext",
              "Rescaled": "ext"}
CASES = []      # (id, target, family, shape, run)


def _wpy(target, d, integrator, shape, forced, n_iter, **kw):
    fam = INT_FAMILY[integrator]
    CASES.append((f"{target}-{fam}-{integrator}-d{d}" + (f"-N{kw['N']}" if "N" in kw else ""), target, fam, S[shape],
                  lambda: run_walnutspy(target, d, integrator, fam, S[shape], forced, n_iter, **kw)))


def _adapt(target, d, shape, warmup, orbit, n_iter, **kw):
    what = "warmup" * warmup + "-" * (warmup and orbit) + "orbit" * orbit
    CASES.append((f"{target}-adapt-{what}-d{d}", target, "adapt", S[shape],
                  lambda: run_adapt(target, d, S[shape], warmup, orbit, n_iter, **kw)))


def _pkg(target, d, shape, n_iter, **kw):
    CASES.append((f"{target}-pkg-d{d}", target, "pkg", S[shape], lambda: run_package(target, d, S[shape], n_iter, **kw)))


# logistic regression: LogRegCoopT (plain kernels, 104 < P <= 128) and the per-warp LogRegT (every other family)
for integ, P, N in (("D", 105, 257), ("R2P", 128, 1001), ("fixed", 105, 1001), ("fixed", 128, 257)):
    _wpy("logreg", P, integ, "warp256", False, 4, N=N)
for P, N in ((7, 257), (100, 1001), (128, 257)):
    _pkg("logreg", P, "warp256", 3, N=N)
_wpy("logreg", 100, "Yoshida", "warp256", False, 4, N=257)
_adapt("logreg", 7, "warp256", True, False, 14, N=1001)
_adapt("logreg", 128, "warp256", False, True, 4, N=257)
for integ in ("Flow", "Midpoint", "Rescaled"):
    for P, N in ((7, 1001), (100, 257)):
        _wpy("logreg", P, integ, "warp256", False, 3, N=N)

# Stock-Watson: 64 threads x 4 time steps up to T = 256, 128 threads (4 warps: cross-warp scans) up to T = 512
for T in (256, 257, 384, 512):
    for integ in ("fixed", "D", "R2P", "Yoshida"):
        _wpy("stock_watson", 3 * T, integ, "sw64" if T <= 256 else "sw128", True, 4, n_chains=2)
for T in (252, 300):
    _pkg("stock_watson", 3 * T, "sw64" if T <= 256 else "sw128", 3, macro_step=0.1)
    _wpy("stock_watson", 3 * T, "Flow", "sw64" if T <= 256 else "sw128", True, 3, n_chains=2)

# funnels: FunnelT on the warp shapes (fixed: the plain-NUTS level loop from d = 33), FunnelPkgT in package mode
for d, shape in ((17, "16x1"), (32, "16x1"), (33, "32x2"), (128, "32x2"), (129, "32x8"), (512, "32x8")):
    _wpy("funnel", d, "fixed", shape, True, 4, n_chains=2)
for integ, ds in (("R2P", (17, 128, 129)), ("Yoshida", (32, 33, 512)), ("Rescaled", (17, 128, 512))):
    for d in ds:
        _wpy("funnel", d, integ, {17: "16x1", 32: "16x1", 33: "32x2", 128: "32x2", 129: "32x8", 512: "32x8"}[d], True,
             4, n_chains=2)
for d, shape in ((13, "16x1"), (33, "32x2"), (129, "32x8"), (512, "32x8")):
    _pkg("funnel_pkg", d, shape, 4)

# large d: the generic 64 x 8, 256 x 4 and 512 x 4 shapes; std_normal is the UNIT instantiation of DiagGaussT
for d, shape in ((513, "64x8"), (1025, "256x4"), (2049, "512x4"), (4096, "512x4")):
    _pkg("std_normal", d, shape, 2)
for d, shape in ((300, "32x8"), (513, "64x8"), (2049, "512x4")):
    _adapt("diag_gauss", d, shape, False, True, 6)
    _adapt("diag_gauss", d, shape, True, False, 12)
for d, shape in ((600, "64x8"), (1500, "256x4"), (3000, "512x4")):
    for integ in ("fixed", "R2P"):
        _wpy("std_normal", d, integ, shape, False, 3)

# dense Gaussian: the per-warp DenseGaussT behind the general and extended kernels
for d in (12, 120):
    for integ in ("Yoshida", "Flow"):
        _wpy("dense_gauss", d, integ, "warp256", False, 6)


# the remaining (target, family, shape) combinations the dispatcher can select, at capacity or one past it: two chains,
# a few transitions each (teacher-forced for the funnels)
for integ, ds in (("Yoshida", ((1, "1x2"), (17, "16x1"), (129, "32x8"), (1024, "64x8"), (2048, "256x4"), (4096, "512x4"))),
                  ("Flow", ((512, "32x8"), (4096, "512x4"))), ("Midpoint", ((1024, "64x8"),)),
                  ("Rescaled", ((1025, "256x4"),))):
    for d, shape in ds:
        _wpy("std_normal", d, integ, shape, False, 3, n_chains=2)
for integ, ds in (("Yoshida", ((4, "1x2"), (16, "8x1"), (32, "16x1"), (128, "32x2"), (1025, "256x4"))),
                  ("Flow", ((13, "8x1"), (512, "32x8"))), ("Midpoint", ((17, "16x1"), (2048, "256x4"))),
                  ("Rescaled", ((1, "1x2"), (33, "32x2"), (2049, "512x4"))),
                  ("fixed", ((129, "32x8"), (1025, "256x4"), (4096, "512x4"))), ("R2P", ((2049, "512x4"),))):
    for d, shape in ds:
        _wpy("diag_gauss", d, integ, shape, False, 3, n_chains=2)
for d, shape in ((1, "1x2"), (12, "1x6"), (13, "16x1"), (128, "32x2"), (129, "32x8"), (1024, "64x8"), (2048, "256x4"),
                 (2049, "512x4")):
    _pkg("diag_gauss", d, shape, 2, n_chains=2)
for d, shape in ((12, "1x6"), (13, "16x1"), (128, "32x2"), (129, "32x8")):
    _pkg("funnel", d, shape, 3, n_chains=2)
for integ, ds in (("fixed", ((12, "1x6"), (32, "16x1"), (33, "32x2"), (512, "32x8"))),
                  ("R2P", ((16, "8x1"), (17, "16x1"), (128, "32x2"), (129, "32x8"))),
                  ("Yoshida", ((5, "8x1"), (32, "16x1"), (33, "32x2"), (512, "32x8"))),
                  ("Rescaled", ((16, "8x1"), (17, "16x1"), (128, "32x2"), (129, "32x8")))):
    for d, shape in ds:
        _wpy("funnel_pkg", d, integ, shape, True, 3, n_chains=2)
_pkg("corr_gauss", 2, "corr", 4, n_chains=2)


@pytest.mark.parametrize("case", [pytest.param(c, id=c[0]) for c in CASES])
def test_dispatched_kernel_parity(cuda_lib, case):
    case[4]()


# ---------------------------------------------------------------------------------------------------------------------
# completeness
# ---------------------------------------------------------------------------------------------------------------------
P = "tests/test_gpu_walnutspy_parity.py::"
E = "tests/test_gpu_ext_integrators.py::"
K = "tests/test_gpu_package_parity.py::"
# (target, family, G, E2, NT) -> an existing test that runs it against the oracle
ALREADY_COVERED = {
    **{("std_normal", f) + S[s]: P + "test_std_normal" for f in ("wpy", "nuts") for s in ("16x1", "32x2", "32x8")},
    ("std_normal", "wpy", 1, 2, 128): P + "test_std_normal", ("std_normal", "nuts", 1, 2, 128): P + "test_std_normal",
    ("std_normal", "wpy", 8, 1, 128): P + "test_std_normal", ("std_normal", "nuts", 1, 6, 128): P + "test_std_normal",
    ("std_normal", "adapt", 8, 1, 128): P + "test_yoshida_integrator",
    ("std_normal", "adapt", 32, 2, 128): P + "test_yoshida_integrator",
    ("std_normal", "ext", 1, 2, 128): E + "test_std_normal", ("std_normal", "ext", 8, 1, 128): E + "test_std_normal",
    ("std_normal", "ext", 16, 1, 128): E + "test_std_normal", ("std_normal", "ext", 32, 2, 128): E + "test_std_normal",
    ("std_normal", "pkg", 1, 2, 128): K + "test_package_golden",
    ("std_normal", "pkg", 1, 6, 128): K + "test_package_vs_oracle_many_chains",
    ("std_normal", "pkg", 16, 1, 128): K + "test_package_small_macro_step_ell_zero_defect_all_kernel_shapes",
    ("std_normal", "pkg", 32, 2, 128): K + "test_package_c1_d100",
    ("std_normal", "pkg", 32, 8, 128): K + "test_package_small_macro_step_ell_zero_defect_all_kernel_shapes",
    **{("diag_gauss", "wpy") + S[s]: P + "test_randomised_configurations"
       for s in ("8x1", "16x1", "32x2", "32x8", "256x4")},
    ("diag_gauss", "wpy", 1, 2, 128): P + "test_randomised_configurations",
    ("diag_gauss", "nuts", 1, 2, 128): P + "test_randomised_configurations",
    ("diag_gauss", "nuts", 1, 6, 128): P + "test_randomised_configurations",
    ("diag_gauss", "nuts", 16, 1, 128): P + "test_randomised_configurations",
    ("diag_gauss", "nuts", 32, 2, 128): P + "test_randomised_configurations",
    ("diag_gauss", "nuts", 32, 16, 64): P + "test_diag_gauss_1000",
    ("diag_gauss", "wpy", 128, 4, 128): P + "test_diag_gauss_1000",
    ("diag_gauss", "ext", 64, 8, 64): E + "test_diag_gauss_block_per_chain",
    ("funnel", "wpy", 8, 1, 128): P + "test_funnel10", ("funnel", "nuts", 8, 1, 128): P + "test_funnel10",
    ("funnel", "adapt", 8, 1, 128): P + "test_yoshida_integrator",
    ("funnel", "ext", 8, 1, 128): E + "test_funnel10_teacher_forced",
    ("funnel_pkg", "pkg", 1, 6, 128): K + "test_package_golden",
    ("logreg", "wpy", 32, 2, 256): P + "test_logreg", ("logreg", "nuts", 32, 2, 256): P + "test_logreg",
    ("stock_watson", "wpy", 64, 7, 64): P + "test_stock_watson",
    ("stock_watson", "nuts", 64, 7, 64): P + "test_stock_watson",
    ("dense_gauss", "wpy", 32, 2, 256): "tests/test_gpu_config_parity.py::test_dense_gauss_tensor_core_target",
    ("dense_gauss", "nuts", 32, 2, 256): "tests/test_gpu_config_parity.py::test_dense_gauss_tensor_core_target",
    ("dense_gauss", "pkg", 32, 2, 256): "tests/test_gpu_config_parity.py::test_dense_gauss_package_mode_and_moments",
    ("corr_gauss", "wpy", 1, 1, 128): P + "test_corr_gauss_minC",
    ("corr_gauss", "nuts", 1, 1, 128): P + "test_corr_gauss_minC",
    ("corr_gauss", "adapt", 1, 1, 128): P + "test_yoshida_integrator",
    ("corr_gauss", "ext", 1, 1, 128): E + "test_corr_gauss",
}
TRIGGERS = ["fixed", "D", "R2P", "Yoshida", "warmup", "orbit", "Flow", "Midpoint", "Rescaled", "package"]
GENERIC_DIMS = [1, 4, 5, 12, 13, 16, 17, 32, 33, 128, 129, 512, 513, 1024, 1025, 2048, 2049, 4096]
# the dimension boundaries of every target (funnels from d = 2, logreg / dense from the smallest tested size: the
# plans below them are the same), and dimensions with no kernel
DIMS = {"std_normal": GENERIC_DIMS, "diag_gauss": GENERIC_DIMS,
        "funnel": [2] + GENERIC_DIMS[1:12], "funnel_pkg": [2] + GENERIC_DIMS[1:12],
        "logreg": [5, 32, 33, 104, 105, 128], "dense_gauss": [7, 32, 33, 104, 105, 128],
        "stock_watson": [3 * 37, 3 * 256, 3 * 257, 3 * 512], "corr_gauss": [2]}
UNSUPPORTED = {"funnel": [513], "funnel_pkg": [513], "logreg": [129], "dense_gauss": [129],
               "stock_watson": [3 * 256 + 1, 3 * 513], "corr_gauss": [3]}
SHAPE_NAME = {v: k for k, v in S.items()}


def _case_keys():
    return {(c[1], c[2]) + tuple(c[3]) for c in CASES}


def _one_transition_plan(target, d, trigger):
    from walnuts_b200 import ChainBatch
    q0, data, scale = problem(target, d, 1, N=40)
    integ = {"warmup": "R2P", "orbit": "R2P", "package": "fixed"}.get(trigger, trigger)
    kw = dict(mode="package", data=dict(data, inv_mass=np.ones(d))) if trigger == "package" else \
        dict(integrator=integ, data=data)
    with ChainBatch(target, d, 1, H0=step_size(target, d, integ, scale), delta=0.3, M=3, seed=3, **kw) as cb:
        if trigger == "warmup":
            cb.set_adapt(5)
        cb.set_state(q0)
        cb.run(1, draws=True, orbit_stats=trigger == "orbit")
        return cb.last_plan()


def test_every_dispatched_plan_has_a_parity_test(cuda_lib):
    """Every plan the dispatcher picks for a built-in target has a parity test:
    a case of this file or an entry of ALREADY_COVERED naming an existing test; unsupported combinations fail
    cleanly with WN_EUNSUPPORTED."""
    import importlib
    from walnuts_b200 import ChainBatch, WalnutsError
    for test in set(ALREADY_COVERED.values()):          # the allow-list names tests that exist
        path, name = test.split("::")
        assert hasattr(importlib.import_module(path[:-3].replace("/", ".")), name), test
    seen = {}
    for target, dims in DIMS.items():
        for d in dims:
            for trigger in TRIGGERS:
                fam, G, E2, NT = _one_transition_plan(target, d, trigger)
                seen.setdefault((target, FAMILY_NAME[fam], G, E2, NT), []).append((d, trigger))
    covered = _case_keys() | set(ALREADY_COVERED)
    missing = {k: v for k, v in seen.items() if k not in covered}
    print(f"{len(seen)} plans dispatched, {len(seen) - len(missing)} covered")
    assert not missing, f"plans without a parity test: {missing}"
    assert not ((set(ALREADY_COVERED) | _case_keys()) - set(seen)), "stale entries"
    for target, dims in UNSUPPORTED.items():
        for d in dims:
            for mode in ("walnutspy", "package"):
                with pytest.raises(WalnutsError, match="WN_EUNSUPPORTED"):
                    ChainBatch(target, d, 1, mode=mode, integrator="R2P")
