"""Gaussian chains above d = 4096 on thread-block clusters (wn_walnutspy.cuh, G > NT).

std_normal and diag_gauss run one chain per cluster of 2, 4 or 8 CTAs of 512 threads (d <= 8192 / 16384 / 32768) in
every WALNUTSpy-mode family: D / R2P ("wpy"), fixedLeapFrog ("nuts"), Yoshida / warm-up adaptation / orbit statistics
("adapt") and Flow / Midpoint / Rescaled ("ext").  Every case asserts the plan it ran on (ChainBatch.last_plan) and
compares against an oracle: the C oracle for fixed / D / R2P (any d), the numpy oracle for the other families.  Draws
are held to 1e-10 relative to each coordinate's sigma and the discrete diagnostics exactly.  Sizes are each cluster
shape's capacity and one past it (the last thread then holds padding lanes).

Cross-CTA paths get their own cases: the stiffest coordinate (which decides the step-size search and, through one
thread's energy partial, the failure-certificate vote) and a coordinate beyond the lazy-energy magnitude bound sit in
the LAST CTA of the cluster, so a vote or reduction that stayed inside rank 0 would change the discrete diagnostics.
"""
import numpy as np
import pytest

from oracle import c_oracle
from oracle import walnutspy_oracle as wo
from tests.helpers import KIND, close, close_diag, oracle_target, oracle_walnutspy
from tests.test_gpu_config_parity import _bonferroni_z
from tests.test_gpu_dispatch_coverage import FAMILY_NAME, TRIGGERS, UNSUPPORTED, _one_transition_plan
from tests.test_gpu_walnutspy_parity import EXACT_COLS, FLOAT_COLS
from walnuts_b200._ffi import FAMILIES

pytestmark = pytest.mark.gpu

NT = 512
SIZES = [4097, 8192, 8193, 16384, 16385, 32768]
C_COLS = [0, 1, 6, 7, 19]          # the columns test_d4096_single_cta_chain holds exactly against the C oracle
INT_FAMILY = {"fixed": "nuts", "D": "wpy", "R2P": "wpy", "Yoshida": "adapt", "Flow": "ext", "Midpoint": "ext",
              "Rescaled": "ext"}
DELTA = {"Yoshida": 0.05, "Flow": 0.02, "Midpoint": 0.05, "Rescaled": 0.3}
COVERED = set()                    # (target, family, G, E2, NT) run by a case of this file


def cluster_of(d):
    return 2 if d <= 8192 else (4 if d <= 16384 else 8)


def plan_for(family, d):
    return (FAMILIES[family], cluster_of(d) * NT, 4, NT)


def cover(target, family, d):
    COVERED.add((target, family) + plan_for(family, d)[1:])


def step(integrator, d, scale=1.0):
    """The reference's Gaussian scalings (mainGaussESS.py): H = 1.4 d^-1/4 for the adaptive integrators, d^-1/2 for
    fixedLeapFrog."""
    return scale * (d ** -0.5 if integrator == "fixed" else 1.4 * d ** -0.25)


def diag_problem(d, n, seed=8):
    rng = np.random.default_rng(seed)
    sigma = np.exp(rng.uniform(-1.0, 1.0, d))
    return rng.standard_normal((n, d)) * sigma, sigma


def run(target, q0, integrator, H0, M, n_iter, seed, sigma=None, delta=0.3, dg=None, plan=None, warmup=0,
        orbit=False):
    from walnuts_b200 import ChainBatch
    n, d = q0.shape
    data = {"inv_var": 1.0 / sigma ** 2} if target == "diag_gauss" else {}
    with ChainBatch(target, d, n, integrator=integrator, H0=H0, delta=delta, M=M, seed=seed, data=data, dg=dg) as cb:
        if warmup:
            cb.set_adapt(warmup)
        cb.set_state(q0)
        out = cb.run(n_iter, draws=True, diag=True, orbit_stats=orbit)
        out["state"] = cb.get_state()
        out["plan"], out["slots"] = cb.last_plan(), cb.last_slots()
    if plan is not None:
        assert out["plan"] == plan, f"ran on plan {out['plan']}, expected {plan}"
    return out


def against_c_oracle(target, out, q0, integrator, H0, M, n_iter, seed, chains, sigma=None, delta=0.3):
    """Draws of `chains` within 1e-10 of sigma, C_COLS and the evaluation counts exact; returns the worst error."""
    iv = None if sigma is None else 1.0 / sigma ** 2
    worst = 0.0
    for c in chains:
        dr, dg, _ = c_oracle.run_chain(target, integrator, q0[c], H0, delta, M, n_iter, seed, c, inv_var=iv)
        ok, err = close(out["draws"][:, c], dr, scale=sigma if sigma is not None else 1.0)
        worst = max(worst, err)
        assert ok, f"chain {c}: draws differ, max rel err {err:.3e}"
        assert np.array_equal(out["diag"][:, c][:, C_COLS], dg[:, C_COLS]), f"chain {c}: discrete diagnostics differ"
        assert int(out["nevalF"][c]) == int(dg[:, 6].sum()) and int(out["nevalB"][c]) == int(dg[:, 7].sum())
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# 1. free-running parity with the C oracle: fixed / D / R2P
# ---------------------------------------------------------------------------------------------------------------------
C_CASES = [("diag_gauss", d, integ) for d in SIZES for integ in ("fixed", "D", "R2P")] + \
          [("std_normal", d, integ) for d in (8192, 16384, 32768) for integ in ("fixed", "D", "R2P")]
for _t, _d, _i in C_CASES:
    cover(_t, INT_FAMILY[_i], _d)


@pytest.mark.parametrize("target,d,integrator", C_CASES)
def test_free_running_vs_c_oracle(cuda_lib, target, d, integrator):
    n_iter, M, seed = (6, 6, 11)
    if target == "diag_gauss":
        q0, sigma = diag_problem(d, 3, seed=d)
        H0 = step(integrator, d, sigma.min())
    else:
        q0, sigma = np.random.default_rng(d).standard_normal((3, d)), None
        H0 = step(integrator, d)
    out = run(target, q0, integrator, H0, M, n_iter, seed, sigma, plan=plan_for(INT_FAMILY[integrator], d))
    worst = against_c_oracle(target, out, q0, integrator, H0, M, n_iter, seed, [0, 2], sigma)
    print(f"{target} d={d} {integrator}: plan {out['plan']}, worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 2. the general ("adapt") and extended ("ext") kernels against the numpy oracle, one size per cluster shape
# ---------------------------------------------------------------------------------------------------------------------
ADAPT_CASES = [("Yoshida", 8192, "diag_gauss"), ("Yoshida", 16384, "std_normal"), ("Yoshida", 32768, "diag_gauss"),
               ("orbit", 8193, "diag_gauss"), ("orbit", 8192, "std_normal"), ("orbit", 32768, "std_normal"),
               ("warmup", 4097, "diag_gauss"), ("warmup", 16384, "diag_gauss"), ("warmup", 32768, "std_normal"),
               ("warmup-fixed", 8192, "std_normal"), ("warmup-fixed", 32768, "diag_gauss"),
               ("Flow", 8192, "std_normal"), ("Flow", 16385, "diag_gauss"), ("Flow", 32768, "diag_gauss"),
               ("Midpoint", 8193, "diag_gauss"), ("Midpoint", 16384, "std_normal"), ("Midpoint", 32768, "diag_gauss"),
               ("Rescaled", 4097, "diag_gauss"), ("Rescaled", 16384, "diag_gauss"), ("Rescaled", 32768, "std_normal")]
for _k, _d, _t in ADAPT_CASES:
    cover(_t, "adapt" if _k in ("Yoshida", "orbit", "warmup", "warmup-fixed") else "ext", _d)


@pytest.mark.parametrize("kind,d,target", ADAPT_CASES)
def test_general_and_extended_kernels_vs_numpy_oracle(cuda_lib, kind, d, target):
    integ = {"orbit": "R2P", "warmup": "R2P", "warmup-fixed": "fixed"}.get(kind, kind)
    warmup, orbit = kind.startswith("warmup"), kind == "orbit"
    # warm-up: 12 adapted transitions, so that the delta update of iterations 11 and 12 takes the quantile of the
    # adaptation-history row (WALNUTS.py:705-707), which thread 0 of rank 0 rewrites and every CTA reads
    n_iter = 12 if warmup else 2
    M, seed, delta = 5, 77, DELTA.get(integ, 0.3)
    if target == "diag_gauss":
        q0, sigma = diag_problem(d, 2, seed=d)
    else:
        q0, sigma = np.random.default_rng(d).standard_normal((2, d)), None
    scale = 1.0 if sigma is None else sigma.min()
    # fixedLeapFrog warm-up starts from the reference's default H0 = 0.2 (scaled), not from d^-1/2: at d^-1/2 the energy
    # error of an orbit is near the rounding level of energies of size d / 2, and adaptH turns it into the next step
    # size through |dH|^(-1/3) -- measured 2.9e-6 (d = 8192) and 2.9e-3 (d = 32768) relative in the draws against the
    # oracle, with every discrete column identical, i.e. summation order, not a different path
    H0 = 0.2 * scale if kind == "warmup-fixed" else step(integ, d, scale)
    family = "adapt" if kind in ("Yoshida", "orbit") or warmup else "ext"
    out = run(target, q0, integ, H0, M, n_iter, seed, sigma, delta=delta, plan=plan_for(family, d),
              warmup=n_iter if warmup else 0, orbit=orbit)
    data = {"inv_var": 1.0 / sigma ** 2} if sigma is not None else None
    lp = oracle_target(target, d, data)
    # Warm-up adaptation feeds each transition's energy error -- a sum over d coordinates whose last bits depend on
    # the summation order -- back into H and delta; the bound of test_gpu_dispatch_coverage.py (1e-6, discrete
    # columns exact) applies.  Without warm-up the 1e-10 bound holds.
    rtol = 1e-6 if warmup else 1e-10
    worst = 0.0
    for c in (0, 1):
        with np.errstate(all="ignore"):
            res = wo.WALNUTS(lp, q0[c], integrator=KIND[integ], H0=H0, delta0=delta, numIter=n_iter, M=M, seed=seed,
                             chain=c, warmupIter=n_iter if warmup else 0, adaptH=warmup, adaptDelta=warmup,
                             recordOrbitStats=orbit)
        so, do = res[0], res[1]
        dgc = out["diag"][:, c]
        assert np.array_equal(dgc[:, EXACT_COLS], do[:, EXACT_COLS]), f"chain {c}: discrete diagnostics differ"
        assert int(out["nevalF"][c]) == int(do[:, 6].sum()) and int(out["nevalB"][c]) == int(do[:, 7].sum())
        ok, err = close(out["draws"][:, c], so[:, 1:].T, rtol=rtol, scale=sigma)
        worst = max(worst, err)
        assert ok, f"chain {c}: draws differ, max rel err {err:.3e}"
        ok, err = close_diag(dgc[:, FLOAT_COLS], do[:, FLOAT_COLS], rtol=max(rtol, 1e-8))
        assert ok, f"chain {c}: float diagnostics differ {err:.3e}"
        if orbit:
            for a, b in ((out["orbit_min"][:, c], res[2].T), (out["orbit_max"][:, c], res[3].T)):
                ok, err = close(a, b, rtol=rtol, scale=sigma)
                worst = max(worst, err)
                assert ok, f"chain {c}: orbit statistics differ {err:.3e}"
    if warmup:
        assert not np.allclose(out["diag"][-1, :, 15], H0), "the adaptation did not move H"
        assert not np.allclose(out["diag"][-1, :, 18], delta), "the quantile update did not move delta"
    print(f"{target} d={d} {kind}: plan {out['plan']}, worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. cross-CTA votes and reductions: the decisive coordinate in the LAST CTA of the cluster
# ---------------------------------------------------------------------------------------------------------------------
def last_cta_coordinate(d):
    """A coordinate owned by cluster rank CL - 1: thread t = (CL - 1) NT + 3 holds coordinates 2 t, 2 t + 1 (pair 0)."""
    return 2 * ((cluster_of(d) - 1) * NT + 3)


@pytest.mark.parametrize("d", [8192, 16384, 32768])
@pytest.mark.parametrize("integrator", ["D", "R2P"])
def test_stiffest_coordinate_in_last_cta(cuda_lib, d, integrator):
    """Unit variances except ONE coordinate of the last CTA with sigma = 0.02: its thread's energy partial alone
    decides every failed step-size attempt (the pass-end failure-certificate vote) and dominates the energy error."""
    sigma = np.ones(d)
    j = last_cta_coordinate(d)
    sigma[j] = 0.02
    q0 = np.random.default_rng(3).standard_normal((3, d)) * sigma
    H0 = step(integrator, d)
    n_iter, M, seed = 6, 6, 5
    out = run("diag_gauss", q0, integrator, H0, M, n_iter, seed, sigma, plan=plan_for("wpy", d))
    worst = against_c_oracle("diag_gauss", out, q0, integrator, H0, M, n_iter, seed, [0, 1, 2], sigma)
    # the stiff coordinate really drives the search: the accepted step size is well below H0
    assert (out["diag"][:, :, 8] > 0).any(), "no step-size halving happened"
    print(f"diag_gauss d={d} {integrator}, stiff coordinate {j}: worst relative error {worst:.2e}")


@pytest.mark.parametrize("d", [8192, 32768])
@pytest.mark.parametrize("integrator", ["D", "R2P"])
def test_magnitude_bound_tripped_in_last_cta(cuda_lib, d, integrator):
    """One chain has a coordinate of the last CTA at 1e150, beyond the lazy-energy magnitude bound (2^300): only that
    thread sees it, and its flag must reach every CTA so that all of them re-run the pass with per-step energies
    (test_forced_reject_non_finite_energy covers the same path inside one CTA).  The draws are compared on each
    coordinate's own magnitude: the 1e150 coordinate carries rounding of order 1e134 in any implementation."""
    sigma = np.exp(np.linspace(-1.0, 1.0, d))
    data = {"inv_var": 1.0 / sigma ** 2}
    q0 = np.random.default_rng(4).standard_normal((2, d)) * sigma
    q0[1, last_cta_coordinate(d)] = 1e150
    H0, M, n_iter, seed = 2.0, 5, 3, 1234
    out = run("diag_gauss", q0, integrator, H0, M, n_iter, seed, sigma, plan=plan_for("wpy", d))
    draws_o, diag_o = oracle_walnutspy("diag_gauss", q0, integrator, H0, 0.3, M, n_iter, seed, [0, 1], 0, 10, data)
    ok, err = close(out["draws"], draws_o)
    assert ok, f"draws differ: max rel err {err:.3e}"
    assert np.array_equal(out["diag"][..., EXACT_COLS], diag_o[..., EXACT_COLS]), "discrete diagnostics differ"
    assert np.array_equal(out["nevalF"], diag_o[..., 6].sum(axis=0).astype(np.uint64))
    assert np.array_equal(out["nevalB"], diag_o[..., 7].sum(axis=0).astype(np.uint64))
    print(f"diag_gauss d={d} {integrator}, 1e150 in the last CTA: worst relative error {err:.2e}, stop codes "
          f"{np.unique(diag_o[:, 1, 19])}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. more chains than resident clusters
# ---------------------------------------------------------------------------------------------------------------------
def test_more_chains_than_resident_clusters(cuda_lib):
    from walnuts_b200 import ChainBatch
    d, integ, M, seed = 16384, "R2P", 6, 21
    H0 = step(integ, d)
    probe = np.random.default_rng(0).standard_normal((512, d))
    with ChainBatch("std_normal", d, 512, integrator=integ, H0=H0, delta=0.3, M=M, seed=seed, dg=1) as cb:
        cb.set_state(probe)
        cb.run(1, draws=False)
        slots = cb.last_slots()
        assert cb.last_plan() == plan_for("wpy", d)
    assert 1 <= slots < 512
    n = slots + 5
    q0 = np.random.default_rng(1).standard_normal((n, d))
    out = run("std_normal", q0, integ, H0, M, 4, seed, plan=plan_for("wpy", d))
    assert out["slots"] == slots
    worst = against_c_oracle("std_normal", out, q0, integ, H0, M, 4, seed, [0, slots - 1, slots, n - 1])
    # chain c does not depend on how many chains share the launch, nor on which cluster served it
    few = run("std_normal", q0[:3], integ, H0, M, 4, seed, plan=plan_for("wpy", d))
    assert np.array_equal(few["draws"], out["draws"][:, :3]) and np.array_equal(few["diag"], out["diag"][:, :3])
    # a continuation (two calls of 2) equals one call of 4
    with ChainBatch("std_normal", d, n, integrator=integ, H0=H0, delta=0.3, M=M, seed=seed) as cb:
        cb.set_state(q0)
        a = cb.run(2, draws=True, diag=True)
        b = cb.run(2, draws=True, diag=True)
        assert cb.last_plan() == plan_for("wpy", d)
        state = cb.get_state()
    assert np.array_equal(np.concatenate([a["draws"], b["draws"]]), out["draws"])
    assert np.array_equal(np.concatenate([a["diag"], b["diag"]]), out["diag"])
    assert np.array_equal(state, out["state"])
    print(f"std_normal d={d}: {slots} resident clusters, {n} chains, worst relative error {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# 5. drop-in surface and statistics
# ---------------------------------------------------------------------------------------------------------------------
def test_walnuts_drop_in_default_adaptation_d8192(cuda_lib):
    """WALNUTS(targets.stdGauss, q0) at d = 8192 with the reference's defaults (fixedLeapFrog, H0 = 0.2, delta0 = 0.05,
    M = 10, adaptH and adaptDelta with their targets), the warm-up shortened to 12 iterations -- enough for the delta
    quantile of iterations 11 and 12 -- and 14 iterations in all, checked against the numpy oracle for chains 0 and 2."""
    import walnuts_b200 as wb
    d, n = 8192, 3
    q0 = np.random.default_rng(6).standard_normal((n, d))
    s, dg = wb.WALNUTS(wb.targets.stdGauss, q0, numIter=14, warmupIter=12, seed=5)
    assert s.shape == (n, d, 15) and dg.shape == (n, 14, 24) and np.isfinite(s).all()
    assert not np.allclose(dg[:, 11, 18], 0.05), "the quantile update did not move delta"
    # the same call's plan: the general kernels of the 2-CTA cluster during warm-up
    from walnuts_b200 import ChainBatch
    with ChainBatch("std_normal", d, n, integrator="fixed", H0=0.2, delta=0.05, M=10, seed=5) as cb:
        cb.set_adapt(12)
        cb.set_state(q0)
        cb.run(1, draws=False)
        assert cb.last_plan() == plan_for("adapt", d)
    worst = 0.0
    for c in (0, 2):
        with np.errstate(all="ignore"):
            so, do = wo.WALNUTS(oracle_target("std_normal", d), q0[c], integrator=wo.FIXED, H0=0.2, delta0=0.05,
                                numIter=14, M=10, seed=5, chain=c, warmupIter=12, adaptH=True, adaptDelta=True)
        assert np.array_equal(dg[c][:, EXACT_COLS], do[:, EXACT_COLS]), f"chain {c}"
        # adapted run (see test_general_and_extended_kernels_...); s[c] is (d, numIter + 1): coordinates on axis 0
        ok, err = close(s[c], so, rtol=1e-6, axis=0)
        worst = max(worst, err)
        assert ok, f"chain {c}: {err:.3e}"
    print(f"WALNUTS(stdGauss) d={d}: worst relative error {worst:.2e}")


def test_long_run_moments_d16384(cuda_lib):
    """Chains started from exact draws of N(0, I) at d = 16384 stay distributed as N(0, I) after 20 R2P transitions:
    the cross-chain mean and variance of every coordinate -- including the first coordinates of each of the 4 CTAs'
    slices, so that a chain whose CTAs drifted apart fails -- within the family-wise 3-MCSE bound of
    test_c2_long_run_100_transitions_moments.  The leading coordinate is also recorded per draw (dg = 1)."""
    from walnuts_b200 import ChainBatch
    d, n, n_iter = 16384, 400, 20
    q0 = np.random.default_rng(12).standard_normal((n, d))
    with ChainBatch("std_normal", d, n, integrator="R2P", H0=step("R2P", d), delta=0.3, M=10, seed=8, dg=1) as cb:
        cb.set_state(q0)
        out = cb.run(n_iter, draws=True)
        assert cb.last_plan() == plan_for("wpy", d)
        z = cb.get_state()
    assert np.array_equal(out["draws"][-1, :, 0], z[:, 0])
    assert np.isfinite(z).all()
    firsts = [r * 2 * NT for r in range(4)]                       # pair 0 of thread 0 of each rank
    zb = _bonferroni_z(2 * d)
    zm = np.abs(z.mean(0)) * np.sqrt(n)
    zv = np.abs(z.var(0, ddof=1) - 1.0) / np.sqrt(2.0 / (n - 1))
    print(f"d={d}: worst mean deviation {zm.max():.2f} SE, worst variance deviation {zv.max():.2f} SE "
          f"(CTA slice starts {zm[firsts].max():.2f} / {zv[firsts].max():.2f}); family-wise bound {zb:.2f} SE")
    assert zm.max() < zb and zv.max() < zb
    corr = np.mean(z * q0, axis=0)
    assert np.abs(corr).mean() < 0.5, "the chains did not move"


# ---------------------------------------------------------------------------------------------------------------------
# 6. refusals and 7. completeness of this file for the new range
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals(cuda_lib):
    import walnuts_b200 as wb
    from walnuts_b200 import WalnutsError
    for target in ("std_normal", "diag_gauss"):
        for trigger in TRIGGERS:
            with pytest.raises(WalnutsError, match="WN_EUNSUPPORTED"):
                _one_transition_plan(target, 32769, trigger)
        with pytest.raises(WalnutsError, match="WN_EUNSUPPORTED"):
            _one_transition_plan(target, 4097, "package")
    for target, dims in UNSUPPORTED.items():
        for d in dims:
            for trigger in ("R2P", "package"):
                with pytest.raises(WalnutsError, match="WN_EUNSUPPORTED"):
                    _one_transition_plan(target, d, trigger)
    with pytest.raises(ValueError):
        wb.targets.cuda_target("WN_TARGET_LP_GRAD(q, g, data, n_data) { return 0.0; }", 513)


def test_every_cluster_plan_has_a_case(cuda_lib):
    """Every plan with G > NT the dispatcher picks for the two Gaussian targets in the new range is run by a case of
    this file."""
    seen = {}
    for target in ("std_normal", "diag_gauss"):
        for d in SIZES:
            for trigger in TRIGGERS:
                if trigger == "package":
                    continue                                      # refused above d = 4096 (test_refusals)
                fam, G, E2, NTB = _one_transition_plan(target, d, trigger)
                assert G > NTB, (target, d, trigger, G, NTB)
                seen.setdefault((target, FAMILY_NAME[fam], G, E2, NTB), []).append((d, trigger))
    missing = {k: v for k, v in seen.items() if k not in COVERED}
    print(f"{len(seen)} cluster plans dispatched, {len(seen) - len(missing)} covered")
    assert not missing, f"cluster plans without a case: {missing}"
