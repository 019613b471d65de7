"""GPU parity of the remaining integrators of adaptiveIntegrators.py (SURVEY.md section 8f, row N3):
adaptLeapFrogFlowD (:246-356), adaptImplicitMidpointD (:478-641, fixed-point variant) and
adaptRescaledLeapFrogD (:660-762), through the C-ABI, against the numpy oracle -- which is bit-identical to
the live reference for these integrators (tests/golden/wpy_*_{Flow,Midpoint,Rescaled}.npz, CPU suite) -- on
the same Philox streams: draws to 1e-10, discrete diagnostics exactly."""
import numpy as np
import pytest

from tests.helpers import close
from tests.test_gpu_walnutspy_parity import check, check_forced, q0_for

pytestmark = pytest.mark.gpu

EXT = ["Flow", "Midpoint", "Rescaled"]
DELTA = {"Flow": 0.02, "Midpoint": 0.05, "Rescaled": 0.3}


@pytest.mark.parametrize("integrator", EXT)
@pytest.mark.parametrize("d", [1, 7, 20, 100])
def test_std_normal(cuda_lib, integrator, d):
    """Group sizes G = 1, 4, 16, 32 (thread, sub-warp and warp per chain)."""
    dg = check("std_normal", q0_for(4, d), integrator, H0=1.3 * d ** -0.25, delta=DELTA[integrator], M=7,
               n_iter=40 if d <= 20 else 15)
    if integrator == "Flow":
        assert (dg[..., 6] % 2 == 0).all()          # two gradient evaluations per micro-step (:262,:266)
    if integrator != "Midpoint":                      # (the implicit midpoint rule conserves quadratic energies: If = 0)
        assert dg[..., 9].max() >= 1                  # the step-size search was exercised


@pytest.mark.parametrize("integrator", EXT)
def test_corr_gauss(cuda_lib, integrator):
    check("corr_gauss", np.tile(np.array([1.0, 0.0]), (4, 1)), integrator, H0=0.9, delta=DELTA[integrator], M=8,
          n_iter=60, minC=1)                           # these integrators ignore minC (their search starts at c = 0)


@pytest.mark.parametrize("integrator", EXT)
def test_diag_gauss_block_per_chain(cuda_lib, integrator):
    """d = 1000 ill-conditioned Gaussian (BASELINE config 2 shape): the ext plan there is 64 threads per chain with 8
    coordinate pairs each, one chain per 64-thread CTA (64 x 8, NT = 64)."""
    d = 1000
    sigma = np.logspace(-2, 2, d)
    data = {"inv_var": 1.0 / sigma ** 2}
    check("diag_gauss", q0_for(3, d) * sigma, integrator, H0=0.02, delta=DELTA[integrator], M=4, n_iter=2, maxC=6,
          data=data)


@pytest.mark.parametrize("integrator", EXT)
def test_funnel10_teacher_forced(cuda_lib, integrator):
    rng = np.random.default_rng(3)
    q0 = np.empty((4, 11))
    q0[:, 0] = 1.5 * rng.standard_normal(4)
    q0[:, 1:] = np.exp(0.5 * q0[:, :1]) * rng.standard_normal((4, 10))
    dg, worst = check_forced("funnel", q0, integrator, H0=0.4, delta=DELTA[integrator], M=8, n_iter=40)
    assert worst < 1e-10


def test_midpoint_not_converged_is_a_forced_reject(cuda_lib):
    """With maxC = 0 and a large step the fixed-point iteration of the only attempt diverges: the reference ends
    the process (sys.exit, adaptiveIntegrators.py:548-550); the kernel and the oracle report stop code 999 and
    leave the chain where it was."""
    q0 = q0_for(3, 5)
    dg = check("std_normal", q0, "Midpoint", H0=4.0, delta=0.05, M=5, n_iter=6, maxC=0)
    assert (dg[..., 19] == 999).any()


def test_aux_parameters_reach_the_kernel(cuda_lib):
    """integratorAuxPar(maxFPiter, FPtol, rescaledGradThresh) through WALNUTS(...)."""
    import walnuts_b200 as wb
    from oracle import targets as ot
    from oracle import walnutspy_oracle as wo
    q0 = q0_for(2, 6)
    for ig, kind, kw in ((wb.adaptImplicitMidpointD, wo.ADAPT_MIDPOINT, dict(maxFPiter=12, FPtol=1e-6)),
                         (wb.adaptRescaledLeapFrogD, wo.ADAPT_RESCALED, dict(rescaledGradThresh=0.8))):
        s, d = wb.WALNUTS(wb.targets.stdGauss, q0, integrator=ig, H0=0.8, delta0=0.2, numIter=30, warmupIter=0, M=6,
                          igrAux=wb.integratorAuxPar(**kw), adaptH=False, adaptDelta=False, seed=9)
        for c in range(2):
            with np.errstate(all="ignore"):
                so, do = wo.WALNUTS(ot.std_normal, q0[c], integrator=kind, H0=0.8, delta0=0.2, numIter=30, M=6,
                                    igrAux=wo.AuxPar(**kw), seed=9, chain=c)
            ok, err = close(s[c], so, axis=-2)
            assert ok, err
            assert np.array_equal(d[c][:, [1, 6, 7, 8, 9, 19]], do[:, [1, 6, 7, 8, 9, 19]])


@pytest.mark.parametrize("integrator", ["Flow", "Rescaled"])
def test_default_adaptation(cuda_lib, integrator):
    """The reference's default call (adaptH, adaptDelta on) with the extended integrators: igrConst of the last
    forward pass feeds the P-squared quantile (:294; adaptRescaledLeapFrogD reports the constant 1, :761)."""
    import walnuts_b200 as wb
    from oracle import targets as ot
    from oracle import walnutspy_oracle as wo
    ig = {"Flow": (wb.adaptLeapFrogFlowD, wo.ADAPT_FLOW), "Rescaled": (wb.adaptRescaledLeapFrogD, wo.ADAPT_RESCALED)}
    q0 = 0.5 * np.random.default_rng(2).standard_normal((3, 6))
    s, d = wb.WALNUTS(wb.targets.stdGauss, q0, integrator=ig[integrator][0], numIter=80, warmupIter=50, M=7, seed=3)
    for c in range(3):
        with np.errstate(all="ignore"):
            so, do = wo.WALNUTS(ot.std_normal, q0[c], integrator=ig[integrator][1], numIter=80, warmupIter=50, M=7,
                                seed=3, chain=c, adaptH=True, adaptDelta=True)
        ok, err = close(s[c], so, rtol=1e-8, axis=-2)
        assert ok, err
        ok, err = close(d[c][:, [15, 18]], do[:, [15, 18]], rtol=1e-8)
        assert ok, err
        assert np.array_equal(d[c][:, [1, 6, 7, 19]], do[:, [1, 6, 7, 19]])
