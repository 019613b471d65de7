"""Load the REAL reference (a checkout named by $WALNUTS_REFERENCE, or the copy staged in oracle/_ref) and run it
under an injected RNG.

TEST / BASELINE INFRASTRUCTURE ONLY; used by tests/golden/make_golden.py to generate the committed fixtures and by
`bench.py --impl reference` (the CPU arm) through the copy staged in oracle/_ref by oracle/stage_ref.py.  The product
(walnuts_b200/) never imports it.

Recipe: SURVEY.md appendix C.  The package `walnuts/__init__.py` imports bridgestan (absent),
so walnuts/walnuts.py is loaded by path; WALNUTSpy/WALNUTS.py imports an unused matplotlib,
so stub modules are pre-inserted.
"""
import contextlib
import importlib.util
import os
import sys
import types

import numpy as np

from . import philox

def _ref_root():
    """$WALNUTS_REFERENCE (a checkout of bob-carpenter/walnuts), else the copy staged by oracle/stage_ref.py
    (oracle/_ref)."""
    return os.environ.get("WALNUTS_REFERENCE") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


REF_ROOT = _ref_root()


def available():
    return os.path.isfile(os.path.join(REF_ROOT, "WALNUTSpy", "WALNUTS.py"))


_cache = {}


def load_walnutspy():
    """Returns (WALNUTS module, adaptiveIntegrators module, targetDistr module)."""
    if "wpy" not in _cache:
        sys.dont_write_bytecode = True
        for name in ("matplotlib", "matplotlib.pyplot"):
            sys.modules.setdefault(name, types.ModuleType(name))
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        p = os.path.join(REF_ROOT, "WALNUTSpy")
        if p not in sys.path:
            sys.path.insert(0, p)
        import WALNUTS as wn                      # noqa: E402
        import adaptiveIntegrators as ai          # noqa: E402
        import targetDistr as td                  # noqa: E402
        _cache["wpy"] = (wn, ai, td)
    return _cache["wpy"]


def load_package():
    """Returns the walnuts/walnuts.py module (tqdm progress bar silenced)."""
    if "pkg" not in _cache:
        sys.dont_write_bytecode = True
        spec = importlib.util.spec_from_file_location(
            "walnuts_ref_pkg", os.path.join(REF_ROOT, "walnuts", "walnuts.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.trange = lambda n, **kw: range(n)
        _cache["pkg"] = mod
    return _cache["pkg"]


def load_test_targets():
    if "tt" not in _cache:
        spec = importlib.util.spec_from_file_location(
            "walnuts_ref_test_targets", os.path.join(REF_ROOT, "test", "targets.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _cache["tt"] = mod
    return _cache["tt"]


@contextlib.contextmanager
def philox_numpy_random(seed, chain, M, first_iteration=1):
    """Patch numpy.random.uniform / numpy.random.normal so that WALNUTS.py and
    adaptiveIntegrators.py draw from the Philox streams of oracle/philox.py.

    Dispatch by call shape (SURVEY.md row A13): `uniform(low=0,high=2,size=M)` is the direction
    block and opens a new iteration; `normal(size=d)` is the momentum block; every other uniform
    call walks the sequential scalar stream."""
    streams = philox.ChainStreams(seed, chain)
    state = {"it": first_iteration - 1}
    old_u, old_n = np.random.uniform, np.random.normal

    def uniform(low=0.0, high=1.0, size=None):
        if size is not None and np.ndim(size) == 0 and int(size) == M and low == 0.0 and high == 2.0:
            state["it"] += 1
            streams.begin_iteration(state["it"])
            return 2.0 * streams.directions(M)
        if size is None:
            return low + (high - low) * streams.uniform()
        return np.array([low + (high - low) * streams.uniform() for _ in range(int(size))])

    def normal(loc=0.0, scale=1.0, size=None):
        assert size is not None
        return loc + scale * streams.momentum(int(size))

    np.random.uniform, np.random.normal = uniform, normal
    try:
        yield streams
    finally:
        np.random.uniform, np.random.normal = old_u, old_n


def run_walnutspy(lpFun, q0, integrator_name, H0, delta0, numIter, M, minC=0, maxC=10,
                  seed=0, chain=0, stepSizeRandScale=0.2, use_philox=True, np_seed=None,
                  generated=None, warmupIter=0, recordOrbitStats=False, first_iteration=1):
    """Run the real WALNUTS.WALNUTS; adaptation off (fixed H, delta) unless warmupIter > 0, which switches on the
    reference's default warm-up adaptation (adaptH, adaptDelta with their default targets, WALNUTS.py:111-129)."""
    wn, ai, _ = load_walnutspy()
    integrator = getattr(ai, integrator_name)
    aux = ai.integratorAuxPar(minC=minC, maxC=maxC)
    kw = dict(q0=np.array(q0, dtype=np.float64), integrator=integrator, H0=H0,
              stepSizeRandScale=stepSizeRandScale, delta0=delta0, numIter=numIter, warmupIter=warmupIter,
              M=M, igrAux=aux, adaptH=warmupIter > 0, adaptDelta=warmupIter > 0)
    if generated is not None:
        kw["generated"] = generated
    if recordOrbitStats:
        kw["recordOrbitStats"] = True      # returns (samples, diagnostics, orbitMin, orbitMax), WALNUTS.py:724-725
    with np.errstate(all="ignore"), contextlib.redirect_stdout(open(os.devnull, "w")):
        if use_philox:
            with philox_numpy_random(seed, chain, M, first_iteration):
                return wn.WALNUTS(lpFun, **kw)
        np.random.seed(np_seed)
        return wn.WALNUTS(lpFun, **kw)
