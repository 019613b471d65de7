"""CUDA target registry: handles that replace the reference's Python target functions
(WALNUTSpy/targetDistr.py, test/targets.py).  A handle names a hand-written CUDA log-density +
gradient (walnuts_b200/csrc/wn_targets.cuh) and carries its data; it is passed where the reference
takes `lpFun` (WALNUTS.py:111) or `logp`/`grad` (walnuts.py:362).
"""
import hashlib
import os
import subprocess

import numpy as np


class Target:
    def __init__(self, name, data=None, d=None, ref="", plugin=None):
        self.name, self.data, self.d, self.ref = name, dict(data or {}), d, ref
        self.plugin = plugin          # path of a user-target plug-in library (cuda_target)

    def __repr__(self):
        return f"<walnuts_b200 target {self.name}{'' if self.d is None else ' d=%d' % self.d} ({self.ref})>"

    def __call__(self, *a, **k):
        raise TypeError(f"target {self.name!r} is a handle for a CUDA log density; it is evaluated "
                        "on the GPU inside walnuts_b200.WALNUTS/walnuts and cannot be called on host arrays")


# names as in the reference -------------------------------------------------------------------------
stdGauss = Target("std_normal", ref="targetDistr.py:18-21")
corrGauss = Target("corr_gauss", d=2, ref="targetDistr.py:25-31")
funnel10 = Target("funnel", d=11, ref="targetDistr.py:74-78")
standard_normal_lpdf = standard_normal_grad = Target("std_normal", ref="test/targets.py:4-7")
funnel_lpdf = funnel_grad = Target("funnel_pkg", ref="test/targets.py:23-29")


def funnel(n=10):
    """Neal's funnel with one log-scale and n conditionally normal coordinates (funnel10 for n=10)."""
    return Target("funnel", d=n + 1, ref="targetDistr.py:74-78")


def diag_gauss(sigma):
    """Zero-mean Gaussian with standard deviations `sigma` (SURVEY.md row T2; not in the reference)."""
    sigma = np.asarray(sigma, dtype=np.float64)
    return Target("diag_gauss", data={"inv_var": 1.0 / (sigma ** 2)}, d=sigma.size, ref="SURVEY.md T2")


def ill_conditioned_gauss(d=1000, lo=-2.0, hi=2.0):
    """BASELINE config 2: sigma = logspace(lo, hi, d)."""
    return diag_gauss(np.logspace(lo, hi, d))


def dense_gauss(precision):
    """Zero-mean Gaussian with a dense symmetric positive-definite PRECISION matrix [d, d], d <= 128 (north_star: the
    target whose gradient -P q is a dense contraction across lock-stepped chains; it runs on the FP64 tensor cores).
    Not in the reference."""
    P = np.ascontiguousarray(precision, dtype=np.float64)
    if P.ndim != 2 or P.shape[0] != P.shape[1]:
        raise ValueError("precision must be a square matrix")
    if not np.allclose(P, P.T, rtol=1e-12, atol=0.0):
        raise ValueError("precision must be symmetric")
    return Target("dense_gauss", data={"precision": P}, d=P.shape[0], ref="north_star (not in the reference)")


def stock_watson(y):
    """Stock-Watson stochastic-volatility model of the reference's example
    (WALNUTSpy_examples/StockWatson/sw_innov.stan:2-52, bridgestan default propto=True) on the
    unconstrained scale; `y` is the observed series (T values), d = 3T."""
    y = np.ascontiguousarray(y, dtype=np.float64)
    return Target("stock_watson", data={"y": y}, d=3 * y.size, ref="sw_innov.stan:2-52")


def logreg(X, y, tau=1.0):
    """Bayesian logistic regression (SURVEY.md row T4): Bernoulli-logit likelihood for rows of X [N, P]
    with responses y in {0, 1} and a N(0, tau^2 I) prior on the P coefficients."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    if X.ndim != 2 or y.shape != (X.shape[0],):
        raise ValueError("X must be [N, P] and y [N]")
    return Target("logreg", data={"X": X, "y": y, "tau": np.array([float(tau)])}, d=X.shape[1], ref="SURVEY.md T4")


# Parallel protocol plans (wn_user_plugin.cuh, UserParT): (largest d, threads per chain G, coordinate pairs per thread
# E2, threads per block NT) -- the shapes the built-in targets run on (wn_dispatch.cuh: pick_generic)
PARALLEL_PLANS = [(256, 32, 4, 128), (512, 32, 8, 128), (1024, 64, 8, 64), (2048, 256, 4, 256), (4096, 512, 4, 512)]
SMEM_MAX = 227 * 1024          # shared memory of one block on sm_100a
_CTL_BYTES = 504               # sizeof(wn::Ctl), the per-warp control block of walnutspy_kernel


def parallel_plan(d):
    """(G, E2, NT) of a parallel-protocol user target of dimension d."""
    for dmax, G, E2, NT in PARALLEL_PLANS:
        if d <= dmax:
            return G, E2, NT
    raise ValueError(f"cuda_target(parallel=True): 1 <= d <= {PARALLEL_PLANS[-1][0]}")


def parallel_smem_bytes(d, scratch):
    """Shared memory per block of a parallel user target's kernels in bytes: the larger of the WALNUTSpy (EXT) and
    package kernels, dynamic part plus static arrays, computed as the plug-in's static_assert computes it."""
    G, E2, NT = parallel_plan(d)
    r16 = lambda b: (b + 15) // 16 * 16
    w = NT // 32
    dyn = 3 * 2 * E2 * NT + 2 * ((G + 31) // 32) * 8 + (NT // G) * (2 * 2 * G * E2 + scratch)
    # the package kernel has the same dynamic part and a smaller static one (its control block is smaller, no table)
    return 8 * dyn + r16(4) + r16(_CTL_BYTES * w) + r16(4 * 32 * w)


def cuda_target(source, d, data=None, name="user", verbose=False, *, parallel=False, scratch=0):
    """A user-defined target: the role of the reference's arbitrary Python `lpFun` (WALNUTSpy/targetDistr.py:18) /
    `logp`, `grad` (walnuts/walnuts.py:296-297) callables and of walnuts_stan.py's compiled Stan model.

    Sequential protocol (parallel=False, 1 <= d <= 512): `source` is CUDA C++ defining the log density and its
    gradient over the whole coordinate vector:

        WN_TARGET_LP_GRAD(q, g, data, n_data) {
            // q[0..WN_D-1] in, g[0..WN_D-1] out; data[0..n_data-1] is the `data` array; return the log density
        }

    d <= 64 runs one thread per chain; 64 < d <= 512 one warp per chain -- leapfrog and tree logic parallel over the
    lanes, the user's function evaluated by every lane on the whole vector.

    Parallel protocol (parallel=True, 1 <= d <= 4096): every thread of the chain's group (32 threads for d <= 512, 64
    for d <= 1024, 256 for d <= 2048, 512 for d <= 4096) calls the function at once and computes its share:

        WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
            // q[0..WN_D-1]: the chain's position in shared memory, readable by every thread of the chain
            for (int j = ctx.rank; j < WN_D; j += ctx.size) g[j] = ...;   // the gradient entries this thread owns
            // ctx.sum(x): sum over the chain's threads (same value on every thread); ctx.sync(): barrier over them;
            // ctx.scratch: `scratch` doubles of per-chain shared memory
            return share;   // this thread's share of lp; the library adds the shares
        }

    Every thread of the chain must call ctx.sum and ctx.sync the same number of times in the same order (a call in a
    branch that differs between threads is undefined behaviour); indices j >= d are never handed out.  `scratch` is
    limited by the 227 KB of shared memory of a block (parallel_smem_bytes).  Defining the macro of the other protocol
    fails to compile with a message naming the right one.

    It is compiled once with nvcc for sm_100a into walnuts_b200/_lib/user/<hash>.so (cached by content), linked
    against the same persistent kernels as the built-in targets, and serves WALNUTS(...) with every integrator and the
    warm-up adaptation as well as walnuts(...) / walnuts_step(...)."""
    from . import build as _build
    d = int(d)
    scratch = int(scratch)
    if parallel:
        if not 1 <= d <= PARALLEL_PLANS[-1][0]:
            raise ValueError(f"cuda_target(parallel=True): 1 <= d <= {PARALLEL_PLANS[-1][0]} (one chain per warp up to "
                             "d = 512, per block of 64 / 256 / 512 threads up to d = 1024 / 2048 / 4096)")
        if scratch < 0:
            raise ValueError("cuda_target: scratch must be >= 0 doubles")
        need = parallel_smem_bytes(d, scratch)
        if need > SMEM_MAX:
            raise ValueError(f"cuda_target: scratch={scratch} needs {need} bytes of shared memory per block at d = {d}, "
                             f"more than the {SMEM_MAX} of a block")
    else:
        if scratch != 0:
            raise ValueError("cuda_target: scratch needs parallel=True")
        if not 1 <= d <= 512:
            raise ValueError("cuda_target: 1 <= d <= 512 (d <= 64: one thread per chain holds the whole vector; "
                             "64 < d <= 512: one warp per chain, the density evaluated by every lane on the whole vector)")
    csrc = os.path.join(_build.HERE, "csrc")
    head = f"#define WN_USER_D {d}\n"
    if parallel:
        head += f"#define WN_USER_PARALLEL 1\n#define WN_USER_SCRATCH {scratch}\n"
    tu = (f"{head}#include \"wn_user_api.cuh\"\n#line 1 \"{name}\"\n{source}\n"
          "#include \"wn_user_plugin.cuh\"\n")
    h = hashlib.sha256()
    h.update(tu.encode())
    for f in _build.HEADERS + [os.path.join(csrc, "wn_user_api.cuh"), os.path.join(csrc, "wn_user_plugin.cuh")]:
        with open(f, "rb") as fh:
            h.update(fh.read())
    out_dir = os.path.join(_build.LIB_DIR, "user")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"{name}_{h.hexdigest()[:16]}.so")
    if not os.path.isfile(so):
        # per-process scratch names + atomic rename: several ranks may build the same plug-in at once
        src = f"{so[:-3]}.{os.getpid()}.cu"
        tmp = f"{so}.{os.getpid()}.tmp"
        with open(src, "w") as fh:
            fh.write(tu)
        cmd = [os.environ.get("NVCC", "nvcc")] + _build.NVCC_FLAGS + ["-shared", "-I", csrc, "-o", tmp, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose:
            print(r.stderr)
        if r.returncode != 0:
            os.remove(src)
            raise RuntimeError("cuda_target: nvcc failed:\n" + r.stdout + r.stderr)
        os.replace(src, so[:-3] + ".cu")
        os.replace(tmp, so)
    dd = {} if data is None else {"data": np.ascontiguousarray(data, dtype=np.float64).ravel()}
    return Target(f"user:{name}", data=dd, d=d, ref="user CUDA source", plugin=so)


class _LazyCudaTarget(Target):
    """A cuda_target() whose plug-in is compiled on first use."""

    def __init__(self, name, d, source, ref):
        super().__init__(f"user:{name}", d=d, ref=ref)
        self._short, self.source = name, source

    def compile(self):
        if self.plugin is None:
            self.plugin = cuda_target(self.source, self.d, name=self._short).plugin
        return self


# The remaining targets of the reference, written as user targets (they double as examples of the protocol).
smileDistr = _LazyCudaTarget("smileDistr", 2, """
WN_TARGET_LP_GRAD(q, g, data, n_data) {                       // q0 ~ N(0,1), q1 | q0 ~ N(q0^2, 1)
  const double r = q[1] - q[0] * q[0];
  g[0] = -q[0] + 2.0 * q[0] * q[1] - 2.0 * q[0] * q[0] * q[0];
  g[1] = q[0] * q[0] - q[1];
  return -0.5 * q[0] * q[0] - 0.5 * r * r;
}""", "targetDistr.py:34-38")
rosenbrock_lpdf = rosenbrock_grad = _LazyCudaTarget("rosenbrock", 2, smileDistr.source, "test/targets.py:17-21")
modFunnel = _LazyCudaTarget("modFunnel", 2, """
WN_TARGET_LP_GRAD(q, g, data, n_data) {
  const double x = q[0], y = q[1];
  const double t1 = exp(-3.0 * x), t2 = 1.0 + t1, t3 = 1.0 / t2, t4 = y * y;
  g[0] = 1.5 * t1 * (t4 - t3) - x;
  g[1] = -y * t2;
  return -0.5 * (t2 * t4 + log(t3) + x * x);
}""", "targetDistr.py:41-51")
funnel1 = _LazyCudaTarget("funnel1", 2, """
WN_TARGET_LP_GRAD(q, g, data, n_data) {                       // q0 ~ N(0, 3^2), q1 | q0 ~ N(0, exp(q0))
  const double L2PI = 0.91893853320467274178, L3 = 1.09861228866810969140;
  const double ex = exp(-q[0]), a = q[0] / 3.0;
  g[0] = -0.5 - q[0] / 9.0 + 0.5 * q[1] * q[1] * ex;
  g[1] = -q[1] * ex;
  return (-(a * a) / 2.0 - L2PI - L3) + (-0.5 * ex * q[1] * q[1] - L2PI - 0.5 * q[0]);
}""", "targetDistr.py:88-92")
funnel10rescaled = _LazyCudaTarget("funnel10rescaled", 11, """
WN_TARGET_LP_GRAD(q, g, data, n_data) {                       // funnel10 evaluated at S q, S = diag(3, 1, ..., 1)
  const double L2PI = 0.91893853320467274178, L3 = 1.09861228866810969140;
  const double q0 = 3.0 * q[0], ex = exp(-q0), a = q0 / 3.0;
  double ss = 0.0;
  for (int i = 1; i < WN_D; ++i) ss += q[i] * q[i];
  for (int i = 1; i < WN_D; ++i) g[i] = -q[i] * ex;
  g[0] = 3.0 * (-5.0 - q0 / 9.0 + 0.5 * ex * ss);
  return (-(a * a) / 2.0 - L2PI - L3) + (-0.5 * ex * ss - 10.0 * L2PI - 10.0 * 0.5 * q0);
}""", "targetDistr.py:81-86")
correlated_normal_lpdf = correlated_normal_grad = _LazyCudaTarget("correlated_normal", 2, """
WN_TARGET_LP_GRAD(q, g, data, n_data) {
  // as written in the reference: the first gradient component is NOT the derivative of the density
  const double rho = 0.5, r = q[1] - rho * q[0];
  g[0] = -q[0] + rho * q[1];
  g[1] = (-q[1] + rho * q[0]) / (1.0 - rho * rho);
  return -0.5 * q[0] * q[0] - 0.5 / (1.0 - rho * rho) * r * r;
}""", "test/targets.py:9-15")


def resolve(target, d):
    """Target handle (or registry name) -> (name, data) after checking the dimension."""
    if isinstance(target, str):
        target = Target(target)
    if not isinstance(target, Target):
        raise TypeError(
            "walnuts_b200 runs CUDA targets only: pass a handle from walnuts_b200.targets (stdGauss, funnel10, "
            "diag_gauss(sigma), ...) or wrap your own density with walnuts_b200.targets.cuda_target(source, d) "
            "where the reference takes a Python log-density callable; Python callables have no GPU "
            "implementation and there is deliberately no CPU fallback")
    if target.d is not None and target.d != d:
        raise ValueError(f"target {target.name} has dimension {target.d}, state has {d}")
    if isinstance(target, _LazyCudaTarget):
        target.compile()
    if target.plugin is not None:
        from . import _ffi
        return _ffi.register_user_target(target.plugin), target.data
    return target.name, target.data
