"""Shared helpers for the parity tests (test infrastructure; may import oracle/)."""
import numpy as np

from oracle import targets as otargets
from oracle import walnutspy_oracle as wo

RTOL = 1e-10   # north_star: per-iteration draws match in fp64 to 1e-10 relative error


def close(a, b, rtol=RTOL, scale=None, axis=-1):
    """TRUE relative agreement, coordinate by coordinate: |a - b| <= rtol * scale_j.

    `axis` is the coordinate axis.  scale=None: scale_j = the largest |b| of coordinate j over all other axes
    (iterations, chains) -- the coordinate's own magnitude, a stand-in for its standard deviation, so that a
    small-sigma coordinate is held to 1e-10 of ITS size (the round-1 harness used max(1, |b|), an absolute
    tolerance for everything below 1) while a value that happens to pass through zero is not held to an impossible
    standard.  Pass `scale` (broadcastable, e.g. sigma) to fix the scales.  Coordinates that are identically zero
    get a floor of 1e-6 of the overall magnitude.  Returns (ok, worst relative error)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if scale is None:
        with np.errstate(invalid="ignore"):
            fin = np.where(np.isfinite(b), np.abs(b), 0.0)
        if b.ndim >= 2:
            ax = axis % b.ndim
            scale = fin.max(axis=tuple(i for i in range(b.ndim) if i != ax), keepdims=True)
            scale = np.maximum(scale, 1e-6 * fin.max()) if fin.size else scale
        else:
            scale = fin.max() if fin.size else 1.0
    scale = np.maximum(np.asarray(scale, dtype=np.float64), 1e-300)
    with np.errstate(invalid="ignore", over="ignore"):
        err = np.abs(a - b) / scale
        same = (np.isnan(a) & np.isnan(b)) | (a == b)
        bad = ~((err <= rtol) | same)
        worst = np.nanmax(np.where(same, 0.0, err)) if a.size else 0.0
    return not bad.any(), float(worst)


def close_diag(a, b, rtol=1e-9):
    """Floating-point diagnostics columns (orbit lengths, log-weights, energy spreads, index statistics): differences
    of O(H) quantities, compared on the scale max(1, |b|) element by element."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return close(a, b, rtol, scale=np.maximum(1.0, np.where(np.isfinite(b), np.abs(b), 1.0)))


def oracle_target(name, d, data=None):
    if name == "std_normal":
        return otargets.std_normal
    if name == "diag_gauss":
        return otargets.make_diag_gauss(1.0 / np.sqrt(data["inv_var"]))
    if name == "funnel":
        return otargets.funnel10
    if name == "corr_gauss":
        return otargets.corr_gauss
    if name == "funnel_pkg":       # the package-mode funnel density under the WALNUTSpy lpFun protocol
        return lambda q, hessian=False: [otargets.funnel_lpdf(q), otargets.funnel_grad(q)]
    if name == "logreg":
        return otargets.make_logreg(data["X"], data["y"], float(np.asarray(data.get("tau", 1.0)).ravel()[0]))
    if name == "dense_gauss":
        return otargets.make_dense_gauss(data["precision"])
    if name == "stock_watson":
        return otargets.make_stock_watson(data["y"])
    raise KeyError(name)


KIND = {"fixed": wo.FIXED, "D": wo.ADAPT_D, "R2P": wo.ADAPT_R2P, "Yoshida": wo.ADAPT_YOSHIDA,
        "Flow": wo.ADAPT_FLOW, "Midpoint": wo.ADAPT_MIDPOINT, "Rescaled": wo.ADAPT_RESCALED}


def oracle_walnutspy(name, q0, integrator, H0, delta, M, n_iter, seed, chains, minC=0, maxC=10, data=None,
                     jitter=0.2, first_iteration=1, lp=None):
    """Run the numpy oracle for the listed chain ids; returns draws (n_iter, len(chains), d), diag."""
    q0 = np.asarray(q0, dtype=np.float64)
    d = q0.shape[-1]
    lp = lp or oracle_target(name, d, data)
    draws = np.empty((n_iter, len(chains), d))
    diag = np.empty((n_iter, len(chains), 24))
    for k, c in enumerate(chains):
        with np.errstate(all="ignore"):
            s, dg = wo.WALNUTS(lp, q0[c] if q0.ndim == 2 else q0, integrator=KIND[integrator], H0=H0,
                               stepSizeRandScale=jitter, delta0=delta, numIter=n_iter, M=M,
                               igrAux=wo.AuxPar(minC, maxC), seed=seed, chain=c,
                               first_iteration=first_iteration)
        draws[:, k, :] = s[:, 1:].T
        diag[:, k, :] = dg
    return draws, diag
