"""CPU restatement of the WALNUTSpy transition kernel.  TEST INFRASTRUCTURE ONLY.

Restates reference WALNUTSpy/WALNUTS.py:111-727 (driver) and
WALNUTSpy/adaptiveIntegrators.py:49-137,361-475 (fixedLeapFrog, adaptLeapFrogD,
adaptLeapFrogR2P) in the streaming form the CUDA kernels use:

  * the post-order sub-U-turn plan (WALNUTS.py:22-41) is derived from the leaf counter
    (after even leaf n: one check per s>=1 with n % 2**s == 0, span [n-2**s+1, n]);
  * only the left-end (q, v) of each pending dyadic level is kept (WALNUTS.py:48-88 keeps
    both ends of every finished subtree; only the left ends are ever read, :575-587);
  * running min/max replace the 2**M arrays Hs/Ifs/Ibs/cs/lwts (WALNUTS.py:170-174).

Pinned against the reference itself: tests/test_oracle_golden.py requires bit-identical samples and diagnostics
against tests/golden/*.npz, outputs of the real WALNUTS.py under the same RNG (tests/golden/make_golden.py).

All reference quirks of SURVEY.md row A14 are reproduced (cited inline).
"""
import math

import numpy as np

LOG_ZERO = -700.0                       # constants.py:13
WT_SUM_THRESH = float(np.exp(LOG_ZERO + 1.0))   # constants.py:14

FIXED, ADAPT_D, ADAPT_R2P, ADAPT_YOSHIDA = 0, 1, 2, 3
ADAPT_FLOW, ADAPT_MIDPOINT, ADAPT_RESCALED = 4, 5, 6   # adaptiveIntegrators.py:246-356, :478-641, :660-762
Y_FIRSTLAST = 1.351207191959658       # adaptiveIntegrators.py:143-144
Y_MIDDLE = -1.702414383919315


class AuxPar:
    """adaptiveIntegrators.integratorAuxPar (adaptiveIntegrators.py:36-44), hot-path fields."""

    def __init__(self, minC=0, maxC=10, R2Pprob0=2.0 / 3.0, maxFPiter=30, FPtol=1.0e-8, rescaledGradThresh=5.0):
        self.minC, self.maxC, self.R2Pprob0 = minC, maxC, R2Pprob0
        self.maxFPiter, self.FPtol, self.rescaledGradThresh = maxFPiter, FPtol, rescaledGradThresh


def _pysum(x):
    # the reference uses the Python builtin sum() (strict left-to-right) for sum(v*v) and the
    # U-turn dots (WALNUTS.py:97,256; adaptiveIntegrators.py:55,84)
    return sum(x)


def stop_condition(qm, vm, qp, vp):
    """WALNUTS.py:95-97."""
    tmp = qp - qm
    return bool(_pysum(vp * tmp) < 0.0 or _pysum(vm * tmp) < 0.0)


def _pass(q, vv, g, h, c, lpFun, track, yoshida=False):
    """2**c leapfrog micro-steps of total length h (adaptiveIntegrators.py:70-84); with `yoshida` each
    micro-step is the 4th-order triple of leapfrogs of adaptYoshidaD (:156-175).
    Returns (q, vv, g, f, H_last, all_finite, max|diff H|, hh, n_evals)."""
    nstep = 2 ** c
    hh = h / nstep
    Hprev = track
    ok = True
    maxd = 0.0
    f = None
    for _ in range(nstep):
        if yoshida:
            for cf in (Y_FIRSTLAST, Y_MIDDLE, Y_FIRSTLAST):
                vh = vv + 0.5 * cf * hh * g
                q = q + cf * hh * vh
                f, g = lpFun(q)
                vv = vh + 0.5 * cf * hh * g
        else:
            vh = vv + 0.5 * hh * g
            q = q + hh * vh
            f, g = lpFun(q)
            vv = vh + 0.5 * hh * g
        Hk = -f + 0.5 * _pysum(vv * vv)
        ok = ok and bool(np.isfinite(Hk))
        dd = abs(Hk - Hprev)
        maxd = dd if (dd > maxd or dd != dd) else maxd
        Hprev = Hk
    return q, vv, g, f, Hprev, ok, maxd, hh


def _pymax(a, b):
    # Python builtin max(a, b): b only if b > a (a NaN in `a` sticks, a NaN in `b` is dropped)
    return b if b > a else a


def _flow_pass(q, vv, g, h, c, lpFun, H0):
    """One attempt of adaptLeapFrogFlowD (adaptiveIntegrators.py:252-287 / :309-339): 2**c leapfrog
    micro-steps, each followed by a midpoint gradient and the 4 flow-error norms.
    Returns (q, vv, g, f, H_last, all_finite, maxErr, max|diff H|, hh)."""
    nstep = 2 ** c
    hh = h / nstep
    Hprev = H0
    ok = True
    maxd = 0.0
    maxErr = None
    f = None
    for _ in range(nstep):
        vh = vv + 0.5 * hh * g
        qold, gold, vold = q, g, vv
        q = q + hh * vh
        f, g = lpFun(q)
        vv = vh + 0.5 * hh * g
        qMid = 0.5 * (q + qold) + (hh / 8.0) * (vold - vv)
        _, gMid = lpFun(qMid)
        qf = qold + hh * vold + hh * hh * ((1.0 / 6.0) * gold + (1.0 / 3.0) * gMid)
        err = np.max(np.abs(qf - q))
        vf = vold + (hh / 6.0) * (gold + g + 4.0 * gMid)
        err = _pymax(err, np.max(np.abs(vf - vv)))
        qb = q - hh * vv + hh * hh * ((1.0 / 6.0) * g + (1.0 / 3.0) * gMid)
        err = _pymax(err, np.max(np.abs(qb - qold)))
        vb = -(-vv + (hh / 6.0) * (gold + g + 4.0 * gMid))
        err = _pymax(err, np.max(np.abs(vb - vold)))
        # np.max(Errs) (:282,337) propagates NaN
        maxErr = err if maxErr is None or (err > maxErr or err != err) else maxErr
        Hk = -f + 0.5 * _pysum(vv * vv)
        ok = ok and bool(np.isfinite(Hk))
        dd = abs(Hk - Hprev)
        maxd = dd if (dd > maxd or dd != dd) else maxd
        Hprev = Hk
    return q, vv, g, f, Hprev, ok, maxErr, maxd, hh


def _macro_flow(q, v, g, Ham0, h, xi, lpFun, delta, aux):
    """adaptLeapFrogFlowD, adaptiveIntegrators.py:246-356 (the search starts at c = 0, not minC)."""
    vv0 = xi * v
    nF = 0
    If = aux.maxC
    for c in range(0, aux.maxC + 1):                # :250-287
        qq, vv, gg, f, Hl, ok, maxErr, maxd, hh = _flow_pass(q, vv0, g, h, c, lpFun, Ham0)
        nF += 2 * 2 ** c
        if ok and maxErr < delta:
            If = c
            break
    with np.errstate(all="ignore"):
        igr = hh * (maxd ** (-1.0 / 3.0)) if maxd > 0 else np.inf      # :294
    Ib = If
    nB = 0
    for c in range(0, If):                          # :300-345
        _, _, _, _, _, okb, maxErrb, _, _ = _flow_pass(qq, -vv, gg, h, c, lpFun, Hl)
        nB += 2 * 2 ** c
        if okb and maxErrb < delta:
            Ib = c
            break
    return dict(q=qq, v=xi * vv, grad=gg, H=Hl, nF=nF, nB=nB, If=If, Ib=Ib, c=If, lwt=(If != Ib) * LOG_ZERO,
                igrConst=igr)


def _midpoint_pass(q, vv, g, h, c, lpFun, H0, aux):
    """One attempt of adaptImplicitMidpointD with fixed-point iterations (FPNewton=False),
    adaptiveIntegrators.py:483-541 / :572-626.  Returns (q, vv, g, f, H_last, all_finite, completed,
    converged_last, max|diff Hams|, hh, n_evals); Hams of steps that were not completed are 0 (:490)."""
    nstep = 2 ** c
    hh = h / nstep
    Hams = np.zeros(nstep + 1)
    Hams[0] = H0
    nev = 0
    f = None
    completed = 0
    converged = False
    for i in range(1, nstep + 1):
        qt = q + hh * (vv + 0.5 * hh * g)            # :494
        converged = False
        oldMaxErr = 1.0e100
        for _ in range(aux.maxFPiter):               # :500-523
            mpq = 0.5 * (qt + q)
            _, gmp = lpFun(mpq)
            qtNew = q + hh * vv + (0.5 * hh * hh) * gmp
            nev += 1
            maxErr = np.max(np.abs(qtNew - qt))
            qt = qtNew
            if maxErr < aux.FPtol:
                converged = True
                break
            if maxErr > 1.1 * oldMaxErr:
                break
            oldMaxErr = maxErr
        if not converged:                            # :525-527
            break
        mpq = 0.5 * (qt + q)                         # :530-540
        _, gmp = lpFun(mpq)
        nev += 1
        q = q + hh * vv + (0.5 * hh * hh) * gmp
        vv = vv + hh * gmp
        f, g = lpFun(q)
        nev += 1
        Hams[i] = -f + 0.5 * _pysum(vv * vv)
        completed += 1
    ok = bool(np.all(np.isfinite(Hams)))
    with np.errstate(all="ignore"):
        maxd = float(np.max(np.abs(np.diff(Hams))))
    return q, vv, g, f, float(Hams[-1]), ok, completed == nstep, converged, maxd, hh, nev


def _macro_midpoint(q, v, g, Ham0, h, xi, lpFun, delta, aux):
    """adaptImplicitMidpointD, adaptiveIntegrators.py:478-641, fixed-point variant.  The reference ends the
    PROCESS (`sys.exit()`, :548-550) when the last attempt (c = maxC) holds a step whose fixed-point iteration
    did not converge; here that macro step reports a NaN energy, which the driver turns into a forced reject
    (stop code 999) -- the same convention as the CUDA kernel (DESIGN.md section 5, deviations)."""
    vv0 = xi * v
    nF = 0
    If = aux.maxC
    for c in range(0, aux.maxC + 1):                # :482-545
        qq, vv, gg, f, Hl, ok, full, conv, maxd, hh, nev = _midpoint_pass(q, vv0, g, h, c, lpFun, Ham0, aux)
        nF += nev
        if ok and abs(Ham0 - Hl) < delta and full:
            If = c
            break
    if not conv:                                    # :548-550 (sys.exit in the reference)
        return dict(q=qq, v=xi * vv, grad=gg, H=float("nan"), nF=nF, nB=0, If=If, Ib=If, c=If, lwt=0.0,
                    igrConst=float("nan"))
    with np.errstate(all="ignore"):
        igr = hh * (maxd ** (-1.0 / 3.0)) if maxd > 0 else np.inf      # :561
    HO = -f + 0.5 * _pysum(vv * vv)                 # :569 (same expression as Hams[-1])
    Ib = aux.maxC                                   # :564
    nB = 0
    for c in range(0, aux.maxC + 1):                # :570-633: the FULL range, not only c < If
        _, _, _, _, Hb, okb, fullb, _, _, _, nev = _midpoint_pass(qq, -vv, gg, h, c, lpFun, HO, aux)
        nB += nev
        if okb and abs(HO - Hb) < delta and fullb:
            Ib = c
            break
    return dict(q=qq, v=xi * vv, grad=gg, H=HO, nF=nF, nB=nB, If=If, Ib=Ib, c=If, lwt=(If != Ib) * LOG_ZERO,
                igrConst=igr)


def _rescaled_attempt(q, vv, g, h, Sd, lpFun):
    """One leapfrog step in coordinates rescaled by Sd, adaptiveIntegrators.py:672-682 / :723-733."""
    qb = q / Sd
    gb = Sd * g
    vh = vv + 0.5 * h * gb
    qbn = qb + h * vh
    q1 = qbn * Sd
    ff, gnew = lpFun(q1)
    gb1 = Sd * gnew
    v1 = vh + 0.5 * h * gb1
    gbmean = 0.5 * (np.abs(gb) + np.abs(gb1))
    Ham1 = -ff + 0.5 * _pysum(v1 * v1)
    return q1, v1, ff, gnew, gbmean, Ham1


def _macro_rescaled(q, v, g, Ham0, h, xi, lpFun, delta, aux):
    """adaptRescaledLeapFrogD, adaptiveIntegrators.py:660-762 (its debugging prints at :720-721 are not
    reproduced)."""
    d = q.size
    thr = aux.rescaledGradThresh
    Sd = np.ones(d)
    Sred = np.zeros(d, dtype=np.int64)
    vv = xi * v
    If = aux.maxC
    nF = nB = 0
    for c in range(0, aux.maxC + 1):                # :669-700
        q1, v1, ff, gnew, gbmean, Ham1 = _rescaled_attempt(q, vv, g, h, Sd, lpFun)
        nF += 1
        big = gbmean > thr
        if not np.isfinite(Ham1):
            Sred += 1
        elif np.any(big):
            Sred[big] += 1
        elif abs(Ham0 - Ham1) > delta:
            Sred += 1
        else:
            If = c
            break
        Sd = 2.0 ** (-Sred)
    qO, vO, gO, HO = q1, v1, gnew, Ham1
    SredForw = Sred
    Sd = np.ones(d)
    Sred = np.zeros(d, dtype=np.int64)
    Ib = If
    if If > 0:                                      # :718-755
        for c in range(0, aux.maxC + 1):
            _, _, _, _, gbmean, Ham1 = _rescaled_attempt(qO, -vO, gO, h, Sd, lpFun)
            nB += 1
            big = gbmean > thr
            if not np.isfinite(Ham1):
                Sred += 1
            elif np.any(big):
                Sred[big] += 1
            elif abs(HO - Ham1) > delta:
                Sred += 1
            else:
                Ib = c
                break
            if np.all(SredForw == Sred):
                Ib = c + 1
                break
            Sd = 2.0 ** (-Sred)
    lwt = LOG_ZERO * (not np.all(Sred == SredForw))     # :762
    return dict(q=qO, v=xi * vO, grad=gO, H=HO, nF=nF, nB=nB, If=If, Ib=Ib, c=If, lwt=lwt, igrConst=1.0)


def macro_step(kind, q, v, g, Ham0, h, xi, lpFun, delta, aux, rng):
    """One macro step.  Returns dict(q, v, grad, H, nF, nB, If, Ib, c, lwt, igrConst).
    `v` is in forward-time convention in and out (adaptiveIntegrators.py:73,135)."""
    if kind == ADAPT_FLOW:
        return _macro_flow(q, v, g, Ham0, h, xi, lpFun, delta, aux)
    if kind == ADAPT_MIDPOINT:
        return _macro_midpoint(q, v, g, Ham0, h, xi, lpFun, delta, aux)
    if kind == ADAPT_RESCALED:
        return _macro_rescaled(q, v, g, Ham0, h, xi, lpFun, delta, aux)
    vv0 = xi * v
    if kind == FIXED:                               # adaptiveIntegrators.py:49-59
        vh = vv0 + 0.5 * h * g
        qq = q + h * vh
        f, gn = lpFun(qq)
        vv = vh + 0.5 * h * gn
        H1 = -f + 0.5 * _pysum(vv * vv)
        with np.errstate(all="ignore"):
            igr = h * (max(1.0e-10, abs(Ham0 - H1)) ** (-1.0 / 3.0))
        return dict(q=qq, v=xi * vv, grad=gn, H=H1, nF=1, nB=0, If=0, Ib=0, c=0, lwt=0.0, igrConst=igr)

    minC, maxC = aux.minC, aux.maxC
    yo = kind == ADAPT_YOSHIDA                      # adaptYoshidaD :142-240 = adaptLeapFrogD with Yoshida steps
    ev = 3 if yo else 1
    nF = 0
    If = maxC
    for c in range(minC, maxC + 1):                 # :69-94 / :365-389
        qq, vv, gg, f, Hl, ok, maxd, hh = _pass(q, vv0, g, h, c, lpFun, Ham0, yo)
        nF += ev * 2 ** c
        if ok and abs(Ham0 - Hl) < delta:
            If = c
            break
    cSim = If
    lwtf = 0.0
    if kind == ADAPT_R2P:
        if rng.uniform() < aux.R2Pprob0:            # :392
            lwtf = math.log(aux.R2Pprob0)
        else:                                       # :400-424 redo at If+1
            cSim = If + 1
            qq, vv, gg, f, Hl, ok, maxd, hh = _pass(q, vv0, g, h, cSim, lpFun, Ham0)
            nF += 2 ** cSim
            lwtf = math.log(1.0 - aux.R2Pprob0)
    qO, vO, gO, HO = qq, vv, gg, Hl
    with np.errstate(all="ignore"):
        igr = hh * (maxd ** (-1.0 / 3.0)) if maxd > 0 else np.inf   # :101,399,424

    if kind in (ADAPT_D, ADAPT_YOSHIDA) or cSim == If:   # :104-132 / :430-433
        maxTry, Ib = If - 1, If
    else:                                           # :434-437
        maxTry, Ib = maxC, maxC
    nB = 0
    for c in range(minC, maxTry + 1):               # :111-132 / :444-464
        _, _, _, _, Hb, okb, _, _ = _pass(qO, -vO, gO, h, c, lpFun, HO, yo)
        nB += ev * 2 ** c
        if okb and abs(HO - Hb) < delta:
            Ib = c
            break
    if kind in (ADAPT_D, ADAPT_YOSHIDA):
        lwt = (If != Ib) * LOG_ZERO                 # :136, :239
    else:                                           # :467-475
        lwtb = LOG_ZERO
        if cSim == Ib:
            lwtb = math.log(aux.R2Pprob0)
        elif cSim == Ib + 1:
            lwtb = math.log(1.0 - aux.R2Pprob0)
        lwt = lwtb - lwtf
    return dict(q=qO, v=xi * vO, grad=gO, H=HO, nF=nF, nB=nB, If=If, Ib=Ib, c=cSim, lwt=lwt, igrConst=igr)


def transition(lpFun, qc, rng, kind, H, delta, M, aux, jitter=0.2, igr_sink=None, orbit=None, compat=True):
    """One WALNUTSpy iteration (WALNUTS.py:196-693).  Returns (q_next, diag[24])."""
    d = qc.size
    B = np.floor(rng.dir_uniform02(M)).astype(int)                      # :216
    v = rng.normal(d)                                                   # :236
    f0, g0 = lpFun(qc)                                                  # :249
    H0 = -f0 + 0.5 * _pysum(v ** 2)                                     # :256
    # ends: index 0 = plus (forward) end, 1 = minus (backward) end
    end_q = [qc, qc]
    end_v = [v, v]
    end_g = [g0, g0]
    end_H = [H0, H0]
    lwtSum = [0.0, 0.0]                 # [f, b]
    timeLen = [0.0, 0.0]                # [F, B]
    maxInt = [0, 0]                     # maxFint, maxBint
    WoldSum = 1.0
    qProp = qc
    L_ = 0
    indexStat = 0.0
    orbitLen = orbitLenSam = 0.0
    nF = nB = 0
    NdS = NdC = 0
    stopCode = 0
    bothEndsPassive = False
    # running statistics over used steps (WALNUTS.py:660-692)
    st = dict(n=0, minIf=None, maxIf=None, minl=None, maxl=None, minc=None, maxc=None,
              nne=0, nz=0, Hmax=H0, Hmin=H0, Hnan=False)
    lo = H * (1 - jitter)
    hi = H * (1 + jitter)
    if orbit is not None:               # recordOrbitStats, WALNUTS.py:274-276
        orbit["min"] = np.array(qc, dtype=np.float64)
        orbit["max"] = np.array(qc, dtype=np.float64)

    def record(o):
        st["n"] += 1
        for k, val in (("If", o["If"]), ("l", o["lwt"]), ("c", o["c"])):
            st["min" + k] = val if st["min" + k] is None else min(st["min" + k], val)
            st["max" + k] = val if st["max" + k] is None else max(st["max" + k], val)
        st["nne"] += int(o["If"] != o["Ib"])
        st["nz"] += int(o["If"] == 0)
        if o["H"] != o["H"]:
            st["Hnan"] = True
        else:
            st["Hmax"] = max(st["Hmax"], o["H"])
            st["Hmin"] = min(st["Hmin"], o["H"])

    forced = False
    for i in range(M):                                                  # :281
        side = int(B[i])                # 0 forward, 1 backward
        xi = 1 - 2 * side
        n_new = 2 ** i
        qPropLast, Lold, indexStatOld = qProp, L_, indexStat
        WnewSum = 0.0
        expand = True
        left = {}                       # level -> (q, v) left ends of pending dyadic spans
        hpair = None
        for n in range(1, n_new + 1):
            if i == 0:
                h = float(rng.uniform_range(lo, hi, 1)[0])              # :298
                orbitLen += h                                           # :300
            elif n % 2 == 1:
                hpair = rng.uniform_range(lo, hi, 2)                    # :395
                h = float(hpair[0])
            else:
                h = float(hpair[1])
            o = macro_step(kind, end_q[side], end_v[side], end_g[side], end_H[side], h, xi,
                           lpFun, delta, aux, rng)
            end_q[side], end_v[side], end_g[side], end_H[side] = o["q"], o["v"], o["grad"], o["H"]
            nF += o["nF"]
            nB += o["nB"]
            if igr_sink is not None:
                igr_sink(o["igrConst"])                                 # :313 (warm-up only)
            idx = maxInt[side] + xi if i > 0 else xi
            maxInt[side] = idx
            if i == 0:
                timeLen[side] = h                                       # :315,349
            else:
                timeLen[side] += h                                      # :413,456,500,543
            record(o)
            if not np.isfinite(o["H"]):                                 # :316,350,414,457,501,544
                forced = True
                if i == 0 or n % 2 == 1:
                    stopCode = 999      # quirk A14(ii): second leaf of a pair leaves stopCode as is
                break
            if i == 0:
                lwtSum[side] = o["lwt"]                                 # :321,354
            elif not compat or not (side == 1 and n % 2 == 0):
                lwtSum[side] += o["lwt"]    # quirk A14(i): :420 has no counterpart after :443-459
            Wnew = float(np.exp(-o["H"] + H0 + lwtSum[side]))           # :322,355,422,462,510,552
            if orbit is not None:       # :331-333,364-366,434-436,474-476,521-523,564-566
                orbit["min"] = np.minimum(orbit["min"], o["q"])
                orbit["max"] = np.maximum(orbit["max"], o["q"])
            if i == 0:
                WnewSum = Wnew
                qProp, L_, indexStat = o["q"], xi, xi * timeLen[side]   # :326-328,359-361
            else:
                WnewSum += Wnew
                if WnewSum > WT_SUM_THRESH and rng.uniform() < Wnew / WnewSum:   # :426,464,512,554
                    qProp, L_, indexStat = o["q"], idx, xi * timeLen[side]
                orbitLen += h                                           # :432,471,519,561
                if n % 2 == 1:
                    # left end of levels 1..tz(n-1) (all levels when n == 1): one slot suffices
                    lvl = i if n == 1 else ((n - 1) & -(n - 1)).bit_length() - 1
                    left[lvl] = (o["q"], o["v"])
                else:
                    s = 1
                    while s <= i and n % (2 ** s) == 0:
                        m = n - 2 ** s + 1
                        lvl = i if m == 1 else ((m - 1) & -(m - 1)).bit_length() - 1
                        ql, vl = left[lvl]
                        if xi == 1:
                            ut = stop_condition(ql, vl, o["q"], o["v"])          # :568,582
                        else:
                            ut = stop_condition(o["q"], o["v"], ql, vl)          # :479,582
                        if ut:
                            expand = False
                            break
                        s += 1
                    if not expand:
                        break
        if forced:                                                      # :590-592 (quirk A14(iii))
            break
        with np.errstate(all="ignore"):
            indexStat = indexStat / (timeLen[0] + timeLen[1])           # :595
        if not expand:                                                  # :597-605
            qProp, L_, indexStat = qPropLast, Lold, indexStatOld
            NdS, NdC, stopCode = i, i + 1, 5
            break
        if not (rng.uniform() < WnewSum / WoldSum):                     # :613
            qProp, L_, indexStat = qPropLast, Lold, indexStatOld
        joined = stop_condition(end_q[1], end_v[1], end_q[0], end_v[0])  # :622
        bothEndsPassive = lwtSum[1] < LOG_ZERO + 1.0 and lwtSum[0] < LOG_ZERO + 1.0   # :624
        if joined or bothEndsPassive:
            stopCode = 4 if joined else -4
            NdS = NdC = i + 1
            orbitLenSam = orbitLen
            break
        WoldSum += WnewSum                                              # :641
        orbitLenSam = orbitLen
        NdS = NdC = i + 1

    diag = np.zeros(24)
    n = st["n"]
    diag[0] = L_
    diag[1] = NdS
    diag[2] = orbitLen
    diag[3] = orbitLenSam
    diag[4] = maxInt[0]
    diag[5] = maxInt[1]
    diag[6] = nF
    diag[7] = nB
    diag[8], diag[9] = st["minIf"], st["maxIf"]
    diag[10], diag[11] = st["minl"], st["maxl"]
    diag[12] = 1.0 * bothEndsPassive
    diag[13] = 1.0 * (lwtSum[1] < LOG_ZERO + 1.0 or lwtSum[0] < LOG_ZERO + 1.0)
    diag[14] = st["nne"] / n
    diag[15] = H
    diag[16] = st["nz"] / n
    diag[17] = np.nan if st["Hnan"] else st["Hmax"] - st["Hmin"]
    diag[18] = delta
    diag[19] = 1.0 * stopCode
    diag[20] = NdC
    diag[21], diag[22] = st["minc"], st["maxc"]
    diag[23] = indexStat
    return qProp, diag


class P2Quantile:
    """Restatement of WALNUTSpy/P2quantile.py:16-92 (P-squared online quantile, Jain & Chlamtac 1985),
    including its behaviour when `findInterval` falls through (xi == q[4]: :31-39 returns None, and
    `n[None:5] += 1` then increments every marker position)."""

    def __init__(self, prob=0.5):
        self.npush = 0
        self.p = prob
        self.q = np.zeros(5)
        self.n = np.arange(1, 6)

    def quantile(self):
        return self.q[2]

    def push(self, xi):
        self.npush += 1
        if self.npush <= 5:
            self.q[self.npush - 1] = xi
            if self.npush == 5:
                self.q = np.sort(self.q)                    # :45-47
            return
        q, n = self.q, self.n
        if xi < q[0]:                                        # :31-39, 49-57
            q[0] = xi
            k = 1
        elif xi > q[4]:
            q[4] = xi
            k = 4
        else:
            k = None
            for i in range(4):
                if xi < q[i + 1]:
                    k = i + 1
                    break
        n[k:5] += 1                                          # :60
        nn, pp = self.npush, self.p
        npp = np.array([1.0, 0.5 * (nn - 1) * pp + 1.0, (nn - 1) * pp + 1.0, (nn - 1) * (1 + pp) / 2.0 + 1, nn])
        with np.errstate(all="ignore"):
            for i in range(2, 5):                            # :70-89
                ni, nip, nim = n[i - 1], n[i], n[i - 2]
                di = npp[i - 1] - ni
                if (di >= 1.0 and nip - ni > 1) or (di <= -1.0 and nim - ni < -1):
                    di = np.sign(di).astype(np.int64)
                    qi = q[i - 1]
                    qip = qi + (di / (nip - nim)) * ((ni - nim + di) * (q[i] - qi) / (nip - ni)
                                                     + (nip - ni - di) * (qi - q[i - 2]) / (ni - nim))
                    if q[i - 2] < qip and qip < q[i]:
                        q[i - 1] = qip
                    else:
                        q[i - 1] = qi + di * (q[i + di - 1] - qi) / (n[i + di - 1] - n[i - 1])
                    n[i - 1] += di


class PhiloxRNG:
    """Adapter: oracle.philox.ChainStreams -> the rng protocol used by transition()."""

    def __init__(self, streams):
        self.s = streams

    def dir_uniform02(self, M):
        return 2.0 * self.s.directions(M)

    def normal(self, d):
        return self.s.momentum(d)

    def uniform_range(self, lo, hi, size):
        return np.array([lo + (hi - lo) * self.s.uniform() for _ in range(size)])

    def uniform(self):
        return self.s.uniform()


class NumpyGlobalRNG:
    """Adapter over numpy's legacy global RNG, call-for-call as the reference uses it."""

    def dir_uniform02(self, M):
        return np.random.uniform(low=0.0, high=2.0, size=M)

    def normal(self, d):
        return np.random.normal(size=d)

    def uniform_range(self, lo, hi, size):
        return np.random.uniform(low=lo, high=hi, size=size)

    def uniform(self):
        return np.random.uniform()


def WALNUTS(lpFun, q0, generated=lambda q: q, integrator=FIXED, H0=0.2, stepSizeRandScale=0.2,
            delta0=0.05, numIter=2000, M=10, igrAux=None, rng=None, seed=0, chain=0,
            first_iteration=1, warmupIter=0, adaptH=False, adaptHtarget=0.8, adaptDelta=False,
            adaptDeltaTarget=0.6, adaptDeltaQuantile=0.9, recordOrbitStats=False, compat=True):
    """WALNUTSpy chain incl. the warm-up adaptation of H and delta (WALNUTS.py:136-147, 313, 701-712).
    Returns (samples (dg, numIter+1), diagnostics (numIter, 24)) like WALNUTS.py:724-727."""
    from . import philox
    aux = igrAux or AuxPar()
    streams = None
    if rng is None:
        streams = philox.ChainStreams(seed, chain)
        rng = PhiloxRNG(streams)
    qc = np.asarray(q0, dtype=np.float64)
    g0 = generated(qc)
    samples = np.zeros((g0.size, numIter + 1))
    samples[:, 0] = g0
    diagnostics = np.zeros((numIter, 24))
    H, delta = H0, delta0
    orbitMin = np.zeros((qc.size, numIter))
    orbitMax = np.zeros((qc.size, numIter))
    p2 = P2Quantile(1.0 - adaptHtarget) if adaptH else None                    # :139-141
    facs = np.zeros(warmupIter) if adaptDelta else None                         # :145-147
    for it in range(1, numIter + 1):
        if streams is not None:
            streams.begin_iteration(first_iteration + it - 1)
        warmup = it <= warmupIter                                               # :209
        sink = None
        if warmup and adaptH:
            with np.errstate(all="ignore"):
                sink = lambda c: p2.push(np.log(c))                             # :313
        with np.errstate(all="ignore"):
            orb = {} if recordOrbitStats else None
            qc, diagnostics[it - 1] = transition(lpFun, qc, rng, integrator, H, delta, M, aux,
                                                 jitter=stepSizeRandScale, igr_sink=sink, orbit=orb, compat=compat)
            if recordOrbitStats:
                orbitMin[:, it - 1], orbitMax[:, it - 1] = orb["min"], orb["max"]
            samples[:, it] = generated(qc)
            if warmup:                                                          # :701-712
                if adaptDelta:
                    facs[it - 1] = diagnostics[it - 1, 17] / delta
                if adaptDelta and it > 10:
                    delta = adaptDeltaTarget / np.quantile(facs[0:it], adaptDeltaQuantile)
                if adaptH and p2.npush > 10:
                    H = (delta ** (1.0 / 3.0)) * np.exp(p2.quantile())
    if recordOrbitStats:
        return samples, diagnostics, orbitMin, orbitMax
    return samples, diagnostics
