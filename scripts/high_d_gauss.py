"""Throughput and ESS of the standard normal above d = 4096 (one chain per thread-block cluster) next to the d = 4096
single-CTA kernel, with the reference's Gaussian scalings (mainGaussESS.py): H = 1.4 d^-1/4 for adaptLeapFrogD /
adaptLeapFrogR2P and H = d^-1/2 for fixedLeapFrog.

Per (d, integrator): gradient evaluations / s and coordinate-steps / s from device time (wn_last_kernel_ms), the share
of the in-run FP64 FMA peak (wn_fp64_peak) at 4 flop per coordinate-step (drift and kick FMA of the merged-kick loop,
counting an FMA as 2 flop), the resident chain groups (clusters above d = 4096), and the bulk ESS of q[0] over the
chains per gradient evaluation (ChainBatch(..., dg=1) draws into wn_ess_rhat), the quantity of mainGaussESS.py.
Chains start from exact N(0, I) draws, so every transition is stationary.  Prints the card and its power limit.

    python scripts/high_d_gauss.py [--chains 592] [--iters 100]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from walnuts_b200 import ChainBatch, _ffi  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=592)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--dims", default="4096,4097,8192,16384,32768")
    a = ap.parse_args()
    lib = _ffi.load()
    import ctypes as C
    peak = C.c_double()
    assert lib.wn_fp64_peak(0, C.byref(peak)) == 0
    print(f"# card: {card()}")
    print(f"# in-run FP64 FMA peak: {peak.value / 1e12:.2f} TFLOP/s; {a.chains} chains x {a.iters} transitions "
          f"(after one warm-up call), std_normal, M = 10, delta = 0.3")
    print(f"{'d':>6} {'int':>5} {'plan (G,E2,NT)':>16} {'slots':>5} {'ms':>9} {'grad/s':>10} {'coord-steps/s':>13} "
          f"{'FP64 %':>6} {'ESS(q0)':>8} {'ESS/grad':>9}")
    for d in (int(x) for x in a.dims.split(",")):
        q0 = np.random.default_rng(d).standard_normal((a.chains, d))
        for integ in ("fixed", "D", "R2P"):
            H0 = d ** -0.5 if integ == "fixed" else 1.4 * d ** -0.25
            with ChainBatch("std_normal", d, a.chains, integrator=integ, H0=H0, delta=0.3, M=10, seed=3, dg=1) as cb:
                cb.set_state(q0)
                cb.run(1, draws=False)                                   # warm-up: module load, scratch
                out = cb.run(a.iters, draws=True)
                ms = cb.last_kernel_ms()
                f, b = cb.last_grad_evals()
                plan, slots = cb.last_plan(), cb.last_slots()
                ess, _ = cb.ess_rhat(out["draws"])
            ev = f + b
            gps = ev / (ms * 1e-3)
            cps = gps * d
            print(f"{d:>6} {integ:>5} {str(plan[1:]):>16} {slots:>5} {ms:>9.2f} {gps:>10.3e} {cps:>13.3e} "
                  f"{100.0 * 4.0 * cps / peak.value:>6.2f} {ess[0]:>8.0f} {ess[0] / ev:>9.2e}", flush=True)


if __name__ == "__main__":
    main()
