"""Gradient evaluations per second of a user CUDA target in the parallel protocol (cuda_target(..., parallel=True))
against the built-in diag_gauss at d = 512, 1024, 2048, 4096, and against the sequential protocol at d = 512 (the
only size both protocols serve).  The three targets are the same diagonal Gaussian, so their draws agree and the
rates compare the cost of a gradient evaluation on the same trajectories.

Rates are from device time (wn_last_kernel_ms) of one call of --iters transitions after a warm-up call, adaptLeapFrogR2P,
H = 1.4 sigma_min d^-1/4, M = 10; chains start from exact draws of the target.  Each (d, target) is measured --reps
times, the targets alternating, and the median is printed with the spread.  Prints the card and its power limit.

    python scripts/user_parallel_bench.py [--chains 2368] [--iters 20] [--reps 3]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import walnuts_b200 as wb  # noqa: E402
from walnuts_b200 import ChainBatch  # noqa: E402

PAR_SRC = """
WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
  double lp = 0.0;
  for (int j = ctx.rank; j < WN_D; j += ctx.size) { g[j] = -q[j] * data[j]; lp += q[j] * g[j]; }
  return 0.5 * lp;
}"""
SEQ_SRC = """
WN_TARGET_LP_GRAD(q, g, data, n_data) {
  double lp = 0.0;
  for (int i = 0; i < WN_D; ++i) { g[i] = -q[i] * data[i]; lp += q[i] * g[i]; }
  return 0.5 * lp;
}"""


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def measure(tg, q0, H0, iters):
    d = q0.shape[1]
    tid, data = wb.targets.resolve(tg, d)
    with ChainBatch(tid, d, q0.shape[0], integrator="R2P", H0=H0, delta=0.3, M=10, seed=3, data=data, dg=1) as cb:
        cb.set_state(q0)
        cb.run(1, draws=False)                      # warm-up: module load, scratch
        cb.run(iters, draws=False)
        ms = cb.last_kernel_ms()
        f, b = cb.last_grad_evals()
        return (f + b) / (ms * 1e-3), cb.last_plan(), cb.last_slots()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=2368)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dims", default="512,1024,2048,4096")
    a = ap.parse_args()
    print(f"# card: {card()}")
    print(f"# {a.chains} chains x {a.iters} transitions (after one warm-up call), diagonal Gaussian "
          f"sigma = exp(U(-1, 1)), adaptLeapFrogR2P, M = 10, delta = 0.3; median of {a.reps} (min .. max)")
    print(f"{'d':>5} {'target':>10} {'plan (fam,G,E2,NT)':>20} {'slots':>5} {'grad/s':>10} {'min':>10} {'max':>10} "
          f"{'vs diag_gauss':>13}")
    for d in (int(x) for x in a.dims.split(",")):
        rng = np.random.default_rng(d)
        sigma = np.exp(rng.uniform(-1.0, 1.0, d))
        q0 = rng.standard_normal((a.chains, d)) * sigma
        iv = 1.0 / sigma ** 2
        tgs = {"diag_gauss": wb.targets.diag_gauss(sigma),
               "parallel": wb.targets.cuda_target(PAR_SRC, d, data=iv, name="bench_par", parallel=True)}
        if d <= 512:
            tgs["sequential"] = wb.targets.cuda_target(SEQ_SRC, d, data=iv, name="bench_seq")
        H0 = 1.4 * sigma.min() * d ** -0.25
        rates = {k: [] for k in tgs}
        info = {}
        for _ in range(a.reps):
            for k, tg in tgs.items():
                r, plan, slots = measure(tg, q0, H0, a.iters)
                rates[k].append(r)
                info[k] = (plan, slots)
        base = float(np.median(rates["diag_gauss"]))
        for k, rs in rates.items():
            med = float(np.median(rs))
            print(f"{d:>5} {k:>10} {str(info[k][0]):>20} {info[k][1]:>5} {med:>10.3e} {min(rs):>10.3e} "
                  f"{max(rs):>10.3e} {med / base:>13.3f}", flush=True)


if __name__ == "__main__":
    main()
