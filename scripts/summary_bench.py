"""Device time of the posterior summary (wn_summary, ChainBatch.summary) against bulk ESS / R-hat (wn_ess_rhat,
ChainBatch.ess_rhat) on the same device-resident draws, at three shapes: 592 chains x 2048 draws x 8 coordinates (the
min-ESS shape of bench.py), 65 536 x 100 x 8 and 1 048 576 x 10 x 4.

Draws are AR(1) chains (rho = 0.9) generated on the device from a seed.  Each call is timed with CUDA events recorded on
the handle's stream around it (both calls end in a stream synchronisation, so the events cover the whole call,
including the per-coordinate host round trip).  Every shape is warmed up with one call of each, then measured --reps
times with the two calls alternating; the median is printed with the spread.  Prints the card and its power limit.

    python scripts/summary_bench.py [--reps 5]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from walnuts_b200 import ChainBatch  # noqa: E402

SHAPES = ((2048, 592, 8), (100, 65536, 8), (10, 1048576, 4))     # (draws, chains, coordinates)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def ar1_draws(n_iter, n_chains, dg, seed, rho=0.9):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.empty((n_iter, n_chains, dg), dtype=torch.float64, device="cuda")
    x[0] = torch.randn((n_chains, dg), generator=g, dtype=torch.float64, device="cuda")
    for t in range(1, n_iter):
        x[t] = rho * x[t - 1] + (1 - rho * rho) ** 0.5 * torch.randn((n_chains, dg), generator=g, dtype=torch.float64,
                                                                    device="cuda")
    torch.cuda.synchronize()
    return x


def timed(cb, fn):
    st = torch.cuda.ExternalStream(cb.stream)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    fn()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    print(f"# card: {card()}")
    print(f"# device-resident AR(1) draws (rho = 0.9); one warm-up call of each, then median of {a.reps} alternating "
          f"calls (min .. max), CUDA events on the handle's stream")
    print(f"{'chains':>8} {'draws':>6} {'dg':>3} {'ess_rhat ms':>12} {'min':>8} {'max':>8} {'summary ms':>11} {'min':>8} "
          f"{'max':>8} {'summary / ess_rhat':>18}")
    for n_iter, n_chains, dg in SHAPES:
        x = ar1_draws(n_iter, n_chains, dg, seed=n_chains)
        with ChainBatch("std_normal", dg, 1, H0=0.5, delta=0.3, M=5, seed=1) as cb:
            cb.ess_rhat(x)
            cb.summary(x)
            t = {"ess_rhat": [], "summary": []}
            for _ in range(a.reps):
                t["ess_rhat"].append(timed(cb, lambda: cb.ess_rhat(x)))
                t["summary"].append(timed(cb, lambda: cb.summary(x)))
        e, s = (float(np.median(t[k])) for k in ("ess_rhat", "summary"))
        print(f"{n_chains:>8} {n_iter:>6} {dg:>3} {e:>12.2f} {min(t['ess_rhat']):>8.2f} {max(t['ess_rhat']):>8.2f} "
              f"{s:>11.2f} {min(t['summary']):>8.2f} {max(t['summary']):>8.2f} {s / e:>18.2f}", flush=True)
        del x
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
