"""Kernel-only throughput of the bench workload (device-resident), for tuning experiments."""
import sys, os, time, argparse
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
from walnuts_b200 import ChainBatch
ap = argparse.ArgumentParser()
ap.add_argument("--chains", type=int, default=16384)
ap.add_argument("--iters", type=int, default=1)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--integrator", default="R2P")
ap.add_argument("--H0", type=float, default=0.5)
a = ap.parse_args()
sigma = bench.sigma_vec()
q0 = bench.init_positions(a.chains, 0, sigma)
cb = ChainBatch("diag_gauss", bench.D, a.chains, integrator=a.integrator, H0=a.H0, delta=0.3, M=10, seed=1, dg=0,
                data={"inv_var": 1.0 / sigma ** 2})
cb.set_state(q0)
cb.run_device(a.iters)
res = []
for r in range(a.reps):
    cb.run_device(a.iters)
    f, b = cb.last_grad_evals(); ms = cb.last_kernel_ms()
    res.append((f + b) / (ms * 1e-3))
print("chains=%d %s: %.4g grad evals/s (%.2f TFLOP/s algorithmic), last %.1f ms" % (
    a.chains, a.integrator, max(res), max(res) * 12e3 / 1e12, ms))
