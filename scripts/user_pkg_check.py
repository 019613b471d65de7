"""User plug-in (standard normal written as a user target) against the built-in standard normal in package mode on the
ell = 0 defect path (small macro step), in the thread layout that user targets with d <= 64 run."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import walnuts_b200 as wb
SRC = """
WN_TARGET_LP_GRAD(q, g, data, n_data) {
  double lp = 0.0;
  for (int i = 0; i < WN_D; ++i) { g[i] = -q[i]; lp += q[i] * q[i]; }
  return -0.5 * lp;
}
"""
for d in (2, 8, 20):
    tg = wb.targets.cuda_target(SRC, d, name=f"sn{d}")
    bi = wb.targets.standard_normal_lpdf
    q0 = 0.4 * np.random.default_rng(1).standard_normal((64, d))
    for macro in (0.9, 0.25):
        p1 = wb.walnuts(None, q0, tg, tg, np.ones(d), macro, 6, 0.3, 0, 6, seed=9)
        p2 = wb.walnuts(None, q0, bi, bi, np.ones(d), macro, 6, 0.3, 0, 6, seed=9)
        same = (np.isnan(p1) & np.isnan(p2)) | (np.abs(p1 - p2) <= 1e-9 * np.maximum(1.0, np.abs(p2)))
        print(d, macro, "chains differing:", int((~same).any(axis=(0, 2)).sum() if p1.ndim == 3 else (~same).any()),
              "of 64; max |diff|", float(np.nanmax(np.abs(p1 - p2))), flush=True)
