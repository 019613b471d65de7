"""Generate the golden fixtures by running the REAL reference (a bob-carpenter/walnuts checkout) under the Philox RNG
shims of oracle/ref_loader.py and oracle/package_oracle.py.  Run from the repo root:

    WALNUTS_REFERENCE=<checkout> PYTHONPATH=. python tests/golden/make_golden.py

Each .npz stores the inputs (config, q0, seed, chain) and the reference's own outputs.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import package_oracle as po   # noqa: E402
from oracle import ref_loader             # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
NAMES = {"fixed": "fixedLeapFrog", "D": "adaptLeapFrogD", "R2P": "adaptLeapFrogR2P", "Yoshida": "adaptYoshidaD",
         "Flow": "adaptLeapFrogFlowD", "Midpoint": "adaptImplicitMidpointD", "Rescaled": "adaptRescaledLeapFrogD"}


def walnutspy_cases():
    rng = np.random.default_rng(2025)
    fq = np.zeros(11)
    fq[0] = 1.3
    fq[1:] = np.exp(0.5 * fq[0]) * rng.standard_normal(10)
    cases = []
    for integ in ("fixed", "D", "R2P"):
        cases.append(dict(name=f"wpy_std7_{integ}", target="std_normal", q0=0.3 * rng.standard_normal(7),
                          integrator=integ, H0=0.6, delta=0.3, M=8, n_iter=100, minC=0, maxC=10, seed=11, chain=3))
        cases.append(dict(name=f"wpy_funnel10_{integ}", target="funnel", q0=fq.copy(), integrator=integ, H0=0.3,
                          delta=0.3, M=12 if integ != "fixed" else 10, n_iter=100, minC=0, maxC=10, seed=12, chain=1))
        cases.append(dict(name=f"wpy_corr_{integ}", target="corr_gauss", q0=np.array([1.0, 0.0]), integrator=integ,
                          H0=0.9, delta=0.1, M=8, n_iter=100, minC=1, maxC=10, seed=13, chain=0))
    # SURVEY.md row N3: the remaining integrators of adaptiveIntegrators.py (added after the cases above; the
    # generator state is re-seeded so that the earlier fixtures stay byte-identical)
    rng2 = np.random.default_rng(2026)
    for integ, dlt in (("Yoshida", 0.05), ("Flow", 0.02), ("Midpoint", 0.05), ("Rescaled", 0.3)):
        cases.append(dict(name=f"wpy_std7_{integ}", target="std_normal", q0=0.3 * rng2.standard_normal(7),
                          integrator=integ, H0=1.1, delta=dlt, M=7, n_iter=60, minC=0, maxC=10, seed=21, chain=2))
        cases.append(dict(name=f"wpy_funnel10_{integ}", target="funnel", q0=fq.copy(), integrator=integ, H0=0.4,
                          delta=dlt, M=8, n_iter=40, minC=0, maxC=10, seed=22, chain=4))
    # warm-up adaptation with the reference's default arguments (P-squared quantile for H, quantile of the energy
    # error for delta, WALNUTS.py:136-147,313,701-712): pins the oracle's adaptation incl. every integrator's igrConst
    rng3 = np.random.default_rng(2027)
    # (adaptImplicitMidpointD is left out: the implicit midpoint rule conserves a quadratic energy exactly, igrConst
    # becomes infinite and the reference itself ends in sys.exit("numerical problems") under its default adaptation)
    for integ in ("fixed", "D", "R2P", "Yoshida", "Flow", "Rescaled"):
        cases.append(dict(name=f"wpy_adapt_std5_{integ}", target="std_normal", q0=0.5 * rng3.standard_normal(5),
                          integrator=integ, H0=0.2, delta=0.05, M=7, n_iter=90, warmup=60, minC=0, maxC=10, seed=31,
                          chain=1))
    cases.append(dict(name="wpy_std100_R2P", target="std_normal", q0=rng.standard_normal(100), integrator="R2P",
                      H0=0.9 * 100 ** -0.25, delta=0.3, M=8, n_iter=40, minC=0, maxC=10, seed=14, chain=7))
    return cases


def package_cases():
    return [
        dict(name="pkg_std2_testpy", target="std_normal", theta0=np.zeros(2), inv_mass=np.ones(2), macro_step=2.0,
             max_depth=10, max_error=0.1, n_iter=40, seed=123, chain=0),       # test/test.py:10-18 settings
        dict(name="pkg_std5_mass", target="std_normal", theta0=np.full(5, 0.3), inv_mass=np.array([.5, 1, 2, 1, .7]),
             macro_step=1.3, max_depth=8, max_error=0.2, n_iter=30, seed=7, chain=2),
        dict(name="pkg_funnel4", target="funnel_pkg", theta0=np.array([0.5, .1, .2, -.3]), inv_mass=np.ones(4),
             macro_step=1.0, max_depth=6, max_error=0.3, n_iter=12, seed=8, chain=5),
        # BASELINE config 1 at its full shape: 100-d standard normal, test/test.py:10-18 settings, depth 10, the
        # first 100 transitions (north_star parity statement)
        dict(name="pkg_std100_c1", target="std_normal", theta0=np.zeros(100), inv_mass=np.ones(100), macro_step=2.0,
             max_depth=10, max_error=0.1, n_iter=100, seed=123, chain=0),
        dict(name="pkg_std3_ell0_defect", target="std_normal", theta0=np.full(3, 0.2), inv_mass=np.ones(3),
             macro_step=0.5, max_depth=5, max_error=0.1, n_iter=12, seed=9, chain=1),
    ]


def main():
    only = sys.argv[1:]          # optional name prefixes: regenerate only the matching fixtures
    want = (lambda name: any(name.startswith(p) for p in only)) if only else (lambda name: True)
    wn, ai, td = ref_loader.load_walnutspy()
    pkg = ref_loader.load_package()
    tt = ref_loader.load_test_targets()
    lp = {"std_normal": td.stdGauss, "funnel": td.funnel10, "corr_gauss": td.corrGauss}
    for c in walnutspy_cases():
        if not want(c["name"]):
            continue
        t0 = time.time()
        s, d = ref_loader.run_walnutspy(lp[c["target"]], c["q0"], NAMES[c["integrator"]], c["H0"], c["delta"],
                                        c["n_iter"], c["M"], c["minC"], c["maxC"], seed=c["seed"], chain=c["chain"],
                                        warmupIter=c.get("warmup", 0))
        meta = {k: v for k, v in c.items() if k != "q0"}
        np.savez_compressed(os.path.join(OUT, c["name"] + ".npz"), meta=json.dumps(meta), q0=c["q0"], samples=s,
                            diagnostics=d)
        print(f"{c['name']}: {time.time() - t0:.1f}s stop codes {np.unique(d[:, 19])}")
    # recordOrbitStats=True (WALNUTS.py:182-184,274-276,...): per-iteration min / max of the states visited by the orbit
    if want("orbit_corr_R2P"):
        q0 = np.array([0.8, -0.3])
        s, d, omin, omax = ref_loader.run_walnutspy(td.corrGauss, q0, "adaptLeapFrogR2P", 0.9, 0.1, 50, 7, 0, 10, seed=41,
                                                    chain=2, recordOrbitStats=True)
        meta = dict(name="orbit_corr_R2P", target="corr_gauss", integrator="R2P", H0=0.9, delta=0.1, M=7, n_iter=50,
                    minC=0, maxC=10, seed=41, chain=2)
        np.savez_compressed(os.path.join(OUT, "orbit_corr_R2P.npz"), meta=json.dumps(meta), q0=q0, samples=s,
                            diagnostics=d, orbit_min=omin, orbit_max=omax)
        print("orbit_corr_R2P: done")
    plp = {"std_normal": (tt.standard_normal_lpdf, tt.standard_normal_grad),
           "funnel_pkg": (tt.funnel_lpdf, tt.funnel_grad)}
    for c in package_cases():
        if not want(c["name"]):
            continue
        t0 = time.time()
        rng = po.KeyedPackageRNG(c["seed"], c["chain"])
        f, g = plp[c["target"]]
        with np.errstate(all="ignore"):
            draws = pkg.walnuts(rng, c["theta0"], f, g, c["inv_mass"], c["macro_step"], c["max_depth"],
                                c["max_error"], 0, c["n_iter"])
        meta = {k: v for k, v in c.items() if k not in ("theta0", "inv_mass")}
        np.savez_compressed(os.path.join(OUT, c["name"] + ".npz"), meta=json.dumps(meta), theta0=c["theta0"],
                            inv_mass=c["inv_mass"], draws=draws)
        print(f"{c['name']}: {time.time() - t0:.1f}s")


if __name__ == "__main__":
    main()
