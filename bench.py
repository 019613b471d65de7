#!/usr/bin/env python
"""Benchmark of the many-chain WALNUTS hot path: gradient evals/sec and min-ESS/sec.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], the config the metric is quoted on): 1000-d ill-conditioned diagonal
Gaussian, sigma = logspace(-2, 2, 1000), 65 536 chains PER GPU (weak scaling), WALNUTSpy driver with
adaptLeapFrogR2P, H0 = 0.5, delta = 0.3, M = 10, minC = 0, maxC = 10 (SURVEY.md section 8(d) row C2).
One "step" = one transition of every chain (one persistent-kernel launch).

ONE JSON line (rank 0):
  value            gradient evaluations per second, chain states resident in HBM, timed with CUDA events on the
                   handle's stream (max over ranks)
  e2e              the same through host buffers (wn_run_host_async on pinned memory: positions H2D, draws /
                   diagnostics / counters / positions D2H inside the timed region; two handles per GPU so that the
                   copies of one overlap the kernel of the other)
  min_ess_per_sec  cross-chain bulk ESS (rank-normalised, split chains; the arviz / Stan estimator) of the slowest
                   monitored coordinate per second of device time, from a dedicated leg with >= 1024 draws per chain
  configs          the OTHER BASELINE configs under the same clock: C1 package-mode 100-d normal, C2 with plain NUTS,
                   C3 funnel, C4 logistic regression, C5 Stock-Watson (131 072 chains per GPU = 1 048 576 on 8 GPUs)
                   and 1 048 576 C2 chains on one GPU -- each with value, e2e, roofline, cpu_baseline, clocks
  strong_scaling   the headline workload with 65 536 chains in TOTAL split over the N GPUs (N > 1)
`--dump-outputs DIR` writes what the headline's last timed step handed back (float64 .npy files, see
headline_outputs) so that two builds can be compared output for output; the inputs depend only on the arguments.
With N > 1 GPUs the dump holds rank 0's chains only.
`--impl reference` times the CPU restatement of the reference's Python implementation (oracle/walnutspy_oracle.py;
the reference itself is Python and cannot travel to the GPU box) on all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if __name__ in ("__main__", "__mp_main__"):      # the script and its CPU-arm workers
    sys.dont_write_bytecode = True    # the bench writes nothing into the tree it runs from (which may be read-only)

SEED = 20251017
D = 1000
CHAINS_PER_GPU = 65536
MONITOR = 16                      # coordinates monitored for ESS (spread over the sigma range)

# Workloads.  flop_per_eval = FP64 work per gradient evaluation (= one leapfrog micro-step incl. the energy) of SURVEY.md
# section 8(d), the roofline numerator -- except for C2 / R2P, whose kernel EXECUTES only 4 flop per coordinate (merged
# kicks, linear gradient folded into the kick, energies only where they are consumed: DESIGN.md section 6): there the
# executed work is the numerator (`frac`), and the figure at SURVEY's 12 flop per coordinate is reported next to it.
WORKLOADS = {
    "c2": dict(target="diag_gauss", d=D, mode="walnutspy", integrator="R2P", H0=0.5, delta=0.3, M=10, minC=0, maxC=10,
               chains=CHAINS_PER_GPU, iters=1, monitor=MONITOR, flop_per_eval=4.0 * D, flop_per_eval_survey=12.0 * D,
               workload="diag_gauss_d1000_sigma_logspace(-2,2)_R2P"),
    "c1": dict(target="std_normal", d=100, mode="package", integrator="fixed", H0=2.0, delta=0.1, M=10, minC=0, maxC=10,
               chains=65536, iters=4, monitor=8, flop_per_eval=12.0 * 100, steps_cap=5, warmup_cap=3,
               workload="package_walnuts_std_normal_d100_macro2.0_depth10_maxerr0.1 (test/test.py:10-18)"),
    "c2_nuts": dict(target="diag_gauss", d=D, mode="walnutspy", integrator="fixed", H0=0.008, delta=0.3, M=10, minC=0,
                    maxC=10, chains=CHAINS_PER_GPU, iters=1, monitor=MONITOR, flop_per_eval=12.0 * D, steps_cap=5,
                    warmup_cap=3, workload="diag_gauss_d1000_fixedLeapFrog_H0.008 (plain NUTS)"),
    "c3": dict(target="funnel", d=11, mode="walnutspy", integrator="R2P", H0=0.3, delta=0.3, M=12, minC=0, maxC=10,
               chains=262144, iters=10, monitor=11, flop_per_eval=200.0, steps_cap=5, warmup_cap=3,
               workload="funnel10_R2P_M12 (mainFunnel.py:24-32)"),
    "c4": dict(target="logreg", d=100, mode="walnutspy", integrator="R2P", H0=0.05, delta=0.3, M=6, minC=0, maxC=10,
               chains=16384, iters=1, monitor=8, flop_per_eval=4.5e7, steps_cap=2, warmup_cap=1,
               workload="logreg_N100000_P100_R2P"),
    "c5": dict(target="stock_watson", d=756, mode="walnutspy", integrator="R2P", H0=0.1, delta=0.3, M=14, minC=3,
               maxC=10, chains=131072, iters=1, monitor=8, flop_per_eval=4.0e4, steps_cap=3, warmup_cap=2,
               workload="stock_watson_T252_R2P_M14_minC3 (mainSW.py:41-49); 131072 chains per GPU"),
    "c2_1m": dict(target="diag_gauss", d=D, mode="walnutspy", integrator="R2P", H0=0.5, delta=0.3, M=10, minC=0,
                  maxC=10, chains=1048576, iters=1, monitor=MONITOR, flop_per_eval=4.0 * D,
                  flop_per_eval_survey=12.0 * D, steps_cap=1, warmup_cap=0,
                  single_gpu_only=True, e2e=False,
                  workload="diag_gauss_d1000_R2P, 1 048 576 concurrent chains on ONE GPU (kernel warm from the headline leg)"),
}
CONFIG_ORDER = ["c1", "c2_nuts", "c3", "c4", "c5", "c2_1m"]
# min-ESS leg: one chain per resident slot of the d = 1000 kernel (148 SMs x 4 blocks) x 2048 draws.  The slowest
# coordinate (sigma = 100) has an autocorrelation time of ~700 transitions at this tuning, so the chains must be long;
# the estimator pools 592 x N_GPU chains that start from exact draws of the target.
ESS_CHAINS, ESS_DRAWS = 592, 2048
# --dump-outputs: draws of up to 65 536 chains and positions of up to 4 096 (one position is 8 KB at d = 1000);
# larger batches are sampled with a fixed seed.  At most 8.4 + 32.8 MB.
DUMP_DRAW_CHAINS, DUMP_STATE_CHAINS = 65536, 4096


def sigma_vec():
    # monitored coordinates first: the sigma ordering is arbitrary for a diagonal target, so the
    # logspace is permuted such that the leading MONITOR coordinates span the whole range
    s = np.logspace(-2, 2, D)
    idx = np.unique(np.round(np.linspace(0, D - 1, MONITOR)).astype(int))
    rest = np.setdiff1d(np.arange(D), idx)
    return np.concatenate([s[idx], s[rest]])


def init_positions(n, rank, sigma):
    """q0 = sigma * z: exact draws from the target, so ESS is measured at stationarity."""
    rng = np.random.Generator(np.random.Philox(key=SEED + 7919 * rank))
    return rng.standard_normal((n, D)) * sigma


def make_inputs(spec, n, rank):
    """(q0 [n, d], data) of a workload; states start in the typical set (SURVEY.md section 8(d))."""
    rng = np.random.Generator(np.random.Philox(key=SEED + 7919 * rank + 13))
    t = spec["target"]
    if t == "diag_gauss":
        sigma = sigma_vec()
        return init_positions(n, rank, sigma), {"inv_var": 1.0 / sigma ** 2}
    if t == "std_normal":
        q0 = rng.standard_normal((n, spec["d"]))
        return q0, ({"inv_mass": np.ones(spec["d"])} if spec["mode"] == "package" else {})
    if t == "funnel":
        q0 = np.empty((n, 11))
        q0[:, 0] = 3.0 * rng.standard_normal(n)
        q0[:, 1:] = np.exp(0.5 * q0[:, :1]) * rng.standard_normal((n, 10))
        return q0, {}
    if t == "logreg":
        from walnuts_b200 import datasets
        X, y, beta = datasets.synth_logreg(100_000, 100, 0)
        return beta + 0.05 * rng.standard_normal((n, 100)), {"X": X, "y": y, "tau": np.array([1.0])}
    if t == "stock_watson":
        from walnuts_b200 import datasets
        y = datasets.stock_watson_series()
        q0 = 0.05 * rng.standard_normal((n, 3 * y.size))
        q0[:, 0] = 2.4
        return q0, {"y": y}
    raise KeyError(t)


# --------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the numpy restatement of the reference (oracle/), one chain per process on every host core.  The only
# place besides tests/ and smoke() that executes anything under oracle/ (as the baseline being timed).
# --------------------------------------------------------------------------------------------------
def _cpu_worker(args):
    """Run transitions of chain `chain` of workload `name` for ~`budget` seconds (at least `min_tr` timed
    transitions after `warm` untimed ones, at most `max_tr`).  Returns (evals, seconds, transitions)."""
    name, chain, budget, min_tr, max_tr, warm, impl = args
    spec = WORKLOADS[name]
    q0, data = make_inputs(spec, chain + 1, 0)
    q = q0[chain]
    from oracle import targets as ot
    evals, n_tr, t_used = 0.0, 0, 0.0
    with np.errstate(all="ignore"):
        if spec["mode"] == "package":
            from oracle import package_oracle as po
            it = 1
            while True:
                cnt = [0]
                t0 = time.perf_counter()
                q = po.walnuts(SEED, chain, q, ot.standard_normal_lpdf, ot.standard_normal_grad, data["inv_mass"],
                               spec["H0"], spec["M"], spec["delta"], 0, 1, first_iteration=it, counter=cnt)[-1]
                dt = time.perf_counter() - t0
                it += 1
                if it - 1 > warm:
                    evals += cnt[0]; t_used += dt; n_tr += 1
                    if (t_used >= budget and n_tr >= min_tr) or n_tr >= max_tr:
                        break
            return evals, t_used, n_tr
        from oracle import walnutspy_oracle as wo
        t = spec["target"]
        if t == "diag_gauss":
            lp = ot.make_diag_gauss(1.0 / np.sqrt(data["inv_var"]))
        elif t == "funnel":
            lp = ot.funnel10
        elif t == "logreg":
            lp = ot.make_logreg(data["X"], data["y"], 1.0)
        elif t == "stock_watson":
            lp = ot.make_stock_watson(data["y"])
        else:
            lp = ot.std_normal
        kind = {"fixed": wo.FIXED, "D": wo.ADAPT_D, "R2P": wo.ADAPT_R2P}[spec["integrator"]]
        ref_name = {"fixed": "fixedLeapFrog", "D": "adaptLeapFrogD", "R2P": "adaptLeapFrogR2P"}[spec["integrator"]]
        if impl == "reference":
            from oracle import ref_loader        # the REAL WALNUTS.py / adaptiveIntegrators.py ($WALNUTS_REFERENCE or oracle/_ref)
        it = 1
        while True:
            t0 = time.perf_counter()
            if impl == "reference":
                s, dg = ref_loader.run_walnutspy(lp, q, ref_name, spec["H0"], spec["delta"], 1, spec["M"], spec["minC"],
                                                 spec["maxC"], seed=SEED, chain=chain, first_iteration=it)
            else:
                s, dg = wo.WALNUTS(lp, q, integrator=kind, H0=spec["H0"], delta0=spec["delta"], numIter=1, M=spec["M"],
                                   igrAux=wo.AuxPar(spec["minC"], spec["maxC"]), seed=SEED, chain=chain,
                                   first_iteration=it)
            dt = time.perf_counter() - t0
            q = s[:, -1]
            it += 1
            if it - 1 > warm:
                evals += float(dg[:, 6].sum() + dg[:, 7].sum()); t_used += dt; n_tr += 1
                if (t_used >= budget and n_tr >= min_tr) or n_tr >= max_tr:
                    break
    return evals, t_used, n_tr


_POOL = None


def _pool(cores):
    global _POOL
    if _POOL is None:
        import atexit
        import multiprocessing as mp
        # the reference is single-threaded: one chain per process and ONE BLAS / OpenMP thread per process (the
        # variables must be in the environment before the children import numpy)
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = "1"
        _POOL = mp.get_context("spawn").Pool(cores)
        atexit.register(_POOL.terminate)
    return _POOL


def reference_available():
    """The real reference's modules are importable here (the build container, or a copy staged by oracle/stage_ref.py)."""
    try:
        from oracle import ref_loader
        return ref_loader.available()
    except Exception:
        return False


def cpu_baseline(name="c2", budget=12.0, min_tr=1, max_tr=10 ** 9, warm=0, cores=None, impl="port"):
    """Gradient evals/sec of the reference algorithm with every host core busy on its own chain: the sum over cores of
    (evaluations / busy seconds).  impl = "port": the numpy restatement (oracle/); "reference": the reference's own
    WALNUTS.py + adaptiveIntegrators.py under the Philox shim (WALNUTSpy-mode workloads, when staged)."""
    cores = cores or os.cpu_count() or 1
    t0 = time.perf_counter()
    res = _pool(cores).map(_cpu_worker, [(name, c, budget, min_tr, max_tr, warm, impl) for c in range(cores)])
    wall = time.perf_counter() - t0
    rate = sum(r[0] / r[1] for r in res)
    n_tr = [r[2] for r in res]
    return {"value": rate, "unit": "grad_evals/s", "cores": cores, "kind": impl,
            "sample": f"{cores} chains (one per process, OMP_NUM_THREADS=1) x {min(n_tr)}..{max(n_tr)} transitions of "
                      f"{WORKLOADS[name]['workload']} on "
                      f"{'the numpy restatement of the reference' if impl == 'port' else 'the reference itself (WALNUTS.py, adaptiveIntegrators.py; Philox shim)'} "
                      f"({sum(r[0] for r in res):.0f} evals, {max(r[1] for r in res):.1f}s busy, wall {wall:.1f}s)",
            "per_core": rate / cores, "transitions_min": min(n_tr), "seconds": float(np.mean([r[1] for r in res])),
            "seconds_per_transition": float(np.mean([r[1] / r[2] for r in res]))}


def cpu_baseline_c(seconds=6.0, cores=None, ess=False):
    """C2 on the C restatement (oracle/c/walnuts_oracle.c, gcc -O3, pthreads): the strong CPU baseline standing in
    for the absent walnuts_cpp.  ess=True: keep going for `seconds` and measure the bulk ESS of the CPU draws."""
    from oracle import c_oracle
    from walnuts_b200 import diagnostics
    cores = cores or os.cpu_count() or 1
    sigma = sigma_vec()
    n = cores
    q = np.ascontiguousarray(init_positions(n, 0, sigma))
    draws, evals, it = [], 0, 1
    t0 = time.perf_counter()
    while True:
        evals += c_oracle.run_many("diag_gauss", "R2P", q, 0.5, 0.3, 10, 1, SEED, cores, minC=0, maxC=10,
                                   inv_var=1.0 / sigma ** 2, jitter=0.2, first_iteration=it)
        it += 1
        draws.append(q[:, :MONITOR].copy())
        if time.perf_counter() - t0 >= seconds and len(draws) >= 4:
            break
    dt = time.perf_counter() - t0
    out = {"value": evals / dt, "unit": "grad_evals/s", "cores": cores, "kind": "port-c",
           "sample": f"{n} chains x {len(draws)} transitions on {cores} pthreads (C restatement of the transition, "
                     f"gcc -O3; {evals} evals in {dt:.1f}s)", "per_core": evals / dt / cores}
    if ess:
        x = np.stack(draws)                                   # (draws, chains, monitor)
        vals = [diagnostics.ess_bulk(x[:, :, j].T)[0] for j in range(MONITOR)]
        out.update(min_ess=float(np.nanmin(vals)), min_ess_per_sec=float(np.nanmin(vals)) / dt,
                   ess_draws_per_chain=len(draws), ess_chains=n,
                   ess_note="bulk ESS of the CPU arm's OWN draws (few draws per chain: a noisy estimate)")
    return out


# --------------------------------------------------------------------------------------------------
# GPU legs
# --------------------------------------------------------------------------------------------------
class Env:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.dev = torch.device("cuda", self.local_rank)
        torch.cuda.set_device(self.dev)
        self.flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)   # 2 x the 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def flush_l2(self):
        self.flush_buf.zero_()

    def reduce(self, maxes, sums):
        t = self.torch
        a = t.tensor(maxes, dtype=t.float64, device=self.dev)
        b = t.tensor(sums, dtype=t.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(a, op=self.dist.ReduceOp.MAX)
            self.dist.all_reduce(b, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in a], [float(x) for x in b]


def make_batch(spec, n, chain_offset, device, data, q0):
    from walnuts_b200 import ChainBatch
    cb = ChainBatch(spec["target"], spec["d"], n, mode=spec["mode"], integrator=spec["integrator"], H0=spec["H0"],
                    jitter=0.2, delta=spec["delta"], M=spec["M"], minC=spec["minC"], maxC=spec["maxC"], seed=SEED,
                    chain_offset=chain_offset, device=device, dg=spec["monitor"], data=data)
    cb.set_state(q0)
    return cb


def _traffic(name, chains, iters):
    """roofline.traffic: DRAM bytes (read + write) of one launch of this workload's kernel, from the committed ncu pass
    over the bench command (profiles/r02_traffic.json, scripts/traffic_from_ncu.py) -- the bench itself never runs under a
    profiler.  null when there is no capture of this workload."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as fh:
            t = json.load(fh)
        w = t["workloads"][name]
        return {"traffic": w["traffic_bytes_per_launch"],
                "traffic_source": "profiles/r02_traffic.json: " + t["source"]}
    except (OSError, KeyError, ValueError):
        return {"traffic": None}


def headline_outputs(env, cb, draws, grad_evals):
    """What a caller of the device-resident path receives from one step: the monitored draws (iters, chains, monitor),
    the chain positions (chains, d) and the gradient evaluations (forward, backward) of the step.  Chains beyond
    DUMP_DRAW_CHAINS / DUMP_STATE_CHAINS are sampled (seed SEED, sorted rows), so the sample depends only on the
    chain count."""
    n = cb.n_chains

    def rows(k):
        return np.arange(n) if n <= k else np.sort(np.random.default_rng(SEED).choice(n, k, replace=False))
    state = env.torch.empty((n, cb.d), dtype=env.torch.float64, device=env.dev)
    cb.get_state(state)
    return {"draws": draws[:, env.torch.as_tensor(rows(DUMP_DRAW_CHAINS), device=env.dev)].cpu().numpy(),
            "positions": state[env.torch.as_tensor(rows(DUMP_STATE_CHAINS), device=env.dev)].cpu().numpy(),
            "grad_evals": np.array(grad_evals, dtype=np.float64)}


def gpu_leg(env, name, steps, warmup, chains=None, e2e=True, fp64_peak=None, dump=False):
    """Device-resident timing (+ e2e through pinned host buffers) of one workload; returns the reduced dict on
    every rank.  dump=True: out["_outputs"] = headline_outputs() of the last timed step."""
    from walnuts_b200.sampler import pinned_empty
    torch = env.torch
    spec = WORKLOADS[name]
    n = chains or spec["chains"]
    iters, mon, pkg = spec["iters"], spec["monitor"], spec["mode"] == "package"
    if spec["target"] == "diag_gauss" and n > 262144:
        # a million chains: exact draws of the target generated on the device (8.4 GB; numpy would take half a minute)
        sigma = sigma_vec()
        gen = torch.Generator(device=env.dev).manual_seed(SEED + 7919 * env.rank)
        q0 = torch.randn((n, D), dtype=torch.float64, device=env.dev, generator=gen) * torch.as_tensor(sigma, device=env.dev)
        data = {"inv_var": 1.0 / sigma ** 2}
    else:
        q0, data = make_inputs(spec, n, env.rank)
    cb = make_batch(spec, n, env.rank * n, env.local_rank, data, q0)
    del q0
    draws = torch.empty((iters, n, mon), dtype=torch.float64, device=env.dev)
    for _ in range(warmup):
        cb.run_device(iters, draws=draws)
    env.barrier()
    sampler = ClockSampler(env.local_rank).start() if env.rank == 0 else None
    kernel_ms, evals = [], 0
    for s in range(steps):
        env.flush_l2()
        cb.run_device(iters, draws=draws)
        kernel_ms.append(cb.last_kernel_ms())
        f, b = cb.last_grad_evals()
        evals += f + b
    env.barrier()
    clocks = sampler.stop() if sampler else None
    launches = steps * cb.last_launches()
    dev_ms = float(sum(kernel_ms))
    outputs = headline_outputs(env, cb, draws, (f, b)) if dump else None

    # ---- e2e: the same steps through HOST buffers, copies inside the timed region; the chains are split over two
    # handles so that the copies of one half overlap the kernel of the other -------------------------------------
    e2e_wall, e2e_evals, h2d, d2h = 0.0, 0, 0, 0
    if e2e and spec.get("e2e", True):
        state = cb.get_state()
        cb.close()
        halves = [(0, n // 2), (n // 2, n - n // 2)] if n >= 2 else [(0, n)]
        hs = []
        for off, m in halves:
            h = make_batch(spec, m, env.rank * n + off, env.local_rank, data, state[off:off + m])
            bufs = dict(q=pinned_empty((m, spec["d"])), dr=pinned_empty((iters, m, mon)),
                        dg=None if pkg else pinned_empty((iters, m, 24)),
                        f=pinned_empty((m,), np.uint64), b=None if pkg else pinned_empty((m,), np.uint64))
            bufs["q"][:] = state[off:off + m]
            hs.append((h, bufs))
        del state

        def enqueue(h, bf):
            h.run_host_async(iters, q_in=bf["q"], draws=bf["dr"], diag=bf["dg"], nevalF=bf["f"], nevalB=bf["b"],
                             q_out=bf["q"])

        def finish(h):
            h.sync()                                          # this half's results are in its host buffers now
            f, b = h.last_grad_evals()
            return f + b

        def run_steps(k):
            # handle-level software pipeline: a half is re-enqueued as soon as ITS results of the previous step have
            # arrived, while the other half's kernel is still running
            tot = 0
            for h, bf in hs:
                enqueue(h, bf)
            for s in range(1, k):
                for h, bf in hs:
                    tot += finish(h)
                    enqueue(h, bf)
            for h, bf in hs:
                tot += finish(h)
            return tot
        run_steps(1)                                          # staging buffers / scratch allocated outside the timing
        env.barrier()
        t1 = time.perf_counter()
        e2e_evals = run_steps(steps)
        env.barrier()
        e2e_wall = time.perf_counter() - t1
        for h, bf in hs:
            h2d += bf["q"].nbytes
            d2h += sum(x.nbytes for x in bf.values() if x is not None)
            h.close()
    else:
        cb.close()

    (dev_ms_max, e2e_wall_max), (evals_all, e2e_evals_all) = env.reduce([dev_ms, e2e_wall], [float(evals), float(e2e_evals)])
    value = evals_all / (dev_ms_max * 1e-3)
    per_launch_flops = spec["flop_per_eval"] * (evals / max(1, steps))
    ach = per_launch_flops / (np.mean(kernel_ms) * 1e-3) / 1e12
    out = {"workload": spec["workload"], "value": value, "unit": "grad_evals/s", "steps": steps, "warmup": warmup,
           "ms_per_step": dev_ms_max / max(1, steps), "chains_per_gpu": n, "chains_total": n * env.world,
           "iters_per_step": iters, "evals_per_transition": evals_all / (steps * iters * n * env.world),
           "gpu_launches": launches, "clocks": clocks,
           "params": {k: spec[k] for k in ("integrator", "H0", "delta", "M", "minC", "maxC", "mode")},
           "roofline": {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
                        "frac": (ach / fp64_peak) if fp64_peak else None, "flop_per_eval": spec["flop_per_eval"],
                        **_traffic(name, n, iters),
                        **({"flop_per_eval_survey": spec["flop_per_eval_survey"],
                            "achieved_at_survey_flop": ach * spec["flop_per_eval_survey"] / spec["flop_per_eval"],
                            "frac_at_survey_flop": (ach * spec["flop_per_eval_survey"] / spec["flop_per_eval"] / fp64_peak)
                            if fp64_peak else None} if "flop_per_eval_survey" in spec else {}),
                        "note": "achieved = flop_per_eval (SURVEY.md 8(d) algorithmic FP64 work per gradient evaluation; "
                                "C2/R2P: the 4 flop per coordinate the kernel executes) x evaluations of one launch / its "
                                "CUDA-event duration; peak = FP64 FMA micro-benchmark of this run (MEASURED_PEAKS.json has "
                                "no FP64 entry); register-resident chains: not HBM-bound"}}
    if e2e_wall_max > 0:
        out["e2e"] = {"value": e2e_evals_all / e2e_wall_max, "unit": "grad_evals/s", "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": d2h, "handles_per_gpu": len(halves)}
    if dump:
        out["_outputs"] = outputs
    return out


def ess_leg(env, chains=ESS_CHAINS, n_draws=ESS_DRAWS):
    """min-ESS/sec: `chains` chains per GPU x `n_draws` transitions of the headline workload in ONE launch; bulk ESS
    (rank-normalised, split chains) and split-R-hat over ALL chains of all GPUs, computed by the library on the device
    (wn_ess_rhat: one NCCL all-gather of the monitored draws, then sort / autocovariance kernels)."""
    from walnuts_b200 import comm_unique_id
    torch = env.torch
    spec = WORKLOADS["c2"]
    q0, data = make_inputs(spec, chains, env.rank)
    cb = make_batch(spec, chains, (1 << 24) + env.rank * chains, env.local_rank, data, q0)
    if env.world > 1:
        box = [comm_unique_id() if env.rank == 0 else None]
        env.dist.broadcast_object_list(box, src=0)            # 128 bytes of rendezvous, not data
        cb.comm_init_rank(env.world, env.rank, box[0])
    draws = torch.empty((n_draws, chains, MONITOR), dtype=torch.float64, device=env.dev)
    env.barrier()
    cb.run_device(n_draws, draws=draws)
    ms = cb.last_kernel_ms()
    f, b = cb.last_grad_evals()
    env.barrier()
    (ms_max,), (evals_all,) = env.reduce([ms], [float(f + b)])
    t0 = time.perf_counter()
    per, rh = cb.ess_rhat(draws)
    stat_s = time.perf_counter() - t0
    half, _ = cb.ess_rhat(draws[:n_draws // 2])
    cb.close()
    per, rh, half = [float(x) for x in per], [float(x) for x in rh], [float(x) for x in half]
    sig = sigma_vec()[:MONITOR]
    if env.rank != 0:
        return None
    k = int(np.nanargmin(per))
    total = chains * env.world * n_draws
    return {"chains_total": chains * env.world, "draws_per_chain": n_draws, "seconds": ms_max * 1e-3,
            "grad_evals": evals_all, "min_ess": per[k], "min_ess_per_sec": per[k] / (ms_max * 1e-3),
            "min_ess_per_grad_eval": per[k] / evals_all, "slowest_sigma": float(sig[k]),
            "tau_max_draws": total / per[k], "split_chain_length": n_draws // 2, "rhat_max": float(np.nanmax(rh)),
            "min_ess_first_half_of_draws": half[k],        # ESS must grow with the draws: ~ half of min_ess
            "ess_per_coordinate": per, "rhat_per_coordinate": rh, "sigma_monitored": [float(x) for x in sig],
            "statistics_seconds": stat_s,
            "estimator": "bulk ESS: rank-normalised, split chains, Geyer initial monotone sequence on chain-averaged "
                         "autocorrelations with all lags available (Vehtari et al. 2021 = arviz.ess default, "
                         "mainGaussESS.py:50-55), computed on the device by wn_ess_rhat over the chains of all GPUs "
                         "(one NCCL all-gather); chains start from exact draws of the target"}


# --------------------------------------------------------------------------------------------------
def reference_arm(args):
    """The reference's own CPU implementation of the path (numpy restatement) on all host cores, headline workload.
    Every core advances its own chain: `warmup` untimed transitions (capped at 1), then timed transitions until the
    time budget is used (at least 4, at most --steps).  One step = one transition of every core's chain; `steps` is
    the number actually executed by every core."""
    impl = "reference" if reference_available() else "port"
    cb = cpu_baseline("c2", budget=args.ref_budget, min_tr=args.ref_min_transitions,
                      max_tr=max(args.ref_min_transitions, args.steps), warm=min(1, args.warmup), impl=impl)
    try:
        extra_c = cpu_baseline_c(6.0)
    except Exception as e:
        extra_c = {"unavailable": str(e)[:200]}
    spec = WORKLOADS["c2"]
    config = {"workload": spec["workload"], "chains": cb["cores"], "d": D,
              **{k: spec[k] for k in ("integrator", "H0", "delta", "M", "minC", "maxC")}, "jitter": 0.2}
    line = {"impl": "reference", "metric": "grad_evals_per_sec", "value": cb["value"], "unit": "grad_evals/s",
            "n_gpus": args.gpus, "steps": cb["transitions_min"], "warmup": min(1, args.warmup),
            "steps_requested": args.steps, "ms_per_step": 1e3 * cb["seconds_per_transition"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config, "cpu_baseline": cb, "cpu_baseline_c": extra_c,
            "e2e": {"value": cb["value"], "unit": "grad_evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8,
                    help="timed steps of the headline workload (exactly); the config legs cap it at their steps_cap, "
                         "strong scaling at 5, and the reference arm takes it as a maximum -- each reports its own count")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chains", type=int, default=CHAINS_PER_GPU, help="headline chains per GPU")
    ap.add_argument("--configs", default="all", help="'all', 'none' or a comma list of " + ",".join(CONFIG_ORDER))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-ess", action="store_true", help="skip the min-ESS/sec leg")
    ap.add_argument("--ess-chains", type=int, default=ESS_CHAINS)
    ap.add_argument("--ess-draws", type=int, default=ESS_DRAWS)
    ap.add_argument("--ref-budget", type=float, default=60.0, help="seconds per core of the reference arm")
    ap.add_argument("--ref-min-transitions", type=int, default=4, help="timed transitions per core of the reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's outputs of its last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.steps < 1):
        ap.error("--dump-outputs needs --impl ours and --steps >= 1")

    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            reference_arm(args)
        return

    env = Env()
    from walnuts_b200 import _ffi, fp64_peak
    try:
        peak = fp64_peak(env.local_rank) / 1e12
        peak_src = "measured FP64 FMA micro-benchmark (wn_fp64_peak) on this GPU, this run"
    except Exception:
        peak, peak_src = 148 * 64 * 2 * 1.965e9 / 1e12, "nominal 148 SM x 64 FMA/clk x 1.965 GHz (fallback)"

    head = gpu_leg(env, "c2", args.steps, args.warmup, chains=args.chains, fp64_peak=peak, dump=bool(args.dump_outputs))
    if args.dump_outputs and env.rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for key, arr in head.pop("_outputs").items():
            np.save(os.path.join(args.dump_outputs, key + ".npy"), arr)
    names = CONFIG_ORDER if args.configs == "all" else ([] if args.configs == "none" else args.configs.split(","))
    configs = {}
    for name in names:
        spec = WORKLOADS[name]
        if spec.get("single_gpu_only") and env.world > 1:
            continue
        configs[name] = gpu_leg(env, name, max(1, min(args.steps, spec["steps_cap"])), min(args.warmup, spec["warmup_cap"]),
                                fp64_peak=peak)
    strong = None
    if env.world > 1:
        st = gpu_leg(env, "c2", min(args.steps, 5), min(args.warmup, 3), chains=CHAINS_PER_GPU // env.world, e2e=False,
                     fp64_peak=peak)
        strong = {k: st[k] for k in ("value", "unit", "ms_per_step", "steps", "warmup", "chains_per_gpu", "chains_total")}
        strong["note"] = "strong scaling: the headline workload with 65 536 chains in TOTAL"
    ess = None if args.no_ess else ess_leg(env, args.ess_chains, args.ess_draws)
    if env.rank != 0:
        if env.world > 1:
            env.dist.destroy_process_group()
        return

    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        hbm_peak = 6650.0
    spec = WORKLOADS["c2"]
    roof = head["roofline"]
    roof.update(peak_source=peak_src,
                hbm={"streaming_model_gbs": head["value"] / env.world * 48 * D / 1e9, "peak_gbs": hbm_peak,
                     "note": "SURVEY.md 8(d) streaming model (48 d bytes per evaluation if q, v, g went through HBM every "
                             "micro-step) vs the measured HBM peak: the chains are register-resident, HBM is not the bound"})
    line = {
        "metric": "grad_evals_per_sec", "value": head["value"], "unit": "grad_evals/s", "n_gpus": env.world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": spec["workload"], "chains_per_gpu": args.chains, "d": D, "iters_per_step": spec["iters"],
                   **{k: spec[k] for k in ("integrator", "H0", "delta", "M", "minC", "maxC")}, "jitter": 0.2,
                   "l2_policy": "a 256 MB buffer is overwritten between timed steps (2 x the 126 MB L2); the headline's "
                                "positions alone are 524 MB"},
        "evals_per_transition": head["evals_per_transition"],
        "e2e": head.get("e2e"), "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "roofline": roof,
        "min_ess_per_sec": ess["min_ess_per_sec"] if ess else None, "ess": ess,
        "configs": configs, "strong_scaling": strong, "lib": os.path.relpath(_ffi.lib_path(), ROOT),
    }
    if env.world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline("c2", budget=12.0, min_tr=1)
        budgets = {"c1": 3.0, "c2_nuts": 4.0, "c3": 4.0, "c4": 8.0, "c5": 5.0}
        for name, c in configs.items():
            if name in budgets:
                try:
                    c["cpu_baseline"] = cpu_baseline(name, budget=budgets[name], min_tr=1)
                except Exception as e:                            # a failed CPU leg must not lose the GPU numbers
                    c["cpu_baseline"] = {"unavailable": str(e)[:200]}
        try:
            line["cpu_baseline_c"] = cpu_baseline_c(20.0 if ess else 6.0, ess=bool(ess))
        except Exception as e:                                    # the C checker is optional for the bench
            line["cpu_baseline_c"] = {"unavailable": str(e)[:200]}
        if ess:
            # the CPU arm runs the identical transition kernel on identical streams (parity tests), so its ESS per
            # gradient evaluation is the GPU leg's; derived figure, next to the one measured on the C port's own draws
            line["cpu_baseline"]["min_ess_per_sec_derived"] = ess["min_ess_per_grad_eval"] * line["cpu_baseline"]["value"]
    print(json.dumps(line))
    if env.world > 1:
        env.dist.destroy_process_group()


if __name__ == "__main__":
    main()
