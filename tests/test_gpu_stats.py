"""Device-side convergence statistics and the multi-GPU entry points of the C-ABI (wn_stats.cu): wn_ess_rhat against the
numpy estimator of walnuts_b200/diagnostics.py, wn_run_host_async against wn_run, and -- on a box with >= 2 GPUs -- the
NCCL paths: pooled ESS / R-hat (one all-gather), wn_moments_all (all-reduce), the single-process launcher
WALNUTS(..., devices=[...]) and the multi-process communicator (wn_comm_unique_id / wn_comm_init_rank)."""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def ar1(n_iter, n_chains, rhos, seed=0):
    rng = np.random.default_rng(seed)
    x = np.empty((n_iter, n_chains, len(rhos)))
    x[0] = rng.standard_normal((n_chains, len(rhos)))
    r = np.asarray(rhos)
    for t in range(1, n_iter):
        x[t] = r * x[t - 1] + np.sqrt(1 - r * r) * rng.standard_normal((n_chains, len(rhos)))
    x[:, :, -1] = np.exp(x[:, :, -1])          # a skewed coordinate: rank normalisation matters
    return x


def n_gpus():
    import torch
    return torch.cuda.device_count()


def test_ess_rhat_matches_numpy_estimator(cuda_lib):
    from walnuts_b200 import ChainBatch, diagnostics
    x = ar1(400, 64, [0.0, 0.5, 0.9, 0.98, 0.7])
    with ChainBatch("std_normal", 5, 64, H0=0.5, delta=0.3, M=5, seed=1) as cb:
        for split in (True, False):
            ess, rhat = cb.ess_rhat(np.ascontiguousarray(x), split=split)
            for j in range(5):
                e, r = diagnostics.ess_bulk(x[:, :, j].T, split=split)
                assert abs(ess[j] - e) <= 1e-8 * e, (j, split, ess[j], e)
                assert abs(rhat[j] - r) <= 1e-10, (j, split, rhat[j], r)
        assert ess[0] > 5 * ess[3]               # the strongly autocorrelated coordinate has far fewer effective draws
        # odd length, device-resident input
        import torch
        xo = np.ascontiguousarray(x[:333])
        e1, r1 = cb.ess_rhat(xo)
        e2, r2 = cb.ess_rhat(torch.from_numpy(xo).cuda())
        assert np.array_equal(e1, e2) and np.array_equal(r1, r2)
        assert abs(e1[2] - diagnostics.ess_bulk(xo[:, :, 2].T)[0]) <= 1e-8 * e1[2]


def test_ess_rhat_of_sampler_draws(cuda_lib):
    """End to end: draws of the sampler on the device -> ESS / R-hat without leaving the GPU."""
    import torch
    from walnuts_b200 import ChainBatch, diagnostics
    n, d, it = 512, 6, 200
    q0 = np.random.default_rng(3).standard_normal((n, d))
    with ChainBatch("std_normal", d, n, integrator="R2P", H0=0.7, delta=0.3, M=6, seed=5) as cb:
        cb.set_state(q0)
        draws = torch.empty((it, n, d), dtype=torch.float64, device="cuda")
        cb.run_device(it, draws=draws)
        ess, rhat = cb.ess_rhat(draws)
    host = draws.cpu().numpy()
    for j in range(d):
        e, r = diagnostics.ess_bulk(host[:, :, j].T)
        assert abs(ess[j] - e) <= 1e-8 * e
    assert (rhat < 1.01).all() and (ess > 0.3 * n * it).all()


def test_moments_equal_moments_all_without_communicator(cuda_lib):
    """Without a communicator wn_moments_all reduces over the handle's own chains: the same bits as wn_moments, and
    numpy's mean and unbiased variance over the chains."""
    from walnuts_b200 import ChainBatch
    n, d = 1000, 37
    rng = np.random.default_rng(21)
    q = rng.standard_normal((n, d)) * np.logspace(-1, 1, d) + np.linspace(1.0, 20.0, d)
    with ChainBatch("std_normal", d, n, H0=0.5, delta=0.3, M=5, seed=1) as cb:
        cb.set_state(q)
        mean, var = cb.moments()
        mean_all, var_all = cb.moments_all()
    assert np.array_equal(mean, mean_all) and np.array_equal(var, var_all)
    assert np.all(np.abs(mean - q.mean(0)) <= 1e-12 * np.abs(q.mean(0)))
    assert np.all(np.abs(var - q.var(0, ddof=1)) <= 1e-12 * q.var(0, ddof=1))


def test_run_host_async_equals_run(cuda_lib):
    from walnuts_b200 import ChainBatch, pinned_empty
    n, d, it = 300, 9, 4
    q0 = np.random.default_rng(4).standard_normal((n, d))
    kw = dict(integrator="R2P", H0=0.6, delta=0.3, M=6, seed=8)
    with ChainBatch("std_normal", d, n, **kw) as cb:
        cb.set_state(q0)
        a = cb.run(it, draws=True, diag=True)
        qa = cb.get_state()
    with ChainBatch("std_normal", d, n, **kw) as cb:
        qin, dr, dg = pinned_empty((n, d)), pinned_empty((it, n, d)), pinned_empty((it, n, 24))
        f, b = pinned_empty((n,), np.uint64), pinned_empty((n,), np.uint64)
        qin[:] = q0
        cb.run_host_async(it, q_in=qin, draws=dr, diag=dg, nevalF=f, nevalB=b, q_out=qin)
        cb.sync()
        assert np.array_equal(dr, a["draws"]) and np.array_equal(dg, a["diag"])
        assert np.array_equal(f, a["nevalF"]) and np.array_equal(b, a["nevalB"]) and np.array_equal(qin, qa)
        with pytest.raises(Exception):
            cb.run_host_async(it, draws=np.empty((it, n, d + 1)))          # wrong size is refused before the call


def test_fixed_seed_walnuts_step_needs_distinct_iterations(cuda_lib):
    """ADVICE r1: walnuts_step with a fixed seed replayed the same streams on every call."""
    import walnuts_b200 as wb
    tg = wb.targets.standard_normal_lpdf
    th = np.full(4, 0.3)
    kw = dict(seed=77)
    a = wb.walnuts_step(None, th, tg, tg, np.ones(4), 1.0, 6, 0.2, iteration=1, **kw)
    b = wb.walnuts_step(None, th, tg, tg, np.ones(4), 1.0, 6, 0.2, iteration=1, **kw)
    c = wb.walnuts_step(None, th, tg, tg, np.ones(4), 1.0, 6, 0.2, iteration=2, **kw)
    assert np.array_equal(a, b) and not np.array_equal(a, c)
    # iteration k of walnuts_step == draw k of walnuts() with the same seed
    d2 = wb.walnuts(None, th, tg, tg, np.ones(4), 1.0, 6, 0.2, 0, 2, seed=77)
    assert np.array_equal(a, d2[0])
    assert np.array_equal(wb.walnuts_step(None, d2[0], tg, tg, np.ones(4), 1.0, 6, 0.2, iteration=2, **kw), d2[1])
    # without an explicit iteration a generator supplies it: a loop never repeats its streams
    rng = np.random.default_rng(0)
    x1 = wb.walnuts_step(rng, th, tg, tg, np.ones(4), 1.0, 6, 0.2, **kw)
    x2 = wb.walnuts_step(rng, th, tg, tg, np.ones(4), 1.0, 6, 0.2, **kw)
    assert not np.array_equal(x1, x2)


# ---- multi-GPU (skipped on a single-GPU box) -----------------------------------------------------------------------
def test_multi_gpu_single_process_comm(cuda_lib):
    if n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    from walnuts_b200 import ChainBatch, comm_init_all, diagnostics
    W = min(n_gpus(), 4)
    n, d, it = 96, 5, 120
    x = ar1(it, n * W, [0.0, 0.6, 0.9, 0.3, 0.8], seed=2)
    q = np.random.default_rng(9).standard_normal((n * W, d))
    cbs = [ChainBatch("std_normal", d, n, H0=0.5, delta=0.3, M=5, seed=1, device=k, chain_offset=k * n) for k in range(W)]
    try:
        comm_init_all(cbs)
        res = [None] * W

        def work(k):
            cbs[k].set_state(q[k * n:(k + 1) * n])
            res[k] = (cbs[k].ess_rhat(np.ascontiguousarray(x[:, k * n:(k + 1) * n])), cbs[k].moments_all())
        th = [threading.Thread(target=work, args=(k,)) for k in range(W)]
        [t.start() for t in th]
        [t.join() for t in th]
        for k in range(W):
            (ess, rhat), (mean, var) = res[k]
            assert np.array_equal(ess, res[0][0][0]) and np.array_equal(rhat, res[0][0][1])      # same on every rank
            for j in range(d):
                e, r = diagnostics.ess_bulk(x[:, :, j].T)
                assert abs(ess[j] - e) <= 1e-8 * e and abs(rhat[j] - r) <= 1e-10
            assert np.allclose(mean, q.mean(0), rtol=1e-12, atol=1e-14) and np.allclose(var, q.var(0, ddof=1), rtol=1e-12)
    finally:
        for cb in cbs:
            cb.close()


def test_multi_gpu_launcher_matches_one_gpu(cuda_lib):
    if n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    import walnuts_b200 as wb
    q0 = np.random.default_rng(5).standard_normal((37, 7))
    kw = dict(integrator=wb.adaptLeapFrogR2P, H0=0.6, delta0=0.3, numIter=25, warmupIter=0, M=6, adaptH=False,
              adaptDelta=False, seed=19)
    s1, d1 = wb.WALNUTS(wb.targets.stdGauss, q0, **kw)
    s2, d2 = wb.WALNUTS(wb.targets.stdGauss, q0, devices=list(range(min(n_gpus(), 4))), **kw)
    assert np.array_equal(s1, s2) and np.array_equal(d1, d2)        # independent of the number of GPUs
    tg = wb.targets.standard_normal_lpdf
    a = wb.walnuts(None, q0, tg, tg, np.ones(7), 1.0, 6, 0.2, 0, 5, seed=3)
    b = wb.walnuts(None, q0, tg, tg, np.ones(7), 1.0, 6, 0.2, 0, 5, seed=3, devices=[0, 1])
    assert np.array_equal(a, b)


def _rank_main(rank, world, uid_q, out_q):
    import numpy as np
    from walnuts_b200 import ChainBatch, comm_unique_id
    if rank == 0:
        uid = comm_unique_id()
        for _ in range(world - 1):
            uid_q.put(uid)
    else:
        uid = uid_q.get()
    n, d, it = 40, 3, 60
    x = ar1(it, n * world, [0.2, 0.8, 0.5], seed=6)
    with ChainBatch("std_normal", d, n, H0=0.5, delta=0.3, M=5, seed=1, device=rank, chain_offset=rank * n) as cb:
        cb.comm_init_rank(world, rank, uid)
        ess, rhat = cb.ess_rhat(np.ascontiguousarray(x[:, rank * n:(rank + 1) * n]))
    out_q.put((rank, ess, rhat))


def test_multi_gpu_multi_process_comm(cuda_lib):
    if n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    import multiprocessing as mp
    from walnuts_b200 import diagnostics
    ctx = mp.get_context("spawn")
    uid_q, out_q = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, uid_q, out_q)) for r in range(2)]
    [p.start() for p in procs]
    got = [out_q.get(timeout=300) for _ in procs]
    [p.join(60) for p in procs]
    x = ar1(60, 80, [0.2, 0.8, 0.5], seed=6)
    for rank, ess, rhat in got:
        for j in range(3):
            e, r = diagnostics.ess_bulk(x[:, :, j].T)
            assert abs(ess[j] - e) <= 1e-8 * e and abs(rhat[j] - r) <= 1e-10


def test_devices_argument_single_gpu(cuda_lib):
    """`devices=[0]` is the plain call; the sharding helper splits chains contiguously with global chain ids."""
    import walnuts_b200 as wb
    from walnuts_b200.api import _over_devices
    q0 = np.random.default_rng(5).standard_normal((9, 5))
    kw = dict(integrator=wb.adaptLeapFrogD, H0=0.6, delta0=0.3, numIter=10, warmupIter=0, M=5, adaptH=False,
              adaptDelta=False, seed=4)
    s1, d1 = wb.WALNUTS(wb.targets.stdGauss, q0, **kw)
    s2, d2 = wb.WALNUTS(wb.targets.stdGauss, q0, devices=[0], **kw)
    assert np.array_equal(s1, s2) and np.array_equal(d1, d2)
    # the same GPU used as two "devices": shards of 5 + 4 chains with chain offsets 0 and 5 reproduce the single call
    parts = _over_devices(lambda xs, dev, off: wb.WALNUTS(wb.targets.stdGauss, xs, device=0, chain_offset=off, **kw),
                          q0, [0, 0], 0)
    assert np.array_equal(np.concatenate([p[0] for p in parts]), s1)


def test_d4096_single_cta_chain(cuda_lib):
    """d = 4096 (one 16-warp CTA per chain): free-running parity with the C oracle for the three integrators."""
    from oracle import c_oracle
    from tests.helpers import close
    from walnuts_b200 import ChainBatch
    d = 4096
    rng = np.random.default_rng(8)
    sigma = np.exp(rng.uniform(-1.0, 1.0, d))
    q0 = rng.standard_normal((3, d)) * sigma
    iv = 1.0 / sigma ** 2
    for integ, H0 in (("fixed", 0.05), ("D", 0.25), ("R2P", 0.25)):
        with ChainBatch("diag_gauss", d, 3, integrator=integ, H0=H0, delta=0.3, M=6, seed=11, data={"inv_var": iv}) as cb:
            cb.set_state(q0)
            out = cb.run(8, draws=True, diag=True)
        for c in (0, 2):
            dr, dg, ne = c_oracle.run_chain("diag_gauss", integ, q0[c], H0, 0.3, 6, 8, 11, c, inv_var=iv)
            ok, err = close(out["draws"][:, c], dr, scale=sigma)
            assert ok, (integ, err)
            assert np.array_equal(out["diag"][:, c][:, [0, 1, 6, 7, 19]], dg[:, [0, 1, 6, 7, 19]])


@pytest.mark.parametrize("mode", ["walnutspy", "package"])
def test_longest_first_queue_order_is_a_hint_only(cuda_lib, mode):
    """wn_sched.cu: from the second call on a handle the chain queue is served in descending order of the previous
    call's evaluation counts.  More chains than resident slots, three calls of three transitions against ONE call of
    nine (which has no history, hence the natural order): bit-identical draws, counters and final states."""
    from walnuts_b200 import ChainBatch
    # more chains than resident chain slots (walnutspy: 148 SMs x 5 blocks x 16 chains; package mode, one thread per
    # chain: up to 148 x 4 x 128)
    n, d = (40000 if mode == "walnutspy" else 100000), 11
    rng = np.random.default_rng(12)
    q0 = rng.standard_normal((n, d))
    q0[:, 0] *= 3.0
    q0[:, 1:] *= np.exp(0.5 * q0[:, :1])
    if mode == "walnutspy":
        kw = dict(integrator="R2P", H0=0.3, delta=0.3, M=8, seed=5)
    else:
        kw = dict(mode="package", H0=0.5, delta=0.3, M=6, seed=5, data={"inv_mass": np.ones(d)})
    target = "funnel" if mode == "walnutspy" else "funnel_pkg"
    with ChainBatch(target, d, n, **kw) as cb:
        cb.set_state(q0)
        whole = cb.run(9, draws=True)
        q_whole = cb.get_state()
    with ChainBatch(target, d, n, **kw) as cb:
        cb.set_state(q0)
        parts = [cb.run(3, draws=True) for _ in range(3)]
        q_parts = cb.get_state()
    assert np.array_equal(np.concatenate([p["draws"] for p in parts]), whole["draws"])
    assert np.array_equal(sum(p["nevalF"] for p in parts), whole["nevalF"])
    assert np.array_equal(q_parts, q_whole)
    assert len(np.unique(parts[0]["nevalF"])) > 10          # the costs do differ between chains: the order is not trivial
