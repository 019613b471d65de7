"""The device posterior summary (wn_summary / ChainBatch.summary) against the host statement diagnostics.summary, its
bulk columns against wn_ess_rhat bit for bit, its determinism, nested R-hat on sampler draws, and -- on a box with
>= 2 GPUs -- the pooled multi-GPU results against one GPU over the concatenated draws."""
import math
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

COLS = ("mean", "sd", "q05", "q50", "q95", "mcse_mean", "mcse_sd", "ess_bulk", "ess_tail", "rhat", "nested_rhat")


def n_gpus():
    import torch
    return torch.cuda.device_count()


def draws3(n_iter, n_chains, seed):
    """[n_iter, n_chains, 3] tie-free draws: an AR(1) coordinate with an offset, one whose chains differ in scale only
    (the folded R-hat is the larger one there) and a skewed one."""
    rng = np.random.default_rng(seed)
    x = np.empty((n_iter, n_chains, 3))
    x[0] = rng.standard_normal((n_chains, 3))
    for t in range(1, n_iter):
        x[t] = 0.7 * x[t - 1] + math.sqrt(1 - 0.49) * rng.standard_normal((n_chains, 3))
    x[:, :, 0] += 2.0
    x[:, :, 1] *= np.where(np.arange(n_chains) % 2 == 0, 1.0, 3.0)
    x[:, :, 2] = np.exp(x[:, :, 2]) + 0.5
    return np.ascontiguousarray(x)


def assert_close(dev, host, where):
    for k in COLS:
        a, b = dev[k], host[k]
        if math.isnan(b):
            assert math.isnan(a), (where, k, a)
        else:
            assert abs(a - b) <= 1e-8 * abs(b), (where, k, a, b)


def batch(dg, **kw):
    from walnuts_b200 import ChainBatch
    return ChainBatch("std_normal", dg, 1, H0=0.5, delta=0.3, M=5, seed=1, **kw)


@pytest.mark.parametrize("n_iter,n_chains,s", [(64, 1, None), (101, 16, 4), (200, 64, 16), (57, 32, 1), (20, 256, 16)])
def test_summary_matches_host(cuda_lib, n_iter, n_chains, s):
    from walnuts_b200 import diagnostics
    x = draws3(n_iter, n_chains, seed=n_iter + n_chains)
    with batch(3) as cb:
        r = cb.summary(x, s)
        ess, rhat = cb.ess_rhat(x)
    for j in range(3):
        host = diagnostics.summary(x[:, :, j].T, s)
        assert_close({k: r[k][j] for k in COLS}, host, (n_iter, n_chains, s, j))
    assert np.array_equal(r["ess_bulk"], ess)                           # wn_ess_rhat's own bits
    assert (r["rhat"] >= rhat).all()
    for j in range(3):
        if r["rhat"][j] != rhat[j]:                                    # the folded R-hat is the larger one
            folded = diagnostics.ess_bulk(np.abs(x[:, :, j].T - r["q50"][j]))[1]
            assert abs(r["rhat"][j] - folded) <= 1e-8 * folded
    if n_chains > 1:
        assert r["rhat"][1] > rhat[1] > 0                             # chains of different scale: the folded R-hat


def test_summary_torch_input_and_repeated_calls_are_identical(cuda_lib):
    import torch
    x = draws3(333, 40, seed=3)
    with batch(3) as cb:
        a = cb.summary(x, 8)
        b = cb.summary(torch.from_numpy(x).cuda(), 8)
        c = cb.summary(x, 8)
    for k in COLS:
        assert np.array_equal(a[k], b[k]) and np.array_equal(a[k], c[k]), k


def test_constant_columns_and_bad_arguments(cuda_lib):
    from walnuts_b200 import diagnostics
    x = draws3(40, 8, seed=4)
    x[:, :, 1] = 2.5
    with batch(3) as cb:
        r = cb.summary(x, 2)
        host = diagnostics.summary(x[:, :, 1].T, 2)
        assert_close({k: r[k][1] for k in COLS}, host, "constant")
        for k in ("mcse_mean", "mcse_sd", "ess_tail", "nested_rhat"):
            assert math.isnan(r[k][1]), k
        assert r["sd"][1] == 0.0 and r["q05"][1] == r["q95"][1] == 2.5
        assert not np.isnan(r["nested_rhat"][[0, 2]]).any()
        for s in (3, 8, 16, -1):                                         # not a divisor / one superchain / negative
            with pytest.raises(ValueError, match="wn_summary"):
                cb.summary(x, s)
        with pytest.raises(ValueError, match="wn_summary"):
            cb.summary(np.ascontiguousarray(x[:3]))                      # fewer than 4 draws
        lib = cuda_lib
        import ctypes as C
        out = np.empty((3, 11))
        rc = lib.wn_summary(cb._h, C.c_void_p(x.ctypes.data), 40, 8, 3, 0, 3, C.c_void_p(out.ctypes.data))
        assert rc == -1                                                  # WN_EINVAL
        assert lib.wn_summary(cb._h, None, 40, 8, 3, 0, 0, C.c_void_p(out.ctypes.data)) == -1


def funnel_draws(n_iter, K=256, s=16, seed=5):
    """funnel10, K superchains of s chains; superchain k starts all its chains at one atypical point of its own."""
    import torch
    from walnuts_b200 import ChainBatch
    d = 11
    rng = np.random.default_rng(7)
    starts = np.empty((K, d))
    starts[:, 0] = rng.uniform(-2.0, 4.0, K)
    starts[:, 1:] = rng.standard_normal((K, d - 1)) * 4 * np.exp(starts[:, :1] / 2)
    q0 = np.repeat(starts, s, 0)                                         # the superchain recipe
    cb = ChainBatch("funnel", d, K * s, integrator="R2P", H0=0.3, delta=0.3, M=8, seed=seed)
    cb.set_state(q0)
    draws = torch.empty((n_iter, K * s, d), dtype=torch.float64, device="cuda")
    cb.run_device(n_iter, draws=draws)
    return cb, draws


def test_nested_rhat_of_funnel_superchains(cuda_lib):
    """4096 chains in 256 superchains of 16: nested R-hat sees the common starting points after 5 transitions and has
    forgotten them after 200 (host calibration with the C oracle on the same starts: >= 1.10 / <= 1.02)."""
    from walnuts_b200 import diagnostics
    cb, draws = funnel_draws(200)
    with cb:
        early = cb.summary(draws[:5].contiguous(), 16)
        late = cb.summary(draws, 16)
    print("nested R-hat after 5:", np.round(early["nested_rhat"], 3), "after 200:", np.round(late["nested_rhat"], 3))
    assert (early["nested_rhat"] > 1.05).all()
    assert (late["nested_rhat"] < 1.05).all()
    host = draws.cpu().numpy()
    for j in (0, 1):                                                   # sampler draws repeat states: ties
        assert_close({k: late[k][j] for k in COLS}, diagnostics.summary(host[:, :, j].T, 16), ("funnel", j))


def test_summary_of_package_mode_walnuts(cuda_lib):
    import walnuts_b200 as wb
    from walnuts_b200 import diagnostics
    K, s, d = 64, 8, 4
    th = np.repeat(np.random.default_rng(8).standard_normal((K, d)) * 4.0, s, 0)
    tg = wb.targets.standard_normal_lpdf
    out = wb.walnuts(None, th, tg, tg, np.ones(d), 0.8, 6, 0.3, 0, 100, seed=9)       # (chains, iter, d)
    x = np.ascontiguousarray(np.transpose(out, (1, 0, 2)))
    with batch(d) as cb:
        r = cb.summary(x, s)
    for j in range(d):
        assert_close({k: r[k][j] for k in COLS}, diagnostics.summary(x[:, :, j].T, s), ("package", j))
    assert (r["nested_rhat"] < 1.05).all() and (np.abs(r["mean"]) < 0.2).all()


# ---- multi-GPU (skipped on a single-GPU box) -----------------------------------------------------------------------
def test_multi_gpu_single_process_summary(cuda_lib):
    if n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    from walnuts_b200 import ChainBatch, comm_init_all
    W = 4 if n_gpus() >= 4 else 2
    n, it, s = 12, 60, 8                                                 # superchains of 8 straddle the shards of 12
    x = draws3(it, n * W, seed=11)
    with batch(3) as cb:
        ref = cb.summary(x, s)
    cbs = [ChainBatch("std_normal", 3, n, H0=0.5, delta=0.3, M=5, seed=1, device=k, chain_offset=k * n) for k in range(W)]
    try:
        comm_init_all(cbs)
        res = [None] * W

        def work(k):
            res[k] = cbs[k].summary(np.ascontiguousarray(x[:, k * n:(k + 1) * n]), s)
        th = [threading.Thread(target=work, args=(k,)) for k in range(W)]
        [t.start() for t in th]
        [t.join() for t in th]
        for k in range(W):
            for c in COLS:
                assert np.array_equal(res[k][c], ref[c], equal_nan=True), (k, c)
    finally:
        for cb in cbs:
            cb.close()


def _rank_main(rank, world, uid_q, out_q):
    import numpy as np
    from walnuts_b200 import ChainBatch, comm_unique_id
    if rank == 0:
        uid = comm_unique_id()
        for _ in range(world - 1):
            uid_q.put(uid)
    else:
        uid = uid_q.get()
    n = 12
    x = draws3(60, n * world, seed=12)
    with ChainBatch("std_normal", 3, n, H0=0.5, delta=0.3, M=5, seed=1, device=rank, chain_offset=rank * n) as cb:
        cb.comm_init_rank(world, rank, uid)
        r = cb.summary(np.ascontiguousarray(x[:, rank * n:(rank + 1) * n]), 8)
    out_q.put((rank, r))


def test_multi_gpu_multi_process_summary(cuda_lib):
    if n_gpus() < 2:
        pytest.skip("needs >= 2 GPUs")
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    uid_q, out_q = ctx.Queue(), ctx.Queue()
    procs = [ctx.Process(target=_rank_main, args=(r, 2, uid_q, out_q)) for r in range(2)]
    [p.start() for p in procs]
    got = [out_q.get(timeout=300) for _ in procs]
    [p.join(60) for p in procs]
    with batch(3) as cb:
        ref = cb.summary(draws3(60, 24, seed=12), 8)
    for rank, r in got:
        for c in COLS:
            assert np.array_equal(r[c], ref[c], equal_nan=True), (rank, c)
