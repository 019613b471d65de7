"""Low-level host wrapper over the C-ABI: one `ChainBatch` = one handle = the chains of one GPU.

numpy arrays are the default I/O; torch CUDA tensors are accepted as optional device-resident I/O
(their data pointers are passed straight through; torch is not imported unless one is given).
Every buffer handed to the library is checked for dtype, contiguity and exact size first: the C-ABI takes raw
pointers and trusts them.
"""
import ctypes as C
import math
import weakref

import numpy as np

from . import _ffi
from . import integrators as _ig
from ._ffi import WalnutsError


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x, numel=None, kind="f8", what="buffer"):
    """(pointer, on_device) of a float64 / uint64 buffer after checking dtype, contiguity and element count."""
    if x is None:
        return None, 0
    if _is_torch(x):
        if not x.is_cuda or not x.is_contiguous():
            raise WalnutsError(f"{what}: torch tensors passed to walnuts_b200 must be contiguous CUDA tensors")
        name = str(x.dtype)
        ok = name == "torch.float64" if kind == "f8" else name in ("torch.uint64", "torch.int64")
        if not ok:
            raise WalnutsError(f"{what}: expected {'float64' if kind == 'f8' else 'uint64/int64'}, got {name}")
        if numel is not None and x.numel() != numel:
            raise WalnutsError(f"{what}: expected {numel} elements, got {x.numel()}")
        return C.c_void_p(x.data_ptr()), 1
    if not isinstance(x, np.ndarray):
        raise WalnutsError(f"{what}: expected a numpy array or a torch CUDA tensor")
    ok = x.dtype == np.float64 if kind == "f8" else x.dtype in (np.uint64, np.int64)
    if not ok:
        raise WalnutsError(f"{what}: expected {'float64' if kind == 'f8' else 'uint64/int64'}, got {x.dtype}")
    if not x.flags.c_contiguous:
        raise WalnutsError(f"{what}: numpy buffers must be C-contiguous")
    if numel is not None and x.size != numel:
        raise WalnutsError(f"{what}: expected {numel} elements, got {x.size}")
    return C.c_void_p(x.ctypes.data), 0


def pinned_empty(shape, dtype=np.float64):
    """numpy array over page-locked host memory (wn_alloc_pinned): copies through wn_run_host_async are then
    truly asynchronous.  The memory is released when the array (and every view of it) is gone."""
    lib = _ffi.load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    rc = lib.wn_alloc_pinned(max(n, 1), C.byref(p))
    if rc != 0:
        raise WalnutsError(f"wn_alloc_pinned({n}): {_ffi.ERRORS.get(rc, rc)}")
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    weakref.finalize(buf, lib.wn_free_pinned, p)
    return arr


class ChainBatch:
    """All chains of one device.  Mirrors wn_create / wn_set_data / wn_set_state / wn_run."""

    def __init__(self, target, d, n_chains, mode="walnutspy", integrator="fixed", H0=0.2, jitter=0.2,
                 delta=0.05, M=10, minC=0, maxC=10, r2p_prob0=2.0 / 3.0, seed=0, chain_offset=0,
                 device=0, dg=None, compat=True, data=None, first_iteration=1):
        self._lib = _ffi.load()
        self._h = C.c_void_p()
        cfg = _ffi.WnConfig()
        cfg.target = _ffi.TARGETS[target] if isinstance(target, str) else int(target)
        cfg.mode = {"walnutspy": _ffi.MODE_WALNUTSPY, "package": _ffi.MODE_PACKAGE}[mode]
        cfg.integrator = _ig.KINDS[integrator] if isinstance(integrator, str) else int(integrator)
        cfg.d, cfg.n_chains, cfg.device = int(d), int(n_chains), int(device)
        cfg.dg = int(d if dg is None else dg)
        cfg.M, cfg.minC, cfg.maxC = int(M), int(minC), int(maxC)
        cfg.compat = int(bool(compat))
        cfg.first_iteration = int(first_iteration)
        cfg.H0, cfg.jitter, cfg.delta = float(H0), float(jitter), float(delta)
        cfg.r2p_prob0 = float(r2p_prob0)
        # logs computed by the host libm exactly as the reference does (adaptiveIntegrators.py:433,437)
        cfg.log_p0 = float(np.log(r2p_prob0)) if 0 < r2p_prob0 else -math.inf
        cfg.log_1mp0 = float(np.log(1.0 - r2p_prob0)) if r2p_prob0 < 1 else -math.inf
        cfg.seed, cfg.chain_offset = int(seed), int(chain_offset)
        self.cfg = cfg
        self.d, self.n_chains, self.dg = cfg.d, cfg.n_chains, cfg.dg
        rc = self._lib.wn_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            msg = self._err()
            self.close()
            if rc == -1:
                raise ValueError(msg)       # the reference raises ValueError (walnuts.py:309-320)
            raise WalnutsError(f"wn_create: {_ffi.ERRORS.get(rc, rc)}: {msg}")
        for k, val in (data or {}).items():
            self.set_data(k, val)

    # -- plumbing ---------------------------------------------------------------------------
    def _err(self):
        return self._lib.wn_last_error(self._h).decode() if self._h else "no handle"

    def _check(self, rc, what):
        if rc != 0:
            msg = self._err()
            if rc == -1:
                raise ValueError(f"{what}: {msg}")
            raise WalnutsError(f"{what}: {_ffi.ERRORS.get(rc, rc)}: {msg}")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.wn_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- data / state -----------------------------------------------------------------------
    def set_data(self, key, arr):
        if not _is_torch(arr):
            arr = np.ascontiguousarray(arr, dtype=np.float64)
            n = arr.size
        else:
            n = arr.numel()
        p, dev = _ptr(arr, what=f"set_data({key})")
        self._check(self._lib.wn_set_data(self._h, key.encode(), p, n, dev), f"wn_set_data({key})")

    def set_aux(self, maxFPiter=None, FPtol=None, rescaledGradThresh=None):
        """integratorAuxPar fields of adaptImplicitMidpointD / adaptRescaledLeapFrogD (adaptiveIntegrators.py:36-44)."""
        for k, val in (("maxFPiter", maxFPiter), ("FPtol", FPtol), ("rescaledGradThresh", rescaledGradThresh)):
            if val is not None:
                self._check(self._lib.wn_set_aux(self._h, k.encode(), float(val)), f"wn_set_aux({k})")

    def set_adapt(self, warmup_iter, adaptH=True, adaptHtarget=0.8, adaptDelta=True, adaptDeltaTarget=0.6,
                  adaptDeltaQuantile=0.9):
        """Warm-up adaptation of H and delta per chain (WALNUTS.py:136-147, 701-712)."""
        rc = self._lib.wn_set_adapt(self._h, int(warmup_iter), int(bool(adaptH)), float(adaptHtarget),
                                    int(bool(adaptDelta)), float(adaptDeltaTarget), float(adaptDeltaQuantile))
        self._check(rc, "wn_set_adapt")

    def set_state(self, q):
        if not _is_torch(q):
            q = np.ascontiguousarray(np.broadcast_to(np.asarray(q, dtype=np.float64), (self.n_chains, self.d)))
        p, dev = _ptr(q, self.n_chains * self.d, what="set_state")
        self._check(self._lib.wn_set_state(self._h, p, dev), "wn_set_state")

    def get_state(self, out=None):
        if out is None:
            out = np.empty((self.n_chains, self.d))
        p, dev = _ptr(out, self.n_chains * self.d, what="get_state(out)")
        self._check(self._lib.wn_get_state(self._h, p, dev), "wn_get_state")
        return out

    # -- sampling ---------------------------------------------------------------------------
    def run(self, n_iter, draws=True, diag=False, nevals=True, orbit_stats=False):
        """Host-buffer path (H2D/D2H inside): returns dict(draws, diag, nevalF, nevalB[, orbit_min, orbit_max])."""
        n_iter = int(n_iter)
        out = {}
        d_arr = np.empty((n_iter, self.n_chains, self.dg)) if draws and self.dg > 0 else None
        g_arr = np.empty((n_iter, self.n_chains, _ffi.DIAG_COLS)) if diag else None
        f_arr = np.zeros(self.n_chains, dtype=np.uint64) if nevals else None
        b_arr = np.zeros(self.n_chains, dtype=np.uint64) if nevals else None
        lo = np.empty((n_iter, self.n_chains, self.dg)) if orbit_stats else None
        hi = np.empty((n_iter, self.n_chains, self.dg)) if orbit_stats else None
        rc = self._lib.wn_run_stats(self._h, n_iter, _ptr(d_arr)[0], _ptr(g_arr)[0], _ptr(f_arr, kind="u8")[0],
                                    _ptr(b_arr, kind="u8")[0], _ptr(lo)[0], _ptr(hi)[0], 0)
        self._check(rc, "wn_run")
        out.update(draws=d_arr, diag=g_arr, nevalF=f_arr, nevalB=b_arr, orbit_min=lo, orbit_max=hi)
        return out

    def _out_ptrs(self, n_iter, draws, diag, nevalF, nevalB, want_device):
        n, k = int(n_iter) * self.n_chains, self.n_chains
        bufs = ((draws, n * self.dg, "f8", "draws"), (diag, n * _ffi.DIAG_COLS, "f8", "diag"),
                (nevalF, k, "u8", "nevalF"), (nevalB, k, "u8", "nevalB"))
        ptrs = []
        for x, numel, kind, what in bufs:
            p, dev = _ptr(x, numel, kind, what)
            if x is not None and dev != want_device:
                raise WalnutsError(f"{what}: expected a {'torch CUDA tensor' if want_device else 'host numpy array'}")
            ptrs.append(p)
        return ptrs

    def run_device(self, n_iter, draws=None, diag=None, nevalF=None, nevalB=None, sync=True):
        """Device-buffer path: torch CUDA tensors (or None) of shapes (n_iter, n_chains, dg), (n_iter, n_chains, 24),
        (n_chains,), (n_chains,) are filled in place."""
        ptrs = self._out_ptrs(n_iter, draws, diag, nevalF, nevalB, 1)
        self._check(self._lib.wn_run_async(self._h, int(n_iter), *ptrs), "wn_run_async")
        if sync:
            self.sync()

    def run_host_async(self, n_iter, q_in=None, draws=None, diag=None, nevalF=None, nevalB=None, q_out=None):
        """The whole step on HOST buffers, enqueued on the handle's stream (wn_run_host_async): positions in,
        n_iter transitions, draws / diag / nevals / positions out.  Use `pinned_empty` buffers and two handles per
        device to overlap the copies of one with the kernel of the other; finish with sync()."""
        ptrs = self._out_ptrs(n_iter, draws, diag, nevalF, nevalB, 0)
        pin, d0 = _ptr(q_in, self.n_chains * self.d, what="q_in")
        pout, d1 = _ptr(q_out, self.n_chains * self.d, what="q_out")
        if d0 or d1:
            raise WalnutsError("run_host_async takes host buffers")
        self._check(self._lib.wn_run_host_async(self._h, int(n_iter), pin, *ptrs, pout), "wn_run_host_async")

    def sync(self):
        self._check(self._lib.wn_sync(self._h), "wn_sync")

    def last_kernel_ms(self):
        ms = C.c_float()
        self._check(self._lib.wn_last_kernel_ms(self._h, C.byref(ms)), "wn_last_kernel_ms")
        return float(ms.value)

    def last_launches(self):
        n = C.c_int64()
        self._check(self._lib.wn_last_launches(self._h, C.byref(n)), "wn_last_launches")
        return int(n.value)

    def last_plan(self):
        """(family, G, E2, NT) of the last run: the kernel family (_ffi.FAMILIES), threads per chain, coordinate pairs
        per thread and threads per block; family -1 before the first run.  G > NT: each chain runs on a thread-block
        cluster of G / NT blocks."""
        out = (C.c_int32 * 4)()
        self._check(self._lib.wn_last_plan(self._h, out), "wn_last_plan")
        return tuple(int(x) for x in out)

    def last_slots(self):
        """Chain slots of the last run: chain groups resident at once (clusters when G > NT), at most n_chains."""
        n = C.c_int64()
        self._check(self._lib.wn_last_slots(self._h, C.byref(n)), "wn_last_slots")
        return int(n.value)

    def last_grad_evals(self):
        f, b = C.c_uint64(), C.c_uint64()
        self._check(self._lib.wn_last_grad_evals(self._h, C.byref(f), C.byref(b)), "wn_last_grad_evals")
        return int(f.value), int(b.value)

    def moments(self, mean=None, var=None):
        mean = np.empty(self.d) if mean is None else mean
        var = np.empty(self.d) if var is None else var
        pm, d0 = _ptr(mean, self.d, what="moments(mean)")
        pv, d1 = _ptr(var, self.d, what="moments(var)")
        if d0 or d1:
            raise WalnutsError("moments() fills host arrays")
        self._check(self._lib.wn_moments(self._h, pm, pv), "wn_moments")
        return mean, var

    # -- cross-GPU statistics (NCCL inside the library) -------------------------------------------
    def comm_init_rank(self, nranks, rank, unique_id):
        """Join the NCCL communicator of a multi-process run (one rank per GPU); `unique_id` = the 128 bytes that
        rank 0 obtained from comm_unique_id() and shipped to every rank."""
        buf = (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        self._check(self._lib.wn_comm_init_rank(self._h, int(nranks), int(rank), buf), "wn_comm_init_rank")

    def ess_rhat(self, draws, split=True):
        """(ess [dg], rhat [dg]): bulk ESS and split-R-hat of draws (n_iter, n_chains, dg) -- numpy or a torch CUDA
        tensor -- computed on the device; pooled over all ranks when a communicator is attached (one all-gather)."""
        n_iter, n_chains, dg = (int(x) for x in draws.shape)
        p, dev = _ptr(draws, n_iter * n_chains * dg, what="ess_rhat(draws)")
        ess, rhat = np.empty(dg), np.empty(dg)
        rc = self._lib.wn_ess_rhat(self._h, p, n_iter, n_chains, dg, dev, int(bool(split)), _ptr(ess)[0], _ptr(rhat)[0])
        self._check(rc, "wn_ess_rhat")
        return ess, rhat

    def summary(self, draws, superchain_size=None):
        """Posterior summary of draws (n_iter, n_chains, dg) -- numpy or a torch CUDA tensor -- computed on the device:
        a dict of [dg] arrays keyed mean, sd, q05, q50, q95, mcse_mean, mcse_sd, ess_bulk, ess_tail, rhat, nested_rhat
        (definitions: include/walnuts_cuda.h at wn_summary; diagnostics.summary is the same on the host).  Pooled over
        all ranks when a communicator is attached (one all-gather; global chain order is rank-major).
        `superchain_size` = s: global chains k*s ... k*s + s - 1 form superchain k (start them from one point: repeat
        each initial point s times in q0) and nested_rhat is computed; None leaves that column NaN.  ValueError if the
        chains of all ranks do not form at least 2 superchains of s."""
        n_iter, n_chains, dg = (int(x) for x in draws.shape)
        p, dev = _ptr(draws, n_iter * n_chains * dg, what="summary(draws)")
        out = np.empty((dg, len(_ffi.SUMMARY_COLS)))
        rc = self._lib.wn_summary(self._h, p, n_iter, n_chains, dg, dev, int(superchain_size or 0), _ptr(out)[0])
        self._check(rc, "wn_summary")
        return {k: np.ascontiguousarray(out[:, i]) for i, k in enumerate(_ffi.SUMMARY_COLS)}

    def moments_all(self):
        """moments() over the chains of every rank of the communicator."""
        mean, var = np.empty(self.d), np.empty(self.d)
        self._check(self._lib.wn_moments_all(self._h, _ptr(mean)[0], _ptr(var)[0]), "wn_moments_all")
        return mean, var

    @property
    def stream(self):
        return self._lib.wn_stream(self._h)


def comm_unique_id():
    """128-byte NCCL unique id (rank 0 of a multi-process run creates it and ships it to the other ranks)."""
    buf = (C.c_char * 128)()
    rc = _ffi.load().wn_comm_unique_id(buf)
    if rc != 0:
        raise WalnutsError(f"wn_comm_unique_id: {_ffi.ERRORS.get(rc, rc)} (is libnccl.so.2 available?)")
    return bytes(buf)


def comm_init_all(batches):
    """One process driving several GPUs: attach a communicator to one ChainBatch per device."""
    arr = (C.c_void_p * len(batches))(*[b._h for b in batches])
    rc = _ffi.load().wn_comm_init_all(arr, len(batches))
    if rc != 0:
        raise WalnutsError(f"wn_comm_init_all: {_ffi.ERRORS.get(rc, rc)}: {batches[0]._err()}")


def fp64_peak(device=0):
    lib = _ffi.load()
    v = C.c_double()
    rc = lib.wn_fp64_peak(int(device), C.byref(v))
    if rc != 0:
        raise WalnutsError(f"wn_fp64_peak: {_ffi.ERRORS.get(rc, rc)}")
    return float(v.value)
