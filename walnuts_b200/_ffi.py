"""ctypes binding of include/walnuts_cuda.h (thin; no torch types cross this boundary)."""
import ctypes as C
import os

from . import build as _build

TARGETS = {"std_normal": 0, "diag_gauss": 1, "funnel": 2, "logreg": 3, "stock_watson": 4,
           "corr_gauss": 5, "funnel_pkg": 6, "dense_gauss": 7}
MODE_WALNUTSPY, MODE_PACKAGE = 0, 1
INT_FIXED, INT_D, INT_R2P = 0, 1, 2
DIAG_COLS = 24
FAMILIES = {"wpy": 0, "pkg": 1, "adapt": 2, "ext": 3, "nuts": 4}      # WN_FAMILY_* (wn_last_plan)
# WN_S_* columns of wn_summary, in order
SUMMARY_COLS = ("mean", "sd", "q05", "q50", "q95", "mcse_mean", "mcse_sd", "ess_bulk", "ess_tail", "rhat", "nested_rhat")
ERRORS = {-1: "WN_EINVAL", -2: "WN_ECUDA", -3: "WN_ENOMEM", -4: "WN_EUNSUPPORTED", -5: "WN_ESTATE"}

# every symbol include/walnuts_cuda.h declares
SYMBOLS = ["wn_abi_version", "wn_target_id", "wn_register_user_target", "wn_create", "wn_destroy", "wn_set_data", "wn_set_aux", "wn_set_adapt", "wn_set_state",
           "wn_get_state", "wn_run", "wn_run_stats", "wn_run_async", "wn_sync", "wn_run_host_async", "wn_alloc_pinned", "wn_free_pinned", "wn_last_kernel_ms", "wn_last_launches",
           "wn_last_plan", "wn_last_slots", "wn_last_grad_evals", "wn_moments", "wn_stream", "wn_last_error", "wn_fp64_peak",
           "wn_comm_load", "wn_comm_unique_id", "wn_comm_init_rank", "wn_comm_init_all", "wn_comm_destroy",
           "wn_ess_rhat", "wn_summary", "wn_moments_all"]


class WnConfig(C.Structure):
    _fields_ = [("target", C.c_int32), ("mode", C.c_int32), ("integrator", C.c_int32), ("d", C.c_int32),
                ("n_chains", C.c_int32), ("device", C.c_int32), ("dg", C.c_int32), ("M", C.c_int32),
                ("minC", C.c_int32), ("maxC", C.c_int32), ("compat", C.c_int32), ("first_iteration", C.c_int32),
                ("H0", C.c_double), ("jitter", C.c_double), ("delta", C.c_double),
                ("r2p_prob0", C.c_double), ("log_p0", C.c_double), ("log_1mp0", C.c_double),
                ("seed", C.c_uint64), ("chain_offset", C.c_uint64)]


class WalnutsError(RuntimeError):
    pass


_lib = None


def lib_path():
    return _build.LIB_PATH


def load():
    """Load the CUDA library; fails loudly if it has not been built (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.isfile(path):
        raise WalnutsError(f"{path} is missing: run `python -m walnuts_b200.build` (the CUDA extension "
                           "is the only implementation; there is no CPU fallback)")
    lib = C.CDLL(path)
    P = C.POINTER
    vp, dp, u64p = C.c_void_p, C.c_void_p, C.c_void_p
    lib.wn_abi_version.restype = C.c_int
    lib.wn_target_id.argtypes = [C.c_char_p]
    lib.wn_create.argtypes = [P(WnConfig), P(vp)]
    lib.wn_destroy.argtypes = [vp]
    lib.wn_destroy.restype = None
    lib.wn_set_data.argtypes = [vp, C.c_char_p, dp, C.c_int64, C.c_int]
    lib.wn_register_user_target.argtypes = [C.c_char_p]
    lib.wn_set_aux.argtypes = [vp, C.c_char_p, C.c_double]
    lib.wn_set_adapt.argtypes = [vp, C.c_int64, C.c_int, C.c_double, C.c_int, C.c_double, C.c_double]
    lib.wn_set_state.argtypes = [vp, dp, C.c_int]
    lib.wn_get_state.argtypes = [vp, dp, C.c_int]
    lib.wn_run.argtypes = [vp, C.c_int64, dp, dp, u64p, u64p, C.c_int]
    lib.wn_run_stats.argtypes = [vp, C.c_int64, dp, dp, u64p, u64p, dp, dp, C.c_int]
    lib.wn_run_async.argtypes = [vp, C.c_int64, dp, dp, u64p, u64p]
    lib.wn_sync.argtypes = [vp]
    lib.wn_run_host_async.argtypes = [vp, C.c_int64, dp, dp, dp, u64p, u64p, dp]
    lib.wn_alloc_pinned.argtypes = [C.c_int64, P(vp)]
    lib.wn_free_pinned.argtypes = [vp]
    lib.wn_last_kernel_ms.argtypes = [vp, P(C.c_float)]
    lib.wn_last_launches.argtypes = [vp, P(C.c_int64)]
    lib.wn_last_plan.argtypes = [vp, P(C.c_int32)]
    lib.wn_last_slots.argtypes = [vp, P(C.c_int64)]
    lib.wn_last_grad_evals.argtypes = [vp, P(C.c_uint64), P(C.c_uint64)]
    lib.wn_moments.argtypes = [vp, dp, dp]
    lib.wn_comm_load.argtypes = [C.c_char_p]
    lib.wn_comm_unique_id.argtypes = [vp]
    lib.wn_comm_init_rank.argtypes = [vp, C.c_int, C.c_int, vp]
    lib.wn_comm_init_all.argtypes = [P(vp), C.c_int]
    lib.wn_comm_destroy.argtypes = [vp]
    lib.wn_ess_rhat.argtypes = [vp, dp, C.c_int64, C.c_int64, C.c_int32, C.c_int, C.c_int32, dp, dp]
    lib.wn_summary.argtypes = [vp, dp, C.c_int64, C.c_int64, C.c_int32, C.c_int, C.c_int32, dp]
    lib.wn_moments_all.argtypes = [vp, dp, dp]
    lib.wn_stream.argtypes = [vp]
    lib.wn_stream.restype = vp
    lib.wn_last_error.argtypes = [vp]
    lib.wn_last_error.restype = C.c_char_p
    lib.wn_fp64_peak.argtypes = [C.c_int, P(C.c_double)]
    for name in SYMBOLS:
        getattr(lib, name)
    _lib = lib
    return lib


_user_ids = {}


def register_user_target(path):
    """Load a user-target plug-in once per process; returns its integer target id."""
    if path not in _user_ids:
        rc = load().wn_register_user_target(os.fsencode(path))
        if rc < 0:
            raise WalnutsError(f"wn_register_user_target({path}): {ERRORS.get(rc, rc)}")
        _user_ids[path] = rc
    return _user_ids[path]
