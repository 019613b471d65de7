"""Host-side checks of the parallel user-target protocol (cuda_target(..., parallel=True)); no GPU needed: the
plug-ins are compiled for sm_100a and their plan entry points are called through ctypes without a device."""
import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import pytest

DIAG_SRC = """
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
FAM_PKG, FAM_EXT = 1, 3

# (d, G, E2, NT): the plan table at every boundary
TABLE = [(1, 32, 4, 128), (256, 32, 4, 128), (257, 32, 8, 128), (512, 32, 8, 128), (513, 64, 8, 64),
         (1024, 64, 8, 64), (1025, 256, 4, 256), (2048, 256, 4, 256), (2049, 512, 4, 512), (4096, 512, 4, 512)]


def _nvcc_ok():
    from walnuts_b200 import build
    try:
        subprocess.run([os.environ.get("NVCC", "nvcc"), "--version"], capture_output=True, check=True)
    except (OSError, subprocess.CalledProcessError):
        return False
    return os.path.isdir(os.path.join(build.HERE, "csrc"))


pytestmark = pytest.mark.skipif(not _nvcc_ok(), reason="needs nvcc")


def _plan(path, family):
    lib = C.CDLL(path)
    lib.wn_user_smem_total.restype = C.c_size_t
    G, E2, NT, pkg = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    smem = C.c_size_t()
    assert lib.wn_user_plan(family, C.byref(G), C.byref(E2), C.byref(NT), C.byref(smem), C.byref(pkg)) == 0
    return (G.value, E2.value, NT.value), smem.value, pkg.value, lib.wn_user_smem_total(family), lib.wn_user_dim()


def test_parallel_plan_table():
    from walnuts_b200 import targets
    with ThreadPoolExecutor(max_workers=min(len(TABLE), os.cpu_count() or 1)) as ex:
        tgs = list(ex.map(lambda r: targets.cuda_target(DIAG_SRC, r[0], name="plan_check", parallel=True), TABLE))
    for (d, G, E2, NT), tg in zip(TABLE, tgs):
        assert targets.parallel_plan(d) == (G, E2, NT)
        totals = []
        for fam, is_pkg in ((FAM_EXT, 0), (FAM_PKG, 1)):
            shape, smem, pkg, total, dim = _plan(tg.plugin, fam)
            assert (shape, pkg, dim) == ((G, E2, NT), is_pkg, d), (d, fam, shape, pkg, dim)
            # dynamic: checkpoint, reduction scratch, and per chain a q row, a g row (2 G E2 doubles each)
            assert smem == 8 * (3 * 2 * E2 * NT + 2 * ((G + 31) // 32) * 8 + (NT // G) * 2 * 2 * G * E2)
            totals.append(total)
        # the host check computes exactly what the plug-in's static_assert computes
        assert targets.parallel_smem_bytes(d, 0) == max(totals) <= targets.SMEM_MAX


def test_parallel_refusals():
    from walnuts_b200 import targets
    with pytest.raises(ValueError, match="4096"):
        targets.cuda_target(DIAG_SRC, 4097, parallel=True)
    with pytest.raises(ValueError, match="4096"):
        targets.cuda_target(DIAG_SRC, 0, parallel=True)
    with pytest.raises(ValueError, match="512"):
        targets.cuda_target(SEQ_SRC, 513)
    with pytest.raises(ValueError, match="scratch"):
        targets.cuda_target(DIAG_SRC, 100, parallel=True, scratch=-1)
    with pytest.raises(ValueError, match="scratch"):
        targets.cuda_target(SEQ_SRC, 100, scratch=8)


def _max_scratch(d):
    from walnuts_b200 import targets
    s = 0
    while targets.parallel_smem_bytes(d, s + 1) <= targets.SMEM_MAX:
        s += 1
    return s


def test_scratch_limit_agrees_with_the_plugin():
    """The largest scratch the host check accepts compiles; one double more is refused by the host check AND by the
    plug-in's static_assert (compiled directly, bypassing the host check)."""
    from walnuts_b200 import build, targets
    d = 4096
    s = _max_scratch(d)
    assert s > 2000
    with pytest.raises(ValueError, match="scratch"):
        targets.cuda_target(DIAG_SRC, d, parallel=True, scratch=s + 1)
    tg = targets.cuda_target(DIAG_SRC, d, name="scratch_max", parallel=True, scratch=s)
    assert _plan(tg.plugin, FAM_EXT)[3] == targets.parallel_smem_bytes(d, s) <= targets.SMEM_MAX
    csrc = os.path.join(build.HERE, "csrc")
    tu = (f"#define WN_USER_D {d}\n#define WN_USER_PARALLEL 1\n#define WN_USER_SCRATCH {s + 1}\n"
          f"#include \"wn_user_api.cuh\"\n{DIAG_SRC}\n#include \"wn_user_plugin.cuh\"\n")
    r = subprocess.run([os.environ.get("NVCC", "nvcc"), "-std=c++17", "-x", "cu", "-gencode",
                        "arch=compute_100a,code=sm_100a", "-I", csrc, "-c", "-o", os.devnull, "-"],
                       input=tu, capture_output=True, text=True)
    assert r.returncode != 0 and "WN_USER_SCRATCH too large" in r.stdout + r.stderr, r.stdout + r.stderr


def test_wrong_macro_names_the_right_one():
    from walnuts_b200 import targets
    with pytest.raises(RuntimeError, match=r"define WN_TARGET_LP_GRAD_PAR\(q, g, data, n_data, ctx\)"):
        targets.cuda_target(SEQ_SRC, 300, name="wrong_macro_par", parallel=True)
    with pytest.raises(RuntimeError, match=r"define WN_TARGET_LP_GRAD\(q, g, data, n_data\), not"):
        targets.cuda_target(DIAG_SRC, 300, name="wrong_macro_seq")
