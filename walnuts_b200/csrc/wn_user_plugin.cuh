// Second half of a user-target plug-in (included AFTER the user's WN_TARGET_LP_GRAD / WN_TARGET_LP_GRAD_PAR
// definition): wraps the user's function as a target of the persistent kernels and exports the plug-in entry points
// that capi.cu binds with dlopen.  Kernel launches happen INSIDE the plug-in: it carries its own statically linked
// CUDA runtime, so its kernels are registered there.  Only the wrapper of the protocol in use is compiled.
#pragma once
#include "wn_dispatch.cuh"

namespace wn {

#if !WN_USER_PARALLEL
// d <= 64: one thread per chain, the whole vector in registers / local memory
template <int G, int E2>
struct UserThreadT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static_assert(G == 1 && E >= WN_USER_D, "user targets up to d = 64 run one thread per chain");
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  const double* data;
  int nd;
  __device__ __forceinline__ int coord(int e, int) const { return e; }
  __device__ __forceinline__ void init(const TargetParams& tp, int, int, double*) { data = tp.p0; nd = tp.n0; }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    double qq[WN_USER_D], gg[WN_USER_D];
#pragma unroll
    for (int e = 0; e < WN_USER_D; ++e) { qq[e] = q[e]; gg[e] = 0.0; }
    const double lp = wn_user_lp_grad(qq, gg, data, nd);
#pragma unroll
    for (int e = 0; e < E; ++e) g[e] = (e < WN_USER_D) ? gg[e < WN_USER_D ? e : 0] : 0.0;
    return lp;
  }
};

// d > 64: ONE WARP per chain.  The chain's coordinates are spread over the 32 lanes (leapfrog, U-turn products, tree
// bookkeeping run in parallel as for the built-in targets); for the density the warp publishes q to its shared-memory
// row and EVERY lane evaluates the user's function on the whole vector -- identical inputs, identical results, the
// lanes write identical gradients -- so the user's source stays a plain sequential function of (q, g).  The
// evaluation itself is not parallelised over the lanes (the price of a generic protocol); d <= 512.
template <int G, int E2>
struct UserWarpT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static constexpr int DPAD = 2 * G * E2;
  static_assert(G == 32 && DPAD >= WN_USER_D, "warp layout: 32 lanes x 2 E2 coordinates must cover d");
  __host__ __device__ static constexpr int smem_doubles(int NT) { return (NT / 32) * 2 * DPAD; }
  const double* data;
  int nd;
  double *qs, *gs;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int, int, double* tsm) {
    data = tp.p0; nd = tp.n0;
    qs = tsm + (threadIdx.x >> 5) * 2 * DPAD;
    gs = qs + DPAD;
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    const int t = threadIdx.x & 31;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; ++e) qs[coord_of<G>(e, t)] = q[e];
    __syncwarp();
    const double lp = wn_user_lp_grad(qs, gs, data, nd);
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      g[e] = (j < WN_USER_D) ? gs[j] : 0.0;
    }
    return (t == 0) ? lp : 0.0;
  }
};
#else

// Parallel protocol (WN_USER_PARALLEL, wn_user_api.cuh): the G threads of a chain evaluate the density TOGETHER.
// Each chain has its own q row, g row and WN_USER_SCRATCH doubles of scratch in shared memory.  lp_grad publishes the
// thread's coordinates to the q row (zero for the padding coordinates j >= d), group barrier, the user's function on
// every thread, group barrier, and reads its coordinates' gradient back from the g row.  No thread keeps a copy of
// the whole vector.  The group barrier is __syncwarp() for G = 32, where four chains share a 128-thread block and
// retire independently (a block barrier there could wait for a warp that has left the kernel), and __syncthreads()
// only when the block is the chain (G == NT): there every thread runs the same control flow up to the exit, which is
// itself decided by a block-wide broadcast (Group::bcast0), as for the built-in targets' reductions.
template <int G>
__device__ __forceinline__ void user_group_sync() {
  if constexpr (G == 32) __syncwarp();
  else __syncthreads();
}

template <int G>
struct UserCtx {
  double* scratch;
  int rank, size;
  double* red;
  int& parity;
  __device__ __forceinline__ double sum(double x) const {
    double v[1] = {x};
    Group<G>::template sum<1>(v, red, parity);
    return v[0];
  }
  __device__ __forceinline__ void sync() const { user_group_sync<G>(); }
};

template <int G, int E2>
struct UserParT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static constexpr int DPAD = 2 * G * E2;
  static_assert(DPAD >= WN_USER_D, "parallel layout: G threads x 2 E2 coordinates must cover d");
  static_assert(WN_USER_SCRATCH >= 0, "WN_USER_SCRATCH: a number of doubles");
  static constexpr int ROW = 2 * DPAD + WN_USER_SCRATCH;   // q, g, scratch of one chain
  __host__ __device__ static constexpr int smem_doubles(int NT) { return (NT / G) * ROW; }
  const double* data;
  int nd;
  double *qs, *gs;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int, int, double* tsm) {
    data = tp.p0; nd = tp.n0;
    qs = tsm + (threadIdx.x / G) * ROW;
    gs = qs + DPAD;
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double* red, int& parity) const {
    const int t = threadIdx.x & (G - 1);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      qs[j] = (j < WN_USER_D) ? q[e] : 0.0;
    }
    user_group_sync<G>();
    const UserCtx<G> ctx{gs + DPAD, t, G, red, parity};
    const double lp = wn_user_lp_grad_par(qs, gs, data, nd, ctx);
    user_group_sync<G>();
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      g[e] = (j < WN_USER_D) ? gs[j] : 0.0;
    }
    return lp;
  }
};
#endif

constexpr int WN_USER_E2 = (WN_USER_D + 1) / 2;
constexpr bool WN_USER_WARP = WN_USER_D > 64;
constexpr int WN_USER_WE2 = (WN_USER_D <= 256) ? 4 : 8;     // 32 lanes x 8 / 16 coordinates

// parallel protocol: the shapes pick_generic ships for the built-in targets (wn_dispatch.cuh) from d = 129 on
constexpr int WN_USER_PG = (WN_USER_D <= 512) ? 32 : (WN_USER_D <= 1024) ? 64 : (WN_USER_D <= 2048) ? 256 : 512;
constexpr int WN_USER_PE2 = (WN_USER_D <= 256) ? 4 : (WN_USER_D <= 1024) ? 8 : 4;
constexpr int WN_USER_PNT = (WN_USER_PG == 32) ? 128 : WN_USER_PG;

#if WN_USER_PARALLEL
static_assert(WN_USER_D >= 1 && WN_USER_D <= 4096, "parallel user targets: 1 <= d <= 4096");
static_assert(WN_USER_PG == 32 || WN_USER_PG == WN_USER_PNT, "a chain is one warp or one whole block");
static_assert(WN_USER_PG <= WN_USER_PNT, "no thread-block clusters for user targets");
#endif

// Shared memory of the user kernels in bytes: the dynamic part of the plan plus the kernels' static __shared__
// arrays (walnutspy_kernel: sh_bcast, sh_ctl, sh_ktab; package_kernel: sh_bcast, sh_ctl), each rounded up to 16 bytes.
// walnuts_b200.targets.cuda_target() checks the same sum before it compiles anything.
constexpr size_t WN_SMEM_MAX = 227 * 1024;
__host__ __device__ constexpr size_t round16(size_t b) { return (b + 15) / 16 * 16; }
__host__ __device__ constexpr size_t user_static_smem(bool package, int G, int NT) {
  const size_t w = (G >= 32) ? NT / 32 : 1;
  return package ? round16(sizeof(uint32_t)) + round16(sizeof(PkgCtl) * w)
                 : round16(sizeof(uint32_t)) + round16(sizeof(Ctl) * w) + round16(sizeof(int) * 32 * w);
}
#if WN_USER_PARALLEL
// dynamic shared memory as plan_wpy (EXT family) / plan_pkg compute it (wn_dispatch.cuh)
constexpr size_t WN_USER_SMEM_EXT =
    (size_t)wpy_smem_doubles<UserParT, WN_USER_PG, WN_USER_PE2, WN_USER_PNT, true, KSET_ANY>() * sizeof(double) +
    user_static_smem(false, WN_USER_PG, WN_USER_PNT);
constexpr size_t WN_USER_SMEM_PKG =
    (size_t)(3 * 2 * WN_USER_PE2 * WN_USER_PNT + 2 * ((WN_USER_PG + 31) / 32) * 8 +
             UserParT<WN_USER_PG, WN_USER_PE2>::smem_doubles(WN_USER_PNT)) * sizeof(double) +
    user_static_smem(true, WN_USER_PG, WN_USER_PNT);
static_assert(WN_USER_SMEM_EXT <= WN_SMEM_MAX && WN_USER_SMEM_PKG <= WN_SMEM_MAX,
              "cuda_target: WN_USER_SCRATCH too large, the plan's shared memory exceeds 227 KB per block");
#endif

// (a template, so that only the layout in use is instantiated)
template <bool WARP>
static LaunchPlan user_plan_t(int family) {
  // FAM_EXT kernels serve every WALNUTSpy integrator and the warm-up adaptation (one instantiation per plug-in)
#if WN_USER_PARALLEL
  if (family == FAM_PKG) return plan_pkg<UserParT, WN_USER_PG, WN_USER_PE2, WN_USER_PNT>();
  return plan_wpy<UserParT, WN_USER_PG, WN_USER_PE2, WN_USER_PNT, 1, true, true>();
#else
  if constexpr (WARP) {
    if (family == FAM_PKG) return plan_pkg<UserWarpT, 32, WN_USER_WE2, 128>();
    return plan_wpy<UserWarpT, 32, WN_USER_WE2, 128, 1, true, true>();
  } else {
    if (family == FAM_PKG) return plan_pkg<UserThreadT, 1, WN_USER_E2, 128>();
    return plan_wpy<UserThreadT, 1, WN_USER_E2, 128, 1, true, true>();
  }
#endif
}
static LaunchPlan user_plan(int family) { return user_plan_t<WN_USER_WARP>(family); }

}  // namespace wn

extern "C" {

int wn_user_abi(void) { return WN_ABI_VERSION; }
int wn_user_dim(void) { return WN_USER_D; }

// fills the launch geometry for `family` (wn::FAM_PKG or anything else = WALNUTSpy driver)
int wn_user_plan(int family, int* G, int* E2, int* NT, size_t* smem, int* package) {
  const wn::LaunchPlan p = wn::user_plan(family);
  *G = p.G; *E2 = p.E2; *NT = p.NT; *smem = p.smem; *package = p.package ? 1 : 0;
  return 0;
}

// shared memory of the family's kernel per block in bytes: the plan's dynamic part plus the kernel's static arrays
// (what cuda_target() checks against the 227 KB of a block before it compiles)
size_t wn_user_smem_total(int family) {
  const wn::LaunchPlan p = wn::user_plan(family);
  return p.smem + wn::user_static_smem(p.package, p.G, p.NT);
}

// resident blocks per SM (after raising the dynamic shared memory limit); < 0: CUDA error code
int wn_user_occupancy(int family, int device) {
  const wn::LaunchPlan p = wn::user_plan(family);
  if (cudaSetDevice(device) != cudaSuccess) return -1;
  if (cudaFuncSetAttribute(p.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem) != cudaSuccess) return -2;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, p.fn, p.NT, p.smem) != cudaSuccess) return -3;
  return occ;
}

// launches the family's kernel on `stream`; params = wn::RunParams or wn::PkgParams of the caller
int wn_user_launch(int family, int device, const void* params, unsigned blocks, void* stream) {
  const wn::LaunchPlan p = wn::user_plan(family);
  if (cudaSetDevice(device) != cudaSuccess) return -1;
  void* args[] = {const_cast<void*>(params)};
  const cudaError_t e = cudaLaunchKernel(p.fn, dim3(blocks), dim3(p.NT), args, p.smem, (cudaStream_t)stream);
  return e == cudaSuccess ? 0 : -(int)e - 100;
}

}  // extern "C"
