// Second half of a user-target plug-in (included AFTER the user's WN_TARGET_LP_GRAD definition): wraps the
// user's function as a target of the persistent kernels (one thread per chain, the whole vector in registers /
// local memory) and exports the plug-in entry points that capi.cu binds with dlopen.  Kernel launches happen
// INSIDE the plug-in: it carries its own statically linked CUDA runtime, so its kernels are registered there.
#pragma once
#include "wn_dispatch.cuh"

namespace wn {

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

constexpr int WN_USER_E2 = (WN_USER_D + 1) / 2;
constexpr bool WN_USER_WARP = WN_USER_D > 64;
constexpr int WN_USER_WE2 = (WN_USER_D <= 256) ? 4 : 8;     // 32 lanes x 8 / 16 coordinates

// (a template, so that only the layout in use is instantiated)
template <bool WARP>
static LaunchPlan user_plan_t(int family) {
  // FAM_EXT kernels serve every WALNUTSpy integrator and the warm-up adaptation (one instantiation per plug-in)
  if constexpr (WARP) {
    if (family == FAM_PKG) return plan_pkg<UserWarpT, 32, WN_USER_WE2, 128>();
    return plan_wpy<UserWarpT, 32, WN_USER_WE2, 128, 1, true, true>();
  } else {
    if (family == FAM_PKG) return plan_pkg<UserThreadT, 1, WN_USER_E2, 128>();
    return plan_wpy<UserThreadT, 1, WN_USER_E2, 128, 1, true, true>();
  }
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
