// User-defined CUDA targets (SURVEY.md section 8f, row N4): the role of the reference's arbitrary Python
// `lpFun(q) -> [lp, grad]` (WALNUTSpy/targetDistr.py:18) / `logp`, `grad` (walnuts/walnuts.py:296-297) and of
// walnuts_stan.py's compiled Stan model.  walnuts_b200.targets.cuda_target() compiles the user's source with nvcc for
// sm_100a into a plug-in library next to the sampler kernels.  This header is included BEFORE the user's source.
//
// Two protocols.
//
// Sequential (cuda_target(..., parallel=False), d <= 512): ONE device function over the whole coordinate vector
//
//     WN_TARGET_LP_GRAD(q, g, data, n_data) {
//       // q[0..WN_D-1] in, g[0..WN_D-1] out, data[0..n_data-1] = the array given to cuda_target(data=...)
//       return lp;      // the log density
//     }
//
// (WN_D <= 64: one thread per chain; 64 < WN_D <= 512: one warp per chain, the function is then called by every lane
// with q and g in shared memory).
//
// Parallel (cuda_target(..., parallel=True, scratch=S), d <= 4096): the function is called by EVERY thread of the
// chain's group at once and each thread computes its share of the density
//
//     WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx) {
//       // q[0..WN_D-1]: the chain's whole position in shared memory, readable by every thread of the chain
//       // g[0..WN_D-1]: shared; this thread writes g[j] for the j it owns:
//       for (int j = ctx.rank; j < WN_D; j += ctx.size) g[j] = ...;
//       // ctx.sum(x)  : sum of x over the chain's threads, the same value on every thread
//       // ctx.sync()  : barrier over the chain's threads (for ctx.scratch)
//       // ctx.scratch : WN_USER_SCRATCH doubles of per-chain shared memory
//       return share;   // this thread's share of lp; the library adds the shares
//     }
//
// Rules of the parallel protocol:
//   - every thread of the chain calls ctx.sum and ctx.sync the same number of times, in the same order; a call inside
//     a branch that differs between threads is undefined behaviour;
//   - the library never hands out an index j >= WN_D (ctx.rank < ctx.size; the loop above stops at WN_D);
//   - g[j] is read back only for j < WN_D, and only the thread that owns j may write it.
// The chain's group is 32, 64, 256 or 512 threads (d <= 512, 1024, 2048, 4096; wn_user_plugin.cuh: UserParT).
//
// A source that defines the macro of the other protocol fails to compile with a message naming the right one.
#pragma once
#include <cmath>
#include <cstdint>

#ifndef WN_USER_D
#error "WN_USER_D (the dimension) must be defined by the generated translation unit"
#endif
#define WN_D WN_USER_D
#ifndef WN_USER_PARALLEL
#define WN_USER_PARALLEL 0
#endif
#ifndef WN_USER_SCRATCH
#define WN_USER_SCRATCH 0
#endif

#if WN_USER_PARALLEL
#define WN_TARGET_LP_GRAD(q, g, data, n_data)                                                              \
  static_assert(wn_user_protocol_sequential_macro_in_parallel_target,                                    \
                "cuda_target(parallel=True): define WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx), "    \
                "not WN_TARGET_LP_GRAD");                                                                 \
  __device__ __forceinline__ double wn_user_lp_grad_unused(const double* q, double* g, const double* data, int n_data)
#define WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx)                                                     \
  template <class WnCtx>                                                                                \
  __device__ __forceinline__ double wn_user_lp_grad_par(const double* __restrict__ q, double* __restrict__ g, \
                                                        const double* __restrict__ data, int n_data,      \
                                                        const WnCtx& ctx)
#else
#define WN_TARGET_LP_GRAD(q, g, data, n_data)                                                              \
  __device__ __forceinline__ double wn_user_lp_grad(const double* __restrict__ q, double* __restrict__ g,   \
                                                    const double* __restrict__ data, int n_data)
#define WN_TARGET_LP_GRAD_PAR(q, g, data, n_data, ctx)                                                     \
  static_assert(wn_user_protocol_parallel_macro_in_sequential_target,                                    \
                "cuda_target(parallel=False): define WN_TARGET_LP_GRAD(q, g, data, n_data), not "        \
                "WN_TARGET_LP_GRAD_PAR (or pass parallel=True)");                                         \
  template <class WnCtx>                                                                                 \
  __device__ __forceinline__ double wn_user_lp_grad_par_unused(const double* q, double* g, const double* data, \
                                                               int n_data, const WnCtx& ctx)
#endif
constexpr bool wn_user_protocol_sequential_macro_in_parallel_target = false;
constexpr bool wn_user_protocol_parallel_macro_in_sequential_target = false;
