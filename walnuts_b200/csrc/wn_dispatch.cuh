// Kernel dispatch by (kernel family, target, dimension).  Each family -- plain WALNUTSpy transition, package
// transition, WALNUTSpy with warm-up adaptation, extended integrators -- is instantiated in its own
// translation unit (plans_*.cu) so that the families compile in parallel; capi.cu only sees the
// wn_pick_plan_* entry points.  The plain family is split by integrator at compile time (wn_walnutspy.cuh: KSET):
// "nuts" = fixedLeapFrog only, "wpy" = adaptLeapFrogD / adaptLeapFrogR2P only; adaptYoshidaD, the warm-up adaptation and
// the orbit statistics run on the "adapt" family (every integrator behind the runtime kind).
#pragma once
#include "../../include/walnuts_cuda.h"
#include "wn_package.cuh"
#include "wn_walnutspy.cuh"

namespace wn {

struct LaunchPlan {
  const void* fn;
  int G, E2, NT;
  size_t smem;
  bool package;
};

enum { FAM_WPY = WN_FAMILY_WPY, FAM_PKG = WN_FAMILY_PKG, FAM_ADAPT = WN_FAMILY_ADAPT, FAM_EXT = WN_FAMILY_EXT,
       FAM_NUTS = WN_FAMILY_NUTS };

template <int G, int E2>
using StdNormalT = DiagGaussT<G, E2, true>;
template <int G, int E2>
using DiagT = DiagGaussT<G, E2, false>;

template <template <int, int> class T, int G, int E2, int NT, int MINB = 1, bool ADAPT = false, bool EXT = false,
          int KSET = KSET_ANY, bool CTLSM = false>
static LaunchPlan plan_wpy() {
  LaunchPlan p;
  p.fn = (const void*)walnutspy_kernel<T, G, E2, NT, MINB, ADAPT, EXT, KSET, CTLSM>;
  p.G = G; p.E2 = E2; p.NT = NT;
  p.smem = (size_t)wpy_smem_doubles<T, G, E2, NT, ADAPT, KSET>() * sizeof(double);
  p.package = false;
  return p;
}
// plain family: the kernel set follows from the family (FAM_NUTS: fixedLeapFrog, FAM_WPY: D / R2P)
template <int FAM, template <int, int> class T, int G, int E2, int NT, int MINB = 1, bool CTLSM = false>
static LaunchPlan plan_plain() {
  return plan_wpy<T, G, E2, NT, MINB, false, false, (FAM == FAM_NUTS) ? KSET_FIXED : KSET_ADAPT, CTLSM>();
}
template <template <int, int> class T, int G, int E2, int NT>
static LaunchPlan plan_pkg() {
  LaunchPlan p;
  p.fn = (const void*)package_kernel<T, G, E2, NT>;
  p.G = G; p.E2 = E2; p.NT = NT;
  p.smem = (size_t)(3 * 2 * E2 * NT + 2 * ((G + 31) / 32) * 8 + T<G, E2>::smem_doubles(NT)) * sizeof(double);
  p.package = true;
  return p;
}

template <int FAM, template <int, int> class T, int G, int E2, int NT>
static LaunchPlan plan_for() {
  if constexpr (FAM == FAM_PKG) return plan_pkg<T, G, E2, NT>();
  else if constexpr (FAM == FAM_ADAPT) return plan_wpy<T, G, E2, NT, 1, true>();
  else if constexpr (FAM == FAM_EXT) return plan_wpy<T, G, E2, NT, 1, true, true>();
  else return plan_plain<FAM, T, G, E2, NT>();
}

#define WN_PICK(G, E2, NT)                                              \
  if (d <= 2 * (G) * (E2)) {                                            \
    p = plan_for<FAM, T, G, E2, NT>();                                  \
    return true;                                                        \
  }
template <int FAM, template <int, int> class T>
static bool pick_generic(int d, LaunchPlan& p) {
  // Threads per chain at small d, measured with scripts/small_d_sweep.py (std normal, 131 072 chains; old = the shapes of
  // round 1: 1 x 12, 4 x 8, 16 x 8): the chains that share a warp sit in different handlers of the state machine most of
  // the time and are served one after the other, so FEWER chains per warp with shorter per-thread code win as soon as
  // the handlers are long (D / R2P: d = 10 1.24x, d = 20 1.6x, d = 100 2.5x; fixedLeapFrog d = 20 2.5x, d = 100 1.7x;
  // package mode d = 100 1.2x, BASELINE config 1 at 65 536 chains 2.78e9 -> 5.18e9 evals/s).  Only the short-handler
  // kernels (fixedLeapFrog, package mode) at d <= 12 still prefer one thread per chain (8 x 2 there: 0.6-0.8x).
  WN_PICK(1, 2, 128)
  if constexpr (FAM == FAM_NUTS || FAM == FAM_PKG) { WN_PICK(1, 6, 128) }
  else { WN_PICK(8, 1, 128) }     // d <= 16: 4 chains per warp, 2 coordinates per thread
  WN_PICK(16, 1, 128)             // d <= 32: 2 chains per warp
  WN_PICK(32, 2, 128)             // d <= 128: ONE chain per warp, 4 coordinates per lane
  WN_PICK(32, 8, 128)
  WN_PICK(64, 8, 64)
  WN_PICK(256, 4, 256)
  WN_PICK(512, 4, 512)     // d <= 4096: one 16-warp CTA per chain, one CTA per SM
  // d <= 8192 / 16384 / 32768: one chain per thread-block CLUSTER of 2 / 4 / 8 such CTAs (G > NT), the reductions
  // finished through distributed shared memory.  Package mode stays at one CTA per chain.  Measured on B200
  // (scripts/high_d_gauss.py, profiles/r03_high_d_gauss.txt): see DESIGN.md section 2.  At 512 threads the register cap
  // is 128, and ptxas spills a little (ptxas -v: 8-144 B of spill stores in the wpy / nuts / adapt kernels, about
  // 1-1.8 KB in the ext kernels, whose extra integrators are not a hot path) -- the same as the 512 x 4 one-CTA rows
  // above, which share the shape.  Other shapes (256 threads per CTA, 2 CTAs per SM) were not measured.
  if constexpr (FAM != FAM_PKG) {
    WN_PICK(1024, 4, 512)
    WN_PICK(2048, 4, 512)
    WN_PICK(4096, 4, 512)
  }
  return false;
}
// targets that need the chain inside one warp; FIRST = false leaves out the first row for a caller that serves those d
// with a plan of its own
template <int FAM, template <int, int> class T, bool FIRST = true>
static bool pick_warp(int d, LaunchPlan& p) {
  if constexpr (FIRST) {
    if constexpr (FAM == FAM_NUTS || FAM == FAM_PKG) { WN_PICK(1, 6, 128) }
    else { WN_PICK(8, 1, 128) }
  }
  WN_PICK(16, 1, 128)
  WN_PICK(32, 2, 128)
  WN_PICK(32, 8, 128)
  return false;
}
#undef WN_PICK

template <int FAM>
static bool pick_plan_family(const wn_config& c, LaunchPlan& p) {
  switch (c.target) {
    case WN_TARGET_STD_NORMAL: return pick_generic<FAM, StdNormalT>(c.d, p);
    case WN_TARGET_DIAG_GAUSS: {
      if constexpr (FAM == FAM_WPY || FAM == FAM_NUTS) {
        if (c.d > 512 && c.d <= 1024) {
          // BASELINE config 2 (d = 1000; the shapes measured against each other are in DESIGN.md section 6).
          // D / R2P: 128 threads x 8 coordinates, 4 blocks / SM at 126 registers.  Plain NUTS (level loop): ONE warp
          // per chain, 32 coordinates per lane, inverse variances in shared memory, gradient recomputed (DiagSmT) --
          // no replicated scalar work, no block barrier per leaf pair: 4.8e8 grad evals/s against 3.5e8 for 4 warps
          // per chain and 1.68e8 for the flat loop of round 1
          if constexpr (FAM == FAM_NUTS) p = plan_plain<FAM, DiagSmT, 32, 16, 64, 4>();
          else p = plan_plain<FAM, DiagT, 128, 4, 128, 4>();
          return true;
        }
      }
      return pick_generic<FAM, DiagT>(c.d, p);
    }
    case WN_TARGET_FUNNEL:
      if constexpr (FAM == FAM_WPY || FAM == FAM_NUTS) {
        if (c.d <= 16) {
          // BASELINE config 3 (funnel10, d = 11): 8 threads per chain with 2 coordinates each (4 chains per warp), the
          // control block of every chain in shared memory, 5 blocks / SM at 92 registers.  The chains of a warp are in
          // different handlers of the state machine most of the time, so a warp issues nearly every instruction for ONE
          // of its chains (measured 1.4 chains per issued instruction with 8 chains per warp): fewer chains per warp
          // with shorter per-thread code win.  Measured at 262 144 chains x 10 transitions, R2P / fixedLeapFrog, ms per
          // call: 1 thread per chain ~330 / --, 4 threads x 4 coordinates (the round-2 default until then) 253 / 99,
          // 8 x 2 (shipped) 204 / 74, 16 x 2 204 / 79, 32 x 2 243 / 87
          p = plan_plain<FAM, FunnelT, 8, 1, 128, 5, true>();
          return true;
        }
        return pick_warp<FAM, FunnelT, false>(c.d, p);
      } else {
        return pick_warp<FAM, FunnelT>(c.d, p);
      }
    case WN_TARGET_FUNNEL_PKG: return pick_warp<FAM, FunnelPkgT>(c.d, p);
    case WN_TARGET_LOGREG: {
      if (c.d > 128) return false;
      // plain WALNUTSpy kernel: FP64 tensor-core gradient with TMA-staged row tiles up to d = 104, the
      // block-cooperative FMA gradient (8 chains per CTA share every load of X) above; the per-warp version serves
      // package mode / warm-up adaptation / the other integrators
      if constexpr (FAM == FAM_WPY || FAM == FAM_NUTS) {
        if (c.d <= 32) p = plan_plain<FAM, LogRegMma32T, 32, 2, 256>();
        else if (c.d <= 104) p = plan_plain<FAM, LogRegMma104T, 32, 2, 256>();
        else p = plan_plain<FAM, LogRegCoopT, 32, 2, 256>();
      } else {
        p = plan_for<FAM, LogRegT, 32, 2, 256>();
      }
      return true;
    }
    case WN_TARGET_STOCK_WATSON: {
      // d = 3T; thread t owns B consecutive time steps: T <= G*B
      if (c.d % 3 != 0) return false;
      const int T = c.d / 3;
      if (T <= 64 * 4) {
        // 6 blocks / SM (168 registers, 12 warps) measured 9 % faster than 4 blocks at 255 registers
        // (8 blocks / SM at 128 registers: spills, same throughput); round 2: see below
        // measured (C5 shape, R2P): launch bounds for 5 blocks / SM 2.65e8, for 6 blocks / SM 2.53e8 grad evals/s
        // (4 warps per chain with 2 time steps per thread, 128 / 96 registers: the same 2.63e8)
        if constexpr (FAM == FAM_WPY || FAM == FAM_NUTS) p = plan_plain<FAM, StockWatsonT, 64, 7, 64, 5>();
        else p = plan_for<FAM, StockWatsonT, 64, 7, 64>();
        return true;
      }
      if (T <= 128 * 4) { p = plan_for<FAM, StockWatsonT, 128, 7, 128>(); return true; }
      return false;
    }
    case WN_TARGET_DENSE_GAUSS: {
      if (c.d > 128) return false;
      // plain WALNUTSpy kernels: the gradient of the CTA's 8 lock-stepped chains on the FP64 tensor cores (DMMA) with
      // TMA-staged rows of P; everything else (package mode, warm-up adaptation, other integrators, d > 104) on the
      // per-warp FMA version
      if constexpr (FAM == FAM_WPY || FAM == FAM_NUTS) {
        if (c.d <= 104) {
          if (c.d <= 32) p = plan_plain<FAM, DenseGaussMma32T, 32, 2, 256>();
          else p = plan_plain<FAM, DenseGaussMma104T, 32, 2, 256>();
          return true;
        }
      }
      p = plan_for<FAM, DenseGaussT, 32, 2, 256>();
      return true;
    }
    case WN_TARGET_CORR_GAUSS:
      if (c.d != 2) return false;
      p = plan_for<FAM, CorrGaussT, 1, 1, 128>();
      return true;
    default: return false;
  }
}

}  // namespace wn

// one definition per translation unit plans_{wpy,nuts,pkg,adapt,ext}.cu
bool wn_pick_plan_wpy(const wn_config& c, wn::LaunchPlan& p);
bool wn_pick_plan_nuts(const wn_config& c, wn::LaunchPlan& p);
bool wn_pick_plan_pkg(const wn_config& c, wn::LaunchPlan& p);
bool wn_pick_plan_adapt(const wn_config& c, wn::LaunchPlan& p);
bool wn_pick_plan_ext(const wn_config& c, wn::LaunchPlan& p);
