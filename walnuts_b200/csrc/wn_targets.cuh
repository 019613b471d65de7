// CUDA target registry: log density + gradient evaluated on the register-resident coordinates
// of a chain group.  Replaces reference WALNUTSpy/targetDistr.py and test/targets.py.
//
// Protocol: `init(tp, d, t)` loads per-thread constants; `lp_grad(q, g, red, parity)` fills the
// gradient of this thread's coordinates and returns this thread's PARTIAL of lp (the sum of the
// partials over the group is lp).  A target may reduce over the group internally; control flow
// is uniform within a group.
#pragma once
#include "wn_common.cuh"

namespace wn {

struct TargetParams {
  const double* p0;  // inv_var [d]      | X [N,P] row-major | y [T]
  const double* p1;  // -                | y [N]             | -
  const double* p2;  // -                | X^T [P,N]         | -
  int n0, n1;        // -                | N, P              | T
  double c0;         // max |inv_var|    | 1/tau^2           | -
  double c1;         // min inv_var      | -                 | -
};

// coordinate index of element e (= 2*e2 + h) held by thread t
template <int G>
__device__ __forceinline__ int coord_of(int e, int t) {
  return 2 * ((e >> 1) * G + t) + (e & 1);
}

// ---- T1/T2: standard normal and diagonal Gaussian -------------------------------------
// lp = -1/2 sum q_i^2 s_i, grad = -q_i s_i (s = 1: reference targetDistr.stdGauss :18-21,
// test/targets.py:4-7).  12 flop per coordinate per leapfrog step including the energy.
template <int G, int E2, bool UNIT>
struct DiagGaussT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  // Energies are only consumed at the end of a pass (adaptiveIntegrators.py:87) plus the
  // all(isfinite(Hams)) test (:92).  While every |q_i|, |v_i| stays below 2^470 (and inv_var <= 2^60, d < 2^23; the
  // dispatcher stops at d = 2^15) each intermediate energy -- every term AND their sum -- is provably finite, so the intermediate
  // steps may skip the two energy FMAs per
  // coordinate; if the bound is ever violated the sampler re-runs the pass with per-step energies.
  static constexpr bool LAZY_ENERGY = true;
  static constexpr bool COOP = false;
  // every thread's partial of H = 1/2 sum s q^2 + 1/2 sum v^2 is non-negative when all inverse variances are
  // (nonneg_ok): a single partial that exceeds the start energy by delta certifies a failed search attempt
  static constexpr bool NONNEG_ENERGY = true;
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  double s[UNIT ? 1 : E];
  double smax;     // max inv_var over ALL coordinates (host-computed, TargetParams::c0)
  bool lazy_ok, nonneg_ok;
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int t, double*) {
    lazy_ok = true;
    nonneg_ok = UNIT ? true : (tp.c1 >= 0.0);    // host-computed minimum of inv_var over ALL coordinates
    smax = UNIT ? 1.0 : tp.c0;
    lazy_ok = (smax <= 0x1p60);
    if constexpr (!UNIT) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int j = coord_of<G>(e, t);
        s[e] = (j < d) ? tp.p0[j] : 0.0;
        lazy_ok = lazy_ok && (fabs(s[e]) <= 0x1p60);
      }
    }
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    double acc0 = 0.0, acc1 = 0.0;   // two partial sums: halves the dependent-FMA chain
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if constexpr (UNIT) g[e] = -q[e];
      else g[e] = -(q[e] * s[e]);
      if (e & 1) acc1 = fma(q[e], g[e], acc1);
      else acc0 = fma(q[e], g[e], acc0);
    }
    return 0.5 * (acc0 + acc1);
  }
  // upper bound of max(|q'|,|v'|) / max(|q|,|v|) over one leapfrog step of size hh on this target:
  // v1 = v - a s q, q' = q + hh v1, v' = v1 - a s q'  with a = hh/2, s <= smax
  __device__ __forceinline__ double step_growth(double hh) const {
    // ... and of the merged-kick form w = v - a s q, q' = q + hh w, w' = w - hh s q' (wn_walnutspy.cuh: drift_kick)
    const double A = 0.5 * hh * smax;
    return fmax(fmax(1.0 + hh + hh * A, 1.0 + 2.0 * A + hh * A + hh * A * A), 1.0 + 2.0 * A + 2.0 * A * hh);
  }
  // The gradient is linear, g = -s q, so the full kick v += h g of the merged-kick loop is ONE FMA v += (-h s) q
  // with the coefficient formed once per pass: 2 FP64 instructions per coordinate and interior step.
  __device__ __forceinline__ void kick_coeffs(double hh, double (&kc)[E]) const {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if constexpr (UNIT) kc[e] = -hh;
      else kc[e] = -(hh * s[e]);
    }
  }
  __device__ __forceinline__ void grad_only(const double (&q)[E], double (&g)[E]) const {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if constexpr (UNIT) g[e] = -q[e];
      else g[e] = -(q[e] * s[e]);
    }
  }
};

// Diagonal Gaussian with the inverse variances in SHARED memory (one table per block) and a gradient that is
// recomputed from q where it is needed (REGRAD): leaves the register file to q and v when ONE warp holds a whole
// high-dimensional chain (plain NUTS at d = 1000: 32 coordinates per lane).
template <int G, int E2>
struct DiagSmT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static constexpr bool REGRAD = true;
  __host__ __device__ static constexpr int smem_doubles(int) { return 2 * G * E2; }
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  const double2* ssm;     // this lane's first pair; pair e2 at ssm[e2 * G]
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int t, double* tsm) {
    for (int j = threadIdx.x; j < 2 * G * E2; j += blockDim.x) tsm[j] = (j < d) ? tp.p0[j] : 0.0;
    __syncthreads();
    ssm = reinterpret_cast<const double2*>(tsm) + t;
  }
  // One leapfrog step (reference adaptiveIntegrators.py:50-55) fused per coordinate, the gradient recomputed from q
  // at both ends instead of being carried: the same operations in the same order as the generic micro_step on this
  // layout (bit-identical), without a gradient array.  Returns this lane's partial of H = -lp + 1/2 sum v^2.
  __device__ __forceinline__ double leapfrog_energy(double (&q)[E], double (&v)[E], double hh, double ha) const {
    double lp0 = 0.0, lp1 = 0.0, ke0 = 0.0, ke1 = 0.0;
#pragma unroll
    for (int e2 = 0; e2 < E2; ++e2) {
      const double2 sv = ssm[e2 * G];
      double q0 = q[2 * e2], q1 = q[2 * e2 + 1], v0 = v[2 * e2], v1 = v[2 * e2 + 1];
      v0 = fma(ha, -(q0 * sv.x), v0);
      v1 = fma(ha, -(q1 * sv.y), v1);
      q0 = fma(hh, v0, q0);
      q1 = fma(hh, v1, q1);
      const double g0 = -(q0 * sv.x), g1 = -(q1 * sv.y);
      lp0 = fma(q0, g0, lp0);
      lp1 = fma(q1, g1, lp1);
      v0 = fma(ha, g0, v0);
      v1 = fma(ha, g1, v1);
      ke0 = fma(v0, v0, ke0);
      ke1 = fma(v1, v1, ke1);
      q[2 * e2] = q0; q[2 * e2 + 1] = q1; v[2 * e2] = v0; v[2 * e2 + 1] = v1;
    }
    return fma(0.5, ke0 + ke1, -(0.5 * (lp0 + lp1)));
  }
  __device__ __forceinline__ double lp_only(const double (&q)[E]) const {
    double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
    for (int e2 = 0; e2 < E2; ++e2) {
      const double2 sv = ssm[e2 * G];
      acc0 = fma(q[2 * e2], -(q[2 * e2] * sv.x), acc0);
      acc1 = fma(q[2 * e2 + 1], -(q[2 * e2 + 1] * sv.y), acc1);
    }
    return 0.5 * (acc0 + acc1);
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    double acc0 = 0.0, acc1 = 0.0;
#pragma unroll
    for (int e2 = 0; e2 < E2; ++e2) {
      const double2 sv = ssm[e2 * G];
      g[2 * e2] = -(q[2 * e2] * sv.x);
      g[2 * e2 + 1] = -(q[2 * e2 + 1] * sv.y);
      acc0 = fma(q[2 * e2], g[2 * e2], acc0);
      acc1 = fma(q[2 * e2 + 1], g[2 * e2 + 1], acc1);
    }
    return 0.5 * (acc0 + acc1);
  }
};

// a / B for a compile-time constant B, correctly rounded (bit-identical to the division): q = a * RN(1 / B) is within one
// ulp, r = a - B q is exact in an FMA, q + r / B rounds to RN(a / B) (Markstein 1990).  3 instructions instead of the ~20
// of the generic division; checked against a / b for 7.8e8 random operands (b = 3, 9).  Operands whose quotient or
// remainder could leave the normal range take the division.
template <int B>
__device__ __forceinline__ double div_const(double a) {
  constexpr double b = (double)B, y = 1.0 / (double)B;
  const double aa = fabs(a);
  if (!(aa > 0x1p-900 && aa < 0x1p900)) return a / b;
  const double q = a * y;
  return fma(fma(-b, q, a), y, q);
}

// ---- T3: Neal's funnel, reference targetDistr.funnel10 :74-78 (d = 1 + n) ---------------
// lp = logN(q0; 0, 3) + sum_i logN(q_i; 0, exp(q0/2));  G <= 32.
template <int G, int E2>
struct FunnelT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  static_assert(G <= 32, "funnel target needs the chain inside one warp");
  int d_;
  double nn;
  __device__ __forceinline__ void init(const TargetParams&, int d, int, double*) {
    d_ = d;
    nn = (double)(d - 1);
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double* red, int& parity) const {
    const int t = threadIdx.x & (G - 1);
    double x[1] = {0.0};
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      if (j >= 1 && j < d_) x[0] = fma(q[e], q[e], x[0]);
    }
    Group<G>::template sum<1>(x, red, parity);
    double q0 = q[0];
    if constexpr (G > 1) q0 = __shfl_sync(Group<G>::mask(), q0, (threadIdx.x & 31u) & ~(unsigned)(G - 1));
    const double ss = x[0];
    const double ex = exp(-q0);
    const double LOG_SQRT_2PI = 0.91893853320467274178;
    const double LOG3 = 1.09861228866810969140;
    const double q03 = div_const<3>(q0);
    const double lp = (-(q03 * q03) / 2.0 - LOG_SQRT_2PI - LOG3) +
                      (-0.5 * ex * ss - nn * LOG_SQRT_2PI - nn * 0.5 * q0);
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      g[e] = (j >= 1 && j < d_) ? -q[e] * ex : 0.0;
    }
    if (t == 0) g[0] = -0.5 * nn - div_const<9>(q0) + 0.5 * ex * ss;
    return (t == 0) ? lp : 0.0;
  }
};

// ---- test/targets.py:23-29 funnel (package protocol; a different density from funnel10) ---
template <int G, int E2>
struct FunnelPkgT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  static_assert(G <= 32, "funnel target needs the chain inside one warp");
  int d_;
  __device__ __forceinline__ void init(const TargetParams&, int d, int, double*) { d_ = d; }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double* red, int& parity) const {
    const int t = threadIdx.x & (G - 1);
    double x[1] = {0.0};
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      if (j >= 1 && j < d_) x[0] = fma(q[e], q[e], x[0]);
    }
    Group<G>::template sum<1>(x, red, parity);
    double q0 = q[0];
    if constexpr (G > 1) q0 = __shfl_sync(Group<G>::mask(), q0, (threadIdx.x & 31u) & ~(unsigned)(G - 1));
    const double ss = x[0];
    const double eh = exp(0.5 * q0);
    const double lp = div_const<9>(-0.5 * q0 * q0) - 0.5 * ss / eh;
    const double m = -1.0 / eh;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int j = coord_of<G>(e, t);
      g[e] = (j >= 1 && j < d_) ? m * q[e] : 0.0;
    }
    if (t == 0) g[0] = -(div_const<9>(q0) - 0.25 * ss / eh);
    return (t == 0) ? lp : 0.0;
  }
};

// ---- reference targetDistr.corrGauss :25-31 (2-d, rho = 0.5); G = 1, E2 = 1 ---------------
template <int G, int E2>
struct CorrGaussT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  static_assert(G == 1 && E2 == 1, "corr_gauss is 2-d");
  __device__ __forceinline__ void init(const TargetParams&, int, int, double*) {}
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    const double rho = 0.5, tmp = 1.0 - rho * rho;
    const double r = q[1] - rho * q[0];
    g[0] = -(q[0] - rho * q[1]) / tmp;
    g[1] = -(q[1] - rho * q[0]) / tmp;
    return -0.5 * q[0] * q[0] - (0.5 / tmp) * (r * r);
  }
};

}  // namespace wn

namespace wn {

// ---- T5: Stock-Watson stochastic volatility ------------------------------------------------------
// Unconstrained parameterisation of reference WALNUTSpy_examples/StockWatson/sw_innov.stan:7-52
// (bridgestan, propto = True); formulas: SURVEY.md appendix B, restated in oracle/targets.py
// (make_stock_watson).  theta = [tS, z1, zinn[T-2], x1, xinn[T-1], tau1, tauinn[T-1]], d = 3T.
//
// Layout: time-aligned.  Thread t owns the B consecutive time indices k = t*B .. t*B+B-1 of the three
// series Z = [z1, zinn...], X = [x1, xinn...], U = [tau1, tauinn...] (elements 0..3B-1) and thread 0
// additionally owns tS (element 3B).  One evaluation = 2 forward and 2 reverse block scans over the
// group (warp shuffles + one shared-memory exchange per scan when the chain spans several warps).
template <int G, int E2>
struct StockWatsonT {
  static constexpr int E = 2 * E2;
  static constexpr int B = (E - 2) / 3;
  static constexpr bool PAIR_LAYOUT = false;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  __host__ __device__ static constexpr int smem_doubles(int) { return 0; }
  static constexpr int WARPS = (G + 31) / 32;
  static_assert(3 * B + 2 == E, "E must be 3B + 2");
  static_assert(G % 32 == 0, "Stock-Watson target needs whole warps per chain");
  int T;
  double y[B];

  __device__ __forceinline__ void init(const TargetParams& tp, int, int t, double*) {
    T = tp.n0;
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const int k = t * B + i;
      y[i] = (k < T) ? tp.p0[k] : 0.0;
    }
  }
  __device__ __forceinline__ int coord(int e, int t) const {
    const int BIG = 1 << 30;
    if (e < B) { const int k = t * B + e; return (k <= T - 2) ? k + 1 : BIG; }                 // z1, zinn
    if (e < 2 * B) { const int k = t * B + (e - B); return (k <= T - 1) ? T + k : BIG; }       // x1, xinn
    if (e < 3 * B) { const int k = t * B + (e - 2 * B); return (k <= T - 1) ? 2 * T + k : BIG; } // tau1, tauinn
    if (e == 3 * B) return (t == 0) ? 0 : BIG;                                                 // tS
    return BIG;
  }

  // inclusive scan over the threads of the group of NV channels; FWD: prefix, else suffix.
  // On return x = inclusive value, ex = exclusive value (sum over strictly preceding / following threads).
  // NB > 0: additionally broadcasts bc[0..NB-1] of the group's thread 0 to every thread; the values ride on the
  // scan's own shared-memory exchange (free slots of warp 0's row) instead of costing a scan channel each.
  template <int NV, bool FWD, int NB = 0>
  __device__ __forceinline__ static void scan(double (&x)[NV], double (&ex)[NV], double* red, int& parity,
                                              double* bc = nullptr) {
    static_assert(NV + NB <= 8, "one row of the exchange buffer per warp");
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const double yv = FWD ? __shfl_up_sync(0xffffffffu, x[k], off) : __shfl_down_sync(0xffffffffu, x[k], off);
        const bool take = FWD ? (lane >= off) : (lane + off < 32);
        x[k] += take ? yv : 0.0;
      }
    }
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const double yv = FWD ? __shfl_up_sync(0xffffffffu, x[k], 1) : __shfl_down_sync(0xffffffffu, x[k], 1);
      ex[k] = (FWD ? (lane >= 1) : (lane < 31)) ? yv : 0.0;
    }
    if constexpr (G > 32) {
      const int w = (threadIdx.x % G) >> 5;
      double* buf = red + parity * (WARPS * 8);
      if (lane == (FWD ? 31 : 0)) {
#pragma unroll
        for (int k = 0; k < NV; ++k) buf[w * 8 + k] = x[k];
      }
      if constexpr (NB > 0) {
        if ((threadIdx.x % G) == 0) {
#pragma unroll
          for (int j = 0; j < NB; ++j) buf[NV + j] = bc[j];
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        double off = 0.0;
        if (FWD) { for (int ww = 0; ww < w; ++ww) off += buf[ww * 8 + k]; }
        else { for (int ww = WARPS - 1; ww > w; --ww) off += buf[ww * 8 + k]; }
        x[k] += off;
        ex[k] += off;
      }
      if constexpr (NB > 0) {
#pragma unroll
        for (int j = 0; j < NB; ++j) bc[j] = buf[NV + j];
      }
      parity ^= 1;
    } else if constexpr (NB > 0) {
#pragma unroll
      for (int j = 0; j < NB; ++j) bc[j] = __shfl_sync(0xffffffffu, bc[j], 0);
    }
  }

  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double* red, int& parity) const {
    const int t = threadIdx.x % G;
    const int k0 = t * B;
    // (temporaries are kept to 8 arrays of B doubles: the kernel is register-bound)
    // ---- phase 1: prefix sums of the innovations; index-0 entries and tS travel as "base" channels ----
    double locZ[B], locX[B];
    double ch[2] = {0.0, 0.0}, ex1[2];
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const int k = k0 + i;
      ch[0] += (k >= 1 && k <= T - 2) ? q[i] : 0.0;
      ch[1] += (k >= 1 && k <= T - 1) ? q[B + i] : 0.0;
      locZ[i] = ch[0];      // local inclusive prefix
      locX[i] = ch[1];
    }
    double b1[3] = {q[0], q[B], q[3 * B]};      // thread 0's z1, x1, tS travel with the scan's exchange
    scan<2, true, 3>(ch, ex1, red, parity, b1);
    const double Z0 = b1[0], X0 = b1[1], tS = b1[2];
    // sigma = exp(-tS / 2) and exp(tS) in ONE instruction stream: even lanes evaluate the first, odd lanes the second
    // (same operation on the same operand as the sequential form: bit-identical)
    const bool oddl = (threadIdx.x & 1) != 0;
    const double e2v = exp(oddl ? tS : -0.5 * tS);
    const double sigma = __shfl_sync(0xffffffffu, e2v, 0), etS = __shfl_sync(0xffffffffu, e2v, 1);
    double lp = 0.0;
    double ez[B], w[B], c[B], locC[B];
    double ch2[1] = {0.0}, ex2[1];
    const double ez_prev = exp(0.5 * fma(sigma, ex1[0], Z0));   // exp(z_{k0-1}/2)
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const int k = k0 + i;
      ez[i] = exp(0.5 * fma(sigma, ex1[0] + locZ[i], Z0));
      const double xx = fma(sigma, ex1[1] + locX[i], X0);
      w[i] = exp(-xx);
      if (k <= T - 1) lp -= 0.5 * xx;
      if (k >= 1 && k <= T - 2) lp -= 0.5 * q[i] * q[i];
      if (k >= 1 && k <= T - 1) lp -= 0.5 * (q[B + i] * q[B + i] + q[2 * B + i] * q[2 * B + i]);
      const double ezm = (i == 0) ? ez_prev : ez[(i > 0) ? i - 1 : 0];
      c[i] = (k >= 1 && k <= T - 1) ? ezm * q[2 * B + i] : 0.0;   // exp(z_{k-1}/2) * tauinn_{k-1}
      ch2[0] += c[i];
      locC[i] = ch2[0];
    }
    // ---- phase 2: tau ----
    double b2[1] = {q[2 * B]};                   // thread 0's tau1
    scan<1, true, 1>(ch2, ex2, red, parity, b2);
    const double U0 = b2[0];
    // residuals and their local suffix sums in one reverse sweep
    double sufR[B], sufA[B];
    double ch3[2] = {0.0, 0.0}, ex3[2];
#pragma unroll
    for (int i = B - 1; i >= 0; --i) {
      const int k = k0 + i;
      const bool obs = (k <= T - 1);
      const double e = y[i] - (U0 + (ex2[0] + locC[i]));
      const double eew = e * e * w[i];
      if (obs) lp -= 0.5 * eew;
      ch3[0] += obs ? e * w[i] : 0.0;
      ch3[1] += obs ? (-0.5 + 0.5 * eew) : 0.0;
      sufR[i] = ch3[0];
      sufA[i] = ch3[1];
    }
    // ---- phase 3: R, A suffix sums ----
    scan<2, false>(ch3, ex3, red, parity);
    double sufB[B];
    double ch4[2] = {0.0, 0.0}, ex4[2];
#pragma unroll
    for (int i = B - 1; i >= 0; --i) {
      const int k = k0 + i;
      const double bb = 0.5 * c[i] * (ex3[0] + sufR[i]);     // b_{k-1} of appendix B (c is already masked)
      sufB[i] = ch4[0];                                      // exclusive local suffix
      ch4[0] += bb;
      // d/dtS partial: sum_k zinn_k Bz_{k+1} + sum_k xinn_k A_{k+1}, with the first sum re-ordered as
      // sum_j b_j * (prefix of zinn before j)
      const double pzex = (ex1[0] + locZ[i]) - ((k >= 1 && k <= T - 2) ? q[i] : 0.0);
      ch4[1] += bb * pzex + ((k >= 1 && k <= T - 1) ? q[B + i] * (ex3[1] + sufA[i]) : 0.0);
    }
    // ---- phase 4: Bz suffix sums and the tS total ----
    scan<2, false>(ch4, ex4, red, parity);
#pragma unroll
    for (int i = 0; i < B; ++i) {
      const int k = k0 + i;
      const double Sx = ex4[0] + sufB[i];     // sum_{j > k} bb_j = Bz of appendix B at the next index
      const double Rk = ex3[0] + sufR[i], Ak = ex3[1] + sufA[i];
      const double ezm = (i == 0) ? ez_prev : ez[(i > 0) ? i - 1 : 0];
      g[i] = (k == 0) ? Sx : ((k <= T - 2) ? fma(sigma, Sx, -q[i]) : 0.0);
      g[B + i] = (k == 0) ? Ak : ((k <= T - 1) ? fma(sigma, Ak, -q[B + i]) : 0.0);
      g[2 * B + i] = (k == 0) ? Rk : ((k <= T - 1) ? fma(ezm, Rk, -q[2 * B + i]) : 0.0);
    }
    g[3 * B] = (t == 0) ? (5.0 - 0.5 * etS - 0.5 * sigma * ch4[1]) : 0.0;
    g[3 * B + 1] = 0.0;
    if (t == 0) lp += 5.0 * tS - 0.5 * etS;
    return lp;
  }
};

}  // namespace wn

namespace wn {

// ---- T4: Bayesian logistic regression (SURVEY.md row T4; not in the reference) -----------------------
// lp = sum_n [y_n eta_n - log(1 + exp(eta_n))] - |beta|^2 / (2 tau^2),  eta = X beta,
// grad = X^T (y - sigmoid(eta)) - beta / tau^2;  X [N,P] row-major plus its transpose X^T [P,N].
// One warp per chain (G = 32, P <= 64*E2).  Rows are processed in tiles of RT: phase 1 computes
// eta / residuals with one lane per row (X^T: coalesced over rows, beta broadcast from shared memory),
// phase 2 accumulates X^T r with one lane per coordinate pair (X: coalesced over coordinates, residuals
// broadcast).  The warps of a block run their evaluations in lock-step (one barrier per trip of the
// sampler's loop), so that the X tiles one warp pulls into L1 are reused by the block's other chains.
template <int G, int E2>
struct LogRegT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = true;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static constexpr int RT = 128, RJ = RT / 32, PMAX = 2 * G * E2;
  static_assert(G == 32, "logistic regression target: one warp per chain");
  __host__ __device__ static constexpr int smem_doubles(int NT) { return (NT / 32) * (PMAX + RT); }
  const double *X, *XT, *y;
  int N, P;
  double itau2;
  double *bs, *rs;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int, double* tsm) {
    X = tp.p0; y = tp.p1; XT = tp.p2; N = tp.n0; P = d; itau2 = tp.c0;
    bs = tsm + (threadIdx.x >> 5) * (PMAX + RT);
    rs = bs + PMAX;
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    const int t = threadIdx.x & 31;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; ++e) bs[coord_of<G>(e, t)] = q[e];
    __syncwarp();
    double lp = 0.0;
    double acc[E];
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] = 0.0;
    for (int n0 = 0; n0 < N; n0 += RT) {
      // phase 1: eta for rows n0 + t + 32 j
      double eta[RJ];
#pragma unroll
      for (int j = 0; j < RJ; ++j) eta[j] = 0.0;
      if (n0 + RT <= N) {
#pragma unroll 4
        for (int k = 0; k < P; ++k) {
          const double b = bs[k];
          const double* col = XT + (size_t)k * N + n0 + t;
#pragma unroll
          for (int j = 0; j < RJ; ++j) eta[j] = fma(__ldg(col + 32 * j), b, eta[j]);
        }
      } else {
        for (int k = 0; k < P; ++k) {
          const double b = bs[k];
          const double* col = XT + (size_t)k * N + n0 + t;
#pragma unroll
          for (int j = 0; j < RJ; ++j)
            if (n0 + t + 32 * j < N) eta[j] = fma(__ldg(col + 32 * j), b, eta[j]);
        }
      }
#pragma unroll
      for (int j = 0; j < RJ; ++j) {
        const int n = n0 + t + 32 * j;
        double r = 0.0;
        if (n < N) {
          const double yy = __ldg(y + n), et = eta[j];
          const double ex = exp(-fabs(et));
          const double inv = 1.0 / (1.0 + ex);
          const double sig = (et >= 0.0) ? inv : ex * inv;
          r = yy - sig;
          lp += yy * et - (fmax(et, 0.0) + log1p(ex));
        }
        rs[t + 32 * j] = r;
      }
      __syncwarp();
      // phase 2: acc_k += X[n][k] * r_n for this lane's coordinates
      const int nend = min(RT, N - n0);
#pragma unroll 4
      for (int i = 0; i < nend; ++i) {
        const double r = rs[i];
        const double* row = X + (size_t)(n0 + i) * P;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int k = coord_of<G>(e, t);
          if (k < P) acc[e] = fma(__ldg(row + k), r, acc[e]);
        }
      }
      __syncwarp();
    }
    double qq = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      g[e] = (k < P) ? fma(-itau2, q[e], acc[e]) : 0.0;
      qq = fma(q[e], q[e], qq);
    }
    return lp - 0.5 * itau2 * qq;
  }
};

}  // namespace wn

namespace wn {

// ---- T4, block-cooperative version: the chains of a CTA evaluate their gradients TOGETHER --------------------
// 8 chains per CTA of 256 threads (one warp owns one chain's coordinates, as in LogRegT).  Every trip of the
// sampler's loop the active chains publish beta to shared memory; then ALL 256 threads stream the rows once:
//   phase 1 (4 rows per thread): eta_n^c = x_n . beta^c for the 8 chains  (X^T coalesced over rows; 32 FMA per
//                                4 loads + 4 shared broadcasts), r_n^c = y_n - sigmoid(eta_n^c),
//                                lp^c += y_n eta - log(1+e^eta) only for chains at the end of a pass -> shared r tile
//   phase 2 (lane = 4 coordinates, warp = row stream): acc[k][c] += X[n][k] r_n^c            (32 FMA per row)
// so every element of X is loaded once per CTA trip instead of once per chain.  Deterministic: partial sums are
// combined in a fixed order (no atomics).
template <int G, int E2>
struct LogRegCoopT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;   // the cooperative evaluation has its own barriers
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = true;
  static constexpr int NTC = 256, C = 8, PMAX = 128, RPT = 4, RT = NTC * RPT;
  static_assert(G == 32 && E2 == 2, "cooperative logistic regression: one warp per chain, P <= 128");
  // Staging ring: S stages of STG doubles, filled by bulk async copies (TMA engine) that complete on a
  // "full" mbarrier per stage; consumers release a stage by arriving on its "empty" mbarrier, and the
  // producer (thread 0) refills it S-1 chunks ahead -- across the phase-1 / phase-2 / row-tile boundaries.
  // Chunk stream of one evaluation: per row tile, P chunks "coordinate k of X^T for the tile's rows"
  // followed by ceil(rows/8) chunks "8 rows of X".
  // Measured on B200 (DESIGN.md section 6): with only 32 FMA per thread between two barrier operations the
  // per-chunk mbarrier wait/arrive costs more than the L2 latency it hides (0.99e5 vs 1.37e5 evals/s with plain
  // read-only loads and 16 loads in flight per thread), so the staging ring is compiled out by default.
  static constexpr bool USE_BULK = false;
  static constexpr int S = 8, STG = 1024, RC = 8;
  // shared: bs[PMAX][C] | rs[RT][C] | gs[C][PMAX] | part[8][PMAX][4] | lps[8 warps][C] | act[C] | need[C]
  //         | full[S] | empty[S] | stage[S][STG]
  __host__ __device__ static constexpr int smem_doubles(int) {
    return PMAX * C + RT * C + C * PMAX + 8 * PMAX * 4 + 8 * C + 2 * C + 2 * S + (USE_BULK ? S * STG : 0);
  }
  const double *X, *XT, *y;
  int N, P;
  double itau2;
  double *bs, *rs, *gs, *part, *lps, *act, *need, *stage;
  uint64_t *full, *empty;
  bool bulk;      // 16-byte alignment of every staged chunk holds (N and P even)
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int, double* tsm) {
    X = tp.p0; y = tp.p1; XT = tp.p2; N = tp.n0; P = d; itau2 = tp.c0;
    bs = tsm; rs = bs + PMAX * C; gs = rs + RT * C; part = gs + C * PMAX; lps = part + 8 * PMAX * 4; act = lps + 8 * C;
    need = act + C;
    full = reinterpret_cast<uint64_t*>(need + C);
    empty = full + S;
    stage = need + C + 2 * S;
    bulk = USE_BULK && ((N & 1) == 0) && ((P & 1) == 0);
    if (USE_BULK && threadIdx.x == 0) {
      for (int i = 0; i < S; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], NTC); }
      mbar_fence_init();
    }
    __syncthreads();
  }
  // not used by COOP kernels (the generic protocol entry point)
  __device__ __forceinline__ double lp_grad(const double (&)[E], double (&)[E], double*, int&) const { return 0.0; }

  // need_lp: the energy of this step is consumed (last step of a pass).  For this target a non-finite
  // intermediate energy implies a non-finite state, which persists to the end of the pass, so skipping the
  // log-likelihood of intermediate steps does not change all(isfinite(Hams)) (adaptiveIntegrators.py:92).
  __device__ __forceinline__ void publish(const double (&q)[E], bool active, bool need_lp) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
#pragma unroll
    for (int e = 0; e < E; ++e) bs[coord_of<G>(e, t) * C + w] = active ? q[e] : 0.0;
    if (t == 0) { act[w] = active ? 1.0 : 0.0; need[w] = (active && need_lp) ? 1.0 : 0.0; }
  }

  // `gch`: number of chunks consumed so far by this CTA (kept by the caller across evaluations); chunk g
  // lives in stage g % S and completes phase (g / S) & 1 of that stage's barriers.
  __device__ __forceinline__ void coop_eval(uint32_t& gch) const {
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    bool any = false;
    bool nl[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { any = any || (act[c] != 0.0); nl[c] = need[c] != 0.0; }
    if (!any) {
      // no chain of the CTA is in a pass: leave through a barrier, so that no warp can publish the NEXT trip's flags
      // while another one is still reading this trip's
      __syncthreads();
      return;
    }
    double acc[4][C];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int c = 0; c < C; ++c) acc[j][c] = 0.0;
    double lp[C];
#pragma unroll
    for (int c = 0; c < C; ++c) lp[c] = 0.0;
    const int k4 = 4 * lane;

    // ---- producer cursor (thread 0 only): next chunk to issue ----
    uint32_t pg = gch;            // global index of the next chunk to issue
    int pn0 = 0, pi = 0;          // its row tile and index inside the tile's chunk list
    auto produce = [&]() {        // issue one chunk if any is left in this evaluation
      if (pn0 >= N) return;
      const int nrows = min(RT, N - pn0);
      const int st_ = pg % S;
      if (pg >= (uint32_t)S) mbar_wait(&empty[st_], ((pg / S) & 1u) ^ 1u);   // previous use released by all
      double* dst = stage + st_ * STG;
      if (pi < P) {
        mbar_expect_tx(&full[st_], (uint32_t)(nrows * 8));
        bulk_g2s(dst, XT + (size_t)pi * N + pn0, (uint32_t)(nrows * 8), &full[st_]);
      } else {
        const int r0 = (pi - P) * RC, rn = min(RC, nrows - r0);
        mbar_expect_tx(&full[st_], (uint32_t)(rn * P * 8));
        bulk_g2s(dst, X + (size_t)(pn0 + r0) * P, (uint32_t)(rn * P * 8), &full[st_]);
      }
      ++pg;
      ++pi;
      if (pi >= P + (nrows + RC - 1) / RC) { pi = 0; pn0 += RT; }
    };
    if (bulk && tid == 0) {
      for (int i = 0; i < S - 1; ++i) produce();
    }
    auto consume_begin = [&]() -> const double* {
      if (tid == 0) produce();                       // keep S-1 chunks in flight
      const int st_ = gch % S;
      mbar_wait(&full[st_], (gch / S) & 1u);
      return stage + st_ * STG;
    };
    auto consume_end = [&]() {
      mbar_arrive(&empty[gch % S]);
      ++gch;
    };

    for (int n0 = 0; n0 < N; n0 += RT) {
      const int nrows = min(RT, N - n0);
      // ---- phase 1: rows n0 + tid + 256 j, j < 4 ----
      {
        double eta[RPT][C];
#pragma unroll
        for (int j = 0; j < RPT; ++j)
#pragma unroll
          for (int c = 0; c < C; ++c) eta[j][c] = 0.0;
        bool in[RPT];
#pragma unroll
        for (int j = 0; j < RPT; ++j) in[j] = tid + NTC * j < nrows;
#pragma unroll 2
        for (int k = 0; k < P; ++k) {
          double x[RPT];
          if (bulk) {
            const double* sb = consume_begin();
#pragma unroll
            for (int j = 0; j < RPT; ++j) x[j] = in[j] ? sb[tid + NTC * j] : 0.0;
            consume_end();
          } else {
#pragma unroll
            for (int j = 0; j < RPT; ++j) x[j] = in[j] ? __ldg(XT + (size_t)k * N + n0 + tid + NTC * j) : 0.0;
          }
          const double2* b2 = reinterpret_cast<const double2*>(bs + k * C);
#pragma unroll
          for (int c2 = 0; c2 < C / 2; ++c2) {
            const double2 bb = b2[c2];
#pragma unroll
            for (int j = 0; j < RPT; ++j) {
              eta[j][2 * c2] = fma(x[j], bb.x, eta[j][2 * c2]);
              eta[j][2 * c2 + 1] = fma(x[j], bb.y, eta[j][2 * c2 + 1]);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < RPT; ++j) {
          const int n = n0 + tid + NTC * j;
          const double yy = in[j] ? __ldg(y + n) : 0.0;
#pragma unroll
          for (int c = 0; c < C; ++c) {
            const double et = eta[j][c];
            const double ex = exp(-fabs(et));
            const double inv = 1.0 / (1.0 + ex);
            const double sig = (et >= 0.0) ? inv : ex * inv;
            eta[j][c] = in[j] ? (yy - sig) : 0.0;                                  // residual
            if (nl[c] && in[j]) lp[c] += yy * et - (fmax(et, 0.0) + log1p(ex));
          }
          double2* r2 = reinterpret_cast<double2*>(rs + (tid + NTC * j) * C);
#pragma unroll
          for (int c2 = 0; c2 < C / 2; ++c2) r2[c2] = make_double2(eta[j][2 * c2], eta[j][2 * c2 + 1]);
        }
      }
      __syncthreads();
      // ---- phase 2: chunks of 8 rows; warp w takes row w of the chunk; lane owns coordinates 4*lane .. +3 ----
      {
        const int nchunk = (nrows + RC - 1) / RC;
#pragma unroll 4
        for (int ch = 0; ch < nchunk; ++ch) {
          const int i = ch * RC + w;                 // row inside the tile
          double x[4];
          if (bulk) {
            const double* sb = consume_begin();
#pragma unroll
            for (int j = 0; j < 4; ++j) x[j] = (i < nrows && k4 + j < P) ? sb[w * P + k4 + j] : 0.0;
            consume_end();
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) x[j] = (i < nrows && k4 + j < P) ? __ldg(X + (size_t)(n0 + i) * P + k4 + j) : 0.0;
          }
          if (i < nrows) {
            const double2* r2 = reinterpret_cast<const double2*>(rs + i * C);
#pragma unroll
            for (int c2 = 0; c2 < C / 2; ++c2) {
              const double2 r = r2[c2];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                acc[j][2 * c2] = fma(x[j], r.x, acc[j][2 * c2]);
                acc[j][2 * c2 + 1] = fma(x[j], r.y, acc[j][2 * c2 + 1]);
              }
            }
          }
        }
      }
      __syncthreads();
    }
    // ---- combine the 8 row streams (fixed order), 4 chains per round ----
#pragma unroll
    for (int half = 0; half < 2; ++half) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) part[(w * PMAX + k4 + j) * 4 + c] = acc[j][4 * half + c];
      __syncthreads();
      {
        const int k = tid & (PMAX - 1), cp = tid >> 7;          // 2 chains per thread
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int c = 2 * cp + cc;
          double s = 0.0;
#pragma unroll
          for (int ww = 0; ww < 8; ++ww) s += part[(ww * PMAX + k) * 4 + c];
          gs[(4 * half + c) * PMAX + k] = s;
        }
      }
      __syncthreads();
    }
    // ---- log-likelihood: lanes -> warp (butterfly), warps -> block (fixed order in collect) ----
#pragma unroll
    for (int c = 0; c < C; ++c) {
      double v = lp[c];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0) lps[w * C + c] = v;
    }
    __syncthreads();
  }

  // gradient of this warp's chain (after coop_eval); returns this thread's partial of lp
  __device__ __forceinline__ double collect(const double (&q)[E], double (&g)[E]) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
    double qq = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      g[e] = (k < P) ? fma(-itau2, q[e], gs[w * PMAX + k]) : 0.0;
      qq = fma(q[e], q[e], qq);
    }
    double lp = -0.5 * itau2 * qq;
    if (t == 0) {
#pragma unroll
      for (int ww = 0; ww < 8; ++ww) lp += lps[ww * C + w];
    }
    return lp;
  }
};

}  // namespace wn

namespace wn {

// Branch-free double-precision helpers for the sigmoid / log-likelihood of the tensor-core logistic regression
// (straight-line code lets the compiler interleave them with the DMMA stream).  Accuracy measured against long-double
// libm over 4e6 arguments: exp 0.87 ulp, reciprocal 0.5 ulp, log1p 2.9 ulp; NaN propagates.
__device__ __forceinline__ double exp_nonpos(double x) {   // exp(x) for x <= 0
  x = (x < -708.0) ? -708.0 : x;                            // below: < 3.4e-308, irrelevant next to 1
  const double z = fma(x, 1.4426950408889634, 6755399441055744.0);
  const int k = __double2loint(z);
  const double t = z - 6755399441055744.0;                  // rint(x log2 e)
  double r = fma(t, -6.93147180369123816490e-01, x);        // Cody-Waite
  r = fma(t, -1.90821492927058770002e-10, r);
  // Taylor to r^13 / 13! (|r| <= 0.347 -> 4e-18): the tail sum_{i>=3} r^(i-3) / i! by Estrin's scheme (dependent depth 4
  // instead of 11), the three leading terms by Horner -- same measured accuracy as the pure Horner form (0.87 ulp
  // against expl over 4e6 arguments), 7 instead of 13 dependent FMAs: the sigmoid's latency is what the DMMA stream
  // of the tensor-core logistic regression waits for
  const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
  const double a0 = fma(r, 4.1666666666666664e-02, 1.6666666666666666e-01);
  const double a1 = fma(r, 1.388888888888889e-03, 8.333333333333333e-03);
  const double a2 = fma(r, 2.48015873015873e-05, 1.984126984126984e-04);
  const double a3 = fma(r, 2.755731922398589e-07, 2.7557319223985893e-06);
  const double a4 = fma(r, 2.08767569878681e-09, 2.505210838544172e-08);
  const double b0 = fma(a1, r2, a0), b1 = fma(a3, r2, a2), b2 = fma(1.6059043836821613e-10, r2, a4);
  const double tl = fma(b2, r8, fma(b1, r4, b0));
  double p = fma(tl, r, 0.5);
  p = fma(p, r, 1.0);
  p = fma(p, r, 1.0);
  return p * __longlong_as_double((long long)(k + 1023) << 52);
}
__device__ __forceinline__ double rcp_pos(double d) {       // 1 / d for a positive normal d of moderate size
  float yf;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(yf) : "f"((float)d));   // MUFU.RCP, no slow path; 2^-22 accurate
  double y = (double)yf;
#pragma unroll
  for (int i = 0; i < 2; ++i) {        // 2^-22 -> 2^-44 -> below the rounding error (0.5 ulp measured against 1 / d)
    const double e = fma(-d, y, 1.0);
    y = fma(y, e, y);
  }
  return y;
}
// log1p(z) for 0 <= z <= 1 given inv = 1 / (1 + z):  log(u) + (z - (u - 1)) / u with u = fl(1 + z),
// log(u) = [u > sqrt 2] ln 2 + 2 atanh(s), s = f / (2 + f), f = m - 1
__device__ __forceinline__ double log1p_unit(double z, double inv) {
  const double u = 1.0 + z, c = z - (u - 1.0);
  const bool big = u > 1.4142135623730951;
  const double m = big ? 0.5 * u : u;
  const double f = m - 1.0;
  const double s = f * rcp_pos(2.0 + f), s2 = s * s;
  // sum_{i=0..9} s2^i / (2 i + 3) by Estrin's scheme (depth 4 instead of 10; same measured accuracy)
  const double s4 = s2 * s2, s8 = s4 * s4, s16 = s8 * s8;
  const double a0 = fma(s2, 1.0 / 5.0, 1.0 / 3.0), a1 = fma(s2, 1.0 / 9.0, 1.0 / 7.0), a2 = fma(s2, 1.0 / 13.0, 1.0 / 11.0);
  const double a3 = fma(s2, 1.0 / 17.0, 1.0 / 15.0), a4 = fma(s2, 1.0 / 21.0, 1.0 / 19.0);
  double q = fma(a4, s16, fma(fma(a3, s4, a2), s8, fma(a1, s4, a0)));
  q *= s2;
  const double two_s = 2.0 * s;
  return (big ? 0.6931471805599453 : 0.0) + fma(two_s, q, two_s) + c * inv;
}

// ---- T4 on the FP64 tensor cores: block-cooperative gradient with DMMA fragments and TMA-staged row tiles ----------
// Same protocol as LogRegCoopT (8 chains per CTA of 8 warps, publish -> coop_eval -> collect), different engine:
//   * the 8 lock-stepped chains of the CTA are the N = 8 dimension of `mma.sync.m8n8k4.f64` (SASS DMMA.8x8x4);
//   * X is streamed in tiles of 8 rows (8 P doubles, contiguous in row-major X) by per-warp bulk async copies
//     (`cp.async.bulk`, TMA engine, SASS UBLKCP) into a private 3-stage ring in shared memory, completing on per-stage
//     mbarriers; the warp that consumes a stage also refills it, so the main loop has no CTA-wide barrier at all;
//   * phase 1: eta[8 rows x 8 chains] = X_tile[8 x P] beta[P x 8]: beta lives in registers as B fragments for the
//     whole evaluation (one double per lane per 4 coordinates), A fragments come from the staged tile
//     (conflict-free: row stride P = 100 doubles puts the 4 rows of a half-warp 8 banks apart); 4 accumulators
//     break the dependent-DMMA chain;
//   * r = y - sigmoid(eta) on the C fragment (2 values per lane; branch-free exp / reciprocal / log1p above),
//     re-laid out as two B fragments by 4 shuffles;
//   * phase 2: grad[P x 8 chains] += X_tile^T[P x 8 rows] r[8 rows x 8]: A fragments are the transposed read of
//     the same staged tile (also conflict-free), accumulators stay in registers (2 doubles per lane per 8 coords);
//   * software pipeline: trip j runs phase 1 of tile j next to sigmoid + phase 2 of tile j - 1 (independent
//     instruction streams in one basic block; loop bounds are compile-time through PCAP >= P);
//   * the 8 warps' partial gradients are combined in a fixed order through the (then idle) stage buffers.
// Per CTA-evaluation X is read once from L2 (80 MB for N = 100 000, P = 100; it fits the 126 MB L2); per 8-row tile
// a warp issues PCAP/4 + PCAP/4 DMMA (52 for PCAP = 104) against as many shared loads.
template <int G, int E2, int PCAP>
struct LogRegMmaTP {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = true;
  static constexpr int NTC = 256, NW = 8, C = 8, PMAX = 128, KS = PCAP / 4, CT = PCAP / 8, RT = 8, S = 3;
  static constexpr int WSTAGE = S * RT * PCAP;      // doubles of stage ring per warp
  static_assert(G == 32 && E2 == 2 && PCAP % 8 == 0 && PCAP <= 104, "tensor-core logistic regression: one warp per chain, P <= 104");
  static_assert(WSTAGE >= CT * 64, "the ring doubles as the reduction buffer");
  // shared: bs[PMAX][C] | gs[C][PMAX] | lps[NW][C] | act[C] | need[C] | full[NW][4] | ring[NW][WSTAGE] | pad[PMAX]
  __host__ __device__ static constexpr int smem_doubles(int) {
    return PMAX * C + C * PMAX + NW * C + 2 * C + NW * 4 + NW * WSTAGE + PMAX;
  }
  const double *X, *y;
  int N, P;
  double itau2;
  double *bs, *gs, *lps, *act, *need, *ring;
  uint64_t* full;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int, double* tsm) {
    X = tp.p0; y = tp.p1; N = tp.n0; P = d; itau2 = tp.c0;
    bs = tsm; gs = bs + PMAX * C; lps = gs + C * PMAX; act = lps + NW * C; need = act + C;
    full = reinterpret_cast<uint64_t*>(need + C);
    ring = need + C + NW * 4;
    for (int i = threadIdx.x; i < PMAX * C; i += NTC) bs[i] = 0.0;
    for (int i = threadIdx.x; i < NW * WSTAGE + PMAX; i += NTC) ring[i] = 0.0;   // stale reads must be finite
    if (threadIdx.x == 0) {
      for (int i = 0; i < NW * 4; ++i) mbar_init(&full[i], 1);
      mbar_fence_init();
    }
    __syncthreads();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __device__ __forceinline__ double lp_grad(const double (&)[E], double (&)[E], double*, int&) const { return 0.0; }

  // see LogRegCoopT::publish
  __device__ __forceinline__ void publish(const double (&q)[E], bool active, bool need_lp) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      if (k < P) bs[k * C + w] = active ? q[e] : 0.0;
    }
    if (t == 0) { act[w] = active ? 1.0 : 0.0; need[w] = (active && need_lp) ? 1.0 : 0.0; }
  }

  __device__ __forceinline__ static void dmma(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
  }

  // `gt`: number of tiles this warp has consumed so far, modulo 2S (kept by the caller across evaluations): tile g
  // lives in stage g % S of the warp's ring and completes phase (g / S) & 1 of that stage's mbarrier.
  __device__ __forceinline__ void coop_eval(uint32_t& gt) const {
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int lr = lane >> 2, lc = lane & 3;       // fragment coordinates
    bool any = false, anyneed = false;
#pragma unroll
    for (int c = 0; c < C; ++c) { any = any || (act[c] != 0.0); anyneed = anyneed || (need[c] != 0.0); }
    if (!any) {
      // no chain of the CTA is in a pass: leave through a barrier, so that no warp can publish the NEXT trip's flags
      // while another one is still reading this trip's
      __syncthreads();
      return;
    }
    const bool nl0 = need[2 * lc] != 0.0, nl1 = need[2 * lc + 1] != 0.0;
    // beta as B fragments: B[k = 4 kk + lc][n = chain lr]
    double bf[KS];
#pragma unroll
    for (int kk = 0; kk < KS; ++kk) bf[kk] = bs[(4 * kk + lc) * C + lr];      // rows >= P of bs are zero
    double ga[CT][2];
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) ga[ct][0] = ga[ct][1] = 0.0;
    double lp0 = 0.0, lp1 = 0.0;

    const int ntile = (N + RT - 1) / RT;
    const int mine = (ntile > w) ? (ntile - w + NW - 1) / NW : 0;     // tiles w, w + NW, ...
    const int stage_d = RT * P;                                       // doubles per stage
    double* myring = ring + w * WSTAGE;
    uint64_t* mybar = full + w * 4;
    auto issue = [&](int j) {     // lane 0: start the copy of my j-th tile
      const uint32_t g = gt + (uint32_t)j;
      const int st_ = (int)(g % (uint32_t)S);
      const int n0 = (w + j * NW) * RT;
      const int nrows = min(RT, N - n0);
      const uint32_t bytes = (uint32_t)(nrows * P * 8);
      if ((bytes & 15u) == 0u) {
        mbar_expect_tx(&mybar[st_], bytes);
        bulk_g2s(myring + st_ * stage_d, X + (size_t)n0 * P, bytes, &mybar[st_]);
      } else {
        // ragged last tile whose byte count is not a multiple of 16: plain copy, then complete the phase
        for (int i = 0; i < nrows * P; ++i) myring[st_ * stage_d + i] = __ldg(X + (size_t)n0 * P + i);
        mbar_arrive(&mybar[st_]);
      }
    };
    if (lane == 0 && mine > 0) issue(0);

    // software pipeline: trip jj = phase 1 of tile jj  ||  sigmoid + phase 2 of tile jj - 1
    double ep[2] = {0.0, 0.0};        // eta of the previous tile (C fragment)
    double yp = 0.0;                  // its y (row lr)
    bool okp = false;                 // its row lr exists
    const double* sxp = myring;       // its stage
    for (int jj = 0; jj <= mine; ++jj) {
      // stage of tile jj + 1 held tile jj - 2, released by the __syncwarp at the end of the previous trip
      if (lane == 0 && jj + 1 < mine) issue(jj + 1);
      double e4[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
      double yn = 0.0;
      bool okn = false;
      const double* sxn = myring;
      if (jj < mine) {
        const uint32_t g = gt + (uint32_t)jj;
        sxn = myring + (g % (uint32_t)S) * stage_d;
        const int n0 = (w + jj * NW) * RT;
        const int nrows = min(RT, N - n0);
        okn = lr < nrows;
        yn = okn ? __ldg(y + n0 + lr) : 0.0;
        mbar_wait(&mybar[g % (uint32_t)S], (g / (uint32_t)S) & 1u);
        if (nrows < RT) {            // partial last tile: rows beyond the data must be finite for phase 2
          for (int i = nrows * P + lane; i < RT * P; i += 32) const_cast<double*>(sxn)[i] = 0.0;
          __syncwarp();
        }
      }
      // ---- phase 1 (tile jj): eta = X_tile beta ----
      {
        const double* ar = sxn + lr * P + lc;
#pragma unroll
        for (int kk = 0; kk < KS; ++kk) {
          const double a = (4 * kk + lc < P) ? ar[4 * kk] : 0.0;
          dmma(e4[kk & 3], a, bf[kk]);
        }
      }
      // ---- tile jj - 1: residuals on the C fragment (row lr, chains 2 lc and 2 lc + 1) ----
      double r[2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const double et = ep[i];
        const double ex = exp_nonpos(-fabs(et));
        const double inv = rcp_pos(1.0 + ex);
        const double sig = (et >= 0.0) ? inv : ex * inv;
        r[i] = okp ? (yp - sig) : 0.0;
        if (anyneed) {               // CTA-uniform: some chain ends a pass with this step
          const double term = yp * et - (fmax(et, 0.0) + log1p_unit(ex, inv));
          if (i == 0) lp0 += (nl0 && okp) ? term : 0.0;
          else lp1 += (nl1 && okp) ? term : 0.0;
        }
      }
      // C fragment -> B fragments: B[k = row lc (+4)][n = chain lr] lives in lane 4 row + lr / 2, element lr & 1
      const int s0 = 4 * lc + (lr >> 1), s1 = 4 * (4 + lc) + (lr >> 1);
      const double x00 = __shfl_sync(0xffffffffu, r[0], s0), x01 = __shfl_sync(0xffffffffu, r[1], s0);
      const double x10 = __shfl_sync(0xffffffffu, r[0], s1), x11 = __shfl_sync(0xffffffffu, r[1], s1);
      const double b0 = (lr & 1) ? x01 : x00, b1 = (lr & 1) ? x11 : x10;
      // ---- phase 2 (tile jj - 1): grad[coord 8 ct + lr][chain] += X[n0 + k][coord] r[k][chain]; r = 0 in trip 0 ----
      {
        const double* at0 = sxp + lc * P + lr;
        const double* at1 = sxp + (4 + lc) * P + lr;
#pragma unroll
        for (int ct = 0; ct < CT; ++ct) dmma(ga[ct], at0[8 * ct], b0);
#pragma unroll
        for (int ct = 0; ct < CT; ++ct) dmma(ga[ct], at1[8 * ct], b1);
      }
      ep[0] = (e4[0][0] + e4[1][0]) + (e4[2][0] + e4[3][0]);
      ep[1] = (e4[0][1] + e4[1][1]) + (e4[2][1] + e4[3][1]);
      yp = yn;
      okp = okn;
      sxp = sxn;
      __syncwarp();      // every lane is done with the stage of tile jj - 1 before lane 0 refills it
    }
    // stage (g % S) and mbarrier phase ((g / S) & 1) only depend on g mod 2S: keep the counter bounded so that a
    // launch of any length never wraps it
    gt = (gt + (uint32_t)mine) % (uint32_t)(2 * S);

    // ---- combine the 8 warps' partial gradients (fixed order) through the idle rings ----
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      myring[(ct * 32 + lane) * 2] = ga[ct][0];
      myring[(ct * 32 + lane) * 2 + 1] = ga[ct][1];
    }
    {
      double v0 = lp0, v1 = lp1;
#pragma unroll
      for (int off = 16; off >= 4; off >>= 1) {
        v0 += __shfl_xor_sync(0xffffffffu, v0, off);
        v1 += __shfl_xor_sync(0xffffffffu, v1, off);
      }
      if (lr == 0) { lps[w * C + 2 * lc] = v0; lps[w * C + 2 * lc + 1] = v1; }
    }
    __syncthreads();
    for (int o = tid; o < C * PMAX; o += NTC) {
      const int c = o / PMAX, k = o % PMAX;
      double s = 0.0;
      if (k < P) {
        // ga[ct = k / 8] of lane (k % 8) * 4 + c / 2, element c & 1
        const int idx = ((k >> 3) * 32 + (k & 7) * 4 + (c >> 1)) * 2 + (c & 1);
#pragma unroll
        for (int ww = 0; ww < NW; ++ww) s += ring[ww * WSTAGE + idx];
      }
      gs[c * PMAX + k] = s;
    }
    __syncthreads();
    // a diverged chain may have left non-finite partials in the ring: stale reads must stay finite
#pragma unroll
    for (int ct = 0; ct < CT; ++ct) {
      myring[(ct * 32 + lane) * 2] = 0.0;
      myring[(ct * 32 + lane) * 2 + 1] = 0.0;
    }
    __syncwarp();
    // the rings are rewritten by bulk copies (async proxy) in the next evaluation
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }

  // gradient of this warp's chain (after coop_eval); returns this thread's partial of lp
  __device__ __forceinline__ double collect(const double (&q)[E], double (&g)[E]) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
    double qq = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      g[e] = (k < P) ? fma(-itau2, q[e], gs[w * PMAX + k]) : 0.0;
      qq = fma(q[e], q[e], qq);
    }
    double lp = -0.5 * itau2 * qq;
    if (t == 0) {
#pragma unroll
      for (int ww = 0; ww < NW; ++ww) lp += lps[ww * C + w];
    }
    return lp;
  }
};
template <int G, int E2>
using LogRegMma32T = LogRegMmaTP<G, E2, 32>;
template <int G, int E2>
using LogRegMma104T = LogRegMmaTP<G, E2, 104>;

}  // namespace wn

namespace wn {

// ---- dense-precision Gaussian (north_star: "tensor cores only where the gradient really is a dense contraction across
// lock-stepped chains"): lp = -1/2 q^T P q, grad = -P q with a dense symmetric positive-definite precision matrix P
// [d, d] (row-major, data key "precision").  Not in the reference (its Gaussians are diagonal or 2-d: targetDistr.py:18-31).
//
// Per-warp version (G = 32): serves package mode, the warm-up adaptation and the extended integrators.  The chain's q is
// published to the warp's shared row; lane t forms the rows of its own coordinates with FMAs, P read through L2.
template <int G, int E2>
struct DenseGaussT {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = true;     // the block's chains stream the same rows of P: keep them in step
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = false;
  static constexpr int PMAX = 2 * G * E2;
  static_assert(G == 32, "dense Gaussian target: one warp per chain");
  __host__ __device__ static constexpr int smem_doubles(int NT) { return (NT / 32) * PMAX; }
  const double* Pm;
  int d_;
  double* qs;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int, double* tsm) {
    Pm = tp.p0; d_ = d;
    qs = tsm + (threadIdx.x >> 5) * PMAX;
  }
  __device__ __forceinline__ double lp_grad(const double (&q)[E], double (&g)[E], double*, int&) const {
    const int t = threadIdx.x & 31;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; ++e) qs[coord_of<G>(e, t)] = q[e];
    __syncwarp();
    double lp = 0.0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int r = coord_of<G>(e, t);
      double acc = 0.0;
      if (r < d_) {
        const double* row = Pm + (size_t)r * d_;
        for (int k = 0; k < d_; ++k) acc = fma(__ldg(row + k), qs[k], acc);
      }
      g[e] = -acc;
      lp = fma(q[e], acc, lp);
    }
    return -0.5 * lp;
  }
};

// Tensor-core version for the plain WALNUTSpy kernels: the 8 lock-stepped chains of a CTA are the N = 8 of
// `mma.sync.m8n8k4.f64` (SASS DMMA.8x8x4), exactly as in LogRegMmaTP: G[d x 8 chains] = P[d x d] Q[d x 8].  P streams in
// tiles of 8 rows (8 d doubles, contiguous) through per-warp 3-stage rings filled by bulk async copies (TMA engine,
// SASS UBLKCP) on per-stage mbarriers; Q lives in registers as B fragments for the whole evaluation; the C fragment of a
// tile IS the gradient of its 8 coordinates for the 8 chains, and q . (P q) accumulates the log density on the way.
template <int G, int E2, int PCAP>
struct DenseGaussMmaTP {
  static constexpr int E = 2 * E2;
  static constexpr bool PAIR_LAYOUT = true;
  static constexpr bool BLOCK_LOCKSTEP = false;
  static constexpr bool LAZY_ENERGY = false;
  static constexpr bool COOP = true;
  static constexpr int NTC = 256, NW = 8, C = 8, PMAX = 128, KS = PCAP / 4, RT = 8, S = 3;
  static constexpr int WSTAGE = S * RT * PCAP;
  static_assert(G == 32 && E2 == 2 && PCAP % 8 == 0 && PCAP <= 104, "tensor-core dense Gaussian: one warp per chain, d <= 104");
  // shared: bs[PMAX][C] | gs[C][PMAX] | lps[NW][C] | act[C] | full[NW][4] | ring[NW][WSTAGE]
  __host__ __device__ static constexpr int smem_doubles(int) { return PMAX * C + C * PMAX + NW * C + C + NW * 4 + NW * WSTAGE; }
  const double* Pm;
  int P;
  double *bs, *gs, *lps, *act, *ring;
  uint64_t* full;
  __device__ __forceinline__ int coord(int e, int t) const { return coord_of<G>(e, t); }
  __device__ __forceinline__ void init(const TargetParams& tp, int d, int, double* tsm) {
    Pm = tp.p0; P = d;
    bs = tsm; gs = bs + PMAX * C; lps = gs + C * PMAX; act = lps + NW * C;
    full = reinterpret_cast<uint64_t*>(act + C);
    ring = act + C + NW * 4;
    for (int i = threadIdx.x; i < PMAX * C; i += NTC) { bs[i] = 0.0; gs[i] = 0.0; }
    for (int i = threadIdx.x; i < NW * WSTAGE; i += NTC) ring[i] = 0.0;      // stale reads must be finite
    if (threadIdx.x == 0) {
      for (int i = 0; i < NW * 4; ++i) mbar_init(&full[i], 1);
      mbar_fence_init();
    }
    __syncthreads();
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __device__ __forceinline__ double lp_grad(const double (&)[E], double (&)[E], double*, int&) const { return 0.0; }

  __device__ __forceinline__ void publish(const double (&q)[E], bool active, bool) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      if (k < P) bs[k * C + w] = active ? q[e] : 0.0;
    }
    if (t == 0) act[w] = active ? 1.0 : 0.0;
  }

  __device__ __forceinline__ static void dmma(double (&c)[2], double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
  }

  // `gt`: tiles consumed so far by this warp modulo 2 S (stage g % S, mbarrier phase (g / S) & 1), kept by the caller
  __device__ __forceinline__ void coop_eval(uint32_t& gt) const {
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int lr = lane >> 2, lc = lane & 3;
    bool any = false;
#pragma unroll
    for (int c = 0; c < C; ++c) any = any || (act[c] != 0.0);
    if (!any) {
      // no chain of the CTA is in a pass: leave through a barrier, so that no warp can publish the NEXT trip's flags
      // while another one is still reading this trip's
      __syncthreads();
      return;
    }
    double bf[KS];                                   // Q as B fragments: B[k = 4 kk + lc][n = chain lr]
#pragma unroll
    for (int kk = 0; kk < KS; ++kk) bf[kk] = bs[(4 * kk + lc) * C + lr];
    double lp0 = 0.0, lp1 = 0.0;
    const int ntile = (P + RT - 1) / RT;
    const int mine = (ntile > w) ? (ntile - w + NW - 1) / NW : 0;
    const int stage_d = RT * P;
    double* myring = ring + w * WSTAGE;
    uint64_t* mybar = full + w * 4;
    auto issue = [&](int j) {
      const uint32_t g = gt + (uint32_t)j;
      const int st_ = (int)(g % (uint32_t)S);
      const int n0 = (w + j * NW) * RT;
      const int nrows = min(RT, P - n0);
      const uint32_t bytes = (uint32_t)(nrows * P * 8);
      if ((bytes & 15u) == 0u && ((((size_t)n0 * P) & 1u) == 0u)) {
        mbar_expect_tx(&mybar[st_], bytes);
        bulk_g2s(myring + st_ * stage_d, Pm + (size_t)n0 * P, bytes, &mybar[st_]);
      } else {       // odd d: a tile is not 16-byte aligned / sized -- plain copy, then complete the phase
        for (int i = 0; i < nrows * P; ++i) myring[st_ * stage_d + i] = __ldg(Pm + (size_t)n0 * P + i);
        mbar_arrive(&mybar[st_]);
      }
    };
    if (lane == 0) {
      if (mine > 0) issue(0);
      if (mine > 1) issue(1);
    }
    for (int jj = 0; jj < mine; ++jj) {
      const uint32_t g = gt + (uint32_t)jj;
      const double* sx = myring + (g % (uint32_t)S) * stage_d;
      const int n0 = (w + jj * NW) * RT;
      const int nrows = min(RT, P - n0);
      mbar_wait(&mybar[g % (uint32_t)S], (g / (uint32_t)S) & 1u);
      double e4[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
      const double* ar = sx + lr * P + lc;
      const bool rowok = lr < nrows;
#pragma unroll
      for (int kk = 0; kk < KS; ++kk) {
        const double a = (rowok && 4 * kk + lc < P) ? ar[4 * kk] : 0.0;
        dmma(e4[kk & 3], a, bf[kk]);
      }
      const double r0 = (e4[0][0] + e4[1][0]) + (e4[2][0] + e4[3][0]);     // (P q)[row n0 + lr][chain 2 lc]
      const double r1 = (e4[0][1] + e4[1][1]) + (e4[2][1] + e4[3][1]);     //                   [chain 2 lc + 1]
      if (rowok) {
        const int row = n0 + lr;
        gs[(2 * lc) * PMAX + row] = -r0;
        gs[(2 * lc + 1) * PMAX + row] = -r1;
        lp0 = fma(bs[row * C + 2 * lc], r0, lp0);
        lp1 = fma(bs[row * C + 2 * lc + 1], r1, lp1);
      }
      __syncwarp();      // every lane is done with this stage before lane 0 refills it
      if (lane == 0 && jj + 2 < mine) issue(jj + 2);
    }
    gt = (gt + (uint32_t)mine) % (uint32_t)(2 * S);
    {
      double v0 = lp0, v1 = lp1;
#pragma unroll
      for (int off = 16; off >= 4; off >>= 1) {
        v0 += __shfl_xor_sync(0xffffffffu, v0, off);
        v1 += __shfl_xor_sync(0xffffffffu, v1, off);
      }
      if (lr == 0) { lps[w * C + 2 * lc] = v0; lps[w * C + 2 * lc + 1] = v1; }
    }
    __syncthreads();
    // the rings are rewritten by bulk copies (async proxy) in the next evaluation
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }

  __device__ __forceinline__ double collect(const double (&)[E], double (&g)[E]) const {
    const int w = threadIdx.x >> 5, t = threadIdx.x & 31;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int k = coord_of<G>(e, t);
      g[e] = (k < P) ? gs[w * PMAX + k] : 0.0;
    }
    double lp = 0.0;
    if (t == 0) {
#pragma unroll
      for (int ww = 0; ww < NW; ++ww) lp += lps[ww * C + w];
      lp *= -0.5;
    }
    return lp;
  }
};
template <int G, int E2>
using DenseGaussMma32T = DenseGaussMmaTP<G, E2, 32>;
template <int G, int E2>
using DenseGaussMma104T = DenseGaussMmaTP<G, E2, 104>;

}  // namespace wn
