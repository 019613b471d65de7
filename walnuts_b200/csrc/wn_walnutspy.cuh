// Persistent many-chain kernel for the WALNUTSpy transition (reference WALNUTSpy/WALNUTS.py:189-695
// driver + WALNUTSpy/adaptiveIntegrators.py:49-137,361-475 macro steps).
//
// One group of G threads owns one chain at a time and keeps (q, v, g) of the active orbit end in
// registers for the whole transition.  The kernel is ONE flat loop whose body is a leapfrog
// micro-step; everything else (step-size search bookkeeping, tree logic, state selection, momentum
// refresh, output) is a small state machine entered only when a pass of 2^c micro-steps ends.  So
// chains that sit at different tree depths / different c never serialise each other's hot loop --
// the SIMT analogue of "lock-free" chains.  Groups pull chains from a global queue.
//
// Per-chain memory outside registers (DESIGN.md section 3):
//   registers : q, v, g of the working state, target constants, 6 hot scalars
//   shared    : checkpoint of the macro-step start state S, later the accepted out state O (3 vectors);
//               the cold control block `Ctl` (one copy per warp; per-thread local copy when G < 32)
//   global    : slot-indexed scratch (other orbit end, two proposal slots, left-end stack of <= M
//               pending dyadic levels) -- indexed by resident slot, not by chain, so it stays L2-sized.
#pragma once
#include <type_traits>

#include "wn_common.cuh"
#include "wn_targets.cuh"

namespace wn {

struct RunParams {
  int n_chains, d, dg, M, kind, minC, maxC;
  int n_iter;
  int compat;           // 1: reproduce reference quirk A14(i) (WALNUTS.py:420 has no counterpart after :443-459)
  uint32_t iter0;       // iteration number of the first transition of this call (1-based)
  uint32_t seed_lo, seed_hi;
  uint32_t chain_offset;
  double H0, delta0, jitter, p0, log_p0, log_1mp0;
  const double* Hstep;  // [n_chains] or null
  const double* delta;  // [n_chains] or null
  double* state;        // [n_chains, d]
  double* draws;        // [n_iter, n_chains, dg] or null
  double* diag;         // [n_iter, n_chains, 24] or null
  double* orbit_min;    // [n_iter, n_chains, dg] or null: recordOrbitStats (WALNUTS.py:182-184,274-276,...)
  double* orbit_max;
  unsigned long long* nevalF;  // [n_chains] or null
  unsigned long long* nevalB;
  unsigned long long* totals;  // [2] grid totals (forward, backward)
  double2* scratch;
  int nslot;
  unsigned int* queue;
  const unsigned int* order;   // queue entries or null (wn_sched.cu): chain index, or 0xffffffff = this group retires
  const unsigned int* order_len;   // device word: number of queue entries
  unsigned int* cost;          // [n_chains] or null: gradient evaluations of the chain in this call (next call's order)
  TargetParams tp;
  // warm-up adaptation (reference WALNUTS.py:136-147, 313, 701-712); ADAPT kernels only
  int warmup_iter, adaptH, adaptDelta;
  double p2prob, adTarget, adQuant;
  double* adapt_state;   // [n_chains, WN_ADAPT_STRIDE]: H, delta, npush, q[5], n[5], hasNaN, nhist
  double* adapt_hist;    // [n_chains, warmup_iter]: sorted history of orbitEnergyError / delta
  // integratorAuxPar fields of the extended integrators (adaptiveIntegrators.py:36-44); EXT kernels only
  int maxFPiter;
  double FPtol, gradThresh;
};
#define WN_ADAPT_STRIDE 16

enum { KIND_FIXED = 0, KIND_D = 1, KIND_R2P = 2, KIND_YOSHIDA = 3 };   // 3: adaptYoshidaD (adaptiveIntegrators.py:142-240)
// EXT kernels: adaptLeapFrogFlowD (:246-356), adaptImplicitMidpointD (:478-641, fixed-point variant),
// adaptRescaledLeapFrogD (:660-762)
enum { KIND_FLOW = 4, KIND_MIDPOINT = 5, KIND_RESCALED = 6 };
#define WN_Y_FIRSTLAST 1.351207191959658
#define WN_Y_MIDDLE (-1.702414383919315)
enum { PH_FWD = 0, PH_REDO = 1, PH_BWD = 2, PH_INIT = 3 };
enum { ST_CHAIN = 0, ST_ITER, ST_ITER2, ST_LEVEL, ST_MACRO, ST_PASS_END, ST_LEAF, ST_LEVEL_END, ST_ITER_END, ST_RUN, ST_EXIT };

// scratch vector ids
enum { V_PARK_Q = 0, V_PARK_V = 1, V_PARK_G = 2, V_PROP0 = 3, V_PROP1 = 4, V_OMIN = 5, V_OMAX = 6, V_STACK = 7 };  // stack: 7 + 2*lvl (+1 for v)
__host__ __device__ inline int scratch_vectors(int M) { return V_STACK + 2 * (M + 1); }

#define WN_LOG_ZERO (-700.0)
#define WN_WT_SUM_THRESH 0x1.78694fe9f73ccp-1009 /* numpy exp(-699) = 2.680137958338607e-304, reference constants.py:14 */

// Cold per-chain control state.  Every thread of a group computes identical values, so a copy may be
// shared by the lanes of one warp (all lanes store the same value, then load it back).  Keeping it
// out of registers leaves the register file to the FP64 working set of the hot loop.
struct Ctl {
  uint32_t chain, iter, nseq, dirbits;
  int it, level, side, phase, c, If, Ib, cSim, maxTry;
  uint32_t nleaf, n_new;
  int maxInt0, maxInt1, L_, Lold, NdS, NdC, stopCode, propCur;
  int bothPassive, candValid, forced, wIntact, sHnan;
  int sN, sMinIf, sMaxIf, sMinC, sMaxC, sNne, sNz;
  double Hbig, delta, jlo, jhi, xi, h, h2, Ham0, Hfwd, H0, lwtf, lwt;
  double endH0, endH1, lwtSum0, lwtSum1, timeLen0, timeLen1;
  double WoldSum, WnewSum, indexStat, indexStatOld, orbitLen, orbitLenSam;
  double sMinL, sMaxL, sHmax, sHmin;
  unsigned long long nF, nB, chainF, chainB;
  // warm-up adaptation
  int warm, p2npush, p2n[5], adNaN, adNhist;
  double p2q[5], igr, maxd, Hprev;
};

// Kernel sets (compile-time knowledge of the integrator: smaller code, no dead search logic):
//   KSET_ANY   every integrator behind the runtime P.kind (warm-up adaptation / extended-integrator families)
//   KSET_FIXED fixedLeapFrog only (plain NUTS); with a whole warp per chain the per-level loop nuts_level() replaces the
//              flat loop + state machine for the leaves
//   KSET_ADAPT adaptLeapFrogD / adaptLeapFrogR2P only
enum { KSET_ANY = 0, KSET_FIXED = 1, KSET_ADAPT = 2 };

// left-end stack levels of the plain-NUTS level loop that live in shared memory (levels 1..NSM; deeper ones in L2 scratch)
template <int G, int E2, int NT>
struct NutsCfg {
  // one level costs 2 * 2 E2 * NT doubles per block; more levels shrink the L1 carve-out (measured for 4 warps per
  // chain at d = 1000: 2 levels 3.45e8, 4 levels 3.15e8 grad evals/s)
  static constexpr int NSM = 2;
};
// one warp holds a whole d = 1000 chain (32 coordinates per lane): a level costs 16 KB per chain, one level fits
template <int NT>
struct NutsCfg<32, 16, NT> {
  static constexpr int NSM = 1;
};
// targets whose per-thread energy partials are non-negative (pass-end failure certificate)
template <class T, class = void>
struct has_nonneg : std::false_type {};
template <class T>
struct has_nonneg<T, std::void_t<decltype(T::NONNEG_ENERGY)>> : std::bool_constant<T::NONNEG_ENERGY> {};
// targets whose gradient is cheap to recompute from q (grad_only) need not keep g in registers between leaves
template <class T, class = void>
struct has_regrad : std::false_type {};
template <class T>
struct has_regrad<T, std::void_t<decltype(T::REGRAD)>> : std::bool_constant<T::REGRAD> {};

template <class Target, int G, int ADAPT, int KSET>
struct NutsFast {
  static constexpr bool value = (KSET == KSET_FIXED) && (G >= 32) && !Target::COOP && !Target::BLOCK_LOCKSTEP && !ADAPT;
};
// dynamic shared memory of walnutspy_kernel in doubles: checkpoint (or the plain-NUTS left-end slots + uniform buffer),
// reduction scratch, target
template <template <int, int> class TargetTT, int G, int E2, int NT, bool ADAPT, int KSET>
__host__ __device__ constexpr int wpy_smem_doubles() {
  using Target = TargetTT<G, E2>;
  constexpr bool NF = NutsFast<Target, G, ADAPT, KSET>::value;
  return (NF ? 2 * NutsCfg<G, E2, NT>::NSM : 3) * 2 * E2 * NT + (NF ? 2 * NT : 0) +
         Group<G, (G > NT) ? NT : G>::RED_DOUBLES + Target::smem_doubles(NT);
}

// CTLSM: the cold control block of chains that SHARE a warp (G < 32) lives in shared memory (one copy per chain)
// instead of per-thread registers / local memory -- fewer registers, more resident warps (G >= 32 always does).
// G > NT: one chain per thread-block CLUSTER of CL = G / NT CTAs (launched with the cluster dimension CL); thread t of
// the chain group is thread threadIdx.x of cluster rank t / NT.  Everything per chain that lives in shared memory
// (control block, checkpoint, left-end slots, uniform buffer) is replicated or split per CTA exactly as for a
// one-CTA group; only the Group<G, NT> reductions, the pass-end vote, the adaptation history and the queue grab cross
// CTAs.
template <template <int, int> class TargetTT, int G, int E2, int NT, int MINB = 1, bool ADAPT = false, bool EXT = false,
          int KSET = KSET_ANY, bool CTLSM = false>
__global__ void __launch_bounds__(NT, MINB) walnutspy_kernel(const __grid_constant__ RunParams P) {
  static_assert(!EXT || ADAPT, "EXT kernels are built with the adaptation code (inactive without wn_set_adapt)");
  static_assert(KSET == KSET_ANY || (!ADAPT && !EXT), "specialised kernel sets exist for the plain family only");
  constexpr int E = 2 * E2;
  constexpr int GPB = NT / G;  // groups per block (0 for a cluster group: unused there)
  static_assert((G <= NT) ? (NT % G == 0 && (G <= 32 || NT == G))
                          : (G % NT == 0 && NT % 32 == 0 && (G / NT == 2 || G / NT == 4 || G / NT == 8)),
                "block must hold whole groups, or a cluster of 2, 4 or 8 blocks one group");
  // Grp::CL: CTAs per chain.  (Read from the group type, not declared as a local constant: an extra constexpr local
  // changed the code ptxas emits for some existing kernels.)
  using Grp = Group<G, (G > NT) ? NT : G>;
  using Target = TargetTT<G, E2>;
  static_assert(Grp::CL == 1 || (!Target::COOP && !Target::BLOCK_LOCKSTEP),
                "block-cooperative and lock-stepped targets need every chain of a block inside that block");
  constexpr bool NUTS_FAST = NutsFast<Target, G, ADAPT, KSET>::value;
  constexpr int NSM = NutsCfg<G, E2, NT>::NSM;
  constexpr bool LAZY = Target::LAZY_ENERGY && KSET != KSET_FIXED;   // plain NUTS consumes every step's energy
  constexpr bool REGRAD = NUTS_FAST && has_regrad<Target>::value;      // g is recomputed, never carried
  // integrator predicates: compile-time where the kernel set fixes them
  auto is_fixed = [&]() -> bool { return KSET == KSET_FIXED || (KSET == KSET_ANY && P.kind == KIND_FIXED); };
  auto is_r2p = [&]() -> bool { return KSET != KSET_FIXED && P.kind == KIND_R2P; };

  extern __shared__ __align__(16) double smem[];
  double* ck = smem;                       // checkpoint: [3*E][NT]  (NUTS_FAST: left-end slots [NSM][2][E][NT])
  double* ubuf = smem + (NUTS_FAST ? 2 * NSM : 3) * E * NT;   // NUTS_FAST: buffered sequential uniforms, 2 per thread
  double* red = ubuf + (NUTS_FAST ? 2 * NT : 0);              // reduction scratch (G > 32; Grp::RED_DOUBLES)
  __shared__ uint32_t sh_bcast;
  constexpr bool CTL_SHARED = (G >= 32) || CTLSM;
  __shared__ Ctl sh_ctl[(G >= 32) ? NT / 32 : (CTLSM ? NT / G : 1)];
  __shared__ int sh_ktab[(G >= 32) ? NT / 32 : 1][32];   // lazy-energy passes: steps between magnitude checks, by c
  // G >= 32: one copy per warp in shared memory (volatile: every lane stores the same value, then reads it
  // back).  G < 32: several chains share a warp; either one shared copy per chain (CTLSM) or each thread keeps a
  // private copy which the compiler is free to hold in registers / spill to local memory as it sees fit.
  Ctl loc_ctl;
  using CtlRef = typename std::conditional<CTL_SHARED, volatile Ctl&, Ctl&>::type;
  CtlRef C = *(CTL_SHARED ? &sh_ctl[(G >= 32) ? (threadIdx.x >> 5) : (threadIdx.x / G)] : &loc_ctl);
  volatile int* ktab = sh_ktab[(G >= 32) ? (threadIdx.x >> 5) : 0];

  const int tid = threadIdx.x;
  const int t = (Grp::CL > 1) ? (int)cluster_rank() * NT + tid : tid % G;
  int parity = 0;

  // scratch addressing: vector vi, pair e2 -> scratch[((vi*E2 + e2) * nslot + slot) * G + t]; slot = chain group
  // (a cluster when G > NT: the grid is 1-D, so cluster c is blocks c CL .. c CL + CL - 1)
  // (computed on demand: a hoisted base pointer + stride would cost four live registers in the hot loop)
  auto sc = [&](int vi, int e2) -> double2* {
    const size_t slot = (Grp::CL > 1) ? (size_t)(blockIdx.x / Grp::CL) : (size_t)blockIdx.x * GPB + tid / G;
    return P.scratch + ((size_t)(vi * E2 + e2) * P.nslot + slot) * G + t;
  };

  Target target;
  target.init(P.tp, P.d, t, red + Grp::RED_DOUBLES);

  // ---- register-resident working state -----------------------------------------------------
  double q[E], v[E], g[E];
  // ---- hot scalars --------------------------------------------------------------------------
  uint32_t steps_left = 0;
  double hh = 0, ha = 0, hp = 0;
  int expmax = 0;          // max over the pass of the exponent field of the per-thread energy partial
  int smax = 0;            // lazy-energy passes: signed / unsigned max of the high words of q, v
  unsigned umax = 0;
  bool lazy = false;       // current pass skips intermediate energies
  int since = 0, lazyK = 2; // skipped steps since the last magnitude check / allowed between checks
  // register copy of the step-size search state: a failed attempt goes straight to the next one
  int rc = 0, rlim = 0;
  bool rsearch = false, rexact = false, rlazyok = false;
  double rh = 0, rHref = 0, rdelta = 0, rsign = 1.0;
  unsigned long long rEv = 0;
  const bool yoshida = (KSET == KSET_ANY) && (P.kind == KIND_YOSHIDA);
  const unsigned long long evmul = yoshida ? 3ull : 1ull;   // gradient evaluations per micro-step
  int ysub = 0;            // Yoshida: index of the next leapfrog inside the triple
  double hh0 = 0;          // Yoshida: the micro-step size the triple is built from
  // ADAPT: per-step energies of the forward passes (igrConst, adaptiveIntegrators.py:101,399,424)
  bool trackH = false;
  double hist[4];
  int nh = 0;
  unsigned long long totF = 0, totB = 0;

  // sequential scalar stream (STREAM_SEQ), draw n of the current iteration.  NUTS_FAST: the stream is counter-based,
  // so the group computes 2 G draws ahead at once (every thread one Philox block) into a shared buffer; a draw is
  // then one shared load instead of ten Philox rounds replicated by every warp of the chain.  A cluster group: every
  // CTA fills its own buffer with the same 2 NT draws (no DSMEM traffic, no cluster barrier).
  uint4 ublk = make_uint4(0u, 0u, 0u, 0u);
  uint32_t ublk_idx = 0xffffffffu;
  auto ufetch = [&](uint32_t n) -> double {
    RngKey key{P.seed_lo, P.seed_hi, C.chain, C.iter};
    if constexpr (NUTS_FAST) {
      constexpr uint32_t UB = 2u * ((Grp::CL > 1) ? NT : G);
      double* ub = ubuf + ((Grp::CL > 1) ? 0 : (tid / G) * UB);
      const int ut = (Grp::CL > 1) ? tid : t;   // this thread's Philox block within the buffer
      if ((n % UB) == 0u) {
        if constexpr (G > 32) __syncthreads(); else __syncwarp();
        double u0, u1;
        rng_uniform_pair(key, STREAM_SEQ, (n >> 1) + (uint32_t)ut, u0, u1);
        ub[2 * ut] = u0;
        ub[2 * ut + 1] = u1;
        if constexpr (G > 32) __syncthreads(); else __syncwarp();
      }
      return ub[n % UB];
    } else {
      // consecutive draws 2b, 2b + 1 share a Philox block: keep the last block (the stream is consumed in order)
      const uint32_t b = n >> 1;
      if (b != ublk_idx) {
        ublk = philox4x32_10(make_uint4(b, key.iter, key.chain, STREAM_SEQ), key.k0, key.k1);
        ublk_idx = b;
      }
      return (n & 1u) ? u53(ublk.z, ublk.w) : u53(ublk.x, ublk.y);
    }
  };
  auto useq = [&]() -> double {
    const uint32_t n = C.nseq;
    C.nseq = n + 1;
    return ufetch(n);
  };
  auto jit = [&](double u) -> double {
    const double lo = C.jlo;
    return __dadd_rn(lo, __dmul_rn(__dadd_rn(C.jhi, -lo), u));
  };
  // magnitude summary (track_state) of the checkpointed state: every attempt of a step-size search restarts from
  // the same checkpoint, so its bound check is done once per checkpoint, not once per pass
  int ckS = 0;
  unsigned ckU = 0;
  bool ckTracked = false;
  auto save_ck = [&]() {
    ckTracked = false;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      ck[(0 * E + e) * NT + tid] = q[e];
      ck[(1 * E + e) * NT + tid] = v[e];
      ck[(2 * E + e) * NT + tid] = g[e];
    }
  };
  auto load_ck = [&](double vsign) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      q[e] = ck[(0 * E + e) * NT + tid];
      v[e] = vsign * ck[(1 * E + e) * NT + tid];
      g[e] = ck[(2 * E + e) * NT + tid];
    }
  };
  auto track_state = [&]() {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const int hq = __double2hiint(q[e]), hv = __double2hiint(v[e]);
      smax = max(smax, max(hq, hv));
      umax = max(umax, max((unsigned)hq, (unsigned)hv));
    }
  };
  // ADAPT: fold the batched per-step energy partials into max |diff(Hams)| (adaptiveIntegrators.py:101)
  auto flush_hist = [&]() {
    if constexpr (ADAPT) {
      if (nh == 0) return;
      double x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = (i < nh) ? hist[i] : 0.0;
      Grp::template sum<4>(x, red, parity);
      double md = C.maxd, hpv = C.Hprev;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (i < nh) {
          const double dd = fabs(x[i] - hpv);
          md = (dd > md || dd != dd) ? dd : md;     // np.max propagates NaN
          hpv = x[i];
        }
      }
      C.maxd = md;
      C.Hprev = hpv;
      nh = 0;
    }
  };
  // ADAPT: P-squared quantile push, reference WALNUTSpy/P2quantile.py:41-89
  auto p2_push = [&](double xi) {
    if constexpr (ADAPT) {
      const int np_ = C.p2npush + 1;
      C.p2npush = np_;
      if (np_ <= 5) {
        C.p2q[np_ - 1] = xi;
        if (np_ == 5) {                       // np.sort(x), :45-47 (NaN sorts last)
          double a[5];
#pragma unroll
          for (int i = 0; i < 5; ++i) a[i] = C.p2q[i];
          // insertion sort, NaN treated as +infinity-like (placed last), stable
          for (int i = 1; i < 5; ++i) {
            const double key = a[i];
            int j = i - 1;
            while (j >= 0 && ((a[j] > key) || (a[j] != a[j] && key == key))) { a[j + 1] = a[j]; --j; }
            a[j + 1] = key;
          }
#pragma unroll
          for (int i = 0; i < 5; ++i) C.p2q[i] = a[i];
        }
        return;
      }
      double q_[5];
      int n_[5];
#pragma unroll
      for (int i = 0; i < 5; ++i) { q_[i] = C.p2q[i]; n_[i] = C.p2n[i]; }
      int k;                                   // findInterval, :31-39,49-57
      if (xi < q_[0]) { q_[0] = xi; k = 1; }
      else if (xi > q_[4]) { q_[4] = xi; k = 4; }
      else {
        k = 0;                                 // fall-through (None): n[None:5] += 1 increments all
        for (int i = 0; i < 4; ++i) if (xi < q_[i + 1]) { k = i + 1; break; }
      }
#pragma unroll
      for (int i = 0; i < 5; ++i) if (i >= k) n_[i] += 1;        // :60
      const double nn = (double)np_, pp = P.p2prob;
      const double npp[5] = {1.0, 0.5 * (nn - 1.0) * pp + 1.0, (nn - 1.0) * pp + 1.0,
                             (nn - 1.0) * (1.0 + pp) / 2.0 + 1.0, nn};
      for (int i = 2; i <= 4; ++i) {           // :70-89
        const int ni = n_[i - 1], nip = n_[i], nim = n_[i - 2];
        double di = npp[i - 1] - (double)ni;
        if ((di >= 1.0 && nip - ni > 1) || (di <= -1.0 && nim - ni < -1)) {
          const int dI = (di > 0.0) ? 1 : -1;
          const double qi = q_[i - 1];
          const double qip = qi + ((double)dI / (double)(nip - nim)) *
                                      ((double)(ni - nim + dI) * (q_[i] - qi) / (double)(nip - ni) +
                                       (double)(nip - ni - dI) * (qi - q_[i - 2]) / (double)(ni - nim));
          if (q_[i - 2] < qip && qip < q_[i]) q_[i - 1] = qip;
          else q_[i - 1] = qi + (double)dI * (q_[i + dI - 1] - qi) / (double)(n_[i + dI - 1] - n_[i - 1]);
          n_[i - 1] += dI;
        }
      }
#pragma unroll
      for (int i = 0; i < 5; ++i) { C.p2q[i] = q_[i]; C.p2n[i] = n_[i]; }
    }
  };
  auto start_pass = [&](int cc) {
    steps_left = (yoshida ? 3u : 1u) << cc;
    hh = rh * __longlong_as_double((long long)(1023 - cc) << 52);   // rh 2^-cc, exact (cc <= 30, rh normal)
    ha = 0.5 * hh;
    hh0 = hh;
    ysub = 0;
    expmax = 0;
    smax = 0;
    umax = 0;
    if constexpr (LAZY) {
      lazy = rlazyok && !rexact && (cc >= 2) && !trackH && !yoshida;
      if (lazy) {
        // the pass starts from a bounded state (registers = checkpoint up to the sign of v, which the two
        // accumulators treat symmetrically)
        if (ckTracked) { smax = ckS; umax = ckU; }
        else { track_state(); ckS = smax; ckU = umax; ckTracked = true; }
        since = 0;
        // One leapfrog step amplifies max(|q|,|v|) by at most Gamma (target-specific bound); checked states are
        // below 2^300, so up to floor(170 / log2 Gamma) steps may pass between checks while every skipped energy
        // stays finite: magnitudes < 2^470, terms q^2 s and v^2 < 2^(940 + 60), so their sum over d <= 2^15
        // coordinates (the largest dispatched) is < 2^1016 -- and below 2^1024 for any d < 2^23.  Gamma grows with
        // the step, so the interval is tabulated per c once per
        // iteration for the LARGEST jittered macro step (ST_ITER: ktab), a conservative bound for every macro step.
        if constexpr (G >= 32) {
          lazyK = ktab[cc];
        } else {
          const int lg = ((__double2hiint(target.step_growth(hh)) >> 20) & 0x7ff) - 1022;
          lazyK = (lg * 66 <= 170) ? 64 : ((int)__fdividef(170.0f, (float)lg) - 2);
          lazyK &= ~1;
        }
        if (lazyK < 2) lazy = false;
      }
    }
    if constexpr (ADAPT) {
      nh = 0;
      if (trackH) { C.maxd = 0.0; C.Hprev = rHref; }
    }
  };
  // U-turn criterion, reference WALNUTS.py:95-97; (ql, vl) read from scratch, the other state is the
  // register-resident end (q, xi*v).  Orientation: minus end = more backward state, tmp = qp - qm = xi (q - ql).
  // The signs are factored out of the sums: (xi v).(xi (q - ql)) = v.(q - ql) term by term, and
  // vl.(xi (q - ql)) = xi (vl.(q - ql)) because negating every product negates every partial sum exactly
  // (round-to-nearest is symmetric) -- bit-identical to the signed form at 3 instead of 5 FP64 instructions per
  // coordinate.
  auto uturn_vs = [&](int viq, int viv) -> bool {
    double x[2] = {0.0, 0.0};
#pragma unroll
    for (int e2 = 0; e2 < E2; ++e2) {
      const double2 ql = *sc(viq, e2), vl = *sc(viv, e2);
      const double t0 = q[2 * e2] - ql.x, t1 = q[2 * e2 + 1] - ql.y;
      x[0] = fma(v[2 * e2], t0, x[0]);
      x[0] = fma(v[2 * e2 + 1], t1, x[0]);  // v_cur(fwd time) . tmp
      x[1] = fma(vl.x, t0, x[1]);
      x[1] = fma(vl.y, t1, x[1]);           // xi (v_left . tmp)
    }
    Grp::template sum<2>(x, red, parity);
    return (x[0] < 0.0) || (C.xi * x[1] < 0.0);
  };
  // one leapfrog micro-step on the registers; reference adaptiveIntegrators.py:79-84 (:50-55 fixed)
  auto micro_step = [&](bool kick1 = true) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (kick1) v[e] = fma(ha, g[e], v[e]);
      q[e] = fma(hh, v[e], q[e]);
    }
    const double lpp = target.lp_grad(q, g, red, parity);
    double ke0 = 0.0, ke1 = 0.0;   // two partial sums: halves the dependent-FMA chain
#pragma unroll
    for (int e = 0; e < E; e += 2) {
      v[e] = fma(ha, g[e], v[e]);
      v[e + 1] = fma(ha, g[e + 1], v[e + 1]);
      ke0 = fma(v[e], v[e], ke0);
      ke1 = fma(v[e + 1], v[e + 1], ke1);
    }
    hp = fma(0.5, ke0 + ke1, -lpp);   // this thread's partial of H_k = -f + 1/2 sum v^2 (:84)
    // all(isfinite(Hams)) (:92) is tracked on the exponent field with integer ops, off the FP64 pipe
    expmax = max(expmax, __double2hiint(hp) & 0x7ff00000);
  };
  // The same step without the energy (targets with LAZY_ENERGY).  Instead, the magnitudes of q and v
  // are bounded: the high words are max-reduced as signed ints (largest positive value) and as
  // unsigned ints (largest-magnitude negative value) -- two 3-input integer max per coordinate, off the
  // FP64 pipe -- at the pass start and after every second skipped step.  With inv_var <= 2^60 and a
  // micro step <= 2^10 one leapfrog step amplifies |q|, |v| by at most 2^142 in the worst case; start_pass() derives the actual per-step bound Gamma and the number of steps
  // that may pass between two checks.
  auto micro_step_lazy = [&]() {
    if constexpr (LAZY) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        v[e] = fma(ha, g[e], v[e]);
        q[e] = fma(hh, v[e], q[e]);
      }
      target.grad_only(q, g);
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = fma(ha, g[e], v[e]);
    }
  };
  // Interior step of a skipped-energy run with MERGED kicks: the closing half kick of one step and the opening half
  // kick of the next use the same gradient, v + a g + a g = v + h g; with the linear gradient of the LAZY_ENERGY
  // targets (g = -s q) that is ONE FMA v + (-h s) q on a coefficient formed once per pass.  2 instead of 4 FP64
  // instructions per coordinate and step: q += h v; v += kc q.  (Rounding differs from the reference's two half
  // kicks by <= 1 ulp of v per step -- the same order as the FMA contraction documented in DESIGN.md section 5;
  // the parity suite, incl. the exact discrete diagnostics over 100 free-running transitions, is unchanged.)
  // v carries the opening half kick of the next step; the run ends with micro_step(false), which recomputes g.
  auto drift_kick = [&](const double (&kc)[E]) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      q[e] = fma(hh, v[e], q[e]);
      v[e] = fma(kc[e], q[e], v[e]);
    }
  };
  constexpr int LAZY_LIMIT = (1023 + 300) << 20;

  uint32_t coop_phase = 0;   // COOP targets: phase bits of the staging mbarriers
  int st = ST_CHAIN;
  // cluster group: no CTA reads a peer's shared memory before the peer runs (the first DSMEM access, in the first
  // queue grab, follows this barrier)
  if constexpr (Grp::CL > 1) cluster_sync();
  // ===================== plain NUTS (fixedLeapFrog), whole warps per chain: one doubling level ======================
  // Replaces ST_MACRO -> ST_RUN -> ST_PASS_END -> ST_LEAF of the flat loop for the n_new = 2^level leaves of a level
  // (reference WALNUTS.py:296-368 for level 0, :392-587 for the leaf pairs; adaptiveIntegrators.py:49-59 per leaf).
  // With lwt = 0, If = Ib = c = 0 for every leaf the bookkeeping collapses, so the level runs as a register-resident
  // loop over LEAF PAIRS (the unit of the reference's plan rows with |a - b| = 1, :394): both leaves are integrated,
  // then ONE group reduction delivers both energies and the two dot products of the pair's own U-turn check (span 2);
  // the bookkeeping of the two leaves follows in the reference's order, with early exit (the second leaf's integration
  // was speculative if the first one force-rejects -- its results are then simply not applied).  The left end of a
  // pending dyadic level <= NSM lives in shared memory (each thread reads back only what it wrote: no barrier), deeper
  // ones in the L2-resident scratch; a leaf m = 3 (mod 4) is only ever the left end of its own pair, i.e. half of all
  // left ends never leave the SM.  Sequential uniforms come from the buffered stream (ufetch).
  auto nuts_level = [&]() {
    if constexpr (NUTS_FAST) {
      const int level = C.level, side = C.side;
      const double H0 = C.H0;
      const uint32_t n_new = C.n_new;
      const double jlo = C.jlo, jhi = C.jhi;
      auto jitl = [&](double u) -> double { return __dadd_rn(jlo, __dmul_rn(__dadd_rn(jhi, -jlo), u)); };
      uint32_t nseq = C.nseq;
      double WnewSum = 0.0;
      double tl = side ? C.timeLen1 : C.timeLen0;
      int mi = side ? C.maxInt1 : C.maxInt0;
      const int dstep = side ? -1 : 1;
      double endH = side ? C.endH1 : C.endH0;
      double orbitLen = C.orbitLen;
      int sN = C.sN, sHnan = C.sHnan;
      double sHmax = C.sHmax, sHmin = C.sHmin;
      int L_ = C.L_, candValid = 0, stop999 = 0;
      double indexStat = C.indexStat;
      const int pvec = V_PROP0 + (C.propCur ^ 1);
      uint32_t nleaf = 0;
      unsigned long long nF = 0;
      int out = 0;   // 0: level complete, 1: forced reject, 2: sub-U-turn
      // scratch vectors of this chain: pair e2 of vector vi at scv(vi)[e2 * sstride] (one 64-bit address computation
      // per vector instead of one per pair)
      const size_t sstride = (size_t)P.nslot * G;
      auto scv = [&](int vi) -> double2* { return sc(vi, 0); };
      // left-end slot `lvl` (>= 1): (q, v) with v in the INTEGRATION convention of the level (forward-time velocity
      // = xi v).  With tmp = qp - qm = xi (q - ql) both products of the U-turn criterion lose their signs:
      // v_cur(fwd).tmp = (xi v).(xi (q - ql)) = v.(q - ql) and v_left(fwd).tmp = (xi vl).(xi (q - ql)) = vl.(q - ql),
      // exactly (multiplications by +-1 are exact), so neither the stores nor the checks multiply by xi.
      auto put_left = [&](int lvl) {
        if (lvl <= NSM) {
          double* b = ck + (size_t)(lvl - 1) * 2 * E * NT + tid;
#pragma unroll
          for (int e = 0; e < E; ++e) { b[e * NT] = q[e]; b[(E + e) * NT] = v[e]; }
        } else {
          double2* pq = scv(V_STACK + 2 * lvl);
          double2* pv = pq + E2 * sstride;
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) {
            pq[e2 * sstride] = make_double2(q[2 * e2], q[2 * e2 + 1]);
            pv[e2 * sstride] = make_double2(v[2 * e2], v[2 * e2 + 1]);
          }
        }
      };
      // partial sums of the U-turn criterion (WALNUTS.py:95-97) between the registers and left-end slot `lvl`:
      // a = v . (q - ql), b = vl . (q - ql); U-turn iff a < 0 or b < 0
      auto dots_left = [&](int lvl, double& a, double& b) {
        constexpr int NA = 1;   // (four interleaved sums measured slower at 254 registers: 4.48e8 against 4.80e8)
        double a0[NA], b0[NA];
#pragma unroll
        for (int k = 0; k < NA; ++k) { a0[k] = 0.0; b0[k] = 0.0; }
        if (lvl <= NSM) {
          const double* p = ck + (size_t)(lvl - 1) * 2 * E * NT + tid;
#pragma unroll
          for (int e = 0; e < E; ++e) {
            const double tt = q[e] - p[e * NT];
            a0[e % NA] = fma(v[e], tt, a0[e % NA]);
            b0[e % NA] = fma(p[(E + e) * NT], tt, b0[e % NA]);
          }
        } else {
          const double2* pq = scv(V_STACK + 2 * lvl);
          const double2* pv = pq + E2 * sstride;
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) {
            const double2 ql = pq[e2 * sstride], vl = pv[e2 * sstride];
            const double t0 = q[2 * e2] - ql.x, t1 = q[2 * e2 + 1] - ql.y;
            a0[(2 * e2) % NA] = fma(v[2 * e2], t0, a0[(2 * e2) % NA]);
            a0[(2 * e2 + 1) % NA] = fma(v[2 * e2 + 1], t1, a0[(2 * e2 + 1) % NA]);
            b0[(2 * e2) % NA] = fma(vl.x, t0, b0[(2 * e2) % NA]);
            b0[(2 * e2 + 1) % NA] = fma(vl.y, t1, b0[(2 * e2 + 1) % NA]);
          }
        }
        if constexpr (NA == 4) {
          a = (a0[0] + a0[1]) + (a0[2] + a0[3]);
          b = (b0[0] + b0[1]) + (b0[2] + b0[3]);
        } else {
          a = a0[0];
          b = b0[0];
        }
      };
      // proposal slot <- left-end slot `lvl` (the picked state is the first leaf of the pair)
      auto prop_from_left = [&](int lvl) {
        double2* dst = scv(pvec);
        if (lvl <= NSM) {
          const double* p = ck + (size_t)(lvl - 1) * 2 * E * NT + tid;
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) dst[e2 * sstride] = make_double2(p[(2 * e2) * NT], p[(2 * e2 + 1) * NT]);
        } else {
          const double2* src = scv(V_STACK + 2 * lvl);
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) dst[e2 * sstride] = src[e2 * sstride];
        }
      };
      // bookkeeping of one leaf with energy Hl, step h and weight Wnew = exp(-Hl + H0) (lwtSum = 0 for fixedLeapFrog,
      // WALNUTS.py:321-322,...; `ratio` = Wnew / (WnewSum + Wnew)): WALNUTS.py:302-328 / :401-429 / :440-467 and the
      // forward twins; returns false on a forced reject.  `pick` tells the caller to store the proposal.
      auto leaf_book = [&](double Hl, double h, double Wnew, double ratio, bool& pick) -> bool {
        ++nleaf;
        ++nF;
        mi += dstep;
        tl = tl + h;
        endH = Hl;
        ++sN;
        if (Hl != Hl) sHnan = 1;
        else { sHmax = fmax(sHmax, Hl); sHmin = fmin(sHmin, Hl); }
        pick = false;
        if (!finite_d(Hl)) {                                     // :316,350,414,457,501,544 (quirks A14 ii, iii)
          if (level == 0 || (nleaf & 1u)) stop999 = 1;
          return false;
        }
        if (level == 0) {
          WnewSum = Wnew;
          pick = true;                                           // :326,359
        } else {
          const double ws = WnewSum + Wnew;
          WnewSum = ws;
          if (ws > WN_WT_SUM_THRESH) pick = ufetch(nseq++) < ratio;   // :426,464,512,554
          orbitLen = orbitLen + h;                               // :432,...
        }
        if (pick) {
          candValid = 1;
          L_ = mi;
          indexStat = side ? -tl : tl;
        }
        return true;
      };
      const bool odd_lane = (tid & 1) != 0;
      // (one code instance each of the leapfrog step and of the dot products: the loops over the pair's two leaves and
      //  over the spans are NOT unrolled -- with 32 coordinates per lane the pair body would otherwise outgrow the
      //  instruction cache)
      do {
        const uint32_t nA = nleaf + 1u;
        const double hA = jitl(ufetch(nseq++));                  // :298 / :395 (two draws per leaf pair)
        double hB = 0.0;
        if (level == 0) orbitLen = orbitLen + hA;                // :300
        else hB = jitl(ufetch(nseq++));
        const int lvlA = (level == 0) ? 0 : ((nA == 1u) ? level : (__ffs(nA - 1u) - 1));
        double x[4] = {0.0, 0.0, 0.0, 0.0};
        const int nl = (level == 0) ? 1 : 2;
#pragma unroll 1
        for (int l = 0; l < nl; ++l) {
          hh = l ? hB : hA;
          ha = 0.5 * hh;
          if constexpr (REGRAD) hp = target.leapfrog_energy(q, v, hh, ha); else micro_step();
          if (l == 0) { x[0] = hp; if (level > 0) put_left(lvlA); }
          else x[1] = hp;
        }
        // post-order sub-U-turn checks ending at the pair's second leaf (WALNUTS.py:22-41 plan; :479,568,582); the
        // first one (the pair itself, span 2) shares its reduction with the two energies, and the leaves' bookkeeping
        // follows it
        bool sub = false;
        int lvl = lvlA;
#pragma unroll 1
        for (int sp = 1;; ++sp) {
          if (level > 0) dots_left(lvl, x[2], x[3]);
          Grp::sum4t(x, red, parity);
          if (sp == 1) {
            // the two leaves' weights and selection ratios in ONE instruction stream: even lanes evaluate leaf A, odd
            // lanes leaf B (same operations on the same operands as the sequential form: bit-identical)
            const double Wl = exp(-(odd_lane ? x[1] : x[0]) + H0);
            const double WA = __shfl_sync(0xffffffffu, Wl, 0), WB = __shfl_sync(0xffffffffu, Wl, 1);
            const double ws1 = WnewSum + WA;
            const double rl = (odd_lane ? WB : WA) / (odd_lane ? ws1 + WB : ws1);
            const double rA = __shfl_sync(0xffffffffu, rl, 0), rB = __shfl_sync(0xffffffffu, rl, 1);
            bool pick;
            if (!leaf_book(x[0], hA, WA, rA, pick)) { out = 1; break; }
            if (pick) {
              if (level == 0) {
                double2* dst = scv(pvec);
#pragma unroll
                for (int e2 = 0; e2 < E2; ++e2) dst[e2 * sstride] = make_double2(q[2 * e2], q[2 * e2 + 1]);
              } else {
                prop_from_left(lvlA);
              }
            }
            if (level == 0) break;
            if (!leaf_book(x[1], hB, WB, rB, pick)) { out = 1; break; }
            if (pick) {
              double2* dst = scv(pvec);
#pragma unroll
              for (int e2 = 0; e2 < E2; ++e2) dst[e2 * sstride] = make_double2(q[2 * e2], q[2 * e2 + 1]);
            }
          }
          sub = (x[2] < 0.0) || (x[3] < 0.0);
          if (sub || sp + 1 > level || (nleaf & ((1u << (sp + 1)) - 1u)) != 0u) break;
          const uint32_t m = nleaf - (1u << (sp + 1)) + 1u;      // left end of the next larger span ending here
          lvl = (m == 1u) ? level : (__ffs(m - 1u) - 1);
          x[0] = 0.0;
          x[1] = 0.0;
        }
        if (out) break;
        if (sub) { out = 2; break; }
      } while (nleaf < n_new);
      // ---- write the level's state back for the shared handlers (level end / iteration end) ----
      C.nseq = nseq;
      C.nleaf = nleaf;
      C.WnewSum = WnewSum;
      if (side) { C.timeLen1 = tl; C.maxInt1 = mi; C.endH1 = endH; }
      else { C.timeLen0 = tl; C.maxInt0 = mi; C.endH0 = endH; }
      C.orbitLen = orbitLen;
      C.sN = sN; C.sNz = sN;                                     // If = 0 for every leaf
      C.sMinIf = 0; C.sMaxIf = 0; C.sMinC = 0; C.sMaxC = 0; C.sMinL = 0.0; C.sMaxL = 0.0;
      C.sHmax = sHmax; C.sHmin = sHmin; C.sHnan = sHnan;
      C.nF = C.nF + nF;
      C.L_ = L_;
      C.indexStat = indexStat;
      C.candValid = candValid;
      if (out == 1) {
        C.forced = 1;
        if (stop999) C.stopCode = 999;
        st = ST_ITER_END;
      } else if (out == 2) {                                     // :597-605
        C.candValid = 0;
        C.L_ = C.Lold;
        C.indexStat = C.indexStatOld;
        C.NdS = level;
        C.NdC = level + 1;
        C.stopCode = 5;
        st = ST_ITER_END;
      } else {
        st = ST_LEVEL_END;
      }
    }
  };
  for (;;) {
    if constexpr (Target::BLOCK_LOCKSTEP) {
      // chains of a block evaluate their gradients in lock-step (shared data tiles stay hot in L1);
      // the same barrier doubles as the block's exit vote
      if (__syncthreads_and(st == ST_EXIT)) break;
    }
    // =============================== hot: leapfrog micro-steps ==================================
    if constexpr (Target::COOP) {
      // block-cooperative gradient: every chain of the CTA that is in a pass takes ONE micro-step per trip;
      // the gradient of all of them is evaluated together by all threads (shared data streamed once)
      const bool act = (st == ST_RUN);
      if (act) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          v[e] = fma(ha, g[e], v[e]);
          q[e] = fma(hh, v[e], q[e]);
        }
      }
      target.publish(q, act, steps_left == 1u);
      if (__syncthreads_and(st == ST_EXIT)) break;      // barrier + exit vote
      target.coop_eval(coop_phase);
      if (act) {
        const double lpp = target.collect(q, g);
        double ke = 0.0;
#pragma unroll
        for (int e = 0; e < E; ++e) {
          v[e] = fma(ha, g[e], v[e]);
          ke = fma(v[e], v[e], ke);
        }
        hp = fma(0.5, ke, -lpp);
        expmax = max(expmax, __double2hiint(hp) & 0x7ff00000);
        if (--steps_left != 0u) continue;
        st = ST_PASS_END;
      }
    } else if (!NUTS_FAST && st == ST_RUN) {
      if (yoshida) {
        // one leapfrog of the 4th-order triple (coefficients firstLast, middle, firstLast, :157-173); the
        // energy (Hams[i], :175) and its finiteness only count after the third
        const double cf = (ysub == 1) ? WN_Y_MIDDLE : WN_Y_FIRSTLAST;
        hh = __dmul_rn(cf, hh0);
        ha = __dmul_rn(__dmul_rn(0.5, cf), hh0);
        const int em = expmax;
        micro_step();
        const bool full = (ysub == 2);
        if (!full) expmax = em;
        ysub = full ? 0 : ysub + 1;
        --steps_left;
        if constexpr (ADAPT) {
          if (trackH && full) {
#pragma unroll
            for (int i = 0; i < 4; ++i) hist[i] = (nh == i) ? hp : hist[i];
            ++nh;
          }
          if (trackH && (nh == 4 || steps_left == 0u)) flush_hist();
        }
      } else if (ADAPT && trackH) {   // warm-up: every step's energy is needed for igrConst
        micro_step();
#pragma unroll
        for (int i = 0; i < 4; ++i) hist[i] = (nh == i) ? hp : hist[i];
        ++nh;
        --steps_left;
        if (nh == 4 || steps_left == 0u) flush_hist();
      } else if (LAZY && lazy && steps_left >= 3u) {
        if constexpr (LAZY && G >= 32 && !Target::BLOCK_LOCKSTEP) {
          // the whole warp follows one chain: stay in a tight loop for the skipped-energy steps (merged kicks),
          // then finish the pass with the one step whose energy is consumed
          double kc[E];
          target.kick_coeffs(hh, kc);
#pragma unroll
          for (int e = 0; e < E; ++e) v[e] = fma(ha, g[e], v[e]);
          // blocks of up to lazyK (even) steps between two magnitude checks; one or two steps are left for the end
          uint32_t n = (steps_left - 1u) & ~1u;
          steps_left -= n;
          do {
            const uint32_t m = min(n, (uint32_t)lazyK);
            n -= m;
#pragma unroll 2
            for (uint32_t i = 0; i < m; i += 2u) {
              drift_kick(kc);
              drift_kick(kc);
            }
            if (n) track_state();
          } while (n);
          if (steps_left == 2u) drift_kick(kc);
          micro_step(false);
          steps_left = 0u;
        } else {
          micro_step_lazy();
          micro_step_lazy();
          steps_left -= 2u;
          since += 2;
          if (since >= lazyK) { track_state(); since = 0; }
        }
      } else if (LAZY && lazy && steps_left == 2u) {
        micro_step_lazy();
        micro_step();
        steps_left = 0u;
      } else if (steps_left >= 2u) {   // two steps per trip: the tail of one overlaps the head of the next
        micro_step();
        micro_step();
        steps_left -= 2u;
      } else {
        micro_step();
        steps_left = 0u;
      }
      if (steps_left != 0u) continue;
      st = ST_PASS_END;
    }
    // =============================== cold: per-chain state machine ==============================
    // Handlers are laid out in transition order (every transition goes DOWN this list), so one straight pass takes
    // a chain from the end of a pass to the start of the next one, and the chains that share a warp (G < 32) run
    // each handler TOGETHER instead of serialising a switch: pass end -> leaf -> level end -> iteration end ->
    // next chain -> iteration setup -> level start -> macro-step start -> (hot loop).
    if constexpr (NUTS_FAST) {
      if (st == ST_MACRO) nuts_level();
    }
    if (!NUTS_FAST && st == ST_PASS_END) do {  // a pass of 2^c micro-steps finished
      if constexpr (has_nonneg<Target>::value && KSET == KSET_ADAPT && !ADAPT) {
        // Local failure certificate of a search attempt (adaptiveIntegrators.py:87-92,129-132).  For targets whose
        // energy partials are non-negative (-lp_t >= 0, kinetic part >= 0) the total satisfies Hend >= hp_t, also in
        // floating point (adding non-negative terms never decreases a running sum, and fl(x - Href) is monotone in
        // x).  So if ONE thread's partial alone is at least delta above the start energy, |Href - Hend| < delta is
        // false whatever the other partials are -- the attempt has failed, with or without non-finite intermediate
        // energies.  The unstable early attempts (c below the stability limit) end this way: one block-wide vote
        // replaces the shuffle tree, the shared exchange and, when the magnitude bound tripped, the exact re-run.
        if (rsearch && rc < rlim && target.nonneg_ok) {
          const bool lf = (hp > rHref) && (fabs(rHref - hp) >= rdelta);
          bool anyf;
          // a cluster group votes over all its CTAs: the failing partial may sit in any of them
          if constexpr (Grp::CL > 1) anyf = Grp::any_cluster(lf, red, parity);
          else if constexpr (G > 32) anyf = __syncthreads_or(lf) != 0;
          else if constexpr (G > 1) anyf = __any_sync(Grp::mask(), lf) != 0;
          else anyf = lf;
          if (anyf) {
            rEv += evmul << rc;
            ++rc;
            rexact = false;
            load_ck(rsign);
            start_pass(rc);
            st = ST_RUN;
            break;
          }
        }
      }
      const bool unbounded = (smax & 0x7ff00000) >= LAZY_LIMIT ||
                             ((umax & 0x80000000u) && (int)(umax & 0x7ff00000u) >= LAZY_LIMIT);
      double Hend = hp;
      unsigned pflags = ((expmax == 0x7ff00000) ? 1u : 0u) | (unbounded ? 2u : 0u);
      Grp::sum1_flags(Hend, pflags, red, parity);
      const bool redo_exact = LAZY && (pflags & 2u);
      const bool anybad = pflags != 0u;
      if (rsearch && !redo_exact) {
        // fast path of the search (adaptiveIntegrators.py:69-94, 111-132): attempt failed -> next c
        const bool ok = !anybad && fabs(rHref - Hend) < rdelta;
        if (!ok && rc < rlim) {
          rEv += evmul << rc;
          ++rc;
          rexact = false;
          load_ck(rsign);
          start_pass(rc);
          st = ST_RUN;
          break;
        }
      }
      const int phase = C.phase;
      if (Target::COOP && phase == PH_INIT) {   // gradient at the current state arrived: H0 = Hend
        C.H0 = Hend;
        st = ST_ITER2;
        break;
      }
      if (rsearch) {   // leave the fast path: write the search state back
        C.c = rc;
        if (phase == PH_FWD) C.nF = C.nF + rEv; else C.nB = C.nB + rEv;
        rEv = 0;
      }
      int c = C.c;
      if (redo_exact) {
        // a skipped energy might have been non-finite: repeat this pass with per-step energies
        rexact = true;
        load_ck(phase == PH_BWD ? -1.0 : 1.0);
        start_pass(phase == PH_REDO ? C.cSim : c);
        st = ST_RUN;
        break;
      }
      rexact = false;
      if (phase == PH_FWD) {
        C.nF = C.nF + (evmul << c);
        const bool ok = !anybad && fabs(C.Ham0 - Hend) < C.delta;   // adaptiveIntegrators.py:87-92
        if (!(is_fixed() || ok || c == P.maxC)) {
          ++c;
          C.c = c;
          rc = c;
          load_ck(1.0);
          start_pass(c);
          st = ST_RUN;
          break;
        }
        C.If = c;
        C.cSim = c;
        C.lwtf = 0.0;
        if (is_r2p()) {
          if (useq() < P.p0) {              // adaptiveIntegrators.py:392
            C.lwtf = P.log_p0;
          } else {                          // :400-424 redo at If+1
            C.cSim = c + 1;
            C.phase = PH_REDO;
            rsearch = false;
            load_ck(1.0);
            start_pass(c + 1);
            st = ST_RUN;
            break;
          }
        }
      } else if (phase == PH_REDO) {
        C.nF = C.nF + (evmul << C.cSim);
        C.lwtf = P.log_1mp0;
      }
      if (phase != PH_BWD) {
        // forward simulation done: registers hold the out state O
        C.Hfwd = Hend;
        if constexpr (ADAPT) {
          if (C.warm && P.adaptH) {
            if (is_fixed()) {      // adaptiveIntegrators.py:59
              const double ad = fabs(C.Ham0 - Hend);
              C.igr = rh * pow((ad > 1.0e-10) ? ad : 1.0e-10, -1.0 / 3.0);
            } else {                         // :101,399,424 (last forward pass)
              const double md = C.maxd;
              C.igr = (md > 0.0 || md != md) ? hh0 * pow(md, -1.0 / 3.0) : INFINITY;
            }
          }
          trackH = false;
        }
        if (is_fixed()) {
          C.Ib = 0;
          C.lwt = 0.0;
          st = ST_LEAF;
          break;
        }
        const int If = C.If, cSim = C.cSim;
        int maxTry, Ib;
        if (!is_r2p() || cSim == If) { maxTry = If - 1; Ib = If; }   // :104-111 / :195-202 / :430-433
        else { maxTry = P.maxC; Ib = P.maxC; }                              // :434-437
        C.maxTry = maxTry;
        C.Ib = Ib;
        if (maxTry >= P.minC) {
          save_ck();             // O replaces S
          C.wIntact = 0;
          C.phase = PH_BWD;
          C.c = P.minC;
          rc = P.minC; rlim = maxTry; rHref = Hend; rsign = -1.0; rsearch = true; rEv = 0;
          if constexpr (ADAPT) trackH = false;
#pragma unroll
          for (int e = 0; e < E; ++e) v[e] = -v[e];
          start_pass(P.minC);
          st = ST_RUN;
          break;
        }
      } else {
        C.nB = C.nB + (evmul << c);
        const bool ok = !anybad && fabs(C.Hfwd - Hend) < C.delta;   // :129-132 / :461-464
        if (ok) C.Ib = c;
        if (!ok && c < C.maxTry) {
          ++c;
          C.c = c;
          rc = c;
          load_ck(-1.0);
          start_pass(c);
          st = ST_RUN;
          break;
        }
      }
      // macro step complete
      {
        const int If = C.If, Ib = C.Ib, cSim = C.cSim;
        if (!is_r2p()) {
          C.lwt = (If != Ib) ? WN_LOG_ZERO : 0.0;                  // :136, :239
        } else {
          double lwtb = WN_LOG_ZERO;                               // :467-471
          if (cSim == Ib) lwtb = P.log_p0;
          else if (cSim == Ib + 1) lwtb = P.log_1mp0;
          C.lwt = lwtb - C.lwtf;
        }
      }
      if (!C.wIntact) load_ck(1.0);
      st = ST_LEAF;
      break;
    } while (0);
    if (!NUTS_FAST && st == ST_LEAF) do {  // driver bookkeeping after a macro step, WALNUTS.py:302-368,398-570
      if constexpr (ADAPT) {
        if (C.warm && P.adaptH) p2_push(log(C.igr));    // :313,347,411,454,498,541
      }
      const int level = C.level, side = C.side;
      const uint32_t nleaf = C.nleaf;
      const double h = C.h, Hfwd = C.Hfwd, lwt = C.lwt;
      const int idx = (level == 0) ? (side ? -1 : 1) : (side ? C.maxInt1 - 1 : C.maxInt0 + 1);
      const double tl = (level == 0) ? h : (side ? C.timeLen1 : C.timeLen0) + h;
      if (side) { C.maxInt1 = idx; C.timeLen1 = tl; C.endH1 = Hfwd; }
      else { C.maxInt0 = idx; C.timeLen0 = tl; C.endH0 = Hfwd; }
      if (ADAPT || P.diag) {  // running statistics over used steps: diagnostics columns 8-11, 14, 16, 17, 21, 22; :704
        const int If = C.If, Ib = C.Ib;
        const int cs = is_fixed() ? 0 : C.cSim;
        if (C.sN == 0) {
          C.sMinIf = If; C.sMaxIf = If;
          C.sMinC = cs; C.sMaxC = cs;
          C.sMinL = lwt; C.sMaxL = lwt;
        } else {
          C.sMinIf = min(C.sMinIf, If); C.sMaxIf = max(C.sMaxIf, If);
          C.sMinC = min(C.sMinC, cs); C.sMaxC = max(C.sMaxC, cs);
          C.sMinL = fmin(C.sMinL, lwt); C.sMaxL = fmax(C.sMaxL, lwt);
        }
        C.sN = C.sN + 1;
        C.sNne = C.sNne + (If != Ib);
        C.sNz = C.sNz + (If == 0);
        if (Hfwd != Hfwd) C.sHnan = 1;
        else { C.sHmax = fmax(C.sHmax, Hfwd); C.sHmin = fmin(C.sHmin, Hfwd); }
      }
      if (!finite_d(Hfwd)) {   // forced reject, :316,350,414,457,501,544 (quirks A14 ii, iii)
        C.forced = 1;
        if (level == 0 || (nleaf & 1u)) C.stopCode = 999;
        st = ST_ITER_END;
        break;
      }
      double ls = side ? C.lwtSum1 : C.lwtSum0;
      if (level == 0) ls = lwt;                                                  // :321,354
      else if (!P.compat || !(side == 1 && !(nleaf & 1u))) ls += lwt;            // :420,507,550; quirk A14(i)
      if (side) C.lwtSum1 = ls; else C.lwtSum0 = ls;
      const double Wnew = exp(-Hfwd + C.H0 + ls);                                // :322,...
      bool pick;
      if (level == 0) {
        C.WnewSum = Wnew;
        pick = true;                                                            // :326,359
      } else {
        const double ws = C.WnewSum + Wnew;
        C.WnewSum = ws;
        pick = false;
        if (ws > WN_WT_SUM_THRESH) pick = useq() < Wnew / ws;                    // :426,464,512,554
        C.orbitLen = C.orbitLen + h;                                            // :432,...
      }
      if (pick) {
        const int pv = V_PROP0 + (C.propCur ^ 1);
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) *sc(pv, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
        C.candValid = 1;
        C.L_ = idx;
        C.indexStat = side ? -tl : tl;
      }
      if (P.orbit_min) {
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) {
          double2 lo = *sc(V_OMIN, e2), hi = *sc(V_OMAX, e2);
          // np.minimum / np.maximum propagate NaN
          lo.x = (q[2 * e2] < lo.x || q[2 * e2] != q[2 * e2]) ? q[2 * e2] : lo.x;
          lo.y = (q[2 * e2 + 1] < lo.y || q[2 * e2 + 1] != q[2 * e2 + 1]) ? q[2 * e2 + 1] : lo.y;
          hi.x = (q[2 * e2] > hi.x || q[2 * e2] != q[2 * e2]) ? q[2 * e2] : hi.x;
          hi.y = (q[2 * e2 + 1] > hi.y || q[2 * e2 + 1] != q[2 * e2 + 1]) ? q[2 * e2 + 1] : hi.y;
          *sc(V_OMIN, e2) = lo;
          *sc(V_OMAX, e2) = hi;
        }
      }
      bool sub = false;
      if (level > 0) {
        const double xi = C.xi;
        if (nleaf & 1u) {
          // left end of the pending dyadic levels 1..ctz(nleaf-1) (all when nleaf == 1)
          const int lvl = (nleaf == 1u) ? level : (__ffs(nleaf - 1u) - 1);
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) {
            *sc(V_STACK + 2 * lvl, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
            *sc(V_STACK + 2 * lvl + 1, e2) = make_double2(xi * v[2 * e2], xi * v[2 * e2 + 1]);
          }
        } else {
          // post-order sub-U-turn checks (WALNUTS.py:22-41 plan; :479,568,582)
          for (int s = 1; s <= level && (nleaf & ((1u << s) - 1u)) == 0u; ++s) {
            const uint32_t m = nleaf - (1u << s) + 1u;
            const int lvl = (m == 1u) ? level : (__ffs(m - 1u) - 1);
            if (uturn_vs(V_STACK + 2 * lvl, V_STACK + 2 * lvl + 1)) {
              sub = true;
              break;
            }
          }
        }
      }
      if (sub) {                         // :597-605
        C.candValid = 0;
        C.L_ = C.Lold;
        C.indexStat = C.indexStatOld;
        C.NdS = level;
        C.NdC = level + 1;
        C.stopCode = 5;
        st = ST_ITER_END;
      } else {
        st = (nleaf == C.n_new) ? ST_LEVEL_END : ST_MACRO;
      }
      break;
    } while (0);
    if (st == ST_LEVEL_END) do {  // WALNUTS.py:595-648
      const int level = C.level;
      const double ws = C.WnewSum, wo = C.WoldSum;
      C.indexStat = C.indexStat / (C.timeLen0 + C.timeLen1);                     // :595
      if (!(useq() < ws / wo)) {                                                 // :613
        C.L_ = C.Lold;
        C.indexStat = C.indexStatOld;
      } else if (C.candValid) {
        C.propCur = C.propCur ^ 1;
      }
      C.candValid = 0;
      const bool joined = uturn_vs(V_PARK_Q, V_PARK_V);                          // :622
      const bool bothPassive = (C.lwtSum1 < WN_LOG_ZERO + 1.0) && (C.lwtSum0 < WN_LOG_ZERO + 1.0);   // :624
      C.bothPassive = bothPassive;
      C.NdS = level + 1;
      C.NdC = level + 1;
      C.orbitLenSam = C.orbitLen;
      if (joined || bothPassive) {
        C.stopCode = joined ? 4 : -4;
        st = ST_ITER_END;
        break;
      }
      C.WoldSum = wo + ws;                                                       // :641
      C.level = level + 1;
      st = (level + 1 == P.M) ? ST_ITER_END : ST_LEVEL;
      break;
    } while (0);
    if (st == ST_ITER_END) do {  // qc = qProp; outputs, WALNUTS.py:653-695
      const int pv = V_PROP0 + ((C.forced && C.candValid) ? (C.propCur ^ 1) : C.propCur);
#pragma unroll
      for (int e2 = 0; e2 < E2; ++e2) {
        const double2 qq = *sc(pv, e2);
        q[2 * e2] = qq.x;
        q[2 * e2 + 1] = qq.y;
      }
      const uint32_t cidx = C.chain - P.chain_offset;
      const int it = C.it;
      const size_t row = (size_t)it * P.n_chains + cidx;
      if (P.draws) {
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const int j = target.coord(e, t);
          if (j < P.dg) P.draws[row * P.dg + j] = q[e];
        }
      }
      if (P.orbit_min) {
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) {
          const double2 lo = *sc(V_OMIN, e2), hi = *sc(V_OMAX, e2);
          const int j0 = target.coord(2 * e2, t), j1 = target.coord(2 * e2 + 1, t);
          if (j0 < P.dg) { P.orbit_min[row * P.dg + j0] = lo.x; P.orbit_max[row * P.dg + j0] = hi.x; }
          if (j1 < P.dg) { P.orbit_min[row * P.dg + j1] = lo.y; P.orbit_max[row * P.dg + j1] = hi.y; }
        }
      }
      const unsigned long long nF = C.nF, nB = C.nB;
      if (P.diag && t == 0) {
        double* dg = P.diag + row * 24;
        const double n = (double)C.sN;
        dg[0] = C.L_; dg[1] = C.NdS; dg[2] = C.orbitLen; dg[3] = C.orbitLenSam;
        dg[4] = C.maxInt0; dg[5] = C.maxInt1; dg[6] = (double)nF; dg[7] = (double)nB;
        dg[8] = C.sMinIf; dg[9] = C.sMaxIf; dg[10] = C.sMinL; dg[11] = C.sMaxL;
        dg[12] = C.bothPassive ? 1.0 : 0.0;
        dg[13] = ((C.lwtSum1 < WN_LOG_ZERO + 1.0) || (C.lwtSum0 < WN_LOG_ZERO + 1.0)) ? 1.0 : 0.0;
        dg[14] = (double)C.sNne / n; dg[15] = C.Hbig; dg[16] = (double)C.sNz / n;
        dg[17] = C.sHnan ? __longlong_as_double(0x7ff8000000000000ll) : C.sHmax - C.sHmin;
        dg[18] = C.delta; dg[19] = C.stopCode; dg[20] = C.NdC; dg[21] = C.sMinC; dg[22] = C.sMaxC;
        dg[23] = C.indexStat;
      }
      if constexpr (ADAPT) {
        if (C.warm) {   // WALNUTS.py:701-712
          double delta = C.delta;
          if (P.adaptDelta) {
            const double fac = (C.sHnan ? __longlong_as_double(0x7ff8000000000000ll) : C.sHmax - C.sHmin) / delta;  // :704
            double* hrow = P.adapt_hist + (size_t)cidx * P.warmup_iter;
            const int n0 = C.adNhist;             // finite / infinite entries stored so far (sorted)
            int pos = n0;
            if (fac != fac) {
              C.adNaN = 1;
            } else {                              // upper-bound position in the sorted row
              int lo = 0, hi = n0;
              while (lo < hi) { const int mid = (lo + hi) >> 1; if (hrow[mid] <= fac) lo = mid + 1; else hi = mid; }
              pos = lo;
            }
            const int n1 = (fac != fac) ? n0 : n0 + 1;
            // element i of the row after insertion, read from the row before insertion
            auto at = [&](int i) -> double { return (fac != fac || i < pos) ? hrow[i] : (i == pos ? fac : hrow[i - 1]); };
            const int iterN = (int)C.iter;
            double newdelta = delta;
            if (iterN > 10) {                     // :705-707, np.quantile(x[0:iterN], q) (method 'linear')
              double qv;
              if (C.adNaN) {
                qv = __longlong_as_double(0x7ff8000000000000ll);
              } else {
                const double nn = (double)n1, qq = P.adQuant;
                // numpy _compute_virtual_index(n, q, 1, 1): n*q + (1 + q*(1-1-1)) - 1
                const double virt = __dadd_rn(__dadd_rn(__dmul_rn(nn, qq), __dadd_rn(1.0, __dmul_rn(qq, -1.0))), -1.0);
                int prev = (int)floor(virt), next = prev + 1;
                if (virt >= nn - 1.0) { prev = n1 - 1; next = n1 - 1; }
                if (prev < 0) { prev = 0; }
                if (next < 0) { next = 0; }
                const double gam = virt - floor(virt);
                const double a = at(prev), b = at(next);
                const double dba = b - a;                                   // numpy _lerp
                qv = (gam >= 0.5) ? (b - dba * (1.0 - gam)) : (a + dba * gam);
              }
              newdelta = P.adTarget / qv;
            }
            // every thread has read the row before thread 0 rewrites it, and sees the new row afterwards; a cluster
            // group's row is read by the other CTAs, so both barriers are cluster barriers (release / acquire at
            // cluster scope order the global-memory row as well)
            if constexpr (Grp::CL > 1) cluster_sync(); else if constexpr (G > 32) __syncthreads(); else if constexpr (G > 1) __syncwarp(Grp::mask());
            if (t == 0 && fac == fac) {           // shift the tail and insert
              for (int i = n0; i > pos; --i) hrow[i] = hrow[i - 1];
              hrow[pos] = fac;
            }
            if constexpr (Grp::CL > 1) cluster_sync(); else if constexpr (G > 32) __syncthreads(); else if constexpr (G > 1) __syncwarp(Grp::mask());
            C.adNhist = n1;
            delta = newdelta;
            C.delta = delta;
          }
          if (P.adaptH && C.p2npush > 10) C.Hbig = pow(delta, 1.0 / 3.0) * exp(C.p2q[2]);   // :711-712
        }
      }
      const unsigned long long cf = C.chainF + nF, cbk = C.chainB + nB;
      C.chainF = cf;
      C.chainB = cbk;
      C.it = it + 1;
      if (it + 1 < P.n_iter) {
        st = ST_ITER;
        break;
      }
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int j = target.coord(e, t);
        if (j < P.d) P.state[(size_t)cidx * P.d + j] = q[e];
      }
      if (t == 0) {
        if (P.nevalF) P.nevalF[cidx] = cf;
        if (P.nevalB) P.nevalB[cidx] = cbk;
        if (P.cost) P.cost[cidx] = (unsigned int)min(cf + cbk, 0xffffffffull);
        if constexpr (ADAPT) if (P.adapt_state) {
          double* as = P.adapt_state + (size_t)cidx * WN_ADAPT_STRIDE;
          as[0] = C.Hbig; as[1] = C.delta; as[2] = (double)C.p2npush;
#pragma unroll
          for (int i = 0; i < 5; ++i) { as[3 + i] = C.p2q[i]; as[8 + i] = (double)C.p2n[i]; }
          as[13] = (double)C.adNaN; as[14] = (double)C.adNhist;
        }
      }
      totF += cf;
      totB += cbk;
      st = ST_CHAIN;
      break;
    } while (0);
    if (st == ST_CHAIN) do {  // grab the next chain from the queue
      // (cluster group: thread 0 of rank 0 grabs, bcast0 hands the SAME index to every CTA, so all CTAs of the cluster
      // serve the same chain and leave the loop at the same trip -- every cluster barrier is reached by all of them)
      uint32_t cidx = 0;
      if (t == 0) {
        cidx = atomicAdd(P.queue, 1u);
        if (P.order) cidx = (cidx < *P.order_len) ? P.order[cidx] : 0xffffffffu;
      }
      cidx = Grp::bcast0(cidx, &sh_bcast);
      if (cidx >= (uint32_t)P.n_chains) {
        st = ST_EXIT;
        break;
      }
      C.chain = P.chain_offset + cidx;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int j = target.coord(e, t);
        q[e] = (j < P.d) ? P.state[(size_t)cidx * P.d + j] : 0.0;
      }
      C.Hbig = P.Hstep ? P.Hstep[cidx] : P.H0;
      C.delta = P.delta ? P.delta[cidx] : P.delta0;
      if constexpr (ADAPT) {
        if (P.adapt_state) {
        const double* as = P.adapt_state + (size_t)cidx * WN_ADAPT_STRIDE;
        C.Hbig = as[0];
        C.delta = as[1];
        C.p2npush = (int)as[2];
#pragma unroll
        for (int i = 0; i < 5; ++i) { C.p2q[i] = as[3 + i]; C.p2n[i] = (int)as[8 + i]; }
        C.adNaN = (int)as[13];
        C.adNhist = (int)as[14];
        }
      }
      C.it = 0;
      C.chainF = 0;
      C.chainB = 0;
      st = ST_ITER;
      break;
    } while (0);
    if (st == ST_ITER) do {  // per-iteration setup, WALNUTS.py:196-276
      RngKey key{P.seed_lo, P.seed_hi, C.chain, P.iter0 + (uint32_t)C.it};
      C.iter = key.iter;
      C.nseq = 0;
      ublk_idx = 0xffffffffu;
      {
        const double Hbig = C.Hbig;
        C.jlo = __dmul_rn(Hbig, __dadd_rn(1.0, -P.jitter));   // WALNUTS.py:298
        C.jhi = __dmul_rn(Hbig, __dadd_rn(1.0, P.jitter));
      }
      if constexpr (LAZY && G >= 32) {
        // steps between two magnitude checks of a skipped-energy pass at c = t (see start_pass); two steps of the
        // budget are reserved for the half kick that the merged-kick loop carries in v; log2 Gamma is bounded
        // from above by the exponent field (Gamma >= 1): integer arithmetic only
        {
          const int cc = tid & 31;
          const double hmax = C.jhi * __longlong_as_double((long long)(1023 - cc) << 52);
          const int lg = ((__double2hiint(target.step_growth(hmax)) >> 20) & 0x7ff) - 1022;
          int k = (lg * 66 <= 170) ? 64 : ((int)__fdividef(170.0f, (float)lg) - 2);
          k &= ~1;
          ktab[cc] = (k < 2) ? 0 : k;
        }
        __syncwarp();
      }
      if constexpr (ADAPT) C.warm = (P.adapt_state && key.iter <= (uint32_t)P.warmup_iter) ? 1 : 0;   // :209
      uint32_t dirbits = 0;
      for (int k = 0; k < P.M; k += 2) {                                // B = floor(U(0,2)), :216
        double u0, u1;                                                  // one Philox block = uniforms k, k + 1
        rng_uniform_pair(key, STREAM_DIR, (uint32_t)k >> 1, u0, u1);
        dirbits |= (u0 >= 0.5 ? 1u : 0u) << k;
        if (k + 1 < P.M) dirbits |= (u1 >= 0.5 ? 1u : 0u) << (k + 1);
      }
      C.dirbits = dirbits;
      double x[1];
      {
        double ke = 0.0;
        if constexpr (Target::PAIR_LAYOUT) {
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) {   // v ~ N(0, I), :236
            double z0, z1;
            const int p = e2 * G + t;
            rng_normal_pair(key, STREAM_MOM, (uint32_t)p, z0, z1);
            v[2 * e2] = (2 * p < P.d) ? z0 : 0.0;
            v[2 * e2 + 1] = (2 * p + 1 < P.d) ? z1 : 0.0;
          }
        } else {
#pragma unroll
          for (int e = 0; e < E; ++e) {       // same normals, addressed by coordinate
            const int j = target.coord(e, t);
            double z0 = 0.0, z1 = 0.0;
            if (j < P.d) rng_normal_pair(key, STREAM_MOM, (uint32_t)(j >> 1), z0, z1);
            v[e] = (j < P.d) ? ((j & 1) ? z1 : z0) : 0.0;
          }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) ke = fma(v[e], v[e], ke);
        if constexpr (Target::COOP) {
          // the gradient at the current state (:249) is requested as a zero-length pass: h = 0 leaves
          // (q, v) untouched and the cooperative evaluation fills g and the energy partial
#pragma unroll
          for (int e = 0; e < E; ++e) g[e] = 0.0;
          C.phase = PH_INIT;
          rsearch = false;
          rh = 0.0;
          start_pass(0);
          st = ST_RUN;
          break;
        }
        double lpp;
        if constexpr (REGRAD) lpp = target.lp_only(q);               // the gradient is recomputed where it is used
        else lpp = target.lp_grad(q, g, red, parity);                // :249
        x[0] = fma(0.5, ke, -lpp);
      }
      Grp::template sum<1>(x, red, parity);
      st = ST_ITER2;
      C.H0 = x[0];
      break;
    } while (0);
    if (st == ST_ITER2) do {  // second half of the per-iteration setup (after the gradient at the current state)
      const double H0 = C.H0;                                         // :256
      C.endH0 = H0;
      C.endH1 = H0;
#pragma unroll
      for (int e2 = 0; e2 < E2; ++e2) {   // origin is both ends; it is also the first proposal
        const double2 qq = make_double2(q[2 * e2], q[2 * e2 + 1]);
        *sc(V_PARK_Q, e2) = qq;
        *sc(V_PARK_V, e2) = make_double2(v[2 * e2], v[2 * e2 + 1]);
        if constexpr (!REGRAD) *sc(V_PARK_G, e2) = make_double2(g[2 * e2], g[2 * e2 + 1]);
        *sc(V_PROP0, e2) = qq;
        if (P.orbit_min) { *sc(V_OMIN, e2) = qq; *sc(V_OMAX, e2) = qq; }   // :274-276
      }
      C.propCur = 0;
      C.lwtSum0 = 0.0; C.lwtSum1 = 0.0;
      C.timeLen0 = 0.0; C.timeLen1 = 0.0;
      C.maxInt0 = 0; C.maxInt1 = 0;
      C.WoldSum = 1.0;
      C.L_ = 0;
      C.indexStat = 0.0;
      C.orbitLen = 0.0; C.orbitLenSam = 0.0;
      C.nF = 0; C.nB = 0;
      C.NdS = 0; C.NdC = 0;
      C.stopCode = 0;
      C.bothPassive = 0;
      C.forced = 0;
      C.sN = 0; C.sNne = 0; C.sNz = 0;
      C.sHmax = H0; C.sHmin = H0;
      C.sHnan = 0;
      C.side = -1;
      C.xi = 1.0;
      C.level = 0;
      st = ST_LEVEL;
      break;
    } while (0);
    if (st == ST_LEVEL) do {  // start doubling `level`, WALNUTS.py:281-294
      const int level = C.level, side = C.side;
      const int ns = (C.dirbits >> level) & 1u;   // 0 forward, 1 backward
      const double nxi = ns ? -1.0 : 1.0;
      if (side < 0) {
        // registers hold the origin with forward-time v; switch to integration convention
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] *= nxi;
      } else if (ns != side) {
        // swap the active end with the parked one (stored in forward-time convention)
        const double xi = C.xi;
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) {
          const double2 pq = *sc(V_PARK_Q, e2), pv = *sc(V_PARK_V, e2);
          *sc(V_PARK_Q, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
          *sc(V_PARK_V, e2) = make_double2(xi * v[2 * e2], xi * v[2 * e2 + 1]);
          if constexpr (!REGRAD) {
            const double2 pg = *sc(V_PARK_G, e2);
            *sc(V_PARK_G, e2) = make_double2(g[2 * e2], g[2 * e2 + 1]);
            g[2 * e2] = pg.x; g[2 * e2 + 1] = pg.y;
          }
          q[2 * e2] = pq.x; q[2 * e2 + 1] = pq.y;
          v[2 * e2] = nxi * pv.x; v[2 * e2 + 1] = nxi * pv.y;
        }
      }
      C.side = ns;
      C.xi = nxi;
      C.nleaf = 0;
      C.n_new = 1u << level;
      C.WnewSum = 0.0;
      C.Lold = C.L_;
      C.indexStatOld = C.indexStat;
      C.candValid = 0;
      st = ST_MACRO;
      break;
    } while (0);
    if (!NUTS_FAST && st == ST_MACRO) do {  // start one macro step from the active end
      const uint32_t nleaf = C.nleaf + 1u;
      C.nleaf = nleaf;
      double h;
      if (C.level == 0) {
        h = jit(useq());              // :298
        C.orbitLen = C.orbitLen + h;  // :300
      } else if (nleaf & 1u) {
        h = jit(useq());              // :395 (two draws per leaf pair)
        C.h2 = jit(useq());
      } else {
        h = C.h2;
      }
      C.h = h;
      const double Ham0 = C.side ? C.endH1 : C.endH0;
      C.Ham0 = Ham0;
      if (EXT && P.kind >= KIND_FLOW) {
        // ---- extended integrators: the whole macro step runs here (simple loops, group reductions); the
        // driver above / below is shared.  Registers hold S = (q, vv = xi v, g).  Not a tuned path.
        // (EXT kernels are supersets: the four hot-path integrators take the flat loop as everywhere else.) ----
        const double delta = C.delta;
        const int maxC = P.maxC;
        const double NaN = __longlong_as_double(0x7ff8000000000000ll);
        unsigned long long nF = 0, nB = 0;
        int If = maxC, Ib = maxC;
        double HO = 0.0, lwt = 0.0, igr = 1.0;
        save_ck();   // S
        if (P.kind == KIND_FLOW) {
          // one attempt, adaptiveIntegrators.py:252-287 / :309-339; returns through the references
          auto flow_pass = [&](int c, double Href, double& Hl, bool& ok, double& maxErr, double& maxd, double& hh_) {
            const uint32_t nstep = 1u << c;
            hh_ = ldexp(h, -c);
            const double ha_ = 0.5 * hh_, h8 = hh_ / 8.0, h6 = hh_ / 6.0, h2_ = hh_ * hh_;
            double Hprev = Href;
            ok = true; maxd = 0.0; maxErr = 0.0;
            for (uint32_t i = 0; i < nstep; ++i) {
              double qo[E], go[E], vo[E], gm[E], qm[E];
#pragma unroll
              for (int e = 0; e < E; ++e) {
                qo[e] = q[e]; go[e] = g[e]; vo[e] = v[e];
                v[e] = fma(ha_, g[e], v[e]);
                q[e] = fma(hh_, v[e], q[e]);
              }
              const double lpp = target.lp_grad(q, g, red, parity);
              double ke = 0.0;
#pragma unroll
              for (int e = 0; e < E; ++e) {
                v[e] = fma(ha_, g[e], v[e]);
                ke = fma(v[e], v[e], ke);
                qm[e] = 0.5 * (q[e] + qo[e]) + h8 * (vo[e] - v[e]);                  // :265
              }
              (void)target.lp_grad(qm, gm, red, parity);                            // :266
              double er[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
              for (int e = 0; e < E; ++e) {
                const double qf = qo[e] + hh_ * vo[e] + h2_ * ((1.0 / 6.0) * go[e] + (1.0 / 3.0) * gm[e]);   // :269
                const double sg = h6 * (go[e] + g[e] + 4.0 * gm[e]);
                const double vf = vo[e] + sg;                                        // :272
                const double qb = q[e] - hh_ * v[e] + h2_ * ((1.0 / 6.0) * g[e] + (1.0 / 3.0) * gm[e]);     // :275
                const double vb = -(-v[e] + sg);                                     // :278
                er[0] = Grp::maxn2(er[0], fabs(qf - q[e]));
                er[1] = Grp::maxn2(er[1], fabs(vf - v[e]));
                er[2] = Grp::maxn2(er[2], fabs(qb - qo[e]));
                er[3] = Grp::maxn2(er[3], fabs(vb - vo[e]));
              }
              Grp::template maxn<4>(er, red, parity);
              double err = er[0];                        // Python max(): a NaN in the first operand sticks
              err = (er[1] > err) ? er[1] : err;
              err = (er[2] > err) ? er[2] : err;
              err = (er[3] > err) ? er[3] : err;
              maxErr = (i == 0) ? err : Grp::maxn2(maxErr, err);                     // np.max(Errs)
              double x[1] = {fma(0.5, ke, -lpp)};
              Grp::template sum<1>(x, red, parity);
              ok = ok && finite_d(x[0]);
              maxd = Grp::maxn2(maxd, fabs(x[0] - Hprev));
              Hprev = x[0];
            }
            Hl = Hprev;
          };
          double Hl = 0, maxErr = 0, maxd = 0, hhl = 0;
          bool ok = false;
          for (int c = 0; c <= maxC; ++c) {              // :250-287 (starts at 0, not minC)
            if (c > 0) load_ck(1.0);
            flow_pass(c, Ham0, Hl, ok, maxErr, maxd, hhl);
            nF += 2ull << c;
            if (ok && maxErr < delta) { If = c; break; }
          }
          HO = Hl;
          igr = (maxd > 0.0 || maxd != maxd) ? hhl * pow(maxd, -1.0 / 3.0) : INFINITY;   // :294
          Ib = If;
          if (If > 0) {                                  // :300-345
            save_ck();   // O replaces S
            for (int c = 0; c < If; ++c) {
              load_ck(-1.0);
              double Hb, eb, mb, hb; bool okb;
              flow_pass(c, HO, Hb, okb, eb, mb, hb);
              nB += 2ull << c;
              if (okb && eb < delta) { Ib = c; break; }
            }
            load_ck(1.0);
          }
          lwt = (If != Ib) ? WN_LOG_ZERO : 0.0;
        } else if (P.kind == KIND_MIDPOINT) {
          // one attempt with fixed-point iterations, adaptiveIntegrators.py:483-541 / :572-626
          auto mid_pass = [&](int c, double Href, double& Hl, bool& ok, bool& full, bool& conv, double& maxd,
                              double& hh_, unsigned long long& nev) {
            const uint32_t nstep = 1u << c;
            hh_ = ldexp(h, -c);
            const double hh2 = 0.5 * hh_ * hh_;
            double Hprev = Href;
            ok = finite_d(Href); maxd = 0.0; conv = false;
            uint32_t done = 0;
            for (uint32_t i = 0; i < nstep; ++i) {
              double qt[E], gm[E], mp[E];
#pragma unroll
              for (int e = 0; e < E; ++e) qt[e] = q[e] + hh_ * (v[e] + 0.5 * hh_ * g[e]);   // :494
              conv = false;
              double oldErr = 1.0e100;
              for (int it = 0; it < P.maxFPiter; ++it) {                                   // :500-523
#pragma unroll
                for (int e = 0; e < E; ++e) mp[e] = 0.5 * (qt[e] + q[e]);
                (void)target.lp_grad(mp, gm, red, parity);
                ++nev;
                double er[1] = {0.0};
#pragma unroll
                for (int e = 0; e < E; ++e) {
                  const double qn = q[e] + hh_ * v[e] + hh2 * gm[e];
                  er[0] = Grp::maxn2(er[0], fabs(qn - qt[e]));
                  qt[e] = qn;
                }
                Grp::template maxn<1>(er, red, parity);
                if (er[0] < P.FPtol) { conv = true; break; }
                if (er[0] > 1.1 * oldErr) break;
                oldErr = er[0];
              }
              if (!conv) break;                                                            // :525-527
#pragma unroll
              for (int e = 0; e < E; ++e) mp[e] = 0.5 * (qt[e] + q[e]);                     // :530
              (void)target.lp_grad(mp, gm, red, parity);
              ++nev;
#pragma unroll
              for (int e = 0; e < E; ++e) {
                q[e] = q[e] + hh_ * v[e] + hh2 * gm[e];                                    // :534
                v[e] = fma(hh_, gm[e], v[e]);                                              // :535
              }
              const double lpp = target.lp_grad(q, g, red, parity);                        // :537
              ++nev;
              double ke = 0.0;
#pragma unroll
              for (int e = 0; e < E; ++e) ke = fma(v[e], v[e], ke);
              double x[1] = {fma(0.5, ke, -lpp)};
              Grp::template sum<1>(x, red, parity);
              ok = ok && finite_d(x[0]);
              maxd = Grp::maxn2(maxd, fabs(x[0] - Hprev));
              Hprev = x[0];
              ++done;
            }
            full = (done == nstep);
            if (!full) {                     // Hams of the missing steps are 0 (:490)
              maxd = Grp::maxn2(maxd, fabs(0.0 - Hprev));
              Hprev = 0.0;
            }
            Hl = Hprev;
          };
          double Hl = 0, maxd = 0, hhl = 0;
          bool ok = false, full = false, conv = false;
          for (int c = 0; c <= maxC; ++c) {              // :482-545
            if (c > 0) load_ck(1.0);
            mid_pass(c, Ham0, Hl, ok, full, conv, maxd, hhl, nF);
            if (ok && fabs(Ham0 - Hl) < delta && full) { If = c; break; }
          }
          if (!conv) {
            // the reference ends the process here (sys.exit, :548-550); per-chain failure instead: NaN energy
            // -> forced reject, stop code 999 (DESIGN.md section 5)
            HO = NaN; Ib = If; lwt = 0.0; igr = NaN;
          } else {
            HO = Hl;                                     // :569 (the same expression as Hams[-1])
            igr = (maxd > 0.0 || maxd != maxd) ? hhl * pow(maxd, -1.0 / 3.0) : INFINITY;   // :561
            Ib = maxC;                                   // :564
            save_ck();   // O replaces S
            for (int c = 0; c <= maxC; ++c) {            // :570-633: the full range
              load_ck(-1.0);
              double Hb, mb, hb; bool okb, fullb, convb;
              mid_pass(c, HO, Hb, okb, fullb, convb, mb, hb, nB);
              if (okb && fabs(HO - Hb) < delta && fullb) { Ib = c; break; }
            }
            load_ck(1.0);
            lwt = (If != Ib) ? WN_LOG_ZERO : 0.0;
          }
        } else {
          // adaptRescaledLeapFrogD, adaptiveIntegrators.py:660-762: one leapfrog step in coordinates rescaled
          // per dimension by Sd = 2^-Sred; from the state in the checkpoint with velocity sign `vs`
          int sred[E], sfw[E];
          double gbm[E];
          auto attempt = [&](double vs, double& Ham1) {
            load_ck(vs);
            const double hah = 0.5 * h;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const double Sd = ldexp(1.0, -sred[e]);
              const double qb = q[e] / Sd, gb = Sd * g[e];                                  // :672-673
              v[e] = fma(hah, gb, v[e]);                                                    // :674
              q[e] = (qb + h * v[e]) * Sd;                                                  // :675-676
              gbm[e] = fabs(gb);
            }
            const double lpp = target.lp_grad(q, g, red, parity);                           // :677
            double ke = 0.0;
#pragma unroll
            for (int e = 0; e < E; ++e) {
              const double gb1 = ldexp(1.0, -sred[e]) * g[e];                               // :679
              v[e] = fma(hah, gb1, v[e]);                                                   // :680
              gbm[e] = 0.5 * (gbm[e] + fabs(gb1));                                          // :681
              ke = fma(v[e], v[e], ke);
            }
            double x[1] = {fma(0.5, ke, -lpp)};
            Grp::template sum<1>(x, red, parity);
            Ham1 = x[0];
          };
          // :687-697: returns true when the attempt is accepted, otherwise updates sred
          auto judge = [&](double Href, double Ham1) -> bool {
            double x[1] = {0.0};
#pragma unroll
            for (int e = 0; e < E; ++e) x[0] += (gbm[e] > P.gradThresh) ? 1.0 : 0.0;
            Grp::template sum<1>(x, red, parity);
            if (!finite_d(Ham1)) {
#pragma unroll
              for (int e = 0; e < E; ++e) sred[e] += 1;
            } else if (x[0] != 0.0) {
#pragma unroll
              for (int e = 0; e < E; ++e) sred[e] += (gbm[e] > P.gradThresh) ? 1 : 0;
            } else if (fabs(Href - Ham1) > delta) {
#pragma unroll
              for (int e = 0; e < E; ++e) sred[e] += 1;
            } else {
              return true;
            }
            return false;
          };
          auto same = [&]() -> bool {
            double x[1] = {0.0};
#pragma unroll
            for (int e = 0; e < E; ++e) x[0] += (sred[e] != sfw[e]) ? 1.0 : 0.0;
            Grp::template sum<1>(x, red, parity);
            return x[0] == 0.0;
          };
#pragma unroll
          for (int e = 0; e < E; ++e) sred[e] = 0;
          double Ham1 = 0.0;
          for (int c = 0; c <= maxC; ++c) {              // :669-700
            attempt(1.0, Ham1);
            ++nF;
            if (judge(Ham0, Ham1)) { If = c; break; }
          }
          HO = Ham1;
          igr = 1.0;
#pragma unroll
          for (int e = 0; e < E; ++e) { sfw[e] = sred[e]; sred[e] = 0; }
          Ib = If;
          if (If > 0) {                                  // :718-755
            save_ck();   // O replaces S
            for (int c = 0; c <= maxC; ++c) {
              double Hb;
              attempt(-1.0, Hb);
              ++nB;
              if (judge(HO, Hb)) { Ib = c; break; }
              if (same()) { Ib = c + 1; break; }
            }
            load_ck(1.0);
          }
          lwt = same() ? 0.0 : WN_LOG_ZERO;              // :762
        }
        C.nF = C.nF + nF;
        C.nB = C.nB + nB;
        C.If = If; C.Ib = Ib; C.cSim = If; C.lwt = lwt; C.Hfwd = HO;
        if constexpr (ADAPT) { C.igr = igr; trackH = false; }
        st = ST_LEAF;
        break;
      }
      C.phase = PH_FWD;
      const int c0 = is_fixed() ? 0 : P.minC;
      C.c = c0;
      rh = h; rc = c0; rlim = P.maxC; rHref = Ham0; rdelta = C.delta; rsign = 1.0;
      rsearch = !is_fixed();
      rexact = false;
      rEv = 0;
      if constexpr (ADAPT) trackH = C.warm && P.adaptH && !is_fixed();
      if constexpr (LAZY) rlazyok = target.lazy_ok && (C.jhi <= 1024.0);
      if (!is_fixed()) save_ck();   // S = start state (integration convention)
      C.wIntact = 1;
      start_pass(c0);
      st = ST_RUN;
      break;
    } while (0);
    if (st == ST_EXIT) {
      if constexpr (Target::BLOCK_LOCKSTEP || Target::COOP) continue;   // keep serving the block's barriers
      break;
    }
  }
  // cluster group: no CTA exits while a peer may still read its shared memory (the last DSMEM access is the exit
  // grab's broadcast, which every CTA passed before leaving the loop at the same trip)
  if constexpr (Grp::CL > 1) cluster_sync();
  if (t == 0 && (totF | totB)) {
    atomicAdd(P.totals, totF);
    atomicAdd(P.totals + 1, totB);
  }
}

}  // namespace wn
