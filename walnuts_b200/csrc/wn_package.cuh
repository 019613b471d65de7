// Persistent many-chain kernel for the `walnuts` PACKAGE transition (reference walnuts/walnuts.py):
//   walnuts_step :279-359, extend_orbit :211-276, stable_steps :144-182, leapfrog :74-95,
//   choose_micro_steps / micro_steps_logp :185-208, uturn / sub_uturn :16-33,62-70, H :127-141.
//
// Same execution model as wn_walnutspy.cuh (one group of G threads per chain, register-resident
// (theta, rho, grad), one flat loop whose body is a leapfrog micro-step, cold state machine around
// it), but with the package's semantics (SURVEY.md section 8 table A):
//   * micro-step criterion: max - min of H over EVERY micro-step <= max_error (:174-181); the
//     per-step energies are reduced over the group in batches of 4 steps;
//   * micro-step law: ell uniform on {ell_s//2, ell_s, 2 ell_s} (:194), log-weight correction
//     logp(ell | ell_next) - logp(ell | ell_s) (:265-271);
//   * diagonal inverse mass matrix in the kinetic energy, the drift and the U-turn metric;
//   * selection: accept the extension w.p. min(1, W_ext / W_old) in log space (:345-347), then a
//     multinomial pick inside it (:349-350) -- done online (reservoir) with keyed uniforms, which
//     has the same law and lets the extension stop at its first sub-U-turn (oracle/package_oracle.py).
// compat != 0 reproduces the reference's two latent defects (SURVEY.md rows B3, B5).
#pragma once
#include "wn_common.cuh"
#include "wn_targets.cuh"

namespace wn {

struct PkgParams {
  int n_chains, d, dg, max_depth, compat, n_iter;
  uint32_t iter0, seed_lo, seed_hi, chain_offset;
  double macro_step, max_error;
  const double* inv_mass;       // [d]
  double* state;                // [n_chains, d]
  double* draws;                // [n_iter, n_chains, dg] or null
  unsigned long long* neval;    // [n_chains] or null: lp/grad evaluations of this call
  unsigned long long* totals;   // [2]
  double2* scratch;
  int nslot;
  unsigned int* queue;
  const unsigned int* order;    // see RunParams
  const unsigned int* order_len;
  unsigned int* cost;
  TargetParams tp;
};

__host__ __device__ inline int package_scratch_vectors(int M) { return 5 + 2 * (M + 1); }

enum { PK_STABLE_F = 0, PK_LEAP = 1, PK_STABLE_B = 2 };
enum { PS_CHAIN = 0, PS_ITER, PS_DEPTH, PS_MACRO, PS_PASS_END, PS_LEAF, PS_DEPTH_END, PS_ITER_END, PS_RUN, PS_EXIT };

struct PkgCtl {
  uint32_t chain, iter;
  int it, depth, back, phase, n, ell_s, ell, ell_n;
  uint32_t k, n_new;
  int propCur, candValid, sub;
  double step, lpS, keS, HS, lpO, keO, lpP, keP, Hmin, Hmax;
  double p0, weight, wL, wR, lse_old, lse_ext;
  unsigned long long nev, chainEv;
};

#define WN_NEG_LOG3 (-1.0986122886681098)

// dynamic shared memory of package_kernel in doubles: checkpoint, reduction scratch, target
template <template <int, int> class TargetTT, int G, int E2, int NT>
__host__ __device__ constexpr int pkg_smem_doubles() {
  return 3 * 2 * E2 * NT + 2 * ((G + 31) / 32) * 8 + TargetTT<G, E2>::smem_doubles(NT);
}

template <template <int, int> class TargetTT, int G, int E2, int NT, int MINB = 1>
__global__ void __launch_bounds__(NT, MINB) package_kernel(const __grid_constant__ PkgParams P) {
  constexpr int E = 2 * E2;
  constexpr int GPB = NT / G;
  constexpr int HB = 4;  // per-step energies are reduced over the group in batches of HB steps
  static_assert(NT % G == 0 && (G <= 32 || NT == G), "block must hold whole groups");
  using Grp = Group<G>;
  using Target = TargetTT<G, E2>;

  extern __shared__ __align__(16) double smem[];
  double* ck = smem;                   // checkpoint [3*E][NT]
  double* red = smem + 3 * E * NT;
  __shared__ uint32_t sh_bcast;
  __shared__ PkgCtl sh_ctl[(G >= 32) ? NT / 32 : 1];
  PkgCtl loc_ctl;
  volatile PkgCtl& C = (G >= 32) ? sh_ctl[threadIdx.x >> 5] : loc_ctl;

  const int tid = threadIdx.x;
  const int t = tid % G;
  int parity = 0;
  auto sc = [&](int vi, int e2) -> double2* {
    const size_t slot = (size_t)blockIdx.x * GPB + tid / G;
    return P.scratch + ((size_t)(vi * E2 + e2) * P.nslot + slot) * G + t;
  };
  enum { V_PARK_Q = 0, V_PARK_V = 1, V_PARK_G = 2, V_PROP0 = 3, V_PROP1 = 4, V_STACK = 5 };

  Target target;
  target.init(P.tp, P.d, t, red + 2 * ((G + 31) / 32) * 8);

  double q[E], v[E], g[E], im[E], sim[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int j = target.coord(e, t);
    im[e] = (j < P.d) ? P.inv_mass[j] : 0.0;
    sim[e] = 0.0;
  }
  // hot scalars
  uint32_t steps_left = 0;
  double step = 0, half = 0, lpp = 0, kep = 0;   // lpp / kep: this thread's partials at the last eval
  double hist[HB];
  int nh = 0;
  bool track = false, merged = false;
  unsigned long long tot = 0;

  auto keyed = [&](uint32_t stream, uint32_t idx) -> double {
    RngKey key{P.seed_lo, P.seed_hi, C.chain, C.iter};
    return rng_uniform(key, stream, idx);
  };
  auto save_ck = [&]() {
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
  // fold a batch of per-step energies into (Hmin, Hmax) with Python min/max semantics (:174,179)
  auto flush_hist = [&]() {
    if (nh == 0) return;
    double x[HB];
#pragma unroll
    for (int i = 0; i < HB; ++i) x[i] = (i < nh) ? hist[i] : 0.0;
    Grp::template sum<HB>(x, red, parity);
    double mn = C.Hmin, mx = C.Hmax;
#pragma unroll
    for (int i = 0; i < HB; ++i) {
      if (i < nh) {
        mn = (x[i] < mn) ? x[i] : mn;
        mx = (x[i] > mx) ? x[i] : mx;
      }
    }
    C.Hmin = mn;
    C.Hmax = mx;
    nh = 0;
  };
  // start a pass of `nsteps` micro-steps of size st_; first half kick is applied here (:168 / :89)
  auto start_pass = [&](double st_, uint32_t nsteps, bool track_, bool merged_) {
    step = st_;
    half = 0.5 * st_;
    steps_left = nsteps;
    track = track_;
    merged = merged_;
    nh = 0;
#pragma unroll
    for (int e = 0; e < E; ++e) {
      sim[e] = st_ * im[e];            // step_inv_mass (:167 / :88)
      v[e] = fma(half, g[e], v[e]);    // rho + half_step_size * grad(theta)
    }
  };
  auto uturn_vs = [&](int viq, int viv, double vcur_sign, bool cur_first) -> bool {
    // walnuts.py:16-33 with state1 = (cur or stored), state2 = the other; diff = inv_mass*(t2 - t1)
    double x[2] = {0.0, 0.0};
    const double sgn = cur_first ? 1.0 : -1.0;   // diff = sgn * inv_mass * (stored - cur)
#pragma unroll
    for (int e2 = 0; e2 < E2; ++e2) {
      const double2 ql = *sc(viq, e2), vl = *sc(viv, e2);
      const double d0 = sgn * (im[2 * e2] * (ql.x - q[2 * e2])), d1 = sgn * (im[2 * e2 + 1] * (ql.y - q[2 * e2 + 1]));
      x[0] = fma(vcur_sign * v[2 * e2], d0, x[0]);
      x[0] = fma(vcur_sign * v[2 * e2 + 1], d1, x[0]);
      x[1] = fma(vl.x, d0, x[1]);
      x[1] = fma(vl.y, d1, x[1]);
    }
    Grp::template sum<2>(x, red, parity);
    return (x[0] < 0.0) || (x[1] < 0.0);
  };
  auto logp_ell = [&](int ell, int es) -> double {   // :197-208
    return (ell == es || ell == es / 2 || ell == es * 2) ? WN_NEG_LOG3 : -INFINITY;
  };
  auto logaddexp = [&](double a, double b) -> double {
    if (a == b) return a + 0.6931471805599453;           // covers (-inf, -inf) and (inf, inf)
    const double dd = a - b;
    if (dd > 0) return a + log1p(exp(-dd));
    if (dd <= 0) return b + log1p(exp(dd));
    return a + b;                                         // NaN
  };

  int st = PS_CHAIN;
  for (;;) {
    if constexpr (Target::BLOCK_LOCKSTEP) {
      if (__syncthreads_and(st == PS_EXIT)) break;
    }
    // =============================== hot: one micro-step ========================================
    if (st == PS_RUN) {
      // drift, gradient, kick (:170-175 stable_steps, :91-94 leapfrog)
#pragma unroll
      for (int e = 0; e < E; ++e) q[e] = fma(sim[e], v[e], q[e]);
      lpp = target.lp_grad(q, g, red, parity);
      const bool last = (steps_left == 1u);
      if (track) {
        double ke0 = 0.0, ke1 = 0.0;
#pragma unroll
        for (int e = 0; e < E; e += 2) {
          v[e] = fma(half, g[e], v[e]);
          v[e + 1] = fma(half, g[e + 1], v[e + 1]);
          ke0 = fma(im[e] * v[e], v[e], ke0);
          ke1 = fma(im[e + 1] * v[e + 1], v[e + 1], ke1);
        }
        kep = ke0 + ke1;
        const double hcur = fma(0.5, kep, -lpp);     // partial of H_current (:173,178)
#pragma unroll
        for (int i = 0; i < HB; ++i) hist[i] = (nh == i) ? hcur : hist[i];
        ++nh;
        if (!last) {
#pragma unroll
          for (int e = 0; e < E; ++e) v[e] = fma(half, g[e], v[e]);   // second half kick (:175)
        }
        if (nh == HB || last) flush_hist();
      } else {
        const double kk = (merged && !last) ? step : half;   // :92 full kick / :94 final half kick
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = fma(kk, g[e], v[e]);
      }
      if (--steps_left != 0u) continue;
      st = PS_PASS_END;
    }
    // =============================== cold state machine ==========================================
    // handlers in transition order (every transition goes down this list): see wn_walnutspy.cuh
    if (st == PS_PASS_END) do {
      const int phase = C.phase;
      if (phase != PK_LEAP) {
        // stable_steps pass n finished (:161-182)
        const int n = C.n;
        C.nev = C.nev + (1ull << n);
        const bool ok = (C.Hmax - C.Hmin) <= P.max_error;                    // :180
        if (!ok && n < 10) {
          C.n = n + 1;
          load_ck(phase == PK_STABLE_F ? 1.0 : -1.0);
          C.Hmin = C.HS;
          C.Hmax = C.HS;
          start_pass(ldexp(P.macro_step, -(n + 1)), 1u << (n + 1), true, false);
          st = PS_RUN;
          break;
        }
        const int es = 1 << n;                                               // :181-182
        if (phase == PK_STABLE_F) {
          C.ell_s = es;
          const double u = keyed(STREAM_PKG_ELL, C.n_new - 1u + C.k - 1u);   // :194,256
          int lo = es / 2;
          if (!P.compat && lo < 1) lo = 1;
          const int pickI = min(2, (int)floor(3.0 * u));
          const int ell = (pickI == 0) ? lo : (pickI == 1 ? es : 2 * es);
          C.ell = ell;
          load_ck(1.0);
          C.phase = PK_LEAP;
          // ell == 0 (defect B3): macro_step / 0 = inf and range(-1) is empty: one step of size inf
          const double stp = (ell > 0) ? P.macro_step / (double)ell : INFINITY;   // :259
          start_pass(stp, ell > 0 ? (uint32_t)ell : 1u, false, true);
          st = PS_RUN;
          break;
        }
        // backward search done: ell_stable_next known; restore O and finish the macro step
        C.ell_n = es;
        load_ck(1.0);
        st = PS_LEAF;
        break;
      }
      // leapfrog (:258) finished: registers hold O = (theta', rho', grad')
      {
        const int ell = C.ell;
        C.nev = C.nev + (unsigned long long)(ell > 0 ? ell : 1);
        double x[2] = {lpp, 0.0};
#pragma unroll
        for (int e = 0; e < E; ++e) x[1] = fma(im[e] * v[e], v[e], x[1]);
        Grp::template sum<2>(x, red, parity);
        C.lpO = x[0];
        C.keO = x[1];
        const double HO = -x[0] + 0.5 * x[1];
        save_ck();                                  // O replaces S
        C.phase = PK_STABLE_B;                      // stable_steps(theta, -rho) (:261)
        C.n = 0;
        C.HS = HO;
        C.Hmin = HO;
        C.Hmax = HO;
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = -v[e];
        start_pass(P.macro_step, 1u, true, false);
        st = PS_RUN;
      }
      break;
    } while (0);
    if (st == PS_LEAF) do {  // weight update, online pick, sub-U-turn checks (:264-273, :343, :349-350)
      const int depth = C.depth, back = C.back, ell = C.ell;
      const uint32_t k = C.k;
      const double p1 = -(-C.lpO + 0.5 * C.keO);                                      // :264
      double w = __dadd_rn(p1, -C.p0);
      w = __dadd_rn(w, logp_ell(ell, C.ell_n));
      w = __dadd_rn(w, -logp_ell(ell, C.ell_s));
      w = __dadd_rn(w, C.weight);                                                      // :265-271
      C.weight = w;
      const double lse = logaddexp(C.lse_ext, w);
      C.lse_ext = lse;
      const double us = keyed(STREAM_PKG_SELECT, C.n_new - 1u + k - 1u);
      if (lse > -INFINITY && us < exp(w - lse)) {
        const int pv = V_PROP0 + (C.propCur ^ 1);
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) *sc(pv, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
        C.candValid = 1;
      }
      // stored momentum: as integrated (reference, :272) or forward-time (compat == 0)
      const double vs = (P.compat || !back) ? 1.0 : -1.0;
      bool sub = false;
      if (depth > 0) {
        if (k & 1u) {
          const int lvl = (k == 1u) ? depth : (__ffs(k - 1u) - 1);
#pragma unroll
          for (int e2 = 0; e2 < E2; ++e2) {
            *sc(V_STACK + 2 * lvl, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
            *sc(V_STACK + 2 * lvl + 1, e2) = make_double2(vs * v[2 * e2], vs * v[2 * e2 + 1]);
          }
        } else {
          for (int s = 1; s <= depth && (k & ((1u << s) - 1u)) == 0u; ++s) {
            const uint32_t m = k - (1u << s) + 1u;
            const int lvl = (m == 1u) ? depth : (__ffs(m - 1u) - 1);
            // list order after the [::-1] of :275: backward -> current state comes first
            if (uturn_vs(V_STACK + 2 * lvl, V_STACK + 2 * lvl + 1, vs, back != 0)) {
              sub = true;
              break;
            }
          }
        }
      }
      if (sub) {                     // :343-344
        C.sub = 1;
        st = PS_ITER_END;
      } else {
        st = (k == C.n_new) ? PS_DEPTH_END : PS_MACRO;
      }
      break;
    } while (0);
    if (st == PS_DEPTH_END) do {  // :345-358
      const int depth = C.depth, back = C.back;
      const double ua = keyed(STREAM_PKG_ACCEPT, (uint32_t)depth);
      const double lse_ext = C.lse_ext, lse_old = C.lse_old;
      if (log(ua) < lse_ext - lse_old) {                                       // :345-347
        if (C.candValid) C.propCur = C.propCur ^ 1;                              // :349-350
      }
      C.candValid = 0;
      // the new end is the last generated state with its stored momentum (:351)
      const double vs = (P.compat || !back) ? 1.0 : -1.0;
#pragma unroll
      for (int e = 0; e < E; ++e) v[e] = vs * v[e];
      if (back) C.wL = C.weight; else C.wR = C.weight;
      // uturn(orbit[0], orbit[-1]) (:352): left first
      const bool joined = uturn_vs(V_PARK_Q, V_PARK_V, 1.0, back != 0);
      if (joined || depth + 1 == P.max_depth) {
        st = PS_ITER_END;
        break;
      }
      C.lse_old = logaddexp(lse_old, lse_ext);                                 // :354-358
      C.depth = depth + 1;
      st = PS_DEPTH;
      break;
    } while (0);
    if (st == PS_ITER_END) do {
      const int pv = V_PROP0 + C.propCur;
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
      const unsigned long long ce = C.chainEv + C.nev;
      C.chainEv = ce;
      C.it = it + 1;
      if (it + 1 < P.n_iter) {
        st = PS_ITER;
        break;
      }
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int j = target.coord(e, t);
        if (j < P.d) P.state[(size_t)cidx * P.d + j] = q[e];
      }
      if (t == 0 && P.neval) P.neval[cidx] = ce;
      if (t == 0 && P.cost) P.cost[cidx] = (unsigned int)min(ce, 0xffffffffull);
      tot += ce;
      st = PS_CHAIN;
      break;
    } while (0);
    if (st == PS_CHAIN) do {
      uint32_t cidx = 0;
      if (t == 0) {
        cidx = atomicAdd(P.queue, 1u);
        if (P.order) cidx = (cidx < *P.order_len) ? P.order[cidx] : 0xffffffffu;
      }
      cidx = Grp::bcast0(cidx, &sh_bcast);
      if (cidx >= (uint32_t)P.n_chains) {
        st = PS_EXIT;
        break;
      }
      C.chain = P.chain_offset + cidx;
#pragma unroll
      for (int e = 0; e < E; ++e) {
        const int j = target.coord(e, t);
        q[e] = (j < P.d) ? P.state[(size_t)cidx * P.d + j] : 0.0;
      }
      C.it = 0;
      C.chainEv = 0;
      st = PS_ITER;
      break;
    } while (0);
    if (st == PS_ITER) do {  // walnuts_step :322-327
      RngKey key{P.seed_lo, P.seed_hi, C.chain, P.iter0 + (uint32_t)C.it};
      C.iter = key.iter;
      double x[2];
      {
        double ke = 0.0;
#pragma unroll
        for (int e = 0; e < E; ++e) {   // rho = inv_mass**-0.5 * N(0, I), :322-325
          const int j = target.coord(e, t);
          double z0 = 0.0, z1 = 0.0;
          if (j < P.d) rng_normal_pair(key, STREAM_MOM, (uint32_t)(j >> 1), z0, z1);
          v[e] = (j < P.d) ? __dmul_rn(pow(im[e], -0.5), (j & 1) ? z1 : z0) : 0.0;
          ke = fma(im[e] * v[e], v[e], ke);
        }
        x[0] = target.lp_grad(q, g, red, parity);
        x[1] = ke;
      }
      C.nev = 1;
      Grp::template sum<2>(x, red, parity);
      const double w0 = -(-x[0] + 0.5 * x[1]);          // -H(theta, rho), :326
      C.lpO = x[0];
      C.keO = x[1];
      C.lpP = x[0];
      C.keP = x[1];
      C.wL = w0;
      C.wR = w0;
      C.lse_old = w0;
#pragma unroll
      for (int e2 = 0; e2 < E2; ++e2) {
        const double2 qq = make_double2(q[2 * e2], q[2 * e2 + 1]);
        *sc(V_PARK_Q, e2) = qq;
        *sc(V_PARK_V, e2) = make_double2(v[2 * e2], v[2 * e2 + 1]);
        *sc(V_PARK_G, e2) = make_double2(g[2 * e2], g[2 * e2 + 1]);
        *sc(V_PROP0, e2) = qq;
      }
      C.propCur = 0;
      C.back = -1;
      C.depth = 0;
      st = PS_DEPTH;
      break;
    } while (0);
    if (st == PS_DEPTH) do {  // :328-342 start of an extension
      const int depth = C.depth, prev = C.back;
      const int back = (keyed(STREAM_PKG_DIR, (uint32_t)depth) >= 0.5) ? 1 : 0;   // :330
      // registers hold the end of side `prev` with its STORED momentum; the other end is parked
      if (prev >= 0 && back != prev) {
#pragma unroll
        for (int e2 = 0; e2 < E2; ++e2) {
          const double2 pq = *sc(V_PARK_Q, e2), pv = *sc(V_PARK_V, e2), pg = *sc(V_PARK_G, e2);
          *sc(V_PARK_Q, e2) = make_double2(q[2 * e2], q[2 * e2 + 1]);
          *sc(V_PARK_V, e2) = make_double2(v[2 * e2], v[2 * e2 + 1]);
          *sc(V_PARK_G, e2) = make_double2(g[2 * e2], g[2 * e2 + 1]);
          q[2 * e2] = pq.x; q[2 * e2 + 1] = pq.y;
          v[2 * e2] = pv.x; v[2 * e2 + 1] = pv.y;
          g[2 * e2] = pg.x; g[2 * e2 + 1] = pg.y;
        }
        // log density / kinetic term of the two ends travel with them
        const double lpo = C.lpO, keo = C.keO;
        C.lpO = C.lpP;
        C.keO = C.keP;
        C.lpP = lpo;
        C.keP = keo;
      }
      if (back) {   // rho = -rho (:245)
#pragma unroll
        for (int e = 0; e < E; ++e) v[e] = -v[e];
      }
      C.back = back;
      C.weight = back ? C.wL : C.wR;      // :244,248
      C.k = 0;
      C.n_new = 1u << depth;
      C.lse_ext = -INFINITY;
      C.candValid = 0;
      C.sub = 0;
      st = PS_MACRO;
      break;
    } while (0);
    if (st == PS_MACRO) do {  // one macro step of extend_orbit (:251-273): start the forward stable_steps search
      C.k = C.k + 1u;
      // registers: (theta, rho in integration convention, grad(theta)); lpO/keO are its lp and rho.M^-1.rho
      const double lpS = C.lpO, keS = C.keO;
      C.lpS = lpS;
      C.keS = keS;
      const double HS = -lpS + 0.5 * keS;
      C.HS = HS;
      C.p0 = -HS;                                  // :252
      save_ck();                                   // S
      C.phase = PK_STABLE_F;
      C.n = 0;
      C.Hmin = HS;                                 // :165
      C.Hmax = HS;
      start_pass(P.macro_step, 1u, true, false);
      st = PS_RUN;
      break;
    } while (0);
    if (st == PS_EXIT) {
      if constexpr (Target::BLOCK_LOCKSTEP) continue;
      break;
    }
  }
  if (t == 0 && tot) atomicAdd(P.totals, tot);
}

}  // namespace wn
