/*
 * walnuts_cuda.h -- C-ABI of the B200-native many-chain WALNUTS/NUTS sampler.
 *
 * The reference (bob-carpenter/walnuts) is pure Python and has no FFI layer for this path, so
 * the boundary below is what its two Python call surfaces bind through ctypes
 * (see INTEGRATION.md for the stub a reference maintainer would add):
 *
 *   walnuts(rng, theta_init, logp, grad, inv_mass, macro_step, max_nuts_depth, max_error,
 *           iter_warmup, iter_sample)                     reference walnuts/walnuts.py:362-408
 *   walnuts_step(...)                                     reference walnuts/walnuts.py:279-359
 *   WALNUTS(lpFun, q0, generated, integrator, H0, stepSizeRandScale, delta0, numIter,
 *           warmupIter, M, igrAux, ...)                   reference WALNUTSpy/WALNUTS.py:111-727
 *   integrator protocol fixedLeapFrog / adaptLeapFrogD / adaptLeapFrogR2P
 *                                                         reference WALNUTSpy/adaptiveIntegrators.py:49-137,361-475
 *   lpFun(q) -> [lp, grad] / logp(theta), grad(theta)     reference WALNUTSpy/targetDistr.py:18-92, test/targets.py:4-29
 *
 * Conventions: every entry point returns 0 on success and a negative WN_E* code on failure
 * (no exceptions / exit() across the ABI; the reference's sys.exit("stack full"),
 * WALNUTS.py:65, and ValueError, walnuts.py:309-320, become error codes + wn_last_error()).
 * The caller owns every buffer.  One handle per (device, host thread); each handle owns one
 * CUDA stream.  Per-chain numerical failures are reported in the diagnostics stop-code column
 * (999, WALNUTS.py:318), never as a call failure.  All floating-point data is IEEE fp64.
 */
#ifndef WALNUTS_CUDA_H
#define WALNUTS_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WN_ABI_VERSION 1

/* error codes */
#define WN_OK 0
#define WN_EINVAL (-1)   /* bad argument (the reference raises ValueError, walnuts.py:309-320) */
#define WN_ECUDA (-2)    /* CUDA runtime error; text in wn_last_error() */
#define WN_ENOMEM (-3)
#define WN_EUNSUPPORTED (-4) /* target/dimension/mode combination has no kernel */
#define WN_ESTATE (-5)   /* call order violation (e.g. wn_run before wn_set_state) */

/* targets: the registry that replaces WALNUTSpy/targetDistr.py and test/targets.py */
#define WN_TARGET_STD_NORMAL 0   /* targetDistr.stdGauss :18-21, test/targets.py:4-7          */
#define WN_TARGET_DIAG_GAUSS 1   /* lp = -1/2 sum q_i^2 inv_var_i; data key "inv_var" [d]     */
#define WN_TARGET_FUNNEL 2       /* targetDistr.funnel10 :74-78 generalised to d = 1 + n      */
#define WN_TARGET_LOGREG 3       /* Bernoulli-logit + N(0,tau^2) prior; keys "X" [N,P], "y" [N] */
#define WN_TARGET_STOCK_WATSON 4 /* WALNUTSpy_examples/StockWatson/sw_innov.stan; key "y" [T] */
#define WN_TARGET_CORR_GAUSS 5   /* targetDistr.corrGauss :25-31 (2-d, rho = 0.5)             */
#define WN_TARGET_FUNNEL_PKG 6   /* test/targets.py:23-29 (different density from funnel10)   */
#define WN_TARGET_DENSE_GAUSS 7  /* lp = -1/2 q^T P q, dense precision P; data key "precision" [d*d]; d <= 128 */

/* User-defined CUDA targets (the role of the reference's arbitrary Python lpFun / logp, grad callables and of
 * walnuts_stan.py's compiled model): ids returned by wn_register_user_target() start here. */
#define WN_TARGET_USER_BASE 1000

/* transition semantics */
#define WN_MODE_WALNUTSPY 0 /* WALNUTSpy/WALNUTS.py + adaptiveIntegrators.py */
#define WN_MODE_PACKAGE 1   /* walnuts/walnuts.py */

/* macro-step integrators (WALNUTSPY mode) */
#define WN_INT_FIXED 0 /* adaptiveIntegrators.fixedLeapFrog     :49-59   (plain NUTS)        */
#define WN_INT_D 1     /* adaptiveIntegrators.adaptLeapFrogD    :65-137                      */
#define WN_INT_R2P 2   /* adaptiveIntegrators.adaptLeapFrogR2P  :361-475                     */
#define WN_INT_YOSHIDA 3 /* adaptiveIntegrators.adaptYoshidaD   :142-240 (4th-order triple)  */
#define WN_INT_FLOW 4     /* adaptiveIntegrators.adaptLeapFrogFlowD      :246-356 (flow-error criterion)      */
#define WN_INT_MIDPOINT 5 /* adaptiveIntegrators.adaptImplicitMidpointD  :478-641 (fixed-point iterations;
                             FPNewton=True, which needs a Hessian, is not built)                            */
#define WN_INT_RESCALED 6 /* adaptiveIntegrators.adaptRescaledLeapFrogD  :660-762 (per-dimension rescaling)  */

#define WN_DIAG_COLS 24 /* WALNUTS.py:180,670-693 */

/* kernel families (wn_last_plan): each is a separate set of template instantiations, picked per call */
#define WN_FAMILY_WPY 0   /* plain WALNUTSpy transition, adaptLeapFrogD / adaptLeapFrogR2P              */
#define WN_FAMILY_PKG 1   /* package mode (walnuts/walnuts.py)                                          */
#define WN_FAMILY_ADAPT 2 /* every integrator behind the runtime kind: adaptYoshidaD, warm-up adaptation,
                             orbit statistics                                                          */
#define WN_FAMILY_EXT 3   /* adaptLeapFrogFlowD / adaptImplicitMidpointD / adaptRescaledLeapFrogD        */
#define WN_FAMILY_NUTS 4  /* plain WALNUTSpy transition, fixedLeapFrog (plain NUTS)                     */

typedef struct wn_handle wn_handle;

typedef struct wn_config {
  int32_t target;      /* WN_TARGET_*                                                    */
  int32_t mode;        /* WN_MODE_*                                                      */
  int32_t integrator;  /* WN_INT_* (WALNUTSPY mode)                                      */
  int32_t d;           /* dimension of q / theta                                         */
  int32_t n_chains;    /* chains held by this handle (this GPU's shard)                  */
  int32_t device;      /* CUDA device ordinal                                            */
  int32_t dg;          /* leading coordinates stored per draw (generated = q[0:dg])      */
  int32_t M;           /* max doublings: WALNUTS(M=) / walnuts(max_nuts_depth=)          */
  int32_t minC, maxC;  /* integratorAuxPar.minC / maxC, adaptiveIntegrators.py:36-44     */
  int32_t compat;      /* 1 = reproduce the reference's latent defects bit-for-bit: PACKAGE mode B3/B5
                          (walnuts.py:194,242-245,272), WALNUTSPY mode A14(i) (WALNUTS.py:420 vs :443-459,
                          biases the funnel, DESIGN.md section 5); 0 = corrected semantics           */
  int32_t first_iteration; /* iteration number of the handle's first transition in the Philox counters; 0 or 1 = start
                          at 1 (WALNUTS.py:196 counts from 1).  A caller that creates a fresh handle per transition with
                          a FIXED seed (walnuts_step) must advance this, or every call replays the same streams */
  double H0;           /* macro step: WALNUTS(H0=) / walnuts(macro_step=)                */
  double jitter;       /* WALNUTS(stepSizeRandScale=), WALNUTS.py:298,395                */
  double delta;        /* WALNUTS(delta0=) / walnuts(max_error=)                         */
  double r2p_prob0;    /* integratorAuxPar.R2Pprob0                                      */
  double log_p0;       /* log(r2p_prob0), computed by the caller's libm (bit parity)     */
  double log_1mp0;     /* log(1 - r2p_prob0)                                             */
  uint64_t seed;       /* Philox key                                                     */
  uint64_t chain_offset; /* global id of this handle's chain 0 (multi-GPU sharding)      */
} wn_config;

int wn_abi_version(void);

/* name -> WN_TARGET_* ("std_normal","diag_gauss","funnel","logreg","stock_watson",
 * "corr_gauss","funnel_pkg","dense_gauss"); <0 if unknown. */
int wn_target_id(const char* name);

/* Load a user-target plug-in (built by walnuts_b200.targets.cuda_target() from csrc/wn_user_api.cuh, the user's
 * WN_TARGET_LP_GRAD function and csrc/wn_user_plugin.cuh) and return its target id (>= WN_TARGET_USER_BASE),
 * or <0.  The plug-in fixes the dimension d; its data array travels with wn_set_data(h, "data", ...).
 * The registry is process-wide and append-only (plug-ins stay loaded); registration is serialised internally. */
int wn_register_user_target(const char* plugin_path);

int wn_create(const wn_config* cfg, wn_handle** out);
void wn_destroy(wn_handle* h);

/* Target data / per-chain tuning.  `key`: "inv_var" [d], "inv_mass" [d] (PACKAGE mode metric,
 * walnuts.py:298), "X" [N*P row-major], "y" [N or T], "tau" [1], "precision" [d*d row-major], "H" [n_chains] and "delta"
 * [n_chains] (per-chain macro step / tolerance, overriding cfg.H0 / cfg.delta).
 * `on_device` != 0: `ptr` is a device pointer on cfg.device. */
int wn_set_data(wn_handle* h, const char* key, const double* ptr, int64_t n, int on_device);

/* Remaining integratorAuxPar fields (adaptiveIntegrators.py:36-44) used by WN_INT_MIDPOINT / WN_INT_RESCALED:
 * `key` = "maxFPiter" (default 30), "FPtol" (1e-8), "rescaledGradThresh" (5.0). */
int wn_set_aux(wn_handle* h, const char* key, double value);

/* Warm-up adaptation of the macro step H and the tolerance delta, per chain, as reference
 * WALNUTS.py:136-147 (setup), :313 (P-squared quantile of log igrConst, P2quantile.py:16-92) and
 * :701-712 (delta <- target / quantile(orbitEnergyError/delta), H <- delta^(1/3) exp(P2 quantile)).
 * Iterations 1..warmup_iter of the handle adapt; later ones use the adapted values.  Must be called
 * before the first wn_run.  WALNUTSPY mode only. */
int wn_set_adapt(wn_handle* h, int64_t warmup_iter, int adaptH, double adaptHtarget, int adaptDelta,
                 double adaptDeltaTarget, double adaptDeltaQuantile);

/* Positions of all chains, row-major [n_chains, d]. */
int wn_set_state(wn_handle* h, const double* q, int on_device);
int wn_get_state(wn_handle* h, double* q, int on_device);

/* Run n_iter transitions of every chain.
 *   draws  [n_iter, n_chains, dg] or NULL
 *   diag   [n_iter, n_chains, WN_DIAG_COLS] or NULL  (columns as WALNUTS.py:670-693)
 *   nevalF, nevalB [n_chains] or NULL: gradient evaluations of this call (forward / reversibility
 *   passes; the one evaluation at the start of each iteration, WALNUTS.py:249, is not counted,
 *   like the reference).
 * Iterations continue the Philox streams of earlier calls on the same handle. */
int wn_run(wn_handle* h, int64_t n_iter, double* draws, double* diag, uint64_t* nevalF,
           uint64_t* nevalB, int on_device);

/* wn_run plus the per-iteration orbit statistics of WALNUTS(recordOrbitStats=True) (WALNUTS.py:182-184,
 * 274-276, 331-333, ...): orbit_min / orbit_max [n_iter, n_chains, dg] = element-wise min / max of the leading
 * dg coordinates over every state visited by the orbit of that iteration (both NULL to skip). */
int wn_run_stats(wn_handle* h, int64_t n_iter, double* draws, double* diag, uint64_t* nevalF,
                 uint64_t* nevalB, double* orbit_min, double* orbit_max, int on_device);

/* Same, asynchronous on the handle's stream with device buffers only; pair with wn_sync(). */
int wn_run_async(wn_handle* h, int64_t n_iter, double* d_draws, double* d_diag,
                 uint64_t* d_nevalF, uint64_t* d_nevalB);
int wn_sync(wn_handle* h);

/* The whole step with HOST buffers, asynchronous on the handle's stream: copy `q_in` [n_chains, d] to the device
 * (NULL: keep the current positions), run n_iter transitions, copy draws / diag / nevalF / nevalB (each may be
 * NULL) and the final positions `q_out` [n_chains, d] (may be NULL) back.  Every buffer is host memory; buffers
 * from wn_alloc_pinned() make the copies truly asynchronous, so that two handles on one device overlap the
 * copies of one with the kernel of the other.  Pair with wn_sync().  This is the host-buffer form of the
 * reference's per-call contract (caller-owned numpy arrays in, fresh arrays out: WALNUTS.py:111,724-727). */
int wn_run_host_async(wn_handle* h, int64_t n_iter, const double* q_in, double* draws, double* diag,
                      uint64_t* nevalF, uint64_t* nevalB, double* q_out);

/* page-locked host memory for the asynchronous host-buffer path */
int wn_alloc_pinned(int64_t bytes, void** out);
int wn_free_pinned(void* p);

/* Device time of the last wn_run / wn_run_async kernel in milliseconds (CUDA events on the
 * handle's stream), its launch count, and the total gradient evaluations it performed. */
int wn_last_kernel_ms(wn_handle* h, float* ms);
int wn_last_launches(wn_handle* h, int64_t* n);
int wn_last_grad_evals(wn_handle* h, uint64_t* forward, uint64_t* backward);

/* The launch plan of the last wn_run* call: out = {WN_FAMILY_*, threads per chain G, coordinate pairs per thread E2,
 * threads per block NT}.  G > NT means one chain per thread-block cluster of G / NT blocks (std_normal and diag_gauss
 * above d = 4096).  A handle that has not run yet reports {-1, 0, 0, 0}.  For testing and tuning. */
int wn_last_plan(wn_handle* h, int32_t out[4]);

/* Chain slots of the last wn_run* launch: the chain groups resident at once (blocks x groups per block, or clusters
 * when G > NT), at most n_chains.  For testing and tuning. */
int wn_last_slots(wn_handle* h, int64_t* n);

/* Cross-chain moments of the current state over this handle's chains: mean[d], var[d]
 * (unbiased).  Multi-GPU callers reduce (n, sum, sumsq) themselves. */
int wn_moments(wn_handle* h, double* mean, double* var);

/* ---- multi-GPU: chains shard across GPUs (cfg.chain_offset) with no exchange while sampling; the collectives below
 * are the only cross-GPU traffic (SURVEY.md section 8(b)/(e): "NCCL inside if multi-GPU").  NCCL is bound at run time
 * (dlopen of libnccl.so.2; a copy already loaded by the process, e.g. torch's, is shared). ----
 * wn_comm_load: optional explicit path of libnccl.so.2.
 * Multi-process (one rank per GPU): rank 0 calls wn_comm_unique_id, ships the 128 bytes to the other ranks by any
 * means, every rank calls wn_comm_init_rank.  Single process: wn_comm_init_all over one handle per GPU (the later
 * collective calls must then be issued concurrently, one host thread per handle). */
int wn_comm_load(const char* libnccl_path);
int wn_comm_unique_id(void* id128);
int wn_comm_init_rank(wn_handle* h, int nranks, int rank, const void* id128);
int wn_comm_init_all(wn_handle** hs, int n);
int wn_comm_destroy(wn_handle* h);

/* Bulk effective sample size and split-R-hat per monitored coordinate (rank-normalised, split chains, Geyer's
 * initial monotone sequence over all lags: Vehtari et al. 2021 = arviz.ess, the quantity of the reference's
 * mainGaussESS.py:50-55) of draws [n_iter, n_chains, dg] as written by wn_run, computed on the device.  With a
 * communicator the draws of ALL ranks are pooled by one NCCL all-gather (every rank passes the same n_iter,
 * n_chains, dg and receives the same result).  split = 0 keeps whole chains.  ess, rhat: host arrays [dg]. */
int wn_ess_rhat(wn_handle* h, const double* draws, int64_t n_iter, int64_t n_chains, int32_t dg, int on_device,
                int32_t split, double* ess, double* rhat);

/* Posterior summary per monitored coordinate, computed on the device: out is a host array [dg][WN_SUMMARY_COLS] with
 * the columns below.  Draws, limits (n_iter >= 4, <= 25 600 draws per split chain, <= 2^31 draws per coordinate) and
 * pooling are those of wn_ess_rhat: with a communicator the draws of all ranks are pooled by the same one all-gather,
 * global chain order is rank-major (the devices= sharding order), and every rank receives the same result.
 * superchain_size = 0: no nested R-hat (that column is NaN).  s > 0: global chains k*s ... k*s + s - 1 form superchain k;
 * the chain count over all ranks must be a multiple of s with at least 2 superchains, else WN_EINVAL.
 *
 * Definitions for one coordinate: x has M chains x N draws, S = M N.  "Split ESS of y" splits every chain of y into
 * [0, h) and [N - h, N), h = N / 2, and applies the estimator of wn_ess_rhat WITHOUT rank normalisation.
 *   WN_S_MEAN, WN_S_SD          mean and sd over all S draws; sd with 1 / (S - 1)
 *   WN_S_Q05, _Q50, _Q95        linear-interpolation quantiles (numpy's default) of the S sorted draws
 *   WN_S_MCSE_MEAN              sd / sqrt(split ESS of x)
 *   WN_S_MCSE_SD                c = (x - mean)^2, E = mean(c), varvar = (mean(c^2) - E^2) / split ESS of c,
 *                               sqrt(varvar / (4 E))
 *   WN_S_ESS_BULK               the ess of wn_ess_rhat with split = 1, bit for bit
 *   WN_S_ESS_TAIL               min(split ESS of 1[x <= q05], split ESS of 1[x <= q95]); indicators not rank-normalised
 *   WN_S_RHAT                   max(the rhat of wn_ess_rhat with split = 1, the same R-hat of |x - q50|)
 *   WN_S_NESTED_RHAT            sqrt(1 + B / W) on the raw draws (Margossian, Hoffman, Sountsov, Riou-Durand, Vehtari,
 *                               Gelman 2024): B = 1/(K-1) sum_k (xbar_k - xbar)^2 over the K superchain means,
 *                               W = 1/K sum_k (Btilde_k + Wtilde_k), Btilde_k = 1/(s-1) sum_m (xbar_mk - xbar_k)^2
 *                               (0 for s = 1), Wtilde_k = 1/s sum_m (within-chain variance with 1 / (N - 1))
 * Conventions, as wn_ess_rhat: ranks are ordinal (ties broken by chain-major position) and taken over all S draws
 * before the split, so for odd N the middle draw is ranked but dropped; an ESS or R-hat of a series with zero variance
 * is NaN, and so is every column computed from one (min and max are NaN when either argument is). */
#define WN_SUMMARY_COLS 11
#define WN_S_MEAN 0
#define WN_S_SD 1
#define WN_S_Q05 2
#define WN_S_Q50 3
#define WN_S_Q95 4
#define WN_S_MCSE_MEAN 5
#define WN_S_MCSE_SD 6
#define WN_S_ESS_BULK 7
#define WN_S_ESS_TAIL 8
#define WN_S_RHAT 9
#define WN_S_NESTED_RHAT 10
int wn_summary(wn_handle* h, const double* draws, int64_t n_iter, int64_t n_chains, int32_t dg, int on_device,
               int32_t superchain_size, double* out);

/* wn_moments over the chains of ALL ranks of the communicator (two all-reduces of d + 1 doubles). */
int wn_moments_all(wn_handle* h, double* mean, double* var);

/* the CUDA stream (cudaStream_t) owned by the handle, for event timing by the caller */
void* wn_stream(wn_handle* h);

const char* wn_last_error(const wn_handle* h);

/* FP64 FMA throughput micro-benchmark (roofline denominator): returns achieved FLOP/s. */
int wn_fp64_peak(int device, double* flops_per_s);

#ifdef __cplusplus
}
#endif
#endif /* WALNUTS_CUDA_H */
