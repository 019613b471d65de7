// C-ABI of the B200-native WALNUTS/NUTS sampler (include/walnuts_cuda.h).
// Host side: handle management, kernel dispatch by (target, dimension), launch + timing.
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/walnuts_cuda.h"
#include "wn_dispatch.cuh"
#include "wn_handle.hpp"

using namespace wn;

// kernel dispatch: wn_dispatch.cuh; one translation unit per kernel family (plans_*.cu) so they compile in parallel

// User targets (SURVEY.md 8f N4): plug-in libraries built by walnuts_b200.targets.cuda_target() from
// csrc/wn_user_api.cuh + the user's source + csrc/wn_user_plugin.cuh.  Target ids >= WN_TARGET_USER_BASE.
struct UserTarget {
  void* dl;
  int d;
  int (*plan)(int, int*, int*, int*, size_t*, int*);
  int (*occupancy)(int, int);
  int (*launch)(int, int, const void*, unsigned, void*);
};
// append-only registry: a deque keeps the addresses of earlier entries stable while wn_register_user_target
// appends from another host thread; the mutex orders appends against look-ups
static std::mutex& user_mutex() {
  static std::mutex m;
  return m;
}
static std::deque<UserTarget>& user_targets() {
  static std::deque<UserTarget> v;
  return v;
}
static const UserTarget* user_target(int id) {
  std::lock_guard<std::mutex> lock(user_mutex());
  const int i = id - WN_TARGET_USER_BASE;
  return (i >= 0 && i < (int)user_targets().size()) ? &user_targets()[i] : nullptr;
}
static int user_family(const wn_config& c) { return c.mode == WN_MODE_PACKAGE ? FAM_PKG : FAM_EXT; }

// `general`: the call needs the kernels that carry every integrator behind the runtime kind plus the adaptation and
// orbit-statistics code ("adapt" family): warm-up iterations, wn_run_stats with orbit buffers, adaptYoshidaD.
// `fam` receives the family (FAM_*) the plan was picked from.
static bool pick_plan(const wn_config& c, bool general, LaunchPlan& p, int& fam) {
  if (c.target >= WN_TARGET_USER_BASE) {
    const UserTarget* u = user_target(c.target);
    if (!u || u->d != c.d) return false;
    int pkg = 0;
    p.fn = nullptr;   // launched inside the plug-in
    fam = user_family(c);
    u->plan(fam, &p.G, &p.E2, &p.NT, &p.smem, &pkg);
    p.package = pkg != 0;
    return true;
  }
  if (c.mode == WN_MODE_PACKAGE) { fam = FAM_PKG; return wn_pick_plan_pkg(c, p); }
  if (c.integrator > WN_INT_YOSHIDA) { fam = FAM_EXT; return wn_pick_plan_ext(c, p); }
  if (general || c.integrator == WN_INT_YOSHIDA) { fam = FAM_ADAPT; return wn_pick_plan_adapt(c, p); }
  if (c.integrator == WN_INT_FIXED) { fam = FAM_NUTS; return wn_pick_plan_nuts(c, p); }
  fam = FAM_WPY;
  return wn_pick_plan_wpy(c, p);
}

// ------------------------------------------------------------------------------------------
// small utility kernels
// ------------------------------------------------------------------------------------------
__global__ void moments_kernel(const double* __restrict__ state, int n_chains, int d,
                               double* __restrict__ mean, double* __restrict__ var) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  double s = 0.0;
  for (int c = 0; c < n_chains; ++c) s += state[(size_t)c * d + j];
  const double m = s / n_chains;
  double ss = 0.0;
  for (int c = 0; c < n_chains; ++c) {
    const double x = state[(size_t)c * d + j] - m;
    ss = fma(x, x, ss);
  }
  mean[j] = m;
  var[j] = n_chains > 1 ? ss / (n_chains - 1) : 0.0;
}

__global__ void transpose_kernel(const double* __restrict__ X, double* __restrict__ XT, int N, int P) {
  __shared__ double tile[32][33];
  const int n0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int n = n0 + i, k = k0 + threadIdx.x;
    tile[i][threadIdx.x] = (n < N && k < P) ? X[(size_t)n * P + k] : 0.0;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int k = k0 + i, n = n0 + threadIdx.x;
    if (k < P && n < N) XT[(size_t)k * N + n] = tile[threadIdx.x][i];
  }
}

__global__ void fp64_fma_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6,
         x7 = x0 + 7;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}

// ------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int wn_abi_version(void) { return WN_ABI_VERSION; }

int wn_register_user_target(const char* path) {
  if (!path) return WN_EINVAL;
  void* dl = dlopen(path, RTLD_NOW | RTLD_LOCAL);
  if (!dl) return WN_EINVAL;
  UserTarget u;
  u.dl = dl;
  auto abi = (int (*)(void))dlsym(dl, "wn_user_abi");
  auto dim = (int (*)(void))dlsym(dl, "wn_user_dim");
  u.plan = (int (*)(int, int*, int*, int*, size_t*, int*))dlsym(dl, "wn_user_plan");
  u.occupancy = (int (*)(int, int))dlsym(dl, "wn_user_occupancy");
  u.launch = (int (*)(int, int, const void*, unsigned, void*))dlsym(dl, "wn_user_launch");
  if (!abi || !dim || !u.plan || !u.occupancy || !u.launch || abi() != WN_ABI_VERSION) {
    dlclose(dl);
    return WN_EUNSUPPORTED;
  }
  u.d = dim();
  std::lock_guard<std::mutex> lock(user_mutex());
  user_targets().push_back(u);
  return WN_TARGET_USER_BASE + (int)user_targets().size() - 1;
}

int wn_target_id(const char* name) {
  if (!name) return WN_EINVAL;
  static const struct { const char* n; int id; } tab[] = {
      {"std_normal", WN_TARGET_STD_NORMAL}, {"diag_gauss", WN_TARGET_DIAG_GAUSS},
      {"funnel", WN_TARGET_FUNNEL},         {"logreg", WN_TARGET_LOGREG},
      {"stock_watson", WN_TARGET_STOCK_WATSON}, {"corr_gauss", WN_TARGET_CORR_GAUSS},
      {"funnel_pkg", WN_TARGET_FUNNEL_PKG}, {"dense_gauss", WN_TARGET_DENSE_GAUSS}};
  for (auto& e : tab)
    if (!strcmp(e.n, name)) return e.id;
  return WN_EINVAL;
}

const char* wn_last_error(const wn_handle* h) { return h ? h->err.c_str() : "null handle"; }

int wn_create(const wn_config* cfg, wn_handle** out) {
  if (!cfg || !out) return WN_EINVAL;
  *out = nullptr;
  wn_handle* h = new wn_handle();
  h->cfg = *cfg;
  *out = h;  // returned even on failure so that wn_last_error() can be read; caller destroys it
  const wn_config& c = h->cfg;
  // argument validation mirrors reference walnuts.py:309-320 (ValueError) and WALNUTS.py:140,146
  if (c.d <= 0 || c.n_chains <= 0) return fail(h, WN_EINVAL, "d and n_chains must be positive");
  if (!(c.H0 > 0)) return fail(h, WN_EINVAL, "non-positive macro_step");
  if (!(c.M > 0) || c.M > 30) return fail(h, WN_EINVAL, "non-positive max_nuts_depth (or > 30)");
  if (!(c.delta > 0)) return fail(h, WN_EINVAL, "non-positive max_error");
  if (c.mode != WN_MODE_WALNUTSPY && c.mode != WN_MODE_PACKAGE) return fail(h, WN_EINVAL, "bad mode");
  if (c.mode == WN_MODE_WALNUTSPY) {
    if (c.integrator < WN_INT_FIXED || c.integrator > WN_INT_RESCALED) return fail(h, WN_EINVAL, "bad integrator");
    if (c.minC < 0 || c.maxC < c.minC || c.maxC > 30) return fail(h, WN_EINVAL, "need 0 <= minC <= maxC <= 30");
    if (!(c.jitter >= 0 && c.jitter < 1)) return fail(h, WN_EINVAL, "stepSizeRandScale must be in [0,1)");
  }
  if (c.dg < 0 || c.dg > c.d) return fail(h, WN_EINVAL, "dg must be in [0, d]");
  if (c.first_iteration < 0) return fail(h, WN_EINVAL, "first_iteration must be >= 0");
  h->iter_done = c.first_iteration > 1 ? (uint32_t)c.first_iteration - 1u : 0u;
  h->iter_base = h->iter_done;
  LaunchPlan p;
  int fam;
  if (!pick_plan(c, false, p, fam)) return fail(h, WN_EUNSUPPORTED, "no CUDA kernel for this target/dimension");
  CUDA_TRY(h, cudaSetDevice(c.device));
  cudaDeviceProp prop;
  CUDA_TRY(h, cudaGetDeviceProperties(&prop, c.device));
  h->num_sms = prop.multiProcessorCount;
  CUDA_TRY(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CUDA_TRY(h, cudaEventCreate(&h->ev0));
  CUDA_TRY(h, cudaEventCreate(&h->ev1));
  CUDA_TRY(h, cudaMalloc(&h->d_state, (size_t)c.n_chains * c.d * sizeof(double)));
  CUDA_TRY(h, cudaMalloc(&h->d_queue, sizeof(unsigned int)));
  CUDA_TRY(h, cudaMalloc(&h->d_totals, 2 * sizeof(unsigned long long)));
  return WN_OK;
}

void wn_destroy(wn_handle* h) {
  if (!h) return;
  wn_comm_destroy(h);
  if (h->stream) {
    cudaSetDevice(h->cfg.device);
    cudaStreamSynchronize(h->stream);
  }
  cudaFree(h->d_state); cudaFree(h->d_scratch); cudaFree(h->d_queue); cudaFree(h->d_totals);
  wn_sched_free(h);
  cudaFree(h->o_draws); cudaFree(h->o_diag); cudaFree(h->o_lo); cudaFree(h->o_hi); cudaFree(h->o_f); cudaFree(h->o_b);
  cudaFree(h->d_p0); cudaFree(h->d_p1); cudaFree(h->d_p2); cudaFree(h->d_inv_mass); cudaFree(h->d_H); cudaFree(h->d_delta); cudaFree(h->d_adapt_state); cudaFree(h->d_adapt_hist);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

static int upload(wn_handle* h, double** dst, const double* src, int64_t n, int on_device) {
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  if (*dst) { cudaFree(*dst); *dst = nullptr; }
  CUDA_TRY(h, cudaMalloc(dst, (size_t)n * sizeof(double)));
  CUDA_TRY(h, cudaMemcpyAsync(*dst, src, (size_t)n * sizeof(double),
                              on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return WN_OK;
}

int wn_set_data(wn_handle* h, const char* key, const double* ptr, int64_t n, int on_device) {
  if (!h || !key || !ptr || n <= 0) return fail(h, WN_EINVAL, "wn_set_data: bad argument");
  const wn_config& c = h->cfg;
  if (!strcmp(key, "inv_var")) {
    if (n != c.d) return fail(h, WN_EINVAL, "inv_var must have d entries");
    h->n_p0 = n;
    int rc = upload(h, &h->d_p0, ptr, n, on_device);
    if (rc) return rc;
    std::vector<double> tmp((size_t)n);
    CUDA_TRY(h, cudaMemcpy(tmp.data(), h->d_p0, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    h->inv_var_max = 0.0;
    h->inv_var_min = tmp.empty() ? 0.0 : tmp[0];
    for (double x : tmp) {
      h->inv_var_max = (fabs(x) > h->inv_var_max || x != x) ? fabs(x) : h->inv_var_max;
      h->inv_var_min = (x < h->inv_var_min || x != x) ? x : h->inv_var_min;     // NaN sticks: no certificate
    }
    return WN_OK;
  }
  if (!strcmp(key, "inv_mass")) {
    if (n != c.d) return fail(h, WN_EINVAL, "size mismatch between theta and inv_mass");
    return upload(h, &h->d_inv_mass, ptr, n, on_device);
  }
  if (!strcmp(key, "H")) {
    if (n != c.n_chains) return fail(h, WN_EINVAL, "H must have n_chains entries");
    return upload(h, &h->d_H, ptr, n, on_device);
  }
  if (!strcmp(key, "delta")) {
    if (n != c.n_chains) return fail(h, WN_EINVAL, "delta must have n_chains entries");
    return upload(h, &h->d_delta, ptr, n, on_device);
  }
  if (!strcmp(key, "X")) {
    if (n % c.d != 0) return fail(h, WN_EINVAL, "X must have N*d entries (row-major [N, d])");
    const int N = (int)(n / c.d);
    int rc = upload(h, &h->d_p0, ptr, n, on_device);
    if (rc) return rc;
    h->n_p0 = N;
    if (h->d_p2) { cudaFree(h->d_p2); h->d_p2 = nullptr; }
    CUDA_TRY(h, cudaMalloc(&h->d_p2, (size_t)n * sizeof(double)));
    transpose_kernel<<<dim3((N + 31) / 32, (c.d + 31) / 32), dim3(32, 8), 0, h->stream>>>(h->d_p0, h->d_p2, N, c.d);
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return WN_OK;
  }
  if (!strcmp(key, "y")) {
    if (c.target == WN_TARGET_STOCK_WATSON) { h->n_p0 = n; return upload(h, &h->d_p0, ptr, n, on_device); }
    h->n_p1 = n;
    return upload(h, &h->d_p1, ptr, n, on_device);
  }
  if (!strcmp(key, "precision")) {
    if (c.target != WN_TARGET_DENSE_GAUSS) return fail(h, WN_EINVAL, "data key \"precision\" belongs to dense_gauss");
    if (n != (int64_t)c.d * c.d) return fail(h, WN_EINVAL, "precision must have d*d entries (row-major [d, d])");
    h->n_p0 = c.d;
    return upload(h, &h->d_p0, ptr, n, on_device);
  }
  if (!strcmp(key, "data")) {   // user targets: the array handed to the user's lp_grad
    if (c.target < WN_TARGET_USER_BASE) return fail(h, WN_EINVAL, "data key \"data\" belongs to user targets");
    h->n_p0 = n;
    return upload(h, &h->d_p0, ptr, n, on_device);
  }
  if (!strcmp(key, "tau")) {
    if (on_device) return fail(h, WN_EINVAL, "tau must be a host scalar");
    h->tau = ptr[0];
    return WN_OK;
  }
  return fail(h, WN_EINVAL, std::string("unknown data key ") + key);
}

int wn_set_aux(wn_handle* h, const char* key, double value) {
  if (!h || !key) return fail(h, WN_EINVAL, "wn_set_aux: bad argument");
  if (!strcmp(key, "maxFPiter")) {
    if (!(value >= 0 && value <= 1e6)) return fail(h, WN_EINVAL, "bad maxFPiter");
    h->maxFPiter = (int)value;
    return WN_OK;
  }
  if (!strcmp(key, "FPtol")) { h->FPtol = value; return WN_OK; }
  if (!strcmp(key, "rescaledGradThresh")) { h->gradThresh = value; return WN_OK; }
  return fail(h, WN_EINVAL, std::string("unknown aux key ") + key);
}

int wn_set_adapt(wn_handle* h, int64_t warmup_iter, int adaptH, double adaptHtarget, int adaptDelta,
                 double adaptDeltaTarget, double adaptDeltaQuantile) {
  if (!h) return WN_EINVAL;
  const wn_config& c = h->cfg;
  if (c.mode != WN_MODE_WALNUTSPY) return fail(h, WN_EINVAL, "warm-up adaptation exists in WALNUTSPY mode only");
  if (warmup_iter < 0 || warmup_iter > (1 << 24)) return fail(h, WN_EINVAL, "bad warmup_iter");
  if (adaptH && (adaptHtarget < 0.0 || adaptHtarget > 1.0)) return fail(h, WN_EINVAL, "bad adaptHtarget");        // WALNUTS.py:140
  if (adaptDelta && adaptDeltaTarget < 0.0) return fail(h, WN_EINVAL, "bad adaptDeltaTarget");                    // WALNUTS.py:146
  if (adaptDelta && !(adaptDeltaQuantile >= 0.0 && adaptDeltaQuantile <= 1.0)) return fail(h, WN_EINVAL, "bad adaptDeltaQuantile");
  if (h->iter_done != h->iter_base) return fail(h, WN_ESTATE, "wn_set_adapt must precede the first wn_run");
  if (h->iter_base != 0 && warmup_iter > 0 && (adaptH || adaptDelta))
    return fail(h, WN_EINVAL, "warm-up adaptation needs first_iteration = 1 (the warm-up window is counted in iterations)");
  CUDA_TRY(h, cudaSetDevice(c.device));
  cudaFree(h->d_adapt_state); cudaFree(h->d_adapt_hist);
  h->d_adapt_state = h->d_adapt_hist = nullptr;
  h->warmup_iter = (int)warmup_iter; h->adaptH = adaptH ? 1 : 0; h->adaptDelta = adaptDelta ? 1 : 0;
  h->adHtarget = adaptHtarget; h->adTarget = adaptDeltaTarget; h->adQuant = adaptDeltaQuantile;
  h->adapt_exported = false;
  if (warmup_iter == 0 || (!adaptH && !adaptDelta)) return WN_OK;
  std::vector<double> init((size_t)c.n_chains * WN_ADAPT_STRIDE, 0.0), Hs, ds;
  if (h->d_H) { Hs.resize(c.n_chains); CUDA_TRY(h, cudaMemcpy(Hs.data(), h->d_H, c.n_chains * sizeof(double), cudaMemcpyDeviceToHost)); }
  if (h->d_delta) { ds.resize(c.n_chains); CUDA_TRY(h, cudaMemcpy(ds.data(), h->d_delta, c.n_chains * sizeof(double), cudaMemcpyDeviceToHost)); }
  for (int i = 0; i < c.n_chains; ++i) {
    double* a = &init[(size_t)i * WN_ADAPT_STRIDE];
    a[0] = Hs.empty() ? c.H0 : Hs[i];
    a[1] = ds.empty() ? c.delta : ds[i];
    for (int k = 0; k < 5; ++k) a[8 + k] = k + 1;     // P2quantile.n = 1..5 (P2quantile.py:22)
  }
  CUDA_TRY(h, cudaMalloc(&h->d_adapt_state, init.size() * sizeof(double)));
  CUDA_TRY(h, cudaMemcpy(h->d_adapt_state, init.data(), init.size() * sizeof(double), cudaMemcpyHostToDevice));
  if (adaptDelta) {
    CUDA_TRY(h, cudaMalloc(&h->d_adapt_hist, (size_t)c.n_chains * warmup_iter * sizeof(double)));
    CUDA_TRY(h, cudaMemset(h->d_adapt_hist, 0, (size_t)c.n_chains * warmup_iter * sizeof(double)));
  }
  return WN_OK;
}

int wn_set_state(wn_handle* h, const double* q, int on_device) {
  if (!h || !q) return fail(h, WN_EINVAL, "wn_set_state: bad argument");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  const size_t bytes = (size_t)h->cfg.n_chains * h->cfg.d * sizeof(double);
  CUDA_TRY(h, cudaMemcpyAsync(h->d_state, q, bytes,
                              on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->have_state = true;
  return WN_OK;
}

int wn_get_state(wn_handle* h, double* q, int on_device) {
  if (!h || !q) return fail(h, WN_EINVAL, "wn_get_state: bad argument");
  if (!h->have_state) return fail(h, WN_ESTATE, "no state set");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  const size_t bytes = (size_t)h->cfg.n_chains * h->cfg.d * sizeof(double);
  CUDA_TRY(h, cudaMemcpyAsync(q, h->d_state, bytes,
                              on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return WN_OK;
}

static int run_async_impl(wn_handle* h, int64_t n_iter, double* d_draws, double* d_diag, uint64_t* d_nevalF,
                          uint64_t* d_nevalB, double* d_omin, double* d_omax);

int wn_run_async(wn_handle* h, int64_t n_iter, double* d_draws, double* d_diag, uint64_t* d_nevalF,
                 uint64_t* d_nevalB) {
  return run_async_impl(h, n_iter, d_draws, d_diag, d_nevalF, d_nevalB, nullptr, nullptr);
}

static int run_async_impl(wn_handle* h, int64_t n_iter, double* d_draws, double* d_diag, uint64_t* d_nevalF,
                          uint64_t* d_nevalB, double* d_omin, double* d_omax) {
  if (!h) return WN_EINVAL;
  if ((d_omin == nullptr) != (d_omax == nullptr)) return fail(h, WN_EINVAL, "orbit_min and orbit_max go together");
  if (d_omin && h->cfg.mode != WN_MODE_WALNUTSPY) return fail(h, WN_EINVAL, "orbit statistics exist in WALNUTSPY mode only");
  if (d_diag && h->cfg.mode != WN_MODE_WALNUTSPY)
    return fail(h, WN_EINVAL, "the 24-column diagnostics exist in WALNUTSPY mode only (walnuts.py returns draws only)");
  if (n_iter <= 0 || n_iter > 0x7fffffff) return fail(h, WN_EINVAL, "n_iter must be positive");
  if (!h->have_state) return fail(h, WN_ESTATE, "wn_run before wn_set_state");
  const wn_config& c = h->cfg;
  if (c.target == WN_TARGET_DIAG_GAUSS && !h->d_p0) return fail(h, WN_ESTATE, "diag_gauss needs data key inv_var");
  if (c.target == WN_TARGET_LOGREG && (!h->d_p0 || !h->d_p1 || h->n_p1 != h->n_p0))
    return fail(h, WN_ESTATE, "logreg needs data keys X [N*d] and y [N]");
  if (c.target == WN_TARGET_STOCK_WATSON && (!h->d_p0 || h->n_p0 * 3 != c.d))
    return fail(h, WN_ESTATE, "stock_watson needs data key y with T = d/3 entries");
  if (c.target == WN_TARGET_DENSE_GAUSS && (!h->d_p0 || h->n_p0 != c.d))
    return fail(h, WN_ESTATE, "dense_gauss needs data key precision [d*d]");
  if (c.mode == WN_MODE_PACKAGE && !h->d_inv_mass) return fail(h, WN_ESTATE, "package mode needs data key inv_mass");
  LaunchPlan p;
  int fam;
  const bool adapting = h->d_adapt_state != nullptr && h->iter_done < (uint32_t)h->warmup_iter;
  if (!pick_plan(c, adapting || d_omin != nullptr, p, fam)) return fail(h, WN_EUNSUPPORTED, "no CUDA kernel for this target/dimension");
  CUDA_TRY(h, cudaSetDevice(c.device));
  const UserTarget* ut = user_target(c.target);
  int occ = 0;
  if (ut) {
    occ = ut->occupancy(user_family(c), c.device);
    if (occ < 0) return fail(h, WN_ECUDA, "user target plug-in: occupancy query failed");
  } else {
    CUDA_TRY(h, cudaFuncSetAttribute(p.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    CUDA_TRY(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, p.fn, p.NT, p.smem));
  }
  if (occ < 1) return fail(h, WN_ECUDA, "kernel does not fit on an SM");
  // G > NT: one chain per cluster of CL = G / NT blocks (wn_walnutspy.cuh); a slot is a cluster, and the resident
  // cluster count comes from the runtime (how many clusters of CL blocks the GPCs hold), not from SMs x blocks per SM
  const int cl = (p.G > p.NT) ? p.G / p.NT : 1;
  cudaLaunchAttribute cattr[1];
  cattr[0].id = cudaLaunchAttributeClusterDimension;
  cattr[0].val.clusterDim.x = (unsigned)cl;
  cattr[0].val.clusterDim.y = 1;
  cattr[0].val.clusterDim.z = 1;
  cudaLaunchConfig_t lcfg = {};
  lcfg.blockDim = dim3(p.NT);
  lcfg.dynamicSmemBytes = p.smem;
  lcfg.stream = h->stream;
  lcfg.attrs = cattr;
  lcfg.numAttrs = 1;
  long long blocks;
  int nslot;
  if (cl > 1) {
    lcfg.gridDim = dim3((unsigned)cl);
    int ncl = 0;
    CUDA_TRY(h, cudaOccupancyMaxActiveClusters(&ncl, p.fn, &lcfg));
    if (ncl < 1) return fail(h, WN_ECUDA, "no cluster of this kernel fits on the GPU");
    const long long clusters = (ncl < c.n_chains) ? ncl : c.n_chains;
    blocks = clusters * cl;
    nslot = (int)clusters;
  } else {
    const int gpb = p.NT / p.G;
    blocks = (long long)h->num_sms * occ;
    const long long need = ((long long)c.n_chains + gpb - 1) / gpb;
    if (blocks > need) blocks = need;
    nslot = (int)blocks * gpb;
  }
  const int nvec = p.package ? package_scratch_vectors(c.M) : scratch_vectors(c.M);
  const size_t sbytes = (size_t)nvec * p.E2 * nslot * p.G * sizeof(double2);
  if (sbytes > h->scratch_bytes) {
    if (h->d_scratch) cudaFree(h->d_scratch);
    h->d_scratch = nullptr;
    h->scratch_bytes = 0;
    CUDA_TRY(h, cudaMalloc(&h->d_scratch, sbytes));
    h->scratch_bytes = sbytes;
  }
  CUDA_TRY(h, cudaMemsetAsync(h->d_queue, 0, sizeof(unsigned int), h->stream));
  CUDA_TRY(h, cudaMemsetAsync(h->d_totals, 0, 2 * sizeof(unsigned long long), h->stream));

  TargetParams tp;
  tp.p0 = h->d_p0; tp.p1 = h->d_p1; tp.p2 = h->d_p2; tp.n0 = (int)h->n_p0; tp.n1 = (int)h->n_p1;
  tp.c0 = (c.target == WN_TARGET_DIAG_GAUSS) ? h->inv_var_max : 1.0 / (h->tau * h->tau);
  tp.c1 = (c.target == WN_TARGET_DIAG_GAUSS) ? h->inv_var_min : 0.0;

  if (h->d_adapt_state && !adapting && !h->adapt_exported) {
    // warm-up is over: freeze the adapted (H, delta) of every chain as its step size / tolerance
    if (!h->d_H) CUDA_TRY(h, cudaMalloc(&h->d_H, (size_t)c.n_chains * sizeof(double)));
    if (!h->d_delta) CUDA_TRY(h, cudaMalloc(&h->d_delta, (size_t)c.n_chains * sizeof(double)));
    CUDA_TRY(h, cudaMemcpy2DAsync(h->d_H, sizeof(double), h->d_adapt_state, WN_ADAPT_STRIDE * sizeof(double),
                                  sizeof(double), c.n_chains, cudaMemcpyDeviceToDevice, h->stream));
    CUDA_TRY(h, cudaMemcpy2DAsync(h->d_delta, sizeof(double), h->d_adapt_state + 1, WN_ADAPT_STRIDE * sizeof(double),
                                  sizeof(double), c.n_chains, cudaMemcpyDeviceToDevice, h->stream));
    h->adapt_exported = true;
  }
  CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
  // queue order of this call: the chains that were longest in the previous call first (wn_sched.cu)
  // -- for kernels whose chains share a warp (small d): there the per-chain cost is heavy-tailed and the gain measured
  // (+3-4 % at config 3); with whole warps per chain it measured neutral (C2) to slightly negative (C4), so those keep
  // the natural order
  const unsigned int* order = nullptr;
  if (p.G < 32)
    if (const int src = wn_sched_prepare(h, nslot, 32 / p.G, &order)) return src;
  if (!p.package) {
    RunParams P;
    memset(&P, 0, sizeof(P));
    P.n_chains = c.n_chains; P.d = c.d; P.dg = c.dg; P.M = c.M; P.kind = c.integrator;
    P.minC = c.minC; P.maxC = c.maxC; P.n_iter = (int)n_iter; P.iter0 = h->iter_done + 1;
    P.compat = c.compat;
    P.seed_lo = (uint32_t)(c.seed & 0xffffffffu); P.seed_hi = (uint32_t)(c.seed >> 32);
    P.chain_offset = (uint32_t)c.chain_offset;
    P.H0 = c.H0; P.delta0 = c.delta; P.jitter = c.jitter; P.p0 = c.r2p_prob0;
    P.log_p0 = c.log_p0; P.log_1mp0 = c.log_1mp0;
    P.warmup_iter = h->warmup_iter; P.adaptH = h->adaptH; P.adaptDelta = h->adaptDelta;
    P.p2prob = 1.0 - h->adHtarget; P.adTarget = h->adTarget; P.adQuant = h->adQuant;
    P.adapt_state = h->d_adapt_state; P.adapt_hist = h->d_adapt_hist;
    P.maxFPiter = h->maxFPiter; P.FPtol = h->FPtol; P.gradThresh = h->gradThresh;
    // once adaptation has run, the adapted per-chain H / delta are the step sizes (WALNUTS.py:137,144)
    P.Hstep = h->d_H; P.delta = h->d_delta; P.state = h->d_state; P.draws = d_draws; P.diag = d_diag;
    P.orbit_min = d_omin; P.orbit_max = d_omax;
    P.nevalF = (unsigned long long*)d_nevalF; P.nevalB = (unsigned long long*)d_nevalB;
    P.totals = h->d_totals; P.scratch = h->d_scratch; P.nslot = nslot; P.queue = h->d_queue; P.order = order; P.order_len = order ? h->d_sched_meta + 1 : nullptr; P.cost = h->d_cost; P.tp = tp;
    void* args[] = {&P};
    if (ut) {
      const int rc = ut->launch(user_family(c), c.device, &P, (unsigned)blocks, h->stream);
      if (rc) return fail(h, WN_ECUDA, "user target plug-in: kernel launch failed (" + std::to_string(rc) + ")");
    } else if (cl > 1) {
      lcfg.gridDim = dim3((unsigned)blocks);
      CUDA_TRY(h, cudaLaunchKernelExC(&lcfg, p.fn, args));
    } else {
      CUDA_TRY(h, cudaLaunchKernel(p.fn, dim3((unsigned)blocks), dim3(p.NT), args, p.smem, h->stream));
    }
  } else {
    PkgParams P;
    memset(&P, 0, sizeof(P));
    P.n_chains = c.n_chains; P.d = c.d; P.dg = c.dg; P.max_depth = c.M; P.compat = c.compat;
    P.n_iter = (int)n_iter; P.iter0 = h->iter_done + 1;
    P.seed_lo = (uint32_t)(c.seed & 0xffffffffu); P.seed_hi = (uint32_t)(c.seed >> 32);
    P.chain_offset = (uint32_t)c.chain_offset;
    P.macro_step = c.H0; P.max_error = c.delta; P.inv_mass = h->d_inv_mass;
    P.state = h->d_state; P.draws = d_draws;
    P.neval = (unsigned long long*)d_nevalF; P.totals = h->d_totals;
    P.scratch = h->d_scratch; P.nslot = nslot; P.queue = h->d_queue; P.order = order; P.order_len = order ? h->d_sched_meta + 1 : nullptr; P.cost = h->d_cost; P.tp = tp;
    void* args[] = {&P};
    if (ut) {
      const int rc = ut->launch(user_family(c), c.device, &P, (unsigned)blocks, h->stream);
      if (rc) return fail(h, WN_ECUDA, "user target plug-in: kernel launch failed (" + std::to_string(rc) + ")");
    } else {
      CUDA_TRY(h, cudaLaunchKernel(p.fn, dim3((unsigned)blocks), dim3(p.NT), args, p.smem, h->stream));
    }
  }
  CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));
  if (h->d_cost) h->have_cost = true;
  h->iter_done += (uint32_t)n_iter;
  h->last_launches = 1;
  h->last_plan[0] = fam; h->last_plan[1] = p.G; h->last_plan[2] = p.E2; h->last_plan[3] = p.NT;
  h->last_slots = nslot;
  return WN_OK;
}

int wn_sync(wn_handle* h) {
  if (!h) return WN_EINVAL;
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  CUDA_TRY(h, cudaEventElapsedTime(&h->last_ms, h->ev0, h->ev1));
  CUDA_TRY(h, cudaMemcpy(h->last_tot, h->d_totals, sizeof(h->last_tot), cudaMemcpyDeviceToHost));
  return WN_OK;
}

int wn_run(wn_handle* h, int64_t n_iter, double* draws, double* diag, uint64_t* nevalF, uint64_t* nevalB,
           int on_device) {
  return wn_run_stats(h, n_iter, draws, diag, nevalF, nevalB, nullptr, nullptr, on_device);
}

// device staging of one output of the host-buffer paths: grow-only, owned by the handle
static int stage(wn_handle* h, double** buf, size_t* cap, size_t n) {
  if (n <= *cap) return WN_OK;
  if (*buf) { cudaFree(*buf); *buf = nullptr; *cap = 0; }
  CUDA_TRY(h, cudaMalloc(buf, n * sizeof(double)));
  *cap = n;
  return WN_OK;
}

static int host_async_impl(wn_handle* h, int64_t n_iter, const double* q_in, double* draws, double* diag,
                           uint64_t* nevalF, uint64_t* nevalB, double* orbit_min, double* orbit_max, double* q_out) {
  if (!h) return WN_EINVAL;
  if ((orbit_min == nullptr) != (orbit_max == nullptr)) return fail(h, WN_EINVAL, "orbit_min and orbit_max go together");
  if (n_iter <= 0 || n_iter > 0x7fffffff) return fail(h, WN_EINVAL, "n_iter must be positive");
  const wn_config& c = h->cfg;
  CUDA_TRY(h, cudaSetDevice(c.device));
  const size_t nd = draws ? (size_t)n_iter * c.n_chains * c.dg : 0;
  const size_t ng = diag ? (size_t)n_iter * c.n_chains * WN_DIAG_COLS : 0;
  const size_t no = orbit_min ? (size_t)n_iter * c.n_chains * c.dg : 0;
  const size_t nc = (size_t)c.n_chains;
  int rc;
  if ((rc = stage(h, &h->o_draws, &h->cap_draws, nd))) return rc;
  if ((rc = stage(h, &h->o_diag, &h->cap_diag, ng))) return rc;
  if ((rc = stage(h, &h->o_lo, &h->cap_lo, no))) return rc;
  if ((rc = stage(h, &h->o_hi, &h->cap_hi, no))) return rc;
  if (nevalF && !h->o_f) CUDA_TRY(h, cudaMalloc(&h->o_f, nc * sizeof(uint64_t)));
  if (nevalB && !h->o_b) CUDA_TRY(h, cudaMalloc(&h->o_b, nc * sizeof(uint64_t)));
  if (q_in) {
    CUDA_TRY(h, cudaMemcpyAsync(h->d_state, q_in, nc * c.d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    h->have_state = true;
  }
  if (nevalB) CUDA_TRY(h, cudaMemsetAsync(h->o_b, 0, nc * sizeof(uint64_t), h->stream));   // package mode leaves it untouched
  rc = run_async_impl(h, n_iter, nd ? h->o_draws : nullptr, ng ? h->o_diag : nullptr, nevalF ? h->o_f : nullptr,
                      nevalB ? h->o_b : nullptr, no ? h->o_lo : nullptr, no ? h->o_hi : nullptr);
  if (rc) return rc;
  if (nd) CUDA_TRY(h, cudaMemcpyAsync(draws, h->o_draws, nd * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (no) {
    CUDA_TRY(h, cudaMemcpyAsync(orbit_min, h->o_lo, no * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(orbit_max, h->o_hi, no * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  }
  if (ng) CUDA_TRY(h, cudaMemcpyAsync(diag, h->o_diag, ng * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  if (nevalF) CUDA_TRY(h, cudaMemcpyAsync(nevalF, h->o_f, nc * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
  if (nevalB) CUDA_TRY(h, cudaMemcpyAsync(nevalB, h->o_b, nc * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
  if (q_out) CUDA_TRY(h, cudaMemcpyAsync(q_out, h->d_state, nc * c.d * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  return WN_OK;
}

int wn_run_host_async(wn_handle* h, int64_t n_iter, const double* q_in, double* draws, double* diag,
                      uint64_t* nevalF, uint64_t* nevalB, double* q_out) {
  return host_async_impl(h, n_iter, q_in, draws, diag, nevalF, nevalB, nullptr, nullptr, q_out);
}

int wn_run_stats(wn_handle* h, int64_t n_iter, double* draws, double* diag, uint64_t* nevalF, uint64_t* nevalB,
                 double* orbit_min, double* orbit_max, int on_device) {
  if (!h) return WN_EINVAL;
  if ((orbit_min == nullptr) != (orbit_max == nullptr)) return fail(h, WN_EINVAL, "orbit_min and orbit_max go together");
  int rc = on_device ? run_async_impl(h, n_iter, draws, diag, nevalF, nevalB, orbit_min, orbit_max)
                     : host_async_impl(h, n_iter, nullptr, draws, diag, nevalF, nevalB, orbit_min, orbit_max, nullptr);
  if (rc) return rc;
  return wn_sync(h);
}

int wn_alloc_pinned(int64_t bytes, void** out) {
  if (!out || bytes <= 0) return WN_EINVAL;
  *out = nullptr;
  return cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable) == cudaSuccess ? WN_OK : WN_ENOMEM;
}
int wn_free_pinned(void* p) { return (!p || cudaFreeHost(p) == cudaSuccess) ? WN_OK : WN_ECUDA; }

int wn_last_kernel_ms(wn_handle* h, float* ms) {
  if (!h || !ms) return WN_EINVAL;
  *ms = h->last_ms;
  return WN_OK;
}
int wn_last_launches(wn_handle* h, int64_t* n) {
  if (!h || !n) return WN_EINVAL;
  *n = h->last_launches;
  return WN_OK;
}
int wn_last_plan(wn_handle* h, int32_t out[4]) {
  if (!h || !out) return WN_EINVAL;
  memcpy(out, h->last_plan, sizeof(h->last_plan));
  return WN_OK;
}
int wn_last_slots(wn_handle* h, int64_t* n) {
  if (!h || !n) return WN_EINVAL;
  *n = h->last_slots;
  return WN_OK;
}
int wn_last_grad_evals(wn_handle* h, uint64_t* forward, uint64_t* backward) {
  if (!h) return WN_EINVAL;
  if (forward) *forward = h->last_tot[0];
  if (backward) *backward = h->last_tot[1];
  return WN_OK;
}

int wn_moments(wn_handle* h, double* mean, double* var) {
  if (!h || !mean || !var) return fail(h, WN_EINVAL, "wn_moments: bad argument");
  if (!h->have_state) return fail(h, WN_ESTATE, "no state set");
  const wn_config& c = h->cfg;
  CUDA_TRY(h, cudaSetDevice(c.device));
  double* buf = nullptr;
  CUDA_TRY(h, cudaMalloc(&buf, 2 * (size_t)c.d * sizeof(double)));
  moments_kernel<<<(c.d + 127) / 128, 128, 0, h->stream>>>(h->d_state, c.n_chains, c.d, buf, buf + c.d);
  cudaError_t e = cudaMemcpyAsync(mean, buf, c.d * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(var, buf + c.d, c.d * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  cudaFree(buf);
  if (e != cudaSuccess) return fail(h, WN_ECUDA, cudaGetErrorString(e));
  return WN_OK;
}

void* wn_stream(wn_handle* h) { return h ? (void*)h->stream : nullptr; }

int wn_fp64_peak(int device, double* flops_per_s) {
  if (!flops_per_s) return WN_EINVAL;
  if (cudaSetDevice(device) != cudaSuccess) return WN_ECUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return WN_ECUDA;
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 16;
  double* out = nullptr;
  if (cudaMalloc(&out, (size_t)blocks * threads * sizeof(double)) != cudaSuccess) return WN_ENOMEM;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  float best = 1e30f;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(a);
    fp64_fma_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-7);
    cudaEventRecord(b);
    if (cudaEventSynchronize(b) != cudaSuccess) { cudaFree(out); return WN_ECUDA; }
    float ms;
    cudaEventElapsedTime(&ms, a, b);
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(out);
  *flops_per_s = 2.0 * 8.0 * (double)iters * blocks * threads / (best * 1e-3);
  return WN_OK;
}

}  // extern "C"
