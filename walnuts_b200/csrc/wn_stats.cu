// Cross-chain convergence statistics on the device, across GPUs: bulk ESS and split-R-hat of the monitored draws
// (Vehtari, Gelman, Simpson, Carpenter, Buerkner 2021 -- the estimator behind arviz.ess, which the reference's
// experiment scripts use: WALNUTSpy_examples/gaussian/mainGaussESS.py:17,50-55) and cross-GPU moments.
//
// Multi-GPU: chains shard across GPUs with no exchange while sampling; the ONE collective is an NCCL all-gather of the
// monitored draws (wn_ess_rhat) or an all-reduce of (n, sum, sum of squares) (wn_moments_all).  NCCL is bound at run
// time with dlopen -- the library has no link-time dependency on it; a process that already loaded libnccl.so.2
// (e.g. through torch) shares that copy.
//
// Pipeline of wn_ess_rhat per coordinate: gather column -> radix sort (cub) -> ranks -> z = Phi^-1((r - 3/8) / (S + 1/4))
// -> split every chain in halves -> per split chain: mean, variance and ALL autocovariances in shared memory -> sums over
// chains in a fixed order -> Geyer's initial monotone sequence on the host (a few thousand numbers).
//
// wn_summary runs the same pipeline per coordinate (its bulk ESS and R-hat are the same bits), then reads the quantiles
// and moments from the sorted column (summary_moments), feeds the raw draws, the two tail indicators and the squared
// deviations through the same split-chain sums, and ranks |x - q50| with a second radix sort.  The second sort rather
// than a merge of the two halves of the sorted column around the median: |x - q50| is rounded, so distinct draws can
// fold to the same value, and ordinal ranks then follow the chain-major position, which the merge does not see; the
// sort gives the ranks the definition asks for in every case.  Nested R-hat: chain moments, one warp per chain, then
// one block over the superchains.  One host synchronisation per coordinate, as in wn_ess_rhat.
#include <dlfcn.h>
#include <nccl.h>   // types and enums only; every function is resolved with dlsym

#include <cmath>
#include <cstring>
#include <cub/cub.cuh>
#include <mutex>
#include <vector>

#include "wn_handle.hpp"

namespace {

struct NcclApi {
  void* dl = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string path;
};
NcclApi g_nccl;
std::mutex g_nccl_mutex;

int nccl_bind(const char* path, std::string* err) {
  std::lock_guard<std::mutex> lock(g_nccl_mutex);
  if (g_nccl.dl) return WN_OK;
  void* dl = nullptr;
  if (path && *path) dl = dlopen(path, RTLD_NOW | RTLD_LOCAL);
  if (!dl) dl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // already in the process (torch's bundled copy)
  if (!dl) dl = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
  if (!dl) dl = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
  if (!dl) {
    if (err) *err = std::string("libnccl.so.2 not found: ") + dlerror();
    return WN_EUNSUPPORTED;
  }
  NcclApi a;
  a.dl = dl;
  a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(dl, "ncclGetUniqueId");
  a.CommInitRank = (decltype(a.CommInitRank))dlsym(dl, "ncclCommInitRank");
  a.CommInitAll = (decltype(a.CommInitAll))dlsym(dl, "ncclCommInitAll");
  a.CommDestroy = (decltype(a.CommDestroy))dlsym(dl, "ncclCommDestroy");
  a.AllGather = (decltype(a.AllGather))dlsym(dl, "ncclAllGather");
  a.AllReduce = (decltype(a.AllReduce))dlsym(dl, "ncclAllReduce");
  a.GetErrorString = (decltype(a.GetErrorString))dlsym(dl, "ncclGetErrorString");
  if (!a.GetUniqueId || !a.CommInitRank || !a.CommInitAll || !a.CommDestroy || !a.AllGather || !a.AllReduce ||
      !a.GetErrorString) {
    if (err) *err = "libnccl.so.2 lacks a required symbol";
    return WN_EUNSUPPORTED;
  }
  g_nccl = a;
  return WN_OK;
}

#define NCCL_TRY(h, expr)                                                                         \
  do {                                                                                            \
    ncclResult_t _r = (expr);                                                                     \
    if (_r != ncclSuccess) return fail(h, WN_ECUDA, std::string(#expr) + ": " + g_nccl.GetErrorString(_r)); \
  } while (0)

// ---- kernels -------------------------------------------------------------------------------------------------------

// column j of draws [W][n_iter][n_chains][dg] -> x[(w * n_chains + c) * n_iter + t]  (chain-major), idx = identity
__global__ void gather_column(const double* __restrict__ draws, int W, int n_iter, int n_chains, int dg, int j,
                              double* __restrict__ x, unsigned* __restrict__ idx) {
  const size_t S = (size_t)W * n_iter * n_chains;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < S; i += (size_t)gridDim.x * blockDim.x) {
    const size_t t = i % n_iter, wc = i / n_iter, c = wc % n_chains, w = wc / n_chains;
    x[i] = draws[(((size_t)w * n_iter + t) * n_chains + c) * dg + j];
    idx[i] = (unsigned)i;
  }
}

// z[idx_sorted[r]] = Phi^-1((r + 1 - 3/8) / (S + 1/4))   (ordinal ranks; ties have probability zero)
__global__ void rank_normalize(const unsigned* __restrict__ idx_sorted, size_t S, double* __restrict__ z) {
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < S; r += (size_t)gridDim.x * blockDim.x)
    z[idx_sorted[r]] = normcdfinv(((double)(r + 1) - 0.375) / ((double)S + 0.25));
}

// One block per split chain: chain c of length n is split into [0, h) and [n - h, n), h = n / 2 (split == 0: the
// whole chain, h = n).  Writes mean, variance (1 / (h - 1)) and the biased autocovariances acov[lag] (1 / h), lag < h.
__global__ void split_chain_stats(const double* __restrict__ z, int n, int h, int split, double* __restrict__ mean,
                                  double* __restrict__ var, double* __restrict__ acov /* [n_split][h] */) {
  extern __shared__ double xs[];
  __shared__ double red[32];
  const int sc = blockIdx.x;
  const int c = split ? (sc >> 1) : sc;
  const int off = (split && (sc & 1)) ? (n - h) : 0;
  const double* src = z + (size_t)c * n + off;
  double s = 0.0;
  for (int i = threadIdx.x; i < h; i += blockDim.x) {
    const double v = src[i];
    xs[i] = v;
    s += v;
  }
  // block sum (fixed order: deterministic)
  for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  double tot = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
  const double m = tot / h;
  __syncthreads();
  for (int i = threadIdx.x; i < h; i += blockDim.x) xs[i] -= m;
  __syncthreads();
  for (int lag = threadIdx.x; lag < h; lag += blockDim.x) {
    double a = 0.0;
    for (int i = 0; i + lag < h; ++i) a = fma(xs[i], xs[i + lag], a);
    acov[(size_t)sc * h + lag] = a / h;
    if (lag == 0) {
      mean[sc] = m;
      var[sc] = a / (h - 1);
    }
  }
}

// out[lag] = sum over split chains of acov[sc][lag] (fixed order); out[h] = sum mean, out[h+1] = sum mean^2, out[h+2] = sum var
__global__ void reduce_chains(const double* __restrict__ acov, const double* __restrict__ mean,
                              const double* __restrict__ var, int n_split, int h, double* __restrict__ out) {
  const int lag = blockIdx.x * blockDim.x + threadIdx.x;
  if (lag < h) {
    double s = 0.0;
    for (int c = 0; c < n_split; ++c) s += acov[(size_t)c * h + lag];
    out[lag] = s;
  } else if (lag == h) {
    double a = 0.0, b = 0.0, v = 0.0;
    for (int c = 0; c < n_split; ++c) { a += mean[c]; b += mean[c] * mean[c]; v += var[c]; }
    out[h] = a; out[h + 1] = b; out[h + 2] = v;
  }
}

// ---- posterior summary (wn_summary) ----

// Sum of one value per thread over the block in a fixed order (shuffle tree per warp, then the warps in order); every
// thread receives the sum.  blockDim.x is a multiple of 32; red holds 32 doubles of shared memory.
__device__ double block_sum(double v, double* red) {
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();   // red may still be read from the previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
  return t;
}

// numpy's default ('linear') quantile p of the sorted xs[0, S): v = (S - 1) p, a = xs[floor v], b = the next draw,
// t = v - floor v, then a + (b - a) t for t < 1/2 and b - (b - a)(1 - t) otherwise, rounded as numpy rounds it (no FMA)
__device__ double quantile_sorted(const double* __restrict__ xs, size_t S, double p) {
  const double v = __dmul_rn((double)(S - 1), p);
  if (v >= (double)(S - 1)) return xs[S - 1];
  const double f = floor(v);
  const size_t i = (size_t)f;
  const double a = xs[i], b = xs[i + 1], t = v - f, d = b - a;
  return t >= 0.5 ? __dsub_rn(b, __dmul_rn(d, 1.0 - t)) : __dadd_rn(a, __dmul_rn(d, t));
}

// Quantiles and central moments of one coordinate from its sorted draws xs[0, S), in a fixed order: the same bits on
// every run and for every rank count, because every rank sorts the same pooled column.  Each block sums the powers
// 1..4 of d = x - q50 over a fixed grid-stride set of draws; the last block to finish adds the partials in block order
// and writes sc = {mean, q05, q50, q95, sum (x - mean)^2, sum (x - mean)^4}.  Centring at the median keeps the power
// sums well conditioned (|mean - median| <= sd).  *done is 0 on entry and is left 0.
__global__ void summary_moments(const double* __restrict__ xs, size_t S, double* __restrict__ part,
                                unsigned* __restrict__ done, double* __restrict__ sc) {
  __shared__ double red[32];
  __shared__ bool last;
  const double q50 = quantile_sorted(xs, S, 0.5);
  double p1 = 0.0, p2 = 0.0, p3 = 0.0, p4 = 0.0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < S; i += (size_t)gridDim.x * blockDim.x) {
    const double d = xs[i] - q50, d2 = d * d;
    p1 += d;
    p2 += d2;
    p3 = fma(d2, d, p3);
    p4 = fma(d2, d2, p4);
  }
  p1 = block_sum(p1, red);
  p2 = block_sum(p2, red);
  p3 = block_sum(p3, red);
  p4 = block_sum(p4, red);
  if (threadIdx.x == 0) {
    double* pb = part + 4 * (size_t)blockIdx.x;
    pb[0] = p1; pb[1] = p2; pb[2] = p3; pb[3] = p4;
    __threadfence();   // the partials are visible to the last block before it counts this one
    last = atomicAdd(done, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  double s1 = 0.0, s2 = 0.0, s3 = 0.0, s4 = 0.0;
  for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
    const double* pb = part + 4 * (size_t)b;
    s1 += __ldcg(pb); s2 += __ldcg(pb + 1); s3 += __ldcg(pb + 2); s4 += __ldcg(pb + 3);
  }
  s1 = block_sum(s1, red);
  s2 = block_sum(s2, red);
  s3 = block_sum(s3, red);
  s4 = block_sum(s4, red);
  if (threadIdx.x == 0) {
    const double n = (double)S, e = s1 / n, e2 = e * e;   // e = mean - q50
    sc[0] = q50 + e;
    sc[1] = quantile_sorted(xs, S, 0.05);
    sc[2] = q50;
    sc[3] = quantile_sorted(xs, S, 0.95);
    sc[4] = s2 - s1 * e;                                        // sum (d - e)^2
    sc[5] = s4 - 4.0 * e * s3 + 6.0 * e2 * s2 - 3.0 * n * e2 * e2;   // sum (d - e)^4
    *done = 0u;
  }
}

// The series of one coordinate whose split-chain statistics the summary needs, element-wise from the chain-major
// column x and sc (summary_moments): kind 0: 1[x <= q05], 1: 1[x <= q95], 2: (x - mean)^2, 3: |x - q50|
__global__ void summary_series(const double* __restrict__ x, size_t S, const double* __restrict__ sc, int kind,
                               double* __restrict__ y) {
  const double mean = sc[0], q05 = sc[1], q50 = sc[2], q95 = sc[3];
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < S; i += (size_t)gridDim.x * blockDim.x) {
    const double v = x[i];
    double r;
    if (kind == 0) r = v <= q05 ? 1.0 : 0.0;
    else if (kind == 1) r = v <= q95 ? 1.0 : 0.0;
    else if (kind == 2) r = (v - mean) * (v - mean);
    else r = fabs(v - q50);
    y[i] = r;
  }
}

// Mean and variance (1 / (n - 1)) of every whole chain of the chain-major column x; one warp per chain, fixed order
__global__ void chain_moments(const double* __restrict__ x, int n, int n_chains, double* __restrict__ mean,
                              double* __restrict__ var) {
  const int c = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (c >= n_chains) return;   // c is uniform over the warp
  const double* v = x + (size_t)c * n;
  double s = 0.0;
  for (int i = lane; i < n; i += 32) s += v[i];
  for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const double m = s / n;
  double q = 0.0;
  for (int i = lane; i < n; i += 32) {
    const double d = v[i] - m;
    q = fma(d, d, q);
  }
  for (int o = 16; o >= 1; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if (lane == 0) {
    mean[c] = m;
    var[c] = q / (n - 1);
  }
}

// Nested R-hat of K superchains of s consecutive chains from the chain moments; one block, fixed order.
// out = sqrt(1 + B / W), B = 1/(K-1) sum_k (xbar_k - xbar)^2, W = 1/K sum_k (Btilde_k + What_k) with
// Btilde_k = 1/(s-1) sum_m (xbar_mk - xbar_k)^2 (0 for s = 1) and What_k = 1/s sum_m var_mk.
__global__ void nested_rhat(const double* __restrict__ mean, const double* __restrict__ var, int K, int s,
                            double* __restrict__ out) {
  __shared__ double red[32];
  auto super_mean = [&](int k) {
    double a = 0.0;
    for (int m = 0; m < s; ++m) a += mean[(size_t)k * s + m];
    return a / s;
  };
  double a = 0.0, w = 0.0;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double mk = super_mean(k);
    double b = 0.0, v = 0.0;
    for (int m = 0; m < s; ++m) {
      const double e = mean[(size_t)k * s + m] - mk;
      b = fma(e, e, b);
      v += var[(size_t)k * s + m];
    }
    a += mk;
    w += (s > 1 ? b / (s - 1) : 0.0) + v / s;
  }
  a = block_sum(a, red);
  w = block_sum(w, red);
  const double xbar = a / K;
  double b = 0.0;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const double e = super_mean(k) - xbar;
    b = fma(e, e, b);
  }
  b = block_sum(b, red);
  if (threadIdx.x == 0) *out = sqrt(1.0 + (b / (K - 1)) / (w / K));
}

// out[j] = sum over chains of state[c][j]  (pass 1)  /  of (state[c][j] - mean[j])^2  (pass 2, mean != null)
__global__ void moment_sums(const double* __restrict__ state, int n_chains, int d, const double* __restrict__ mean,
                            double* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  const double m = mean ? mean[j] : 0.0;
  double s = 0.0;
  for (int c = 0; c < n_chains; ++c) {
    const double x = state[(size_t)c * d + j] - m;
    s = mean ? fma(x, x, s) : s + x;
  }
  out[j] = s;
}

// Geyer's initial positive + monotone sequence on chain-averaged autocorrelations (the arviz / Stan rule);
// acov_sum[lag] = sum over the m chains of the biased lag autocovariance, n = draws per chain
void ess_from_sums(const double* acov_sum, int T, int m, int n, double sum_mean, double sum_mean2, double sum_var,
                   double* ess, double* rhat) {
  const double nan = std::nan("");
  *ess = nan;
  *rhat = nan;
  if (n < 4 || T < 2) return;
  const double mean_var = sum_var / m;
  const double mom = sum_mean / m;
  double var_plus = mean_var * (n - 1.0) / n;
  if (m > 1) var_plus += (sum_mean2 - m * mom * mom) / (m - 1);
  if (!(var_plus > 0)) return;
  auto rho = [&](int t) { return t < T ? 1.0 - (mean_var - acov_sum[t] / m) / var_plus : 0.0; };
  std::vector<double> rh((size_t)n + 2, 0.0);
  double even = 1.0, odd = rho(1);
  rh[0] = even;
  rh[1] = odd;
  int t = 1;
  while (t < n - 3 && (even + odd) > 0.0) {
    even = rho(t + 1);
    odd = rho(t + 2);
    if (even + odd >= 0) { rh[t + 1] = even; rh[t + 2] = odd; }
    t += 2;
  }
  const int max_t = t - 2;
  if (even > 0) rh[max_t + 1] = even;
  t = 1;
  while (t <= max_t - 2) {
    if (rh[t + 1] + rh[t + 2] > rh[t - 1] + rh[t]) {
      rh[t + 1] = (rh[t - 1] + rh[t]) / 2.0;
      rh[t + 2] = rh[t + 1];
    }
    t += 2;
  }
  const double total = (double)m * n;
  double tau = -1.0;
  for (int i = 0; i <= max_t; ++i) tau += 2.0 * rh[i];
  tau += rh[max_t + 1];
  tau = std::fmax(tau, 1.0 / std::log10(total));
  *ess = total / tau;
  *rhat = mean_var > 0 ? std::sqrt(var_plus / mean_var) : nan;
}

// Device buffers of one statistics call, freed when the call returns
struct DevBufs {
  std::vector<void*> ptrs;
  ~DevBufs() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T>
  cudaError_t alloc(T** out, size_t n) {
    *out = nullptr;
    const cudaError_t e = cudaMalloc((void**)out, n * sizeof(T));
    if (e == cudaSuccess) ptrs.push_back(*out);
    return e;
  }
};

#define ST_TRY(expr)                                                                           \
  do {                                                                                         \
    const cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) return fail(h, WN_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e)); \
  } while (0)

// The draws of every rank on this device, [W][n_iter][n_chains][dg]: a copy of host draws, then the one all-gather of
// a multi-GPU run (every rank receives the monitored draws of all chains).
int pooled_draws(wn_handle* h, const double* draws, size_t per_rank, int on_device, DevBufs& bufs,
                 const double** src) {
  cudaStream_t st = h->stream;
  *src = draws;
  if (!on_device) {
    double* d_in = nullptr;
    ST_TRY(bufs.alloc(&d_in, per_rank));
    ST_TRY(cudaMemcpyAsync(d_in, draws, per_rank * sizeof(double), cudaMemcpyHostToDevice, st));
    *src = d_in;
  }
  if (h->comm) {
    double* d_all = nullptr;
    ST_TRY(bufs.alloc(&d_all, per_rank * h->comm_size));
    const ncclResult_t r = g_nccl.AllGather(*src, d_all, per_rank, ncclDouble, (ncclComm_t)h->comm, st);
    if (r != ncclSuccess) return fail(h, WN_ECUDA, std::string("ncclAllGather: ") + g_nccl.GetErrorString(r));
    *src = d_all;
  }
  return WN_OK;
}

// The per-coordinate pipeline of wn_ess_rhat, which wn_summary runs too (so that its bulk ESS and R-hat are the same
// bits): gather a column of the pooled draws, sort it, rank-normalise, split-chain sums.
struct ColumnWork {
  int W, n, n_chains, dg, hlen, split, n_split, nb;
  size_t S;
  cudaStream_t st;
  double *x, *xs, *z, *mean, *var, *acov;
  unsigned *idx, *idxs;
  char* tmp = nullptr;
  size_t tmp_bytes = 0;

  ColumnWork(int W_, int n_, int n_chains_, int dg_, int split_, cudaStream_t st_)
      : W(W_), n(n_), n_chains(n_chains_), dg(dg_), hlen(split_ ? n_ / 2 : n_), split(split_ ? 1 : 0),
        n_split(W_ * n_chains_ * (split_ ? 2 : 1)), S((size_t)W_ * n_ * n_chains_), st(st_) {
    nb = (int)((S + 255) / 256 < 4096 ? (S + 255) / 256 : 4096);
  }
  cudaError_t alloc(DevBufs& b) {
    cudaError_t e;
    if ((e = b.alloc(&x, S)) || (e = b.alloc(&xs, S)) || (e = b.alloc(&z, S)) || (e = b.alloc(&idx, S)) ||
        (e = b.alloc(&idxs, S)) || (e = b.alloc(&mean, n_split)) || (e = b.alloc(&var, n_split)) ||
        (e = b.alloc(&acov, (size_t)n_split * hlen)))
      return e;
    if ((e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, x, xs, idx, idxs, (int)S, 0, 64, st))) return e;
    if ((e = b.alloc(&tmp, tmp_bytes))) return e;
    return cudaFuncSetAttribute(split_chain_stats, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(hlen * sizeof(double)));
  }
  // column j of the pooled draws -> x (chain-major), idx = identity
  void gather(const double* src, int j) { gather_column<<<nb, 256, 0, st>>>(src, W, n, n_chains, dg, j, x, idx); }
  // keys (chain-major) sorted with idx into xs / idxs; z = the rank-normalised keys, chain-major.  idx stays identity.
  cudaError_t sort_rank(const double* keys) {
    const cudaError_t e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, xs, idx, idxs, (int)S, 0, 64, st);
    if (e) return e;
    rank_normalize<<<nb, 256, 0, st>>>(idxs, S, z);
    return cudaSuccess;
  }
  // split-chain sums of y (chain-major) into out[0, hlen + 3), as ess_from_sums takes them
  void chain_sums(const double* y, double* out) {
    split_chain_stats<<<n_split, 256, hlen * sizeof(double), st>>>(y, n, hlen, split, mean, var, acov);
    reduce_chains<<<(hlen + 1 + 255) / 256, 256, 0, st>>>(acov, mean, var, n_split, hlen, out);
  }
  void ess_rhat(const double* o, double* ess, double* rhat) const {
    ess_from_sums(o, hlen, n_split, hlen, o[hlen], o[hlen + 1], o[hlen + 2], ess, rhat);
  }
};

}  // namespace

extern "C" {

int wn_comm_load(const char* libnccl_path) { return nccl_bind(libnccl_path, nullptr); }

int wn_comm_unique_id(void* id128) {
  if (!id128) return WN_EINVAL;
  int rc = nccl_bind(nullptr, nullptr);
  if (rc) return rc;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return WN_ECUDA;
  memcpy(id128, &id, sizeof(id));
  return WN_OK;
}

int wn_comm_init_rank(wn_handle* h, int nranks, int rank, const void* id128) {
  if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return fail(h, WN_EINVAL, "wn_comm_init_rank: bad argument");
  if (h->comm) return fail(h, WN_ESTATE, "the handle already has a communicator");
  int rc = nccl_bind(nullptr, &h->err);
  if (rc) return rc;
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  NCCL_TRY(h, g_nccl.CommInitRank(&comm, nranks, id, rank));
  h->comm = comm;
  h->comm_rank = rank;
  h->comm_size = nranks;
  return WN_OK;
}

int wn_comm_init_all(wn_handle** hs, int n) {
  if (!hs || n < 1) return WN_EINVAL;
  for (int i = 0; i < n; ++i)
    if (!hs[i] || hs[i]->comm) return fail(hs[i], WN_ESTATE, "wn_comm_init_all: null handle or communicator already set");
  int rc = nccl_bind(nullptr, &hs[0]->err);
  if (rc) return rc;
  std::vector<int> devs(n);
  for (int i = 0; i < n; ++i) devs[i] = hs[i]->cfg.device;
  std::vector<ncclComm_t> comms(n, nullptr);
  NCCL_TRY(hs[0], g_nccl.CommInitAll(comms.data(), n, devs.data()));
  for (int i = 0; i < n; ++i) {
    hs[i]->comm = comms[i];
    hs[i]->comm_rank = i;
    hs[i]->comm_size = n;
  }
  return WN_OK;
}

int wn_comm_destroy(wn_handle* h) {
  if (!h) return WN_EINVAL;
  if (h->comm) {
    cudaSetDevice(h->cfg.device);
    g_nccl.CommDestroy((ncclComm_t)h->comm);
    h->comm = nullptr;
    h->comm_size = 1;
    h->comm_rank = 0;
  }
  return WN_OK;
}

int wn_ess_rhat(wn_handle* h, const double* draws, int64_t n_iter, int64_t n_chains, int32_t dg, int on_device,
                int32_t split, double* ess, double* rhat) {
  if (!h || !draws || !ess || !rhat || n_iter < 4 || n_chains < 1 || dg < 1)
    return fail(h, WN_EINVAL, "wn_ess_rhat: need draws [n_iter >= 4, n_chains, dg] and ess / rhat [dg]");
  const int W = h->comm ? h->comm_size : 1;
  const int n = (int)n_iter;
  const int hlen = split ? n / 2 : n;
  if ((size_t)hlen * sizeof(double) > 200 * 1024) return fail(h, WN_EUNSUPPORTED, "wn_ess_rhat: more than 25 600 draws per (split) chain");
  const size_t per_rank = (size_t)n_iter * n_chains * dg;
  const size_t S = (size_t)W * n_iter * n_chains;
  if (S > 0x7ffffff0ull) return fail(h, WN_EUNSUPPORTED, "wn_ess_rhat: more than 2^31 draws per coordinate");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  DevBufs bufs;
  const double* src = nullptr;
  int rc = pooled_draws(h, draws, per_rank, on_device, bufs, &src);
  if (rc) return rc;
  ColumnWork cw(W, n, (int)n_chains, dg, split, st);
  double* d_out = nullptr;
  ST_TRY(cw.alloc(bufs));
  ST_TRY(bufs.alloc(&d_out, (size_t)hlen + 3));
  std::vector<double> out((size_t)hlen + 3);
  for (int j = 0; j < dg; ++j) {
    cw.gather(src, j);
    ST_TRY(cw.sort_rank(cw.x));
    cw.chain_sums(cw.z, d_out);
    ST_TRY(cudaMemcpyAsync(out.data(), d_out, ((size_t)hlen + 3) * sizeof(double), cudaMemcpyDeviceToHost, st));
    ST_TRY(cudaStreamSynchronize(st));
    cw.ess_rhat(out.data(), &ess[j], &rhat[j]);
  }
  return WN_OK;
}

int wn_summary(wn_handle* h, const double* draws, int64_t n_iter, int64_t n_chains, int32_t dg, int on_device,
               int32_t superchain_size, double* out) {
  if (!h || !draws || !out || n_iter < 4 || n_chains < 1 || dg < 1 || superchain_size < 0)
    return fail(h, WN_EINVAL, "wn_summary: need draws [n_iter >= 4, n_chains, dg], out [dg][WN_SUMMARY_COLS] and "
                              "superchain_size >= 0");
  const int W = h->comm ? h->comm_size : 1;
  const int n = (int)n_iter;
  const int hlen = n / 2;
  if ((size_t)hlen * sizeof(double) > 200 * 1024) return fail(h, WN_EUNSUPPORTED, "wn_summary: more than 25 600 draws per split chain");
  const size_t per_rank = (size_t)n_iter * n_chains * dg;
  const size_t S = (size_t)W * n_iter * n_chains;
  if (S > 0x7ffffff0ull) return fail(h, WN_EUNSUPPORTED, "wn_summary: more than 2^31 draws per coordinate");
  const int M = W * (int)n_chains;   // chains over all ranks
  const int s = superchain_size;
  if (s > 0 && (M % s != 0 || M / s < 2))
    return fail(h, WN_EINVAL, "wn_summary: the chains of all ranks must form at least 2 superchains of superchain_size");
  CUDA_TRY(h, cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->stream;
  DevBufs bufs;
  const double* src = nullptr;
  int rc = pooled_draws(h, draws, per_rank, on_device, bufs, &src);
  if (rc) return rc;
  ColumnWork cw(W, n, (int)n_chains, dg, 1, st);
  ST_TRY(cw.alloc(bufs));
  // split-chain sums of six series: the ranks (bulk), x, 1[x <= q05], 1[x <= q95], (x - mean)^2 and the ranks of
  // |x - q50|; then summary_moments' sc[6] and the nested R-hat
  enum { BULK, RAW, I05, I95, SQ, FOLD, NSER };
  const size_t L = (size_t)hlen + 3, n_out = NSER * L + 7;
  double *d_out = nullptr, *d_y = nullptr, *d_part = nullptr;
  unsigned* d_done = nullptr;
  ST_TRY(bufs.alloc(&d_out, n_out));
  ST_TRY(bufs.alloc(&d_y, S));
  ST_TRY(bufs.alloc(&d_part, 4 * (size_t)cw.nb));
  ST_TRY(bufs.alloc(&d_done, 1));
  ST_TRY(cudaMemsetAsync(d_done, 0, sizeof(unsigned), st));
  double* d_sc = d_out + NSER * L;
  std::vector<double> o(n_out);
  const double nan = std::nan("");
  for (int j = 0; j < dg; ++j) {
    cw.gather(src, j);
    ST_TRY(cw.sort_rank(cw.x));
    cw.chain_sums(cw.z, d_out + BULK * L);
    summary_moments<<<cw.nb, 256, 0, st>>>(cw.xs, S, d_part, d_done, d_sc);
    cw.chain_sums(cw.x, d_out + RAW * L);
    for (int k = 0; k < 3; ++k) {
      summary_series<<<cw.nb, 256, 0, st>>>(cw.x, S, d_sc, k, d_y);
      cw.chain_sums(d_y, d_out + (I05 + k) * L);
    }
    summary_series<<<cw.nb, 256, 0, st>>>(cw.x, S, d_sc, 3, d_y);
    ST_TRY(cw.sort_rank(d_y));   // overwrites the sorted column, which summary_moments has read
    cw.chain_sums(cw.z, d_out + FOLD * L);
    if (s > 0) {
      chain_moments<<<(M + 7) / 8, 256, 0, st>>>(cw.x, n, M, cw.mean, cw.var);
      nested_rhat<<<1, 256, 0, st>>>(cw.mean, cw.var, M / s, s, d_sc + 6);
    }
    ST_TRY(cudaMemcpyAsync(o.data(), d_out, n_out * sizeof(double), cudaMemcpyDeviceToHost, st));
    ST_TRY(cudaStreamSynchronize(st));
    double ess[NSER], rhat[NSER];
    for (int k = 0; k < NSER; ++k) cw.ess_rhat(o.data() + k * L, &ess[k], &rhat[k]);
    const double* sc = o.data() + NSER * L;
    const double Sd = (double)S, sd = std::sqrt(sc[4] / (Sd - 1.0)), E = sc[4] / Sd;
    double* r = out + (size_t)j * WN_SUMMARY_COLS;
    r[WN_S_MEAN] = sc[0];
    r[WN_S_SD] = sd;
    r[WN_S_Q05] = sc[1];
    r[WN_S_Q50] = sc[2];
    r[WN_S_Q95] = sc[3];
    r[WN_S_MCSE_MEAN] = sd / std::sqrt(ess[RAW]);
    r[WN_S_MCSE_SD] = std::sqrt((sc[5] / Sd - E * E) / ess[SQ] / (4.0 * E));
    r[WN_S_ESS_BULK] = ess[BULK];
    r[WN_S_ESS_TAIL] = std::isnan(ess[I05]) || std::isnan(ess[I95]) ? nan : std::fmin(ess[I05], ess[I95]);
    r[WN_S_RHAT] = std::isnan(rhat[BULK]) || std::isnan(rhat[FOLD]) ? nan : std::fmax(rhat[BULK], rhat[FOLD]);
    r[WN_S_NESTED_RHAT] = s > 0 ? sc[6] : nan;
  }
  return WN_OK;
}
#undef ST_TRY

int wn_moments_all(wn_handle* h, double* mean, double* var) {
  if (!h || !mean || !var) return fail(h, WN_EINVAL, "wn_moments_all: bad argument");
  if (!h->have_state) return fail(h, WN_ESTATE, "no state set");
  const wn_config& c = h->cfg;
  CUDA_TRY(h, cudaSetDevice(c.device));
  const int d = c.d;
  double* buf = nullptr;   // [d + 1] sums (+ chain count) | [d] means
  CUDA_TRY(h, cudaMalloc(&buf, (2 * (size_t)d + 1) * sizeof(double)));
  std::vector<double> host((size_t)d + 1);
  auto bail = [&](const std::string& msg) {
    cudaFree(buf);
    return fail(h, WN_ECUDA, msg);
  };
  // two passes (sum -> mean, then centred sum of squares), each followed by ONE all-reduce when a communicator is set
  for (int pass = 0; pass < 2; ++pass) {
    moment_sums<<<(d + 127) / 128, 128, 0, h->stream>>>(h->d_state, c.n_chains, d, pass ? buf + d + 1 : nullptr, buf);
    const double nloc = (double)c.n_chains;
    cudaError_t e = cudaMemcpyAsync(buf + d, &nloc, sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);      // nloc is a stack variable
    if (e != cudaSuccess) return bail(cudaGetErrorString(e));
    if (h->comm) {
      ncclResult_t r = g_nccl.AllReduce(buf, buf, (size_t)d + 1, ncclDouble, ncclSum, (ncclComm_t)h->comm, h->stream);
      if (r != ncclSuccess) return bail(std::string("ncclAllReduce: ") + g_nccl.GetErrorString(r));
    }
    e = cudaMemcpyAsync(host.data(), buf, host.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) return bail(cudaGetErrorString(e));
    const double n = host[d];
    if (pass == 0) {
      for (int j = 0; j < d; ++j) mean[j] = host[j] / n;
      e = cudaMemcpyAsync(buf + d + 1, mean, (size_t)d * sizeof(double), cudaMemcpyHostToDevice, h->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
      if (e != cudaSuccess) return bail(cudaGetErrorString(e));
    } else {
      for (int j = 0; j < d; ++j) var[j] = n > 1 ? host[j] / (n - 1) : 0.0;
    }
  }
  cudaFree(buf);
  return WN_OK;
}

}  // extern "C"
