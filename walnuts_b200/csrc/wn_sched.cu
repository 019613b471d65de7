// Chain scheduling across calls, for kernels whose chains SHARE a warp (G < 32 threads per chain: funnel, small user
// targets): longest chains first, the very longest alone in their warp.
//
// The persistent kernels hand chains to thread groups from a global queue; a call ends when the LAST chain ends.  The cost
// of a transition varies by orders of magnitude between chains (funnel neck: up to 2^10 micro-steps per macro step and
// 2^12 leaves, reference WALNUTSpy_examples/funnel/mainFunnel.py:24-32).  Measured at BASELINE config 3 (funnel10,
// R2P, 10 transitions per call): 147 / 258 / 743 ms at 65 536 / 262 144 / 1 048 576 chains, i.e. 0.62 ms per 1000 chains
// plus ~95 ms that do not depend on the chain count -- the slowest chains, whose ten transitions are one sequential
// dependence chain of ~10^6 micro-steps, and which advance at a fraction of a warp's speed while the W - 1 other chains
// of their warp (W = 32 / G) diverge from them.
//
// Successive calls on one handle continue the same chains, and a chain that was slow in the previous call (still in the
// neck) is very likely slow in the next one.  Every kernel records the gradient evaluations of each chain (`cost`); the
// next call builds its queue from the descending list of those counts:
//   1. the K chains whose cost exceeds half the per-slot share (total cost / resident chain slots) -- the ones that would
//      outlast the balanced part of the call -- get a warp to themselves: W queue entries (chain, retire, ..., retire).  The
//      lanes of a warp take W consecutive entries at launch (the queue's atomicAdd is warp-aggregated in lane order), so
//      the other W - 1 groups of that warp retire at once and the chain runs undiluted.  K <= 1/16 of the resident warps.
//   2. the rest is dealt out in W columns: entry k W + j is the k-th longest chain of the j-th W-quantile, so every warp
//      starts with one chain of each cost class (the plain descending order would put the W slowest chains into ONE warp,
//      where they run one after the other: measured 1.5x slower than the natural order).
//
// The queue is a scheduling hint only: every chain appears in it exactly once, its random numbers are keyed by (seed,
// chain id, iteration) and its state is its own, so the draws are bit-identical with and without it
// (tests/test_gpu_stats.py).  The sort (cub radix sort of n_chains 32-bit keys) and the two small kernels run on the
// handle's stream inside the timed region of the call (~40 us at 262 144 chains).
#include <cub/cub.cuh>

#include "wn_handle.hpp"

namespace {
constexpr unsigned int RETIRE = 0xffffffffu;

__global__ void iota_kernel(unsigned int* x, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = (unsigned int)i;
}

// meta[0] = K: number of chains with cost > total / (2 nslot), at most kmax;  meta[1] = queue length n + K (W - 1)
__global__ void plan_kernel(const unsigned int* cost_desc, int n, int nslot, int W, int kmax, unsigned int* meta) {
  __shared__ unsigned long long part[32];
  unsigned long long s = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += cost_desc[i];
  for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += part[w];
    const unsigned long long thr = tot / (2ull * (unsigned long long)nslot);
    int lo = 0, hi = n;                    // first index whose cost is <= thr (the list is descending)
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if ((unsigned long long)cost_desc[mid] > thr) lo = mid + 1; else hi = mid;
    }
    const int K = min(lo, kmax);
    meta[0] = (unsigned int)K;
    meta[1] = (unsigned int)(n + K * (W - 1));
  }
}

// rank r of the descending list -> queue entry
__global__ void deal_kernel(const unsigned int* sorted, unsigned int* order, int n, int W, const unsigned int* meta) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const int K = (int)meta[0];
  if (r < K) {
    order[r * W] = sorted[r];
    for (int j = 1; j < W; ++j) order[r * W + j] = RETIRE;
    return;
  }
  // column rr / m, row rr % m of an [m, W] table; the lightest chains beyond m W keep their place at the end
  const int rr = r - K, nn = n - K, m = nn / W;
  const int p = (rr < m * W) ? (rr % m) * W + rr / m : rr;
  order[K * W + p] = sorted[r];
}
}  // namespace

int wn_sched_prepare(wn_handle* h, int nslot, int chains_per_warp, const unsigned int** order) {
  *order = nullptr;
  const int n = h->cfg.n_chains;
  const int W = chains_per_warp < 1 ? 1 : chains_per_warp;
  // every chain has its own slot from the start: the order cannot matter; and a call of a few milliseconds is not
  // worth the sort (the previous call's duration is known after wn_sync)
  if (n <= nslot || (h->last_ms > 0.f && h->last_ms < 5.f)) return WN_OK;
  const int kmax = (W > 1) ? (nslot / W) / 16 : 0;
  if (!h->d_cost) {
    CUDA_TRY(h, cudaMalloc(&h->d_cost, (size_t)n * sizeof(unsigned int)));
    CUDA_TRY(h, cudaMalloc(&h->d_cost_sorted, (size_t)n * sizeof(unsigned int)));
    CUDA_TRY(h, cudaMalloc(&h->d_iota, (size_t)n * sizeof(unsigned int)));
    // K W <= nslot / 16 < n / 16 entries of exclusive warps on top of the n chains, whatever kernel the later calls use
    CUDA_TRY(h, cudaMalloc(&h->d_order, ((size_t)n + (size_t)n / 16 + 32) * sizeof(unsigned int)));
    CUDA_TRY(h, cudaMalloc(&h->d_order_sorted, (size_t)n * sizeof(unsigned int)));
    CUDA_TRY(h, cudaMalloc(&h->d_sched_meta, 2 * sizeof(unsigned int)));
    iota_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_iota, n);
    CUDA_TRY(h, cudaGetLastError());
    size_t bytes = 0;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, h->d_cost, h->d_cost_sorted, h->d_iota,
                                                          h->d_order_sorted, n, 0, 32, h->stream));
    CUDA_TRY(h, cudaMalloc(&h->d_sort_tmp, bytes));
    h->sort_tmp_bytes = bytes;
    h->have_cost = false;
  }
  if (!h->have_cost) return WN_OK;   // first call: queue order = chain order; the kernel records the costs
  size_t bytes = h->sort_tmp_bytes;
  CUDA_TRY(h, cub::DeviceRadixSort::SortPairsDescending(h->d_sort_tmp, bytes, h->d_cost, h->d_cost_sorted, h->d_iota,
                                                        h->d_order_sorted, n, 0, 32, h->stream));
  plan_kernel<<<1, 1024, 0, h->stream>>>(h->d_cost_sorted, n, nslot, W, kmax, h->d_sched_meta);
  deal_kernel<<<(n + 255) / 256, 256, 0, h->stream>>>(h->d_order_sorted, h->d_order, n, W, h->d_sched_meta);
  CUDA_TRY(h, cudaGetLastError());
  *order = h->d_order;
  return WN_OK;
}

void wn_sched_free(wn_handle* h) {
  cudaFree(h->d_cost); cudaFree(h->d_cost_sorted); cudaFree(h->d_iota); cudaFree(h->d_order); cudaFree(h->d_order_sorted);
  cudaFree(h->d_sort_tmp); cudaFree(h->d_sched_meta);
  h->d_cost = h->d_cost_sorted = h->d_iota = h->d_order = h->d_order_sorted = h->d_sched_meta = nullptr;
  h->d_sort_tmp = nullptr;
  h->have_cost = false;
}
