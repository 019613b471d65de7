// Private to the library: the handle behind the C-ABI (include/walnuts_cuda.h), shared by capi.cu and wn_stats.cu.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/walnuts_cuda.h"

struct wn_handle {
  wn_config cfg;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double* d_state = nullptr;
  bool have_state = false;
  double2* d_scratch = nullptr;
  size_t scratch_bytes = 0;
  unsigned int* d_queue = nullptr;
  unsigned long long* d_totals = nullptr;
  double* d_p0 = nullptr;  // inv_var | X | y(T)
  double* d_p1 = nullptr;  // y(N)
  double* d_p2 = nullptr;  // X^T (logreg)
  double* d_inv_mass = nullptr;
  double* d_H = nullptr;
  double* d_delta = nullptr;
  double* d_adapt_state = nullptr;   // warm-up adaptation (wn_set_adapt)
  double* d_adapt_hist = nullptr;
  int warmup_iter = 0, adaptH = 0, adaptDelta = 0;
  bool adapt_exported = false;
  double adHtarget = 0.8, adTarget = 0.6, adQuant = 0.9;
  int maxFPiter = 30;                       // integratorAuxPar defaults, adaptiveIntegrators.py:37
  double FPtol = 1.0e-8, gradThresh = 5.0;
  int64_t n_p0 = 0, n_p1 = 0;
  double tau = 1.0;
  double inv_var_max = 1.0, inv_var_min = 1.0;
  uint32_t iter_done = 0, iter_base = 0;   // iter_base: iter_done at creation (cfg.first_iteration - 1)
  float last_ms = 0.f;
  int64_t last_launches = 0;
  int32_t last_plan[4] = {-1, 0, 0, 0};   // {WN_FAMILY_*, G, E2, NT} of the last launch (wn_last_plan)
  int64_t last_slots = 0;                  // chain slots of the last launch (wn_last_slots)
  unsigned long long last_tot[2] = {0, 0};
  int num_sms = 148;
  // grow-only device staging of the host-buffer paths (wn_run / wn_run_stats / wn_run_host_async)
  double *o_draws = nullptr, *o_diag = nullptr, *o_lo = nullptr, *o_hi = nullptr;
  uint64_t *o_f = nullptr, *o_b = nullptr;
  size_t cap_draws = 0, cap_diag = 0, cap_lo = 0, cap_hi = 0;
  // chain scheduling (wn_sched.cu): evaluations of every chain in the previous call -> launch order of the next one
  unsigned int *d_cost = nullptr, *d_cost_sorted = nullptr, *d_iota = nullptr, *d_order = nullptr, *d_order_sorted = nullptr;
  unsigned int* d_sched_meta = nullptr;   // [2]: exclusive warps K, queue length
  void* d_sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;
  bool have_cost = false;
  // cross-GPU statistics (wn_stats.cu): NCCL communicator of this handle's rank, or null
  void* comm = nullptr;
  int comm_rank = 0, comm_size = 1;
  std::string err;
};

static inline int fail(wn_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg;
  return code;
}
// wn_sched.cu: (re)builds h->d_order from h->d_cost on h->stream; *order = the queue order for this launch or null
int wn_sched_prepare(wn_handle* h, int nslot, int chains_per_warp, const unsigned int** order);
void wn_sched_free(wn_handle* h);

#define CUDA_TRY(h, expr)                                                                \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      return fail(h, WN_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));      \
  } while (0)

