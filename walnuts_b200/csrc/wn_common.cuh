// Common device helpers: Philox4x32-10 streams, chain-group reductions, scratch addressing.
//
// Layout idea (DESIGN.md section 3): a chain is owned by a group of G threads (G = 1 .. 512 in one CTA, 1024 .. 4096 on
// a thread-block cluster).
// Thread t of the group holds E = 2*E2 coordinates in registers: the pairs p = e2*G + t,
// i.e. coordinates 2p and 2p+1.  All per-chain control state is replicated in the registers of
// the G threads and is bit-identical across them (reductions return identical values to every
// thread), so control flow is uniform within a group and never needs a broadcast.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace wn {

// --------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011); the same integer function as oracle/philox.py.
// key = (seed_lo, seed_hi); counter = (block, iteration, chain, stream).
// --------------------------------------------------------------------------------------
enum : uint32_t {
  STREAM_DIR = 0,   // M direction uniforms            (reference WALNUTS.py:216)
  STREAM_MOM = 1,   // d momentum normals              (WALNUTS.py:236, walnuts.py:325)
  STREAM_SEQ = 2,   // sequential scalar uniforms      (WALNUTS.py:298,395,426,...,613; adaptiveIntegrators.py:392)
  STREAM_INIT = 3,
  STREAM_PKG_DIR = 4,     // walnuts.py:330
  STREAM_PKG_ELL = 5,     // walnuts.py:194
  STREAM_PKG_ACCEPT = 6,  // walnuts.py:346
  STREAM_PKG_SELECT = 7   // walnuts.py:350
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  // ((a >> 5) * 2^26 + (b >> 6)) * 2^-53, exact in fp64
  return __dmul_rn(__dadd_rn(__dmul_rn((double)(a >> 5), 67108864.0), (double)(b >> 6)),
                   1.1102230246251565404e-16);
}

struct RngKey {
  uint32_t k0, k1, chain, iter;
};

__device__ __forceinline__ double rng_uniform(const RngKey& k, uint32_t stream, uint32_t idx) {
  const uint4 w = philox4x32_10(make_uint4(idx >> 1, k.iter, k.chain, stream), k.k0, k.k1);
  return (idx & 1u) ? u53(w.z, w.w) : u53(w.x, w.y);
}

// uniforms 2b and 2b+1 of a stream (one Philox block)
__device__ __forceinline__ void rng_uniform_pair(const RngKey& k, uint32_t stream, uint32_t b, double& u0, double& u1) {
  const uint4 w = philox4x32_10(make_uint4(b, k.iter, k.chain, stream), k.k0, k.k1);
  u0 = u53(w.x, w.y);
  u1 = u53(w.z, w.w);
}

// normal pair p of a stream: z[2p], z[2p+1]  (Box-Muller, same formula as oracle/philox.py)
__device__ __forceinline__ void rng_normal_pair(const RngKey& k, uint32_t stream, uint32_t p,
                                                double& z0, double& z1) {
  const uint4 w = philox4x32_10(make_uint4(p, k.iter, k.chain, stream), k.k0, k.k1);
  const double u1 = u53(w.x, w.y), u2 = u53(w.z, w.w);
  const double r = sqrt(__dmul_rn(-2.0, log(__dadd_rn(1.0, -u1))));
  double s, c;
  sincos(__dmul_rn(6.283185307179586, u2), &s, &c);
  z0 = __dmul_rn(r, c);
  z1 = __dmul_rn(r, s);
}

// --------------------------------------------------------------------------------------
// Thread-block clusters: barrier and distributed shared memory (DSMEM) reads.
// --------------------------------------------------------------------------------------
// Every thread of every CTA of the cluster arrives (release: its earlier shared AND global writes become visible at
// cluster scope) and waits for all of them (acquire).  Not `.aligned`: correctness does not rest on warp convergence.
// SASS (sm_100a, CUDA 12.9): MEMBAR.ALL.GPU + UCGABAR_ARV, then UCGABAR_WAIT + CCTL.IVALL (the release fences at GPU
// scope, the acquire invalidates L1), and ld.shared::cluster below becomes a generic LD.E.64 -- the same as the
// cooperative_groups form (this_cluster().sync(), map_shared_rank), so the explicit PTX saves neither.
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release;\n\tbarrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t dsmem_addr(const void* p, uint32_t rank) {
  uint32_t a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"((uint32_t)__cvta_generic_to_shared(p)), "r"(rank));
  return a;
}
__device__ __forceinline__ double ld_dsmem(const double* p, uint32_t rank) {
  double v;
  asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(dsmem_addr(p, rank)) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t ld_dsmem(const uint32_t* p, uint32_t rank) {
  uint32_t v;
  asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(v) : "r"(dsmem_addr(p, rank)) : "memory");
  return v;
}

// --------------------------------------------------------------------------------------
// Group reductions.  Every thread of the group receives bit-identical results.
// NTB: threads of the group in ONE CTA.  G > NTB: the group spans a cluster of CL = G / NTB CTAs (one chain per
// cluster); each reduction first reduces within the CTA exactly as a one-CTA group does, then folds the CL partials
// through DSMEM in rank order, so every thread of every CTA computes the same sum in the same order.
// --------------------------------------------------------------------------------------
template <int G, int NTB = G>
struct Group {
  static constexpr int CL = (G > NTB) ? G / NTB : 1;
  static constexpr int LANES = (G < 32) ? G : 32;
  static constexpr int WARPS = (((CL > 1) ? NTB : G) + 31) / 32;   // warps of the group in one CTA
  // shared reduction scratch: two halves of WARPS * 8 doubles, and for a cluster group two halves of 8 doubles that
  // the other CTAs read (the CTA's published partials)
  static constexpr int RED_DOUBLES = 2 * WARPS * 8 + ((CL > 1) ? 2 * 8 : 0);

  // Cluster stage (CL > 1): x holds the CTA's NV partials, identical in every thread of the CTA.  Thread 0 publishes
  // them in half `parity` of the CTA's exchange, one cluster barrier, then every thread folds the CL CTAs' partials in
  // rank order.  The caller flips `parity` afterwards.
  // Reuse of a half: reduction n + 2 rewrites the half that reduction n published.  Its writer (thread 0) has passed
  // the cluster barrier of reduction n + 1 by then, and no thread arrives there before it has finished its DSMEM
  // reads of reduction n -- so every read of a half precedes its next write.  (Further cluster barriers in between,
  // e.g. a broadcast or a vote, only add order.)
  template <int NV, class Op>
  __device__ __forceinline__ static void cluster_fold(double (&x)[NV], double* red, int parity, Op op) {
    double* xb = red + 2 * WARPS * 8 + parity * 8;
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < NV; ++k) xb[k] = x[k];
    }
    cluster_sync();
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double s = ld_dsmem(xb + k, 0u);
#pragma unroll
      for (int r = 1; r < CL; ++r) s = op(s, ld_dsmem(xb + k, (uint32_t)r));
      x[k] = s;
    }
  }
  struct Plus {
    __device__ __forceinline__ double operator()(double a, double b) const { return a + b; }
  };
  struct MaxN {
    __device__ __forceinline__ double operator()(double a, double b) const { return maxn2(a, b); }
  };

  __device__ __forceinline__ static unsigned mask() {
    if constexpr (G >= 32) return 0xffffffffu;
    else return ((1u << G) - 1u) << ((threadIdx.x & 31u) & ~(unsigned)(G - 1));
  }

  // red: shared scratch of RED_DOUBLES doubles (G > 32 only: one chain per block, or per cluster when CL > 1 -- then
  // each CTA holds its own scratch, with the cluster exchange after the two CTA halves), two halves used alternately
  // (`parity`).  EVERY reduction, whatever its number of values, takes the half at red + parity * WARPS * 8: with a
  // value-count-dependent offset the half of one reduction overlapped the other half of the previous one, and a warp
  // that had passed the barrier could overwrite partial sums a slower warp was still reading (racecheck, round 2).
  template <int NV>
  __device__ __forceinline__ static void sum(double (&x)[NV], double* red, int& parity) {
    if constexpr (G == 1) {
      return;
    } else {
      const unsigned m = mask();
#pragma unroll
      for (int off = LANES / 2; off >= 1; off >>= 1) {
#pragma unroll
        for (int k = 0; k < NV; ++k) x[k] += __shfl_xor_sync(m, x[k], off);
      }
      if constexpr (G > 32) {
        const int w = threadIdx.x >> 5;
        double* buf = red + parity * (WARPS * 8);
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
          for (int k = 0; k < NV; ++k) buf[w * NV + k] = x[k];
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          double s = buf[k];
#pragma unroll
          for (int ww = 1; ww < WARPS; ++ww) s += buf[ww * NV + k];
          x[k] = s;
        }
        if constexpr (CL > 1) cluster_fold<NV>(x, red, parity, Plus());
        parity ^= 1;
      }
    }
  }

  // Sum of FOUR doubles over a group of whole warps with a transposing butterfly: the first two exchange steps hand
  // every lane ONE of the four values (6 instead of 20 64-bit shuffles and additions); lanes 0..3 of each warp then hold
  // the warp totals, which are combined across warps in a fixed order through shared memory.
  __device__ __forceinline__ static void sum4t(double (&x)[4], double* red, int& parity) {
    static_assert(G >= 32, "sum4t: whole warps per chain");
    const unsigned lane = threadIdx.x & 31u;
    const bool b0 = lane & 1u, b1 = lane & 2u;
    double k0 = b0 ? x[2] : x[0], k1 = b0 ? x[3] : x[1];
    k0 += __shfl_xor_sync(0xffffffffu, b0 ? x[0] : x[2], 1);
    k1 += __shfl_xor_sync(0xffffffffu, b0 ? x[1] : x[3], 1);
    double k = b1 ? k1 : k0;
    k += __shfl_xor_sync(0xffffffffu, b1 ? k0 : k1, 2);
    k += __shfl_xor_sync(0xffffffffu, k, 4);
    k += __shfl_xor_sync(0xffffffffu, k, 8);
    k += __shfl_xor_sync(0xffffffffu, k, 16);
    // lane l < 4 holds value 2 (l & 1) + (l >> 1)
    if constexpr (G > 32) {
      const int w = threadIdx.x >> 5;
      double* buf = red + parity * (WARPS * 8);
      if (lane < 4u) buf[w * 4 + 2 * (lane & 1u) + (lane >> 1)] = k;
      __syncthreads();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        double s = buf[i];
#pragma unroll
        for (int ww = 1; ww < WARPS; ++ww) s += buf[ww * 4 + i];
        x[i] = s;
      }
      if constexpr (CL > 1) cluster_fold<4>(x, red, parity, Plus());
      parity ^= 1;
    } else {
      x[0] = __shfl_sync(0xffffffffu, k, 0);
      x[1] = __shfl_sync(0xffffffffu, k, 2);
      x[2] = __shfl_sync(0xffffffffu, k, 1);
      x[3] = __shfl_sync(0xffffffffu, k, 3);
    }
  }

  // sum of one double plus OR of a small flag word over the group: the flags ride on a warp-wide integer OR
  // (redux.sync, one instruction) and on the second slot of the shared exchange instead of a second shuffle tree
  __device__ __forceinline__ static void sum1_flags(double& x, unsigned& flags, double* red, int& parity) {
    if constexpr (G == 1) {
      return;
    } else {
      const unsigned m = mask();
#pragma unroll
      for (int off = LANES / 2; off >= 1; off >>= 1) x += __shfl_xor_sync(m, x, off);
      flags = __reduce_or_sync(m, flags);
      if constexpr (G > 32) {
        const int w = threadIdx.x >> 5;
        double* buf = red + parity * (WARPS * 8);
        if ((threadIdx.x & 31) == 0) {
          buf[w * 2] = x;
          buf[w * 2 + 1] = __hiloint2double(0, (int)flags);
        }
        __syncthreads();
        double s = buf[0];
        unsigned f = (unsigned)__double2loint(buf[1]);
#pragma unroll
        for (int ww = 1; ww < WARPS; ++ww) {
          s += buf[ww * 2];
          f |= (unsigned)__double2loint(buf[ww * 2 + 1]);
        }
        if constexpr (CL > 1) {   // the flag word rides as the low half of a double (OR-folded, never added)
          double* xb = red + 2 * WARPS * 8 + parity * 8;
          if (threadIdx.x == 0) {
            xb[0] = s;
            xb[1] = __hiloint2double(0, (int)f);
          }
          cluster_sync();
          s = ld_dsmem(xb, 0u);
          f = (unsigned)__double2loint(ld_dsmem(xb + 1, 0u));
#pragma unroll
          for (int r = 1; r < CL; ++r) {
            s += ld_dsmem(xb, (uint32_t)r);
            f |= (unsigned)__double2loint(ld_dsmem(xb + 1, (uint32_t)r));
          }
        }
        x = s;
        flags = f;
        parity ^= 1;
      }
    }
  }

  // NaN-propagating maximum (numpy's np.max) over the group, same protocol as sum()
  __device__ __forceinline__ static double maxn2(double a, double b) { return (b > a || b != b) ? b : a; }
  template <int NV>
  __device__ __forceinline__ static void maxn(double (&x)[NV], double* red, int& parity) {
    if constexpr (G == 1) {
      return;
    } else {
      const unsigned m = mask();
#pragma unroll
      for (int off = LANES / 2; off >= 1; off >>= 1) {
#pragma unroll
        for (int k = 0; k < NV; ++k) x[k] = maxn2(x[k], __shfl_xor_sync(m, x[k], off));
      }
      if constexpr (G > 32) {
        const int w = threadIdx.x >> 5;
        double* buf = red + parity * (WARPS * 8);
        if ((threadIdx.x & 31) == 0) {
#pragma unroll
          for (int k = 0; k < NV; ++k) buf[w * NV + k] = x[k];
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          double s = buf[k];
#pragma unroll
          for (int ww = 1; ww < WARPS; ++ww) s = maxn2(s, buf[ww * NV + k]);
          x[k] = s;
        }
        if constexpr (CL > 1) cluster_fold<NV>(x, red, parity, MaxN());
        parity ^= 1;
      }
    }
  }

  // OR of a predicate over a cluster group (CL > 1): CTA vote, then the CTAs' votes folded like a sum
  __device__ __forceinline__ static bool any_cluster(bool p, double* red, int& parity) {
    static_assert(CL > 1, "any_cluster: a group that spans a cluster");
    double x[1] = {__syncthreads_or(p) ? 1.0 : 0.0};
    cluster_fold<1>(x, red, parity, Plus());
    parity ^= 1;
    return x[0] != 0.0;
  }

  // broadcast a value chosen by thread 0 of the group (used for queue grabs)
  __device__ __forceinline__ static uint32_t bcast0(uint32_t v, uint32_t* sh) {
    if constexpr (G == 1) {
      return v;
    } else if constexpr (G <= 32) {
      return __shfl_sync(mask(), v, (threadIdx.x & 31u) & ~(unsigned)(G - 1));
    } else if constexpr (CL > 1) {
      // thread 0 of rank 0 chose v; every CTA reads it from rank 0's shared memory.  The first barrier orders this
      // write after every read of the previous broadcast -- and, at the first call of the kernel, after every CTA of
      // the cluster has started (no DSMEM access reaches a CTA that is not running).
      cluster_sync();
      if (threadIdx.x == 0 && cluster_rank() == 0u) *sh = v;
      cluster_sync();
      return ld_dsmem(sh, 0u);
    } else {
      __syncthreads();
      if (threadIdx.x == 0) *sh = v;
      __syncthreads();
      return *sh;
    }
  }
};

// --------------------------------------------------------------------------------------
// Bulk asynchronous global -> shared copies (TMA engine, `cp.async.bulk`, SASS UBLKCP) completing on an
// mbarrier; used to stage data tiles that every chain of a CTA reuses.
// --------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WN_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WN_DONE;\n"
      "bra WN_WAIT;\n"
      "WN_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

__device__ __forceinline__ bool finite_d(double x) { return fabs(x) <= 1.7976931348623157e308; }

}  // namespace wn
