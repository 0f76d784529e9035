// common.cuh -- shared helpers for the hmvec_b200 CUDA kernels (sm_100a, FP64 throughout).
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <cmath>
#include "../../include/hmvec_b200.h"

namespace hmv {

// thread-local error text returned by hmv_last_error()
char* err_buf();
int fail(int code, const char* fmt, ...);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return HMV_OK;
}

#define HMV_REQUIRE(cond, ...)                          \
  do {                                                  \
    if (!(cond)) return hmv::fail(HMV_E_ARG, __VA_ARGS__); \
  } while (0)

// device-side bounds checks of the debug build (make EXTRA=-DHMV_DEBUG; compute-sanitizer is not available on the pool):
// a failed check prints its location and traps, which the next CUDA call reports as an error
#ifdef HMV_DEBUG
#define HMV_DEV_ASSERT(cond)                                                                         \
  do {                                                                                               \
    if (!(cond)) {                                                                                   \
      printf("HMV_DEV_ASSERT failed: %s  (%s:%d, block %d thread %d)\n", #cond, __FILE__, __LINE__, \
             (int)blockIdx.x, (int)threadIdx.x);                                                     \
      __trap();                                                                                      \
    }                                                                                                \
  } while (0)
#else
#define HMV_DEV_ASSERT(cond) ((void)0)
#endif

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum for blockDim.x <= 1024 (multiple of 32); result valid in every thread.
__device__ __forceinline__ double block_sum(double v, double* smem_warp /* >= 32 doubles */) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem_warp[w] = v;
  __syncthreads();
  double r = (threadIdx.x < nw) ? smem_warp[threadIdx.x] : 0.0;
  if (w == 0) {
    r = warp_sum(r);
    if (lane == 0) smem_warp[0] = r;
  }
  __syncthreads();
  r = smem_warp[0];
  return r;
}

// trapezoid weight of sample i on a (non-uniform) grid x[0..n): trapz(y,x) == sum_i y_i * w_i
__device__ __forceinline__ double trapz_weight(const double* __restrict__ x, int i, int n) {
  if (n < 2) return 0.0;
  const double lo = (i > 0) ? x[i - 1] : x[0];
  const double hi = (i < n - 1) ? x[i + 1] : x[n - 1];
  return 0.5 * (hi - lo);
}

__device__ __forceinline__ int interval(const double* __restrict__ x, int n, double v) {
  // largest i in [0, n-2] with x[i] <= v  (v already clamped to [x[0], x[n-1]])
  int lo = 0, hi = n - 1;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (x[mid] <= v) lo = mid; else hi = mid;
  }
  return lo;
}

// ---- mbarrier / bulk-copy primitives (PTX; SASS: SYNCS.*, UBLKCP) ----------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!ok);
}
// producer-side wait: back off between polls so the spinning lane does not eat the consumers' issue slots
__device__ __forceinline__ void mbar_wait_sleep(unsigned long long* bar, unsigned parity) {
  unsigned ok;
  for (;;) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) break;
    __nanosleep(64);
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- stage ring fed by bulk async copies -------------------------------------------------------------------------
// Dynamic shared memory holds nst stages of stage_doubles, then full[nst] and empty[nst] mbarriers.  One producer lane
// acquires a stage (waits until every consumer warp has released it), announces the bytes it will copy and issues the
// copies on the stage's full barrier; each consumer warp waits on full and releases the stage with one arrive on empty.
// Producer and every consumer walk the stages in the same order; a RingSlot names a stage and the parity of its lap.
struct RingSlot {
  int s = 0;           // stage
  unsigned ph = 0;     // parity of the current lap
};
struct RingStage {
  double* p;
  unsigned long long* full;   // the barrier the stage's copies complete on
};

struct BulkRing {
  double* base;
  unsigned long long *full, *empty;
  int nst, stage_doubles;

  __host__ __device__ static constexpr size_t smem_bytes(int nst, int stage_doubles) {
    return (size_t)nst * stage_doubles * sizeof(double) + 2 * (size_t)nst * sizeof(unsigned long long);
  }
  // carves the ring out of `smem`; thread 0 initialises the barriers, which the block may use after a __syncthreads()
  __device__ __forceinline__ BulkRing(void* smem, int nst_, int stage_doubles_, unsigned consumer_warps)
      : base(reinterpret_cast<double*>(smem)), nst(nst_), stage_doubles(stage_doubles_) {
    full = reinterpret_cast<unsigned long long*>(base + (size_t)nst * stage_doubles);
    empty = full + nst;
    if (threadIdx.x == 0) {
      for (int s = 0; s < nst; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, consumer_warps); }
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
  }
  __device__ __forceinline__ double* stage(const RingSlot& c) const { return base + (size_t)c.s * stage_doubles; }
  // Two ways to the same sequence of slots: slot(it) of the it-th fill, or a cursor stepped by advance().  With a
  // compile-time nst the division is a multiply; which one a kernel uses is a register-allocation choice (ptxas spills).
  __device__ __forceinline__ RingSlot slot(int it) const {
    RingSlot c;
    c.s = it % nst;
    c.ph = (unsigned)(it / nst) & 1u;
    return c;
  }
  __device__ __forceinline__ void advance(RingSlot& c) const {
    if (++c.s == nst) { c.s = 0; c.ph ^= 1u; }
  }
  // producer: the empty barrier of a stage completes its phase ph ^ 1 before the first lap, so that lap passes at once.
  // kSleep backs off between polls (mbar_wait_sleep) where the spinning lane would take the consumers' issue slots.
  template <bool kSleep = false>
  __device__ __forceinline__ RingStage acquire(const RingSlot& c, unsigned bytes) const {
    if (kSleep) mbar_wait_sleep(empty + c.s, c.ph ^ 1u);
    else mbar_wait(empty + c.s, c.ph ^ 1u);
    mbar_expect_tx(full + c.s, bytes);
    return {stage(c), full + c.s};
  }
  // consumer: wait until the stage's copies have landed
  __device__ __forceinline__ const double* wait(const RingSlot& c) const {
    mbar_wait(full + c.s, c.ph);
    return stage(c);
  }
  // consumer warp: done with the stage
  __device__ __forceinline__ void release(const RingSlot& c) const {
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(empty + c.s);
  }
};

}  // namespace hmv
