// gemm_f64.cuh -- the FP64 tensor-core contraction shared by K3 (sigma^2, k_sigma2.cu) and the 1-halo trispectrum
// (k_trispec.cu).  Included by each translation unit that launches it; every instantiation is local to its unit.
#pragma once
#include "common.cuh"

namespace hmv {

// ---- contraction C[z][m] = sum_k A[z][k] * B[k][m] : FP64 tensor-core GEMM -------------------------------------
// K3 (sigma^2): A = sPzk (the k' weights ride on B = W2T).  The z extent is small (200 on the LARGE grid, 25 per rank
// on eight GPUs), so a CTA takes ALL redshifts of a z tile (8 MT rows, MT <= 26) against a 64-wide strip of masses: the
// 160 MB W^2 table is read once per z tile instead of once per 32 redshifts.  Warp w owns the strip's columns
// 8w..8w+7 for every row: MT accumulator tiles of mma.sync m8n8k4, fed from a cp.async double-buffered pair of
// shared-memory tiles (A as [z][k] rows of 16-byte copies, B as [k][m]).  Split-k across blockIdx.z fills the SMs;
// the partial sums are added in a fixed order.
// AK = true takes A K-major, A[k][z] with an even row stride lda >= nz (the 1-halo trispectrum's panels, k_trispec.cu):
// A is then staged as [k][z] like B.  lda comes last so that the sigma^2 instantiations keep their parameter offsets
// and compile to the same instructions.  blockIdx.z * kchunk is the first k of a CTA and its partial sums go to
// out + blockIdx.z * out_split_stride: with kchunk = the k extent of one batch item that is a batched product.
constexpr int SG_BN = 64, SG_BK = 16, SG_T = 256, SG_ALD = SG_BK + 4, SG_BLD = SG_BN + 8;

__device__ __forceinline__ void cp_async16_sg(void* dst, const void* src, bool pred) {
  const int bytes = pred ? 16 : 0;                        // zero-fill when out of range
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes) : "memory");
}

// shared memory of one instantiation, in doubles
template <int MT, bool AK>
constexpr int sg_smem_doubles() { return 2 * (AK ? SG_BK * (8 * MT + 8) : 8 * MT * SG_ALD) + 2 * SG_BK * SG_BLD; }

template <int MT, bool AK = false>
__global__ void __launch_bounds__(SG_T, MT > 16 ? 1 : 2) sigma2_gemm_kernel(int nz, int nm, int nks, int kchunk,
                                                                            const double* __restrict__ sPzk,
                                                                            const double* __restrict__ W2T,
                                                                            double* __restrict__ out,
                                                                            long long out_split_stride, int lda = 0) {
  constexpr int BM = 8 * MT;
  constexpr int ATILE = AK ? SG_BK * (BM + 8) : BM * SG_ALD;   // one A buffer: [SG_BK][BM+8] or [BM][SG_ALD]
  extern __shared__ __align__(16) double sg_smem[];
  double* As = sg_smem;                                  // [2][ATILE]
  double* Bs = As + 2 * ATILE;                           // [2][SG_BK][SG_BLD]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int kq = lane & 3, nq = lane >> 2;
  const int z0 = blockIdx.y * BM, m0 = blockIdx.x * SG_BN;
  const int kbeg = blockIdx.z * kchunk, kend = min(nks, kbeg + kchunk);
  double c[MT][2];
#pragma unroll
  for (int t = 0; t < MT; ++t) c[t][0] = c[t][1] = 0.0;
  // nks and nm are even and the rows 16-byte aligned (checked on the host): every copy is a whole 16-byte word
  auto load = [&](int k0, int buf) {
    double* Ab = As + buf * ATILE;
    if constexpr (AK) {
      for (int i = tid; i < SG_BK * (BM / 2); i += SG_T) {          // A: 16 k rows x BM/2 words
        const int r = i / (BM / 2), zw = (i - r * (BM / 2)) * 2;
        const int k = k0 + r, z = z0 + zw;
        HMV_DEV_ASSERT(!(k < kend && z < nz) || (k < nks && z + 1 < lda));
        cp_async16_sg(Ab + r * (BM + 8) + zw, sPzk + (long long)min(k, nks - 1) * lda + min(z, lda - 2),
                      k < kend && z < nz);
      }
    } else {
      for (int i = tid; i < BM * (SG_BK / 2); i += SG_T) {          // A: BM rows x 8 words
        const int r = i / (SG_BK / 2), kw2 = (i - r * (SG_BK / 2)) * 2;
        const int z = z0 + r, k = k0 + kw2;
        cp_async16_sg(Ab + r * SG_ALD + kw2, sPzk + (long long)min(z, nz - 1) * nks + min(k, nks - 2), z < nz && k < kend);
      }
    }
    double* Bb = Bs + buf * SG_BK * SG_BLD;
    for (int i = tid; i < SG_BK * (SG_BN / 2); i += SG_T) {         // B: 16 rows x 32 words
      const int r = i / (SG_BN / 2), mw = (i - r * (SG_BN / 2)) * 2;
      const int k = k0 + r, m = m0 + mw;
      cp_async16_sg(Bb + r * SG_BLD + mw, W2T + (long long)min(k, nks - 1) * nm + min(m, nm - 2), k < kend && m < nm);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  int buf = 0;
  load(kbeg, 0);
  for (int k0 = kbeg; k0 < kend; k0 += SG_BK) {
    if (k0 + SG_BK < kend) {
      load(k0 + SG_BK, buf ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const double* Ab = As + buf * ATILE;
    const double* Bb = Bs + buf * SG_BK * SG_BLD;
#pragma unroll
    for (int kk = 0; kk < SG_BK; kk += 4) {
      const double bv = Bb[(kk + kq) * SG_BLD + 8 * w + nq];
#pragma unroll
      for (int t = 0; t < MT; ++t) {
        const double av = AK ? Ab[(kk + kq) * (BM + 8) + 8 * t + nq] : Ab[(8 * t + nq) * SG_ALD + kk + kq];
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(c[t][0]), "+d"(c[t][1]) : "d"(av), "d"(bv));
      }
    }
    __syncthreads();
    buf ^= 1;
  }
  double* o = out + (long long)blockIdx.z * out_split_stride;
  const int m = m0 + 8 * w + 2 * kq;
#pragma unroll
  for (int t = 0; t < MT; ++t) {
    const int z = z0 + 8 * t + nq;
    if (z < nz) {
      if (m < nm) o[(long long)z * nm + m] = c[t][0];
      if (m + 1 < nm) o[(long long)z * nm + m + 1] = c[t][1];
    }
  }
}

}  // namespace hmv
