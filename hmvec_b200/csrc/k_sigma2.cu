// k_sigma2.cu -- K3: sigma^2(R,z) contraction (FP64 tensor cores), K3b: Sheth-Tormen mass function and bias.
// Reference arithmetic: cosmology.py:30-38 (Wkr), :245-269 (get_sigma2_R), hmvec.py:133-185.
#include "common.cuh"
#include "gemm_f64.cuh"

namespace hmv {

// ---- W^2 table: W2T[k'][m] = W(ks[k'] R[m])^2, k' major so the contraction reads it coalesced in m ----
__global__ void w2_table_kernel(int nm, int nks, const double* __restrict__ ks, const double* __restrict__ R,
                                const double* __restrict__ kw, double taylor_switch, double* __restrict__ W2T) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)nm * nks) return;
  const int k = (int)(idx / nm), m = (int)(idx - (long long)k * nm);
  const double x = ks[k] * R[m];
  double w;
  if (x < taylor_switch) {
    const double xx = x * x;
    w = 1.0 - 0.1 * xx + 0.00357142857143 * xx * xx;  // cosmology.py:30-32
  } else {
    double s, c;
    sincos(x, &s, &c);
    w = 3.0 * (s - x * c) / (x * x * x);  // cosmology.py:36
  }
  W2T[idx] = w * w * kw[k];     // the integration weight of k' rides on the table (one multiply here, none in the GEMM)
}

// fallback for odd nks / nm or unaligned inputs: the scalar-load kernel of round 1
constexpr int BM = 32, BN = 64, BK = 16, GT = 256;
#ifndef HMV_SIGMA2_CTAS
#define HMV_SIGMA2_CTAS (16 * 148)
#endif
__global__ void __launch_bounds__(GT) sigma2_gemm_plain_kernel(int nz, int nm, int nks, int kchunk,
                                                               const double* __restrict__ sPzk,
                                                               const double* __restrict__ W2T, double* __restrict__ out,
                                                               long long out_split_stride) {
  __shared__ double As[BK][BM + 1];
  __shared__ double Bs[BK][BN + 8];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int kq = lane & 3, nq = lane >> 2;
  const int wz = (w & 3) * 8, wn = (w >> 2) * 32;
  const int z0 = blockIdx.y * BM, m0 = blockIdx.x * BN;
  const int kbeg = blockIdx.z * kchunk, kend = min(nks, kbeg + kchunk);
  double c[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
  const int az = tid >> 3, ak = (tid & 7) * 2;     // A: 32 z x 16 k, 2 k per thread
  const int bk = tid >> 4, bm = (tid & 15) * 4;    // B: 16 k x 64 m, 4 m per thread
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int z = z0 + az, k = k0 + ak + i;
      As[ak + i][az] = (z < nz && k < kend) ? sPzk[(long long)z * nks + k] : 0.0;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int k = k0 + bk, m = m0 + bm + i;
      Bs[bk][bm + i] = (k < kend && m < nm) ? W2T[(long long)k * nm + m] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      const double a = As[kk + kq][wz + nq];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const double b = Bs[kk + kq][wn + 8 * t + nq];
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                     : "+d"(c[t][0]), "+d"(c[t][1]) : "d"(a), "d"(b));
      }
    }
    __syncthreads();
  }
  double* o = out + (long long)blockIdx.z * out_split_stride;
  const int z = z0 + wz + nq;
  if (z < nz) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int m = m0 + wn + 8 * t + 2 * kq;
      if (m < nm) o[(long long)z * nm + m] = c[t][0];
      if (m + 1 < nm) o[(long long)z * nm + m + 1] = c[t][1];
    }
  }
}

__global__ void splitk_reduce_kernel(long long n, int nsplit, const double* __restrict__ part,
                                     double* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double s = 0.0;
  for (int p = 0; p < nsplit; ++p) s += part[(long long)p * n + i];  // fixed order: deterministic
  out[i] = s;
}

// z rows per CTA of the all-z kernel: the smallest of 32 / 64 / 128 / 208 that covers nz (several z tiles beyond 208)
static int sigma2_mt(int nz) { return nz <= 32 ? 4 : nz <= 64 ? 8 : nz <= 128 ? 16 : 26; }

// split-k factor.  The workspace is sized for the larger of the two plans (all-z kernel / fallback kernel).
static int sigma2_splits(int nz, int nm, int nks, bool allz) {
  long long s;
  if (allz) {
    const int mt = sigma2_mt(nz);
    const long long tiles = (long long)cdiv(nm, SG_BN) * cdiv(nz, 8 * mt);
    const long long slots = 148LL * (mt > 16 ? 1 : 2) * 2;        // at most two full waves of resident CTAs
    s = slots / tiles;
  } else {
    const long long tiles = (long long)cdiv(nm, BN) * cdiv(nz, BM);
    s = (HMV_SIGMA2_CTAS + tiles - 1) / tiles;   // enough resident CTAs per SM to hide the un-pipelined loads
  }
  if (s < 1) s = 1;
  if (s > 32) s = 32;
  const long long maxs = (nks + BK - 1) / BK;
  if (s > maxs) s = maxs;
  return (int)s;
}

// ---- mass function and bias --------------------------------------------------------------------------
// TINKER = false: Sheth-Tormen f(sigma), b(sigma) (hmvec.py:137-141, 152-156).
// TINKER = true:  Tinker et al. 2010 (hmvec.py:142-145, 157-159 -> tinker.py:26-67): multiplicity nu f(nu) with the
//                 per-redshift parameters tk[z] = (alpha, beta, phi, eta, gamma) prepared on the host (alpha from the
//                 normalisation table), bias of eq. 6 for Delta = 200.
template <bool TINKER>
__global__ void mass_function_kernel(int nz, int nm, const double* __restrict__ sigma2,
                                     const double* __restrict__ ms, double rho_m0, double A, double a, double p,
                                     double dc, const double* __restrict__ tk, double* __restrict__ nzm,
                                     double* __restrict__ bh) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)nz * nm) return;
  const int z = (int)(idx / nm), m = (int)(idx - (long long)z * nm);
  const double* s2row = sigma2 + (long long)z * nm;
  const double s2 = s2row[m];
  // d ln(sigma^-1) / d ln M with numpy.gradient's stencil (hmvec.py:181-183)
  const double f0 = -0.5 * log(s2), x0 = log(ms[m]);
  double g;
  if (m == 0) {
    g = (-0.5 * log(s2row[1]) - f0) / (log(ms[1]) - x0);
  } else if (m == nm - 1) {
    g = (f0 + 0.5 * log(s2row[m - 1])) / (x0 - log(ms[m - 1]));
  } else {
    const double fm = -0.5 * log(s2row[m - 1]), fp = -0.5 * log(s2row[m + 1]);
    const double hs = x0 - log(ms[m - 1]), hd = log(ms[m + 1]) - x0;
    const double ca = -hd / (hs * (hd + hs)), cb = (hd - hs) / (hd * hs), cc = hs / (hd * (hd + hs));
    g = ca * fm + cb * f0 + cc * fp;
  }
  const double sig = sqrt(s2);
  double f, b;
  if constexpr (!TINKER) {
    const double nu2a = a * dc * dc / s2;
    // hmvec.py:141
    f = A * sqrt(2.0 * a / M_PI) * (1.0 + pow(s2 / a / (dc * dc), p)) * (dc / sig) * exp(-0.5 * nu2a);
    // hmvec.py:156
    b = 1.0 + (nu2a - 1.0) / dc + (2.0 * p / dc) / (1.0 + pow(nu2a, p));
  } else {
    const double nu = dc / sig;
    const double* t = tk + 5 * z;
    const double al = t[0], be = t[1], ph = t[2], et = t[3], ga = t[4];
    // tinker.py:62 times nu (hmvec.py:145: "f is actually nu*fnu")
    f = nu * al * (1.0 + pow(be * nu, -2.0 * ph)) * pow(nu, 2.0 * et) * exp(-0.5 * ga * nu * nu);
    // tinker.py:28-40 with delta = 200 and tinker's own deltac = 1.686 (its constants dict, not st_deltac)
    const double y = log10(200.0), ey = exp(-pow(4.0 / y, 4.0));
    const double tA = 1.0 + 0.24 * y * ey, ta = 0.44 * y - 0.88, tC = 0.019 + 0.107 * y + 0.19 * ey;
    const double nua = pow(nu, ta);
    b = 1.0 - tA * nua / (nua + pow(1.686, ta)) + 0.183 * pow(nu, 1.5) + tC * pow(nu, 2.4);
  }
  const double M = ms[m];
  nzm[idx] = rho_m0 * f * g / (M * M);
  bh[idx] = b;
}

}  // namespace hmv

using namespace hmv;

extern "C" long long hmv_sigma2_ws_doubles(int nz, int nm, int nks) {
  if (nz <= 0 || nm <= 0 || nks <= 0) return 0;
  const int s0 = sigma2_splits(nz, nm, nks, true), s1 = sigma2_splits(nz, nm, nks, false);
  const int s = s0 > s1 ? s0 : s1;
  return (long long)nks * nm + (long long)s * nz * nm;
}

extern "C" int hmv_sigma2(int nz, int nm, int nks, const double* sPzk_d, const double* kw_d, const double* ks_sig_d,
                          const double* R_d, double taylor_switch, double* w2_ws_d, double* sigma2_d, void* stream) {
  HMV_REQUIRE(nz > 0 && nm > 0 && nks > 0, "hmv_sigma2: sizes must be positive (nz=%d nm=%d nks=%d)", nz, nm, nks);
  HMV_REQUIRE(sPzk_d && kw_d && ks_sig_d && R_d && w2_ws_d && sigma2_d, "hmv_sigma2: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const long long nw = (long long)nm * nks;
  w2_table_kernel<<<cdiv(nw, 256), 256, 0, st>>>(nm, nks, ks_sig_d, R_d, kw_d, taylor_switch, w2_ws_d);
  int rc = check_launch("w2_table_kernel");
  if (rc) return rc;
  const bool allz = (nks & 1) == 0 && (nm & 1) == 0 && (((size_t)sPzk_d | (size_t)w2_ws_d) & 15) == 0;
  const int splits = sigma2_splits(nz, nm, nks, allz);
  int kchunk = cdiv(nks, splits);
  kchunk = cdiv(kchunk, BK) * BK;
  double* part = w2_ws_d + nw;
  const long long n = (long long)nz * nm;
  double* dst = splits == 1 ? sigma2_d : part;
  if (allz) {
    const int mt = sigma2_mt(nz);
    dim3 grid(cdiv(nm, SG_BN), cdiv(nz, 8 * mt), splits);
    const size_t smem = (size_t)(2 * 8 * mt * SG_ALD + 2 * SG_BK * SG_BLD) * sizeof(double);
    cudaError_t e = cudaSuccess;
#define HMV_SG(MTV)                                                                                                  \
    case MTV:                                                                                                        \
      e = cudaFuncSetAttribute(sigma2_gemm_kernel<MTV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);     \
      if (e == cudaSuccess) sigma2_gemm_kernel<MTV><<<grid, SG_T, smem, st>>>(nz, nm, nks, kchunk, sPzk_d, w2_ws_d, dst, n); \
      break;
    switch (mt) { HMV_SG(4) HMV_SG(8) HMV_SG(16) default: HMV_SG(26) }
#undef HMV_SG
    if (e != cudaSuccess) return fail(HMV_E_CUDA, "sigma2_gemm_kernel smem opt-in (%zu B): %s", smem, cudaGetErrorString(e));
    rc = check_launch("sigma2_gemm_kernel");
  } else {
    dim3 grid(cdiv(nm, BN), cdiv(nz, BM), splits);
    sigma2_gemm_plain_kernel<<<grid, GT, 0, st>>>(nz, nm, nks, kchunk, sPzk_d, w2_ws_d, dst, n);
    rc = check_launch("sigma2_gemm_plain_kernel");
  }
  if (rc || splits == 1) return rc;
  splitk_reduce_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, splits, part, sigma2_d);
  return check_launch("splitk_reduce_kernel");
}

extern "C" int hmv_mass_function(int nz, int nm, const double* sigma2_d, const double* ms_d, double rho_m0,
                                 double st_A, double st_a, double st_p, double st_deltac, double* nzm_d, double* bh_d,
                                 void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2, "hmv_mass_function: need nz>0 and nm>=2 (numpy.gradient needs two samples)");
  HMV_REQUIRE(sigma2_d && ms_d && nzm_d && bh_d, "hmv_mass_function: null pointer");
  const long long n = (long long)nz * nm;
  mass_function_kernel<false><<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(nz, nm, sigma2_d, ms_d, rho_m0, st_A, st_a,
                                                                               st_p, st_deltac, nullptr, nzm_d, bh_d);
  return check_launch("mass_function_kernel");
}

extern "C" int hmv_mass_function_tinker(int nz, int nm, const double* sigma2_d, const double* ms_d, double rho_m0,
                                        double deltac, const double* tinker_z_d, double* nzm_d, double* bh_d,
                                        void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2, "hmv_mass_function_tinker: need nz>0 and nm>=2 (numpy.gradient needs two samples)");
  HMV_REQUIRE(sigma2_d && ms_d && tinker_z_d && nzm_d && bh_d, "hmv_mass_function_tinker: null pointer");
  const long long n = (long long)nz * nm;
  mass_function_kernel<true><<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(nz, nm, sigma2_d, ms_d, rho_m0, 0.0, 0.0,
                                                                              0.0, deltac, tinker_z_d, nzm_d, bh_d);
  return check_launch("mass_function_kernel<tinker>");
}
