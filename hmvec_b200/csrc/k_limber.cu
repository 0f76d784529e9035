// k_limber.cu -- K6: Limber projection (reference cosmology.py:867-904).
// One warp per multipole: lanes stride over the window redshifts, each doing a clamped bilinear lookup of P(k,z)
// at k = (l + 1/2)/chi (the FITPACK kx=ky=1 evaluation the reference obtains through interp2d + bispeu), then
// a trapezoid in z reduced with warp shuffles.
#include "common.cuh"

namespace hmv {

__device__ __forceinline__ void limber_warp(int nl, const double* __restrict__ ells, int nzp, int nk, int ldp,
                                            const double* __restrict__ zs, const double* __restrict__ ks,
                                            const double* __restrict__ P, const double* __restrict__ P2, int ngz,
                                            const double* __restrict__ gzs,
                                            const double* __restrict__ pref, const double* __restrict__ chis,
                                            double* __restrict__ cl) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= nl) return;
  const double ell = ells[warp];
  double acc = 0.0;
  for (int g = lane; g < ngz; g += 32) {
    double kq = (ell + 0.5) / chis[g];                          // cosmology.py:895
    kq = fmin(fmax(kq, ks[0]), ks[nk - 1]);
    const int ik = interval(ks, nk, kq);
    const double tk = (kq - ks[ik]) / (ks[ik + 1] - ks[ik]);
    double val;
    if (nzp > 1) {
      const double zq = fmin(fmax(gzs[g], zs[0]), zs[nzp - 1]);
      const int iz = interval(zs, nzp, zq);
      const double tz = (zq - zs[iz]) / (zs[iz + 1] - zs[iz]);
      const long long o0 = (long long)iz * ldp + ik, o1 = o0 + ldp;
      double a0 = P[o0], a1 = P[o0 + 1], b0 = P[o1], b1 = P[o1 + 1];
      if (P2) { a0 += P2[o0]; a1 += P2[o0 + 1]; b0 += P2[o1]; b1 += P2[o1 + 1]; }   // P = P1h + P2h
      const double v0 = fma(tk, a1 - a0, a0);
      const double v1 = fma(tk, b1 - b0, b0);
      val = fma(tz, v1 - v0, v0);
    } else {
      double a0 = P[ik], a1 = P[ik + 1];
      if (P2) { a0 += P2[ik]; a1 += P2[ik + 1]; }
      val = fma(tk, a1 - a0, a0);
    }
    const double w = (ngz > 1) ? trapz_weight(gzs, g, ngz) : 1.0;   // cosmology.py:902-903
    acc = fma(w, val * pref[g], acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) cl[warp] = acc;
}

__global__ void limber_kernel(int nl, const double* __restrict__ ells, int nzp, int nk, int ldp,
                              const double* __restrict__ zs, const double* __restrict__ ks,
                              const double* __restrict__ P, const double* __restrict__ P2, int ngz,
                              const double* __restrict__ gzs,
                              const double* __restrict__ pref, const double* __restrict__ chis,
                              double* __restrict__ cl) {
  limber_warp(nl, ells, nzp, nk, ldp, zs, ks, P, P2, ngz, gzs, pref, chis, cl);
}

// several projections of tables on one (z, k) grid in ONE launch (blockIdx.y = job): each is latency-bound (two
// binary searches and a bilinear lookup per redshift), so C_kk, C_kg and C_yy take the time of one
struct LimberJobs { hmv_limber_job j[HMV_LIMBER_MAXJOBS]; };
__global__ void limber_multi_kernel(int nl, const double* __restrict__ ells, int nzp, int nk, int ldp,
                                    const double* __restrict__ zs, const double* __restrict__ ks, const LimberJobs q) {
  const hmv_limber_job& j = q.j[blockIdx.y];
  limber_warp(nl, ells, nzp, nk, ldp, zs, ks, j.P_d, j.P2_d, j.ngz, j.gzs_d, j.pref_d, j.chis_d, j.cl_d);
}

// ---- measurement helpers -----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dfma_kernel(int iters, double seed, double* __restrict__ sink) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double m = 0.999999, c = 1e-9;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 1.2345) sink[0] = s;   // never true; keeps the chains alive
}

__global__ void __launch_bounds__(256) dmma_kernel(int iters, double* __restrict__ sink) {
  const double a = 1.0 + threadIdx.x * 1e-9, b = 1.0 - threadIdx.x * 1e-9;
  double c[8][2];
#pragma unroll
  for (int q = 0; q < 8; ++q) { c[q][0] = 0.0; c[q][1] = 0.0; }
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int q = 0; q < 8; ++q)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[q][0]), "+d"(c[q][1]) : "d"(a), "d"(b));
  }
  double s = 0.0;
#pragma unroll
  for (int q = 0; q < 8; ++q) s += c[q][0] + c[q][1];
  if (s == 1.2345) sink[0] = s;   // never true; keeps the chains alive
}

__global__ void __launch_bounds__(256) copy_kernel(const double2* __restrict__ src, double2* __restrict__ dst,
                                                    long long n2) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride) dst[i] = src[i];
}


// ---- kSZ velocity-reconstruction noise: the short-wavelength integral of Nvv_core_integral (ksz.py:299-336) ----------
//   I[b] = trapz_kS( sanitize( kS * Pge[b,kS]^2 / (Pgg_tot[b,kS] * Cl_tot(chi* kS)) [* Pgg_photo_tot/Pgg_tot] ) )
// b runs over the (mu, kL) plane when the spectra carry the photo-z window and is a single row otherwise; non-finite
// integrand values (C_l = inf beyond the table, C_l = 0 below l = 2) count as zero (ksz.py:98-100).  One warp per b.
__global__ void ksz_nvv_integral_kernel(int nb, int nk, const double* __restrict__ ks, const double* __restrict__ pge,
                                        long long pge_stride, const double* __restrict__ pgg, long long pgg_stride,
                                        const double* __restrict__ pgg_photo, long long photo_stride,
                                        const double* __restrict__ clk, double* __restrict__ out) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= nb) return;
  const double* e = pge ? pge + b * pge_stride : nullptr;
  const double* g = pgg + b * pgg_stride;
  const double* ph = pgg_photo ? pgg_photo + b * photo_stride : nullptr;
  double acc = 0.0;
  for (int k = lane; k < nk; k += 32) {
    const double pe = e ? e[k] : 1.0;
    double v = ks[k] * (pe * pe / (g[k] * clk[k]));
    if (!isfinite(v)) v = 0.0;
    if (ph) {
      v *= ph[k] / g[k];
      if (!isfinite(v)) v = 0.0;
    }
    acc = fma(v, trapz_weight(ks, k, nk), acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[b] = acc;
}

// out[z][s][k] = a_s[z][k] + b_s[z][k]: the P = P1h + P2h tables Limber needs, summed and packed z-major so that ONE
// all-gather over the redshift slabs yields [nz_total][nsp][nk] (each spectrum is then a table of row stride nsp*nk)
struct PackPtrs { const double* a[4]; const double* b[4]; };
__global__ void pack_sum_kernel(int nz, int nk, int nsp, PackPtrs q, double* __restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x, z = blockIdx.y;
  if (k >= nk) return;
  const long long i = (long long)z * nk + k;
  for (int s = 0; s < nsp; ++s) out[((long long)z * nsp + s) * nk + k] = q.a[s][i] + (q.b[s] ? q.b[s][i] : 0.0);
}

}  // namespace hmv
using namespace hmv;

extern "C" int hmv_limber(int nl, const double* ells_d, int nzp, int nk, int ldp, const double* zs_d,
                          const double* ks_d, const double* P_d, const double* P2_d, int ngz, const double* gzs_d,
                          const double* pref_d, const double* chis_d, double* cl_d, void* stream) {
  HMV_REQUIRE(nl > 0 && nzp > 0 && nk >= 2 && ldp >= nk && ngz > 0, "hmv_limber: bad sizes");
  HMV_REQUIRE(ells_d && zs_d && ks_d && P_d && gzs_d && pref_d && chis_d && cl_d, "hmv_limber: null pointer");
  const int wpb = 4;  // warps per block
  limber_kernel<<<cdiv(nl, wpb), wpb * 32, 0, (cudaStream_t)stream>>>(nl, ells_d, nzp, nk, ldp, zs_d, ks_d, P_d, P2_d,
                                                                      ngz, gzs_d, pref_d, chis_d, cl_d);
  return check_launch("limber_kernel");
}

extern "C" int hmv_limber_multi(int njobs, const hmv_limber_job* jobs_h, int nl, const double* ells_d, int nzp, int nk,
                                int ldp, const double* zs_d, const double* ks_d, void* stream) {
  HMV_REQUIRE(njobs >= 1 && njobs <= HMV_LIMBER_MAXJOBS && jobs_h, "hmv_limber_multi: 1..%d jobs", HMV_LIMBER_MAXJOBS);
  HMV_REQUIRE(nl > 0 && nzp > 0 && nk >= 2 && ldp >= nk && ells_d && zs_d && ks_d, "hmv_limber_multi: bad sizes");
  LimberJobs q;
  memset(&q, 0, sizeof(q));
  for (int i = 0; i < njobs; ++i) {
    q.j[i] = jobs_h[i];
    HMV_REQUIRE(q.j[i].P_d && q.j[i].gzs_d && q.j[i].pref_d && q.j[i].chis_d && q.j[i].cl_d && q.j[i].ngz > 0,
                "hmv_limber_multi: job %d: null pointer or ngz <= 0", i);
  }
  const int wpb = 4;
  dim3 grid(cdiv(nl, wpb), njobs);
  limber_multi_kernel<<<grid, wpb * 32, 0, (cudaStream_t)stream>>>(nl, ells_d, nzp, nk, ldp, zs_d, ks_d, q);
  return check_launch("limber_multi_kernel");
}

extern "C" int hmv_ksz_nvv_integral(int nb, int nk, const double* ks_d, const double* pge_d, long long pge_stride,
                                    const double* pgg_d, long long pgg_stride, const double* pgg_photo_d,
                                    long long photo_stride, const double* clk_d, double* out_d, void* stream) {
  HMV_REQUIRE(nb > 0 && nk >= 2 && ks_d && pgg_d && clk_d && out_d, "hmv_ksz_nvv_integral: bad arguments");
  ksz_nvv_integral_kernel<<<cdiv((long long)nb * 32, 128), 128, 0, (cudaStream_t)stream>>>(
      nb, nk, ks_d, pge_d, pge_stride, pgg_d, pgg_stride, pgg_photo_d, photo_stride, clk_d, out_d);
  return check_launch("ksz_nvv_integral_kernel");
}

extern "C" int hmv_pack_sum(int nz, int nk, int nsp, const double* const* a_h, const double* const* b_h, double* out_d,
                            void* stream) {
  HMV_REQUIRE(nz > 0 && nz <= 65535 && nk > 0 && nsp >= 1 && nsp <= 4 && a_h && out_d, "hmv_pack_sum: bad arguments");
  PackPtrs q;
  for (int s = 0; s < 4; ++s) {
    q.a[s] = s < nsp ? a_h[s] : nullptr;
    q.b[s] = (s < nsp && b_h) ? b_h[s] : nullptr;
    HMV_REQUIRE(s >= nsp || q.a[s], "hmv_pack_sum: null table");
  }
  dim3 grid(cdiv(nk, 256), nz);
  pack_sum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(nz, nk, nsp, q, out_d);
  return check_launch("pack_sum_kernel");
}

extern "C" double hmv_bench_dfma(int iters, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* sink = nullptr;
  if (cudaMalloc(&sink, 8) != cudaSuccess) return -1.0;
  const int blocks = sms * 8, threads = 256;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  dfma_kernel<<<blocks, threads, 0, st>>>(iters / 8 + 1, 1.0, sink);  // warm-up
  float best = 1e30f;
  for (int r = 0; r < 3; ++r) {
    cudaEventRecord(e0, st);
    dfma_kernel<<<blocks, threads, 0, st>>>(iters, 1.0, sink);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(sink);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  const double flop = 2.0 * 8.0 * (double)iters * blocks * threads;
  return flop / (best * 1e-3) / 1e12;
}

extern "C" double hmv_bench_dmma(int iters, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* sink = nullptr;
  if (cudaMalloc(&sink, 8) != cudaSuccess) return -1.0;
  const int blocks = sms * 8, threads = 256;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  dmma_kernel<<<blocks, threads, 0, st>>>(iters / 8 + 1, sink);  // warm-up
  float best = 1e30f;
  for (int r = 0; r < 3; ++r) {
    cudaEventRecord(e0, st);
    dmma_kernel<<<blocks, threads, 0, st>>>(iters, sink);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(sink);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  // one m8n8k4 = 256 FMA = 512 flop per warp instruction, 8 per iteration per warp
  const double flop = 512.0 * 8.0 * (double)iters * blocks * (threads / 32);
  return flop / (best * 1e-3) / 1e12;
}

extern "C" double hmv_bench_copy(const double* src_d, double* dst_d, long long n, int reps, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (!src_d || !dst_d || n < 2 || reps < 1) return -1.0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  const long long n2 = n / 2;
  copy_kernel<<<sms * 16, 256, 0, st>>>((const double2*)src_d, (double2*)dst_d, n2);
  float best = 1e30f;
  for (int r = 0; r < reps; ++r) {
    cudaEventRecord(e0, st);
    copy_kernel<<<sms * 16, 256, 0, st>>>((const double2*)src_d, (double2*)dst_d, n2);
    cudaEventRecord(e1, st);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (ms < best) best = ms;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  return 2.0 * 16.0 * (double)n2 / (best * 1e-3) / 1e9;
}
