// k_trispec.cu -- the 1-halo trispectrum of profile tracers and the non-Gaussian Limber covariance of C_l it projects to.
// The reference has no counterpart.  Definitions (DESIGN.md §3.7): with legs t_X(z,m,k) = a_X(z,m) u_X(z,m,k),
// a = M/rho_m0 (matter) or 1 (pressure), u linear in k on the ks grid and clamped to its ends,
//   T^{ABCD}(k1,k2;z) = sum_m w_m n(z,m) t_A(k1) t_B(k1) t_C(k2) t_D(k2)                         (w_m: trapezoid on ms)
//   Cov^{AB,CD}(l,l') = sum_z zeta_z pref_z T((l+1/2)/chi_z, (l'+1/2)/chi_z; z),  pref = H^3 W_A W_B W_C W_D/chi^6/(4 pi fsky)
// (zeta_z: trapezoid on zs, 1 for a single redshift).  No 1-halo damping factor is applied.
//
// Both are one FP64 contraction over K = (z, m): a panel kernel writes P1[K][l] = w_m n (zeta pref) t_A t_B at k1 and
// P2[K][l'] = t_C t_D at k2, and sigma2_gemm_kernel<MT, A K-major> forms C = P1^T P2 on the tensor pipe -- over all of
// K with a fixed-order split-k reduction for the covariance, batched over z (K = m, one batch item per split index)
// for the trispectrum.  A last kernel sums the splits in a fixed order and drops the padding column.  Galaxy (HOD) legs
// of the 1-halo term (DESIGN.md §4.8) have their own panel kernel and feed the same contraction.
// The super-sample covariance (DESIGN.md §4.5) reuses the projection with K = z; sigma_b^2 of a disc is here too.
// The 2-halo trispectrum and its covariance (DESIGN.md §4.6) run the trispectrum's batched product three times per pass
// of redshifts and combine the blocks per (z, k1, k2) with P_lin and its angle average; see the section below.
// The 3- and 4-halo trispectra (DESIGN.md §4.7) add the angle-averaged tree-level bispectrum and trispectrum: exact
// window moments of P_lin per (z, k1, k2), the 2-halo I2 product for the 3-halo term.
#include "common.cuh"
#include "gemm_f64.cuh"

namespace hmv {

constexpr int TP_T = 256, TP_MROWS = 32;   // panel kernel: columns per CTA, mass rows per CTA

struct TrispecLegs {
  const double* u[4];   // cubes [nz][nm][ldk] of A, B (k1 panel) and C, D (k2 panel)
  int matter[4];        // 1: a = M/rho_m0, 0: a = 1
};

// interpolation interval and weight of k on ks, k clamped to [ks[0], ks[nk-1]] (as hmv_limber)
__device__ __forceinline__ void k_locate(const double* __restrict__ ks, int nk, double k, int& j, double& f) {
  k = fmin(fmax(k, ks[0]), ks[nk - 1]);
  j = interval(ks, nk, k);
  HMV_DEV_ASSERT(j >= 0 && j + 1 < nk);
  f = (k - ks[j]) / (ks[j + 1] - ks[j]);
}

__device__ __forceinline__ double k_lerp(const double* __restrict__ row, int j, double f) {
  const double a = row[j];
  return fma(f, row[j + 1] - a, a);
}

// One CTA: redshift blockIdx.y, columns blockIdx.x*TP_T.., mass rows blockIdx.z*TP_MROWS.. of both panels.  A column's
// interval and weight are the same on every mass row, so each thread locates its k once.  Rows m in [nm, nmp) and
// columns in [n, ld) are written as zeros (the contraction reads whole 16-byte words).  chis == nullptr: 3D mode, q
// are wavenumbers; otherwise q are multipoles, k = (q + 1/2)/chi_z and row weights carry zeta_z pref_z.
__global__ void __launch_bounds__(TP_T) trispec_panel_kernel(int nz, int nm, int nmp, int nk, int ldk,
                                                             const double* __restrict__ ks, const double* __restrict__ ms,
                                                             const double* __restrict__ nzm, double rho_m0,
                                                             const TrispecLegs L, int n1, int ld1,
                                                             const double* __restrict__ q1, int n2, int ld2,
                                                             const double* __restrict__ q2, const double* __restrict__ zs,
                                                             const double* __restrict__ chis,
                                                             const double* __restrict__ pref, double* __restrict__ P1,
                                                             double* __restrict__ P2) {
  const int z = blockIdx.y, l = blockIdx.x * TP_T + threadIdx.x;
  const int m0 = blockIdx.z * TP_MROWS, m1 = min(nmp, m0 + TP_MROWS);
  HMV_DEV_ASSERT(z < nz && (nmp == nm || nmp == nm + 1));
  const bool c1 = l < n1, c2 = l < n2;
  double zfac = 1.0, inv_chi = 0.0;
  if (chis) {
    zfac = pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0);
    inv_chi = 1.0 / chis[z];
  }
  int j1 = 0, j2 = 0;
  double f1 = 0.0, f2 = 0.0;
  if (c1) k_locate(ks, nk, chis ? (q1[l] + 0.5) * inv_chi : q1[l], j1, f1);
  if (c2) k_locate(ks, nk, chis ? (q2[l] + 0.5) * inv_chi : q2[l], j2, f2);
  for (int m = m0; m < m1; ++m) {
    const long long K = (long long)z * nmp + m;
    double v1 = 0.0, v2 = 0.0;
    if (m < nm) {
      const long long row = ((long long)z * nm + m) * ldk;
      const double a = ms[m] / rho_m0;
      if (c1) {
        const double wn = trapz_weight(ms, m, nm) * nzm[(long long)z * nm + m] * zfac;
        v1 = wn * (L.matter[0] ? a : 1.0) * k_lerp(L.u[0] + row, j1, f1) * (L.matter[1] ? a : 1.0) *
             k_lerp(L.u[1] + row, j1, f1);
      }
      if (c2) v2 = (L.matter[2] ? a : 1.0) * k_lerp(L.u[2] + row, j2, f2) * (L.matter[3] ? a : 1.0) *
                   k_lerp(L.u[3] + row, j2, f2);
    }
    if (l < ld1) P1[K * ld1 + l] = v1;
    if (l < ld2) P2[K * ld2 + l] = v2;
  }
}

// out[b][i][j] = sum_s part[b*ns + s][i][j] (fixed order: deterministic), j < n2 of the ld2-wide rows
__global__ void trispec_reduce_kernel(long long n, int ns, int n1, int n2, int ld2, const double* __restrict__ part,
                                      double* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long per = (long long)n1 * n2;
  const long long b = i / per, r = i - b * per;
  const long long row = r / n2, col = r - row * n2;
  const long long stride = (long long)n1 * ld2;
  const double* p = part + b * ns * stride + row * ld2 + col;
  double s = 0.0;
  for (int q = 0; q < ns; ++q) s += p[q * stride];
  out[i] = s;
}

// ---- launch plan: a function of the shapes only, so that the workspace size and the launch agree ----------------------
struct TrispecPlan {
  int mt;               // 8*mt output rows per CTA
  int nmp, ld1, ld2;    // rows per redshift (nseg segments of the even-padded mass rows) and panel widths, padded to even
  long long K;          // nz * nmp
  int kchunk, nsplit;   // K range of one split index, split indices per batch item
  int nbatch;           // 1 (covariance) or nz (trispectrum)
};

// output rows per CTA, padded widths and K = nz * rows_z of the contraction of an n1 x n2 result
static TrispecPlan base_plan(int nz, int rows_z, int n1, int n2) {
  TrispecPlan p;
  p.mt = n1 <= 32 ? 4 : n1 <= 64 ? 8 : n1 <= 128 ? 16 : 26;
  p.nmp = rows_z;
  p.ld1 = n1 + (n1 & 1);
  p.ld2 = n2 + (n2 & 1);
  p.K = (long long)nz * p.nmp;
  return p;
}

// The projection's split of K: fills kchunk, nsplit and nbatch = 1 of a plan whose mt, ld1, ld2 and K are set.
static TrispecPlan split_k(TrispecPlan p, int n1) {
  // Split K so that the grid is about sixteen waves of resident CTAs (148 SMs; MT = 26 runs one CTA per SM): the last
  // wave is then a small fraction of the run.  CTAs are issued tile-fastest, so the resident ones walk the same K range
  // together and every panel row comes from HBM about once, the other tiles finding it in L2.  At least eight k
  // steps per split.
  const long long tiles = (long long)cdiv(p.ld2, SG_BN) * cdiv(n1, 8 * p.mt);
  const long long slots = 148LL * (p.mt > 16 ? 1 : 2);
  long long s = 16 * slots / tiles;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  const long long maxs = (p.K + 8 * SG_BK - 1) / (8 * SG_BK);
  if (s > maxs) s = maxs;
  p.kchunk = cdiv(cdiv(p.K, s), SG_BK) * SG_BK;
  p.nsplit = cdiv(p.K, p.kchunk);
  p.nbatch = 1;
  return p;
}

// nseg: segments of mass rows per redshift (2 for the split galaxy pair of the tracer panels, else 1)
static TrispecPlan trispec_plan(bool proj, int nz, int nm, int n1, int n2, int nseg = 1) {
  TrispecPlan p = base_plan(nz, nseg * (nm + (nm & 1)), n1, n2);
  if (!proj) {                       // one batch item per redshift: its K range is its nmp rows
    p.kchunk = p.nmp;
    p.nsplit = 1;
    p.nbatch = nz;
    return p;
  }
  return split_k(p, n1);
}

static long long trispec_ws(const TrispecPlan& p, int n1) {
  return p.K * (p.ld1 + p.ld2) + (long long)p.nbatch * p.nsplit * n1 * p.ld2;
}

static long long trispec_ws_doubles(bool proj, int nz, int nm, int n1, int n2, int nseg = 1) {
  if (nz <= 0 || nm <= 0 || n1 <= 0 || n2 <= 0) return 0;
  return trispec_ws(trispec_plan(proj, nz, nm, n1, n2, nseg), n1);
}

template <int MT>
static cudaError_t trispec_gemm(const TrispecPlan& p, int n1, const double* P1, const double* P2, double* part,
                                cudaStream_t st) {
  const size_t smem = (size_t)sg_smem_doubles<MT, true>() * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(sigma2_gemm_kernel<MT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem);
  if (e != cudaSuccess) return e;
  dim3 grid(cdiv(p.ld2, SG_BN), cdiv(n1, 8 * MT), p.nbatch * p.nsplit);
  sigma2_gemm_kernel<MT, true><<<grid, SG_T, smem, st>>>(n1, p.ld2, (int)p.K, p.kchunk, P1, P2, part,
                                                         (long long)n1 * p.ld2, p.ld1);
  return cudaSuccess;
}

// part = P1^T P2 of a plan's panels at the plan's MT: split-k partial sums [nbatch * nsplit][n1][ld2]
static int trispec_product(const char* who, const TrispecPlan& p, int n1, const double* P1, const double* P2,
                           double* part, cudaStream_t st) {
  cudaError_t e;
  switch (p.mt) {
    case 4: e = trispec_gemm<4>(p, n1, P1, P2, part, st); break;
    case 8: e = trispec_gemm<8>(p, n1, P1, P2, part, st); break;
    case 16: e = trispec_gemm<16>(p, n1, P1, P2, part, st); break;
    default: e = trispec_gemm<26>(p, n1, P1, P2, part, st); break;
  }
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "%s: sigma2_gemm_kernel smem opt-in: %s", who, cudaGetErrorString(e));
  return check_launch("sigma2_gemm_kernel<A K-major>");
}

// C = P1^T P2 of a plan's panels: the contraction into the split-k partial sums, then their fixed-order reduction into
// out [nbatch][n1][n2] without the padding column
static int trispec_contract(const char* who, const TrispecPlan& p, int n1, int n2, const double* P1, const double* P2,
                            double* part, double* out_d, cudaStream_t st) {
  int rc = trispec_product(who, p, n1, P1, P2, part, st);
  if (rc) return rc;
  const long long n = (long long)p.nbatch * n1 * n2;
  trispec_reduce_kernel<<<cdiv(n, 256), 256, 0, st>>>(n, p.nsplit, n1, n2, p.ld2, part, out_d);
  return check_launch("trispec_reduce_kernel");
}

// The size, pointer and limit checks shared by every trispectrum entry point, made before any launch.  check_legs() runs
// between the pointer and the limit checks and sets nseg, the segments of mass rows per redshift that K counts.
template <class LegCheck>
static int trispec_check_args(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                              const double* ms_d, const double* nzm_d, bool legs, int n1, const double* q1_d, int n2,
                              const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                              const double* ws_d, const double* out_d, int& nseg, LegCheck check_legs) {
  HMV_REQUIRE(nz >= 1 && nm >= 1 && nk >= 2 && n1 >= 1 && n2 >= 1,
              "%s: sizes must be >= 1 and nk >= 2 (nz=%d nm=%d nk=%d n1=%d n2=%d)", who, nz, nm, nk, n1, n2);
  HMV_REQUIRE(ldk >= nk && (ldk & 1) == 0, "%s: ldk must be even and >= nk (ldk=%d nk=%d)", who, ldk, nk);
  HMV_REQUIRE(ks_d && ms_d && nzm_d && legs && q1_d && q2_d && ws_d && out_d, "%s: null pointer", who);
  HMV_REQUIRE(!proj || (zs_d && chis_d && pref_d), "%s: null pointer (zs, chis or pref)", who);
  nseg = 1;
  const int rc = check_legs();
  if (rc) return rc;
  HMV_REQUIRE(((size_t)ws_d & 15) == 0, "%s: workspace must be 16-byte aligned", who);
  if (nz > 65535) return fail(HMV_E_LIMIT, "%s: nz=%d exceeds 65535 (grid y of the panel kernel)", who, nz);
  const long long K = (long long)nz * nseg * (nm + (nm & 1));
  if (K > (1LL << 30))
    return fail(HMV_E_LIMIT, "%s: nz * nm%s = %lld exceeds 2^30 (32-bit k index of the contraction)", who,
                nseg > 1 ? " * segments" : "", K);
  return HMV_OK;
}

// The argument checks of every profile-leg trispectrum entry point (1- to 4-halo), made before any launch; fills L.
static int trispec_check(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                         const double* ms_d, const double* nzm_d, const double* const* u_h, const int* kind_h, int n1,
                         const double* q1_d, int n2, const double* q2_d, const double* zs_d, const double* chis_d,
                         const double* pref_d, const double* ws_d, const double* out_d, TrispecLegs& L) {
  int nseg;
  return trispec_check_args(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, u_h && kind_h, n1, q1_d, n2, q2_d, zs_d,
                            chis_d, pref_d, ws_d, out_d, nseg, [&]() -> int {
    for (int i = 0; i < 4; ++i) {
      HMV_REQUIRE(u_h[i], "%s: null pointer (cube %d)", who, i);
      HMV_REQUIRE(kind_h[i] == 0 || kind_h[i] == 2, "%s: cube %d: kind %d is neither 0 (matter) nor 2 (pressure)", who,
                  i, kind_h[i]);
      HMV_REQUIRE(((size_t)u_h[i] & 15) == 0, "%s: cube %d must be 16-byte aligned", who, i);
      L.u[i] = u_h[i];
      L.matter[i] = kind_h[i] == 0;
    }
    return HMV_OK;
  });
}

static int trispec_run(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                       const double* ms_d, const double* nzm_d, double rho_m0, const double* const* u_h,
                       const int* kind_h, int n1, const double* q1_d, int n2, const double* q2_d, const double* zs_d,
                       const double* chis_d, const double* pref_d, double* ws_d, double* out_d, void* stream) {
  TrispecLegs L;
  const int chk = trispec_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, u_h, kind_h, n1, q1_d, n2, q2_d, zs_d,
                                chis_d, pref_d, ws_d, out_d, L);
  if (chk) return chk;
  const TrispecPlan p = trispec_plan(proj, nz, nm, n1, n2);
  double* P1 = ws_d;
  double* P2 = P1 + p.K * p.ld1;
  double* part = P2 + p.K * p.ld2;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 pg(cdiv(p.ld1 > p.ld2 ? p.ld1 : p.ld2, TP_T), nz, cdiv(p.nmp, TP_MROWS));
  trispec_panel_kernel<<<pg, TP_T, 0, st>>>(nz, nm, p.nmp, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, L, n1, p.ld1, q1_d, n2,
                                            p.ld2, q2_d, zs_d, proj ? chis_d : nullptr, pref_d, P1, P2);
  int rc = check_launch("trispec_panel_kernel");
  if (rc) return rc;
  return trispec_contract(who, p, n1, n2, P1, P2, part, out_d, st);
}

// ---- 1-halo trispectrum with galaxy (HOD) legs (DESIGN.md §4.8) ------------------------------------------------------
// A galaxy leg is t_g = (Nc u_c + Ns u_s)/ngal (u_c = 1 without a central profile), hmv_power's HOD leg.  Two galaxy
// legs in one halo take the pair moment without self-pairs,
//   <g g>(k, k') = [NsNsm1 u_s(k) u_s(k') + NcNs (u_c(k) u_s(k') + u_s(k) u_c(k'))] / ngal^2,
// so that with both on one side the panel column is w n <g g>(k, k) (hmv_power's form-1 integrand) and the panels stay
// rank-1.  With one on each side (legs g X at k1, g Y at k2) <g g>(k1, k2) has rank 2 and each redshift gets two
// segments of mass rows, K = (z, segment, m):
//   segment 0:  P1 = w n u_s t_X / ngal^2 (k1)           P2 = (NsNsm1 u_s + NcNs u_c) t_Y (k2)
//   segment 1:  P1 = w n NcNs u_c t_X / ngal^2 (k1)      P2 = u_s t_Y (k2)
// Three or four galaxy legs need higher occupation moments than the HOD defines and are refused.
struct TracerLegs {
  const double* us[4];
  const double* uc[4];                            // kind 1: central profile or null (u_c = 1)
  int kind[4];
  const double *Nc, *Ns, *NcNs, *NsNsm1, *ngal;   // the one HOD of the kind-1 legs
  int pair1, pair2;                               // 1: both legs of side 1 (A, B) / side 2 (C, D) are galaxies
  int g1, g2;                                     // split pair: the galaxy leg of side 1 (0, 1) and side 2 (2, 3); else -1
};

// u_s and u_c of leg x at (row, j, f)
__device__ __forceinline__ void hod_profiles(const TracerLegs& L, int x, long long row, int j, double f, double& us,
                                             double& uc) {
  us = k_lerp(L.us[x] + row, j, f);
  uc = L.uc[x] ? k_lerp(L.uc[x] + row, j, f) : 1.0;
}

// t_x at (row, j, f) of mass element i: a u_s (kind 0 a = M/rho_m0, kind 2 a = 1) or (Nc u_c + Ns u_s)/ngal
__device__ __forceinline__ double tracer_leg(const TracerLegs& L, int x, long long i, long long row, int j, double f,
                                             double a, double ig) {
  if (L.kind[x] == 1) {
    double us, uc;
    hod_profiles(L, x, row, j, f, us, uc);
    return (L.Nc[i] * uc + L.Ns[i] * us) * ig;
  }
  return (L.kind[x] == 0 ? a : 1.0) * k_lerp(L.us[x] + row, j, f);
}

// t_x t_{x+1} of one side, or the pair moment <g g>(k, k) = u_s (2 NcNs u_c + NsNsm1 u_s)/ngal^2 when both are galaxies
__device__ __forceinline__ double tracer_side(const TracerLegs& L, int x, int pair, long long i, long long row, int j,
                                              double f, double a, double ig) {
  if (pair) {
    double us, uc;
    hod_profiles(L, x, row, j, f, us, uc);
    return us * (2.0 * L.NcNs[i] * uc + L.NsNsm1[i] * us) * (ig * ig);
  }
  return tracer_leg(L, x, i, row, j, f, a, ig) * tracer_leg(L, x + 1, i, row, j, f, a, ig);
}

// trispec_panel_kernel for tracer legs: the same grid, columns and padding, with nseg (1 or 2) segments of nmp rows per
// redshift; the split pair (L.g1 >= 0) writes both segments of a mass row from one pair of interval searches.
__global__ void __launch_bounds__(TP_T) trispec_tracer_panel_kernel(int nz, int nm, int nmp, int nseg, int nk, int ldk,
                                                                    const double* __restrict__ ks,
                                                                    const double* __restrict__ ms,
                                                                    const double* __restrict__ nzm, double rho_m0,
                                                                    const TracerLegs L, int n1, int ld1,
                                                                    const double* __restrict__ q1, int n2, int ld2,
                                                                    const double* __restrict__ q2,
                                                                    const double* __restrict__ zs,
                                                                    const double* __restrict__ chis,
                                                                    const double* __restrict__ pref,
                                                                    double* __restrict__ P1, double* __restrict__ P2) {
  const int z = blockIdx.y, l = blockIdx.x * TP_T + threadIdx.x;
  const int m0 = blockIdx.z * TP_MROWS, m1 = min(nmp, m0 + TP_MROWS);
  HMV_DEV_ASSERT(z < nz && (nmp == nm || nmp == nm + 1) && nseg == (L.g1 >= 0 ? 2 : 1));
  const bool c1 = l < n1, c2 = l < n2;
  double zfac = 1.0, inv_chi = 0.0;
  if (chis) {
    zfac = pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0);
    inv_chi = 1.0 / chis[z];
  }
  const double ig = L.ngal ? 1.0 / L.ngal[z] : 1.0;
  int j1 = 0, j2 = 0;
  double f1 = 0.0, f2 = 0.0;
  if (c1) k_locate(ks, nk, chis ? (q1[l] + 0.5) * inv_chi : q1[l], j1, f1);
  if (c2) k_locate(ks, nk, chis ? (q2[l] + 0.5) * inv_chi : q2[l], j2, f2);
  for (int m = m0; m < m1; ++m) {
    double v10 = 0.0, v11 = 0.0, v20 = 0.0, v21 = 0.0;   // panel values of segments 0 and 1
    if (m < nm) {
      const long long i = (long long)z * nm + m, row = i * ldk;
      const double a = ms[m] / rho_m0;
      if (c1) {
        const double wn = trapz_weight(ms, m, nm) * nzm[i] * zfac;
        if (L.g1 >= 0) {
          double us, uc;
          hod_profiles(L, L.g1, row, j1, f1, us, uc);
          const double wx = wn * (ig * ig) * tracer_leg(L, 1 - L.g1, i, row, j1, f1, a, ig);
          v10 = wx * us;
          v11 = wx * L.NcNs[i] * uc;
        } else {
          v10 = wn * tracer_side(L, 0, L.pair1, i, row, j1, f1, a, ig);
        }
      }
      if (c2) {
        if (L.g2 >= 0) {
          double us, uc;
          hod_profiles(L, L.g2, row, j2, f2, us, uc);
          const double ty = tracer_leg(L, 5 - L.g2, i, row, j2, f2, a, ig);
          v20 = (L.NsNsm1[i] * us + L.NcNs[i] * uc) * ty;
          v21 = us * ty;
        } else {
          v20 = tracer_side(L, 2, L.pair2, i, row, j2, f2, a, ig);
        }
      }
    }
    const long long K = (long long)z * nseg * nmp + m;
    if (l < ld1) P1[K * ld1 + l] = v10;
    if (l < ld2) P2[K * ld2 + l] = v20;
    if (nseg == 2) {
      if (l < ld1) P1[(K + nmp) * ld1 + l] = v11;
      if (l < ld2) P2[(K + nmp) * ld2 + l] = v21;
    }
  }
}

// segments per redshift of a leg set: 2 for one galaxy leg on each side, else 1
static int tracer_nseg(const hmv_tracer* legs_h) {
  const bool g1 = legs_h[0].kind == 1 || legs_h[1].kind == 1, g2 = legs_h[2].kind == 1 || legs_h[3].kind == 1;
  const int ng = (legs_h[0].kind == 1) + (legs_h[1].kind == 1) + (legs_h[2].kind == 1) + (legs_h[3].kind == 1);
  return ng == 2 && g1 && g2 ? 2 : 1;
}

static long long tracer_ws_doubles(bool proj, int nz, int nm, int n1, int n2, const hmv_tracer* legs_h) {
  if (!legs_h) return 0;
  return trispec_ws_doubles(proj, nz, nm, n1, n2, tracer_nseg(legs_h));
}

// Checks of the tracer entry points, before any launch: fills L and nseg, ng = the number of galaxy legs.
static int tracer_check(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                        const double* ms_d, const double* nzm_d, const hmv_tracer* legs_h, int n1, const double* q1_d,
                        int n2, const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                        const double* ws_d, const double* out_d, TracerLegs& L, int& nseg, int& ng) {
  return trispec_check_args(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, legs_h != nullptr, n1, q1_d, n2, q2_d, zs_d,
                            chis_d, pref_d, ws_d, out_d, nseg, [&]() -> int {
    const hmv_tracer* g = nullptr;
    ng = 0;
    L.Nc = L.Ns = L.NcNs = L.NsNsm1 = L.ngal = nullptr;
    for (int i = 0; i < 4; ++i) {
      const hmv_tracer& t = legs_h[i];
      HMV_REQUIRE(t.us_d, "%s: null pointer (cube %d)", who, i);
      HMV_REQUIRE(t.kind >= 0 && t.kind <= 2, "%s: leg %d: kind %d is not 0 (matter), 1 (HOD) or 2 (pressure)", who,
                  i, t.kind);
      HMV_REQUIRE(((size_t)t.us_d & 15) == 0 && ((size_t)t.uc_d & 15) == 0, "%s: cube %d must be 16-byte aligned",
                  who, i);
      HMV_REQUIRE(!t.bias_d, "%s: leg %d: bias_d has no meaning in the 1-halo trispectrum; pass NULL", who, i);
      L.us[i] = t.us_d;
      L.uc[i] = t.kind == 1 ? t.uc_d : nullptr;
      L.kind[i] = t.kind;
      if (t.kind != 1) continue;
      HMV_REQUIRE(t.Nc_d && t.Ns_d && t.NcNs_d && t.NsNsm1_d && t.ngal_d, "%s: HOD leg %d lacks occupation arrays", who,
                  i);
      if (g) {
        HMV_REQUIRE(t.us_d == g->us_d && t.uc_d == g->uc_d && t.Nc_d == g->Nc_d && t.Ns_d == g->Ns_d &&
                        t.NcNs_d == g->NcNs_d && t.NsNsm1_d == g->NsNsm1_d && t.ngal_d == g->ngal_d,
                    "%s: HOD legs %d and %d differ: the joint occupation of two HODs is not defined", who,
                    (int)(g - legs_h), i);
      } else {
        g = &t;
        L.Nc = t.Nc_d; L.Ns = t.Ns_d; L.NcNs = t.NcNs_d; L.NsNsm1 = t.NsNsm1_d; L.ngal = t.ngal_d;
      }
      ++ng;
    }
    HMV_REQUIRE(ng <= 2, "%s: %d HOD legs need occupation moments of order %d, which the HOD does not define", who, ng,
                ng);
    L.pair1 = L.kind[0] == 1 && L.kind[1] == 1;
    L.pair2 = L.kind[2] == 1 && L.kind[3] == 1;
    nseg = tracer_nseg(legs_h);
    L.g1 = nseg == 2 ? (L.kind[0] == 1 ? 0 : 1) : -1;
    L.g2 = nseg == 2 ? (L.kind[2] == 1 ? 2 : 3) : -1;
    return HMV_OK;
  });
}

// Profile legs only: trispec_run, so that the result is the profile entry point's to the bit.
static int tracer_run(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                      const double* ms_d, const double* nzm_d, double rho_m0, const hmv_tracer* legs_h, int n1,
                      const double* q1_d, int n2, const double* q2_d, const double* zs_d, const double* chis_d,
                      const double* pref_d, double* ws_d, double* out_d, void* stream) {
  TracerLegs L;
  int nseg = 1, ng = 0;
  const int chk = tracer_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, legs_h, n1, q1_d, n2, q2_d, zs_d, chis_d,
                               pref_d, ws_d, out_d, L, nseg, ng);
  if (chk) return chk;
  if (ng == 0) {
    const double* u_h[4] = {legs_h[0].us_d, legs_h[1].us_d, legs_h[2].us_d, legs_h[3].us_d};
    const int kind_h[4] = {legs_h[0].kind, legs_h[1].kind, legs_h[2].kind, legs_h[3].kind};
    return trispec_run(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, u_h, kind_h, n1, q1_d, n2, q2_d, zs_d,
                       chis_d, pref_d, ws_d, out_d, stream);
  }
  const TrispecPlan p = trispec_plan(proj, nz, nm, n1, n2, nseg);
  const int nmp = nm + (nm & 1);
  double* P1 = ws_d;
  double* P2 = P1 + p.K * p.ld1;
  double* part = P2 + p.K * p.ld2;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 pg(cdiv(p.ld1 > p.ld2 ? p.ld1 : p.ld2, TP_T), nz, cdiv(nmp, TP_MROWS));
  trispec_tracer_panel_kernel<<<pg, TP_T, 0, st>>>(nz, nm, nmp, nseg, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, L, n1,
                                                   p.ld1, q1_d, n2, p.ld2, q2_d, zs_d, proj ? chis_d : nullptr, pref_d,
                                                   P1, P2);
  int rc = check_launch("trispec_tracer_panel_kernel");
  if (rc) return rc;
  return trispec_contract(who, p, n1, n2, P1, P2, part, out_d, st);
}

// ---- 2-halo trispectrum (DESIGN.md §4.6)-------------------------------------------------------------------------------
//   T2h^{ABCD}(k1,k2;z) = P(k1) [I1~A(k1) I3^{BCD}(k1,k2,k2) + I1~B(k1) I3^{ACD}(k1,k2,k2)]
//                       + P(k2) [I1~C(k2) I3^{ABD}(k1,k1,k2) + I1~D(k2) I3^{ABC}(k1,k1,k2)]
//                       + Pbar(k1,k2) [I2^{AC}(k1,k2) I2^{BD}(k1,k2) + I2^{AD}(k1,k2) I2^{BC}(k1,k2)]
// with I2, I3 = sum_m w_m n b t t (t), I1~X = sum_m w_m n b t_X + b_X - C_X (hmv_power's 2-halo legs), P = P_lin linear
// in k on ks and clamped, Pbar its angle average from a per-redshift prefix table of int q P dq.  Per chunk of zc
// redshifts, four panels over K = (z, m), with w^ = w_m n b:
//   P1s [K][nA1 n1p] = w^ t_A | w^ t_B (k1)        P1p [K][n1q] = w^ t_A t_B (k1) | w^
//   P2s [K][nC1 n2p] = t_C | t_D (k2)              P2p [K][n2q] = t_C t_D (k2) | 1
// (nA1 = 1 when A and B coincide, nC1 likewise; n1p = n1 rounded up to even, n1q = n1 + 1 rounded up to even) and three
// batched products, one batch item per redshift:
//   O22 = P1s^T P2s: I2^{XY}      O3a = P1s^T P2p: I3^{XCD} and, in column n2, sum w^ t_X(k1)
//   O3b = P1p^T P2s: I3^{ABY} and, in row n1, sum w^ t_Y(k2)
// The contraction reads B with the row stride of its output, so each product's operands are whole panels; a product per
// pair of panels keeps every block in [k1][k2] order for the assembly.  nA1 nC1 + nA1 + nC1 blocks: 8, 5 or 3.
struct Legs2h {
  const double* u[4];
  int matter[4];
  int nA1, nC1;          // distinct legs at k1 (1: A == B) and at k2 (1: C == D)
};

struct Plan2h {
  int zc, nmp, n1, n2, n1p, n1q, n2p, n2q, nk, nA1, nC1;
  __host__ __device__ long long m1s() const { return (long long)nA1 * n1p; }   // rows of O22 and O3a
  __host__ __device__ long long m2s() const { return (long long)nC1 * n2p; }   // columns of O22 and O3b
  // per-redshift sizes (all even, so that every region stays 16-byte aligned)
  __host__ __device__ long long panels() const { return (long long)nmp * (m1s() + n1q + m2s() + n2q); }
  __host__ __device__ long long blocks() const { return m1s() * m2s() + m1s() * n2q + (long long)n1q * m2s(); }
  __host__ __device__ long long sides() const { return (n1 + (n1 & 1)) + (n2 + (n2 & 1)) + (nk + (nk & 1)) + 2; }
  __host__ __device__ long long ws() const { return (long long)zc * (panels() + blocks() + sides()); }
};

static Plan2h plan_2h(int nm, int nk, int n1, int n2, int nA1, int nC1, int zc) {
  Plan2h p;
  p.zc = zc;
  p.nmp = nm + (nm & 1);
  p.n1 = n1;
  p.n2 = n2;
  p.n1p = n1 + (n1 & 1);
  p.n2p = n2 + (n2 & 1);
  p.n1q = (n1 + 1) + ((n1 + 1) & 1);
  p.n2q = (n2 + 1) + ((n2 + 1) & 1);
  p.nk = nk;
  p.nA1 = nA1;
  p.nC1 = nC1;
  return p;
}

// legs coincide when they read the same cube with the same kind
static void distinct_2h(const double* const* u_h, const int* kind_h, int& nA1, int& nC1) {
  nA1 = (u_h[0] == u_h[1] && kind_h[0] == kind_h[1]) ? 1 : 2;
  nC1 = (u_h[2] == u_h[3] && kind_h[2] == kind_h[3]) ? 1 : 2;
}

static long long trispec2h_ws_doubles(int nz, int nm, int nk, int n1, int n2, const double* const* u_h,
                                      const int* kind_h, int zchunk) {
  if (nz <= 0 || nm <= 0 || nk < 2 || n1 <= 0 || n2 <= 0 || !u_h || !kind_h || zchunk < 1 || zchunk > nz) return 0;
  int nA1, nC1;
  distinct_2h(u_h, kind_h, nA1, nC1);
  return plan_2h(nm, nk, n1, n2, nA1, nC1, zchunk).ws();
}

// One CTA per chunk redshift: C = sum_m w_m n b M/rho_m0 (the matter consistency integral of hmv_power) into Cm[zl], and
// S[zl][j] = int_{ks[0]}^{ks[j]} q P(q) dq, exact for P linear on each interval.  Each thread sums a contiguous run of
// intervals, thread 0 scans the run totals: a fixed order, so every chunking gives the same bits.
__global__ void __launch_bounds__(256) trispec2h_prep_kernel(int z0, int nm, int nk, const double* __restrict__ ks,
                                                             const double* __restrict__ ms,
                                                             const double* __restrict__ nzm,
                                                             const double* __restrict__ bh,
                                                             const double* __restrict__ Pzk, double rho_m0,
                                                             double* __restrict__ Cm, double* __restrict__ S) {
  __shared__ double red[256];
  const int zl = blockIdx.x, z = z0 + zl, t = threadIdx.x;
  double c = 0.0;
  for (int m = t; m < nm; m += blockDim.x) {
    const long long i = (long long)z * nm + m;
    c = fma(trapz_weight(ms, m, nm) * nzm[i] * bh[i], ms[m] / rho_m0, c);
  }
  c = block_sum(c, red);
  if (t == 0) Cm[zl] = c;
  const double* P = Pzk + (long long)z * nk;
  double* Sz = S + (long long)zl * nk;
  const int per = (nk - 1 + blockDim.x - 1) / blockDim.x, j0 = min(nk - 1, t * per), j1 = min(nk - 1, j0 + per);
  double run = 0.0;
  for (int j = j0; j < j1; ++j) {
    const double x0 = ks[j], x1 = ks[j + 1];
    run += (x1 - x0) * (x0 * (2.0 * P[j] + P[j + 1]) + x1 * (P[j] + 2.0 * P[j + 1])) / 6.0;
  }
  __syncthreads();
  red[t] = run;
  __syncthreads();
  if (t == 0) {
    double s = 0.0;
    for (int q = 0; q < (int)blockDim.x; ++q) {
      const double v = red[q];
      red[q] = s;
      s += v;
    }
    Sz[0] = 0.0;
  }
  __syncthreads();
  run = red[t];
  for (int j = j0; j < j1; ++j) {
    const double x0 = ks[j], x1 = ks[j + 1];
    run += (x1 - x0) * (x0 * (2.0 * P[j] + P[j + 1]) + x1 * (P[j] + 2.0 * P[j + 1])) / 6.0;
    Sz[j + 1] = run;
  }
}

// One CTA: chunk redshift blockIdx.y, columns blockIdx.x*TP_T.., mass rows blockIdx.z*TP_MROWS.. of the four panels;
// one interval search per column and side.  The first mass group also writes P(k1) and P(k2) of its columns.  Padding
// rows (m = nm) and columns are zeros; the sum columns (w^ in P1p, 1 in P2p) sit at n1 and n2.
__global__ void __launch_bounds__(TP_T) trispec2h_panel_kernel(int z0, int nm, int nk, int ldk,
                                                               const double* __restrict__ ks,
                                                               const double* __restrict__ ms,
                                                               const double* __restrict__ nzm,
                                                               const double* __restrict__ bh,
                                                               const double* __restrict__ Pzk, double rho_m0,
                                                               const Legs2h L, const Plan2h p,
                                                               const double* __restrict__ q1,
                                                               const double* __restrict__ q2,
                                                               const double* __restrict__ chis, double* __restrict__ P1s,
                                                               double* __restrict__ P1p, double* __restrict__ P2s,
                                                               double* __restrict__ P2p, double* __restrict__ Pk1,
                                                               double* __restrict__ Pk2) {
  const int zl = blockIdx.y, z = z0 + zl, l = blockIdx.x * TP_T + threadIdx.x;
  const int m0 = blockIdx.z * TP_MROWS, m1 = min(p.nmp, m0 + TP_MROWS);
  const bool c1 = l < p.n1, c2 = l < p.n2;
  const double inv_chi = chis ? 1.0 / chis[z] : 0.0;
  int j1 = 0, j2 = 0;
  double f1 = 0.0, f2 = 0.0;
  if (c1) k_locate(ks, nk, chis ? (q1[l] + 0.5) * inv_chi : q1[l], j1, f1);
  if (c2) k_locate(ks, nk, chis ? (q2[l] + 0.5) * inv_chi : q2[l], j2, f2);
  if (blockIdx.z == 0) {
    if (c1) Pk1[(long long)zl * p.n1 + l] = k_lerp(Pzk + (long long)z * nk, j1, f1);
    if (c2) Pk2[(long long)zl * p.n2 + l] = k_lerp(Pzk + (long long)z * nk, j2, f2);
  }
  const long long w1s = p.m1s(), w2s = p.m2s();
  for (int m = m0; m < m1; ++m) {
    const long long K = (long long)zl * p.nmp + m;
    double tA = 0.0, tB = 0.0, tC = 0.0, tD = 0.0, w = 0.0, one = 0.0;
    if (m < nm) {
      const long long row = ((long long)z * nm + m) * ldk, i = (long long)z * nm + m;
      const double a = ms[m] / rho_m0;
      w = trapz_weight(ms, m, nm) * nzm[i] * bh[i];
      one = 1.0;
      if (c1) {
        tA = (L.matter[0] ? a : 1.0) * k_lerp(L.u[0] + row, j1, f1);
        tB = (L.matter[1] ? a : 1.0) * k_lerp(L.u[1] + row, j1, f1);
      }
      if (c2) {
        tC = (L.matter[2] ? a : 1.0) * k_lerp(L.u[2] + row, j2, f2);
        tD = (L.matter[3] ? a : 1.0) * k_lerp(L.u[3] + row, j2, f2);
      }
    }
    if (l < p.n1p) {
      P1s[K * w1s + l] = w * tA;
      if (p.nA1 == 2) P1s[K * w1s + p.n1p + l] = w * tB;
    }
    if (l < p.n1q) P1p[K * p.n1q + l] = c1 ? w * tA * tB : (l == p.n1 ? w : 0.0);
    if (l < p.n2p) {
      P2s[K * w2s + l] = tC;
      if (p.nC1 == 2) P2s[K * w2s + p.n2p + l] = tD;
    }
    if (l < p.n2q) P2p[K * p.n2q + l] = c2 ? tC * tD : (l == p.n2 ? one : 0.0);
  }
}

// P linear on each interval of ks and held at the end values outside: its value at x >= 0, and the region of x
// (-1: below ks[0], nk - 1: at or above ks[nk-1], else the interval)
__device__ __forceinline__ double plin_at(const double* __restrict__ ks, const double* __restrict__ P, int nk, double x,
                                          int& r) {
  if (x < ks[0]) { r = -1; return P[0]; }
  if (x >= ks[nk - 1]) { r = nk - 1; return P[nk - 1]; }
  r = interval(ks, nk, x);
  const double f = (x - ks[r]) / (ks[r + 1] - ks[r]);
  return fma(f, P[r + 1] - P[r], P[r]);
}

// int_{x0}^{x1} q P(q) dq for P linear on [x0, x1] with end values p0, p1; h = x1 - x0, formed by the caller
__device__ __forceinline__ double qp_piece(double h, double x0, double x1, double p0, double p1) {
  return h * (x0 * (2.0 * p0 + p1) + x1 * (p0 + 2.0 * p1)) / 6.0;
}

// Pbar(k1,k2) = (1/2k1k2) int_{|k1-k2|}^{k1+k2} q P(q) dq.  Ends in one region: the piece alone, with b - a = 2 min(k1,k2)
// cancelled against the prefactor.  Adjacent regions: two pieces.  Otherwise two pieces and a difference of prefixes
// S over at least one whole interval.  The pieces' widths xa - a and b - xb are formed as (xa - hi) + lo and
// (hi - xb) + lo: a and b themselves carry a rounding error of hi, which is large against the width when lo << hi.
__device__ __forceinline__ double pbar(const double* __restrict__ ks, const double* __restrict__ P,
                                       const double* __restrict__ S, int nk, double k1, double k2) {
  const double lo = fmin(k1, k2), hi = fmax(k1, k2), a = hi - lo, b = hi + lo;
  int ra, rb;
  const double pa = plin_at(ks, P, nk, a, ra), pb = plin_at(ks, P, nk, b, rb);
  if (ra == rb) return (a * (2.0 * pa + pb) + b * (pa + 2.0 * pb)) / (6.0 * hi);
  const double xa = ks[ra + 1], xb = ks[rb];
  double s = qp_piece((xa - hi) + lo, a, xa, pa, P[ra + 1]) + qp_piece((hi - xb) + lo, xb, b, P[rb], pb);
  if (rb > ra + 1) s += S[rb] - S[ra + 1];
  return s / (2.0 * k1 * k2);
}

// One thread per output element (i, j): the chunk's redshifts in increasing z.  3D mode writes T2h per redshift into
// out[z][i][j]; projection mode adds zeta_z pref_z T2h onto the previous chunk's value (first == 1: onto zero).
__global__ void __launch_bounds__(256) trispec2h_assemble_kernel(int z0, int zc, int nz, int nk,
                                                                 const double* __restrict__ ks,
                                                                 const double* __restrict__ Pzk, const Legs2h L,
                                                                 const Plan2h p, const double* __restrict__ q1,
                                                                 const double* __restrict__ q2,
                                                                 const double* __restrict__ zs,
                                                                 const double* __restrict__ chis,
                                                                 const double* __restrict__ pref,
                                                                 const double* __restrict__ O22,
                                                                 const double* __restrict__ O3a,
                                                                 const double* __restrict__ O3b,
                                                                 const double* __restrict__ Pk1,
                                                                 const double* __restrict__ Pk2,
                                                                 const double* __restrict__ Cm,
                                                                 const double* __restrict__ S, int first,
                                                                 double* __restrict__ out) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x, n = (long long)p.n1 * p.n2;
  if (e >= n) return;
  const int i = (int)(e / p.n2), j = (int)(e - (long long)i * p.n2);
  const long long w22 = p.m2s(), w3b = p.m2s();
  const long long s22 = p.m1s() * w22, s3a = p.m1s() * p.n2q, s3b = (long long)p.n1q * w3b;
  const long long rB = (p.nA1 == 2 ? p.n1p : 0), cD = (p.nC1 == 2 ? p.n2p : 0);
  double acc = (chis && !first) ? out[e] : 0.0;
  for (int zl = 0; zl < zc; ++zl) {
    const int z = z0 + zl;
    const double* o22 = O22 + zl * s22;
    const double* o3a = O3a + zl * s3a;
    const double* o3b = O3b + zl * s3b;
    const double cm = 1.0 - Cm[zl];
    const long long il = i;
    const double I1A = o3a[il * p.n2q + p.n2] + (L.matter[0] ? cm : 0.0);
    const double I1B = o3a[(rB + i) * p.n2q + p.n2] + (L.matter[1] ? cm : 0.0);
    const double I1C = o3b[p.n1 * w3b + j] + (L.matter[2] ? cm : 0.0);
    const double I1D = o3b[p.n1 * w3b + cD + j] + (L.matter[3] ? cm : 0.0);
    const double I3ACD = o3a[il * p.n2q + j], I3BCD = o3a[(rB + i) * p.n2q + j];
    const double I3ABC = o3b[il * w3b + j], I3ABD = o3b[il * w3b + cD + j];
    const double I2AC = o22[il * w22 + j], I2AD = o22[il * w22 + cD + j];
    const double I2BC = o22[(rB + i) * w22 + j], I2BD = o22[(rB + i) * w22 + cD + j];
    const double inv_chi = chis ? 1.0 / chis[z] : 0.0;
    const double k1 = chis ? (q1[i] + 0.5) * inv_chi : q1[i], k2 = chis ? (q2[j] + 0.5) * inv_chi : q2[j];
    const double pb = pbar(ks, Pzk + (long long)z * nk, S + (long long)zl * nk, nk, k1, k2);
    const double T = Pk1[(long long)zl * p.n1 + i] * (I1A * I3BCD + I1B * I3ACD) +
                     Pk2[(long long)zl * p.n2 + j] * (I1C * I3ABD + I1D * I3ABC) + pb * (I2AC * I2BD + I2AD * I2BC);
    if (chis) acc += pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0) * T;
    else out[(long long)z * n + e] = T;
  }
  if (chis) out[e] = acc;
}

static int trispec2h_run(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                         const double* ms_d, const double* nzm_d, const double* bh_d, const double* Pzk_d,
                         double rho_m0, const double* const* u_h, const int* kind_h, int n1, const double* q1_d, int n2,
                         const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                         int zchunk, double* ws_d, double* out_d, void* stream) {
  Legs2h L;
  {
    TrispecLegs L4;
    const int chk = trispec_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, u_h, kind_h, n1, q1_d, n2, q2_d, zs_d,
                                  chis_d, pref_d, ws_d, out_d, L4);
    if (chk) return chk;
    for (int i = 0; i < 4; ++i) {
      L.u[i] = L4.u[i];
      L.matter[i] = L4.matter[i];
    }
  }
  HMV_REQUIRE(bh_d && Pzk_d, "%s: null pointer (bh or Pzk)", who);
  HMV_REQUIRE(zchunk >= 1 && zchunk <= nz, "%s: zchunk must lie in [1, nz] (zchunk=%d nz=%d)", who, zchunk, nz);
  distinct_2h(u_h, kind_h, L.nA1, L.nC1);
  const Plan2h full = plan_2h(nm, nk, n1, n2, L.nA1, L.nC1, zchunk);
  const long long zc = zchunk;
  double* P1s = ws_d;
  double* P1p = P1s + zc * full.nmp * full.m1s();
  double* P2s = P1p + zc * full.nmp * full.n1q;
  double* P2p = P2s + zc * full.nmp * full.m2s();
  double* O22 = P2p + zc * full.nmp * full.n2q;
  double* O3a = O22 + zc * full.m1s() * full.m2s();
  double* O3b = O3a + zc * full.m1s() * full.n2q;
  double* Pk1 = O3b + zc * full.n1q * full.m2s();
  double* Pk2 = Pk1 + zc * (n1 + (n1 & 1));
  double* S = Pk2 + zc * (n2 + (n2 & 1));
  double* Cm = S + zc * (nk + (nk & 1));
  cudaStream_t st = (cudaStream_t)stream;
  const long long nout = (long long)n1 * n2;
  for (int z0 = 0; z0 < nz; z0 += zchunk) {
    const int zn = min(zchunk, nz - z0);
    Plan2h p = full;
    p.zc = zn;
    trispec2h_prep_kernel<<<zn, 256, 0, st>>>(z0, nm, nk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, Cm, S);
    int rc = check_launch("trispec2h_prep_kernel");
    if (rc) return rc;
    dim3 pg(cdiv(p.n1q > p.n2q ? p.n1q : p.n2q, TP_T), zn, cdiv(p.nmp, TP_MROWS));
    trispec2h_panel_kernel<<<pg, TP_T, 0, st>>>(z0, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, L, p, q1_d,
                                                q2_d, proj ? chis_d : nullptr, P1s, P1p, P2s, P2p, Pk1, Pk2);
    rc = check_launch("trispec2h_panel_kernel");
    if (rc) return rc;
    // the three batched products: rows x columns = m1s x m2s, m1s x n2q, n1q x m2s, K = the nmp rows of each redshift
    const struct { int rows, cols; const double *A, *B; double* C; } prod[3] = {
        {(int)p.m1s(), (int)p.m2s(), P1s, P2s, O22},
        {(int)p.m1s(), p.n2q, P1s, P2p, O3a},
        {p.n1q, (int)p.m2s(), P1p, P2s, O3b}};
    for (const auto& g : prod) {
      rc = trispec_product(who, trispec_plan(false, zn, nm, g.rows, g.cols), g.rows, g.A, g.B, g.C, st);
      if (rc) return rc;
    }
    trispec2h_assemble_kernel<<<cdiv(nout, 256), 256, 0, st>>>(z0, zn, nz, nk, ks_d, Pzk_d, L, p, q1_d, q2_d, zs_d,
                                                               proj ? chis_d : nullptr, pref_d, O22, O3a, O3b, Pk1, Pk2,
                                                               Cm, S, z0 == 0, out_d);
    rc = check_launch("trispec2h_assemble_kernel");
    if (rc) return rc;
  }
  return HMV_OK;
}

// ---- 3- and 4-halo trispectra (DESIGN.md §4.7) ------------------------------------------------------------------------
//   T3h^{ABCD}(k1,k2;z) = Bbar [I2^{AC} I1~B I1~D + I2^{AD} I1~B I1~C + I2^{BC} I1~A I1~D + I2^{BD} I1~A I1~C]
//   T4h^{ABCD}(k1,k2;z) = I1~A I1~B I1~C I1~D Tbar
//   Bbar = (34/21) P1 P2 + 2 <G P(q)>,   Tbar = 12 P1 P2^2 F3bar(k2/k1) + 12 P1^2 P2 F3bar(k1/k2) + 8 <G^2 P(q)>
// with I1~, I2 as in the 2-halo section, P1 = P(k1), P2 = P(k2), q = |k1 + k2| and, for x = q^2 and d = k1^2 - k2^2,
//   G = P1 F2(-k1, k1+k2) + P2 F2(-k2, k1+k2) = g1 x + g0 + gm / x,
//   g1 = -5/28 (P1/k1^2 + P2/k2^2),  g0 = 13/28 (P1 + P2) - 3d/28 (P1/k1^2 - P2/k2^2),
//   gm = -d/4 (P1 - P2) + d^2/14 (P1/k1^2 + P2/k2^2).
// <f> = (1/(2 k1 k2)) int_{|k1-k2|}^{k1+k2} q f(q) dq, so <G P> and <G^2 P> are sums of gn M_n with the window moments
// M_n = int q^n P(q) dq, n = -3, -1, 1, 3, 5: exact for P linear on each interval of ks and held at its end values.

// double-double accumulation of the moment tables: a window's moment is a difference of two table entries, and a
// double table would lose (window / whole range) of it
struct DD {
  double hi, lo;
};

__device__ __forceinline__ DD dd_add(DD a, double b) {
  const double s = a.hi + b, bb = s - a.hi, e = ((a.hi - (s - bb)) + (b - bb)) + a.lo, h = s + e;
  return {h, e - (h - s)};
}

__device__ __forceinline__ DD dd_add(DD a, DD b) {
  const double s = a.hi + b.hi, bb = s - a.hi, e = ((a.hi - (s - bb)) + (b.hi - bb)) + (a.lo + b.lo), h = s + e;
  return {h, e - (h - s)};
}

// a - b rounded to double
__device__ __forceinline__ double dd_diff(DD a, DD b) {
  const double s = a.hi - b.hi, bb = s - a.hi, e = (a.hi - (s - bb)) + (-b.hi - bb);
  return s + (e + (a.lo - b.lo));
}

constexpr int PT_NMOM = 5;   // moments q^-3, q^-1, q^1, q^3, q^5

// int_{x0}^{x1} q^n P(q) dq, n = -3, -1, 1, 3, 5, for P linear from p0 at x0 to p1 at x1; h = x1 - x0 formed by the
// caller.  The negative powers in closed forms without cancellation (x0 = 0 gives 0: their coefficients vanish there);
// the positive ones by 4-node Gauss-Legendre, exact for these polynomials of degree <= 6.
__device__ __forceinline__ void qmom_piece(double x0, double x1, double h, double p0, double p1, double m[PT_NMOM]) {
  if (x0 > 0.0) {
    const double y = h / x0, L = log1p(y);
    m[0] = h * (p0 * (x1 / x0) + p1) / (2.0 * x0 * x1 * x1);
    m[1] = p0 * L + (p1 - p0) * (1.0 - L / y);
  } else {
    m[0] = m[1] = 0.0;
  }
  const double t[4] = {0.06943184420297371, 0.33000947820757187, 0.66999052179242813, 0.93056815579702629};
  const double w[4] = {0.17392742256872693, 0.32607257743127307, 0.32607257743127307, 0.17392742256872693};
  m[2] = m[3] = m[4] = 0.0;
  for (int i = 0; i < 4; ++i) {
    const double q = fma(h, t[i], x0), q2 = q * q, v = h * w[i] * q * fma(t[i], p1 - p0, p0);
    m[2] += v;
    m[3] = fma(v, q2, m[3]);
    m[4] = fma(v * q2, q2, m[4]);
  }
}

// One CTA per chunk redshift: tab[zl][n][j] (double-double) = int_{ks[0]}^{ks[j]} q^n P for n = 1, 3, 5 and
// int_{ks[j]}^{ks[nk-1]} q^n P for n = -3, -1 (each accumulated from the end where it is small, so that a difference is
// dominated by its own window).  Each thread sums a contiguous run of intervals, thread 0 scans the run totals: a fixed
// order, so every chunking gives the same bits.
__global__ void __launch_bounds__(256) trispec_pt_moments_kernel(int z0, int nk, const double* __restrict__ ks,
                                                                 const double* __restrict__ Pzk,
                                                                 DD* __restrict__ tab) {
  __shared__ DD red[256][PT_NMOM];
  const int zl = blockIdx.x, z = z0 + zl, t = threadIdx.x;
  const double* P = Pzk + (long long)z * nk;
  DD* T = tab + (long long)zl * PT_NMOM * nk;
  const int per = (nk - 1 + blockDim.x - 1) / blockDim.x, j0 = min(nk - 1, t * per), j1 = min(nk - 1, j0 + per);
  DD run[PT_NMOM];
  double m[PT_NMOM];
  for (int n = 0; n < PT_NMOM; ++n) run[n] = {0.0, 0.0};
  for (int j = j0; j < j1; ++j) {
    qmom_piece(ks[j], ks[j + 1], ks[j + 1] - ks[j], P[j], P[j + 1], m);
    for (int n = 0; n < PT_NMOM; ++n) run[n] = dd_add(run[n], m[n]);
  }
  for (int n = 0; n < PT_NMOM; ++n) red[t][n] = run[n];
  __syncthreads();
  if (t == 0) {   // exclusive scans: forward for the positive powers, backward for the negative ones
    for (int n = 0; n < PT_NMOM; ++n) {
      DD s = {0.0, 0.0};
      for (int i = 0; i < (int)blockDim.x; ++i) {
        const int q = n < 2 ? (int)blockDim.x - 1 - i : i;
        const DD v = red[q][n];
        red[q][n] = s;
        s = dd_add(s, v);
      }
      T[(long long)n * nk + (n < 2 ? nk - 1 : 0)] = {0.0, 0.0};
    }
  }
  __syncthreads();
  for (int n = 0; n < PT_NMOM; ++n) run[n] = red[t][n];
  for (int j = j0; j < j1; ++j) {
    qmom_piece(ks[j], ks[j + 1], ks[j + 1] - ks[j], P[j], P[j + 1], m);
    for (int n = 2; n < PT_NMOM; ++n) {
      run[n] = dd_add(run[n], m[n]);
      T[(long long)n * nk + j + 1] = run[n];
    }
  }
  for (int j = j1 - 1; j >= j0; --j) {
    qmom_piece(ks[j], ks[j + 1], ks[j + 1] - ks[j], P[j], P[j + 1], m);
    for (int n = 0; n < 2; ++n) {
      run[n] = dd_add(run[n], m[n]);
      T[(long long)n * nk + j] = run[n];
    }
  }
}

// Ratios max(k1,k2)/min(k1,k2) >= PT_R0 take the local branch of pt_averages (below).  The Laurent sums' terms grow
// like r^2 times <G^2 P>, and Tbar is a further r^2 below its two leading pieces (12 P_lo^2 P_hi F3bar(lo/hi) ->
// -(2/3) r^2 P_lo^2 P_hi and 8 <G^2 P> -> +(2/3) r^2 P_lo^2 P_hi), so there the Laurent route would lose eps r^4 of
// Tbar; below PT_R0 that is <~1e-9.  The local branch costs 8 evaluations per interval its window crosses, so PT_R0 is
// as large as that loss allows.  The decision uses the caller's q values, so the F3 table and the assembly agree.
constexpr double PT_R0 = 100.0;

__device__ __forceinline__ bool pt_local(double x1, double x2) { return fmax(x1, x2) >= PT_R0 * fmin(x1, x2); }

// The local branch, in t = q - hi on the window t in [-lo, lo] (r = hi/lo >= PT_R0).  With A = -(1/2) r mu P_lo, the
// large part of P_lo F2(-k_lo, s), and R = G - A (bounded):
//   <G P>   = <A (P(q) - P_hi) + R P(q)>                       (<A> P_hi = 0)
//   <D>     = <G^2 P> - (r^2/12) P_lo^2 P_hi = <A^2 (P(q) - P_hi) + (2A + R) R P(q)>
// and the caller's Tbar = 12 P1 P2 (P2 F12 + P1 F21) + 8 <D> holds with the table entry of the small ratio x = lo/hi
// taken as F3bar(x) + 1/(18 x^2) (f3bar's tail): the two -(2/3) r^2 P_lo^2 P_hi pieces cancel in closed form.  Every
// factor is formed from local differences: mu r = (t (2 hi + t) - lo^2)/(2 lo^2); P(q) - P_hi from node differences
// and slopes times local lengths.  Each piece of the window between nodes takes 8-node Gauss-Legendre: the integrand
// is a polynomial of degree <= 6 in t plus a rational part whose poles (q = 0) lie r half-widths away, so the rule's
// error is below (2 r)^-16 of the terms.  Pointwise terms are O(r) times the result: the error is a few eps r.
__device__ __noinline__ void pt_averages_local(const double* __restrict__ ks, const double* __restrict__ P, int nk,
                                               double k1, double k2, double P1, double P2, double& gp, double& g2p) {
  const double x[4] = {0.1834346424956498, 0.5255324099163290, 0.7966664774136267, 0.9602898564975363};
  const double w[4] = {0.3626837833783620, 0.3137066458778873, 0.2223810344533745, 0.1012285362903763};
  const double lo = fmin(k1, k2), hi = fmax(k1, k2), Plo = k1 <= k2 ? P1 : P2, Phi = k1 <= k2 ? P2 : P1;
  int ra, rb, m;
  plin_at(ks, P, nk, hi - lo, ra);
  plin_at(ks, P, nk, hi + lo, rb);
  plin_at(ks, P, nk, hi, m);
  const double sm = (m < 0 || m >= nk - 1) ? 0.0 : (P[m + 1] - P[m]) / (ks[m + 1] - ks[m]);
  const double lo2 = lo * lo;
  double sg = 0.0, sd = 0.0;
  for (int j = ra; j <= rb; ++j) {
    const bool held = j < 0 || j >= nk - 1;
    const double sj = held ? 0.0 : (P[j + 1] - P[j]) / (ks[j + 1] - ks[j]);
    const double t0 = j == ra ? -lo : ks[j] - hi, t1 = j == rb ? lo : ks[j + 1] - hi;
    const double hw = 0.5 * (t1 - t0), c = t0 + hw;
    // P(q) - P_hi = base + sj * (t - tj): from the node next to hi, so that no term is larger than the window needs
    double base = 0.0, tj = 0.0;
    if (j > m) {
      base = sm * (ks[m + 1] - hi) + (P[j] - P[m + 1]);
      tj = ks[j] - hi;
    } else if (j < m) {
      base = (P[j + 1] - P[m]) - sm * (hi - ks[m]);
      tj = ks[j + 1] - hi;
    }
    for (int g = 0; g < 8; ++g) {
      const double t = fma(hw, g < 4 ? -x[3 - g] : x[g - 4], c), wt = hw * w[g < 4 ? 3 - g : g - 4];
      const double dP = base + sj * (t - tj), Pq = Phi + dP;
      const double u = t * (2.0 * hi + t), q = hi + t, q2 = q * q;
      const double A = -0.25 * (u - lo2) / lo2 * Plo;
      const double v = (u + lo2) / (2.0 * lo), ww = hi + t + (t * t - lo2) / (2.0 * hi);
      const double R = Plo * (3.0 / 14.0 - 0.5 * lo * v / q2 + (2.0 / 7.0) * v * v / q2) +
                       Phi * (5.0 / 7.0 - 0.5 * ww / hi - 0.5 * hi * ww / q2 + (2.0 / 7.0) * ww * ww / q2);
      const double f = wt * q;
      sg = fma(f, A * dP + R * Pq, sg);
      sd = fma(f, A * A * dP + (2.0 * A + R) * R * Pq, sd);
    }
  }
  const double inv = 1.0 / (2.0 * lo * hi);
  gp = sg * inv;
  g2p = sd * inv;
}

// <G P> and <G^2 P> at (k1, k2) from one redshift's P and moment table; local (pt_local of the caller's q): the local
// branch, whose g2p is <D>.  Window [a, b] = [|k1-k2|, k1+k2]: ends in one region give one piece; otherwise an end
// piece on each side (widths formed as in pbar) and, over whole intervals between them, a difference of table entries.
__device__ __forceinline__ void pt_averages(const double* __restrict__ ks, const double* __restrict__ P,
                                            const DD* __restrict__ T, int nk, double k1, double k2, double P1,
                                            double P2, bool local, double& gp, double& g2p) {
  if (local) {
    pt_averages_local(ks, P, nk, k1, k2, P1, P2, gp, g2p);
    return;
  }
  const double lo = fmin(k1, k2), hi = fmax(k1, k2), a = hi - lo, b = hi + lo;
  int ra, rb;
  const double pa = plin_at(ks, P, nk, a, ra), pb = plin_at(ks, P, nk, b, rb);
  double M[PT_NMOM], m[PT_NMOM];
  if (ra == rb) {
    qmom_piece(a, b, 2.0 * lo, pa, pb, M);
  } else {
    const double xa = ks[ra + 1], xb = ks[rb];
    qmom_piece(a, xa, (xa - hi) + lo, pa, P[ra + 1], M);
    qmom_piece(xb, b, (hi - xb) + lo, P[rb], pb, m);
    for (int n = 0; n < PT_NMOM; ++n) M[n] += m[n];
    if (rb > ra + 1)
      for (int n = 0; n < PT_NMOM; ++n)
        M[n] += n < 2 ? dd_diff(T[(long long)n * nk + ra + 1], T[(long long)n * nk + rb])
                      : dd_diff(T[(long long)n * nk + rb], T[(long long)n * nk + ra + 1]);
  }
  const double d = (k1 - k2) * (k1 + k2), r1 = P1 / (k1 * k1), r2 = P2 / (k2 * k2);
  const double g1 = (-5.0 / 28.0) * (r1 + r2);
  const double g0 = (13.0 / 28.0) * (P1 + P2) - (3.0 / 28.0) * d * (r1 - r2);
  const double gm = -0.25 * d * (P1 - P2) + (d * d / 14.0) * (r1 + r2);
  const double inv = 1.0 / (2.0 * k1 * k2);
  gp = (g1 * M[3] + g0 * M[2] + gm * M[1]) * inv;
  g2p = (g1 * g1 * M[4] + 2.0 * g1 * g0 * M[3] + (g0 * g0 + 2.0 * g1 * gm) * M[2] + 2.0 * g0 * gm * M[1] +
         gm * gm * M[0]) * inv;
}

// F3bar(r) = <F3_sym(k, q, -q)> over the angle, r = q/k:
//   [12/r^2 - 158 + 100 r^2 - 42 r^4 + (3/r^3)(r^2-1)^3 (7r^2+2) ln|(1+r)/(1-r)|] / (3024 r^2).
// The closed form cancels for small and large r: series in r^2 below 0.4 and in 1/r^2 above 2.5 (26 terms each, exact
// rationals rounded once, truncation below 1e-20); -11/378 at r = 1.  tail (r < 0.4 only): F3bar(r) + 1/(18 r^2), the
// small-r series without its leading term (see pt_averages_local).
__device__ double f3bar(double r, bool tail) {
  constexpr double cs[26] = {
      -0.05555555555555555, 0.061375661375661375, -0.042630385487528344, 0.00655076845553036,
      0.000760438855676951, 0.00021354307068592783, 8.38667505334172e-05, 3.975690250200054e-05,
      2.130652285451047e-05, 1.2456624575156199e-05, 7.773259316439517e-06, 5.103490671630971e-06,
      3.4900532521396275e-06, 2.467901851543364e-06, 1.7946309316753127e-06, 1.3364096913719952e-06,
      1.0157257186584305e-06, 7.8582630624582e-07, 6.175121382494654e-07, 4.919865547043248e-07,
      3.9682399296693115e-07, 3.2361537371936314e-07, 2.665494674200016e-07, 2.2153424371892526e-07,
      1.856390527643294e-07, 1.567325245090209e-07};
  constexpr double cl[26] = {
      -0.032275132275132276, 0.006349206349206349, -0.0025195263290501385, -0.0003939622987242035,
      -0.0001289715575429861, -5.567624615243663e-05, -2.8149047756890894e-05, -1.580806534366906e-05,
      -9.57648016471546e-06, -6.145351606190404e-06, -4.126746045481503e-06, -2.875065894934407e-06,
      -2.0649791002709783e-06, -1.521683261458535e-06, -1.146173436372423e-06, -8.798426793730217e-07,
      -6.866684127132244e-07, -5.437793456226636e-07, -4.3623737003527943e-07, -3.540397349651057e-07,
      -2.9033872860683223e-07, -2.40352959565456e-07, -2.0068396195714407e-07, -1.6887706154407393e-07,
      -1.4313317314164382e-07, -1.2211599375569742e-07};
  if (r < 0.4 || r > 2.5) {   // F = sum cs[k] r^(2k-2)  or  sum cl[k] r^(-2k-2)
    const double y = r < 0.4 ? r * r : 1.0 / (r * r);
    const double* c = r < 0.4 ? cs : cl;
    double s = c[25];
    for (int k = 24; k >= (tail ? 1 : 0); --k) s = fma(s, y, c[k]);
    return tail ? s : r < 0.4 ? s / y : s * y;
  }
  if (r == 1.0) return -11.0 / 378.0;
  const double r2 = r * r, L = 2.0 * atanh(r < 1.0 ? r : 1.0 / r), u = r2 - 1.0;
  return (12.0 / r2 - 158.0 + r2 * (100.0 - 42.0 * r2) + (3.0 / (r2 * r)) * (u * u * u) * (7.0 * r2 + 2.0) * L) /
         (3024.0 * r2);
}

// F3[0][i][j] = F3bar(k2/k1), F3[1][i][j] = F3bar(k1/k2): the ratio is the same at every redshift, (l'+1/2)/(l+1/2) in
// projection.  Where pt_local holds, the entry of the small ratio is f3bar's tail (see pt_averages_local).
__global__ void __launch_bounds__(256) trispec4h_f3_kernel(int n1, int n2, const double* __restrict__ q1,
                                                           const double* __restrict__ q2, int proj,
                                                           double* __restrict__ F3) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x, n = (long long)n1 * n2;
  if (e >= n) return;
  const int i = (int)(e / n2), j = (int)(e - (long long)i * n2);
  const double s = proj ? 0.5 : 0.0, x1 = q1[i] + s, x2 = q2[j] + s;
  const bool local = pt_local(x1, x2);
  F3[e] = f3bar(x2 / x1, local && x2 < x1);
  F3[n + e] = f3bar(x1 / x2, local && x1 < x2);
}

// One thread per chunk redshift blockIdx.y, side blockIdx.z (0: k1 legs A, B; 1: k2 legs C, D) and column: P(k) into
// Pk[zl][l] and I1~ of the side's distinct legs into I1[zl][leg][ld] by a mass sum in increasing m.
__global__ void __launch_bounds__(TP_T) trispec_pt_side_kernel(int z0, int nm, int nk, int ldk,
                                                               const double* __restrict__ ks,
                                                               const double* __restrict__ ms,
                                                               const double* __restrict__ nzm,
                                                               const double* __restrict__ bh,
                                                               const double* __restrict__ Pzk, double rho_m0,
                                                               const Legs2h L, int n1, int ld1,
                                                               const double* __restrict__ q1, int n2, int ld2,
                                                               const double* __restrict__ q2,
                                                               const double* __restrict__ chis, double* __restrict__ Pk1,
                                                               double* __restrict__ Pk2, double* __restrict__ I1a,
                                                               double* __restrict__ I1c) {
  const int zl = blockIdx.y, z = z0 + zl, side = blockIdx.z, l = blockIdx.x * TP_T + threadIdx.x;
  const int n = side ? n2 : n1, ld = side ? ld2 : ld1, X = 2 * side, nleg = side ? L.nC1 : L.nA1;
  if (l >= n) return;
  const double q = side ? q2[l] : q1[l], inv_chi = chis ? 1.0 / chis[z] : 0.0;
  int j;
  double f;
  k_locate(ks, nk, chis ? (q + 0.5) * inv_chi : q, j, f);
  (side ? Pk2 : Pk1)[(long long)zl * n + l] = k_lerp(Pzk + (long long)z * nk, j, f);
  double c = 0.0, s0 = 0.0, s1 = 0.0;
  for (int m = 0; m < nm; ++m) {
    const long long i = (long long)z * nm + m, row = i * ldk;
    const double a = ms[m] / rho_m0, w = trapz_weight(ms, m, nm) * nzm[i] * bh[i];
    c = fma(w, a, c);
    s0 = fma(w, (L.matter[X] ? a : 1.0) * k_lerp(L.u[X] + row, j, f), s0);
    if (nleg == 2) s1 = fma(w, (L.matter[X + 1] ? a : 1.0) * k_lerp(L.u[X + 1] + row, j, f), s1);
  }
  double* I1 = (side ? I1c : I1a) + (long long)zl * 2 * ld;
  I1[l] = s0 + (L.matter[X] ? 1.0 - c : 0.0);
  if (nleg == 2) I1[ld + l] = s1 + (L.matter[X + 1] ? 1.0 - c : 0.0);
}

// The side vectors of a pass of zc redshifts: Pk1 [zc][n1p], Pk2 [zc][n2p], I1a [zc][2][n1p], I1c [zc][2][n2p] and the
// moment table [zc][5][nk] in double-double
struct PtSides {
  double *Pk1, *Pk2, *I1a, *I1c;
  DD* tab;
};

static long long pt_sides_doubles(int zc, int nk, int n1, int n2) {
  return (long long)zc * (3LL * (n1 + (n1 & 1)) + 3LL * (n2 + (n2 & 1)) + 2LL * PT_NMOM * nk);
}

static PtSides pt_sides(double* ws, int zc, int nk, int n1, int n2) {
  PtSides s;
  const long long n1p = n1 + (n1 & 1), n2p = n2 + (n2 & 1);
  s.Pk1 = ws;
  s.Pk2 = s.Pk1 + zc * n1p;
  s.I1a = s.Pk2 + zc * n2p;
  s.I1c = s.I1a + 2LL * zc * n1p;
  s.tab = reinterpret_cast<DD*>(s.I1c + 2LL * zc * n2p);
  return s;
}

static int pt_sides_run(int z0, int zn, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                        const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0, const Legs2h& L,
                        int n1, const double* q1_d, int n2, const double* q2_d, const double* chis_d,
                        const PtSides& s, cudaStream_t st) {
  trispec_pt_moments_kernel<<<zn, 256, 0, st>>>(z0, nk, ks_d, Pzk_d, s.tab);
  int rc = check_launch("trispec_pt_moments_kernel");
  if (rc) return rc;
  dim3 g(cdiv(n1 > n2 ? n1 : n2, TP_T), zn, 2);
  trispec_pt_side_kernel<<<g, TP_T, 0, st>>>(z0, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, L, n1,
                                             n1 + (n1 & 1), q1_d, n2, n2 + (n2 & 1), q2_d, chis_d, s.Pk1, s.Pk2,
                                             s.I1a, s.I1c);
  return check_launch("trispec_pt_side_kernel");
}

// One thread per output element (i, j): the chunk's redshifts in increasing z (3D: T3h into out[z][i][j]; projection:
// zeta_z pref_z T3h added onto the previous chunk's value, onto zero when first == 1).
__global__ void __launch_bounds__(256) trispec3h_assemble_kernel(int z0, int zc, int nz, int nk,
                                                                 const double* __restrict__ ks,
                                                                 const double* __restrict__ Pzk, const Plan2h p, const double* __restrict__ q1,
                                                                 const double* __restrict__ q2,
                                                                 const double* __restrict__ zs,
                                                                 const double* __restrict__ chis,
                                                                 const double* __restrict__ pref,
                                                                 const double* __restrict__ O22, const PtSides s,
                                                                 int first, double* __restrict__ out) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x, n = (long long)p.n1 * p.n2;
  if (e >= n) return;
  const int i = (int)(e / p.n2), j = (int)(e - (long long)i * p.n2);
  const long long w22 = p.m2s(), s22 = p.m1s() * w22;
  const long long rB = (p.nA1 == 2 ? p.n1p : 0), cD = (p.nC1 == 2 ? p.n2p : 0);   // B and D rows/columns, also in I1
  const bool local = chis ? pt_local(q1[i] + 0.5, q2[j] + 0.5) : pt_local(q1[i], q2[j]);
  double acc = (chis && !first) ? out[e] : 0.0;
  for (int zl = 0; zl < zc; ++zl) {
    const int z = z0 + zl;
    const double* o22 = O22 + zl * s22;
    const double* Ia = s.I1a + 2LL * zl * p.n1p;
    const double* Ic = s.I1c + 2LL * zl * p.n2p;
    const double I1A = Ia[i], I1B = Ia[rB + i], I1C = Ic[j], I1D = Ic[cD + j];
    const double I2AC = o22[i * w22 + j], I2AD = o22[i * w22 + cD + j];
    const double I2BC = o22[(rB + i) * w22 + j], I2BD = o22[(rB + i) * w22 + cD + j];
    const double inv_chi = chis ? 1.0 / chis[z] : 0.0;
    const double k1 = chis ? (q1[i] + 0.5) * inv_chi : q1[i], k2 = chis ? (q2[j] + 0.5) * inv_chi : q2[j];
    const double P1 = s.Pk1[(long long)zl * p.n1 + i], P2 = s.Pk2[(long long)zl * p.n2 + j];
    double gp, g2p;
    pt_averages(ks, Pzk + (long long)z * nk, s.tab + (long long)zl * PT_NMOM * nk, nk, k1, k2, P1, P2, local, gp,
                g2p);
    const double B = (34.0 / 21.0) * P1 * P2 + 2.0 * gp;
    const double T = B * (I2AC * I1B * I1D + I2AD * I1B * I1C + I2BC * I1A * I1D + I2BD * I1A * I1C);
    if (chis) acc += pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0) * T;
    else out[(long long)z * n + e] = T;
  }
  if (chis) out[e] = acc;
}

// One thread per output element (i, j), all redshifts in increasing z
__global__ void __launch_bounds__(256) trispec4h_assemble_kernel(int nz, int nk, int n1, int n2,
                                                                 const double* __restrict__ ks,
                                                                 const double* __restrict__ Pzk, const Legs2h L,
                                                                 const double* __restrict__ q1,
                                                                 const double* __restrict__ q2,
                                                                 const double* __restrict__ zs,
                                                                 const double* __restrict__ chis,
                                                                 const double* __restrict__ pref, const PtSides s,
                                                                 const double* __restrict__ F3,
                                                                 double* __restrict__ out) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x, n = (long long)n1 * n2;
  if (e >= n) return;
  const int i = (int)(e / n2), j = (int)(e - (long long)i * n2);
  const long long n1p = n1 + (n1 & 1), n2p = n2 + (n2 & 1);
  const long long bB = (L.nA1 == 2 ? n1p : 0), bD = (L.nC1 == 2 ? n2p : 0);
  const double F12 = F3[e], F21 = F3[n + e];
  const bool local = chis ? pt_local(q1[i] + 0.5, q2[j] + 0.5) : pt_local(q1[i], q2[j]);
  double acc = 0.0;
  for (int z = 0; z < nz; ++z) {
    const double* Ia = s.I1a + 2LL * z * n1p;
    const double* Ic = s.I1c + 2LL * z * n2p;
    const double inv_chi = chis ? 1.0 / chis[z] : 0.0;
    const double k1 = chis ? (q1[i] + 0.5) * inv_chi : q1[i], k2 = chis ? (q2[j] + 0.5) * inv_chi : q2[j];
    const double P1 = s.Pk1[(long long)z * n1 + i], P2 = s.Pk2[(long long)z * n2 + j];
    double gp, g2p;
    pt_averages(ks, Pzk + (long long)z * nk, s.tab + (long long)z * PT_NMOM * nk, nk, k1, k2, P1, P2, local, gp,
                g2p);
    const double Tb = 12.0 * P1 * P2 * (P2 * F12 + P1 * F21) + 8.0 * g2p;
    const double T = Ia[i] * Ia[bB + i] * Ic[j] * Ic[bD + j] * Tb;
    if (chis) acc += pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0) * T;
    else out[(long long)z * n + e] = T;
  }
  if (chis) out[e] = acc;
}

// The checks shared by the 3- and 4-halo entry points (those of the 2-halo ones without zchunk); fills L
static int trispec_pt_check(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                            const double* ms_d, const double* nzm_d, const double* bh_d, const double* Pzk_d,
                            const double* const* u_h, const int* kind_h, int n1, const double* q1_d, int n2,
                            const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                            const double* ws_d, const double* out_d, Legs2h& L) {
  TrispecLegs L4;
  const int chk = trispec_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, u_h, kind_h, n1, q1_d, n2, q2_d, zs_d,
                                chis_d, pref_d, ws_d, out_d, L4);
  if (chk) return chk;
  for (int i = 0; i < 4; ++i) {
    L.u[i] = L4.u[i];
    L.matter[i] = L4.matter[i];
  }
  HMV_REQUIRE(bh_d && Pzk_d, "%s: null pointer (bh or Pzk)", who);
  distinct_2h(u_h, kind_h, L.nA1, L.nC1);
  return HMV_OK;
}

// 3-halo workspace: the 2-halo panels P1s P1p P2s P2p and the I2 block O22 of a pass, then its side vectors
static long long trispec3h_ws(const Plan2h& p) {
  return (long long)p.zc * (p.nmp * (p.m1s() + p.n1q + p.m2s() + p.n2q) + p.m1s() * p.m2s()) +
         pt_sides_doubles(p.zc, p.nk, p.n1, p.n2);
}

static long long trispec3h_ws_doubles(int nz, int nm, int nk, int n1, int n2, const double* const* u_h,
                                      const int* kind_h, int zchunk) {
  if (nz <= 0 || nm <= 0 || nk < 2 || n1 <= 0 || n2 <= 0 || !u_h || !kind_h || zchunk < 1 || zchunk > nz) return 0;
  int nA1, nC1;
  distinct_2h(u_h, kind_h, nA1, nC1);
  return trispec3h_ws(plan_2h(nm, nk, n1, n2, nA1, nC1, zchunk));
}

static int trispec3h_run(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                         const double* ms_d, const double* nzm_d, const double* bh_d, const double* Pzk_d,
                         double rho_m0, const double* const* u_h, const int* kind_h, int n1, const double* q1_d, int n2,
                         const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                         int zchunk, double* ws_d, double* out_d, void* stream) {
  Legs2h L;
  const int chk = trispec_pt_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, u_h, kind_h, n1, q1_d,
                                   n2, q2_d, zs_d, chis_d, pref_d, ws_d, out_d, L);
  if (chk) return chk;
  HMV_REQUIRE(zchunk >= 1 && zchunk <= nz, "%s: zchunk must lie in [1, nz] (zchunk=%d nz=%d)", who, zchunk, nz);
  const Plan2h full = plan_2h(nm, nk, n1, n2, L.nA1, L.nC1, zchunk);
  const long long zc = zchunk;
  double* P1s = ws_d;
  double* P1p = P1s + zc * full.nmp * full.m1s();
  double* P2s = P1p + zc * full.nmp * full.n1q;
  double* P2p = P2s + zc * full.nmp * full.m2s();
  double* O22 = P2p + zc * full.nmp * full.n2q;
  const PtSides s = pt_sides(O22 + zc * full.m1s() * full.m2s(), zchunk, nk, n1, n2);
  cudaStream_t st = (cudaStream_t)stream;
  const double* chis = proj ? chis_d : nullptr;
  const long long nout = (long long)n1 * n2;
  for (int z0 = 0; z0 < nz; z0 += zchunk) {
    const int zn = min(zchunk, nz - z0);
    Plan2h p = full;
    p.zc = zn;
    int rc = pt_sides_run(z0, zn, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, L, n1, q1_d, n2, q2_d, chis, s,
                          st);
    if (rc) return rc;
    // The 2-halo panel kernel, unchanged: of its outputs only P1s and P2s are read here.  Its P(k1), P(k2) go to the
    // side kernel's Pk1, Pk2, rewriting them with the same bits (the same k_locate and k_lerp); P1p and P2p are unused.
    dim3 pg(cdiv(p.n1q > p.n2q ? p.n1q : p.n2q, TP_T), zn, cdiv(p.nmp, TP_MROWS));
    trispec2h_panel_kernel<<<pg, TP_T, 0, st>>>(z0, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, L, p, q1_d,
                                                q2_d, chis, P1s, P1p, P2s, P2p, s.Pk1, s.Pk2);
    rc = check_launch("trispec2h_panel_kernel");
    if (rc) return rc;
    rc = trispec_product(who, trispec_plan(false, zn, nm, (int)p.m1s(), (int)p.m2s()), (int)p.m1s(), P1s, P2s, O22,
                         st);
    if (rc) return rc;
    trispec3h_assemble_kernel<<<cdiv(nout, 256), 256, 0, st>>>(z0, zn, nz, nk, ks_d, Pzk_d, p, q1_d, q2_d, zs_d, chis,
                                                               pref_d, O22, s, z0 == 0, out_d);
    rc = check_launch("trispec3h_assemble_kernel");
    if (rc) return rc;
  }
  return HMV_OK;
}

static long long trispec4h_ws_doubles(int nz, int nk, int n1, int n2) {
  if (nz <= 0 || nk < 2 || n1 <= 0 || n2 <= 0) return 0;
  return pt_sides_doubles(nz, nk, n1, n2) + 2LL * n1 * n2;
}

static int trispec4h_run(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                         const double* ms_d, const double* nzm_d, const double* bh_d, const double* Pzk_d,
                         double rho_m0, const double* const* u_h, const int* kind_h, int n1, const double* q1_d, int n2,
                         const double* q2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                         double* ws_d, double* out_d, void* stream) {
  Legs2h L;
  const int chk = trispec_pt_check(who, proj, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, u_h, kind_h, n1, q1_d,
                                   n2, q2_d, zs_d, chis_d, pref_d, ws_d, out_d, L);
  if (chk) return chk;
  const PtSides s = pt_sides(ws_d, nz, nk, n1, n2);
  double* F3 = ws_d + pt_sides_doubles(nz, nk, n1, n2);
  cudaStream_t st = (cudaStream_t)stream;
  const double* chis = proj ? chis_d : nullptr;
  const long long nout = (long long)n1 * n2;
  int rc = pt_sides_run(0, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, L, n1, q1_d, n2, q2_d, chis, s,
                        st);
  if (rc) return rc;
  trispec4h_f3_kernel<<<cdiv(nout, 256), 256, 0, st>>>(n1, n2, q1_d, q2_d, proj, F3);
  rc = check_launch("trispec4h_f3_kernel");
  if (rc) return rc;
  trispec4h_assemble_kernel<<<cdiv(nout, 256), 256, 0, st>>>(nz, nk, n1, n2, ks_d, Pzk_d, L, q1_d, q2_d, zs_d, chis,
                                                             pref_d, s, F3, out_d);
  return check_launch("trispec4h_assemble_kernel");
}

// ---- super-sample covariance (DESIGN.md §4.5) -------------------------------------------------------------------------
//   sigma_b^2(z)        = sum_j kw_j P[z][j] W(k_j R_z)^2,  W(x) = 2 J1(x)/x, kw_j = s_j k_j/(2 pi) from the caller
//   Cov^{AB,CD}(l,l')   = sum_z zeta_z pref_z R^{AB}((l+1/2)/chi_z, z) R^{CD}((l'+1/2)/chi_z, z)
// with pref = H^3 W_A W_B W_C W_D sigma_b^2/chi^4 from the caller and R linear in k on ks, clamped to its ends.  The
// covariance is the trispectrum's contraction with K = z: one panel row per redshift.

// 2 J1(x)/x, the Fourier transform of a disc; its Taylor series near x = 0 (error below 1e-16 for |x| < 1e-2)
__device__ __forceinline__ double disc_window(double x) {
  if (fabs(x) < 1e-2) {
    const double x2 = x * x;
    return fma(x2, fma(x2, 1.0 / 192.0, -1.0 / 8.0), 1.0);
  }
  return 2.0 * j1(x) / x;
}

// one CTA per redshift; a fixed-order block reduction, so repeated calls give identical results
__global__ void __launch_bounds__(256) sigma_b2_kernel(int nks, const double* __restrict__ ks,
                                                       const double* __restrict__ kw, const double* __restrict__ P,
                                                       const double* __restrict__ R, double* __restrict__ out) {
  __shared__ double red[32];
  const int z = blockIdx.x;
  const double Rz = R[z];
  const double* Pz = P + (long long)z * nks;
  double s = 0.0;
  for (int j = threadIdx.x; j < nks; j += blockDim.x) {
    const double W = disc_window(ks[j] * Rz);
    s = fma(kw[j] * Pz[j], W * W, s);
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) out[z] = s;
}

// P1[z][l] = zeta_z pref_z R^{AB}(z, (l+1/2)/chi_z), P2[z][l'] = R^{CD}(z, (l'+1/2)/chi_z); columns in [n, ld) are zero.
// One thread per column and redshift: one interval search each.
__global__ void __launch_bounds__(TP_T) ssc_panel_kernel(int nz, int nk, const double* __restrict__ ks,
                                                         const double* __restrict__ rAB, const double* __restrict__ rCD,
                                                         int n1, int ld1, const double* __restrict__ l1, int n2,
                                                         int ld2, const double* __restrict__ l2,
                                                         const double* __restrict__ zs, const double* __restrict__ chis,
                                                         const double* __restrict__ pref, double* __restrict__ P1,
                                                         double* __restrict__ P2) {
  const int z = blockIdx.y, l = blockIdx.x * TP_T + threadIdx.x;
  const double inv_chi = 1.0 / chis[z];
  int j;
  double f;
  if (l < ld1) {
    double v = 0.0;
    if (l < n1) {
      k_locate(ks, nk, (l1[l] + 0.5) * inv_chi, j, f);
      v = pref[z] * (nz > 1 ? trapz_weight(zs, z, nz) : 1.0) * k_lerp(rAB + (long long)z * nk, j, f);
    }
    P1[(long long)z * ld1 + l] = v;
  }
  if (l < ld2) {
    double v = 0.0;
    if (l < n2) {
      k_locate(ks, nk, (l2[l] + 0.5) * inv_chi, j, f);
      v = k_lerp(rCD + (long long)z * nk, j, f);
    }
    P2[(long long)z * ld2 + l] = v;
  }
}

static TrispecPlan ssc_plan(int nz, int n1, int n2) { return split_k(base_plan(nz, 1, n1, n2), n1); }

}  // namespace hmv

using namespace hmv;

extern "C" long long hmv_trispec_1h_ws_doubles(int nz, int nm, int nk1, int nk2) {
  return trispec_ws_doubles(false, nz, nm, nk1, nk2);
}

extern "C" int hmv_trispec_1h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                              const double* nzm_d, double rho_m0, const double* const* u_h, const int* kind_h, int nk1,
                              const double* k1_d, int nk2, const double* k2_d, double* ws_d, double* out_d,
                              void* stream) {
  return trispec_run("hmv_trispec_1h", false, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, u_h, kind_h, nk1, k1_d, nk2,
                     k2_d, nullptr, nullptr, nullptr, ws_d, out_d, stream);
}

extern "C" long long hmv_cl_cov_1h_ws_doubles(int nz, int nm, int nl1, int nl2) {
  return trispec_ws_doubles(true, nz, nm, nl1, nl2);
}

extern "C" int hmv_cl_cov_1h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                             const double* nzm_d, double rho_m0, const double* const* u_h, const int* kind_h, int nl1,
                             const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                             const double* chis_d, const double* pref_d, double* ws_d, double* out_d, void* stream) {
  return trispec_run("hmv_cl_cov_1h", true, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, u_h, kind_h, nl1, ells1_d, nl2,
                     ells2_d, zs_d, chis_d, pref_d, ws_d, out_d, stream);
}

extern "C" long long hmv_trispec_1h_tracers_ws_doubles(int nz, int nm, int nk1, int nk2, const hmv_tracer* legs_h) {
  return tracer_ws_doubles(false, nz, nm, nk1, nk2, legs_h);
}

extern "C" int hmv_trispec_1h_tracers(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                                      const double* nzm_d, double rho_m0, const hmv_tracer* legs_h, int nk1,
                                      const double* k1_d, int nk2, const double* k2_d, double* ws_d, double* out_d,
                                      void* stream) {
  return tracer_run("hmv_trispec_1h_tracers", false, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, legs_h, nk1, k1_d,
                    nk2, k2_d, nullptr, nullptr, nullptr, ws_d, out_d, stream);
}

extern "C" long long hmv_cl_cov_1h_tracers_ws_doubles(int nz, int nm, int nl1, int nl2, const hmv_tracer* legs_h) {
  return tracer_ws_doubles(true, nz, nm, nl1, nl2, legs_h);
}

extern "C" int hmv_cl_cov_1h_tracers(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                                     const double* nzm_d, double rho_m0, const hmv_tracer* legs_h, int nl1,
                                     const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                                     const double* chis_d, const double* pref_d, double* ws_d, double* out_d,
                                     void* stream) {
  return tracer_run("hmv_cl_cov_1h_tracers", true, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, rho_m0, legs_h, nl1, ells1_d,
                    nl2, ells2_d, zs_d, chis_d, pref_d, ws_d, out_d, stream);
}

extern "C" long long hmv_trispec_2h_ws_doubles(int nz, int nm, int nk, int nk1, int nk2, const double* const* u_h,
                                                const int* kind_h, int zchunk) {
  return trispec2h_ws_doubles(nz, nm, nk, nk1, nk2, u_h, kind_h, zchunk);
}

extern "C" int hmv_trispec_2h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                              const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                              const double* const* u_h, const int* kind_h, int nk1, const double* k1_d, int nk2,
                              const double* k2_d, int zchunk, double* ws_d, double* out_d, void* stream) {
  return trispec2h_run("hmv_trispec_2h", false, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nk1, k1_d, nk2, k2_d, nullptr, nullptr, nullptr, zchunk, ws_d, out_d, stream);
}

extern "C" long long hmv_cl_cov_2h_ws_doubles(int nz, int nm, int nk, int nl1, int nl2, const double* const* u_h,
                                               const int* kind_h, int zchunk) {
  return trispec2h_ws_doubles(nz, nm, nk, nl1, nl2, u_h, kind_h, zchunk);
}

extern "C" int hmv_cl_cov_2h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                             const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                             const double* const* u_h, const int* kind_h, int nl1, const double* ells1_d, int nl2,
                             const double* ells2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                             int zchunk, double* ws_d, double* out_d, void* stream) {
  return trispec2h_run("hmv_cl_cov_2h", true, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nl1, ells1_d, nl2, ells2_d, zs_d, chis_d, pref_d, zchunk, ws_d, out_d, stream);
}

extern "C" long long hmv_trispec_3h_ws_doubles(int nz, int nm, int nk, int nk1, int nk2, const double* const* u_h,
                                                const int* kind_h, int zchunk) {
  return trispec3h_ws_doubles(nz, nm, nk, nk1, nk2, u_h, kind_h, zchunk);
}

extern "C" int hmv_trispec_3h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                              const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                              const double* const* u_h, const int* kind_h, int nk1, const double* k1_d, int nk2,
                              const double* k2_d, int zchunk, double* ws_d, double* out_d, void* stream) {
  return trispec3h_run("hmv_trispec_3h", false, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nk1, k1_d, nk2, k2_d, nullptr, nullptr, nullptr, zchunk, ws_d, out_d, stream);
}

extern "C" long long hmv_cl_cov_3h_ws_doubles(int nz, int nm, int nk, int nl1, int nl2, const double* const* u_h,
                                               const int* kind_h, int zchunk) {
  return trispec3h_ws_doubles(nz, nm, nk, nl1, nl2, u_h, kind_h, zchunk);
}

extern "C" int hmv_cl_cov_3h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                             const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                             const double* const* u_h, const int* kind_h, int nl1, const double* ells1_d, int nl2,
                             const double* ells2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                             int zchunk, double* ws_d, double* out_d, void* stream) {
  return trispec3h_run("hmv_cl_cov_3h", true, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nl1, ells1_d, nl2, ells2_d, zs_d, chis_d, pref_d, zchunk, ws_d, out_d, stream);
}

extern "C" long long hmv_trispec_4h_ws_doubles(int nz, int nk, int nk1, int nk2) {
  return trispec4h_ws_doubles(nz, nk, nk1, nk2);
}

extern "C" int hmv_trispec_4h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                              const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                              const double* const* u_h, const int* kind_h, int nk1, const double* k1_d, int nk2,
                              const double* k2_d, double* ws_d, double* out_d, void* stream) {
  return trispec4h_run("hmv_trispec_4h", false, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nk1, k1_d, nk2, k2_d, nullptr, nullptr, nullptr, ws_d, out_d, stream);
}

extern "C" long long hmv_cl_cov_4h_ws_doubles(int nz, int nk, int nl1, int nl2) {
  return trispec4h_ws_doubles(nz, nk, nl1, nl2);
}

extern "C" int hmv_cl_cov_4h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                             const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                             const double* const* u_h, const int* kind_h, int nl1, const double* ells1_d, int nl2,
                             const double* ells2_d, const double* zs_d, const double* chis_d, const double* pref_d,
                             double* ws_d, double* out_d, void* stream) {
  return trispec4h_run("hmv_cl_cov_4h", true, nz, nm, nk, ldk, ks_d, ms_d, nzm_d, bh_d, Pzk_d, rho_m0, u_h, kind_h,
                       nl1, ells1_d, nl2, ells2_d, zs_d, chis_d, pref_d, ws_d, out_d, stream);
}

extern "C" int hmv_sigma_b2(int nz, int nks, const double* ks_d, const double* kw_d, const double* P_d,
                            const double* R_d, double* out_d, void* stream) {
  HMV_REQUIRE(nz >= 1 && nks >= 1, "hmv_sigma_b2: sizes must be >= 1 (nz=%d nks=%d)", nz, nks);
  HMV_REQUIRE(ks_d && kw_d && P_d && R_d && out_d, "hmv_sigma_b2: null pointer");
  sigma_b2_kernel<<<nz, 256, 0, (cudaStream_t)stream>>>(nks, ks_d, kw_d, P_d, R_d, out_d);
  return check_launch("sigma_b2_kernel");
}

extern "C" long long hmv_cl_cov_ssc_ws_doubles(int nz, int nl1, int nl2) {
  if (nz <= 0 || nl1 <= 0 || nl2 <= 0) return 0;
  return trispec_ws(ssc_plan(nz, nl1, nl2), nl1);
}

extern "C" int hmv_cl_cov_ssc(int nz, int nk, const double* ks_d, const double* rAB_d, const double* rCD_d, int nl1,
                              const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                              const double* chis_d, const double* pref_d, double* ws_d, double* out_d, void* stream) {
  const char* who = "hmv_cl_cov_ssc";
  HMV_REQUIRE(nz >= 1 && nk >= 2 && nl1 >= 1 && nl2 >= 1,
              "%s: sizes must be >= 1 and nk >= 2 (nz=%d nk=%d n1=%d n2=%d)", who, nz, nk, nl1, nl2);
  HMV_REQUIRE(ks_d && rAB_d && rCD_d && ells1_d && ells2_d && ws_d && out_d, "%s: null pointer", who);
  HMV_REQUIRE(zs_d && chis_d && pref_d, "%s: null pointer (zs, chis or pref)", who);
  HMV_REQUIRE(((size_t)ws_d & 15) == 0, "%s: workspace must be 16-byte aligned", who);
  if (nz > 65535) return fail(HMV_E_LIMIT, "%s: nz=%d exceeds 65535 (grid y of the panel kernel)", who, nz);
  const TrispecPlan p = ssc_plan(nz, nl1, nl2);
  double* P1 = ws_d;
  double* P2 = P1 + p.K * p.ld1;
  double* part = P2 + p.K * p.ld2;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 pg(cdiv(p.ld1 > p.ld2 ? p.ld1 : p.ld2, TP_T), nz);
  ssc_panel_kernel<<<pg, TP_T, 0, st>>>(nz, nk, ks_d, rAB_d, rCD_d, nl1, p.ld1, ells1_d, nl2, p.ld2, ells2_d, zs_d,
                                        chis_d, pref_d, P1, P2);
  const int rc = check_launch("ssc_panel_kernel");
  if (rc) return rc;
  return trispec_contract(who, p, nl1, nl2, P1, P2, part, out_d, st);
}
