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
// for the trispectrum.  A last kernel sums the splits in a fixed order and drops the padding column.
// The super-sample covariance (DESIGN.md §4.5) reuses the projection with K = z; sigma_b^2 of a disc is here too.
// The 2-halo trispectrum and its covariance (DESIGN.md §4.6) run the trispectrum's batched product three times per pass
// of redshifts and combine the blocks per (z, k1, k2) with P_lin and its angle average; see the section below.
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
  int nmp, ld1, ld2;    // mass rows and panel widths, padded to even
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

static TrispecPlan trispec_plan(bool proj, int nz, int nm, int n1, int n2) {
  TrispecPlan p = base_plan(nz, nm + (nm & 1), n1, n2);
  if (!proj) {                       // one batch item per redshift: its K range is its nmp mass rows
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

static long long trispec_ws_doubles(bool proj, int nz, int nm, int n1, int n2) {
  if (nz <= 0 || nm <= 0 || n1 <= 0 || n2 <= 0) return 0;
  return trispec_ws(trispec_plan(proj, nz, nm, n1, n2), n1);
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

// The argument checks of every trispectrum entry point (1- and 2-halo), made before any launch; fills L.
static int trispec_check(const char* who, bool proj, int nz, int nm, int nk, int ldk, const double* ks_d,
                         const double* ms_d, const double* nzm_d, const double* const* u_h, const int* kind_h, int n1,
                         const double* q1_d, int n2, const double* q2_d, const double* zs_d, const double* chis_d,
                         const double* pref_d, const double* ws_d, const double* out_d, TrispecLegs& L) {
  HMV_REQUIRE(nz >= 1 && nm >= 1 && nk >= 2 && n1 >= 1 && n2 >= 1,
              "%s: sizes must be >= 1 and nk >= 2 (nz=%d nm=%d nk=%d n1=%d n2=%d)", who, nz, nm, nk, n1, n2);
  HMV_REQUIRE(ldk >= nk && (ldk & 1) == 0, "%s: ldk must be even and >= nk (ldk=%d nk=%d)", who, ldk, nk);
  HMV_REQUIRE(ks_d && ms_d && nzm_d && u_h && kind_h && q1_d && q2_d && ws_d && out_d, "%s: null pointer", who);
  HMV_REQUIRE(!proj || (zs_d && chis_d && pref_d), "%s: null pointer (zs, chis or pref)", who);
  for (int i = 0; i < 4; ++i) {
    HMV_REQUIRE(u_h[i], "%s: null pointer (cube %d)", who, i);
    HMV_REQUIRE(kind_h[i] == 0 || kind_h[i] == 2, "%s: cube %d: kind %d is neither 0 (matter) nor 2 (pressure)", who, i,
                kind_h[i]);
    HMV_REQUIRE(((size_t)u_h[i] & 15) == 0, "%s: cube %d must be 16-byte aligned", who, i);
    L.u[i] = u_h[i];
    L.matter[i] = kind_h[i] == 0;
  }
  HMV_REQUIRE(((size_t)ws_d & 15) == 0, "%s: workspace must be 16-byte aligned", who);
  if (nz > 65535) return fail(HMV_E_LIMIT, "%s: nz=%d exceeds 65535 (grid y of the panel kernel)", who, nz);
  const long long K = (long long)nz * (nm + (nm & 1));
  if (K > (1LL << 30))
    return fail(HMV_E_LIMIT, "%s: nz * nm = %lld exceeds 2^30 (32-bit k index of the contraction)", who, K);
  return HMV_OK;
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

// ---- 2-halo trispectrum (DESIGN.md §4.6) -------------------------------------------------------------------------------
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
