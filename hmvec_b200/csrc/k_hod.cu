// k_hod.cu -- K4: HOD occupations (table-inverse SHMR, erf central, power-law satellites) and their mass
// integrals; K4b: the mthresh <-> ngal bisection.  Reference arithmetic: hmvec.py:634-731 (SHMR, Nc, Ns,
// moments), :462-466, :936-957 (ngal, bg), utils.py:9-42 (vectorized_bisection_search), hmvec.py:415-433.
// One CTA per redshift; the 4000-point SHMR table, the inverse-SHMR of the mass grid and the trapezoid x n(M)
// weights are staged in shared memory once and re-used by every bisection iteration.
#include "common.cuh"

namespace hmv {

constexpr int HT = 1024;   // one CTA per redshift: the bisection is latency-bound, so use the whole CTA width
constexpr int NTAB = 4000;  // hmvec.py:641

struct HodP { double sig, alphasat, Bsat, betasat, Bcut, betacut, Msat_ov, Mcut_ov; };

struct Shmr { double lM1, lMs0, beta, gamma, delta; };

__device__ __forceinline__ Shmr shmr_params(double z) {
  // Leauthaud-style SHMR, two redshift branches (hmvec.py:668-694); every parameter is p0 + pa (a-1)
  const double am1 = 1.0 / (1.0 + z) - 1.0;
  Shmr s;
  if (z <= 0.8) {
    s.lMs0 = 10.72 + 0.55 * am1; s.lM1 = 12.35 + 0.28 * am1; s.beta = 0.44 + 0.18 * am1;
    s.gamma = 1.56 + 2.51 * am1; s.delta = 0.57 + 0.17 * am1;
  } else {
    s.lMs0 = 11.09 + 0.56 * am1; s.lM1 = 12.27 + (-0.84) * am1; s.beta = 0.65 + 0.31 * am1;
    s.gamma = 1.12 + (-0.53) * am1; s.delta = 0.56 + (-0.12) * am1;
  }
  return s;
}

__device__ __forceinline__ double shmr_log10mh(const Shmr& s, double L) {  // hmvec.py:655
  const double d = L - s.lMs0;
  return -0.5 + s.lM1 + s.beta * d + exp10(s.delta * d) / (1.0 + exp10(-s.gamma * d));
}

// np.interp(x, tab, L_i) with clamped ends (hmvec.py:645); tab is increasing
__device__ __forceinline__ double shmr_inverse(const double* tab, double x) {
  const double Lstep = 36.0 / (NTAB - 1);
  if (x <= tab[0]) return -18.0;
  if (x >= tab[NTAB - 1]) return 18.0;
  int lo = 0, hi = NTAB - 1;  // tab[lo] <= x < tab[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (tab[mid] <= x) lo = mid; else hi = mid;
  }
  const double L0 = -18.0 + lo * Lstep;
  const double L1 = (lo + 1 == NTAB - 1) ? 18.0 : -18.0 + (lo + 1) * Lstep;
  const double slope = (L1 - L0) / (tab[lo + 1] - tab[lo]);
  return slope * (x - tab[lo]) + L0;
}

struct SatScale { double Msat, Mcut; };

__device__ __forceinline__ SatScale sat_scales(const Shmr& s, const HodP& hp, double lth) {
  const double mth = shmr_log10mh(s, lth);  // hmvec.py:711
  SatScale r;
  r.Msat = hp.Msat_ov > 0 ? hp.Msat_ov : 1e12 * hp.Bsat * exp10((mth - 12.0) * hp.betasat);  // :706,712
  r.Mcut = hp.Mcut_ov > 0 ? hp.Mcut_ov : 1e12 * hp.Bcut * exp10((mth - 12.0) * hp.betacut);
  return r;
}

__device__ __forceinline__ void occupations(double M, double lmstar, double lth, const HodP& hp, const SatScale& sc,
                                            double& Nc, double& Ns) {
  Nc = 0.5 * (1.0 - erf((lth - lmstar) / (M_SQRT2 * hp.sig)));               // hmvec.py:701-703
  const double r = M / sc.Msat;
  Ns = Nc * (hp.alphasat == 1.0 ? r : pow(r, hp.alphasat)) * exp(-sc.Mcut / M);   // hmvec.py:716
}

// shared staging used by both kernels: tab[NTAB], lmstar[nm], wn[nm] = trapz_weight * nzm
__device__ __forceinline__ void stage(int z, int nm, const double* __restrict__ ms, const double* __restrict__ nzm,
                                      const Shmr& s, double* tab, double* lmstar, double* wn) {
  const double Lstep = 36.0 / (NTAB - 1);
  for (int i = threadIdx.x; i < NTAB; i += blockDim.x)
    tab[i] = shmr_log10mh(s, (i == NTAB - 1) ? 18.0 : -18.0 + i * Lstep);
  __syncthreads();
  for (int m = threadIdx.x; m < nm; m += blockDim.x) {
    lmstar[m] = shmr_inverse(tab, log10(ms[m]));
    wn[m] = trapz_weight(ms, m, nm) * nzm[(long long)z * nm + m];
  }
  __syncthreads();
}

__global__ void __launch_bounds__(HT) hod_kernel(int nm, const double* __restrict__ zs, const double* __restrict__ ms,
                                                  const double* __restrict__ lth_in, HodP hp, int corr,
                                                  const double* __restrict__ nzm, const double* __restrict__ bh,
                                                  double* __restrict__ Nc_o, double* __restrict__ Ns_o,
                                                  double* __restrict__ NsNsm1_o, double* __restrict__ NcNs_o,
                                                  double* __restrict__ ngal_o, double* __restrict__ bg_o) {
  extern __shared__ double sm[];
  double *tab = sm, *lmstar = tab + NTAB, *wn = lmstar + nm, *red = wn + nm;
  const int z = blockIdx.x;
  const Shmr s = shmr_params(zs[z]);
  stage(z, nm, ms, nzm, s, tab, lmstar, wn);
  const double lth = lth_in[z];
  const SatScale sc = sat_scales(s, hp, lth);
  double sn = 0.0, sb = 0.0;
  for (int m = threadIdx.x; m < nm; m += blockDim.x) {
    const long long i = (long long)z * nm + m;
    double Nc, Ns;
    occupations(ms[m], lmstar[m], lth, hp, sc, Nc, Ns);
    double nn, cn;
    if (corr == 0) {               // "max": hmvec.py:720-723, 728-729
      nn = (fabs(Nc) <= 1e-8) ? 0.0 : Ns * Ns / Nc;   // np.isclose(Nc, 0) -> 0
      cn = Ns;
    } else {                       // "min": hmvec.py:724-725, 730-731
      nn = Ns * Ns;
      cn = Ns * Nc;
    }
    Nc_o[i] = Nc; Ns_o[i] = Ns; NsNsm1_o[i] = nn; NcNs_o[i] = cn;
    const double t = wn[m] * (Nc + Ns);
    sn += t;
    sb = fma(t, bh[i], sb);
  }
  sn = block_sum(sn, red);
  sb = block_sum(sb, red);
  if (threadIdx.x == 0) {
    ngal_o[z] = sn;               // hmvec.py:956-957
    bg_o[z] = sb / sn;            // hmvec.py:464-466
  }
}

// Every z bisects for HMV_BISECT_MAXIT iterations; ys[z][it] = midpoint, bit `it` of pass[z] = |err|<=rtol.
__global__ void __launch_bounds__(HT) hod_bisect_kernel(int nm, const double* __restrict__ zs,
                                                         const double* __restrict__ ms,
                                                         const double* __restrict__ nzm,
                                                         const double* __restrict__ target, HodP hp, double ylo,
                                                         double yhi, double rtol, int it0, int it1,
                                                         const unsigned long long* __restrict__ gmask,
                                                         double* __restrict__ ys, unsigned long long* __restrict__ pass,
                                                         double* __restrict__ ylr) {
  extern __shared__ double sm[];
  double *tab = sm, *lmstar = tab + NTAB, *wn = lmstar + nm, *red = wn + nm;
  const int z = blockIdx.x;
  // a continuation round has nothing to do once every redshift (of every rank) has converged in an earlier round
  if (it0 > 0 && gmask[0] != 0ull) return;
  const Shmr s = shmr_params(zs[z]);
  stage(z, nm, ms, nzm, s, tab, lmstar, wn);
  const double x = target[z];
  double yl = ylo, yr = yhi;
  unsigned long long mask = 0ull;
  if (it0 > 0) { yl = ylr[2 * z]; yr = ylr[2 * z + 1]; mask = pass[z]; }
  for (int it = it0; it < it1; ++it) {
    const double y = 0.5 * (yl + yr);                       // utils.py:27
    const SatScale sc = sat_scales(s, hp, y);
    double sn = 0.0;
    for (int m = threadIdx.x; m < nm; m += blockDim.x) {
      double Nc, Ns;
      occupations(ms[m], lmstar[m], y, hp, sc, Nc, Ns);
      sn = fma(wn[m], Nc + Ns, sn);
    }
    sn = block_sum(sn, red);
    const double err = (sn - x) / x;                        // utils.py:29
    if (err > 0) yl = y; else if (err <= 0) yr = y;         // "decreasing", utils.py:30-32
    if (!(fabs(err) > rtol)) mask |= (1ull << it);          // utils.py:26
    if (threadIdx.x == 0) ys[(long long)z * HMV_BISECT_MAXIT + it] = y;
  }
  if (threadIdx.x == 0) { pass[z] = mask; ylr[2 * z] = yl; ylr[2 * z + 1] = yr; }
}

// AND of the per-z pass masks of this device's redshifts -> mask[0] (bit it = every local z passes at iteration it)
__global__ void hod_mask_reduce_kernel(int nz, const unsigned long long* __restrict__ pass,
                                       unsigned long long* __restrict__ mask) {
  __shared__ unsigned long long all;
  if (threadIdx.x == 0) all = ~0ull;
  __syncthreads();
  unsigned long long mine = ~0ull;
  for (int z = threadIdx.x; z < nz; z += blockDim.x) mine &= pass[z];
  atomicAnd(&all, mine);
  __syncthreads();
  if (threadIdx.x == 0) mask[0] = all;
}

// mask[0] is the AND over ALL redshifts (all ranks when z is sharded): pick the first iteration every z passes
__global__ void hod_bisect_pick_kernel(int nz, const double* __restrict__ ys,
                                       const unsigned long long* __restrict__ mask, double A,
                                       double* __restrict__ lth_out, int* __restrict__ iters) {
  const unsigned long long a = mask[0];
  const int T = a ? (__ffsll((long long)a) - 1) : -1;
  if (blockIdx.x == 0 && threadIdx.x == 0) *iters = T + 1;
  const int use = T >= 0 ? T : HMV_BISECT_MAXIT - 1;
  for (int z = blockIdx.x * blockDim.x + threadIdx.x; z < nz; z += gridDim.x * blockDim.x)
    lth_out[z] = ys[(long long)z * HMV_BISECT_MAXIT + use] * A;  // hmvec.py:433
}

static int hod_smem(int nm, size_t* bytes) {
  *bytes = ((size_t)NTAB + 2 * (size_t)nm + 32) * sizeof(double);
  if (*bytes > 200 * 1024)
    return fail(HMV_E_LIMIT, "HOD kernels stage %d + 2*nm + 32 doubles (at most 200 KiB) in shared memory: nm=%d too "
                "large (max 10784)", NTAB, nm);
  return HMV_OK;
}

static HodP load_hodp(const double* h) {
  HodP p;
  p.sig = h[0]; p.alphasat = h[1]; p.Bsat = h[2]; p.betasat = h[3]; p.Bcut = h[4]; p.betacut = h[5];
  p.Msat_ov = h[6]; p.Mcut_ov = h[7];
  return p;
}

}  // namespace hmv
using namespace hmv;

extern "C" int hmv_hod(int nz, int nm, const double* zs_d, const double* ms_d, const double* log10mthresh_d,
                       const double* hodp_h, int corr, const double* nzm_d, const double* bh_d, double* Nc_d,
                       double* Ns_d, double* NsNsm1_d, double* NcNs_d, double* ngal_d, double* bg_d, void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2, "hmv_hod: need nz>0, nm>=2");
  HMV_REQUIRE(corr == 0 || corr == 1, "hmv_hod: corr must be 0 (max) or 1 (min)");
  HMV_REQUIRE(zs_d && ms_d && log10mthresh_d && hodp_h && nzm_d && bh_d && Nc_d && Ns_d && NsNsm1_d && NcNs_d &&
                  ngal_d && bg_d, "hmv_hod: null pointer");
  size_t smem;
  int rc = hod_smem(nm, &smem);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(hod_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "hod_kernel smem opt-in: %s", cudaGetErrorString(e));
  hod_kernel<<<nz, HT, smem, (cudaStream_t)stream>>>(nm, zs_d, ms_d, log10mthresh_d, load_hodp(hodp_h), corr, nzm_d,
                                                     bh_d, Nc_d, Ns_d, NsNsm1_d, NcNs_d, ngal_d, bg_d);
  return check_launch("hod_kernel");
}

extern "C" int hmv_hod_bisect(int nz, int nm, const double* zs_d, const double* ms_d, const double* nzm_d,
                              const double* ngal_target_d, const double* hodp_h, double ylo, double yhi, double rtol,
                              int it_begin, int it_end, double* ws_d, unsigned long long* mask_d, void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2, "hmv_hod_bisect: need nz>0, nm>=2");
  HMV_REQUIRE(0 <= it_begin && it_begin < it_end && it_end <= HMV_BISECT_MAXIT,
              "hmv_hod_bisect: iteration range [%d,%d) must lie in [0,%d]", it_begin, it_end, HMV_BISECT_MAXIT);
  HMV_REQUIRE(zs_d && ms_d && nzm_d && ngal_target_d && hodp_h && ws_d && mask_d, "hmv_hod_bisect: null pointer");
  size_t smem;
  int rc = hod_smem(nm, &smem);
  if (rc) return rc;
  cudaError_t e = cudaFuncSetAttribute(hod_bisect_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "hod_bisect_kernel smem opt-in: %s", cudaGetErrorString(e));
  double* ys = ws_d;
  unsigned long long* pass = (unsigned long long*)(ws_d + (size_t)nz * HMV_BISECT_MAXIT);
  cudaStream_t st = (cudaStream_t)stream;
  double* ylr = ws_d + (size_t)nz * (HMV_BISECT_MAXIT + 1);
  hod_bisect_kernel<<<nz, HT, smem, st>>>(nm, zs_d, ms_d, nzm_d, ngal_target_d, load_hodp(hodp_h), ylo, yhi, rtol,
                                          it_begin, it_end, mask_d, ys, pass, ylr);
  rc = check_launch("hod_bisect_kernel");
  if (rc) return rc;
  hod_mask_reduce_kernel<<<1, 256, 0, st>>>(nz, pass, mask_d);
  return check_launch("hod_mask_reduce_kernel");
}

extern "C" int hmv_hod_pick(int nz, const double* ws_d, const unsigned long long* mask_d, double A_log10mthresh,
                            double* log10mthresh_d, int* iters_d, void* stream) {
  HMV_REQUIRE(nz > 0, "hmv_hod_pick: need nz>0");
  HMV_REQUIRE(ws_d && mask_d && log10mthresh_d && iters_d, "hmv_hod_pick: null pointer");
  hod_bisect_pick_kernel<<<cdiv(nz, 256), 256, 0, (cudaStream_t)stream>>>(nz, ws_d, mask_d, A_log10mthresh,
                                                                         log10mthresh_d, iters_d);
  return check_launch("hod_bisect_pick_kernel");
}

extern "C" int hmv_hod_solve(int nz, int nm, const double* zs_d, const double* ms_d, const double* nzm_d,
                             const double* ngal_target_d, const double* hodp_h, double ylo, double yhi, double rtol,
                             double A_log10mthresh, double* ws_d, double* log10mthresh_d, int* iters_d, void* stream) {
  HMV_REQUIRE(ws_d != nullptr, "hmv_hod_solve: null workspace");
  unsigned long long* mask = (unsigned long long*)(ws_d + (size_t)nz * (HMV_BISECT_MAXIT + 3));
  int rc = hmv_hod_bisect(nz, nm, zs_d, ms_d, nzm_d, ngal_target_d, hodp_h, ylo, yhi, rtol, 0, HMV_BISECT_MAXIT, ws_d,
                          mask, stream);
  if (rc) return rc;
  return hmv_hod_pick(nz, ws_d, mask, A_log10mthresh, log10mthresh_d, iters_d, stream);
}
