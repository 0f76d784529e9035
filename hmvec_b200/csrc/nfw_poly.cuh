// nfw_poly.cuh -- device helpers of the piecewise-polynomial NFW evaluation shared by the cube kernel (k_nfw.cu) and
// the fused spectra kernel (k_power.cu).  See k_nfw.cu for the method.
#pragma once
#include "sici.cuh"

namespace hmv {
#include "nfw_poly_tables.inc"

constexpr int NFWP_REC = NFWP_NI * NFWP_STRIDE;          // polynomial coefficients per halo
constexpr int NFW_REC = NFWP_REC + 6;                    // per-halo record: the polynomial coefficients, then
                                                         // {c, a = r_s (1+z), a c, ln(1+c), 1/m_c, 0}

__device__ __forceinline__ int nfwp_interval(double s) {
  const int si = __double2int_rz(fmin(s, 1.0e6));
  return si < 1 ? 0 : si < 2 ? 1 : si < 16 ? 1 + (si >> 1) : si < 64 ? 5 + (si >> 2) : NFWP_NI;
}

struct NfwpTables {                        // per-CTA copies of the interval tables (lane-divergent lookups)
  double2 map[NFWP_NI];                    // t = y*map.x + map.y
  double hi[NFWP_NI + 1];                  // end of the range the interval's polynomial is valid on (a little past its
                                           // upper edge; last entry: +inf for "beyond")
  int deg[NFWP_NI];
  unsigned char idx[72];                   // interval of floor(s) for floor(s) <= 64 (64: beyond)
};

// filled by the first 72 threads of a CTA; callers synchronise afterwards
__device__ __forceinline__ void nfwp_tables_init(NfwpTables& T, int tid) {
  if (tid < NFWP_NI) { T.map[tid] = g_nfwp_map[tid]; T.deg[tid] = g_nfwp_deg[tid]; }
  if (tid <= NFWP_NI) T.hi[tid] = tid < NFWP_NI ? g_nfwp_hix[tid] : 1.0e300;
  if (tid < 72) T.idx[tid] = (unsigned char)(tid < 64 ? nfwp_interval((double)tid + 0.5) : NFWP_NI);
}

__device__ __forceinline__ int nfwp_lookup(const NfwpTables& T, double s) {
  return T.idx[min(__double2int_rz(s), 64)];            // the conversion saturates for huge s
}

// host: per-halo records rec[rows][NFW_REC] from ONE tensor-core contraction (k_nfw.cu).  kmax_d: device scalar
// >= max(ks), or the per-chunk maxima (nkmax entries).
int nfw_poly_records(long long rows, int nm, int nkmax, const double* kmax_d, const double* zs_d, const double* cs_d,
                     const double* rvir_d, double* rec, cudaStream_t st);

}  // namespace hmv
