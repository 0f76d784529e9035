// k_power.cu -- K5: fused 1-halo + 2-halo mass integrals (reference hmvec.py:469-572).
//
// HBM-bound streaming reductions over the mass axis of the u(z,M,k) cubes.  A CTA owns one redshift and a k tile and
// walks the whole mass axis: one producer lane issues 1-D bulk async copies (cp.async.bulk -> TMA unit) of a few rows of
// every cube it needs plus the rows' 64-byte coefficient records into a shared-memory stage ring (BulkRing,
// common.cuh); the consumer warps read the ring, each thread owning adjacent k for ALL masses (no cross-thread
// reduction).  The trapezoid-in-linear-M weights, n(M,z), b(M,z) and the tracer amplitudes are folded into the
// per-(z,M) records by a small prep kernel; the epilogue applies the 1-halo damping, the consistency terms and P_lin.
// Algorithmic traffic: 8*nm bytes per (z,k) per distinct cube read.
//   power_prep_kernel      coefficient records of a tracer pair (hmv_power, hmv_power_tab)
//   power_pair_kernel      any tracer pair (matter / HOD / pressure), up to four distinct cubes
//   power_one_kernel       a pair whose two legs read the same single cube and no central-profile cube
//   power_resp_prep_kernel, power_one_resp_kernel, power_pair_resp_kernel
//                          the same bodies with the response's records and epilogue (hmv_power_response, DESIGN.md §4.5)
//   power_six_prep_kernel  coefficient records of the six spectra (hmv_power_six, _six_tab, _six_nfw)
//   power_six_kernel       {mm, ee, me, gg, gm, ge} in one pass over two cubes
//   power_six_tab_kernel   the same with the electron profile interpolated from its bin tables
//   power_one_tab_kernel   the auto spectrum of one profile given as bin tables (P_yy); nothing is streamed
//   tile_range_kernel      {min, max} of ks, the range of power_six_nfw_kernel's polynomial records
//   power_six_nfw_kernel   the six spectra with the NFW profile evaluated in-kernel (spectra-only fusion)
#include <cstdlib>
#include <initializer_list>
#include <math_constants.h>
#include "common.cuh"
#include "nfw_poly.cuh"

namespace hmv {

// 1-halo damping 1 - exp(-(k/kstar)^2) (hmvec.py:526)
__device__ __forceinline__ double damp_1h(double k, double kstar) {
  const double r = k / kstar;
  return 1.0 - exp(-r * r);
}

// ---------------------------------------------------------------------------------------------------------
// prep: per-(z,M) coefficient rows + per-z offsets
//   generic pair (form 0):  coef = {aA, bA, aB, bB, w1, w2, -}     1h += w1 (aA UC_A + bA US_A)(aB UC_B + bB US_B)
//   hod square   (form 1):  coef = {aA, bA, aB, bB, c1, w2, c2}    1h += US_A (c1 UC_A + c2 US_A)
//   w1 = trapzw*n, w2 = trapzw*n*b_h ;  zoff[z] = {b_A - C_A, b_B - C_B}
// ---------------------------------------------------------------------------------------------------------
struct TracerArgs {
  int kind;
  const double *Nc, *Ns, *NcNs, *NsNsm1, *ngal, *bias;
};

__device__ __forceinline__ void leg_coeffs(const TracerArgs& t, int z, long long i, double mu, double& a, double& b,
                                           double& t0) {
  if (t.kind == 0) {            // matter: M u / rho_m0 (hmvec.py:488-492)
    a = 0.0; b = mu; t0 = mu;
  } else if (t.kind == 1) {     // hod: (u_c Nc + u_s Ns)/ngal (hmvec.py:481-486)
    const double ig = 1.0 / t.ngal[z];
    a = t.Nc[i] * ig; b = t.Ns[i] * ig; t0 = (t.Nc[i] + t.Ns[i]) * ig;
  } else {                      // pressure (hmvec.py:494-497, 541-545)
    a = 0.0; b = 1.0; t0 = 0.0;
  }
}

// kResp: the records of the response to a long mode (hmv_power_response): c4 = w2, so that the 1-halo sum of the
// consumers is R1h = sum_m w n b t_A t_B.  Only form 0 occurs there.
template <bool kResp>
__device__ __forceinline__ void power_prep_body(int nm, const double* __restrict__ ms, const double* __restrict__ nzm,
                                                const double* __restrict__ bh, double rho_m0, TracerArgs A,
                                                TracerArgs B, int form, double* __restrict__ coef,
                                                double* __restrict__ zoff) {
  __shared__ double red[32];
  const int z = blockIdx.x;
  double cA = 0.0, cB = 0.0, gA = 0.0, gB = 0.0;
  for (int m = threadIdx.x; m < nm; m += blockDim.x) {
    const long long i = (long long)z * nm + m;
    const double wt = trapz_weight(ms, m, nm);
    const double w1 = wt * nzm[i], w2 = w1 * bh[i], mu = ms[m] / rho_m0;
    double aA, bA, tA0, aB, bB, tB0;
    leg_coeffs(A, z, i, mu, aA, bA, tA0);
    leg_coeffs(B, z, i, mu, aB, bB, tB0);
    double c4 = kResp ? w2 : w1, c6 = 0.0;
    if (!kResp && form == 1) {            // hmvec.py:477-479
      const double ig = 1.0 / A.ngal[z], ig2 = ig * ig;
      c4 = w1 * 2.0 * A.NcNs[i] * ig2;
      c6 = w1 * A.NsNsm1[i] * ig2;
    }
    double2* rec = reinterpret_cast<double2*>(coef + i * 8);     // 64-byte record per (z,M): one bulk copy per stage
    rec[0] = make_double2(aA, bA);
    rec[1] = make_double2(aB, bB);
    rec[2] = make_double2(c4, w2);
    rec[3] = make_double2(c6, 0.0);
    cA = fma(w2, tA0, cA);      // consistency integrals (hmvec.py:567-568)
    cB = fma(w2, tB0, cB);
    if (A.kind == 1) gA = fma(w2, A.Nc[i] + A.Ns[i], gA);   // get_bg numerator (hmvec.py:465)
    if (B.kind == 1) gB = fma(w2, B.Nc[i] + B.Ns[i], gB);
  }
  cA = block_sum(cA, red); cB = block_sum(cB, red); gA = block_sum(gA, red); gB = block_sum(gB, red);
  if (threadIdx.x == 0) {
    double bA = (A.kind == 0) ? 1.0 : (A.kind == 1 ? gA / A.ngal[z] : 0.0);
    double bB = (B.kind == 0) ? 1.0 : (B.kind == 1 ? gB / B.ngal[z] : 0.0);
    if (A.bias) bA = A.bias[z];   // b1_in / b2_in (hmvec.py:558-561)
    if (B.bias) bB = B.bias[z];
    zoff[2 * z + 0] = bA - cA;
    zoff[2 * z + 1] = bB - cB;
  }
}

__global__ void __launch_bounds__(256) power_prep_kernel(int nm, const double* __restrict__ ms,
                                                          const double* __restrict__ nzm,
                                                          const double* __restrict__ bh, double rho_m0,
                                                          TracerArgs A, TracerArgs B, int form,
                                                          double* __restrict__ coef, double* __restrict__ zoff) {
  power_prep_body<false>(nm, ms, nzm, bh, rho_m0, A, B, form, coef, zoff);
}

__global__ void __launch_bounds__(256) power_resp_prep_kernel(int nm, const double* __restrict__ ms,
                                                               const double* __restrict__ nzm,
                                                               const double* __restrict__ bh, double rho_m0,
                                                               TracerArgs A, TracerArgs B,
                                                               double* __restrict__ coef, double* __restrict__ zoff) {
  power_prep_body<true>(nm, ms, nzm, bh, rho_m0, A, B, 0, coef, zoff);
}

// Generic tracer pair on the same ring as power_six_kernel: up to four distinct cubes (us_A, uc_A, us_B, uc_B,
// de-duplicated by pointer) are streamed once; a stage holds PR_R rows of every cube plus the rows' 64-byte records.
constexpr int PR_K = 512, PR_R = 4, PR_CT = 256;

struct PairArgs {
  int nm, nk, ldk, form, ncube, nst;
  const double* cube[4];
  int rusA, rucA, rusB, rucB;            // index into cube[] of each role; -1 = the profile is identically 1
  const double* coef;
  const double *zoff, *ks, *Pzk;
  double kstar;
  double *p1h, *p2h;
};

// P1h and P2h of one (z, k) of a tracer pair (hmvec.py:526, 572)
__device__ __forceinline__ void pair_epilogue(const PairArgs& a, int z, int k, double p1, double iA, double iB) {
  const long long o = (long long)z * a.nk + k;
  if (a.p1h) a.p1h[o] = p1 * damp_1h(a.ks[k], a.kstar);
  if (a.p2h) a.p2h[o] = a.Pzk[o] * (iA + a.zoff[2 * z]) * (iB + a.zoff[2 * z + 1]);
}

// n_eff = d ln P_lin / d ln k at column k of the row P (nk >= 2), as np.gradient(np.log(P), np.log(ks)): the
// second-order stencil of a non-uniform grid inside, first-order one-sided differences at both ends.  A P that is not
// positive at the column or at a neighbour the stencil reads gives NaN.
__device__ __forceinline__ double n_eff(const double* __restrict__ ks, const double* __restrict__ P, int nk, int k) {
  const int lo = k > 0 ? k - 1 : 0, hi = k < nk - 1 ? k + 1 : nk - 1;
  const double Pl = P[lo], Pc = P[k], Ph = P[hi];
  if (!(Pl > 0.0 && Pc > 0.0 && Ph > 0.0)) return CUDART_NAN;
  const double xl = log(ks[lo]), xc = log(ks[k]), xh = log(ks[hi]);
  const double fl = log(Pl), fc = log(Pc), fh = log(Ph);
  if (k == 0) return (fh - fc) / (xh - xc);
  if (k == nk - 1) return (fc - fl) / (xc - xl);
  const double d1 = xc - xl, d2 = xh - xc;
  return -d2 / (d1 * (d1 + d2)) * fl + (d2 - d1) / (d1 * d2) * fc + d1 / (d2 * (d1 + d2)) * fh;
}

// The response of one (z, k) to a long-wavelength mode (hmv_power_response): R1h = the 1-halo sum of the response
// records (c4 = w2, no damping) into p1h, R2h = (47/21 - n_eff/3) P_lin (I_A + b_A - C_A)(I_B + b_B - C_B) into p2h.
__device__ __forceinline__ void response_epilogue(const PairArgs& a, int z, int k, double p1, double iA, double iB) {
  const long long o = (long long)z * a.nk + k;
  if (a.p1h) a.p1h[o] = p1;
  if (a.p2h) {
    const double P2h = a.Pzk[o] * (iA + a.zoff[2 * z]) * (iB + a.zoff[2 * z + 1]);
    a.p2h[o] = (47.0 / 21.0 - n_eff(a.ks, a.Pzk + (long long)z * a.nk, a.nk, k) / 3.0) * P2h;
  }
}

// the epilogue of the two streaming bodies: the spectra (hmv_power) or the response (hmv_power_response)
template <bool kResp>
__device__ __forceinline__ void pair_out(const PairArgs& a, int z, int k, double p1, double iA, double iB) {
  if (kResp) response_epilogue(a, z, k, p1, iA, iB);
  else pair_epilogue(a, z, k, p1, iA, iB);
}

template <bool kResp>
__device__ __forceinline__ void power_pair_body(const PairArgs a) {
  __builtin_assume(threadIdx.x < PR_CT + 32);            // the kernels' launch bounds, which the body does not see
  extern __shared__ __align__(128) unsigned char pair_smem[];
  const BulkRing ring(pair_smem, a.nst, a.ncube * PR_R * PR_K + PR_R * 8, PR_CT / 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int z = blockIdx.y, k0 = blockIdx.x * PR_K;
  const int segk = min(PR_K, a.ldk - k0);
  const long long zrow = (long long)z * a.nm;
  const int nit = (a.nm + PR_R - 1) / PR_R;
  __syncthreads();
  RingSlot slot;

  if (warp == PR_CT / 32) {            // ---- producer warp ----
    if (lane == 0) {
      const unsigned segb = (unsigned)segk * 8u;
      for (int it = 0; it < nit; ++it, ring.advance(slot)) {
        const int m0 = it * PR_R, rows = min(PR_R, a.nm - m0);
        const RingStage st = ring.acquire(slot, (unsigned)rows * ((unsigned)a.ncube * segb + 64u));
        for (int c = 0; c < a.ncube; ++c)
          for (int r = 0; r < rows; ++r)
            bulk_g2s(st.p + (c * PR_R + r) * PR_K, a.cube[c] + (zrow + m0 + r) * (long long)a.ldk + k0, segb, st.full);
        bulk_g2s(st.p + a.ncube * PR_R * PR_K, a.coef + (zrow + m0) * 8, (unsigned)rows * 64u, st.full);
      }
    }
    return;
  }

  const bool active = 2 * tid < segk;
  double2 p1 = {0, 0}, iA = {0, 0}, iB = {0, 0};
  const double2 one = make_double2(1.0, 1.0);
  for (int it = 0; it < nit; ++it, ring.advance(slot)) {
    const int rows = min(PR_R, a.nm - it * PR_R);
    const double* st = ring.wait(slot);
    if (active) {
#pragma unroll
      for (int r = 0; r < PR_R; ++r) {
        if (r < rows) {
          auto ld = [&](int role) { return *reinterpret_cast<const double2*>(st + (role * PR_R + r) * PR_K + 2 * tid); };
          const double2 usA = ld(a.rusA);
          const double2 ucA = a.rucA >= 0 ? ld(a.rucA) : one;
          const double2 usB = a.rusB == a.rusA ? usA : ld(a.rusB);
          const double2 ucB = a.rucB >= 0 ? (a.rucB == a.rucA ? ucA : ld(a.rucB)) : one;
          const double2* c = reinterpret_cast<const double2*>(st + a.ncube * PR_R * PR_K + r * 8);
          const double2 c01 = c[0], c23 = c[1], c45 = c[2], c67 = c[3];
          const double aA = c01.x, bA = c01.y, aB = c23.x, bB = c23.y, c4 = c45.x, w2 = c45.y, c6 = c67.x;
          double2 tA, tB;
          tA.x = fma(aA, ucA.x, bA * usA.x); tA.y = fma(aA, ucA.y, bA * usA.y);
          tB.x = fma(aB, ucB.x, bB * usB.x); tB.y = fma(aB, ucB.y, bB * usB.y);
          if (a.form == 0) {
            p1.x = fma(c4 * tA.x, tB.x, p1.x); p1.y = fma(c4 * tA.y, tB.y, p1.y);
          } else {
            p1.x = fma(usA.x, fma(c4, ucA.x, c6 * usA.x), p1.x);
            p1.y = fma(usA.y, fma(c4, ucA.y, c6 * usA.y), p1.y);
          }
          iA.x = fma(w2, tA.x, iA.x); iA.y = fma(w2, tA.y, iA.y);
          iB.x = fma(w2, tB.x, iB.x); iB.y = fma(w2, tB.y, iB.y);
        }
      }
    }
    ring.release(slot);
  }
  if (!active) return;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = k0 + 2 * tid + e;
    if (k >= a.nk) break;
    pair_out<kResp>(a, z, k, e ? p1.y : p1.x, e ? iA.y : iA.x, e ? iB.y : iB.x);
  }
}

__global__ void __launch_bounds__(PR_CT + 32, 1) power_pair_kernel(const PairArgs a) { power_pair_body<false>(a); }
__global__ void __launch_bounds__(PR_CT + 32, 1) power_pair_resp_kernel(const PairArgs a) { power_pair_body<true>(a); }

// Tracer pairs whose two legs read the SAME single cube and have no central-profile cube (mm, ee, yy autos; galaxies x
// their own satellite profile): t_A = aA + bA u, t_B = aB + bB u.  Same ring as power_pair_kernel, but a thread owns
// four adjacent k of a 1024-wide tile and the role bookkeeping is gone: 6 FP64 instructions per element and the per-row
// record loads shared by four elements.  power_pair_kernel was issue-bound on this case (ncu: 70 % issue slots active,
// 5.9 TB/s); this one streams at the HBM rate.
constexpr int ONE_K = 1024, ONE_R = 4, ONE_NST = 5, ONE_CT = 256;
constexpr int ONE_STAGE_DOUBLES = ONE_R * ONE_K + ONE_R * 8;

template <bool kResp>
__device__ __forceinline__ void power_one_body(const PairArgs a) {
  __builtin_assume(threadIdx.x < ONE_CT + 32);           // the kernels' launch bounds, which the body does not see
  extern __shared__ __align__(128) unsigned char one_smem[];
  const BulkRing ring(one_smem, ONE_NST, ONE_STAGE_DOUBLES, ONE_CT / 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int z = blockIdx.y, k0 = blockIdx.x * ONE_K;
  const int segk = min(ONE_K, a.ldk - k0);                 // doubles per row segment (multiple of 2)
  const long long zrow = (long long)z * a.nm;
  const int nit = (a.nm + ONE_R - 1) / ONE_R;
  __syncthreads();

  if (warp == ONE_CT / 32) {            // ---- producer warp ----
    if (lane == 0) {
      const unsigned segb = (unsigned)segk * 8u;
      for (int it = 0; it < nit; ++it) {
        const int m0 = it * ONE_R, rows = min(ONE_R, a.nm - m0);
        const RingStage st = ring.acquire(ring.slot(it), (unsigned)rows * (segb + 64u));
        for (int r = 0; r < rows; ++r)
          bulk_g2s(st.p + r * ONE_K, a.cube[0] + (zrow + m0 + r) * (long long)a.ldk + k0, segb, st.full);
        bulk_g2s(st.p + ONE_R * ONE_K, a.coef + (zrow + m0) * 8, (unsigned)rows * 64u, st.full);
      }
    }
    return;
  }

  // thread owns k0 + 2 tid, +1 and k0 + 512 + 2 tid, +1 (two conflict-free 16-byte loads per row)
  const bool act0 = 2 * tid < segk, act1 = 512 + 2 * tid < segk;
  double p1[4] = {0, 0, 0, 0}, iA[4] = {0, 0, 0, 0}, iB[4] = {0, 0, 0, 0};
  for (int it = 0; it < nit; ++it) {
    const RingSlot slot = ring.slot(it);
    const int rows = min(ONE_R, a.nm - it * ONE_R);
    const double* st = ring.wait(slot);
    if (act0) {
#pragma unroll
      for (int r = 0; r < ONE_R; ++r) {
        if (r < rows) {
          const double2 u0 = *reinterpret_cast<const double2*>(st + r * ONE_K + 2 * tid);
          const double2 u1 = act1 ? *reinterpret_cast<const double2*>(st + r * ONE_K + 512 + 2 * tid) : make_double2(0.0, 0.0);
          const double2* c = reinterpret_cast<const double2*>(st + ONE_R * ONE_K + r * 8);
          const double2 c01 = c[0], c23 = c[1], c45 = c[2];
          const double aA = c01.x, bA = c01.y, aB = c23.x, bB = c23.y, c4 = c45.x, w2 = c45.y;
          const double u[4] = {u0.x, u0.y, u1.x, u1.y};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const double tA = fma(bA, u[e], aA), tB = fma(bB, u[e], aB);
            p1[e] = fma(c4 * tA, tB, p1[e]);
            iA[e] = fma(w2, tA, iA[e]);
            iB[e] = fma(w2, tB, iB[e]);
          }
        }
      }
    }
    ring.release(slot);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int k = k0 + (e >> 1) * 512 + 2 * tid + (e & 1);
    if (k >= a.nk || (e < 2 ? !act0 : !act1)) continue;
    pair_out<kResp>(a, z, k, p1[e], iA[e], iB[e]);
  }
}

__global__ void __launch_bounds__(ONE_CT + 32, 1) power_one_kernel(const PairArgs a) { power_one_body<false>(a); }
__global__ void __launch_bounds__(ONE_CT + 32, 1) power_one_resp_kernel(const PairArgs a) { power_one_body<true>(a); }

// ---------------------------------------------------------------------------------------------------------
// six spectra {mm, ee, me, gg, gm, ge} in one pass over (u_m, u_e); HOD satellites follow u_m, centrals u_c = 1
//   coef[z][m][8]: A1 = w1 mu^2, c1 = w1 2 NcNs/ngal^2, c2 = w1 NsNsm1/ngal^2, B1 = w1 mu Nc/ngal, B2 = w1 mu Ns/ngal,
//                  D1 = w2 mu, D2 = w2 Ns/ngal, (pad) ;  zoff6[z] = {1 - C_m, bg - C_g + sum w2 Nc/ngal}
//
// HBM-bound stream: a CTA owns one redshift and a 512-wide k tile and walks the whole mass axis.  One producer
// lane issues 1-D bulk async copies (cp.async.bulk -> the TMA unit) of SIX_R rows x 4 KB from each cube plus the
// rows' 64-byte coefficient records into a SIX_NST-deep shared-memory ring, completion tracked by mbarriers
// (full/empty pair per stage); eight consumer warps read the ring (each thread owns two adjacent k for ALL masses, so
// there is no cross-thread reduction) and keep 18 FP64 accumulators in registers.  Memory-level parallelism comes
// from the ring (up to 96 KB in flight per SM), not from registers or occupancy.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) power_six_prep_kernel(int nm, const double* __restrict__ ms,
                                                              const double* __restrict__ nzm,
                                                              const double* __restrict__ bh, double rho_m0,
                                                              const double* __restrict__ Nc, const double* __restrict__ Ns,
                                                              const double* __restrict__ NcNs,
                                                              const double* __restrict__ NsNsm1,
                                                              const double* __restrict__ ngal,
                                                              double* __restrict__ coef, double* __restrict__ zoff) {
  __shared__ double red[32];
  const int z = blockIdx.x;
  const double ig = 1.0 / ngal[z], ig2 = ig * ig;
  double cm = 0.0, cg = 0.0, gb = 0.0, gc = 0.0;
  for (int m = threadIdx.x; m < nm; m += blockDim.x) {
    const long long i = (long long)z * nm + m;
    const double wt = trapz_weight(ms, m, nm);
    const double w1 = wt * nzm[i], w2 = w1 * bh[i], mu = ms[m] / rho_m0;
    const double nc = Nc[i] * ig, ns = Ns[i] * ig;
    double2* c = reinterpret_cast<double2*>(coef + i * 8);
    c[0] = make_double2(w1 * mu * mu, w1 * 2.0 * NcNs[i] * ig2);
    c[1] = make_double2(w1 * NsNsm1[i] * ig2, w1 * mu * nc);
    c[2] = make_double2(w1 * mu * ns, w2 * mu);
    c[3] = make_double2(w2 * ns, 0.0);
    cm = fma(w2, mu, cm);
    cg = fma(w2, (Nc[i] + Ns[i]) * ig, cg);
    gb = fma(w2, Nc[i] + Ns[i], gb);
    gc = fma(w2, nc, gc);
  }
  cm = block_sum(cm, red); cg = block_sum(cg, red); gb = block_sum(gb, red); gc = block_sum(gc, red);
  if (threadIdx.x == 0) {
    zoff[2 * z + 0] = 1.0 - cm;
    zoff[2 * z + 1] = gb * ig - cg + gc;   // bias - consistency + the k-independent central part of I_g
  }
}

// k-tile width for a grid of nz x ceil(ldk / tile) CTAs on `per_sm` CTA slots per SM.  Measured on B200
// (gpurun_out/r2_k5_tiles.txt): a wave of 512-column CTAs is HBM-bound (0.33 ms for 2000 masses); narrower CTAs do not
// get proportionally faster -- below ~440 columns a wave takes 0.285 ms whatever its width, because every consumer warp
// still walks the whole mass axis for its 64 columns -- and a CTA in a thin last wave takes ~0.24 ms.  So a narrower
// tile pays only when it moves CTAs out of a thin last wave of a grid that is a few waves deep: a 25-z slab (one rank
// of an 8-GPU run) has 500 CTAs = 3 waves + 56 at 512 columns, 575 = 3 waves + 131 at 448 (1.25 -> 1.15 ms); 100 or
// 200 redshifts stay at 512 (a predicted gain below 3 % is not taken).  Multiples of 16 doubles keep rows 128-B aligned.
static int wave_tile(int nz, int ldk, int tile_max, int per_sm) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        sms <= 0)
      sms = 148;
  }
  if (const char* e = getenv("HMV_TILE")) {                 // measurement knob: force a width
    const int t = atoi(e);
    if (t >= 16 && t <= tile_max && t % 16 == 0) return t;
  }
  const long long slots = (long long)sms * per_sm;
  const double unit = tile_max / 0.33;                      // columns of a full-width wave per millisecond
  const double floor_w = 0.285 * unit, lone = 0.24 * unit;
  auto cost = [&](int t) {
    const long long ctas = (long long)nz * cdiv(ldk, t);
    const long long full = ctas / slots, rem = ctas % slots;
    return (double)full * fmax((double)t, floor_w) + (rem ? fmax(lone, (double)rem / (double)slots * t) : 0.0);
  };
  int best = tile_max;
  double best_cost = cost(tile_max);
  const double need = 0.97 * best_cost;
  for (int t = tile_max - 16; t >= tile_max * 7 / 8; t -= 16) {
    const double c = cost(t);
    if (c < need && c < best_cost) { best_cost = c; best = t; }
  }
  return best;
}

constexpr int SIX_K = 512, SIX_R = 4, SIX_NST = 6, SIX_CT = 256;   // k per CTA, rows per stage, stages, consumers
constexpr int SIX_STAGE_DOUBLES = 2 * SIX_R * SIX_K + SIX_R * 8;

// what the six-spectra epilogue reads besides the sums, and where it writes P1h / P2h of {mm, ee, me, gg, gm, ge}
struct SixOut {
  long long spec_stride;   // doubles between consecutive spectra in p1h/p2h
  const double *zoff, *ks, *Pzk;
  double kstar;
  double *p1h, *p2h;
};

struct SixArgs {
  int nm, nk, ldk;
  int tk;                  // k per CTA (multiple of 16, <= SIX_K): chosen per launch so that the grid fills whole waves
  const double *um, *ue, *coef;
  SixOut out;
};

// the seven coefficients of a mass row's 64-byte record (power_six_prep_kernel)
struct SixCoef { double A1, c1, c2, B1, B2, D1, D2; };

__device__ __forceinline__ SixCoef six_coef(const double* rec) {
  const double2* c = reinterpret_cast<const double2*>(rec);
  const double2 c01 = c[0], c23 = c[1], c45 = c[2], c67 = c[3];
  return {c01.x, c01.y, c23.x, c23.y, c45.x, c45.y, c67.x};
}

// one mass row at one wavenumber: 18 FMAs into the six 1-halo sums acc[0..6) and the 2-halo legs acc[6..9) (m, e, g)
__device__ __forceinline__ void six_fma(double (&acc)[9], const SixCoef& c, double um, double ue) {
  const double q1 = um * um, q2 = ue * ue, q3 = um * ue;
  acc[0] = fma(c.A1, q1, acc[0]);
  acc[1] = fma(c.A1, q2, acc[1]);
  acc[2] = fma(c.A1, q3, acc[2]);
  acc[3] = fma(c.c1, um, fma(c.c2, q1, acc[3]));
  acc[4] = fma(c.B1, um, fma(c.B2, q1, acc[4]));
  acc[5] = fma(c.B1, ue, fma(c.B2, q3, acc[5]));
  acc[6] = fma(c.D1, um, acc[6]);
  acc[7] = fma(c.D1, ue, acc[7]);
  acc[8] = fma(c.D2, um, acc[8]);
}

// the six spectra of redshift z at wavenumber index k < nk (hmvec.py:526, 572)
__device__ __forceinline__ void six_epilogue(const SixOut& a, int z, int nk, int k, const double (&acc)[9]) {
  const long long S = a.spec_stride, o = (long long)z * nk + k;
  const double zo0 = a.zoff[2 * z], zo1 = a.zoff[2 * z + 1];
  if (a.p1h) {
    const double damp = damp_1h(a.ks[k], a.kstar);
#pragma unroll
    for (int q = 0; q < 6; ++q) a.p1h[q * S + o] = acc[q] * damp;
  }
  if (a.p2h) {
    const double P = a.Pzk[o];
    const double Lm = acc[6] + zo0, Le = acc[7] + zo0, Lg = acc[8] + zo1;
    a.p2h[0 * S + o] = P * Lm * Lm; a.p2h[1 * S + o] = P * Le * Le; a.p2h[2 * S + o] = P * Lm * Le;
    a.p2h[3 * S + o] = P * Lg * Lg; a.p2h[4 * S + o] = P * Lg * Lm; a.p2h[5 * S + o] = P * Lg * Le;
  }
}

__global__ void __launch_bounds__(SIX_CT + 32, 1) power_six_kernel(const SixArgs a) {
  extern __shared__ __align__(128) unsigned char six_smem[];
  const BulkRing ring(six_smem, SIX_NST, SIX_STAGE_DOUBLES, SIX_CT / 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int z = blockIdx.y, k0 = blockIdx.x * a.tk;
  const int segk = min(a.tk, a.ldk - k0);                  // doubles per row segment (multiple of 2)
  const long long zrow = (long long)z * a.nm;
  const int nit = (a.nm + SIX_R - 1) / SIX_R;
  __syncthreads();

  if (warp == SIX_CT / 32) {            // ---- producer warp: one elected lane drives the TMA unit ----
    if (lane == 0) {
      const unsigned segb = (unsigned)segk * 8u;
      for (int it = 0; it < nit; ++it) {
        const int m0 = it * SIX_R, rows = min(SIX_R, a.nm - m0);
        const RingStage st = ring.acquire(ring.slot(it), (unsigned)rows * (2u * segb + 64u));
        for (int r = 0; r < rows; ++r) {
          const long long off = (zrow + m0 + r) * (long long)a.ldk + k0;
          bulk_g2s(st.p + r * SIX_K, a.um + off, segb, st.full);
          bulk_g2s(st.p + (SIX_R + r) * SIX_K, a.ue + off, segb, st.full);
        }
        bulk_g2s(st.p + 2 * SIX_R * SIX_K, a.coef + (zrow + m0) * 8, (unsigned)rows * 64u, st.full);
      }
    }
    return;
  }

  // ---- consumers: thread owns k = k0 + 2 tid, +1 over the whole mass axis ----
  const bool active = 2 * tid < segk;
  double acc[2][9] = {};
  for (int it = 0; it < nit; ++it) {
    const RingSlot slot = ring.slot(it);
    const int rows = min(SIX_R, a.nm - it * SIX_R);
    const double* st = ring.wait(slot);
    if (active) {
#pragma unroll
      for (int r = 0; r < SIX_R; ++r) {
        if (r < rows) {
          const double2 um = *reinterpret_cast<const double2*>(st + r * SIX_K + 2 * tid);
          const double2 ue = *reinterpret_cast<const double2*>(st + (SIX_R + r) * SIX_K + 2 * tid);
          const SixCoef c = six_coef(st + 2 * SIX_R * SIX_K + r * 8);
          six_fma(acc[0], c, um.x, ue.x);
          six_fma(acc[1], c, um.y, ue.y);
        }
      }
    }
    ring.release(slot);
  }
  if (!active) return;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = k0 + 2 * tid + e;
    if (k >= a.nk) break;
    six_epilogue(a.out, z, a.nk, k, acc[e]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// The six spectra with the ELECTRON profile interpolated from its bin tables inside the reduction (hmv_profile_tables:
// the transform's result before the expansion onto ks) instead of read from a cube: the 32 GB cube is neither written
// nor re-read, the kernel streams the matter cube plus the rows' table parameters, and gathers the two bins around
// each wavenumber from the tables (which the redshift's CTAs share in L2).  A row whose t = k * inv lies below the
// first bin holds u_e = u_1, above the last one u_e = 0.  Consumers interpolate exactly as the transform's own
// expansion does (np.interp semantics of fft.py:102-107).
// ---------------------------------------------------------------------------------------------------------
constexpr int TAB_R = 4, TAB_CT = 256, TAB_NST = 6;
constexpr int TAB_STAGE_DOUBLES = TAB_R * SIX_K + TAB_R * 8 + TAB_R * 4;       // matter rows, coefficient records, table parameters

struct SixTabArgs {
  int nm, nk, ldk, nmp, JS, J;
  const double *um, *coef, *tab, *tmeta;
  SixOut out;
};

// what a thread keeps of one (row, wavenumber) between issuing the two table loads and using them
struct TabLerp { double ua, ub, fr; };   // fr: t - j inside [1, J]; -1: below the first bin (hold u_1); -2: above the last (zero)

__device__ __forceinline__ TabLerp tab_fetch(const double* __restrict__ row, double inv, int jcap, double k, double tJ) {
  const double t = k * inv;
  const int jj = min(max(__double2int_rz(fmin(t, tJ)), 1), jcap);       // always inside the bins the transform wrote
  HMV_DEV_ASSERT(jj >= 1 && jj + 1 <= (int)tJ + 1);
  TabLerp r;
  r.fr = (t >= 1.0) ? ((t > tJ) ? -2.0 : t - (double)jj) : -1.0;
  r.ua = 0.0; r.ub = 0.0;
  if (r.fr >= 0.0) { r.ua = row[jj]; r.ub = row[jj + 1]; }              // plain loads: the tables of a redshift live in L2
  return r;
}
__device__ __forceinline__ double tab_value(const TabLerp& r, double u1) {
  const double v = fma(r.fr, r.ub - r.ua, r.ua);
  return (r.fr >= 0.0) ? v : ((r.fr > -1.5) ? u1 : 0.0);                // np.interp left=puks[0], right=0 (fft.py:102-107)
}

__global__ void __launch_bounds__(TAB_CT + 32, 1) power_six_tab_kernel(const SixTabArgs a) {
  extern __shared__ __align__(128) unsigned char tab_smem[];
  const BulkRing ring(tab_smem, TAB_NST, TAB_STAGE_DOUBLES, TAB_CT / 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int z = blockIdx.y, k0 = blockIdx.x * SIX_K;
  const int segk = min(SIX_K, a.ldk - k0);
  const long long zrow = (long long)z * a.nm, zrowp = (long long)z * a.nmp;
  const double tJ = (double)a.J;
  const int nit = (a.nm + TAB_R - 1) / TAB_R;
  __syncthreads();

  if (warp == TAB_CT / 32) {            // ---- producer warp: one elected lane drives the TMA unit ----
    if (lane == 0) {
      const unsigned segb = (unsigned)segk * 8u;
      for (int it = 0; it < nit; ++it) {
        const int m0 = it * TAB_R, rows = min(TAB_R, a.nm - m0);
        const RingStage st = ring.acquire(ring.slot(it), (unsigned)rows * (segb + 64u + 32u));
        for (int r = 0; r < rows; ++r)
          bulk_g2s(st.p + r * SIX_K, a.um + (zrow + m0 + r) * (long long)a.ldk + k0, segb, st.full);
        bulk_g2s(st.p + TAB_R * SIX_K, a.coef + (zrow + m0) * 8, (unsigned)rows * 64u, st.full);
        bulk_g2s(st.p + TAB_R * SIX_K + TAB_R * 8, a.tmeta + (zrowp + m0) * 4, (unsigned)rows * 32u, st.full);
      }
    }
    return;
  }

  // ---- consumers: thread owns k = k0 + 2 tid, +1 over the whole mass axis.  The table reads of stage i+1 are issued
  //      (from the stage's parameter records, as soon as they have landed) before stage i is accumulated ----
  const bool active = 2 * tid < segk;
  const int kc = min(k0 + 2 * tid, a.nk - 1), kc1 = min(k0 + 2 * tid + 1, a.nk - 1);
  const double kx = a.out.ks[kc], ky = a.out.ks[kc1];
  double acc[2][9] = {};
  TabLerp cur[TAB_R][2], nxt[TAB_R][2];
  auto issue = [&](int it, TabLerp (&dst)[TAB_R][2]) {
    const double4* pm = reinterpret_cast<const double4*>(ring.wait(ring.slot(it)) + TAB_R * SIX_K + TAB_R * 8);
    const int m0 = it * TAB_R, rows = min(TAB_R, a.nm - m0);
#pragma unroll
    for (int r = 0; r < TAB_R; ++r) {
      const double4 mt = pm[r < rows ? r : 0];
      const double* row = a.tab + (zrowp + m0 + (r < rows ? r : 0)) * (long long)a.JS;
      const int jcap = min(a.J - 1, (int)mt.z);
      dst[r][0] = tab_fetch(row, mt.x, jcap, kx, tJ);
      dst[r][1] = tab_fetch(row, mt.x, jcap, ky, tJ);
    }
  };
  if (active) issue(0, cur);
  for (int it = 0; it < nit; ++it) {
    const RingSlot slot = ring.slot(it);
    const int rows = min(TAB_R, a.nm - it * TAB_R);
    const double* st = ring.stage(slot);
    if (active) {
      if (it + 1 < nit) issue(it + 1, nxt);
    } else {
      ring.wait(slot);
    }
    if (active) {
      const double4* pm = reinterpret_cast<const double4*>(st + TAB_R * SIX_K + TAB_R * 8);
#pragma unroll
      for (int r = 0; r < TAB_R; ++r) {
        if (r < rows) {
          const double2 um = *reinterpret_cast<const double2*>(st + r * SIX_K + 2 * tid);
          const double u1 = pm[r].y;
          const SixCoef c = six_coef(st + TAB_R * SIX_K + r * 8);
          six_fma(acc[0], c, um.x, tab_value(cur[r][0], u1));
          six_fma(acc[1], c, um.y, tab_value(cur[r][1], u1));
        }
      }
#pragma unroll
      for (int r = 0; r < TAB_R; ++r) { cur[r][0] = nxt[r][0]; cur[r][1] = nxt[r][1]; }
    }
    ring.release(slot);
  }
  if (!active) return;
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = k0 + 2 * tid + e;
    if (k >= a.nk) break;
    six_epilogue(a.out, z, a.nk, k, acc[e]);
  }
}

// ---------------------------------------------------------------------------------------------------------
// Auto spectrum of ONE profile given as bin tables (hmv_profile_tables) -- the tSZ case: P_yy needs the Compton-y
// profile only under the mass integral, so its 32 GB cube is neither written nor read.  Nothing is streamed: a CTA
// (z, 512-wide k tile) keeps the redshift's per-halo parameters in shared memory, sorts the halos into those whose
// whole tile lies below the first bin (u = u_1: their contribution does not depend on k and is summed once per CTA),
// above the last bin (u = 0: nothing) and the rest, and loops over the rest only, each thread interpolating its two
// wavenumbers from the halo's table row in L2 exactly as the transform's expansion does (fft.py:102-107).
// Work is proportional to the interpolated elements (37 % on the LARGE grid).
// ---------------------------------------------------------------------------------------------------------
// 256 threads per CTA (a thread owns two adjacent wavenumbers), register allocation for 2 CTAs per SM, 6 halos in
// flight per thread in the interior loop.  Measured on a B200 on a 67-z slab: 6 halos in flight
// 1.02 ms against 1.10 with 4 (8 spills); prefetch instructions (L1 or L2) for the table line of the halo 4 / 8 / 16
// positions ahead: 1.20-1.25 ms -- slower, the extra address arithmetic costs more than the earlier arrival saves.  A
// ninth warp that walks the halo lists ahead of the others and asks L2 for every halo's whole table segment with
// coalesced prefetches (32 / 96 / 256 halos ahead): 1.60 ms against 1.03 -- the gathers are
// not waiting for DRAM alone.
constexpr int OT_T = 256, OT_K = 2 * OT_T, OT_MINB = 2, OT_UNROLL = 6;
// CTA order: k tiles are the slow index, highest k first, within chunks of OT_ZC redshifts.  A tile's cost is the
// number of halos it has to interpolate (none at low k, where every halo holds u_1), so the expensive tiles of every
// redshift go first and the launch drains on the trivial ones.  Measured on a B200 against redshift-slow
// order: 25 z 0.454 -> 0.385 ms, 67 z 1.013 -> 0.858, 100 z 1.49 -> 1.33, 200 z 2.63 -> 2.52 (chunks of
// 100; 2.58 unchunked, 2.74 with chunks of 32 or 64).
constexpr int OT_ZC = 100;

// launch position -> (redshift, first wavenumber of the tile) of power_one_tab_kernel's tile-slow order
__host__ __device__ __forceinline__ void ot_cta(int id, int nz, int nk, int& z, int& k0) {
  const int T = (nk + OT_K - 1) / OT_K, per = OT_ZC * T;
  const int c = id / per, r = id - c * per;
  const int left = nz - c * OT_ZC;
  const int nzc = left < OT_ZC ? left : OT_ZC;
  const int tr = r / nzc;
  z = c * OT_ZC + (r - tr * nzc);
  k0 = (T - 1 - tr) * OT_K;
}

struct OneTabArgs {
  int nm, nk, nmp, JS, J, nz;
  const double *coef, *zoff, *ks, *Pzk, *tab, *tmeta;
  double kstar;
  double *p1h, *p2h;
};

__global__ void __launch_bounds__(OT_T, OT_MINB) power_one_tab_kernel(const OneTabArgs a) {
  extern __shared__ __align__(16) unsigned char ot_smem[];
  double4* prm = reinterpret_cast<double4*>(ot_smem);              // per interpolated halo: {inv, u_1, a, b} (t = a + b u)
  double2* prm2 = reinterpret_cast<double2*>(prm + a.nm);          //                        {c4, w2}
  int* rowid = reinterpret_cast<int*>(prm2 + a.nm);
  __shared__ double red[3][OT_T / 32];
  __shared__ int nlist, nlist2, wcnt[OT_T / 32], wcnt2[OT_T / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int z, k0;
  ot_cta(blockIdx.x, a.nz, a.nk, z, k0);
  const long long zrow = (long long)z * a.nm, zrowp = (long long)z * a.nmp;
  const double tJ = (double)a.J;
  // wavenumber range of the tile (any order of ks)
  double kmn = 1.0e300, kmx = 0.0;
  for (int k = k0 + tid; k < min(a.nk, k0 + OT_K); k += OT_T) { const double v = a.ks[k]; kmn = fmin(kmn, v); kmx = fmax(kmx, v); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    kmn = fmin(kmn, __shfl_xor_sync(0xffffffffu, kmn, o));
    kmx = fmax(kmx, __shfl_xor_sync(0xffffffffu, kmx, o));
  }
  if (lane == 0) { red[0][warp] = kmn; red[1][warp] = kmx; }
  if (tid == 0) { nlist = 0; nlist2 = 0; }
  __syncthreads();
#pragma unroll
  for (int w = 0; w < OT_T / 32; ++w) { kmn = fmin(kmn, red[0][w]); kmx = fmax(kmx, red[1][w]); }
  __syncthreads();
  // classify the halos; hold-u_1 halos are summed here.  Halos whose whole tile lies inside [1, J] and inside the bins
  // the transform wrote are appended from the front of the list (no classification or clamping per element), the
  // other interpolated ones from the back -- both in halo order, which keeps the sums bit-reproducible
  double h1 = 0.0, hA = 0.0;
  for (int m0 = 0; m0 < a.nm; m0 += OT_T) {
    const int m = m0 + tid;
    int cls = 0;                                               // 1: interior, 2: mixed
    double4 mt = make_double4(0.0, 0.0, 0.0, 0.0);
    double aA = 0, bA = 0, c4 = 0, w2 = 0;
    if (m < a.nm) {
      mt = *reinterpret_cast<const double4*>(a.tmeta + (zrowp + m) * 4);
      const double2* c = reinterpret_cast<const double2*>(a.coef + (zrow + m) * 8);
      const double2 c01 = c[0], c45 = c[2];
      aA = c01.x; bA = c01.y; c4 = c45.x; w2 = c45.y;         // both legs are the same tracer
      const double tlo = kmn * mt.x, thi = kmx * mt.x;
      if (thi < 1.0 || tlo > tJ) {
        const double u = (thi < 1.0) ? mt.y : 0.0;              // the whole tile holds u_1, or is zero
        const double tA = fma(bA, u, aA);
        h1 = fma(c4 * tA, tA, h1); hA = fma(w2, tA, hA);
      } else {
        cls = (tlo >= 1.0 && thi <= tJ && thi < (double)min(a.J - 1, (int)mt.z) + 1.0) ? 1 : 2;
      }
    }
    const unsigned balI = __ballot_sync(0xffffffffu, cls == 1), balM = __ballot_sync(0xffffffffu, cls == 2);
    if (lane == 0) { wcnt[warp] = __popc(balI); wcnt2[warp] = __popc(balM); }
    __syncthreads();
    int baseI = nlist, baseM = nlist2, totI = 0, totM = 0;
#pragma unroll
    for (int w = 0; w < OT_T / 32; ++w) {
      baseI += (w < warp) ? wcnt[w] : 0; totI += wcnt[w];
      baseM += (w < warp) ? wcnt2[w] : 0; totM += wcnt2[w];
    }
    __syncthreads();                                       // everyone has read the list lengths and the counts
    if (tid == 0) { nlist += totI; nlist2 += totM; }
    if (cls) {
      const unsigned bal = cls == 1 ? balI : balM;
      const int pos = (cls == 1 ? baseI : baseM) + __popc(bal & ((1u << lane) - 1u));
      const int slot = cls == 1 ? pos : a.nm - 1 - pos;
      HMV_DEV_ASSERT(slot >= 0 && slot < a.nm);
      prm[slot] = make_double4(mt.x, mt.y, aA, bA);
      prm2[slot] = make_double2(c4, w2);
      rowid[slot] = (m << 12) | min(a.J - 1, (int)mt.z);         // halo index and bin cap (J - 1 < 4096 checked on the host)
    }
  }
  h1 = warp_sum(h1); hA = warp_sum(hA);
  if (lane == 0) { red[0][warp] = h1; red[1][warp] = hA; }
  __syncthreads();
  h1 = hA = 0.0;
#pragma unroll
  for (int w = 0; w < OT_T / 32; ++w) { h1 += red[0][w]; hA += red[1][w]; }
  const int nI = nlist, nM = nlist2;

  const int kc = min(k0 + 2 * tid, a.nk - 1), kc1 = min(k0 + 2 * tid + 1, a.nk - 1);
  const double kx = a.ks[kc], ky = a.ks[kc1];
  double p1x = 0, p1y = 0, iAx = 0, iAy = 0;
  // interior halos: j = floor(t) needs no clamp, the value no classification
#pragma unroll OT_UNROLL
  for (int i = 0; i < nI; ++i) {
    const double4 q = prm[i];
    const double2 q2 = prm2[i];
    const double* row = a.tab + (zrowp + (rowid[i] >> 12)) * (long long)a.JS;
    const double tx = kx * q.x, ty = ky * q.x;
    const int jx = __double2int_rz(tx), jy = __double2int_rz(ty);
    HMV_DEV_ASSERT(jx >= 1 && jy >= 1 && jx + 1 < a.JS && jy + 1 < a.JS && jx <= (rowid[i] & 4095) && jy <= (rowid[i] & 4095));
    const double uax = __ldg(row + jx), ubx = __ldg(row + jx + 1), uay = __ldg(row + jy), uby = __ldg(row + jy + 1);
    const double ux = fma(tx - (double)jx, ubx - uax, uax), uy = fma(ty - (double)jy, uby - uay, uay);
    const double tAx = fma(q.w, ux, q.z), tAy = fma(q.w, uy, q.z);
    p1x = fma(q2.x * tAx, tAx, p1x); p1y = fma(q2.x * tAy, tAy, p1y);
    iAx = fma(q2.y, tAx, iAx); iAy = fma(q2.y, tAy, iAy);
  }
  // halos whose tile crosses the first or the last bin
#pragma unroll 2
  for (int i = a.nm - 1; i > a.nm - 1 - nM; --i) {
    const double4 q = prm[i];
    const double2 q2 = prm2[i];
    const int id = rowid[i];
    const int jcap = id & 4095;
    const double* row = a.tab + (zrowp + (id >> 12)) * (long long)a.JS;
    const double inv = q.x, u1 = q.y;
    double ue[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const double t = (e ? ky : kx) * inv;
      const int jj = min(max(__double2int_rz(fmin(t, tJ)), 1), jcap);
      const double ua = __ldg(row + jj), ub = __ldg(row + jj + 1);
      double v = fma(t - (double)jj, ub - ua, ua);
      v = (t > tJ) ? 0.0 : v;
      ue[e] = (t >= 1.0) ? v : u1;
    }
    const double tAx = fma(q.w, ue[0], q.z), tAy = fma(q.w, ue[1], q.z);
    p1x = fma(q2.x * tAx, tAx, p1x); p1y = fma(q2.x * tAy, tAy, p1y);
    iAx = fma(q2.y, tAx, iAx); iAy = fma(q2.y, tAy, iAy);
  }
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    const int k = k0 + 2 * tid + e;
    if (k >= a.nk) break;
    const long long o = (long long)z * a.nk + k;
    if (a.p1h) a.p1h[o] = ((e ? p1y : p1x) + h1) * damp_1h(a.ks[k], a.kstar);
    if (a.p2h) {
      const double I = (e ? iAy : iAx) + hA + a.zoff[2 * z];
      a.p2h[o] = a.Pzk[o] * I * I;                                                                           // hmvec.py:572
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Spectra-only fusion: the six spectra with the NFW matter profile evaluated IN the reduction instead of being read
// from a cube.  u_NFW(k|M,z) is a function of s = k r_s c (1+z) given by piecewise polynomials (nfw_poly.cuh,
// k_nfw.cu), so a per-halo record of NFW_REC doubles -- the halo's NFWP_REC polynomial coefficients, then
// {c, a = r_s (1+z), a c, ln(1+c), 1/m_c, 0} -- replaces an 8*nk-byte cube row: the kernel streams only the electron
// cube (half the HBM traffic of power_six_kernel and no 32 GB NFW store/reload) and spends the freed time in the FP64
// pipe on the Horner chains.  Beyond the last polynomial interval (s > 64) u_NFW takes its closed form (Si/Ci).
// Same ring as power_six_kernel; stage = SIX_R rows x (4 KB of u_e + 64 B coefficients + NFW_REC doubles of NFW record).
// k tiles are the slow grid dimension, highest k first: the tiles that reach the closed form are scheduled first.
// ---------------------------------------------------------------------------------------------------------
// {min, max} of ks over [b*tile, (b+1)*tile) for each block b (one warp per block)
__global__ void tile_range_kernel(int nk, int tile, const double* __restrict__ ks, double* __restrict__ tilek) {
  const int b = blockIdx.x, lane = threadIdx.x;
  double mn = 1.0e300, mx = 0.0;
  for (int k = b * tile + lane; k < min(nk, (b + 1) * tile); k += 32) { mn = fmin(mn, ks[k]); mx = fmax(mx, ks[k]); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if (lane == 0) { tilek[2 * b] = mn; tilek[2 * b + 1] = mx; }
}

constexpr int FSX_NST = 6;
constexpr int FSX_STAGE_DOUBLES = SIX_R * SIX_K + SIX_R * 8 + SIX_R * NFW_REC;

struct FusedArgs {
  int nm, nk, ldk;
  const double *ue, *coef, *rec;
  SixOut out;
};

constexpr int FSX_CT = 512;   // consumer threads: one k each (16 warps keep the FP64 pipe fed through the Horner chains)

// u_NFW of one wavenumber for two halo rows at once (two interleaved Horner chains).  The 32 adjacent wavenumbers of a
// warp almost always share an interval, so the per-lane coefficient loads are shared-memory broadcasts; the loop runs
// to the highest degree present in the warp (lower ones are zero padded); beyond s = 64: the closed form.
__device__ __forceinline__ void nfw_poly_pair(const NfwpTables& T, const double* __restrict__ r0,
                                              const double* __restrict__ r1, double kk, double& um0, double& um1) {
  const double s0 = kk * r0[NFWP_REC + 2], s1 = kk * r1[NFWP_REC + 2];
  const int i0 = nfwp_lookup(T, s0), i1 = nfwp_lookup(T, s1);
  const int j0 = min(i0, NFWP_NI - 1), j1 = min(i1, NFWP_NI - 1);
  const double2 m0 = T.map[j0], m1 = T.map[j1];
  const double t0 = fma(s0 * s0, m0.x, m0.y), t1 = fma(s1 * s1, m1.x, m1.y);
  const int D = __reduce_max_sync(0xffffffffu, max(T.deg[j0], T.deg[j1]));
  const double* c0 = r0 + j0 * NFWP_STRIDE;
  const double* c1 = r1 + j1 * NFWP_STRIDE;
  double2 a0 = *reinterpret_cast<const double2*>(c0 + D - 1), a1 = *reinterpret_cast<const double2*>(c1 + D - 1);
  double u0 = fma(a0.y, t0, a0.x), u1 = fma(a1.y, t1, a1.x);
  for (int j = D - 3; j >= 0; j -= 2) {
    a0 = *reinterpret_cast<const double2*>(c0 + j);
    a1 = *reinterpret_cast<const double2*>(c1 + j);
    u0 = fma(fma(u0, t0, a0.y), t0, a0.x);
    u1 = fma(fma(u1, t1, a1.y), t1, a1.x);
  }
  if (i0 >= NFWP_NI) {
    const double x = kk * r0[NFWP_REC + 1], c = r0[NFWP_REC];
    u0 = (x > 4.0 ? nfw_bracket_far(x, c) : nfw_bracket(x, c, r0[NFWP_REC + 3])) * r0[NFWP_REC + 4];
  }
  if (i1 >= NFWP_NI) {
    const double x = kk * r1[NFWP_REC + 1], c = r1[NFWP_REC];
    u1 = (x > 4.0 ? nfw_bracket_far(x, c) : nfw_bracket(x, c, r1[NFWP_REC + 3])) * r1[NFWP_REC + 4];
  }
  um0 = u0; um1 = u1;
}

__global__ void __launch_bounds__(FSX_CT + 32, 1) power_six_nfw_kernel(const FusedArgs a) {
  extern __shared__ __align__(128) unsigned char six_smem[];
  __shared__ NfwpTables T;
  const BulkRing ring(six_smem, FSX_NST, FSX_STAGE_DOUBLES, FSX_CT / 32);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int z = blockIdx.x, k0 = (gridDim.y - 1 - blockIdx.y) * SIX_K;
  const int segk = min(SIX_K, a.ldk - k0);
  const long long zrow = (long long)z * a.nm;
  const int nit = (a.nm + SIX_R - 1) / SIX_R;
  const int k = k0 + tid;
  const bool active = tid < FSX_CT && k < a.nk;
  const double kk = __ldg(a.out.ks + min(k, a.nk - 1));   // idle lanes evaluate a valid wavenumber and discard it
  nfwp_tables_init(T, tid);
  __syncthreads();
  RingSlot slot;

  if (warp == FSX_CT / 32) {            // ---- producer warp ----
    if (lane == 0) {
      const unsigned segb = (unsigned)segk * 8u;
      for (int it = 0; it < nit; ++it, ring.advance(slot)) {
        const int m0 = it * SIX_R, rows = min(SIX_R, a.nm - m0);
        const RingStage st = ring.acquire<true>(slot, (unsigned)rows * (segb + 64u + NFW_REC * 8u));
        for (int r = 0; r < rows; ++r) {
          bulk_g2s(st.p + r * SIX_K, a.ue + (zrow + m0 + r) * (long long)a.ldk + k0, segb, st.full);
          double* rr = st.p + SIX_R * SIX_K + SIX_R * 8 + r * NFW_REC;
          bulk_g2s(rr, a.rec + (zrow + m0 + r) * NFW_REC, NFW_REC * 8u, st.full);
        }
        bulk_g2s(st.p + SIX_R * SIX_K, a.coef + (zrow + m0) * 8, (unsigned)rows * 64u, st.full);
      }
    }
    return;
  }

  // ---- consumers: thread owns wavenumber k over the whole mass axis ----
  double acc[9] = {};
  for (int it = 0, mleft = a.nm; it < nit; ++it, mleft -= SIX_R, ring.advance(slot)) {
    const int rows = min(SIX_R, mleft);
    const double* st = ring.wait(slot);
    const double* recs = st + SIX_R * SIX_K + SIX_R * 8;
    const double* cfs = st + SIX_R * SIX_K;
#pragma unroll 1
    for (int r = 0; r < rows; r += 2) {
      const double* r0 = recs + r * NFW_REC;
      const bool two = r + 1 < rows;
      const double* r1 = two ? r0 + NFW_REC : r0;
      double um0, um1;
      nfw_poly_pair(T, r0, r1, kk, um0, um1);
      six_fma(acc, six_coef(cfs + r * 8), um0, st[r * SIX_K + min(tid, segk - 1)]);
      if (two) six_fma(acc, six_coef(cfs + (r + 1) * 8), um1, st[(r + 1) * SIX_K + min(tid, segk - 1)]);
    }
    ring.release(slot);
  }
  if (!active) return;
  six_epilogue(a.out, z, a.nk, k, acc);
}

static bool aligned16(const void* p) { return ((unsigned long long)p & 15ull) == 0; }

static int tracer_args(const hmv_tracer* t, const char* which, TracerArgs* out) {
  HMV_REQUIRE(t != nullptr, "hmv_power: tracer %s is null", which);
  HMV_REQUIRE(t->kind >= 0 && t->kind <= 2, "hmv_power: tracer %s has unknown kind %d", which, t->kind);
  HMV_REQUIRE(t->us_d != nullptr, "hmv_power: tracer %s has no profile cube", which);
  HMV_REQUIRE(aligned16(t->us_d) && aligned16(t->uc_d), "hmv_power: cubes must be 16-byte aligned (tracer %s)", which);
  if (t->kind == 1)
    HMV_REQUIRE(t->Nc_d && t->Ns_d && t->NcNs_d && t->NsNsm1_d && t->ngal_d, "hmv_power: hod tracer %s lacks occupation arrays", which);
  out->kind = t->kind; out->Nc = t->Nc_d; out->Ns = t->Ns_d; out->NcNs = t->NcNs_d; out->NsNsm1 = t->NsNsm1_d;
  out->ngal = t->ngal_d; out->bias = t->bias_d;
  return HMV_OK;
}

// lets `kernel` use `bytes` of dynamic shared memory
template <class Kernel>
static int smem_opt_in(Kernel kernel, const char* name, size_t bytes) {
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "%s smem opt-in (%zu B): %s", name, bytes, cudaGetErrorString(e));
  return HMV_OK;
}

// The part the three six-spectra entry points share: the checks of the common arguments (after the caller's own, so
// that a rejected call launches nothing), the spec_stride default and the coefficient prep.  `streamed` are the cubes
// or tables the kernel reads with bulk copies: non-null and 16-byte aligned.  The prep writes ws[z][m][8] and zoff.
static int six_setup(const char* fn, int nz, int nm, int nk, int ldk, std::initializer_list<const double*> streamed,
                     const double* ms_d, const double* ks_d, const double* nzm_d, const double* bh_d,
                     const double* Pzk_d, double rho_m0, double kstar, const double* Nc_d, const double* Ns_d,
                     const double* NcNs_d, const double* NsNsm1_d, const double* ngal_d, double* ws_d, double* zoff,
                     long long spec_stride, double* p1h_d, double* p2h_d, cudaStream_t st, SixOut& out) {
  HMV_REQUIRE(nz > 0 && nm >= 2 && nk > 0 && ldk >= nk, "%s: bad sizes (nz=%d nm=%d nk=%d ldk=%d)", fn, nz, nm, nk, ldk);
  HMV_REQUIRE(ms_d && ks_d && nzm_d && bh_d && Nc_d && Ns_d && NcNs_d && NsNsm1_d && ngal_d && ws_d, "%s: null pointer", fn);
  for (const double* p : streamed) HMV_REQUIRE(p != nullptr, "%s: null pointer", fn);
  HMV_REQUIRE(p2h_d == nullptr || Pzk_d != nullptr, "%s: P2h requested without Pzk", fn);
  bool al = (ldk & 1) == 0 && aligned16(ws_d);
  for (const double* p : streamed) al = al && aligned16(p);
  HMV_REQUIRE(al, "%s: cubes, tables and workspace must be 16-byte aligned with even ldk (bulk async copies)", fn);
  HMV_REQUIRE(spec_stride == 0 || spec_stride >= (long long)nz * nk, "%s: spec_stride smaller than nz*nk", fn);
  out.spec_stride = spec_stride ? spec_stride : (long long)nz * nk;
  out.zoff = zoff; out.ks = ks_d; out.Pzk = Pzk_d; out.kstar = kstar; out.p1h = p1h_d; out.p2h = p2h_d;
  power_six_prep_kernel<<<nz, 256, 0, st>>>(nm, ms_d, nzm_d, bh_d, rho_m0, Nc_d, Ns_d, NcNs_d, NsNsm1_d, ngal_d, ws_d,
                                            zoff);
  return check_launch("power_six_prep_kernel");
}

}  // namespace hmv
using namespace hmv;

extern "C" long long hmv_power_ws_doubles(int nz, int nm) {
  if (nz <= 0 || nm <= 0) return 0;
  return 8LL * nz * nm + 2LL * nz;   // [z][m][8] coefficient records + zoff[z][2]
}

extern "C" int hmv_power(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d,
                         const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0, double kstar,
                         const hmv_tracer* A, const hmv_tracer* B, double* ws_d, double* p1h_d, double* p2h_d,
                         void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2 && nk > 0 && ldk >= nk, "hmv_power: bad sizes (nz=%d nm=%d nk=%d ldk=%d)", nz, nm, nk, ldk);
  HMV_REQUIRE((ldk & 1) == 0 && aligned16(ws_d),
              "hmv_power: ldk must be even and the workspace 16-byte aligned (bulk async copies); ldk=%d", ldk);
  HMV_REQUIRE(nz <= 65535, "hmv_power: nz=%d exceeds grid.y limit 65535", nz);
  HMV_REQUIRE(ms_d && ks_d && nzm_d && bh_d && ws_d, "hmv_power: null pointer");
  HMV_REQUIRE(p2h_d == nullptr || Pzk_d != nullptr, "hmv_power: P2h requested without Pzk");
  TracerArgs ta, tb;
  int rc = tracer_args(A, "A", &ta);
  if (rc) return rc;
  rc = tracer_args(B, "B", &tb);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long cs = (long long)nz * nm;
  double* coef = ws_d;
  double* zoff = ws_d + 8 * cs;
  int form = 0;
  if (A->kind == 1 && B->kind == 1) form = 1;            // hmvec.py:510-511 (uses leg A's HOD only)
  power_prep_kernel<<<nz, 256, 0, st>>>(nm, ms_d, nzm_d, bh_d, rho_m0, ta, tb, form, coef, zoff);
  rc = check_launch("power_prep_kernel");
  if (rc) return rc;
  PairArgs a;
  a.nm = nm; a.nk = nk; a.ldk = ldk; a.form = form;
  a.coef = coef; a.zoff = zoff; a.ks = ks_d; a.Pzk = Pzk_d; a.kstar = kstar;
  a.p1h = p1h_d; a.p2h = p2h_d;
  auto launch = [&](const double* usA, const double* ucA, const double* usB, const double* ucB, PairArgs q) -> int {
    q.ncube = 0;
    auto role = [&](const double* ptr) -> int {
      if (!ptr) return -1;
      for (int c = 0; c < q.ncube; ++c)
        if (q.cube[c] == ptr) return c;
      q.cube[q.ncube] = ptr;
      return q.ncube++;
    };
    q.rusA = role(usA); q.rucA = role(ucA); q.rusB = role(usB); q.rucB = role(ucB);
    if (q.form == 0 && q.ncube == 1 && q.rusA == 0 && q.rusB == 0 && q.rucA < 0 && q.rucB < 0) {
      // one cube, no central-profile cube: the streamlined kernel (uc == 1 is folded into aA, aB)
      const size_t smem = BulkRing::smem_bytes(ONE_NST, ONE_STAGE_DOUBLES);
      int r = smem_opt_in(power_one_kernel, "power_one_kernel", smem);
      if (r) return r;
      dim3 grid(cdiv(ldk, ONE_K), nz);
      power_one_kernel<<<grid, ONE_CT + 32, smem, st>>>(q);
      return check_launch("power_one_kernel");
    }
    const int stage_doubles = q.ncube * PR_R * PR_K + PR_R * 8;
    q.nst = (int)((200 * 1024) / (stage_doubles * sizeof(double)));
    if (q.nst > 6) q.nst = 6;
    const size_t smem = BulkRing::smem_bytes(q.nst, stage_doubles);
    int r = smem_opt_in(power_pair_kernel, "power_pair_kernel", smem);
    if (r) return r;
    dim3 grid(cdiv(ldk, PR_K), nz);
    power_pair_kernel<<<grid, PR_CT + 32, smem, st>>>(q);
    return check_launch("power_pair_kernel");
  };
  if (A->kind == 2 && B->kind == 2 && A->us_d != B->us_d && p1h_d) {
    // both pressure: the 1h integrand is pk_A^2 (hmvec.py:512-513) while the 2h legs stay A and B.
    // Leg-B coefficient records equal leg A's for pressure (a=0, b=1), so one prep serves both passes.
    PairArgs a1 = a;
    a1.p2h = nullptr;
    rc = launch(A->us_d, A->uc_d, A->us_d, A->uc_d, a1);
    if (rc) return rc;
    a.p1h = nullptr;
    if (!p2h_d) return HMV_OK;
  }
  return launch(A->us_d, A->uc_d, B->us_d, B->uc_d, a);
}

extern "C" int hmv_power_response(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d,
                                  const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                                  const double* uA_d, int kindA, const double* uB_d, int kindB, double* ws_d,
                                  double* r1h_d, double* r2h_d, void* stream) {
  const char* fn = "hmv_power_response";
  HMV_REQUIRE(nz >= 1 && nm >= 1 && nk >= 2, "%s: sizes must be >= 1 and nk >= 2 (nz=%d nm=%d nk=%d)", fn, nz, nm, nk);
  HMV_REQUIRE(ldk >= nk && (ldk & 1) == 0, "%s: ldk must be even and >= nk (ldk=%d nk=%d)", fn, ldk, nk);
  HMV_REQUIRE(ms_d && ks_d && nzm_d && bh_d && Pzk_d && uA_d && uB_d && ws_d, "%s: null pointer", fn);
  HMV_REQUIRE(r1h_d || r2h_d, "%s: null pointer (r1h and r2h are both NULL)", fn);
  HMV_REQUIRE(kindA == 0 || kindA == 2, "%s: cube A: kind %d is neither 0 (matter) nor 2 (pressure)", fn, kindA);
  HMV_REQUIRE(kindB == 0 || kindB == 2, "%s: cube B: kind %d is neither 0 (matter) nor 2 (pressure)", fn, kindB);
  HMV_REQUIRE(aligned16(uA_d), "%s: cube A must be 16-byte aligned", fn);
  HMV_REQUIRE(aligned16(uB_d), "%s: cube B must be 16-byte aligned", fn);
  HMV_REQUIRE(aligned16(ws_d), "%s: workspace must be 16-byte aligned", fn);
  if (nz > 65535) return fail(HMV_E_LIMIT, "%s: nz=%d exceeds 65535 (grid y of the streaming kernel)", fn, nz);
  cudaStream_t st = (cudaStream_t)stream;
  double* coef = ws_d;
  double* zoff = ws_d + 8LL * nz * nm;
  TracerArgs ta, tb;
  ta.kind = kindA; tb.kind = kindB;
  ta.Nc = ta.Ns = ta.NcNs = ta.NsNsm1 = ta.ngal = ta.bias = nullptr;
  tb.Nc = tb.Ns = tb.NcNs = tb.NsNsm1 = tb.ngal = tb.bias = nullptr;
  PairArgs a;
  a.nm = nm; a.nk = nk; a.ldk = ldk; a.form = 0;
  a.coef = coef; a.zoff = zoff; a.ks = ks_d; a.Pzk = Pzk_d; a.kstar = 0.0;
  a.p1h = r1h_d; a.p2h = r2h_d;
  a.cube[0] = uA_d; a.cube[1] = uB_d; a.cube[2] = a.cube[3] = nullptr;
  a.rusA = 0; a.rusB = uB_d == uA_d ? 0 : 1; a.rucA = a.rucB = -1;
  a.ncube = a.rusB + 1;
  const int stage_doubles = a.ncube * PR_R * PR_K + PR_R * 8;
  a.nst = a.ncube == 1 ? ONE_NST : (int)((200 * 1024) / (stage_doubles * sizeof(double)));
  if (a.nst > 6) a.nst = 6;
  const size_t smem = a.ncube == 1 ? BulkRing::smem_bytes(ONE_NST, ONE_STAGE_DOUBLES) : BulkRing::smem_bytes(a.nst, stage_doubles);
  int rc = a.ncube == 1 ? smem_opt_in(power_one_resp_kernel, "power_one_resp_kernel", smem)
                        : smem_opt_in(power_pair_resp_kernel, "power_pair_resp_kernel", smem);
  if (rc) return rc;
  power_resp_prep_kernel<<<nz, 256, 0, st>>>(nm, ms_d, nzm_d, bh_d, rho_m0, ta, tb, coef, zoff);
  rc = check_launch("power_resp_prep_kernel");
  if (rc) return rc;
  if (a.ncube == 1) {             // one cube: power_one's body (t = a + b u folded into the records)
    power_one_resp_kernel<<<dim3(cdiv(ldk, ONE_K), nz), ONE_CT + 32, smem, st>>>(a);
    return check_launch("power_one_resp_kernel");
  }
  power_pair_resp_kernel<<<dim3(cdiv(ldk, PR_K), nz), PR_CT + 32, smem, st>>>(a);
  return check_launch("power_pair_resp_kernel");
}

extern "C" int hmv_power_six(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d,
                             const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                             double kstar, const double* um_d, const double* ue_d, const double* Nc_d,
                             const double* Ns_d, const double* NcNs_d, const double* NsNsm1_d, const double* ngal_d,
                             double* ws_d, long long spec_stride, double* p1h_d, double* p2h_d, void* stream) {
  HMV_REQUIRE(nz <= 65535, "hmv_power_six: nz=%d exceeds grid.y limit 65535", nz);
  cudaStream_t st = (cudaStream_t)stream;
  SixArgs a;
  int rc = six_setup("hmv_power_six", nz, nm, nk, ldk, {um_d, ue_d}, ms_d, ks_d, nzm_d, bh_d, Pzk_d, rho_m0, kstar,
                     Nc_d, Ns_d, NcNs_d, NsNsm1_d, ngal_d, ws_d, ws_d + 8LL * nz * nm, spec_stride, p1h_d, p2h_d, st,
                     a.out);
  if (rc) return rc;
  a.nm = nm; a.nk = nk; a.ldk = ldk; a.um = um_d; a.ue = ue_d; a.coef = ws_d;
  const size_t smem = BulkRing::smem_bytes(SIX_NST, SIX_STAGE_DOUBLES);
  rc = smem_opt_in(power_six_kernel, "power_six_kernel", smem);
  if (rc) return rc;
  a.tk = wave_tile(nz, ldk, SIX_K, 1);
  dim3 grid(cdiv(ldk, a.tk), nz);
  power_six_kernel<<<grid, SIX_CT + 32, smem, st>>>(a);
  return check_launch("power_six_kernel");
}

extern "C" long long hmv_power_six_tab_ws_doubles(int nz, int nm, int nk) {
  if (nz <= 0 || nm <= 0 || nk <= 0) return 0;
  return hmv_power_ws_doubles(nz, nm);
}

extern "C" int hmv_power_six_tab(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d,
                                 const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0,
                                 double kstar, const double* um_d, const double* etab_d, int nxs, const double* Nc_d,
                                 const double* Ns_d, const double* NcNs_d, const double* NsNsm1_d, const double* ngal_d,
                                 double* ws_d, long long spec_stride, double* p1h_d, double* p2h_d, void* stream) {
  HMV_REQUIRE(nxs >= 4, "hmv_power_six_tab: bad sizes (nxs=%d)", nxs);
  HMV_REQUIRE(nz <= 65535, "hmv_power_six_tab: nz=%d exceeds grid.y limit 65535", nz);
  cudaStream_t st = (cudaStream_t)stream;
  SixTabArgs a;
  int rc = six_setup("hmv_power_six_tab", nz, nm, nk, ldk, {um_d, etab_d}, ms_d, ks_d, nzm_d, bh_d, Pzk_d, rho_m0,
                     kstar, Nc_d, Ns_d, NcNs_d, NsNsm1_d, ngal_d, ws_d, ws_d + 8LL * nz * nm, spec_stride, p1h_d,
                     p2h_d, st, a.out);
  if (rc) return rc;
  a.nm = nm; a.nk = nk; a.ldk = ldk; a.um = um_d; a.coef = ws_d;
  a.JS = (int)hmv_profile_table_stride(nxs); a.J = nxs / 2; a.nmp = cdiv(nm, 16) * 16;
  a.tab = etab_d; a.tmeta = etab_d + (size_t)nz * a.nmp * (size_t)a.JS;
  const size_t smem = BulkRing::smem_bytes(TAB_NST, TAB_STAGE_DOUBLES);
  rc = smem_opt_in(power_six_tab_kernel, "power_six_tab_kernel", smem);
  if (rc) return rc;
  dim3 grid(cdiv(ldk, SIX_K), nz);
  power_six_tab_kernel<<<grid, TAB_CT + 32, smem, st>>>(a);
  return check_launch("power_six_tab_kernel");
}

extern "C" int hmv_power_tab(int nz, int nm, int nk, const double* ms_d, const double* ks_d, const double* nzm_d,
                             const double* bh_d, const double* Pzk_d, double rho_m0, double kstar, int kind,
                             const double* tab_d, int nxs, double* ws_d, double* p1h_d, double* p2h_d, void* stream) {
  HMV_REQUIRE(nz > 0 && nm >= 2 && nk > 0 && nxs >= 4, "hmv_power_tab: bad sizes");
  HMV_REQUIRE(nz <= 65535, "hmv_power_tab: nz=%d exceeds grid.y limit 65535", nz);
  HMV_REQUIRE(kind == 0 || kind == 2, "hmv_power_tab: kind must be 0 (matter profile) or 2 (pressure profile)");
  HMV_REQUIRE(ms_d && ks_d && nzm_d && bh_d && tab_d && ws_d, "hmv_power_tab: null pointer");
  HMV_REQUIRE(p2h_d == nullptr || Pzk_d != nullptr, "hmv_power_tab: P2h requested without Pzk");
  HMV_REQUIRE(aligned16(tab_d) && aligned16(ws_d), "hmv_power_tab: tables and workspace must be 16-byte aligned");
  HMV_REQUIRE(nxs / 2 <= 4096 && nm < (1 << 19), "hmv_power_tab: nxs <= 8192 and nm < 2^19 (packed row ids)");
  const size_t smem = (size_t)nm * (sizeof(double4) + sizeof(double2) + sizeof(int)) + 16;
  if (smem > 200 * 1024) return fail(HMV_E_LIMIT, "hmv_power_tab: nm=%d needs %zu B of shared memory", nm, smem);
  cudaStream_t st = (cudaStream_t)stream;
  const long long cs = (long long)nz * nm;
  double* coef = ws_d;
  double* zoff = ws_d + 8 * cs;
  TracerArgs t;
  t.kind = kind; t.Nc = t.Ns = t.NcNs = t.NsNsm1 = t.ngal = t.bias = nullptr;
  power_prep_kernel<<<nz, 256, 0, st>>>(nm, ms_d, nzm_d, bh_d, rho_m0, t, t, 0, coef, zoff);
  int rc = check_launch("power_prep_kernel");
  if (rc) return rc;
  OneTabArgs a;
  a.nm = nm; a.nk = nk; a.nz = nz; a.coef = coef; a.zoff = zoff; a.ks = ks_d; a.Pzk = Pzk_d; a.kstar = kstar;
  a.p1h = p1h_d; a.p2h = p2h_d;
  a.JS = (int)hmv_profile_table_stride(nxs); a.J = nxs / 2; a.nmp = cdiv(nm, 16) * 16;
  a.tab = tab_d; a.tmeta = tab_d + (size_t)nz * a.nmp * (size_t)a.JS;
  rc = smem_opt_in(power_one_tab_kernel, "power_one_tab_kernel", smem);
  if (rc) return rc;
  power_one_tab_kernel<<<(unsigned)nz * cdiv(nk, OT_K), OT_T, smem, st>>>(a);
  return check_launch("power_one_tab_kernel");
}

extern "C" long long hmv_power_six_nfw_ws_doubles(int nz, int nm) {
  if (nz <= 0 || nm <= 0) return 0;
  return (8LL + NFW_REC) * nz * nm + 2LL * nz + 4;   // coefficient records + NFW records + zoff + max(ks)
}

extern "C" int hmv_power_six_nfw(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ms_d,
                                 const double* ks_d, const double* nzm_d, const double* bh_d, const double* Pzk_d,
                                 double rho_m0, double kstar, const double* cs_d, const double* rvir_d,
                                 const double* ue_d, const double* Nc_d, const double* Ns_d, const double* NcNs_d,
                                 const double* NsNsm1_d, const double* ngal_d, double* ws_d, long long spec_stride,
                                 double* p1h_d, double* p2h_d, void* stream) {
  HMV_REQUIRE(cdiv(ldk, SIX_K) <= 65535, "hmv_power_six_nfw: grid limit");
  HMV_REQUIRE(zs_d && cs_d && rvir_d, "hmv_power_six_nfw: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const long long cs = (long long)nz * nm;
  double* coef = ws_d;
  double* rec = ws_d + 8 * cs;
  double* zoff = rec + NFW_REC * cs;
  double* kmax_dev = zoff + 2 * nz + ((2 * nz) & 1);
  FusedArgs a;
  int rc = six_setup("hmv_power_six_nfw", nz, nm, nk, ldk, {ue_d}, ms_d, ks_d, nzm_d, bh_d, Pzk_d, rho_m0, kstar, Nc_d,
                     Ns_d, NcNs_d, NsNsm1_d, ngal_d, ws_d, zoff, spec_stride, p1h_d, p2h_d, st, a.out);
  if (rc) return rc;
  tile_range_kernel<<<1, 32, 0, st>>>(nk, nk, ks_d, kmax_dev);          // {min, max} of ks
  rc = check_launch("tile_range_kernel");
  if (rc) return rc;
  rc = nfw_poly_records(cs, nm, 1, kmax_dev + 1, zs_d, cs_d, rvir_d, rec, st);
  if (rc) return rc;
  a.nm = nm; a.nk = nk; a.ldk = ldk; a.ue = ue_d; a.coef = coef; a.rec = rec;
  const size_t smem = BulkRing::smem_bytes(FSX_NST, FSX_STAGE_DOUBLES);
  rc = smem_opt_in(power_six_nfw_kernel, "power_six_nfw_kernel", smem);
  if (rc) return rc;
  dim3 grid(nz, cdiv(ldk, SIX_K));
  power_six_nfw_kernel<<<grid, FSX_CT + 32, smem, st>>>(a);
  return check_launch("power_six_nfw_kernel");
}

// host-side introspection for the CPU tests: the k-tile width hmv_power_six picks for an nz x ldk launch, and the
// (z, k0) of every CTA of hmv_power_tab's launch order (returns the tile width of that kernel)
extern "C" int hmv_debug_wave_tile(int nz, int ldk) {
  HMV_REQUIRE(nz > 0 && ldk > 0, "hmv_debug_wave_tile: bad sizes");
  return wave_tile(nz, ldk, SIX_K, 1);
}
extern "C" int hmv_debug_tab_order(int nz, int nk, int* z_out, int* k0_out) {
  HMV_REQUIRE(nz > 0 && nk > 0 && z_out && k0_out, "hmv_debug_tab_order: bad arguments");
  const int T = cdiv(nk, OT_K);
  for (int i = 0; i < nz * T; ++i) ot_cta(i, nz, nk, z_out[i], k0_out[i]);
  return OT_K;
}
