// k_nfw.cu -- K2: analytic truncated-NFW Fourier profile u(k|M,z) (reference hmvec.py:339-353).
//
// The reference evaluates  u = [sin x (Si X - Si x) - sin(cx)/X + cos x (Ci X - Ci x)]/m_c,  X=(1+c)x, x = k r_s (1+z),
// with two scipy.special.sici calls per (z,M,k).  That closed form is the integral
//        u(x; c) = (1/m_c) int_0^c  t/(1+t)^2  sinc(x t) dt .
//
// Here it is evaluated as piecewise polynomials.  u_NFW depends on the halo through c alone once written in s = x c,
// and is smooth in y = s^2: on 21 fixed intervals of s (edges 0,1,2,4,...,16,20,...,64) a per-halo polynomial of degree
// 5..13 in the interval's local variable t reproduces it to < 2e-11 of the interval's max|u| for 0.6 <= c <= 25
// (tools/gen_nfw_poly_tables.py --check, mpmath), at ~13 FP64 instructions per element on the LARGE grid (66 % of the
// elements have s <= 1: degree 5) where the closed form costs ~90: the kernel is store-bound.  Beyond s = 64 u_NFW
// takes the closed form (nfw_bracket / nfw_bracket_far of sici.cuh).
//   nfw_chunk_kernel       : per 256-wide k chunk, min and max of ks, and padded copies of ks and ks^2
//   nfw_poly_gemm_kernel   : per halo, one record of NFW_REC doubles (polynomial coefficients and halo constants) from
//                            one FP64 tensor-core contraction
//   uk_nfw_poly_kernel     : one warp per halo row, 256-wide k chunks; a chunk whose min and max s fall into one
//                            interval runs Horner with warp-uniform coefficients (one shared-memory load per 16 FMAs);
//                            a chunk that straddles interval edges looks the coefficients up per element; elements
//                            beyond s = 64 (6.8 % on the LARGE grid, all with x > 4) take the closed form's asymptotic
//                            branch.  No assumption on the order of ks (chunk min/max come from a pre-pass).
#include "common.cuh"
#include "nfw_poly.cuh"

namespace hmv {

constexpr int NFW_T = 256, NFW_CH = 256;              // threads per CTA, wavenumbers per chunk

// per 256-wide chunk: min and max of ks; copies of ks and ks^2 padded to whole chunks (last value repeated), so the
// cube kernel reads 16-byte pairs without bounds checks
__global__ void nfw_chunk_kernel(int nk, const double* __restrict__ ks, double* __restrict__ kcmin,
                                 double* __restrict__ kcmax, double* __restrict__ ksp, double* __restrict__ k2p) {
  const int chunk = blockIdx.x, lane = threadIdx.x;
  double mx = 0.0, mn = 1.0e300;
  for (int k = chunk * NFW_CH + lane; k < (chunk + 1) * NFW_CH; k += 32) {
    const double v = ks[min(k, nk - 1)];
    mx = fmax(mx, v); mn = fmin(mn, v);
    ksp[k] = v;
    k2p[k] = v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, o));
  }
  if (lane == 0) { kcmax[chunk] = mx; kcmin[chunk] = mn; }
}

// Pre-pass: the polynomial coefficients of every halo as ONE dense contraction on the FP64 tensor cores.
// u(s; c) = (c^2/m_c) int_0^1 tau/(1 + c tau)^2 sinc(s tau) dtau; with 64-point Gauss-Legendre in tau and the (linear)
// map "values at an interval's Chebyshev nodes -> monomial coefficients", coefficient r = (interval, j) of a halo is
//        coef[halo][r] = sum_q R[halo][q] W[q][r],     R[halo][q] = (c^2/m_c) w_q tau_q / (1 + c tau_q)^2,
// where W (64 x 294, tools/gen_nfw_poly_tables.py, 50-digit arithmetic) holds the monomial coefficients of the
// interpolants of s -> sinc(s tau_q): O(1) numbers, so nothing is amplified (the 1e4-sized entries of the
// node->monomial matrices cancel inside W).  No Si/Ci, no series, no per-node branches: per 16 halos, 64 reciprocals
// per lane and 37 x 16 x 2 mma.sync m8n8k4 (SASS DMMA) with W resident in shared memory.  Checked against mpmath for
// 0.6 <= c <= 25: same error as exact node values (< 2e-11 of an interval's max|u|, the truncation error).
// The coefficients fill slots [0, NFWP_REC) of the halo's record, the constants {c, a = r_s (1+z), a c, ln(1+c), 1/m_c, 0}
// the last six.
constexpr int NFWP_MAXCH = 128;                          // chunks whose min/max the cube kernel keeps in shared memory
constexpr int NFWP_NT = (NFWP_REC + 7) / 8;              // 8-wide coefficient tiles
constexpr size_t NFWP_GEMM_SMEM = ((size_t)NFWP_Q * NFWP_WLD + 2 * NFWP_Q) * sizeof(double);

__global__ void __launch_bounds__(256, 1) nfw_poly_gemm_kernel(long long rows, int nm, int nchunks,
                                                               const double* __restrict__ kcmax,
                                                               const double* __restrict__ zs,
                                                               const double* __restrict__ cs,
                                                               const double* __restrict__ rvir,
                                                               double* __restrict__ rec) {
  extern __shared__ __align__(16) double gsm[];
  double* Wsm = gsm;                                     // [Q][WLD]
  double2* gl = reinterpret_cast<double2*>(gsm + (size_t)NFWP_Q * NFWP_WLD);   // {tau_q, w_q tau_q}
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  {
    const double2* src = reinterpret_cast<const double2*>(g_nfwp_W);
    double2* dst = reinterpret_cast<double2*>(Wsm);
    for (int i = tid; i < NFWP_Q * NFWP_WLD / 2; i += 256) dst[i] = src[i];
    if (tid < NFWP_Q) gl[tid] = g_nfwp_gl[tid];
  }
  double kmax = 0.0;                                     // max(ks) from the chunk pre-pass, not from the caller
  for (int i = lane; i < nchunks; i += 32) kmax = fmax(kmax, __ldg(kcmax + i));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) kmax = fmax(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
  __syncthreads();
  const long long ngroups = (rows + 15) / 16;
  for (long long grp = (long long)blockIdx.x * 8 + warp; grp < ngroups; grp += (long long)gridDim.x * 8) {
    double a0[NFWP_Q / 4], a1[NFWP_Q / 4];
    int ivtop = 0;
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const long long row = grp * 16 + g + 8 * mt;
      const bool ok = row < rows;
      const double c = ok ? __ldg(cs + row) : 1.0;
      const double ln1pc = log1p(c), mc = ln1pc - c / (1.0 + c);        // hmvec.py:348
      const double inv_mc = 1.0 / mc, pref = c * c * inv_mc;
      const double av = ok ? __ldg(rvir + row) / c * (1.0 + __ldg(zs + row / nm)) : 0.0;   // x = k r_s (1+z), hmvec.py:342,349
      if (ok && t4 == 0) {
        double2* r = reinterpret_cast<double2*>(rec + row * NFW_REC + NFWP_REC);
        r[0] = make_double2(c, av); r[1] = make_double2(av * c, ln1pc); r[2] = make_double2(inv_mc, 0.0);
      }
      ivtop = max(ivtop, ok ? min(NFWP_NI - 1, nfwp_interval(kmax * av * c)) : 0);
#pragma unroll
      for (int ks = 0; ks < NFWP_Q / 4; ++ks) {
        const double2 q = gl[4 * ks + t4];
        const double rd = rcp_fast(fma(c, q.x, 1.0));
        const double v = pref * q.y * (rd * rd);
        if (mt == 0) a0[ks] = v; else a1[ks] = v;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ivtop = max(ivtop, __shfl_xor_sync(0xffffffffu, ivtop, o));
    const int ntiles = min(NFWP_NT, ((ivtop + 1) * NFWP_STRIDE + 7) >> 3);   // intervals no halo of the group reaches are skipped
    for (int nt0 = 0; nt0 < ntiles; nt0 += 4) {
      double acc[4][2][2];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j][0][0] = acc[j][0][1] = acc[j][1][0] = acc[j][1][1] = 0.0;
      const double* Wb = Wsm + (size_t)t4 * NFWP_WLD + 8 * nt0 + g;
#pragma unroll
      for (int ks = 0; ks < NFWP_Q / 4; ++ks) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double bv = Wb[(size_t)(4 * ks) * NFWP_WLD + 8 * j];     // columns past 294 are zero padding (WLD = 296) ...
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                       : "+d"(acc[j][0][0]), "+d"(acc[j][0][1]) : "d"(a0[ks]), "d"(bv));
          asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                       : "+d"(acc[j][1][0]), "+d"(acc[j][1][1]) : "d"(a1[ks]), "d"(bv));
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = 8 * (nt0 + j) + 2 * t4;                              // ... and tiles past the table are not stored
        if (r < NFWP_REC) {
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            const long long row = grp * 16 + g + 8 * mt;
            if (row < rows) *reinterpret_cast<double2*>(rec + row * NFW_REC + r) = make_double2(acc[j][mt][0], acc[j][mt][1]);
          }
        }
      }
    }
  }
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}

// one element through the general route: the polynomial of its own interval, or the closed form beyond s = 64
__device__ __noinline__ double nfwp_element(const double* R, const NfwpTables& T, double kk, double ac, double a,
                                            double c, double ln1pc, double inv_mc) {
  const double s = kk * ac;
  const int iv = nfwp_lookup(T, s);
  if (iv >= NFWP_NI) {
    const double x = kk * a;
    return (x > 4.0 ? nfw_bracket_far(x, c) : nfw_bracket(x, c, ln1pc)) * inv_mc;
  }
  const double2 mp = T.map[iv];
  const double t = fma(s * s, mp.x, mp.y);
  const double* m = R + iv * NFWP_STRIDE;
  double u = 0.0;
#pragma unroll
  for (int j = NFWP_STRIDE - 1; j >= 0; --j) u = fma(u, t, m[j]);
  return u;
}

// One WARP per halo row, eight rows per CTA, no block-level synchronisation after the tables are staged: a warp copies
// its row's record into its own shared-memory slice, sweeps the leading chunks that lie entirely below s = 1 (two
// thirds of the LARGE grid's elements) in a tight loop with the six coefficients in registers, and takes the remaining
// chunks through the general route.  A lane owns four 16-byte pairs of a 256-wide chunk (coalesced 16-byte stores).
// Three CTAs per SM is what the register allocation aims at (four would cap it at 64 registers).
__global__ void __launch_bounds__(NFW_T, 3) uk_nfw_poly_kernel(long long rows, int nk, int ldk,
                                                                const double* __restrict__ ksp,
                                                                const double* __restrict__ k2p,
                                                                const double* __restrict__ rec,
                                                                const double* __restrict__ kcmin,
                                                                const double* __restrict__ kcmax,
                                                                double* __restrict__ uk) {
  __shared__ __align__(16) double Rall[NFW_T / 32][NFW_REC];
  __shared__ NfwpTables T;
  __shared__ double2 cmm[NFWP_MAXCH];                       // {min, max} of ks per chunk (when they fit)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long row = (long long)blockIdx.x * (NFW_T / 32) + warp;
  double* Rr = Rall[warp];
  const double* src = rec + min(row, rows - 1) * NFW_REC;   // a warp past the last row copies that row, then returns
  for (int i = lane; i < NFW_REC / 2; i += 32) cp_async16(Rr + 2 * i, src + 2 * i);
  asm volatile("cp.async.commit_group;" ::: "memory");
  nfwp_tables_init(T, tid);
  const int nchunks = (nk + NFW_CH - 1) / NFW_CH;
  const bool cmm_sm = nchunks <= NFWP_MAXCH;
  if (cmm_sm)
    for (int i = tid; i < nchunks; i += NFW_T) cmm[i] = make_double2(__ldg(kcmin + i), __ldg(kcmax + i));
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if (row >= rows) return;
  const double c = Rr[NFWP_REC], a = Rr[NFWP_REC + 1], ac = Rr[NFWP_REC + 2], ln1pc = Rr[NFWP_REC + 3],
               inv_mc = Rr[NFWP_REC + 4];
  const double ac2 = ac * ac;
  const int npair = nk >> 1;
  const double2* ks2 = reinterpret_cast<const double2*>(ksp);
  const double2* kq2 = reinterpret_cast<const double2*>(k2p);
  double* out = uk + row * (long long)ldk;
  double2* out2 = reinterpret_cast<double2*>(out);

  // ---- leading chunks entirely inside the first interval: degree 5, coefficients in registers ----
  int nA = 0;
  for (int b0 = 0; b0 < nchunks - 1; b0 += 32) {            // the last (possibly partial) chunk is left to the general loop
    const int b = b0 + lane;
    const double bmax = cmm_sm ? cmm[min(b, nchunks - 1)].y : __ldg(kcmax + min(b, nchunks - 1));
    const unsigned in0 = __ballot_sync(0xffffffffu, b < nchunks - 1 && bmax * ac < T.hi[0]);
    const int run = in0 == 0xffffffffu ? 32 : __ffs(~in0) - 1;
    nA += run;
    if (run < 32) break;
  }
  {
    static_assert(NFWP_STRIDE >= 6, "first interval");
    const double m0 = Rr[0], m1 = Rr[1], m2 = Rr[2], m3 = Rr[3], m4 = Rr[4], m5 = Rr[5];
    HMV_DEV_ASSERT(T.deg[0] == 5);
    const double ts = T.map[0].x * ac2, to = T.map[0].y;
    double2 kn[4];                                            // next chunk's k^2, loaded one trip ahead
#pragma unroll
    for (int q = 0; q < 4; ++q) kn[q] = __ldg(kq2 + lane + 32 * q);
    for (int chunk = 0; chunk < nA; ++chunk) {
      const int pbase = chunk * (NFW_CH / 2) + lane;
      HMV_DEV_ASSERT(chunk + 1 < nchunks && pbase + 96 < npair);
      double2 t[4], u[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) t[q] = make_double2(fma(kn[q].x, ts, to), fma(kn[q].y, ts, to));
#pragma unroll
      for (int q = 0; q < 4; ++q) kn[q] = __ldg(kq2 + pbase + NFW_CH / 2 + 32 * q);   // chunk + 1 < nchunks: in range
#pragma unroll
      for (int q = 0; q < 4; ++q) u[q] = make_double2(fma(m5, t[q].x, m4), fma(m5, t[q].y, m4));
#define HMV_STEP(mm)                                                                       \
  _Pragma("unroll") for (int q = 0; q < 4; ++q) { u[q].x = fma(u[q].x, t[q].x, mm); u[q].y = fma(u[q].y, t[q].y, mm); }
      HMV_STEP(m3) HMV_STEP(m2) HMV_STEP(m1) HMV_STEP(m0)
#undef HMV_STEP
#pragma unroll
      for (int q = 0; q < 4; ++q) __stcs(out2 + pbase + 32 * q, u[q]);   // streaming: keeps k, k^2 in L1
    }
  }

  // ---- the other chunks ----
  for (int chunk = nA; chunk < nchunks; ++chunk) {
    const double2 mm = cmm_sm ? cmm[chunk] : make_double2(__ldg(kcmin + chunk), __ldg(kcmax + chunk));
    const double smin = mm.x * ac, smax = mm.y * ac;
    const int pbase = chunk * (NFW_CH / 2) + lane;        // pair index of this lane's first pair
    double2 u[4];
    if (smin >= NFWP_SMAX) {                              // the whole chunk is beyond the polynomials: closed form
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const double2 kk = __ldg(ks2 + pbase + 32 * q);
        const double x0 = kk.x * a, x1 = kk.y * a;
        double2 v;
        if (x0 > 4.0 && x1 > 4.0) {
          v.x = nfw_bracket_far(x0, c) * inv_mc;
          v.y = nfw_bracket_far(x1, c) * inv_mc;
        } else {
          v.x = nfw_bracket(x0, c, ln1pc) * inv_mc;
          v.y = nfw_bracket(x1, c, ln1pc) * inv_mc;
        }
#pragma unroll
        for (int w = 0; w < 4; ++w)
          if (w == q) u[w] = v;
      }
    } else {
      const int ivlo = nfwp_lookup(T, smin), ivhi = nfwp_lookup(T, smax);
      double2 t[4];
      if (smax < T.hi[ivlo]) {                            // one interval (or just past its edge): warp-uniform coefficients
        const double2 mp = T.map[ivlo];
        const double ts = mp.x * ac2, to = mp.y;
        const int D = T.deg[ivlo];                        // odd
        HMV_DEV_ASSERT(ivlo >= 0 && ivlo < NFWP_NI && (D & 1) && D < NFWP_STRIDE);
        const double* m = Rr + ivlo * NFWP_STRIDE;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double2 k2 = __ldg(kq2 + pbase + 32 * q);
          t[q] = make_double2(fma(k2.x, ts, to), fma(k2.y, ts, to));
        }
        double2 a2 = *reinterpret_cast<const double2*>(m + D - 1);
#pragma unroll
        for (int q = 0; q < 4; ++q) u[q] = make_double2(fma(a2.y, t[q].x, a2.x), fma(a2.y, t[q].y, a2.x));
        for (int j = D - 3; j >= 0; j -= 2) {
          a2 = *reinterpret_cast<const double2*>(m + j);
#pragma unroll
          for (int q = 0; q < 4; ++q) { u[q].x = fma(u[q].x, t[q].x, a2.y); u[q].y = fma(u[q].y, t[q].y, a2.y); }
#pragma unroll
          for (int q = 0; q < 4; ++q) { u[q].x = fma(u[q].x, t[q].x, a2.x); u[q].y = fma(u[q].y, t[q].y, a2.x); }
        }
      } else {
        // several intervals: every pair looks up the interval of its smaller element; a pair that straddles an edge,
        // or reaches beyond s = 64, is redone element by element afterwards
        int off[4];
        unsigned redo = 0u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double2 kk = __ldg(ks2 + pbase + 32 * q);
          const double s0 = kk.x * ac, s1 = kk.y * ac;
          const int iv0 = nfwp_lookup(T, fmin(s0, s1));
          if (fmax(s0, s1) >= T.hi[iv0] || iv0 >= NFWP_NI) redo |= 1u << q;
          const int iv = min(iv0, NFWP_NI - 1);
          const double2 mp = T.map[iv];
          t[q] = make_double2(fma(s0 * s0, mp.x, mp.y), fma(s1 * s1, mp.x, mp.y));
          off[q] = iv * NFWP_STRIDE;
          HMV_DEV_ASSERT(iv >= 0 && iv < NFWP_NI);
          u[q] = make_double2(0.0, 0.0);
        }
        const int D = T.deg[min(ivhi, NFWP_NI - 1)];      // degrees do not decrease with s; lower ones are zero padded
        for (int j = D - 1; j >= 0; j -= 2) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const double2 a2 = *reinterpret_cast<const double2*>(Rr + off[q] + j);
            u[q].x = fma(fma(u[q].x, t[q].x, a2.y), t[q].x, a2.x);
            u[q].y = fma(fma(u[q].y, t[q].y, a2.y), t[q].y, a2.x);
          }
        }
        if (__any_sync(0xffffffffu, redo != 0u)) {
#pragma unroll 1
          for (int q = 0; q < 4; ++q)
            if (redo & (1u << q)) {
              const double2 kk = __ldg(ks2 + pbase + 32 * q);
              double2 v;
              v.x = nfwp_element(Rr, T, kk.x, ac, a, c, ln1pc, inv_mc);
              v.y = nfwp_element(Rr, T, kk.y, ac, a, c, ln1pc, inv_mc);
#pragma unroll
              for (int w = 0; w < 4; ++w)
                if (w == q) u[w] = v;
            }
        }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int pp = pbase + 32 * q;
      if (pp < npair) __stcs(out2 + pp, u[q]);
      else if (2 * pp < nk) out[2 * pp] = u[q].x;          // odd nk: the last wavenumber
    }
  }
}

int nfw_poly_records(long long rows, int nm, int nkmax, const double* kmax_d, const double* zs_d, const double* cs_d,
                     const double* rvir_d, double* rec, cudaStream_t st) {
  int dev = 0, nsm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(nfw_poly_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NFWP_GEMM_SMEM);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "nfw_poly_records: %s", cudaGetErrorString(e));
  const long long ngroups = (rows + 15) / 16;
  const int grid = (int)((ngroups + 7) / 8 < nsm ? (ngroups + 7) / 8 : nsm);
  nfw_poly_gemm_kernel<<<grid, 256, NFWP_GEMM_SMEM, st>>>(rows, nm, nkmax, kmax_d, zs_d, cs_d, rvir_d, rec);
  return check_launch("nfw_poly_gemm_kernel");
}

__global__ void sici_test_kernel(int n, const double* __restrict__ x, double* __restrict__ si,
                                 double* __restrict__ ci) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) sici(x[i], si[i], ci[i]);
}

}  // namespace hmv
using namespace hmv;

extern "C" int hmv_set_nfw_mode(int mode) {
  HMV_REQUIRE(mode == 0, "hmv_set_nfw_mode: mode %d does not exist; 0 (piecewise polynomials) is the only evaluation "
              "(the series + Si/Ci path, mode 1, was removed)", mode);
  return HMV_OK;
}

extern "C" long long hmv_uk_nfw_ws_doubles(int nz, int nm, int nk) {
  if (nz <= 0 || nm <= 0 || nk <= 0) return 0;
  // per-halo records, per-chunk min(k) and max(k), padded copies of k and k^2
  const long long nchunks = (nk + NFW_CH - 1) / NFW_CH;
  return (long long)nz * nm * NFW_REC + 2 * nchunks + 2 * nchunks * NFW_CH + 4;
}

extern "C" int hmv_uk_nfw(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
                          double kmax, const double* cs_d, const double* rvir_d, double* ws_d, double* uk_d,
                          void* stream) {
  HMV_REQUIRE(nz > 0 && nm > 0 && nk > 0 && ldk >= nk, "hmv_uk_nfw: bad sizes (nz=%d nm=%d nk=%d ldk=%d)", nz, nm, nk, ldk);
  HMV_REQUIRE(zs_d && ks_d && cs_d && rvir_d && ws_d && uk_d, "hmv_uk_nfw: null pointer");
  // the kernels move 16-byte words: an even row stride and 16-byte aligned rows and workspace
  HMV_REQUIRE((ldk & 1) == 0 && (((size_t)uk_d | (size_t)ws_d) & 15) == 0,
              "hmv_uk_nfw: uk_d and ws_d must be 16-byte aligned and ldk even (ldk=%d)", ldk);
  const long long rows = (long long)nz * nm;
  if (rows > 2147483647LL) return fail(HMV_E_LIMIT, "hmv_uk_nfw: %lld halo rows exceed the 2^31-1 grid limit", rows);
  cudaStream_t st = (cudaStream_t)stream;
  const int nchunks = (nk + NFW_CH - 1) / NFW_CH;
  double* rec = ws_d;                                    // NFW_REC is even: what follows stays 16-byte aligned
  double* ksp = rec + rows * NFW_REC;
  double* k2p = ksp + (size_t)nchunks * NFW_CH;
  double* kcmin = k2p + (size_t)nchunks * NFW_CH;
  double* kcmax = kcmin + nchunks;
  nfw_chunk_kernel<<<nchunks, 32, 0, st>>>(nk, ks_d, kcmin, kcmax, ksp, k2p);
  int rc = check_launch("nfw_chunk_kernel");
  if (rc) return rc;
  rc = nfw_poly_records(rows, nm, nchunks, kcmax, zs_d, cs_d, rvir_d, rec, st);
  if (rc) return rc;
  uk_nfw_poly_kernel<<<cdiv(rows, NFW_T / 32), NFW_T, 0, st>>>(rows, nk, ldk, ksp, k2p, rec, kcmin, kcmax, uk_d);
  return check_launch("uk_nfw_poly_kernel");
}

// test hook: elementwise Si/Ci of the device routine (x > 0)
extern "C" int hmv_sici_test(int n, const double* x_d, double* si_d, double* ci_d, void* stream) {
  HMV_REQUIRE(n > 0 && x_d && si_d && ci_d, "hmv_sici_test: bad arguments");
  sici_test_kernel<<<cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(n, x_d, si_d, ci_d);
  return check_launch("sici_test_kernel");
}
