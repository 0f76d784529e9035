// k_transform.cu -- K1: batched numerical profile transform fused with on-the-fly GNFW evaluation and the
// interpolation onto the target wavenumbers.  Replaces generic_profile_fft + fft_integral + _interp_loop
// (reference fft.py:35-115) and rho_gas_generic_x / P_e_generic_x (hmvec.py:856-860, 918-927).
//
// The (z,M,x) profile cube never exists: samples are evaluated chunk by chunk into shared memory, the sine sums
//        U_j = step * sum_n x_n y_n sin(2 pi j n / N)          ( == -Im rfft(x*y) * step, fft.py:49 )
// are accumulated only for the bins j the target k-range needs (bin skipping; the theta-cut bounds n), then
// u_j = U_j/kt_j/mnorm is linearly interpolated onto ks (direct index j = floor(k/kout_1), no search) and written
// once, coalesced.
//
// The sine matrix S[n][j] = sin(2 pi n j/N) is halo independent, so the sums are a dense contraction
// [halos x samples] x [samples x bins] and run on the FP64 tensor cores (mma.sync m8n8k4 -> SASS DMMA.8x8x4).
// A lane's B-operand element is sin(phi_j (s + 4 i)) for its fixed (bin j, sample offset): an arithmetic sequence of
// angles, advanced with the three-term recurrence  b_{i+1} = 2 cos(4 phi_j) b_i - b_{i-1}  and re-seeded exactly from
// a {sin,cos} table (global memory) at every sample chunk, which bounds the recurrence round-off at (chunk/4)^2 ulp/2
// (3e-12 for 704 samples).  Why tensor cores: DMMA has the DFMA pipe's peak on B200 (36.9 vs 35.0 TFLOP/s,
// tools/micro/dmma_bench.cu) but takes ONE issue slot per 256 FMAs; the per-thread DFMA form was issue-bound on
// phase-index arithmetic and a DMMA form fed from a shared-memory sine table was shared-memory bandwidth bound
// (0.74 wavefronts/cycle/SM: the 32 table addresses of a B fragment are effectively random, ~6 wavefronts per
// fragment) -- ncu evidence in profiles/.
//
// One launch plan: profile_transform_ws_kernel, ONE persistent kernel -- two independent 8-warp groups per SM, each
// evaluating + transforming 16 halos and then interpolating + storing their rows, so that one group's tensor-core phase
// overlaps the other's store phase.  The same kernel also runs the two phases as separate launches around a resident
// table array (hmv_profile_tables / hmv_profile_expand: consumers that only integrate over M read the tables and never
// need the cube).  Every entry point reads ks, the workspace and the cube / tables with 16-byte accesses.
#include <cstdlib>
#include "common.cuh"
#include "gnfw_eval.cuh"

namespace hmv {

struct TParams {
  int nz, nm, nk, ldk, N, J, JS, nmg, do_mass_norm;
  int jlo, jhi;           // unused; removing them shifts every later field's constant-bank offset in the kernel
  double gamma, dx, step, kt1, kmax;
  const double *zs, *ks, *rs, *cmax, *xc, *alpha, *expo, *amp, *outscale, *sintab, *rkt;
  const double* rho;      // user-supplied samples rho[z][m][n] = rho(x_n) (generic_profile_fft with any profile), or NULL
  // two-stage (Cooley-Tukey) form of the sine sums for items with many bins: N = TS_P * ts_Q
  int ts_Q, ts_QT;        // Q = N / TS_P (0: not available for this N), number of 8-wide q tiles
  const double *ts_a1, *ts_tw, *ts_a2;   // fragment-ordered twiddle tables (global)
  const int* jn_cta;
  double* uk;
  // table mode: the finished bin tables go to tab[z][nmp][JS] (nmp = nm rounded up to 16) with
  // {k -> bin factor, u_1, bin count, 0} per halo in tmeta[z][nmp][4], instead of a per-CTA slot that is reused
  double *tab, *tmeta;
  int phases;             // bit 0: compute the tables, bit 1: interpolate + store the rows
};

// samples evaluated per chunk: every Battaglia/README halo has <= 690 samples inside its theta-cut, so one chunk = one
// evaluation phase and one seeding of the sine recurrences per item; longer profiles simply take more chunks.
constexpr int NCH_MMA = 704;

// {sin, cos}(2 pi m/N) for m < N: seeds of the tensor-core path (read with __ldg, 16 bytes per entry)
__global__ void sine_table_kernel(int N, double2* __restrict__ tab, double kt1, double* __restrict__ rkt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) {
    double sn, cs;
    sincospi(2.0 * (double)i / (double)N, &sn, &cs);
    tab[i] = make_double2(sn, cs);
    if (rkt && i <= N / 2 + 1) rkt[i] = i ? 1.0 / ((double)i * kt1) : 0.0;   // 1/kt_j  (fft.py:91)
  }
}

// max(ks) on the device: the bin counts must cover the largest wavenumber whatever kmax the caller passed
__global__ void kmax_kernel(int nk, const double* __restrict__ ks, double* __restrict__ out) {
  __shared__ double red[32];
  double m = 0.0;
  for (int k = threadIdx.x; k < nk; k += blockDim.x) m = fmax(m, ks[k]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, red[w]);
    *out = m;
  }
}

// bins needed by each item (group of HB halos): jn = floor(kmax * max_h(rs (1+z)) / kt_1) + 2, capped at N/2
__global__ void bin_count_kernel(int nz, int nm, int nmg, int HB, int J, double kmax_host, double kt1,
                                 const double* __restrict__ zs, const double* __restrict__ rs,
                                 int* __restrict__ jn_cta, int* __restrict__ work_counter,
                                 const double* __restrict__ kmax_dev) {
  const double kmax = fmax(kmax_host, *kmax_dev);
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) *work_counter = 0;                // queue head of the persistent kernel
  if (b >= nz * nmg) return;
  const int z = b / nmg, mg = nmg - 1 - (b - z * nmg);
  double amax = 0.0;
  for (int h = 0; h < HB; ++h) {
    const int m = mg * HB + h;
    if (m < nm) amax = fmax(amax, rs[(long long)z * nm + m] * (1.0 + zs[z]));
  }
  jn_cta[b] = (int)fmin((double)J, floor(kmax * amax / kt1) + 2.0);
}

// =====================================================================================================================
// The persistent, warp-specialised transform kernel.
//
// Why two groups: an earlier design ran evaluation, sine sums and stores one after the other in one CTA per SM, and the
// FP64 pipe idled while rows were stored and the store path idled while the pipe worked (ncu: 48 % tensor-pipe active,
// 8 % DRAM on its heaviest halos).  ONE 512-thread CTA per SM holds TWO independent groups of 8 warps, each with its
// own 90 KB sample buffer and its own bin table in global memory (only the bins an item needs are touched, so the
// tables live in the 126 MB L2).  A group pulls (z, 16-halo group) items from a global atomic queue and runs, for
// each item,
//   phase 1: evaluate the samples into its buffer, run the DMMA sine sums, write the normalised bin table u_j;
//   phase 2: interpolate the 16 rows onto the target ks and store them.  A warp owns 256-wide k blocks and walks the 16
//            rows of the item for each block: the wavenumbers stay in registers for all rows (no shared-memory copy of
//            ks: that space holds the second sample buffer), and one pair of products per (row, block) classifies a
//            block of a sorted k axis as hold-u_1 / zero / interior / general -- fills are plain 16-byte streaming
//            stores, interior blocks interpolate without classification.
// The two groups run free of each other ("ping-pong"): while one stores rows (HBM-bound) or sits in the latencies of
// its phase changes, the other one's DMMAs keep the FP64 pipe busy.  There are no consumer warps, no ring and no
// mbarriers: a group synchronises with itself through one named barrier.  Measured on a 64-z slab (tools/kbench.py):
// phase 1 alone 2.66 ms, phase 2 alone 1.75 ms (pure fills: 1.56 ms = the HBM roof), both 3.87 ms.
// Sixteen halos per item = two 8-row M tiles per B fragment: every sine value the recurrence produces feeds two DMMAs
// (tools/micro/dmma_sweep.cu: one recurrence DFMA per DMMA caps the loop at 28 of 36 TFLOP/s), and a warp with 4 bin
// tiles runs 8 independent accumulator chains (DMMA dependent-issue latency ~49 cycles, 16 cycles of pipe each).
// Items are issued in an order that strides through the mass axis (golden-ratio step), so light (store-bound) and heavy
// (DMMA-bound) groups alternate in every SM's queue instead of arriving as one heavy and one light phase; the last
// redshifts behind a short mixed head (see ws_item, launch_transform_ws) run jointly heavy-first so the queue drains on light items.
// The parameters of the next item are fetched into registers while the current one is being transformed.
constexpr int WS_HB = 16, WS_NG = 2, WS_GT = 256, WS_MAXCTA = 192;
constexpr int WS_GS_DOUBLES = (NCH_MMA / 4) * 64;      // one sample buffer: 16 halos x NCH_MMA samples
// sum over the lanes of the caller's parity (even lanes hold halos 0-7, odd lanes halos 8-15)
__device__ __forceinline__ double warp_sum_parity(double v) {
#pragma unroll
  for (int o = 16; o > 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// barrier among the 128 threads of producer group g (named barriers 1 and 2; 0 is __syncthreads)
__device__ __forceinline__ void group_bar(int g) { asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(WS_GT) : "memory"); }

// sample n of halo h inside a chunk: [n/4][h%8][n%4][h/8] -- the A fragments (sample kq of halo nq, both M tiles) of a
// 4-sample MMA step are 32 consecutive 16-byte words, one conflict-free LDS.128 per lane
// (WS_GSB = doubles per 4-sample block; padding it to 72 to spread the evaluation's stores over more banks was
// measured: no gain, the A-fragment loads then straddle an extra bank row)
constexpr int WS_GSB = 64;
__device__ __forceinline__ int ws_gs_index(int sn, int h) {
  return (sn >> 2) * WS_GSB + ((h & 7) << 3) + ((sn & 3) << 1) + (h >> 3);
}

// D[16 halos][8 bins] += A[16][4 samples] B[4][8] as two m8n8k4 DMMAs sharing the B fragment; NT bin tiles per warp.
// First chunk stores, later chunks add; when the whole profile fits one chunk (fuse) the mass norm and 1/kt_j are
// applied on the way out and bin 1 is published as u1.
template <int NT>
__device__ __forceinline__ void accum_mma_ws(const double2* __restrict__ tab, const double* __restrict__ gs, double* U,
                                             int JS, int N, int n0, int nlen, int jw, int jn, int lane, bool first,
                                             bool fuse, double scale0, double scale1, const double* __restrict__ rkt,
                                             double* u1_out) {
  const int kq = lane & 3, nq = lane >> 2;
  double bc[NT], bp[NT], tc[NT], c[NT][2][2];
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int jj = jw + 8 * t + nq;
    const unsigned j = (jj <= jn) ? (unsigned)jj : 0u;          // bin 0: sin == 0, contributes nothing
    const unsigned ph = (j * (unsigned)(n0 + kq)) % (unsigned)N;  // j*n < 2^31 (checked on the host)
    const unsigned st = (4u * j) % (unsigned)N;                   // phase advance per 4 samples
    const unsigned pp = ph >= st ? ph - st : ph + (unsigned)N - st;
    bc[t] = __ldg(tab + ph).x;
    bp[t] = __ldg(tab + pp).x;
    tc[t] = 2.0 * __ldg(tab + st).y;
    c[t][0][0] = 0.0; c[t][0][1] = 0.0; c[t][1][0] = 0.0; c[t][1][1] = 0.0;
  }
  const double2* ga = reinterpret_cast<const double2*>(gs) + (nq << 2) + kq;
#pragma unroll 2
  for (int nn = 0; nn < nlen; nn += 4) {
    const double2 a = ga[(nn >> 2) * (WS_GSB / 2)];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[t][0][0]), "+d"(c[t][0][1]) : "d"(a.x), "d"(bc[t]));
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[t][1][0]), "+d"(c[t][1][1]) : "d"(a.y), "d"(bc[t]));
      const double bn = fma(tc[t], bc[t], -bp[t]);
      bp[t] = bc[t];
      bc[t] = bn;
    }
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    double* Uh = U + (size_t)(nq + 8 * mt) * JS;
    const double sc = mt ? scale1 : scale0;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int b = jw + 8 * t + 2 * kq + e;
        if (b <= jn) {
          double v = c[t][mt][e];
          HMV_DEV_ASSERT(b >= 1 && b < JS - 1);
          if (!first) v += Uh[b];
          if (fuse) {
            v *= sc * __ldg(rkt + b);
            if (b == 1) u1_out[nq + 8 * mt] = v;
          }
          Uh[b] = v;
        }
      }
    }
  }
}

__device__ __forceinline__ double ws_interp(const double* U, double t, double u1, double tJ, int jcap) {
  const int j = min(max((int)fmin(t, tJ), 1), jcap);       // always inside the bins the producer wrote
  const double ua = U[j], ub = U[j + 1];
  double v = fma(t - (double)j, ub - ua, ua);
  v = (t > tJ) ? 0.0 : v;                                    // np.interp right=0
  return (t >= 1.0) ? v : u1;                                // np.interp left=puks[0]
}

// The same interpolation with 5 FP64-pipe instructions (the pipe is shared with the producers' DMMAs, so every FP64
// compare, min or conversion here is taken from the sine sums): rint(t) by the 2^52 magic-number add, the offset
// from the nearest bin by an exact fma, classification (t < 1, t > J) and clamping on integer registers, and
// v = U[jn] + |t - jn| (U[jn +- 1] - U[jn]), the line through the two bins around t.  Split in two steps so that a
// lane can issue the table loads of all its elements before the first use (one L2 round trip per block, not eight).
struct WsLerp {
  int jc, jo;         // nearest bin and its neighbour on t's side, clamped to the computed bins
  int cls;            // 0: interpolate, 1: below the first bin (hold u_1), 2: above the last bin (zero)
  double af;          // |t - rint(t)|
};
__device__ __forceinline__ WsLerp ws_lerp_setup(double k, double inv, int J, int jcap) {
  const double MAGIC = 6755399441055744.0;                   // 1.5 * 2^52
  const double tm = fma(k, inv, MAGIC);
  const unsigned jr = (unsigned)__double2loint(tm);          // rint(t) for t < 2^32
  const int huge = __double2hiint(tm) != 0x43380000;         // t >= 2^32 (or negative / NaN)
  const double frac = fma(k, inv, -(tm - MAGIC));            // t - rint(t), exact
  const int fh = __double2hiint(frac), fl = __double2loint(frac);
  const int neg = fh < 0, pos = (fh >= 0) & ((fh | fl) != 0);
  const int below = (huge ^ 1) & ((jr < 1u) | ((jr == 1u) & neg));                  // t < 1
  const int above = huge | (jr > (unsigned)J) | ((jr == (unsigned)J) & pos);        // t > J
  WsLerp r;
  r.jc = min(max((int)min(jr, (unsigned)(jcap + 1)), 1), jcap + 1);
  r.jo = min(r.jc + 1 - 2 * neg, jcap + 1);
  r.cls = below | (above << 1);
  r.af = __hiloint2double(fh & 0x7fffffff, fl);
  return r;
}
__device__ __forceinline__ double ws_lerp_finish(const WsLerp& r, double ua, double uo, double u1) {
  const double v = fma(r.af, uo - ua, ua);
  return (r.cls & 1) ? u1 : ((r.cls & 2) ? 0.0 : v);
}

// Interior of a sorted row (every t of the block inside [1, J], bins inside the computed range): no classification.
__device__ __forceinline__ void ws_lerp_interior(double k, double inv, unsigned jmax, unsigned& jc, unsigned& jo, double& af) {
  // four FP64-pipe instructions (t, t - rint t, and the two of the lerp); the rounding and its way back to FP64 are
  // conversion instructions, which do not queue behind the producers' DMMAs
  const double t = k * inv;
  const int jr = __double2int_rn(t);
  const double frac = t - (double)jr;
  const int fh = __double2hiint(frac);
  jc = min((unsigned)jr, jmax);
  jo = jc + 1u + (unsigned)((fh >> 31) << 1);                // +1, or -1 when t is left of its nearest bin
  af = __hiloint2double(fh & 0x7fffffff, __double2loint(frac));
}

// queue position -> (z, mass-group index counted from the heavy end)
// The last `ntail` redshifts are issued jointly heavy-first -- mass group by mass group across those redshifts -- so
// that the queue drains on the lightest items of the launch whatever the slab size; the redshifts in front of them
// stride through the mass axis (a mixed head that desynchronises the groups' phases).
__host__ __device__ __forceinline__ void ws_item(int item, int nz, int nmg, int stride, int ntail, int& z, int& q) {
  if (ntail < 0) {                       // measurement variant: heaviest and lightest items of the launch alternate
    const int n = nz * nmg, idx = (item & 1) ? n - 1 - (item >> 1) : (item >> 1);
    q = idx / nz;
    z = idx - q * nz;
    return;
  }
  const int nhead = (nz - ntail) * nmg;
  if (item < nhead) {
    z = item / nmg;
    const int r = item - z * nmg;
    q = (int)(((long long)r * stride) % nmg);
  } else {
    const int r = item - nhead;
    q = r / ntail;
    z = nz - ntail + (r - q * ntail);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Two-stage form of the sine sums (the Cooley-Tukey factorisation of the zero-padded, output-pruned transform), used
// for items that need many bins.  With N = P Q, samples n = P n1 + n0 and bins j = q + Q j1:
//     stage 1   H(q, n0)  = sum_n1 g[P n1 + n0] exp(i 2 pi q n1 / Q)               [q < Q, n0 < P; n1 < nb/P <= 18]
//     twiddle   H'(q, n0) = H(q, n0) exp(i 2 pi q n0 / N)
//     stage 2   U[q + Q j1] = Im sum_n0 H'(q, n0) exp(i 2 pi j1 n0 / P)            [j1 <= jn/Q]
// Both stages are small dense contractions with HALO-INDEPENDENT matrices, so they run on the same FP64 tensor-core
// instruction: stage 1 as D[q][n0] += A1[q][n1] B[n1][n0] (B = the halo's samples), stage 2 as
// D[j1][q] += A2[j1][(n0, re/im)] B[(n0, re/im)][q], where the B fragment of stage 2 is exactly what a lane holds of the
// stage-1 result after the twiddle (the k index of stage 2 is ordered to match), so nothing is shuffled or stored in
// between.  Work per halo: 16 q-tiles x (50 + 20 R) DMMAs (R = ceil((jn/Q + 1)/8) <= 3) instead of
// ceil(nb/4) ceil(jn/8)/8 x 2: 3.4 x fewer for the heaviest halos (jn = 2207), break-even near jn = 410; the heavy
// third of the items carries three quarters of the direct form's DMMAs.  No recurrences: every twiddle is exact.
// All 8 warps of a group work on the same q tile (two halos each); the tile's A1 / twiddle slice (7.5 KB) is staged in
// shared memory once per tile for the whole group, the A2 table (15 KB) once per kernel.
constexpr int TS_P = 40, TS_U = TS_P / 8, TS_S = 5, TS_RMAX = 3;      // n0 tiles, stage-1 k-steps (n1 < 20), j1 tiles
constexpr int TS_A1_SLICE = TS_S * 2 * 32, TS_TW_SLICE = TS_U * 2 * 32 * 2, TS_SLICE = TS_A1_SLICE + TS_TW_SLICE;
constexpr int TS_A2_DOUBLES = TS_RMAX * TS_U * 4 * 32;

// fragment-ordered tables: a1[qt][s][cos|sin][lane], tw[qt][u][e][lane]{cos,sin}, a2[r][u][a][lane]
__global__ void twostage_tables_kernel(int N, int Q, int QT, double* __restrict__ a1, double* __restrict__ tw,
                                       double* __restrict__ a2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = i & 31, g = lane >> 2, t = lane & 3;
  if (i < QT * TS_S * 32) {
    const int s = (i >> 5) % TS_S, qt = (i >> 5) / TS_S;
    const long long q = 8 * qt + g, n1 = 4 * s + t;
    double sn, cs;
    sincospi(2.0 * (double)((q * n1) % Q) / (double)Q, &sn, &cs);
    a1[((qt * TS_S + s) * 2 + 0) * 32 + lane] = cs;
    a1[((qt * TS_S + s) * 2 + 1) * 32 + lane] = sn;
  }
  if (i < QT * TS_U * 2 * 32) {
    const int e = (i >> 5) & 1, u = ((i >> 5) >> 1) % TS_U, qt = ((i >> 5) >> 1) / TS_U;
    const long long q = 8 * qt + g, n0 = 8 * u + 2 * t + e;
    double sn, cs;
    sincospi(2.0 * (double)((q * n0) % N) / (double)N, &sn, &cs);
    reinterpret_cast<double2*>(tw)[((qt * TS_U + u) * 2 + e) * 32 + lane] = make_double2(cs, sn);
  }
  if (i < TS_A2_DOUBLES) {
    const int a = (i >> 5) & 3, u = ((i >> 5) >> 2) % TS_U, r = ((i >> 5) >> 2) / TS_U;
    const long long j1 = 8 * r + g, n0 = 8 * u + 2 * t + (a & 1);
    double sn, cs;
    sincospi(2.0 * (double)((j1 * n0) % TS_P) / (double)TS_P, &sn, &cs);
    a2[i] = (a < 2) ? sn : cs;
  }
}

__device__ __forceinline__ void dmma(double (&d)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

// One item (16 halos, one sample chunk) by a group of 8 warps; warp w owns halos 2w and 2w+1.  gs is halo-major
// [16][NCH_MMA]; slice = this group's staging buffer; a2s = the A2 table in shared memory.
template <int R>
__device__ __forceinline__ void accum_two_stage(const TParams& p, const double* __restrict__ gs, int nfill, int ksteps,
                                                const double* __restrict__ a2s, double* slice, double* U, int JS,
                                                int jn, int g_id, int gt, double sc0, double sc1, double* u1_out) {
  const int warp = gt >> 5, lane = gt & 31, gq = lane >> 2, t = lane & 3;
  const int Q = p.ts_Q, QT = p.ts_QT;
  const double* a1g = p.ts_a1;
  const double* twg = p.ts_tw;
  const double* g0 = gs + (size_t)(2 * warp) * NCH_MMA;
  const double* g1 = g0 + NCH_MMA;
  double* U0 = U + (size_t)(2 * warp) * JS;
  double* U1 = U0 + JS;
  // stage the slice of q tile 0
  for (int i = gt; i < TS_SLICE; i += WS_GT)
    slice[i] = (i < TS_A1_SLICE) ? __ldg(a1g + i) : __ldg(twg + (i - TS_A1_SLICE));
  group_bar(g_id);
  for (int qt = 0; qt < QT; ++qt) {
    // next tile's slice travels through registers while this one is being used
    double nx[(TS_SLICE + WS_GT - 1) / WS_GT];
    if (qt + 1 < QT) {
#pragma unroll
      for (int i = 0; i < (TS_SLICE + WS_GT - 1) / WS_GT; ++i) {
        const int idx = gt + i * WS_GT;
        if (idx < TS_SLICE)
          nx[i] = (idx < TS_A1_SLICE) ? __ldg(a1g + (size_t)(qt + 1) * TS_A1_SLICE + idx)
                                      : __ldg(twg + (size_t)(qt + 1) * TS_TW_SLICE + (idx - TS_A1_SLICE));
      }
    }
    double rk[R][2];                     // 1/kt_j of this lane's bins, in flight behind the tile's DMMAs
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int q = 8 * qt + 2 * t + e, j = q + Q * (8 * r + gq);
        rk[r][e] = (q < Q && j >= 1 && j <= jn) ? __ldg(p.rkt + j) : 0.0;
      }
    double a1c[TS_S], a1s[TS_S];
#pragma unroll
    for (int s = 0; s < TS_S; ++s) { a1c[s] = slice[(s * 2 + 0) * 32 + lane]; a1s[s] = slice[(s * 2 + 1) * 32 + lane]; }
    const double2* tws = reinterpret_cast<const double2*>(slice + TS_A1_SLICE);
    // stage-2 accumulators [halo][j1 tile][k split]: with one j1 tile the k index is split over two accumulators per
    // halo, so that an accumulator is never reused by the next DMMA but one (dependent-issue latency ~49 cycles)
    constexpr int KS = (R == 1) ? 2 : 1;
    double acc[2][R][KS][2];
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
      for (int r = 0; r < R; ++r)
#pragma unroll
        for (int k = 0; k < KS; ++k) acc[x][r][k][0] = acc[x][r][k][1] = 0.0;
#pragma unroll
    for (int u = 0; u < TS_U; ++u) {
      double hr[2][2] = {{0.0, 0.0}, {0.0, 0.0}}, hi[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
      for (int s = 0; s < TS_S; ++s) {
        if (s < ksteps) {
          const int n = TS_P * (4 * s + t) + 8 * u + gq;
          const bool in = n < nfill;
          const double b0 = in ? g0[n] : 0.0, b1 = in ? g1[n] : 0.0;
          dmma(hr[0], a1c[s], b0);
          dmma(hr[1], a1c[s], b1);
          dmma(hi[0], a1s[s], b0);
          dmma(hi[1], a1s[s], b1);
        }
      }
      const double2 w0 = tws[(u * 2 + 0) * 32 + lane], w1 = tws[(u * 2 + 1) * 32 + lane];
      double v[2][4];
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        v[x][0] = fma(hr[x][0], w0.x, -hi[x][0] * w0.y);      // Re H' at n0 = 8u+2t
        v[x][1] = fma(hr[x][1], w1.x, -hi[x][1] * w1.y);      // Re H' at n0 = 8u+2t+1
        v[x][2] = fma(hr[x][0], w0.y, hi[x][0] * w0.x);       // Im H' at n0 = 8u+2t
        v[x][3] = fma(hr[x][1], w1.y, hi[x][1] * w1.x);       // Im H' at n0 = 8u+2t+1
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double* af = a2s + ((r * TS_U + u) * 4) * 32 + lane;
        const double f0 = af[0], f1 = af[32], f2 = af[64], f3 = af[96];
        dmma(acc[0][r][0], f0, v[0][0]);
        dmma(acc[1][r][0], f0, v[1][0]);
        dmma(acc[0][r][KS - 1], f1, v[0][1]);
        dmma(acc[1][r][KS - 1], f1, v[1][1]);
        dmma(acc[0][r][0], f2, v[0][2]);
        dmma(acc[1][r][0], f2, v[1][2]);
        dmma(acc[0][r][KS - 1], f3, v[0][3]);
        dmma(acc[1][r][KS - 1], f3, v[1][3]);
      }
    }
    // bins of this q tile: lane holds rows j1 = 8r + gq, columns q = 8 qt + 2t + e
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int q = 8 * qt + 2 * t + e, j = q + Q * (8 * r + gq);
        if (q < Q && j >= 1 && j <= jn) {
          const double v0 = (KS == 2 ? acc[0][r][0][e] + acc[0][r][KS - 1][e] : acc[0][r][0][e]) * (sc0 * rk[r][e]);
          const double v1 = (KS == 2 ? acc[1][r][0][e] + acc[1][r][KS - 1][e] : acc[1][r][0][e]) * (sc1 * rk[r][e]);
          U0[j] = v0;
          U1[j] = v1;
          if (j == 1) { u1_out[2 * warp] = v0; u1_out[2 * warp + 1] = v1; }
        }
      }
    group_bar(g_id);                     // everyone is done reading this tile's slice
    if (qt + 1 < QT) {
#pragma unroll
      for (int i = 0; i < (TS_SLICE + WS_GT - 1) / WS_GT; ++i) {
        const int idx = gt + i * WS_GT;
        if (idx < TS_SLICE) slice[idx] = nx[i];
      }
      group_bar(g_id);
    }
  }
}

struct WsGroupShared {                        // per group
  double h_cmax[WS_HB], h_lxc[WS_HB], h_alpha[WS_HB], h_expo[WS_HB], h_amp[WS_HB], h_oscale[WS_HB], h_inv[WS_HB];
  double u1[WS_HB];                           // bin 1 of the finished table (np.interp's left value)
  double redm[WS_GT / 32][WS_HB];
  int nxt_item;
  int blk_next, blk_rot;                      // phase 2: next k block to hand out, first block that is not a pure hold-u_1 fill
};

__global__ void __launch_bounds__(WS_NG * WS_GT, 1)
profile_transform_ws_kernel(const TParams p, double* ring, int* work_counter, int nitems, int stride, int ntail) {
  extern __shared__ double smem[];            // [WS_NG] sample buffers, each [NCH_MMA/4][8][4][2]
  __shared__ WsGroupShared gsh[WS_NG];
  __shared__ GnfwTables tabs;

  const int tid = threadIdx.x;
  if (tid < WS_NG) gsh[tid].nxt_item = atomicAdd(work_counter, 1);
  gnfw_tables_init(tabs, tid, WS_NG * WS_GT);
  if (p.ts_Q > 0)
    for (int i = tid; i < TS_A2_DOUBLES; i += WS_NG * WS_GT)
      smem[(size_t)WS_NG * WS_GS_DOUBLES + i] = __ldg(p.ts_a2 + i);
  int ascending = 1;
  for (int k = tid; k + 1 < p.nk; k += WS_NG * WS_GT)
    if (!(__ldg(p.ks + k) <= __ldg(p.ks + k + 1))) ascending = 0;
  const int sorted = __syncthreads_and(ascending);     // also publishes the tables and nxt_item
  const int JS = p.JS;

  const int g = tid / WS_GT, gt = tid - g * WS_GT;
  WsGroupShared& G = gsh[g];
  double* gs = smem + (size_t)g * WS_GS_DOUBLES;
  double* a2s = smem + (size_t)WS_NG * WS_GS_DOUBLES;                    // two-stage form: A2 table, then one slice
  double* slice = a2s + TS_A2_DOUBLES + (size_t)g * TS_SLICE;            // per group (present only when ts_Q > 0)
  double* Uslot = ring + ((size_t)blockIdx.x * WS_NG + g) * WS_HB * JS;    // this group's bin table (L2-resident)
  const int nmp = p.nmg * WS_HB;
  const double2* T = reinterpret_cast<const double2*>(p.sintab);
  const int warp = gt >> 5, lane = gt & 31, hoff = (gt & 1) << 3;
  const int npair = p.nk >> 1;
  const int nblk = (npair + 127) >> 7;
  const double2* ks2 = reinterpret_cast<const double2*>(p.ks);
  const double tJ = (double)p.J;
  // parameters of halo `gt` (gt < 16) of an item, fetched one item ahead
  double f_cmax = -1.0, f_xc = 1.0, f_alpha = 0.0, f_expo = 0.0, f_amp = 0.0, f_oscale = 1.0, f_inv = 0.0;
  int f_jn = 0;
  auto fetch = [&](int item) {
    if (item >= nitems) return;
    int z, q;
    ws_item(item, p.nz, p.nmg, stride, ntail, z, q);
    f_jn = p.jn_cta[z * p.nmg + q];
    if (gt < WS_HB) {
      const int m = (p.nmg - 1 - q) * WS_HB + gt;
      const bool ok = m < p.nm;
      const long long rr = (long long)z * p.nm + (ok ? m : p.nm - 1);
      if (p.phases & 1) f_cmax = ok ? p.cmax[rr] : -1.0;
      if (!p.rho && (p.phases & 1)) {
        f_xc = p.xc[rr];
        f_alpha = p.alpha[rr];
        f_expo = p.expo[rr];
        f_amp = p.amp[rr];
      }
      f_oscale = p.outscale ? p.outscale[rr] : 1.0;
      f_inv = p.rs[rr] * (1.0 + p.zs[z]) / p.kt1;            // k -> fractional bin index   (fft.py:92)
    }
  };
  auto publish = [&]() {
    if (gt < WS_HB) {
      G.h_cmax[gt] = f_cmax; G.h_lxc[gt] = log(f_xc); G.h_alpha[gt] = f_alpha; G.h_expo[gt] = f_expo;
      G.h_amp[gt] = f_amp; G.h_oscale[gt] = f_oscale; G.h_inv[gt] = f_inv;
    }
  };
  int item = G.nxt_item;
  fetch(item);
  publish();
  group_bar(g);
  while (item < nitems) {
    if (gt == 0) G.nxt_item = atomicAdd(work_counter, 1);
    int z, q;
    ws_item(item, p.nz, p.nmg, stride, ntail, z, q);
    const int jn = f_jn;
    const int m0 = (p.nmg - 1 - q) * WS_HB;
    HMV_DEV_ASSERT(jn >= 2 && jn <= p.J && m0 >= 0 && m0 < p.nm && z >= 0 && z < p.nz);
    double* U = p.tab ? p.tab + ((size_t)z * nmp + m0) * JS : Uslot;
    group_bar(g);                            // h_* of this item and nxt_item are visible
    const int nxt = G.nxt_item;
    fetch(nxt);                              // loads in flight behind the whole transform of this item

    // ======================== phase 1: samples -> sine sums -> bin table of the item ========================
    if (p.phases & 1) {
    double cmx = -1.0;
#pragma unroll
    for (int h = 0; h < WS_HB; ++h) cmx = fmax(cmx, G.h_cmax[h]);
    const int nb = (cmx > 0.0) ? (int)fmin((double)p.N, floor(cmx / p.dx) + 2.0) : 0;
    const bool single = nb > 0 && nb <= NCH_MMA;
    if (nb == 0)
      for (int i = gt; i < WS_HB * (jn + 1); i += WS_GT) U[(size_t)(i / (jn + 1)) * JS + 1 + i % (jn + 1)] = 0.0;
    // two-stage form when it needs clearly fewer DMMAs than the direct one (both counted for the whole item)
    const int ts_k = (((nb + TS_P - 1) / TS_P) + 3) >> 2;                       // stage-1 k-steps: n1 < 4 ts_k
    const int ts_r = p.ts_Q > 0 ? ((jn / p.ts_Q + 1) + 7) >> 3 : 0;             // j1 tiles
    bool two = false;
    if (single && p.ts_Q > 0 && ts_k <= TS_S && ts_r <= TS_RMAX) {
      const long long direct = 2LL * ((nb + 3) >> 2) * ((jn + 7) >> 3);
      const long long staged = (long long)WS_HB * p.ts_QT * (2 * TS_U * ts_k + 4 * TS_U * ts_r);
      // a 5/4 margin, because the two-stage form also pays for slice staging, twiddles and group barriers; 5/4
      // measured best among the thresholds tried
      two = 5 * staged < 4 * direct;
    }

    double msum[8];                          // this lane's half of the halos (hoff ...)
#pragma unroll
    for (int h = 0; h < 8; ++h) msum[h] = 0.0;
    double scale0 = 1.0, scale1 = 1.0;

    for (int n0 = 0; n0 < nb; n0 += NCH_MMA) {
      const int nfill = min(NCH_MMA, ((nb - n0) + 3) & ~3);
      // thread pair (2i, 2i+1) shares a sample: even lanes evaluate halos 0-7, odd lanes halos 8-15, the eight
      // chains of a thread in lock-step (gnfw_eval.cuh); samples outside a halo's theta-cut are masked afterwards
      if (p.rho) {
        // samples supplied by the caller (rhofunc_x evaluated elsewhere, fft.py:76-81): x * rho(x) inside the cut
        for (int sn = gt >> 1; sn < nfill; sn += WS_GT / 2) {
          const int n = n0 + sn;
          const double x = (double)(n + 1) * p.dx;
          const double wx = ((n == 0 || n == p.N - 1) ? 0.5 * p.dx : p.dx) * x;
#pragma unroll
          for (int hh = 0; hh < 8; ++hh) {
            const int h = hh + hoff;
            const long long row = (long long)z * p.nm + min(m0 + h, p.nm - 1);
            const double v = (n < p.N && x <= G.h_cmax[h]) ? x * __ldg(p.rho + row * p.N + n) : 0.0;
            msum[hh] = fma(wx, v, msum[hh]);
            gs[two ? h * NCH_MMA + sn : ws_gs_index(sn, h)] = v;
          }
        }
      } else
      for (int sn = gt >> 1; sn < nfill; sn += WS_GT / 2) {
        const int n = n0 + sn;
        const double x = (double)(n + 1) * p.dx;
        const double wx = ((n == 0 || n == p.N - 1) ? 0.5 * p.dx : p.dx) * x;   // np.trapz weights on xs (fft.py:84)
        double lt[8], y[8], f[8];
        {
          const double xv[1] = {x};
          double lxv[1];
          log_lockstep<1>(tabs, xv, 0.0, lxv);
#pragma unroll
          for (int hh = 0; hh < 8; ++hh) { lt[hh] = lxv[0] - G.h_lxc[hh + hoff]; y[hh] = G.h_alpha[hh + hoff] * lt[hh]; }
        }
        exp_lockstep<8>(tabs, y, f);                       // t^alpha
        log_lockstep<8>(tabs, f, 1.0, y);                  // log(1 + t^alpha)
#pragma unroll
        for (int hh = 0; hh < 8; ++hh) y[hh] = fma(-G.h_expo[hh + hoff], y[hh], p.gamma * lt[hh]);
        exp_lockstep<8>(tabs, y, f);                       // t^gamma (1 + t^alpha)^(-expo)
#pragma unroll
        for (int hh = 0; hh < 8; ++hh) {
          const int h = hh + hoff;
          const double v = (n < p.N && x <= G.h_cmax[h]) ? (x * G.h_amp[h]) * f[hh] : 0.0;   // x * rho(x) inside the cut
          msum[hh] = fma(wx, v, msum[hh]);
          HMV_DEV_ASSERT(ws_gs_index(sn, h) >= 0 && ws_gs_index(sn, h) < WS_GS_DOUBLES);
          gs[two ? h * NCH_MMA + sn : ws_gs_index(sn, h)] = v;
        }
      }
      if (single && p.do_mass_norm) {
#pragma unroll
        for (int h = 0; h < 8; ++h) {
          const double v = warp_sum_parity(msum[h]);
          if (lane < 2) G.redm[warp][h + hoff] = v;
        }
      }
      group_bar(g);
      if (single) {
        const int nq = lane >> 2;
        double mn0 = 1.0, mn1 = 1.0;
        if (p.do_mass_norm) {
          mn0 = 0.0; mn1 = 0.0;
#pragma unroll
          for (int w8 = 0; w8 < WS_GT / 32; ++w8) { mn0 += G.redm[w8][nq]; mn1 += G.redm[w8][nq + 8]; }
        }
        scale0 = p.step / mn0 * G.h_oscale[nq];
        scale1 = p.step / mn1 * G.h_oscale[nq + 8];
      }
      const int nlen = min(NCH_MMA, nb - n0);
      constexpr int NW = WS_GT / 32;
      const int ntile = (jn + 7) >> 3;
#define HMV_WS_ACC(NTV) accum_mma_ws<NTV>(T, gs, U, JS, p.N, n0, nlen, jw, jn, lane, first, single, scale0, scale1, p.rkt, G.u1)
      const bool first = n0 == 0;
      if (two) {
        // scale of this warp's two halos (the direct form applies them per lane row instead)
        double m0 = 1.0, m1 = 1.0;
        if (p.do_mass_norm) {
          m0 = 0.0; m1 = 0.0;
#pragma unroll
          for (int w8 = 0; w8 < WS_GT / 32; ++w8) { m0 += G.redm[w8][2 * warp]; m1 += G.redm[w8][2 * warp + 1]; }
        }
        const double s0 = p.step / m0 * G.h_oscale[2 * warp], s1 = p.step / m1 * G.h_oscale[2 * warp + 1];
        switch (ts_r) {
          case 1: accum_two_stage<1>(p, gs, nfill, ts_k, a2s, slice, U, JS, jn, g, gt, s0, s1, G.u1); break;
          case 2: accum_two_stage<2>(p, gs, nfill, ts_k, a2s, slice, U, JS, jn, g, gt, s0, s1, G.u1); break;
          default: accum_two_stage<3>(p, gs, nfill, ts_k, a2s, slice, U, JS, jn, g, gt, s0, s1, G.u1); break;
        }
      } else {
      // bin tiles split evenly over the warps (counts differ by at most one), each warp's share in passes of up to
      // four tiles of equal size (5 tiles: 3 + 2, not 4 + 1, so that no pass runs on two accumulator chains)
      int rem = ntile / NW + (warp < ntile % NW);
      int tb = warp * (ntile / NW) + min(warp, ntile % NW);
      for (int passes = (rem + 3) >> 2; passes > 0; --passes) {
        const int ntc = (rem + passes - 1) / passes;
        const int jw = 1 + 8 * tb;
        switch (ntc) {
          case 4: HMV_WS_ACC(4); break;
          case 3: HMV_WS_ACC(3); break;
          case 2: HMV_WS_ACC(2); break;
          default: HMV_WS_ACC(1); break;
        }
        tb += ntc;
        rem -= ntc;
      }
      }
#undef HMV_WS_ACC
      group_bar(g);                          // the chunk's samples are consumed, its sums are in the table
    }

    if (!single) {
      // profile longer than one chunk (or empty): normalise the finished table in a separate pass
      if (p.do_mass_norm) {
#pragma unroll
        for (int h = 0; h < 8; ++h) {
          const double v = warp_sum_parity(msum[h]);
          if (lane < 2) G.redm[warp][h + hoff] = v;
        }
      }
      group_bar(g);
      for (int i = gt; i < WS_HB * jn; i += WS_GT) {
        const int h = i / jn, j = 1 + (i - h * jn);
        double mn = 1.0;
        if (p.do_mass_norm) {
          mn = 0.0;
          for (int w8 = 0; w8 < WS_GT / 32; ++w8) mn += G.redm[w8][h];
        }
        const double v = U[(size_t)h * JS + j] * (p.step / mn * G.h_oscale[h]) * __ldg(p.rkt + j);
        U[(size_t)h * JS + j] = v;
        if (j == 1) G.u1[h] = v;
      }
    }
    if (gt < WS_HB) U[(size_t)gt * JS + jn + 1] = 0.0;     // guard bin behind the last computed one
    __threadfence_block();
    group_bar(g);                            // table complete and visible to the whole group
    if (p.tmeta && gt < WS_HB)               // what a later reader of the table needs to know about the halo
      *reinterpret_cast<double4*>(p.tmeta + ((size_t)z * nmp + m0 + gt) * 4) = make_double4(G.h_inv[gt], G.u1[gt], (double)jn, 0.0);
    } else {                                 // tables computed by an earlier launch: only u_1 has to be fetched
      if (gt < WS_HB) G.u1[gt] = p.tmeta[((size_t)z * nmp + m0 + gt) * 4 + 1];
      group_bar(g);
    }

    // ======================== phase 2: interpolate the 16 rows onto ks, store them ========================
    // The finished table moves from L2 into the (now dead) sample buffer, as many rows per pass as fit (all 16 for
    // jn <= 702: four fifths of the items of the LARGE grid; at least 4 for N <= 5000), so the two table reads of every
    // interpolated element are shared-memory loads instead of L2 round trips -- with eight warps a group cannot keep
    // enough of those in flight (ncu: long_scoreboard was the top stall of this phase).  k blocks are handed out
    // through a counter in shared memory, starting at the first block that is not a pure hold-u_1 fill: the expensive
    // (interpolated) blocks go first and the group's warps finish within one cheap fill block of each other.
    if (p.phases & 2) {
      const int nvalid = min(WS_HB, p.nm - m0);
      double* out0 = p.uk + ((long long)z * p.nm + m0) * (long long)p.ldk;
      const int jcap = min(p.J - 1, jn);
      const int tw = (jn + 3) & ~1;                      // bins 0 .. jn+1, rounded up to whole 16-byte words
      const bool staged = tw <= WS_GS_DOUBLES;           // a row longer than the buffer (N > 22500) is read from L2
      const int rpp = staged ? min(WS_HB, WS_GS_DOUBLES / tw) : WS_HB;    // rows per pass
      const int nwhole = npair >> 7;
      if (warp == 0) {
        int rot = 0;
        if (sorted) {
          double invmax = 0.0;
          for (int h = 0; h < nvalid; ++h) invmax = fmax(invmax, G.h_inv[h]);
          for (int b0 = 0; b0 < nwhole; b0 += 32) {
            const int b = b0 + lane;
            const unsigned hold = __ballot_sync(0xffffffffu, b < nwhole && __ldg(p.ks + 256 * b + 255) * invmax < 1.0);
            rot += __popc(hold);
            if (hold != 0xffffffffu) break;
          }
        }
        if (lane == 0) G.blk_rot = rot < nblk ? rot : 0;
      }
      for (int r0 = 0; r0 < nvalid; r0 += rpp) {
        const int r1 = min(nvalid, r0 + rpp);
        if (r0 > 0) group_bar(g);                        // the previous pass is done with the staged rows
        if (staged) {
          const int hw = tw >> 1;
          double2* dst = reinterpret_cast<double2*>(gs);
          for (int row = r0 + warp; row < r1; row += WS_GT / 32) {
            const double2* src = reinterpret_cast<const double2*>(U + (size_t)row * JS);
            double2* d = dst + (size_t)(row - r0) * hw;
            for (int i = lane; i < hw; i += 32) d[i] = src[i];
          }
        }
        if (gt == 0) G.blk_next = 0;
        group_bar(g);
        const int rot = G.blk_rot;
      // (the two callers differ in the table pointer's address space: shared-memory loads for staged rows)
      auto blocks = [&](const double* __restrict__ tabbase, const int tabstride) {
      for (;;) {
        int blk = 0;
        if (lane == 0) blk = atomicAdd(&G.blk_next, 1);
        blk = __shfl_sync(0xffffffffu, blk, 0);
        if (blk >= nblk) break;
        blk += rot;
        if (blk >= nblk) blk -= nblk;
        const int base = blk << 7;                       // first pair of the block
        const bool whole = base + 128 <= npair;
        double2 kk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) kk[u] = __ldg(ks2 + min(base + lane + 32 * u, npair - 1));
        // lane r (and r + 16) classifies the block for row r: 0 all below the first bin (hold u_1), 1 all above the
        // last bin (zero), 2 all inside [1, J] (interior), 3 mixed / unsorted ks / last partial block
        int cls = 3;
        if (sorted && whole) {
          const double kf = __ldg(p.ks + 2 * base), kl = __ldg(p.ks + 2 * base + 255);
          const double inv_r = G.h_inv[lane & 15];
          const double tf = kf * inv_r, tl = kl * inv_r;
          cls = (tl < 1.0) ? 0 : (tf > tJ) ? 1 : (tf >= 1.0 && tl <= tJ) ? 2 : 3;
        }
        for (int row = r0; row < r1; ++row) {
          const int c = __shfl_sync(0xffffffffu, cls, row);
          double2* orow = reinterpret_cast<double2*>(out0 + (long long)row * p.ldk) + base + lane;
          const double* Uh = tabbase + (size_t)(row - r0) * tabstride;
          if (c < 2) {
            const double fv = c ? 0.0 : G.u1[row];
            const double2 v = make_double2(fv, fv);
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (whole || base + lane + 32 * u < npair) __stcs(orow + 32 * u, v);
          } else if (c == 2) {
            const double inv = G.h_inv[row];
            unsigned jc[8], jo[8];
            double af[8];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              ws_lerp_interior(kk[u].x, inv, (unsigned)(jcap + 1), jc[2 * u], jo[2 * u], af[2 * u]);
              ws_lerp_interior(kk[u].y, inv, (unsigned)(jcap + 1), jc[2 * u + 1], jo[2 * u + 1], af[2 * u + 1]);
            }
            double ua[8], uo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              HMV_DEV_ASSERT(jc[i] >= 1u && jc[i] <= (unsigned)(jn + 1) && jo[i] <= (unsigned)(jn + 1));
              ua[i] = Uh[jc[i]]; uo[i] = Uh[jo[i]];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
              __stcs(orow + 32 * u, make_double2(fma(af[2 * u], uo[2 * u] - ua[2 * u], ua[2 * u]),
                                                fma(af[2 * u + 1], uo[2 * u + 1] - ua[2 * u + 1], ua[2 * u + 1])));
          } else {
            const double inv = G.h_inv[row], u1 = G.u1[row];
            WsLerp e[8];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              e[2 * u] = ws_lerp_setup(kk[u].x, inv, p.J, jcap);
              e[2 * u + 1] = ws_lerp_setup(kk[u].y, inv, p.J, jcap);
            }
            double ua[8], uo[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              HMV_DEV_ASSERT(e[i].jc >= 1 && e[i].jc <= jn + 1 && e[i].jo >= 0 && e[i].jo <= jn + 1);
              ua[i] = Uh[e[i].jc]; uo[i] = Uh[e[i].jo];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const double2 v = make_double2(ws_lerp_finish(e[2 * u], ua[2 * u], uo[2 * u], u1),
                                             ws_lerp_finish(e[2 * u + 1], ua[2 * u + 1], uo[2 * u + 1], u1));
              if (whole || base + lane + 32 * u < npair) __stcs(orow + 32 * u, v);
            }
          }
        }
      }
      };
      if (staged) blocks(gs, tw); else blocks(U + (size_t)r0 * JS, JS);
        if ((p.nk & 1) && warp == 0 && lane >= r0 && lane < r1) {   // odd nk: the last wavenumber, one row per lane
          const int k = p.nk - 1;
          out0[(long long)lane * p.ldk + k] = ws_interp(staged ? gs + (size_t)(lane - r0) * tw : U + (size_t)lane * JS, __ldg(p.ks + k) * G.h_inv[lane], G.u1[lane], tJ, jcap);
        }
      }
    }
    group_bar(g);                            // every warp is done with the table, u1 and this item's h_*
    publish();                               // next item's parameters (ordered by the next trip's first barrier)
    item = nxt;
  }
}

// row stride of the bin tables: bins 0 .. J+1, rounded up to whole 16-byte words
static int ws_js(int nxs) { return (nxs / 2 + 3) & ~1; }

// two-stage form available: N divisible by TS_P (tables: QT q tiles)
static int ts_qtiles(int nxs) { return (nxs % TS_P == 0 && nxs / TS_P >= 16) ? (nxs / TS_P + 7) / 8 : 0; }

// Workspace of the transform, as offsets in doubles from ws_d (16-byte aligned): the {sin,cos} table, the bin count of
// every (z, 16-halo item) as ints, the queue head (int) + the device max(ks), 1/kt_j for j <= J+1, one [16][JS] bin
// table per group of the persistent kernel, the two-stage tables.  The bin tables and the two-stage tables are read as
// double2, so they start on even offsets.
struct K1Ws {
  size_t jn, head, rkt, ring, ts, total;
};
static K1Ws k1_ws_layout(int nz, int nm, int nxs) {
  auto even = [](size_t n) { return (n + 1) & ~(size_t)1; };
  const int QT = ts_qtiles(nxs);
  K1Ws w;
  w.jn = 2 * (size_t)nxs;
  w.head = w.jn + ((size_t)nz * cdiv(nm, WS_HB) + 1) / 2;
  w.rkt = w.head + 2;
  w.ring = even(w.rkt + nxs / 2 + 2);
  w.ts = even(w.ring + (size_t)WS_MAXCTA * WS_NG * WS_HB * ws_js(nxs));
  w.total = w.ts + (QT ? (size_t)QT * TS_SLICE + TS_A2_DOUBLES : 0);
  return w;
}

// stride through the mass groups with a step near nmg/phi^2 that is coprime to nmg (a permutation of 0..nmg-1)
static int ws_stride(int nmg) {
  auto gcd = [](int a, int b) { while (b) { const int t = a % b; a = b; b = t; } return a; };
  int stride = (int)(0.381966 * nmg);
  if (stride < 1) stride = 1;
  while (gcd(stride, nmg) != 1) ++stride;
  return stride;
}

// how many redshifts the queue issues jointly heavy-first (see ws_item)
static int ws_tail(int nz, int nmg, int grid) {
  // Measured (gpurun_out/r2_k1_tail*.txt, electron profile): heavy-first behind a short mixed head of 4-6 redshifts
  // beats both the all-mixed order with a one-redshift heavy-first tail (25 z: 1.33 -> 1.19 ms, 64 z: 3.06 -> 2.90,
  // 200 z: 9.18 -> 8.90) and heavy-first from the start (1.26 / 2.99 ms on 25 / 64 z: every group then begins with
  // the sine sums of a heaviest item and nothing is stored for the first third of a millisecond); the head's length
  // matters little beyond that (a quarter of the redshifts: 1.20 / 2.93 / 8.94 ms)
  int head = nz / 8;
  head = head < 4 ? 4 : (head > 6 ? 6 : head);
  int ntail = nz - head;
  if (ntail < cdiv(2LL * grid * WS_NG, nmg)) ntail = cdiv(2LL * grid * WS_NG, nmg);
  if (const char* ev = getenv("HMV_K1_TAIL"))                            // measurement knob
    if (*ev) ntail = atoi(ev);
  if (ntail >= 0) ntail = ntail < 1 ? 1 : (ntail > nz ? nz : ntail);
  return ntail;
}

static int launch_transform_ws(const TParams& p, double* ring, int* counter, cudaStream_t st) {
  int dev = 0, nsm = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "profile_transform: %s", cudaGetErrorString(e));
  const int nitems = p.nz * p.nmg;
  const int grid = nitems < nsm ? nitems : (nsm < WS_MAXCTA ? nsm : WS_MAXCTA);
  const int stride = ws_stride(p.nmg);
  size_t smem = (size_t)WS_NG * WS_GS_DOUBLES * sizeof(double);
  if (p.ts_Q > 0) smem += (size_t)(TS_A2_DOUBLES + WS_NG * TS_SLICE) * sizeof(double);
  e = cudaFuncSetAttribute(profile_transform_ws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return fail(HMV_E_CUDA, "profile_transform smem opt-in (%zu B): %s", smem, cudaGetErrorString(e));
  const int ntail = ws_tail(p.nz, p.nmg, grid);
  profile_transform_ws_kernel<<<grid, WS_NG * WS_GT, smem, st>>>(p, ring, counter, nitems, stride, ntail);
  return check_launch("profile_transform_ws_kernel");
}

}  // namespace hmv
using namespace hmv;

extern "C" long long hmv_profile_transform_ws_doubles(int nz, int nm, int nxs) {
  if (nz <= 0 || nm <= 0 || nxs <= 0) return 0;
  return (long long)k1_ws_layout(nz, nm, nxs).total;
}

// Kept for ABI stability: 0 selects the persistent kernel, the one launch plan there is.
extern "C" int hmv_set_transform_mode(int mode) {
  HMV_REQUIRE(mode == 0, "hmv_set_transform_mode: mode %d does not exist; 0 is the only launch plan (the "
              "bin-count-class plan, mode 1, was removed)", mode);
  return HMV_OK;
}

static int profile_transform_impl(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
                                  double kmax, const double* rs_d, const double* cmax_d, const double* xc_d,
                                  const double* alpha_d, const double* expo_d, const double* amp_d,
                                  const double* outscale_d, const double* rho_d, double gamma, double xmax, int nxs,
                                  int do_mass_norm, double* ws_d, double* uk_d, void* stream, double* tab_d = nullptr,
                                  int phases = 3) {
  HMV_REQUIRE(nz > 0 && nm > 0 && nk > 0 && ldk >= nk, "hmv_profile_transform: bad sizes");
  HMV_REQUIRE(nxs >= 4 && xmax > 0, "hmv_profile_transform: need nxs>=4 and xmax>0");
  HMV_REQUIRE((long long)nxs * (nxs / 2) < 2147483647LL, "hmv_profile_transform: nxs=%d too large (phase index overflow)", nxs);
  HMV_REQUIRE(zs_d && ks_d && rs_d && ws_d && ((phases & 2) == 0 || uk_d) &&
              ((phases & 1) == 0 || (cmax_d && (rho_d || (xc_d && alpha_d && expo_d && amp_d)))),
              "hmv_profile_transform: null pointer");
  HMV_REQUIRE((((size_t)ks_d | (size_t)ws_d | (size_t)uk_d | (size_t)tab_d) & 15) == 0 && (ldk & 1) == 0,
              "hmv_profile_transform: ks, ws, uk and tab must be 16-byte aligned with even ldk (16-byte loads and "
              "stores); ldk=%d", ldk);
  const K1Ws w = k1_ws_layout(nz, nm, nxs);
  TParams p = {};                              // jlo, jhi stay 0
  p.nz = nz; p.nm = nm; p.nk = nk; p.ldk = ldk; p.N = nxs; p.J = nxs / 2; p.JS = ws_js(nxs); p.nmg = cdiv(nm, WS_HB);
  p.do_mass_norm = do_mass_norm;
  p.gamma = gamma;
  p.dx = xmax / nxs;                           // xs = linspace(0,xmax,nxs+1)[1:]           (fft.py:73)
  p.step = (xmax - 1.0 * p.dx) / nxs;          // (x[-1]-x[0])/N                            (fft.py:44-46)
  p.kt1 = (1.0 * (1.0 / (nxs * p.step))) * 2.0 * M_PI;  // rfftfreq(N,step)[1]*2pi          (fft.py:50)
  p.kmax = kmax;
  p.zs = zs_d; p.ks = ks_d; p.rs = rs_d; p.cmax = cmax_d; p.xc = xc_d; p.alpha = alpha_d; p.expo = expo_d;
  p.amp = amp_d; p.outscale = outscale_d; p.uk = uk_d; p.sintab = ws_d;
  p.rho = rho_d;
  p.tab = tab_d; p.phases = phases;
  p.tmeta = tab_d ? tab_d + (size_t)nz * (size_t)(p.nmg * WS_HB) * (size_t)p.JS : nullptr;
  int* jn_cta = reinterpret_cast<int*>(ws_d + w.jn);
  p.jn_cta = jn_cta;
  int* counter = reinterpret_cast<int*>(ws_d + w.head);
  double* kmax_dev = ws_d + w.head + 1;
  p.rkt = ws_d + w.rkt;
  cudaStream_t st = (cudaStream_t)stream;
  sine_table_kernel<<<cdiv(nxs, 256), 256, 0, st>>>(nxs, reinterpret_cast<double2*>(ws_d), p.kt1, ws_d + w.rkt);
  int rc = check_launch("sine_table_kernel");
  if (rc) return rc;
  kmax_kernel<<<1, 1024, 0, st>>>(nk, ks_d, kmax_dev);
  bin_count_kernel<<<cdiv((long long)nz * p.nmg, 256), 256, 0, st>>>(nz, nm, p.nmg, WS_HB, p.J, kmax, p.kt1, zs_d, rs_d,
                                                                       jn_cta, counter, kmax_dev);
  rc = check_launch("bin_count_kernel");
  if (rc) return rc;
  const int QT = ts_qtiles(nxs);
  if (QT) {
    double* tabs = ws_d + w.ts;
    p.ts_Q = nxs / TS_P; p.ts_QT = QT;
    p.ts_a1 = tabs; p.ts_tw = tabs + (size_t)QT * TS_A1_SLICE; p.ts_a2 = tabs + (size_t)QT * (TS_A1_SLICE + TS_TW_SLICE);
    const int nthr = QT * TS_U * 2 * 32 > TS_A2_DOUBLES ? QT * TS_U * 2 * 32 : TS_A2_DOUBLES;
    twostage_tables_kernel<<<cdiv(nthr, 256), 256, 0, st>>>(nxs, p.ts_Q, QT, tabs, tabs + (size_t)QT * TS_A1_SLICE,
                                                           tabs + (size_t)QT * (TS_A1_SLICE + TS_TW_SLICE));
    rc = check_launch("twostage_tables_kernel");
    if (rc) return rc;
  }
  return launch_transform_ws(p, ws_d + w.ring, counter, st);
}

extern "C" int hmv_profile_transform(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
                                     double kmax, const double* rs_d, const double* cmax_d, const double* xc_d,
                                     const double* alpha_d, const double* expo_d, const double* amp_d,
                                     const double* outscale_d, double gamma, double xmax, int nxs, int do_mass_norm,
                                     double* ws_d, double* uk_d, void* stream) {
  return profile_transform_impl(nz, nm, nk, ldk, zs_d, ks_d, kmax, rs_d, cmax_d, xc_d, alpha_d, expo_d, amp_d, outscale_d,
                                nullptr, gamma, xmax, nxs, do_mass_norm, ws_d, uk_d, stream);
}

extern "C" int hmv_profile_transform_samples(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
                                             double kmax, const double* rs_d, const double* cmax_d,
                                             const double* rho_d, const double* outscale_d, double xmax, int nxs,
                                             int do_mass_norm, double* ws_d, double* uk_d, void* stream) {
  HMV_REQUIRE(rho_d, "hmv_profile_transform_samples: null samples");
  return profile_transform_impl(nz, nm, nk, ldk, zs_d, ks_d, kmax, rs_d, cmax_d, nullptr, nullptr, nullptr, nullptr,
                                outscale_d, rho_d, 0.0, xmax, nxs, do_mass_norm, ws_d, uk_d, stream);
}

// ---- table mode: the transform split in two launches around a persistent table array -------------------------------
extern "C" long long hmv_profile_table_stride(int nxs) { return nxs > 0 ? ws_js(nxs) : 0; }

extern "C" long long hmv_profile_table_doubles(int nz, int nm, int nxs) {
  if (nz <= 0 || nm <= 0 || nxs <= 0) return 0;
  const long long nmp = (long long)cdiv(nm, WS_HB) * WS_HB;
  return (long long)nz * nmp * (ws_js(nxs) + 4) + 2;       // tab[z][nmp][JS], tmeta[z][nmp][4], slack for 16-byte reads past a row
}

extern "C" int hmv_profile_tables(int nz, int nm, int nk, const double* zs_d, const double* ks_d, double kmax,
                                  const double* rs_d, const double* cmax_d, const double* xc_d, const double* alpha_d,
                                  const double* expo_d, const double* amp_d, const double* outscale_d, double gamma,
                                  double xmax, int nxs, int do_mass_norm, double* ws_d, double* tab_d, void* stream) {
  HMV_REQUIRE(tab_d, "hmv_profile_tables: null table array");
  return profile_transform_impl(nz, nm, nk, (nk + 1) & ~1, zs_d, ks_d, kmax, rs_d, cmax_d, xc_d, alpha_d, expo_d, amp_d,
                                outscale_d, nullptr, gamma, xmax, nxs, do_mass_norm, ws_d, nullptr, stream, tab_d, 1);
}

extern "C" int hmv_profile_expand(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d, double kmax,
                                  const double* rs_d, double xmax, int nxs, double* ws_d, const double* tab_d,
                                  double* uk_d, void* stream) {
  HMV_REQUIRE(tab_d, "hmv_profile_expand: null table array");
  return profile_transform_impl(nz, nm, nk, ldk, zs_d, ks_d, kmax, rs_d, nullptr, nullptr, nullptr, nullptr, nullptr,
                                nullptr, nullptr, 0.0, xmax, nxs, 0, ws_d, uk_d, stream, const_cast<double*>(tab_d), 2);
}

// host-side introspection for the CPU tests: the (z, mass group) of every queue position of the persistent kernel for
// an nz x nm grid on `grid` CTAs (0 = 148) -- the order must be a permutation of all items
extern "C" int hmv_debug_k1_order(int nz, int nm, int grid, int* z_out, int* q_out) {
  HMV_REQUIRE(nz > 0 && nm > 0 && z_out && q_out, "hmv_debug_k1_order: bad arguments");
  const int nmg = cdiv(nm, WS_HB);
  if (grid <= 0) grid = 148;
  const int stride = ws_stride(nmg), ntail = ws_tail(nz, nmg, grid);
  for (int i = 0; i < nz * nmg; ++i) ws_item(i, nz, nmg, stride, ntail, z_out[i], q_out[i]);
  return nmg;
}
