/* hmvec_b200.h -- C ABI of the B200 (sm_100a) halo-model hot path.
 *
 * The reference (simonsobs/hmvec) has no FFI of its own: its boundary is the Python class API
 * (HaloModel / Cosmology, hmvec/hmvec.py:75-572, hmvec/cosmology.py:506-597,867-904).  This header is
 * the boundary a maintainer would bind underneath that API (ctypes stub in INTEGRATION.md); every
 * entry point names the reference lines whose arithmetic it replaces.
 *
 * Conventions
 *   - every `*_d` pointer is a DEVICE pointer to float64 (or int32 where typed so); the caller owns
 *     every buffer, including workspaces; the library never allocates device memory (exceptions: hmv_peer_alloc,
 *     whose blocks must come from cudaMalloc to be exportable to the other ranks, and the self-timing hmv_bench_*);
 *   - `stream` is a cudaStream_t passed as void*; every call is stream-ordered and asynchronous,
 *     no hidden synchronisation (except hmv_bench_* which time themselves with events);
 *   - return value 0 = ok, <0 = error (HMV_E_*); hmv_last_error() gives a thread-local message;
 *   - cubes u(z,M,k) are laid out [nz][nm][ldk] with k fastest and ldk >= nk the padded row stride
 *     (the Python facade uses ldk = nk rounded up to 16 doubles = 128 B so every row starts on a line);
 *   - [nz,nm] arrays are row-major with M fastest.
 */
#ifndef HMVEC_B200_H
#define HMVEC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define HMV_OK 0
#define HMV_E_ARG (-1)     /* bad argument (null pointer, non-positive size, ...) */
#define HMV_E_CUDA (-2)    /* CUDA launch / runtime error; text in hmv_last_error() */
#define HMV_E_LIMIT (-3)   /* size exceeds a compiled-in limit (stated in the message) */

int hmv_abi_version(void);
const char* hmv_last_error(void);
/* Device sanity: returns compute capability major*10+minor of `device` (100 on B200), <0 on error. */
int hmv_device_cc(int device);

/* ---- a1: sigma^2(R,z)  (cosmology.py:245-269, Wkr :30-38) -------------------------------------------
 * sigma2[z,m] = sum_k' sPzk[z,k'] * kw[k'] * W^2(ks_sig[k'] * R[m]),  kw = simpson_weight * k'^2 / (2 pi^2)
 * (the Simpson rule is linear in the integrand, so the host supplies one weight vector).
 * w2_ws_d: workspace of hmv_sigma2_ws_doubles() doubles (the W^2 table, k' major, + split-k partials). */
long long hmv_sigma2_ws_doubles(int nz, int nm, int nks);
int hmv_sigma2(int nz, int nm, int nks, const double* sPzk_d, const double* kw_d, const double* ks_sig_d,
               const double* R_d, double taylor_switch, double* w2_ws_d, double* sigma2_d, void* stream);

/* ---- a2: Sheth-Tormen f(sigma), bias, n(M,z)  (hmvec.py:133-185) ------------------------------------
 * nzm = rho_m0 * f * dln(sigma^-1)/dlnM / M^2 with numpy.gradient's non-uniform stencil along M. */
int hmv_mass_function(int nz, int nm, const double* sigma2_d, const double* ms_d, double rho_m0, double st_A,
                      double st_a, double st_p, double st_deltac, double* nzm_d, double* bh_d, void* stream);
/* f3: the same with the Tinker et al. 2010 multiplicity function nu f(nu) and bias (hmvec.py:142-145,157-159 ->
 * tinker.py:26-67; mass_function="tinker").  tinker_z_d: [nz][5] = (alpha, beta, phi, eta, gamma) of f(nu) at each
 * redshift -- O(nz) host work: redshifts clamped at 3, alpha from the reference's normalisation table
 * hmvec/data/alpha_consistency.txt (tinker.py:56-66).  nu = deltac/sigma; the bias uses Delta = 200. */
int hmv_mass_function_tinker(int nz, int nm, const double* sigma2_d, const double* ms_d, double rho_m0, double deltac,
                             const double* tinker_z_d, double* nzm_d, double* bh_d, void* stream);

/* ---- a3: Duffy concentration and r_vir  (hmvec.py:68-73,111-115,163-176,627) ------------------------
 * cs = A (h M/2e12)^alpha (1+z)^beta ; rvir = (3M/(4 pi drho1[z]))^(1/3), drho1 = Delta_vir rho_c or 200 rho_m. */
int hmv_halo_geometry(int nz, int nm, const double* zs_d, const double* ms_d, const double* drho1_d, double duffy_A,
                      double duffy_alpha, double duffy_beta, double h, double* cs_d, double* rvir_d, void* stream);

/* ---- a5: mass-definition conversion  (hmvec.py:748-798) ---------------------------------------------
 * Solves M1/mc(C1) = M2/mc(C2(M2)) for M2 by the secant method in ln M2 (start values as scipy.optimize.newton). */
int hmv_mdelta(int nz, int nm, const double* ms_d, const double* cs_d, const double* drho1_d,
               const double* drho2_d, double* m2_d, void* stream);

/* ---- a4: analytic NFW u(k|M,z)  (hmvec.py:346-353) --------------------------------------------------
 * u is evaluated as per-halo piecewise polynomials in (x c)^2 up to x c = 64 and the closed form's asymptotic branch
 * beyond; ks need not be sorted.  uk_d and ws_d must be 16-byte aligned and ldk even (HMV_E_ARG otherwise).
 * ws_d: workspace of hmv_uk_nfw_ws_doubles() doubles (one record of 300 doubles per halo -- its polynomial coefficients
 * and constants -- and per-256-wavenumber chunk bounds and padded copies of ks and ks^2, see k_nfw.cu). */
long long hmv_uk_nfw_ws_doubles(int nz, int nm, int nk);
/* The analytic NFW profile has one evaluation, the piecewise polynomials.  Mode 0 selects it and is accepted for ABI
 * stability; any other mode returns HMV_E_ARG. */
int hmv_set_nfw_mode(int mode);
int hmv_uk_nfw(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
               double kmax /* ignored: max(ks) is reduced on the device */, const double* cs_d,
               const double* rvir_d, double* ws_d, double* uk_d, void* stream);

/* ---- a6: Battaglia GNFW per-halo shape parameters  (hmvec.py:215-249,278-316,800-802,856-860,918-927)
 * The transform kernel evaluates  rho(x) = amp * (x/xc)^gamma * (1 + (x/xc)^alpha)^(-expo)  per halo.
 * kind 0 (density): xc=1, alpha=fit, expo=(beta+gamma)/alpha, amp=1 (cancels against the mass norm),
 *                   rs = r200c/2, outscale = 1.
 * kind 1 (pressure): xc=fit, alpha=pres_alpha, expo=beta, amp = eFrac (omb/omm) 200 m200c G rho_c /(2 r200c) P0,
 *                   rs = r200c, outscale = 4 pi sigmaT/(me c^2) r200c^3 (1+z)^2 / H(z)   (const passed in `pref`).
 * fit[9] = (A0, alpha_m, alpha_z) x 3 in the order (rho0|P0, alpha|xc, beta).
 * Outputs are [nz,nm]: rs, cmax = rvir/rs, xc, alpha, expo, amp, outscale. */
int hmv_gnfw_params(int kind, int nz, int nm, const double* zs_d, const double* m200c_d, const double* rvir_d,
                    const double* rhocrit_d, const double* hofz_d, const double* fit9_h, double gamma,
                    double pres_alpha, double amp_const, double pref, double* rs_d, double* cmax_d, double* xc_d,
                    double* alpha_d, double* expo_d, double* amp_d, double* outscale_d, void* stream);

/* ---- a7+a8: numerical profile transform + interpolation  (fft.py:35-115) ----------------------------
 * Per halo: samples x_n=(n+1) xmax/nxs, theta-cut at cmax, trapezoid mass norm, the rFFT-equivalent sine
 * sums U_j = step sum_n x_n y_n sin(2 pi j n/N), u_j = U_j/kt_j/mnorm, kout_j = kt_j/rs/(1+z), then linear
 * interpolation onto ks (hold u_1 below the first bin, 0 above the last).  The (z,M,x) cube is never stored.
 * outscale_d may be NULL (=1).  do_mass_norm as in generic_profile_fft.  ks need not be sorted.  ks_d, uk_d and ws_d
 * must be 16-byte aligned and ldk even (HMV_E_ARG otherwise), as for the other three transform entry points.
 * ws_d: workspace of hmv_profile_transform_ws_doubles(nz,nm,nxs) doubles (sine table, per-item bin counts, work-queue
 * head and the per-group bin tables of the persistent kernel). */
long long hmv_profile_transform_ws_doubles(int nz, int nm, int nxs);
/* The transform has one launch plan: a persistent kernel with two 8-warp groups per SM, each group evaluating the
 * samples and running the tensor-core sine sums of 16 halos and then interpolating and storing their rows, so that one
 * group's sums overlap the other's stores.  Mode 0 selects it and is accepted for ABI stability; any other mode
 * returns HMV_E_ARG. */
int hmv_set_transform_mode(int mode);
int hmv_profile_transform(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d,
                          double kmax /* hint for max(ks); the kernels also reduce ks on the device and use the larger of the two */, const double* rs_d,
                          const double* cmax_d, const double* xc_d, const double* alpha_d, const double* expo_d,
                          const double* amp_d, const double* outscale_d, double gamma, double xmax, int nxs,
                          int do_mass_norm, double* ws_d, double* uk_d, void* stream);
/* a7 in its general form, generic_profile_fft(rhofunc_x, ...) for ANY radial profile (fft.py:56-94): the samples
 * rho_d[z][m][n] = rho(x_n), x_n = (n+1) xmax/nxs, are supplied by the caller (the reference evaluates a Python
 * callable); theta-cut at cmax, mass norm, sine transform, interpolation onto ks exactly as above.  Needs the
 * persistent kernel (16-byte aligned ks_d / uk_d / ws_d, even ldk); same workspace size. */
int hmv_profile_transform_samples(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d, double kmax,
                                  const double* rs_d, const double* cmax_d, const double* rho_d,
                                  const double* outscale_d, double xmax, int nxs, int do_mass_norm, double* ws_d,
                                  double* uk_d, void* stream);

/* ---- Table mode of the transform: the same persistent kernel split around a table array that stays on the device ----
 * hmv_profile_tables runs the evaluation + sine sums only and leaves, per halo, the normalised bins u_j (j <= the bin
 * count the k range needs) in tab_d[z][nmp][JS] (nmp = nm rounded up to 16, JS = hmv_profile_table_stride(nxs)) followed
 * by {k -> bin factor r_s(1+z)/kt_1, u_1, bin count, 0} per halo; hmv_profile_expand interpolates such tables onto ks
 * (fft.py:97-115) and writes the cube.  tables + expand == hmv_profile_transform bit for bit.  hmv_profile_expand
 * recomputes the bin count from its own ks and kmax and does not read the one stored with the table: it must be
 * called with the ks and kmax the tables were built with (or a range that needs no more bins), since a wider k range
 * would interpolate from bins that were never written.  Consumers that only
 * need sums over M (hmv_power_six_tab, hmv_power_tab) interpolate from the tables themselves: the 8*nk-byte row of
 * every halo is then neither written nor re-read. */
long long hmv_profile_table_stride(int nxs);
long long hmv_profile_table_doubles(int nz, int nm, int nxs);
int hmv_profile_tables(int nz, int nm, int nk, const double* zs_d, const double* ks_d, double kmax,
                       const double* rs_d, const double* cmax_d, const double* xc_d, const double* alpha_d,
                       const double* expo_d, const double* amp_d, const double* outscale_d, double gamma,
                       double xmax, int nxs, int do_mass_norm, double* ws_d, double* tab_d, void* stream);
int hmv_profile_expand(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ks_d, double kmax,
                       const double* rs_d, double xmax, int nxs, double* ws_d, const double* tab_d, double* uk_d,
                       void* stream);

/* ---- a9: HOD occupations and their mass integrals  (hmvec.py:634-731, 462-466, 936-957) -------------
 * hodp[8] = (sig_log_mstellar, alphasat, Bsat, betasat, Bcut, betacut, Msat_override or <=0, Mcut_override or <=0)
 * corr: 0 = "max", 1 = "min".  Outputs [nz,nm]: Nc, Ns, NsNsm1, NcNs; [nz]: ngal, bg. */
int hmv_hod(int nz, int nm, const double* zs_d, const double* ms_d, const double* log10mthresh_d,
            const double* hodp_h, int corr, const double* nzm_d, const double* bh_d, double* Nc_d, double* Ns_d,
            double* NsNsm1_d, double* NcNs_d, double* ngal_d, double* bg_d, void* stream);

/* ---- a10: mthresh <-> ngal bisection  (utils.py:9-42, hmvec.py:415-433) -----------------------------
 * Reproduces the reference's all-z loop exactly: every z bisects independently for HMV_BISECT_MAXIT
 * iterations recording its midpoint and whether |x/x_target - 1| <= rtol (bit `it` of its pass mask); the
 * result is the midpoint of the first iteration at which ALL z pass.
 *   hmv_hod_bisect : runs iterations [it_begin, it_end) (first call from 0; a continuation call resumes from the
 *                    interval state kept in ws_d and returns at once when mask_d[0] != 0, i.e. when an earlier round
 *                    already converged everywhere -- so the usual ~20-iteration solve does not pay for 64);
 *                    ws_d = nz*(HMV_BISECT_MAXIT+4) doubles (midpoints, per-z masks, bracket state);
 *                    mask_d[0] (uint64, device) = AND of the masks of THIS call's redshifts.
 *   (z-sharded runs AND-reduce mask_d over the ranks here -- the reference's loop condition is global in z.)
 *   hmv_hod_pick   : log10mthresh_d[z] = midpoint(z, first set bit of mask_d[0]) * A_log10mthresh;
 *                    iters_d: int32[1], the iteration count (0 = never converged within HMV_BISECT_MAXIT).
 *   hmv_hod_solve  : both steps on one device (all HMV_BISECT_MAXIT iterations in one round; same ws_d size). */
#define HMV_BISECT_MAXIT 64
int hmv_hod_bisect(int nz, int nm, const double* zs_d, const double* ms_d, const double* nzm_d,
                   const double* ngal_target_d, const double* hodp_h, double ylo, double yhi, double rtol,
                   int it_begin, int it_end, double* ws_d, unsigned long long* mask_d, void* stream);
int hmv_hod_pick(int nz, const double* ws_d, const unsigned long long* mask_d, double A_log10mthresh,
                 double* log10mthresh_d, int* iters_d, void* stream);
int hmv_hod_solve(int nz, int nm, const double* zs_d, const double* ms_d, const double* nzm_d,
                  const double* ngal_target_d, const double* hodp_h, double ylo, double yhi, double rtol,
                  double A_log10mthresh, double* ws_d, double* log10mthresh_d, int* iters_d, void* stream);

/* ---- a12-a14: 1-halo + 2-halo mass integrals  (hmvec.py:469-572) ------------------------------------
 * A tracer leg t(z,M,k) = a[z,M]*UC + b[z,M]*US with UC = uc cube (or 1 when uc_d == NULL) and US = us cube:
 *   kind 0 matter   : a=0,        b=M/rho_m0         (hmvec.py:488-492)   bias 1
 *   kind 1 hod      : a=Nc/ngal,  b=Ns/ngal          (hmvec.py:481-486)   bias bg(z)
 *   kind 2 pressure : a=0,        b=1                (hmvec.py:494-497)   bias 0, no consistency term
 * Both legs hod   -> 1h integrand (2 UC US NcNs + NsNsm1 US^2)/ngal^2 of leg A     (hmvec.py:477-479,510-511)
 * Both pressure   -> 1h integrand US_A^2                                          (hmvec.py:512-513)
 * P1h = trapz_M(n * integrand) * (1-exp(-(k/kstar)^2)) ; P2h = Pzk (I_A + b_A - C_A)(I_B + b_B - C_B). */
typedef struct {
  int kind;              /* 0 matter, 1 hod, 2 pressure */
  const double* us_d;    /* [nz][nm][ldk] */
  const double* uc_d;    /* [nz][nm][ldk] or NULL */
  const double* Nc_d;    /* hod only, [nz,nm] */
  const double* Ns_d;
  const double* NcNs_d;
  const double* NsNsm1_d;
  const double* ngal_d;  /* hod only, [nz] */
  const double* bias_d;  /* [nz] override (b1_in/b2_in) or NULL: matter 1, hod bg, pressure 0 */
} hmv_tracer;

/* Workspace size (in doubles) for hmv_power. */
long long hmv_power_ws_doubles(int nz, int nm);
/* p1h_d / p2h_d: [nz][nk] dense outputs (either may be NULL). */
int hmv_power(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d, const double* nzm_d,
              const double* bh_d, const double* Pzk_d, double rho_m0, double kstar, const hmv_tracer* A,
              const hmv_tracer* B, double* ws_d, double* p1h_d, double* p2h_d, void* stream);

/* Six spectra {mm, ee, me, gg, gm, ge} in ONE pass over two cubes (u_m = matter profile, also the HOD's
 * satellite profile with u_c = 1; u_e = second matter-like profile).  Outputs p1h_d/p2h_d: [6][nz][nk]. */
int hmv_power_six(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d, const double* nzm_d,
                  const double* bh_d, const double* Pzk_d, double rho_m0, double kstar, const double* um_d,
                  const double* ue_d, const double* Nc_d, const double* Ns_d, const double* NcNs_d,
                  const double* NsNsm1_d, const double* ngal_d, double* ws_d,
                  long long spec_stride /* doubles between spectra in the outputs; 0 = nz*nk.  A caller working
                                           through z in chunks passes the full-grid stride and offset pointers */,
                  double* p1h_d, double* p2h_d, void* stream);

/* hmv_power_six with the electron profile given as bin tables (hmv_profile_tables, same nxs) instead of a cube:
 * reference hmvec.py:504-572 for the six pairs, fft.py:97-115 for the interpolation done inside the reduction. */
/* Auto spectrum (1h + 2h) of ONE matter (kind 0) or pressure (kind 2) profile given as bin tables: nothing of size
 * nz*nm*nk is read or written (hmvec.py:504-572 with fft.py:97-115 folded in).  ws_d: hmv_power_ws_doubles(nz,nm). */
int hmv_power_tab(int nz, int nm, int nk, const double* ms_d, const double* ks_d, const double* nzm_d,
                  const double* bh_d, const double* Pzk_d, double rho_m0, double kstar, int kind, const double* tab_d,
                  int nxs, double* ws_d, double* p1h_d, double* p2h_d, void* stream);
long long hmv_power_six_tab_ws_doubles(int nz, int nm, int nk);
int hmv_power_six_tab(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d, const double* nzm_d,
                      const double* bh_d, const double* Pzk_d, double rho_m0, double kstar, const double* um_d,
                      const double* etab_d, int nxs, const double* Nc_d, const double* Ns_d, const double* NcNs_d,
                      const double* NsNsm1_d, const double* ngal_d, double* ws_d, long long spec_stride,
                      double* p1h_d, double* p2h_d, void* stream);

/* Spectra-only fusion of a4 + a12-a14: the same six spectra with the analytic NFW matter profile (hmvec.py:346-353,
 * from cs_d, rvir_d as in hmv_uk_nfw) evaluated inside the mass reduction instead of read from a cube; only the
 * electron cube ue_d is streamed.  For callers that want the spectra and never look at uk_profiles['nfw'].
 * ws_d: hmv_power_six_nfw_ws_doubles(nz,nm) doubles. */
long long hmv_power_six_nfw_ws_doubles(int nz, int nm);
int hmv_power_six_nfw(int nz, int nm, int nk, int ldk, const double* zs_d, const double* ms_d, const double* ks_d,
                      const double* nzm_d, const double* bh_d, const double* Pzk_d, double rho_m0, double kstar,
                      const double* cs_d, const double* rvir_d, const double* ue_d, const double* Nc_d,
                      const double* Ns_d, const double* NcNs_d, const double* NsNsm1_d, const double* ngal_d,
                      double* ws_d, long long spec_stride, double* p1h_d, double* p2h_d, void* stream);

/* ---- a16: Limber integral  (cosmology.py:867-904) ---------------------------------------------------
 * C_l = trapz_gz( pref[gz] * P(k=(l+1/2)/chi[gz], gz) )  (ngz>1) or pref*P (ngz==1); P by bilinear
 * interpolation in linear (k,z) with out-of-range coordinates clamped to the table edge. pref = H W1 W2/chi^2.
 * P2_d: optional second [nzp][ldp] table added to P_d at lookup (P = P1h + P2h without a temporary), or NULL.
 * ks_d [nk] and the table's redshifts zs_d [nzp] must be strictly increasing (both are binary-searched; unsorted axes
 * give wrong C_l without an error).  The window redshifts gzs_d may come in either order: the trapezoid follows them,
 * so a decreasing gzs gives -C_l, as numpy.trapz does. */
int hmv_limber(int nl, const double* ells_d, int nzp, int nk, int ldp, const double* zs_d, const double* ks_d,
               const double* P_d, const double* P2_d, int ngz, const double* gzs_d, const double* pref_d,
               const double* chis_d, double* cl_d, void* stream);

/* The same for up to HMV_LIMBER_MAXJOBS projections of tables that share the (zs, ks) grid and the multipoles, in one
 * launch (C_kk, C_kg, C_yy of one step: cosmology.py:536-597).  jobs_h: HOST array; fields as in hmv_limber, and
 * ks_d and zs_d strictly increasing as there. */
#define HMV_LIMBER_MAXJOBS 4
typedef struct hmv_limber_job {
  const double* P_d;     /* [nzp][ldp] table */
  const double* P2_d;    /* optional second table added at lookup, or NULL */
  int ngz;               /* window redshifts (1: no z integral) */
  const double* gzs_d;   /* [ngz] */
  const double* pref_d;  /* [ngz] H W1 W2 / chi^2 */
  const double* chis_d;  /* [ngz] */
  double* cl_d;          /* [nl] result */
} hmv_limber_job;
int hmv_limber_multi(int njobs, const hmv_limber_job* jobs_h, int nl, const double* ells_d, int nzp, int nk, int ldp,
                     const double* zs_d, const double* ks_d, void* stream);

/* Sum-and-pack in front of the one all-gather of a z-sharded run: out_d[z][s][k] = a_s[z][k] + b_s[z][k] for up to
 * four spectra (P1h + P2h of C_kk's P_mm, C_kg's P_gm, C_yy's P_yy, cosmology.py:536-597).  a_h / b_h: HOST arrays of
 * nsp device pointers to [nz][nk] tables (b_h or any b_h[s] may be NULL).  After all_gather the table of spectrum s is
 * out + s*nk with row stride ldp = nsp*nk for hmv_limber. */
int hmv_pack_sum(int nz, int nk, int nsp, const double* const* a_h, const double* const* b_h, double* out_d,
                 void* stream);

/* ---- (e) multi-GPU: the z-sharded run's one exchange, fused into the kernel that forms the tables -----------------
 * (cosmology.py:867-904 integrates P(k,z) over ALL redshifts; zshard.py shards z over the GPUs of one box.)
 * hmv_peer_scatter is hmv_pack_sum whose stores go over NVLink into the gathered [nrow_total][nsp][ncol] table of
 * EVERY rank: peer_buf_h[p] / peer_flag_h[p] are this process's mappings of rank p's table and of its flag array
 * (HMV_MAX_PEERS x uint64, zero-initialised), obtained with hmv_peer_alloc on the owner and hmv_peer_open (CUDA IPC,
 * one box) on the others; entry `rank` is the local allocation.  The last CTA stores `step` (> 0, increasing) to
 * flag[rank] on every peer; hmv_peer_wait queues a one-CTA kernel that returns once all npeers flags have reached
 * `step` (or sets *status_d = 1 + the missing rank after timeout_s; it never hangs).  Alternate two tables by step
 * parity; scatter, wait and the consumers of one rank must be queued on one stream.  done_d: one zeroed uint32.
 * These are the only entry points that allocate: peer buffers must come from cudaMalloc to be exportable. */
#define HMV_MAX_PEERS 16
int hmv_peer_alloc(long long bytes, void** ptr_out, unsigned char* handle64_out);
int hmv_peer_open(const unsigned char* handle64, void** ptr_out);
int hmv_peer_close(void* ptr);
int hmv_peer_free(void* ptr);
int hmv_peer_scatter(int nrow, int ncol, int nsp, const double* const* a_h, const double* const* b_h, int npeers,
                     int rank, void* const* peer_buf_h, void* const* peer_flag_h, long long row0,
                     unsigned long long step, unsigned int* done_d, void* stream);
int hmv_peer_wait(const void* flags_d, int npeers, unsigned long long step, double timeout_s, int* status_d,
                  void* stream);

/* ---- launch-order introspection (host only, no device work): what the CPU tests check --------------------------
 * hmv_debug_k1_order: (z, mass group counted from the heavy end) of every position of hmv_profile_transform's work
 *   queue on an nz x nm grid with `grid` CTAs (0 = 148); z_out/q_out: HOST arrays of nz*ceil(nm/16) ints; returns the
 *   number of mass groups.  hmv_debug_wave_tile: the k-tile width hmv_power_six picks for nz redshifts of ldk columns.
 * hmv_debug_tab_order: (z, first wavenumber) of every CTA of hmv_power_tab in launch order; HOST arrays of
 *   nz*ceil(nk/tile) ints; returns the tile width.  Every (z, group) / (z, tile) must occur exactly once. */
int hmv_debug_k1_order(int nz, int nm, int grid, int* z_out, int* q_out);
int hmv_debug_wave_tile(int nz, int ldk);
int hmv_debug_tab_order(int nz, int nk, int* z_out, int* k0_out);

/* ---- 1-halo trispectrum and the non-Gaussian Limber covariance of C_l ----------------------------------------------
 * No counterpart in the reference.  The 1-halo term of the power-spectrum covariance (Cooray & Hu 2001, ApJ 554, 56,
 * eq. 17; Cooray & Sheth 2002, Phys. Rep. 372, 1, §6.2) and its Limber projection (Komatsu & Seljak 2002, MNRAS 336,
 * 1256, eq. 14 for the tSZ), with the window convention of hmv_limber (C = int dz H W1 W2/chi^2 P).  A profile
 * tracer's leg is t_X(z,m,k) = a_X u_X(z,m,k): kind 0 (matter) a = M/rho_m0, kind 2 (pressure) a = 1, as in hmv_power;
 * u is linear in k on ks (strictly increasing, nk >= 2) with k clamped to [ks[0], ks[nk-1]] as in hmv_limber.
 *   T^{ABCD}(k1,k2;z) = sum_m w_m n(z,m) t_A(k1) t_B(k1) t_C(k2) t_D(k2)      w_m: trapezoid weight on ms
 *   Cov^{AB,CD}(l,l') = sum_z zeta_z pref[z] T((l+1/2)/chi[z], (l'+1/2)/chi[z]; z)
 * with zeta_z the trapezoid weight on zs (1 when nz == 1) and pref[z] = H^3 W_A W_B W_C W_D / chi^6 / (4 pi f_sky)
 * supplied by the caller (W = the lensing window for kappa, 1 for Compton-y).  No 1-halo damping (1 - e^{-(k/k*)^2}).
 * u_h / kind_h: HOST arrays of the four cubes [nz][nm][ldk] (A, B at k1; C, D at k2) and their kinds (0 or 2).
 * k1/k2 and ells1/ells2 need not be sorted.  Cubes and ws_d must be 16-byte aligned and ldk even (HMV_E_ARG);
 * nz <= 65535 and nz * nm <= 2^30 (HMV_E_LIMIT).  Every check is made before the first launch.
 * One FP64 tensor-core contraction over (z, m): panels of t_A t_B (weights folded in) and t_C t_D in ws_d, then the
 * sigma^2 GEMM (mma.sync m8n8k4) with a fixed-order split-k reduction: repeated calls give identical results.
 * hmv_trispec_1h: out_d [nz][nk1][nk2].  hmv_cl_cov_1h: out_d [nl1][nl2].  ws_d: *_ws_doubles() doubles. */
long long hmv_trispec_1h_ws_doubles(int nz, int nm, int nk1, int nk2);
int hmv_trispec_1h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                   double rho_m0, const double* const* u_h, const int* kind_h, int nk1, const double* k1_d, int nk2,
                   const double* k2_d, double* ws_d, double* out_d, void* stream);
long long hmv_cl_cov_1h_ws_doubles(int nz, int nm, int nl1, int nl2);
int hmv_cl_cov_1h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                  double rho_m0, const double* const* u_h, const int* kind_h, int nl1, const double* ells1_d, int nl2,
                  const double* ells2_d, const double* zs_d, const double* chis_d, const double* pref_d, double* ws_d,
                  double* out_d, void* stream);

/* The same with galaxy (HOD) legs (DESIGN.md §4.8).  legs_h: HOST array of four hmv_tracer (A, B at k1; C, D at k2)
 * in place of u_h / kind_h; the other arguments as in hmv_trispec_1h / hmv_cl_cov_1h.  Kind 0 and 2 legs are the
 * profile legs above (us_d the cube; uc_d and the occupation arrays are not read); a kind-1 leg is the HOD leg of
 * hmv_power, t_g = (Nc UC + Ns US)/ngal with UC = 1 when uc_d is NULL.  Two galaxy legs take the pair moment without
 * self-pairs, <g g>(k,k') = [NsNsm1 US(k) US(k') + NcNs (UC(k) US(k') + US(k) UC(k'))]/ngal^2, in place of t_g t_g:
 * on one side (A, B or C, D) it is formed per column; one on each side runs the contraction over two segments of mass
 * rows per redshift, K = nz * 2 * nm (even-padded) <= 2^30.  HMV_E_ARG before any launch for: a kind-1 leg with a
 * NULL occupation array, three or four kind-1 legs (moments the HOD does not define), kind-1 legs that differ in any
 * cube or occupation pointer (two HODs: no joint occupation), a non-NULL bias_d, and the checks of hmv_trispec_1h.
 * Profile legs only give hmv_trispec_1h / hmv_cl_cov_1h's result to the bit.  The workspace functions take the legs
 * (the segment count depends on them) and return 0 on invalid sizes or NULL legs_h. */
long long hmv_trispec_1h_tracers_ws_doubles(int nz, int nm, int nk1, int nk2, const hmv_tracer* legs_h);
int hmv_trispec_1h_tracers(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                           const double* nzm_d, double rho_m0, const hmv_tracer* legs_h, int nk1, const double* k1_d,
                           int nk2, const double* k2_d, double* ws_d, double* out_d, void* stream);
long long hmv_cl_cov_1h_tracers_ws_doubles(int nz, int nm, int nl1, int nl2, const hmv_tracer* legs_h);
int hmv_cl_cov_1h_tracers(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d,
                          const double* nzm_d, double rho_m0, const hmv_tracer* legs_h, int nl1,
                          const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                          const double* chis_d, const double* pref_d, double* ws_d, double* out_d, void* stream);

/* ---- 2-halo trispectrum and its non-Gaussian Limber covariance of C_l (DESIGN.md §4.6) ----------------------------
 * No counterpart in the reference.  Cooray & Hu 2001, ApJ 554, 56; Cooray & Sheth 2002, Phys. Rep. 372, 1, §6.2.  Legs,
 * kinds, ks and the projection as in hmv_trispec_1h / hmv_cl_cov_1h; w^ = w_m n(z,m) b(z,m) (bh_d [nz][nm]).  For
 * T(k1,-k1,k2,-k2) averaged over the angle between k1 and k2, legs A, B at k1 and C, D at k2:
 *   I2^{XY}(k,k')      = sum_m w^ t_X(k) t_Y(k')          I3^{XYZ}(k,k',k'') = sum_m w^ t_X(k) t_Y(k') t_Z(k'')
 *   I1~X(k)            = sum_m w^ t_X(k) + b_X - C_X       (matter b = 1, C = sum_m w^ M/rho_m0; pressure 0, 0)
 *   P(k)               = Pzk[z] linear in k on ks, held at the end values outside
 *   Pbar(k1,k2)        = (1/(2 k1 k2)) int_{|k1-k2|}^{k1+k2} q P(q) dq        (closed form; P piecewise linear)
 *   T2h(k1,k2;z)       = P(k1) [I1~A I3^{BCD} + I1~B I3^{ACD}] + P(k2) [I1~C I3^{ABD} + I1~D I3^{ABC}]
 *                      + Pbar [I2^{AC} I2^{BD} + I2^{AD} I2^{BC}]
 *   Cov2h(l,l')        = sum_z zeta_z pref[z] T2h((l+1/2)/chi[z], (l'+1/2)/chi[z]; z),  pref as in hmv_cl_cov_1h
 * The (AB)(CD) pairing carries P_lin(0) and is dropped; I2 and I3 carry no consistency term; no 1-halo damping.
 * zchunk (1 <= zchunk <= nz) redshifts per pass bound the workspace; the result is bit-identical for every zchunk and
 * for repeated calls.  Legs coincide when they have the same cube pointer and kind: 8 contracted blocks when neither
 * side coincides, 5 when A == B or C == D, 3 when both.  The workspace functions take the legs for that reason and nk
 * for the per-redshift Pbar prefix table; they return 0 on invalid sizes or zchunk.  Argument checks, codes and
 * messages as hmv_trispec_1h, plus bh_d / Pzk_d non-null and the zchunk range, all before the first launch.
 * hmv_trispec_2h: out_d [nz][nk1][nk2].  hmv_cl_cov_2h: out_d [nl1][nl2]. */
long long hmv_trispec_2h_ws_doubles(int nz, int nm, int nk, int nk1, int nk2, const double* const* u_h,
                                    const int* kind_h, int zchunk);
int hmv_trispec_2h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                   const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                   int nk1, const double* k1_d, int nk2, const double* k2_d, int zchunk, double* ws_d, double* out_d,
                   void* stream);
long long hmv_cl_cov_2h_ws_doubles(int nz, int nm, int nk, int nl1, int nl2, const double* const* u_h,
                                   const int* kind_h, int zchunk);
int hmv_cl_cov_2h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                  const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                  int nl1, const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                  const double* chis_d, const double* pref_d, int zchunk, double* ws_d, double* out_d, void* stream);

/* ---- 3- and 4-halo trispectra and their non-Gaussian Limber covariance of C_l (DESIGN.md §4.7) ----------------------
 * No counterpart in the reference.  Cooray & Hu 2001, ApJ 554, 56; Takada & Jain 2009, MNRAS 395, 2065.  Legs, kinds,
 * w^, I1~X, I2^{XY}, P and the projection as in hmv_trispec_2h / hmv_cl_cov_2h; P1 = P(k1), P2 = P(k2).  For
 * T(k1,-k1,k2,-k2) averaged over mu = k1^.k2^ (<.> = (1/2) int_{-1}^{1} dmu), q = |k1 + k2|:
 *   G(mu)        = P1 F2(-k1, k1+k2) + P2 F2(-k2, k1+k2),  F2 the symmetric second-order PT kernel
 *   F3bar(r)     = <F3_sym(k, q', -q')>, r = q'/k (the P13 kernel divided by 3024 r^2)
 *   Bbar(k1,k2)  = (34/21) P1 P2 + 2 <G P(q)>
 *   Tbar(k1,k2)  = 12 P1 P2^2 F3bar(k2/k1) + 12 P1^2 P2 F3bar(k1/k2) + 8 <G^2 P(q)>
 *   T3h(k1,k2;z) = Bbar [I2^{AC} I1~B I1~D + I2^{AD} I1~B I1~C + I2^{BC} I1~A I1~D + I2^{BD} I1~A I1~C]
 *   T4h(k1,k2;z) = I1~A I1~B I1~C I1~D Tbar
 * Terms carrying P(0) are dropped.  <G P> and <G^2 P> are exact for P piecewise linear (per-redshift moment tables of
 * int q^n P dq, n = -3, -1, 1, 3, 5); ks must be positive and k1, k2 > 0.  hmv_*_3h: zchunk and the workspace as in
 * hmv_trispec_2h, with 1, 2 or 4 contracted I2 blocks (A == B and C == D, one of them, neither).  hmv_*_4h: one pass,
 * no contraction; the workspace depends on the sizes only.  The workspace functions return 0 on invalid sizes or
 * zchunk.  Argument checks, codes and messages as hmv_trispec_2h, all before the first launch; the result is
 * bit-identical for every zchunk and for repeated calls.  hmv_trispec_3h/4h: out_d [nz][nk1][nk2];
 * hmv_cl_cov_3h/4h: out_d [nl1][nl2]. */
long long hmv_trispec_3h_ws_doubles(int nz, int nm, int nk, int nk1, int nk2, const double* const* u_h,
                                    const int* kind_h, int zchunk);
int hmv_trispec_3h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                   const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                   int nk1, const double* k1_d, int nk2, const double* k2_d, int zchunk, double* ws_d, double* out_d,
                   void* stream);
long long hmv_cl_cov_3h_ws_doubles(int nz, int nm, int nk, int nl1, int nl2, const double* const* u_h,
                                   const int* kind_h, int zchunk);
int hmv_cl_cov_3h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                  const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                  int nl1, const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                  const double* chis_d, const double* pref_d, int zchunk, double* ws_d, double* out_d, void* stream);
long long hmv_trispec_4h_ws_doubles(int nz, int nk, int nk1, int nk2);
int hmv_trispec_4h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                   const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                   int nk1, const double* k1_d, int nk2, const double* k2_d, double* ws_d, double* out_d,
                   void* stream);
long long hmv_cl_cov_4h_ws_doubles(int nz, int nk, int nl1, int nl2);
int hmv_cl_cov_4h(int nz, int nm, int nk, int ldk, const double* ks_d, const double* ms_d, const double* nzm_d,
                  const double* bh_d, const double* Pzk_d, double rho_m0, const double* const* u_h, const int* kind_h,
                  int nl1, const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d,
                  const double* chis_d, const double* pref_d, double* ws_d, double* out_d, void* stream);

/* ---- super-sample covariance of C_l (matter and pressure profiles) ---------------------------------------------------
 * No counterpart in the reference.  Takada & Hu 2013, PRD 87, 123504; Li, Hu & Takada 2014, PRD 89, 083519.  Legs t_X
 * and kinds as in hmv_trispec_1h (0: matter, a = M/rho_m0; 2: pressure, a = 1); w_m the trapezoid weight on ms.
 * hmv_power_response: the response of P^{AB}(k,z) to a long-wavelength mode, on ks (strictly increasing, nk >= 2):
 *   r1h[z][k] = sum_m w_m n(z,m) b(z,m) t_A(z,m,k) t_B(z,m,k)                 (no 1-halo damping)
 *   r2h[z][k] = [47/21 - n_eff(z,k)/3] P2h^{AB}(z,k)
 * P2h is hmv_power's 2-halo term, P_lin (I_A + b_A - C_A)(I_B + b_B - C_B) (pressure: b = 0, no consistency term);
 * n_eff = d ln P_lin/d ln k as np.gradient(log Pzk, log ks, axis=1): second-order non-uniform stencil inside,
 * one-sided at the ends.  A Pzk that is not positive at a column or at a neighbour the stencil reads gives NaN there.
 * One pass over the cube (uA_d == uB_d) or the two cubes, as hmv_power's power_one / power_pair.  r1h_d or r2h_d may
 * be NULL, not both; ws_d: hmv_power_ws_doubles(nz, nm) doubles.  Cubes and ws_d 16-byte aligned, ldk even (HMV_E_ARG);
 * nz <= 65535 (HMV_E_LIMIT).  Every check is made before the first launch.
 * hmv_sigma_b2: out[z] = sum_j kw[j] P[z][j] (2 J1(ks[j] R[z]) / (ks[j] R[z]))^2, P [nz][nks]: the variance of the
 *   background mode over a disc of radius R (flat sky) when kw = Simpson weight * k / (2 pi).  x = 0 gives W = 1.
 * hmv_cl_cov_ssc: Cov^{AB,CD}(l,l') = sum_z zeta_z pref[z] R^{AB}((l+1/2)/chi[z], z) R^{CD}((l'+1/2)/chi[z], z),
 *   rAB/rCD [nz][nk] (R1h + R2h), linear in k on ks with k clamped to its ends, zeta_z the trapezoid weight on zs (1 when
 *   nz == 1), pref[z] = H^3 W_A W_B W_C W_D sigma_b^2 / chi^4 from the caller.  out_d [nl1][nl2]; ws_d:
 *   hmv_cl_cov_ssc_ws_doubles() doubles, 16-byte aligned; nz <= 65535.  The contraction of hmv_cl_cov_1h with one K
 *   row per redshift; repeated calls give identical results. */
int hmv_power_response(int nz, int nm, int nk, int ldk, const double* ms_d, const double* ks_d, const double* nzm_d,
                       const double* bh_d, const double* Pzk_d, double rho_m0, const double* uA_d, int kindA,
                       const double* uB_d, int kindB, double* ws_d, double* r1h_d, double* r2h_d, void* stream);
int hmv_sigma_b2(int nz, int nks, const double* ks_d, const double* kw_d, const double* P_d, const double* R_d,
                 double* out_d, void* stream);
long long hmv_cl_cov_ssc_ws_doubles(int nz, int nl1, int nl2);
int hmv_cl_cov_ssc(int nz, int nk, const double* ks_d, const double* rAB_d, const double* rCD_d, int nl1,
                   const double* ells1_d, int nl2, const double* ells2_d, const double* zs_d, const double* chis_d,
                   const double* pref_d, double* ws_d, double* out_d, void* stream);

/* ---- f2: kSZ consumer -- the short-wavelength integral of the velocity-reconstruction noise
 * (ksz.py:299-336, Nvv_core_integral):  out[b] = trapz_kS( kS Pge[b,kS]^2 / (Pgg_tot[b,kS] C_tot(chi* kS)) ) with
 * non-finite integrand values set to zero (ksz.py:98-100).  b = 0..nb-1 runs over the (mu,kL) plane when the spectra
 * carry the photo-z window (stride nk) or is one row (nb = 1).  pge_d NULL = 1 (errs mode); pgg_photo_d optional
 * (robust term: integrand * Pgg_photo_tot/Pgg_tot).  clk_d[k] = C_tot at l = chi* kS[k] (host lookup, O(nk)). */
int hmv_ksz_nvv_integral(int nb, int nk, const double* ks_d, const double* pge_d, long long pge_stride,
                         const double* pgg_d, long long pgg_stride, const double* pgg_photo_d, long long photo_stride,
                         const double* clk_d, double* out_d, void* stream);

/* ---- next row (SURVEY 8f-1): P(z,k) from a matter-power interpolator  (cosmology.py:227-229, 353-382;
 *      utils.py:95-103 `PKInterpolator.P`; CAMB get_matter_power_interpolator) -------------------------------
 * out[z][k] = scale * (islog ? exp(s) : s),  s = the tensor-product B-spline (knots tx[nx], ty[ny], degrees kx, ky,
 * coefficients c[(nx-kx-1)(ny-ky-1)], as in scipy RectBivariateSpline.tck) evaluated at (zs[z], ln ks[k]) with
 * FITPACK bispev's conventions (arguments clamped to the knot range).  The fit itself stays on the host.
 * scale carries logsign * as8^2. */
int hmv_pk_spline(int nz, int nk, const double* zs_d, const double* ks_d, int nx, int ny, int kx, int ky,
                  const double* tx_d, const double* ty_d, const double* c_d, int islog, double scale, double* out_d,
                  void* stream);

/* v(k) = pref k (k/kp)^(ns-1) T_EH98(k)^2: the wavenumber factor of the separable accuracy='low' linear power
 * (reference cosmology.py:391-402, Tk :404-504; Eisenstein & Hu 1998 with oscillations, or the no-wiggle fit). */
int hmv_eh98_factor(int nk, const double* ks_d, double h, double omch2, double ombh2, double omm0, int wiggles,
                    double pref, double kp, double ns, double* out_d, void* stream);
/* accuracy='low' linear power (cosmology.py:391-402) is separable, P(z,k) = D(z)^2 * [pref k (k/kp)^(ns-1) T(k)^2]:
 * out[z][k] = a[z] * b[k] from the two host-side factor vectors, so that neither Pzk [nz,nk] nor the sigma^2 spectrum
 * [nz,sigma2_numks] crosses PCIe. */
int hmv_outer(int nz, int nk, const double* a_d, const double* b_d, double* out_d, void* stream);
/* out = a + b elementwise: P = P1h + P2h of get_power (hmvec.py:500-502) formed on the device before the download. */
int hmv_sum2(long long n, const double* a_d, const double* b_d, double* out_d, void* stream);

/* ---- test hook: elementwise Si(x), Ci(x) of the device routine used by hmv_uk_nfw (x > 0) -----------*/
int hmv_sici_test(int n, const double* x_d, double* si_d, double* ci_d, void* stream);

/* ---- measurement helpers (bench.py) -------------------------------------------------------------------
 * hmv_bench_dfma: dependent-chain-free DFMA micro-benchmark; returns achieved FP64 TFLOP/s (2 flop per FMA)
 * on the current device, timed with CUDA events.  hmv_bench_copy: device copy GB/s (read+write bytes). */
double hmv_bench_dfma(int iters, void* stream);
/* hmv_bench_dmma: the same for FP64 tensor-core mma.sync m8n8k4 (512 flop per warp instruction). */
double hmv_bench_dmma(int iters, void* stream);
double hmv_bench_copy(const double* src_d, double* dst_d, long long n, int reps, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HMVEC_B200_H */
