"""GridSix: the whole hot path for one z-slab as a stream-ordered, allocation-free launch sequence.

    sigma^2 -> n(M,z), b(M,z) -> halo geometry -> u_NFW cube -> M200c, GNFW parameters -> u_electron cube ->
    Compton-y pressure cube -> HOD (mthresh<->ngal bisection + occupations) -> {mm,ee,me,gg,gm,ge} 1h+2h spectra ->
    yy 1h+2h spectrum -> [all-gather over z] -> Limber C_kk, C_kg, C_yy

This is what `HaloModel(...)`, `add_battaglia_profile`, `add_battaglia_pres_profile`, `add_hod(ngal=...)`, seven
`get_power` calls and `C_kk`/`C_kg`/`C_yy` do in the reference (hmvec.py:76-572, cosmology.py:536-568,867-904), arranged B200-first: every buffer
(two [nz][nm][ldk] cubes, ~20 [nz,nm] arrays, workspaces, outputs) is allocated once in __init__, `run()` only issues
kernel launches through the C ABI on the current stream with no host synchronisation, host inputs arrive through
pinned staging buffers (`upload`) and results leave through pinned buffers (`download`).  Host-side inputs (the CAMB
products and O(nz) background scalars) are prepared by `make_inputs`.
"""
import ctypes as C

import numpy as np
import torch

from . import _capi as capi
from .cosmology import Cosmology, simpson_weights
from .params import default_params, battaglia_defaults

TAGS = ("mm", "ee", "me", "gg", "gm", "ge")
_KIND_PRESSURE = 2

# host inputs that change with the cosmology / redshift slab (uploaded every e2e step), name -> shape key
_PER_STEP = ("Pzk", "sPzk", "drho1", "drho2", "rhocrit", "hofz", "ngal_target")


def make_inputs(zs, ms, ks, params=None, mdef='vir', ngal=None, ells=None, lzs=2.5, gz=0.8, accuracy='low'):
    """Host-side producers: linear power on `ks` and on the sigma^2 grid, Simpson weights, background scalars per z,
    Limber prefactors.  Everything here is O(nz*nk) numpy work on inputs of the path (north_star: "Linear P(k) from
    CAMB stays a host-side input")."""
    zs = np.asarray(zs, dtype=np.float64).reshape(-1)
    ms = np.asarray(ms, dtype=np.float64).reshape(-1)
    ks = np.asarray(ks, dtype=np.float64).reshape(-1)
    c = Cosmology(dict(params or {}), accuracy=accuracy)
    p = c.p
    ks_sig = np.geomspace(p['sigma2_kmin'], p['sigma2_kmax'], int(p['sigma2_numks']))
    rho_m0 = float(np.atleast_1d(c.rho_matter_z(0.))[0])
    rhoc = np.asarray(c.rho_critical_z(zs), dtype=np.float64)
    if mdef == 'vir':
        x = c.omz(zs) - 1.
        drho1 = rhoc * (18. * np.pi ** 2. + 82. * x - 39. * x ** 2.)
    elif mdef == 'mean':
        drho1 = c.rho_matter_z(zs) * 200.
    else:
        raise ValueError("mdef must be 'vir' or 'mean'")
    inp = dict(zs=zs, ms=ms, ks=ks, ks_sig=ks_sig,
               kw=simpson_weights(ks_sig) * ks_sig ** 2. / 2. / np.pi ** 2.,
               R=(3. * ms / 4. / np.pi / rho_m0) ** (1. / 3.),
               Pzk=c.P_lin_approx(ks, zs), sPzk=c.P_lin_approx(ks_sig, zs),
               drho1=np.asarray(drho1, dtype=np.float64), drho2=200. * rhoc, rhocrit=rhoc,
               hofz=np.asarray(c.h_of_z(zs), dtype=np.float64),
               ngal_target=np.geomspace(1e-3, 1e-5, zs.size) if ngal is None else np.asarray(ngal, dtype=np.float64),
               rho_m0=rho_m0, h=c.h, p=p, mdef=mdef)
    if ells is not None:
        chis = c.comoving_radial_distance(zs)
        W = c.lensing_window(zs, lzs)
        with np.errstate(all="ignore"):
            inp["ells"] = np.asarray(ells, dtype=np.float64)
            inp["chis"] = chis
            inp["pref_kk"] = inp["hofz"] * W * W / chis ** 2.                  # cosmology.py:887 with C_kk's windows
            chig = c.comoving_radial_distance(np.array([gz]))
            inp["gz"] = np.array([gz])
            inp["chig"] = chig
            inp["pref_kg"] = c.h_of_z(np.array([gz])) * c.lensing_window(np.array([gz]), lzs) / chig ** 2.
            inp["pref_yy"] = inp["hofz"] / chis ** 2.                         # cosmology.py:591-597: both windows 1
    inp["omm0"] = c.omm0
    return inp


def slab_inputs(inp, sl):
    """The rows of the per-redshift inputs owned by slab `sl` (everything else is replicated)."""
    out = dict(inp)
    for k in ("zs", "Pzk", "sPzk", "drho1", "drho2", "rhocrit", "hofz", "ngal_target"):
        out[k] = np.ascontiguousarray(inp[k][sl])
    return out


class GridSix(object):
    STAGES = ("sigma2", "massfn", "uk_nfw", "uk_electron", "uk_pressure", "hod", "power_six", "power_yy", "limber")

    def __init__(self, inp, device=None, zcomm=None, family="AGN", xmax=None, nxs=None, nz_total_zs=None,
                 fused_nfw=False, tsz=True, tsz_tables=True):
        """inp: this rank's slab of `make_inputs` (see slab_inputs).  zcomm: zshard.ZComm for a sharded z axis;
        nz_total_zs: the full redshift vector (needed for Limber after the all-gather).  fused_nfw: spectra-only
        variant -- the NFW profile is evaluated inside the mass reduction (hmv_power_six_nfw), its cube is never
        written and 32 GB of HBM stay free; the default materialises it first (hmv_uk_nfw + hmv_power_six), which
        measured FASTER on B200 (10.9 + 8.9 ms vs 21.5 ms: the fused kernel trades HBM traffic for issue slots --
        one k per thread instead of eight k per lane sharing each coefficient load -- see DESIGN.md).
        tsz_tables (default): the Compton-y profile stays in the transform's bin tables (hmv_profile_tables) and P_yy is
        reduced straight from them (hmv_power_tab) -- its 32 GB cube is never written or read (measured 3.0 vs 4.6 ms on
        a 64-z slab); False materialises the cube (hmv_profile_transform + hmv_power) as every other consumer needs."""
        if "ells" in inp:
            # hmv_limber_multi binary-searches ks and the table's redshifts; sorting them here would cost a gather of
            # the packed table every step, so a Limber grid must come sorted
            for name, x in (("ks", inp["ks"]), ("zs", inp["zs"] if nz_total_zs is None else nz_total_zs)):
                if not np.all(np.diff(np.asarray(x, dtype=np.float64).reshape(-1)) > 0):
                    raise ValueError("GridSix with ells: %s must be strictly increasing" % name)
        if not torch.cuda.is_available():
            raise RuntimeError("hmvec_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback.")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.zcomm = zcomm
        p = self.p = inp["p"]
        self.nz, self.nm, self.nk = inp["zs"].size, inp["ms"].size, inp["ks"].size
        self.nks = inp["ks_sig"].size
        self.ldk = ((self.nk + 15) // 16) * 16
        self.rho_m0, self.h = inp["rho_m0"], inp["h"]
        self.kmax = float(np.max(inp["ks"]))
        self.xmax = float(p['electron_density_profile_integral_xmax'] if xmax is None else xmax)
        self.nxs = int(p['electron_density_profile_integral_numxs'] if nxs is None else nxs)
        tag = 'mean' if inp["mdef"] == 'mean' else 'vir'
        self.duffy = (p['duffy_A_' + tag], p['duffy_alpha_' + tag], p['duffy_beta_' + tag])
        fam = battaglia_defaults[family]
        self.gamma = float(p['battaglia_gas_gamma'])
        self.fit9 = capi.darr([fam[q + s] for q in ('rho0', 'alpha', 'beta') for s in ('_A0', '_alpham', '_alphaz')])
        # tSZ leg (BASELINE.json configs[4]): Battaglia-2012 pressure profile -> P_yy -> C_yy
        self.tsz = bool(tsz)
        self.tsz_tables = bool(tsz_tables) and self.tsz
        pf = battaglia_defaults[p['battaglia_pres_family']]
        self.pfit9 = capi.darr([pf[q + s] for q in ('P0', 'xc', 'beta') for s in ('_A0', '_alpham', '_alphaz')])
        from .hmvec import pressure_constants
        self.p_amp, self.p_pref = pressure_constants(p['ombh2'] / inp["h"] ** 2., inp["omm0"])
        self.p_xmax = float(p['electron_pressure_profile_integral_xmax'])
        self.p_nxs = int(p['electron_pressure_profile_integral_numxs'])
        self.hodp = capi.darr([p['hod_sig_log_mstellar'], p['hod_alphasat'], p['hod_Bsat'], p['hod_betasat'],
                               p['hod_Bcut'], p['hod_betacut'], 0.0, 0.0])
        f64 = dict(dtype=torch.float64, device=self.device)
        E = lambda *s: torch.empty(s, **f64)
        nz, nm, nk = self.nz, self.nm, self.nk
        # replicated inputs (uploaded once)
        self.d = {k: torch.as_tensor(np.array(inp[k], dtype=np.float64), device=self.device)
                  for k in ("zs", "ms", "ks", "ks_sig", "kw", "R")}
        # per-step inputs: pinned host staging + device buffers
        self.h_in = {k: torch.as_tensor(np.array(inp[k], dtype=np.float64)).pin_memory() for k in _PER_STEP}
        for k in _PER_STEP:
            self.d[k] = torch.empty_like(self.h_in[k], device=self.device)
        # intermediates
        for k in ("sigma2", "nzm", "bh", "cs", "rvir", "m200c", "rs", "cmax", "xc", "alpha", "expo", "amp", "oscale",
                  "Nc", "Ns", "NsNsm1", "NcNs"):
            self.d[k] = E(nz, nm)
        self.d["ngal"], self.d["bg"], self.d["l10"] = E(nz), E(nz), E(nz)
        self.d["sig_ws"] = E(int(capi.lib.hmv_sigma2_ws_doubles(nz, nm, self.nks)))
        self.d["nfw_ws"] = E(int(capi.lib.hmv_uk_nfw_ws_doubles(nz, nm, nk)))
        self.d["tr_ws"] = E(int(capi.lib.hmv_profile_transform_ws_doubles(nz, nm, max(self.nxs, self.p_nxs if self.tsz else 0))))
        self.d["pow_ws"] = E(int(capi.lib.hmv_power_ws_doubles(nz, nm)))
        self.d["bis_ws"] = E(nz * (capi.HMV_BISECT_MAXIT + 4))
        self.mask = torch.empty(1, dtype=torch.int64, device=self.device)
        self.iters = torch.zeros(1, dtype=torch.int32, device=self.device)
        # the two cubes: [nz][nm][ldk]; pad columns (if any) zeroed once, never written by the kernels
        self.fused_nfw = bool(fused_nfw)
        self.um = None if self.fused_nfw else torch.empty((nz, nm, self.ldk), **f64)
        self.ue = torch.empty((nz, nm, self.ldk), **f64)
        if self.ldk > nk:
            self.ue[..., nk:] = 0.0
            if self.um is not None:
                self.um[..., nk:] = 0.0
        if self.fused_nfw:
            self.d["pow_ws"] = E(int(capi.lib.hmv_power_six_nfw_ws_doubles(nz, nm)))
        # spectra: rows 0-5 = TAGS, row 6 = yy (Compton-y auto spectrum) when the tSZ leg is on
        self.nsp = 7 if self.tsz else 6
        self.p1 = E(self.nsp, nz, nk)
        self.p2 = E(self.nsp, nz, nk)
        self.h_p1 = torch.empty((self.nsp, nz, nk), dtype=torch.float64).pin_memory()
        self.h_p2 = torch.empty((self.nsp, nz, nk), dtype=torch.float64).pin_memory()
        if self.tsz:
            if self.tsz_tables:
                self.uy = None
                self.ytab = E(int(capi.lib.hmv_profile_table_doubles(nz, nm, self.p_nxs)))
            else:
                self.uy = torch.empty((nz, nm, self.ldk), **f64)
                if self.ldk > nk:
                    self.uy[..., nk:] = 0.0
            for k in ("y_rs", "y_cmax", "y_xc", "y_alpha", "y_expo", "y_amp", "y_oscale"):
                self.d[k] = E(nz, nm)
            self.d["pair_ws"] = E(int(capi.lib.hmv_power_ws_doubles(nz, nm)))
            self.ty = capi.Tracer()
            self.ty.kind = _KIND_PRESSURE
            self.ty.us_d = self.uy.data_ptr() if self.uy is not None else None
        # Limber (replicated on every rank after the all-gather)
        self.has_limber = "ells" in inp
        if self.has_limber:
            self.zs_all = torch.as_tensor(np.array(inp["zs"] if nz_total_zs is None else nz_total_zs, dtype=np.float64),
                                          device=self.device)
            self.nl = inp["ells"].size
            for k in ("ells", "chis", "pref_kk", "gz", "chig", "pref_kg", "pref_yy"):
                self.d[k] = torch.as_tensor(np.array(inp[k], dtype=np.float64), device=self.device)
            self.ncl = 3 if self.tsz else 2
            self.cl = E(self.ncl, self.nl)
            self.h_cl = torch.empty((self.ncl, self.nl), dtype=torch.float64).pin_memory()
        self.launches_per_run = 0
        self.transform_mode = 0      # the transform's only launch plan; bench.py sets this attribute and reads it back
        self._ev = None
        self._Pfull = None
        self._Ppack = None
        self._peer = None
        # the download (224 MB on the full grid) takes about as long as the reduction: start it early, end it small.
        # >= 12 redshifts per reduction launch: a 25-z slab (8 GPUs) still runs as two launches of ~1.7 waves each --
        # the same four wave-times as one launch of 3.4 -- and the first half's copy hides behind the second half
        self.d2h_chunks = int(min(10, max(1, self.nz // 12)))
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.ev_chunk = [torch.cuda.Event() for _ in range(self.d2h_chunks)]
        self.ev_pzk = torch.cuda.Event()
        self.ev_yy = torch.cuda.Event()
        self.hod_stream = torch.cuda.Stream(device=self.device)
        self.ev_mf, self.ev_hod = torch.cuda.Event(), torch.cuda.Event()
        self.hod_overlap = True
        # `overlap` (used when run() is not asked for per-stage events): 1 = the whole sigma^2 -> n(M), b(M) -> HOD leg runs
        # on the side stream next to the NFW cube (which needs only the halo geometry) and rejoins in front of the mass
        # integrals; 2 = also the electron transform and the tSZ leg (pressure tables -> P_yy) on streams of their own.
        # The big kernels still run one after the other (each fills every SM), but a kernel's drain -- SMs idle while
        # its last CTAs finish -- is taken by the next leg's first CTAs and the small kernels disappear behind the cubes.
        # That pays on small slabs only (tools/slab_skew.py, medians of interleaved runs, levels 0 / 1 / 2:
        # 25 z 4.80 / 4.73 / 4.54 ms, 50 z 9.13 / 9.09 / 8.92, 100 z 17.69 / 17.61 / 17.79, 200 z 35.02 / 35.27 / 35.18 --
        # on long slabs P_yy's table gathers and the six-spectra stream evict each other from L2).
        self.overlap = 2 if nz <= 64 else (1 if nz <= 128 else 0)
        self.ev_geo = torch.cuda.Event()
        self.e_stream = torch.cuda.Stream(device=self.device)
        self.y_stream = torch.cuda.Stream(device=self.device)
        self.ev_geo2, self.ev_m200, self.ev_e, self.ev_ydone = (torch.cuda.Event() for _ in range(4))
        if self.tsz:
            self.d["tr_ws_y"] = E(int(capi.lib.hmv_profile_transform_ws_doubles(nz, nm, self.p_nxs)))
        self.h_iters = torch.zeros(1, dtype=torch.int32).pin_memory()

    # ------------------------------------------------------------------ host <-> device
    def h2d_bytes(self):
        return int(sum(t.numel() * 8 for t in self.h_in.values()))

    def d2h_bytes(self):
        n = self.h_p1.numel() * 8 + self.h_p2.numel() * 8
        return int(n + (self.h_cl.numel() * 8 if self.has_limber else 0))

    def upload(self):
        """Pinned host -> HBM.  Pzk is first needed by the spectra at the end of the step, so it travels on the copy
        stream behind the kernels (run() waits for it in front of hmv_power_six); everything else is needed at once."""
        self.copy_stream.wait_stream(torch.cuda.current_stream())      # the previous step no longer reads Pzk
        with torch.cuda.stream(self.copy_stream):
            self.d["Pzk"].copy_(self.h_in["Pzk"], non_blocking=True)
            self.ev_pzk.record()
        for k in _PER_STEP:
            if k != "Pzk":
                self.d[k].copy_(self.h_in[k], non_blocking=True)

    def download(self):
        self.h_p1.copy_(self.p1, non_blocking=True)
        self.h_p2.copy_(self.p2, non_blocking=True)
        self.h_iters.copy_(self.iters, non_blocking=True)
        if self.has_limber:
            self.h_cl.copy_(self.cl, non_blocking=True)

    def _check_converged(self):
        """hmv_hod_pick reports 0 iterations when the all-z bisection never met rtol (target outside the mthresh
        bracket, NaN n(M)); spectra built on that midpoint are meaningless, so this is an error as in HaloModel."""
        if int(self.h_iters[0]) == 0:
            raise capi.HmvError("mthresh<->ngal bisection did not converge within %d iterations" % capi.HMV_BISECT_MAXIT)

    def finish_e2e(self):
        """After run(overlap_d2h=True): copy the C_ell and wait until every result is in the pinned host buffers."""
        self.h_iters.copy_(self.iters, non_blocking=True)
        if self.has_limber:
            self.h_cl.copy_(self.cl, non_blocking=True)
        self.copy_stream.synchronize()
        torch.cuda.current_stream().synchronize()
        self._check_converged()
        if self._peer is not None:
            self._peer.check()

    # ------------------------------------------------------------------ the launch sequence
    def _mark(self, i):
        if self._ev is not None:
            self._ev[i].record()

    def run(self, events=None, overlap_d2h=False):
        """Issue the whole path.  `events`: optional list of len(STAGES)+1 CUDA events recorded at the stage boundaries
        (per-kernel timing for the roofline report) -- the stages then run strictly one after the other on the current
        stream; without them the sigma^2 -> n(M), b(M) -> HOD leg runs on a side stream next to the NFW cube (see
        `overlap` in __init__) and rejoins in front of the mass integrals.  overlap_d2h: end-to-end mode -- the spectra
        leave for the pinned host buffers chunk by chunk on a copy stream while later chunks compute; finish with
        `finish_e2e()`."""
        self._ev = events
        self._n = 0
        main = torch.cuda.current_stream()
        # with stage events everything, the HOD solve included, runs on the current stream: its stage time is then a
        # kernel time, not the time it takes to queue work on a side stream
        hod_side = self.hod_overlap and events is None
        level = self.overlap if hod_side else 0
        side, legs = level >= 1, level >= 2 and not self.fused_nfw
        self._mark(0)
        if side:
            self.ev_geo.record(main)               # this step's inputs are queued on `main`
            with torch.cuda.stream(self.hod_stream):
                self.hod_stream.wait_event(self.ev_geo)
                self._st_sigma2()
                self._st_massfn()
                self._hod_stage(self.hod_stream, self.hod_stream)
        else:
            self._st_sigma2()
            self._mark(1)
            self._st_massfn()
        self._st_geometry()
        self._mark(2)
        if hod_side and not side:
            self._hod_stage(main, self.hod_stream)     # side stream, concurrent with the cube kernels
        if legs:
            self.ev_geo2.record(main)
        if not self.fused_nfw:
            self._st_nfw()
        self._mark(3)
        if legs:
            with torch.cuda.stream(self.e_stream):
                self.e_stream.wait_event(self.ev_geo2)
                self._st_m200c()
                self.ev_m200.record(self.e_stream)
                self._st_electron()
                self.ev_e.record(self.e_stream)
        else:
            self._st_m200c()
            self._st_electron()
        self._mark(4)
        if self.tsz:
            if legs:
                with torch.cuda.stream(self.y_stream):
                    self.y_stream.wait_event(self.ev_m200)
                    self._st_pressure(self.d["tr_ws_y"])
                    self.y_stream.wait_event(self.ev_mf)      # n(M), b(M): recorded by _hod_stage on the side stream
                    self.y_stream.wait_event(self.ev_pzk)
                    self._st_yy(overlap_d2h)
                    self.ev_ydone.record(self.y_stream)
            else:
                self._st_pressure(self.d["tr_ws"])
        self._mark(5)
        if not hod_side:
            self._hod_stage(main, main)
        self._n += 6
        self._mark(6)
        main.wait_event(self.ev_pzk)                 # Pzk of this step has arrived (see upload)
        if hod_side:
            main.wait_event(self.ev_hod)             # n(M), b(M), occupations, ngal, bg are in place
        if legs:
            main.wait_event(self.ev_e)
        self._st_six(overlap_d2h)
        self._mark(7)
        if self.tsz:
            if legs:
                main.wait_event(self.ev_ydone)
            else:
                self._st_yy(overlap_d2h)
        self._mark(8)
        if self.has_limber:
            self._n += self._limber(capi.stream())
        self._mark(9)
        self.launches_per_run = self._n
        self._ev = None

    # ---- the stages (each issues on the CURRENT stream) ----
    def _st_sigma2(self):
        L, d, ptr, p = capi.lib, self.d, capi.ptr, self.p
        capi.check(L.hmv_sigma2(self.nz, self.nm, self.nks, ptr(d["sPzk"]), ptr(d["kw"]), ptr(d["ks_sig"]), ptr(d["R"]),
                                float(p['Wkr_taylor_switch']), ptr(d["sig_ws"]), ptr(d["sigma2"]), capi.stream()),
                   "hmv_sigma2")
        self._n += 3

    def _st_massfn(self):
        L, d, ptr, p, st = capi.lib, self.d, capi.ptr, self.p, capi.stream()
        capi.check(L.hmv_mass_function(self.nz, self.nm, ptr(d["sigma2"]), ptr(d["ms"]), self.rho_m0, p['st_A'], p['st_a'],
                                       p['st_p'], p['st_deltac'], ptr(d["nzm"]), ptr(d["bh"]), st), "hmv_mass_function")
        self._n += 1

    def _st_geometry(self):
        L, d, ptr, st = capi.lib, self.d, capi.ptr, capi.stream()
        capi.check(L.hmv_halo_geometry(self.nz, self.nm, ptr(d["zs"]), ptr(d["ms"]), ptr(d["drho1"]), self.duffy[0],
                                       self.duffy[1], self.duffy[2], self.h, ptr(d["cs"]), ptr(d["rvir"]), st),
                   "hmv_halo_geometry")
        self._n += 1

    def _st_nfw(self):
        L, d, ptr = capi.lib, self.d, capi.ptr
        capi.check(L.hmv_uk_nfw(self.nz, self.nm, self.nk, self.ldk, ptr(d["zs"]), ptr(d["ks"]), self.kmax, ptr(d["cs"]),
                                ptr(d["rvir"]), ptr(d["nfw_ws"]), ptr(self.um), capi.stream()), "hmv_uk_nfw")
        self._n += 3

    def _st_m200c(self):
        L, d, ptr = capi.lib, self.d, capi.ptr
        capi.check(L.hmv_mdelta(self.nz, self.nm, ptr(d["ms"]), ptr(d["cs"]), ptr(d["drho1"]), ptr(d["drho2"]),
                                ptr(d["m200c"]), capi.stream()), "hmv_mdelta")
        self._n += 1

    def _st_electron(self):
        L, d, ptr, st = capi.lib, self.d, capi.ptr, capi.stream()
        nz, nm = self.nz, self.nm
        capi.check(L.hmv_gnfw_params(0, nz, nm, ptr(d["zs"]), ptr(d["m200c"]), ptr(d["rvir"]), ptr(d["rhocrit"]),
                                     ptr(d["hofz"]), self.fit9, self.gamma, 1.0, 1.0, 1.0, ptr(d["rs"]), ptr(d["cmax"]),
                                     ptr(d["xc"]), ptr(d["alpha"]), ptr(d["expo"]), ptr(d["amp"]), ptr(d["oscale"]),
                                     st), "hmv_gnfw_params")
        capi.check(L.hmv_profile_transform(nz, nm, self.nk, self.ldk, ptr(d["zs"]), ptr(d["ks"]), self.kmax, ptr(d["rs"]),
                                           ptr(d["cmax"]), ptr(d["xc"]), ptr(d["alpha"]), ptr(d["expo"]), ptr(d["amp"]),
                                           ptr(d["oscale"]), self.gamma, self.xmax, self.nxs, 1, ptr(d["tr_ws"]),
                                           ptr(self.ue), st), "hmv_profile_transform")
        self._n += 4                 # gnfw_params, sine_table, bin_count + the persistent transform kernel

    def _st_pressure(self, ws):
        # Compton-y profile (hmvec.py:252-316): pressure GNFW, no mass norm, scaled by 4 pi sigma_T/(m_e c^2)
        # r200c^3 (1+z)^2/H -- the second invocation of the transform kernel
        L, d, ptr, p, st = capi.lib, self.d, capi.ptr, self.p, capi.stream()
        nz, nm, nk = self.nz, self.nm, self.nk
        capi.check(L.hmv_gnfw_params(1, nz, nm, ptr(d["zs"]), ptr(d["m200c"]), ptr(d["rvir"]), ptr(d["rhocrit"]),
                                     ptr(d["hofz"]), self.pfit9, float(p['battaglia_pres_gamma']),
                                     float(p['battaglia_pres_alpha']), self.p_amp, self.p_pref, ptr(d["y_rs"]),
                                     ptr(d["y_cmax"]), ptr(d["y_xc"]), ptr(d["y_alpha"]), ptr(d["y_expo"]),
                                     ptr(d["y_amp"]), ptr(d["y_oscale"]), st), "hmv_gnfw_params(pressure)")
        if self.tsz_tables:
            capi.check(L.hmv_profile_tables(nz, nm, nk, ptr(d["zs"]), ptr(d["ks"]), self.kmax, ptr(d["y_rs"]),
                                            ptr(d["y_cmax"]), ptr(d["y_xc"]), ptr(d["y_alpha"]), ptr(d["y_expo"]),
                                            ptr(d["y_amp"]), ptr(d["y_oscale"]), float(p['battaglia_pres_gamma']),
                                            self.p_xmax, self.p_nxs, 0, ptr(ws), ptr(self.ytab), st),
                       "hmv_profile_tables(pressure)")
        else:
            capi.check(L.hmv_profile_transform(nz, nm, nk, self.ldk, ptr(d["zs"]), ptr(d["ks"]), self.kmax, ptr(d["y_rs"]),
                                               ptr(d["y_cmax"]), ptr(d["y_xc"]), ptr(d["y_alpha"]), ptr(d["y_expo"]),
                                               ptr(d["y_amp"]), ptr(d["y_oscale"]), float(p['battaglia_pres_gamma']),
                                               self.p_xmax, self.p_nxs, 0, ptr(ws), ptr(self.uy), st),
                       "hmv_profile_transform(pressure)")
        self._n += 4

    def _st_six(self, overlap_d2h):
        # z-chunked so that (in e2e mode) the device->host copy of a finished chunk overlaps the next chunk's kernel
        L, d, ptr, p, st = capi.lib, self.d, capi.ptr, self.p, capi.stream()
        nz, nm, nk, ldk = self.nz, self.nm, self.nk, self.ldk
        nchunk = self.d2h_chunks if overlap_d2h else 1
        zb = np.linspace(0, nz, nchunk + 1).round().astype(int)
        S = nz * nk
        off = lambda t, z0, w: C.c_void_p(t.data_ptr() + 8 * z0 * w)
        for ci in range(nchunk):
            z0, z1 = int(zb[ci]), int(zb[ci + 1])
            if z1 == z0:
                continue
            if self.fused_nfw:
                capi.check(L.hmv_power_six_nfw(z1 - z0, nm, nk, ldk, off(d["zs"], z0, 1), ptr(d["ms"]), ptr(d["ks"]),
                                               off(d["nzm"], z0, nm), off(d["bh"], z0, nm), off(d["Pzk"], z0, nk),
                                               self.rho_m0, float(p['kstar_damping']), off(d["cs"], z0, nm),
                                               off(d["rvir"], z0, nm), off(self.ue, z0, nm * ldk),
                                               off(d["Nc"], z0, nm), off(d["Ns"], z0, nm), off(d["NcNs"], z0, nm),
                                               off(d["NsNsm1"], z0, nm), off(d["ngal"], z0, 1), ptr(d["pow_ws"]), S,
                                               off(self.p1, z0, nk), off(self.p2, z0, nk), st), "hmv_power_six_nfw")
                self._n += 3
            else:
                capi.check(L.hmv_power_six(z1 - z0, nm, nk, ldk, ptr(d["ms"]), ptr(d["ks"]), off(d["nzm"], z0, nm),
                                           off(d["bh"], z0, nm), off(d["Pzk"], z0, nk), self.rho_m0,
                                           float(p['kstar_damping']), off(self.um, z0, nm * ldk),
                                           off(self.ue, z0, nm * ldk), off(d["Nc"], z0, nm), off(d["Ns"], z0, nm),
                                           off(d["NcNs"], z0, nm), off(d["NsNsm1"], z0, nm), off(d["ngal"], z0, 1),
                                           ptr(d["pow_ws"]), S, off(self.p1, z0, nk), off(self.p2, z0, nk), st),
                           "hmv_power_six")
            self._n += 2
            if overlap_d2h:
                self.ev_chunk[ci].record()
                self.copy_stream.wait_event(self.ev_chunk[ci])
                with torch.cuda.stream(self.copy_stream):
                    for q in range(6):       # one contiguous [z1-z0, nk] block per spectrum: plain async memcpys
                        self.h_p1[q, z0:z1].copy_(self.p1[q, z0:z1], non_blocking=True)
                        self.h_p2[q, z0:z1].copy_(self.p2[q, z0:z1], non_blocking=True)

    def _st_yy(self, overlap_d2h):
        # P_yy 1h+2h (hmvec.py:512-514, 541-545: pressure tracers, b = 0, no consistency terms)
        L, d, ptr, p, st = capi.lib, self.d, capi.ptr, self.p, capi.stream()
        nz, nm, nk = self.nz, self.nm, self.nk
        if self.tsz_tables:
            capi.check(L.hmv_power_tab(nz, nm, nk, ptr(d["ms"]), ptr(d["ks"]), ptr(d["nzm"]), ptr(d["bh"]),
                                       ptr(d["Pzk"]), self.rho_m0, float(p['kstar_damping']), _KIND_PRESSURE,
                                       ptr(self.ytab), self.p_nxs, ptr(d["pair_ws"]), ptr(self.p1[6]),
                                       ptr(self.p2[6]), st), "hmv_power_tab(yy)")
        else:
            capi.check(L.hmv_power(nz, nm, nk, self.ldk, ptr(d["ms"]), ptr(d["ks"]), ptr(d["nzm"]), ptr(d["bh"]),
                                   ptr(d["Pzk"]), self.rho_m0, float(p['kstar_damping']), C.byref(self.ty),
                                   C.byref(self.ty), ptr(d["pair_ws"]), ptr(self.p1[6]), ptr(self.p2[6]), st),
                       "hmv_power(yy)")
        self._n += 2
        if overlap_d2h:
            self.ev_yy.record()
            self.copy_stream.wait_event(self.ev_yy)
            with torch.cuda.stream(self.copy_stream):
                self.h_p1[6].copy_(self.p1[6], non_blocking=True)
                self.h_p2[6].copy_(self.p2[6], non_blocking=True)

    def _hod_stage(self, main, hs):
        # The HOD solve needs only n(M,z) and b(M,z), is latency-bound (one CTA per redshift, 24 + 40 bisection
        # iterations, two flag all-reduces when z is sharded) and writes only [nz,nm] arrays: it runs on a side stream
        # next to the two cube kernels and rejoins in front of the mass integrals.
        self.ev_mf.record(main)
        L, d, ptr, p, nz, nm = capi.lib, self.d, capi.ptr, self.p, self.nz, self.nm
        with torch.cuda.stream(hs):
            hs.wait_event(self.ev_mf)
            sth = capi.stream()
            for it0, it1 in ((0, capi.HMV_BISECT_ROUND1), (capi.HMV_BISECT_ROUND1, capi.HMV_BISECT_MAXIT)):
                capi.check(L.hmv_hod_bisect(nz, nm, ptr(d["zs"]), ptr(d["ms"]), ptr(d["nzm"]), ptr(d["ngal_target"]),
                                            self.hodp, float(p['hod_bisection_search_min_log10mthresh']),
                                            float(p['hod_bisection_search_max_log10mthresh']),
                                            float(p['hod_bisection_search_rtol']), it0, it1, ptr(d["bis_ws"]),
                                            C.c_void_p(self.mask.data_ptr()), sth), "hmv_hod_bisect")
                if self.zcomm is not None:
                    self.zcomm.all_reduce_and(self.mask)
            capi.check(L.hmv_hod_pick(nz, ptr(d["bis_ws"]), C.c_void_p(self.mask.data_ptr()),
                                      float(p['hod_A_log10mthresh']), ptr(d["l10"]), ptr(self.iters), sth), "hmv_hod_pick")
            capi.check(L.hmv_hod(nz, nm, ptr(d["zs"]), ptr(d["ms"]), ptr(d["l10"]), self.hodp, 0, ptr(d["nzm"]), ptr(d["bh"]),
                                 ptr(d["Nc"]), ptr(d["Ns"]), ptr(d["NsNsm1"]), ptr(d["NcNs"]), ptr(d["ngal"]), ptr(d["bg"]),
                                 sth), "hmv_hod")
            self.ev_hod.record(hs)

    def _limber(self, st):
        """P = P1h + P2h of mm, gm (and yy) summed and packed z-major by one kernel, all-gathered over z when sharded
        (ONE collective), then C_kk, C_kg (and C_yy) (cosmology.py:536-597)."""
        L, d, ptr = capi.lib, self.d, capi.ptr
        nk, nq = self.nk, self.ncl
        rows = (0, 4, 6)[:nq]                                # mm, gm, yy in self.p1 / self.p2
        pg = self.zcomm.peer_gather(nq * nk) if hasattr(self.zcomm, "peer_gather") else None
        if pg is not None:
            # fused pack + all-gather: the summing kernel stores this slab's rows into every rank's table over NVLink
            full = pg.gather([self.p1[r] for r in rows], [self.p2[r] for r in rows])
            self._peer = pg
            nl0 = 2
        else:
            if self._Ppack is None:
                self._Ppack = torch.empty((self.nz, nq, nk), dtype=torch.float64, device=self.device)
                self._pa = (C.c_void_p * nq)(*[self.p1[r].data_ptr() for r in rows])
                self._pb = (C.c_void_p * nq)(*[self.p2[r].data_ptr() for r in rows])
            capi.check(L.hmv_pack_sum(self.nz, nk, nq, self._pa, self._pb, ptr(self._Ppack), st), "hmv_pack_sum")
            full = self._Ppack
            nl0 = 1
            if self.zcomm is not None:
                # rank order is z order, so the gathered buffer is [nz_total][nq][nk]: each spectrum is a table with
                # row stride nq*nk (hmv_limber's ldp)
                if self._Pfull is None:
                    self._Pfull = torch.empty((self.zs_all.numel(), nq, nk), dtype=torch.float64, device=self.device)
                self.zcomm.all_gather_rows(self._Ppack.view(self.nz, nq * nk), self._Pfull.view(-1, nq * nk))
                full = self._Pfull
        base, ldp, nzt = full.data_ptr(), nq * nk, full.shape[0]
        # C_kk, C_kg (and C_yy) in one launch: each projection is latency-bound, so three cost the time of one
        dp = lambda t: t.data_ptr()
        jobs = (capi.LimberJob * nq)()
        specs = [(nzt, self.zs_all, d["pref_kk"], d["chis"]), (1, d["gz"], d["pref_kg"], d["chig"]),
                 (nzt, self.zs_all, d["pref_yy"], d["chis"])][:nq]
        for q, (ngz, gzs, pref, chis) in enumerate(specs):
            jobs[q].P_d, jobs[q].P2_d, jobs[q].ngz = base + 8 * q * nk, None, ngz
            jobs[q].gzs_d, jobs[q].pref_d, jobs[q].chis_d, jobs[q].cl_d = dp(gzs), dp(pref), dp(chis), dp(self.cl[q])
        capi.check(L.hmv_limber_multi(nq, jobs, self.nl, ptr(d["ells"]), nzt, nk, ldp, ptr(self.zs_all), ptr(d["ks"]), st),
                   "hmv_limber_multi")
        return nl0 + 1


    def spectra(self):
        """Download and return ({tag: P1h}, {tag: P2h}, C_kk, C_kg) as numpy (synchronises); with the tSZ leg the
        dicts also hold 'yy' and `self.last_cyy` is C_yy."""
        self.download()
        torch.cuda.current_stream().synchronize()
        self._check_converged()
        p1, p2 = self.h_p1.numpy().copy(), self.h_p2.numpy().copy()
        tags = TAGS + (("yy",) if self.tsz else ())
        out1 = {t: p1[i] for i, t in enumerate(tags)}
        out2 = {t: p2[i] for i, t in enumerate(tags)}
        if self.has_limber:
            cl = self.h_cl.numpy().copy()
            self.last_cyy = cl[2] if self.tsz else None
            return out1, out2, cl[0], cl[1]
        return out1, out2, None, None
