"""HaloModel: drop-in for `hmvec.hmvec.HaloModel` (reference hmvec/hmvec.py:75-572) on one B200.

Same constructor and method signatures, same attributes (`zs, ks, ms, p, params, h, omm0, Pzk, sigma2, nzm, bh,
uk_profiles, pk_profiles, hods`), same numpy float64 return types -- but nothing on the path is computed by numpy.
The host side prepares O(nz)+O(nk) inputs (background scalars, linear P(k), Simpson weights), uploads them once and
every [nz,nm] / [nz,nm,nk] quantity is produced by the sm_100a kernels behind the C ABI (include/hmvec_b200.h):

    init_mass_function   -> hmv_sigma2, hmv_mass_function, hmv_halo_geometry
    add_nfw_profile      -> hmv_uk_nfw                      (numeric=True -> hmv_profile_transform)
    add_battaglia_*      -> hmv_mdelta, hmv_gnfw_params, hmv_profile_transform
    add_hod              -> hmv_hod_bisect/hmv_hod_pick (ngal given), hmv_hod
    get_power_1halo/2halo/get_power/get_power_six -> hmv_power / hmv_power_six

Data layout in HBM: cubes are [nz][nm][ldk] float64, k fastest, ldk = nk rounded up to 16 doubles.  The cubes stay
resident on the device; `uk_profiles[name]` / `pk_profiles[name]` download a numpy copy on access (at the LARGE grid
one cube is 32 GB, which is why they are not mirrored eagerly).  There is no CPU fallback.
"""
from collections.abc import MutableMapping
import ctypes as C
import weakref

import numpy as np
import torch
from scipy import constants

from . import _capi as capi
from . import utils  # noqa: F401  (reference exports `utils` through `from .hmvec import *`)
from .cosmology import Cosmology, limber_integral, Wkr, a2z, _trapz  # noqa: F401
from .params import default_params, battaglia_defaults

_KIND_MATTER, _KIND_HOD, _KIND_PRESSURE = 0, 1, 2


from .hostfuncs import *  # noqa: F401,F403,E402  (module-level helpers of hmvec.py:627-957)
from .hostfuncs import R_from_M, duffy_concentration, Fcon  # noqa: F401,E402
from . import tinker  # noqa: F401,E402  (reference: `from . import tinker,utils`)
from .fft import generic_profile_fft  # noqa: F401,E402  (hmvec.py:13)


def pressure_constants(omb, omm):
    """Constant factors of the Battaglia pressure profile and of its Compton-y normalisation (hmvec.py:313-316,
    918-927): amp_const = eFrac (omb/omm) 200 G [x m200c rho_c/(2 r200c) P0 on the device],
    pref = 4 pi sigma_T/(m_e c^2) [x r200c^3 (1+z)^2/H on the device], m_e in solar masses."""
    XH = .76
    eFrac = 2.0 * (XH + 1.0) / (5.0 * XH + 3.0)
    G_newt = constants.G / (default_params['parsec'] * 1e6) ** 3 * default_params['mSun']
    sigmaT = constants.physical_constants['Thomson cross section'][0]
    mElect = constants.physical_constants['electron mass'][0] / default_params['mSun']
    return eFrac * (omb / omm) * 200 * G_newt, 4 * np.pi * (sigmaT / (mElect * constants.c ** 2))


class TableProfile(object):
    """A profile kept as the transform's bin tables (hmv_profile_tables) instead of a [nz,nm,nk] cube: ~1 GB instead of
    32 GB on the LARGE grid.  Consumers that only integrate over M (the auto spectrum: hmv_power_tab) read the tables;
    anything that needs u(k|M,z) itself gets the cube, expanded on first use (hmv_profile_expand) and kept."""

    def __init__(self, owner, tab, rs_d, xmax, nxs):
        self._owner = weakref.proxy(owner)
        self.tab, self.rs_d, self.xmax, self.nxs = tab, rs_d, float(xmax), int(nxs)
        self.cube = None

    def materialize(self):
        if self.cube is None:
            o = self._owner
            out = o._cube()
            ws = o._workspace('transform', capi.lib.hmv_profile_transform_ws_doubles(o._nz, o._nm, self.nxs))
            capi.check(capi.lib.hmv_profile_expand(o._nz, o._nm, o._nk, o._ldk, capi.ptr(o._zs_d), capi.ptr(o._ks_d),
                                                   o._kmax, capi.ptr(self.rs_d), self.xmax, self.nxs, capi.ptr(ws),
                                                   capi.ptr(self.tab), capi.ptr(out), capi.stream()),
                       "hmv_profile_expand")
            self.cube = out
        return self.cube


class DeviceCubes(MutableMapping):
    """name -> u(z,M,k) cube resident in HBM ([nz][nm][ldk] float64).  Reading an item returns a numpy
    [nz,nm,nk] copy (what reference callers index); assigning a numpy/torch [nz,nm,nk] array uploads it."""

    def __init__(self, owner):
        self._owner = weakref.proxy(owner) if owner is not None else None    # no reference cycle: dropping the model frees its cubes at once
        self._t = {}

    def device(self, name):
        t = self._t[name]
        return t.materialize() if isinstance(t, TableProfile) else t

    def tables(self, name):
        """The TableProfile behind `name`, or None when the profile is held as a cube."""
        t = self._t.get(name)
        return t if isinstance(t, TableProfile) else None

    def __getitem__(self, name):
        t = self.device(name)
        o = self._owner
        if o._ldk == o._nk:
            return o._host(t)
        return o._host(t[..., :o._nk].contiguous())

    def __setitem__(self, name, value):
        o = self._owner
        o._invalidate_spectra()
        if isinstance(value, TableProfile):
            self._t[name] = value
            return
        if isinstance(value, torch.Tensor) and value.is_cuda:
            # zero-copy only for exactly the layout the kernels read: float64, contiguous [nz][nm][ldk], this device,
            # 16-byte aligned (cp.async.bulk sources); anything else is converted and copied into a fresh cube
            if (value.dtype == torch.float64 and value.is_contiguous() and tuple(value.shape) == (o._nz, o._nm, o._ldk)
                    and value.device == o.device and value.data_ptr() % 16 == 0):
                self._t[name] = value
                return
            if tuple(value.shape) not in ((o._nz, o._nm, o._nk), (o._nz, o._nm, o._ldk)):
                raise ValueError("profile cube must have shape (nz,nm,nk)=%s" % ((o._nz, o._nm, o._nk),))
            t = o._cube()
            t[..., :o._nk] = value[..., :o._nk].to(device=o.device, dtype=torch.float64)
            self._t[name] = t
            return
        arr = torch.as_tensor(np.asarray(value, dtype=np.float64))
        if tuple(arr.shape) != (o._nz, o._nm, o._nk):
            raise ValueError("profile cube must have shape (nz,nm,nk)=%s" % ((o._nz, o._nm, o._nk),))
        t = o._cube()
        capi.count_h2d(arr.numel() * 8)
        t[..., :o._nk] = arr.to(o.device)
        self._t[name] = t

    def __contains__(self, name):
        # Mapping's default would call __getitem__, i.e. download a whole cube, just to test membership
        return name in self._t

    def __delitem__(self, name):
        self._owner._invalidate_spectra()
        del self._t[name]

    def __iter__(self):
        return iter(self._t)

    def __len__(self):
        return len(self._t)


def _lazy_host(name, dev_attr):
    """Public numpy attribute mirrored from a device tensor: downloaded (through pinned memory) on first read,
    uploaded when assigned.  The reference holds these as plain numpy attributes (hmvec.py:99-131)."""

    def fget(self):
        c = self._hostc
        if name not in c:
            t = getattr(self, dev_attr, None)
            if t is None:
                raise AttributeError(name)
            c[name] = self._host(t)
        return c[name]

    def fset(self, value):
        arr = np.array(value, dtype=np.float64)
        self._hostc[name] = arr
        setattr(self, dev_attr, self._dev(arr))
        self._invalidate_spectra()

    return property(fget, fset)


_side_streams = {}


def _side_stream(device, which):
    """One HOD stream and one download stream per device, shared by every object (creating a stream per HaloModel
    costs a millisecond while kernels are running)."""
    key = (str(device), which)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device)
    return _side_streams[key]


class HodRecord(dict):
    """hods[name] (hmvec.py:452-460): 'Nc','Ns','NsNsm1','NcNs' [nz,nm], 'ngal','bg' [nz], 'log10mthresh' [nz,1] plus
    the profile names.  The arrays live on the device; each one is downloaded the first time it is read."""

    def __init__(self, owner, dev, pending=None, **plain):
        dict.__init__(self, **plain)
        self._owner, self._dev = weakref.proxy(owner), dev
        self._pending = pending                 # (pinned int32 tensor, event): iteration count of the ngal bisection

    def _resolve(self):
        """Iteration count of the all-z bisection, read when first needed (add_hod itself does not wait for the
        device).  0 means the search never met rtol: HmvError, as the reference's convergence loop would never end."""
        if self._pending is not None:
            h, ev = self._pending
            ev.synchronize()
            self._pending = None
            iters = int(h.item())
            dict.__setitem__(self, 'iterations', iters)
            if iters == 0:
                raise capi.HmvError("mthresh<->ngal bisection did not converge within %d iterations"
                                    % capi.HMV_BISECT_MAXIT)
            print("Bisection search converged in ", iters, " iterations.")   # utils.py:41
        return dict.__getitem__(self, 'iterations')

    def __missing__(self, key):
        if key == 'iterations' and self._pending is not None:
            return self._resolve()
        if key in self._dev:
            v = self._owner._host(self._dev[key])
            if self._pending is not None:
                self._resolve()                  # the download has waited for the solve: check it converged
            if key == 'log10mthresh':
                v = v[:, None]
            dict.__setitem__(self, key, v)
            return v
        raise KeyError(key)

    def _all(self):
        for k in self._dev:
            self[k]
        if self._pending is not None:
            self._resolve()
        return self

    def get(self, key, default=None):
        return self[key] if key in self else default

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in self._dev or (key == 'iterations' and self._pending is not None)

    def keys(self):
        return dict.keys(self._all())

    def items(self):
        return dict.items(self._all())

    def values(self):
        return dict.values(self._all())

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return len(self.keys())


class HaloModel(Cosmology):
    Pzk = _lazy_host('Pzk', '_Pzk_d')
    sPzk = _lazy_host('sPzk', '_sPzk_d')
    sigma2 = _lazy_host('sigma2', '_sigma2_d')
    nzm = _lazy_host('nzm', '_nzm_d')
    bh = _lazy_host('bh', '_bh_d')

    def __init__(self, zs, ks, ms=None, params={}, mass_function="sheth-torman", halofit=None, mdef='vir',
                 nfw_numeric=False, skip_nfw=False, accuracy='medium', engine='camb', device=None, Pzk=None,
                 sPzk=None, zcomm=None):
        """Reference signature (hmvec.py:76-77) plus keyword-only extensions:
        device -- CUDA device (default: current); Pzk [nz,nk], sPzk [nz,sigma2_numks] -- host-supplied linear power
        on `ks` and on the sigma^2 grid (the CAMB products; skips the internal producer); zcomm -- a
        `zshard.ZComm` when `zs` is this rank's slab of a redshift axis sharded over several GPUs."""
        self._hostc = {}
        self._six = {}
        self._six_host = {}
        self._pairs = {}
        self._ws = {}
        self.zs = np.asarray(zs, dtype=np.float64).reshape(-1)
        self.ks = ks
        self._ks64 = np.asarray(ks, dtype=np.float64).reshape(-1)
        self._kmax = float(np.max(self._ks64))
        self._Pzk_in, self._sPzk_in = Pzk, sPzk
        self._zcomm = zcomm
        self._nz, self._nk = self.zs.size, self._ks64.size
        self._ldk = ((self._nk + 15) // 16) * 16
        self._defer_pzk = True                  # the linear power is formed after the NFW cube kernel has been queued
        Cosmology.__init__(self, params, halofit, accuracy=accuracy, engine=engine, device=device)
        if mdef not in ('vir', 'mean'):
            raise ValueError("mdef must be 'vir' or 'mean'")
        self.mdef = mdef
        self.mode = mass_function
        self.hods = {}
        self._hod_d = {}
        self._zs_d = self._dev(self.zs)
        self._ks_d = self._dev(self._ks64)
        self._rho_m0 = float(np.atleast_1d(self.rho_matter_z(0.))[0])
        self._hod_stream = None
        self._ev_mf = self._ev_hod = None
        self.uk_profiles = DeviceCubes(self)
        self.pk_profiles = DeviceCubes(self)
        # Launch order: per-halo geometry and the NFW cube first (they need only zs, ms and the background), so that
        # the host-side preparation of the linear power and of the sigma^2 integral (EH98 transfer function, growth,
        # Simpson weights: a few ms of numpy) runs while the GPU is already busy.  The reference's order
        # (hmvec.py:98-131: P(z,k), mass function, NFW) yields the same state.
        if ms is not None:
            self.ms = np.asarray(ms, dtype=np.float64).reshape(-1)
            self._init_geometry(self.ms)
            if not skip_nfw:
                self.add_nfw_profile("nfw", numeric=nfw_numeric)
        self._defer_pzk = False
        self._make_pzk(halofit)
        if ms is not None:
            self._init_sigma2_massfn()
        elif not skip_nfw:
            self.add_nfw_profile("nfw", numeric=nfw_numeric)      # raises as the reference does without a mass grid

    # ------------------------------------------------------------------ host-side inputs
    def _plin_device(self, ks, zs):
        """accuracy='low': EH98 P(z,k) = D(z)^2 v(k) (cosmology.py:391-402) formed on the device from its two factor
        vectors -- O(nz)+O(nk) host work, no [nz,nk] array on the host or on PCIe."""
        ks_d = self._ks_d if ks is self._ks64 else self._dev(np.asarray(ks, dtype=np.float64).reshape(-1))
        d2, v_d = self.P_lin_approx_factors_device(ks_d, zs)       # EH98 itself runs on the device too
        out = self._empty(d2.size, v_d.numel())
        d2_d = self._dev(d2)                             # named: a temporary's block would be recycled at once
        capi.check(capi.lib.hmv_outer(d2.size, v_d.numel(), capi.ptr(d2_d), capi.ptr(v_d), capi.ptr(out), capi.stream()),
                   "hmv_outer")
        return out

    def _init_cosmology(self, params, halofit):
        Cosmology._init_cosmology(self, params, halofit)
        if not self._defer_pzk:
            self._make_pzk(halofit)

    def _make_pzk(self, halofit):
        if self._Pzk_in is not None:
            P = np.array(self._Pzk_in, dtype=np.float64)
            if P.shape != (self.zs.size, self._ks64.size):
                raise ValueError("Pzk must have shape (nz,nk)")
            self.Pzk = P
        elif self.accuracy == 'low':
            self._Pzk_d = self._plin_device(self._ks64, self.zs)             # hmvec.py:98-99
        else:
            self.Pzk = self._get_matter_power(self.zs, self._ks64, nonlinear=False)
        if halofit is not None and self._Pzk_in is None:
            self.nPzk = self._get_matter_power(self.zs, self._ks64, nonlinear=True)

    def _sigma2_inputs(self, zs, kmin=None, kmax=None, numks=None):
        from .cosmology import simpson_weights
        ks_sigma2 = np.geomspace(self.p['sigma2_kmin'] if kmin is None else kmin,
                                 self.p['sigma2_kmax'] if kmax is None else kmax,
                                 int(self.p['sigma2_numks'] if numks is None else numks))
        same_z = np.size(zs) == self.zs.size and np.array_equal(np.asarray(zs, dtype=np.float64).reshape(-1), self.zs)
        if self._sPzk_in is not None and same_z:
            sP = np.array(self._sPzk_in, dtype=np.float64)
            if sP.shape != (np.size(zs), ks_sigma2.size):
                raise ValueError("sPzk must have shape (nz, sigma2_numks)")
            self.sPzk = sP
        elif self.accuracy == 'low' and same_z:
            self._hostc.pop('sPzk', None)
            self._sPzk_d = self._plin_device(ks_sigma2, self.zs)              # cosmology.py:259-260
        else:
            return Cosmology._sigma2_inputs(self, zs, kmin, kmax, numks)
        return ks_sigma2, simpson_weights(ks_sigma2) * ks_sigma2 ** 2. / 2. / np.pi ** 2.

    def deltav(self, z):
        """Bryan & Norman virial overdensity (hmvec.py:105-109)."""
        x = self.omz(z) - 1.
        return 18. * np.pi ** 2. + 82. * x - 39. * x ** 2.

    def rvir(self, m, z):
        if self.mdef == 'vir':
            return R_from_M(m, self.rho_critical_z(z), delta=self.deltav(z))
        return R_from_M(m, self.rho_matter_z(z), delta=200.)

    def R_of_m(self, ms):
        return R_from_M(ms, self.rho_matter_z(0), delta=1.)

    def _delta_rhos1(self):
        rhocritz = self.rho_critical_z(self.zs)
        if self.mdef == 'vir':
            return rhocritz * self.deltav(self.zs)
        return self.rho_matter_z(self.zs) * 200.

    # ------------------------------------------------------------------ device plumbing
    def _cube(self):
        t = torch.empty((self._nz, self._nm, self._ldk), dtype=torch.float64, device=self.device)
        if self._ldk > self._nk:
            t[..., self._nk:] = 0.0          # pad columns are read (and ignored) by the 16-byte loads of hmv_power
        return t

    def _workspace(self, kind, ndoubles):
        """Per-object scratch buffers, allocated once per kind and reused by every later call (all calls of one object
        are ordered on one stream)."""
        t = self._ws.get(kind)
        if t is None or t.numel() < ndoubles:
            t = self._ws[kind] = self._empty(int(ndoubles))
        return t

    @staticmethod
    def _host(t):
        """Device tensor -> numpy through pinned memory (a pageable `.cpu()` runs at ~2 GB/s, pinned at PCIe speed).
        The pinned block comes from torch's caching host allocator and is owned by the returned array."""
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t, non_blocking=True)
        capi.count_d2h(h.numel() * h.element_size())
        torch.cuda.current_stream().synchronize()
        return h.numpy()

    def _invalidate_spectra(self):
        self._six = {}
        self._six_host = {}
        self._pairs = {}

    def _duffy(self):
        tag = 'mean' if self.mdef == 'mean' else 'vir'
        return self.p['duffy_A_' + tag], self.p['duffy_alpha_' + tag], self.p['duffy_beta_' + tag]

    # ------------------------------------------------------------------ mass function (K3, K3b, geometry)
    def get_sigma2(self):
        return self._host(self._sigma2_d)

    def init_mass_function(self, ms):
        """sigma^2 -> n(M,z), b(M,z) and the per-halo geometry, all on the device (hmvec.py:127-185).  The numpy
        attributes `sigma2`, `nzm`, `bh` are downloaded when first read."""
        self._init_geometry(ms)
        self._init_sigma2_massfn()

    def _init_geometry(self, ms):
        """c(M,z) and r_vir(M,z) (hmvec.py:148-165): everything the profile kernels need of the mass grid."""
        if self.mode not in ("sheth-torman", "tinker"):
            raise NotImplementedError("mass_function=%r" % (self.mode,))
        self.ms = np.asarray(ms, dtype=np.float64).reshape(-1)
        self._nm = self.ms.size
        self._ms_d = self._dev(self.ms)
        self._invalidate_spectra()
        A, alpha, beta = self._duffy()
        self._drho1_d = self._dev(self._delta_rhos1())
        self._cs_d, self._rvir_d = self._empty(self._nz, self._nm), self._empty(self._nz, self._nm)
        capi.check(capi.lib.hmv_halo_geometry(self._nz, self._nm, capi.ptr(self._zs_d), capi.ptr(self._ms_d),
                                              capi.ptr(self._drho1_d), A, alpha, beta, self.h, capi.ptr(self._cs_d),
                                              capi.ptr(self._rvir_d), capi.stream()), "hmv_halo_geometry")

    def _init_sigma2_massfn(self):
        for k in ('sigma2', 'nzm', 'bh'):
            self._hostc.pop(k, None)
        ks_sig, kw = self._sigma2_inputs(self.zs)
        R = np.asarray(self.R_of_m(self.ms), dtype=np.float64).reshape(-1)
        self._sigma2_d = self._sigma2_device(self._dev(R), self._sPzk_d, self._dev(ks_sig), self._dev(kw))
        self._nzm_d, self._bh_d = self._empty(self._nz, self._nm), self._empty(self._nz, self._nm)
        p = self.p
        if self.mode == "tinker":
            from . import tinker
            tk = self._dev(tinker.redshift_parameters(self.zs))                # [nz,5], hmvec.py:142-145 -> tinker.py
            capi.check(capi.lib.hmv_mass_function_tinker(self._nz, self._nm, capi.ptr(self._sigma2_d),
                                                         capi.ptr(self._ms_d), self._rho_m0, p['st_deltac'],
                                                         capi.ptr(tk), capi.ptr(self._nzm_d), capi.ptr(self._bh_d),
                                                         capi.stream()), "hmv_mass_function_tinker")
        else:
            capi.check(capi.lib.hmv_mass_function(self._nz, self._nm, capi.ptr(self._sigma2_d), capi.ptr(self._ms_d),
                                                  self._rho_m0, p['st_A'], p['st_a'], p['st_p'], p['st_deltac'],
                                                  capi.ptr(self._nzm_d), capi.ptr(self._bh_d), capi.stream()),
                       "hmv_mass_function")
        self._ev_mf = torch.cuda.Event()
        self._ev_mf.record()                                                  # the HOD side stream starts from here

    def get_nzm(self):
        return self._host(self._nzm_d)

    def get_bh(self):
        return self._host(self._bh_d)

    def concentration(self, mode='duffy'):
        if mode != 'duffy':
            raise NotImplementedError
        return self._host(self._cs_d)

    # ------------------------------------------------------------------ profiles (K0, K1, K2)
    def _m200c_device(self):
        rhoc = np.asarray(self.rho_critical_z(self.zs), dtype=np.float64)
        drho2_d = self._dev(200. * rhoc)
        m200_d = self._empty(self._nz, self._nm)
        capi.check(capi.lib.hmv_mdelta(self._nz, self._nm, capi.ptr(self._ms_d), capi.ptr(self._cs_d),
                                       capi.ptr(self._drho1_d), capi.ptr(drho2_d), capi.ptr(m200_d), capi.stream()),
                   "hmv_mdelta")
        return m200_d, self._dev(rhoc)

    def _transform(self, rs_d, cmax_d, xc_d, alpha_d, expo_d, amp_d, oscale_d, gamma, xmax, nxs, mass_norm,
                   tables=False):
        ws = self._workspace('transform', capi.lib.hmv_profile_transform_ws_doubles(self._nz, self._nm, int(nxs)))
        if tables and int(nxs) // 2 <= 4096 and self._nm * 28 + 16 <= 200 * 1024:
            # keep the bin tables only (see TableProfile); limits are those of hmv_power_tab
            tab = self._empty(int(capi.lib.hmv_profile_table_doubles(self._nz, self._nm, int(nxs))))
            capi.check(capi.lib.hmv_profile_tables(
                self._nz, self._nm, self._nk, capi.ptr(self._zs_d), capi.ptr(self._ks_d), self._kmax, capi.ptr(rs_d),
                capi.ptr(cmax_d), capi.ptr(xc_d), capi.ptr(alpha_d), capi.ptr(expo_d), capi.ptr(amp_d),
                capi.ptr(oscale_d), float(gamma), float(xmax), int(nxs), int(bool(mass_norm)), capi.ptr(ws),
                capi.ptr(tab), capi.stream()), "hmv_profile_tables")
            return TableProfile(self, tab, rs_d, xmax, nxs)
        out = self._cube()
        capi.check(capi.lib.hmv_profile_transform(
            self._nz, self._nm, self._nk, self._ldk, capi.ptr(self._zs_d), capi.ptr(self._ks_d),
            self._kmax, capi.ptr(rs_d), capi.ptr(cmax_d), capi.ptr(xc_d), capi.ptr(alpha_d),
            capi.ptr(expo_d), capi.ptr(amp_d), capi.ptr(oscale_d), float(gamma), float(xmax), int(nxs),
            int(bool(mass_norm)), capi.ptr(ws), capi.ptr(out), capi.stream()), "hmv_profile_transform")
        return out

    def _gnfw(self, kind, fit9, gamma, pres_alpha, amp_const, pref, xmax, nxs, tables=False):
        m200_d, rhoc_d = self._m200c_device()
        hofz_d = self._dev(self.h_of_z(self.zs))
        outs = [self._empty(self._nz, self._nm) for _ in range(7)]
        capi.check(capi.lib.hmv_gnfw_params(kind, self._nz, self._nm, capi.ptr(self._zs_d), capi.ptr(m200_d),
                                            capi.ptr(self._rvir_d), capi.ptr(rhoc_d), capi.ptr(hofz_d),
                                            capi.darr(fit9), float(gamma), float(pres_alpha), float(amp_const),
                                            float(pref), *[capi.ptr(o) for o in outs], capi.stream()),
                   "hmv_gnfw_params")
        rs, cmax, xc, alpha, expo, amp, oscale = outs
        return self._transform(rs, cmax, xc, alpha, expo, amp, oscale, gamma, xmax, nxs, mass_norm=(kind == 0),
                               tables=tables)

    def add_battaglia_profile(self, name, family=None, param_override=None, nxs=None, xmax=None,
                              ignore_existing=False):
        """Battaglia-2016 GNFW electron density u(k|M,z) (hmvec.py:188-250 + fft.py:56-115), one fused kernel."""
        if not ignore_existing:
            assert name not in self.uk_profiles.keys(), "Profile name already exists."
        assert name != 'nfw', "Name nfw is reserved."
        if nxs is None:
            nxs = self.p['electron_density_profile_integral_numxs']
        if xmax is None:
            xmax = self.p['electron_density_profile_integral_xmax']
        if family is None:
            family = self.p['battaglia_gas_family']
        pparams = {'battaglia_gas_gamma': self.p['battaglia_gas_gamma']}
        pparams.update(battaglia_defaults[family])
        if param_override is not None:
            print(param_override)                                           # hmvec.py:205
            for key in param_override.keys():                               # unknown keys are ignored (:204-213)
                if key == 'battaglia_gas_gamma' or key in battaglia_defaults[family]:
                    pparams[key] = param_override[key]
        fit9 = [pparams[q + s] for q in ('rho0', 'alpha', 'beta') for s in ('_A0', '_alpham', '_alphaz')]
        self.uk_profiles[name] = self._gnfw(0, fit9, pparams['battaglia_gas_gamma'], 1.0, 1.0, 1.0, xmax, nxs)

    def add_battaglia_pres_profile(self, name, family=None, param_override=None, nxs=None, xmax=None,
                                   ignore_existing=False):
        """Battaglia-2012 GNFW electron pressure -> Compton-y profile (hmvec.py:252-316, 906-927)."""
        if not ignore_existing:
            assert name not in self.pk_profiles.keys(), "Profile name already exists."
        assert name != 'nfw', "Name nfw is reserved."
        if nxs is None:
            nxs = self.p['electron_pressure_profile_integral_numxs']
        if xmax is None:
            xmax = self.p['electron_pressure_profile_integral_xmax']
        if family is None:
            family = self.p['battaglia_pres_family']
        pparams = {'battaglia_pres_gamma': self.p['battaglia_pres_gamma'],
                   'battaglia_pres_alpha': self.p['battaglia_pres_alpha']}
        pparams.update(battaglia_defaults[family])
        if param_override is not None:
            for key in param_override.keys():
                if key in ('battaglia_pres_gamma', 'battaglia_pres_alpha') or key in battaglia_defaults[family]:
                    pparams[key] = param_override[key]
        fit9 = [pparams[q + s] for q in ('P0', 'xc', 'beta') for s in ('_A0', '_alpham', '_alphaz')]
        amp_const, pref = pressure_constants(self.p['ombh2'] / self.h ** 2., self.omm0)
        # kept as bin tables: the tSZ auto spectrum -- what a Compton-y profile is for (hmvec.py:512-514, C_yy) -- is
        # reduced straight from them; pk_profiles[name] and cross spectra expand the cube on first use
        self.pk_profiles[name] = self._gnfw(1, fit9, pparams['battaglia_pres_gamma'],
                                            pparams['battaglia_pres_alpha'], amp_const, pref, xmax, nxs, tables=True)

    def add_nfw_profile(self, name, numeric=False, nxs=None, xmax=None, ignore_existing=False):
        """Truncated-NFW u(k|M,z): analytic Si/Ci kernel, or the numerical transform (hmvec.py:318-355)."""
        if not ignore_existing:
            assert name not in self.uk_profiles.keys(), "Profile name already exists."
        if nxs is None:
            nxs = self.p['nfw_integral_numxs']
        if xmax is None:
            xmax = self.p['nfw_integral_xmax']
        if numeric:
            # rho_nfw_x = 1/x/(1+x)^2 is the GNFW form with gamma=-1, alpha=1, exponent 2; cmax = c, rs = rvir/c
            one = torch.ones((self._nz, self._nm), dtype=torch.float64, device=self.device)
            rs_d = self._rvir_d / self._cs_d
            out = self._transform(rs_d, self._cs_d, one, one, 2.0 * one, one, one, -1.0, xmax, nxs, mass_norm=True)
        else:
            out = self._cube()
            ws = self._workspace('nfw', capi.lib.hmv_uk_nfw_ws_doubles(self._nz, self._nm, self._nk))
            capi.check(capi.lib.hmv_uk_nfw(self._nz, self._nm, self._nk, self._ldk, capi.ptr(self._zs_d),
                                           capi.ptr(self._ks_d), self._kmax, capi.ptr(self._cs_d),
                                           capi.ptr(self._rvir_d), capi.ptr(ws), capi.ptr(out), capi.stream()),
                       "hmv_uk_nfw")
        self.uk_profiles[name] = out
        return self.ks, LazyCube(self.uk_profiles, name)

    # ------------------------------------------------------------------ HOD (K4, K4b)
    def add_hod(self, name, mthresh=None, ngal=None, corr="max", satellite_profile_name='nfw',
                central_profile_name=None, ignore_existing=False, param_override=None):
        """Leauthaud-SHMR HOD from a stellar-mass threshold or a number density (hmvec.py:357-460)."""
        if not ignore_existing:
            assert name not in self.uk_profiles.keys(), "HOD name already used by profile."
        assert satellite_profile_name in self.uk_profiles.keys(), "No matter profile by that name exists."
        if central_profile_name is not None:
            assert central_profile_name in self.uk_profiles.keys(), "No matter profile by that name exists."
        if not ignore_existing:
            assert name not in self.hods.keys(), "HOD with that name already exists."
        if corr not in ("max", "min"):
            raise ValueError("corr must be 'max' or 'min'")
        hod_params = ['hod_sig_log_mstellar', 'hod_bisection_search_min_log10mthresh',
                      'hod_bisection_search_max_log10mthresh', 'hod_bisection_search_rtol',
                      'hod_bisection_search_warn_iter', 'hod_alphasat', 'hod_Bsat', 'hod_betasat', 'hod_Bcut',
                      'hod_betacut', 'hod_A_log10mthresh']
        pp = {k: self.p[k] for k in hod_params}
        if param_override is not None:
            for key in param_override.keys():
                if key in hod_params:
                    pp[key] = param_override[key]
                else:
                    raise ValueError("%r is not an HOD parameter" % (key,))
        hodp = capi.darr([pp['hod_sig_log_mstellar'], pp['hod_alphasat'], pp['hod_Bsat'], pp['hod_betasat'],
                          pp['hod_Bcut'], pp['hod_betacut'], 0.0, 0.0])
        nz, nm = self._nz, self._nm
        self._invalidate_spectra()
        # The HOD solve needs only n(M,z) and b(M,z) and is latency-bound: it runs on a side stream that forks after
        # the mass function, next to the profile-cube kernels of the main stream, and rejoins in front of the spectra.
        if self._hod_stream is None:
            self._hod_stream = _side_stream(self.device, 'hod')
        main = torch.cuda.current_stream()
        hs = self._hod_stream
        pending = None
        with torch.cuda.stream(hs):
            hs.wait_event(self._ev_mf)
            if ngal is not None:
                ngal = np.asarray(ngal, dtype=np.float64)
                if ngal.size != nz:
                    raise ValueError("ngal has to be a vector of size self.zs")
                assert mthresh is None
                l10_d, pending = self._solve_mthresh(self._dev(ngal.reshape(-1)), hodp, pp)
            else:
                mthresh = np.asarray(mthresh, dtype=np.float64)
                if mthresh.size != nz:
                    raise ValueError("mthresh has to be a vector of size self.zs")
                l10_d = self._dev(np.log10(mthresh.reshape(-1)))
            d = {k: self._empty(nz, nm) for k in ('Nc', 'Ns', 'NsNsm1', 'NcNs')}
            d['ngal'], d['bg'] = self._empty(nz), self._empty(nz)
            capi.check(capi.lib.hmv_hod(nz, nm, capi.ptr(self._zs_d), capi.ptr(self._ms_d), capi.ptr(l10_d), hodp,
                                        0 if corr == "max" else 1, capi.ptr(self._nzm_d), capi.ptr(self._bh_d),
                                        capi.ptr(d['Nc']), capi.ptr(d['Ns']), capi.ptr(d['NsNsm1']), capi.ptr(d['NcNs']),
                                        capi.ptr(d['ngal']), capi.ptr(d['bg']), capi.stream()), "hmv_hod")
            d['log10mthresh'] = l10_d
            for t in d.values():
                t.record_stream(main)
            ev = torch.cuda.Event()
            ev.record(hs)
        main.wait_event(ev)                    # later work on the main stream (spectra, downloads) sees the HOD arrays
        self._hod_d[name] = d
        rec = HodRecord(self, d, pending, satellite_profile=satellite_profile_name,
                        central_profile=central_profile_name)
        if pending is None:
            rec['iterations'] = 0
        self.hods[name] = rec

    def _solve_mthresh(self, target_d, hodp, pp):
        """All-z bisection (utils.py:9-42): every redshift bisects on the device and records, per iteration,
        its midpoint and a pass bit; the answer is the midpoint of the first iteration at which EVERY redshift
        passes -- across all ranks when the z axis is sharded (one 8-byte all-reduce)."""
        nz, nm = self._nz, self._nm
        ws = self._empty(nz * (capi.HMV_BISECT_MAXIT + 4))
        mask_d = torch.empty(1, dtype=torch.int64, device=self.device)
        # two rounds: the usual solve converges within the first (rtol 1e-4 on [7,14] takes ~19 iterations), and the
        # continuation returns immediately on the device when it did -- no host synchronisation in between
        for it0, it1 in ((0, capi.HMV_BISECT_ROUND1), (capi.HMV_BISECT_ROUND1, capi.HMV_BISECT_MAXIT)):
            capi.check(capi.lib.hmv_hod_bisect(nz, nm, capi.ptr(self._zs_d), capi.ptr(self._ms_d),
                                               capi.ptr(self._nzm_d), capi.ptr(target_d), hodp,
                                               float(pp['hod_bisection_search_min_log10mthresh']),
                                               float(pp['hod_bisection_search_max_log10mthresh']),
                                               float(pp['hod_bisection_search_rtol']), it0, it1, capi.ptr(ws),
                                               C.c_void_p(mask_d.data_ptr()), capi.stream()), "hmv_hod_bisect")
            if self._zcomm is not None:
                self._zcomm.all_reduce_and(mask_d)
        l10_d = self._empty(nz)
        iters_d = torch.zeros(1, dtype=torch.int32, device=self.device)
        capi.check(capi.lib.hmv_hod_pick(nz, capi.ptr(ws), C.c_void_p(mask_d.data_ptr()),
                                         float(pp['hod_A_log10mthresh']), capi.ptr(l10_d), capi.ptr(iters_d),
                                         capi.stream()), "hmv_hod_pick")
        # the count goes to pinned memory behind the solve; nobody waits for it here: it is read (and a search that
        # never converged raises) when the HOD is first consumed -- get_power & co., hods[name]['iterations']
        h = torch.empty(1, dtype=torch.int32, pin_memory=True)
        h.copy_(iters_d, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return l10_d, (h, ev)

    def get_ngal(self, Nc, Ns):
        return _trapz(self.nzm * (Nc + Ns), self.ms, axis=-1)

    def get_bg(self, Nc, Ns, ngal):
        return _trapz(self.nzm * (Nc + Ns) * self.bh, self.ms, axis=-1) / ngal

    # ------------------------------------------------------------------ spectra (K5)
    def _kind(self, name, order):
        for k in order:
            if k == 'h' and name in self.hods:
                return _KIND_HOD
            if k == 'm' and name in self.uk_profiles:
                return _KIND_MATTER
            if k == 'p' and name in self.pk_profiles:
                return _KIND_PRESSURE
        raise ValueError("no profile or HOD named %r" % (name,))

    def _tracer(self, name, kind, bias_d=None):
        t = capi.Tracer()
        t.kind = kind
        keep = []
        if kind == _KIND_HOD:
            hod, d = self.hods[name], self._hod_d[name]
            t.us_d = capi.ptr(self.uk_profiles.device(hod['satellite_profile'])).value
            cen = hod['central_profile']
            t.uc_d = capi.ptr(self.uk_profiles.device(cen)).value if cen is not None else None
            t.Nc_d, t.Ns_d = d['Nc'].data_ptr(), d['Ns'].data_ptr()
            t.NcNs_d, t.NsNsm1_d = d['NcNs'].data_ptr(), d['NsNsm1'].data_ptr()
            t.ngal_d = d['ngal'].data_ptr()
        elif kind == _KIND_MATTER:
            t.us_d = capi.ptr(self.uk_profiles.device(name)).value
        else:
            t.us_d = capi.ptr(self.pk_profiles.device(name)).value
        if bias_d is not None:
            t.bias_d = bias_d.data_ptr()
            keep.append(bias_d)
        return t, keep

    def _power(self, name, name2, want1, want2, b1_in=None, b2_in=None, kinds=None, to_host=True, add=False):
        name2 = name if name2 is None else name2
        kA, kB = kinds
        bA = self._dev(np.asarray(b1_in, dtype=np.float64).reshape(-1)) if b1_in is not None else None
        bB = self._dev(np.asarray(b2_in, dtype=np.float64).reshape(-1)) if b2_in is not None else None
        for b in (bA, bB):
            if b is not None and b.numel() != self._nz:
                raise ValueError("b1_in/b2_in must have one value per redshift")
        if bA is None and bB is None:
            six = self._six_lookup(name, name2, kA, kB)
            if six is not None:
                p1, p2, tag = six
                if add and to_host and tag in self._six_host:
                    h, ev = self._six_host.pop(tag)           # handed out once: the caller owns the memory
                    ev.synchronize()
                    self._check_hods()
                    return h
                return self._power_out(p1 if want1 else None, p2 if want2 else None, to_host, add)
            hit = self._pairs.get((name, kA, name2, kB))             # prefetched next to the six-spectra pass
            if hit is not None:
                return self._power_out(hit[0] if want1 else None, hit[1] if want2 else None, to_host, add)
        p1, p2 = self._power_pair(name, kA, bA, name2, kB, bB, want1, want2)
        return self._power_out(p1, p2, to_host, add)

    def _power_pair(self, name, kA, bA, name2, kB, bB, want1=True, want2=True):
        """One generic tracer pair: hmv_power on the resident cubes; returns device [nz,nk] tensors."""
        if name == name2 and kA == kB and bA is None and bB is None and kA in (_KIND_MATTER, _KIND_PRESSURE):
            tp = (self.uk_profiles if kA == _KIND_MATTER else self.pk_profiles).tables(name)
            if tp is not None and tp.cube is None:
                # auto spectrum of a table-backed profile: no cube is built
                ws = self._workspace('power', capi.lib.hmv_power_ws_doubles(self._nz, self._nm))
                p1 = self._empty(self._nz, self._nk) if want1 else None
                p2 = self._empty(self._nz, self._nk) if want2 else None
                capi.check(capi.lib.hmv_power_tab(self._nz, self._nm, self._nk, capi.ptr(self._ms_d), capi.ptr(self._ks_d),
                                                  capi.ptr(self._nzm_d), capi.ptr(self._bh_d), capi.ptr(self._Pzk_d),
                                                  self._rho_m0, float(self.p['kstar_damping']), kA, capi.ptr(tp.tab),
                                                  tp.nxs, capi.ptr(ws), capi.ptr(p1), capi.ptr(p2), capi.stream()),
                           "hmv_power_tab")
                return p1, p2
        A, keepA = self._tracer(name, kA, bA)
        B, keepB = self._tracer(name2, kB, bB)
        ws = self._workspace('power', capi.lib.hmv_power_ws_doubles(self._nz, self._nm))
        p1 = self._empty(self._nz, self._nk) if want1 else None
        p2 = self._empty(self._nz, self._nk) if want2 else None
        capi.check(capi.lib.hmv_power(self._nz, self._nm, self._nk, self._ldk, capi.ptr(self._ms_d),
                                      capi.ptr(self._ks_d), capi.ptr(self._nzm_d), capi.ptr(self._bh_d),
                                      capi.ptr(self._Pzk_d), self._rho_m0, float(self.p['kstar_damping']),
                                      C.byref(A), C.byref(B), capi.ptr(ws), capi.ptr(p1), capi.ptr(p2),
                                      capi.stream()), "hmv_power")
        return p1, p2

    def _check_hods(self):
        """Called after a download has synchronised the stream: every ngal bisection queued before it has finished,
        so its iteration count is read for free here -- and a search that did not converge raises before any
        spectrum built on it is handed out."""
        for rec in self.hods.values():
            if rec._pending is not None:
                rec._resolve()

    def _power_out(self, p1, p2, to_host, add):
        if add:                                  # get_power: P1h + P2h formed on the device, one download
            out = self._empty(self._nz, self._nk)
            capi.check(capi.lib.hmv_sum2(out.numel(), capi.ptr(p1), capi.ptr(p2), capi.ptr(out), capi.stream()),
                       "hmv_sum2")
            if not to_host:
                return out
            res = self._host(out)
            self._check_hods()
            return res
        if not to_host:
            return p1, p2
        res = (self._host(p1) if p1 is not None else None), (self._host(p2) if p2 is not None else None)
        self._check_hods()
        return res

    # The usual workflow asks for the six auto/cross spectra of (matter, electron, galaxies) one after the other
    # (README.rst:75-100); each of them alone streams one or two 32 GB cubes.  The first such request runs ONE pass
    # over the two cubes (hmv_power_six) and keeps the twelve [nz,nk] results on the device; the others are lookups.
    _SIX = ("mm", "ee", "me", "gg", "gm", "ge")

    def _six_lookup(self, name, name2, kA, kB):
        if _KIND_PRESSURE in (kA, kB):
            return None
        hod = [n for n, k in ((name, kA), (name2, kB)) if k == _KIND_HOD]
        mat = [n for n, k in ((name, kA), (name2, kB)) if k == _KIND_MATTER]
        if len(set(hod)) > 1:
            return None
        g = hod[0] if hod else next((n for n in reversed(list(self.hods)) if self.hods[n]['central_profile'] is None), None)
        if g is None or self.hods[g]['central_profile'] is not None:
            return None
        m = self.hods[g]['satellite_profile']
        others = [n for n in mat if n != m]
        if len(set(others)) > 1:
            return None
        e = others[0] if others else next((n for n in reversed(list(self.uk_profiles)) if n != m), None)
        if e is None:
            return None
        tag = "".join("g" if n == g and k == _KIND_HOD else ("m" if n == m else "e") for n, k in ((name, kA), (name2, kB)))
        tag = {"em": "me", "mg": "gm", "eg": "ge"}.get(tag, tag)
        if tag not in self._SIX:
            return None
        key = (m, e, g)
        if key not in self._six:
            self._six = {key: self.get_power_six(m, e, g, to_host=False, stacked=True)}
            # P = P1h + P2h of all six goes to pinned host memory on the download stream, behind the pass but beside
            # whatever the main stream runs next (the tSZ pair below): get_power then finds its array on the host
            self._prefetch_six_totals(*self._six[key])
            # The caller is about to block on a download of one of these spectra; whatever is launched now runs behind
            # that wait for free.  A Compton-y profile next to the six tracers means the tSZ auto spectrum follows
            # (BASELINE configs[4]): queue it now, the request for it then finds it ready.
            self._pairs = {}
            for y in list(self.pk_profiles)[-1:]:
                self._pairs[(y, _KIND_PRESSURE, y, _KIND_PRESSURE)] = self._power_pair(
                    y, _KIND_PRESSURE, None, y, _KIND_PRESSURE, None)
        p1, p2 = self._six[key]
        i = self._SIX.index(tag)
        return p1[i], p2[i], tag

    def _prefetch_six_totals(self, p1, p2):
        tot = self._empty(6, self._nz, self._nk)
        capi.check(capi.lib.hmv_sum2(tot.numel(), capi.ptr(p1), capi.ptr(p2), capi.ptr(tot), capi.stream()), "hmv_sum2")
        ready = torch.cuda.Event()
        ready.record()
        cs = _side_stream(self.device, 'd2h')
        self._six_host = {}
        with torch.cuda.stream(cs):
            cs.wait_event(ready)
            for i, tag in enumerate(self._SIX):
                h = torch.empty((self._nz, self._nk), dtype=torch.float64, pin_memory=True)
                h.copy_(tot[i], non_blocking=True)
                capi.count_d2h(h.numel() * 8)
                ev = torch.cuda.Event()
                ev.record(cs)
                self._six_host[tag] = (h.numpy(), ev)
        tot.record_stream(cs)

    # 1-halo looks names up as HOD first (hmvec.py:510-523); 2-halo as matter profile first (hmvec.py:536-550)
    def _kinds_1h(self, name, name2):
        return self._kind(name, 'hmp'), self._kind(name2, 'hmp')

    def _kinds_2h(self, name, name2):
        return self._kind(name, 'mph'), self._kind(name2, 'mph')

    def get_power_1halo(self, name="nfw", name2=None):
        name2 = name if name2 is None else name2
        return self._power(name, name2, True, False, kinds=self._kinds_1h(name, name2))[0]

    def get_power_2halo(self, name="nfw", name2=None, verbose=False, b1_in=None, b2_in=None):
        name2 = name if name2 is None else name2
        kinds = self._kinds_2h(name, name2)
        if _KIND_PRESSURE in kinds:
            print('Check the consistency relation for tSZ')                 # hmvec.py:544
        return self._power(name, name2, False, True, b1_in, b2_in, kinds=kinds)[1]

    def get_power(self, name, name2=None, verbose=False, b1=None, b2=None):
        """P1h + P2h (hmvec.py:500-502); one pass over the cubes produces both terms, summed on the device."""
        name2 = name if name2 is None else name2
        k1, k2 = self._kinds_1h(name, name2), self._kinds_2h(name, name2)
        if k1 == k2:
            if _KIND_PRESSURE in k1:
                print('Check the consistency relation for tSZ')             # hmvec.py:544
            return self._power(name, name2, True, True, b1, b2, kinds=k1, add=True)
        return self.get_power_1halo(name, name2) + self.get_power_2halo(name, name2, verbose, b1, b2)

    def get_power_device(self, name, name2=None):
        """get_power without the download: P1h + P2h as a CUDA tensor [nz,nk] (an extension of the reference's API for
        device-side consumers -- the gather over the z-shards, C_kk & co., which accept CUDA tensors).  After
        get_power on the standard pairs this is a lookup of the resident spectra."""
        name2 = name if name2 is None else name2
        k1, k2 = self._kinds_1h(name, name2), self._kinds_2h(name, name2)
        if k1 != k2:
            raise ValueError("get_power_device: %r x %r resolve to different tracers for the 1-halo and 2-halo terms"
                             % (name, name2))
        return self._power(name, name2, True, True, kinds=k1, to_host=False, add=True)

    def get_power_six(self, matter="nfw", electron="electron", hod="g", to_host=True, stacked=False):
        """{mm, ee, me, gg, gm, ge} 1h and 2h spectra in ONE pass over the two cubes (hmv_power_six).

        Requires the HOD's satellite profile to be `matter` and its central profile to be None.  Returns
        (P1h, P2h), each a dict tag -> [nz,nk] (numpy, or CUDA tensors when to_host=False; stacked=True returns the
        two [6,nz,nk] device tensors themselves)."""
        h = self.hods[hod]
        if h['satellite_profile'] != matter or h['central_profile'] is not None:
            raise ValueError("get_power_six needs satellite_profile == matter profile and no central profile")
        d = self._hod_d[hod]
        ws = self._workspace('power', capi.lib.hmv_power_ws_doubles(self._nz, self._nm))
        p1, p2 = self._empty(6, self._nz, self._nk), self._empty(6, self._nz, self._nk)
        capi.check(capi.lib.hmv_power_six(self._nz, self._nm, self._nk, self._ldk, capi.ptr(self._ms_d),
                                          capi.ptr(self._ks_d), capi.ptr(self._nzm_d), capi.ptr(self._bh_d),
                                          capi.ptr(self._Pzk_d), self._rho_m0, float(self.p['kstar_damping']),
                                          capi.ptr(self.uk_profiles.device(matter)),
                                          capi.ptr(self.uk_profiles.device(electron)), capi.ptr(d['Nc']),
                                          capi.ptr(d['Ns']), capi.ptr(d['NcNs']), capi.ptr(d['NsNsm1']),
                                          capi.ptr(d['ngal']), capi.ptr(ws), 0, capi.ptr(p1), capi.ptr(p2),
                                          capi.stream()), "hmv_power_six")
        if stacked:
            return p1, p2
        tags = self._SIX
        if not to_host:
            return {t: p1[i] for i, t in enumerate(tags)}, {t: p2[i] for i, t in enumerate(tags)}
        h1, h2 = self._host(p1), self._host(p2)
        self._check_hods()
        return {t: h1[i] for i, t in enumerate(tags)}, {t: h2[i] for i, t in enumerate(tags)}

    # ------------------------------------------------------------------ 1-halo trispectrum and C_l covariance
    def _trispec_legs(self, names, what="1-halo trispectrum",
                      hod_why="needs occupation moments up to fourth order, which the HOD does not define"):
        """Device cubes and kinds of profile tracers: matter profile first, then pressure profile.  A table-backed
        profile is expanded to its cube (DeviceCubes.device)."""
        cubes, kinds = [], []
        for n in names:
            if n in self.uk_profiles:
                cubes.append(self.uk_profiles.device(n))
                kinds.append(_KIND_MATTER)
            elif n in self.pk_profiles:
                cubes.append(self.pk_profiles.device(n))
                kinds.append(_KIND_PRESSURE)
            elif n in self.hods:
                raise ValueError("%r is an HOD: its %s %s" % (n, what, hod_why))
            else:
                raise ValueError("no matter or pressure profile named %r" % (n,))
        if not np.all(np.diff(self._ks64) > 0):
            raise ValueError("the model's ks must be strictly increasing for the %s's interpolation" % what)
        return cubes, kinds

    @staticmethod
    def _positive(x, what):
        x = np.asarray(x, dtype=np.float64).reshape(-1)
        if x.size == 0 or not np.all(np.isfinite(x)) or not np.all(x > 0):
            raise ValueError("%s must be a non-empty list of positive finite values" % what)
        return x

    def _trispec_call(self, fn, names, q1, q2, extra, out_shape):
        cubes, kinds = self._trispec_legs(names)
        nz, nm = self._nz, self._nm
        ws = self._workspace('trispec', getattr(capi.lib, fn + '_ws_doubles')(nz, nm, q1.size, q2.size))
        out = self._empty(*out_shape)
        q1_d, q2_d = self._dev(q1), self._dev(q2)
        u_h = (C.c_void_p * 4)(*[c.data_ptr() for c in cubes])
        capi.check(getattr(capi.lib, fn)(nz, nm, self._nk, self._ldk, capi.ptr(self._ks_d), capi.ptr(self._ms_d),
                                         capi.ptr(self._nzm_d), self._rho_m0, u_h, (C.c_int * 4)(*kinds), q1.size,
                                         capi.ptr(q1_d), q2.size, capi.ptr(q2_d), *[capi.ptr(e) for e in extra],
                                         capi.ptr(ws), capi.ptr(out), capi.stream()), fn)
        return self._host(out)

    def _trispec1h_call(self, fn, names, q1, q2, extra, out_shape):
        """The 1-halo term of four legs resolved as matter profile, then pressure profile, then HOD.  Profile legs only:
        `fn` (_trispec_call).  One or two legs of one HOD: fn + '_tracers' with hmv_power's tracer records."""
        kinds = []
        for n in names:
            if n in self.uk_profiles:
                kinds.append(_KIND_MATTER)
            elif n in self.pk_profiles:
                kinds.append(_KIND_PRESSURE)
            elif n in self.hods:
                kinds.append(_KIND_HOD)
            else:
                raise ValueError("no matter or pressure profile or HOD named %r" % (n,))
        hods = [n for n, k in zip(names, kinds) if k == _KIND_HOD]
        if not hods:
            return self._trispec_call(fn, names, q1, q2, extra, out_shape)
        if len(hods) > 2:
            raise ValueError("%d HOD legs: the 1-halo trispectrum needs occupation moments of order %d, which the HOD "
                             "does not define" % (len(hods), len(hods)))
        if len(set(hods)) > 1:
            raise ValueError("HOD legs %r and %r: the 1-halo trispectrum of two HODs needs their joint occupation, "
                             "which is not defined" % tuple(hods))
        if not np.all(np.diff(self._ks64) > 0):
            raise ValueError("the model's ks must be strictly increasing for the 1-halo trispectrum's interpolation")
        legs = (capi.Tracer * 4)(*[self._tracer(n, k)[0] for n, k in zip(names, kinds)])
        nz, nm = self._nz, self._nm
        fn = fn + '_tracers'
        ws = self._workspace('trispec', getattr(capi.lib, fn + '_ws_doubles')(nz, nm, q1.size, q2.size, legs))
        out = self._empty(*out_shape)
        q1_d, q2_d = self._dev(q1), self._dev(q2)
        capi.check(getattr(capi.lib, fn)(nz, nm, self._nk, self._ldk, capi.ptr(self._ks_d), capi.ptr(self._ms_d),
                                         capi.ptr(self._nzm_d), self._rho_m0, legs, q1.size, capi.ptr(q1_d), q2.size,
                                         capi.ptr(q2_d), *[capi.ptr(e) for e in extra], capi.ptr(ws), capi.ptr(out),
                                         capi.stream()), fn)
        res = self._host(out)
        self._check_hods()
        return res

    def get_trispectrum_1halo(self, ks1, ks2=None, name="nfw", name2=None, name3=None, name4=None):
        """1-halo trispectrum T^{ABCD}(k1, k2; z) = sum_M w_M n(z,M) t_A(k1) t_B(k1) t_C(k2) t_D(k2), [nz, nk1, nk2].

        No counterpart in the reference (Cooray & Hu 2001, eq. 17).  A profile tracer's leg is t = (M/rho_m0) u(k|M,z)
        for a matter profile and u(k|M,z) for a pressure profile, the weights of get_power_1halo; w_M is the trapezoid
        weight on ms.  u is interpolated linearly in k on `ks`, and k outside [ks[0], ks[-1]] is clamped to the edge.
        No 1-halo damping factor (1 - exp(-(k/k*)^2)) is applied.  Names resolve as matter profile, then pressure
        profile, then HOD.  A galaxy leg is t_g = (Nc u_c + Ns u_s)/ngal, get_power's (u_c = 1 without a central
        profile).  Two galaxy legs in one halo take the pair moment without self-pairs, as get_power_1halo("g", "g"):
        t_g(k) t_g(k') is replaced by [NsNsm1 u_s(k) u_s(k') + NcNs (u_c(k) u_s(k') + u_s(k) u_c(k'))] / ngal^2, on one
        side (k = k') or across the two (k = k1, k' = k2).  Three or four galaxy legs, which need occupation moments
        the HOD does not define, and galaxy legs of two different HODs raise ValueError.  Defaults: name2 = name,
        name3 = name, name4 = name3, ks2 = ks1.  ks1 and ks2 need not be sorted."""
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        k1 = self._positive(ks1, "ks1")
        k2 = k1 if ks2 is None else self._positive(ks2, "ks2")
        return self._trispec1h_call('hmv_trispec_1h', (name, name2, name3, name4), k1, k2, (),
                                    (self._nz, k1.size, k2.size))

    def get_cl_cov_1halo(self, ells, name="nfw", name2=None, name3=None, name4=None, windows=(1., 1., 1., 1.), fsky=1.,
                         ells2=None):
        """Non-Gaussian (1-halo) Limber covariance Cov(C_l^{AB}, C_l'^{CD}), [len(ells), len(ells2)]:

            1/(4 pi fsky) sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 T^{ABCD}((l+1/2)/chi, (l'+1/2)/chi; z)

        with the window convention of limber_integral (C = int dz H W1 W2/chi^2 P), zeta_z the trapezoid weight on
        self.zs (1 for a single redshift) and T as in get_trispectrum_1halo (no 1-halo damping; galaxy legs of one
        HOD, at most two).  Each window is a scalar or an [nz] array on self.zs: lensing_window(zs, lzs) for kappa, 1
        for Compton-y (1/H is inside the y profile), the normalised dN/dz on self.zs for galaxies (as C_kg and C_gg
        take it).  Defaults: name2 = name, name3 = name, name4 = name3, ells2 = ells; multipoles need not be sorted.
        Not available on a z-sharded model (the z sum would need a cross-rank reduction)."""
        if self._zcomm is not None:
            raise NotImplementedError("get_cl_cov_1halo on a z-sharded model: the z sum spans the ranks")
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        l1 = self._positive(ells, "ells")
        l2 = l1 if ells2 is None else self._positive(ells2, "ells2")
        fsky = self._fsky(fsky)
        W = self._window_product(windows)
        chis = np.asarray(self.comoving_radial_distance(self.zs), dtype=np.float64).reshape(-1)
        H = np.asarray(self.h_of_z(self.zs), dtype=np.float64).reshape(-1)
        pref = H ** 3 * W / chis ** 6 / (4.0 * np.pi * fsky)
        extra = (self._zs_d, self._dev(chis), self._dev(pref))
        return self._trispec1h_call('hmv_cl_cov_1h', (name, name2, name3, name4), l1, l2, extra, (l1.size, l2.size))

    # ------------------------------------------------------------------ 2-halo trispectrum and C_l covariance
    # Workspace budget of one 2-halo call, in doubles (8 GiB): the largest number of redshifts per pass that fits
    _TRISPEC_2H_WS_BUDGET = 1 << 30

    def _trispec2h_call(self, fn, names, q1, q2, extra, out_shape, what="2-halo trispectrum",
                        hod_why="needs occupation moments up to third order, which the HOD does not define",
                        budget=None):
        budget = self._TRISPEC_2H_WS_BUDGET if budget is None else budget
        cubes, kinds = self._trispec_legs(names, what, hod_why)
        nz, nm = self._nz, self._nm
        u_h = (C.c_void_p * 4)(*[c.data_ptr() for c in cubes])
        k_h = (C.c_int * 4)(*kinds)
        size = getattr(capi.lib, fn + '_ws_doubles')
        lo, hi = 1, nz                   # the workspace grows with zchunk: the largest zchunk within the budget
        while lo < hi:
            mid = (lo + hi + 1) // 2
            if size(nz, nm, self._nk, q1.size, q2.size, u_h, k_h, mid) <= budget:
                lo = mid
            else:
                hi = mid - 1
        ws = self._workspace('trispec', size(nz, nm, self._nk, q1.size, q2.size, u_h, k_h, lo))
        out = self._empty(*out_shape)
        q1_d, q2_d = self._dev(q1), self._dev(q2)
        capi.check(getattr(capi.lib, fn)(nz, nm, self._nk, self._ldk, capi.ptr(self._ks_d), capi.ptr(self._ms_d),
                                         capi.ptr(self._nzm_d), capi.ptr(self._bh_d), capi.ptr(self._Pzk_d),
                                         self._rho_m0, u_h, k_h, q1.size, capi.ptr(q1_d), q2.size, capi.ptr(q2_d),
                                         *[capi.ptr(e) for e in extra], lo, capi.ptr(ws), capi.ptr(out), capi.stream()),
                   fn)
        return self._host(out)

    def get_trispectrum_2halo(self, ks1, ks2=None, name="nfw", name2=None, name3=None, name4=None):
        """2-halo trispectrum of T(k1, -k1, k2, -k2) averaged over the angle between k1 and k2, [nz, nk1, nk2]:

            P(k1) [I1~A(k1) I3^{BCD}(k1,k2,k2) + I1~B(k1) I3^{ACD}(k1,k2,k2)]
          + P(k2) [I1~C(k2) I3^{ABD}(k1,k1,k2) + I1~D(k2) I3^{ABC}(k1,k1,k2)]
          + Pbar(k1,k2) [I2^{AC}(k1,k2) I2^{BD}(k1,k2) + I2^{AD}(k1,k2) I2^{BC}(k1,k2)]

        No counterpart in the reference (Cooray & Hu 2001, ApJ 554, 56).  I2^{XY} = sum_M w_M n b t_X t_Y, I3^{XYZ} =
        sum_M w_M n b t_X t_Y t_Z, I1~X = sum_M w_M n b t_X + b_X - C_X with the consistency terms of get_power_2halo
        (matter: b = 1, C = sum_M w_M n b M/rho_m0; pressure: 0, 0), so that P I1~A I1~B is get_power_2halo's P2h.  P is
        Pzk interpolated linearly in k on `ks` and held at its end values outside; Pbar(k1,k2) = (1/(2 k1 k2))
        int_{|k1-k2|}^{k1+k2} q P(q) dq, in closed form.  The (AB)(CD) pairing carries P(0) and is dropped; I2 and I3
        carry no consistency term; no 1-halo damping.  Legs t, names, defaults and k handling as get_trispectrum_1halo;
        HODs raise ValueError.  The redshifts run in passes whose workspace fits _TRISPEC_2H_WS_BUDGET doubles; the
        result does not depend on the pass size."""
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        k1 = self._positive(ks1, "ks1")
        k2 = k1 if ks2 is None else self._positive(ks2, "ks2")
        return self._trispec2h_call('hmv_trispec_2h', (name, name2, name3, name4), k1, k2, (),
                                    (self._nz, k1.size, k2.size))

    def get_cl_cov_2halo(self, ells, name="nfw", name2=None, name3=None, name4=None, windows=(1., 1., 1., 1.), fsky=1.,
                         ells2=None):
        """Non-Gaussian 2-halo Limber covariance Cov(C_l^{AB}, C_l'^{CD}), [len(ells), len(ells2)]:

            1/(4 pi fsky) sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 T2h^{ABCD}((l+1/2)/chi, (l'+1/2)/chi; z)

        with T2h from get_trispectrum_2halo and the projection, windows, names and defaults of get_cl_cov_1halo.  Not
        available on a z-sharded model (the z sum would need a cross-rank reduction)."""
        if self._zcomm is not None:
            raise NotImplementedError("get_cl_cov_2halo on a z-sharded model: the z sum spans the ranks")
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        l1 = self._positive(ells, "ells")
        l2 = l1 if ells2 is None else self._positive(ells2, "ells2")
        fsky = self._fsky(fsky)
        W = self._window_product(windows)
        chis = np.asarray(self.comoving_radial_distance(self.zs), dtype=np.float64).reshape(-1)
        H = np.asarray(self.h_of_z(self.zs), dtype=np.float64).reshape(-1)
        pref = H ** 3 * W / chis ** 6 / (4.0 * np.pi * fsky)
        extra = (self._zs_d, self._dev(chis), self._dev(pref))
        return self._trispec2h_call('hmv_cl_cov_2h', (name, name2, name3, name4), l1, l2, extra, (l1.size, l2.size))

    # ------------------------------------------------------------------ 3- and 4-halo trispectra and C_l covariance
    # Workspace budget of one 3-halo call, in doubles (8 GiB): the largest number of redshifts per pass that fits
    _TRISPEC_3H_WS_BUDGET = 1 << 30
    _PT_HOD_WHY = "is not implemented for HOD tracers (matter and pressure profiles only)"

    def _trispec4h_call(self, fn, names, q1, q2, extra, out_shape):
        cubes, kinds = self._trispec_legs(names, "4-halo trispectrum", self._PT_HOD_WHY)
        nz, nm = self._nz, self._nm
        ws = self._workspace('trispec', getattr(capi.lib, fn + '_ws_doubles')(nz, self._nk, q1.size, q2.size))
        out = self._empty(*out_shape)
        q1_d, q2_d = self._dev(q1), self._dev(q2)
        u_h = (C.c_void_p * 4)(*[c.data_ptr() for c in cubes])
        capi.check(getattr(capi.lib, fn)(nz, nm, self._nk, self._ldk, capi.ptr(self._ks_d), capi.ptr(self._ms_d),
                                         capi.ptr(self._nzm_d), capi.ptr(self._bh_d), capi.ptr(self._Pzk_d),
                                         self._rho_m0, u_h, (C.c_int * 4)(*kinds), q1.size, capi.ptr(q1_d), q2.size,
                                         capi.ptr(q2_d), *[capi.ptr(e) for e in extra], capi.ptr(ws), capi.ptr(out),
                                         capi.stream()),
                   fn)
        return self._host(out)

    def _pt_args(self, ks1, ks2, name, name2, name3, name4):
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        k1 = self._positive(ks1, "ks1")
        k2 = k1 if ks2 is None else self._positive(ks2, "ks2")
        return (name, name2, name3, name4), k1, k2

    def _pt_cov_args(self, what, ells, name, name2, name3, name4, windows, fsky, ells2):
        if self._zcomm is not None:
            raise NotImplementedError("%s on a z-sharded model: the z sum spans the ranks" % what)
        names, l1, l2 = self._pt_args(ells, ells2, name, name2, name3, name4)
        fsky = self._fsky(fsky)
        W = self._window_product(windows)
        chis = np.asarray(self.comoving_radial_distance(self.zs), dtype=np.float64).reshape(-1)
        H = np.asarray(self.h_of_z(self.zs), dtype=np.float64).reshape(-1)
        pref = H ** 3 * W / chis ** 6 / (4.0 * np.pi * fsky)
        return names, l1, l2, (self._zs_d, self._dev(chis), self._dev(pref))

    def get_trispectrum_3halo(self, ks1, ks2=None, name="nfw", name2=None, name3=None, name4=None):
        """3-halo trispectrum of T(k1, -k1, k2, -k2) averaged over mu = k1^.k2^, [nz, nk1, nk2]:

            Bbar(k1,k2) [I2^{AC} I1~B I1~D + I2^{AD} I1~B I1~C + I2^{BC} I1~A I1~D + I2^{BD} I1~A I1~C]
            Bbar = (34/21) P(k1) P(k2) + 2 <G P(|k1+k2|)>,  G = P(k1) F2(-k1, k1+k2) + P(k2) F2(-k2, k1+k2)

        No counterpart in the reference (Cooray & Hu 2001, ApJ 554, 56).  Bbar is the angle-averaged tree-level
        bispectrum with the pairings that carry P(0) dropped; <.> = (1/2) int dmu, exact for P linear on `ks` (held at
        its end values outside).  I2 and I1~ as in get_trispectrum_2halo (I2 carries no consistency term).  Legs,
        names, defaults and k handling as get_trispectrum_2halo; HODs raise ValueError.  The redshifts run in passes
        whose workspace fits _TRISPEC_3H_WS_BUDGET doubles; the result does not depend on the pass size."""
        names, k1, k2 = self._pt_args(ks1, ks2, name, name2, name3, name4)
        return self._trispec2h_call('hmv_trispec_3h', names, k1, k2, (), (self._nz, k1.size, k2.size),
                                    "3-halo trispectrum", self._PT_HOD_WHY, self._TRISPEC_3H_WS_BUDGET)

    def get_cl_cov_3halo(self, ells, name="nfw", name2=None, name3=None, name4=None, windows=(1., 1., 1., 1.), fsky=1.,
                         ells2=None):
        """Non-Gaussian 3-halo Limber covariance Cov(C_l^{AB}, C_l'^{CD}), [len(ells), len(ells2)]:

            1/(4 pi fsky) sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 T3h^{ABCD}((l+1/2)/chi, (l'+1/2)/chi; z)

        with T3h from get_trispectrum_3halo and the projection, windows, names and defaults of get_cl_cov_1halo.  Not
        available on a z-sharded model (the z sum would need a cross-rank reduction)."""
        names, l1, l2, extra = self._pt_cov_args("get_cl_cov_3halo", ells, name, name2, name3, name4, windows, fsky,
                                                 ells2)
        return self._trispec2h_call('hmv_cl_cov_3h', names, l1, l2, extra, (l1.size, l2.size), "3-halo trispectrum",
                                    self._PT_HOD_WHY, self._TRISPEC_3H_WS_BUDGET)

    def get_trispectrum_4halo(self, ks1, ks2=None, name="nfw", name2=None, name3=None, name4=None):
        """4-halo trispectrum of T(k1, -k1, k2, -k2) averaged over mu = k1^.k2^, [nz, nk1, nk2]:

            I1~A(k1) I1~B(k1) I1~C(k2) I1~D(k2) Tbar(k1,k2)
            Tbar = 12 P1 P2^2 F3bar(k2/k1) + 12 P1^2 P2 F3bar(k1/k2) + 8 <G^2 P(|k1+k2|)>

        No counterpart in the reference (Cooray & Hu 2001, ApJ 554, 56).  Tbar is the angle-averaged tree-level
        trispectrum with the pairings that carry P(0) dropped; F3bar(r) = <F3_sym(k, q, -q)>, r = q/k; G and <.> as in
        get_trispectrum_3halo; I1~ as in get_trispectrum_2halo.  Legs, names, defaults and k handling as
        get_trispectrum_2halo; HODs raise ValueError."""
        names, k1, k2 = self._pt_args(ks1, ks2, name, name2, name3, name4)
        return self._trispec4h_call('hmv_trispec_4h', names, k1, k2, (), (self._nz, k1.size, k2.size))

    def get_cl_cov_4halo(self, ells, name="nfw", name2=None, name3=None, name4=None, windows=(1., 1., 1., 1.), fsky=1.,
                         ells2=None):
        """Non-Gaussian 4-halo Limber covariance Cov(C_l^{AB}, C_l'^{CD}), [len(ells), len(ells2)]:

            1/(4 pi fsky) sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 T4h^{ABCD}((l+1/2)/chi, (l'+1/2)/chi; z)

        with T4h from get_trispectrum_4halo and the projection, windows, names and defaults of get_cl_cov_1halo.  Not
        available on a z-sharded model (the z sum would need a cross-rank reduction)."""
        names, l1, l2, extra = self._pt_cov_args("get_cl_cov_4halo", ells, name, name2, name3, name4, windows, fsky,
                                                 ells2)
        return self._trispec4h_call('hmv_cl_cov_4h', names, l1, l2, extra, (l1.size, l2.size))

    @staticmethod
    def _fsky(fsky):
        fsky = float(fsky)
        if not (0.0 < fsky <= 1.0):
            raise ValueError("fsky must lie in (0, 1]")
        return fsky

    def _window_product(self, windows):
        """W_A W_B W_C W_D on self.zs; each window is a scalar or an [nz] array."""
        if len(windows) != 4:
            raise ValueError("windows must hold four entries (A, B, C, D)")
        W = np.ones(self._nz)
        for w in windows:
            w = np.asarray(w, dtype=np.float64)
            if w.ndim > 1 or (w.ndim == 1 and w.size != self._nz):
                raise ValueError("each window must be a scalar or an array of length nz=%d" % self._nz)
            W = W * w
        return W

    # ------------------------------------------------------------------ super-sample covariance (DESIGN.md §4.5)
    def _response_legs(self, names):
        cubes, kinds = self._trispec_legs(names, "response", "needs the number-density term -(b_A + b_B) P, which is "
                                                             "not part of the response of profile tracers")
        if self._nk < 2:
            raise ValueError("the response needs at least two wavenumbers (n_eff)")
        return cubes, kinds

    def _response_device(self, cubes, kinds):
        """R1h + R2h of a pair of profile legs as a device tensor [nz, nk] (hmv_power_response)."""
        nz, nm = self._nz, self._nm
        ws = self._workspace('power', capi.lib.hmv_power_ws_doubles(nz, nm))
        r1, r2 = self._empty(nz, self._nk), self._empty(nz, self._nk)
        capi.check(capi.lib.hmv_power_response(nz, nm, self._nk, self._ldk, capi.ptr(self._ms_d), capi.ptr(self._ks_d),
                                               capi.ptr(self._nzm_d), capi.ptr(self._bh_d), capi.ptr(self._Pzk_d),
                                               self._rho_m0, capi.ptr(cubes[0]), kinds[0], capi.ptr(cubes[1]), kinds[1],
                                               capi.ptr(ws), capi.ptr(r1), capi.ptr(r2), capi.stream()),
                   "hmv_power_response")
        capi.check(capi.lib.hmv_sum2(r1.numel(), capi.ptr(r1), capi.ptr(r2), capi.ptr(r1), capi.stream()), "hmv_sum2")
        return r1

    def get_power_response(self, name="nfw", name2=None):
        """Response of P^{AB}(k, z) to a long-wavelength density mode, dP/d delta_b on self.ks, [nz, nk]:

            R1h = sum_M w_M n(z,M) b(z,M) t_A(k) t_B(k)                (no 1-halo damping)
            R2h = [47/21 - n_eff(z,k)/3] P2h^{AB}(k, z),   n_eff = d ln P_lin / d ln k

        (Takada & Hu 2013, PRD 87, 123504).  No counterpart in the reference.  t as in get_trispectrum_1halo: (M/rho_m0) u
        for a matter profile, u for a pressure profile; P2h is get_power_2halo's.  n_eff follows
        np.gradient(np.log(Pzk), np.log(ks), axis=1); a P_lin that is not positive at a column or a neighbour gives NaN
        there.  HODs raise ValueError.  On a z-sharded model: this rank's slab."""
        name2 = name if name2 is None else name2
        cubes, kinds = self._response_legs((name, name2))
        return self._host(self._response_device(cubes, kinds))

    def _sigma_b2_grid(self, fsky):
        """Disc radius R_z = chi(z) theta_s (cos theta_s = 1 - 2 fsky), the k grid geomspace(k_b, sigma2_kmax,
        sigma2_numks) with k_b = min(sigma2_kmin, 1e-3 / max_z R_z), and its weights simpson * k / (2 pi)."""
        from .cosmology import simpson_weights
        chis = np.asarray(self.comoving_radial_distance(self.zs), dtype=np.float64).reshape(-1)
        R = chis * np.arccos(1.0 - 2.0 * fsky)
        kb = float(self.p['sigma2_kmin'])
        if R.max() > 0:
            kb = min(kb, 1e-3 / R.max())
        kg = np.geomspace(kb, self.p['sigma2_kmax'], int(self.p['sigma2_numks']))
        return R, kg, simpson_weights(kg) * kg / (2.0 * np.pi)

    def get_sigma_b2(self, fsky):
        """Variance of the background density mode over a disc of area 4 pi fsky, flat sky, [nz]:

            sigma_b^2(z) = 1/(2 pi) int dk k P_lin(k, z) [2 J1(k R_z) / (k R_z)]^2,   R_z = chi(z) theta_s

        Simpson on geomspace(k_b, sigma2_kmax, sigma2_numks), k_b = min(sigma2_kmin, 1e-3 / max_z R_z); P_lin from the
        producer of sPzk (accuracy 'low': EH98 on the device; otherwise P_lin / P_lin_slow).  The model's sPzk, sigma2
        and mass function are not touched.  On a z-sharded model: this rank's slab (k_b from the slab's redshifts)."""
        fsky = self._fsky(fsky)
        R, kg, kw = self._sigma_b2_grid(fsky)
        if self.accuracy == 'low':
            P_d = self._plin_device(kg, self.zs)
        elif self.accuracy == 'high':
            P_d = self._dev(np.asarray(self.P_lin_slow(kg, self.zs, kmax=self.p['sigma2_kmax']), dtype=np.float64))
        else:
            P_d = self._dev(np.asarray(self.P_lin(kg, self.zs), dtype=np.float64))
        out = self._empty(self._nz)
        kg_d, kw_d, R_d = self._dev(kg), self._dev(kw), self._dev(R)
        capi.check(capi.lib.hmv_sigma_b2(self._nz, kg.size, capi.ptr(kg_d), capi.ptr(kw_d), capi.ptr(P_d),
                                         capi.ptr(R_d), capi.ptr(out), capi.stream()), "hmv_sigma_b2")
        return self._host(out)

    def get_cl_cov_ssc(self, ells, name="nfw", name2=None, name3=None, name4=None, windows=(1., 1., 1., 1.), fsky=1.,
                       ells2=None, sigma_b2=None):
        """Super-sample covariance Cov_SSC(C_l^{AB}, C_l'^{CD}), [len(ells), len(ells2)]:

            sum_z zeta_z H^3 W_A W_B W_C W_D sigma_b^2(z) / chi^4 R^{AB}((l+1/2)/chi, z) R^{CD}((l'+1/2)/chi, z)

        (Takada & Hu 2013; Li, Hu & Takada 2014), with R from get_power_response interpolated linearly in k on `ks` (k
        clamped to the grid's ends), sigma_b^2 from get_sigma_b2(fsky) and the window convention of get_cl_cov_1halo.
        fsky enters only through sigma_b^2.  sigma_b2: an optional [nz] array (e.g. from a mask's power spectrum) that
        replaces the disc.  Names, windows, ells2 and the defaults behave as in get_cl_cov_1halo; HODs raise ValueError.
        Not available on a z-sharded model (the z sum would need a cross-rank reduction)."""
        if self._zcomm is not None:
            raise NotImplementedError("get_cl_cov_ssc on a z-sharded model: the z sum spans the ranks")
        name2 = name if name2 is None else name2
        name3 = name if name3 is None else name3
        name4 = name3 if name4 is None else name4
        l1 = self._positive(ells, "ells")
        l2 = l1 if ells2 is None else self._positive(ells2, "ells2")
        fsky = self._fsky(fsky)
        W = self._window_product(windows)
        if sigma_b2 is not None:
            sb2 = np.array(sigma_b2, dtype=np.float64).reshape(-1)
            if sb2.size != self._nz or not np.all(np.isfinite(sb2)) or np.any(sb2 < 0):
                raise ValueError("sigma_b2 must hold nz=%d finite non-negative values" % self._nz)
        legAB = self._response_legs((name, name2))
        legCD = self._response_legs((name3, name4))
        if sigma_b2 is None:
            sb2 = self.get_sigma_b2(fsky)
        chis = np.asarray(self.comoving_radial_distance(self.zs), dtype=np.float64).reshape(-1)
        H = np.asarray(self.h_of_z(self.zs), dtype=np.float64).reshape(-1)
        pref = H ** 3 * W * sb2 / chis ** 4
        rAB = self._response_device(*legAB)
        rCD = rAB if (name3, name4) == (name, name2) else self._response_device(*legCD)
        nz = self._nz
        ws = self._workspace('ssc', capi.lib.hmv_cl_cov_ssc_ws_doubles(nz, l1.size, l2.size))
        out = self._empty(l1.size, l2.size)
        l1_d, l2_d, chis_d, pref_d = self._dev(l1), self._dev(l2), self._dev(chis), self._dev(pref)
        capi.check(capi.lib.hmv_cl_cov_ssc(nz, self._nk, capi.ptr(self._ks_d), capi.ptr(rAB), capi.ptr(rCD), l1.size,
                                           capi.ptr(l1_d), l2.size, capi.ptr(l2_d), capi.ptr(self._zs_d),
                                           capi.ptr(chis_d), capi.ptr(pref_d), capi.ptr(ws), capi.ptr(out),
                                           capi.stream()), "hmv_cl_cov_ssc")
        return self._host(out)


    # ------------------------------------------------------------------ cluster-lensing helper
    def kappa_2h_profiles(self, thetas, Ms, zsource, delta=200, rho='mean', rho_at_z=True, lmin=100, lmax=10000,
                          verbose=True):
        """Two-halo convergence profile kappa_2h(theta) of a halo of mass Ms at the lens redshift (hmvec.py:598-622):
        rho_m b_h / (1+z)^3 / Sigma_cr / D_A^2 * int dl l/(2 pi) J0(l theta) P_lin(k = l/chi), trapezoid over the
        l = k chi inside (lmin, lmax).  Returns [n_theta, nz].  The reference forms `self.ks*chis`, which only
        broadcasts for ONE lens redshift (zs of length 1); that case is reproduced exactly, and several lens redshifts
        are handled one by one with the same expression.  Host-side O(n_theta nk) Hankel sum on [nz,nk] inputs; the
        bias b_h it interpolates is the device mass function's."""
        from scipy.special import j0
        zlens = self.zs
        Ms = np.broadcast_to(np.asarray(Ms, dtype=np.float64).reshape(-1), (zlens.size,)) if np.size(Ms) in (1, zlens.size) \
            else np.asarray(Ms, dtype=np.float64).reshape(-1)
        if Ms.size != zlens.size:
            raise ValueError("Ms must be a scalar or one mass per lens redshift")
        sigmac = np.atleast_1d(self.sigma_crit(zlens, zsource))
        rhomz = np.atleast_1d(self.rho_matter_z(zlens))
        chis = np.atleast_1d(np.asarray(self.comoving_radial_distance(zlens), dtype=np.float64))
        DAz = np.atleast_1d(self.angular_diameter_distance(zlens))
        Pzk, bh = self.Pzk, self.bh
        bhs = np.array([np.interp(Ms[i], self.ms, bh[i]) for i in range(zlens.size)])
        if verbose:
            print("bias ", bhs)
            print("sigmacr ", sigmac)
        thetas = np.atleast_1d(np.asarray(thetas, dtype=np.float64))
        out = np.zeros((thetas.size, zlens.size))
        for i in range(zlens.size):
            ells = self._ks64 * chis[i]
            sel = np.logical_and(ells > lmin, ells < lmax)
            l = ells[sel]
            pref = rhomz[i] * bhs[i] / (1 + zlens[i]) ** 3. / sigmac[i] / DAz[i] ** 2
            for it, theta in enumerate(thetas):
                out[it, i] = _trapz(pref * Pzk[i, sel] * j0(l * theta) * l / 2. / np.pi, l)
        return out


class LazyCube(object):
    """Second return value of add_nfw_profile: behaves as the [nz,nm,nk] numpy array when converted or indexed,
    without forcing a 32 GB device->host copy when the caller ignores it."""

    def __init__(self, cubes, name):
        self._cubes, self._name = cubes, name

    def __array__(self, dtype=None, copy=None):
        a = self._cubes[self._name]
        return a if dtype is None else a.astype(dtype)

    def __getitem__(self, idx):
        return self._cubes[self._name][idx]

    @property
    def shape(self):
        o = self._cubes._owner
        return (o._nz, o._nm, o._nk)
