"""Cosmology: host-side background / linear-power producers + device sigma^2 and Limber kernels.

Drop-in for the reference `hmvec.cosmology.Cosmology` on the hot path (cosmology.py:51-597, 867-904):
same constructor, same method names and argument meaning.  What runs where:

  host (numpy, O(nz)+O(nk) work, inputs to the path -- "Linear P(k) from CAMB stays a host-side input"):
      background H(z), chi(z) [camb if installed, else the analytic flat-LCDM background], EH98 transfer
      function / P_lin_approx, growth factor, lensing windows, Simpson weight vector
  device (hand-written sm_100a kernels through the C ABI, no CPU fallback):
      get_sigma2_R  -> hmv_sigma2        (cosmology.py:245-269)
      limber_integral / C_kk / C_kg / C_gg / C_ky / C_yy -> hmv_limber   (cosmology.py:536-597, 867-904)
"""
import warnings

import numpy as np
import torch

from . import _capi as capi
from .background import AnalyticBackground
from .params import default_params

cspeed = 299792.458  # km/s


def _trapz(y, x, axis=-1):
    f = getattr(np, "trapezoid", None) or np.trapz
    return f(y, x, axis=axis)


def Wkr_taylor(kR):
    xx = kR * kR
    return 1 - .1 * xx + .00357142857143 * xx * xx


def Wkr(k, R, taylor_switch=default_params['Wkr_taylor_switch']):
    """Top-hat window (host helper kept for API compatibility, cosmology.py:30-38); the device path evaluates the
    same expression inside hmv_sigma2."""
    kR = np.asarray(k * R, dtype=np.float64)
    with np.errstate(all="ignore"):
        ans = 3. * (np.sin(kR) - kR * np.cos(kR)) / (kR ** 3.)
    small = kR < taylor_switch
    ans[small] = Wkr_taylor(kR[small])
    return ans


def simpson_weights(x):
    """Weight vector w with scipy.integrate.simpson(y, x=x) == y @ w  (SciPy >= 1.11 rule).

    Odd N: composite non-uniform Simpson over interval pairs.  Even N: the same on the first N-1 points plus the
    Cartwright correction on the last interval.  Linear in y, so sigma^2 becomes one contraction on the device."""
    x = np.asarray(x, dtype=np.float64)
    N = x.size
    w = np.zeros(N)
    if N == 1:
        return w
    if N == 2:
        w[:] = 0.5 * (x[1] - x[0])
        return w
    h = np.diff(x)
    last = N if N % 2 == 1 else N - 1
    h0, h1 = h[0:last - 1:2], h[1:last - 1:2]
    hs = h0 + h1
    w[0:last - 2:2] += hs / 6.0 * (2.0 - h1 / h0)
    w[1:last - 1:2] += hs / 6.0 * (hs * hs / (h0 * h1))
    w[2:last:2] += hs / 6.0 * (2.0 - h0 / h1)
    if N % 2 == 0:
        a0, a1 = h[-2], h[-1]
        w[-1] += (2.0 * a1 ** 2 + 3.0 * a0 * a1) / (6.0 * (a0 + a1))
        w[-2] += (a1 ** 2 + 3.0 * a0 * a1) / (6.0 * a0)
        w[-3] -= a1 ** 3 / (6.0 * a0 * (a0 + a1))
    return w


def get_eds_model(fb=0.15, H0=68.0, YHe=0.25):
    """Einstein-de Sitter parameter set (cosmology.py:40-49)."""
    h0 = H0 / 100
    return {'omch2': (1 - fb) * h0 ** 2, 'ombh2': fb * h0 ** 2, 'H0': H0, 'mnu': 0., 'YHe': YHe}


def _default_device():
    if not torch.cuda.is_available():
        raise RuntimeError("hmvec_b200 needs a CUDA device (B200, sm_100a): there is no CPU fallback.")
    return torch.device("cuda", torch.cuda.current_device())


class Cosmology(object):

    def __init__(self, params={}, halofit=None, engine='camb', accuracy='medium', device=None):
        engine = engine.lower()
        if not (engine in ['camb', 'class']):
            raise ValueError
        self.accuracy = accuracy
        self.engine = engine
        if self.accuracy == 'low' and (('S8' in params.keys()) or ('sigma8' in params.keys())):
            raise ValueError("Can't use S8 or sigma8 with low accuracy.")
        self.p = dict(params) if params is not None else {}
        for key, val in default_params.items():
            self.p.setdefault(key, val)
        self._device = torch.device(device) if device is not None else None
        self._bg_cache = {}
        self._init_cosmology(self.p, halofit)

    # ------------------------------------------------------------------ device plumbing
    @property
    def device(self):
        """CUDA device of this object; resolved on first use so that the host-side producers (background, P_lin,
        windows) work on a machine without a GPU while every device op still fails loudly there."""
        if self._device is None:
            self._device = _default_device()
        return self._device

    def _dev(self, a):
        """numpy -> device through a pinned staging block, asynchronously on the current stream: a pageable copy
        would block the host until every kernel queued before it has finished (torch's caching host allocator keeps
        the block alive until the copy has been carried out)."""
        return _upload(a, self.device)

    def _empty(self, *shape):
        return torch.empty(shape, dtype=torch.float64, device=self.device)

    # ------------------------------------------------------------------ background (host input)
    def _init_cosmology(self, params, halofit):
        if 'theta100' in params:
            raise NotImplementedError("theta100 parameterisation needs CAMB's solver; pass H0")
        H0 = params['H0']
        h = H0 / 100.
        if 'omm' in params:
            params['omch2'] = params['omm'] * h ** 2 - params['ombh2']
            print("WARNING: omm specified. Ignoring omch2.")
        self._camb_results = None
        if self.engine == 'camb':
            try:
                import camb
            except ImportError:
                camb = None
            if camb is not None:
                YHe = params.get('YHe')
                self._camb_pars = camb.set_params(
                    ns=params['ns'], As=params['As'], r=params.get('r', 0.), H0=H0, cosmomc_theta=None,
                    ombh2=params['ombh2'], omch2=params['omch2'], mnu=params['mnu'], omk=params['omk'],
                    tau=params['tau'], nnu=params['nnu'], num_massive_neutrinos=params['num_massive_neutrinos'],
                    w=params['w0'], wa=params['wa'], dark_energy_model='ppf',
                    halofit_version=self.p['default_halofit'] if halofit is None else halofit,
                    AccuracyBoost=2, pivot_scalar=params['pivot_scalar'], YHe=YHe)
                self._camb_pars.WantTransfer = True
                self._camb_pars.WantTensors = True
                self._camb_results = camb.get_background(self._camb_pars)
            else:
                if self.accuracy != 'low':
                    raise ImportError("camb is not installed: accuracy='%s' needs CAMB's linear P(k). Use "
                                      "accuracy='low' (EH98 P(k) + analytic flat-LCDM background) or install camb."
                                      % self.accuracy)
                warnings.warn("camb not installed: using the analytic flat-LCDM background (H0, Om only).")
                self._camb_results = AnalyticBackground(H0, params['ombh2'], params['omch2'])
        else:
            raise NotImplementedError("engine='class' is a host-side P(k) producer outside the B200 hot path")
        self.params = params
        omh2 = self.params['omch2'] + self.params['ombh2']
        self.h = h
        self.omm0 = omh2 / (self.params['H0'] / 100.) ** 2.
        self.omk0 = self.params['omk']
        self.oml0 = 1 - self.omm0 - self.omk0
        self.as8 = self.params.get('as8', 1)
        self.ombh2 = self.params['ombh2']
        self.YHe = getattr(getattr(self, '_camb_pars', None), 'YHe', params.get('YHe', 0.24))

    def _bg(self, what, z):
        """Background quantity `what` at z, memoised per argument: the same redshift vector is asked for again and
        again (every window, every Limber call), and each evaluation is a quadrature (or a CAMB call)."""
        if np.ndim(z) == 0:
            return getattr(self._camb_results, what)(z)
        za = np.ascontiguousarray(z, dtype=np.float64)
        key = (what, za.shape, za.tobytes())
        hit = self._bg_cache.get(key)
        if hit is None:
            if len(self._bg_cache) > 64:
                self._bg_cache.clear()
            hit = self._bg_cache[key] = np.asarray(getattr(self._camb_results, what)(z))
        return hit.copy()

    def angular_diameter_distance(self, z1, z2=None):
        if z2 is not None:
            return self._camb_results.angular_diameter_distance2(z1, z2)
        return self._bg('angular_diameter_distance', z1)

    def comoving_radial_distance(self, z):
        return self._bg('comoving_radial_distance', z)

    def hubble_parameter(self, z):  # km/s/Mpc
        return self._bg('hubble_parameter', z)

    def h_of_z(self, z):  # 1/Mpc
        return self._bg('h_of_z', z)

    def get_growth_rate_f(self, zs):
        """Logarithmic growth rate f = dlnD/dlna.  The reference takes it from CLASS and raises for engine='camb'
        (cosmology.py:345-350); here it is the derivative of the closed-form growing mode D_growth_approx
        (cosmology.py:297-313, flat LCDM), by central differences in ln a."""
        a = 1. / (1. + np.atleast_1d(np.asarray(zs, dtype=np.float64)))
        e = 1e-4
        return (np.log(self.D_growth_approx(a * np.exp(e))) - np.log(self.D_growth_approx(a * np.exp(-e)))) / (2. * e)

    def get_Omega_nu(self):
        return self._camb_results.get_Omega('nu')

    def sigma_crit(self, zlens, zsource):
        Gval = 4.517e-48
        cval = 9.716e-15
        Dd = self.angular_diameter_distance(zlens)
        Ds = self.angular_diameter_distance(zsource)
        Dds = np.asarray([self.angular_diameter_distance(zl, zsource) for zl in zlens])
        return cval ** 2 * Ds / 4 / np.pi / Gval / Dd / Dds

    # cosmology.py:232-243
    def rho_matter_z(self, z):
        return self.rho_critical_z(0.) * self.omm0 * (1 + np.atleast_1d(z)) ** 3.

    def omz(self, z):
        return self.rho_matter_z(z) / self.rho_critical_z(z)

    def rho_critical_z(self, z):
        Hz = self.hubble_parameter(z) * 3.241e-20
        G = 6.67259e-11
        return 3. * (Hz ** 2.) / 8. / np.pi / G * 1.477543e37

    # ------------------------------------------------------------------ linear power (host input)
    def _pk_grid(self, PK, zs, ks):
        """PK.P(zs, ks, grid=True) of a RectBivariateSpline-based interpolator, evaluated on the GPU (hmv_pk_spline)."""
        from .utils import PKInterpolatorDevice
        if not isinstance(PK, PKInterpolatorDevice):
            if not hasattr(PK, "tck"):                   # single-redshift interp1d objects: tiny, host
                return PK.P(zs, ks, grid=True)
            PK = PKInterpolatorDevice.from_spline(PK, device=self.device)
        return PK.P(np.atleast_1d(zs), np.atleast_1d(ks), grid=True)

    def _get_matter_power(self, zs, ks, nonlinear=False):
        PK = self.get_pk_interpolator(zs, kmax=np.max(ks), var='total', nonlinear=nonlinear)
        return (self.as8 ** 2.) * self._pk_grid(PK, zs, ks)

    def get_pk_interpolator(self, zs, kmax, var='total', nonlinear=False):
        if not hasattr(self, '_camb_pars'):
            raise ImportError("CAMB is required for interpolated linear/non-linear P(k) (accuracy medium/high)")
        import camb
        from camb import model
        self._camb_pars.set_matter_power(redshifts=list(zs), kmax=kmax + 1., silent=True)
        self._camb_pars.NonLinear = model.NonLinear_both if nonlinear else model.NonLinear_none
        var = {'total': 'delta_tot', 'weyl': 'Weyl'}.get(var, var)
        return camb.get_matter_power_interpolator(self._camb_pars, nonlinear=nonlinear, hubble_units=False,
                                                  k_hunit=False, kmax=kmax + 1., zmax=max(zs) + 1., var1=var, var2=var)

    def D_growth_approx(self, a):
        """Heath 1977 growing mode, normalised to a in matter domination (cosmology.py:297-313)."""
        from scipy.special import hyp2f1
        a = np.asarray(a)
        x = (self.oml0 / self.omm0) ** (1. / 3.) * a
        return np.sqrt(1. + x ** 3.) * hyp2f1(5 / 6., 3 / 2., 11 / 6., -x ** 3.) * a

    def D_growth(self, a, type="anorm", exact=False, k_camb=1e-5):
        if exact:
            raise NotImplementedError("exact growth needs CAMB transfer evolution (host-side, out of the hot path)")
        val = self.D_growth_approx(a) / self.D_growth_approx(1)
        if type == "z0norm":
            return val
        if type == "anorm":
            return val * self.D_growth_approx(1)
        raise ValueError

    def Tk(self, ks, type='eisenhu_osc'):
        """Eisenstein & Hu 1998 transfer function (cosmology.py:404-504); host-side P_lin producer."""
        from .linear_power import eisenstein_hu
        return eisenstein_hu(np.asarray(ks, dtype=np.float64), self.h, self.params['omch2'], self.params['ombh2'],
                             self.omm0, wiggles=(type == 'eisenhu_osc'))

    def P_lin_approx_factors(self, ks, zs, type='eisenhu_osc'):
        """The two factors of the separable EH98 power of cosmology.py:391-402: (D(z)^2 [nz], pref k (k/kp)^(ns-1)
        T(k)^2 [nk]); P(z,k) is their outer product (host: P_lin_approx, device: hmv_outer)."""
        zs = np.atleast_1d(np.asarray(zs, dtype=np.float64))
        ks = np.asarray(ks, dtype=np.float64).reshape(-1)
        tk = self.Tk(ks, type=type)
        Dzs = self.D_growth(1 / (1 + zs), type='anorm')
        kp, ns = self.params['pivot_scalar'], self.params['ns']
        omh2 = (self.params['omch2'] + self.params['ombh2']) * 100 ** 2. + self.get_Omega_nu() * self.params['H0'] ** 2.
        kfacts = (ks / kp) ** (ns - 1.) * ks
        pref = 8 * np.pi ** 2 * self.params['As'] / 25. / omh2 ** 2. * cspeed ** 4.
        return Dzs ** 2., pref * kfacts * tk ** 2.

    def P_lin_approx_factors_device(self, ks_d, zs, type='eisenhu_osc'):
        """The same two factors with the O(nk) one -- EH98 transfer function included -- evaluated on the device
        (hmv_eh98_factor) from a wavenumber tensor; returns (D(z)^2 as numpy [nz], v(k) as a CUDA tensor [nk])."""
        zs = np.atleast_1d(np.asarray(zs, dtype=np.float64))
        Dzs = self.D_growth(1 / (1 + zs), type='anorm')
        kp, ns = self.params['pivot_scalar'], self.params['ns']
        omh2 = (self.params['omch2'] + self.params['ombh2']) * 100 ** 2. + self.get_Omega_nu() * self.params['H0'] ** 2.
        pref = 8 * np.pi ** 2 * self.params['As'] / 25. / omh2 ** 2. * cspeed ** 4.
        v_d = torch.empty(ks_d.numel(), dtype=torch.float64, device=ks_d.device)
        capi.check(capi.lib.hmv_eh98_factor(ks_d.numel(), capi.ptr(ks_d), float(self.h), float(self.params['omch2']),
                                            float(self.params['ombh2']), float(self.omm0), int(type == 'eisenhu_osc'),
                                            float(pref), float(kp), float(ns), capi.ptr(v_d), capi.stream()),
                   "hmv_eh98_factor")
        return Dzs ** 2., v_d

    def P_lin_approx(self, ks, zs, type='eisenhu_osc'):
        """cosmology.py:391-402"""
        d2, v = self.P_lin_approx_factors(ks, zs, type=type)
        return d2[:, None] * v[None, :]

    def P_lin(self, ks, zs, knorm=1e-4, kmax=None):
        """cosmology.py:353-374 (needs CAMB for the normalisation)."""
        zs, ks = np.asarray(zs), np.asarray(ks)
        tk = self.Tk(ks, 'eisenhu_osc')
        if kmax is None:
            kmax = ks.max()
        if knorm >= kmax:
            raise ValueError
        PK = self.get_pk_interpolator(zs, kmax=kmax, var='total', nonlinear=False)
        pnorm = self._pk_grid(PK, zs, knorm)
        tnorm = self.Tk(knorm, 'eisenhu_osc') * knorm ** (self.params['ns'])
        return (self.as8 ** 2.) * (pnorm / tnorm) * tk ** 2. * ks ** (self.params['ns'])

    def P_lin_slow(self, ks, zs, kmax=None):
        zs, ks = np.asarray(zs), np.asarray(ks)
        if kmax is None:
            kmax = ks.max()
        PK = self.get_pk_interpolator(zs, kmax=kmax, var='total', nonlinear=False)
        return (self.as8 ** 2.) * self._pk_grid(PK, zs, ks)

    # ------------------------------------------------------------------ sigma^2 (device, K3)
    def _sigma2_inputs(self, zs, kmin=None, kmax=None, numks=None):
        kmin = self.p['sigma2_kmin'] if kmin is None else kmin
        kmax = self.p['sigma2_kmax'] if kmax is None else kmax
        numks = self.p['sigma2_numks'] if numks is None else numks
        ks_sigma2 = np.geomspace(kmin, kmax, int(numks))
        if self.accuracy == 'high':
            self.sPzk = self.P_lin_slow(ks_sigma2, zs, kmax=kmax)
        elif self.accuracy == 'medium':
            self.sPzk = self.P_lin(ks_sigma2, zs)
        elif self.accuracy == 'low':
            self.sPzk = self.P_lin_approx(ks_sigma2, zs)
        kw = simpson_weights(ks_sigma2) * ks_sigma2 ** 2. / 2. / np.pi ** 2.
        return ks_sigma2, kw

    def _sigma2_device(self, R_d, sPzk_d, ks_sig_d, kw_d):
        """sigma2[z,m] on the device from device inputs (hmv_sigma2); returns a [nz,nm] tensor."""
        nz, nks = sPzk_d.shape
        nm = R_d.numel()
        ws = self._empty(int(capi.lib.hmv_sigma2_ws_doubles(nz, nm, nks)))
        out = self._empty(nz, nm)
        capi.check(capi.lib.hmv_sigma2(nz, nm, nks, capi.ptr(sPzk_d), capi.ptr(kw_d), capi.ptr(ks_sig_d),
                                       capi.ptr(R_d), float(self.p['Wkr_taylor_switch']), capi.ptr(ws),
                                       capi.ptr(out), capi.stream()), "hmv_sigma2")
        return out

    def get_sigma2_R(self, R, zs, kmin=None, kmax=None, numks=None, Ws=None, ret_pk=False):
        """sigma^2(R,z), Simpson over a geomspace k grid (cosmology.py:245-269).  R: [nm] (or [1,nm,1])."""
        if Ws is not None:
            raise NotImplementedError("custom window arrays are not part of the device path")
        zs = np.atleast_1d(zs)
        Rflat = np.asarray(R, dtype=np.float64).reshape(-1)
        ks_sigma2, kw = self._sigma2_inputs(zs, kmin, kmax, numks)
        s2 = self._sigma2_device(self._dev(Rflat), self._dev(self.sPzk), self._dev(ks_sigma2), self._dev(kw))
        sigma2 = s2.cpu().numpy()
        if ret_pk:
            return sigma2, ks_sigma2[None, None, :], self.sPzk[:, None, :]
        return sigma2

    def get_sigma8(self, zs, exact=False, kmin=1e-4, kmax=None, Ws=None, numks=1000, ret_pk=False):
        if exact:
            raise NotImplementedError
        r = self.get_sigma2_R(np.array([8. / self.params['H0'] * 100.]), zs, kmin=kmin, kmax=kmax, numks=numks)
        return np.sqrt(r)

    # ------------------------------------------------------------------ windows (host) and Limber (device, K6)
    def lensing_window(self, ezs, zs, dndz=None):
        """W_kappa(z) (cosmology.py:506-534): delta-function source or dn/dz-weighted."""
        ezs = np.asarray(ezs, dtype=np.float64)
        zs = np.array(zs, dtype=np.float64).reshape(-1)
        H0 = self.h_of_z(0.)
        H = self.h_of_z(ezs)
        chis = self.comoving_radial_distance(ezs)
        chistar = self.comoving_radial_distance(zs)
        if zs.size == 1:
            assert dndz is None
            integral = (chistar - chis) / chistar
            integral[ezs > zs] = 0
        else:
            dndz = np.asarray(dndz, dtype=np.float64)
            dndz = dndz / _trapz(dndz, zs)
            integrand = (chistar[None, :] - chis[:, None]) / chistar[None, :] * dndz[None, :]
            integrand[zs[None, :] < ezs[:, None]] = 0
            integral = _trapz(integrand, zs, axis=-1)
        return 1.5 * self.omm0 * H0 ** 2. * (1. + ezs) * chis / H * integral

    def C_kg(self, ells, zs, ks, Pgm, gzs, gdndz=None, lzs=None, ldndz=None, lwindow=None):
        gzs = np.array(gzs, dtype=np.float64).reshape(-1)
        Wz1s = self.lensing_window(gzs, lzs, ldndz) if lwindow is None else lwindow
        chis = self.comoving_radial_distance(gzs)
        hzs = self.h_of_z(gzs)
        Wz2s = np.asarray(gdndz) / _trapz(gdndz, gzs) if gzs.size > 1 else 1.
        return limber_integral(ells, zs, ks, Pgm, gzs, Wz1s, Wz2s, hzs, chis, device=self.device)

    def C_gg(self, ells, zs, ks, Pgg, gzs, gdndz=None, zmin=None, zmax=None):
        gzs = np.asarray(gzs, dtype=np.float64).reshape(-1)
        chis = self.comoving_radial_distance(gzs)
        hzs = self.h_of_z(gzs)
        if gzs.size > 1:
            Wz1s = Wz2s = np.asarray(gdndz) / _trapz(gdndz, gzs)
        else:
            dchi = self.comoving_radial_distance(zmax) - self.comoving_radial_distance(zmin)
            Wz1s = 1.
            Wz2s = 1. / dchi / hzs
        return limber_integral(ells, zs, ks, Pgg, gzs, Wz1s, Wz2s, hzs, chis, device=self.device)

    def C_kk(self, ells, zs, ks, Pmm, lzs1=None, ldndz1=None, lzs2=None, ldndz2=None, lwindow1=None, lwindow2=None):
        own1 = lwindow1 is None
        if own1:
            lwindow1 = self.lensing_window(zs, lzs1, ldndz1)
        if lwindow2 is None:
            same = (own1 and ldndz1 is None and ldndz2 is None and lzs1 is not None and np.ndim(lzs1) == 0
                    and np.ndim(lzs2) == 0 and lzs1 == lzs2)
            lwindow2 = lwindow1 if same else self.lensing_window(zs, lzs2, ldndz2)     # the auto spectrum: one window
        chis = self.comoving_radial_distance(zs)
        hzs = self.h_of_z(zs)
        return limber_integral(ells, zs, ks, Pmm, zs, lwindow1, lwindow2, hzs, chis, device=self.device)

    def C_ky(self, ells, zs, ks, Pym, lzs1=None, ldndz1=None, lzs2=None, ldndz2=None, lwindow1=None):
        if lwindow1 is None:
            lwindow1 = self.lensing_window(zs, lzs1, ldndz1)
        chis = self.comoving_radial_distance(zs)
        hzs = self.h_of_z(zs)
        return limber_integral(ells, zs, ks, Pym, zs, lwindow1, 1, hzs, chis, device=self.device)

    def C_yy(self, ells, zs, ks, Ppp, dndz=None, zmin=None, zmax=None):
        chis = self.comoving_radial_distance(zs)
        hzs = self.h_of_z(zs)
        return limber_integral(ells, zs, ks, Ppp, zs, 1, 1, hzs, chis, device=self.device)

    def total_matter_power_spectrum(self, Pnn, Pne, Pee):
        omtoth2 = self.p['omch2'] + self.p['ombh2']
        fc = self.p['omch2'] / omtoth2
        fb = self.p['ombh2'] / omtoth2
        return fc ** 2. * Pnn + 2. * fc * fb * Pne + fb * fb * Pee


def a2z(a):
    return (1.0 / np.atleast_1d(a)) - 1.0


def _upload(a, device):
    a = np.asarray(a, dtype=np.float64)
    h = torch.empty(a.shape, dtype=torch.float64, pin_memory=True)
    if a.size:
        np.copyto(h.numpy(), a)
    capi.count_h2d(a.nbytes)
    return h.to(device, non_blocking=True)


def _upload_many(arrays, device):
    """Several small float64 vectors through ONE pinned staging block and ONE host->device copy (a copy per vector
    costs ~25 us of launch overhead each); returns device views, every one 16-byte aligned."""
    arrays = [np.asarray(a, dtype=np.float64).reshape(-1) for a in arrays]
    offs, n = [], 0
    for a in arrays:
        offs.append(n)
        n += (a.size + 1) & ~1
    h = torch.empty(max(n, 2), dtype=torch.float64, pin_memory=True)
    hv = h.numpy()
    for a, o in zip(arrays, offs):
        if a.size:
            hv[o:o + a.size] = a
    capi.count_h2d(8 * sum(a.size for a in arrays))
    d = h.to(device, non_blocking=True)
    return [d[o:o + a.size] for a, o in zip(arrays, offs)]


def _sort_order(x, name):
    """None when x is strictly increasing, else the permutation that sorts it; repeated values are an error."""
    if np.all(np.diff(x) > 0):
        return None
    order = np.argsort(x, kind="stable")
    if not np.all(np.diff(x[order]) > 0):
        raise ValueError("limber_integral: %s must not hold repeated values" % name)
    return order


def limber_integral(ells, zs, ks, Pzks, gzs, Wz1s, Wz2s, hzs, chis, device=None):
    r"""C(ell) = \int dz (H(z)/c) W1(z) W2(z) P(z, k=(ell+1/2)/chi) / chi^2   (cosmology.py:867-904) on the device.

    Pzks may be a numpy array [npzs,nk] or a CUDA tensor of that shape (kept on the device after an all-gather).
    ks and zs may come in any order (a HaloModel on shuffled ks hands out spectra in that order): the kernel looks
    them up by binary search, so they are sorted here and the table's columns and rows permuted to match, as the
    reference's interp2d does.  The window redshifts gzs are integrated over in the order given."""
    ells = np.asarray(ells, dtype=np.float64).reshape(-1)
    zs = np.asarray(zs, dtype=np.float64).reshape(-1)
    ks = np.asarray(ks, dtype=np.float64).reshape(-1)
    kord, zord = _sort_order(ks, "ks"), _sort_order(zs, "zs")
    device = torch.device(device) if device is not None else _default_device()
    gzs = np.asarray(gzs, dtype=np.float64).reshape(-1)
    hzs = np.array(hzs, dtype=np.float64).reshape(-1)
    chis = np.array(chis, dtype=np.float64).reshape(-1)
    with np.errstate(all="ignore"):
        pref = hzs * np.array(Wz1s, dtype=np.float64).reshape(-1) * np.array(Wz2s, dtype=np.float64).reshape(-1) / chis ** 2.
    pref = np.broadcast_to(pref, gzs.shape)

    if isinstance(Pzks, torch.Tensor):
        P_d = Pzks.to(device=device, dtype=torch.float64).contiguous()
    else:
        # the [nz,nk] table: arrays handed out by get_power live in pinned memory and go up at PCIe speed; anything
        # else is a pageable copy
        h = torch.from_numpy(np.ascontiguousarray(Pzks, dtype=np.float64))
        capi.count_h2d(h.numel() * 8)
        P_d = torch.empty(h.shape, dtype=torch.float64, device=device)
        P_d.copy_(h, non_blocking=h.is_pinned())
    if P_d.dim() != 2 or P_d.shape[0] != zs.size or P_d.shape[1] != ks.size:
        raise ValueError("Pzks must have shape (zs.size, ks.size)")
    if kord is not None or zord is not None:
        # one gather on the device puts the table in the sorted (z, k) order
        zi = np.arange(zs.size) if zord is None else zord
        ki = np.arange(ks.size) if kord is None else kord
        idx = torch.from_numpy((zi[:, None] * ks.size + ki[None, :]).reshape(-1)).to(device)
        capi.count_h2d(idx.numel() * 8)
        P_d = P_d.reshape(-1).index_select(0, idx).view(zs.size, ks.size)
        zs, ks = zs[zi], ks[ki]
    out = torch.empty(ells.size, dtype=torch.float64, device=device)
    # keep every temporary alive until the launch has been issued (the caching allocator may otherwise recycle it)
    ells_d, zs_d, ks_d, gzs_d, pref_d, chis_d = _upload_many((ells, zs, ks, gzs, pref, chis), device)
    capi.check(capi.lib.hmv_limber(ells.size, capi.ptr(ells_d), zs.size, ks.size, ks.size, capi.ptr(zs_d),
                                   capi.ptr(ks_d), capi.ptr(P_d), None, gzs.size, capi.ptr(gzs_d), capi.ptr(pref_d),
                                   capi.ptr(chis_d), capi.ptr(out), capi.stream()), "hmv_limber")
    capi.count_d2h(out.numel() * 8)
    h = torch.empty(out.shape, dtype=torch.float64, pin_memory=True)
    h.copy_(out, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return h.numpy()
