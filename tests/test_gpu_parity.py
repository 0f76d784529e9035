"""Parity of the CUDA path (through the drop-in HaloModel / C ABI) against the golden vectors produced by the
unmodified reference and against the CPU oracle.  Tolerance: rtol 1e-6 (FP64 kernels; BASELINE.json north_star) on
every [nz,nk] spectrum and [nz,nm] weight; u(k) cubes, which oscillate through zero, add an absolute floor of
1e-9 * max|cube| (u is O(1); the spectra built from them are still compared with pure rtol)."""
import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

OSC = 1e-9
# Occupations are 0.5*(1-erf(x)): where Nc < 1e-10 the result is a difference of two numbers that agree to 11+ digits,
# so one ulp of erf (CUDA libm vs cephes) is a 1e-5 relative change of a 1e-12 value.  Floor: 1e-14 * max|array|.
HOD_FLOOR = 1e-14
SPECTRA = [("mm", "nfw", "nfw"), ("ee", "electron", "electron"), ("me", "nfw", "electron"),
           ("gg", "g", "g"), ("gm", "g", "nfw"), ("ge", "g", "electron")]


@pytest.fixture(scope="module")
def hm():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    import hmvec_b200
    return hmvec_b200


@pytest.fixture(scope="module")
def mini(hm, golden_mini):
    g = golden_mini
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    return h


def test_background_and_plin(mini, golden_mini):
    g, h = golden_mini, mini
    assert_close(h.hubble_parameter(g["zs"]), g["hubble"], 1e-12)
    assert_close(h.comoving_radial_distance(g["zs"]), g["chi"], 1e-12)
    assert_close(h.rho_critical_z(g["zs"]), g["rho_crit"], 1e-12)
    assert_close(h.deltav(g["zs"]), g["deltav"], 1e-12)
    assert_close(h.Pzk, g["Pzk"], 1e-9, name="Pzk")
    assert_close(h.sPzk[:, ::10], g["sPzk_sub"], 1e-9, name="sPzk")


def test_mass_function(mini, golden_mini):
    g, h = golden_mini, mini
    assert_close(h.sigma2, g["sigma2"], 1e-9, name="sigma2")
    assert_close(h.nzm, g["nzm"], 1e-6, name="nzm")
    assert_close(h.bh, g["bh"], 1e-9, name="bh")
    assert_close(h.concentration(), g["cs"], 1e-12, name="cs")
    assert_close(h._rvir_d.cpu().numpy(), g["rvirs"], 1e-12, name="rvir")
    m200, _ = h._m200c_device()
    assert_close(m200.cpu().numpy(), g["m200c"], 1e-9, name="m200c")


def test_profiles(mini, golden_mini):
    g, h = golden_mini, mini
    assert_close(h.uk_profiles["nfw"], g["uk_nfw"], 1e-6, OSC, "uk_nfw")
    assert_close(h.uk_profiles["electron"], g["uk_e"], 1e-6, OSC, "uk_e")
    h.add_battaglia_profile("esh", family="SH", xmax=10, nxs=2000)
    assert_close(h.uk_profiles["esh"], g["uk_e_sh"], 1e-6, OSC, "uk_e_sh")
    h.add_battaglia_profile("eov", family="AGN", xmax=20, nxs=5000,
                            param_override={"battaglia_gas_gamma": -0.3, "rho0_A0": 3000., "alpha_alphaz": 0.25,
                                            "not_a_key": 1.0})
    assert_close(h.uk_profiles["eov"], g["uk_e_ov"], 1e-6, OSC, "uk_e_ov")
    h.add_nfw_profile("nfwnum", numeric=True, nxs=8000, xmax=100)
    assert_close(h.uk_profiles["nfwnum"], g["uk_nfwnum"], 1e-6, OSC, "uk_nfwnum")
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    assert_close(h.pk_profiles["y"], g["pk_y"], 1e-6, OSC, "pk_y")
    for tag, a, b in [("shsh", "esh", "esh"), ("ovm", "eov", "nfw")]:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)


def test_hod_and_spectra(mini, golden_mini):
    g, h = golden_mini, mini
    zs = g["zs"]
    h.add_hod("g2", ngal=g["g2_ngal_target"])
    h.add_hod("gmin", mthresh=10 ** (10.2 + 0.1 * zs), corr="min")
    for n in ("g", "g2", "gmin"):
        for k in ("Nc", "Ns", "NsNsm1", "NcNs", "ngal", "bg", "log10mthresh"):
            assert_close(h.hods[n][k], g["hod_%s_%s" % (n, k)], 1e-6, HOD_FLOOR, name="%s.%s" % (n, k))
    pairs = SPECTRA + [("g2g2", "g2", "g2"), ("g2e", "g2", "electron"), ("gming", "gmin", "gmin"),
                       ("gminm", "gmin", "nfw"), ("gg2", "g", "g2"), ("eg", "electron", "g")]
    for tag, a, b in pairs:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)
        assert_close(h.get_power(a, b), g["P1h_" + tag] + g["P2h_" + tag], 1e-6, name="P_" + tag)
    assert_close(h.get_power_2halo("g", "electron", b1_in=g["b1_in"], b2_in=g["b2_in"]), g["P2h_ge_bin"], 1e-6)
    p1, p2 = h.get_power_six("nfw", "electron", "g")
    for tag, _, _ in SPECTRA:
        assert_close(p1[tag], g["P1h_" + tag], 1e-6, name="six P1h_" + tag)
        assert_close(p2[tag], g["P2h_" + tag], 1e-6, name="six P2h_" + tag)


def test_central_profile_override_and_pressure_spectra(mini, golden_mini):
    g, h = golden_mini, mini
    zs = g["zs"]
    if "nfwnum" not in h.uk_profiles:
        h.add_nfw_profile("nfwnum", numeric=True, nxs=8000, xmax=100)
    if "y" not in h.pk_profiles:
        h.add_battaglia_pres_profile("y")
    h.add_hod("gcen", mthresh=10 ** 10.8 + zs * 0., central_profile_name="electron", satellite_profile_name="nfwnum")
    h.add_hod("gov", mthresh=10 ** 10.5 + zs * 0.,
              param_override={"hod_sig_log_mstellar": 0.3, "hod_alphasat": 1.1, "hod_Bsat": 8.0, "hod_betacut": 0.5})
    for n in ("gcen", "gov"):
        for k in ("Nc", "Ns", "NsNsm1", "ngal", "bg"):
            assert_close(h.hods[n][k], g["hod_%s_%s" % (n, k)], 1e-6, HOD_FLOOR, name="%s.%s" % (n, k))
    for tag, a, b in [("gcengcen", "gcen", "gcen"), ("gcene", "gcen", "electron"), ("govgov", "gov", "gov"),
                      ("yy", "y", "y"), ("ym", "y", "nfw"), ("yg", "y", "g"), ("nn", "nfwnum", "nfwnum")]:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)


def test_limber(mini, golden_mini):
    g, h = golden_mini, mini
    zs, ks, ells = g["zs"], g["ks"], g["ells"]
    Pmm = g["P1h_mm"] + g["P2h_mm"]
    Pgm = g["P1h_gm"] + g["P2h_gm"]
    Pgg = g["P1h_gg"] + g["P2h_gg"]
    Pyy = g["P1h_yy"] + g["P2h_yy"]
    assert_close(h.lensing_window(zs, 2.5), g["lens_window_25"], 1e-9)
    assert_close(h.lensing_window(zs, g["lz"], g["ldndz"]), g["lens_window_dndz"], 1e-9)
    assert_close(h.C_kk(ells, zs, ks, Pmm, lzs1=2.5, lzs2=2.5), g["C_kk"], 1e-6)
    assert_close(h.C_kg(ells, zs, ks, Pgm, gzs=0.8, lzs=2.5), g["C_kg"], 1e-6)
    assert_close(h.C_yy(ells, zs, ks, Pyy), g["C_yy"], 1e-6)
    assert_close(h.C_kk(ells, zs, ks, Pmm, lzs1=g["lz"], ldndz1=g["ldndz"], lzs2=1.1), g["C_kk_dndz"], 1e-6)
    assert_close(h.C_kg(ells, zs, ks, Pgm, gzs=g["gz"], gdndz=g["gdndz"], lzs=1100.), g["C_kg_dndz"], 1e-6)
    assert_close(h.C_gg(ells, zs, ks, Pgg, g["gz"], g["gdndz"]), g["C_gg_dndz"], 1e-6)


def test_mean_mdef(hm, golden_mini_mean):
    g = golden_mini_mean
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low', mdef='mean',
                     params={"omch2": 0.125, "H0": 70.0, "ns": 0.97, "st_a": 0.75, "kstar_damping": 0.02})
    h.add_battaglia_profile("electron", xmax=20, nxs=5000)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    assert_close(h.sigma2, g["sigma2"], 1e-9)
    assert_close(h.nzm, g["nzm"], 1e-6)
    assert_close(h.concentration(), g["cs"], 1e-12)
    assert_close(h.uk_profiles["nfw"], g["uk_nfw"], 1e-6, OSC)
    assert_close(h.uk_profiles["electron"], g["uk_e"], 1e-6, OSC)
    for tag, a, b in SPECTRA:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)


def test_readme_grid(hm, golden_readme):
    """C1-C3 (README.rst:55-84): zs[0]=0, 19-iteration ngal bisection."""
    g = golden_readme
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    assert_close(h.sigma2, g["sigma2"], 1e-9)
    assert_close(h.nzm, g["nzm"], 1e-6)
    assert_close(h.bh, g["bh"], 1e-9)
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    assert_close(h.uk_profiles["nfw"][:, ::8, ::4], g["uk_nfw_sub"], 1e-6, OSC)
    assert_close(h.uk_profiles["electron"][:, ::8, ::4], g["uk_e_sub"], 1e-6, OSC)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    h.add_hod("g2", ngal=g["g2_ngal_target"])
    assert h.hods["g2"]["iterations"] == 19
    for n in ("g", "g2"):
        for k in ("Nc", "Ns", "NsNsm1", "NcNs", "ngal", "bg", "log10mthresh"):
            assert_close(h.hods[n][k], g["hod_%s_%s" % (n, k)], 1e-6, HOD_FLOOR, name="%s.%s" % (n, k))
    for tag, a, b in SPECTRA + [("g2g2", "g2", "g2"), ("g2e", "g2", "electron")]:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)


def test_large_slab(hm, golden_largeslab):
    """Two redshifts at the LARGE grid's M and k resolution (2000 M x 10000 k)."""
    g = golden_largeslab
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    assert_close(h.sigma2, g["sigma2"], 1e-9)
    assert_close(h.nzm, g["nzm"], 1e-6)
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    assert_close(h.uk_profiles["nfw"][:, ::400], g["uk_nfw_rows"], 1e-6, OSC)
    assert_close(h.uk_profiles["electron"][:, ::400], g["uk_e_rows"], 1e-6, OSC)
    p1, p2 = h.get_power_six("nfw", "electron", "g")
    for tag, a, b in SPECTRA:
        assert_close(p1[tag], g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(p2[tag], g["P2h_" + tag], 1e-6, name="P2h_" + tag)
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="pair P1h_" + tag)


def test_known_answers(hm, golden_kat):
    """Device Si/Ci against scipy, and structural invariants the reference's code implies."""
    import torch
    from scipy.special import sici
    from hmvec_b200 import _capi as capi
    x = np.concatenate([np.geomspace(1e-8, 4.0, 4000), np.linspace(4.0, 60.0, 4000), np.geomspace(60, 1e6, 2000)])
    xd = torch.as_tensor(x, device="cuda")
    si, ci = torch.empty_like(xd), torch.empty_like(xd)
    capi.check(capi.lib.hmv_sici_test(x.size, capi.ptr(xd), capi.ptr(si), capi.ptr(ci), capi.stream()), "sici")
    S, Cc = sici(x)
    np.testing.assert_allclose(si.cpu().numpy(), S, rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(ci.cpu().numpy(), Cc, rtol=1e-12, atol=3e-15)


def test_bisection_continuation_round(hm, golden_mini):
    """A tight rtol needs more iterations than the first bisection round (24): the continuation round resumes from
    the saved brackets and must land on the same iteration count and midpoints as the reference's loop."""
    from oracle import hmvec_oracle as orc
    g = golden_mini
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low', skip_nfw=True)
    h.uk_profiles["nfw"] = np.ones((g["zs"].size, g["ms"].size, g["ks"].size))
    h.add_hod("gt", ngal=g["g2_ngal_target"], param_override={"hod_bisection_search_rtol": 1e-9})
    o = orc.OracleHaloModel(g["zs"], g["ks"], g["ms"], params={"hod_bisect_rtol": 1e-9}, skip_nfw=True)
    l10, iters = orc.hod_solve_mthresh(g["g2_ngal_target"], o.zs, o.ms, o.nzm, o.p)
    assert iters > 24
    assert h.hods["gt"]["iterations"] == iters
    assert_close(h.hods["gt"]["log10mthresh"][:, 0], l10, 1e-12, name="log10mthresh (rtol 1e-9)")


def test_two_halo_consistency_invariant(mini):
    """P2h(k->0) -> b1 b2 P_lin by construction of the consistency term (hmvec.py:566-572): at the lowest k the
    matter u(k) -> 1, so I - C -> 0 and P2h_mm -> Pzk."""
    p2 = mini.get_power_2halo("nfw", "nfw")
    np.testing.assert_allclose(p2[:, 0], mini.Pzk[:, 0], rtol=2e-3)


def test_errors(hm, mini):
    with pytest.raises(AssertionError):
        mini.add_battaglia_profile("nfw")
    with pytest.raises(AssertionError):
        mini.add_battaglia_profile("electron")
    with pytest.raises(ValueError):
        mini.add_hod("gbad", mthresh=np.ones(3))
    with pytest.raises(ValueError):
        mini.add_hod("gbad2", ngal=np.ones(3))
    with pytest.raises(ValueError):
        mini.add_hod("gbad3", mthresh=10 ** 10.5 + mini.zs * 0, param_override={"nope": 1})
    with pytest.raises(ValueError):
        mini.get_power_1halo("nfw", "doesnotexist")
    with pytest.raises(NotImplementedError):
        hm.HaloModel(mini.zs, mini.ks, ms=mini.ms, accuracy='low', mass_function="press-schechter")
    from hmvec_b200 import _capi as capi
    assert capi.lib.hmv_uk_nfw(0, 1, 1, 16, None, None, 1.0, None, None, None, None, None) == -1
    assert "bad sizes" in capi.last_error()


def test_unsorted_wavenumbers(hm, golden_mini):
    """The cube kernels take ks in any order (the reference's np.interp / elementwise maths do not care either):
    a shuffled k vector must give the shuffled spectra."""
    g = golden_mini
    rng = np.random.default_rng(0)
    perm = rng.permutation(g["ks"].size)
    h = hm.HaloModel(g["zs"], g["ks"][perm], ms=g["ms"], accuracy='low')
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    assert_close(h.uk_profiles["nfw"], g["uk_nfw"][:, :, perm], 1e-6, OSC, "uk_nfw (shuffled k)")
    assert_close(h.uk_profiles["electron"], g["uk_e"][:, :, perm], 1e-6, OSC, "uk_e (shuffled k)")
    for tag, a, b in SPECTRA:
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag][:, perm], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag][:, perm], 1e-6, name="P2h_" + tag)


def test_transform_ragged_grid_and_long_profile(hm):
    """Shapes the golden grids do not hold, against the CPU oracle: a mass axis that is not a multiple of the
    16-halo item (last item partly empty), an odd number of wavenumbers (scalar tail behind the 16-byte pairs),
    a k-range that starts above some halos' first bin and ends beyond the last bin of the big ones (all three
    interpolation zones), and a profile of ~2000 samples inside the theta-cut (three 704-sample chunks: the
    accumulate-then-normalise path)."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from oracle.hmvec_oracle import OracleHaloModel
    zs = np.array([0.0, 0.7, 2.5])
    ms = np.geomspace(3e10, 8e16, 37)
    ks = np.geomspace(2e-3, 4e3, 333)
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
    o = OracleHaloModel(zs, ks, ms)
    for name, kw in (("e5", dict(xmax=20, nxs=5000)), ("elong", dict(xmax=20, nxs=14000)), ("eodd", dict(xmax=15, nxs=3001))):
        h.add_battaglia_profile(name, family="AGN", **kw)
        o.add_battaglia_profile(name, family="AGN", **kw)
        assert_close(h.uk_profiles[name], o.uk_profiles[name], 1e-6, OSC, "uk_%s" % name)
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    o.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    assert_close(h.pk_profiles["y"], o.pk_profiles["y"], 1e-6, OSC, "pk_y")
    # numeric NFW at the package defaults (nxs=40000, xmax=200; params.py:59-60): a 20000-bin table per halo,
    # ~2000 samples inside the cut
    h.add_nfw_profile("nfwnum", numeric=True)
    o.add_nfw_profile("nfwnum", numeric=True)
    assert_close(h.uk_profiles["nfwnum"], o.uk_profiles["nfwnum"], 1e-6, OSC, "uk_nfwnum default")


def test_pk_spline_device(hm, golden_pkspline):
    """hmv_pk_spline (P(z,k) from a matter-power interpolator, SURVEY 8f-1) against the reference's own
    get_matter_power_interpolator_generic(...).P(z, k, grid=True): bicubic log-interpolation, power-law extension,
    sign-changing and negative tables, a 3-redshift (kx=2) table, scalar arguments, and a scipy spline handed over
    as CAMB's interpolator would be."""
    from conftest import PKSPLINE_CASES
    g = golden_pkspline
    gen = hm.utils.get_matter_power_interpolator_generic
    for key, tab, zq, kq, zt, kw in PKSPLINE_CASES:
        pk = -g[tab[1:]] if tab.startswith("-") else g[tab]
        PK = gen(g["ks_tab"], g[zt], pk, silent=True, **kw)
        assert_close(PK.P(g[zq], g[kq], grid=True), g[key], 1e-11, name=key)
    PK = gen(g["ks_tab"], g["zs_tab"], g["pk_tab"])
    assert (PK.kmin, PK.kmax, PK.zmin, PK.zmax) == (g["ks_tab"].min(), g["ks_tab"][-1], 0.0, 4.0) and PK.islog
    assert_close(PK.P(1.2345, g["kq"]), g["P_log_scalar_z"], 1e-11, name="P(z scalar, k)")
    assert np.isclose(PK.P(1.2345, 0.1), g["P_log_scalar_z"][np.argmin(np.abs(g["kq"] - 0.1))], rtol=0.2)
    # unsorted query points are fine on the device (scipy's grid=True refuses them)
    perm = np.random.default_rng(1).permutation(g["kq"].size)
    assert_close(PK.P(g["zq"][::-1], g["kq"][perm]), g["P_log"][::-1][:, perm], 1e-11, name="shuffled grid")
    # a scipy interpolator object (what camb.get_matter_power_interpolator returns) goes through from_spline
    from scipy.interpolate import RectBivariateSpline
    spl = RectBivariateSpline(g["zs_tab"], np.log(g["ks_tab"]), np.log(g["pk_tab"]))
    spl.islog, spl.logsign = True, 1
    c = hm.Cosmology(accuracy='low')
    assert_close(c._pk_grid(spl, g["zq"], g["kq"]), g["P_log"], 1e-11, name="from_spline")
    z3 = g["zs_tab3"]
    PK3 = gen(g["ks_tab"], z3, c.P_lin_approx(g["ks_tab"], z3))
    assert_close(PK3.P(g["zq3"], g["kq"]), g["P_kx2"], 1e-9, name="P_kx2")


def test_c_ky(hm, golden_cky):
    """tSZ x CMB lensing through the drop-in API (cosmology.py:585-589)."""
    g = golden_cky
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    assert_close(h.get_power_1halo("y", "nfw"), g["P1h_ym"], 1e-6, name="P1h_ym")
    assert_close(h.get_power_2halo("y", "nfw"), g["P2h_ym"], 1e-6, name="P2h_ym")
    Pym = h.get_power("y", "nfw")
    assert_close(h.C_ky(g["ells"], g["zs"], g["ks"], Pym, lzs1=2.5), g["C_ky"], 1e-6)
    assert_close(h.C_ky(g["ells"], g["zs"], g["ks"], Pym, lzs1=g["lz"], ldndz1=g["ldndz"]), g["C_ky_dndz"], 1e-6)
    h.add_hod("g", mthresh=10 ** 10.5 + g["zs"] * 0.0)
    assert_close(h.get_power("g", "g"), g["Pgg"], 1e-6, name="Pgg")
    assert_close(h.C_gg(g["ells"], g["zs"], g["ks"], g["Pgg"], 0.8, zmin=0.7, zmax=0.9), g["C_gg_tophat"], 1e-6)


@pytest.mark.parametrize("nz,nm,nk", [(1, 2, 1), (1, 16, 2), (2, 17, 31), (3, 33, 100), (5, 5, 257), (1, 48, 3)])
def test_small_and_degenerate_grids(hm, nz, nm, nk):
    """Edge shapes through the whole drop-in path against the CPU oracle: a single redshift, two masses (the minimum
    numpy.gradient accepts), one or two wavenumbers (no 16-byte pair / a single pair), mass counts around the 16-halo
    item size, and k grids shorter than one interpolation block."""
    from oracle.hmvec_oracle import OracleHaloModel
    zs = np.linspace(0.2, 2.2, nz) if nz > 1 else np.array([0.7])
    ms = np.geomspace(5e11, 3e15, nm)
    ks = np.geomspace(3e-3, 40.0, nk) if nk > 1 else np.array([0.5])
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
    o = OracleHaloModel(zs, ks, ms)
    assert_close(h.nzm, o.nzm, 1e-6, name="nzm")
    assert_close(h.uk_profiles["nfw"], o.uk_profiles["nfw"], 1e-6, OSC, "uk_nfw")
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    o.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    assert_close(h.uk_profiles["electron"], o.uk_profiles["electron"], 1e-6, OSC, "uk_e")
    h.add_hod("g", mthresh=10 ** 11.0 + zs * 0.0)
    o.add_hod("g", mthresh=10 ** 11.0 + zs * 0.0)
    for a, b in (("nfw", "nfw"), ("g", "electron"), ("electron", "electron")):
        assert_close(h.get_power_1halo(a, b), o.get_power_1halo(a, b), 1e-6, name="P1h %s %s" % (a, b))
        assert_close(h.get_power_2halo(a, b), o.get_power_2halo(a, b), 1e-6, name="P2h %s %s" % (a, b))
