"""CPU tests of the host-side mirrors: the free functions of hmvec.py:627-957 and tinker.py against values produced
by the unmodified reference (tests/golden/hostfuncs.npz, tinker.npz), the oracle's Tinker restatement against the
same fixture, and the export surface (`from hmvec_b200 import *` offers every public name of `from hmvec import *`)."""
import os
import re

import numpy as np
import pytest

from conftest import load_golden, assert_close, ROOT

# public def/class names of the reference's hmvec/hmvec.py (what `from .hmvec import *` in hmvec/__init__.py:1 exports
# besides re-exported modules); checked against the installed reference (oracle/_ref) when it is present
REFERENCE_NAMES = """HaloModel Fcon Mhalo_stellar Mhalo_stellar_core Mstellar_halo P_e P_e_generic P_e_generic_x R_from_M a2z avg_Nc
avg_NcNs avg_Ns avg_NsNsm1 battaglia_gas_fit duffy_concentration hod_default_mfunc mdelta_from_mdelta
mdelta_from_mdelta_unvectorized ngal_from_mthresh rho_gas rho_gas_generic rho_gas_generic_x rho_nfw rho_nfw_x
rhoscale_nfw Cosmology default_params battaglia_defaults tinker utils generic_profile_fft""".split()


@pytest.fixture(scope="module")
def hm():
    import warnings
    warnings.filterwarnings("ignore")
    import hmvec_b200
    return hmvec_b200


def test_export_surface(hm):
    names = set(REFERENCE_NAMES)
    ref = os.path.join(ROOT, "oracle", "_ref", "hmvec", "hmvec.py")
    if os.path.exists(ref):
        found = set(re.findall(r"^(?:def|class) (\w+)", open(ref).read(), re.M))
        assert found <= names, "REFERENCE_NAMES is stale: %s" % sorted(found - names)
    missing = sorted(n for n in names if not hasattr(hm, n))
    assert not missing, "hmvec_b200 lacks reference names: %s" % missing
    star = {}
    exec("from hmvec_b200 import *", star)
    assert not [n for n in names if n not in star], "not reachable through `from hmvec_b200 import *`"


def test_free_functions_match_reference(hm):
    g = load_golden("hostfuncs")
    z, lmh, thr = g["z"], g["log10mhalo"], g["thresh"]
    assert_close(hm.Mhalo_stellar(z[:, None], np.linspace(8., 12., 9)[None, :]), g["Mhalo_stellar"], 1e-13)
    assert_close(hm.Mstellar_halo(z[:, None], lmh), g["Mstellar_halo"], 1e-13)
    Nc = hm.avg_Nc(lmh, z[:, None], thr, 0.2)
    Ns = hm.avg_Ns(lmh, z[:, None], thr, Nc, 0.2, 1.0, 9.04, 0.74, 1.65, 0.59)
    assert_close(Nc, g["avg_Nc"], 1e-12, 1e-15)
    assert_close(Ns, g["avg_Ns"], 1e-12, 1e-15)
    for corr in ("max", "min"):
        assert_close(hm.avg_NsNsm1(Nc, Ns, corr), g["avg_NsNsm1_" + corr], 1e-12, 1e-15)
        assert_close(hm.avg_NcNs(Nc, Ns, corr), g["avg_NcNs_" + corr], 1e-12, 1e-15)
    assert_close(hm.hod_default_mfunc(np.array([11.5, 12.0, 13.0]), 9.04, 0.74), g["hod_default_mfunc"], 1e-14)
    ms, C1, d1, d2 = g["ms"], g["C1"], g["d1"], g["d2"]
    assert_close(hm.duffy_concentration(ms[None, :], z[:, None], 7.85, -0.081, -0.71, 0.673), C1, 1e-14)
    assert_close(hm.duffy_concentration(ms, 0.5), g["duffy_default"], 1e-14)
    assert_close(hm.mdelta_from_mdelta_unvectorized(ms[3], C1[1, 3], d1[1], d2[1]), g["mdelta_unvec"], 1e-9)
    assert_close(hm.mdelta_from_mdelta_unvectorized(ms[None, :] + 0 * C1, C1, d1[:, None], d2[:, None]), g["mdelta"], 1e-9)
    assert_close(hm.R_from_M(ms, 3e10, 200.), g["R_from_M"], 1e-14)
    assert_close(hm.Fcon(np.array([0.5, 4., 11.])), g["Fcon"], 1e-14)
    assert_close(hm.rho_nfw(np.array([0.1, 1., 3.]), 2e15, 0.4), g["rho_nfw"], 1e-14)
    x, m200 = g["x"], g["m200"]
    assert_close(hm.battaglia_gas_fit(m200, 0.7, 4000., 0.29, -0.66), g["battaglia_gas_fit"], 1e-14)
    assert_close(hm.rho_gas_generic_x(x[None, :], m200, 0.7, 0.049, 0.31, 1.5e11), g["rho_gas_generic_x"], 1e-13)
    assert_close(hm.rho_gas(x[None, :], m200, 0.7, 0.049, 0.31, 1.5e11, profile="SH"), g["rho_gas_SH"], 1e-13)
    assert_close(hm.P_e_generic_x(x[None, :], m200, 1.3, 0.7, 0.049, 0.31, 1.5e11), g["P_e_generic_x"], 1e-13)
    assert_close(hm.P_e(x[None, :], m200, 0.7, 0.049, 0.31, 1.5e11), g["P_e"], 1e-13)
    assert_close(hm.a2z(np.array([0.2, 0.5, 1.0])), g["a2z"], 1e-15)
    nzm = np.ones((4, lmh.shape[1]))
    got = hm.ngal_from_mthresh(thr[:, 0], z, nzm, 10 ** lmh[0], 0.2, alphasat=1.0, Bsat=9.04, betasat=0.74, Bcut=1.65,
                               betacut=0.59)
    trapz = getattr(np, "trapezoid", None) or np.trapz
    assert_close(got, trapz(g["avg_Nc"] + g["avg_Ns"], 10 ** lmh[0], axis=-1), 1e-12)


def test_tinker_module_and_oracle(hm):
    g = load_golden("tinker")
    t = hm.tinker
    nu, zs = g["kat_nu"], g["zs"]
    assert_close(t.bias(nu), g["kat_bias"], 1e-13)
    assert_close(t.f_nu(nu, zs[:, None]), g["kat_f_nu"], 1e-13)
    assert_close(t.f_nu(nu, zs[:, None], norm_consistency=False), g["kat_f_nu_nonorm"], 1e-13)
    assert_close(t.simple_f_nu(nu), g["kat_simple_f_nu"], 1e-13)
    assert_close(t.NlnMsub(np.geomspace(1e9, 1e13, 7), np.geomspace(1e12, 1e15, 5)), g["kat_NlnMsub"], 1e-13)
    with pytest.raises(ValueError):
        t.f_nu(nu, -0.1 + 0 * zs[:, None])
    # device-kernel input: nu f(nu) from the [nz,5] parameter rows must reproduce f_nu
    p = t.redshift_parameters(zs)
    al, be, ph, et, ga = (p[:, i][:, None] for i in range(5))
    assert_close(al * (1 + (be * nu) ** (-2 * ph)) * nu ** (2 * et) * np.exp(-ga * nu ** 2 / 2), g["kat_f_nu"], 1e-13)
    # oracle restatement of the tinker branch (hmvec.py:142-145,157-159) against the reference's arrays
    from oracle import hmvec_oracle as orc
    table = np.loadtxt(os.path.join(ROOT, "hmvec_b200", "data", "alpha_consistency.txt"), unpack=True)
    o = orc.OracleHaloModel(g["zs"], g["ks"], g["ms"], mdef="mean", skip_nfw=True, mass_function_mode="tinker",
                            alpha_table=table)
    assert_close(o.sigma2, g["sigma2"], 1e-10)
    assert_close(o.nzm, g["nzm"], 1e-9)
    assert_close(o.bh, g["bh"], 1e-10)
