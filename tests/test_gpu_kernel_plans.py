"""The reductions behind every spectrum, checked kernel by kernel against float64 host restatements of the same
operation on the same inputs, at the shapes that select each launch plan.

The golden-fixture tests pin the user-visible results at rtol 1e-6, and the kernel-vs-kernel tests share the
prep kernels, `trapz_weight` and the interpolation, so neither notices a dropped mass row, a misplaced tile seam or
a wrong tile classification whose effect on a physical grid stays below 1e-6.  Here every call goes through the C
ABI, so it is known which kernel ran, and the reference is a plain numpy reduction of the downloaded inputs:

* K5 mass integrals (`hmv_power_six`, `hmv_power` in its `power_pair_kernel` and `power_one_kernel` plans,
  `hmv_power_tab`, `hmv_power_six_tab`, `hmv_power_six_nfw`) against `oracle.hmvec_oracle.power_1halo` /
  `power_2halo`.  Inputs are seeded random -- cubes in [-0.3, 1.2] (sign changes), n(M), b(M) and the HOD moments of
  order one on every mass row, masses with O(1) trapezoid weights -- so that the last mass rows and every k column
  matter as much as any other.  One physical case (a 25-redshift slab from the pipeline) is a sanity check.
  Each element is held to an error bound rather than a bare rtol: |got - want| <= tau * B, where B is the same
  reduction over absolute values (|u|, and the 2-halo legs as I(|u|) + |b| + C, so the consistency subtraction is
  bounded by what was subtracted).  k* is set at the low end of ks, so the damping 1 - exp(-(k/k*)^2) is not itself a
  cancellation (device and numpy exp may differ in the last bit).
* sigma^2 (`hmv_sigma2`): the contraction against the W^2 table the kernel itself wrote (isolates the GEMM, split-k
  and the z tiles), and the whole result against a host W^2 @ sPzk (adds the top-hat window) at a pure rtol: every
  term is non-negative except the Cartwright correction of an even-length Simpson rule.
* HOD occupations, ngal, b_g and the all-z bisection at nm around the 1024-thread CTA width.
* K2, the analytic NFW cube (`hmv_uk_nfw`), against `oracle.hmvec_oracle.uk_nfw_analytic`, the reference's Si/Ci
  closed form in float64 (2.3e-14 absolute from 40-digit mpmath for 0.6 <= c <= 25), at inputs chosen so that every
  plan of the cube kernel runs (`_k2_plans` restates the kernel's choices and each case asserts the ones it is for).

Largest error-to-bound ratios measured on one B200 (1000 W power limit); the tolerances below keep about 10x headroom
over them and stay far below the effect of the faults these tests exist for (dropping the last mass row of the
random inputs moves the ratio to 0.3 - 1):

    power_six 6.7e-15 (incl. the physical slab), power_pair 4.3e-15, power_one 4.7e-15, power_six_tab 1.3e-15,
    power_tab 1.4e-15 -> tau = 7e-14;
    power_six_nfw 2.0e-12 -> tau = 2e-11: the in-kernel NFW evaluation and hmv_uk_nfw's cube are two evaluations of
    the same piecewise polynomials (t from (k a c)^2 or from k^2 (a c)^2, and near an interval edge one or the other
    interval's polynomial), which agree to ~1e-11 of max|u|, not to rounding;
    hmv_profile_expand vs np.interp 2.1e-16 of the row's max|u| -> 2e-15;
    sigma^2 against its own W^2 table 5.1e-15 -> rtol 5e-14; sigma^2 against the host window 3.0e-13 -> rtol 3e-12:
    the floor is the top-hat window's cancellation 3 (sin x - x cos x) / x^3 just above the Taylor switch x = 0.01
    (device and numpy sin / cos differ in the last bit, amplified by 1/x^2);
    HOD occupations 4.2e-13 -> rtol 4e-12 (above the 1e-14 max floor of N_c ~ 0); ngal and b_g 4.2e-16 -> 5e-15;
    uk_nfw 3.5e-13 of the row's max|u| -> tau = 4e-12: the polynomials' truncation error, not rounding.
The whole file runs in about 10 s and allocates under 0.4 GB of device memory.

Also here: NaN in the cube padding columns [nk, ldk) must not reach any output; outputs are written between NaN
guards (and, for the six-spectra kernels, with spec_stride > nz*nk and a poisoned gap between spectra) that must
survive bit for bit; every launch is repeated and must give bit-identical outputs."""
import ctypes as C

import numpy as np
import pytest

from conftest import assert_close

pytestmark = pytest.mark.gpu

TAU_K5 = 7e-14          # power_six / power_pair / power_one / power_six_tab / power_tab
TAU_NFW = 2e-11         # power_six_nfw against the hmv_uk_nfw cube (two evaluations of u_NFW)
TAU_K2 = 4e-12          # hmv_uk_nfw against the Si/Ci closed form, as a fraction of the row's max|u|
TOL_EXPAND = 2e-15      # hmv_profile_expand against np.interp, as a fraction of the row's max|u|
RTOL_SIGMA2_GEMM = 5e-14
RTOL_SIGMA2 = 3e-12
RTOL_HOD, HOD_FLOOR = 4e-12, 1e-14
RTOL_HOD_SUMS = 5e-15
SIX = ("mm", "ee", "me", "gg", "gm", "ge")
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64

OBSERVED = {}           # largest error-to-bound ratio seen per kernel in this session


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    from oracle import hmvec_oracle as orc
    return torch, capi, orc


def _dev(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def _vp(t, off=0):
    return C.c_void_p(t.data_ptr() + 8 * off)


def _ldk(nk):
    return (nk + 15) // 16 * 16


def _record(kind, ratio):
    OBSERVED[kind] = max(OBSERVED.get(kind, 0.0), float(ratio))


def _assert_bound(kind, name, got, want, bound, tau):
    got, want, bound = (np.asarray(a, dtype=np.float64) for a in (got, want, bound))
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    err = np.abs(got - want)
    zero = bound == 0.0
    assert np.all(err[zero] == 0.0), "%s: error where every term is zero" % name
    ratio = float(np.max(err[~zero] / bound[~zero])) if (~zero).any() else 0.0
    _record(kind, ratio)
    assert ratio <= tau, "%s: max |got-want| / sum|terms| = %.3g > %.1g" % (name, ratio, tau)


def _assert_rtol(kind, name, got, want, rtol):
    got, want = np.asarray(got), np.asarray(want)
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    ratio = float(np.max(np.abs(got - want) / np.abs(want)))
    _record(kind, ratio)
    assert ratio <= rtol, "%s: max relative error %.3g > %.1g" % (name, ratio, rtol)


class Out(object):
    """nspec outputs of nz*nk doubles, spectrum q at [q*stride, q*stride + n), between NaN guards."""

    def __init__(self, torch, nspec, n, stride=None):
        self.nspec, self.n, self.stride = nspec, n, stride or n
        self.buf = torch.full((2 * GUARD + nspec * self.stride,), float("nan"), dtype=torch.float64, device="cuda")
        self.ptr = _vp(self.buf, GUARD)
        keep = np.ones(self.buf.numel(), dtype=bool)
        for q in range(nspec):
            keep[GUARD + q * self.stride:GUARD + q * self.stride + n] = False
        self.poison = keep

    def host(self, shape):
        b = self.buf.cpu().numpy()
        assert np.all(b.view(np.int64)[self.poison] == NAN_BITS), "a guard or the gap between spectra was written"
        return np.stack([b[GUARD + q * self.stride:GUARD + q * self.stride + self.n].reshape(shape)
                         for q in range(self.nspec)])


def _twice(torch, launch, outs):
    """Launch, snapshot, launch again: every output (guards included) must be bit-identical."""
    launch()
    torch.cuda.synchronize()
    first = [o.buf.clone() for o in outs]
    launch()
    torch.cuda.synchronize()
    for a, o in zip(first, outs):
        assert torch.equal(a.view(torch.int64), o.buf.view(torch.int64)), "second launch differs"


# ------------------------------------------------------------------------------------------------- K5 inputs
def _k5_inputs(torch, nz, nm, nk, seed, ncube=2):
    """Seeded random inputs with O(1) weight on every mass row; cubes on the device with NaN padding columns."""
    rng = np.random.default_rng(seed)
    ldk = _ldk(nk)
    ms = 1e13 * (1.0 + np.cumsum(rng.uniform(0.5, 1.5, nm)) / nm)          # increasing, non-uniform spacing
    inp = dict(nz=nz, nm=nm, nk=nk, ldk=ldk, ms=ms, rho_m0=2e13,
               ks=np.geomspace(1e-2, 10.0, nk) if nk > 1 else np.array([0.3]),
               nzm=_flat_nzm(rng, ms, nz), bh=rng.uniform(0.5, 3.0, (nz, nm)), Pzk=rng.uniform(0.5, 2.0, (nz, nk)),
               hod=dict(Nc=rng.uniform(0.0, 1.0, (nz, nm)), Ns=rng.uniform(0.0, 2.0, (nz, nm)),
                        NcNs=rng.uniform(0.0, 2.0, (nz, nm)), NsNsm1=rng.uniform(0.0, 2.0, (nz, nm)),
                        ngal=rng.uniform(0.5, 2.0, nz)))
    inp["kstar"] = 0.5 * inp["ks"].min()
    inp["cubes"] = [rng.uniform(-0.3, 1.2, (nz, nm, nk)) for _ in range(ncube)]
    inp["d"] = {k: _dev(torch, inp[k]) for k in ("ms", "ks", "nzm", "bh", "Pzk")}
    inp["d"].update({k: _dev(torch, v) for k, v in inp["hod"].items()})
    inp["dcubes"] = [_cube(torch, c, ldk) for c in inp["cubes"]]
    return inp


def _flat_nzm(rng, ms, nz):
    """n(M) that gives every mass row a trapezoid weight w_m n(M) of order one."""
    wt = 0.5 * (np.r_[ms[1:], ms[-1]] - np.r_[ms[0], ms[:-1]])
    return rng.uniform(0.5, 2.0, (nz, ms.size)) / wt


def _cube(torch, c, ldk):
    t = torch.full(c.shape[:2] + (ldk,), float("nan"), dtype=torch.float64, device="cuda")
    t[..., :c.shape[2]] = _dev(torch, c)
    return t


# ------------------------------------------------------------------------------------------------- host references
def _leg_bound(orc, T, inp):
    """I(|u|) + |b| + C: what the 2-halo leg I + b - C is made of, in absolute value."""
    nzm, bh, ms, rho = inp["nzm"], inp["bh"], inp["ms"], inp["rho_m0"]
    I = orc._trapz(nzm[..., None] * np.abs(T.term(ms, rho)) * bh[..., None], ms[:, None], axis=-2)
    if T.kind == "pressure":
        return I
    Cc = orc._trapz(nzm[..., None] * np.abs(T.term(ms, rho, lowk=True)) * bh[..., None], ms[:, None], axis=-2)
    b = 1.0 if T.kind == "matter" else np.abs(orc.hod_bias(nzm, bh, ms, T.hod["Nc"], T.hod["Ns"], T.hod["ngal"]))[:, None]
    return I + b + Cc


def _abs(orc, T):
    return orc.Tracer(T.kind, None if T.u is None else np.abs(T.u), None if T.uc is None else np.abs(T.uc), T.hod)


def _pair_ref(orc, A, B, inp):
    """(P1h, P2h, bound1, bound2) of one tracer pair, [nz, nk] each."""
    args1 = (inp["nzm"], inp["ms"], inp["ks"], inp["rho_m0"], inp["kstar"])
    p1 = orc.power_1halo(A, B, *args1)
    b1 = orc.power_1halo(_abs(orc, A), _abs(orc, B), *args1)
    p2 = orc.power_2halo(A, B, inp["nzm"], inp["bh"], inp["ms"], inp["Pzk"], inp["rho_m0"])
    b2 = np.abs(inp["Pzk"]) * _leg_bound(orc, A, inp) * _leg_bound(orc, B, inp)
    return p1, p2, b1, b2


def _six_ref(orc, inp, um, ue):
    m, e = orc.Tracer("matter", um), orc.Tracer("matter", ue)
    g = orc.Tracer("hod", u=um, hod=inp["hod"])             # central profile 1, satellites follow u_m
    refs = [_pair_ref(orc, A, B, inp) for A, B in ((m, m), (e, e), (m, e), (g, g), (g, m), (g, e))]
    return [np.stack([r[i] for r in refs]) for i in range(4)]


def _check_six(kind, name, p1, p2, ref, tau):
    for q, tag in enumerate(SIX):
        _assert_bound(kind, "%s P1h_%s" % (name, tag), p1[q], ref[0][q], ref[2][q], tau)
        _assert_bound(kind, "%s P2h_%s" % (name, tag), p2[q], ref[1][q], ref[3][q], tau)


# ------------------------------------------------------------------------------------------------- K5 launchers
def _run_six(env, inp, stride_pad=37):
    """hmv_power_six on (cube 0, cube 1) with spec_stride > nz*nk; returns host (p1h, p2h) [6, nz, nk]."""
    torch, capi, _ = env
    nz, nm, nk, ldk, d = inp["nz"], inp["nm"], inp["nk"], inp["ldk"], inp["d"]
    S = nz * nk + stride_pad
    o1, o2 = Out(torch, 6, nz * nk, S), Out(torch, 6, nz * nk, S)
    ws = torch.empty(int(capi.lib.hmv_power_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")
    um, ue = inp["dcubes"][:2]
    L, p = capi.lib, capi.ptr

    def launch():
        capi.check(L.hmv_power_six(nz, nm, nk, ldk, p(d["ms"]), p(d["ks"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]),
                                   inp["rho_m0"], inp["kstar"], p(um), p(ue), p(d["Nc"]), p(d["Ns"]), p(d["NcNs"]),
                                   p(d["NsNsm1"]), p(d["ngal"]), p(ws), S, o1.ptr, o2.ptr, capi.stream()),
                   "hmv_power_six")
    _twice(torch, launch, (o1, o2))
    return o1.host((nz, nk)), o2.host((nz, nk))


def _tracer(capi, kind, us, uc=None, d=None):
    t = capi.Tracer()
    t.kind, t.us_d, t.uc_d = kind, us.data_ptr(), (uc.data_ptr() if uc is not None else None)
    if kind == 1:
        t.Nc_d, t.Ns_d, t.NcNs_d, t.NsNsm1_d, t.ngal_d = (d[k].data_ptr() for k in ("Nc", "Ns", "NcNs", "NsNsm1", "ngal"))
    return t


def _run_power(env, inp, A, B):
    """hmv_power with the C tracers A, B; returns host (p1h, p2h) [nz, nk]."""
    torch, capi, _ = env
    nz, nm, nk, ldk, d = inp["nz"], inp["nm"], inp["nk"], inp["ldk"], inp["d"]
    o1, o2 = Out(torch, 1, nz * nk), Out(torch, 1, nz * nk)
    ws = torch.empty(int(capi.lib.hmv_power_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")
    L, p = capi.lib, capi.ptr

    def launch():
        capi.check(L.hmv_power(nz, nm, nk, ldk, p(d["ms"]), p(d["ks"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]),
                               inp["rho_m0"], inp["kstar"], C.byref(A), C.byref(B), p(ws), o1.ptr, o2.ptr,
                               capi.stream()), "hmv_power")
    _twice(torch, launch, (o1, o2))
    return o1.host((nz, nk))[0], o2.host((nz, nk))[0]


def _check_kernel(env, inp, which, name):
    """One of the three cube-streaming plans on `inp` against the host reduction."""
    torch, capi, orc = env
    um, ue = inp["cubes"][:2]
    if which == "six":
        p1, p2 = _run_six(env, inp)
        _check_six("power_six", name, p1, p2, _six_ref(orc, inp, um, ue), TAU_K5)
        return
    d, dc = inp["d"], inp["dcubes"]
    if which == "one":              # one matter cube on both legs: power_one_kernel
        A = _tracer(capi, 0, dc[0])
        ref = _pair_ref(orc, orc.Tracer("matter", um), orc.Tracer("matter", um), inp)
        got = _run_power(env, inp, A, A)
    else:                           # matter x HOD with a central-profile cube: power_pair_kernel, three cubes
        A, B = _tracer(capi, 0, dc[0]), _tracer(capi, 1, dc[1], dc[2], d)
        ref = _pair_ref(orc, orc.Tracer("matter", um), orc.Tracer("hod", u=ue, uc=inp["cubes"][2], hod=inp["hod"]), inp)
        got = _run_power(env, inp, A, B)
    kind = "power_" + which
    _assert_bound(kind, name + " P1h", got[0], ref[0], ref[2], TAU_K5)
    _assert_bound(kind, name + " P2h", got[1], ref[1], ref[3], TAU_K5)


# ------------------------------------------------------------------------------------------------- K5: k and M extents
@pytest.mark.parametrize("which", ["six", "pair", "one"])
@pytest.mark.parametrize("nk", [1, 2, 447, 448, 449, 511, 512, 513, 1023, 1024, 1025, 10000])
def test_k5_k_extents(env, nk, which):
    """Every k-tile seam of the 512-wide (power_six, power_pair) and 1024-wide (power_one: two 512-column halves per
    thread) tiles, partial last tiles, and a 20-tile row."""
    inp = _k5_inputs(env[0], 2, 5, nk, seed=nk, ncube=3)
    _check_kernel(env, inp, which, "%s nk=%d" % (which, nk))


@pytest.mark.parametrize("which", ["six", "pair", "one"])
@pytest.mark.parametrize("nm", [2, 3, 4, 5, 1025, 2001])
def test_k5_mass_extents(env, nm, which):
    """Mass axes that end on a full stage and 1 / 2 / 3 rows into the last one (SIX_R = PR_R = ONE_R = 4), and long
    ones; nk = 600 has a partial second half of power_one's tile."""
    inp = _k5_inputs(env[0], 2, nm, 600, seed=1000 + nm, ncube=3)
    _check_kernel(env, inp, which, "%s nm=%d" % (which, nm))


@pytest.mark.parametrize("tile", [16, 448, 496, 512])
def test_power_six_tile_widths(env, monkeypatch, tile):
    """power_six_kernel at forced k-tile widths (HMV_TILE is read on every launch): narrow tiles, the 448 of a
    25-redshift slab on 148 SMs, a width that does not divide nk."""
    torch, capi, orc = env
    monkeypatch.setenv("HMV_TILE", str(tile))
    assert capi.lib.hmv_debug_wave_tile(3, _ldk(1025)) == tile
    inp = _k5_inputs(torch, 3, 6, 1025, seed=tile)
    p1, p2 = _run_six(env, inp)
    _check_six("power_six", "tile=%d" % tile, p1, p2, _six_ref(orc, inp, *inp["cubes"]), TAU_K5)


def test_power_six_natural_tile_of_a_slab(env, monkeypatch):
    """Without HMV_TILE, a 25-redshift slab of 10000 k (one rank of an 8-GPU run) takes 448-wide tiles on a 148-SM
    B200 (DESIGN section 5); the unforced launch at that shape against the host reduction."""
    torch, capi, orc = env
    monkeypatch.delenv("HMV_TILE", raising=False)
    tile = capi.lib.hmv_debug_wave_tile(25, 10000)
    if torch.cuda.get_device_properties(0).multi_processor_count == 148:
        assert tile == 448
    inp = _k5_inputs(torch, 25, 3, 10000, seed=25)
    assert inp["ldk"] == 10000
    p1, p2 = _run_six(env, inp)
    _check_six("power_six", "natural tile %d" % tile, p1, p2, _six_ref(orc, inp, *inp["cubes"]), TAU_K5)


def test_power_pair_four_cubes_and_pressure_pair(env):
    """power_pair_kernel with three and four distinct cubes at nk > 512 (HOD with a central-profile cube x an electron
    tracer; HOD x HOD with their own satellite and central cubes), and the pressure x pressure two-pass branch
    (1-halo from leg A alone, 2-halo from both legs)."""
    torch, capi, orc = env
    inp = _k5_inputs(torch, 3, 37, 1300, seed=77, ncube=4)
    d, dc, c, hod = inp["d"], inp["dcubes"], inp["cubes"], inp["hod"]
    cases = [("hod(us,uc) x electron", _tracer(capi, 1, dc[0], dc[1], d), _tracer(capi, 0, dc[2]),
              orc.Tracer("hod", u=c[0], uc=c[1], hod=hod), orc.Tracer("matter", c[2])),
             ("hod(us,uc) x hod(us',uc')", _tracer(capi, 1, dc[0], dc[1], d), _tracer(capi, 1, dc[2], dc[3], d),
              orc.Tracer("hod", u=c[0], uc=c[1], hod=hod), orc.Tracer("hod", u=c[2], uc=c[3], hod=hod)),
             ("pressure x pressure", _tracer(capi, 2, dc[0]), _tracer(capi, 2, dc[3]),
              orc.Tracer("pressure", c[0]), orc.Tracer("pressure", c[3]))]
    for name, A, B, TA, TB in cases:
        got = _run_power(env, inp, A, B)
        ref = _pair_ref(orc, TA, TB, inp)
        _assert_bound("power_pair", name + " P1h", got[0], ref[0], ref[2], TAU_K5)
        _assert_bound("power_pair", name + " P2h", got[1], ref[1], ref[3], TAU_K5)


def test_power_six_physical_slab(env):
    """Sanity check on physical inputs: the NFW and electron cubes, n(M), b(M) and HOD of a 25-redshift pipeline slab."""
    torch, capi, orc = env
    from hmvec_b200 import pipeline
    zs = np.linspace(0.05, 3.0, 25)
    g = pipeline.GridSix(pipeline.make_inputs(zs, np.geomspace(1e11, 5e15, 150), np.geomspace(1e-3, 30.0, 700)),
                         tsz=False)
    g.upload(); g.run(); torch.cuda.synchronize()
    host = {k: g.d[k].cpu().numpy() for k in ("ms", "ks", "nzm", "bh", "Pzk", "Nc", "Ns", "NcNs", "NsNsm1", "ngal")}
    inp = dict(nz=g.nz, nm=g.nm, nk=g.nk, ldk=g.ldk, rho_m0=g.rho_m0, kstar=float(host["ks"].min()),
               d={k: g.d[k] for k in host}, dcubes=[g.um, g.ue],
               hod={k: host[k] for k in ("Nc", "Ns", "NcNs", "NsNsm1", "ngal")},
               **{k: host[k] for k in ("ms", "ks", "nzm", "bh", "Pzk")})
    um, ue = (c[..., :g.nk].cpu().numpy() for c in (g.um, g.ue))
    p1, p2 = _run_six(env, inp)
    _check_six("power_six", "physical slab", p1, p2, _six_ref(orc, inp, um, ue), TAU_K5)


def test_power_six_nfw_multi_tile(env):
    """power_six_nfw_kernel (NFW evaluated inside the reduction, k tiles highest first) with three k tiles, against
    the host reduction over the hmv_uk_nfw cube of the same halos."""
    torch, capi, orc = env
    nz, nm, nk = 3, 45, 1100
    rng = np.random.default_rng(11)
    inp = _k5_inputs(torch, nz, nm, nk, seed=11)
    inp["ks"] = np.geomspace(1e-3, 200.0, nk)
    inp["kstar"] = 0.5e-3
    d = inp["d"]
    d["ks"] = _dev(torch, inp["ks"])
    zs, cs, rv = np.array([0.1, 1.0, 2.5]), rng.uniform(1.0, 20.0, (nz, nm)), rng.uniform(0.05, 3.0, (nz, nm))
    dz, dcs, drv = _dev(torch, zs), _dev(torch, cs), _dev(torch, rv)
    ldk, L, p = inp["ldk"], capi.lib, capi.ptr
    um = torch.zeros((nz, nm, ldk), dtype=torch.float64, device="cuda")
    ws = torch.empty(int(L.hmv_uk_nfw_ws_doubles(nz, nm, nk)), dtype=torch.float64, device="cuda")
    capi.check(L.hmv_uk_nfw(nz, nm, nk, ldk, p(dz), p(d["ks"]), float(inp["ks"].max()), p(dcs), p(drv), p(ws), p(um),
                            capi.stream()), "hmv_uk_nfw")
    S = nz * nk + 19
    o1, o2 = Out(torch, 6, nz * nk, S), Out(torch, 6, nz * nk, S)
    ws2 = torch.empty(int(L.hmv_power_six_nfw_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")
    ue = inp["dcubes"][1]

    def launch():
        capi.check(L.hmv_power_six_nfw(nz, nm, nk, ldk, p(dz), p(d["ms"]), p(d["ks"]), p(d["nzm"]), p(d["bh"]),
                                       p(d["Pzk"]), inp["rho_m0"], inp["kstar"], p(dcs), p(drv), p(ue), p(d["Nc"]),
                                       p(d["Ns"]), p(d["NcNs"]), p(d["NsNsm1"]), p(d["ngal"]), p(ws2), S, o1.ptr,
                                       o2.ptr, capi.stream()), "hmv_power_six_nfw")
    _twice(torch, launch, (o1, o2))
    ref = _six_ref(orc, inp, um[..., :nk].cpu().numpy(), inp["cubes"][1])
    _check_six("power_six_nfw", "six_nfw", o1.host((nz, nk)), o2.host((nz, nk)), ref, TAU_NFW)


# ------------------------------------------------------------------------------------------------- K5 from bin tables
def _expand_host(tab, meta, ks, J):
    """np.interp expansion of bin tables onto ks (fft.py:102-107): hold u_1 below bin 1, zero above bin J."""
    nz, nm = meta.shape[:2]
    out = np.empty((nz, nm, ks.size))
    for z in range(nz):
        for m in range(nm):
            inv, u1, jn = meta[z, m, 0], meta[z, m, 1], int(meta[z, m, 2])
            n = min(J, jn)
            t = ks * inv
            assert np.all((t <= n) | (t > J)), "a wavenumber needs a bin the transform did not write"
            j = np.arange(1, n + 1, dtype=np.float64)
            out[z, m] = np.interp(t, j, tab[z, m, 1:n + 1], left=u1, right=0.0)
    return out


def _tables(env, g, which, ks, nxs):
    """hmv_profile_tables of the pipeline's electron (mass-normalised) or pressure profiles on `ks`."""
    torch, capi, _ = env
    L, d, p = capi.lib, g.d, capi.ptr
    pre = "" if which == "electron" else "y_"
    gamma = g.gamma if which == "electron" else float(g.p['battaglia_pres_gamma'])
    nz, nm = g.nz, g.nm
    dks = _dev(torch, ks)
    tab = torch.zeros(int(L.hmv_profile_table_doubles(nz, nm, nxs)), dtype=torch.float64, device="cuda")
    ws = torch.empty(int(L.hmv_profile_transform_ws_doubles(nz, nm, nxs)), dtype=torch.float64, device="cuda")
    capi.check(L.hmv_profile_tables(nz, nm, ks.size, p(d["zs"]), p(dks), float(ks.max()), p(d[pre + "rs"]),
                                    p(d[pre + "cmax"]), p(d[pre + "xc"]), p(d[pre + "alpha"]), p(d[pre + "expo"]),
                                    p(d[pre + "amp"]), p(d[pre + "oscale"]), gamma, 20.0, nxs,
                                    1 if which == "electron" else 0, p(ws), p(tab), capi.stream()), "hmv_profile_tables")
    JS, nmp = int(L.hmv_profile_table_stride(nxs)), (nm + 15) // 16 * 16
    h = tab.cpu().numpy()
    rows = h[:nz * nmp * JS].reshape(nz, nmp, JS)[:, :nm]
    meta = h[nz * nmp * JS:nz * nmp * (JS + 4)].reshape(nz, nmp, 4)[:, :nm]
    return dict(tab=tab, rows=rows, meta=meta, ws=ws, dks=dks, J=nxs // 2)


@pytest.fixture(scope="module")
def tab_grid(env):
    """Pressure and electron GNFW parameters from the pipeline (masses 1e10..1e16 Msun: first-bin wavenumbers over
    two decades), tables with nxs = 100 (J = 50 bins), and a 1600-point k axis (four 512-wide tiles) placed so that in
    its second tile some halos lie wholly below their first bin, some wholly above their last and the rest in between."""
    torch, capi, _ = env
    from hmvec_b200 import pipeline
    zs, nxs = np.array([0.2, 0.6]), 100
    g = pipeline.GridSix(pipeline.make_inputs(zs, np.geomspace(1e10, 1e16, 61), np.geomspace(1e-2, 10.0, 64),
                                              ngal=np.array([1e-3, 1e-4])))
    g.upload(); g.run(); torch.cuda.synchronize()
    k1 = 1.0 / _tables(env, g, "pressure", np.geomspace(1e-2, 10.0, 64), nxs)["meta"][0, :, 0]   # first-bin k, z = 0
    lo, hi = np.log(nxs // 2 * k1.min()), np.log(k1.max())
    assert hi - lo > 0.3
    step = 0.5 * (hi - lo) / 511
    ks = np.exp(lo + 0.25 * (hi - lo) + (np.arange(1600) - 512) * step)
    return g, ks, nxs


def _classes(meta, ks, J, tile=512):
    """Per (z, tile): numbers of halos below the first bin, above the last, interpolated, and switching inside."""
    out = []
    for z in range(meta.shape[0]):
        inv = meta[z, :, 0]
        for k0 in range(0, ks.size, tile):
            kk = ks[k0:k0 + tile]
            tlo, thi = kk.min() * inv, kk.max() * inv
            below, above = thi < 1.0, tlo > J
            switch = ((tlo < 1.0) & (thi >= 1.0)) | ((tlo <= J) & (thi > J))
            out.append((z, k0, int(below.sum()), int(above.sum()), int((~below & ~above).sum()), int(switch.sum())))
    return out


@pytest.mark.parametrize("order", ["sorted", "shuffled"])
def test_power_tab_tiles_and_classes(env, tab_grid, order):
    """power_one_tab_kernel (P_yy from tables) over four k tiles in its descending launch order: per-tile halo
    classification (hold u_1 / zero / interpolate), with a tile holding all three classes and tiles in which a halo
    changes class; the expansion hmv_profile_expand writes is checked against the same host expansion."""
    torch, capi, orc = env
    g, ks, nxs = tab_grid
    if order == "shuffled":
        ks = np.random.default_rng(3).permutation(ks)
    T = _tables(env, g, "pressure", ks, nxs)
    J, nz, nm, nk = T["J"], g.nz, g.nm, ks.size
    cls = _classes(T["meta"], ks, J)
    if order == "sorted":
        assert any(b and a and i for _, _, b, a, i, _ in cls), cls
        assert any(s for *_, s in cls), cls
    u = _expand_host(T["rows"], T["meta"], ks, J)
    ldk = _ldk(nk)
    cube = torch.full((nz, nm, ldk), float("nan"), dtype=torch.float64, device="cuda")
    L, p, d = capi.lib, capi.ptr, g.d
    capi.check(L.hmv_profile_expand(nz, nm, nk, ldk, p(d["zs"]), p(T["dks"]), float(ks.max()), p(d["y_rs"]), 20.0, nxs,
                                    p(T["ws"]), p(T["tab"]), p(cube), capi.stream()), "hmv_profile_expand")
    ce = cube[..., :nk].cpu().numpy()
    scale = np.abs(T["rows"]).max(axis=-1, keepdims=True)
    ratio = float(np.max(np.abs(ce - u) / scale))
    _record("profile_expand", ratio)
    assert ratio <= TOL_EXPAND, "hmv_profile_expand vs host np.interp: %.3g of max|u|" % ratio
    rng = np.random.default_rng(8)
    inp = dict(nz=nz, nm=nm, nk=nk, ms=g.d["ms"].cpu().numpy(), rho_m0=g.rho_m0, ks=ks,
               nzm=_flat_nzm(rng, g.d["ms"].cpu().numpy(), nz), bh=rng.uniform(0.5, 3.0, (nz, nm)),
               Pzk=rng.uniform(0.5, 2.0, (nz, nk)))
    inp["kstar"] = 0.5 * ks.min()
    dd = {k: _dev(torch, inp[k]) for k in ("ms", "nzm", "bh", "Pzk")}
    o1, o2 = Out(torch, 1, nz * nk), Out(torch, 1, nz * nk)
    ws = torch.empty(int(L.hmv_power_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")

    def launch():
        capi.check(L.hmv_power_tab(nz, nm, nk, p(dd["ms"]), p(T["dks"]), p(dd["nzm"]), p(dd["bh"]), p(dd["Pzk"]),
                                   inp["rho_m0"], inp["kstar"], 2, p(T["tab"]), nxs, p(ws), o1.ptr, o2.ptr,
                                   capi.stream()), "hmv_power_tab")
    _twice(torch, launch, (o1, o2))
    y = orc.Tracer("pressure", u)
    ref = _pair_ref(orc, y, y, inp)
    _assert_bound("power_tab", order + " P1h_yy", o1.host((nz, nk))[0], ref[0], ref[2], TAU_K5)
    _assert_bound("power_tab", order + " P2h_yy", o2.host((nz, nk))[0], ref[1], ref[3], TAU_K5)


@pytest.mark.parametrize("order", ["sorted", "shuffled"])
def test_power_six_tab_tiles(env, tab_grid, order):
    """power_six_tab_kernel (electron profile interpolated from its tables inside the reduction) over four k tiles,
    against the host expansion of the downloaded tables reduced on the host."""
    torch, capi, orc = env
    g, ks, nxs = tab_grid
    if order == "shuffled":
        ks = np.random.default_rng(4).permutation(ks)
    T = _tables(env, g, "electron", ks, nxs)
    nz, nm, nk = g.nz, g.nm, ks.size
    ue = _expand_host(T["rows"], T["meta"], ks, T["J"])
    inp = _k5_inputs(torch, nz, nm, nk, seed=21, ncube=1)
    ms = g.d["ms"].cpu().numpy()
    inp.update(ks=ks, kstar=0.5 * ks.min(), ms=ms, nzm=_flat_nzm(np.random.default_rng(22), ms, nz))
    d, ldk, L, p = inp["d"], inp["ldk"], capi.lib, capi.ptr
    d["ms"], d["ks"], d["nzm"] = g.d["ms"], T["dks"], _dev(torch, inp["nzm"])
    S = nz * nk + 5
    o1, o2 = Out(torch, 6, nz * nk, S), Out(torch, 6, nz * nk, S)
    ws = torch.empty(int(L.hmv_power_six_tab_ws_doubles(nz, nm, nk)), dtype=torch.float64, device="cuda")

    def launch():
        capi.check(L.hmv_power_six_tab(nz, nm, nk, ldk, p(d["ms"]), p(d["ks"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]),
                                       inp["rho_m0"], inp["kstar"], p(inp["dcubes"][0]), p(T["tab"]), nxs, p(d["Nc"]),
                                       p(d["Ns"]), p(d["NcNs"]), p(d["NsNsm1"]), p(d["ngal"]), p(ws), S, o1.ptr,
                                       o2.ptr, capi.stream()), "hmv_power_six_tab")
    _twice(torch, launch, (o1, o2))
    ref = _six_ref(orc, inp, inp["cubes"][0], ue)
    _check_six("power_six_tab", "six_tab " + order, o1.host((nz, nk)), o2.host((nz, nk)), ref, TAU_K5)


# ------------------------------------------------------------------------------------------------- sigma^2
def _sigma2_splits(nz, nm, nks, allz):
    """sigma2_splits of k_sigma2.cu restated: the split-k factor of each launch plan."""
    cd = lambda a, b: -(-a // b)
    if allz:
        mt = 4 if nz <= 32 else 8 if nz <= 64 else 16 if nz <= 128 else 26
        s = (148 * (1 if mt > 16 else 2) * 2) // (cd(nm, 64) * cd(nz, 8 * mt))
    else:
        s = cd(16 * 148, cd(nm, 64) * cd(nz, 32))
    return int(min(max(s, 1), 32, cd(nks, 16)))


SIGMA2_CASES = [  # (nz, nm, nks, misaligned sPzk, expected split-k > 1)
    (1, 130, 512, False, True), (32, 130, 512, False, True), (33, 130, 512, False, True),
    (64, 130, 512, False, True), (65, 130, 512, False, True), (128, 130, 512, False, True),
    (129, 130, 512, False, True), (208, 130, 512, False, True), (209, 130, 512, False, True),
    (417, 130, 512, False, True),
    (417, 6336, 512, False, False),          # 3 z tiles x 99 mass strips > 296 resident CTAs: no split
    (417, 130, 16, False, False),            # one k chunk
    (33, 131, 512, False, True),             # odd nm: sigma2_gemm_plain_kernel
    (33, 130, 511, False, True),             # odd nks: plain
    (65, 130, 512, True, True),              # sPzk 8 bytes off 16-byte alignment: plain
    (40, 131, 15, False, False),             # plain, one k chunk
]


@pytest.mark.parametrize("nz,nm,nks,misaligned,split", SIGMA2_CASES)
def test_sigma2_plans(env, nz, nm, nks, misaligned, split):
    """hmv_sigma2 in every plan: sigma2_gemm_kernel<MT> for MT = 4 / 8 / 16 / 26 with one to three z tiles, the plain
    fallback (odd nm, odd nks, misaligned input), split-k with the fixed-order reduction and without."""
    torch, capi, orc = env
    from hmvec_b200.cosmology import simpson_weights
    allz = nm % 2 == 0 and nks % 2 == 0 and not misaligned
    assert (_sigma2_splits(nz, nm, nks, allz) > 1) == split
    rng = np.random.default_rng(nz * 7 + nm + nks)
    ks = np.geomspace(1e-4, 2000.0, nks)
    kw = simpson_weights(ks) * ks ** 2 / 2.0 / np.pi ** 2
    R = (3.0 * np.geomspace(1e10, 1e16, nm) / 4.0 / np.pi / 4e10) ** (1.0 / 3.0)
    sP = rng.uniform(0.5, 2.0, (nz, 1)) * ks / (1.0 + (ks / 0.02) ** 2.6)
    buf = torch.full((nz * nks + 2,), float("nan"), dtype=torch.float64, device="cuda")
    off = 1 if misaligned else 0
    buf[off:off + nz * nks] = _dev(torch, sP.ravel())
    L, p = capi.lib, capi.ptr
    dk, dkw, dR = _dev(torch, ks), _dev(torch, kw), _dev(torch, R)
    ws = torch.empty(int(L.hmv_sigma2_ws_doubles(nz, nm, nks)), dtype=torch.float64, device="cuda")
    out = Out(torch, 1, nz * nm)

    def launch():
        capi.check(L.hmv_sigma2(nz, nm, nks, _vp(buf, off), p(dkw), p(dk), p(dR), 0.01, p(ws), out.ptr,
                                capi.stream()), "hmv_sigma2")
    _twice(torch, launch, (out,))
    got = out.host((nz, nm))[0]
    w2t = ws[:nks * nm].cpu().numpy().reshape(nks, nm)
    _assert_rtol("sigma2_gemm", "sigma2 vs its W^2 table", got, sP @ w2t, RTOL_SIGMA2_GEMM)
    W2 = orc.tophat_window(ks[:, None] * R[None, :], 0.01) ** 2 * kw[:, None]
    _assert_rtol("sigma2", "sigma2 vs host W^2 @ sPzk", got, sP @ W2, RTOL_SIGMA2)


# ------------------------------------------------------------------------------------------------- HOD
def _hod_inputs(nm):
    zs = np.array([0.3, 1.2])
    ms = np.geomspace(1e10, 1e16, nm)
    nzm = (ms / 1e12) ** -1.9 / 1e12 * np.exp(-ms / 5e14) * (1.0 + zs[:, None]) ** -1
    return zs, ms, nzm, 1.0 + (ms / 1e13) ** 0.5 + 0.0 * zs[:, None]


@pytest.mark.parametrize("nm", [1023, 1024, 1025, 2000])
def test_hod_around_cta_width(env, nm):
    """hod_kernel and hod_bisect_kernel (one 1024-thread CTA per redshift, strided mass loops) at nm below, at and
    above the CTA width: occupations, ngal and b_g against the oracle; the all-z bisection's log10 mthresh and its
    iteration count against oracle.hod_solve_mthresh."""
    torch, capi, orc = env
    hp = dict(orc.DEFAULTS)
    zs, ms, nzm, bh = _hod_inputs(nm)
    l10 = np.array([10.6, 11.1])
    L, p, st = capi.lib, capi.ptr, capi.stream()
    dz, dm, dn, db, dl = (_dev(torch, a) for a in (zs, ms, nzm, bh, l10))
    hodp = capi.darr([hp[k] for k in ("hod_sig_log_mstellar", "hod_alphasat", "hod_Bsat", "hod_betasat", "hod_Bcut",
                                      "hod_betacut")] + [0.0, 0.0])
    outs = [Out(torch, 1, zs.size * nm) for _ in range(4)] + [Out(torch, 1, zs.size) for _ in range(2)]

    def launch():
        capi.check(L.hmv_hod(zs.size, nm, p(dz), p(dm), p(dl), hodp, 0, p(dn), p(db), *(o.ptr for o in outs), st),
                   "hmv_hod")
    _twice(torch, launch, outs)
    got = [o.host((zs.size, nm) if i < 4 else (zs.size,))[0] for i, o in enumerate(outs)]
    want = orc.hod_occupations(zs, ms, l10, hp, "max")
    for name, a, b in zip(("Nc", "Ns", "NsNsm1", "NcNs"), got[:4], want):
        assert_close(a, b, RTOL_HOD, HOD_FLOOR, name="%s nm=%d" % (name, nm))
        big = np.abs(b) > HOD_FLOOR * np.abs(b).max() / RTOL_HOD
        if big.any():
            _record("hod_occupations", np.max(np.abs(a - b)[big] / np.abs(b)[big]))
    ngal = orc.hod_ngal(nzm, ms, want[0], want[1])
    _assert_rtol("hod_ngal", "ngal nm=%d" % nm, got[4], ngal, RTOL_HOD_SUMS)
    bg = orc.hod_bias(nzm, bh, ms, want[0], want[1], ngal)
    _assert_rtol("hod_ngal", "bg nm=%d" % nm, got[5], bg, RTOL_HOD_SUMS)
    # the bisection: targets from the host ngal at other thresholds
    target = orc.hod_ngal(nzm, ms, *orc.hod_occupations(zs, ms, np.array([10.23, 11.71]), hp)[:2])
    l10_want, it_want = orc.hod_solve_mthresh(target, zs, ms, nzm, hp)
    dt = _dev(torch, target)
    ws = torch.zeros(zs.size * (capi.HMV_BISECT_MAXIT + 4), dtype=torch.float64, device="cuda")
    res, iters = Out(torch, 1, zs.size), torch.zeros(1, dtype=torch.int32, device="cuda")
    capi.check(L.hmv_hod_solve(zs.size, nm, p(dz), p(dm), p(dn), p(dt), hodp, hp["hod_bisect_lo"], hp["hod_bisect_hi"],
                               hp["hod_bisect_rtol"], hp["hod_A_log10mthresh"], p(ws), res.ptr, p(iters), st),
               "hmv_hod_solve")
    torch.cuda.synchronize()
    assert int(iters[0]) == it_want
    assert_close(res.host((zs.size,))[0], l10_want, 1e-12, name="log10mthresh nm=%d" % nm)


# ------------------------------------------------------------------------------------------------- K2: the NFW cube
NFWP_HI = 1.005 * np.array([1, 2, 4, 6, 8, 10, 12, 14, 16, 20, 24, 28, 32, 36, 40, 44, 48, 52, 56, 60, 64.0])
NFWP_NI, NFW_CH = 21, 256


def _nfwp_interval(s):
    """nfwp_interval of nfw_poly.cuh: the polynomial interval of s = x c (NFWP_NI: beyond s = 64)."""
    si = np.floor(np.minimum(s, 1e6)).astype(np.int64)
    return np.where(si < 1, 0, np.where(si < 2, 1, np.where(si < 16, 1 + (si >> 1),
                                                            np.where(si < 64, 5 + (si >> 2), NFWP_NI))))


def _k2_plans(ks, sr, xr):
    """The plans uk_nfw_poly_kernel takes (k_nfw.cu restated) over all halo rows, s = k sr and x = k xr per row:
    the leading run below s = 1 (fast), a chunk inside one interval (one), a chunk over several (several) with pairs
    that straddle an edge or reach s = 64 (redo), whole chunks beyond s = 64 with every x > 4 (far) or some x <= 4
    (near)."""
    nch = -(-ks.size // NFW_CH)
    kp = np.concatenate([ks, np.full(nch * NFW_CH - ks.size, ks[-1])]).reshape(nch, NFW_CH)  # as nfw_chunk_kernel pads
    kmin, kmax = kp.min(axis=1), kp.max(axis=1)
    sr, xr = sr.ravel()[:, None], xr.ravel()[:, None]
    smin, smax = kmin * sr, kmax * sr
    fast = np.cumprod((smax < NFWP_HI[0]) & (np.arange(nch) < nch - 1), axis=1).astype(bool)
    beyond = ~fast & (smin >= 64.0)
    iv = _nfwp_interval(smin)
    one = ~fast & ~beyond & (smax < NFWP_HI[np.minimum(iv, NFWP_NI - 1)])
    several = ~fast & ~beyond & ~one
    pairs = kp.reshape(nch, NFW_CH // 2, 2)
    plo, phi = pairs.min(axis=2)[None] * sr[..., None], pairs.max(axis=2)[None] * sr[..., None]
    ivp = _nfwp_interval(plo)
    redo = several & ((phi >= NFWP_HI[np.minimum(ivp, NFWP_NI - 1)]) | (ivp >= NFWP_NI)).any(axis=2)
    return {name for name, hit in (("fast", fast), ("one", one), ("several", several), ("redo", redo),
                                   ("far", beyond & (kmin * xr > 4.0)), ("near", beyond & (kmin * xr <= 4.0)))
            if hit.any()}


def _k2_inputs(case, nsm):
    """(zs, cs, rvir, ks, plans the case must take).  c spans [0.6, 25] with both ends in every case."""
    rng = np.random.default_rng(len(case))
    if case == "sorted":                # every in-row plan, 37 masses: 111 rows, not a multiple of the 8 per CTA;
        zs, nm = np.array([0.0, 0.7, 3.0]), 37      # c >= 16 at s >= 64 gives whole chunks with x <= 4 (near)
        ks, plans = np.geomspace(1e-4, 300.0, 4097), {"fast", "one", "several", "redo", "far", "near"}
    elif case == "shuffled":            # unsorted ks: every chunk spans many intervals, pairs straddle edges
        zs, nm = np.array([0.3, 2.0]), 21
        ks, plans = rng.permutation(np.geomspace(1e-3, 100.0, 515)), {"several", "redo"}
    elif case == "partial":             # nk < 256: one partial chunk, the general loop only
        zs, nm = np.array([0.5]), 16
        ks, plans = np.geomspace(1e-2, 5.0, 200), {"one", "several"}
    elif case == "global":              # 129 chunks > 128: chunk bounds read from global memory, in every plan
        zs, nm = np.array([0.1]), 5
        ks, plans = np.geomspace(1e-4, 100.0, 33001), {"fast", "one", "several", "redo", "far"}
    elif case == "global_shuffled":
        zs, nm = np.array([1.0]), 5
        ks, plans = rng.permutation(np.geomspace(1e-4, 100.0, 33001)), {"several", "redo"}
    else:                               # "gridstride": more rows than nfw_poly_gemm_kernel's grid covers in one
        zs, nm = np.array([0.2, 1.5]), 64 * nsm + 37        # pass (16 rows x 8 warps x SM count)
        ks, plans = np.geomspace(1e-3, 30.0, 33), set()
    nz = zs.size
    cs = np.stack([rng.permutation(np.linspace(0.6, 25.0, nm)) for _ in range(nz)])
    rv = np.broadcast_to(np.geomspace(0.05, 3.0, nm), (nz, nm)).copy()
    return zs, cs, rv, ks, plans


@pytest.mark.parametrize("case", ["sorted", "shuffled", "partial", "global", "global_shuffled", "gridstride"])
def test_k2_uk_nfw_plans(env, case):
    """hmv_uk_nfw (chunk pre-pass, tensor-core record pre-pass, cube kernel) against the float64 Si/Ci closed form
    of the same halos, in every plan of the cube kernel; every case has odd nk or padding columns [nk, ldk)."""
    torch, capi, orc = env
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    zs, cs, rv, ks, plans = _k2_inputs(case, nsm)
    nz, nm, nk = cs.shape[0], cs.shape[1], ks.size
    sr = rv * (1.0 + zs[:, None])                   # s = k r_vir (1+z),  x = s / c
    assert plans <= _k2_plans(ks, sr, sr / cs), case
    nch = -(-nk // NFW_CH)
    assert {"partial": nch == 1 and nk < NFW_CH, "global": nch > 128, "global_shuffled": nch > 128,
            "gridstride": nz * nm > 16 * 8 * nsm and (nz * nm) % 8 != 0}.get(case, True)
    ldk = _ldk(nk)
    assert ldk > nk
    out = Out(torch, 1, nz * nm * ldk)
    out.poison[GUARD:GUARD + nz * nm * ldk].reshape(nz * nm, ldk)[:, nk:] = True     # NaN padding must survive
    dz, dk, dc, dr = (_dev(torch, a) for a in (zs, ks, cs, rv))
    L, p = capi.lib, capi.ptr
    ws = torch.empty(int(L.hmv_uk_nfw_ws_doubles(nz, nm, nk)), dtype=torch.float64, device="cuda")

    def launch():
        capi.check(L.hmv_uk_nfw(nz, nm, nk, ldk, p(dz), p(dk), float(ks.max()), p(dc), p(dr), p(ws), out.ptr,
                                capi.stream()), "hmv_uk_nfw")
    _twice(torch, launch, (out,))
    got = out.host((nz, nm, ldk))[0][..., :nk]
    want = orc.uk_nfw_analytic(ks, zs, cs, rv)
    bound = np.broadcast_to(np.abs(want).max(axis=-1, keepdims=True), want.shape)       # max|u| of the row (= 1)
    _assert_bound("uk_nfw", "uk_nfw " + case, got, want, bound, TAU_K2)
