"""The front and the end of the path, checked kernel by kernel against float64 host restatements of the same
operation on the same inputs, at the shapes and edges where these kernels go wrong.

The golden grids check these kernels only through the spectra, at rtol 1e-6, and every golden mass grid is a
geomspace, every golden Limber table sorted and dense.  Here every call goes through the C ABI, inputs are seeded
random, and the reference is numpy / scipy on the downloaded inputs:

* K6, Limber (`hmv_limber`, `hmv_limber_multi`): against `oracle.bilinear_clamped` with explicit trapezoid weights,
  and against `oracle.limber` (FITPACK) where the grid allows it.  Window redshifts above one warp's 32 lanes,
  multipole counts that are not a multiple of the 4 warps per CTA, queries below ks[0], above ks[-1], exactly on
  interior nodes and on the last node, window redshifts outside the table's, descending window redshifts (the
  trapezoid changes sign, as numpy.trapz), tables with a row stride ldp > nk and NaN in the columns [nk, ldp), with
  and without the second table P2.  `hmv_limber_multi` on the packed [nz][nsp][nk] layout of GridSix._limber (with
  and without a poisoned gap between spectra), each job bit-identical to its own `hmv_limber` launch.
  `hmv_pack_sum` bit-exact against numpy a + b.  Each C_l is held to |got - want| <= tau * sum_g |w_g pref_g| P_g.
* The unsorted-k fix: C_kk, C_kg and C_yy of a HaloModel on shuffled ks, bit-identical to the same calls on the
  sorted axis; GridSix refuses an unsorted Limber grid.
* a2, the mass function (`hmv_mass_function`, `hmv_mass_function_tinker`) on a mass grid with jittered log spacing,
  so that numpy.gradient's non-uniform stencil has asymmetric coefficients.  n(M) is held to the same stencil over
  |-ln(sigma)/2| (the gradient cancels) times |f(sigma)| (1 + nu^2/2), the condition number of f's exponential
  (sigma reaches 0.05 at z = 4 here, where the exponent is -400); b(M) to a plain rtol.
* K0 (`hmv_halo_geometry`, `hmv_mdelta`, `hmv_gnfw_params`): Duffy c and r_vir; the mass-definition secant solve
  against a bracketed brentq root per element, and its residual; all seven GNFW outputs of both kinds against the
  closed forms with non-default fit triples.
* K4, the HOD paths `test_hod_around_cta_width` does not reach: corr = "min", the Msat / Mcut overrides,
  alphasat == 1 exactly and one ulp either side, the shared-memory limit nm = 10784, and `hmv_hod_bisect` split
  into two rounds at several points, bit-identical to one `hmv_hod_solve`.
* `hmv_pk_spline` at every degree pair 1..5 against scipy's FITPACK evaluation (bispeu) of the same tck.

Largest error ratios measured on one B200 (1000 W power limit); each tolerance keeps about 10x headroom:

    limber (bilinear restatement) 4.3e-16 -> tau 5e-15; limber vs FITPACK 6.1e-16 -> 6e-15;
    mass function n(M) 3.3e-16 (Sheth-Tormen), 3.5e-16 (Tinker) of the bound -> tau 4e-15;
    b(M) 4.8e-16 (both) -> rtol 5e-15; halo geometry (c and r_vir) 4.5e-16 -> rtol 5e-15;
    mdelta M2 against brentq 7.2e-15 -> rtol 7e-14; its residual 3.3e-15 of M1/mc(C1) -> 3e-14;
    gnfw_params 4.3e-16 -> rtol 5e-15;
    HOD occupations 6.7e-14 -> rtol 7e-13 (with the N_c ~ 0 floor 1e-14 of test_gpu_kernel_plans);
    ngal and b_g 2.8e-16 -> rtol 3e-15;
    pk_spline 6.9e-16 of the |c| spline (islog 0) and relative (islog 1) -> tau 7e-15.
The whole file runs in a few seconds.

Outputs are written between NaN guards that must survive bit for bit, every launch is repeated and must give
bit-identical outputs, and each argument check must return its code before anything is launched (the outputs stay
NaN)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import assert_close

gpu = pytest.mark.gpu

TAU_LIMBER = 5e-15
TAU_LIMBER_FITPACK = 6e-15
TAU_MASSFN = 4e-15
RTOL_BIAS = 5e-15
RTOL_GEOMETRY = 5e-15
RTOL_MDELTA = 7e-14
TOL_MDELTA_RESID = 3e-14
RTOL_GNFW = 5e-15
RTOL_HOD, HOD_FLOOR = 7e-13, 1e-14
RTOL_HOD_SUMS = 3e-15
TAU_PKS = 7e-15
HMV_E_ARG, HMV_E_LIMIT = -1, -3
HOD_NM_MAX = 10784           # (4000 + 2 nm + 32) doubles = 200 KiB of shared memory
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64

OBSERVED = {}           # largest error ratio seen per comparison in this session


@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    from oracle import hmvec_oracle as orc
    yield torch, capi, orc
    print("\nlargest measured ratios:", ", ".join("%s %.2g" % kv for kv in sorted(OBSERVED.items())))


def _dev(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def _vp(t, off=0):
    return C.c_void_p(t.data_ptr() + 8 * off)


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
    assert ratio <= tau, "%s: max |got-want| / bound = %.3g > %.1g" % (name, ratio, tau)


def _assert_rtol(kind, name, got, want, rtol):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    ratio = float(np.max(np.abs(got - want) / np.abs(want)))
    _record(kind, ratio)
    assert ratio <= rtol, "%s: max relative error %.3g > %.1g" % (name, ratio, rtol)


class Out(object):
    """nspec outputs of n doubles, output q at [q*stride, q*stride + n), between NaN guards."""

    def __init__(self, torch, nspec, n, stride=None):
        self.nspec, self.n, self.stride = nspec, n, stride or n
        self.buf = torch.full((2 * GUARD + nspec * self.stride,), float("nan"), dtype=torch.float64, device="cuda")
        self.ptr = _vp(self.buf, GUARD)
        keep = np.ones(self.buf.numel(), dtype=bool)
        for q in range(nspec):
            keep[GUARD + q * self.stride:GUARD + q * self.stride + n] = False
        self.poison = keep

    def host(self, shape=None):
        b = self.buf.cpu().numpy()
        assert np.all(b.view(np.int64)[self.poison] == NAN_BITS), "a guard or the gap between outputs was written"
        out = np.stack([b[GUARD + q * self.stride:GUARD + q * self.stride + self.n] for q in range(self.nspec)])
        return out if shape is None else out.reshape((self.nspec,) + tuple(shape))

    def untouched(self):
        return bool(np.all(self.buf.cpu().numpy().view(np.int64) == NAN_BITS))


def _twice(torch, launch, outs):
    """Launch, snapshot, launch again: every output (guards included) must be bit-identical."""
    launch()
    torch.cuda.synchronize()
    first = [o.buf.clone() for o in outs]
    launch()
    torch.cuda.synchronize()
    for a, o in zip(first, outs):
        assert torch.equal(a.view(torch.int64), o.buf.view(torch.int64)), "second launch differs"


def _refused(torch, capi, rc, code, outs, what):
    torch.cuda.synchronize()
    assert rc == code, "%s: returned %d, expected %d (%s)" % (what, rc, code, capi.last_error())
    assert all(o.untouched() for o in outs), "%s: an output was written although the call was refused" % what


# ================================================================================================= K6: Limber
def _k_nodes(rng, Q, nk):
    """An increasing k axis of nk nodes for the queries Q: some queries below the first node and above the last,
    some exactly on an interior node and on the last node (IEEE division is exact-rounded on both sides)."""
    q = np.unique(Q)
    if q.size < 4:
        return np.geomspace(0.6 * q.min(), 1.7 * q.max(), nk)
    pick = lambda f: q[int(f * (q.size - 1))]
    exact = [pick(0.3), pick(0.5), pick(0.8)]
    if nk == 2:
        return np.array([exact[0], exact[2]])
    fill = np.exp(rng.uniform(np.log(pick(0.1)), np.log(exact[2]), nk - 3))
    ks = np.unique(np.r_[exact, fill])
    assert ks.size == nk and ks[-1] == exact[2]
    return ks


def _limber_case(seed, nl, ngz, nzp, nk, desc=False):
    """ells (non-integer, unsorted), the table's zs and ks, window redshifts, pref (both signs), chis."""
    rng = np.random.default_rng(seed)
    ells = rng.uniform(2.0, 3000.0, nl) + 0.37
    chis = rng.uniform(200.0, 6000.0, ngz)
    Q = (ells[:, None] + 0.5) / chis[None, :]                        # the kernel's k, bit for bit
    ks = _k_nodes(rng, Q, nk)
    zs = np.array([0.7]) if nzp == 1 else np.array([0.3, 1.9]) if nzp == 2 else \
        np.unique(rng.uniform(0.1, 3.0, nzp))
    assert zs.size == nzp
    gzs = rng.uniform(zs[0] - 0.3, zs[-1] + 0.4, ngz)                # some outside [zs[0], zs[-1]]
    if nzp > 2 and ngz > 3:
        gzs[:3] = (zs[nzp // 3], zs[nzp // 2], zs[-1])                # on interior table redshifts and the last
    elif nzp == 2 and ngz > 2:
        gzs[:1] = zs[-1]
    gzs = np.sort(gzs)[::-1].copy() if desc else np.sort(gzs)
    pref = rng.uniform(-1.0, 1.0, ngz)
    return dict(ells=ells, zs=zs, ks=ks, gzs=gzs, pref=pref, chis=chis, Q=Q)


def _trapz_w(x):
    n = x.size
    if n == 1:
        return np.ones(1)
    return 0.5 * (x[np.minimum(np.arange(n) + 1, n - 1)] - x[np.maximum(np.arange(n) - 1, 0)])


def _limber_ref(orc, c, P):
    """(C_l, bound): the clamped bilinear lookup of P [nzp, nk] at every (ell, window z), trapezoid-weighted."""
    Q, zs, ks = c["Q"], c["zs"], c["ks"]
    if zs.size > 1:
        val = orc.bilinear_clamped(ks, zs, P, Q, np.broadcast_to(c["gzs"], Q.shape))
    else:
        val = np.interp(Q, ks, P[0])
    wp = _trapz_w(c["gzs"]) * c["pref"]
    return val @ wp, np.abs(val) @ np.abs(wp)


def _table(torch, rng, nzp, nk, ldp):
    """A positive [nzp, nk] table and its device copy with row stride ldp, NaN in the columns [nk, ldp)."""
    P = rng.uniform(0.5, 2.0, (nzp, nk))
    t = torch.full((nzp, ldp), float("nan"), dtype=torch.float64, device="cuda")
    t[:, :nk] = _dev(torch, P)
    return P, t


LIMBER_SHAPES = [  # (nl, ngz, nzp, nk)
    (1, 1, 1, 2), (3, 2, 2, 3), (4, 31, 200, 10000), (5, 32, 2, 10000), (1001, 33, 200, 3), (1001, 1000, 200, 10000),
    (4, 1000, 1, 10000), (5, 33, 200, 2), (3, 32, 1, 3), (1001, 2, 2, 2), (1, 31, 200, 10000), (5, 1, 200, 10000),
]


@gpu
@pytest.mark.parametrize("p2", [False, True])
@pytest.mark.parametrize("order", ["ascending", "descending"])
@pytest.mark.parametrize("nl,ngz,nzp,nk", LIMBER_SHAPES)
def test_limber_shapes_and_edges(env, nl, ngz, nzp, nk, order, p2):
    """hmv_limber against the bilinear restatement (and FITPACK on the smaller grids): warps with 1, 31, 32, 33 and
    1000 window redshifts, multipole counts around the 4 warps per CTA, clamps at both ends in k and z, exact nodes,
    a row stride ldp > nk with NaN padding, P2 = NULL and not."""
    torch, capi, orc = env
    seed = nl * 7919 + ngz * 31 + nzp * 7 + nk + (order == "descending") * 3 + p2
    c = _limber_case(seed, nl, ngz, nzp, nk, desc=(order == "descending"))
    rng = np.random.default_rng(seed + 1)
    ldp = nk + 5
    P, dP = _table(torch, rng, nzp, nk, ldp)
    P2, dP2 = _table(torch, rng, nzp, nk, ldp) if p2 else (None, None)
    ks, Q = c["ks"], c["Q"]
    if nl * ngz >= 20:
        assert (Q < ks[0]).any() and (Q > ks[-1]).any() and (Q == ks[-1]).any(), "k edges not reached"
        if nk > 2:
            assert np.isin(Q, ks[1:-1]).any(), "no query on an interior node"
    d = {k: _dev(torch, c[k]) for k in ("ells", "zs", "ks", "gzs", "pref", "chis")}
    out = Out(torch, 1, nl)
    L, p = capi.lib, capi.ptr

    def launch():
        capi.check(L.hmv_limber(nl, p(d["ells"]), nzp, nk, ldp, p(d["zs"]), p(d["ks"]), p(dP), p(dP2), ngz,
                                p(d["gzs"]), p(d["pref"]), p(d["chis"]), out.ptr, capi.stream()), "hmv_limber")
    _twice(torch, launch, (out,))
    got = out.host()[0]
    Pt = P if P2 is None else P + P2
    want, bound = _limber_ref(orc, c, Pt)
    name = "limber nl=%d ngz=%d nzp=%d nk=%d %s P2=%s" % (nl, ngz, nzp, nk, order, p2)
    _assert_bound("limber", name, got, want, bound, TAU_LIMBER)
    if nzp * nk <= 20000:
        fp = orc.limber(c["ells"], c["zs"], ks, Pt, c["gzs"], np.ones(ngz), np.ones(ngz), c["pref"] * c["chis"] ** 2,
                        c["chis"])
        _assert_bound("limber_fitpack", name + " vs FITPACK", got, fp, bound, TAU_LIMBER_FITPACK)


def _packed(torch, rng, nz, nsp, nk, gap):
    """nsp tables in one [nz][nsp][nk + gap] buffer (GridSix._limber's layout; NaN in the gaps)."""
    Ps = [rng.uniform(0.5, 2.0, (nz, nk)) for _ in range(nsp)]
    buf = torch.full((nz, nsp, nk + gap), float("nan"), dtype=torch.float64, device="cuda")
    for q in range(nsp):
        buf[:, q, :nk] = _dev(torch, Ps[q])
    return Ps, buf


@gpu
@pytest.mark.parametrize("gap", [0, 6])
@pytest.mark.parametrize("njobs", [1, 2, 3, 4])
def test_limber_multi_jobs(env, njobs, gap):
    """hmv_limber_multi with 1..4 jobs that differ in ngz, table, P2 and pref, on the packed [nz][nsp][nk] layout
    (ldp = nsp (nk + gap)): each job is bit-identical to its own hmv_limber launch and matches the restatement."""
    torch, capi, orc = env
    nl, nz, nk, nsp = 37, 60, 700, 4
    ldp = nsp * (nk + gap)
    rng = np.random.default_rng(100 * njobs + gap)
    base = _limber_case(17, nl, nz, nz, nk)                       # shared ells, zs, ks
    zs, ks, ells = base["zs"], base["ks"], base["ells"]
    Ps, buf = _packed(torch, rng, nz, nsp, nk, gap)
    P2s, buf2 = _packed(torch, rng, nz, nsp, nk, gap)
    dz, dk, de = _dev(torch, zs), _dev(torch, ks), _dev(torch, ells)
    jobs, keep, refs = (capi.LimberJob * njobs)(), [], []
    outs = [Out(torch, 1, nl) for _ in range(njobs)]
    for q in range(njobs):
        ngz = (nz, 1, 33, 100)[q]
        c = _limber_case(1000 + q, nl, ngz, nz, nk, desc=(q == 3))
        gzs = zs.copy() if q == 0 else c["gzs"]
        chis = c["chis"] * (1.0 + 0.1 * q)
        pref = rng.uniform(-1.0, 1.0, ngz)
        tab = (q + 1) % nsp                                        # not the job's own index
        use2 = q % 2 == 1
        dg, dpf, dch = _dev(torch, gzs), _dev(torch, pref), _dev(torch, chis)
        keep += [dg, dpf, dch]
        jobs[q].P_d = buf.data_ptr() + 8 * tab * (nk + gap)
        jobs[q].P2_d = buf2.data_ptr() + 8 * tab * (nk + gap) if use2 else None
        jobs[q].ngz, jobs[q].gzs_d, jobs[q].pref_d, jobs[q].chis_d = ngz, dg.data_ptr(), dpf.data_ptr(), dch.data_ptr()
        jobs[q].cl_d = outs[q].ptr.value
        cq = dict(Q=(ells[:, None] + 0.5) / chis[None, :], zs=zs, ks=ks, gzs=gzs, pref=pref)
        refs.append(_limber_ref(orc, cq, Ps[tab] + P2s[tab] if use2 else Ps[tab]))
    L, p = capi.lib, capi.ptr

    def launch():
        capi.check(L.hmv_limber_multi(njobs, jobs, nl, p(de), nz, nk, ldp, p(dz), p(dk), capi.stream()),
                   "hmv_limber_multi")
    _twice(torch, launch, outs)
    for q in range(njobs):
        got = outs[q].host()[0]
        _assert_bound("limber", "limber_multi job %d/%d gap %d" % (q, njobs, gap), got, *refs[q], TAU_LIMBER)
        one = Out(torch, 1, nl)
        j = jobs[q]
        capi.check(L.hmv_limber(nl, p(de), nz, nk, ldp, p(dz), p(dk), C.c_void_p(j.P_d), C.c_void_p(j.P2_d), j.ngz,
                                C.c_void_p(j.gzs_d), C.c_void_p(j.pref_d), C.c_void_p(j.chis_d), one.ptr,
                                capi.stream()), "hmv_limber")
        torch.cuda.synchronize()
        assert np.array_equal(one.host()[0].view(np.int64), got.view(np.int64)), "job %d differs from hmv_limber" % q


@gpu
def test_limber_argument_checks(env):
    """hmv_limber_multi refuses 0 or 5 jobs, ldp < nk, nk < 2, a NULL job array and a job without a table, and
    hmv_limber refuses ldp < nk and nk < 2, each before anything is launched."""
    torch, capi, _ = env
    nl, nz, nk = 8, 5, 40
    c = _limber_case(5, nl, nz, nz, nk)
    d = {k: _dev(torch, c[k]) for k in ("ells", "zs", "ks", "gzs", "pref", "chis")}
    P = _dev(torch, np.ones((nz, nk)))
    outs = [Out(torch, 1, nl) for _ in range(5)]
    jobs = (capi.LimberJob * 5)()
    for q in range(5):
        jobs[q].P_d, jobs[q].P2_d, jobs[q].ngz = P.data_ptr(), None, nz
        jobs[q].gzs_d, jobs[q].pref_d, jobs[q].chis_d = d["gzs"].data_ptr(), d["pref"].data_ptr(), d["chis"].data_ptr()
        jobs[q].cl_d = outs[q].ptr.value
    L, p, st = capi.lib, capi.ptr, capi.stream()
    multi = lambda nj, jb, nk_, ldp: L.hmv_limber_multi(nj, jb, nl, p(d["ells"]), nz, nk_, ldp, p(d["zs"]), p(d["ks"]), st)
    _refused(torch, capi, multi(0, jobs, nk, nk), HMV_E_ARG, outs, "njobs = 0")
    _refused(torch, capi, multi(5, jobs, nk, nk), HMV_E_ARG, outs, "njobs = 5")
    _refused(torch, capi, multi(4, jobs, nk, nk - 1), HMV_E_ARG, outs, "ldp < nk")
    _refused(torch, capi, multi(4, jobs, 1, 1), HMV_E_ARG, outs, "nk = 1")
    _refused(torch, capi, multi(4, None, nk, nk), HMV_E_ARG, outs, "NULL jobs")
    jobs[2].P_d = None
    _refused(torch, capi, multi(4, jobs, nk, nk), HMV_E_ARG, outs, "job without a table")
    one = lambda nk_, ldp: L.hmv_limber(nl, p(d["ells"]), nz, nk_, ldp, p(d["zs"]), p(d["ks"]), p(P), None, nz,
                                        p(d["gzs"]), p(d["pref"]), p(d["chis"]), outs[0].ptr, st)
    _refused(torch, capi, one(nk, nk - 1), HMV_E_ARG, outs, "hmv_limber ldp < nk")
    _refused(torch, capi, one(1, 1), HMV_E_ARG, outs, "hmv_limber nk = 1")


@gpu
@pytest.mark.parametrize("bmode", ["all", "none", "some"])
@pytest.mark.parametrize("nsp", [1, 2, 3, 4])
def test_pack_sum(env, nsp, bmode):
    """hmv_pack_sum: out[z][s][k] = a_s[z][k] + b_s[z][k] bit for bit, with b_h NULL or some b_h[s] NULL, on k rows
    that end inside a 256-wide block."""
    torch, capi, _ = env
    for nz, nk in ((3, 300), (2, 257), (1, 1)):
        rng = np.random.default_rng(nz * 1000 + nk + nsp)
        a = [rng.standard_normal((nz, nk)) for _ in range(nsp)]
        a[0].flat[0] = -0.0                                        # -0.0 + 0.0 = +0.0 on both sides
        b = [rng.standard_normal((nz, nk)) if (bmode == "all" or (bmode == "some" and s % 2 == 0)) else None
             for s in range(nsp)]
        da = [_dev(torch, x) for x in a]
        db = [None if x is None else _dev(torch, x) for x in b]
        ah = (C.c_void_p * nsp)(*[t.data_ptr() for t in da])
        bh = None if bmode == "none" else (C.c_void_p * nsp)(*[None if t is None else t.data_ptr() for t in db])
        out = Out(torch, 1, nz * nsp * nk)

        def launch():
            capi.check(capi.lib.hmv_pack_sum(nz, nk, nsp, ah, bh, out.ptr, capi.stream()), "hmv_pack_sum")
        _twice(torch, launch, (out,))
        got = out.host((nz, nsp, nk))[0]
        want = np.stack([a[s] + (0.0 if b[s] is None else b[s]) for s in range(nsp)], axis=1)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), "pack_sum nsp=%d %s nz=%d nk=%d" % (
            nsp, bmode, nz, nk)


@gpu
def test_limber_unsorted_wavenumbers(env):
    """C_kk, C_kg and C_yy of a HaloModel on shuffled ks, from the shuffled spectra: bit-identical to the same calls on
    the sorted axis and columns (after the sort the kernel sees identical inputs), and within the 1e-6 of
    test_unsorted_wavenumbers of a model built on sorted ks.  GridSix refuses an unsorted Limber grid."""
    torch, capi, _ = env
    import hmvec_b200 as hm
    from hmvec_b200 import pipeline
    zs = np.linspace(0.1, 3.0, 14)
    ms = np.geomspace(1e11, 1e16, 40)
    ks = np.geomspace(1e-3, 30.0, 300)
    perm = np.random.default_rng(0).permutation(ks.size)
    ells = np.array([10.0, 100.0, 1000.0, 3000.0, 37.5])
    gzs = np.linspace(0.2, 2.0, 25)
    gdndz = np.exp(-(gzs - 0.8) ** 2 / 0.1)

    def model(kk):
        h = hm.HaloModel(zs, kk, ms=ms, accuracy='low')
        h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
        h.add_hod("g", mthresh=10 ** 10.5 + zs * 0.0)
        return h, {"C_kk": h.get_power("nfw", "nfw"), "C_kg": h.get_power("g", "nfw"), "C_yy": h.get_power("y", "y")}

    def cls(h, kk, P):
        return {"C_kk": h.C_kk(ells, zs, kk, P["C_kk"], lzs1=2.5, lzs2=2.5),
                "C_kg": h.C_kg(ells, zs, kk, P["C_kg"], gzs, gdndz, lzs=2.5),
                "C_yy": h.C_yy(ells, zs, kk, P["C_yy"])}

    hs, Ps = model(ks[perm])
    ksh = np.asarray(hs.ks)
    assert np.array_equal(ksh, ks[perm])
    order = np.argsort(ksh)
    got = cls(hs, ksh, Ps)
    srt = cls(hs, ksh[order], {k: np.ascontiguousarray(v[:, order]) for k, v in Ps.items()})
    h0, P0 = model(ks)
    ref = cls(h0, ks, P0)
    for k in got:
        assert np.array_equal(got[k].view(np.int64), srt[k].view(np.int64)), "%s: shuffled ks differ from sorted" % k
        assert_close(got[k], ref[k], 1e-6, name=k + " (shuffled ks vs a sorted-ks model)")
    with pytest.raises(ValueError):
        pipeline.GridSix(pipeline.make_inputs(zs, ms, ks[perm], ells=ells))
    pipeline.GridSix(pipeline.make_inputs(zs, ms, ks, ells=ells))          # the sorted grid is accepted


def test_limber_integral_refuses_repeated_axes():
    """A Limber axis with a repeated value has no order to sort into: ValueError before any device work."""
    from hmvec_b200.cosmology import limber_integral
    zs, ks = np.array([0.5, 1.0, 2.0]), np.array([0.1, 0.3, 0.2, 0.3])
    P = np.ones((3, 4))
    args = (np.array([100.0]), zs, ks, P, zs, 1.0, 1.0, np.ones(3), np.ones(3))
    with pytest.raises(ValueError, match="ks"):
        limber_integral(*args, device="cpu")
    with pytest.raises(ValueError, match="zs"):
        limber_integral(np.array([100.0]), np.array([0.5, 2.0, 0.5]), ks[:3], P[:, :3], zs, 1.0, 1.0, np.ones(3),
                        np.ones(3), device="cpu")


# ================================================================================================= a2: mass function
def _jittered_ms(rng, nm, lo=1e9, hi=1e16):
    """ln M on a grid with each step perturbed by up to +-30 %: the non-uniform stencil's coefficients differ."""
    x = np.linspace(np.log(lo), np.log(hi), nm)
    h = x[1] - x[0]
    x = x + rng.uniform(-0.3, 0.3, nm) * h
    assert np.all(np.diff(x) > 0)
    return np.exp(x)


def _sigma2(rng, zs, ms):
    """sigma^2(M, z) from ~0.05 to ~20 with 3 % point-to-point noise (the gradient then cancels)."""
    u = np.log(ms / 1e12)
    s2 = np.exp(2.0 * (np.log(3.0) - 0.12 * u - 0.004 * u ** 2))[None, :] / (1.0 + zs[:, None]) ** 2
    return s2 * rng.uniform(0.97, 1.03, s2.shape)


def _stencil_bound(s2, ms):
    """numpy.gradient's stencil applied to |-ln(sigma^2)/2|: the sum the n(M) error is bounded by."""
    f, x = np.abs(-0.5 * np.log(s2)), np.log(ms)
    b = np.empty_like(f)
    b[:, 0] = (f[:, 1] + f[:, 0]) / (x[1] - x[0])
    b[:, -1] = (f[:, -1] + f[:, -2]) / (x[-1] - x[-2])
    if ms.size > 2:
        hs, hd = x[1:-1] - x[:-2], x[2:] - x[1:-1]
        ca, cb, cc = -hd / (hs * (hd + hs)), (hd - hs) / (hd * hs), hs / (hd * (hd + hs))
        b[:, 1:-1] = np.abs(ca) * f[:, :-2] + np.abs(cb) * f[:, 1:-1] + np.abs(cc) * f[:, 2:]
    return b


MASSFN_SHAPES = [(1, 2), (4, 3), (3, 17), (15, 17), (85, 3), (128, 2), (16, 16), (1, 257)]   # nz*nm 255/256/257
TINKER_Z = np.array([0.0, 0.5, 1.7, np.nextafter(3.0, 0.0), 2.9999, 3.0, 3.4, 6.0])


@gpu
@pytest.mark.parametrize("fit", ["sheth-tormen", "tinker"])
@pytest.mark.parametrize("nz,nm", MASSFN_SHAPES)
def test_mass_function(env, nz, nm, fit):
    """hmv_mass_function / hmv_mass_function_tinker against oracle.mass_function on a jittered ln M grid, with nz*nm
    below, at and above the 256-thread block; Tinker at z = 0, just below 3, exactly 3 (mapped to 0) and above 3."""
    torch, capi, orc = env
    rng = np.random.default_rng(nz * 1000 + nm + (fit == "tinker"))
    ms = _jittered_ms(rng, nm)
    zs = TINKER_Z[np.arange(nz) % TINKER_Z.size] if fit == "tinker" else rng.uniform(0.0, 4.0, nz)
    s2 = _sigma2(rng, zs, ms)
    rho = 4.1e10
    ds2, dm = _dev(torch, s2), _dev(torch, ms)
    o_n, o_b = Out(torch, 1, nz * nm), Out(torch, 1, nz * nm)
    L, p = capi.lib, capi.ptr
    if fit == "tinker":
        from hmvec_b200 import tinker
        dc = 1.686
        dtk = _dev(torch, tinker.redshift_parameters(zs))
        alpha_table = np.loadtxt(os.path.join(os.path.dirname(tinker.__file__), "data", "alpha_consistency.txt"),
                                 unpack=True)
        F = orc.tinker_fsigma(s2, zs, alpha_table, dc)
        want_b = orc.tinker_bias(s2, dc)

        def launch():
            capi.check(L.hmv_mass_function_tinker(nz, nm, p(ds2), p(dm), rho, dc, p(dtk), o_n.ptr, o_b.ptr,
                                                  capi.stream()), "hmv_mass_function_tinker")
    else:
        st = dict(A=0.33, a=0.75, p=0.28, dc=1.68)                   # non-default: every parameter must arrive
        F = orc.st_fsigma(s2, **st)
        want_b = orc.st_bias(s2, a=st["a"], p=st["p"], dc=st["dc"])

        def launch():
            capi.check(L.hmv_mass_function(nz, nm, p(ds2), p(dm), rho, st["A"], st["a"], st["p"], st["dc"], o_n.ptr,
                                           o_b.ptr, capi.stream()), "hmv_mass_function")
    _twice(torch, launch, (o_n, o_b))
    want_n = orc.mass_function(s2, ms, rho, fsigma=F)
    # f(sigma) carries exp(-a nu^2 / 2) (Sheth-Tormen) or exp(-gamma nu^2 / 2) (Tinker), a, gamma < 1: rounding of
    # the exponent is amplified by its condition number, at most 1 + nu^2 / 2
    cond = 1.0 + 0.5 * (st["dc"] if fit != "tinker" else dc) ** 2 / s2
    bound = rho * np.abs(F) * cond * _stencil_bound(s2, ms) / ms[None, :] ** 2
    name = "%s nz=%d nm=%d" % (fit, nz, nm)
    _assert_bound("massfn_" + fit, name + " n(M)", o_n.host((nz, nm))[0], want_n, bound, TAU_MASSFN)
    _assert_rtol("bias_" + fit, name + " b(M)", o_b.host((nz, nm))[0], want_b, RTOL_BIAS)


# ================================================================================================= K0: halo prep
@gpu
def test_halo_geometry(env):
    """hmv_halo_geometry: Duffy c = A (h M / 2e12)^alpha (1+z)^beta and r_vir = cbrt(3 M / (4 pi Delta rho)) with
    non-default Duffy parameters, over 1e8..1e17 Msun and nz*nm = 1001 (a partial last block)."""
    torch, capi, orc = env
    rng = np.random.default_rng(3)
    zs, ms = rng.uniform(0.0, 6.0, 7), _jittered_ms(rng, 143, 1e8, 1e17)
    drho = rng.uniform(1e10, 1e13, zs.size)
    A, al, be, h = 6.71, -0.091, -0.44, 0.68
    oc, orv = Out(torch, 1, zs.size * ms.size), Out(torch, 1, zs.size * ms.size)
    dz, dm, dd = _dev(torch, zs), _dev(torch, ms), _dev(torch, drho)

    def launch():
        capi.check(capi.lib.hmv_halo_geometry(zs.size, ms.size, capi.ptr(dz), capi.ptr(dm), capi.ptr(dd), A, al, be, h,
                                              oc.ptr, orv.ptr, capi.stream()), "hmv_halo_geometry")
    _twice(torch, launch, (oc, orv))
    shape = (zs.size, ms.size)
    _assert_rtol("geometry", "Duffy c", oc.host(shape)[0], orc.duffy(ms, zs, h, A, al, be), RTOL_GEOMETRY)
    rv = np.cbrt(3.0 * ms[None, :] / (4.0 * np.pi * drho[:, None]))
    _assert_rtol("geometry", "r_vir", orv.host(shape)[0], rv, RTOL_GEOMETRY)


@gpu
def test_mdelta_against_bracketed_root(env):
    """hmv_mdelta's secant solve of M1/mc(C1) = M2/mc(C2(M2)) in ln M2 against brentq to the float64 floor per
    element, for c in [0.3, 40], M in [1e8, 1e17] and Delta rho1 / Delta rho2 in [0.3, 3] (vir -> 200c and
    200m -> 200c at every redshift the grids use); the residual at the device's root is at the rounding level."""
    torch, capi, orc = env
    from scipy.optimize import brentq
    rng = np.random.default_rng(4)
    nz, nm = 9, 47
    ms = np.exp(rng.uniform(np.log(1e8), np.log(1e17), nm))
    cs = np.exp(rng.uniform(np.log(0.3), np.log(40.0), (nz, nm)))
    cs[0, :2], cs[1, :2] = (0.3, 40.0), (40.0, 0.3)
    d2 = rng.uniform(1e10, 1e12, nz)
    r = np.r_[0.3, 3.0, rng.uniform(0.3, 3.0, nz - 2)]
    d1 = r * d2
    out = Out(torch, 1, nz * nm)
    dm, dc, dd1, dd2 = (_dev(torch, a) for a in (ms, cs, d1, d2))

    def launch():
        capi.check(capi.lib.hmv_mdelta(nz, nm, capi.ptr(dm), capi.ptr(dc), capi.ptr(dd1), capi.ptr(dd2), out.ptr,
                                       capi.stream()), "hmv_mdelta")
    _twice(torch, launch, (out,))
    got = out.host((nz, nm))[0]
    rr = d1 / d2
    mc = lambda c: np.log1p(c) - c / (1.0 + c)                     # hmvec.py:737, as the kernel forms it
    want, resid = np.empty((nz, nm)), np.empty((nz, nm))
    for z in range(nz):
        for m in range(nm):
            M1, C1, lnM1 = ms[m], cs[z, m], np.log(ms[m])
            lhs = M1 / mc(C1)
            g = lambda x: lhs - np.exp(x) / mc(C1 * np.cbrt(np.exp(x - lnM1) * rr[z]))
            want[z, m] = np.exp(brentq(g, lnM1 - 8.0, lnM1 + 8.0, xtol=1e-300, rtol=4 * np.finfo(float).eps,
                                       maxiter=500))
            resid[z, m] = abs(g(np.log(got[z, m]))) / lhs
    _assert_rtol("mdelta", "M2 vs brentq", got, want, RTOL_MDELTA)
    _record("mdelta_residual", resid.max())
    assert resid.max() <= TOL_MDELTA_RESID, "residual %.3g of M1/mc(C1)" % resid.max()


@gpu
@pytest.mark.parametrize("kind", [0, 1])
def test_gnfw_params(env, kind):
    """hmv_gnfw_params, density (0) and pressure (1): all seven outputs against the closed forms with
    oracle._plaw and non-default fit triples (every power of m200 and 1+z non-zero)."""
    torch, capi, orc = env
    rng = np.random.default_rng(5 + kind)
    nz, nm = 5, 53
    zs = rng.uniform(0.0, 4.0, nz)
    m200 = np.exp(rng.uniform(np.log(1e10), np.log(1e16), (nz, nm)))
    rvir = rng.uniform(0.05, 3.0, (nz, nm))
    rhoc = rng.uniform(1e11, 1e12, nz)
    hofz = rng.uniform(2e-4, 2e-3, nz)
    trip = [(3.7e3, 0.14, -0.52), (1.13, -0.031, 0.27), (3.9, 0.051, -0.33)] if kind == 0 else \
        [(17.3, 0.161, -0.71), (0.52, -0.011, 0.69), (4.1, 0.046, 0.39)]
    fit9 = [v for t in trip for v in t]
    gamma, pres_alpha, amp_const, pref = -0.23, 1.07, 3.3e-19, 2.9e-7
    outs = [Out(torch, 1, nz * nm) for _ in range(7)]
    dz, dm, dr, drc, dh = (_dev(torch, a) for a in (zs, m200, rvir, rhoc, hofz))

    def launch():
        capi.check(capi.lib.hmv_gnfw_params(kind, nz, nm, capi.ptr(dz), capi.ptr(dm), capi.ptr(dr), capi.ptr(drc),
                                            capi.ptr(dh), capi.darr(fit9), gamma, pres_alpha, amp_const, pref,
                                            *(o.ptr for o in outs), capi.stream()), "hmv_gnfw_params")
    _twice(torch, launch, outs)
    got = [o.host((nz, nm))[0] for o in outs]
    z = zs[:, None]
    r200 = np.cbrt(3.0 * m200 / (4.0 * np.pi * 200.0 * rhoc[:, None]))
    q0, q1, q2 = (orc._plaw(m200, z, t) for t in trip)
    one = np.ones((nz, nm))
    if kind == 0:
        want = [0.5 * r200, rvir / (0.5 * r200), one, q1, (q2 + gamma) / q1, one, one]
    else:
        want = [r200, rvir / r200, q1, pres_alpha * one, q2, amp_const * m200 * rhoc[:, None] / (2.0 * r200) * q0,
                pref * r200 ** 3 * (1.0 + z) ** 2 / hofz[:, None]]
    for name, g, w in zip(("rs", "cmax", "xc", "alpha", "expo", "amp", "outscale"), got, want):
        if np.all(w == 1.0) or (kind == 1 and name == "alpha"):
            assert np.array_equal(g, w), "gnfw kind %d %s: constant output differs" % (kind, name)
        else:
            _assert_rtol("gnfw", "gnfw kind %d %s" % (kind, name), g, w, RTOL_GNFW)


# ================================================================================================= K4: HOD
def _hod_inputs(nm):
    zs = np.array([0.3, 1.2])
    ms = np.geomspace(1e10, 1e16, nm)
    nzm = (ms / 1e12) ** -1.9 / 1e12 * np.exp(-ms / 5e14) * (1.0 + zs[:, None]) ** -1
    return zs, ms, nzm, 1.0 + (ms / 1e13) ** 0.5 + 0.0 * zs[:, None]


def _hod_host(orc, zs, ms, l10, hp, corr, msat, mcut):
    """hmvec.py:698-731 with the Msat / Mcut overrides of hmv_hod (a value > 0 replaces the SHMR scaling)."""
    Nc = orc.hod_occupations(zs, ms, l10, hp)[0]
    mth = orc.shmr_log10mhalo(zs, np.asarray(l10)[:, None])
    Msat = np.full_like(mth, msat) if msat > 0 else 1e12 * hp["hod_Bsat"] * 10.0 ** ((mth - 12.0) * hp["hod_betasat"])
    Mcut = np.full_like(mth, mcut) if mcut > 0 else 1e12 * hp["hod_Bcut"] * 10.0 ** ((mth - 12.0) * hp["hod_betacut"])
    Ns = Nc * (ms[None, :] / Msat) ** hp["hod_alphasat"] * np.exp(-Mcut / ms[None, :])
    if corr == 0:
        with np.errstate(all="ignore"):
            nn = Ns ** 2 / Nc
        nn[np.isclose(Nc, 0.0)] = 0.0
        return Nc, Ns, nn, Ns
    return Nc, Ns, Ns ** 2, Ns * Nc


def _hodp(capi, hp, msat=0.0, mcut=0.0):
    return capi.darr([hp[k] for k in ("hod_sig_log_mstellar", "hod_alphasat", "hod_Bsat", "hod_betasat", "hod_Bcut",
                                      "hod_betacut")] + [msat, mcut])


def _run_hod(env, nm, hp, corr, msat, mcut, name):
    torch, capi, orc = env
    zs, ms, nzm, bh = _hod_inputs(nm)
    l10 = np.array([10.6, 11.1])
    L, p = capi.lib, capi.ptr
    dz, dm, dn, db, dl = (_dev(torch, a) for a in (zs, ms, nzm, bh, l10))
    hodp = _hodp(capi, hp, msat, mcut)
    outs = [Out(torch, 1, zs.size * nm) for _ in range(4)] + [Out(torch, 1, zs.size) for _ in range(2)]

    def launch():
        capi.check(L.hmv_hod(zs.size, nm, p(dz), p(dm), p(dl), hodp, corr, p(dn), p(db), *(o.ptr for o in outs),
                             capi.stream()), "hmv_hod")
    _twice(torch, launch, outs)
    got = [o.host((zs.size, nm) if i < 4 else (zs.size,))[0] for i, o in enumerate(outs)]
    want = _hod_host(orc, zs, ms, l10, hp, corr, msat, mcut)
    for tag, a, b in zip(("Nc", "Ns", "NsNsm1", "NcNs"), got[:4], want):
        assert_close(a, b, RTOL_HOD, HOD_FLOOR, name="%s %s" % (name, tag))
        big = np.abs(b) > HOD_FLOOR * np.abs(b).max() / RTOL_HOD
        if big.any():
            _record("hod_occupations", np.max(np.abs(a - b)[big] / np.abs(b)[big]))
    ngal = orc.hod_ngal(nzm, ms, want[0], want[1])
    _assert_rtol("hod_sums", name + " ngal", got[4], ngal, RTOL_HOD_SUMS)
    _assert_rtol("hod_sums", name + " b_g", got[5], orc.hod_bias(nzm, bh, ms, want[0], want[1], ngal), RTOL_HOD_SUMS)


HOD_CASES = {  # name: (corr, Msat override, Mcut override, alphasat)
    "min": (1, 0.0, 0.0, None),
    "overrides": (0, 3.1e13, 2.3e11, None),
    "overrides_min": (1, 8.0e12, 4.0e12, None),
    "alphasat_1": (0, 0.0, 0.0, 1.0),
    "alphasat_1_plus_ulp": (0, 0.0, 0.0, np.nextafter(1.0, 2.0)),
    "alphasat_1_minus_ulp": (1, 0.0, 0.0, np.nextafter(1.0, 0.0)),
}


@gpu
@pytest.mark.parametrize("case", sorted(HOD_CASES))
def test_hod_branches(env, case):
    """hod_kernel's branches that the default HOD does not take: corr = "min", the Msat / Mcut overrides, and the
    exact alphasat == 1 shortcut next to pow() one ulp either side of it."""
    _, _, orc = env
    corr, msat, mcut, alpha = HOD_CASES[case]
    hp = dict(orc.DEFAULTS)
    if alpha is not None:
        hp["hod_alphasat"] = alpha
    _run_hod(env, 700, hp, corr, msat, mcut, case)


@gpu
def test_hod_shared_memory_limit(env):
    """nm = 10784 fills the 200 KiB of staged shared memory exactly and must run and match; nm = 10785 must return
    HMV_E_LIMIT from hmv_hod, hmv_hod_bisect and hmv_hod_solve before anything is launched."""
    torch, capi, orc = env
    hp = dict(orc.DEFAULTS)
    _run_hod(env, HOD_NM_MAX, hp, 0, 0.0, 0.0, "nm=%d" % HOD_NM_MAX)
    nm = HOD_NM_MAX + 1
    zs, ms, nzm, bh = _hod_inputs(nm)
    L, p, st = capi.lib, capi.ptr, capi.stream()
    dz, dm, dn, db, dl = (_dev(torch, a) for a in (zs, ms, nzm, bh, np.array([10.6, 11.1])))
    hodp = _hodp(capi, hp)
    outs = [Out(torch, 1, zs.size * nm) for _ in range(4)] + [Out(torch, 1, zs.size) for _ in range(2)]
    rc = L.hmv_hod(zs.size, nm, p(dz), p(dm), p(dl), hodp, 0, p(dn), p(db), *(o.ptr for o in outs), st)
    _refused(torch, capi, rc, HMV_E_LIMIT, outs, "hmv_hod nm=%d" % nm)
    assert "10784" in capi.last_error()
    ws, mask = Out(torch, 1, zs.size * (capi.HMV_BISECT_MAXIT + 4)), Out(torch, 1, 1)
    rc = L.hmv_hod_bisect(zs.size, nm, p(dz), p(dm), p(dn), p(dl), hodp, 7.0, 14.0, 1e-4, 0, 64, ws.ptr, mask.ptr, st)
    _refused(torch, capi, rc, HMV_E_LIMIT, (ws, mask), "hmv_hod_bisect nm=%d" % nm)
    res, it = Out(torch, 1, zs.size), Out(torch, 1, 1)
    rc = L.hmv_hod_solve(zs.size, nm, p(dz), p(dm), p(dn), p(dl), hodp, 7.0, 14.0, 1e-4, 1.0, ws.ptr, res.ptr, it.ptr,
                         st)
    _refused(torch, capi, rc, HMV_E_LIMIT, (ws, res, it), "hmv_hod_solve nm=%d" % nm)


@gpu
def test_hod_bisect_rounds(env):
    """hmv_hod_bisect over [0, a) then [a, 64), then hmv_hod_pick, for split points a before and after convergence,
    against one hmv_hod_solve: before convergence every workspace word (midpoints, pass masks, brackets) is
    bit-identical; after it the second round returns at once (later midpoints stay unwritten) and the first passing
    iteration is the same.  log10 mthresh and the iteration count are bit-identical either way."""
    torch, capi, orc = env
    hp = dict(orc.DEFAULTS)
    zs = np.array([0.1, 0.5, 0.9, 1.6, 2.4])
    nz, nm = zs.size, 500
    ms = np.geomspace(1e10, 1e16, nm)
    nzm = (ms / 1e12) ** -1.9 / 1e12 * np.exp(-ms / 5e14) * (1.0 + zs[:, None]) ** -1
    target = orc.hod_ngal(nzm, ms, *orc.hod_occupations(zs, ms, np.linspace(10.2, 11.6, nz), hp)[:2])
    L, p, st = capi.lib, capi.ptr, capi.stream()
    dz, dm, dn, dt = (_dev(torch, a) for a in (zs, ms, nzm, target))
    hodp = _hodp(capi, hp)
    lo, hi, rtol, A = hp["hod_bisect_lo"], hp["hod_bisect_hi"], 1e-7, hp["hod_A_log10mthresh"]
    MAXIT = capi.HMV_BISECT_MAXIT
    nws = nz * (MAXIT + 3)                                          # midpoints, pass masks, brackets

    ws_s = torch.full((nz * (MAXIT + 4),), float("nan"), dtype=torch.float64, device="cuda")
    l10_s, it_s = torch.zeros(nz, dtype=torch.float64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    capi.check(L.hmv_hod_solve(nz, nm, p(dz), p(dm), p(dn), p(dt), hodp, lo, hi, rtol, A, p(ws_s), p(l10_s),
                               p(it_s), st), "hmv_hod_solve")
    torch.cuda.synchronize()
    T = int(it_s[0])
    assert 2 <= T < MAXIT
    ref = ws_s.cpu().numpy()
    ref_bits = ref.view(np.int64)
    ref_pass = ref_bits[nz * MAXIT:nz * (MAXIT + 1)]
    for a in sorted({1, T - 1, T, T + 1, 40, MAXIT - 1} & set(range(1, MAXIT))):
        ws = torch.full((nws,), float("nan"), dtype=torch.float64, device="cuda")
        mask = torch.zeros(1, dtype=torch.int64, device="cuda")
        l10, it = torch.zeros(nz, dtype=torch.float64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
        for i0, i1 in ((0, a), (a, MAXIT)):
            capi.check(L.hmv_hod_bisect(nz, nm, p(dz), p(dm), p(dn), p(dt), hodp, lo, hi, rtol, i0, i1, p(ws),
                                        _vp(mask), st), "hmv_hod_bisect [%d,%d)" % (i0, i1))
        capi.check(L.hmv_hod_pick(nz, p(ws), _vp(mask), A, p(l10), p(it), st), "hmv_hod_pick")
        torch.cuda.synchronize()
        bits = ws.cpu().numpy().view(np.int64)
        ys, ys_ref = bits[:nz * MAXIT].reshape(nz, MAXIT), ref_bits[:nz * MAXIT].reshape(nz, MAXIT)
        if a < T:               # not converged before a: the continuation round resumes from the saved state
            assert np.array_equal(bits, ref_bits[:nws]), "a=%d: workspace differs from hmv_hod_solve" % a
            assert int(mask[0]) == int(ref_bits[nz * (MAXIT + 3)]), "a=%d: mask differs" % a
        else:                   # converged at iteration T-1 < a: the second round returns at once
            assert np.array_equal(ys[:, :a], ys_ref[:, :a]), "a=%d: midpoints differ" % a
            assert np.all(ys[:, a:] == NAN_BITS), "a=%d: the continuation round ran after convergence" % a
            low = (1 << a) - 1
            assert np.array_equal(bits[nz * MAXIT:nz * (MAXIT + 1)] & low, ref_pass & low), "a=%d: pass masks" % a
            assert (int(mask[0]) & -int(mask[0])) == 1 << (T - 1), "a=%d: first passing iteration" % a
        assert int(it[0]) == T, "a=%d: iterations %d vs %d" % (a, int(it[0]), T)
        assert torch.equal(l10.view(torch.int64), l10_s.view(torch.int64)), "a=%d: log10 mthresh differs" % a


# ================================================================================================= hmv_pk_spline
def _pks_case(torch, rng, kx, ky, ninterior):
    """tck with (kx, ky) and `ninterior` interior knots per axis (0: the minimum 2(k+1) knots); z queries below,
    above, on interior knots and on the last knot, unsorted; ln k knots taken from the device's own log so the
    kernel's log(ks) lands exactly on them."""
    zk = np.sort(rng.uniform(0.0, 5.0, ninterior + 2))
    tx = np.r_[[zk[0]] * (kx + 1), zk[1:-1], [zk[-1]] * (kx + 1)]
    kn = np.sort(np.exp(rng.uniform(np.log(1e-3), np.log(20.0), ninterior + 2)))
    yk = torch.log(_dev(torch, kn)).cpu().numpy()
    ty = np.r_[[yk[0]] * (ky + 1), yk[1:-1], [yk[-1]] * (ky + 1)]
    zq = rng.permutation(np.r_[zk, zk[0] - 0.7, zk[-1] + 1.3, rng.uniform(zk[0], zk[-1], 9)])
    kq = rng.permutation(np.r_[kn, 1e-5, 300.0, np.exp(rng.uniform(np.log(1e-3), np.log(20.0), 291 - kn.size))])
    return tx, ty, zq, kq


@gpu
@pytest.mark.parametrize("ky", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("kx", [1, 2, 3, 4, 5])
def test_pk_spline_degrees(env, kx, ky):
    """hmv_pk_spline at every degree pair against FITPACK's bispeu on the same tck, with the minimum knot count and
    with interior knots, islog 0 and 1, nk = 293 (not a multiple of the 128-thread block)."""
    torch, capi, _ = env
    from scipy.interpolate import BivariateSpline
    rng = np.random.default_rng(10 * kx + ky)
    for ninterior in (0, 1 + (kx + ky) % 5):
        tx, ty, zq, kq = _pks_case(torch, rng, kx, ky, ninterior)
        nx, ny = tx.size, ty.size
        ncoef = (nx - kx - 1) * (ny - ky - 1)
        yq = torch.log(_dev(torch, kq)).cpu().numpy()
        Z, Y = np.meshgrid(zq, yq, indexing="ij")
        for islog in (0, 1):
            c = rng.uniform(-2.0, 2.0, ncoef) if islog else rng.standard_normal(ncoef)
            scale = -1.7 if islog else 1.3
            sp = BivariateSpline._from_tck((tx, ty, c, kx, ky)).ev(Z.ravel(), Y.ravel()).reshape(Z.shape)
            sab = BivariateSpline._from_tck((tx, ty, np.abs(c), kx, ky)).ev(Z.ravel(), Y.ravel()).reshape(Z.shape)
            d = [_dev(torch, a) for a in (zq, kq, tx, ty, c)]
            out = Out(torch, 1, zq.size * kq.size)

            def launch():
                capi.check(capi.lib.hmv_pk_spline(zq.size, kq.size, *(capi.ptr(t) for t in d[:2]), nx, ny, kx, ky,
                                                  *(capi.ptr(t) for t in d[2:]), islog, scale, out.ptr, capi.stream()),
                           "hmv_pk_spline")
            _twice(torch, launch, (out,))
            got = out.host((zq.size, kq.size))[0]
            if islog:
                want = scale * np.exp(sp)
                bound = np.abs(want) * (sab + 1.0)
            else:
                want, bound = scale * sp, abs(scale) * sab
            _assert_bound("pk_spline", "pk_spline kx=%d ky=%d interior=%d islog=%d" % (kx, ky, ninterior, islog),
                          got, want, bound, TAU_PKS)


@gpu
def test_pk_spline_argument_checks(env):
    """Degree 0 or 6, too few knots and nz > 65535 return HMV_E_ARG before anything is launched."""
    torch, capi, _ = env
    tx = np.r_[[0.0] * 7, [1.0] * 7]
    d = [_dev(torch, a) for a in (np.zeros(4), np.ones(4), tx, tx, np.zeros(64))]
    out = Out(torch, 1, 16)
    call = lambda nz, nx, ny, kx, ky: capi.lib.hmv_pk_spline(nz, 4, *(capi.ptr(t) for t in d[:2]), nx, ny, kx, ky,
                                                             *(capi.ptr(t) for t in d[2:]), 0, 1.0, out.ptr,
                                                             capi.stream())
    for args, what in (((4, 14, 14, 0, 3), "kx = 0"), ((4, 14, 14, 3, 0), "ky = 0"), ((4, 14, 14, 6, 3), "kx = 6"),
                       ((4, 14, 14, 3, 6), "ky = 6"), ((4, 7, 14, 3, 3), "nx < 2(kx+1)"),
                       ((4, 14, 5, 3, 2), "ny < 2(ky+1)"), ((65536, 14, 14, 3, 3), "nz > 65535")):
        _refused(torch, capi, call(*args), HMV_E_ARG, (out,), what)
