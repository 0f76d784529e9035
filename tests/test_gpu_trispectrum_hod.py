"""The 1-halo trispectrum and its non-Gaussian Limber covariance with galaxy (HOD) legs (hmv_trispec_1h_tracers,
hmv_cl_cov_1h_tracers, HaloModel.get_trispectrum_1halo / get_cl_cov_1halo with HOD names), against a float64 numpy
restatement on the same downloaded cubes and occupations: np.interp for u(k), explicit trapezoid weights on ms and zs.

    t_g(k)        = (Nc u_c(k) + Ns u_s(k)) / ngal                 (u_c = 1 without a central profile)
    <g g>(k, k')  = [NsNsm1 u_s(k) u_s(k') + NcNs (u_c(k) u_s(k') + u_s(k) u_c(k'))] / ngal^2
    T^{ABCD}(k1,k2;z) = sum_m w_m n(z,m) t_A(k1) t_B(k1) t_C(k2) t_D(k2), a pair of galaxy legs replaced by <g g>

The reference expands <g g> into its three separable terms and each element is held to |got - want| <= TAU * B, B the
same sums over absolute values.  The ABI cases use seeded random cubes in [-0.3, 1.2] with NaN padding columns, random
positive occupations, and NaN guards around the output; every launch runs twice and must give bit-identical output.
They cover every MT plan of the contraction with one and two segments of mass rows per redshift, with and without
split-k, K chunks that cross segment and redshift boundaries, nm = 1 and odd nm.
"""
import ctypes as C

import numpy as np
import pytest

HMV_E_ARG, HMV_E_LIMIT = -1, -3
TAU = 1e-12
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64
KIND_MATTER, KIND_HOD, KIND_PRESSURE = 0, 1, 2


# ------------------------------------------------------------------------------------------------- host restatement
def _trapz_w(x):
    x = np.asarray(x, dtype=np.float64)
    n = x.size
    if n < 2:
        return np.zeros(n)
    return 0.5 * (x[np.minimum(np.arange(n) + 1, n - 1)] - x[np.maximum(np.arange(n) - 1, 0)])


def _interp(cube, ks, kq):
    """u(z, m, l) at kq[z, l], linear on ks and clamped (np.interp)."""
    nz, nm = cube.shape[:2]
    out = np.empty((nz, nm, kq.shape[1]))
    for z in range(nz):
        for m in range(nm):
            out[z, m] = np.interp(kq[z], ks, cube[z, m])
    return out


def _reference(legs, hod, ms, nzm, rho, ks, q1, q2, chis=None, zs=None, pref=None):
    """(value, bound) of four legs, each (kind, us cube, uc cube or None); hod = dict(Nc, Ns, NcNs, NsNsm1 [nz, nm],
    ngal [nz]) for the kind-1 legs.  T [nz, n1, n2] when chis is None, else Cov [n1, n2]."""
    nz, nm = legs[0][1].shape[:2]
    if chis is None:
        kq1, kq2 = np.broadcast_to(q1, (nz, q1.size)), np.broadcast_to(q2, (nz, q2.size))
        zw = np.ones(nz)
    else:
        kq1, kq2 = (q1[None, :] + 0.5) / chis[:, None], (q2[None, :] + 0.5) / chis[:, None]
        zw = (_trapz_w(zs) if nz > 1 else np.ones(1)) * pref
    wn = _trapz_w(ms)[None, :] * nzm * zw[:, None]
    kqs = (kq1, kq1, kq2, kq2)
    us = [_interp(c, ks, kqs[i]) for i, (_, c, _) in enumerate(legs)]
    uc = [_interp(c, ks, kqs[i]) if c is not None else np.ones_like(us[i]) for i, (_, _, c) in enumerate(legs)]
    t = []
    for i, (kind, _, _) in enumerate(legs):
        if kind == KIND_HOD:
            t.append((hod["Nc"][..., None] * uc[i] + hod["Ns"][..., None] * us[i]) / hod["ngal"][:, None, None])
        else:
            t.append((ms / rho)[None, :, None] * us[i] if kind == KIND_MATTER else us[i])
    gal = [i for i, (kind, _, _) in enumerate(legs) if kind == KIND_HOD]
    terms = []                        # (coefficient [nz, nm], factor at k1 [nz, nm, n1], factor at k2 [nz, nm, n2])
    if len(gal) <= 1:
        terms.append((wn, t[0] * t[1], t[2] * t[3]))
    else:
        p, q = gal
        ig2 = 1.0 / hod["ngal"][:, None] ** 2
        rest = [i for i in range(4) if i not in gal]

        def side(fp, fq):             # the k1 and k2 factors of u_?(p) u_?(q) times the other legs
            f = {p: fp, q: fq}
            for i in rest:
                f[i] = t[i]
            return f[0] * f[1], f[2] * f[3]

        for c, fp, fq in ((hod["NsNsm1"], us[p], us[q]), (hod["NcNs"], uc[p], us[q]), (hod["NcNs"], us[p], uc[q])):
            terms.append((wn * c * ig2, *side(fp, fq)))
    val = bnd = 0.0
    for c, f1, f2 in terms:
        P1, P2 = c[..., None] * f1, f2
        if chis is None:
            v = np.einsum("zml,zmn->zln", P1, P2)
            b = np.einsum("zml,zmn->zln", np.abs(P1), np.abs(P2))
        else:
            A, B = P1.reshape(-1, q1.size), P2.reshape(-1, q2.size)
            v, b = A.T @ B, np.abs(A).T @ np.abs(B)
        val, bnd = val + v, bnd + b
    return val, bnd


def _assert_bound(name, got, want, bound, tau=TAU):
    got, want, bound = (np.asarray(a, dtype=np.float64) for a in (got, want, bound))
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    err = np.abs(got - want)
    zero = bound == 0.0
    assert np.all(err[zero] == 0.0), "%s: error where every term is zero" % name
    ratio = float(np.max(err[~zero] / bound[~zero])) if (~zero).any() else 0.0
    assert ratio <= tau, "%s: max |got-want| / sum|terms| = %.3g > %.1g" % (name, ratio, tau)


def _nseg(kinds):
    g1 = KIND_HOD in kinds[:2]
    g2 = KIND_HOD in kinds[2:]
    return 2 if list(kinds).count(KIND_HOD) == 2 and g1 and g2 else 1


def _plan(proj, nz, nm, n1, n2, nseg):
    """trispec_plan of k_trispec.cu restated with nseg segments of mass rows per redshift: (MT, splits, K chunk)."""
    cd = lambda a, b: -(-a // b)
    mt = 4 if n1 <= 32 else 8 if n1 <= 64 else 16 if n1 <= 128 else 26
    rows = nseg * (nm + nm % 2)
    if not proj:
        return mt, 1, rows
    K = nz * rows
    s = (16 * 148 * (1 if mt > 16 else 2)) // (cd(n2 + n2 % 2, 64) * cd(n1, 8 * mt))
    s = min(max(s, 1), 64, cd(K, 128))
    kchunk = cd(cd(K, s), 16) * 16
    return mt, cd(K, kchunk), kchunk


def _ws_expected(proj, nz, nm, n1, n2, nseg):
    mt, ns, _ = _plan(proj, nz, nm, n1, n2, nseg)
    K, ld1, ld2 = nz * nseg * (nm + nm % 2), n1 + n1 % 2, n2 + n2 % 2
    return K * (ld1 + ld2) + (1 if proj else nz) * ns * n1 * ld2


# ------------------------------------------------------------------------------------------------- CPU-only
def _dummy_legs(capi, p, kinds, occ=None, uc=None):
    legs = (capi.Tracer * 4)()
    for i, k in enumerate(kinds):
        legs[i].kind = k
        legs[i].us_d = p[3 + i].value if k != KIND_HOD else p[3].value
        if k == KIND_HOD:
            o = occ if occ is not None else p[12:17]
            legs[i].uc_d = uc
            legs[i].Nc_d, legs[i].Ns_d, legs[i].NcNs_d, legs[i].NsNsm1_d, legs[i].ngal_d = [x.value for x in o]
    return legs


def test_tracer_trispec_rejects_before_any_launch():
    """Every refusal of the tracer entry points returns its own code and message before the first launch (valid-looking
    dummy device pointers, no GPU); the workspace functions agree with the plan restated in _plan, counting segments;
    the API refuses three or four HOD legs and two HODs before touching the device."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    p = [C.c_void_p(0x10000 + 0x100 * i) for i in range(20)]          # non-null, 16-byte aligned, never dereferenced
    ok = _dummy_legs(capi, p, (KIND_HOD, KIND_MATTER, KIND_HOD, KIND_PRESSURE))

    def tri(legs=ok, nz=2, nm=40, nk=30, ldk=32, ws=p[9]):
        return L.hmv_trispec_1h_tracers(nz, nm, nk, ldk, p[0], p[1], p[2], 1.0, legs, 5, p[7], 6, p[8], ws, p[10], None)

    def cov(legs=ok, nz=2, nm=40, chis=p[11]):
        return L.hmv_cl_cov_1h_tracers(nz, nm, 30, 32, p[0], p[1], p[2], 1.0, legs, 5, p[7], 6, p[8], p[1], chis, p[2],
                                       p[9], p[10], None)

    def edit(legs, i, **kw):
        out = (capi.Tracer * 4)(*legs)
        for k, v in kw.items():
            setattr(out[i], k, v)
        return out

    three = _dummy_legs(capi, p, (KIND_HOD, KIND_HOD, KIND_HOD, KIND_MATTER))
    four = _dummy_legs(capi, p, (KIND_HOD,) * 4)
    cases = {
        "null Nc": (lambda: tri(edit(ok, 2, Nc_d=None)), HMV_E_ARG, "HOD leg 2 lacks occupation arrays"),
        "null ngal": (lambda: tri(edit(ok, 0, ngal_d=None)), HMV_E_ARG, "HOD leg 0 lacks occupation arrays"),
        "three HOD legs": (lambda: tri(three), HMV_E_ARG, "3 HOD legs"),
        "four HOD legs": (lambda: cov(four), HMV_E_ARG, "4 HOD legs"),
        "two HODs (occupation)": (lambda: tri(edit(ok, 2, NcNs_d=p[18].value)), HMV_E_ARG, "legs 0 and 2 differ"),
        "two HODs (central)": (lambda: tri(edit(ok, 2, uc_d=p[19].value)), HMV_E_ARG, "legs 0 and 2 differ"),
        "bias": (lambda: tri(edit(ok, 1, bias_d=p[18].value)), HMV_E_ARG, "leg 1: bias_d"),
        "hod bias": (lambda: cov(edit(ok, 0, bias_d=p[18].value)), HMV_E_ARG, "leg 0: bias_d"),
        "kind 3": (lambda: tri(edit(ok, 3, kind=3)), HMV_E_ARG, "leg 3: kind 3"),
        "null legs": (lambda: tri(legs=None), HMV_E_ARG, "hmv_trispec_1h_tracers: null pointer"),
        "null cube": (lambda: tri(edit(ok, 1, us_d=None)), HMV_E_ARG, "null pointer (cube 1)"),
        "misaligned cube": (lambda: tri(edit(ok, 3, us_d=0x20008)), HMV_E_ARG, "cube 3 must be 16-byte aligned"),
        "misaligned central": (lambda: tri(edit(edit(ok, 0, uc_d=0x20008), 2, uc_d=0x20008)), HMV_E_ARG,
                               "cube 0 must be 16-byte aligned"),
        "odd ldk": (lambda: tri(ldk=31), HMV_E_ARG, "ldk must be even"),
        "nz = 0": (lambda: tri(nz=0), HMV_E_ARG, "sizes must be >= 1"),
        "misaligned ws": (lambda: tri(ws=C.c_void_p(0x20008)), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "cov null chis": (lambda: cov(chis=None), HMV_E_ARG, "hmv_cl_cov_1h_tracers: null pointer (zs, chis or pref)"),
        "nz > 65535": (lambda: tri(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        # 40000 * 2 * 14000 > 2^30 > 40000 * 14000: only the two segments of the split pair exceed the limit
        "K > 2^30 with segments": (lambda: cov(nz=40000, nm=14000), HMV_E_LIMIT, "nz * nm * segments"),
    }
    for what, (call, code, msg) in cases.items():
        rc = call()
        assert rc == code and msg in capi.last_error(), (what, rc, capi.last_error())
    same_side = _dummy_legs(capi, p, (KIND_HOD, KIND_HOD, KIND_MATTER, KIND_PRESSURE))
    assert cov(same_side, nz=60000, nm=20000) == HMV_E_LIMIT and "nz * nm = " in capi.last_error()
    # the profile entry points still refuse kind 1 with the same message
    u = (C.c_void_p * 4)(*p[3:7])
    rc = L.hmv_trispec_1h(2, 40, 30, 32, p[0], p[1], p[2], 1.0, u, (C.c_int * 4)(0, 1, 2, 2), 5, p[7], 6, p[8], p[9],
                          p[10], None)
    assert rc == HMV_E_ARG and "kind 1 is neither" in capi.last_error()

    for proj, fn in ((False, L.hmv_trispec_1h_tracers_ws_doubles), (True, L.hmv_cl_cov_1h_tracers_ws_doubles)):
        assert fn(0, 4, 3, 3, ok) == 0 and fn(2, 4, 3, 3, None) == 0
        for kinds in ((0, 0, 2, 2), (1, 0, 0, 0), (1, 1, 0, 2), (0, 2, 1, 1), (1, 0, 1, 2), (0, 1, 1, 0)):
            legs = _dummy_legs(capi, p, kinds)
            for nz, nm, n1, n2 in [(1, 1, 1, 1), (3, 41, 7, 65), (6, 101, 1000, 1000), (200, 2000, 1000, 1000)]:
                assert fn(nz, nm, n1, n2, legs) == _ws_expected(proj, nz, nm, n1, n2, _nseg(kinds)), \
                    (proj, kinds, nz, nm, n1, n2)
            old = (L.hmv_cl_cov_1h_ws_doubles if proj else L.hmv_trispec_1h_ws_doubles)(6, 101, 1000, 1000)
            assert (fn(6, 101, 1000, 1000, legs) == old) == (_nseg(kinds) == 1)

    from hmvec_b200.hmvec import HaloModel

    class Stub(HaloModel):
        def __init__(self):
            self._zcomm, self.uk_profiles, self.pk_profiles = None, {"nfw": None}, {"y": None}
            self.hods, self._ks64, self._nz = {"g": None, "g2": None}, np.geomspace(1e-3, 10, 20), 4
    h = Stub()
    for call, match in ((lambda: h.get_trispectrum_1halo([0.1], name="g"), "4 HOD legs"),
                        (lambda: h.get_trispectrum_1halo([0.1], name="g", name2="g", name3="g", name4="nfw"),
                         "3 HOD legs"),
                        (lambda: h.get_trispectrum_1halo([0.1], ks2=[0.2], name="g", name2="nfw", name3="g2",
                                                         name4="nfw"), "two HODs"),
                        (lambda: h.get_trispectrum_1halo([0.1], name="g", name2="g2", name3="y"), "two HODs"),
                        (lambda: h.get_trispectrum_1halo([0.1], name="g", name2="nope"), "no matter or pressure")):
        with pytest.raises(ValueError, match=match):
            call()


# ------------------------------------------------------------------------------------------------- GPU: the C ABI
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    return torch, capi


def _dev(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def _guarded(torch, n):
    buf = torch.full((2 * GUARD + n,), float("nan"), dtype=torch.float64, device="cuda")
    return buf, C.c_void_p(buf.data_ptr() + 8 * GUARD)


def _read_guarded(buf, n, shape):
    b = buf.cpu().numpy()
    g = np.r_[b[:GUARD], b[GUARD + n:]]
    assert np.all(g.view(np.int64) == NAN_BITS), "a guard around the output was written"
    return b[GUARD:GUARD + n].reshape(shape)


class AbiInputs(object):
    """Seeded cubes (NaN padding columns), mass function, occupations and multipoles or wavenumbers on the device."""

    def __init__(self, torch, nz, nm, n1, n2, seed, proj, central=True, pad=float("nan"), lo=-0.3):
        rng = np.random.default_rng(seed)
        self.nz, self.nm, self.n1, self.n2, self.proj = nz, nm, n1, n2, proj
        self.nk = nk = 37
        self.ldk = (nk + 15) // 16 * 16
        self.ks = np.geomspace(1e-2, 10.0, nk)
        self.ms = 1e13 * (1.0 + np.cumsum(rng.uniform(0.5, 1.5, nm)) / nm)
        wt = _trapz_w(self.ms) if nm > 1 else np.ones(1)
        self.nzm = rng.uniform(0.5, 2.0, (nz, nm)) / wt
        self.rho = 2e13
        self.cubes = {c: rng.uniform(lo, 1.2, (nz, nm, nk)) for c in ("a", "b", "s", "c")}
        self.cubes["one"] = np.ones((nz, nm, nk))
        self.central = central
        Nc = rng.uniform(0.0, 1.0, (nz, nm))
        Ns = rng.uniform(0.0, 4.0, (nz, nm))
        self.hod = dict(Nc=Nc, Ns=Ns, NcNs=Nc * Ns * rng.uniform(0.5, 1.0, (nz, nm)),
                        NsNsm1=Ns * Ns * rng.uniform(0.5, 1.0, (nz, nm)), ngal=rng.uniform(0.5, 2.0, nz))
        self.zs = np.sort(rng.uniform(0.1, 3.0, nz)) if nz > 1 else np.array([0.7])
        self.chis = 1000.0 + 2000.0 * self.zs
        self.pref = rng.uniform(0.5, 2.0, nz)
        if proj:
            self.q1, self.q2 = rng.uniform(2.0, 2e4, n1), rng.uniform(2.0, 2e4, n2)
        else:
            self.q1, self.q2 = rng.uniform(3e-3, 20.0, n1), rng.uniform(3e-3, 20.0, n2)
        self.dcubes = {}
        for k, c in self.cubes.items():
            t = torch.full((nz, nm, self.ldk), pad, dtype=torch.float64, device="cuda")
            t[..., :nk] = _dev(torch, c)
            self.dcubes[k] = t
        self.d = {k: _dev(torch, getattr(self, k)) for k in ("ks", "ms", "nzm", "zs", "chis", "pref", "q1", "q2")}
        self.dhod = {k: _dev(torch, v) for k, v in self.hod.items()}

    def legs(self, capi, spec):
        """spec: four of 'g' (the HOD: satellite cube 's', central cube 'c' or none), ('m', cube) or ('p', cube)."""
        legs = (capi.Tracer * 4)()
        host = []
        for i, s in enumerate(spec):
            if s == "g":
                legs[i].kind = KIND_HOD
                legs[i].us_d = self.dcubes["s"].data_ptr()
                legs[i].uc_d = self.dcubes["c"].data_ptr() if self.central else None
                h = self.dhod
                legs[i].Nc_d, legs[i].Ns_d = h["Nc"].data_ptr(), h["Ns"].data_ptr()
                legs[i].NcNs_d, legs[i].NsNsm1_d, legs[i].ngal_d = (h["NcNs"].data_ptr(), h["NsNsm1"].data_ptr(),
                                                                    h["ngal"].data_ptr())
                host.append((KIND_HOD, self.cubes["s"], self.cubes["c"] if self.central else None))
            else:
                kind = KIND_MATTER if s[0] == "m" else KIND_PRESSURE
                legs[i].kind = kind
                legs[i].us_d = self.dcubes[s[1]].data_ptr()
                host.append((kind, self.cubes[s[1]], None))
        return legs, host

    def shape(self):
        return (self.n1, self.n2) if self.proj else (self.nz, self.n1, self.n2)

    def run(self, torch, capi, legs, old=None):
        """One tracer ABI launch twice (bit-identical, guards intact); old = (u_h, kind_h) runs the profile entry point
        instead."""
        L, p, d = capi.lib, capi.ptr, self.d
        nz, nm, n1, n2 = self.nz, self.nm, self.n1, self.n2
        if old is None:
            nws = (L.hmv_cl_cov_1h_tracers_ws_doubles if self.proj else L.hmv_trispec_1h_tracers_ws_doubles)(
                nz, nm, n1, n2, legs)
            assert nws == _ws_expected(self.proj, nz, nm, n1, n2, _nseg([legs[i].kind for i in range(4)]))
        else:
            nws = (L.hmv_cl_cov_1h_ws_doubles if self.proj else L.hmv_trispec_1h_ws_doubles)(nz, nm, n1, n2)
        ws = torch.empty(int(nws), dtype=torch.float64, device="cuda")
        shape = self.shape()
        n = int(np.prod(shape))
        buf, optr = _guarded(torch, n)

        def launch():
            common = (nz, nm, self.nk, self.ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), self.rho)
            proj = (p(d["zs"]), p(d["chis"]), p(d["pref"])) if self.proj else ()
            if old is None:
                fn = L.hmv_cl_cov_1h_tracers if self.proj else L.hmv_trispec_1h_tracers
                rc = fn(*common, legs, n1, p(d["q1"]), n2, p(d["q2"]), *proj, p(ws), optr, capi.stream())
            else:
                fn = L.hmv_cl_cov_1h if self.proj else L.hmv_trispec_1h
                rc = fn(*common, old[0], old[1], n1, p(d["q1"]), n2, p(d["q2"]), *proj, p(ws), optr, capi.stream())
            capi.check(rc, "trispectrum ABI")

        launch()
        torch.cuda.synchronize()
        first = buf.clone()
        launch()
        torch.cuda.synchronize()
        assert torch.equal(first.view(torch.int64), buf.view(torch.int64)), "second launch differs"
        return _read_guarded(buf, n, shape)

    def reference(self, host):
        extra = (self.chis, self.zs, self.pref) if self.proj else ()
        return _reference(host, self.hod, self.ms, self.nzm, self.rho, self.ks, self.q1, self.q2, *extra)


SPLIT = ("g", ("m", "a"), ("p", "b"), "g")          # one galaxy leg on each side: two segments
SAME = (("m", "a"), ("p", "b"), "g", "g")           # both on side 2: one segment

COV_CASES = [  # (n1, n2, nz, nm, MT, split-k > 1)
    (1, 1, 1, 2, 4, False),
    (7, 7, 3, 41, 4, False),
    (63, 64, 2, 30, 8, False),
    (64, 63, 1, 1, 8, False),           # nm = 1: trapz over one mass is zero
    (65, 65, 4, 17, 16, False),
    (7, 209, 9, 33, 4, True),           # K chunks of 16 rows cross the 34-row segments and the redshift blocks
    (209, 7, 5, 40, 26, True),
    (1000, 1000, 6, 101, 26, True),
    (1000, 1, 1, 300, 26, True),        # nz = 1: split-k over the segments of the mass axis
    (63, 1000, 12, 21, 8, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [SPLIT, SAME], ids=["split", "same"])
@pytest.mark.parametrize("n1,n2,nz,nm,mt,split", COV_CASES)
def test_tracer_cov_plans(env, n1, n2, nz, nm, mt, split, spec):
    torch, capi = env
    nseg = _nseg([KIND_HOD if s == "g" else 0 for s in spec])
    got_mt, ns, kchunk = _plan(True, nz, nm, n1, n2, nseg)
    assert got_mt == mt and (nseg == 2 or (ns > 1) == split), (got_mt, ns)    # two segments double K
    if ns > 1 and nz * nseg > 1:
        assert kchunk % (nm + nm % 2) != 0, "K chunks should cross segment boundaries"
    inp = AbiInputs(torch, nz, nm, n1, n2, seed=n1 * 31 + n2 + nz * 7 + nm + nseg, proj=True)
    legs, host = inp.legs(capi, spec)
    got = inp.run(torch, capi, legs)
    want, bnd = inp.reference(host)
    _assert_bound("cov_abi %s n1=%d n2=%d nz=%d nm=%d" % (spec, n1, n2, nz, nm), got, want, bnd)


TRI_CASES = [  # (n1, n2, nz, nm, MT)
    (1, 1, 1, 1, 4),
    (7, 65, 3, 41, 4),
    (65, 64, 2, 30, 16),
    (209, 63, 4, 21, 26),
    (1000, 7, 2, 33, 26),
    (63, 1000, 1, 40, 8),
]

TRI_SPECS = [SPLIT, SAME, (("p", "a"), "g", "g", ("m", "b")), ("g", "g", ("m", "a"), ("m", "a")),
             (("m", "a"), "g", ("p", "b"), ("m", "a"))]


@pytest.mark.gpu
@pytest.mark.parametrize("spec", TRI_SPECS, ids=["split", "same2", "split2", "same1", "single"])
@pytest.mark.parametrize("n1,n2,nz,nm,mt", TRI_CASES)
def test_tracer_trispec_plans(env, n1, n2, nz, nm, mt, spec):
    torch, capi = env
    nseg = _nseg([KIND_HOD if s == "g" else 0 for s in spec])
    assert _plan(False, nz, nm, n1, n2, nseg)[:2] == (mt, 1)
    for central in (True, False):
        inp = AbiInputs(torch, nz, nm, n1, n2, seed=n1 + 17 * n2 + nz + nm, proj=False, central=central)
        legs, host = inp.legs(capi, spec)
        got = inp.run(torch, capi, legs)
        want, bnd = inp.reference(host)
        _assert_bound("trispec_abi %s central=%s n1=%d n2=%d nz=%d nm=%d" % (spec, central, n1, n2, nz, nm), got,
                      want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("proj", [False, True], ids=["trispec", "cov"])
def test_profile_legs_match_profile_entry_points(env, proj):
    """Profile legs through the tracer entry points give the profile entry points' result to the bit."""
    torch, capi = env
    for n1, n2, nz, nm in ((7, 65, 3, 41), (1000, 1000, 6, 101)):
        inp = AbiInputs(torch, nz, nm, n1, n2, seed=nz * nm, proj=proj)
        spec = (("m", "a"), ("p", "b"), ("m", "b"), ("p", "a"))
        legs, _ = inp.legs(capi, spec)
        new = inp.run(torch, capi, legs)
        u_h = (C.c_void_p * 4)(*[legs[i].us_d for i in range(4)])
        k_h = (C.c_int * 4)(*[legs[i].kind for i in range(4)])
        old = inp.run(torch, capi, None, old=(u_h, k_h))
        assert np.array_equal(new.view(np.int64), old.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("central", [False, True], ids=["no-central", "central"])
def test_pair_moment_is_power_1halo(env, central):
    """Legs (g, g) at k1 and cubes of ones (kind 2) for C and D: T[z][i][j] = hmv_power's P1h of (g, g) divided by its
    damping factor 1 - exp(-(k/k*)^2), at grid k where that factor is >= 1/2."""
    torch, capi = env
    nz, nm, kstar = 3, 29, 0.1
    inp = AbiInputs(torch, nz, nm, 1, 3, seed=11, proj=False, central=central, pad=0.0, lo=0.05)   # no cancellation
    inp.q1 = inp.ks.copy()
    inp.n1 = inp.nk
    inp.d["q1"] = _dev(torch, inp.q1)
    legs, _ = inp.legs(capi, ("g", "g", ("p", "one"), ("p", "one")))
    got = inp.run(torch, capi, legs)
    L, p = capi.lib, capi.ptr
    A = legs[0]
    bh = _dev(torch, np.ones((nz, nm)))
    Pzk = _dev(torch, np.ones((nz, inp.nk)))
    ws = torch.empty(int(L.hmv_power_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")
    p1h = torch.empty((nz, inp.nk), dtype=torch.float64, device="cuda")
    capi.check(L.hmv_power(nz, nm, inp.nk, inp.ldk, p(inp.d["ms"]), p(inp.d["ks"]), p(inp.d["nzm"]), p(bh), p(Pzk),
                           inp.rho, kstar, C.byref(A), C.byref(A), p(ws), p(p1h), None, capi.stream()), "hmv_power")
    torch.cuda.synchronize()
    damp = 1.0 - np.exp(-(inp.ks / kstar) ** 2)
    use = damp >= 0.5
    assert use.sum() >= 20
    want = p1h.cpu().numpy()[:, use] / damp[use]
    for j in range(inp.n2):
        np.testing.assert_allclose(got[:, use, j], want, rtol=TAU, atol=0)


# ------------------------------------------------------------------------------------------------- GPU: HaloModel API
@pytest.fixture(scope="module")
def model(env):
    import hmvec_b200 as hm
    zs = np.array([0.05, 0.7, 1.5, 2.8])
    ms = np.geomspace(1e11, 1e16, 47)
    ks = np.geomspace(1e-3, 30, 130)
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low', device="cuda:0")
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)   # table-backed Compton-y
    h.add_hod("g", ngal=np.geomspace(2e-3, 5e-5, zs.size))                # the bisection is resolved at the download
    h.add_hod("gc", mthresh=np.geomspace(3e10, 1e10, zs.size), corr="min", central_profile_name="electron")
    host = dict(zs=zs, ms=h.ms, ks=h._ks64, nzm=h.nzm, rho=h._rho_m0,
                chis=np.asarray(h.comoving_radial_distance(zs), dtype=np.float64),
                H=np.asarray(h.h_of_z(zs), dtype=np.float64), Wk=h.lensing_window(zs, 3.0))
    dndz = np.exp(-0.5 * ((zs - 0.8) / 0.6) ** 2)
    host["Wg"] = dndz / np.sum(_trapz_w(zs) * dndz)
    host["cube"] = {"nfw": (KIND_MATTER, h.uk_profiles["nfw"], None), "electron": (KIND_MATTER,
                                                                                  h.uk_profiles["electron"], None),
                    "y": (KIND_PRESSURE, h.pk_profiles["y"], None),
                    "g": (KIND_HOD, h.uk_profiles["nfw"], None), "gc": (KIND_HOD, h.uk_profiles["nfw"],
                                                                      h.uk_profiles["electron"])}
    host["hod"] = {n: {k: h.hods[n][k] for k in ("Nc", "Ns", "NcNs", "NsNsm1", "ngal")} for n in ("g", "gc")}
    return h, host


COMBOS = [("nfw", "g", "nfw", "g"), ("nfw", "nfw", "nfw", "g"), ("nfw", "nfw", "g", "g"), ("g", "g", "nfw", "nfw"),
          ("y", "g", "y", "g"), ("g", "y", "nfw", "nfw"), ("gc", "nfw", "gc", "nfw"), ("nfw", "y", "gc", "gc"),
          ("gc", "gc", "y", "electron")]


def _model_ref(host, names, q1, q2, windows=None, fsky=1.0):
    legs = [host["cube"][n] for n in names]
    hn = [n for n in names if n in host["hod"]]
    hod = host["hod"][hn[0]] if hn else None
    if windows is None:
        return _reference(legs, hod, host["ms"], host["nzm"], host["rho"], host["ks"], q1, q2)
    W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), host["zs"].shape) for w in windows], axis=0)
    pref = host["H"] ** 3 * W / host["chis"] ** 6 / (4 * np.pi * fsky)
    return _reference(legs, hod, host["ms"], host["nzm"], host["rho"], host["ks"], q1, q2, host["chis"], host["zs"],
                      pref)


def _win(host, names):
    return tuple(1.0 if n == "y" else host["Wg"] if n in ("g", "gc") else host["Wk"] for n in names)


@pytest.mark.gpu
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_trispectrum_hod_tracers(model, names):
    """3D mode: k on the grid, between grid points, below and above the grid (clamped), unsorted."""
    h, host = model
    ks = host["ks"]
    k1 = np.array([ks[40], np.sqrt(ks[10] * ks[11]), 1e-5, 100.0, ks[0], ks[-1], 0.5 * (ks[3] + ks[4])])
    k2 = np.array([3.0, ks[70], 2e-4, np.sqrt(ks[100] * ks[101]), 45.0])
    got = h.get_trispectrum_1halo(k1, k2, *names)
    want, bnd = _model_ref(host, names, k1, k2)
    _assert_bound("trispec_model %s" % "-".join(names), got, want, bnd)
    assert got.shape == (4, k1.size, k2.size)


@pytest.mark.gpu
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_cl_cov_hod_tracers(model, names):
    """Projected mode: unsorted multipoles, l = 2 (k below ks at high z) and l = 2e4 (k above ks at low z), ells2 !=
    ells, fsky < 1; kappa windows from lensing_window, galaxy windows a normalised dN/dz, y windows of 1."""
    h, host = model
    ells = np.array([300.0, 2.0, 20000.0, 45.5, 1000.0, 7.0, 3000.0])
    ells2 = np.array([10.0, 5000.0, 2.0, 150.0])
    win = _win(host, names)
    got = h.get_cl_cov_1halo(ells, *names, windows=win, fsky=0.4, ells2=ells2)
    want, bnd = _model_ref(host, names, ells, ells2, win, 0.4)
    _assert_bound("cov_model %s" % "-".join(names), got, want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("g", ["g", "gc"])
def test_split_pair_equals_same_side_pair_at_equal_k(model, g):
    """<g g>(k, k) is the same whether the two galaxy legs sit on one side or on both: T^{gX,gY}(k,k) = T^{gg,XY}(k,k)."""
    h, host = model
    ks = host["ks"]
    k = np.array([ks[5], 0.37, ks[64], 2.2, ks[120], 1e-4, 50.0])
    a = h.get_trispectrum_1halo(k, k, g, "nfw", g, "y")
    b = h.get_trispectrum_1halo(k, k, g, g, "nfw", "y")
    _, bnd = _model_ref(host, (g, "nfw", g, "y"), k, k)
    i = np.arange(k.size)
    _assert_bound("split_vs_same %s" % g, a[:, i, i], b[:, i, i], bnd[:, i, i])


@pytest.mark.gpu
def test_cl_cov_hod_structure(model):
    """Cov^{AB,CD}(l,l') = Cov^{CD,AB}(l',l), A <-> B leaves it unchanged, and the C_kg x C_kg auto covariance is
    symmetric with the spectrum of the host restatement.  It is positive semi-definite only up to the central self-pairs
    that <g g> excludes (NcNs (u_c u_s' + u_s u_c') is indefinite): on this model the exact matrix has eigenvalues near
    -5e-11 of its trace, far above the eigensolver's and the kernel's error, so its smallest eigenvalue is held to the
    restatement's rather than to zero."""
    h, host = model
    ells = np.geomspace(10, 1e4, 40)
    ells2 = np.geomspace(30, 3e3, 25)
    Wk, Wg = host["Wk"], host["Wg"]
    for names in (("nfw", "g", "nfw", "nfw"), ("nfw", "gc", "y", "gc"), ("g", "g", "nfw", "y")):
        win = _win(host, names)
        a = h.get_cl_cov_1halo(ells, *names, windows=win, ells2=ells2)
        b = h.get_cl_cov_1halo(ells2, *names[2:], *names[:2], windows=win[2:] + win[:2], ells2=ells)
        c = h.get_cl_cov_1halo(ells, names[1], names[0], *names[2:], windows=(win[1], win[0]) + win[2:], ells2=ells2)
        _, bnd = _model_ref(host, names, ells, ells2, win)
        _assert_bound("cov_transpose %s" % "-".join(names), a, b.T, bnd)
        _assert_bound("cov_swap %s" % "-".join(names), a, c, bnd)
    for g in ("g", "gc"):
        c = h.get_cl_cov_1halo(ells, "nfw", g, "nfw", g, windows=(Wk, Wg, Wk, Wg))
        want, bnd = _model_ref(host, ("nfw", g, "nfw", g), ells, ells, (Wk, Wg, Wk, Wg))
        _assert_bound("cov_symmetric %s" % g, c, c.T, bnd)
        ev = np.linalg.eigvalsh(0.5 * (c + c.T))
        ev_ref = np.linalg.eigvalsh(0.5 * (want + want.T))
        tol = ells.size * TAU * bnd.max() + 1e-14 * ev_ref.max()     # ||error||_2 <= n max|error| (Weyl)
        assert np.all(np.abs(ev - ev_ref) <= tol), (g, np.abs(ev - ev_ref).max(), tol)


@pytest.mark.gpu
def test_api_hod_defaults_and_rejections(model):
    h, host = model
    ells = np.array([100.0, 1000.0])
    np.testing.assert_array_equal(h.get_cl_cov_1halo(ells, "nfw", "g"),
                                  h.get_cl_cov_1halo(ells, "nfw", "g", "nfw", "nfw", ells2=ells))
    np.testing.assert_array_equal(h.get_trispectrum_1halo([0.1, 1.0], name="g", name3="nfw"),
                                  h.get_trispectrum_1halo([0.1, 1.0], [0.1, 1.0], "g", "g", "nfw", "nfw"))
    with pytest.raises(ValueError, match="HOD"):
        h.get_cl_cov_1halo(ells, "g")
    with pytest.raises(ValueError, match="two HODs"):
        h.get_trispectrum_1halo([0.1], name="g", name2="nfw", name3="gc", name4="nfw")
    with pytest.raises(ValueError, match="HOD"):
        h.get_trispectrum_2halo([0.1], name="nfw", name4="g")
    with pytest.raises(ValueError, match="HOD"):
        h.get_cl_cov_ssc(ells, "g")
