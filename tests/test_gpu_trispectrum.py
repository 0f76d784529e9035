"""The 1-halo trispectrum (hmv_trispec_1h, HaloModel.get_trispectrum_1halo) and the non-Gaussian Limber covariance of
C_l (hmv_cl_cov_1h, HaloModel.get_cl_cov_1halo), against a float64 numpy restatement of their definitions on the same
downloaded inputs: np.interp for u(k), explicit trapezoid weights on ms and zs.

    T^{ABCD}(k1,k2;z) = sum_m w_m n(z,m) t_A(k1) t_B(k1) t_C(k2) t_D(k2),   t = (M/rho_m0 or 1) u
    Cov(l,l') = sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 / (4 pi fsky) T((l+1/2)/chi, (l'+1/2)/chi; z)

Each element is held to |got - want| <= tau * B, B the same reduction over absolute values.  Largest ratio measured on
one B200 (1000 W power limit): see TAU.  The ABI-driven cases use seeded random cubes in [-0.3, 1.2] with NaN padding
columns, n(M) with O(1) weight on every mass row, and NaN guards around the output; each is launched twice and must
give bit-identical output.  The shapes hit every launch plan of k_trispec.cu: MT = 4 / 8 / 16 / 26 output rows per
CTA with one to five row tiles, odd and even widths, nm = 1 and odd nm, a single split and split-k whose K chunks cross
redshift boundaries, and the trispectrum's batch over z.
"""
import ctypes as C

import numpy as np
import pytest

HMV_E_ARG, HMV_E_LIMIT = -1, -3
TAU = 1e-12             # largest ratio measured: see the module docstring of the commit that set it
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64
OBSERVED = {}


# ------------------------------------------------------------------------------------------------- host restatement
def _trapz_w(x):
    x = np.asarray(x, dtype=np.float64)
    n = x.size
    if n < 2:
        return np.zeros(n)
    return 0.5 * (x[np.minimum(np.arange(n) + 1, n - 1)] - x[np.maximum(np.arange(n) - 1, 0)])


def _legs(cube, kind, ms, rho, ks, kq):
    """t(z, m, l) = a(m) u(z, m, kq[z, l]) with np.interp (clamps to the end values outside ks)."""
    nz, nm = cube.shape[:2]
    a = ms / rho if kind == 0 else np.ones(nm)
    out = np.empty((nz, nm, kq.shape[1]))
    for z in range(nz):
        for m in range(nm):
            out[z, m] = a[m] * np.interp(kq[z], ks, cube[z, m])
    return out


def _reference(cubes, kinds, ms, nzm, rho, ks, q1, q2, chis=None, zs=None, pref=None):
    """(value, bound): T [nz, n1, n2] when chis is None, else Cov [n1, n2]."""
    nz, nm = cubes[0].shape[:2]
    if chis is None:
        kq1, kq2 = np.broadcast_to(q1, (nz, q1.size)), np.broadcast_to(q2, (nz, q2.size))
        zw = np.ones(nz)
    else:
        kq1, kq2 = (q1[None, :] + 0.5) / chis[:, None], (q2[None, :] + 0.5) / chis[:, None]
        zw = (_trapz_w(zs) if nz > 1 else np.ones(1)) * pref
    t = [_legs(c, k, ms, rho, ks, kq1 if i < 2 else kq2) for i, (c, k) in enumerate(zip(cubes, kinds))]
    wn = _trapz_w(ms)[None, :] * nzm * zw[:, None]
    P1, P2 = wn[..., None] * t[0] * t[1], t[2] * t[3]
    if chis is None:
        val = np.einsum("zml,zmn->zln", P1, P2)
        bnd = np.einsum("zml,zmn->zln", np.abs(P1), np.abs(P2))
    else:
        A, B = P1.reshape(-1, q1.size), P2.reshape(-1, q2.size)
        val, bnd = A.T @ B, np.abs(A).T @ np.abs(B)
    return val, bnd


def _assert_bound(name, got, want, bound, tau=TAU):
    got, want, bound = (np.asarray(a, dtype=np.float64) for a in (got, want, bound))
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    err = np.abs(got - want)
    zero = bound == 0.0
    assert np.all(err[zero] == 0.0), "%s: error where every term is zero" % name
    ratio = float(np.max(err[~zero] / bound[~zero])) if (~zero).any() else 0.0
    OBSERVED[name.split(" ")[0]] = max(OBSERVED.get(name.split(" ")[0], 0.0), ratio)
    assert ratio <= tau, "%s: max |got-want| / sum|terms| = %.3g > %.1g" % (name, ratio, tau)


def _plan(proj, nz, nm, n1, n2):
    """trispec_plan of k_trispec.cu restated: (MT, split-k factor, K chunk)."""
    cd = lambda a, b: -(-a // b)
    mt = 4 if n1 <= 32 else 8 if n1 <= 64 else 16 if n1 <= 128 else 26
    nmp = nm + nm % 2
    if not proj:
        return mt, 1, nmp
    K = nz * nmp
    s = (16 * 148 * (1 if mt > 16 else 2)) // (cd(n2 + n2 % 2, 64) * cd(n1, 8 * mt))
    s = min(max(s, 1), 64, cd(K, 128))
    kchunk = cd(cd(K, s), 16) * 16
    return mt, cd(K, kchunk), kchunk


def _ws_expected(proj, nz, nm, n1, n2):
    mt, ns, _ = _plan(proj, nz, nm, n1, n2)
    K, ld1, ld2 = nz * (nm + nm % 2), n1 + n1 % 2, n2 + n2 % 2
    return K * (ld1 + ld2) + (1 if proj else nz) * ns * n1 * ld2


# ------------------------------------------------------------------------------------------------- CPU-only
def test_trispec_rejects_before_any_launch():
    """Every argument and limit check of both entry points runs before the first launch: with valid-looking dummy
    device pointers and no GPU, each rejected call returns its own code and message, never a CUDA error.  The workspace
    functions agree with the launch plan restated in _plan."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    p = [C.c_void_p(0x10000 + 0x100 * i) for i in range(12)]          # non-null, 16-byte aligned, never dereferenced
    bad = C.c_void_p(0x20008)

    def cubes(*ptrs):
        return (C.c_void_p * 4)(*ptrs)

    def kinds(*k):
        return (C.c_int * 4)(*k)

    ok_u, ok_k = cubes(*p[3:7]), kinds(0, 0, 2, 2)

    def tri(nz=2, nm=40, nk=30, ldk=32, ks=p[0], u=ok_u, k=ok_k, ws=p[9]):
        return L.hmv_trispec_1h(nz, nm, nk, ldk, ks, p[1], p[2], 1.0, u, k, 5, p[7], 6, p[8], ws, p[10], None)

    def cov(chis=p[11], **kw):
        nz, nm, nk, ldk = kw.get("nz", 2), kw.get("nm", 40), kw.get("nk", 30), kw.get("ldk", 32)
        return L.hmv_cl_cov_1h(nz, nm, nk, ldk, p[0], p[1], p[2], 1.0, ok_u, ok_k, 5, p[7], 6, p[8], p[1], chis,
                               p[2], p[9], p[10], None)

    cases = {
        "nz = 0": (lambda: tri(nz=0), HMV_E_ARG, "sizes must be >= 1"),
        "nk = 1": (lambda: tri(nk=1, ldk=2), HMV_E_ARG, "nk >= 2"),
        "odd ldk": (lambda: tri(ldk=31), HMV_E_ARG, "ldk must be even"),
        "ldk < nk": (lambda: tri(ldk=28), HMV_E_ARG, "ldk must be even and >= nk"),
        "null ks": (lambda: tri(ks=None), HMV_E_ARG, "hmv_trispec_1h: null pointer"),
        "null cube": (lambda: tri(u=cubes(p[3], p[4], None, p[6])), HMV_E_ARG, "null pointer (cube 2)"),
        "hod kind": (lambda: tri(k=kinds(0, 1, 2, 2)), HMV_E_ARG, "kind 1 is neither"),
        "misaligned cube": (lambda: tri(u=cubes(p[3], bad, p[5], p[6])), HMV_E_ARG, "cube 1 must be 16-byte aligned"),
        "misaligned ws": (lambda: tri(ws=bad), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "cov null chis": (lambda: cov(chis=None), HMV_E_ARG, "hmv_cl_cov_1h: null pointer (zs, chis or pref)"),
        "cov odd ldk": (lambda: cov(ldk=33), HMV_E_ARG, "hmv_cl_cov_1h: ldk"),
        "nz > 65535": (lambda: tri(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        "K > 2^30": (lambda: cov(nz=60000, nm=20000), HMV_E_LIMIT, "exceeds 2^30"),
    }
    for what, (call, code, msg) in cases.items():
        rc = call()
        assert rc == code and msg in capi.last_error(), (what, rc, capi.last_error())
    assert L.hmv_trispec_1h_ws_doubles(0, 4, 3, 3) == 0 and L.hmv_cl_cov_1h_ws_doubles(2, 4, 0, 3) == 0
    for proj, fn in ((False, L.hmv_trispec_1h_ws_doubles), (True, L.hmv_cl_cov_1h_ws_doubles)):
        for nz, nm, n1, n2 in [(1, 1, 1, 1), (3, 41, 7, 65), (6, 101, 1000, 1000), (200, 2000, 1000, 1000)]:
            assert fn(nz, nm, n1, n2) == _ws_expected(proj, nz, nm, n1, n2), (proj, nz, nm, n1, n2)


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


def _abi_run(torch, capi, proj, nz, nm, n1, n2, kinds, seed, ones=False):
    """Seeded inputs, one ABI launch twice (bit-identical, guards intact), and the host reference."""
    rng = np.random.default_rng(seed)
    nk = 37
    ldk = (nk + 15) // 16 * 16
    ks = np.geomspace(1e-2, 10.0, nk)
    ms = 1e13 * (1.0 + np.cumsum(rng.uniform(0.5, 1.5, nm)) / nm)
    wt = _trapz_w(ms) if nm > 1 else np.ones(1)
    nzm = rng.uniform(0.5, 2.0, (nz, nm)) / wt
    rho = 2e13
    cubes = [np.ones((nz, nm, nk)) if ones else rng.uniform(-0.3, 1.2, (nz, nm, nk)) for _ in range(4)]
    dcubes = []
    for c in cubes:
        t = torch.full((nz, nm, ldk), float("nan"), dtype=torch.float64, device="cuda")   # NaN padding columns
        t[..., :nk] = _dev(torch, c)
        dcubes.append(t)
    zs = np.sort(rng.uniform(0.1, 3.0, nz)) if nz > 1 else np.array([0.7])
    chis = 1000.0 + 2000.0 * zs
    pref = rng.uniform(0.5, 2.0, nz)
    if proj:
        q1, q2 = rng.uniform(2.0, 2e4, n1), rng.uniform(2.0, 2e4, n2)      # k spans below ks[0] to above ks[-1]
    else:
        q1, q2 = rng.uniform(3e-3, 20.0, n1), rng.uniform(3e-3, 20.0, n2)
    d = {k: _dev(torch, v) for k, v in dict(ks=ks, ms=ms, nzm=nzm, zs=zs, chis=chis, pref=pref, q1=q1, q2=q2).items()}
    L, p = capi.lib, capi.ptr
    nws = (L.hmv_cl_cov_1h_ws_doubles if proj else L.hmv_trispec_1h_ws_doubles)(nz, nm, n1, n2)
    assert nws == _ws_expected(proj, nz, nm, n1, n2)
    ws = torch.empty(int(nws), dtype=torch.float64, device="cuda")
    shape = (n1, n2) if proj else (nz, n1, n2)
    n = int(np.prod(shape))
    buf, optr = _guarded(torch, n)
    u_h = (C.c_void_p * 4)(*[t.data_ptr() for t in dcubes])
    k_h = (C.c_int * 4)(*kinds)

    def launch():
        if proj:
            rc = L.hmv_cl_cov_1h(nz, nm, nk, ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), rho, u_h, k_h, n1, p(d["q1"]),
                                 n2, p(d["q2"]), p(d["zs"]), p(d["chis"]), p(d["pref"]), p(ws), optr, capi.stream())
        else:
            rc = L.hmv_trispec_1h(nz, nm, nk, ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), rho, u_h, k_h, n1, p(d["q1"]),
                                  n2, p(d["q2"]), p(ws), optr, capi.stream())
        capi.check(rc, "trispectrum ABI")

    launch()
    torch.cuda.synchronize()
    first = buf.clone()
    launch()
    torch.cuda.synchronize()
    assert torch.equal(first.view(torch.int64), buf.view(torch.int64)), "second launch differs"
    got = _read_guarded(buf, n, shape)
    ref = _reference(cubes, kinds, ms, nzm, rho, ks, q1, q2, *((chis, zs, pref) if proj else ()))
    return got, ref, dict(ms=ms, nzm=nzm, rho=rho)


COV_CASES = [  # (n1, n2, nz, nm, MT, split-k > 1)
    (1, 1, 1, 2, 4, False),
    (7, 7, 3, 41, 4, False),
    (63, 64, 2, 30, 8, False),
    (64, 63, 1, 1, 8, False),           # nm = 1: trapz over one mass is zero
    (65, 65, 4, 17, 16, False),
    (7, 209, 9, 33, 4, True),           # K chunks of 16 rows cross the 34-row redshift blocks
    (209, 7, 5, 40, 26, True),
    (1000, 1000, 6, 101, 26, True),     # five row tiles, 16 column strips, K chunks across redshifts
    (1000, 1, 1, 300, 26, True),        # nz = 1 with split-k over the mass axis
    (63, 1000, 12, 21, 8, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n1,n2,nz,nm,mt,split", COV_CASES)
def test_cov_plans(env, n1, n2, nz, nm, mt, split):
    torch, capi = env
    got_mt, ns, kchunk = _plan(True, nz, nm, n1, n2)
    assert got_mt == mt and (ns > 1) == split, (got_mt, ns)
    if split and nz > 1:
        assert kchunk % (nm + nm % 2) != 0, "K chunks should cross redshift boundaries"
    got, (want, bnd), _ = _abi_run(torch, capi, True, nz, nm, n1, n2, (0, 2, 0, 0), seed=n1 * 31 + n2 + nz * 7 + nm)
    _assert_bound("cov_abi n1=%d n2=%d nz=%d nm=%d" % (n1, n2, nz, nm), got, want, bnd)


TRI_CASES = [  # (n1, n2, nz, nm, MT)
    (1, 1, 1, 1, 4),
    (7, 65, 3, 41, 4),
    (65, 64, 2, 30, 16),
    (209, 63, 4, 21, 26),
    (1000, 7, 2, 33, 26),
    (63, 1000, 1, 40, 8),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n1,n2,nz,nm,mt", TRI_CASES)
def test_trispec_plans(env, n1, n2, nz, nm, mt):
    torch, capi = env
    assert _plan(False, nz, nm, n1, n2)[:2] == (mt, 1)
    got, (want, bnd), _ = _abi_run(torch, capi, False, nz, nm, n1, n2, (2, 0, 0, 2), seed=n1 + 17 * n2 + nz + nm)
    _assert_bound("trispec_abi n1=%d n2=%d nz=%d nm=%d" % (n1, n2, nz, nm), got, want, bnd)


@pytest.mark.gpu
def test_trispec_of_unit_cubes(env):
    """u = 1 on every cube: T = sum_m w_m n (M/rho_m0)^4 at every (k1, k2)."""
    torch, capi = env
    got, _, inp = _abi_run(torch, capi, False, 3, 25, 9, 70, (0, 0, 0, 0), seed=5, ones=True)
    want = (_trapz_w(inp["ms"])[None, :] * inp["nzm"] * (inp["ms"] / inp["rho"]) ** 4).sum(axis=1)
    bnd = (np.abs(_trapz_w(inp["ms"])[None, :] * inp["nzm"]) * (inp["ms"] / inp["rho"]) ** 4).sum(axis=1)
    _assert_bound("unit_cubes", got, np.broadcast_to(want[:, None, None], got.shape),
                  np.broadcast_to(bnd[:, None, None], got.shape))


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
    h.add_hod("g", ngal=np.geomspace(2e-3, 5e-5, zs.size))
    host = dict(zs=zs, ms=h.ms, ks=h._ks64, nzm=h.nzm, rho=h._rho_m0,
                chis=np.asarray(h.comoving_radial_distance(zs), dtype=np.float64),
                H=np.asarray(h.h_of_z(zs), dtype=np.float64), Wk=h.lensing_window(zs, 3.0))
    host["cube"] = {"nfw": (h.uk_profiles["nfw"], 0), "electron": (h.uk_profiles["electron"], 0),
                    "y": (h.pk_profiles["y"], 2)}
    return h, host


COMBOS = [("nfw", "nfw", "nfw", "nfw"), ("electron", "electron", "nfw", "nfw"), ("y", "y", "y", "y"),
          ("nfw", "y", "nfw", "y")]


def _model_ref(host, names, q1, q2, windows=None, fsky=1.0):
    cubes, kinds = zip(*[host["cube"][n] for n in names])
    if windows is None:
        return _reference(cubes, kinds, host["ms"], host["nzm"], host["rho"], host["ks"], q1, q2)
    W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), host["zs"].shape) for w in windows], axis=0)
    pref = host["H"] ** 3 * W / host["chis"] ** 6 / (4 * np.pi * fsky)
    return _reference(cubes, kinds, host["ms"], host["nzm"], host["rho"], host["ks"], q1, q2, host["chis"],
                      host["zs"], pref)


def _win(host, names):
    return tuple(1.0 if n == "y" else host["Wk"] for n in names)


@pytest.mark.gpu
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_trispectrum_tracers(model, names):
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
def test_cl_cov_tracers(model, names):
    """Projected mode: unsorted multipoles, l = 2 (k below ks at high z) and l = 2e4 (k above ks at low z), ells2 !=
    ells, fsky < 1, kappa windows from lensing_window and y windows of 1."""
    h, host = model
    ells = np.array([300.0, 2.0, 20000.0, 45.5, 1000.0, 7.0, 3000.0])
    ells2 = np.array([10.0, 5000.0, 2.0, 150.0])
    win = _win(host, names)
    got = h.get_cl_cov_1halo(ells, *names, windows=win, fsky=0.4, ells2=ells2)
    want, bnd = _model_ref(host, names, ells, ells2, win, 0.4)
    _assert_bound("cov_model %s" % "-".join(names), got, want, bnd)


@pytest.mark.gpu
def test_cl_cov_structure(model):
    """Cov^{AB,CD}(l,l') = Cov^{CD,AB}(l',l); the auto covariance is positive semi-definite."""
    h, host = model
    ells = np.geomspace(10, 1e4, 40)
    ells2 = np.geomspace(30, 3e3, 25)
    Wk = host["Wk"]
    a = h.get_cl_cov_1halo(ells, "nfw", "nfw", "y", "y", windows=(Wk, Wk, 1., 1.), ells2=ells2)
    b = h.get_cl_cov_1halo(ells2, "y", "y", "nfw", "nfw", windows=(1., 1., Wk, Wk), ells2=ells)
    _, bnd = _model_ref(host, ("nfw", "nfw", "y", "y"), ells, ells2, (Wk, Wk, 1., 1.))
    _assert_bound("cov_transpose", a, b.T, bnd)
    for names, win in ((("nfw",) * 4, (Wk,) * 4), (("y",) * 4, (1.,) * 4)):
        c = h.get_cl_cov_1halo(ells, *names, windows=win)
        ev = np.linalg.eigvalsh(0.5 * (c + c.T))
        assert ev.min() >= -TAU * np.trace(c), (names, ev.min(), np.trace(c))


@pytest.mark.gpu
def test_api_defaults_and_rejections(model):
    h, host = model
    ells = np.array([100.0, 1000.0])
    np.testing.assert_array_equal(h.get_cl_cov_1halo(ells, "nfw"), h.get_cl_cov_1halo(ells, "nfw", "nfw", "nfw", "nfw",
                                                                                        ells2=ells))
    np.testing.assert_array_equal(h.get_trispectrum_1halo([0.1, 1.0], name="y", name3="nfw"),
                                  h.get_trispectrum_1halo([0.1, 1.0], [0.1, 1.0], "y", "y", "nfw", "nfw"))
    with pytest.raises(ValueError, match="HOD"):
        h.get_cl_cov_1halo(ells, "g")
    with pytest.raises(ValueError, match="no matter or pressure profile"):
        h.get_trispectrum_1halo([0.1], name="nope")
    for bad in ([0.0, 1.0], [np.inf], [-3.0], []):
        with pytest.raises(ValueError, match="positive finite"):
            h.get_cl_cov_1halo(bad)
        with pytest.raises(ValueError, match="positive finite"):
            h.get_trispectrum_1halo([0.1], ks2=bad)
    for fsky in (0.0, 1.5, -0.1):
        with pytest.raises(ValueError, match="fsky"):
            h.get_cl_cov_1halo(ells, fsky=fsky)
    with pytest.raises(ValueError, match="length nz"):
        h.get_cl_cov_1halo(ells, windows=(1., np.ones(3), 1., 1.))
    ks = h._ks64
    try:
        h._ks64 = ks[::-1].copy()
        with pytest.raises(ValueError, match="strictly increasing"):
            h.get_trispectrum_1halo([0.1])
    finally:
        h._ks64 = ks
    try:
        h._zcomm = object()
        with pytest.raises(NotImplementedError):
            h.get_cl_cov_1halo(ells)
    finally:
        h._zcomm = None

