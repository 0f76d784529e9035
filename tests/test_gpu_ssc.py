"""The super-sample covariance (SSC) of C_l: the response of P^{AB} to a long-wavelength mode (hmv_power_response,
HaloModel.get_power_response), the variance of that mode over a disc (hmv_sigma_b2, HaloModel.get_sigma_b2) and the
Limber projection (hmv_cl_cov_ssc, HaloModel.get_cl_cov_ssc), against float64 numpy restatements of their definitions on
the same downloaded inputs: np.gradient, scipy.special.j1, simpson_weights, np.interp and explicit trapezoids.

    R1h(k,z) = sum_m w_m n b t_A t_B,   R2h(k,z) = [47/21 - n_eff/3] P_lin (I_A + b_A - C_A)(I_B + b_B - C_B)
    sigma_b^2(z) = sum_j s_j k_j/(2 pi) P(k_j, z) [2 J1(k_j R_z)/(k_j R_z)]^2
    Cov(l,l') = sum_z zeta_z H^3 W_A W_B W_C W_D sigma_b^2 / chi^4 R^{AB}((l+1/2)/chi, z) R^{CD}((l'+1/2)/chi, z)

Each element is held to |got - want| <= tau * B, B the same reduction over absolute values (for R2h: the bracket's and
n_eff's stencil terms taken in absolute value).  Largest ratio measured on one B200 (1000 W power limit): 9.5e-16
(response), 1.5e-14 (covariance), TAU = 1e-12; sigma_b^2 against scipy's j1 1.2e-11, TAU_J1 = 1e-10.  The ABI cases use seeded signed random cubes with NaN padding
columns, n(M) b(M) with O(1) weight on every mass row, a positive random P_lin on a non-uniform ks, and NaN guards
around every output; each is launched twice and must give bit-identical output.
"""
import ctypes as C

import numpy as np
import pytest

HMV_E_ARG, HMV_E_LIMIT = -1, -3
TAU = 1e-12
TAU_J1 = 1e-10          # sigma_b^2 against scipy: CUDA's j1 is held to an absolute error of 5e-12 for |x| >= 8, not ulps
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


def _neff(P, ks):
    """(n_eff, bound): np.gradient(log P, log ks, axis=1), and the same stencil over absolute values plus |n_eff| times
    the spacings' own terms, |ln k| / (its spacing)."""
    x, f = np.log(ks), np.log(P)
    n = np.gradient(f, x, axis=1)
    nb = np.empty_like(n)
    d = np.diff(x)
    ax = np.abs(x)
    nb[:, 0] = (np.abs(f[:, 1]) + np.abs(f[:, 0])) / d[0] + np.abs(n[:, 0]) * max(ax[0], ax[1]) / d[0]
    nb[:, -1] = (np.abs(f[:, -1]) + np.abs(f[:, -2])) / d[-1] + np.abs(n[:, -1]) * max(ax[-1], ax[-2]) / d[-1]
    if ks.size > 2:
        d1, d2 = d[:-1], d[1:]
        a, b, c = -d2 / (d1 * (d1 + d2)), (d2 - d1) / (d1 * d2), d1 / (d2 * (d1 + d2))
        xs = np.maximum(np.maximum(ax[:-2], ax[1:-1]), ax[2:]) / np.minimum(d1, d2)
        nb[:, 1:-1] = (np.abs(a) * np.abs(f[:, :-2]) + np.abs(b) * np.abs(f[:, 1:-1]) + np.abs(c) * np.abs(f[:, 2:]) +
                       np.abs(n[:, 1:-1]) * xs)
    return n, nb


def _response_ref(cubes, kinds, ms, nzm, bh, rho, ks, P):
    """(R1h, R2h) and their bounds on the [nz, nm, nk] cubes of legs A, B."""
    wnb = _trapz_w(ms)[None, :] * nzm * bh
    t, lab, lbd = [], [], []
    for cube, kind in zip(cubes, kinds):
        a = ms / rho if kind == 0 else np.ones(ms.size)
        tx = a[None, :, None] * cube
        I = np.einsum("zm,zmk->zk", wnb, tx)
        Ib = np.einsum("zm,zmk->zk", np.abs(wnb), np.abs(tx))
        if kind == 0:
            Cc = (wnb * a[None, :]).sum(axis=1)
            Cb = (np.abs(wnb) * a[None, :]).sum(axis=1)
            lab.append(I + 1.0 - Cc[:, None])
            lbd.append(Ib + 1.0 + Cb[:, None])
        else:
            lab.append(I)
            lbd.append(Ib)
        t.append(tx)
    r1 = np.einsum("zm,zmk,zmk->zk", wnb, t[0], t[1])
    r1b = np.einsum("zm,zmk,zmk->zk", np.abs(wnb), np.abs(t[0]), np.abs(t[1]))
    n, nb = _neff(P, ks)
    r2 = (47.0 / 21.0 - n / 3.0) * (P * lab[0] * lab[1])
    r2b = (47.0 / 21.0 + nb / 3.0) * (P * lbd[0] * lbd[1])
    return (r1, r1b), (r2, r2b)


def _disc_w2(x):
    from scipy.special import j1
    x = np.asarray(x, dtype=np.float64)
    w = np.ones_like(x)
    nz = x != 0
    w[nz] = 2.0 * j1(x[nz]) / x[nz]
    return w * w


def _sigma_b2_ref(ks, kw, P, R):
    terms = kw[None, :] * P * _disc_w2(ks[None, :] * R[:, None])
    return terms.sum(axis=1), np.abs(terms).sum(axis=1)


def _cov_ref(ks, rAB, rCD, l1, l2, zs, chis, pref):
    nz = zs.size
    zw = (_trapz_w(zs) if nz > 1 else np.ones(1)) * pref
    A = np.array([zw[z] * np.interp((l1 + 0.5) / chis[z], ks, rAB[z]) for z in range(nz)])
    B = np.array([np.interp((l2 + 0.5) / chis[z], ks, rCD[z]) for z in range(nz)])
    return A.T @ B, np.abs(A).T @ np.abs(B)


def _assert_bound(name, got, want, bound, tau=TAU):
    got, want, bound = (np.asarray(a, dtype=np.float64) for a in (got, want, bound))
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    err = np.abs(got - want)
    zero = bound == 0.0
    assert np.all(err[zero] == 0.0), "%s: error where every term is zero" % name
    ratio = float(np.max(err[~zero] / bound[~zero])) if (~zero).any() else 0.0
    key = name.split(" ")[0]
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), ratio)
    assert ratio <= tau, "%s: max |got-want| / sum|terms| = %.3g > %.1g" % (name, ratio, tau)


def _plan(nz, n1, n2):
    """ssc_plan of k_trispec.cu restated: (MT, split-k factor, K chunk); K = nz, one row per redshift."""
    cd = lambda a, b: -(-a // b)
    mt = 4 if n1 <= 32 else 8 if n1 <= 64 else 16 if n1 <= 128 else 26
    s = (16 * 148 * (1 if mt > 16 else 2)) // (cd(n2 + n2 % 2, 64) * cd(n1, 8 * mt))
    s = min(max(s, 1), 64, cd(nz, 128))
    kchunk = cd(cd(nz, s), 16) * 16
    return mt, cd(nz, kchunk), kchunk


def _ws_expected(nz, n1, n2):
    _, ns, _ = _plan(nz, n1, n2)
    return nz * (n1 + n1 % 2 + n2 + n2 % 2) + ns * n1 * (n2 + n2 % 2)


# ------------------------------------------------------------------------------------------------- CPU-only
def test_ssc_rejects_before_any_launch():
    """Every argument and limit check of the three entry points runs before the first launch: with valid-looking dummy
    device pointers and no GPU, each rejected call returns its own code and message, never a CUDA error.  The workspace
    function agrees with the plan restated in _plan."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    p = [C.c_void_p(0x10000 + 0x100 * i) for i in range(16)]          # non-null, 16-byte aligned, never dereferenced
    bad = C.c_void_p(0x20008)

    def resp(nz=2, nm=40, nk=30, ldk=32, ks=p[1], P=p[4], uA=p[5], kA=0, uB=p[6], kB=2, ws=p[7], r1=p[8], r2=p[9]):
        return L.hmv_power_response(nz, nm, nk, ldk, p[0], ks, p[2], p[3], P, 1.0, uA, kA, uB, kB, ws, r1, r2, None)

    def sb2(nz=3, nks=100, ks=p[0], R=p[3], out=p[4]):
        return L.hmv_sigma_b2(nz, nks, ks, p[1], p[2], R, out, None)

    def cov(nz=3, nk=30, n1=5, n2=6, rAB=p[1], chis=p[8], ws=p[10]):
        return L.hmv_cl_cov_ssc(nz, nk, p[0], rAB, p[2], n1, p[3], n2, p[4], p[5], chis, p[9], ws, p[11], None)

    cases = {
        "resp nz = 0": (lambda: resp(nz=0), HMV_E_ARG, "hmv_power_response: sizes must be >= 1"),
        "resp nm = 0": (lambda: resp(nm=0), HMV_E_ARG, "sizes must be >= 1"),
        "resp nk = 1": (lambda: resp(nk=1, ldk=2), HMV_E_ARG, "nk >= 2"),
        "resp odd ldk": (lambda: resp(ldk=31), HMV_E_ARG, "ldk must be even"),
        "resp ldk < nk": (lambda: resp(ldk=28), HMV_E_ARG, "ldk must be even and >= nk"),
        "resp null ks": (lambda: resp(ks=None), HMV_E_ARG, "hmv_power_response: null pointer"),
        "resp null Pzk": (lambda: resp(P=None), HMV_E_ARG, "hmv_power_response: null pointer"),
        "resp null cube": (lambda: resp(uB=None), HMV_E_ARG, "hmv_power_response: null pointer"),
        "resp no output": (lambda: resp(r1=None, r2=None), HMV_E_ARG, "r1h and r2h are both NULL"),
        "resp hod kind A": (lambda: resp(kA=1), HMV_E_ARG, "cube A: kind 1 is neither"),
        "resp bad kind B": (lambda: resp(kB=3), HMV_E_ARG, "cube B: kind 3 is neither"),
        "resp misaligned A": (lambda: resp(uA=bad), HMV_E_ARG, "cube A must be 16-byte aligned"),
        "resp misaligned B": (lambda: resp(uB=bad), HMV_E_ARG, "cube B must be 16-byte aligned"),
        "resp misaligned ws": (lambda: resp(ws=bad), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "resp nz > 65535": (lambda: resp(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        "sb2 nz = 0": (lambda: sb2(nz=0), HMV_E_ARG, "hmv_sigma_b2: sizes must be >= 1"),
        "sb2 nks = 0": (lambda: sb2(nks=0), HMV_E_ARG, "hmv_sigma_b2: sizes must be >= 1"),
        "sb2 null ks": (lambda: sb2(ks=None), HMV_E_ARG, "hmv_sigma_b2: null pointer"),
        "sb2 null R": (lambda: sb2(R=None), HMV_E_ARG, "hmv_sigma_b2: null pointer"),
        "sb2 null out": (lambda: sb2(out=None), HMV_E_ARG, "hmv_sigma_b2: null pointer"),
        "cov nz = 0": (lambda: cov(nz=0), HMV_E_ARG, "hmv_cl_cov_ssc: sizes must be >= 1"),
        "cov nk = 1": (lambda: cov(nk=1), HMV_E_ARG, "nk >= 2"),
        "cov n2 = 0": (lambda: cov(n2=0), HMV_E_ARG, "sizes must be >= 1"),
        "cov null r": (lambda: cov(rAB=None), HMV_E_ARG, "hmv_cl_cov_ssc: null pointer"),
        "cov null chis": (lambda: cov(chis=None), HMV_E_ARG, "hmv_cl_cov_ssc: null pointer (zs, chis or pref)"),
        "cov misaligned ws": (lambda: cov(ws=bad), HMV_E_ARG, "hmv_cl_cov_ssc: workspace must be 16-byte aligned"),
        "cov nz > 65535": (lambda: cov(nz=70000), HMV_E_LIMIT, "exceeds 65535"),
    }
    for what, (call, code, msg) in cases.items():
        rc = call()
        assert rc == code and msg in capi.last_error(), (what, rc, capi.last_error())
    assert L.hmv_cl_cov_ssc_ws_doubles(0, 4, 3) == 0 and L.hmv_cl_cov_ssc_ws_doubles(2, 0, 3) == 0
    for nz, n1, n2 in [(1, 1, 1), (3, 7, 65), (200, 1000, 1000), (2000, 33, 129), (5000, 5, 5)]:
        assert L.hmv_cl_cov_ssc_ws_doubles(nz, n1, n2) == _ws_expected(nz, n1, n2), (nz, n1, n2)


# ------------------------------------------------------------------------------------------------- GPU: the C ABI
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    yield torch, capi
    print("\nlargest |got - want| / bound:", {k: "%.2g" % v for k, v in sorted(OBSERVED.items())})


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


def _twice(torch, launch, bufs):
    """Launch, snapshot, launch again: the outputs must be bit-identical."""
    launch()
    torch.cuda.synchronize()
    first = [b.clone() for b in bufs]
    launch()
    torch.cuda.synchronize()
    for a, b in zip(first, bufs):
        assert torch.equal(a.view(torch.int64), b.view(torch.int64)), "second launch differs"


def _response_abi(torch, capi, nz, nm, nk, ncube, kinds, seed, ones=False, P=None, ks=None):
    rng = np.random.default_rng(seed)
    ldk = (nk + 15) // 16 * 16
    if ks is None:
        ks = 1e-3 * np.cumsum(rng.uniform(0.2, 1.8, nk))                  # non-uniform, strictly increasing
    ms = 1e13 * (1.0 + np.cumsum(rng.uniform(0.5, 1.5, nm)) / nm)
    wt = _trapz_w(ms) if nm > 1 else np.ones(1)
    nzm = rng.uniform(0.5, 2.0, (nz, nm)) / wt
    bh = rng.uniform(0.5, 2.0, (nz, nm))
    rho = 2e13
    if P is None:
        P = rng.uniform(0.5, 2.0, (nz, nk)) * 1e3
    cubes = [np.ones((nz, nm, nk)) if ones else rng.uniform(-0.3, 1.2, (nz, nm, nk)) for _ in range(ncube)]
    dcubes = []
    for c in cubes:
        t = torch.full((nz, nm, ldk), float("nan"), dtype=torch.float64, device="cuda")   # NaN padding columns
        t[..., :nk] = _dev(torch, c)
        dcubes.append(t)
    if ncube == 1:
        cubes, dcubes = cubes * 2, dcubes * 2
    d = {k: _dev(torch, v) for k, v in dict(ks=ks, ms=ms, nzm=nzm, bh=bh, P=P).items()}
    L, p = capi.lib, capi.ptr
    ws = torch.empty(int(L.hmv_power_ws_doubles(nz, nm)), dtype=torch.float64, device="cuda")
    n = nz * nk
    (b1, o1), (b2, o2) = _guarded(torch, n), _guarded(torch, n)

    def launch():
        capi.check(L.hmv_power_response(nz, nm, nk, ldk, p(d["ms"]), p(d["ks"]), p(d["nzm"]), p(d["bh"]), p(d["P"]),
                                        rho, p(dcubes[0]), kinds[0], p(dcubes[1]), kinds[1], p(ws), o1, o2,
                                        capi.stream()), "hmv_power_response")

    _twice(torch, launch, [b1, b2])
    got = _read_guarded(b1, n, (nz, nk)), _read_guarded(b2, n, (nz, nk))
    ref = _response_ref(cubes, kinds, ms, nzm, bh, rho, ks, P)
    return got, ref, dict(ms=ms, nzm=nzm, bh=bh, rho=rho, ks=ks, P=P)


RESP_CASES = [  # (nz, nm, nk, distinct cubes, kinds): k-tile seams of power_one (1024) and power_pair (512)
    (2, 7, 1023, 1, (0, 0)),
    (1, 4, 1024, 1, (2, 2)),
    (2, 5, 1025, 1, (0, 0)),
    (3, 6, 2049, 1, (0, 2)),
    (2, 1, 2, 1, (0, 0)),            # nm = 1 (no trapezoid weight), nk = 2 (both columns one-sided)
    (1, 3, 17, 1, (2, 2)),
    (2, 7, 511, 2, (0, 2)),
    (1, 4, 512, 2, (0, 0)),
    (2, 6, 513, 2, (2, 2)),
    (3, 5, 1025, 2, (0, 2)),
    (2, 5, 2, 2, (2, 0)),
    (1, 1, 40, 2, (0, 0)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("nz,nm,nk,ncube,kinds", RESP_CASES)
def test_response_plans(env, nz, nm, nk, ncube, kinds):
    torch, capi = env
    (r1, r2), ((w1, b1), (w2, b2)), _ = _response_abi(torch, capi, nz, nm, nk, ncube, kinds, seed=nz * 7 + nm * 31 + nk)
    tag = "nz=%d nm=%d nk=%d cubes=%d kinds=%s" % (nz, nm, nk, ncube, kinds)
    _assert_bound("response_r1h " + tag, r1, w1, b1)
    _assert_bound("response_r2h " + tag, r2, w2, b2)


@pytest.mark.gpu
def test_response_known_answers(env):
    """A power law P = A k^n gives n_eff = n at every column, edges included; unit cubes give R1h = sum w n b a_A a_B."""
    torch, capi = env
    nk, nexp = 300, -1.37
    ks = np.geomspace(1e-3, 5.0, nk) * (1.0 + 0.005 * np.sin(np.arange(nk)))    # non-uniform in ln k, increasing
    P = np.broadcast_to(2e4 * ks ** nexp, (2, nk)).copy()
    for kinds in ((2, 2), (0, 0), (0, 2)):
        (r1, r2), _, inp = _response_abi(torch, capi, 2, 9, nk, 1, kinds, seed=11, ones=True, P=P, ks=ks)
        wnb = _trapz_w(inp["ms"])[None, :] * inp["nzm"] * inp["bh"]
        a = [inp["ms"] / inp["rho"] if k == 0 else np.ones(inp["ms"].size) for k in kinds]
        want1 = (wnb * a[0] * a[1]).sum(axis=1)
        _assert_bound("unit_r1h", r1, np.broadcast_to(want1[:, None], r1.shape),
                      np.broadcast_to((np.abs(wnb) * a[0] * a[1]).sum(axis=1)[:, None], r1.shape))
        lab = [(wnb * ax).sum(axis=1) + (1.0 - (wnb * ax).sum(axis=1) if k == 0 else 0.0) for ax, k in zip(a, kinds)]
        p2h = P * (lab[0] * lab[1])[:, None]
        neff = 3.0 * (47.0 / 21.0 - r2 / p2h)
        assert np.max(np.abs(neff - nexp)) < 1e-9, (kinds, np.max(np.abs(neff - nexp)))


@pytest.mark.gpu
def test_response_nonpositive_plin_gives_nan(env):
    torch, capi = env
    rng = np.random.default_rng(3)
    P = rng.uniform(0.5, 2.0, (1, 40)) * 1e3
    P[0, 20] = 0.0
    P[0, 0] = -1.0
    (r1, r2), _, _ = _response_abi(torch, capi, 1, 5, 40, 1, (0, 0), seed=3, P=P)
    bad = np.zeros(40, dtype=bool)
    bad[[0, 1, 19, 20, 21]] = True
    assert np.all(np.isnan(r2[0, bad])) and np.all(np.isfinite(r2[0, ~bad])) and np.all(np.isfinite(r1))


# ---- sigma_b^2
@pytest.mark.gpu
@pytest.mark.parametrize("nks", [1, 255, 256, 257, 10000])
def test_sigma_b2_abi(env, nks):
    """Against the numpy restatement; R = 0 (chi = 0) gives W = 1 and a finite value; tiny x takes the Taylor form."""
    torch, capi = env
    from hmvec_b200.cosmology import simpson_weights
    rng = np.random.default_rng(nks)
    ks = np.geomspace(1e-6, 50.0, nks) if nks > 1 else np.array([0.3])
    kw = simpson_weights(ks) * ks / (2 * np.pi) if nks > 1 else np.array([0.7])
    R = np.array([0.0, 1e-7, 3.0, 150.0, 4000.0, 7000.0])
    P = rng.uniform(0.5, 2.0, (R.size, nks)) * 1e4
    d = {k: _dev(torch, v) for k, v in dict(ks=ks, kw=kw, P=P, R=R).items()}
    buf, optr = _guarded(torch, R.size)
    p = capi.ptr

    def launch():
        capi.check(capi.lib.hmv_sigma_b2(R.size, nks, p(d["ks"]), p(d["kw"]), p(d["P"]), p(d["R"]), optr,
                                         capi.stream()), "hmv_sigma_b2")

    _twice(torch, launch, [buf])
    got = _read_guarded(buf, R.size, (R.size,))
    want, bnd = _sigma_b2_ref(ks, kw, P, R)
    _assert_bound("sigma_b2_abi nks=%d" % nks, got, want, bnd, TAU_J1)
    assert got[0] == pytest.approx((kw * P[0]).sum(), rel=1e-13)


@pytest.mark.gpu
def test_sigma_b2_white_spectrum(env):
    """P = P0: sigma_b^2 -> P0/(pi R^2), up to the grid's truncation (below k_b: P0 k_b^2/(4 pi); above k_max the window's
    envelope 8/(pi (kR)^3) gives P0 4/(pi^2 R^3 k_max)) and the quadrature error (half the grid's against the grid's)."""
    torch, capi = env
    from hmvec_b200.cosmology import simpson_weights
    R = np.array([50.0, 100.0, 500.0])
    P0, kb, kmax = 3e4, 1e-6, 20.0          # 1e5 points: the window's oscillation is resolved up to k_max at every R
    vals = []
    for n in (50001, 100001):
        ks = np.geomspace(kb, kmax, n)
        kw = simpson_weights(ks) * ks / (2 * np.pi)
        out = torch.empty(R.size, dtype=torch.float64, device="cuda")
        d = [_dev(torch, v) for v in (ks, kw, np.full((R.size, n), P0), R)]     # alive until the kernel has run
        capi.check(capi.lib.hmv_sigma_b2(R.size, n, *[capi.ptr(t) for t in d], capi.ptr(out), capi.stream()),
                   "hmv_sigma_b2")
        vals.append(out.cpu().numpy())
    exact = P0 / (np.pi * R ** 2)
    bound = P0 * kb ** 2 / (4 * np.pi) + P0 * 4 / (np.pi ** 2 * R ** 3 * kmax) + np.abs(vals[1] - vals[0])
    assert np.all(np.abs(vals[1] - exact) <= bound), (vals[1] / exact - 1, bound / exact)
    assert np.all(bound / exact < 2e-3)


# ---- projection
@pytest.mark.gpu
@pytest.mark.parametrize("n1,n2,nz,mt,split", [
    (1, 1, 1, 4, False),
    (7, 33, 3, 4, False),
    (63, 64, 2, 8, False),
    (65, 65, 25, 16, False),
    (129, 7, 200, 26, True),
    (1000, 1000, 6, 26, False),
    (209, 1000, 300, 26, True),
    (32, 1, 2001, 4, True),
])
def test_cov_ssc_plans(env, n1, n2, nz, mt, split):
    torch, capi = env
    got_mt, ns, _ = _plan(nz, n1, n2)
    assert got_mt == mt and (ns > 1) == split, (got_mt, ns)
    rng = np.random.default_rng(n1 + 7 * n2 + nz)
    nk = 37
    ks = np.geomspace(1e-2, 10.0, nk)
    rAB, rCD = rng.uniform(-1.0, 3.0, (nz, nk)), rng.uniform(-1.0, 3.0, (nz, nk))
    zs = np.sort(rng.uniform(0.1, 3.0, nz)) if nz > 1 else np.array([0.7])
    chis = 1000.0 + 2000.0 * zs
    pref = rng.uniform(0.5, 2.0, nz)
    l1, l2 = rng.uniform(2.0, 2e4, n1), rng.uniform(2.0, 2e4, n2)        # k spans below ks[0] to above ks[-1]
    d = {k: _dev(torch, v) for k, v in dict(ks=ks, a=rAB, c=rCD, zs=zs, chis=chis, pref=pref, l1=l1, l2=l2).items()}
    nws = capi.lib.hmv_cl_cov_ssc_ws_doubles(nz, n1, n2)
    assert nws == _ws_expected(nz, n1, n2)
    ws = torch.empty(int(nws), dtype=torch.float64, device="cuda")
    buf, optr = _guarded(torch, n1 * n2)
    p = capi.ptr

    def launch():
        capi.check(capi.lib.hmv_cl_cov_ssc(nz, nk, p(d["ks"]), p(d["a"]), p(d["c"]), n1, p(d["l1"]), n2, p(d["l2"]),
                                           p(d["zs"]), p(d["chis"]), p(d["pref"]), p(ws), optr, capi.stream()),
                   "hmv_cl_cov_ssc")

    _twice(torch, launch, [buf])
    got = _read_guarded(buf, n1 * n2, (n1, n2))
    want, bnd = _cov_ref(ks, rAB, rCD, l1, l2, zs, chis, pref)
    _assert_bound("cov_ssc_abi n1=%d n2=%d nz=%d" % (n1, n2, nz), got, want, bnd)


# ------------------------------------------------------------------------------------------------- GPU: HaloModel API
def _make_model(zs):
    import hmvec_b200 as hm
    ms = np.geomspace(1e11, 1e16, 47)
    ks = np.geomspace(1e-3, 30, 130)
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low', device="cuda:0")
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)   # table-backed Compton-y
    h.add_hod("g", ngal=np.geomspace(2e-3, 5e-5, zs.size))
    host = dict(zs=zs, ms=h.ms, ks=h._ks64, nzm=h.nzm, bh=h.bh, rho=h._rho_m0, P=h.Pzk,
                chis=np.asarray(h.comoving_radial_distance(zs), dtype=np.float64),
                H=np.asarray(h.h_of_z(zs), dtype=np.float64), Wk=h.lensing_window(zs, 3.0))
    host["cube"] = {"nfw": (h.uk_profiles["nfw"], 0), "y": (h.pk_profiles["y"], 2)}
    return h, host


@pytest.fixture(scope="module")
def model(env):
    return _make_model(np.array([0.05, 0.7, 1.5, 2.8]))


def _sigma_b2_model_ref(h, host, fsky):
    """The disc's grid and weights restated; P_lin on it from the same producer (the device EH98), downloaded."""
    from hmvec_b200.cosmology import simpson_weights
    R = host["chis"] * np.arccos(1.0 - 2.0 * fsky)
    kb = min(h.p['sigma2_kmin'], 1e-3 / R.max())
    kg = np.geomspace(kb, h.p['sigma2_kmax'], int(h.p['sigma2_numks']))
    kw = simpson_weights(kg) * kg / (2 * np.pi)
    P = h._plin_device(kg, host["zs"]).cpu().numpy()
    return _sigma_b2_ref(kg, kw, P, R)


@pytest.mark.gpu
@pytest.mark.parametrize("names", [("nfw", "nfw"), ("y", "y"), ("nfw", "y")], ids=["nfw-nfw", "y-y", "nfw-y"])
def test_power_response_model(model, names):
    h, host = model
    got = h.get_power_response(*names)
    cubes, kinds = zip(*[host["cube"][n] for n in names])
    (w1, b1), (w2, b2) = _response_ref(cubes, kinds, host["ms"], host["nzm"], host["bh"], host["rho"], host["ks"],
                                       host["P"])
    _assert_bound("response_model %s" % "-".join(names), got, w1 + w2, b1 + b2)


@pytest.mark.gpu
def test_response_nfw_large_scale_limit(model):
    """For a physical NFW auto the consistency-corrected bracket -> 1 as u -> 1: R2h(ks[0]) / P_lin(ks[0]) =
    47/21 - n_eff/3."""
    h, host = model
    import torch
    from hmvec_b200 import _capi as capi
    nz, nk = h._nz, h._nk
    r2 = torch.empty(nz, nk, dtype=torch.float64, device="cuda")
    ws = torch.empty(int(capi.lib.hmv_power_ws_doubles(nz, h._nm)), dtype=torch.float64, device="cuda")
    cube = h.uk_profiles.device("nfw")
    capi.check(capi.lib.hmv_power_response(nz, h._nm, nk, h._ldk, capi.ptr(h._ms_d), capi.ptr(h._ks_d),
                                           capi.ptr(h._nzm_d), capi.ptr(h._bh_d), capi.ptr(h._Pzk_d), h._rho_m0,
                                           capi.ptr(cube), 0, capi.ptr(cube), 0, capi.ptr(ws), None, capi.ptr(r2),
                                           capi.stream()), "hmv_power_response")
    ratio = r2.cpu().numpy()[:, 0] / host["P"][:, 0]
    neff = np.gradient(np.log(host["P"]), np.log(host["ks"]), axis=1)[:, 0]
    np.testing.assert_allclose(ratio, 47.0 / 21.0 - neff / 3.0, rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("fsky", [0.05, 0.4, 1.0])
def test_sigma_b2_model(model, fsky):
    h, host = model
    got = h.get_sigma_b2(fsky)
    want, bnd = _sigma_b2_model_ref(h, host, fsky)
    _assert_bound("sigma_b2_model fsky=%g" % fsky, got, want, bnd, TAU_J1)
    assert np.all(got > 0) and np.all(np.diff(got) < 0)          # a larger disc at higher z: less variance


def _cov_model_ref(h, host, names, l1, l2, windows, fsky, sb2=None):
    rAB = h.get_power_response(names[0], names[1])
    rCD = h.get_power_response(names[2], names[3])
    if sb2 is None:
        sb2 = h.get_sigma_b2(fsky)
    W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), host["zs"].shape) for w in windows], axis=0)
    pref = host["H"] ** 3 * W * sb2 / host["chis"] ** 4
    return _cov_ref(host["ks"], rAB, rCD, l1, l2, host["zs"], host["chis"], pref)


COMBOS = [("nfw", "nfw", "nfw", "nfw"), ("y", "y", "y", "y"), ("nfw", "nfw", "y", "y")]


@pytest.mark.gpu
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_cl_cov_ssc_tracers(model, names):
    """Unsorted multipoles, l = 2 (k below ks at high z) and l = 2e4 (k above ks at low z), ells2 != ells, fsky < 1,
    kappa windows from lensing_window and y windows of 1."""
    h, host = model
    ells = np.array([300.0, 2.0, 20000.0, 45.5, 1000.0, 7.0, 3000.0])
    ells2 = np.array([10.0, 5000.0, 2.0, 150.0, 20000.0])
    win = tuple(1.0 if n == "y" else host["Wk"] for n in names)
    got = h.get_cl_cov_ssc(ells, *names, windows=win, fsky=0.4, ells2=ells2)
    want, bnd = _cov_model_ref(h, host, names, ells, ells2, win, 0.4)
    _assert_bound("cov_ssc_model %s" % "-".join(names), got, want, bnd)
    sb2 = h.get_sigma_b2(0.4)
    again = h.get_cl_cov_ssc(ells, *names, windows=win, fsky=0.4, ells2=ells2, sigma_b2=sb2)
    assert np.array_equal(got.view(np.int64), again.view(np.int64)), "sigma_b2= of the disc's own values differs"
    scaled = h.get_cl_cov_ssc(ells, *names, windows=win, ells2=ells2, sigma_b2=2.0 * sb2)
    _assert_bound("cov_ssc_override %s" % "-".join(names), scaled, 2.0 * want, 2.0 * bnd)


@pytest.mark.gpu
def test_cl_cov_ssc_structure(model):
    """The auto covariances are symmetric and positive semi-definite; the cross is the transpose of its mirror."""
    h, host = model
    ells = np.geomspace(10, 1e4, 40)
    Wk = host["Wk"]
    for names, win in ((("nfw",) * 4, (Wk,) * 4), (("y",) * 4, (1.,) * 4)):
        c = h.get_cl_cov_ssc(ells, *names, windows=win, fsky=0.1)
        _, bnd = _cov_model_ref(h, host, names, ells, ells, win, 0.1)
        _assert_bound("cov_ssc_symmetry", c, c.T, bnd)
        ev = np.linalg.eigvalsh(0.5 * (c + c.T))
        assert ev.min() >= -TAU * np.trace(c), (names, ev.min(), np.trace(c))
    ells2 = np.geomspace(30, 3e3, 25)
    a = h.get_cl_cov_ssc(ells, "nfw", "nfw", "y", "y", windows=(Wk, Wk, 1., 1.), ells2=ells2)
    b = h.get_cl_cov_ssc(ells2, "y", "y", "nfw", "nfw", windows=(1., 1., Wk, Wk), ells2=ells)
    _, bnd = _cov_model_ref(h, host, ("nfw", "nfw", "y", "y"), ells, ells2, (Wk, Wk, 1., 1.), 1.0)
    _assert_bound("cov_ssc_transpose", a, b.T, bnd)


@pytest.mark.gpu
def test_cl_cov_ssc_single_redshift_is_rank_one(env):
    """nz = 1: Cov = pref R^{AB}(l) R^{CD}(l'), an outer product."""
    h, host = _make_model(np.array([0.9]))
    ells = np.geomspace(20, 8000, 30)
    c = h.get_cl_cov_ssc(ells, "nfw", "nfw", "y", "y", windows=(host["Wk"], host["Wk"], 1., 1.), fsky=0.3)
    want, bnd = _cov_model_ref(h, host, ("nfw", "nfw", "y", "y"), ells, ells, (host["Wk"], host["Wk"], 1., 1.), 0.3)
    _assert_bound("cov_ssc_rank1", c, want, bnd)
    s = np.linalg.svd(c, compute_uv=False)
    assert s[1] <= 1e-12 * s[0], s[:3]


@pytest.mark.gpu
def test_ssc_api_defaults_and_rejections(model):
    h, host = model
    ells = np.array([100.0, 1000.0])
    np.testing.assert_array_equal(h.get_cl_cov_ssc(ells, "nfw"),
                                  h.get_cl_cov_ssc(ells, "nfw", "nfw", "nfw", "nfw", ells2=ells, fsky=1.0))
    np.testing.assert_array_equal(h.get_power_response("y"), h.get_power_response("y", "y"))
    with pytest.raises(ValueError, match="HOD"):
        h.get_cl_cov_ssc(ells, "g")
    with pytest.raises(ValueError, match="HOD"):
        h.get_power_response("nfw", "g")
    with pytest.raises(ValueError, match="no matter or pressure profile"):
        h.get_power_response("nope")
    for bad in ([0.0, 1.0], [np.inf], [-3.0], []):
        with pytest.raises(ValueError, match="positive finite"):
            h.get_cl_cov_ssc(bad)
        with pytest.raises(ValueError, match="positive finite"):
            h.get_cl_cov_ssc(ells, ells2=bad)
    for fsky in (0.0, 1.5, -0.1):
        with pytest.raises(ValueError, match="fsky"):
            h.get_cl_cov_ssc(ells, fsky=fsky)
        with pytest.raises(ValueError, match="fsky"):
            h.get_sigma_b2(fsky)
    with pytest.raises(ValueError, match="length nz"):
        h.get_cl_cov_ssc(ells, windows=(1., np.ones(3), 1., 1.))
    with pytest.raises(ValueError, match="four entries"):
        h.get_cl_cov_ssc(ells, windows=(1., 1., 1.))
    for sb2 in (np.ones(3), np.array([1.0, -1e-9, 1.0, 1.0]), np.array([1.0, np.nan, 1.0, 1.0]), np.full(4, np.inf)):
        with pytest.raises(ValueError, match="sigma_b2"):
            h.get_cl_cov_ssc(ells, sigma_b2=sb2)
    ks = h._ks64
    try:
        h._ks64 = ks[::-1].copy()
        with pytest.raises(ValueError, match="strictly increasing"):
            h.get_power_response()
        with pytest.raises(ValueError, match="strictly increasing"):
            h.get_cl_cov_ssc(ells)
    finally:
        h._ks64 = ks
    try:
        h._zcomm = object()
        with pytest.raises(NotImplementedError):
            h.get_cl_cov_ssc(ells)
        assert h.get_sigma_b2(0.4).shape == (h._nz,) and h.get_power_response().shape == (h._nz, h._nk)
    finally:
        h._zcomm = None
