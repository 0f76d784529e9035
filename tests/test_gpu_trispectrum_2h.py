"""The 2-halo trispectrum (hmv_trispec_2h, HaloModel.get_trispectrum_2halo) and its non-Gaussian Limber covariance of
C_l (hmv_cl_cov_2h, HaloModel.get_cl_cov_2halo), against a float64 numpy restatement of the definitions on the same
downloaded inputs: np.interp for u(k) and P(k), explicit trapezoid weights on ms and zs, and Pbar from the closed form
with a long-double prefix of int q P dq.

    T2h = P(k1) [I1~A I3^{BCD} + I1~B I3^{ACD}] + P(k2) [I1~C I3^{ABD} + I1~D I3^{ABC}] + Pbar [I2^{AC} I2^{BD} + I2^{AD} I2^{BC}]
    Cov2h(l,l') = sum_z zeta_z H^3 W_A W_B W_C W_D / chi^6 / (4 pi fsky) T2h((l+1/2)/chi, (l'+1/2)/chi; z)

Each element is held to |got - want| <= TAU * B, B the same expression over absolute values.  Largest ratio measured on
one B200 (1000 W power limit): 1.2e-15 (TAU = 1e-12).  Pbar alone is held to 1e-12 of scipy.integrate.quad over the same
piecewise-linear P.  The ABI cases use seeded random cubes in [-0.3, 1.2] with NaN padding columns, NaN guards around
the output and several zchunk values, each launched twice: every output must be bit-identical.  Their shapes take the
contraction's MT = 4 / 8 / 16 / 26 with one to ten row tiles, odd and even widths, nm = 1 and odd nm, and the 8-, 5- and
3-block leg patterns.
"""
import ctypes as C

import numpy as np
import pytest

HMV_E_ARG, HMV_E_LIMIT = -1, -3
TAU = 1e-12
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


def _ev(n):
    return n + n % 2


def _ws2h(nz, nm, nk, n1, n2, nA1, nC1, zc):
    """The workspace of k_trispec.cu's Plan2h restated: four panels, nA1 nC1 + nA1 + nC1 blocks, the side vectors."""
    nmp, n1p, n2p, n1q, n2q = _ev(nm), _ev(n1), _ev(n2), _ev(n1 + 1), _ev(n2 + 1)
    m1, m2 = nA1 * n1p, nC1 * n2p
    panels = nmp * (m1 + n1q + m2 + n2q)
    blocks = m1 * m2 + m1 * n2q + n1q * m2
    return zc * (panels + blocks + _ev(n1) + _ev(n2) + _ev(nk) + 2)


def _qp_prefix(ks, P):
    """F(x) = int_0^x q P(q) dq for P linear on ks and held at its end values, in long double."""
    ks, P = ks.astype(np.longdouble), P.astype(np.longdouble)
    pieces = (ks[1:] - ks[:-1]) * (ks[:-1] * (2 * P[:-1] + P[1:]) + ks[1:] * (P[:-1] + 2 * P[1:])) / 6
    S = np.concatenate([[P[0] * ks[0] ** 2 / 2], P[0] * ks[0] ** 2 / 2 + np.cumsum(pieces)])

    def F(x):
        x = np.asarray(x, dtype=np.longdouble)
        r = np.clip(np.searchsorted(ks, x, side="right") - 1, 0, ks.size - 2)
        f = (x - ks[r]) / (ks[r + 1] - ks[r])
        px = P[r] + f * (P[r + 1] - P[r])
        mid = S[r] + (x - ks[r]) * (ks[r] * (2 * P[r] + px) + x * (P[r] + 2 * px)) / 6
        lo = P[0] * x * x / 2
        hi = S[-1] + P[-1] * (x * x - ks[-1] ** 2) / 2
        return np.where(x < ks[0], lo, np.where(x >= ks[-1], hi, mid))
    return F


def _pbar(ks, P, k1, k2):
    F = _qp_prefix(ks, P)
    k1, k2 = np.broadcast_arrays(np.asarray(k1, dtype=np.float64), np.asarray(k2, dtype=np.float64))
    k1l, k2l = k1.astype(np.longdouble), k2.astype(np.longdouble)
    a, b = np.abs(k1l - k2l), k1l + k2l
    return np.asarray((F(b) - F(a)) / (2 * k1.astype(np.longdouble) * k2), dtype=np.float64)


def _reference(cubes, kinds, ms, nzm, bh, Pzk, rho, ks, q1, q2, chis=None, zs=None, pref=None):
    """(value, bound): T2h [nz, n1, n2] when chis is None, else Cov2h [n1, n2]."""
    nz, nm = cubes[0].shape[:2]
    w = _trapz_w(ms)[None, :] * nzm * bh
    a = [ms / rho if k == 0 else np.ones(nm) for k in kinds]
    T, B = np.empty((nz, q1.size, q2.size)), np.empty((nz, q1.size, q2.size))
    for z in range(nz):
        k1 = q1 if chis is None else (q1 + 0.5) / chis[z]
        k2 = q2 if chis is None else (q2 + 0.5) / chis[z]
        t = [a[i][:, None] * np.array([np.interp(k1 if i < 2 else k2, ks, cubes[i][z, m]) for m in range(nm)])
             for i in range(4)]
        A, Bl, Cc, D = t
        W, Wa = w[z][:, None], np.abs(w[z])[:, None]
        cons = 1.0 - np.sum(w[z] * ms / rho)
        zo = [cons if k == 0 else 0.0 for k in kinds]

        def I1(x, i):
            return (W * x).sum(0) + zo[i], (Wa * np.abs(x)).sum(0) + abs(zo[i])

        def I2(x, y):
            return (W * x).T @ y, (Wa * np.abs(x)).T @ np.abs(y)

        def I3(x, y, u, v):       # sum_m w x(k1) y(.) [u v](k2) or [x y](k1) u(k2)
            return (W * x * y).T @ (u * v), (Wa * np.abs(x * y)).T @ np.abs(u * v)
        one = np.ones((nm, 1))
        I1A, I1B, I1C, I1D = I1(A, 0), I1(Bl, 1), I1(Cc, 2), I1(D, 3)
        I3BCD, I3ACD = I3(Bl, one, Cc, D), I3(A, one, Cc, D)
        I3ABD, I3ABC = I3(A, Bl, D, one), I3(A, Bl, Cc, one)
        I2AC, I2BD, I2AD, I2BC = I2(A, Cc), I2(Bl, D), I2(A, D), I2(Bl, Cc)
        P1, P2 = np.interp(k1, ks, Pzk[z]), np.interp(k2, ks, Pzk[z])
        pb = _pbar(ks, Pzk[z], k1[:, None], k2[None, :])
        pba = _pbar(ks, np.abs(Pzk[z]), k1[:, None], k2[None, :])
        for s, (o, P1_, P2_, pb_) in enumerate(((0, P1, P2, pb), (1, np.abs(P1), np.abs(P2), pba))):
            v = P1_[:, None] * (I1A[s][:, None] * I3BCD[s] + I1B[s][:, None] * I3ACD[s]) \
                + P2_[None, :] * (I1C[s][None, :] * I3ABD[s] + I1D[s][None, :] * I3ABC[s]) \
                + pb_ * (I2AC[s] * I2BD[s] + I2AD[s] * I2BC[s])
            (T if s == 0 else B)[z] = v if s == 0 else np.abs(v)
    if chis is None:
        return T, B
    zw = (_trapz_w(zs) if nz > 1 else np.ones(1)) * pref
    return np.einsum("z,zln->ln", zw, T), np.einsum("z,zln->ln", np.abs(zw), B)


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


# ------------------------------------------------------------------------------------------------- CPU-only
def test_trispec_2h_rejects_before_any_launch():
    """Every argument and limit check of both entry points runs before the first launch: with valid-looking dummy
    device pointers and no GPU, each rejected call returns its own code and message, never a CUDA error.  The workspace
    functions agree with the plan restated in _ws2h, with 8, 5 or 3 blocks by leg coincidence."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    p = [C.c_void_p(0x10000 + 0x100 * i) for i in range(14)]          # non-null, 16-byte aligned, never dereferenced
    bad = C.c_void_p(0x20008)

    def cubes(*ptrs):
        return (C.c_void_p * 4)(*ptrs)

    def kinds(*k):
        return (C.c_int * 4)(*k)

    ok_u, ok_k = cubes(*p[3:7]), kinds(0, 0, 2, 2)

    def tri(nz=2, nm=40, nk=30, ldk=32, ks=p[0], u=ok_u, k=ok_k, ws=p[9], bh=p[12], Pzk=p[13], zchunk=1):
        return L.hmv_trispec_2h(nz, nm, nk, ldk, ks, p[1], p[2], bh, Pzk, 1.0, u, k, 5, p[7], 6, p[8], zchunk, ws,
                                p[10], None)

    def cov(chis=p[11], zchunk=2, **kw):
        nz, nm, nk, ldk = kw.get("nz", 2), kw.get("nm", 40), kw.get("nk", 30), kw.get("ldk", 32)
        return L.hmv_cl_cov_2h(nz, nm, nk, ldk, p[0], p[1], p[2], p[12], p[13], 1.0, ok_u, ok_k, 5, p[7], 6, p[8],
                               p[1], chis, p[2], zchunk, p[9], p[10], None)

    cases = {
        "nz = 0": (lambda: tri(nz=0), HMV_E_ARG, "sizes must be >= 1"),
        "nk = 1": (lambda: tri(nk=1, ldk=2), HMV_E_ARG, "nk >= 2"),
        "odd ldk": (lambda: tri(ldk=31), HMV_E_ARG, "ldk must be even"),
        "ldk < nk": (lambda: tri(ldk=28), HMV_E_ARG, "ldk must be even and >= nk"),
        "null ks": (lambda: tri(ks=None), HMV_E_ARG, "hmv_trispec_2h: null pointer"),
        "null cube": (lambda: tri(u=cubes(p[3], p[4], None, p[6])), HMV_E_ARG, "null pointer (cube 2)"),
        "hod kind": (lambda: tri(k=kinds(0, 1, 2, 2)), HMV_E_ARG, "kind 1 is neither"),
        "misaligned cube": (lambda: tri(u=cubes(p[3], bad, p[5], p[6])), HMV_E_ARG, "cube 1 must be 16-byte aligned"),
        "misaligned ws": (lambda: tri(ws=bad), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "null bh": (lambda: tri(bh=None), HMV_E_ARG, "null pointer (bh or Pzk)"),
        "null Pzk": (lambda: tri(Pzk=None), HMV_E_ARG, "null pointer (bh or Pzk)"),
        "zchunk = 0": (lambda: tri(zchunk=0), HMV_E_ARG, "zchunk must lie in [1, nz]"),
        "zchunk > nz": (lambda: tri(zchunk=3), HMV_E_ARG, "zchunk must lie in [1, nz]"),
        "cov null chis": (lambda: cov(chis=None), HMV_E_ARG, "hmv_cl_cov_2h: null pointer (zs, chis or pref)"),
        "cov odd ldk": (lambda: cov(ldk=33), HMV_E_ARG, "hmv_cl_cov_2h: ldk"),
        "cov zchunk": (lambda: cov(zchunk=-1), HMV_E_ARG, "hmv_cl_cov_2h: zchunk"),
        "nz > 65535": (lambda: tri(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        "K > 2^30": (lambda: cov(nz=60000, nm=20000), HMV_E_LIMIT, "exceeds 2^30"),
    }
    for what, (call, code, msg) in cases.items():
        rc = call()
        assert rc == code and msg in capi.last_error(), (what, rc, capi.last_error())
    patterns = [  # (cubes, kinds, nA1, nC1, blocks)
        ((3, 4, 5, 6), (0, 0, 2, 2), 2, 2, 8),
        ((3, 4, 3, 4), (0, 2, 0, 2), 2, 2, 8),          # NFW y NFW y: neither side coincides
        ((3, 3, 5, 5), (0, 2, 0, 0), 2, 1, 5),          # same cube, different kind: distinct legs
        ((3, 3, 5, 6), (0, 0, 2, 2), 1, 2, 5),
        ((3, 4, 5, 5), (0, 0, 2, 2), 2, 1, 5),
        ((3, 3, 3, 3), (2, 2, 2, 2), 1, 1, 3),
        ((3, 3, 5, 5), (0, 0, 2, 2), 1, 1, 3),
    ]
    for fn in (L.hmv_trispec_2h_ws_doubles, L.hmv_cl_cov_2h_ws_doubles):
        assert fn(0, 4, 10, 3, 3, ok_u, ok_k, 1) == 0 and fn(2, 4, 1, 3, 3, ok_u, ok_k, 1) == 0
        assert fn(3, 4, 10, 3, 3, ok_u, ok_k, 0) == 0 and fn(3, 4, 10, 3, 3, ok_u, ok_k, 4) == 0
        for idx, kk, nA1, nC1, nb in patterns:
            assert nA1 * nC1 + nA1 + nC1 == nb
            for nz, nm, nk, n1, n2, zc in [(1, 1, 2, 1, 1, 1), (3, 41, 37, 7, 65, 2), (200, 2000, 10000, 1000, 1000, 53)]:
                got = fn(nz, nm, nk, n1, n2, cubes(*[p[i] for i in idx]), kinds(*kk), zc)
                assert got == _ws2h(nz, nm, nk, n1, n2, nA1, nC1, zc), (idx, kk, nz, nm, n1, n2, zc)


# ------------------------------------------------------------------------------------------------- GPU: the C ABI
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    yield torch, capi
    print("\n2-halo largest measured ratios:", {k: "%.2g" % v for k, v in sorted(OBSERVED.items())})


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


def _inputs(rng, nz, nm, nk=37, cube_fn=None, P=None):
    ks = np.geomspace(1e-2, 10.0, nk)
    ms = 1e13 * (1.0 + np.cumsum(rng.uniform(0.5, 1.5, nm)) / nm)
    wt = _trapz_w(ms) if nm > 1 else np.ones(1)
    nzm = rng.uniform(0.5, 2.0, (nz, nm)) / wt
    bh = rng.uniform(0.5, 3.0, (nz, nm))
    if P is None:
        P = (ks / 0.05) / (1.0 + (ks / 0.05) ** 2.5)[None, :] * rng.uniform(0.5, 2.0, (nz, 1))
    zs = np.sort(rng.uniform(0.1, 3.0, nz)) if nz > 1 else np.array([0.7])
    return dict(ks=ks, ms=ms, nzm=nzm, bh=bh, Pzk=np.ascontiguousarray(np.broadcast_to(P, (nz, nk))), zs=zs,
                chis=1000.0 + 2000.0 * zs, pref=rng.uniform(0.5, 2.0, nz), rho=2e13)


def _abi(torch, capi, proj, inp, cubes, kinds, q1, q2, zchunks, same=None):
    """One launch per zchunk, each twice: bit-identical across every launch, guards intact.  same: which cube each leg
    reads ((0, 0, 2, 2): A = B and C = D share one device cube)."""
    nz, nm, nk = cubes[0].shape
    ldk = (nk + 15) // 16 * 16
    same = same or (0, 1, 2, 3)
    dcubes = {}
    for i in sorted(set(same)):
        t = torch.full((nz, nm, ldk), float("nan"), dtype=torch.float64, device="cuda")   # NaN padding columns
        t[..., :nk] = _dev(torch, cubes[i])
        dcubes[i] = t
    d = {k: _dev(torch, inp[k]) for k in ("ks", "ms", "nzm", "bh", "Pzk", "zs", "chis", "pref")}
    d["q1"], d["q2"] = _dev(torch, q1), _dev(torch, q2)
    L, p = capi.lib, capi.ptr
    u_h = (C.c_void_p * 4)(*[dcubes[s].data_ptr() for s in same])
    k_h = (C.c_int * 4)(*kinds)
    n1, n2 = q1.size, q2.size
    shape = (n1, n2) if proj else (nz, n1, n2)
    n = int(np.prod(shape))
    outs = []
    for zc in zchunks:
        nws = (L.hmv_cl_cov_2h_ws_doubles if proj else L.hmv_trispec_2h_ws_doubles)(nz, nm, nk, n1, n2, u_h, k_h, zc)
        nA1 = 1 if same[0] == same[1] and kinds[0] == kinds[1] else 2
        nC1 = 1 if same[2] == same[3] and kinds[2] == kinds[3] else 2
        assert nws == _ws2h(nz, nm, nk, n1, n2, nA1, nC1, zc)
        ws = torch.full((int(nws),), float("nan"), dtype=torch.float64, device="cuda")
        buf, optr = _guarded(torch, n)
        for _ in range(2):
            if proj:
                rc = L.hmv_cl_cov_2h(nz, nm, nk, ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]),
                                     inp["rho"], u_h, k_h, n1, p(d["q1"]), n2, p(d["q2"]), p(d["zs"]), p(d["chis"]),
                                     p(d["pref"]), zc, p(ws), optr, capi.stream())
            else:
                rc = L.hmv_trispec_2h(nz, nm, nk, ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]),
                                      inp["rho"], u_h, k_h, n1, p(d["q1"]), n2, p(d["q2"]), zc, p(ws), optr,
                                      capi.stream())
            capi.check(rc, "2-halo ABI")
            torch.cuda.synchronize()
            outs.append(buf.clone())
    for o in outs[1:]:
        assert torch.equal(outs[0].view(torch.int64), o.view(torch.int64)), "launches or zchunks differ"
    return _read_guarded(outs[0], n, shape)


def _abi_ref(inp, cubes, kinds, q1, q2, proj):
    extra = (inp["chis"], inp["zs"], inp["pref"]) if proj else ()
    return _reference(cubes, kinds, inp["ms"], inp["nzm"], inp["bh"], inp["Pzk"], inp["rho"], inp["ks"], q1, q2,
                      *extra)


PLAN_CASES = [  # (n1, n2, nz, nm, same, zchunks) -- product rows nA1 n1p / n1q pick MT
    (1, 1, 1, 1, (0, 1, 2, 3), (1,)),                 # MT 4, nm = 1 (trapezoid weight zero)
    (7, 9, 5, 41, (0, 1, 2, 3), (1, 2, 5)),           # MT 4, 8 blocks, zchunk 2 does not divide 5
    (31, 64, 3, 30, (0, 0, 2, 3), (1, 2, 3)),         # rows 32 / 32: MT 4; 5 blocks (A = B)
    (63, 7, 4, 17, (0, 1, 2, 2), (1, 3, 4)),          # rows 128 / 64: MT 16 / 8; 5 blocks (C = D)
    (100, 33, 2, 25, (0, 0, 2, 2), (1, 2)),           # rows 100 / 102: MT 16 / 26; 3 blocks
    (209, 63, 3, 21, (0, 1, 2, 3), (1, 2, 3)),        # rows 418 / 210: MT 26, two to three row tiles
    (1000, 5, 2, 9, (0, 1, 2, 3), (1, 2)),            # rows 2000: MT 26, ten row tiles
]


@pytest.mark.gpu
@pytest.mark.parametrize("proj", [False, True], ids=["trispec", "cov"])
@pytest.mark.parametrize("n1,n2,nz,nm,same,zchunks", PLAN_CASES)
def test_plans(env, proj, n1, n2, nz, nm, same, zchunks):
    torch, capi = env
    rng = np.random.default_rng(n1 * 31 + n2 + nz * 7 + nm + proj)
    inp = _inputs(rng, nz, nm)
    base = [rng.uniform(-0.3, 1.2, (nz, nm, 37)) for _ in range(4)]
    cubes = [base[s] for s in same]
    kinds = (0, 0, 2, 2) if same[0] == same[1] or same[2] == same[3] else (0, 2, 0, 2)
    if proj:
        q1, q2 = rng.uniform(2.0, 2e4, n1), rng.uniform(2.0, 2e4, n2)    # k spans below ks[0] to above ks[-1]
    else:
        q1, q2 = rng.uniform(3e-3, 20.0, n1), rng.uniform(3e-3, 20.0, n2)
    got = _abi(torch, capi, proj, inp, cubes, kinds, q1, q2, zchunks, same)
    want, bnd = _abi_ref(inp, cubes, kinds, q1, q2, proj)
    _assert_bound("abi n1=%d n2=%d nz=%d nm=%d proj=%d" % (n1, n2, nz, nm, proj), got, want, bnd)


@pytest.mark.gpu
def test_pbar_against_quad(env):
    """Pbar alone: pressure legs u = +1 and -1 on two masses with equal w^ give I1~ = I3 = 0 and I2 = 2 w^ exactly, so
    T2h = 2 Pbar I2^2.  Rows of P: constant (Pbar = P0), P = k (Pbar = ((k1+k2)^3 - |k1-k2|^3)/(6 k1 k2) inside the
    grid) and a peaked spectrum, against the definition (1/2) int dmu P(|k1 + k2|) by scipy.integrate.quad over
    np.interp's interpolant."""
    from scipy.integrate import quad
    torch, capi = env
    nk, nz = 40, 3
    ks = np.geomspace(1e-2, 10.0, nk)
    P = np.stack([np.full(nk, 3.7), ks.copy(), (ks / 0.05) / (1.0 + (ks / 0.05) ** 2.5)])
    inp = dict(ks=ks, ms=np.array([1.0, 3.0]), nzm=np.ones((nz, 2)), bh=np.ones((nz, 2)), Pzk=P, zs=np.array([0.1, 0.5, 1.]),
               chis=np.ones(nz), pref=np.ones(nz), rho=1.0)
    cube = np.empty((nz, 2, nk))
    cube[:, 0], cube[:, 1] = 1.0, -1.0
    k1 = np.array([0.5, 1e-3 * 2.0, 6.0, 0.013, 2.0, 0.3, 9.0, 0.02, 0.5, 0.05])
    k2 = np.array([0.5, 2.0, 7.5, 0.012, 2.0 + 1e-9, 0.3001, 9.5, 3.0, 1.5, 0.2])
    got = _abi(torch, capi, False, inp, [cube] * 4, (2, 2, 2, 2), k1, k2, (1, 3), same=(0, 0, 0, 0))
    pb = np.array([np.diag(g) for g in got]) / 8.0          # w^ = 1 on each mass, I2 = 2
    for z in range(nz):
        for i in range(k1.size):
            c, s2 = 2 * k1[i] * k2[i], k1[i] ** 2 + k2[i] ** 2       # q^2 = k1^2 + k2^2 + 2 k1 k2 mu
            pts = [m for m in (ks ** 2 - s2) / c if -1 < m < 1]
            f = lambda mu: 0.5 * np.interp(np.sqrt(max(s2 + c * mu, 0.0)), ks, P[z])
            want = quad(f, -1, 1, points=pts or None, limit=400, epsabs=0, epsrel=1e-13)[0]
            assert abs(pb[z, i] - want) <= 1e-12 * abs(want), (z, i, pb[z, i], want)
    np.testing.assert_allclose(pb[0], 3.7, rtol=1e-13)
    inside = (np.abs(k1 - k2) >= ks[0]) & (k1 + k2 <= ks[-1])
    lin = ((k1 + k2) ** 3 - np.abs(k1 - k2) ** 3) / (6 * k1 * k2)
    np.testing.assert_allclose(pb[1][inside], lin[inside], rtol=1e-12)
    assert inside.sum() >= 3 and (~inside).sum() >= 3


@pytest.mark.gpu
def test_unit_cubes_constant_power(env):
    """u = 1, matter legs: I1~ = 1, so with P_lin = P0 everywhere T2h = 2 P0 I2^2 + 4 P0 I3, I2 = sum w^ (M/rho)^2,
    I3 = sum w^ (M/rho)^3."""
    torch, capi = env
    rng = np.random.default_rng(3)
    nz, nm = 3, 25
    inp = _inputs(rng, nz, nm, P=np.full(37, 2.5))
    cube = np.ones((nz, nm, 37))
    k1, k2 = rng.uniform(3e-3, 20.0, 9), rng.uniform(3e-3, 20.0, 70)
    got = _abi(torch, capi, False, inp, [cube] * 4, (0, 0, 0, 0), k1, k2, (2,), same=(0, 0, 0, 0))
    w = _trapz_w(inp["ms"])[None, :] * inp["nzm"] * inp["bh"]
    a = inp["ms"] / inp["rho"]
    I2, I3 = (w * a ** 2).sum(1), (w * a ** 3).sum(1)
    want = 2 * 2.5 * I2 ** 2 + 4 * 2.5 * I3
    cons = 1.0 - (w * a).sum(1)
    bnd = 2 * 2.5 * I2 ** 2 + 4 * 2.5 * I3 * (1 + (w * a).sum(1) + np.abs(cons))
    _assert_bound("unit_cubes", got, np.broadcast_to(want[:, None, None], got.shape),
                  np.broadcast_to(bnd[:, None, None], got.shape))


@pytest.mark.gpu
def test_single_redshift_cov_is_pref_times_trispectrum(env):
    """nz = 1: Cov2h(l, l') = pref T2h((l+1/2)/chi, (l'+1/2)/chi) to rounding."""
    torch, capi = env
    rng = np.random.default_rng(11)
    inp = _inputs(rng, 1, 19)
    cubes = [rng.uniform(-0.3, 1.2, (1, 19, 37)) for _ in range(4)]
    ells, ells2 = rng.uniform(2.0, 2e4, 13), rng.uniform(2.0, 2e4, 6)
    cov = _abi(torch, capi, True, inp, cubes, (0, 2, 0, 2), ells, ells2, (1,))
    chi = inp["chis"][0]
    T = _abi(torch, capi, False, inp, cubes, (0, 2, 0, 2), (ells + 0.5) / chi, (ells2 + 0.5) / chi, (1,))
    _, bnd = _abi_ref(inp, cubes, (0, 2, 0, 2), ells, ells2, True)
    _assert_bound("nz1_cov", cov, inp["pref"][0] * T[0], bnd)


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
    host = dict(zs=zs, ms=h.ms, ks=h._ks64, nzm=h.nzm, bh=h.bh, Pzk=h.Pzk, rho=h._rho_m0,
                chis=np.asarray(h.comoving_radial_distance(zs), dtype=np.float64),
                H=np.asarray(h.h_of_z(zs), dtype=np.float64), Wk=h.lensing_window(zs, 3.0))
    host["cube"] = {"nfw": (h.uk_profiles["nfw"], 0), "electron": (h.uk_profiles["electron"], 0),
                    "y": (h.pk_profiles["y"], 2)}
    return h, host


COMBOS = [("nfw",) * 4, ("y",) * 4, ("nfw", "nfw", "y", "y"), ("nfw", "y", "nfw", "y"), ("nfw", "electron", "y", "nfw")]


def _model_ref(host, names, q1, q2, windows=None, fsky=1.0):
    cubes, kinds = zip(*[host["cube"][n] for n in names])
    args = (cubes, kinds, host["ms"], host["nzm"], host["bh"], host["Pzk"], host["rho"], host["ks"], q1, q2)
    if windows is None:
        return _reference(*args)
    W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), host["zs"].shape) for w in windows], axis=0)
    pref = host["H"] ** 3 * W / host["chis"] ** 6 / (4 * np.pi * fsky)
    return _reference(*args, host["chis"], host["zs"], pref)


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
    got = h.get_trispectrum_2halo(k1, k2, *names)
    assert got.shape == (4, k1.size, k2.size)
    want, bnd = _model_ref(host, names, k1, k2)
    _assert_bound("trispec_model %s" % "-".join(names), got, want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_cl_cov_tracers(model, names):
    """Projected mode: unsorted multipoles, l = 2 (k below ks at high z) and l = 2e4 (k above ks at low z), ells2 !=
    ells, fsky < 1, kappa windows from lensing_window and y windows of 1."""
    h, host = model
    ells = np.array([300.0, 2.0, 20000.0, 45.5, 1000.0, 7.0, 3000.0])
    ells2 = np.array([10.0, 5000.0, 2.0, 150.0])
    win = _win(host, names)
    got = h.get_cl_cov_2halo(ells, *names, windows=win, fsky=0.4, ells2=ells2)
    want, bnd = _model_ref(host, names, ells, ells2, win, 0.4)
    _assert_bound("cov_model %s" % "-".join(names), got, want, bnd)


@pytest.mark.gpu
def test_structure(model):
    """T^{ABCD}(k1,k2) = T^{CDAB}(k2,k1)^T; T is invariant under A <-> B; the auto covariance is symmetric; a budget
    small enough to force one redshift per pass gives the same bits."""
    h, host = model
    k1, k2 = np.geomspace(2e-3, 20, 11), np.geomspace(5e-3, 8, 6)
    a = h.get_trispectrum_2halo(k1, k2, "nfw", "y", "electron", "nfw")
    b = h.get_trispectrum_2halo(k2, k1, "electron", "nfw", "nfw", "y")
    _, bnd = _model_ref(host, ("nfw", "y", "electron", "nfw"), k1, k2)
    _assert_bound("transpose", a, b.transpose(0, 2, 1), bnd)
    c = h.get_trispectrum_2halo(k1, k2, "y", "nfw", "electron", "nfw")
    _assert_bound("swap_AB", a, c, bnd)
    ells = np.geomspace(10, 1e4, 30)
    Wk = host["Wk"]
    for names, win in ((("nfw",) * 4, (Wk,) * 4), (("y",) * 4, (1.,) * 4)):
        cov = h.get_cl_cov_2halo(ells, *names, windows=win)
        _, bnd = _model_ref(host, names, ells, ells, win)
        _assert_bound("symmetric", cov, cov.T, bnd)
    full = h.get_cl_cov_2halo(ells, "nfw", "y", windows=(Wk, 1., Wk, Wk))
    try:
        h._TRISPEC_2H_WS_BUDGET = 1
        one = h.get_cl_cov_2halo(ells, "nfw", "y", windows=(Wk, 1., Wk, Wk))
    finally:
        del h._TRISPEC_2H_WS_BUDGET
    assert np.array_equal(full.view(np.int64), one.view(np.int64))


@pytest.mark.gpu
def test_api_defaults_and_rejections(model):
    h, host = model
    ells = np.array([100.0, 1000.0])
    np.testing.assert_array_equal(h.get_cl_cov_2halo(ells, "nfw"),
                                  h.get_cl_cov_2halo(ells, "nfw", "nfw", "nfw", "nfw", ells2=ells))
    np.testing.assert_array_equal(h.get_trispectrum_2halo([0.1, 1.0], name="y", name3="nfw"),
                                  h.get_trispectrum_2halo([0.1, 1.0], [0.1, 1.0], "y", "y", "nfw", "nfw"))
    with pytest.raises(ValueError, match="HOD"):
        h.get_cl_cov_2halo(ells, "g")
    with pytest.raises(ValueError, match="HOD"):
        h.get_trispectrum_2halo([0.1], name="nfw", name4="g")
    with pytest.raises(ValueError, match="no matter or pressure profile"):
        h.get_trispectrum_2halo([0.1], name="nope")
    for bad in ([0.0, 1.0], [np.inf], [-3.0], []):
        with pytest.raises(ValueError, match="positive finite"):
            h.get_cl_cov_2halo(bad)
        with pytest.raises(ValueError, match="positive finite"):
            h.get_trispectrum_2halo([0.1], ks2=bad)
    for fsky in (0.0, 1.5, -0.1):
        with pytest.raises(ValueError, match="fsky"):
            h.get_cl_cov_2halo(ells, fsky=fsky)
    with pytest.raises(ValueError, match="length nz"):
        h.get_cl_cov_2halo(ells, windows=(1., np.ones(3), 1., 1.))
    with pytest.raises(ValueError, match="four entries"):
        h.get_cl_cov_2halo(ells, windows=(1., 1., 1.))
    ks = h._ks64
    try:
        h._ks64 = ks[::-1].copy()
        with pytest.raises(ValueError, match="strictly increasing"):
            h.get_trispectrum_2halo([0.1])
    finally:
        h._ks64 = ks
    try:
        h._zcomm = object()
        with pytest.raises(NotImplementedError):
            h.get_cl_cov_2halo(ells)
    finally:
        h._zcomm = None
