"""The 3- and 4-halo trispectra (hmv_trispec_3h/4h, HaloModel.get_trispectrum_3halo/4halo) and their non-Gaussian
Limber covariance of C_l (hmv_cl_cov_3h/4h, HaloModel.get_cl_cov_3halo/4halo).

    T3h = Bbar [I2^{AC} I1~B I1~D + I2^{AD} I1~B I1~C + I2^{BC} I1~A I1~D + I2^{BD} I1~A I1~C],  Bbar = 34/21 P1 P2 + 2<G P>
    T4h = I1~A I1~B I1~C I1~D Tbar,  Tbar = 12 P1 P2^2 F3bar(k2/k1) + 12 P1^2 P2 F3bar(k1/k2) + 8 <G^2 P>

Two references:
- The perturbation-theory kernels against their definition: the generic tree-level bispectrum and trispectrum at
  explicit vectors (symmetrised F2 and F3 from the standard recursion, P(0) pairings dropped), averaged over mu by
  scipy.integrate.quad with the ks nodes as breakpoints.  Unit pressure cubes isolate them: T4h = (sum w^)^4 Tbar and
  T3h = 4 (sum w^)^3 Bbar.  <G P> and <G^2 P> are held to 1e-8 of <|G| |P|> and <G^2 |P|>; F3bar, read from the 4-halo
  workspace, to 1e-12 of its mpmath value.
- The full terms against a float64 numpy restatement on the same inputs (np.interp, explicit trapezoids) whose mu
  averages are the same Laurent sums over long-double window moments of the piecewise-linear P.  Each element is held to
  TAU * B, B the same expression over absolute values (including |g_n| M_n(|P|) inside the mu averages).

Largest ratios measured on one B200 (1000 W power limit) are in DESIGN.md §4.7.
"""
import ctypes as C

import numpy as np
import pytest

HMV_E_ARG, HMV_E_LIMIT = -1, -3
TAU = 1e-12
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64
OBSERVED = {}
LD = np.longdouble


# ------------------------------------------------------------------------------------------------- host restatement
def _trapz_w(x):
    x = np.asarray(x, dtype=np.float64)
    n = x.size
    if n < 2:
        return np.zeros(n)
    return 0.5 * (x[np.minimum(np.arange(n) + 1, n - 1)] - x[np.maximum(np.arange(n) - 1, 0)])


def _ev(n):
    return n + n % 2


def _sides(zc, nk, n1, n2):
    return zc * (3 * _ev(n1) + 3 * _ev(n2) + 10 * nk)


def _ws3h(nz, nm, nk, n1, n2, nA1, nC1, zc):
    """k_trispec.cu's 3-halo workspace restated: the 2-halo panels, nA1 nC1 I2 blocks, the side vectors and tables."""
    nmp, n1p, n2p, n1q, n2q = _ev(nm), _ev(n1), _ev(n2), _ev(n1 + 1), _ev(n2 + 1)
    m1, m2 = nA1 * n1p, nC1 * n2p
    return zc * (nmp * (m1 + n1q + m2 + n2q) + m1 * m2) + _sides(zc, nk, n1, n2)


def _ws4h(nz, nk, n1, n2):
    return _sides(nz, nk, n1, n2) + 2 * n1 * n2


def _int_pow(n, u, v):
    """int_u^v q^n dq in long double without cancellation (u > 0 for n < 0)."""
    h = v - u
    if n >= 0:
        return h * sum(v ** i * u ** (n - i) for i in range(n + 1)) / (n + 1)
    if n == -1:
        return np.log1p(h / u)
    m = -n - 1                      # (u^-m - v^-m)/m = (v^m - u^m)/(m u^m v^m)
    return h * sum(v ** i * u ** (m - 1 - i) for i in range(m)) / (m * u ** m * v ** m)


def _window_moments(ks, P, a, b):
    """int_a^b q^n P(q) dq, n = -3, -1, 1, 3, 5 (rows), P linear on ks and held at its end values; long double."""
    ks, P = ks.astype(LD), P.astype(LD)
    edges = [(LD(0), ks[0], P[0], LD(0))] + [
        (ks[j], ks[j + 1], P[j] - (P[j + 1] - P[j]) / (ks[j + 1] - ks[j]) * ks[j], (P[j + 1] - P[j]) / (ks[j + 1] - ks[j]))
        for j in range(ks.size - 1)] + [(ks[-1], LD(np.inf), P[-1], LD(0))]
    M = np.zeros((5,) + a.shape, dtype=LD)
    for x0, x1, al, be in edges:             # P = al + be q on [x0, x1]
        u, v = np.maximum(a, x0), np.minimum(b, x1)
        on = v > u
        if not on.any():
            continue
        u, v = u[on], v[on]
        for r, n in enumerate((-3, -1, 1, 3, 5)):
            if n < 0:
                ok = u > 0
                val = np.zeros(u.shape, dtype=LD)
                val[ok] = al * _int_pow(n, u[ok], v[ok]) + (be * _int_pow(n + 1, u[ok], v[ok]) if be != 0 else 0)
            else:
                val = al * _int_pow(n, u, v) + be * _int_pow(n + 1, u, v)
            M[r][on] += val
    return M


def _mu_averages(ks, P, k1, k2, P1, P2):
    """(<G P>, <G^2 P>, bound of each): the Laurent sums over exact window moments, in long double.  Bounds: sum of
    |coefficient| M_n(|P|)."""
    k1, k2 = np.broadcast_arrays(np.asarray(k1, dtype=np.float64), np.asarray(k2, dtype=np.float64))
    P1, P2 = np.broadcast_to(P1, k1.shape).astype(LD), np.broadcast_to(P2, k1.shape).astype(LD)
    K1, K2 = k1.astype(LD), k2.astype(LD)
    lo, hi = np.minimum(K1, K2), np.maximum(K1, K2)
    a, b = hi - lo, hi + lo
    M, Ma = _window_moments(ks, P, a, b), _window_moments(ks, np.abs(P), a, b)
    d = (K1 - K2) * (K1 + K2)
    r1, r2 = P1 / K1 ** 2, P2 / K2 ** 2
    g1 = -LD(5) / 28 * (r1 + r2)
    g0 = LD(13) / 28 * (P1 + P2) - LD(3) / 28 * d * (r1 - r2)
    gm = -d / 4 * (P1 - P2) + d * d / 14 * (r1 + r2)
    inv = 1 / (2 * K1 * K2)
    t1 = [g1 * M[3], g0 * M[2], gm * M[1]]
    b1 = [abs(g1) * Ma[3], abs(g0) * Ma[2], abs(gm) * Ma[1]]
    t2 = [g1 * g1 * M[4], 2 * g1 * g0 * M[3], (g0 * g0 + 2 * g1 * gm) * M[2], 2 * g0 * gm * M[1], gm * gm * M[0]]
    b2 = [g1 * g1 * Ma[4], abs(2 * g1 * g0) * Ma[3], (g0 * g0 + abs(2 * g1 * gm)) * Ma[2], abs(2 * g0 * gm) * Ma[1],
          gm * gm * Ma[0]]
    f = lambda t: np.asarray(sum(t) * inv, dtype=np.float64)
    return f(t1), f(t2), f(b1), f(b2)


def _f3bar_mp(r, tail=False, as_mp=False):
    """F3bar(r) in mpmath; tail: F3bar(r) + 1/(18 r^2), the 4-halo table's entry for a small ratio of the large-ratio
    branch."""
    import mpmath as mp
    with mp.workdps(80):
        r = r if isinstance(r, mp.mpf) else mp.mpf(float(r))     # an mpf ratio stays exact: Tbar weighs it with r^2
        if r == 1:
            v = mp.mpf(-11) / 378
        else:
            L = mp.log(abs((1 + r) / (1 - r)))
            v = (12 / r ** 2 - 158 + 100 * r ** 2 - 42 * r ** 4 + (3 / r ** 3) * (r ** 2 - 1) ** 3 * (7 * r ** 2 + 2) * L) \
                / (3024 * r ** 2)
        if tail:
            v += 1 / (18 * r ** 2)
        return v if as_mp else float(v)


R_LOCAL = 100.0      # k_trispec.cu's PT_R0: ratios max/min at or above it take the local large-ratio branch


def _pt_mp(ks, P, k1, k2):
    """(Bbar, Tbar) in mpmath (80 digits): the Laurent sums over exact window moments of the piecewise-linear P and
    F3bar from its closed form.  At r = 1e6 Tbar is 1e-12 of its two leading pieces; 80 digits keep it exact."""
    import bisect
    import mpmath as mp
    with mp.workdps(80):
        K, PP = [mp.mpf(float(x)) for x in ks], [mp.mpf(float(x)) for x in P]

        def Pi(x):
            if x < K[0]:
                return PP[0]
            if x >= K[-1]:
                return PP[-1]
            r = bisect.bisect_right(K, x) - 1
            return PP[r] + (PP[r + 1] - PP[r]) / (K[r + 1] - K[r]) * (x - K[r])
        k1, k2 = mp.mpf(float(k1)), mp.mpf(float(k2))
        P1, P2 = Pi(k1), Pi(k2)
        a, b = abs(k1 - k2), k1 + k2
        edges = [(mp.mpf(0), K[0], PP[0], mp.mpf(0))] + [
            (K[j], K[j + 1], PP[j] - (PP[j + 1] - PP[j]) / (K[j + 1] - K[j]) * K[j], (PP[j + 1] - PP[j]) / (K[j + 1] - K[j]))
            for j in range(len(K) - 1)] + [(K[-1], mp.inf, PP[-1], mp.mpf(0))]

        def F(n, x):
            return mp.log(x) if n == -1 else x ** (n + 1) / (n + 1)
        M = {}
        for n in (-3, -1, 1, 3, 5):
            s = mp.mpf(0)
            for x0, x1, al, be in edges:
                u, v = max(a, x0), min(b, x1)
                if v <= u or (n < 0 and u == 0):
                    continue
                s += al * (F(n, v) - F(n, u)) + be * (F(n + 1, v) - F(n + 1, u))
            M[n] = s
        d, r1, r2 = k1 * k1 - k2 * k2, P1 / k1 ** 2, P2 / k2 ** 2
        g1 = -mp.mpf(5) / 28 * (r1 + r2)
        g0 = mp.mpf(13) / 28 * (P1 + P2) - mp.mpf(3) / 28 * d * (r1 - r2)
        gm = -d / 4 * (P1 - P2) + d * d / 14 * (r1 + r2)
        inv = 1 / (2 * k1 * k2)
        gp = (g1 * M[3] + g0 * M[1] + gm * M[-1]) * inv
        g2p = (g1 * g1 * M[5] + 2 * g1 * g0 * M[3] + (g0 * g0 + 2 * g1 * gm) * M[1] + 2 * g0 * gm * M[-1]
               + gm * gm * M[-3]) * inv
        Tb = 12 * P1 * P2 * P2 * _f3bar_mp(k2 / k1, as_mp=True) + 12 * P1 * P1 * P2 * _f3bar_mp(k1 / k2, as_mp=True) \
            + 8 * g2p
        return float(mp.mpf(34) / 21 * P1 * P2 + 2 * gp), float(Tb)


def _f3_table(q1, q2, proj):
    s = 0.5 if proj else 0.0
    x1, x2 = q1 + s, q2 + s
    F12 = np.array([[_f3bar_mp(b / a) for b in x2] for a in x1])
    F21 = np.array([[_f3bar_mp(a / b) for b in x2] for a in x1])
    return F12, F21


def _reference(order, cubes, kinds, ms, nzm, bh, Pzk, rho, ks, q1, q2, chis=None, zs=None, pref=None):
    """(value, bound): T3h or T4h (order 3 or 4) [nz, n1, n2] when chis is None, else the covariance [n1, n2]."""
    nz, nm = cubes[0].shape[:2]
    w = _trapz_w(ms)[None, :] * nzm * bh
    a = [ms / rho if k == 0 else np.ones(nm) for k in kinds]
    T, B = np.empty((nz, q1.size, q2.size)), np.empty((nz, q1.size, q2.size))
    if order == 4:
        F12, F21 = _f3_table(q1, q2, chis is not None)
    for z in range(nz):
        k1 = q1 if chis is None else (q1 + 0.5) * (1.0 / chis[z])
        k2 = q2 if chis is None else (q2 + 0.5) * (1.0 / chis[z])
        t = [a[i][:, None] * np.array([np.interp(k1 if i < 2 else k2, ks, cubes[i][z, m]) for m in range(nm)])
             for i in range(4)]
        W, Wa = w[z][:, None], np.abs(w[z])[:, None]
        cons = 1.0 - np.sum(w[z] * ms / rho)
        I1 = [((W * t[i]).sum(0) + (cons if kinds[i] == 0 else 0.0),
               (Wa * np.abs(t[i])).sum(0) + (abs(cons) if kinds[i] == 0 else 0.0)) for i in range(4)]
        P1, P2 = np.interp(k1, ks, Pzk[z]), np.interp(k2, ks, Pzk[z])
        gp, g2p, gpb, g2pb = _mu_averages(ks, Pzk[z], k1[:, None], k2[None, :], P1[:, None], P2[None, :])
        A, Bi, Cc, D = [(x[0], x[1]) for x in I1]
        if order == 3:
            def I2(x, y):
                return (W * x).T @ y, (Wa * np.abs(x)).T @ np.abs(y)
            I2AC, I2AD, I2BC, I2BD = I2(t[0], t[2]), I2(t[0], t[3]), I2(t[1], t[2]), I2(t[1], t[3])
            Bb = (34 / 21 * P1[:, None] * P2[None, :] + 2 * gp, 34 / 21 * np.abs(P1[:, None] * P2[None, :]) + 2 * gpb)
            for s in range(2):
                v = Bb[s] * (I2AC[s] * Bi[s][:, None] * D[s][None, :] + I2AD[s] * Bi[s][:, None] * Cc[s][None, :]
                             + I2BC[s] * A[s][:, None] * D[s][None, :] + I2BD[s] * A[s][:, None] * Cc[s][None, :])
                (T if s == 0 else B)[z] = v if s == 0 else np.abs(v)
        else:
            p1, p2 = P1[:, None], P2[None, :]
            Tb = (12 * p1 * p2 * (p2 * F12 + p1 * F21) + 8 * g2p,
                  12 * np.abs(p1 * p2) * (np.abs(p2 * F12) + np.abs(p1 * F21)) + 8 * g2pb)
            for s in range(2):
                v = A[s][:, None] * Bi[s][:, None] * Cc[s][None, :] * D[s][None, :] * Tb[s]
                (T if s == 0 else B)[z] = v if s == 0 else np.abs(v)
    if chis is None:
        return T, B
    zw = (_trapz_w(zs) if nz > 1 else np.ones(1)) * pref
    return np.einsum("z,zln->ln", zw, T), np.einsum("z,zln->ln", np.abs(zw), B)


def _assert_bound(name, got, want, bound, tau=TAU):
    got, want, bound = (np.asarray(x, dtype=np.float64) for x in (got, want, bound))
    assert got.shape == want.shape, name
    assert np.all(np.isfinite(got)), "%s: non-finite output" % name
    err = np.abs(got - want)
    zero = bound == 0.0
    assert np.all(err[zero] == 0.0), "%s: error where every term is zero" % name
    ratio = float(np.max(err[~zero] / bound[~zero])) if (~zero).any() else 0.0
    key = name.split(" ")[0]
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), ratio)
    assert ratio <= tau, "%s: max |got-want| / bound = %.3g > %.1g" % (name, ratio, tau)


# ------------------------------------------------------------------------------------------------- generic tree level
def _F2(a, b):
    ab, a2, b2 = a @ b, a @ a, b @ b
    return 5 / 7 + 0.5 * ab * (1 / a2 + 1 / b2) + 2 / 7 * ab * ab / (a2 * b2)


def _G2(a, b):
    ab, a2, b2 = a @ b, a @ a, b @ b
    return 3 / 7 + 0.5 * ab * (1 / a2 + 1 / b2) + 4 / 7 * ab * ab / (a2 * b2)


def _F3u(q1, q2, q3):
    """Unsymmetrised F3 of the standard recursion; terms whose partial sum vanishes are zero (their G2 factor vanishes
    faster than alpha, beta diverge)."""
    def al(a, b):
        return (a + b) @ a / (a @ a)

    def be(a, b):
        s = a + b
        return (s @ s) * (a @ b) / (2 * (a @ a) * (b @ b))
    q23, q12 = q2 + q3, q1 + q2
    t = 0.0
    if q23 @ q23 > 0:
        t += 7 * al(q1, q23) * _F2(q2, q3) + 2 * be(q1, q23) * _G2(q2, q3)
    if q12 @ q12 > 0:
        t += (7 * al(q12, q3) + 2 * be(q12, q3)) * _G2(q1, q2)
    return t / 18


def _F3s(a, b, c):
    from itertools import permutations
    return sum(_F3u(*p) for p in permutations((a, b, c))) / 6


def _tree(ks, P, k1, k2, mu):
    """(B(k1+k2, -k1, -k2), T(k1, -k1, k2, -k2) without P(0) pairings, G) at the angle mu."""
    Pf = lambda k: np.interp(k, ks, P)
    v1 = np.array([0.0, 0.0, k1])
    v2 = k2 * np.array([np.sqrt(max(1 - mu * mu, 0.0)), 0.0, mu])
    s = v1 + v2
    q = np.sqrt(s @ s)
    P1, P2, Pq = Pf(k1), Pf(k2), Pf(q)
    G = P1 * _F2(-v1, s) + P2 * _F2(-v2, s)
    Bt = 2 * (_F2(-v1, -v2) * P1 * P2 + _F2(s, -v1) * Pq * P1 + _F2(s, -v2) * Pq * P2)
    legs = [v1, -v1, v2, -v2]
    Pl = [P1, P1, P2, P2]
    T = 0.0
    for d in range(4):
        o = [i for i in range(4) if i != d]
        T += 6 * _F3s(*[legs[i] for i in o]) * Pl[o[0]] * Pl[o[1]] * Pl[o[2]]
    for c in range(4):
        for dd in range(c + 1, 4):
            a_, b_ = [i for i in range(4) if i not in (c, dd)]
            for x, y in ((a_, b_), (b_, a_)):
                kc = legs[c] + legs[x]
                n = np.sqrt(kc @ kc)
                if n == 0:
                    continue
                T += 4 * _F2(-legs[x], kc) * _F2(-legs[y], legs[dd] + legs[y]) * Pl[x] * Pl[y] * Pf(n)
    return Bt, T, G, Pq


def _tree_averages(ks, P, k1, k2):
    """(Bbar, Tbar, <|G| |P|>, <G^2 |P|>) by quad over mu with breakpoints where |k1 +- k2| crosses a node."""
    from scipy.integrate import quad
    c, s2 = 2 * k1 * k2, k1 * k1 + k2 * k2
    pts = sorted({m for kn in ks for m in ((kn * kn - s2) / c, -(kn * kn - s2) / c) if -1 < m < 1})
    kw = dict(points=pts or None, limit=2000, epsabs=0, epsrel=1e-13)
    out = []
    for f in (lambda m: _tree(ks, P, k1, k2, m)[0], lambda m: _tree(ks, P, k1, k2, m)[1],
              lambda m: abs(_tree(ks, P, k1, k2, m)[2] * _tree(ks, P, k1, k2, m)[3]),
              lambda m: _tree(ks, P, k1, k2, m)[2] ** 2 * abs(_tree(ks, P, k1, k2, m)[3])):
        out.append(0.5 * quad(f, -1, 1, **kw)[0])
    return out


# ------------------------------------------------------------------------------------------------- CPU-only
def test_trispec_pt_rejects_before_any_launch():
    """Every argument and limit check of the four entry points runs before the first launch; the workspace functions
    agree with the plans restated in _ws3h / _ws4h; HODs raise ValueError and a z-sharded model NotImplementedError
    before any device work."""
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

    def t3(nz=2, nm=40, nk=30, ldk=32, ks=p[0], u=ok_u, k=ok_k, ws=p[9], bh=p[12], Pzk=p[13], zchunk=1):
        return L.hmv_trispec_3h(nz, nm, nk, ldk, ks, p[1], p[2], bh, Pzk, 1.0, u, k, 5, p[7], 6, p[8], zchunk, ws,
                                p[10], None)

    def c3(chis=p[11], zchunk=2, nz=2, nm=40, ldk=32):
        return L.hmv_cl_cov_3h(nz, nm, 30, ldk, p[0], p[1], p[2], p[12], p[13], 1.0, ok_u, ok_k, 5, p[7], 6, p[8],
                               p[1], chis, p[2], zchunk, p[9], p[10], None)

    def t4(nz=2, nm=40, nk=30, ldk=32, ks=p[0], u=ok_u, k=ok_k, ws=p[9], bh=p[12], Pzk=p[13], out=p[10]):
        return L.hmv_trispec_4h(nz, nm, nk, ldk, ks, p[1], p[2], bh, Pzk, 1.0, u, k, 5, p[7], 6, p[8], ws, out, None)

    def c4(chis=p[11], nz=2, nm=40, ldk=32, ws=p[9]):
        return L.hmv_cl_cov_4h(nz, nm, 30, ldk, p[0], p[1], p[2], p[12], p[13], 1.0, ok_u, ok_k, 5, p[7], 6, p[8],
                               p[1], chis, p[2], ws, p[10], None)

    cases = {
        "3h nz = 0": (lambda: t3(nz=0), HMV_E_ARG, "sizes must be >= 1"),
        "3h nk = 1": (lambda: t3(nk=1, ldk=2), HMV_E_ARG, "nk >= 2"),
        "3h odd ldk": (lambda: t3(ldk=31), HMV_E_ARG, "ldk must be even"),
        "3h null ks": (lambda: t3(ks=None), HMV_E_ARG, "hmv_trispec_3h: null pointer"),
        "3h null cube": (lambda: t3(u=cubes(p[3], p[4], None, p[6])), HMV_E_ARG, "null pointer (cube 2)"),
        "3h hod kind": (lambda: t3(k=kinds(0, 1, 2, 2)), HMV_E_ARG, "kind 1 is neither"),
        "3h misaligned cube": (lambda: t3(u=cubes(p[3], bad, p[5], p[6])), HMV_E_ARG, "cube 1 must be 16-byte"),
        "3h misaligned ws": (lambda: t3(ws=bad), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "3h null bh": (lambda: t3(bh=None), HMV_E_ARG, "null pointer (bh or Pzk)"),
        "3h null Pzk": (lambda: t3(Pzk=None), HMV_E_ARG, "null pointer (bh or Pzk)"),
        "3h zchunk = 0": (lambda: t3(zchunk=0), HMV_E_ARG, "zchunk must lie in [1, nz]"),
        "3h zchunk > nz": (lambda: t3(zchunk=3), HMV_E_ARG, "zchunk must lie in [1, nz]"),
        "3h nz > 65535": (lambda: t3(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        "cov3 null chis": (lambda: c3(chis=None), HMV_E_ARG, "hmv_cl_cov_3h: null pointer (zs, chis or pref)"),
        "cov3 zchunk": (lambda: c3(zchunk=-1), HMV_E_ARG, "hmv_cl_cov_3h: zchunk"),
        "cov3 K > 2^30": (lambda: c3(nz=60000, nm=20000, zchunk=1), HMV_E_LIMIT, "exceeds 2^30"),
        "4h nz = 0": (lambda: t4(nz=0), HMV_E_ARG, "hmv_trispec_4h: sizes must be >= 1"),
        "4h odd ldk": (lambda: t4(ldk=33), HMV_E_ARG, "ldk must be even"),
        "4h null ks": (lambda: t4(ks=None), HMV_E_ARG, "hmv_trispec_4h: null pointer"),
        "4h null out": (lambda: t4(out=None), HMV_E_ARG, "hmv_trispec_4h: null pointer"),
        "4h hod kind": (lambda: t4(k=kinds(0, 0, 1, 2)), HMV_E_ARG, "kind 1 is neither"),
        "4h misaligned ws": (lambda: t4(ws=bad), HMV_E_ARG, "workspace must be 16-byte aligned"),
        "4h null bh": (lambda: t4(bh=None), HMV_E_ARG, "null pointer (bh or Pzk)"),
        "4h nz > 65535": (lambda: t4(nz=70000, nm=2), HMV_E_LIMIT, "exceeds 65535"),
        "cov4 null chis": (lambda: c4(chis=None), HMV_E_ARG, "hmv_cl_cov_4h: null pointer (zs, chis or pref)"),
        "cov4 misaligned ws": (lambda: c4(ws=bad), HMV_E_ARG, "hmv_cl_cov_4h: workspace must be 16-byte aligned"),
    }
    for what, (call, code, msg) in cases.items():
        rc = call()
        assert rc == code and msg in capi.last_error(), (what, rc, capi.last_error())
    patterns = [((3, 4, 5, 6), (0, 0, 2, 2), 2, 2), ((3, 4, 3, 4), (0, 2, 0, 2), 2, 2),
                ((3, 3, 5, 5), (0, 2, 0, 0), 2, 1), ((3, 3, 5, 6), (0, 0, 2, 2), 1, 2),
                ((3, 3, 3, 3), (2, 2, 2, 2), 1, 1)]
    for fn in (L.hmv_trispec_3h_ws_doubles, L.hmv_cl_cov_3h_ws_doubles):
        assert fn(0, 4, 10, 3, 3, ok_u, ok_k, 1) == 0 and fn(2, 4, 1, 3, 3, ok_u, ok_k, 1) == 0
        assert fn(3, 4, 10, 3, 3, ok_u, ok_k, 0) == 0 and fn(3, 4, 10, 3, 3, ok_u, ok_k, 4) == 0
        for idx, kk, nA1, nC1 in patterns:
            for nz, nm, nk, n1, n2, zc in [(1, 1, 2, 1, 1, 1), (3, 41, 37, 7, 65, 2), (200, 2000, 10000, 1000, 1000, 53)]:
                got = fn(nz, nm, nk, n1, n2, cubes(*[p[i] for i in idx]), kinds(*kk), zc)
                assert got == _ws3h(nz, nm, nk, n1, n2, nA1, nC1, zc), (idx, kk, nz, nm, n1, n2, zc)
    for fn in (L.hmv_trispec_4h_ws_doubles, L.hmv_cl_cov_4h_ws_doubles):
        assert fn(0, 10, 3, 3) == 0 and fn(2, 1, 3, 3) == 0 and fn(2, 10, 0, 3) == 0
        for nz, nk, n1, n2 in [(1, 2, 1, 1), (3, 37, 7, 65), (200, 10000, 1000, 1000)]:
            assert fn(nz, nk, n1, n2) == _ws4h(nz, nk, n1, n2)

    from hmvec_b200.hmvec import HaloModel

    class Stub(HaloModel):
        def __init__(self):
            self._zcomm, self.uk_profiles, self.pk_profiles = None, {}, {}
            self.hods, self._ks64, self._nz = {"g": None}, np.geomspace(1e-3, 10, 20), 4
    h = Stub()
    for f in (h.get_trispectrum_3halo, h.get_trispectrum_4halo):
        with pytest.raises(ValueError, match="HOD"):
            f([0.1], name="g")
    h._zcomm = object()
    for f in (h.get_cl_cov_3halo, h.get_cl_cov_4halo):
        with pytest.raises(NotImplementedError):
            f(np.array([100.0]))


# ------------------------------------------------------------------------------------------------- GPU: the C ABI
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    yield torch, capi
    print("\n3-/4-halo largest measured ratios:", {k: "%.2g" % v for k, v in sorted(OBSERVED.items())})


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


def _inputs(rng, nz, nm, nk=37, P=None):
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


def _abi(torch, capi, order, proj, inp, cubes, kinds, q1, q2, zchunks=(1,), same=None, want_ws=False):
    """One launch per zchunk (4h: one plan), each twice: bit-identical across every launch, guards intact.  same:
    which cube each leg reads ((0, 0, 2, 2): A = B and C = D share one device cube)."""
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
    nA1 = 1 if same[0] == same[1] and kinds[0] == kinds[1] else 2
    nC1 = 1 if same[2] == same[3] and kinds[2] == kinds[3] else 2
    outs = []
    for zc in (zchunks if order == 3 else (None,)):
        if order == 3:
            nws = (L.hmv_cl_cov_3h_ws_doubles if proj else L.hmv_trispec_3h_ws_doubles)(nz, nm, nk, n1, n2, u_h, k_h,
                                                                                      zc)
            assert nws == _ws3h(nz, nm, nk, n1, n2, nA1, nC1, zc)
        else:
            nws = (L.hmv_cl_cov_4h_ws_doubles if proj else L.hmv_trispec_4h_ws_doubles)(nz, nk, n1, n2)
            assert nws == _ws4h(nz, nk, n1, n2)
        ws = torch.full((int(nws),), float("nan"), dtype=torch.float64, device="cuda")
        buf, optr = _guarded(torch, n)
        base = [nz, nm, nk, ldk, p(d["ks"]), p(d["ms"]), p(d["nzm"]), p(d["bh"]), p(d["Pzk"]), inp["rho"], u_h, k_h,
                n1, p(d["q1"]), n2, p(d["q2"])]
        extra = [p(d["zs"]), p(d["chis"]), p(d["pref"])] if proj else []
        zarg = [zc] if order == 3 else []
        fn = getattr(L, "hmv_%s_%dh" % ("cl_cov" if proj else "trispec", order))
        for _ in range(2):
            capi.check(fn(*base, *extra, *zarg, p(ws), optr, capi.stream()), "pt ABI")
            torch.cuda.synchronize()
            outs.append(buf.clone())
    for o in outs[1:]:
        assert torch.equal(outs[0].view(torch.int64), o.view(torch.int64)), "launches or zchunks differ"
    got = _read_guarded(outs[0], n, shape)
    return (got, ws.cpu().numpy()) if want_ws else got


def _abi_ref(order, inp, cubes, kinds, q1, q2, proj):
    extra = (inp["chis"], inp["zs"], inp["pref"]) if proj else ()
    return _reference(order, cubes, kinds, inp["ms"], inp["nzm"], inp["bh"], inp["Pzk"], inp["rho"], inp["ks"], q1, q2,
                      *extra)


def _unit_inputs(nz, nk, P):
    ks = np.geomspace(1e-2, 10.0, nk)
    return ks, dict(ks=ks, ms=np.array([1.0, 3.0]), nzm=np.ones((nz, 2)), bh=np.ones((nz, 2)), Pzk=P,
                    zs=np.linspace(0.1, 1.0, nz), chis=np.ones(nz), pref=np.ones(nz), rho=1.0)


@pytest.mark.gpu
def test_pt_kernels_against_tree_level(env):
    """Unit pressure cubes on two masses with w^ = 1: I1~ = I2 = 2, so T4h = 16 Tbar and T3h = 32 Bbar, against the
    generic tree-level B and T averaged over mu by quad.  Pairs: k1 = k2, k1/k2 = 1e-3 and 1e3, windows crossing ks[0]
    and ks[-1], k outside the grid."""
    torch, capi = env
    nk, nz = 30, 1
    ks0 = np.geomspace(1e-2, 10.0, nk)
    P = ((ks0 / 0.05) / (1.0 + (ks0 / 0.05) ** 2.5))[None, :]
    ks, inp = _unit_inputs(nz, nk, P)
    cube = np.ones((nz, 2, nk))
    k1 = np.array([0.5, 0.5, 2e-3, 2.0, 0.013, 6.0, 0.02, 0.3, 4e-3, 30.0, 0.05])
    k2 = np.array([0.5, 0.5 + 1e-7, 2.0, 2e-3, 0.012, 7.5, 3.0, 0.3001, 5e-3, 0.2, 40.0])
    T4 = _abi(torch, capi, 4, False, inp, [cube] * 4, (2, 2, 2, 2), k1, k2, same=(0, 0, 0, 0))
    T3 = _abi(torch, capi, 3, False, inp, [cube] * 4, (2, 2, 2, 2), k1, k2, same=(0, 0, 0, 0))
    for z in range(nz):
        for i in range(k1.size):
            Bb, Tb, gabs, g2abs = _tree_averages(ks, P[z], k1[i], k2[i])
            P1, P2 = np.interp(k1[i], ks, P[z]), np.interp(k2[i], ks, P[z])
            bB = 2e-8 * gabs + 1e-13 * 34 / 21 * abs(P1 * P2)
            f12, f21 = _f3bar_mp(k2[i] / k1[i]), _f3bar_mp(k1[i] / k2[i])
            bT = 8e-8 * g2abs + 1e-10 * 12 * (abs(P1 * P2 * P2 * f12) + abs(P1 * P1 * P2 * f21))
            eB, eT = abs(T3[z, i, i] / 32 - Bb), abs(T4[z, i, i] / 16 - Tb)
            OBSERVED["tree_B/1e-8"] = max(OBSERVED.get("tree_B/1e-8", 0.0), eB / bB)
            OBSERVED["tree_T/1e-8"] = max(OBSERVED.get("tree_T/1e-8", 0.0), eT / bT)
            assert eB <= bB, (z, i, T3[z, i, i] / 32, Bb)
            assert eT <= bT, (z, i, T4[z, i, i] / 16, Tb)


@pytest.mark.gpu
def test_f3bar_against_mpmath(env):
    """The F3bar table of the 4-halo workspace at r = k2/k1 in [1e-6, 1e6], both series switches and r = 1."""
    torch, capi = env
    ks, inp = _unit_inputs(1, 8, np.ones((1, 8)))
    r = np.r_[np.geomspace(1e-6, 1e6, 121), 1.0, 0.4, 0.4 * (1 - 1e-15), 2.5, 2.5 * (1 + 1e-15), 1 - 1e-9, 1 + 1e-9,
              0.999, 1.001, 0.05, 20.0]
    k1 = np.array([1.0])
    _, ws = _abi(torch, capi, 4, False, inp, [np.ones((1, 2, 8))] * 4, (2, 2, 2, 2), k1, r, same=(0, 0, 0, 0),
                 want_ws=True)
    off = _sides(1, 8, 1, r.size)
    F12, F21 = ws[off:off + r.size], ws[off + r.size:off + 2 * r.size]
    local = np.maximum(r, 1.0) >= R_LOCAL * np.minimum(r, 1.0)
    assert local.sum() >= 40 and (~local).sum() >= 40
    for got, rr in ((F12, r / 1.0), (F21, 1.0 / r)):
        want = np.array([_f3bar_mp(x, tail=bool(loc and x < 1)) for x, loc in zip(rr, local)])
        _assert_bound("f3bar", got, want, np.abs(want))


@pytest.mark.gpu
def test_large_ratio_against_mpmath(env):
    """Tbar and Bbar at max/min ratios 1e3 ... 1e6 (and on both sides of the switch to the local branch), each held to
    a small multiple of |Tbar| and |Bbar| themselves against an 80-digit mpmath evaluation: Tbar is there up to 1e-12 of
    its two leading pieces, which cancel.  Unit pressure cubes: T4h = 16 Tbar, T3h = 32 Bbar.  A P_lin-like P on
    geomspace(1e-4, 100, 400); windows inside one interval, across nodes and across ks[-1]; k below the grid."""
    torch, capi = env
    nk = 400
    ks0 = np.geomspace(1e-4, 100.0, nk)
    P = (ks0 / (1.0 + (ks0 / 0.02) ** 2.6) * 1e4)[None, :]
    ks, inp = _unit_inputs(1, nk, P)
    inp["ks"] = ks = ks0
    k1 = np.array([3e-4, 0.3, 2.6e-4, 1e-4, 20.0, 2e-5, 1.7e-3, 0.01, 0.01, 0.05, 1e-3, 6e-4])
    k2 = np.array([0.3, 3e-4, 2.6, 100.0, 2e-5, 20.0, 170.0, 1.01, 0.99, 0.05 * 99.5, 10.0, 3.3])
    r = np.maximum(k1, k2) / np.minimum(k1, k2)
    assert r.max() >= 1e6 and ((r > 95) & (r < R_LOCAL)).any() and ((r > R_LOCAL) & (r < 105)).any()
    cube = np.ones((1, 2, nk))
    T4 = _abi(torch, capi, 4, False, inp, [cube] * 4, (2, 2, 2, 2), k1, k2, same=(0, 0, 0, 0))
    T3 = _abi(torch, capi, 3, False, inp, [cube] * 4, (2, 2, 2, 2), k1, k2, same=(0, 0, 0, 0))
    for i in range(k1.size):
        Bb, Tb = _pt_mp(ks, P[0], k1[i], k2[i])
        eB, eT = abs(T3[0, i, i] / 32 - Bb) / abs(Bb), abs(T4[0, i, i] / 16 - Tb) / abs(Tb)
        OBSERVED["large_ratio_B"] = max(OBSERVED.get("large_ratio_B", 0.0), eB)
        OBSERVED["large_ratio_T"] = max(OBSERVED.get("large_ratio_T", 0.0), eT)
        assert eB <= 1e-11, (r[i], T3[0, i, i] / 32, Bb)
        assert eT <= 1e-8, (r[i], T4[0, i, i] / 16, Tb)


PLAN_CASES = [  # (n1, n2, nz, nm, same, zchunks) -- 3h rows nA1 n1p pick MT 4 / 8 / 16 / 26
    (1, 1, 1, 1, (0, 1, 2, 3), (1,)),                 # MT 4, nm = 1
    (7, 9, 5, 41, (0, 1, 2, 3), (1, 2, 5)),           # MT 4, 4 blocks, zchunk 2 does not divide 5
    (31, 20, 3, 30, (0, 0, 2, 3), (1, 3)),            # rows 32: MT 4; 2 blocks (A = B)
    (40, 7, 4, 17, (0, 1, 2, 2), (1, 3, 4)),          # rows 80: MT 16; 2 blocks (C = D)
    (60, 33, 2, 25, (0, 0, 2, 2), (1, 2)),            # rows 60: MT 8; 1 block
    (140, 13, 3, 21, (0, 1, 2, 3), (1, 2, 3)),        # rows 280: MT 26, two row tiles
]


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
@pytest.mark.parametrize("proj", [False, True], ids=["trispec", "cov"])
@pytest.mark.parametrize("n1,n2,nz,nm,same,zchunks", PLAN_CASES)
def test_plans(env, order, proj, n1, n2, nz, nm, same, zchunks):
    torch, capi = env
    rng = np.random.default_rng(n1 * 31 + n2 + nz * 7 + nm + proj + 100 * order)
    inp = _inputs(rng, nz, nm)
    base = [rng.uniform(-0.3, 1.2, (nz, nm, 37)) for _ in range(4)]
    cubes = [base[s] for s in same]
    kinds = (0, 0, 2, 2) if same[0] == same[1] or same[2] == same[3] else (0, 2, 0, 2)
    if proj:
        q1, q2 = rng.uniform(2.0, 2e4, n1), rng.uniform(2.0, 2e4, n2)    # k spans below ks[0] to above ks[-1]
    else:
        q1, q2 = rng.uniform(3e-3, 20.0, n1), rng.uniform(3e-3, 20.0, n2)
    got = _abi(torch, capi, order, proj, inp, cubes, kinds, q1, q2, zchunks, same)
    want, bnd = _abi_ref(order, inp, cubes, kinds, q1, q2, proj)
    _assert_bound("abi%dh n1=%d n2=%d nz=%d nm=%d proj=%d" % (order, n1, n2, nz, nm, proj), got, want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
def test_single_redshift_cov_is_pref_times_trispectrum(env, order):
    torch, capi = env
    rng = np.random.default_rng(11 + order)
    inp = _inputs(rng, 1, 19)
    cubes = [rng.uniform(-0.3, 1.2, (1, 19, 37)) for _ in range(4)]
    ells, ells2 = rng.uniform(2.0, 2e4, 13), rng.uniform(2.0, 2e4, 6)
    cov = _abi(torch, capi, order, True, inp, cubes, (0, 2, 0, 2), ells, ells2)
    chi = inp["chis"][0]
    T = _abi(torch, capi, order, False, inp, cubes, (0, 2, 0, 2), (ells + 0.5) * (1.0 / chi), (ells2 + 0.5) * (1.0 / chi))
    _, bnd = _abi_ref(order, inp, cubes, (0, 2, 0, 2), ells, ells2, True)
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


def _model_ref(order, host, names, q1, q2, windows=None, fsky=1.0):
    cubes, kinds = zip(*[host["cube"][n] for n in names])
    args = (order, cubes, kinds, host["ms"], host["nzm"], host["bh"], host["Pzk"], host["rho"], host["ks"], q1, q2)
    if windows is None:
        return _reference(*args)
    W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), host["zs"].shape) for w in windows], axis=0)
    pref = host["H"] ** 3 * W / host["chis"] ** 6 / (4 * np.pi * fsky)
    return _reference(*args, host["chis"], host["zs"], pref)


def _win(host, names):
    return tuple(1.0 if n == "y" else host["Wk"] for n in names)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_trispectrum_tracers(model, order, names):
    """3D mode: k on the grid, between grid points, below and above the grid (clamped), unsorted."""
    h, host = model
    ks = host["ks"]
    k1 = np.array([ks[40], np.sqrt(ks[10] * ks[11]), 1e-5, 100.0, ks[0], ks[-1], 0.5 * (ks[3] + ks[4])])
    k2 = np.array([3.0, ks[70], 2e-4, np.sqrt(ks[100] * ks[101]), 45.0])
    got = getattr(h, "get_trispectrum_%dhalo" % order)(k1, k2, *names)
    assert got.shape == (4, k1.size, k2.size)
    want, bnd = _model_ref(order, host, names, k1, k2)
    _assert_bound("trispec_model%dh %s" % (order, "-".join(names)), got, want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
@pytest.mark.parametrize("names", COMBOS, ids=["-".join(c) for c in COMBOS])
def test_cl_cov_tracers(model, order, names):
    """Projected mode: unsorted multipoles, l = 2 (k below ks at high z) and l = 2e4 (k above ks at low z), ells2 !=
    ells, fsky < 1, kappa windows from lensing_window and y windows of 1."""
    h, host = model
    ells = np.array([300.0, 2.0, 20000.0, 45.5, 1000.0, 7.0, 3000.0])
    ells2 = np.array([10.0, 5000.0, 2.0, 150.0])
    win = _win(host, names)
    got = getattr(h, "get_cl_cov_%dhalo" % order)(ells, *names, windows=win, fsky=0.4, ells2=ells2)
    want, bnd = _model_ref(order, host, names, ells, ells2, win, 0.4)
    _assert_bound("cov_model%dh %s" % (order, "-".join(names)), got, want, bnd)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
def test_structure(model, order):
    """T^{ABCD}(k1,k2) = T^{CDAB}(k2,k1)^T; T is invariant under A <-> B; the auto covariance is symmetric; for the
    3-halo term a budget small enough to force one redshift per pass gives the same bits."""
    h, host = model
    tri = getattr(h, "get_trispectrum_%dhalo" % order)
    cov = getattr(h, "get_cl_cov_%dhalo" % order)
    k1, k2 = np.geomspace(2e-3, 20, 11), np.geomspace(5e-3, 8, 6)
    a = tri(k1, k2, "nfw", "y", "electron", "nfw")
    b = tri(k2, k1, "electron", "nfw", "nfw", "y")
    _, bnd = _model_ref(order, host, ("nfw", "y", "electron", "nfw"), k1, k2)
    _assert_bound("transpose", a, b.transpose(0, 2, 1), bnd)
    c = tri(k1, k2, "y", "nfw", "electron", "nfw")
    _assert_bound("swap_AB", a, c, bnd)
    ells = np.geomspace(10, 1e4, 30)
    Wk = host["Wk"]
    for names, win in ((("nfw",) * 4, (Wk,) * 4), (("y",) * 4, (1.,) * 4)):
        cv = cov(ells, *names, windows=win)
        _, bnd = _model_ref(order, host, names, ells, ells, win)
        _assert_bound("symmetric", cv, cv.T, bnd)
    if order == 3:
        full = cov(ells, "nfw", "y", windows=(Wk, 1., Wk, Wk))
        try:
            h._TRISPEC_3H_WS_BUDGET = 1
            one = cov(ells, "nfw", "y", windows=(Wk, 1., Wk, Wk))
        finally:
            del h._TRISPEC_3H_WS_BUDGET
        assert np.array_equal(full.view(np.int64), one.view(np.int64))


@pytest.mark.gpu
@pytest.mark.parametrize("order", [3, 4])
def test_api_defaults_and_rejections(model, order):
    h, host = model
    tri = getattr(h, "get_trispectrum_%dhalo" % order)
    cov = getattr(h, "get_cl_cov_%dhalo" % order)
    ells = np.array([100.0, 1000.0])
    np.testing.assert_array_equal(cov(ells, "nfw"), cov(ells, "nfw", "nfw", "nfw", "nfw", ells2=ells))
    np.testing.assert_array_equal(tri([0.1, 1.0], name="y", name3="nfw"),
                                  tri([0.1, 1.0], [0.1, 1.0], "y", "y", "nfw", "nfw"))
    with pytest.raises(ValueError, match="HOD"):
        cov(ells, "g")
    with pytest.raises(ValueError, match="HOD"):
        tri([0.1], name="nfw", name4="g")
    with pytest.raises(ValueError, match="no matter or pressure profile"):
        tri([0.1], name="nope")
    for bad in ([0.0, 1.0], [np.inf], [-3.0], []):
        with pytest.raises(ValueError, match="positive finite"):
            cov(bad)
        with pytest.raises(ValueError, match="positive finite"):
            tri([0.1], ks2=bad)
    for fsky in (0.0, 1.5):
        with pytest.raises(ValueError, match="fsky"):
            cov(ells, fsky=fsky)
    with pytest.raises(ValueError, match="four entries"):
        cov(ells, windows=(1., 1., 1.))
    ks = h._ks64
    try:
        h._ks64 = ks[::-1].copy()
        with pytest.raises(ValueError, match="strictly increasing"):
            tri([0.1])
    finally:
        h._ks64 = ks
    try:
        h._zcomm = object()
        with pytest.raises(NotImplementedError):
            cov(ells)
    finally:
        h._zcomm = None
