"""K1, the profile transform (k_transform.cu), checked plan by plan against float64 host restatements of the same
operation on seeded synthetic inputs.

Phase 1 (`hmv_profile_tables`): every bin 1..jn of every halo's table against a host sine transform,
    u_j = step sum_n g_n sin(2 pi j n / N) / kt_j / mnorm * outscale,    g_n = x_n rho(x_n) inside the theta-cut,
at the kernel's own sample positions x_n = (n+1) xmax/nxs, with the trapezoid mass norm (half weights at n = 0 and
n = N-1), the sums by float64 np.fft.rfft and rho by a float64 numpy evaluation of amp t^gamma (1 + t^alpha)^-expo.
Each bin is held to |got - want| <= tau * B_j, B_j = step sum_n |g_n| / kt_j / |mnorm| * |outscale| (times
1 + sum_n w_n x_n |g_n| / |mnorm|, the condition number of the mass norm).  The per-halo record {inv, u_1, bin
count, 0} is checked exactly: the bin count against the restated rule, u_1 bit for bit against bin 1, inv to within
one rounding of r_s(1+z)/kt_1, and the guard bin jn+1 must be 0.
Phase 2 (`hmv_profile_expand`, `hmv_profile_transform`): the cube against the host np.interp expansion of the
kernel's own tables in its coordinate t = k inv (left = u_1, right = 0): values below bin 1 must be u_1 and values
above bin J must be 0 bit for bit, interpolated ones within a fraction of the row's max|u|; the fused kernel must equal
tables + expand bit for bit.  The samples path (`hmv_profile_transform_samples`) has no table entry point, so its cube
is held to the host expansion of the host tables, with the bound B interpolated the same way.

`_k1_plans` restates the kernel's launch decisions (bin counts, chunks, direct or two-stage sine sums, the direct
form's tile split, phase 2's staging, block classes and rotation, the queue), and every case asserts the plans it exists
for; `test_plan_union` checks on the host that together the cases take every plan in `ALL_PLANS`.

Largest error-to-bound ratios measured on one B200 (1000 W power limit); each tolerance keeps about 10x headroom and
stays more than six orders of magnitude below the effect of the faults these tests exist for (a trapezoid end weight
on the wrong sample, a later chunk that overwrites instead of adding, a dropped bin tile of either form, a conjugated
twiddle, a bin count without max(ks), a misread log table: 5e-5 to 10; a misclassified block or a tail that reads the
wrong staged row: a value where 0 is required, or 3.5e-4 of max|u|):

    phase 1, direct form (three-term sine recurrence re-seeded every 704-sample chunk): 8.0e-14 (tables), 6.7e-14
    (samples path) -> TAU_DIRECT = 1e-12;  the GNFW halos with t^alpha ~ 1e+-200 reach 1.7e-14;
    phase 1, two-stage form (exact twiddles): 5.2e-16 (tables), 2.8e-16 (samples path) -> TAU_TWO = 1.5e-14;
    phase 2 interpolation against np.interp: 2.8e-16 of the row's max|u| -> TOL_EXPAND = 3e-15.
The whole file runs in about 6 s and allocates 0.6 GB of device memory (the workspace of the nxs = 24000 case
holds 192 x 2 ring slots of 16 x 12004 doubles).

Also here: NaN in the cube padding [nk, ldk) and in guards around the cube must survive; every launch is repeated and
must be bit-identical; a workspace and a table array pre-filled with NaN must give the same output bits as zero-filled
ones (nothing stale is read: the ring slot of a group keeps the previous item's bins above jn+1); and with many more
items than SMs the cube must not depend on the queue order (HMV_K1_TAIL unset, 1 and -1)."""
import ctypes as C

import numpy as np
import pytest

TAU_DIRECT = 1e-12      # phase 1, direct form
TAU_TWO = 1.5e-14       # phase 1, two-stage form
TOL_EXPAND = 3e-15      # phase 2 against np.interp, as a fraction of the row's max|u|
NAN_BITS = np.array([np.nan]).view(np.int64)[0]
GUARD = 64
HB, NCH, TS_P, GS_DOUBLES, MAXCTA = 16, 704, 40, 11264, 192     # k_transform.cu: WS_HB, NCH_MMA, TS_P, WS_GS_DOUBLES
NSM_B200 = 148

OBSERVED = {}           # largest error-to-bound ratio seen per comparison in this session

ALL_PLANS = {
    "direct", "direct_ts_available", "two_stage_R1", "two_stage_R2", "two_stage_R3",   # sine-sum forms
    "idle_warps", "nt1", "nt2", "nt3", "nt4", "split_3_2", "jn_partial_tile",          # direct form's tile split
    "chunks_2", "chunks_3", "last_chunk_ragged",                                       # multi-chunk profiles
    "staged16", "staged_rpp<16", "unstaged",                                           # phase 2 table reads
    "cls_hold", "cls_zero", "cls_interior", "cls_mixed", "cls_rows_differ", "cls_mixed_at_J",
    "rotation", "partial_block", "odd_nk", "odd_nk_later_pass", "unsorted",
    "grid_nitems", "ring_reuse", "cmax_over_xmax",
}


# ------------------------------------------------------------------------------------------------- host restatement
def _geom(xmax, nxs):
    """dx, step and kt_1 exactly as profile_transform_impl computes them."""
    dx = xmax / nxs
    step = (xmax - 1.0 * dx) / nxs
    kt1 = (1.0 * (1.0 / (nxs * step))) * 2.0 * np.pi
    return dx, step, kt1


def _k1_plans(c, nsm=NSM_B200):
    """The launch decisions of profile_transform_ws_kernel (k_transform.cu restated) for case c: (plans, jn[z, mass
    group], form[z, mass group] in {"direct", "two"}).  A mass group is 16 consecutive halos of one redshift."""
    N, J = c["nxs"], c["nxs"] // 2
    dx, _, kt1 = _geom(c["xmax"], N)
    zs, rs, cmax, ks = c["zs"], c["rs"], c["cmax"], c["ks"]
    nz, nm = rs.shape
    nmg = -(-nm // HB)
    kmax = max(c["hint"], float(ks.max()))
    Q = N // TS_P if (N % TS_P == 0 and N // TS_P >= 16) else 0
    QT = (Q + 7) // 8
    nk = ks.size
    npair, nwhole = nk >> 1, (nk >> 1) >> 7
    nblk = (npair + 127) >> 7
    srt = bool(np.all(ks[:-1] <= ks[1:]))
    inv = rs * (1.0 + zs[:, None]) / kt1
    plans, jn, form = set(), np.zeros((nz, nmg), dtype=np.int64), np.empty((nz, nmg), dtype=object)
    if (cmax >= c["xmax"]).any():
        plans.add("cmax_over_xmax")
    for z in range(nz):
        for mg in range(nmg):
            m0, m1 = mg * HB, min(nm, mg * HB + HB)
            amax = max(rs[z, m] * (1.0 + zs[z]) for m in range(m0, m1))
            n = int(min(J, np.floor(kmax * amax / kt1) + 2.0))              # bin_count_kernel
            jn[z, mg] = n
            cmx = cmax[z, m0:m1].max()
            nb = int(min(N, np.floor(cmx / dx) + 2.0)) if cmx > 0 else 0
            single = 0 < nb <= NCH
            ts_k = (-(-nb // TS_P) + 3) >> 2
            ts_r = ((n // Q + 1) + 7) >> 3 if Q else 0
            two = False
            if single and Q and ts_k <= 5 and ts_r <= 3:
                direct = 2 * ((nb + 3) >> 2) * ((n + 7) >> 3)
                staged = HB * QT * (2 * 5 * ts_k + 4 * 5 * ts_r)
                two = 5 * staged < 4 * direct
                if not two:
                    plans.add("direct_ts_available")
            form[z, mg] = "two" if two else "direct"
            if two:
                plans.add("two_stage_R%d" % ts_r)
            else:
                plans.add("direct")
                ntile = (n + 7) >> 3
                if ntile < 8:
                    plans.add("idle_warps")
                if n % 8:
                    plans.add("jn_partial_tile")
                for w in range(8):                   # tiles split over the warps, passes of <= 4 equal tiles
                    rem = ntile // 8 + (w < ntile % 8)
                    split = []
                    for passes in range((rem + 3) >> 2, 0, -1):
                        split.append((rem + passes - 1) // passes)
                        rem -= split[-1]
                    plans.update("nt%d" % t for t in split)
                    if split == [3, 2]:
                        plans.add("split_3_2")
            if nb > NCH:
                nch = -(-nb // NCH)
                plans.add("chunks_%d" % nch)
                if (nb - NCH * (nch - 1)) % 4:
                    plans.add("last_chunk_ragged")
            # phase 2
            tw = (n + 3) & ~1
            staged = tw <= GS_DOUBLES
            rpp = min(HB, GS_DOUBLES // tw) if staged else HB
            plans.add(("staged16" if rpp == HB else "staged_rpp<16") if staged else "unstaged")
            iv = inv[z, m0:m1]
            if nk & 1:
                plans.add("odd_nk")
                tl = ks[-1] * iv[rpp:]
                if ((tl >= 1.0) & (tl <= J)).any():
                    plans.add("odd_nk_later_pass")        # the tail interpolates a row of a later staging pass
            if nblk > nwhole:
                plans.add("partial_block")
            if not srt:
                plans.add("unsorted")
                continue
            for b in range(nwhole):
                tf, tl = ks[256 * b] * iv, ks[256 * b + 255] * iv
                cls = np.where(tl < 1.0, 0, np.where(tf > J, 1, np.where((tf >= 1.0) & (tl <= J), 2, 3)))
                plans.update(("cls_hold", "cls_zero", "cls_interior", "cls_mixed")[k] for k in set(cls.tolist()))
                if len(set(cls.tolist())) > 1:
                    plans.add("cls_rows_differ")
                if ((tf >= 1.0) & (tl > J) & (tl <= J + 1)).any():
                    plans.add("cls_mixed_at_J")           # an interior test with tl <= J + 1 would take it
            rot = sum(1 for b in range(nwhole) if ks[256 * b + 255] * iv.max() < 1.0)
            if 0 < rot < nblk:
                plans.add("rotation")
    nitems = nz * nmg
    grid = nitems if nitems < nsm else min(nsm, MAXCTA)
    if nitems < nsm:
        plans.add("grid_nitems")
    if nitems > 2 * grid:
        plans.add("ring_reuse")
    return plans, jn, form


def _case(name, nxs, zs, nm, jns, cmxs, nk, seed, xmax=20.0, span=1e-3, order="sorted", hint="zero", norm=1,
          oscale=True, gamma=0.0, samples=False, spread=0.3, extreme=False, plans=()):
    """A synthetic case.  jns[z][mg] is the bin count the kernel must give mass group mg of redshift z (J or more: the
    cap), cmxs[z][mg] the largest theta-cut of the group; r_s is chosen from the bin count and the k range."""
    rng = np.random.default_rng(seed)
    zs = np.asarray(zs, dtype=np.float64)
    nz, nmg, J = zs.size, -(-nm // HB), nxs // 2
    _, _, kt1 = _geom(xmax, nxs)
    ks = np.geomspace(10.0 * span, 10.0, nk) if nk > 1 else np.array([10.0])
    if order == "shuffled":
        ks = rng.permutation(ks)
    kmax = 10.0 * (1.3 if hint == "above" else 1.0)
    rs, cmax = np.zeros((nz, nm)), np.zeros((nz, nm))
    for z in range(nz):
        for mg in range(nmg):
            m0, m1 = mg * HB, min(nm, mg * HB + HB)
            a = ((jns[z][mg] - 1.5) if jns[z][mg] < J else 1.5 * J) * kt1 / kmax
            f = rng.uniform(spread, 1.0, m1 - m0)
            f[rng.integers(m1 - m0)] = 1.0
            rs[z, m0:m1] = a * f / (1.0 + zs[z])
            cm = rng.uniform(0.3, 1.0, m1 - m0) * cmxs[z][mg]
            cm[rng.integers(m1 - m0)] = cmxs[z][mg]
            cmax[z, m0:m1] = cm
    c = dict(name=name, nxs=nxs, xmax=xmax, zs=zs, rs=rs, cmax=cmax, ks=ks, norm=norm, gamma=gamma,
             hint={"zero": 0.0, "equal": float(ks.max()), "above": kmax}[hint], plans=set(plans))
    c["oscale"] = rng.uniform(-2.0, 3.0, (nz, nm)) if oscale else None
    if samples:
        c["rho"] = rng.uniform(-0.3, 1.2, (nz, nm, nxs))            # signed samples, mass norm of order sum|g|
    else:
        c["gnfw"] = dict(xc=rng.uniform(0.05, 1.0, (nz, nm)), alpha=rng.uniform(0.8, 2.0, (nz, nm)),
                         expo=rng.uniform(1.5, 4.0, (nz, nm)), amp=rng.uniform(0.5, 2.0, (nz, nm)))
        if extreme:      # t^alpha up to ~1e+200 (xc << x) and down to ~1e-200 (t << 1)
            g = c["gnfw"]
            lo = np.arange(nm) % 2 == 0
            g["xc"] = np.where(lo, rng.uniform(0.008, 0.012, (nz, nm)), rng.uniform(10.0, 30.0, (nz, nm)))
            g["alpha"] = np.where(lo, rng.uniform(55.0, 62.0, (nz, nm)), rng.uniform(60.0, 70.0, (nz, nm)))
            g["expo"] = np.where(lo, rng.uniform(0.04, 0.07, (nz, nm)), rng.uniform(0.5, 1.0, (nz, nm)))
    return c


def _edge_row(c, z, m, b):
    """Move halo (z, m) so that the last wavenumber of whole block b sits at t = J + 0.5 (a block that ends just past
    bin J); the halo's group must already have the capped bin count."""
    J = c["nxs"] // 2
    _, _, kt1 = _geom(c["xmax"], c["nxs"])
    c["rs"][z, m] = (J + 0.5) / c["ks"][256 * b + 255] * kt1 / (1.0 + c["zs"][z])
    return c


def _cases():
    C_ = []
    # direct form only (700 = 40 x 17.5: no two-stage form): 1 tile (7 idle warps), 2 tiles, 33 tiles (3 + 2 split),
    # 13 tiles, the capped count J = 350 (44 tiles, two passes), jn % 8 != 0; nm = 37 (last item 5 halos)
    C_.append(_case("direct", 700, [0.0, 1.2], 37, [[2, 13, 263], [100, 999, 41]], [[9.0, 14.0, 5.0]] * 2, 257,
                    seed=1, span=0.1, gamma=-0.3, plans={"direct", "idle_warps", "nt1", "nt2", "nt3", "nt4",
                                                         "split_3_2", "jn_partial_tile", "staged16", "odd_nk",
                                                         "cls_hold", "cls_interior", "cls_mixed", "grid_nitems"}))
    # two-stage form at R = 1, 2, 3 and just below its threshold (jn = 56: direct, though available); theta-cuts past
    # xmax (the trapezoid end weight at n = N-1); sorted 10000-point axis over six decades: leading pure hold-u_1
    # blocks (rotation), blocks past bin J of the capped group, rows of one block in different classes
    C_.append(_case("two_stage", 640, [0.3, 2.0], 48, [[56, 57, 200], [127, 300, 999]], [[25.0, 21.0, 22.0],
                                                                                           [23.0, 30.0, 20.5]],
                    10000, seed=2, span=1e-6, hint="equal", gamma=0.2, spread=0.1,
                    plans={"direct_ts_available", "two_stage_R1", "two_stage_R2", "two_stage_R3", "cmax_over_xmax",
                           "rotation", "cls_hold", "cls_zero", "cls_interior", "cls_mixed", "cls_rows_differ"}))
    # several sample chunks (odd N = 3001: no two-stage form, and u_J != 0): 2 chunks with a last chunk of 299, 3 with
    # one of 2, 5 (cut past xmax); jn = 1000 and the capped 1500 stage fewer than 16 rows per pass; one block ends just
    # past bin J; kmax hint above max(ks)
    dx = 20.0 / 3001
    c = _case("multichunk", 3001, [0.1, 0.9], 17, [[1000, 40], [2000, 150]],
              [[1001.5 * dx, 25.0], [1408.5 * dx, 3.0]], 512, seed=3, span=1e-2, hint="above", norm=0,
              plans={"chunks_2", "chunks_3", "last_chunk_ragged", "staged_rpp<16", "cls_mixed_at_J",
                     "cmax_over_xmax"})
    C_.append(_edge_row(c, 1, 3, 0))
    # odd nk with 14 staged rows per pass (jn = 790): the last wavenumber of rows 14 and 15 is interpolated from the
    # second pass's staged rows
    C_.append(_case("odd_tail", 1600, [0.6], 16, [[790]], [[6.0]], 511, seed=11, gamma=0.1,
                    plans={"staged_rpp<16", "odd_nk", "odd_nk_later_pass", "partial_block"}))
    # rows longer than the sample buffer (jn >= 11263: table rows read from L2), two-stage R = 3 at jn >= 9600, and
    # jn = 9000 (two-stage R = 2, one staged row per pass); nm = 40: last item of 8 halos
    C_.append(_case("unstaged", 24000, [0.5], 40, [[11263, 999999, 9000]], [[0.55, 0.5, 0.3]], 256, seed=4,
                    gamma=-0.5, plans={"unstaged", "staged_rpp<16", "two_stage_R3", "two_stage_R2"}))
    # GNFW at t^alpha ~ 1e+-200, nm = 15, nk = 2, no outscale
    C_.append(_case("gnfw_extreme", 640, [0.2, 1.0], 15, [[200], [40]], [[30.0], [8.0]], 2, seed=5, gamma=0.4,
                    extreme=True, oscale=False, hint="above", plans={"two_stage_R2", "direct", "partial_block"}))
    return C_


def _samples_cases():
    return [
        _case("samples_norm", 640, [0.1, 0.5, 1.1, 2.3], 16, [[30], [100], [250], [300]], [[22.0], [12.0], [30.0], [7.0]],
              4001, seed=6, oscale=False, samples=True,
              plans={"direct", "two_stage_R1", "two_stage_R2", "two_stage_R3", "odd_nk", "cls_hold"}),
        _case("samples_chunks", 3001, [0.7], 1, [[400]], [[26.0]], 255, seed=7, order="shuffled", hint="above",
              norm=0, samples=True, plans={"direct", "unsorted", "odd_nk"}),
        _case("samples_one_k", 1000, [0.4], 16, [[300]], [[12.0]], 1, seed=8, hint="above", samples=True,
              plans={"odd_nk"}),
    ]


def _queue_case():
    """Many more items than SMs (40 x 16 = 640), bin counts from 2 to J over the items: ring slots are reused."""
    rng = np.random.default_rng(9)
    jns = [list(rng.integers(2, 340, 16)) for _ in range(40)]
    cmxs = [list(rng.uniform(2.0, 25.0, 16)) for _ in range(40)]
    return _case("queue", 640, np.linspace(0.0, 3.0, 40), 256, jns, cmxs, 255, seed=10, hint="zero",
                 plans={"ring_reuse", "direct", "two_stage_R1", "two_stage_R2", "two_stage_R3"})


# ------------------------------------------------------------------------------------------------- host references
def _samples(c):
    """x_n and rho(x_n) [nz, nm, N] (float64 GNFW, or the case's samples)."""
    N = c["nxs"]
    dx, _, _ = _geom(c["xmax"], N)
    x = (np.arange(N) + 1.0) * dx
    if "rho" in c:
        return x, c["rho"]
    g = c["gnfw"]
    lt = np.log(x)[None, None, :] - np.log(g["xc"])[..., None]
    with np.errstate(over="ignore"):
        y = c["gamma"] * lt - g["expo"][..., None] * np.log1p(np.exp(g["alpha"][..., None] * lt))
    return x, g["amp"][..., None] * np.exp(y)


def _host_tables(c):
    """(want, bound) [nz, nm, J+1]: u_j and B_j of every halo (bin 0 unused)."""
    N, J = c["nxs"], c["nxs"] // 2
    dx, step, kt1 = _geom(c["xmax"], N)
    x, rho = _samples(c)
    g = np.where(x[None, None, :] <= c["cmax"][..., None], x[None, None, :] * rho, 0.0)
    w = np.full(N, dx)
    w[0] = w[-1] = 0.5 * dx
    if c["norm"]:
        mn = (w * x * g).sum(axis=-1)
        cond = 1.0 + (w * x * np.abs(g)).sum(axis=-1) / np.abs(mn)
    else:
        mn, cond = np.ones(g.shape[:2]), np.ones(g.shape[:2])
    os_ = c["oscale"] if c["oscale"] is not None else np.ones(g.shape[:2])
    S = -np.fft.rfft(g, axis=-1).imag[..., :J + 1]
    j = np.arange(J + 1, dtype=np.float64)
    with np.errstate(divide="ignore"):
        rkt = np.where(j > 0, 1.0 / (j * kt1), 0.0)
    fac = (step / mn * os_)[..., None]
    want = S * rkt * fac
    bound = np.abs(g).sum(axis=-1)[..., None] * rkt * np.abs(fac) * cond[..., None]
    return want, bound


def _expand(tab, inv, u1, jn, ks, J):
    """np.interp expansion of one halo's bins 1..jn onto ks in t = k inv (fft.py:102-107)."""
    t = ks * inv
    assert np.all((t <= jn) | (t > J)), "a wavenumber needs a bin the transform did not write"
    return t, np.interp(t, np.arange(1, jn + 1, dtype=np.float64), tab[1:jn + 1], left=u1, right=0.0)


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


# ------------------------------------------------------------------------------------------------- device side
@pytest.fixture(scope="module")
def env():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    from hmvec_b200 import _capi as capi
    torch.cuda.reset_peak_memory_stats()
    yield torch, capi
    print("\nK1 largest error-to-bound ratios: %s; peak device memory %.2f GB" % (
        ", ".join("%s %.2g" % kv for kv in sorted(OBSERVED.items())), torch.cuda.max_memory_allocated() / 1e9))


def _dev(torch, x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def _vp(t, off=0):
    return C.c_void_p(t.data_ptr() + 8 * off)


class Cube(object):
    """[nz][nm][ldk] output with ldk > nk, between NaN guards; the guards and the padding [nk, ldk) must stay NaN."""

    def __init__(self, torch, nz, nm, nk):
        self.shape, self.nk, self.ldk = (nz, nm), nk, (nk // 16 + 1) * 16
        self.buf = torch.full((2 * GUARD + nz * nm * self.ldk,), float("nan"), dtype=torch.float64, device="cuda")
        self.ptr = _vp(self.buf, GUARD)

    def host(self):
        b = self.buf.cpu().numpy()
        bits = b.view(np.int64)
        assert np.all(bits[:GUARD] == NAN_BITS) and np.all(bits[-GUARD:] == NAN_BITS), "a guard around the cube was written"
        cube = b[GUARD:-GUARD].reshape(self.shape + (self.ldk,))
        assert np.all(cube[..., self.nk:].view(np.int64) == NAN_BITS), "the padding [nk, ldk) was written"
        return cube[..., :self.nk]


class Dev(object):
    """The case's inputs on the device."""

    def __init__(self, torch, c):
        self.zs, self.ks, self.rs, self.cmax = (_dev(torch, c[k]) for k in ("zs", "ks", "rs", "cmax"))
        self.os = _dev(torch, c["oscale"]) if c["oscale"] is not None else None
        if "gnfw" in c:
            self.g = [_dev(torch, c["gnfw"][k]) for k in ("xc", "alpha", "expo", "amp")]
        else:
            self.rho = _dev(torch, c["rho"])


def _ws(torch, capi, c, fill):
    nz, nm = c["rs"].shape
    return torch.full((int(capi.lib.hmv_profile_transform_ws_doubles(nz, nm, c["nxs"])),), fill, dtype=torch.float64,
                      device="cuda")


def _tables(env, c, d, fill):
    """hmv_profile_tables into a table array pre-filled with `fill`; returns (tab tensor, rows, meta)."""
    torch, capi = env
    L, p = capi.lib, capi.ptr
    nz, nm = c["rs"].shape
    N, nk = c["nxs"], c["ks"].size
    tab = torch.full((int(L.hmv_profile_table_doubles(nz, nm, N)),), fill, dtype=torch.float64, device="cuda")
    ws = _ws(torch, capi, c, fill)
    capi.check(L.hmv_profile_tables(nz, nm, nk, p(d.zs), p(d.ks), c["hint"], p(d.rs), p(d.cmax), *(p(a) for a in d.g),
                                    p(d.os), c["gamma"], c["xmax"], N, c["norm"], p(ws), p(tab), capi.stream()),
               "hmv_profile_tables")
    JS, nmp = int(L.hmv_profile_table_stride(N)), -(-nm // HB) * HB
    h = tab.cpu().numpy()
    rows = h[:nz * nmp * JS].reshape(nz, nmp, JS)[:, :nm]
    meta = h[nz * nmp * JS:nz * nmp * (JS + 4)].reshape(nz, nmp, 4)[:, :nm]
    del ws
    return tab, rows, meta


def _expand_dev(env, c, d, tab, fill):
    torch, capi = env
    L, p = capi.lib, capi.ptr
    nz, nm = c["rs"].shape
    out, ws = Cube(torch, nz, nm, c["ks"].size), _ws(torch, capi, c, fill)
    capi.check(L.hmv_profile_expand(nz, nm, c["ks"].size, out.ldk, p(d.zs), p(d.ks), c["hint"], p(d.rs), c["xmax"],
                                    c["nxs"], p(ws), p(tab), out.ptr, capi.stream()), "hmv_profile_expand")
    return out.host()


def _fused_dev(env, c, d, fill, twice=False):
    """hmv_profile_transform or hmv_profile_transform_samples with a workspace pre-filled with `fill`."""
    torch, capi = env
    L, p = capi.lib, capi.ptr
    nz, nm = c["rs"].shape
    nk = c["ks"].size
    out, ws = Cube(torch, nz, nm, nk), _ws(torch, capi, c, fill)

    def launch():
        if "gnfw" in c:
            rc = L.hmv_profile_transform(nz, nm, nk, out.ldk, p(d.zs), p(d.ks), c["hint"], p(d.rs), p(d.cmax),
                                         *(p(a) for a in d.g), p(d.os), c["gamma"], c["xmax"], c["nxs"], c["norm"],
                                         p(ws), out.ptr, capi.stream())
        else:
            rc = L.hmv_profile_transform_samples(nz, nm, nk, out.ldk, p(d.zs), p(d.ks), c["hint"], p(d.rs), p(d.cmax),
                                                 p(d.rho), p(d.os), c["xmax"], c["nxs"], c["norm"], p(ws), out.ptr,
                                                 capi.stream())
        capi.check(rc, "hmv_profile_transform")
    launch()
    torch.cuda.synchronize()
    if twice:
        first = out.buf.clone()
        launch()
        torch.cuda.synchronize()
        assert torch.equal(first.view(torch.int64), out.buf.view(torch.int64)), "second launch differs"
    return out.host()


def _same_bits(a, b, what):
    assert np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64)), what


# ------------------------------------------------------------------------------------------------- checks
def _check_tables(c, rows, meta, jn, form):
    """Phase 1: bins 1..jn against the host transform, and the per-halo record."""
    nz, nm = c["rs"].shape
    J = c["nxs"] // 2
    _, _, kt1 = _geom(c["xmax"], c["nxs"])
    want, bound = _host_tables(c)
    inv = c["rs"] * (1.0 + c["zs"][:, None]) / kt1
    jm = jn[:, np.arange(nm) // HB]                          # bin count of every halo's group
    assert np.array_equal(meta[..., 2], jm.astype(np.float64)), "bin count of the table record"
    assert np.all(meta[..., 3] == 0.0)
    _same_bits(meta[..., 1], rows[..., 1], "u_1 of the record is bin 1")
    assert np.all(np.abs(meta[..., 0] - inv) <= np.spacing(inv)), "k -> bin factor of the record"
    assert np.all(np.take_along_axis(rows, (jm + 1)[..., None], axis=-1) == 0.0), "guard bin jn+1"
    fm = form[:, np.arange(nm) // HB]
    for kind, tau in (("direct", TAU_DIRECT), ("two", TAU_TWO)):
        sel = (fm == kind)[..., None] & (np.arange(J + 1) >= 1) & (np.arange(J + 1) <= jm[..., None])
        if sel.any():
            _assert_bound("tables_" + kind, "%s tables (%s form)" % (c["name"], kind), rows[..., :J + 1][sel],
                          want[sel], bound[sel], tau)


def _check_cube(c, cube, rows, meta):
    """Phase 2: the cube against the np.interp expansion of the tables; hold and zero values bit for bit."""
    nz, nm = c["rs"].shape
    J, ks = c["nxs"] // 2, c["ks"]
    worst = 0.0
    for z in range(nz):
        for m in range(nm):
            inv, u1, jn = meta[z, m, 0], meta[z, m, 1], int(meta[z, m, 2])
            t, want = _expand(rows[z, m], inv, u1, jn, ks, J)
            got = cube[z, m]
            _same_bits(got[t < 1.0], np.full(int((t < 1.0).sum()), u1), "%s: hold u_1 below bin 1" % c["name"])
            assert np.all(got[t > J] == 0.0), "%s: zero above bin J" % c["name"]
            mid = (t >= 1.0) & (t <= J)
            if mid.any():
                scale = np.abs(rows[z, m, 1:jn + 1]).max()
                worst = max(worst, float(np.max(np.abs(got[mid] - want[mid]))) / scale)
    _record("expand", worst)
    assert worst <= TOL_EXPAND, "%s: cube vs np.interp of the tables %.3g of max|u|" % (c["name"], worst)


def _check_samples_cube(c, cube, form, jn):
    """The samples path: the cube against the expansion of the host tables, bound interpolated alike."""
    nz, nm = c["rs"].shape
    J, ks = c["nxs"] // 2, c["ks"]
    _, _, kt1 = _geom(c["xmax"], c["nxs"])
    want, bound = _host_tables(c)
    for z in range(nz):
        for m in range(nm):
            n = int(jn[z, m // HB])
            tau = TAU_DIRECT if form[z, m // HB] == "direct" else TAU_TWO
            inv = c["rs"][z, m] * (1.0 + c["zs"][z]) / kt1
            t, w = _expand(want[z, m], inv, want[z, m, 1], n, ks, J)
            _, b = _expand(bound[z, m], inv, bound[z, m, 1], n, ks, J)
            b = b + np.abs(want[z, m, 1:n + 1]).max() * TOL_EXPAND / tau
            _assert_bound("samples_" + form[z, m // HB], "%s z=%d m=%d" % (c["name"], z, m), cube[z, m], w, b, tau)


# ------------------------------------------------------------------------------------------------- tests
def test_plan_union():
    """Host only: every case takes the plans it is for, and together the cases take every plan of the kernel."""
    union = set()
    for c in _cases() + _samples_cases() + [_queue_case()]:
        plans, _, _ = _k1_plans(c)
        assert c["plans"] <= plans, (c["name"], c["plans"] - plans)
        union |= c["plans"]
    assert union == ALL_PLANS, (ALL_PLANS - union, union - ALL_PLANS)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in _cases()])
def test_transform_plans(env, name):
    """hmv_profile_tables against the host transform, hmv_profile_expand against np.interp of those tables,
    hmv_profile_transform == tables + expand bit for bit; NaN-filled workspace and tables give the same bits."""
    torch, _ = env
    c = next(c for c in _cases() if c["name"] == name)
    plans, jn, form = _k1_plans(c, torch.cuda.get_device_properties(0).multi_processor_count)
    assert c["plans"] <= plans, c["plans"] - plans
    d = Dev(torch, c)
    tab, rows, meta = _tables(env, c, d, 0.0)
    _check_tables(c, rows, meta, jn, form)
    tabn, rowsn, metan = _tables(env, c, d, float("nan"))
    _same_bits(metan, meta, "table record with a NaN-filled table array")
    jm = jn[:, np.arange(c["rs"].shape[1]) // HB][..., None]
    sel = (np.arange(rows.shape[-1]) >= 1) & (np.arange(rows.shape[-1]) <= jm + 1)
    _same_bits(rowsn[np.broadcast_to(sel, rows.shape)], rows[np.broadcast_to(sel, rows.shape)],
               "bins 1..jn+1 with a NaN-filled table array")
    cube = _expand_dev(env, c, d, tab, 0.0)
    _check_cube(c, cube, rows, meta)
    _same_bits(_expand_dev(env, c, d, tabn, float("nan")), cube, "expand of NaN-filled tables and workspace")
    del tabn
    _same_bits(_fused_dev(env, c, d, 0.0, twice=True), cube, "hmv_profile_transform vs tables + expand")
    _same_bits(_fused_dev(env, c, d, float("nan")), cube, "hmv_profile_transform with a NaN-filled workspace")


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in _samples_cases()])
def test_transform_samples_plans(env, name):
    """hmv_profile_transform_samples (caller-supplied signed samples) against the expansion of the host transform."""
    torch, _ = env
    c = next(c for c in _samples_cases() if c["name"] == name)
    plans, jn, form = _k1_plans(c, torch.cuda.get_device_properties(0).multi_processor_count)
    assert c["plans"] <= plans, c["plans"] - plans
    d = Dev(torch, c)
    cube = _fused_dev(env, c, d, 0.0, twice=True)
    _check_samples_cube(c, cube, form, jn)
    _same_bits(_fused_dev(env, c, d, float("nan")), cube, "NaN-filled workspace")


@pytest.mark.gpu
def test_transform_queue_order(env, monkeypatch):
    """640 items (over 2 per group of 148 SMs: ring slots reused) with bin counts 2..J: the tables against the host
    transform, the cube against them, and the cube bit for bit the same in every queue order (HMV_K1_TAIL is read on
    every launch: unset, 1 = one heavy-first redshift, -1 = heaviest and lightest alternating)."""
    torch, _ = env
    c = _queue_case()
    plans, jn, form = _k1_plans(c, torch.cuda.get_device_properties(0).multi_processor_count)
    assert c["plans"] <= plans, c["plans"] - plans
    assert jn.max() - jn.min() > 250
    d = Dev(torch, c)
    _, rows, meta = _tables(env, c, d, 0.0)
    _check_tables(c, rows, meta, jn, form)
    monkeypatch.delenv("HMV_K1_TAIL", raising=False)
    cube = _fused_dev(env, c, d, float("nan"), twice=True)
    _check_cube(c, cube, rows, meta)
    for tail in ("1", "-1"):
        monkeypatch.setenv("HMV_K1_TAIL", tail)
        _same_bits(_fused_dev(env, c, d, float("nan")), cube, "queue order HMV_K1_TAIL=%s" % tail)
