"""Time the non-Gaussian C_l covariances on the LARGE grid: the 1-halo term (hmv_cl_cov_1h, also on a 25-redshift slab),
its galaxy (HOD) legs (hmv_cl_cov_1h_tracers) and the 2-halo term (hmv_cl_cov_2h).

Cases: C_kk x C_kk (NFW, lensing window of a source at z = 2.5) and C_yy x C_yy (Battaglia pressure) at
ells = geomspace(10, 1e4, nl) on zs = linspace(0.01, 3, nz), ms = geomspace(2e10, 1e17, nm), ks = geomspace(1e-4, 100,
nk) (bench.py's grid), and C_kk on the slab zs[:25].  For each case it reports, from one run on one device:

  * the whole call from CUDA events over --reps launches after two warm-up launches (panels, contraction, reduction);
  * the panel kernel and the contraction separately, from torch.profiler over three further launches;
  * flop = 2 n1 n2 nz nm, the contraction's TFLOP/s and its ratio to hmv_bench_dmma measured in the same run;
  * a check of a seeded sample of (l, l') entries against a float64 host reduction over the same cubes;

with the card's name and power limit read in the same run.  2-halo cases: C_kk and C_yy autos (3 contracted blocks)
and the C_ky x C_ky cross (NFW, y, NFW, y: 8 blocks), zchunk as HaloModel.get_cl_cov_2halo picks it; flop = 2 nz nm
n1 n2 per block; the split into prep, panel, contraction and assembly kernels; a seeded sample of entries against a
float64 host evaluation (long-double Pbar prefix).  HOD cases: C_kg x C_kg (NFW and an HOD with ngal from 2e-3 to
5e-5 over z, NFW satellites, no central profile: one galaxy leg on each side, two segments of mass rows per redshift)
and C_kk x C_gg (both galaxy legs on one side: one segment), galaxy window a normalised Gaussian dN/dz; flop = 2 n1 n2
nz nm per segment.  Prints one JSON document (and writes it to --out).

    python tools/trispec_bench.py [--nz 200 --nm 2000 --nk 10000 --nl 1000 --reps 10 --cases TAG,... --out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:        # the numbers are still reported, without the card's settings
        return {"error": repr(e)}


class Case(object):
    """The ABI call of one covariance, with every input resident on the device."""

    def __init__(self, h, name, kind, windows, ells):
        from hmvec_b200 import _capi as capi
        self.capi, self.h = capi, h
        cube = (h.uk_profiles if kind == 0 else h.pk_profiles).device(name)
        self.cube, self.kind = cube, kind
        self.ells = ells
        zs = h.zs
        self.chis = np.asarray(h.comoving_radial_distance(zs), dtype=np.float64)
        self.H = np.asarray(h.h_of_z(zs), dtype=np.float64)
        W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), zs.shape) for w in windows], axis=0)
        self.pref = self.H ** 3 * W / self.chis ** 6 / (4 * np.pi)
        self.d = {k: h._dev(v) for k, v in dict(ells=ells, chis=self.chis, pref=self.pref).items()}
        n = ells.size
        self.ws = h._empty(int(capi.lib.hmv_cl_cov_1h_ws_doubles(h._nz, h._nm, n, n)))
        self.out = h._empty(n, n)
        self.u_h = (C.c_void_p * 4)(*([cube.data_ptr()] * 4))
        self.k_h = (C.c_int * 4)(*([kind] * 4))

    def launch(self):
        h, p, d, n = self.h, self.capi.ptr, self.d, self.ells.size
        self.capi.check(self.capi.lib.hmv_cl_cov_1h(h._nz, h._nm, h._nk, h._ldk, p(h._ks_d), p(h._ms_d), p(h._nzm_d),
                                                    h._rho_m0, self.u_h, self.k_h, n, p(d["ells"]), n, p(d["ells"]),
                                                    p(h._zs_d), p(d["chis"]), p(d["pref"]), p(self.ws), p(self.out),
                                                    self.capi.stream()), "hmv_cl_cov_1h")

    def check_sample(self, rng, npairs=8):
        """Max |got - want| / sum|terms| over seeded (l, l') entries, want from a float64 host reduction over the cube
        columns that the entries need (gathered on the device, reduced on the host)."""
        import torch
        h = self.h
        got = self.out.cpu().numpy()
        ks, ms, nzm = h._ks64, h.ms, h.nzm
        wm = 0.5 * (ms[np.minimum(np.arange(ms.size) + 1, ms.size - 1)] - ms[np.maximum(np.arange(ms.size) - 1, 0)])
        zs = h.zs
        zw = 0.5 * (zs[np.minimum(np.arange(zs.size) + 1, zs.size - 1)] - zs[np.maximum(np.arange(zs.size) - 1, 0)]) \
            if zs.size > 1 else np.ones(1)
        a = ms / h._rho_m0 if self.kind == 0 else np.ones(ms.size)
        zi = torch.arange(zs.size, device=self.cube.device)

        def leg(ell):                     # t(z, m) at k = (l + 1/2)/chi_z, linear in k, clamped
            k = np.clip((ell + 0.5) / self.chis, ks[0], ks[-1])
            j = np.clip(np.searchsorted(ks, k, side="right") - 1, 0, ks.size - 2)
            f = (k - ks[j]) / (ks[j + 1] - ks[j])
            jd = torch.as_tensor(j, device=self.cube.device)
            u0 = self.cube[zi, :, jd].cpu().numpy()
            u1 = self.cube[zi, :, jd + 1].cpu().numpy()
            return a[None, :] * (u0 + f[:, None] * (u1 - u0))

        worst = 0.0
        for _ in range(npairs):
            i, j = rng.integers(0, self.ells.size, 2)
            ti, tj = leg(self.ells[i]), leg(self.ells[j])
            c = (zw * self.pref)[:, None] * wm[None, :] * nzm
            want = np.sum(c * ti ** 2 * tj ** 2)
            bound = np.sum(np.abs(c) * ti ** 2 * tj ** 2)
            worst = max(worst, abs(got[i, j] - want) / bound if bound > 0 else abs(got[i, j] - want))
        return worst


class CaseHod(object):
    """The ABI call of one 1-halo covariance with galaxy legs (hmv_cl_cov_1h_tracers), inputs resident on the device."""

    def __init__(self, h, names, windows, ells):
        from hmvec_b200 import _capi as capi
        self.capi, self.h, self.names, self.ells = capi, h, names, ells
        self.kinds = [0 if n in h.uk_profiles else 1 for n in names]
        self.legs = (capi.Tracer * 4)(*[h._tracer(n, k)[0] for n, k in zip(names, self.kinds)])
        zs = h.zs
        self.chis = np.asarray(h.comoving_radial_distance(zs), dtype=np.float64)
        H = np.asarray(h.h_of_z(zs), dtype=np.float64)
        W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), zs.shape) for w in windows], axis=0)
        self.pref = H ** 3 * W / self.chis ** 6 / (4 * np.pi)
        self.d = {k: h._dev(v) for k, v in dict(ells=ells, chis=self.chis, pref=self.pref).items()}
        n = ells.size
        self.ws = h._empty(int(capi.lib.hmv_cl_cov_1h_tracers_ws_doubles(h._nz, h._nm, n, n, self.legs)))
        self.out = h._empty(n, n)
        self.nseg = 2 if 1 in self.kinds[:2] and 1 in self.kinds[2:] else 1

    def launch(self):
        h, p, d, n = self.h, self.capi.ptr, self.d, self.ells.size
        self.capi.check(self.capi.lib.hmv_cl_cov_1h_tracers(h._nz, h._nm, h._nk, h._ldk, p(h._ks_d), p(h._ms_d),
                                                            p(h._nzm_d), h._rho_m0, self.legs, n, p(d["ells"]), n,
                                                            p(d["ells"]), p(h._zs_d), p(d["chis"]), p(d["pref"]),
                                                            p(self.ws), p(self.out), self.capi.stream()),
                        "hmv_cl_cov_1h_tracers")

    def check_sample(self, rng, npairs=8):
        """Max |got - want| / sum|terms| over seeded (l, l') entries: u_s of the NFW cube gathered on the device at the
        columns the entries need, t and <g g> formed on the host in float64 (u_c = 1)."""
        import torch
        h = self.h
        got = self.out.cpu().numpy()
        ks, ms, nzm, zs = h._ks64, h.ms, h.nzm, h.zs
        hod = h.hods[next(n for n, k in zip(self.names, self.kinds) if k == 1)]
        Nc, Ns, NcNs, NsNsm1, ig = hod["Nc"], hod["Ns"], hod["NcNs"], hod["NsNsm1"], 1.0 / hod["ngal"][:, None]
        wm = 0.5 * (ms[np.minimum(np.arange(ms.size) + 1, ms.size - 1)] - ms[np.maximum(np.arange(ms.size) - 1, 0)])
        zw = 0.5 * (zs[np.minimum(np.arange(zs.size) + 1, zs.size - 1)] - zs[np.maximum(np.arange(zs.size) - 1, 0)])
        cube = h.uk_profiles.device("nfw")
        zi = torch.arange(zs.size, device=cube.device)

        def us(ell):                       # u_s(z, m) at k = (l + 1/2)/chi_z, linear in k, clamped
            k = np.clip((ell + 0.5) / self.chis, ks[0], ks[-1])
            j = np.clip(np.searchsorted(ks, k, side="right") - 1, 0, ks.size - 2)
            f = (k - ks[j]) / (ks[j + 1] - ks[j])
            jd = torch.as_tensor(j, device=cube.device)
            u0, u1 = cube[zi, :, jd].cpu().numpy(), cube[zi, :, jd + 1].cpu().numpy()
            return u0 + f[:, None] * (u1 - u0)

        c = (zw * self.pref)[:, None] * wm[None, :] * nzm
        worst = 0.0
        for _ in range(npairs):
            i, j = rng.integers(0, self.ells.size, 2)
            u1, u2 = us(self.ells[i]), us(self.ells[j])
            tk1, tk2 = ms[None, :] / h._rho_m0 * u1, ms[None, :] / h._rho_m0 * u2
            if self.nseg == 2:             # kappa g x kappa g: t_k(k1) t_k(k2) <g g>(k1, k2)
                terms = [NsNsm1 * u1 * u2, NcNs * u2, NcNs * u1]
                terms = [tk1 * tk2 * ig ** 2 * t for t in terms]
            else:                          # kappa kappa x g g: t_k(k1)^2 <g g>(k2, k2)
                terms = [tk1 ** 2 * ig ** 2 * t for t in (NsNsm1 * u2 ** 2, 2 * NcNs * u2)]
            want = sum(np.sum(c * t) for t in terms)
            bound = sum(np.sum(np.abs(c * t)) for t in terms)
            worst = max(worst, abs(got[i, j] - want) / bound if bound > 0 else abs(got[i, j] - want))
        return worst


class Case2h(object):
    """The ABI call of one 2-halo covariance, with every input resident on the device."""

    def __init__(self, h, names, windows, ells):
        from hmvec_b200 import _capi as capi
        self.capi, self.h, self.names, self.ells = capi, h, names, ells
        self.cubes, self.kinds = h._trispec_legs(names)
        zs = h.zs
        self.chis = np.asarray(h.comoving_radial_distance(zs), dtype=np.float64)
        H = np.asarray(h.h_of_z(zs), dtype=np.float64)
        W = np.prod([np.broadcast_to(np.asarray(w, dtype=np.float64), zs.shape) for w in windows], axis=0)
        self.pref = H ** 3 * W / self.chis ** 6 / (4 * np.pi)
        self.d = {k: h._dev(v) for k, v in dict(ells=ells, chis=self.chis, pref=self.pref).items()}
        n = ells.size
        self.u_h = (C.c_void_p * 4)(*[c.data_ptr() for c in self.cubes])
        self.k_h = (C.c_int * 4)(*self.kinds)
        size = lambda zc: capi.lib.hmv_cl_cov_2h_ws_doubles(h._nz, h._nm, h._nk, n, n, self.u_h, self.k_h, zc)
        self.zchunk = max([zc for zc in range(1, h._nz + 1) if size(zc) <= h._TRISPEC_2H_WS_BUDGET] or [1])
        self.ws = h._empty(int(size(self.zchunk)))
        self.out = h._empty(n, n)
        self.blocks = (1 if self.u_h[0] == self.u_h[1] and self.kinds[0] == self.kinds[1] else 2)
        nc = (1 if self.u_h[2] == self.u_h[3] and self.kinds[2] == self.kinds[3] else 2)
        self.blocks = self.blocks * nc + self.blocks + nc

    def launch(self):
        h, p, d, n = self.h, self.capi.ptr, self.d, self.ells.size
        self.capi.check(self.capi.lib.hmv_cl_cov_2h(h._nz, h._nm, h._nk, h._ldk, p(h._ks_d), p(h._ms_d), p(h._nzm_d),
                                                    p(h._bh_d), p(h._Pzk_d), h._rho_m0, self.u_h, self.k_h, n,
                                                    p(d["ells"]), n, p(d["ells"]), p(h._zs_d), p(d["chis"]),
                                                    p(d["pref"]), self.zchunk, p(self.ws), p(self.out),
                                                    self.capi.stream()), "hmv_cl_cov_2h")

    def check_sample(self, rng, npairs=6):
        """Max |got - want| / sum|terms| over seeded (l, l') entries: T2h per redshift from the cube columns the entries
        need (gathered on the device), I2, I3, I1~ and P by float64 host sums, Pbar from a long-double prefix."""
        import torch
        h = self.h
        got = self.out.cpu().numpy()
        ks, ms, nzm, bh, Pzk = h._ks64, h.ms, h.nzm, h.bh, h.Pzk
        wm = 0.5 * (ms[np.minimum(np.arange(ms.size) + 1, ms.size - 1)] - ms[np.maximum(np.arange(ms.size) - 1, 0)])
        zs = h.zs
        zw = 0.5 * (zs[np.minimum(np.arange(zs.size) + 1, zs.size - 1)] - zs[np.maximum(np.arange(zs.size) - 1, 0)])
        w = wm[None, :] * nzm * bh
        cons = 1.0 - (w * ms[None, :] / h._rho_m0).sum(1)
        zi = torch.arange(zs.size, device=self.cubes[0].device)
        kl = ks.astype(np.longdouble)

        def leg(c, ell):                   # t(z, m) at k = (l + 1/2)/chi_z, linear in k, clamped
            k = np.clip((ell + 0.5) / self.chis, ks[0], ks[-1])
            j = np.clip(np.searchsorted(ks, k, side="right") - 1, 0, ks.size - 2)
            f = (k - ks[j]) / (ks[j + 1] - ks[j])
            jd = torch.as_tensor(j, device=self.cubes[c].device)
            u0, u1 = self.cubes[c][zi, :, jd].cpu().numpy(), self.cubes[c][zi, :, jd + 1].cpu().numpy()
            a = ms / h._rho_m0 if self.kinds[c] == 0 else np.ones(ms.size)
            return a[None, :] * (u0 + f[:, None] * (u1 - u0))

        def F(z, x):                       # int_0^x q P dq, P linear on ks and held at its ends, long double
            P = Pzk[z].astype(np.longdouble)
            S = np.concatenate([[0], np.cumsum((kl[1:] - kl[:-1]) * (kl[:-1] * (2 * P[:-1] + P[1:]) +
                                                                      kl[1:] * (P[:-1] + 2 * P[1:])) / 6)])
            x = np.longdouble(x)
            if x < kl[0]:
                return P[0] * x * x / 2
            base = P[0] * kl[0] ** 2 / 2
            if x >= kl[-1]:
                return base + S[-1] + P[-1] * (x * x - kl[-1] ** 2) / 2
            r = min(max(np.searchsorted(kl, x, side="right") - 1, 0), ks.size - 2)
            px = P[r] + (x - kl[r]) / (kl[r + 1] - kl[r]) * (P[r + 1] - P[r])
            return base + S[r] + (x - kl[r]) * (kl[r] * (2 * P[r] + px) + x * (P[r] + 2 * px)) / 6

        worst = 0.0
        for _ in range(npairs):
            i, j = rng.integers(0, self.ells.size, 2)
            tA, tB = leg(0, self.ells[i]), leg(1, self.ells[i])
            tC, tD = leg(2, self.ells[j]), leg(3, self.ells[j])
            want = bound = 0.0
            for z in range(zs.size):
                k1, k2 = (self.ells[i] + 0.5) / self.chis[z], (self.ells[j] + 0.5) / self.chis[z]
                k1l, k2l = np.longdouble(k1), np.longdouble(k2)
                pb = float((F(z, k1l + k2l) - F(z, abs(k1l - k2l))) / (2 * k1l * k2l))
                P1, P2 = np.interp(k1, ks, Pzk[z]), np.interp(k2, ks, Pzk[z])
                W, Wa = w[z], np.abs(w[z])
                zo = [cons[z] if k == 0 else 0.0 for k in self.kinds]
                t = (tA[z], tB[z], tC[z], tD[z])
                vals = []
                for s, (Ww, f) in enumerate(((W, lambda x: x), (Wa, np.abs))):
                    I1 = [np.sum(Ww * f(t[q])) + f(zo[q]) for q in range(4)]
                    I3 = lambda x, y, u: np.sum(Ww * f(t[x] * t[y] * t[u]))
                    I2 = lambda x, y: np.sum(Ww * f(t[x] * t[y]))
                    v = f(P1) * (I1[0] * I3(1, 2, 3) + I1[1] * I3(0, 2, 3)) \
                        + f(P2) * (I1[2] * I3(0, 1, 3) + I1[3] * I3(0, 1, 2)) \
                        + f(pb) * (I2(0, 2) * I2(1, 3) + I2(0, 3) * I2(1, 2))
                    vals.append(v)
                want += zw[z] * self.pref[z] * vals[0]
                bound += abs(zw[z] * self.pref[z]) * abs(vals[1])
            worst = max(worst, abs(got[i, j] - want) / bound if bound > 0 else abs(got[i, j] - want))
        return worst


def time_case(case, reps, dmma_tflops):
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        case.launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        case.launch()
    e1.record()
    e1.synchronize()
    total_ms = e0.elapsed_time(e1) / reps
    nprof = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            case.launch()
        torch.cuda.synchronize()
    per = {}
    names = (("trispec2h_prep_kernel", "prep"), ("trispec2h_panel_kernel", "panel"), ("trispec_panel_kernel", "panel"),
             ("trispec_tracer_panel_kernel", "panel"),
             ("sigma2_gemm_kernel", "contraction"), ("trispec_reduce_kernel", "reduce"),
             ("trispec2h_assemble_kernel", "assemble"))
    for ev in prof.key_averages():
        key = next((k for n, k in names if n in ev.key), None)
        if key:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            per[key] = per.get(key, 0.0) + t / 1e3 / nprof
    h, n = case.h, case.ells.size
    blocks, nseg = getattr(case, "blocks", 1), getattr(case, "nseg", 1)
    flop = 2.0 * n * n * h._nz * h._nm * blocks * nseg
    K, ld = h._nz * nseg * (h._nm + h._nm % 2), n + n % 2
    res = {"nz": h._nz, "nm": h._nm, "nk": h._nk, "nl": n, "call_ms": total_ms, "reps": reps,
           "panel_ms": per.get("panel"), "contraction_ms": per.get("contraction"), "reduce_ms": per.get("reduce"),
           "flop": flop, "blocks": blocks, "segments": nseg}
    if blocks == 1:
        res["panel_bytes_written"] = 2.0 * K * ld * 8
    else:
        res.update(prep_ms=per.get("prep"), assemble_ms=per.get("assemble"), zchunk=case.zchunk,
                   names=list(case.names))
    if per.get("contraction"):
        res["contraction_tflops"] = flop / (per["contraction"] * 1e-3) / 1e12
        res["contraction_over_dmma"] = res["contraction_tflops"] / dmma_tflops
    if per.get("panel") and "panel_bytes_written" in res:
        res["panel_write_gbs"] = res["panel_bytes_written"] / (per["panel"] * 1e-3) / 1e9
    res["call_tflops"] = flop / (total_ms * 1e-3) / 1e12
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--nz", type=int, default=200)
    ap.add_argument("--nm", type=int, default=2000)
    ap.add_argument("--nk", type=int, default=10000)
    ap.add_argument("--nl", type=int, default=1000)
    ap.add_argument("--slab", type=int, default=25)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cases", default=None, help="comma-separated result tags to run (default: all)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    want = None if a.cases is None else set(a.cases.split(","))
    run = lambda tag: want is None or tag in want
    import torch
    if not torch.cuda.is_available():
        sys.exit("trispec_bench needs a CUDA device")
    import hmvec_b200 as hm
    from hmvec_b200 import _capi as capi
    info = {"card": card(), "torch": torch.__version__, "device": torch.cuda.get_device_name(0)}
    zs = np.linspace(0.01, 3., a.nz)
    ms = np.geomspace(2e10, 1e17, a.nm)
    ks = np.geomspace(1e-4, 100, a.nk)
    ells = np.geomspace(10, 1e4, a.nl)
    rng = np.random.default_rng(1234)
    dmma = capi.lib.hmv_bench_dmma(20000, capi.stream())
    info["dmma_tflops"] = dmma
    results = {}
    t = time.perf_counter()
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    h.add_hod("g", ngal=np.geomspace(2e-3, 5e-5, a.nz))
    Wk = h.lensing_window(zs, 2.5)
    dndz = np.exp(-0.5 * ((zs - 0.8) / 0.5) ** 2)
    Wg = dndz / np.sum(0.5 * (np.r_[zs[1:], zs[-1]] - np.r_[zs[0], zs[:-1]]) * dndz)
    torch.cuda.synchronize()
    info["model_setup_s"] = time.perf_counter() - t
    for tag, name, kind, win in (("large_kk", "nfw", 0, (Wk,) * 4), ("large_yy", "y", 2, (1.,) * 4)):
        if not run(tag):
            continue
        c = Case(h, name, kind, win, ells)
        results[tag] = time_case(c, a.reps, dmma)
        results[tag]["sample_max_err_over_bound"] = c.check_sample(rng)
        del c
        torch.cuda.empty_cache()
    for tag, names, win in (("large_kg_kg", ("nfw", "g", "nfw", "g"), (Wk, Wg, Wk, Wg)),
                            ("large_kk_gg", ("nfw", "nfw", "g", "g"), (Wk, Wk, Wg, Wg))):
        if not run(tag):
            continue
        c = CaseHod(h, names, win, ells)
        results[tag] = time_case(c, a.reps, dmma)
        results[tag]["names"] = list(names)
        results[tag]["sample_max_err_over_bound"] = c.check_sample(rng)
        del c
        torch.cuda.empty_cache()
    for tag, names, win in (("large_kk_2h", ("nfw",) * 4, (Wk,) * 4), ("large_yy_2h", ("y",) * 4, (1.,) * 4),
                            ("large_ky_ky_2h", ("nfw", "y", "nfw", "y"), (Wk, 1., Wk, 1.))):
        if not run(tag):
            continue
        c = Case2h(h, names, win, ells)
        results[tag] = time_case(c, a.reps, dmma)
        results[tag]["sample_max_err_over_bound"] = c.check_sample(rng)
        del c
        h._ws.clear()
        torch.cuda.empty_cache()
    del h
    torch.cuda.empty_cache()
    if run("slab_kk"):
        hs = hm.HaloModel(zs[:a.slab], ks, ms=ms, accuracy='low')
        c = Case(hs, "nfw", 0, (hs.lensing_window(zs[:a.slab], 2.5),) * 4, ells)
        results["slab_kk"] = time_case(c, a.reps, dmma)
        results["slab_kk"]["sample_max_err_over_bound"] = c.check_sample(rng)
    info["dmma_tflops_after"] = capi.lib.hmv_bench_dmma(20000, capi.stream())
    info["results"] = results
    txt = json.dumps(info, indent=1, sort_keys=True)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
