"""Time the non-Gaussian (1-halo) C_l covariance, hmv_cl_cov_1h, on the LARGE grid and on a 25-redshift slab.

Cases: C_kk x C_kk (NFW, lensing window of a source at z = 2.5) and C_yy x C_yy (Battaglia pressure) at
ells = geomspace(10, 1e4, nl) on zs = linspace(0.01, 3, nz), ms = geomspace(2e10, 1e17, nm), ks = geomspace(1e-4, 100,
nk) (bench.py's grid), and C_kk on the slab zs[:25].  For each case it reports, from one run on one device:

  * the whole call from CUDA events over --reps launches after two warm-up launches (panels, contraction, reduction);
  * the panel kernel and the contraction separately, from torch.profiler over three further launches;
  * flop = 2 n1 n2 nz nm, the contraction's TFLOP/s and its ratio to hmv_bench_dmma measured in the same run;
  * a check of a seeded sample of (l, l') entries against a float64 host reduction over the same cubes;

with the card's name and power limit read in the same run.  Prints one JSON document (and writes it to --out).

    python tools/trispec_bench.py [--nz 200 --nm 2000 --nk 10000 --nl 1000 --reps 10 --out FILE]
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
    for ev in prof.key_averages():
        key = "panel" if "trispec_panel_kernel" in ev.key else "contraction" if "sigma2_gemm_kernel" in ev.key else \
            "reduce" if "trispec_reduce_kernel" in ev.key else None
        if key:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            per[key] = per.get(key, 0.0) + t / 1e3 / nprof
    h, n = case.h, case.ells.size
    flop = 2.0 * n * n * h._nz * h._nm
    K, ld = h._nz * (h._nm + h._nm % 2), n + n % 2
    res = {"nz": h._nz, "nm": h._nm, "nk": h._nk, "nl": n, "call_ms": total_ms, "reps": reps,
           "panel_ms": per.get("panel"), "contraction_ms": per.get("contraction"), "reduce_ms": per.get("reduce"),
           "flop": flop, "panel_bytes_written": 2.0 * K * ld * 8}
    if per.get("contraction"):
        res["contraction_tflops"] = flop / (per["contraction"] * 1e-3) / 1e12
        res["contraction_over_dmma"] = res["contraction_tflops"] / dmma_tflops
    if per.get("panel"):
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
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
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
    Wk = h.lensing_window(zs, 2.5)
    torch.cuda.synchronize()
    info["model_setup_s"] = time.perf_counter() - t
    for tag, name, kind, win in (("large_kk", "nfw", 0, (Wk,) * 4), ("large_yy", "y", 2, (1.,) * 4)):
        c = Case(h, name, kind, win, ells)
        results[tag] = time_case(c, a.reps, dmma)
        results[tag]["sample_max_err_over_bound"] = c.check_sample(rng)
        del c
        torch.cuda.empty_cache()
    del h
    torch.cuda.empty_cache()
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
