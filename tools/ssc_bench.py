"""Time the super-sample covariance of C_l on the LARGE grid: the response pass, sigma_b^2 and the projection.

Grid: zs = linspace(0.01, 3, nz), ms = geomspace(2e10, 1e17, nm), ks = geomspace(1e-4, 100, nk) (bench.py's grid), the
NFW cube and the Battaglia pressure profile expanded to its cube.  From one run on one device it reports:

  * hmv_power_response for NFW x NFW (one cube, power_one's body) and NFW x y (two cubes, power_pair's body), beside
    hmv_power on the same cubes: the call from CUDA events over --reps launches after two warm-up launches, and the
    streaming kernel alone from torch.profiler over three further launches.  bytes = 8 nz nm nk per distinct cube;
    bytes / kernel time is reported as GB/s and as a fraction of the 6551 GB/s device copy rate of DESIGN.md §4;
  * hmv_sigma_b2 at f_sky = 0.4 on the sigma^2 grid's 10000 wavenumbers (CUDA events);
  * hmv_cl_cov_ssc for nl x nl multipoles (CUDA events; panel, contraction and reduction from torch.profiler);

with the card's name and power limit read in the same run.  Prints one JSON document (and writes it to --out).

    python tools/ssc_bench.py [--nz 200 --nm 2000 --nk 10000 --nl 1000 --reps 10 --out FILE]
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
COPY_GBS = 6551.0           # device copy rate of DESIGN.md §4


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:        # the numbers are still reported, without the card's settings
        return {"error": repr(e)}


def timed(launch, reps, kernels):
    """(ms per call from CUDA events, {key: ms per call of the kernels whose name contains key} from torch.profiler)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    e1.synchronize()
    call = e0.elapsed_time(e1) / reps
    nprof = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            launch()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        for key in kernels:
            if key in ev.key:
                t = getattr(ev, "device_time_total", None)
                if t is None:
                    t = ev.cuda_time_total
                per[key] = per.get(key, 0.0) + t / 1e3 / nprof
    return call, per


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--nz", type=int, default=200)
    ap.add_argument("--nm", type=int, default=2000)
    ap.add_argument("--nk", type=int, default=10000)
    ap.add_argument("--nl", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("ssc_bench needs a CUDA device")
    import hmvec_b200 as hm
    from hmvec_b200 import _capi as capi
    L, p = capi.lib, capi.ptr
    info = {"card": card(), "torch": torch.__version__, "device": torch.cuda.get_device_name(0)}
    zs = np.linspace(0.01, 3., a.nz)
    ms = np.geomspace(2e10, 1e17, a.nm)
    ks = np.geomspace(1e-4, 100, a.nk)
    t = time.perf_counter()
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    u_m, u_y = h.uk_profiles.device("nfw"), h.pk_profiles.device("y")       # the y tables expanded to their cube
    torch.cuda.synchronize()
    info["model_setup_s"] = time.perf_counter() - t
    nz, nm, nk, ldk = h._nz, h._nm, h._nk, h._ldk
    ws = h._empty(int(L.hmv_power_ws_doubles(nz, nm)))
    r1, r2 = h._empty(nz, nk), h._empty(nz, nk)
    results = {}

    def resp(uB, kB):
        return lambda: capi.check(L.hmv_power_response(nz, nm, nk, ldk, p(h._ms_d), p(h._ks_d), p(h._nzm_d),
                                                       p(h._bh_d), p(h._Pzk_d), h._rho_m0, p(u_m), 0, p(uB), kB,
                                                       p(ws), p(r1), p(r2), capi.stream()), "hmv_power_response")

    def power(uB, kB):
        A, B = capi.Tracer(), capi.Tracer()
        A.kind, A.us_d = 0, u_m.data_ptr()
        B.kind, B.us_d = kB, uB.data_ptr()
        return lambda: capi.check(L.hmv_power(nz, nm, nk, ldk, p(h._ms_d), p(h._ks_d), p(h._nzm_d), p(h._bh_d),
                                              p(h._Pzk_d), h._rho_m0, float(h.p['kstar_damping']), C.byref(A),
                                              C.byref(B), p(ws), p(r1), p(r2), capi.stream()), "hmv_power")

    cases = (("response_nfw_nfw", resp(u_m, 0), "power_one_resp_kernel", 1),
             ("power_nfw_nfw", power(u_m, 0), "power_one_kernel", 1),
             ("response_nfw_y", resp(u_y, 2), "power_pair_resp_kernel", 2),
             ("power_nfw_y", power(u_y, 2), "power_pair_kernel", 2))
    for tag, launch, kname, ncube in cases:
        call, per = timed(launch, a.reps, [kname + "("])
        kms = per.get(kname + "(")
        nbytes = 8.0 * nz * nm * nk * ncube
        results[tag] = {"call_ms": call, "kernel": kname, "kernel_ms": kms, "bytes": nbytes, "cubes": ncube}
        if kms:
            results[tag]["gbs"] = nbytes / (kms * 1e-3) / 1e9
            results[tag]["fraction_of_copy_rate"] = results[tag]["gbs"] / COPY_GBS

    # sigma_b^2 at f_sky = 0.4 on the disc's grid, the kernel alone
    R, kg, kw = h._sigma_b2_grid(0.4)
    P_d = h._plin_device(kg, zs)
    d = {k: h._dev(v) for k, v in dict(kg=kg, kw=kw, R=R).items()}
    sb2 = h._empty(nz)
    call, _ = timed(lambda: capi.check(L.hmv_sigma_b2(nz, kg.size, p(d["kg"]), p(d["kw"]), p(P_d), p(d["R"]), p(sb2),
                                                      capi.stream()), "hmv_sigma_b2"), a.reps, [])
    results["sigma_b2"] = {"call_ms": call, "nks": int(kg.size), "k_b": float(kg[0])}

    # the nl x nl projection of the NFW x NFW response
    resp(u_m, 0)()
    rAB = h._empty(nz, nk)
    capi.check(L.hmv_sum2(rAB.numel(), p(r1), p(r2), p(rAB), capi.stream()), "hmv_sum2")
    ells = np.geomspace(10, 1e4, a.nl)
    chis = np.asarray(h.comoving_radial_distance(zs), dtype=np.float64)
    H = np.asarray(h.h_of_z(zs), dtype=np.float64)
    Wk = h.lensing_window(zs, 2.5)
    pref = H ** 3 * Wk ** 4 * sb2.cpu().numpy() / chis ** 4
    d = {k: h._dev(v) for k, v in dict(ells=ells, chis=chis, pref=pref).items()}
    n = ells.size
    cws = h._empty(int(L.hmv_cl_cov_ssc_ws_doubles(nz, n, n)))
    out = h._empty(n, n)
    call, per = timed(lambda: capi.check(L.hmv_cl_cov_ssc(nz, nk, p(h._ks_d), p(rAB), p(rAB), n, p(d["ells"]), n,
                                                          p(d["ells"]), p(h._zs_d), p(d["chis"]), p(d["pref"]), p(cws),
                                                          p(out), capi.stream()), "hmv_cl_cov_ssc"),
                      a.reps, ["ssc_panel_kernel", "sigma2_gemm_kernel", "trispec_reduce_kernel"])
    results["projection"] = {"call_ms": call, "nl": n, "panel_ms": per.get("ssc_panel_kernel"),
                             "contraction_ms": per.get("sigma2_gemm_kernel"),
                             "reduce_ms": per.get("trispec_reduce_kernel"), "flop": 2.0 * n * n * nz}
    c = out.cpu().numpy()
    results["projection"]["finite"] = bool(np.all(np.isfinite(c)))
    results["projection"]["max_asymmetry_over_max"] = float(np.max(np.abs(c - c.T)) / np.max(np.abs(c)))
    info["results"] = results
    txt = json.dumps(info, indent=1, sort_keys=True)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
