"""Time the 3- and 4-halo covariances of C_l (HaloModel.get_cl_cov_3halo / get_cl_cov_4halo) on the LARGE grid.

Grid: zs = linspace(0.01, 3, nz), ms = geomspace(2e10, 1e17, nm), ks = geomspace(1e-4, 100, nk) (bench.py's grid),
ells = geomspace(10, 1e4, nl).  Cases: C_kk auto (NFW, lensing window of a source at z = 2.5), C_yy auto (Battaglia
pressure) and C_ky x C_ky (NFW, y, NFW, y), each for the 3- and the 4-halo term.  For each case, from one run on one
device:

  * the whole API call (device work, the copy of the result to the host) from CUDA events over --reps calls after two
    warm-up calls;
  * the per-kernel split from torch.profiler over three further calls;
  * for 3h: flop = 2 nz nm n1 n2 per contracted I2 block (1 for the autos, 4 for C_ky x C_ky), the contraction's
    TFLOP/s and its ratio to hmv_bench_dmma measured in the same run;
  * the assembly kernel's time per (z, l, l') point;

with the card's name and power limit read in the same run.  Prints one JSON document (and writes it to --out).

    python tools/trispec_pt_bench.py [--nz 200 --nm 2000 --nk 10000 --nl 1000 --reps 5 --out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tools.trispec_bench import card  # noqa: E402

KERNELS = (("trispec_pt_moments_kernel", "moments"), ("trispec_pt_side_kernel", "sides"),
           ("trispec2h_panel_kernel", "panel"), ("sigma2_gemm_kernel", "contraction"),
           ("trispec4h_f3_kernel", "f3"), ("trispec3h_assemble_kernel", "assemble"),
           ("trispec4h_assemble_kernel", "assemble"))


def time_case(call, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        call()
    e1.record()
    e1.synchronize()
    total_ms = e0.elapsed_time(e1) / reps
    nprof = 3
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(nprof):
            call()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.key_averages():
        key = next((k for n, k in KERNELS if n in ev.key), None)
        if key:
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = ev.cuda_time_total
            per[key] = per.get(key, 0.0) + t / 1e3 / nprof
    return total_ms, per


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--nz", type=int, default=200)
    ap.add_argument("--nm", type=int, default=2000)
    ap.add_argument("--nk", type=int, default=10000)
    ap.add_argument("--nl", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("trispec_pt_bench needs a CUDA device")
    import hmvec_b200 as hm
    from hmvec_b200 import _capi as capi
    info = {"card": card(), "torch": torch.__version__, "device": torch.cuda.get_device_name(0)}
    zs = np.linspace(0.01, 3., a.nz)
    ms = np.geomspace(2e10, 1e17, a.nm)
    ks = np.geomspace(1e-4, 100, a.nk)
    ells = np.geomspace(10, 1e4, a.nl)
    info["dmma_tflops"] = dmma = capi.lib.hmv_bench_dmma(20000, capi.stream())
    t = time.perf_counter()
    h = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    Wk = h.lensing_window(zs, 2.5)
    torch.cuda.synchronize()
    info["model_setup_s"] = time.perf_counter() - t
    results = {}
    cases = (("kk", ("nfw",) * 4, (Wk,) * 4, 1), ("yy", ("y",) * 4, (1.,) * 4, 1),
             ("ky_ky", ("nfw", "y", "nfw", "y"), (Wk, 1., Wk, 1.), 4))
    for order in (3, 4):
        for tag, names, win, blocks in cases:
            fn = getattr(h, "get_cl_cov_%dhalo" % order)
            total, per = time_case(lambda: fn(ells, *names, windows=win), a.reps)
            r = {"names": list(names), "call_ms": total, "kernels_ms": per, "nz": a.nz, "nm": a.nm, "nk": a.nk,
                 "nl": a.nl, "points": a.nz * a.nl * a.nl}
            if per.get("assemble"):
                r["assemble_ns_per_point"] = per["assemble"] * 1e6 / r["points"]
            if order == 3:
                r["blocks"] = blocks
                r["flop"] = 2.0 * a.nz * a.nm * a.nl * a.nl * blocks
                if per.get("contraction"):
                    r["contraction_tflops"] = r["flop"] / (per["contraction"] * 1e-3) / 1e12
                    r["contraction_over_dmma"] = r["contraction_tflops"] / dmma
            results["large_%s_%dh" % (tag, order)] = r
            h._ws.clear()
            torch.cuda.empty_cache()
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
