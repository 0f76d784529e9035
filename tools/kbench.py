#!/usr/bin/env python
"""Kernel-level A/B bench on a z-slab of the LARGE grid: times hmv_profile_transform (K1), hmv_uk_nfw (K2) and every
K5 mass-integral entry point alone with CUDA events, for one or several builds of the library (same C ABI), and
compares the cubes and spectra each build writes with those of the first one.

    python tools/kbench.py --nz 25 --libs hmvec_b200/libhmvec_b200.so,variants/lib_v2.so [--reps 10]
    python tools/kbench.py --kernels k5 --libs old,new,old,new      # variants/lib_old.so, ... (tools/build_variant.sh)

Each build runs in its own process (HMV_LIB selects the library).  Run on a GPU box."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def child(a):
    import torch
    from hmvec_b200 import _capi as capi, pipeline
    zs_all = np.linspace(0.01, 3., 200)
    pick = np.linspace(0, 199, a.nz).round().astype(int)          # spread over the whole redshift range
    zs = zs_all[pick]
    ms = np.geomspace(2e10, 1e17, a.nm)
    ks = np.geomspace(1e-4, 100, a.nk)
    inp = pipeline.make_inputs(zs, ms, ks, ngal=np.geomspace(1e-3, 1e-5, 200)[pick])
    g = pipeline.GridSix(inp)
    g.upload()
    g.run()
    torch.cuda.synchronize()
    L, d, ptr, st = capi.lib, g.d, capi.ptr, capi.stream()
    nz, nm, nk, ldk = g.nz, g.nm, g.nk, g.ldk

    def k1():
        capi.check(L.hmv_profile_transform(nz, nm, nk, ldk, ptr(d["zs"]), ptr(d["ks"]), g.kmax, ptr(d["rs"]),
                                           ptr(d["cmax"]), ptr(d["xc"]), ptr(d["alpha"]), ptr(d["expo"]), ptr(d["amp"]),
                                           ptr(d["oscale"]), g.gamma, g.xmax, g.nxs, 1, ptr(d["tr_ws"]), ptr(g.ue), st),
                   "hmv_profile_transform")

    def k2():
        capi.check(L.hmv_uk_nfw(nz, nm, nk, ldk, ptr(d["zs"]), ptr(d["ks"]), g.kmax, ptr(d["cs"]), ptr(d["rvir"]),
                                ptr(d["nfw_ws"]), ptr(g.um), st), "hmv_uk_nfw")

    # K5 on the same slab: hmv_power for mm / gg / me / ge runs power_one_kernel, and power_pair_kernel with one and
    # with two cubes; hmv_power_tab reads the pipeline's pressure tables, hmv_power_six_tab electron tables made here
    E = lambda *s: torch.empty(s, dtype=torch.float64, device="cuda")
    ws, ws_nfw = E(int(L.hmv_power_ws_doubles(nz, nm))), E(int(L.hmv_power_six_nfw_ws_doubles(nz, nm)))
    etab = torch.zeros(int(L.hmv_profile_table_doubles(nz, nm, g.nxs)), dtype=torch.float64, device="cuda")
    tr_ws = E(int(L.hmv_profile_transform_ws_doubles(nz, nm, g.nxs)))
    capi.check(L.hmv_profile_tables(nz, nm, nk, ptr(d["zs"]), ptr(d["ks"]), g.kmax, ptr(d["rs"]), ptr(d["cmax"]),
                                    ptr(d["xc"]), ptr(d["alpha"]), ptr(d["expo"]), ptr(d["amp"]), ptr(d["oscale"]),
                                    g.gamma, g.xmax, g.nxs, 1, ptr(tr_ws), ptr(etab), st), "hmv_profile_tables")
    hod = [ptr(d[k]) for k in ("Nc", "Ns", "NcNs", "NsNsm1", "ngal")]

    def tracer(kind, u):
        t = capi.Tracer()
        t.kind, t.us_d = kind, u.data_ptr()
        if kind == 1:
            t.Nc_d, t.Ns_d, t.NcNs_d, t.NsNsm1_d, t.ngal_d = (d[k].data_ptr() for k in ("Nc", "Ns", "NcNs", "NsNsm1", "ngal"))
        return t

    tm, te, tg = tracer(0, g.um), tracer(0, g.ue), tracer(1, g.um)
    k5_out = {}

    def spectra(name, n):
        k5_out[name] = (E(n, nz, nk), E(n, nz, nk))
        return [ptr(x) for x in k5_out[name]]

    base = (ptr(d["ms"]), ptr(d["ks"]), ptr(d["nzm"]), ptr(d["bh"]), ptr(d["Pzk"]), g.rho_m0, float(g.p['kstar_damping']))
    k5_calls = {
        "k5_six": (L.hmv_power_six, (nz, nm, nk, ldk, *base, ptr(g.um), ptr(g.ue), *hod, ptr(ws), 0,
                                     *spectra("k5_six", 6), st)),
        "k5_six_tab": (L.hmv_power_six_tab, (nz, nm, nk, ldk, *base, ptr(g.um), ptr(etab), g.nxs, *hod, ptr(ws), 0,
                                             *spectra("k5_six_tab", 6), st)),
        "k5_six_nfw": (L.hmv_power_six_nfw, (nz, nm, nk, ldk, ptr(d["zs"]), *base, ptr(d["cs"]), ptr(d["rvir"]),
                                             ptr(g.ue), *hod, ptr(ws_nfw), 0, *spectra("k5_six_nfw", 6), st)),
        "k5_tab_yy": (L.hmv_power_tab, (nz, nm, nk, *base, 2, ptr(g.ytab), g.p_nxs, ptr(ws), *spectra("k5_tab_yy", 1),
                                        st)),
    }
    for name, A, B in (("mm", tm, tm), ("gg", tg, tg), ("me", tm, te), ("ge", tg, te)):
        k5_calls["k5_" + name] = (L.hmv_power, (nz, nm, nk, ldk, *base, C.byref(A), C.byref(B), ptr(ws),
                                                *spectra("k5_" + name, 1), st))

    def k5(name):
        fn, args = k5_calls[name]
        return lambda: capi.check(fn(*args), name)

    out = {"lib": os.environ.get("HMV_LIB", "default"), "nz": nz}
    for name, fn in [("k1", k1), ("k2", k2)] + [(name, k5(name)) for name in k5_calls]:
        if name.split("_")[0] not in a.kernels:
            continue
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        out[name + "_ms"] = float(np.median(ts))
        out[name + "_min"] = float(np.min(ts))
    # samples of the cubes for the parity comparison between builds
    rows = slice(None, None, 37)
    dump = dict(ue=g.ue[:, rows, :nk].cpu().numpy(), um=g.um[:, rows, :nk].cpu().numpy())
    for name, (p1, p2) in k5_out.items():
        if name + "_ms" in out:
            dump[name + "_p1"], dump[name + "_p2"] = p1.cpu().numpy(), p2.cpu().numpy()
    np.savez(a.dump, **dump)
    print("KBENCH " + json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nz", type=int, default=25)
    ap.add_argument("--nm", type=int, default=2000)
    ap.add_argument("--nk", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--kernels", default="k1,k2,k5")
    ap.add_argument("--libs", default="")
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--dump", default="/tmp/kbench_dump.npz")
    a = ap.parse_args()
    a.kernels = a.kernels.split(",")
    if a.child:
        return child(a)
    libs = [l if os.path.exists(l) else os.path.join(ROOT, "variants", "lib_%s.so" % l) for l in a.libs.split(",") if l]
    libs = libs or [os.path.join(ROOT, "hmvec_b200", "libhmvec_b200.so")]
    ref = None
    for i, lib in enumerate(libs):
        env = dict(os.environ, HMV_LIB=os.path.abspath(lib))
        dump = "/tmp/kbench_dump_%d.npz" % i
        cmd = [sys.executable, os.path.abspath(__file__), "--child", "--nz", str(a.nz), "--nm", str(a.nm), "--nk", str(a.nk),
               "--reps", str(a.reps), "--kernels", ",".join(a.kernels), "--dump", dump]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
        line = [l for l in r.stdout.splitlines() if l.startswith("KBENCH ")]
        if r.returncode != 0 or not line:
            print("KBENCH-FAIL %s rc=%d\n%s" % (lib, r.returncode, (r.stdout + r.stderr)[-2000:]), flush=True)
            continue
        res = json.loads(line[0][7:])
        cur = dict(np.load(dump))
        os.remove(dump)
        if ref is None:
            ref = cur
        else:
            for k in ref:
                sc = np.max(np.abs(ref[k]))
                res["dmax_" + k] = float(np.max(np.abs(cur[k] - ref[k])) / sc)
                if k not in ("ue", "um"):
                    with np.errstate(all="ignore"):
                        rel = np.abs(cur[k] - ref[k]) / np.abs(ref[k])
                    res["rel_" + k] = float(np.nanmax(np.where(np.isfinite(rel), rel, 0.0)))
        print("KBENCH " + json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
