#!/usr/bin/env python
"""bench.py -- P(k,z) grid points per second for the hmvec hot path on B200 (BASELINE.json metric).

A step = one pass of the whole path over the LARGE synthetic grid (BASELINE.json configs[3]+[4]):
    zs=linspace(0.01,3,200), ms=geomspace(2e10,1e17,2000), ks=geomspace(1e-4,100,10000), EH98 linear power;
    sigma^2 -> n(M,z), b -> u_NFW cube -> Battaglia-AGN electron cube (xmax=20, nxs=5000) -> Battaglia pressure
    (Compton-y) cube -> ngal-solved HOD -> {mm,ee,me,gg,gm,ge,yy} 1h+2h spectra -> [all-gather over z] ->
    Limber C_kk, C_kg, C_yy at 1000 ells.
One "grid point" = one (z,k) of one spectrum with both its 1-halo and 2-halo terms: 7*nz*nk points per step.
With N GPUs the z axis is sharded (nz/N redshifts per rank, total work fixed -> "strong" scaling).

  value : device-resident inputs, the allocation-free launch sequence (pipeline.GridSix), CUDA events around K steps,
          max over ranks
  e2e   : the same step through the drop-in API a user calls -- HaloModel(zs,ks,ms) -> add_battaglia_profile ->
          add_battaglia_pres_profile -> add_hod(ngal=...) -> seven get_power -> C_kk / C_kg / C_yy -- numpy in, numpy
          out, every host<->device copy inside the timed region
  --impl reference : the reference's own CPU implementation on the host cores: the unmodified simonsobs/hmvec installed
          under oracle/_ref (oracle/build_ref.sh) when present, else the oracle port; one z-slab per worker process
  --dump-outputs DIR : the outputs of the last timed step as .npy files.  The inputs depend only on the arguments, so
          two builds of the project run with the same arguments can be compared array for array.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "P(k,z) grid pts/s, Battaglia+HOD 1h+2h"
UNIT = "pts/s"
NSPEC = 7
PAIRS = (("nfw", "nfw"), ("electron", "electron"), ("nfw", "electron"), ("g", "g"), ("g", "nfw"), ("g", "electron"),
         ("y", "y"))
SHARD_REF = os.path.join(ROOT, "profiles", "r02_shard_reference.json")


def grids(a):
    zs = np.linspace(0.01, 3., a.nz)
    ms = np.geomspace(2e10, 1e17, a.nm)
    ks = np.geomspace(1e-4, 100, a.nk)
    ells = np.geomspace(10, 1e4, a.nl)
    return zs, ms, ks, ells


def workload_name(a):
    return "C4+C5: zs=%d, ms=%d (2e10-1e17), ks=%d (1e-4-100), Battaglia AGN electron (xmax=20,nxs=5000) + Battaglia " \
           "pressure (tSZ) + ngal-HOD, seven spectra 1h+2h (mm,ee,me,gg,gm,ge,yy), Limber C_kk/C_kg/C_yy at %d ells" \
           % (a.nz, a.nm, a.nk, a.nl)


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's numpy path on a z-slab, one slab per worker process
# ---------------------------------------------------------------------------------------------------------
def _reference_kind():
    from oracle import ref_loader
    return "reference" if ref_loader.available() else "port"


def _cpu_slab(job):
    """The whole path on one z-slab at full k resolution: the unmodified reference when oracle/_ref holds it, else the
    oracle port.  Returns (seconds, checksum)."""
    zs, ms, ks, ngal, ells, kind = job
    import warnings
    warnings.filterwarnings("ignore")
    sink = io.StringIO()
    t = time.perf_counter()
    with contextlib.redirect_stdout(sink):
        if kind == "reference":
            from oracle import ref_loader
            hm = ref_loader.load()
            o = hm.HaloModel(zs, ks, ms=ms, accuracy='low')
            o.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
            o.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
        else:
            from oracle import hmvec_oracle as orc
            o = orc.OracleHaloModel(zs, ks, ms)
            o.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
            o.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
        o.add_hod("g", ngal=ngal)
        chk, P = 0.0, {}
        for a, b in PAIRS:
            P[(a, b)] = o.get_power_1halo(a, b) + o.get_power_2halo(a, b)
            chk += float(np.sum(P[(a, b)][:, ::97]))
        # Limber on this slab's own P(k,z) table (cost scales with the number of redshifts, as the full table's does).
        # The reference's single-redshift branch (interp1d with bounds_error) rejects k=(l+1/2)/chi outside ks, so a
        # one-redshift slab is handed over as a two-row table, which takes the clamping 2-D branch like the full grid.
        zl = zs if zs.size > 1 else np.array([zs[0], zs[0] + 0.01])
        tab = lambda p: P[p] if zs.size > 1 else np.vstack([P[p], P[p]])
        chk += float(np.sum(o.C_kk(ells, zl, ks, tab(("nfw", "nfw")), lzs1=2.5, lzs2=2.5)))
        chk += float(np.sum(o.C_kg(ells, zl, ks, tab(("g", "nfw")), gzs=0.8, lzs=2.5)))
        chk += float(np.sum(o.C_yy(ells, zl, ks, tab(("y", "y")))))
    return time.perf_counter() - t, chk


def cpu_workers():
    n = os.cpu_count() or 1
    try:
        import psutil
        n = min(n, max(1, int(psutil.virtual_memory().available / 5e9)))   # ~4 GB peak RSS per 1-z slab
    except Exception:
        pass
    return max(1, min(n, 64))


def cpu_sample(a, nworkers, zper=1, kind=None, mstride=1):
    """Time `nworkers` concurrent slabs of `zper` redshifts each at full k resolution on every `mstride`-th mass (every
    stage of the path costs time proportional to the number of masses, so the rate is scaled back by nm_sample/nm);
    returns (pts/s at the full mass resolution, seconds)."""
    kind = kind or _reference_kind()
    zs, ms_full, ks, ells = grids(a)
    ms = ms_full[::mstride]
    ngal = np.geomspace(1e-3, 1e-5, zs.size)
    pick = np.linspace(0, zs.size - 1, nworkers * zper).round().astype(int)
    jobs = [(zs[pick[i * zper:(i + 1) * zper]], ms, ks, ngal[pick[i * zper:(i + 1) * zper]], ells, kind)
            for i in range(nworkers)]
    t = time.perf_counter()
    if nworkers == 1:
        _cpu_slab(jobs[0])
    else:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(nworkers) as pool:
            pool.map(_cpu_slab, jobs)
    dt = time.perf_counter() - t
    return float(NSPEC) * nworkers * zper * ks.size / dt * (ms.size / float(ms_full.size)), dt


REFERENCE_BUDGET_S = 240.0      # the K timed steps of --impl reference are sized to end within about this


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    P = cpu_workers()
    kind = _reference_kind()
    # one warm-up step at the full mass resolution pages numpy/scipy in and sizes the per-step sample: if K such steps
    # would overrun the budget, every later step keeps all k and thins the mass axis (cost is linear in nm)
    t_full = cpu_sample(a, P, kind=kind)[1]
    mstride = max(1, int(np.ceil(a.steps * t_full / REFERENCE_BUDGET_S)))
    nm_s = len(range(0, a.nm, mstride))
    secs, vals = [], []
    for _ in range(a.steps):
        v, dt = cpu_sample(a, P, kind=kind, mstride=mstride)
        secs.append(dt)
        vals.append(v)
    value = float(NSPEC) * P * a.nk * a.steps / sum(secs) * (nm_s / float(a.nm))
    what = "the unmodified reference (oracle/_ref)" if kind == "reference" else "the oracle port of the reference"
    sample = "%s: %d concurrent 1-redshift slabs (of %d z) per step at full %d k resolution on %d of %d masses (rate " \
             "scaled by %d/%d: every stage is linear in the number of masses), whole path incl. tSZ and Limber; the " \
             "warm-up step at all %d masses took %.1f s" % (what, P, a.nz, a.nk, nm_s, a.nm, nm_s, a.nm, a.nm, t_full)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * sum(secs) / a.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(a), "parallelism": "host processes x%d" % P},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": P, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """Polls SM clock and throttle reasons through NVML from a thread while the timed region runs."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
               ("hw_thermal_slowdown", 0x40), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, index, period=0.01):
        import threading
        self.sm, self.bits, self.mx, self.power = [], 0, None, []
        self._stop = threading.Event()
        self._ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._ok = True
        except Exception:
            return
        self.period = period
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self._stop.wait(self.period)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": [], "samples": 0}
        if not self._ok:
            return out
        self._stop.set()
        self.t.join(timeout=2)
        if self.sm:
            out.update(sm_mhz=float(np.median(self.sm)), samples=len(self.sm),
                       power_w_max=float(np.max(self.power)) if self.power else None)
        out["reasons"] = [n for n, b in self.REASONS if self.bits & b]
        return out


def api_step(hm, zc, zs, ms, ks, ells, ngal):
    """The drop-in workflow (README.rst:55-123 + the tSZ notebook's profile) on this rank's redshift slab: numpy in,
    numpy out.  With a sharded z axis the three P(k,z) tables Limber integrates are gathered over the ranks."""
    sl = zc.slab if zc is not None else slice(None)
    with contextlib.redirect_stdout(io.StringIO()):       # the reference prints the bisection's iteration count
        h = hm.HaloModel(zs[sl], ks, ms=ms, accuracy='low', zcomm=zc)
        h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
        h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
        h.add_hod("g", ngal=ngal[sl])
        P = {p: h.get_power(*p) for p in PAIRS}
        if zc is not None:
            # sharded: the three tables Limber integrates are gathered from their device copies and stay on the
            # device (C_kk & co. accept CUDA tensors) -- no round trip through the host
            Pmm, Pgm, Pyy = zc.all_gather_tables([h.get_power_device(*p)
                                                  for p in (("nfw", "nfw"), ("g", "nfw"), ("y", "y"))])
        else:
            Pmm, Pgm, Pyy = P[("nfw", "nfw")], P[("g", "nfw")], P[("y", "y")]
    ckk = h.C_kk(ells, zs, ks, Pmm, lzs1=2.5, lzs2=2.5)
    ckg = h.C_kg(ells, zs, ks, Pgm, gzs=0.8, lzs=2.5)
    cyy = h.C_yy(ells, zs, ks, Pyy)
    return P, ckk, ckg, cyy


def summary_for_shard_check(P_local, cl, world, dist, dev):
    """Numbers that must not depend on how the z axis is sharded: the three C_ell vectors (replicated after the
    all-gather) and the sum over ALL redshifts of a strided sample of every spectrum (summed over the ranks)."""
    import torch
    sums = torch.tensor([float(np.sum(P_local[p][:, ::97])) for p in PAIRS], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(sums)
    return {"cl": [np.asarray(c)[::100].tolist() for c in cl], "spectra_sums": sums.cpu().tolist()}


DUMP_BUDGET = 60 * 10 ** 6     # bytes of array data --dump-outputs writes at most


def sample_outputs(g, ks, nz_total, world, dist):
    """What the caller of the timed launch sequence receives from its last step (GridSix.spectra()): P1h and P2h of
    the seven spectra [nz, nk] and C_kk, C_kg, C_yy, all float64.  When the whole set exceeds DUMP_BUDGET the spectra
    keep a fixed, seeded subset of their k columns, listed in `ks`.  With a sharded z axis the slabs are gathered."""
    p1, p2, ckk, ckg = g.spectra()
    tags, nk = tuple(p1), ks.size
    ncol = min(nk, max(1, (DUMP_BUDGET - 8 * 3 * ckk.size) // (16 * len(tags) * nz_total + 8)))
    cols = np.arange(nk) if ncol == nk else np.sort(np.random.default_rng(0).choice(nk, ncol, replace=False))
    out = {}
    for t in tags:
        out["P1h_" + t] = p1[t][:, cols]
        out["P2h_" + t] = p2[t][:, cols]
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, out)          # rank order is z order
        out = {n: np.concatenate([p[n] for p in parts]) for n in out}
    out.update(C_kk=ckk, C_kg=ckg, C_yy=g.last_cyy, ks=ks[cols])
    return out


def run_b200(a):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import warnings
    warnings.filterwarnings("ignore", message="camb not installed")
    import hmvec_b200 as hm
    from hmvec_b200 import _capi as capi, pipeline, zshard

    zs, ms, ks, ells = grids(a)
    ngal = np.geomspace(1e-3, 1e-5, zs.size)
    inp = pipeline.make_inputs(zs, ms, ks, ells=ells, ngal=ngal)
    zc = zshard.ZComm(a.nz, None) if world > 1 else None
    sl = zc.slab if zc is not None else slice(0, a.nz)
    g = pipeline.GridSix(pipeline.slab_inputs(inp, sl), device=dev, zcomm=zc, nz_total_zs=zs,
                         fused_nfw=a.fused_nfw, tsz_tables=not a.tsz_cube)
    capi.check(capi.lib.hmv_set_transform_mode(a.transform_mode), "hmv_set_transform_mode")
    g.transform_mode = a.transform_mode
    g.upload()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms_):
        if world == 1:
            return ms_
        t = torch.tensor([ms_], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(a.warmup, 3)):
        g.run()
    barrier()

    # ---- device-resident timing: the launch sequence as it ships (independent legs on their own streams) ---------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local) if rank == 0 else None
    barrier()
    e0.record()
    for s in range(a.steps):
        g.run()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler is not None else None
    dump = sample_outputs(g, ks, a.nz, world, dist) if a.dump_outputs else None

    # ---- per-stage times: the same steps again with the stages strictly one after the other on one stream and an
    # event at every stage boundary (a kernel's own duration, for the roofline entries; their sum is `serial_ms`) ----
    nst = len(g.STAGES) + 1
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(nst)] for _ in range(a.steps)]
    barrier()
    e0.record()
    for s in range(a.steps):
        g.run(events=evs[s])
    e1.record()
    barrier()
    ms_serial = max_over_ranks(e0.elapsed_time(e1))
    stage_ms = np.array([[evs[s][i].elapsed_time(evs[s][i + 1]) for i in range(nst - 1)] for s in range(a.steps)])
    stage_ms = stage_ms.mean(axis=0)

    # ---- the same launch sequence through pinned host buffers (kept as a second end-to-end figure) --------------
    for _ in range(2):
        g.upload(); g.run(overlap_d2h=True); g.finish_e2e()
    barrier()
    e0.record()
    for s in range(a.steps):
        g.upload()                   # pinned host -> HBM: linear power, background, ngal targets
        g.run(overlap_d2h=True)      # spectra go back chunk by chunk while later z-chunks are still being reduced
        g.finish_e2e()               # the step's results are on the host before the next one starts
    e1.record()
    barrier()
    ms_pinned = max_over_ranks(e0.elapsed_time(e1))
    g1, g2, gkk, gkg = g.spectra()
    launches = int(g.launches_per_run)
    pin_h2d, pin_d2h = g.h2d_bytes(), g.d2h_bytes()
    gyy = g.last_cyy

    # ---- per-stage roofline inputs taken from the resident state, then free the slab for the API leg ------------
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json)") if peaks.get("hbm_gbs") else (6650.0, "fallback")
    nzl, nm, nk = g.nz, g.nm, g.nk
    fp64_tf = float(capi.lib.hmv_bench_dfma(20000, capi.stream()))
    dmma_tf = float(capi.lib.hmv_bench_dmma(2000, capi.stream()))

    def k1_flops(rs_t, cmax_t, xmax, nxs):
        dx = xmax / nxs
        kt1 = 2.0 * np.pi / (nxs * ((xmax - dx) / nxs))
        rs_h, cmax_h, zs_h = rs_t.cpu().numpy(), cmax_t.cpu().numpy(), g.d["zs"].cpu().numpy()
        ncut = np.minimum(nxs, np.floor(cmax_h / dx))
        jneed = np.minimum(nxs // 2, np.floor(g.kmax * rs_h * (1.0 + zs_h[:, None]) / kt1) + 1.0)
        return float(2.0 * np.sum(ncut * jneed))

    k1_flop = k1_flops(g.d["rs"], g.d["cmax"], g.xmax, g.nxs)
    k1p_flop = k1_flops(g.d["y_rs"], g.d["y_cmax"], g.p_xmax, g.p_nxs) if g.tsz else 0.0
    fused_nfw, ldk, mode = g.fused_nfw, g.ldk, g.transform_mode
    overlap_level = int(g.overlap)
    tsz_tables = g.tsz_tables
    ytab_bytes = 0.0
    if tsz_tables:      # bins the Compton-y tables actually hold: sum over halos of (bin count + 2) doubles
        ytab_bytes = 8.0 * float(np.sum(np.minimum(g.p_nxs // 2, np.floor(g.kmax * g.d["y_rs"].cpu().numpy() *
                                 (1.0 + g.d["zs"].cpu().numpy()[:, None]) / (2.0 * np.pi / (g.p_nxs * ((g.p_xmax - g.p_xmax / g.p_nxs) / g.p_nxs)))) + 2.0) + 2.0))
    del g
    torch.cuda.empty_cache()

    # ---- end to end through the drop-in API: numpy in, numpy out ---------------------------------------------------
    for _ in range(2):
        out = api_step(hm, zc, zs, ms, ks, ells, ngal)
    barrier()
    capi.reset_copy_counters()
    e0.record()
    t0 = time.perf_counter()
    for s in range(a.steps):
        out = api_step(hm, zc, zs, ms, ks, ells, ngal)
    e1.record()
    barrier()
    wall_api = (time.perf_counter() - t0) * 1e3
    ms_api = max_over_ranks(max(e0.elapsed_time(e1), wall_api))
    h2d_api, d2h_api = capi.copy_counters()
    aP, akk, akg, ayy = out
    # the two paths must agree (the API routes the six standard pairs through the same kernels)
    api_vs_launchseq = max(float(np.max(np.abs(akk / gkk - 1.0))), float(np.max(np.abs(akg / gkg - 1.0))),
                           float(np.max(np.abs(ayy / gyy - 1.0))) if gyy is not None else 0.0)
    summ = summary_for_shard_check(aP, (akk, akg, ayy), world, dist, dev)

    if zc is not None:
        zc.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pts_per_step = float(NSPEC) * a.nz * a.nk
    value = pts_per_step * a.steps / (ms_total * 1e-3)
    e2e = pts_per_step * a.steps / (ms_api * 1e-3)

    shard = {"reference": None, "cl_max_rel": None, "spectra_sums_max_rel": None}
    if a.write_shard_ref and world == 1:
        with open(SHARD_REF, "w") as f:
            json.dump({"grid": [a.nz, a.nm, a.nk, a.nl], **summ}, f)
    try:
        with open(SHARD_REF) as f:
            ref = json.load(f)
        if ref.get("grid") == [a.nz, a.nm, a.nk, a.nl]:
            rel = lambda x, y: float(np.max(np.abs(np.asarray(x) / np.asarray(y) - 1.0)))
            shard = {"reference": "profiles/r02_shard_reference.json (written by a 1-GPU run)",
                     "cl_max_rel": max(rel(x, y) for x, y in zip(summ["cl"], ref["cl"])),
                     "spectra_sums_max_rel": rel(summ["spectra_sums"], ref["spectra_sums"])}
    except Exception:
        pass

    # ---- roofline per stage (algorithmic bytes per launch of the stage's main kernel; this rank's slab) ------
    alg_bytes = {
        "uk_nfw": 8.0 * nzl * nm * nk,                                  # store of the cube (K2; FP64-pipe bound)
        "uk_electron": 8.0 * nzl * nm * nk,                             # store of the cube (K1; FP64-pipe bound)
        # second K1 launch (tSZ): the cube, or -- table mode -- only the bin tables (then FP64-bound, not a store)
        "uk_pressure": ytab_bytes if tsz_tables else 8.0 * nzl * nm * nk,
        # two-cube kernel: read 2 cubes once, write 12 spectra, read Pzk.  Fused kernel: one cube + 448 B of per-halo
        # coefficient/NFW records per (z,M) for each of the ceil(nk/512) k tiles
        "power_six": (nzl * nk * (16.0 * nm + 96.0 + 8.0) if not fused_nfw else
                      nzl * nk * (8.0 * nm + 96.0 + 8.0) + 448.0 * nzl * nm * ((ldk + 511) // 512)),
        # one cube read, P1h + P2h written; table mode: every k tile reads its segment of the tables (~ the tables once)
        "power_yy": (ytab_bytes + nzl * nk * 24.0) if tsz_tables else nzl * nk * (8.0 * nm + 16.0 + 8.0),
        "sigma2": 8.0 * (nzl * 10000 + 2.0 * 10000 * nm + nzl * nm),    # sPzk + W2 table write/read + sigma2 out
    }
    if fused_nfw:
        del alg_bytes["uk_nfw"]          # no NFW cube in the spectra-only fusion
    kernels = {}
    for name, ms_ in zip(pipeline.GridSix.STAGES, stage_ms):
        k = {"ms": float(ms_)}
        if name in alg_bytes and ms_ > 0:
            gbs = alg_bytes[name] / (ms_ * 1e-3) / 1e9
            k.update(alg_bytes=alg_bytes[name], gbs=gbs, frac_hbm=gbs / hbm_peak)
        kernels[name] = k
    # K1 runs on the FP64 tensor cores: algorithmic flops = 2 * sum over halos of (samples inside the theta-cut) x
    # (bins the k-range needs), from the per-halo parameters the step just produced
    for name, fl in (("uk_electron", k1_flop), ("uk_pressure", k1p_flop)):
        k = kernels[name]
        if fl > 0 and k["ms"] > 0:
            k.update(alg_flop=fl, tflops=fl / (k["ms"] * 1e-3) / 1e12)
            k["frac_fp64_tensor"] = k["tflops"] / dmma_tf
    k1 = kernels["uk_electron"]
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)     # ncu dram__bytes_read+write per launch of each stage's main kernel (full grid)
    except Exception:
        pass
    dom = max(alg_bytes, key=lambda n: kernels[n]["ms"])
    if dom in ("uk_electron", "uk_pressure"):
        # the transform kernel is launched once (electron) or twice (electron + pressure) per step: the roofline entry
        # is the kernel's AVERAGE launch -- algorithmic flops per launch over the average launch duration
        launches_k1 = [kernels[n] for n in ("uk_electron", "uk_pressure") if kernels[n].get("alg_flop")]
        nl = len(launches_k1)
        fl = sum(k["alg_flop"] for k in launches_k1) / nl
        msl = sum(k["ms"] for k in launches_k1) / nl
        tf = fl / (msl * 1e-3) / 1e12
        roof = {"kernel": "%s (K1, FP64 mma.sync m8n8k4; average of its %d launches per step)" % (
                    "profile_transform_ws_kernel" if mode == 0 else "profile_transform_kernel", nl),
                "bound": "tensor", "achieved": tf, "peak": dmma_tf, "unit": "TFLOP/s", "frac": tf / dmma_tf,
                "peak_source": "FP64 DMMA peak measured in this run (hmv_bench_dmma); MEASURED_PEAKS.json has no FP64 figure",
                "alg_flop_per_launch": fl,
                "hbm_store_frac": kernels["uk_electron"]["frac_hbm"],     # of the launch that stores a cube
                "launches": {n: {"ms": kernels[n]["ms"], "frac": kernels[n]["frac_fp64_tensor"]}
                             for n in ("uk_electron", "uk_pressure") if kernels[n].get("alg_flop")}}
        kernels_dom_ms = msl
    else:
        roof = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": kernels[dom]["frac_hbm"], "peak_source": peak_src, "alg_bytes_per_launch": alg_bytes[dom]}
    roof.update(ms_per_launch=kernels_dom_ms if dom in ("uk_electron", "uk_pressure") else kernels[dom]["ms"],
                traffic=traffic.get(dom) if world == 1 else None,
                fp64_dfma_peak_tflops_measured=fp64_tf, fp64_dmma_peak_tflops_measured=dmma_tf)
    # the HBM-bound kernel of the path, for reference beside the dominant one
    roof["hbm_kernel"] = {"kernel": "power_six_nfw_kernel (K5+K2 fused)" if fused_nfw else "power_six_kernel (K5)", "achieved": kernels["power_six"]["gbs"], "peak": hbm_peak,
                          "unit": "GB/s", "frac": kernels["power_six"]["frac_hbm"],
                          "traffic": traffic.get("power_six") if world == 1 else None}

    # SURVEY 8(d) whole-workload traffic, extended by the tSZ leg: 3 cubes written once; NFW + electron read once by the
    # six-spectra pass, pressure read once by the yy pass; 14 spectra written
    wl_bytes = 8.0 * a.nz * a.nm * a.nk * (4 if tsz_tables else 6) + 2 * NSPEC * 8.0 * a.nz * a.nk + 2.0 * ytab_bytes * world
    roof["workload"] = {"alg_bytes_per_step": wl_bytes, "achieved": wl_bytes / (ms_total / a.steps * 1e-3) / 1e9 / world,
                        "peak": hbm_peak, "unit": "GB/s per GPU",
                        "frac": wl_bytes / (ms_total / a.steps * 1e-3) / 1e9 / world / hbm_peak,
                        "note": ("table mode: the Compton-y profile stays in its bin tables, 2 cubes written + read once; " if tsz_tables else "") +
                                "SURVEY 8(d) algorithmic traffic of the whole step incl. the tSZ leg (3 cubes written + "
                                "read once, 14 spectra) over the step time"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_total / a.steps, "serial_ms_per_step": ms_serial / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "parallelism": "z-sharded x%d" % world,
                       "nfw": "evaluated inside the mass reduction (spectra-only fusion)" if fused_nfw else
                              "cube materialised in HBM",
                       "tsz": "Compton-y profile kept as bin tables, P_yy reduced from them (no third cube)" if tsz_tables else
                              "Compton-y cube materialised",
                       "streams": ("overlap level %d (0: one stream + HOD side stream; 1: sigma^2/n(M)/HOD leg beside the NFW "
                                   "cube; 2: + electron transform and tSZ leg on their own streams), chosen from the slab "
                                   "size; kernels{} and roofline from a second pass with the stages serialised "
                                   "(serial_ms_per_step)") % overlap_level,
                       "l2": "inputs exceed L2 (%s %.1f GB cubes per rank)" % ("two" if tsz_tables else "three", 8e-9 * nzl * nm * ldk)},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d_api * world / a.steps),
                    "d2h_bytes_per_step": int(d2h_api * world / a.steps), "ms_per_step": ms_api / a.steps,
                    "path": "drop-in API: HaloModel -> add_battaglia_profile -> add_battaglia_pres_profile -> "
                            "add_hod(ngal) -> 7x get_power -> C_kk/C_kg/C_yy, numpy in / numpy out",
                    "api_vs_launch_sequence_max_rel": api_vs_launchseq},
            "e2e_launch_sequence": {"value": pts_per_step * a.steps / (ms_pinned * 1e-3), "unit": UNIT,
                                    "ms_per_step": ms_pinned / a.steps, "h2d_bytes_per_step": pin_h2d * world,
                                    "d2h_bytes_per_step": pin_d2h * world,
                                    "path": "pipeline.GridSix through pinned host buffers"},
            "gpu_launches": int(launches * a.steps * world), "clocks": clocks, "roofline": roof, "kernels": kernels,
            "shard_check": shard}

    if world == 1 and not a.no_cpu:
        kind = _reference_kind()
        v, dt = cpu_sample(a, 1, zper=a.cpu_nz, kind=kind)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": kind, "seconds": dt,
                                "sample": "%d of %d redshifts at full %d M x %d k resolution, whole path incl. tSZ and "
                                          "Limber, single numpy thread, %s" % (
                                              a.cpu_nz, a.nz, a.nm, a.nk,
                                              "unmodified reference from oracle/_ref" if kind == "reference" else "oracle port")}
    if dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float64))
        line["dump_outputs"] = {"dir": a.dump_outputs, "arrays": len(dump), "k_columns": int(dump["ks"].size),
                                "bytes": int(sum(v.nbytes for v in dump.values()))}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nz", type=int, default=200)
    ap.add_argument("--nm", type=int, default=2000)
    ap.add_argument("--nk", type=int, default=10000)
    ap.add_argument("--nl", type=int, default=1000)
    ap.add_argument("--cpu-nz", type=int, default=1, help="redshifts in the cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--transform-mode", type=int, default=0, choices=[0, 1],
                    help="K1 launch plan: 0 = persistent kernel (default), 1 = bin-count-class kernels")
    ap.add_argument("--tsz-cube", action="store_true",
                    help="materialise the Compton-y cube (hmv_profile_transform + hmv_power) instead of the table path")
    ap.add_argument("--fused-nfw", action="store_true",
                    help="evaluate the NFW profile inside the mass reduction (hmv_power_six_nfw) instead of writing "
                         "its cube to HBM and reading it back (hmv_uk_nfw + hmv_power_six, the faster default)")
    ap.add_argument("--write-shard-ref", action="store_true",
                    help="(1 GPU) write profiles/r02_shard_reference.json: the C_ell and spectra sums N>1 runs are checked against")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed (the seven P1h/P2h spectra, k-sampled "
                         "to at most 60 MB, and C_kk, C_kg, C_yy) as DIR/<name>.npy, float64")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        # the reference arm times a sample of one-redshift slabs on a thinned mass axis, not the grid itself
        ap.error("--dump-outputs applies to the B200 path (--impl b200)")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
