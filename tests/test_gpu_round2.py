"""Round-2 additions, GPU side (all through the drop-in API / C ABI):
Tinker-2010 mass function (SURVEY 8f-3), generic_profile_fft on caller-supplied samples, device mdelta_from_mdelta,
kappa_2h_profiles (8f-4), the lazily mirrored attributes and the cached six-spectra pass behind get_power."""
import numpy as np
import pytest

from conftest import assert_close, load_golden

pytestmark = pytest.mark.gpu
OSC, HOD_FLOOR = 1e-9, 1e-14


@pytest.fixture(scope="module")
def hm():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback")
    import hmvec_b200
    return hmvec_b200


def test_tinker_mass_function_and_tsz_config(hm):
    """mass_function='tinker', mdef='mean' -- the tSZ notebook's configuration -- against the reference's arrays."""
    g = load_golden("tinker")
    zs = g["zs"]
    h = hm.HaloModel(zs, g["ks"], ms=g["ms"], accuracy='low', mass_function='tinker', mdef='mean')
    assert_close(h.sigma2, g["sigma2"], 1e-9, name="sigma2")
    assert_close(h.nzm, g["nzm"], 1e-6, name="nzm")
    assert_close(h.bh, g["bh"], 1e-9, name="bh")
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    h.add_hod("g", mthresh=10 ** 10.5 + zs * 0.)
    for k in ("Nc", "Ns", "ngal", "bg"):
        assert_close(h.hods["g"][k], g["hod_g_" + k], 1e-6, HOD_FLOOR, name=k)
    for tag, a, b in (("mm", "nfw", "nfw"), ("gg", "g", "g"), ("gm", "g", "nfw"), ("yy", "y", "y"), ("ym", "y", "nfw")):
        assert_close(h.get_power_1halo(a, b), g["P1h_" + tag], 1e-6, name="P1h_" + tag)
        assert_close(h.get_power_2halo(a, b), g["P2h_" + tag], 1e-6, name="P2h_" + tag)
    with pytest.raises(ValueError):          # alpha(z) table ends at z = 3... negative z is outside, as in the reference
        hm.HaloModel(np.array([-0.05, 0.5]), g["ks"], ms=g["ms"], accuracy='low', mass_function='tinker')
    with pytest.raises(NotImplementedError):
        hm.HaloModel(zs, g["ks"], ms=g["ms"], accuracy='low', mass_function='press-schechter')


def test_generic_profile_fft_any_profile(hm):
    """generic_profile_fft with a caller-supplied callable (here an Einasto-like profile with per-halo shape) against
    the oracle's restatement of fft.py:56-115; also the 1-D helpers against the reference's known answer."""
    from oracle import hmvec_oracle as orc
    zs = np.array([0.1, 1.0, 2.2])
    nm = 21                                    # not a multiple of 16: ragged last item
    rss = np.geomspace(0.02, 1.5, nm)[None, :] * (1 + 0.1 * zs[:, None])
    cmaxs = np.linspace(3.0, 9.0, nm)[None, :] + zs[:, None]
    ks = np.geomspace(1e-3, 80., 333)
    al = np.linspace(0.15, 0.3, nm)[None, :, None]
    prof = lambda x: np.exp(-2. / al * (x[None, None, :] ** al - 1.)) * (1 + zs[:, None, None])
    for norm in (True, False):
        kk, u = hm.generic_profile_fft(prof, cmaxs, rss, zs, ks, 30., 3000, do_mass_norm=norm)
        want = orc.profile_transform(prof, cmaxs, rss, zs, ks, 30., 3000, mass_norm=norm)
        assert kk is ks
        assert_close(u, want, 1e-6, OSC, name="generic_profile_fft norm=%s" % norm)
    xs = np.linspace(0., 30., 6001)[1:]
    kt, U = hm.fft_integral(xs, np.exp(-xs ** 2 / 2.))
    g = load_golden("kat")
    assert_close(kt, g["gauss_kt"], 1e-13)
    assert_close(U, g["gauss_U"], 1e-9, 1e-12)
    assert_close(hm.analytic_fft_integral(kt), g["gauss_analytic"], 1e-13)


def test_device_mdelta_and_kappa2h(hm):
    g = load_golden("hostfuncs")
    got = hm.mdelta_from_mdelta(g["ms"], g["C1"], g["d1"], g["d2"])
    assert_close(got, g["mdelta"], 1e-9, name="mdelta_from_mdelta")
    h = hm.HaloModel(g["k2h_zl"], g["k2h_ks"], ms=np.geomspace(1e11, 1e16, 64), accuracy='low', skip_nfw=True)
    k2 = h.kappa_2h_profiles(g["k2h_thetas"], 3e14, 1.1, verbose=False)
    assert_close(k2, g["k2h"], 1e-6, name="kappa_2h_profiles")


def test_lazy_mirrors_and_six_cache(hm, golden_mini):
    g = golden_mini
    zs = g["zs"]
    h = hm.HaloModel(zs, g["ks"], ms=g["ms"], accuracy='low')
    assert not h._hostc                          # nothing has crossed PCIe yet
    h.add_battaglia_profile("electron", family="AGN", xmax=20, nxs=5000)
    h.add_hod("g2", ngal=g["g2_ngal_target"])
    rec = h.hods["g2"]
    assert set(rec.keys()) >= {"Nc", "Ns", "NsNsm1", "NcNs", "ngal", "bg", "log10mthresh", "satellite_profile",
                               "central_profile"}
    assert rec["log10mthresh"].shape == (zs.size, 1) and rec["satellite_profile"] == "nfw"
    assert_close(rec["ngal"], g["g2_ngal_target"], 2e-4)
    # six standard pairs: first request runs hmv_power_six once, the rest are lookups; compare with the generic pair kernel
    pairs = [("nfw", "nfw"), ("electron", "electron"), ("nfw", "electron"), ("g2", "g2"), ("g2", "nfw"), ("electron", "g2")]
    cached = {p: h.get_power(*p) for p in pairs}
    assert len(h._six) == 1
    c1 = h.get_power_1halo("g2", "electron")
    h._six_lookup = lambda *a: None              # force the generic hmv_power path
    for p in pairs:
        assert_close(cached[p], h.get_power(*p), 1e-12, name="six-cache %s x %s" % p)
    assert_close(c1, h.get_power_1halo("g2", "electron"), 1e-12)
    assert_close(cached[("g2", "g2")], g["P1h_g2g2"] + g["P2h_g2g2"], 1e-6)
    assert_close(cached[("electron", "g2")], g["P1h_g2e"] + g["P2h_g2e"], 1e-6)
    del h._six_lookup
    # assigning a mirrored attribute uploads it and drops cached spectra
    P0 = h.get_power("nfw", "nfw")
    h.Pzk = 2.0 * h.Pzk
    P1 = h.get_power("nfw", "nfw")
    p1h = h.get_power_1halo("nfw", "nfw")
    assert_close(P1 - p1h, 2.0 * (P0 - p1h), 1e-9, 1e-12)


def test_device_cubes_validate_user_tensors(hm, golden_mini):
    """ADVICE r1: only float64 contiguous [nz,nm,ldk] tensors on the owner's device are aliased; others are copied."""
    import torch
    g = golden_mini
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    u = h.uk_profiles.device("nfw")
    h.uk_profiles["alias"] = u
    assert h.uk_profiles.device("alias").data_ptr() == u.data_ptr()
    h.uk_profiles["f32"] = u[..., :h._nk].to(torch.float32)
    t = h.uk_profiles.device("f32")
    assert t.dtype == torch.float64 and t.is_contiguous() and tuple(t.shape) == (h._nz, h._nm, h._ldk)
    assert_close(h.get_power("f32", "f32"), h.get_power("nfw", "nfw"), 1e-5)
    h.uk_profiles["view"] = u.permute(0, 1, 2)[..., :h._nk]            # non-contiguous slice of the right shape
    assert_close(h.get_power_1halo("view"), h.get_power_1halo("nfw"), 1e-12)
    with pytest.raises(ValueError):
        h.uk_profiles["bad"] = torch.zeros((h._nz, h._nm + 1, h._ldk), dtype=torch.float64, device=u.device)


def test_transform_table_mode_and_fused_six():
    """hmv_profile_tables + hmv_profile_expand reproduce hmv_profile_transform bit for bit (ragged grid: nm not a
    multiple of 16, odd nk), and hmv_power_six_tab -- the electron profile interpolated from the tables inside the mass
    reduction -- gives the spectra of hmv_power_six on the expanded cube."""
    import torch
    from hmvec_b200 import _capi as capi, pipeline
    zs = np.array([0.1, 1.3, 2.9]); ms = np.geomspace(1e11, 5e15, 41); ks = np.geomspace(1e-3, 30., 333)
    g = pipeline.GridSix(pipeline.make_inputs(zs, ms, ks, ngal=np.array([1e-3, 1e-4, 1e-5])))
    g.upload(); g.run(); torch.cuda.synchronize()
    L, d, ptr, st = capi.lib, g.d, capi.ptr, capi.stream()
    nz, nm, nk, ldk = g.nz, g.nm, g.nk, g.ldk
    E = lambda n: torch.empty(int(n), dtype=torch.float64, device=g.ue.device)
    tab = E(L.hmv_profile_table_doubles(nz, nm, g.nxs))
    capi.check(L.hmv_profile_tables(nz, nm, nk, ptr(d["zs"]), ptr(d["ks"]), g.kmax, ptr(d["rs"]), ptr(d["cmax"]),
                                    ptr(d["xc"]), ptr(d["alpha"]), ptr(d["expo"]), ptr(d["amp"]), ptr(d["oscale"]),
                                    g.gamma, g.xmax, g.nxs, 1, ptr(d["tr_ws"]), ptr(tab), st), "tables")
    cube = torch.zeros_like(g.ue)
    capi.check(L.hmv_profile_expand(nz, nm, nk, ldk, ptr(d["zs"]), ptr(d["ks"]), g.kmax, ptr(d["rs"]), g.xmax, g.nxs,
                                    ptr(d["tr_ws"]), ptr(tab), ptr(cube), st), "expand")
    assert torch.equal(cube[..., :nk], g.ue[..., :nk])
    p1, p2 = torch.zeros(6, nz, nk, dtype=torch.float64, device=cube.device), torch.zeros(6, nz, nk, dtype=torch.float64, device=cube.device)
    ws = E(L.hmv_power_six_tab_ws_doubles(nz, nm, nk))
    capi.check(L.hmv_power_six_tab(nz, nm, nk, ldk, ptr(d["ms"]), ptr(d["ks"]), ptr(d["nzm"]), ptr(d["bh"]), ptr(d["Pzk"]),
                                   g.rho_m0, float(g.p['kstar_damping']), ptr(g.um), ptr(tab), g.nxs, ptr(d["Nc"]),
                                   ptr(d["Ns"]), ptr(d["NcNs"]), ptr(d["NsNsm1"]), ptr(d["ngal"]), ptr(ws), 0, ptr(p1),
                                   ptr(p2), st), "six_tab")
    g1, g2, _, _ = g.spectra()
    for i, tag in enumerate(("mm", "ee", "me", "gg", "gm", "ge")):
        assert_close(p1[i].cpu().numpy(), g1[tag], 1e-12, name="P1h_" + tag)
        assert_close(p2[i].cpu().numpy(), g2[tag], 1e-12, name="P2h_" + tag)


def test_eh98_on_the_device(hm):
    """hmv_eh98_factor (Eisenstein & Hu 1998 on the device, both the oscillating and the no-wiggle form) against the
    host-side factors, which tests/test_host_logic.py pins to the reference's Tk / P_lin_approx."""
    import torch
    c = hm.Cosmology({}, None, accuracy='low')
    ks = np.geomspace(1e-5, 300., 4001)
    zs = np.array([0.0, 0.5, 3.0])
    ks_d = torch.as_tensor(ks, device="cuda")
    for typ in ('eisenhu_osc', 'eisenhu'):
        d2h, vh = c.P_lin_approx_factors(ks, zs, type=typ)
        d2d, vd = c.P_lin_approx_factors_device(ks_d, zs, type=typ)
        assert_close(d2d, d2h, 1e-14, name="growth")
        assert_close(vd.cpu().numpy(), vh, 1e-11, name="EH98 " + typ)


def test_pressure_profile_tables_and_lazy_cube(hm, golden_mini):
    """add_battaglia_pres_profile keeps bin tables: P_yy comes straight from them (hmv_power_tab), the cube appears
    when something asks for it (pk_profiles[name], cross spectra) and then gives the same auto spectrum."""
    g = golden_mini
    h = hm.HaloModel(g["zs"], g["ks"], ms=g["ms"], accuracy='low')
    h.add_battaglia_pres_profile("y", family="pres", xmax=20, nxs=5000)
    tp = h.pk_profiles.tables("y")
    assert tp is not None and tp.cube is None
    p1, p2 = h.get_power_1halo("y", "y"), h.get_power_2halo("y", "y")
    assert tp.cube is None                                   # the auto spectrum did not build the cube
    assert_close(p1, g["P1h_yy"], 1e-6, name="P1h_yy from tables")
    assert_close(p2, g["P2h_yy"], 1e-6, name="P2h_yy from tables")
    assert_close(h.pk_profiles["y"], g["pk_y"], 1e-6, OSC, name="pk_y")      # expands the cube
    assert tp.cube is not None
    assert_close(h.get_power_1halo("y", "y"), p1, 1e-12, name="P1h_yy cube vs tables")
    assert_close(h.get_power_2halo("y", "y"), p2, 1e-12, name="P2h_yy cube vs tables")
    assert_close(h.get_power_1halo("y", "nfw"), g["P1h_ym"], 1e-6, name="P1h_ym")


def test_peer_exchange_on_one_rank_and_wait_timeout():
    """The peer-store exchange (csrc/k_peer.cu) with a single rank whose 'peer' table is its own: hmv_peer_scatter packs
    a_s + b_s into [nrow][nsp][ncol] (odd and even row lengths: scalar and 16-byte stores), publishes the step flag,
    hmv_peer_wait passes; a wait for a flag nobody raises gives up after its timeout with the missing rank in the
    status word instead of hanging, and every later wait returns at once."""
    import ctypes as C
    import time
    import torch
    from hmvec_b200 import _capi as capi
    dev = torch.device("cuda")
    gen = torch.Generator(device="cuda").manual_seed(3)
    for ncol in (130, 37):
        nrow, nsp = 5, 3
        a = [torch.rand((nrow, ncol), dtype=torch.float64, device=dev, generator=gen) for _ in range(nsp)]
        b = [torch.rand((nrow, ncol), dtype=torch.float64, device=dev, generator=gen), None, a[0]]
        out = torch.zeros((nrow + 2, nsp, ncol), dtype=torch.float64, device=dev)          # this rank's rows start at 1
        flags = torch.zeros(16, dtype=torch.int64, device=dev)
        done = torch.zeros(1, dtype=torch.int32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        pa = (C.c_void_p * nsp)(*[t.data_ptr() for t in a])
        pb = (C.c_void_p * nsp)(*[t.data_ptr() if t is not None else None for t in b])
        bufs, flg = (C.c_void_p * 1)(out.data_ptr()), (C.c_void_p * 1)(flags.data_ptr())
        for step in (1, 2):
            capi.check(capi.lib.hmv_peer_scatter(nrow, ncol, nsp, pa, pb, 1, 0, bufs, flg, 1, step,
                                                 C.c_void_p(done.data_ptr()), capi.stream()), "hmv_peer_scatter")
            capi.check(capi.lib.hmv_peer_wait(C.c_void_p(flags.data_ptr()), 1, step, 5.0,
                                              C.c_void_p(status.data_ptr()), capi.stream()), "hmv_peer_wait")
        torch.cuda.synchronize()
        want = torch.stack([a[0] + b[0], a[1], a[2] + a[0]], dim=1)
        assert torch.equal(out[1:1 + nrow], want) and float(out[0].abs().sum()) == 0.0 and float(out[-1].abs().sum()) == 0.0
        assert int(flags[0]) == 2 and int(done[0]) == 0 and int(status[0]) == 0
    # nobody raises flag 1 of a two-rank set: the wait gives up after 0.05 s
    t0 = time.perf_counter()
    capi.check(capi.lib.hmv_peer_wait(C.c_void_p(flags.data_ptr()), 2, 2, 0.05, C.c_void_p(status.data_ptr()),
                                      capi.stream()), "hmv_peer_wait")
    torch.cuda.synchronize()
    assert int(status[0]) == 2 and time.perf_counter() - t0 < 2.0
    t0 = time.perf_counter()
    capi.check(capi.lib.hmv_peer_wait(C.c_void_p(flags.data_ptr()), 2, 3, 30.0, C.c_void_p(status.data_ptr()),
                                      capi.stream()), "hmv_peer_wait")
    torch.cuda.synchronize()
    assert time.perf_counter() - t0 < 1.0, "a wait behind a failed one must return at once"
    with pytest.raises(capi.HmvError):
        capi.check(capi.lib.hmv_peer_scatter(nrow, ncol, 5, pa, pb, 1, 0, bufs, flg, 0, 1,
                                             C.c_void_p(done.data_ptr()), capi.stream()), "hmv_peer_scatter")
