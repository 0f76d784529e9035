"""The C-ABI library loads and exports every symbol include/hmvec_b200.h declares (no compute calls: CPU-only)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HMV_E_ARG, HMV_E_LIMIT = -1, -3             # include/hmvec_b200.h


def _declared():
    src = open(os.path.join(ROOT, "include", "hmvec_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hmv_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported():
    names = _declared()
    assert len(names) >= 20
    lib = ctypes.CDLL(os.path.join(ROOT, "hmvec_b200", "libhmvec_b200.so"))
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, "declared in include/hmvec_b200.h but not exported: %s" % missing


def test_binding_covers_header_and_reports_errors():
    from hmvec_b200 import _capi as capi
    assert set(_declared()) == set(capi.EXPORTS)
    assert capi.lib.hmv_abi_version() == 1
    # argument validation happens before any CUDA call, so it can be exercised without a GPU
    assert capi.lib.hmv_power_ws_doubles(0, 5) == 0
    assert capi.lib.hmv_sigma2_ws_doubles(4, 64, 1000) >= 64 * 1000
    rc = capi.lib.hmv_limber(0, None, 1, 2, 2, None, None, None, None, 1, None, None, None, None, None)
    assert rc == -1 and "bad sizes" in capi.last_error()
    rc = capi.lib.hmv_hod(3, 10, None, None, None, None, 0, None, None, None, None, None, None, None, None, None)
    assert rc == -1 and "null pointer" in capi.last_error()


def test_k5_rejects_before_any_launch():
    """Every argument and limit check of the mass-integral entry points runs before their first launch: with valid-
    looking dummy device pointers and no GPU, a rejected call returns its own error, never a CUDA one."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    ptr = [ctypes.c_void_p(0x10000 + 0x100 * i) for i in range(16)]     # non-null, 16-byte aligned, never dereferenced
    nz, nm, nk, ldk = 2, 40, 30, 32
    t = capi.Tracer()
    t.kind = 0
    t.us_d = 0x20008                                                     # misaligned cube
    rc = L.hmv_power(nz, nm, nk, ldk, *ptr[:5], 1.0, 1.0, ctypes.byref(t), ctypes.byref(t), *ptr[5:8], None)
    assert rc == HMV_E_ARG and "16-byte aligned" in capi.last_error()
    rc = L.hmv_power_six(nz, nm, nk, ldk, *ptr[:5], 1.0, 1.0, *ptr[5:13], nz * nk - 1, *ptr[13:15], None)
    assert rc == HMV_E_ARG and "hmv_power_six: spec_stride" in capi.last_error()
    rc = L.hmv_power_six_tab(nz, nm, nk, ldk, *ptr[:5], 1.0, 1.0, *ptr[5:7], 64, *ptr[7:13], nz * nk - 1,
                             *ptr[13:15], None)
    assert rc == HMV_E_ARG and "hmv_power_six_tab: spec_stride" in capi.last_error()
    rc = L.hmv_power_tab(nz, 4000, nk, *ptr[:5], 1.0, 1.0, 2, ptr[5], 64, *ptr[6:9], None)
    assert rc == HMV_E_LIMIT and "shared memory" in capi.last_error()


def test_k1_rejects_before_any_launch():
    """The transform has one launch plan, selected by mode 0 alone, and its four entry points all read ks, the workspace
    and the cube or tables with 16-byte accesses: a misaligned pointer or an odd ldk is refused before the first
    launch (dummy device pointers, no GPU), never routed to another kernel."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    assert L.hmv_set_transform_mode(0) == 0
    assert L.hmv_set_transform_mode(1) == HMV_E_ARG
    ptr = [ctypes.c_void_p(0x10000 + 0x100 * i) for i in range(12)]     # non-null, 16-byte aligned, never dereferenced
    bad = ctypes.c_void_p(0x20008)                                       # misaligned
    nz, nm, nk, nxs = 2, 40, 30, 5000
    calls = {
        "transform, odd ldk": lambda: L.hmv_profile_transform(nz, nm, nk, 31, ptr[0], ptr[1], 1.0, *ptr[2:9], 1.0,
                                                              20.0, nxs, 1, ptr[9], ptr[10], None),
        "transform, misaligned ks": lambda: L.hmv_profile_transform(nz, nm, nk, 32, ptr[0], bad, 1.0, *ptr[2:9], 1.0,
                                                                    20.0, nxs, 1, ptr[9], ptr[10], None),
        "tables, misaligned ws": lambda: L.hmv_profile_tables(nz, nm, nk, ptr[0], ptr[1], 1.0, *ptr[2:9], 1.0, 20.0,
                                                              nxs, 1, bad, ptr[10], None),
        "expand, misaligned ws": lambda: L.hmv_profile_expand(nz, nm, nk, 32, ptr[0], ptr[1], 1.0, ptr[2], 20.0, nxs,
                                                              bad, ptr[3], ptr[4], None),
        "samples, misaligned ws": lambda: L.hmv_profile_transform_samples(nz, nm, nk, 32, ptr[0], ptr[1], 1.0,
                                                                          *ptr[2:6], 20.0, nxs, 1, bad, ptr[6], None),
    }
    for what, call in calls.items():
        rc = call()
        assert rc == HMV_E_ARG and "16-byte aligned" in capi.last_error(), (what, rc, capi.last_error())


def test_k2_rejects_before_any_launch():
    """The analytic NFW profile has one evaluation, selected by mode 0 alone, and hmv_uk_nfw moves 16-byte words of
    the cube and the workspace: an odd ldk or a misaligned cube or workspace is refused before the first launch (dummy
    device pointers, no GPU), never routed to another kernel."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("dummy device pointers must never reach a launch on a GPU")
    from hmvec_b200 import _capi as capi
    L = capi.lib
    assert L.hmv_set_nfw_mode(0) == 0
    assert L.hmv_set_nfw_mode(1) == HMV_E_ARG
    ptr = [ctypes.c_void_p(0x10000 + 0x100 * i) for i in range(6)]      # non-null, 16-byte aligned, never dereferenced
    bad = ctypes.c_void_p(0x20008)                                       # misaligned
    nz, nm, nk = 2, 40, 30
    zs, ks, cs, rvir, ws, uk = ptr
    calls = {
        "odd ldk": lambda: L.hmv_uk_nfw(nz, nm, nk, 31, zs, ks, 1.0, cs, rvir, ws, uk, None),
        "misaligned uk": lambda: L.hmv_uk_nfw(nz, nm, nk, 32, zs, ks, 1.0, cs, rvir, ws, bad, None),
        "misaligned ws": lambda: L.hmv_uk_nfw(nz, nm, nk, 32, zs, ks, 1.0, cs, rvir, bad, uk, None),
    }
    for what, call in calls.items():
        rc = call()
        assert rc == HMV_E_ARG and "16-byte aligned" in capi.last_error(), (what, rc, capi.last_error())


def test_no_cpu_fallback_in_product():
    """The product package must not import the oracle (or the reference) anywhere."""
    pkg = os.path.join(ROOT, "hmvec_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            txt = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in txt.replace("test-side oracle", ""), fn
            assert "/root/reference" not in txt, fn
