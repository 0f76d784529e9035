"""ctypes binding of libhmvec_b200.so (C ABI declared in include/hmvec_b200.h).

PyTorch is used only to own device memory and to hand out `data_ptr()` / the current stream.  There is NO CPU
fallback: if the shared library has not been built (python -c "import __graft_entry__ as g; g.build()") importing
this module raises, and every entry point raises HmvError on a non-zero return code.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HMV_LIB") or os.path.join(_HERE, "libhmvec_b200.so")   # HMV_LIB: A/B builds of the same ABI

HMV_BISECT_MAXIT = 64
HMV_BISECT_ROUND1 = 24      # iterations of the first bisection round (rtol 1e-4 on [7,14] needs ~19)


class HmvError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "hmvec_b200: %s not found. The CUDA extension is the only compute path (no CPU fallback); build it with\n"
        "    python -c 'import __graft_entry__ as g; g.build()'   (or: make -C hmvec_b200/csrc)" % LIB_PATH)

lib = C.CDLL(LIB_PATH)

_p = C.c_void_p
_i = C.c_int
_d = C.c_double
_ll = C.c_longlong


class Tracer(C.Structure):
    """struct hmv_tracer (include/hmvec_b200.h)"""
    _fields_ = [("kind", _i), ("us_d", _p), ("uc_d", _p), ("Nc_d", _p), ("Ns_d", _p), ("NcNs_d", _p),
                ("NsNsm1_d", _p), ("ngal_d", _p), ("bias_d", _p)]


class LimberJob(C.Structure):
    """struct hmv_limber_job (include/hmvec_b200.h)"""
    _fields_ = [("P_d", _p), ("P2_d", _p), ("ngz", _i), ("gzs_d", _p), ("pref_d", _p), ("chis_d", _p), ("cl_d", _p)]


_SIGS = {
    "hmv_abi_version": (_i, []),
    "hmv_last_error": (C.c_char_p, []),
    "hmv_device_cc": (_i, [_i]),
    "hmv_sigma2_ws_doubles": (_ll, [_i, _i, _i]),
    "hmv_sigma2": (_i, [_i, _i, _i, _p, _p, _p, _p, _d, _p, _p, _p]),
    "hmv_mass_function": (_i, [_i, _i, _p, _p, _d, _d, _d, _d, _d, _p, _p, _p]),
    "hmv_mass_function_tinker": (_i, [_i, _i, _p, _p, _d, _d, _p, _p, _p, _p]),
    "hmv_halo_geometry": (_i, [_i, _i, _p, _p, _p, _d, _d, _d, _d, _p, _p, _p]),
    "hmv_mdelta": (_i, [_i, _i, _p, _p, _p, _p, _p, _p]),
    "hmv_uk_nfw_ws_doubles": (_ll, [_i, _i, _i]),
    "hmv_uk_nfw": (_i, [_i, _i, _i, _i, _p, _p, _d, _p, _p, _p, _p, _p]),
    "hmv_gnfw_params": (_i, [_i, _i, _i, _p, _p, _p, _p, _p, C.POINTER(_d), _d, _d, _d, _d,
                             _p, _p, _p, _p, _p, _p, _p, _p]),
    "hmv_profile_transform_ws_doubles": (_ll, [_i, _i, _i]),
    "hmv_set_transform_mode": (_i, [_i]),
    "hmv_eh98_factor": (_i, [_i, _p, _d, _d, _d, _d, _i, _d, _d, _d, _p, _p]),
    "hmv_profile_table_stride": (_ll, [_i]),
    "hmv_profile_table_doubles": (_ll, [_i, _i, _i]),
    "hmv_profile_tables": (_i, [_i, _i, _i, _p, _p, _d, _p, _p, _p, _p, _p, _p, _p, _d, _d, _i, _i, _p, _p, _p]),
    "hmv_profile_expand": (_i, [_i, _i, _i, _i, _p, _p, _d, _p, _d, _i, _p, _p, _p, _p]),
    "hmv_power_tab": (_i, [_i, _i, _i, _p, _p, _p, _p, _p, _d, _d, _i, _p, _i, _p, _p, _p, _p]),
    "hmv_power_six_tab_ws_doubles": (_ll, [_i, _i, _i]),
    "hmv_power_six_tab": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, _d, _p, _p, _i, _p, _p, _p, _p, _p, _p, _ll, _p, _p, _p]),
    "hmv_set_nfw_mode": (_i, [_i]),
    "hmv_profile_transform": (_i, [_i, _i, _i, _i, _p, _p, _d, _p, _p, _p, _p, _p, _p, _p, _d, _d, _i, _i, _p, _p, _p]),
    "hmv_profile_transform_samples": (_i, [_i, _i, _i, _i, _p, _p, _d, _p, _p, _p, _p, _d, _i, _i, _p, _p, _p]),
    "hmv_hod": (_i, [_i, _i, _p, _p, _p, C.POINTER(_d), _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "hmv_hod_bisect": (_i, [_i, _i, _p, _p, _p, _p, C.POINTER(_d), _d, _d, _d, _i, _i, _p, _p, _p]),
    "hmv_hod_pick": (_i, [_i, _p, _p, _d, _p, _p, _p]),
    "hmv_hod_solve": (_i, [_i, _i, _p, _p, _p, _p, C.POINTER(_d), _d, _d, _d, _d, _p, _p, _p, _p]),
    "hmv_power_ws_doubles": (_ll, [_i, _i]),
    "hmv_power": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, _d, C.POINTER(Tracer), C.POINTER(Tracer), _p, _p, _p, _p]),
    "hmv_power_six": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, _d, _p, _p, _p, _p, _p, _p, _p, _p, _ll, _p, _p, _p]),
    "hmv_power_six_nfw_ws_doubles": (_ll, [_i, _i]),
    "hmv_power_six_nfw": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _d, _d, _p, _p, _p, _p, _p, _p, _p, _p, _p, _ll,
                               _p, _p, _p]),
    "hmv_limber": (_i, [_i, _p, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p, _p, _p, _p]),
    "hmv_limber_multi": (_i, [_i, C.POINTER(LimberJob), _i, _p, _i, _i, _i, _p, _p, _p]),
    "hmv_trispec_1h_ws_doubles": (_ll, [_i, _i, _i, _i]),
    "hmv_trispec_1h": (_i, [_i, _i, _i, _i, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p, _p, _p]),
    "hmv_cl_cov_1h_ws_doubles": (_ll, [_i, _i, _i, _i]),
    "hmv_cl_cov_1h": (_i, [_i, _i, _i, _i, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p, _p, _p,
                           _p, _p, _p]),
    "hmv_trispec_1h_tracers_ws_doubles": (_ll, [_i, _i, _i, _i, C.POINTER(Tracer)]),
    "hmv_trispec_1h_tracers": (_i, [_i, _i, _i, _i, _p, _p, _p, _d, C.POINTER(Tracer), _i, _p, _i, _p, _p, _p, _p]),
    "hmv_cl_cov_1h_tracers_ws_doubles": (_ll, [_i, _i, _i, _i, C.POINTER(Tracer)]),
    "hmv_cl_cov_1h_tracers": (_i, [_i, _i, _i, _i, _p, _p, _p, _d, C.POINTER(Tracer), _i, _p, _i, _p, _p, _p, _p, _p,
                                   _p, _p]),
    "hmv_trispec_2h_ws_doubles": (_ll, [_i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_i), _i]),
    "hmv_trispec_2h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _i,
                            _p, _p, _p]),
    "hmv_cl_cov_2h_ws_doubles": (_ll, [_i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_i), _i]),
    "hmv_cl_cov_2h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p,
                           _p, _p, _i, _p, _p, _p]),
    "hmv_trispec_3h_ws_doubles": (_ll, [_i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_i), _i]),
    "hmv_trispec_3h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _i,
                            _p, _p, _p]),
    "hmv_cl_cov_3h_ws_doubles": (_ll, [_i, _i, _i, _i, _i, C.POINTER(_p), C.POINTER(_i), _i]),
    "hmv_cl_cov_3h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p,
                           _p, _p, _i, _p, _p, _p]),
    "hmv_trispec_4h_ws_doubles": (_ll, [_i, _i, _i, _i]),
    "hmv_trispec_4h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p,
                            _p, _p]),
    "hmv_cl_cov_4h_ws_doubles": (_ll, [_i, _i, _i, _i]),
    "hmv_cl_cov_4h": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, C.POINTER(_p), C.POINTER(_i), _i, _p, _i, _p, _p,
                           _p, _p, _p, _p, _p]),
    "hmv_power_response": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _d, _p, _i, _p, _i, _p, _p, _p, _p]),
    "hmv_sigma_b2": (_i, [_i, _i, _p, _p, _p, _p, _p, _p]),
    "hmv_cl_cov_ssc_ws_doubles": (_ll, [_i, _i, _i]),
    "hmv_cl_cov_ssc": (_i, [_i, _i, _p, _p, _p, _i, _p, _i, _p, _p, _p, _p, _p, _p, _p]),
    "hmv_ksz_nvv_integral": (_i, [_i, _i, _p, _p, _ll, _p, _ll, _p, _ll, _p, _p, _p]),
    "hmv_pack_sum": (_i, [_i, _i, _i, C.POINTER(_p), C.POINTER(_p), _p, _p]),
    "hmv_peer_alloc": (_i, [_ll, C.POINTER(_p), C.c_char_p]),
    "hmv_peer_open": (_i, [C.c_char_p, C.POINTER(_p)]),
    "hmv_peer_close": (_i, [_p]),
    "hmv_peer_free": (_i, [_p]),
    "hmv_peer_scatter": (_i, [_i, _i, _i, C.POINTER(_p), C.POINTER(_p), _i, _i, C.POINTER(_p), C.POINTER(_p), _ll,
                              C.c_ulonglong, _p, _p]),
    "hmv_peer_wait": (_i, [_p, _i, C.c_ulonglong, _d, _p, _p]),
    "hmv_debug_k1_order": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "hmv_debug_wave_tile": (_i, [_i, _i]),
    "hmv_debug_tab_order": (_i, [_i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "hmv_pk_spline": (_i, [_i, _i, _p, _p, _i, _i, _i, _i, _p, _p, _p, _i, _d, _p, _p]),
    "hmv_outer": (_i, [_i, _i, _p, _p, _p, _p]),
    "hmv_sum2": (_i, [_ll, _p, _p, _p, _p]),
    "hmv_bench_dfma": (_d, [_i, _p]),
    "hmv_bench_dmma": (_d, [_i, _p]),
    "hmv_bench_copy": (_d, [_p, _p, _ll, _i, _p]),
    "hmv_sici_test": (_i, [_i, _p, _p, _p, _p]),
}

for _name, (_res, _args) in _SIGS.items():
    _f = getattr(lib, _name)      # AttributeError here == header/library mismatch: fail loudly
    _f.restype = _res
    _f.argtypes = _args

EXPORTS = tuple(_SIGS)


def last_error():
    return lib.hmv_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise HmvError("%s failed (code %d): %s" % (what, rc, last_error()))


def ptr(t):
    """Device pointer of a contiguous float64 (or int32) CUDA tensor; None -> NULL."""
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise HmvError("expected a CUDA tensor, got %r" % (type(t),))
    if not t.is_contiguous():
        raise HmvError("tensor must be contiguous")
    if t.dtype not in (torch.float64, torch.int32):
        raise HmvError("tensor must be float64 (or int32), got %s" % t.dtype)
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def darr(vals):
    return (C.c_double * len(vals))(*[float(v) for v in vals])


# ---- host<->device copy accounting (bench.py reports the bytes the API moved per step) ----------------------------
_copied = [0, 0]


def count_h2d(nbytes):
    _copied[0] += int(nbytes)


def count_d2h(nbytes):
    _copied[1] += int(nbytes)


def reset_copy_counters():
    _copied[0] = _copied[1] = 0


def copy_counters():
    return tuple(_copied)

