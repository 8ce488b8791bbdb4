"""ctypes binding of libproxtv_b200.so (the C ABI declared in include/proxtv_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C proxtv_b200/csrc``.  There is no CPU fallback:
if the shared object is missing, or no CUDA device is usable when a compute entry point is called, this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libproxtv_b200.so")

_dp = C.POINTER(C.c_double)
_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)
_vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/proxtv_b200.h one to one (tests/test_abi.py checks the header against this)
SIGNATURES = {
    # Part 1: drop-in symbols (src/TVopt.h:88-141)
    "hybridTautString_TV1": (None, [_vp, C.c_int, C.c_double, _vp]),
    "hybridTautString_TV1_custom": (None, [_vp, C.c_int, C.c_double, _vp, C.c_double]),
    "classicTautString_TV1": (C.c_int, [_vp, C.c_int, C.c_double, _vp]),
    "linearizedTautString_TV1": (C.c_int, [_vp, C.c_double, _vp, C.c_int]),
    "TV1D_denoise": (None, [_vp, _vp, C.c_int, C.c_double]),
    "tautString_TV1_Weighted": (C.c_int, [_vp, _vp, _vp, C.c_int]),
    "PN_TV1": (C.c_int, [_vp, C.c_double, _vp, _vp, C.c_int, C.c_double, _vp]),
    "PN_TV1_Weighted": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_double, _vp]),
    "TV1D_denoise_tautstring": (None, [_vp, _vp, C.c_int, C.c_double]),
    "SolveTVConvexQuadratic_a1_nw": (None, [C.c_int, _vp, C.c_double, _vp]),
    "SolveTVConvexQuadratic_a1": (None, [C.c_int, _vp, _vp, _vp]),
    "dp": (None, [C.c_int, _vp, C.c_double, _vp]),
    "TV": (C.c_int, [_vp, C.c_double, _vp, _vp, C.c_int, C.c_double, _vp]),
    "DR2_TV": (C.c_int, [C.c_size_t, C.c_size_t, _vp, C.c_double, C.c_double, C.c_double, C.c_double, _vp, C.c_int,
                         C.c_int, _vp]),
    "DR2L1W_TV": (C.c_int, [C.c_size_t, C.c_size_t, _vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "PD2_TV": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "PD_TV": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    "PDR_TV": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int]),
    # Part 2: extensions
    "proxtv_device_count": (C.c_int, []),
    "proxtv_last_error": (C.c_char_p, []),
    "proxtv_version": (C.c_char_p, []),
    "proxtv_set_engine": (C.c_int, [C.c_int]),
    "proxtv_prox_fibers_dev_f64": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_double, _vp, _vp]),
    "proxtv_prox_fibers_dev_f32": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_float, _vp, _vp]),
    "proxtv_prox_fibers_f64": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_double, _vp]),
    "proxtv_prox_fibers_f32": (C.c_int, [_vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_float, _vp]),
    "proxtv_DR2_TV_dev_f64": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, C.c_int, _vp, C.c_double, C.c_double, _vp, C.c_int, _vp, _vp]),
    "proxtv_DR2_TV_dev_f32": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, C.c_int, _vp, C.c_float, C.c_float, _vp, C.c_int, _vp, _vp]),
    "proxtv_DR2L1W_TV_dev_f64": (C.c_int, [C.c_size_t, C.c_size_t, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp]),
    "proxtv_DR2L1W_TV_dev_f32": (C.c_int, [C.c_size_t, C.c_size_t, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp]),
    "proxtv_DR2_TV_batched_f64": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, _vp, C.c_double, C.c_double, _vp, C.c_int, _vp]),
    "proxtv_DR2_TV_batched_f32": (C.c_int, [C.c_size_t, C.c_size_t, C.c_int, _vp, C.c_float, C.c_float, _vp, C.c_int, _vp]),
    "proxtv_PD2_TV_dev_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_PD2_TV_dev_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_PD_TV_dev_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_PD_TV_dev_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_PD_TV_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int]),
    "proxtv_PDR_TV_dev_f64": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_PDR_TV_dev_f32": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "proxtv_lane_prox_dev_f64": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_double, _vp]),
    "proxtv_lane_prox_dev_f32": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_float, _vp]),
    "proxtv_lane_prox2_dev_f64": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_double, _vp]),
    "proxtv_lane_prox2_dev_f32": (C.c_int, [C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_longlong, C.c_int, C.c_longlong, C.c_float, _vp]),
    "proxtv_lane_tuning": (None, [C.c_int, C.c_int, C.c_int]),
    "proxtv_lane_stats": (C.c_ulonglong, [C.c_int]),
    "proxtv_lane_guard_last": (C.c_int, []),
    "proxtv_lane_tasklog": (None, [_vp, C.c_longlong]),
    "proxtv_profile_enable": (None, [C.c_int]),
    "proxtv_profile_reset": (None, []),
    "proxtv_profile_read": (None, [_vp, _vp, _vp]),
    "proxtv_host_alloc": (_vp, [C.c_size_t]),
    "proxtv_host_free": (None, [_vp]),
    "proxtv_release_workspace": (None, []),
}

_lib = None


class ProxTVError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises ProxTVError if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ProxTVError(
            "proxtv_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C proxtv_b200/csrc` (there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def require_device():
    lib = load()
    if lib.proxtv_device_count() <= 0:
        raise ProxTVError("proxtv_b200: no usable CUDA device; the B200 path has no CPU fallback")
    return lib


def last_error():
    return load().proxtv_last_error().decode()
