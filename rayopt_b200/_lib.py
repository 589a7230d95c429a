"""ctypes binding of librtx.so (include/rtx.h).  No CPU fallback: importing
this module without the built library raises; using it without a CUDA device
raises at context creation."""
import ctypes as C
import os


from .surface_table import SURFACE_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librtx.so")

RTX_F64, RTX_F32 = 0, 1
RTX_KEEP_ALL, RTX_KEEP_LAST = 0, 1
RTX_EXACT, RTX_STORE_DIRECT, RTX_RPT1, RTX_RPT2, RTX_GATHER_XY = 1, 2, 4, 8, 16

# every symbol include/rtx.h declares: name -> (restype, argtypes)
_vp, _i, _i64, _sz, _u = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_uint
_pp = C.POINTER(C.c_void_p)
SYMBOLS = {
    "rtx_abi_version": (_i, []),
    "rtx_sizeof_surface": (_sz, []),
    "rtx_sizeof_aim": (_sz, []),
    "rtx_sizeof_opd": (_sz, []),
    "rtx_device_count": (_i, []),
    "rtx_strerror": (C.c_char_p, [_i]),
    "rtx_surface_finalize": (_i, [_vp, _i, _vp]),
    "rtx_init": (_i, [_i, _pp]),
    "rtx_free": (_i, [_vp]),
    "rtx_sync": (_i, [_vp]),
    "rtx_device_info": (_i, [_vp, C.POINTER(_i), C.POINTER(_sz), C.POINTER(_sz),
                            C.c_char_p, _i]),
    "rtx_malloc": (_i, [_vp, _sz, _pp]),
    "rtx_free_device": (_i, [_vp, _vp]),
    "rtx_host_alloc": (_i, [_vp, _sz, _pp]),
    "rtx_host_free": (_i, [_vp, _vp]),
    "rtx_memcpy_h2d": (_i, [_vp, _vp, _vp, _sz]),
    "rtx_memcpy_d2h": (_i, [_vp, _vp, _vp, _sz]),
    "rtx_memcpy_d2d": (_i, [_vp, _vp, _vp, _sz]),
    "rtx_numa_bind": (_i, [_vp, _i, C.POINTER(_i)]),
    "rtx_memcpy2d_d2h": (_i, [_vp, _vp, _sz, _vp, _sz, _sz, _sz]),
    "rtx_memset": (_i, [_vp, _vp, _i, _sz]),
    "rtx_timer_start": (_i, [_vp]),
    "rtx_timer_stop": (_i, [_vp, C.POINTER(C.c_float)]),
    "rtx_last_kernel_ms": (_i, [_vp, C.POINTER(C.c_float)]),
    "rtx_launch_count": (_i64, [_vp]),
    "rtx_trace": (_i, [_vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _i, _i, _i64,
                       _vp, _vp, _vp, _vp, _u]),
    "rtx_trace_batch": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i64,
                             _vp, _vp, _vp, _vp, _u]),
    "rtx_trace_batch_host": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i,
                                  _vp, _vp, _vp, _vp, _u]),
    "rtx_set_mask_output": (_i, [_vp, _vp]),
    "rtx_set_path_sum_output": (_i, [_vp, _vp, _i]),
    "rtx_trace_host": (_i, [_vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _i, _i,
                            _vp, _vp, _vp, _vp, _u]),
    "rtx_moments": (_i, [_vp, _i, _i64, _vp, _vp, _vp, _vp]),
    "rtx_trace_reduce": (_i, [_vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _i, _vp, _vp, _vp, _u]),
    "rtx_trace_opd": (_i, [_vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _i, _vp, _vp, _vp, _u]),
    "rtx_selftest_math": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "rtx_aim_infinite": (_i, [_vp, _i, _i64, _vp, _i, _vp, C.c_double, _vp, _vp]),
    "rtx_aim_finite": (_i, [_vp, _i, _i64, _vp, _i, _vp, C.c_double, C.c_double, _vp, _vp]),
    "rtx_aim_plan": (_i, [_vp, _vp, _i64, _vp, C.POINTER(_i64)]),
    "rtx_aim_rays": (_i, [_vp, _vp, _i64, _vp, _i, _i64, _i64, _vp, _vp, _vp]),
    "rtx_focus_moments": (_i, [_vp, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "rtx_ipc_export": (_i, [_vp, _vp, _vp]),
    "rtx_ipc_open": (_i, [_vp, _vp, _pp]),
    "rtx_ipc_close": (_i, [_vp, _vp]),
    "rtx_trace_gather": (_i, [_vp, _vp, _i, _vp, _i, _i64, _vp, _vp, _i, _i, _vp, _vp, _i64,
                              _u]),
    "rtx_opd_regrid": (_i, [_vp, _i64, _vp, _vp, C.c_double, _vp, C.c_double, _i, _i64, _vp,
                            _vp, _vp]),
    "rtx_psf": (_i, [_vp, _i64, _vp, _i, _vp]),
    "rtx_psf_lines": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "rtx_psf_encircled": (_i, [_vp, _i64, _vp, C.c_double, C.c_double, _i64, _vp]),
    "rtx_psf_mtf": (_i, [_vp, _i64, _vp, _vp]),
    "rtx_psf_window": (_i, [_vp, _i64, _vp, _i64, _i64, _i64, _vp]),
}

_lib = None


class RtxError(RuntimeError):
    pass


def load():
    """dlopen librtx.so and bind every symbol (raises if missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RtxError(
            "%s not built: run `python -m rayopt_b200.build` (needs nvcc). "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.rtx_sizeof_surface() != SURFACE_DTYPE.itemsize:
        raise RtxError("rtx_surface layout mismatch: C %d, numpy %d" % (
            lib.rtx_sizeof_surface(), SURFACE_DTYPE.itemsize))
    from .rays import aim_dtype
    if lib.rtx_sizeof_aim() != aim_dtype().itemsize:
        raise RtxError("rtx_aim layout mismatch: C %d, numpy %d" % (
            lib.rtx_sizeof_aim(), aim_dtype().itemsize))
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().rtx_strerror(code)
        raise RtxError("rtx error %d: %s" % (code, msg.decode() if msg else "?"))


def ptr(a):
    """void* of a numpy array (or None)"""
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)
