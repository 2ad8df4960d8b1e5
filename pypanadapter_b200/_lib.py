"""ctypes binding of the C ABI in include/zoomfft_b200.h.

The product library is ``pypanadapter_b200/libzoomfft_b200.so`` (built in-tree
by ``pypanadapter_b200/build.py`` with nvcc for sm_100a).  There is no CPU
fallback: if the library is missing, or no CUDA device is present, loading /
engine creation raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libzoomfft_b200.so"
LIB_PATH = os.path.join(HERE, LIB_NAME)

ZFB_OK = 0
ZFB_EINVAL = -22
ZFB_ENOMEM = -12
ZFB_ENODEV = -19
ZFB_ECUDA = -5
ZFB_ESTATE = -1
ZFB_ETOOSHORT = -34

ZFB_DTYPE_C64 = 0
ZFB_DTYPE_U8 = 1
ZFB_DTYPE_CS16 = 2
ZFB_MODE_EXACT = 0
ZFB_MODE_FAST = 1
FAST_MAX_STAGES = 12
ZFB_FLAG_NO_LO = 1
ZFB_FLAG_LINEAR = 2
ZFB_FLAG_ONESIDED = 4

ABI_VERSION = 3
PROF_CLASSES = 21
ZFB_IMAGE_F32 = 0
ZFB_IMAGE_U8 = 1
ZFB_IMAGE_RGBA = 2
ZFB_TRACE_LAST = 0
ZFB_TRACE_MAX = 1
ZFB_TRACE_MIN = 2
ZFB_TRACE_AVG = 3


class ZfbConfig(C.Structure):
    """struct zfb_config (include/zoomfft_b200.h)."""
    _fields_ = [
        ("fs", C.c_double),
        ("fft_size", C.c_int32),
        ("fft_ratio", C.c_int32),
        ("frame_len", C.c_int32),
        ("row_width", C.c_int32),
        ("nperseg", C.c_int32),
        ("dtype", C.c_int32),
        ("flip", C.c_int32),
        ("mode", C.c_int32),
        ("flags", C.c_int32),
        ("f_demod", C.c_double),
        ("ema_alpha", C.c_double),
        ("window", C.POINTER(C.c_double)),
    ]


class ZfbFastPlan(C.Structure):
    """struct zfb_fast_plan (include/zoomfft_b200.h)."""
    _fields_ = [
        ("nstages", C.c_int32),
        ("half", C.c_int32 * FAST_MAX_STAGES),
        ("taps", C.POINTER(C.c_double) * FAST_MAX_STAGES),
        ("comp_half", C.c_int32),
        ("comp_taps", C.POINTER(C.c_double)),
        ("strip", C.c_int32),
    ]


# every symbol the header declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "zfb_abi_version": (C.c_int, []),
    "zfb_build_kind": (C.c_char_p, []),
    "zfb_source_hash": (C.c_char_p, []),
    "zfb_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "zfb_destroy": (None, [_P]),
    "zfb_last_error": (C.c_char_p, [_P]),
    "zfb_configure": (C.c_int, [_P, C.POINTER(ZfbConfig)]),
    "zfb_set_fast_plan": (C.c_int, [_P, C.POINTER(ZfbFastPlan)]),
    "zfb_fast_active": (C.c_int, [_P]),
    "zfb_set_stream": (C.c_int, [_P, _P]),
    "zfb_set_group": (C.c_int, [_P, C.c_int]),
    "zfb_reset_ema": (C.c_int, [_P]),
    "zfb_set_option": (C.c_int, [_P, C.c_char_p, C.c_longlong]),
    "zfb_slab_lanes": (C.c_int, [_P]),
    "zfb_join": (C.c_int, [_P, _P]),
    "zfb_process_device": (C.c_int, [_P, _P, C.c_int, _P]),
    "zfb_process_host": (C.c_int, [_P, _P, C.c_int, _P]),
    "zfb_process_channels_device": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_double), C.c_int, _P]),
    "zfb_process_channels_host": (C.c_int, [_P, _P, C.c_int, C.POINTER(C.c_double), C.c_int, _P]),
    "zfb_synchronize": (C.c_int, [_P]),
    "zfb_debug_read_decimated": (C.c_int, [_P, _P, C.c_int]),
    "zfb_ring_configure": (C.c_int, [_P, C.c_int]),
    "zfb_ring_configure_width": (C.c_int, [_P, C.c_int, C.c_int]),
    "zfb_ring_width": (C.c_int, [_P]),
    "zfb_ring_rows_written": (C.c_int64, [_P]),
    "zfb_read_rows": (C.c_int, [_P, C.c_int, C.c_int, _P]),
    "zfb_ring_push_rows": (C.c_int, [_P, _P, C.c_int]),
    "zfb_traces_enable": (C.c_int, [_P, C.c_int]),
    "zfb_traces_reset": (C.c_int, [_P]),
    "zfb_traces_count": (C.c_int64, [_P]),
    "zfb_trace_read": (C.c_int, [_P, C.c_int, C.POINTER(C.c_float)]),
    "zfb_trace_peaks": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int32),
                                  C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "zfb_find_peaks_device": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int32),
                                        C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "zfb_ring_image": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_double, C.c_double, _P, _P, C.c_int]),
    "zfb_ring_quantiles": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_double), C.c_int,
                                     C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "zfb_taper_design": (C.c_int, [_P, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "zfb_taper_preview": (C.c_int, [_P, C.POINTER(C.c_double), C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "zfb_samples_create": (C.c_int, [_P, C.c_int64, C.c_int]),
    "zfb_samples_host_ptr": (_P, [_P]),
    "zfb_samples_begin_write": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "zfb_samples_commit": (C.c_int, [_P, C.c_int64, C.c_int64]),
    "zfb_samples_process": (C.c_int, [_P, _P]),
    "zfb_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "zfb_free_pinned": (C.c_int, [_P]),
    "zfb_decim_sos": (C.c_int, [C.POINTER(C.c_double)]),
    "zfb_plan_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "zfb_get_counters": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "zfb_set_profiling": (C.c_int, [_P, C.c_int]),
    "zfb_get_profile": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
}


class ZoomFFTLibraryMissing(ImportError):
    pass


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen the C-ABI library and declare every prototype.

    ``path=None`` loads the product library next to this file and insists it
    was built for sm_100a.  (tests/emu passes an explicit path to its own
    CPU emulation build of the same sources; the package never does.)
    """
    product = path is None
    path = LIB_PATH if product else path
    if not os.path.isfile(path):
        raise ZoomFFTLibraryMissing(
            "%s not found: build it with `python -m pypanadapter_b200.build` "
            "(nvcc, sm_100a).  pypanadapter_b200 has no CPU fallback." % path)
    lib = C.CDLL(path, mode=C.RTLD_LOCAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.zfb_abi_version() != ABI_VERSION:
        raise ZoomFFTLibraryMissing("ABI version mismatch: library %d, binding %d"
                                    % (lib.zfb_abi_version(), ABI_VERSION))
    kind = lib.zfb_build_kind().decode()
    if product and kind != "sm_100a":
        raise ZoomFFTLibraryMissing("%s is a %r build, not the sm_100a product" % (path, kind))
    return lib


_product_lib = None


def product_library() -> C.CDLL:
    global _product_lib
    if _product_lib is None:
        _product_lib = load_library(None)
    return _product_lib
