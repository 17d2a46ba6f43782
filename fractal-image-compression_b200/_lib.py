"""ctypes binding of libfic_b200.so -- exactly the entry points of include/fic_b200.h.

This is the binding a maintainer of the reference would write against the C ABI (the
Java FFM / JNI equivalent is shown in INTEGRATION.md).  There is no CPU fallback: if
the library has not been built the import of a compute entry raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libfic_b200.so")

FIC_OK = 0
FIC_E_ARG, FIC_E_CUDA, FIC_E_NOMEM, FIC_E_STREAM, FIC_E_INTERNAL = -1, -2, -3, -4, -5
FIC_ENGINE_AUTO, FIC_ENGINE_DIRECT, FIC_ENGINE_UMMA, FIC_ENGINE_FUSED = 0, 1, 2, 3
FIC_UMMA_KIND_AUTO, FIC_UMMA_KIND_I8, FIC_UMMA_KIND_F16 = 0, 1, 2
FIC_MODE_GREY, FIC_MODE_RGB, FIC_MODE_GREY_ISO = 0, 1, 2
FIC_OPT_ENGINE = 1
FIC_OPT_UMMA_KIND = 2
FIC_OPT_F16_EXACT = 3
FIC_OPT_UMMA_PAIR = 4
FIC_OPT_UMMA_PAIR_USED = 5
FIC_UMMA_PAIR_AUTO, FIC_UMMA_PAIR_OFF, FIC_UMMA_PAIR_ON = 0, 1, 2

# every symbol include/fic_b200.h declares (tests check the library exports them all)
ABI_SYMBOLS = [
    "fic_create", "fic_destroy", "fic_last_error", "fic_version", "fic_set_option", "fic_get_option", "fic_set_stream",
    "fic_get_timings", "fic_geometry", "fic_encode_grey", "fic_encode_rgb", "fic_encode_grey_iso", "fic_encode_planes_dev",
    "fic_sync", "fic_decode", "fic_collage", "fic_build_pool", "fic_stream_size", "fic_stream_write",
    "fic_stream_read_header", "fic_stream_read_codes", "fic_measure_int8_peak", "fic_measure_mma_peak", "fic_measure_mma_peak_pair",
    "fic_pin_host_buffer", "fic_unpin_host_buffer", "fic_debug_float_sum",
    "fic_encode_grey_u8", "fic_encode_rgb_planes", "fic_decode_u8", "fic_decode_planes_dev",
    "fic_create_multi", "fic_destroy_multi", "fic_multi_last_error", "fic_multi_device_count", "fic_multi_handle",
    "fic_multi_set_option", "fic_multi_get_timings", "fic_multi_range_slice", "fic_multi_encode_grey",
    "fic_multi_encode_rgb", "fic_multi_encode_grey_iso", "fic_multi_encode_grey_u8", "fic_multi_encode_rgb_planes",
    "fic_encode_batch", "fic_encode_batch_u8", "fic_decode_batch", "fic_decode_batch_u8",
]


class Timings(C.Structure):
    _fields_ = [
        ("h2d_ms", C.c_float), ("pool_ms", C.c_float), ("search_ms", C.c_float), ("kernel_ms", C.c_float), ("solve_ms", C.c_float),
        ("d2h_ms", C.c_float), ("total_ms", C.c_float), ("engine", C.c_int), ("launches", C.c_int),
        ("search_evals", C.c_double),
    ]


class FicError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libfic_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Loads the shared library; raises (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python fractal-image-compression_b200/build.py` "
            "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i32p, f32p, u8p = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_uint8)
    i64 = C.c_int64
    L.fic_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.fic_destroy.argtypes = [vp]
    L.fic_destroy.restype = None
    L.fic_last_error.argtypes = [vp]
    L.fic_last_error.restype = C.c_char_p
    L.fic_version.restype = C.c_char_p
    L.fic_set_option.argtypes = [vp, C.c_int, C.c_int]
    L.fic_get_option.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.fic_set_stream.argtypes = [vp, vp]
    L.fic_get_timings.argtypes = [vp, C.POINTER(Timings)]
    L.fic_geometry.argtypes = [C.c_int] * 4 + [C.POINTER(i64), C.POINTER(i64)]
    for fn in (L.fic_encode_grey, L.fic_encode_rgb, L.fic_encode_grey_iso):
        fn.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, i64, i64, vp, vp]
    for fn in (L.fic_encode_grey_u8, L.fic_encode_rgb_planes):
        fn.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, i64, i64, vp, vp]
    for fn in (L.fic_decode_u8, L.fic_decode_planes_dev):
        fn.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, f32p, C.POINTER(C.c_int)]
    for fn in (L.fic_encode_batch, L.fic_encode_batch_u8):
        fn.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    for fn in (L.fic_decode_batch, L.fic_decode_batch_u8):
        fn.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, vp]
    L.fic_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.fic_destroy_multi.argtypes = [vp]
    L.fic_destroy_multi.restype = None
    L.fic_multi_last_error.argtypes = [vp]
    L.fic_multi_last_error.restype = C.c_char_p
    L.fic_multi_device_count.argtypes = [vp]
    L.fic_multi_handle.argtypes = [vp, C.c_int]
    L.fic_multi_handle.restype = vp
    L.fic_multi_set_option.argtypes = [vp, C.c_int, C.c_int]
    L.fic_multi_get_timings.argtypes = [vp, C.c_int, C.POINTER(Timings)]
    L.fic_multi_range_slice.argtypes = [vp, C.c_int, C.POINTER(i64), C.POINTER(i64)]
    for fn in (L.fic_multi_encode_grey, L.fic_multi_encode_rgb, L.fic_multi_encode_grey_iso, L.fic_multi_encode_grey_u8,
               L.fic_multi_encode_rgb_planes):
        fn.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    L.fic_encode_planes_dev.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, i64, i64, vp, vp]
    L.fic_sync.argtypes = [vp]
    L.fic_decode.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, f32p,
                             C.POINTER(C.c_int)]
    L.fic_collage.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    L.fic_build_pool.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.fic_measure_int8_peak.argtypes = [vp, C.POINTER(C.c_double)]
    L.fic_measure_mma_peak.argtypes = [vp, C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.fic_measure_mma_peak_pair.argtypes = [vp, C.c_int, C.POINTER(C.c_double)]
    L.fic_pin_host_buffer.argtypes = [vp, vp, C.c_size_t]
    L.fic_unpin_host_buffer.argtypes = [vp, vp]
    L.fic_debug_float_sum.argtypes = [vp, vp, i64, C.c_float, f32p]
    L.fic_stream_size.argtypes = [C.c_int] * 4
    L.fic_stream_size.restype = C.c_size_t
    L.fic_stream_write.argtypes = [C.c_int] * 5 + [vp, vp, C.c_size_t]
    L.fic_stream_read_header.argtypes = [vp, C.c_size_t] + [C.POINTER(C.c_int)] * 5 + [C.POINTER(C.c_size_t)]
    L.fic_stream_read_codes.argtypes = [vp, C.c_size_t, vp]
    for name in ABI_SYMBOLS:
        fn = getattr(L, name)
        if fn.restype is C.c_int and name not in ("fic_version", "fic_last_error", "fic_stream_size", "fic_multi_last_error",
                                                   "fic_multi_handle"):
            fn.restype = C.c_int
    _lib = L
    return L
