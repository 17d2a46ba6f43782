"""ctypes binding of the CPU oracle (oracle/fic_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Nothing under
fractal-image-compression_b200/ may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libfic_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile oracle/_build/libfic_oracle.so with the committed Makefile."""
    src = os.path.join(_HERE, "fic_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE], stdout=subprocess.DEVNULL)
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        i32p, f32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_uint8)
        L.fic_oracle_domain_block_index.argtypes = [C.c_int] * 6
        L.fic_oracle_domain_block_index.restype = C.c_int
        L.fic_oracle_generate_kernel.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_int)] * 2
        L.fic_oracle_generate_kernel.restype = None
        for fn in (L.fic_oracle_scale_image, L.fic_oracle_scale_image_rgb):
            fn.argtypes = [i32p, C.c_int, C.c_int, i32p]
            fn.restype = None
        L.fic_oracle_create_codebook.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, f32p]
        L.fic_oracle_create_codebook.restype = C.c_long
        for fn in (L.fic_oracle_encode_grey, L.fic_oracle_encode_rgb, L.fic_oracle_encode_grey_iso):
            fn.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_long, C.c_long, C.c_int, f32p]
            fn.restype = C.c_int
        L.fic_oracle_encode_list.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_long), C.c_long,
                                             C.c_int, f32p]
        L.fic_oracle_encode_list.restype = C.c_int
        L.fic_oracle_write_data.argtypes = [C.c_int] * 5 + [f32p, u8p]
        L.fic_oracle_write_data.restype = C.c_size_t
        L.fic_oracle_decode.argtypes = [u8p, C.c_size_t, i32p, f32p, C.POINTER(C.c_int)]
        L.fic_oracle_decode.restype = C.c_int
        L.fic_oracle_decode_iters.argtypes = [u8p, C.c_size_t, C.c_int, i32p, f32p, C.POINTER(C.c_int)]
        L.fic_oracle_decode_iters.restype = C.c_int
        L.fic_oracle_collage.argtypes = [i32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, f32p, i32p]
        L.fic_oracle_collage.restype = C.c_int
        L.fic_oracle_is_grey.argtypes = [i32p, C.c_int, C.c_int]
        L.fic_oracle_is_grey.restype = C.c_int
        _lib = L
    return _lib


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def _argb(a) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.int32)
    assert a.ndim == 2
    return a


def domain_block_index(x, y, rpw, rph, dpw, B) -> int:
    return lib().fic_oracle_domain_block_index(x, y, rpw, rph, dpw, B)


def generate_kernel(dpw, dph, index, wk):
    dy, dx = C.c_int(), C.c_int()
    lib().fic_oracle_generate_kernel(dpw, dph, index, wk, C.byref(dy), C.byref(dx))
    return dy.value, dx.value


def scale_image(argb, rgb: bool = False) -> np.ndarray:
    a = _argb(argb)
    H, W = a.shape
    out = np.empty((H // 2, W // 2), np.int32)
    fn = lib().fic_oracle_scale_image_rgb if rgb else lib().fic_oracle_scale_image
    fn(_p(a, C.c_int32), W, H, _p(out, C.c_int32))
    return out


def create_codebook(argb, B: int, rgb: bool = False):
    """Returns (pool[ND, B*B] int32, mean, var) as the reference's Domainblock fields."""
    a = _argb(argb)
    H, W = a.shape
    nd = (2 * W // B - 3) * (2 * H // B - 3)
    pool = np.empty((nd, B * B), np.int32)
    mean = np.empty((nd, 4) if rgb else (nd,), np.int32)
    var = np.empty((nd, 3) if rgb else (nd,), np.float32)
    got = lib().fic_oracle_create_codebook(_p(a, C.c_int32), W, H, B, int(rgb), _p(pool, C.c_int32),
                                           _p(mean, C.c_int32), _p(var, C.c_float))
    if got != nd:
        raise RuntimeError(f"codebook size {got} != {nd}")
    return pool, mean, var


def _mode(rgb: bool, iso: bool) -> int:
    """Stream / code layout: 0 grey (3 per range), 1 RGB (5), 2 grey + isometry index (4; extension)."""
    assert not (rgb and iso)
    return 2 if iso else int(bool(rgb))


def encode(argb, B: int, wk: int, rgb: bool = False, range_begin: int = 0, range_end: int | None = None,
           nthreads: int = 1, iso: bool = False) -> np.ndarray:
    """imageInfo[NR][3] (grey) or imageInfoRGB[NR][5]: {window-local idx, a, b...} floats; iso=True (extension,
    not in the reference): 8 isometries per candidate -> [NR][4] = {idx, a, b, isometry}."""
    a = _argb(argb)
    H, W = a.shape
    nr = (W // B) * (H // B)
    if range_end is None:
        range_end = nr
    info = np.zeros((nr, (3, 5, 4)[_mode(rgb, iso)]), np.float32)
    fn = (lib().fic_oracle_encode_grey, lib().fic_oracle_encode_rgb, lib().fic_oracle_encode_grey_iso)[_mode(rgb, iso)]
    rc = fn(_p(a, C.c_int32), W, H, B, wk, range_begin, range_end, nthreads, _p(info, C.c_float))
    if rc:
        raise ValueError(f"oracle encode rejected arguments (rc={rc})")
    return info


def encode_list(argb, B: int, wk: int, ranges, rgb: bool = False, iso: bool = False, nthreads: int = 1) -> np.ndarray:
    """Codes of the listed range blocks only (the codebook is built once): returns info[len(ranges)][3|5|4] in the
    order of `ranges`.  For spot checks of images whose full encode the CPU cannot finish."""
    a = _argb(argb)
    H, W = a.shape
    nr = (W // B) * (H // B)
    mode = _mode(rgb, iso)
    S = (3, 5, 4)[mode]
    r = np.ascontiguousarray(ranges, dtype=np.int64)
    info = np.zeros((nr, S), np.float32)
    rc = lib().fic_oracle_encode_list(_p(a, C.c_int32), W, H, B, wk, mode, r.ctypes.data_as(C.POINTER(C.c_long)), len(r),
                                      nthreads, _p(info, C.c_float))
    if rc:
        raise ValueError(f"oracle encode_list rejected arguments (rc={rc})")
    return info[r]


def write_data(info: np.ndarray, W: int, H: int, B: int, wk: int, rgb: bool = False, iso: bool = False) -> bytes:
    info = np.ascontiguousarray(info, np.float32)
    n = lib().fic_oracle_write_data(_mode(rgb, iso), W, H, B, wk, _p(info, C.c_float), None)
    buf = np.empty(n, np.uint8)
    lib().fic_oracle_write_data(_mode(rgb, iso), W, H, B, wk, _p(info, C.c_float), _p(buf, C.c_uint8))
    return buf.tobytes()


def decode(stream: bytes, avg_error_in: float = 0.0, max_iters: int = 50):
    """Returns (argb[H, W] int32, avgError float32, iterations); max_iters replaces the reference's limit of 50."""
    import struct

    _, W, H, _, _ = struct.unpack(">5i", stream[:20])
    buf = np.frombuffer(stream, np.uint8).copy()
    out = np.empty((H, W), np.int32)
    avg = C.c_float(avg_error_in)
    it = C.c_int(0)
    rc = lib().fic_oracle_decode_iters(_p(buf, C.c_uint8), len(buf), max_iters, _p(out, C.c_int32), C.byref(avg),
                                       C.byref(it))
    if rc:
        raise ValueError(f"oracle decode failed (rc={rc})")
    return out, np.float32(avg.value), it.value


def collage(argb, info: np.ndarray, B: int, wk: int, rgb: bool = False, iso: bool = False) -> np.ndarray:
    a = _argb(argb)
    H, W = a.shape
    info = np.ascontiguousarray(info, np.float32).copy()
    out = np.empty((H, W), np.int32)
    rc = lib().fic_oracle_collage(_p(a, C.c_int32), W, H, B, wk, _mode(rgb, iso), _p(info, C.c_float), _p(out, C.c_int32))
    if rc:
        raise ValueError(f"oracle collage failed (rc={rc})")
    return out


def is_grey(argb) -> bool:
    a = _argb(argb)
    H, W = a.shape
    return bool(lib().fic_oracle_is_grey(_p(a, C.c_int32), W, H))
