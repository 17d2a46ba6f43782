"""ctypes binding of the RGB quadtree extension's CPU oracle (oracle/fic_oracle_quadtree_rgb.c, linked with fic_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/.  Nothing under fractal-image-compression_b200/ may import this
module.  The library is compiled on first use with the flags of oracle/Makefile (Java float semantics: no FMA
contraction, no fast-math) into oracle/_build, or into a per-user temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes as C
import os
import struct
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, f) for f in ("fic_oracle_quadtree_rgb.c", "fic_oracle.c")]
_DEPS = _SRCS + [os.path.join(_HERE, f) for f in ("fic_oracle_quadtree_rgb.h", "fic_oracle.h")]
_CFLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra"]
_NAME = "libfic_oracle_quadtree_rgb.so"
_lib = None


def _stale(so: str) -> bool:
    return not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in _DEPS)


def build() -> str:
    """Compiles the library (when missing or older than its sources) and returns its path."""
    for d in (os.path.join(_HERE, "_build"), os.path.join(tempfile.gettempdir(), f"fic_oracle_{os.getuid()}")):
        so = os.path.join(d, _NAME)
        if not _stale(so):
            return so
        try:
            os.makedirs(d, exist_ok=True)
            if not os.access(d, os.W_OK):
                continue
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-o", tmp] + _SRCS + ["-lm", "-lpthread"])
            os.replace(tmp, so)
            return so
        except OSError:
            continue  # not writable: the next directory
    raise RuntimeError("no writable directory to build the RGB quadtree oracle in")


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        i32p, f32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_float), C.POINTER(C.c_uint8)
        L.fic_oracle_quadtree_rgb_bound.argtypes = [C.c_int] * 4
        L.fic_oracle_quadtree_rgb_bound.restype = C.c_size_t
        L.fic_oracle_encode_quadtree_rgb.argtypes = [i32p] + [C.c_int] * 5 + [C.c_double, C.c_int, u8p, C.POINTER(C.c_size_t)]
        L.fic_oracle_encode_quadtree_rgb.restype = C.c_int
        L.fic_oracle_decode_quadtree_rgb.argtypes = [u8p, C.c_size_t, C.c_int, i32p, f32p, C.POINTER(C.c_int)]
        L.fic_oracle_decode_quadtree_rgb.restype = C.c_int
        _lib = L
    return _lib


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(C.POINTER(t))


def planes_to_argb(planes) -> np.ndarray:
    """uint8 [3, H, W] planes (R, G, B) -> ARGB int32 [H, W]."""
    p = np.asarray(planes).astype(np.uint32)
    assert p.ndim == 3 and p.shape[0] == 3
    return (np.uint32(0xFF000000) | (p[0] << np.uint32(16)) | (p[1] << np.uint32(8)) | p[2]).view(np.int32)


def argb_to_planes(argb) -> np.ndarray:
    """ARGB int32 [H, W] -> uint8 [3, H, W] planes (R, G, B)."""
    a = np.asarray(argb).view(np.uint32)
    return np.stack([(a >> np.uint32(s)) & np.uint32(0xFF) for s in (16, 8, 0)]).astype(np.uint8)


def encode_quadtree_rgb(image, b_max: int, b_min: int, wk: int, max_mse: float, nthreads: int = 1) -> bytes:
    """The FIC_MODE_RGB_QT stream of an RGB image (ARGB ints [H, W], or uint8 planes [3, H, W]) with levels
    b_max .. b_min; wk == 0: each level's whole pool."""
    a = np.asarray(image)
    if a.dtype == np.uint8:
        a = planes_to_argb(a)
    a = np.ascontiguousarray(a, dtype=np.int32)
    assert a.ndim == 2
    H, W = a.shape
    cap = lib().fic_oracle_quadtree_rgb_bound(W, H, b_max, b_min)
    buf = np.zeros(max(cap, 1), np.uint8)
    n = C.c_size_t(0)
    rc = lib().fic_oracle_encode_quadtree_rgb(_p(a, C.c_int32), W, H, b_max, b_min, wk, float(max_mse), nthreads,
                                              _p(buf, C.c_uint8), C.byref(n))
    if rc:
        raise ValueError(f"oracle RGB quadtree encode rejected arguments (rc={rc})")
    return buf[:n.value].tobytes()


def decode_quadtree_rgb(stream: bytes, max_iters: int = 50):
    """Returns (planes uint8[3, H, W], avgError float32, iterations) of an RGB quadtree stream."""
    W, H = struct.unpack(">2i", stream[4:12]) if len(stream) >= 12 else (0, 0)
    buf = np.frombuffer(stream, np.uint8).copy()
    out = np.empty((H, W) if 0 < W <= 32768 and 0 < H <= 32768 else (1, 1), np.int32)
    avg = C.c_float(0.0)
    it = C.c_int(0)
    rc = lib().fic_oracle_decode_quadtree_rgb(_p(buf, C.c_uint8), len(buf), max_iters, _p(out, C.c_int32), C.byref(avg),
                                              C.byref(it))
    if rc:
        raise ValueError(f"oracle RGB quadtree decode failed (rc={rc})")
    return argb_to_planes(out), np.float32(avg.value), it.value
