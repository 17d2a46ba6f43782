"""ctypes binding of the quadtree oracles' encode to a byte budget (oracle/fic_oracle_quadtree_budget.c and
oracle/fic_oracle_quadtree_rgb_budget.c, linked with fic_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/ and tools/.  Nothing under fractal-image-compression_b200/ may import this
module.  The library is compiled on first use with the flags of oracle/Makefile (Java float semantics: no FMA
contraction, no fast-math) into oracle/_build, or into a per-user temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from .quadtree_rgb import planes_to_argb

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRCS = [os.path.join(_HERE, f) for f in ("fic_oracle_quadtree_budget.c", "fic_oracle_quadtree_rgb_budget.c", "fic_oracle.c")]
_DEPS = _SRCS + [os.path.join(_HERE, f) for f in ("fic_oracle_quadtree.c", "fic_oracle_quadtree_rgb.c", "fic_oracle_quadtree.h",
                                                   "fic_oracle_quadtree_rgb.h", "fic_oracle_quadtree_budget.h",
                                                   "fic_oracle_quadtree_budget_core.h", "fic_oracle.h")]
_CFLAGS = ["-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra"]
_NAME = "libfic_oracle_quadtree_budget.so"
_lib = None

E_INFEASIBLE = -9  # max_bytes below the unsplit tree's size


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
    raise RuntimeError("no writable directory to build the quadtree budget oracle in")


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        i32p, u8p = C.POINTER(C.c_int32), C.POINTER(C.c_uint8)
        for fn in (L.fic_oracle_encode_quadtree_budget, L.fic_oracle_encode_quadtree_rgb_budget):
            fn.argtypes = [i32p] + [C.c_int] * 5 + [C.c_size_t, C.c_int, u8p, C.POINTER(C.c_size_t), C.POINTER(C.c_double)]
            fn.restype = C.c_int
        _lib = L
    return _lib


class BudgetInfeasible(ValueError):
    """max_bytes is below the unsplit tree's size (min_bytes)."""

    def __init__(self, min_bytes: int):
        super().__init__(f"the unsplit tree needs {min_bytes} bytes")
        self.min_bytes = min_bytes


def _bound(W: int, H: int, b_max: int, b_min: int, leaf: int) -> int:
    top = (W // b_max) * (H // b_max)
    return 32 + ((top + 3) & ~3) + leaf * (W // b_min) * (H // b_min)


def _run(fn, a: np.ndarray, b_max: int, b_min: int, wk: int, max_bytes: int, nthreads: int, leaf: int):
    H, W = a.shape
    buf = np.zeros(max(_bound(W, H, b_max, b_min, leaf), 1), np.uint8)
    n, m = C.c_size_t(0), C.c_double(0.0)
    rc = fn(a.ctypes.data_as(C.POINTER(C.c_int32)), W, H, b_max, b_min, wk, int(max_bytes), nthreads,
            buf.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(n), C.byref(m))
    if rc == E_INFEASIBLE:
        raise BudgetInfeasible(n.value)
    if rc:
        raise ValueError(f"oracle quadtree budget encode rejected arguments (rc={rc})")
    return buf[:n.value].tobytes(), m.value


def encode_quadtree_budget(argb, b_max: int, b_min: int, wk: int, max_bytes: int, nthreads: int = 1):
    """(stream, m*) of a grey image (ARGB ints, or an 8-bit plane): the FIC_MODE_GREY_QT stream at the smallest max_mse
    m* whose stream has at most max_bytes bytes.  Raises BudgetInfeasible below the unsplit tree's size."""
    a = np.asarray(argb)
    if a.dtype == np.uint8:
        a = (np.uint32(0xFF000000) | a.astype(np.uint32) * np.uint32(0x010101)).view(np.int32)
    a = np.ascontiguousarray(a, dtype=np.int32)
    assert a.ndim == 2
    return _run(lib().fic_oracle_encode_quadtree_budget, a, b_max, b_min, wk, max_bytes, nthreads, 12)


def encode_quadtree_rgb_budget(image, b_max: int, b_min: int, wk: int, max_bytes: int, nthreads: int = 1):
    """(stream, m*) of an RGB image (ARGB ints [H, W], or uint8 planes [3, H, W]), as encode_quadtree_budget for
    FIC_MODE_RGB_QT."""
    a = np.asarray(image)
    if a.dtype == np.uint8:
        a = planes_to_argb(a)
    a = np.ascontiguousarray(a, dtype=np.int32)
    assert a.ndim == 2
    return _run(lib().fic_oracle_encode_quadtree_rgb_budget, a, b_max, b_min, wk, max_bytes, nthreads, 20)
