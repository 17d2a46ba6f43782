"""Host-side mirror of the reference's codec interface on top of the C ABI.

The reference is Java (src/bvk_ss19/FractalCompression.java = FC, RasterImage.java = RI)
and no JVM exists in the build environment, so the host side that stays in Java
(image container, grey/RGB dispatch, stream writer, decoder entry) is mirrored here
with the reference's own names and argument meaning; the hot path is the native
library.  Nothing in this module computes codes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import io
import struct

import numpy as np

from . import _lib
from ._lib import FicError, Timings


class RasterImage:
    """RI:18-72: `argb` int32 0xAARRGGBB pixels in scanline order, `width`, `height`."""

    GRAY = np.int32(np.uint32(0xFFA0A0A0).view(np.int32))  # RI:19

    def __init__(self, width: int, height: int):
        self.width, self.height = int(width), int(height)
        self.argb = np.full((self.height, self.width), self.GRAY, np.int32)  # RI:31

    @classmethod
    def from_argb(cls, argb) -> "RasterImage":
        a = np.ascontiguousarray(argb, dtype=np.int32)
        im = cls.__new__(cls)
        im.height, im.width = a.shape
        im.argb = a
        return im

    @classmethod
    def from_grey(cls, plane) -> "RasterImage":
        v = np.ascontiguousarray(plane, dtype=np.uint8).astype(np.uint32)
        return cls.from_argb((0xFF000000 | (v << 16) | (v << 8) | v).view(np.int32))

    @classmethod
    def from_rgb(cls, rgb) -> "RasterImage":
        a = np.ascontiguousarray(rgb, dtype=np.uint8).astype(np.uint32)
        return cls.from_argb((0xFF000000 | (a[..., 0] << 16) | (a[..., 1] << 8) | a[..., 2]).view(np.int32))

    @classmethod
    def from_file(cls, path: str) -> "RasterImage":
        """RI:34-52 (JavaFX Image + getIntArgbInstance); PIL decodes the bundled images identically."""
        from PIL import Image

        return cls.from_rgb(np.asarray(Image.open(path).convert("RGB")))

    def red(self) -> np.ndarray:
        return ((self.argb.view(np.uint32) >> 16) & 0xFF).astype(np.uint8)

    def rgb(self) -> np.ndarray:
        u = self.argb.view(np.uint32)
        return np.stack([(u >> 16) & 0xFF, (u >> 8) & 0xFF, u & 0xFF], -1).astype(np.uint8)


class ByteSink(io.BytesIO):
    """A DataOutputStream stand-in whose contents survive close() (FC:259 closes `out`)."""

    def close(self):  # noqa: D401
        self.closed_by_codec = True


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Handle:
    """One libfic_b200 context (device memory, stream) on one GPU."""

    def __init__(self, device: int = 0):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = self._L.fic_create(int(device), C.byref(h))
        if rc:
            raise FicError(rc, self._L.fic_last_error(None).decode())
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._L.fic_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc: int):
        if rc:
            raise FicError(rc, self._L.fic_last_error(self._h).decode())

    def set_engine(self, engine: int):
        self._check(self._L.fic_set_option(self._h, _lib.FIC_OPT_ENGINE, int(engine)))

    def set_umma_kind(self, kind: int):
        """Tensor-core instruction kind of the tcgen05 search: FIC_UMMA_KIND_AUTO / _I8 / _F16."""
        self._check(self._L.fic_set_option(self._h, _lib.FIC_OPT_UMMA_KIND, int(kind)))

    def set_umma_pair(self, pair: int):
        """CTA pairs (tcgen05 cta_group::2) of the tcgen05 search: FIC_UMMA_PAIR_AUTO / _OFF / _ON."""
        self._check(self._L.fic_set_option(self._h, _lib.FIC_OPT_UMMA_PAIR, int(pair)))

    def umma_pair_used(self) -> bool:
        """True if the last tcgen05 search of this handle ran the CTA-pair kernel."""
        v = C.c_int(0)
        self._check(self._L.fic_get_option(self._h, _lib.FIC_OPT_UMMA_PAIR_USED, C.byref(v)))
        return bool(v.value)

    def pin(self, array: np.ndarray):
        """Page-locks a caller-owned contiguous array (fic_pin_host_buffer) so encode/decode copies run at full PCIe
        rate; pair with unpin() before the array is freed."""
        assert array.flags["C_CONTIGUOUS"]
        self._check(self._L.fic_pin_host_buffer(self._h, array.ctypes.data, array.nbytes))

    def unpin(self, array: np.ndarray):
        self._check(self._L.fic_unpin_host_buffer(self._h, array.ctypes.data))

    def f16_exact(self) -> bool:
        """True if this device's kind::f16 tensor path reproduced the exact integer covariances in the
        library's self-test (run once per handle); False means the handle runs kind::i8 instead."""
        v = C.c_int(0)
        self._check(self._L.fic_get_option(self._h, _lib.FIC_OPT_F16_EXACT, C.byref(v)))
        return bool(v.value)

    def set_stream(self, cuda_stream: int | None):
        """None -> the handle's own stream; an integer cudaStream_t otherwise.  torch reports its default
        stream as 0, which the C ABI reads as "own stream": pass the legacy-default handle instead."""
        if cuda_stream is None:
            v = 0
        else:
            v = int(cuda_stream) or 1  # cudaStreamLegacy == (cudaStream_t)0x1
        self._check(self._L.fic_set_stream(self._h, C.c_void_p(v)))

    def sync(self):
        self._check(self._L.fic_sync(self._h))

    def timings(self) -> Timings:
        t = Timings()
        self._check(self._L.fic_get_timings(self._h, C.byref(t)))
        return t

    def geometry(self, W, H, B, wk):
        nr, nd = C.c_int64(), C.c_int64()
        self._check(self._L.fic_geometry(W, H, B, wk, C.byref(nr), C.byref(nd)))
        return nr.value, nd.value

    def encode(self, argb: np.ndarray, B: int, wk: int, rgb, range_begin: int = 0,
               range_end: int | None = None, info: np.ndarray | None = None, q: np.ndarray | None = None):
        """Runs fic_encode_grey / fic_encode_rgb (rgb = False / True) or the isometry extension fic_encode_grey_iso
        (rgb = FIC_MODE_GREY_ISO); returns (imageInfo float32[NR][S], qcodes int32[NR][S]), S = 3 / 5 / 4."""
        a = np.ascontiguousarray(argb, dtype=np.int32)
        H, W = a.shape
        S = (3, 5, 4)[int(rgb)]
        nr = (W // B) * (H // B) if B > 0 else 0
        if range_end is None:
            range_end = nr
        if info is None:
            info = np.zeros((max(nr, 0), S), np.float32)
        if q is None:
            q = np.zeros((max(nr, 0), S), np.int32)
        fn = (self._L.fic_encode_grey, self._L.fic_encode_rgb, self._L.fic_encode_grey_iso)[int(rgb)]
        self._check(fn(self._h, _ptr(a), W, H, B, wk, range_begin, range_end, _ptr(info), _ptr(q)))
        return info, q

    def encode_u8(self, planes: np.ndarray, B: int, wk: int, range_begin: int = 0, range_end: int | None = None,
                  info: np.ndarray | None = None, q: np.ndarray | None = None):
        """fic_encode_grey_u8 (planes: uint8 [H, W]) / fic_encode_rgb_planes (uint8 [3, H, W]): the 8-bit host entries."""
        a = np.ascontiguousarray(planes, dtype=np.uint8)
        rgb = a.ndim == 3
        assert not rgb or a.shape[0] == 3
        H, W = a.shape[-2:]
        S = 5 if rgb else 3
        nr = (W // B) * (H // B) if B > 0 else 0
        if range_end is None:
            range_end = nr
        if info is None:
            info = np.zeros((max(nr, 0), S), np.float32)
        if q is None:
            q = np.zeros((max(nr, 0), S), np.int32)
        fn = self._L.fic_encode_rgb_planes if rgb else self._L.fic_encode_grey_u8
        self._check(fn(self._h, _ptr(a), W, H, B, wk, range_begin, range_end, _ptr(info), _ptr(q)))
        return info, q

    def encode_planes_dev(self, d_planes: int, rgb, W: int, H: int, B: int, wk: int, range_begin: int,
                          range_end: int, d_info: int | None, d_q: int | None):
        """Asynchronous device-pointer entry (fic_encode_planes_dev)."""
        self._check(self._L.fic_encode_planes_dev(self._h, C.c_void_p(d_planes), int(rgb), W, H, B, wk,
                                                  range_begin, range_end, C.c_void_p(d_info or 0),
                                                  C.c_void_p(d_q or 0)))

    def decode(self, q: np.ndarray, W: int, H: int, B: int, wk: int, rgb, avg_error: float = 0.0,
               max_iters: int = 50, out: np.ndarray | None = None):
        """fic_decode.  `out` (int32 [H, W], e.g. a view of pinned memory) receives the ARGB image; allocated if None."""
        qq = np.ascontiguousarray(q, dtype=np.int32)
        if out is None:
            out = np.empty((H, W), np.int32)
        assert out.dtype == np.int32 and out.shape == (H, W) and out.flags["C_CONTIGUOUS"]
        avg = C.c_float(avg_error)
        it = C.c_int(0)
        self._check(self._L.fic_decode(self._h, int(rgb), W, H, B, wk, _ptr(qq), max_iters, _ptr(out),
                                       C.byref(avg), C.byref(it)))
        return out, np.float32(avg.value), it.value

    def encode_batch(self, argb: np.ndarray, B: int, wk: int, rgb, info: np.ndarray | None = None,
                     q: np.ndarray | None = None):
        """fic_encode_batch: n same-size images, int32 ARGB [n, H, W], mode rgb = False / True / FIC_MODE_GREY_ISO;
        returns (info float32 [n, NR, S], qcodes int32 [n, NR, S]), each image's rows equal to encode() of that image."""
        a = np.ascontiguousarray(argb, dtype=np.int32)
        assert a.ndim == 3, "argb must be [n, H, W]"
        n, H, W = a.shape
        info, q = self._batch_codes(n, W, H, B, (3, 5, 4)[int(rgb)], info, q)
        self._check(self._L.fic_encode_batch(self._h, int(rgb), _ptr(a), n, W, H, B, wk, _ptr(info), _ptr(q)))
        return info, q

    def encode_batch_u8(self, planes: np.ndarray, B: int, wk: int, rgb=None, info: np.ndarray | None = None,
                        q: np.ndarray | None = None):
        """fic_encode_batch_u8: uint8 [n, H, W] (grey: the red channel; rgb may be FIC_MODE_GREY_ISO) or [n, 3, H, W]
        (RGB).  rgb=None takes the mode from the shape."""
        a = np.ascontiguousarray(planes, dtype=np.uint8)
        assert a.ndim in (3, 4) and (a.ndim == 3 or a.shape[1] == 3), "planes must be [n, H, W] or [n, 3, H, W]"
        if rgb is None:
            rgb = a.ndim == 4
        assert (a.ndim == 4) == (int(rgb) == 1), "RGB takes [n, 3, H, W] planes, grey [n, H, W]"
        n, H, W = a.shape[0], a.shape[-2], a.shape[-1]
        info, q = self._batch_codes(n, W, H, B, (3, 5, 4)[int(rgb)], info, q)
        self._check(self._L.fic_encode_batch_u8(self._h, int(rgb), _ptr(a), n, W, H, B, wk, _ptr(info), _ptr(q)))
        return info, q

    @staticmethod
    def _batch_codes(n, W, H, B, S, info, q):
        nr = (W // B) * (H // B) if B > 0 else 0
        if info is None:
            info = np.zeros((n, max(nr, 0), S), np.float32)
        if q is None:
            q = np.zeros((n, max(nr, 0), S), np.int32)
        for t, dt in ((info, np.float32), (q, np.int32)):
            assert t.dtype == dt and t.shape == (n, max(nr, 0), S) and t.flags["C_CONTIGUOUS"]
        return info, q

    def _decode_batch(self, fn, q, W, H, B, wk, rgb, avg_error, max_iters, out):
        qq = np.ascontiguousarray(q, dtype=np.int32)
        assert qq.ndim == 3, "q must be [n, NR, S]"
        n = qq.shape[0]
        avg = np.zeros(n, np.float32) if avg_error is None else np.array(avg_error, np.float32).reshape(n)
        it = np.zeros(n, np.int32)
        self._check(fn(self._h, int(rgb), n, W, H, B, wk, _ptr(qq), max_iters, _ptr(out), _ptr(avg), _ptr(it)))
        return out, avg, it

    def decode_batch(self, q: np.ndarray, W: int, H: int, B: int, wk: int, rgb, avg_error=None, max_iters: int = 50,
                     out: np.ndarray | None = None):
        """fic_decode_batch: codes [n, NR, S] -> (ARGB int32 [n, H, W], avgError float32 [n], iterations int32 [n]).
        avg_error: each image's carry-in (the reference's never-reset static, FC:20), None for 0."""
        n = np.shape(q)[0]
        if out is None:
            out = np.empty((n, H, W), np.int32)
        assert out.dtype == np.int32 and out.shape == (n, H, W) and out.flags["C_CONTIGUOUS"]
        return self._decode_batch(self._L.fic_decode_batch, q, W, H, B, wk, rgb, avg_error, max_iters, out)

    def decode_batch_u8(self, q: np.ndarray, W: int, H: int, B: int, wk: int, rgb, avg_error=None, max_iters: int = 50,
                        out: np.ndarray | None = None):
        """fic_decode_batch_u8: as decode_batch with 8-bit planes, uint8 [n, H, W] (grey) or [n, 3, H, W] (RGB)."""
        n = np.shape(q)[0]
        shape = (n, 3, H, W) if int(rgb) == 1 else (n, H, W)
        if out is None:
            out = np.empty(shape, np.uint8)
        assert out.dtype == np.uint8 and out.shape == shape and out.flags["C_CONTIGUOUS"]
        return self._decode_batch(self._L.fic_decode_batch_u8, q, W, H, B, wk, rgb, avg_error, max_iters, out)

    def float_sum(self, terms: np.ndarray, carry: float = 0.0) -> np.float32:
        """fic_debug_float_sum: the reference's sequential binary32 running sum (FC:407) over integer terms, computed
        the way the decoder folds a sweep."""
        t = np.ascontiguousarray(terms, dtype=np.int32)
        out = C.c_float(0)
        self._check(self._L.fic_debug_float_sum(self._h, _ptr(t), t.size, C.c_float(carry), C.byref(out)))
        return np.float32(out.value)

    def decode_u8(self, q: np.ndarray, W: int, H: int, B: int, wk: int, rgb, avg_error: float = 0.0,
                  max_iters: int = 50, out: np.ndarray | None = None):
        """fic_decode_u8: the image as 8-bit planes, uint8 [H, W] (grey) or [3, H, W] (RGB)."""
        qq = np.ascontiguousarray(q, dtype=np.int32)
        shape = (3, H, W) if int(rgb) == 1 else (H, W)
        if out is None:
            out = np.empty(shape, np.uint8)
        assert out.dtype == np.uint8 and out.shape == shape and out.flags["C_CONTIGUOUS"]
        avg = C.c_float(avg_error)
        it = C.c_int(0)
        self._check(self._L.fic_decode_u8(self._h, int(rgb), W, H, B, wk, _ptr(qq), max_iters, _ptr(out),
                                          C.byref(avg), C.byref(it)))
        return out, np.float32(avg.value), it.value

    def decode_planes_dev(self, d_q: int, W: int, H: int, B: int, wk: int, rgb, d_planes_out: int,
                          avg_error: float = 0.0, max_iters: int = 50):
        """fic_decode_planes_dev: device codes in, device 8-bit planes out; returns (avgError, iterations)."""
        avg = C.c_float(avg_error)
        it = C.c_int(0)
        self._check(self._L.fic_decode_planes_dev(self._h, int(rgb), W, H, B, wk, C.c_void_p(d_q), max_iters,
                                                  C.c_void_p(d_planes_out), C.byref(avg), C.byref(it)))
        return np.float32(avg.value), it.value

    def collage(self, argb: np.ndarray, info: np.ndarray, B: int, wk: int, rgb: bool):
        """fic_collage; `info` is rewritten in place (window-local -> codebook index, FC:273)."""
        a = np.ascontiguousarray(argb, dtype=np.int32)
        H, W = a.shape
        assert info.dtype == np.float32 and info.flags["C_CONTIGUOUS"]
        out = np.empty((H, W), np.int32)
        self._check(self._L.fic_collage(self._h, int(rgb), _ptr(a), W, H, B, wk, _ptr(info), _ptr(out)))
        return out

    def measure_int8_peak(self) -> float:
        """Dense int8 tensor-pipe rate of this GPU in TOP/s, from a bare tcgen05.mma.kind::i8 loop."""
        v = C.c_double(0.0)
        self._check(self._L.fic_measure_int8_peak(self._h, C.byref(v)))
        return v.value

    def measure_mma_peak(self, kind: int, n_cols: int = 128) -> float:
        """Dense tensor-pipe rate in TOP/s of kind::i8 / kind::f16 at the MMA shape M = 128 x N = n_cols."""
        v = C.c_double(0.0)
        self._check(self._L.fic_measure_mma_peak(self._h, int(kind), int(n_cols), C.byref(v)))
        return v.value

    def measure_mma_peak_pair(self, kind: int) -> float:
        """The same for the CTA-pair shape (cta_group::2, M = 256 x N = 128)."""
        v = C.c_double(0.0)
        self._check(self._L.fic_measure_mma_peak_pair(self._h, int(kind), C.byref(v)))
        return v.value

    def build_pool(self, argb: np.ndarray, B: int, rgb: bool):
        a = np.ascontiguousarray(argb, dtype=np.int32)
        H, W = a.shape
        Cn = 3 if rgb else 1
        nd = (2 * W // B - 3) * (2 * H // B - 3)
        dec = np.empty((Cn, H // 2, W // 2), np.uint8)
        s1 = np.empty((Cn, nd), np.int32)
        s2 = np.empty((Cn, nd), np.int32)
        self._check(self._L.fic_build_pool(self._h, _ptr(a), int(rgb), W, H, B, _ptr(dec), _ptr(s1), _ptr(s2)))
        return dec, s1, s2


class _BorrowedHandle(Handle):
    """A per-device context owned by a MultiHandle (fic_multi_handle): never destroyed from here."""

    def __init__(self, L, h, device):
        self._L, self._h, self.device = L, h, int(device)

    def close(self):
        self._h = None

    __del__ = close


class MultiHandle:
    """One libfic_b200 context over several GPUs of this process (fic_create_multi): the image is uploaded once,
    broadcast with NCCL over NVLink, every device searches a slice of range rows and writes its codes straight into
    the caller's arrays.  Results equal Handle.encode byte for byte."""

    def __init__(self, devices):
        self._L = _lib.load()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        m = C.c_void_p()
        rc = self._L.fic_create_multi(devs, len(devices), C.byref(m))
        if rc:
            raise FicError(rc, self._L.fic_multi_last_error(None).decode())
        self._m = m
        self.devices = [int(d) for d in devices]

    def close(self):
        if getattr(self, "_m", None):
            self._L.fic_destroy_multi(self._m)
            self._m = None

    __del__ = close

    def _check(self, rc: int):
        if rc:
            raise FicError(rc, self._L.fic_multi_last_error(self._m).decode())

    def handle(self, rank: int = 0) -> Handle:
        h = self._L.fic_multi_handle(self._m, int(rank))
        if not h:
            raise IndexError(rank)
        return _BorrowedHandle(self._L, C.c_void_p(h), self.devices[rank])

    def set_engine(self, engine: int):
        self._check(self._L.fic_multi_set_option(self._m, _lib.FIC_OPT_ENGINE, int(engine)))

    def set_umma_kind(self, kind: int):
        self._check(self._L.fic_multi_set_option(self._m, _lib.FIC_OPT_UMMA_KIND, int(kind)))

    def set_umma_pair(self, pair: int):
        self._check(self._L.fic_multi_set_option(self._m, _lib.FIC_OPT_UMMA_PAIR, int(pair)))

    def timings(self, rank: int = -1) -> Timings:
        t = Timings()
        self._check(self._L.fic_multi_get_timings(self._m, int(rank), C.byref(t)))
        return t

    def range_slice(self, rank: int):
        a, b = C.c_int64(), C.c_int64()
        self._check(self._L.fic_multi_range_slice(self._m, int(rank), C.byref(a), C.byref(b)))
        return a.value, b.value

    def encode(self, pixels: np.ndarray, B: int, wk: int, rgb=False, info: np.ndarray | None = None,
               q: np.ndarray | None = None):
        """int32 ARGB [H, W] -> fic_multi_encode_grey / _rgb / _grey_iso (rgb = False / True / FIC_MODE_GREY_ISO);
        uint8 [H, W] / [3, H, W] -> fic_multi_encode_grey_u8 / _rgb_planes."""
        a = np.ascontiguousarray(pixels)
        if a.dtype == np.uint8:
            rgb = a.ndim == 3
            fn = self._L.fic_multi_encode_rgb_planes if rgb else self._L.fic_multi_encode_grey_u8
        else:
            a = np.ascontiguousarray(a, dtype=np.int32)
            fn = (self._L.fic_multi_encode_grey, self._L.fic_multi_encode_rgb, self._L.fic_multi_encode_grey_iso)[int(rgb)]
        H, W = a.shape[-2:]
        S = (3, 5, 4)[int(rgb)]
        nr = (W // B) * (H // B) if B > 0 else 0
        if info is None:
            info = np.zeros((max(nr, 0), S), np.float32)
        if q is None:
            q = np.zeros((max(nr, 0), S), np.int32)
        self._check(fn(self._m, _ptr(a), W, H, B, wk, _ptr(info), _ptr(q)))
        return info, q


# ---- .run stream helpers (native) ---------------------------------------------------

def stream_write(q: np.ndarray, W: int, H: int, B: int, wk: int, rgb: bool) -> bytes:
    L = _lib.load()
    n = L.fic_stream_size(int(rgb), W, H, B)
    buf = np.empty(n, np.uint8)
    qq = np.ascontiguousarray(q, dtype=np.int32)
    rc = L.fic_stream_write(int(rgb), W, H, B, wk, _ptr(qq), _ptr(buf), n)
    if rc:
        raise FicError(rc, "fic_stream_write rejected its arguments")
    return buf.tobytes()


def stream_read(stream: bytes):
    """Returns (mode, W, H, B, wk, qcodes int32[NR][S]); mode is False (grey), True (RGB) or FIC_MODE_GREY_ISO (2)."""
    L = _lib.load()
    buf = np.frombuffer(stream, np.uint8)
    v = [C.c_int() for _ in range(5)]
    off = C.c_size_t()
    rc = L.fic_stream_read_header(_ptr(buf), len(buf), *[C.byref(x) for x in v], C.byref(off))
    if rc:
        raise FicError(rc, "malformed .run stream")
    rgb, W, H, B, wk = [x.value for x in v]
    S = (3, 5, 4)[rgb]
    q = np.empty(((W // B) * (H // B), S), np.int32)
    rc = L.fic_stream_read_codes(_ptr(buf), len(buf), _ptr(q))
    if rc:
        raise FicError(rc, "malformed .run stream")
    return (rgb if rgb == _lib.FIC_MODE_GREY_ISO else bool(rgb)), W, H, B, wk, q


class FractalCompression:
    """Mirror of the reference's static codec facade (FC:12-59, FC:230-261, FC:547-553).

    The mutable statics `blockgroesse`, `widthKernel` (FC:14-15) and `avgError` (FC:20) are
    class attributes, as in the reference; the native handle is created on first use.
    """

    blockgroesse = 8
    widthKernel = 2
    avgError = np.float32(0.0)
    imageInfo: np.ndarray | None = None      # FC:17
    imageInfoRGB: np.ndarray | None = None   # FC:18
    _handle: Handle | None = None
    device = 0
    isometries = False   # extension (not in the reference): 8 isometries per candidate domain, grey images only

    @classmethod
    def handle(cls) -> Handle:
        if cls._handle is None:
            cls._handle = Handle(cls.device)
        return cls._handle

    @classmethod
    def getAvgError(cls):  # FC:22-24
        return cls.avgError

    @staticmethod
    def isGreyScale(input: RasterImage) -> bool:  # FC:32-45
        u = input.argb.view(np.uint32)
        r, g, b = (u >> 16) & 0xFF, (u >> 8) & 0xFF, u & 0xFF
        return bool(np.all(r == g) and np.all(g == b))

    @classmethod
    def encode(cls, input: RasterImage, out) -> RasterImage:  # FC:54-59
        if cls.isGreyScale(input):
            return cls.encodeGrayScale(input, out)
        return cls.encodeRGB(input, out)

    @classmethod
    def encodeGrayScale(cls, input: RasterImage, out) -> RasterImage:  # FC:109-162
        mode = _lib.FIC_MODE_GREY_ISO if cls.isometries else _lib.FIC_MODE_GREY
        info, q = cls.handle().encode(input.argb, cls.blockgroesse, cls.widthKernel, rgb=mode)
        cls.imageInfo, cls._q = info, q
        cls.writeData(out, mode, input.width, input.height)
        return cls.getBestGeneratedCollage(input)

    @classmethod
    def encodeRGB(cls, input: RasterImage, out) -> RasterImage:  # FC:171-219
        info, q = cls.handle().encode(input.argb, cls.blockgroesse, cls.widthKernel, rgb=True)
        cls.imageInfoRGB, cls._q = info, q
        cls.writeData(out, 1, input.width, input.height)
        return cls.getBestGeneratedCollageRGB(input)

    @classmethod
    def writeData(cls, out, isRGB: int, width: int, height: int):  # FC:230-261
        out.write(stream_write(cls._q, width, height, cls.blockgroesse, cls.widthKernel, int(isRGB)))
        out.close()  # FC:259

    @classmethod
    def getBestGeneratedCollage(cls, originalImage: RasterImage) -> RasterImage:  # FC:269-300
        mode = _lib.FIC_MODE_GREY_ISO if cls.imageInfo.shape[1] == 4 else _lib.FIC_MODE_GREY
        out = cls.handle().collage(originalImage.argb, cls.imageInfo, cls.blockgroesse, cls.widthKernel, rgb=mode)
        return RasterImage.from_argb(out)

    @classmethod
    def getBestGeneratedCollageRGB(cls, originalImage: RasterImage) -> RasterImage:  # FC:308-347
        out = cls.handle().collage(originalImage.argb, cls.imageInfoRGB, cls.blockgroesse, cls.widthKernel, rgb=True)
        return RasterImage.from_argb(out)

    @classmethod
    def decode(cls, inputStream) -> RasterImage:  # FC:547-553 -> FC:356-421 / FC:430-508
        data = inputStream.read() if hasattr(inputStream, "read") else bytes(inputStream)
        rgb, W, H, B, wk, q = stream_read(data)
        img, avg, _ = cls.handle().decode(q, W, H, B, wk, rgb, avg_error=float(cls.avgError))
        cls.avgError = avg
        return RasterImage.from_argb(img)


def parse_header(stream: bytes):
    return struct.unpack(">5i", stream[:20])
