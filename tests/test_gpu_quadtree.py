"""The quadtree extension (FIC_MODE_GREY_QT) on the GPU: streams and decodes bit-identical to the CPU oracle, the
degenerate trees against the fixed-block entries, the 4096^2 full pool against per-level GPU encodes, and the
rejections."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

from conftest import GOLD

pytestmark = pytest.mark.gpu

MSES = [-1.0, 0.0, 4.0, 25.0, 100.0, np.inf]


def _plane(name):
    from fractal_image_compression_b200 import synth

    if name == "lena":
        return np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    if name == "lena64":
        return np.fromfile(os.path.join(GOLD, "lena64.u8"), np.uint8).reshape(64, 64)
    if name == "structured512":
        return synth.structured(512, 512, 7)
    if name == "noise512":
        return synth.noise(512, 512, 9)
    if name == "structured512x256":
        return synth.structured(512, 256, 11)
    if name == "flat":
        return np.full((128, 128), 77, np.uint8)
    if name == "binary":
        return ((synth.noise(128, 128, 13) >> 7) * 255).astype(np.uint8)
    if name == "ties":  # a few repeated 8 x 8 tiles: many equal scores
        t = synth.noise(8, 8, 17)
        return np.tile(np.concatenate([t, t[::-1]], 0), (8, 16))
    raise KeyError(name)


@pytest.fixture(scope="module")
def h():
    import fractal_image_compression_b200 as fic

    hh = fic.Handle(0)
    yield hh
    hh.close()


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree

    quadtree.build()
    return quadtree


CASES = [("lena", 16, 8, 2), ("lena", 16, 4, 0), ("lena", 8, 4, 4), ("lena64", 16, 4, 0), ("lena64", 8, 4, 2),
         ("structured512", 16, 8, 0), ("noise512", 16, 8, 0), ("structured512x256", 16, 4, 3), ("flat", 16, 4, 0),
         ("binary", 8, 4, 5), ("ties", 16, 4, 0)]


@pytest.mark.parametrize("name,b_max,b_min,wk", CASES)
def test_stream_and_decode_match_oracle(h, oracle, name, b_max, b_min, wk, qt):
    plane = _plane(name)
    for mse in MSES:
        got = h.encode_quadtree(plane, b_max, b_min, wk, mse)
        want = qt.encode_quadtree(plane, b_max, b_min, wk, mse, nthreads=16)
        assert got == want, (name, mse)
        img, avg, it = h.decode_quadtree(got)
        oimg, oavg, oit = qt.decode_quadtree(want)
        assert (img == oimg).all() and it == oit and avg.tobytes() == oavg.tobytes(), (name, mse)


def test_decode_1024_matches_oracle(h, oracle, qt):
    from fractal_image_compression_b200 import synth

    plane = synth.structured(1024, 1024, 21)
    for b_max, b_min, mse in [(16, 4, 25.0), (16, 8, 4.0)]:
        s = h.encode_quadtree(plane, b_max, b_min, 2, mse)
        img, avg, it = h.decode_quadtree(s)
        oimg, oavg, oit = qt.decode_quadtree(s)
        assert (img == oimg).all() and it == oit and avg.tobytes() == oavg.tobytes()


def _leaves(s):
    n = struct.unpack(">i", s[28:32])[0]
    ntop = (struct.unpack(">i", s[4:8])[0] // struct.unpack(">i", s[20:24])[0]) * \
        (struct.unpack(">i", s[8:12])[0] // struct.unpack(">i", s[20:24])[0])
    return np.frombuffer(s, ">i4", count=3 * n, offset=32 + ntop + (-ntop % 4)).reshape(n, 3).astype(np.int32), ntop


@pytest.mark.parametrize("b_max,b_min,wk", [(16, 8, 2), (16, 4, 0), (8, 4, 0)])
def test_degenerate_trees(h, b_max, b_min, wk):
    plane = _plane("lena")
    full = lambda B: wk or 2 * (256 // B) - 3  # noqa: E731
    _, q_max = h.encode_u8(plane, b_max, full(b_max))
    _, q_min = h.encode_u8(plane, b_min, full(b_min))
    leaves, ntop = _leaves(h.encode_quadtree(plane, b_max, b_min, wk, np.inf))
    assert (leaves == q_max).all()
    leaves, _ = _leaves(h.encode_quadtree(plane, b_max, b_min, wk, -1.0))
    assert sorted(map(tuple, leaves.tolist())) == sorted(map(tuple, q_min.tolist()))
    s = h.encode_quadtree(plane, b_max, b_min, wk, np.inf)
    img, avg, it = h.decode_quadtree(s)
    fimg, favg, fit = h.decode_u8(q_max, 256, 256, b_max, full(b_max), False)
    assert (img == fimg).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == np.float32(favg).tobytes()


def test_direct_engine_gives_the_same_stream(h):
    import fractal_image_compression_b200 as fic

    plane = _plane("lena")
    want = [h.encode_quadtree(plane, 16, 4, wk, 25.0) for wk in (2, 0)]
    h.set_engine(fic.FIC_ENGINE_DIRECT)
    try:
        assert [h.encode_quadtree(plane, 16, 4, wk, 25.0) for wk in (2, 0)] == want
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)


def test_4096_full_pool_against_level_encodes(h):
    from fractal_image_compression_b200 import synth

    plane = synth.structured(4096, 4096, 5)
    mse = 20.0
    s = h.encode_quadtree(plane, 16, 8, 0, mse)
    t = h.timings()
    assert t.launches > 0 and t.search_evals > 0
    q16 = h.encode_u8(plane, 16, 2 * 256 - 3)[1]
    q8 = h.encode_u8(plane, 8, 2 * 512 - 3)[1]
    leaves, ntop = _leaves(s)
    flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
    # every flag from a numpy recomputation of E of the 16 x 16 codes on the source
    p = plane.astype(np.int64)
    dec = (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]) // 4
    wk, dpw = 509, 509
    c = q16[:, 0].astype(np.float32)
    # the whole pool: the window origin is 0 (generateKernel clamps it), so the codebook index is c itself
    idx = (np.trunc(c / np.float32(wk)).astype(np.int64) * dpw + np.trunc(np.fmod(c, np.float32(wk))).astype(np.int64))
    a = q16[:, 1].astype(np.float32) / np.float32(100)
    b = q16[:, 2].astype(np.float32)
    r, col = (idx // dpw) * 4, (idx % dpw) * 4
    ii = np.arange(16)
    dblk = dec[(r[:, None, None] + ii[None, :, None]), (col[:, None, None] + ii[None, None, :])]
    v = np.clip(np.trunc(a[:, None, None] * dblk.astype(np.float32) + b[:, None, None]), 0, 255).astype(np.int64)
    j = np.arange(ntop)
    src = p.reshape(256, 16, 256, 16).transpose(0, 2, 1, 3).reshape(-1, 16, 16)
    E = ((v - src[j]) ** 2).sum(axis=(1, 2))
    assert ((flags & 1) == (E.astype(np.float64) > mse * 256.0)).all()
    assert not (flags & ~np.uint8(1)).any()
    # every leaf: the level encode's code of that range
    k = 0
    for t_ in range(ntop):
        if not flags[t_] & 1:
            assert (leaves[k] == q16[t_]).all()
            k += 1
            continue
        y, x = divmod(t_, 256)
        for kk in range(4):
            assert (leaves[k] == q8[(2 * y + (kk >> 1)) * 512 + 2 * x + (kk & 1)]).all()
            k += 1
    assert k == len(leaves)


def test_rejections(h):
    import fractal_image_compression_b200 as fic

    L = fic._lib.load()
    plane = _plane("lena")
    ap = plane.ctypes.data_as(C.c_void_p)
    cap = L.fic_quadtree_stream_bound(256, 256, 16, 4)
    buf = np.zeros(cap, np.uint8)
    n = C.c_size_t(0)

    def enc(W, H, bmax, bmin, wk, mse, capacity=cap):
        return L.fic_encode_quadtree(h._h, ap, W, H, bmax, bmin, wk, mse, buf.ctypes.data_as(C.c_void_p), capacity, C.byref(n))

    assert enc(256, 256, 32, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 4, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 8, 16, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 2, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(248, 256, 16, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 128, 16, 4, 0, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 4, 2, float("nan")) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 4, 2, 25.0) == fic._lib.FIC_OK
    need = n.value
    assert enc(256, 256, 16, 4, 2, 25.0, need - 1) == fic._lib.FIC_E_ARG and n.value == need
    s = buf[:need].tobytes()
    assert fic.quadtree_stream_info(s) == (256, 256, 16, 4, 2, struct.unpack(">i", s[28:32])[0])

    def refused(stream):
        with pytest.raises(fic.FicError) as e:
            fic.quadtree_stream_info(stream)
        assert e.value.code == fic._lib.FIC_E_STREAM
        with pytest.raises(fic.FicError) as e:
            h.decode_quadtree(stream)
        assert e.value.code == fic._lib.FIC_E_STREAM

    refused(s[:-1])
    refused(s[:31])
    ntop = 256
    flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
    bad = bytearray(s)
    bad[32] |= 0x20  # bit 5 is never meaningful
    refused(bytes(bad))
    unsplit = np.flatnonzero((flags & 1) == 0)
    assert len(unsplit)
    bad = bytearray(s)
    bad[32 + int(unsplit[0])] |= 0x04  # a child split under a top block that is not split
    refused(bytes(bad))
    bad = bytearray(s)
    bad[28:32] = struct.pack(">i", struct.unpack(">i", s[28:32])[0] - 1)
    refused(bytes(bad))
    bad = bytearray(s)
    bad[32 + ntop:36 + ntop] = struct.pack(">i", 1 << 24)
    refused(bytes(bad))
    # the device's own out-of-pool check (the host decoder entry parses flags only)
    bad = bytes(bad)
    out = np.zeros((256, 256), np.uint8)
    rc = L.fic_decode_quadtree(h._h, np.frombuffer(bad, np.uint8).ctypes.data_as(C.c_void_p), len(bad), 50,
                               out.ctypes.data_as(C.c_void_p), None, None)
    assert rc == fic._lib.FIC_E_STREAM
    # the fixed-block header parser refuses a quadtree stream (blockgroesse 0)
    v = [C.c_int() for _ in range(5)]
    off = C.c_size_t()
    sb = np.frombuffer(s, np.uint8)
    assert L.fic_stream_read_header(sb.ctypes.data_as(C.c_void_p), len(s), *[C.byref(x) for x in v], C.byref(off)) == fic._lib.FIC_E_STREAM
