"""Quadtree batches (fic_encode_quadtree_batch, fic_decode_quadtree_batch) on the GPU: every stream, size, decoded image,
avgError and sweep count equal to the single entries' for that image, grey and RGB, across level pairs, windows, engines,
thresholds, batch sizes and mixed content; a few streams against the CPU oracle; the rejections; and launch counts that
do not grow with the batch."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

from conftest import GOLD

pytestmark = pytest.mark.gpu

MSES = [-1.0, 0.0, 25.0, 200.0, np.inf]
PAIRS = [(16, 8), (16, 4), (8, 4), (16, 16)]


@pytest.fixture(scope="module")
def fic():
    import fractal_image_compression_b200 as f

    return f


@pytest.fixture(scope="module")
def h(fic):
    hh = fic.Handle(0)
    yield hh
    hh.close()


@pytest.fixture(autouse=True)
def _auto(h, fic):
    h.set_engine(fic.FIC_ENGINE_AUTO)
    yield
    h.set_engine(fic.FIC_ENGINE_AUTO)


def _grey(name, W=256, seed=0):
    from fractal_image_compression_b200 import synth

    if name == "lena":
        p = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
        return np.roll(p, 8 * seed, axis=1)[:W, :W].copy()
    if name == "noise":
        return synth.noise(W, W, 31 + seed)
    if name == "flat":
        return np.full((W, W), (77 + 3 * seed) % 256, np.uint8)
    if name == "binary":
        return ((synth.noise(W, W, 13 + seed) >> 7) * 255).astype(np.uint8)
    if name == "ties":  # a few repeated 8 x 8 tiles: many equal scores
        t = synth.noise(8, 8, 17 + seed)
        return np.tile(np.concatenate([t, t[::-1]], 0), (W // 16, W // 8))
    if name == "structured":
        return synth.structured(W, W, 7 + seed)
    raise KeyError(name)


def _image(name, rgb, W=256, seed=0):
    if not rgb:
        return _grey(name, W, seed)
    if name == "lena":
        p = np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1)
        return np.roll(p, 8 * seed, axis=2)[:, :W, :W].copy()
    return np.stack([_grey(name, W, 3 * seed + k) for k in range(3)])


MIX = ["lena", "noise", "flat", "binary", "ties"]


def _batch(names, rgb, W=256):
    return np.stack([_image(n, rgb, W, i) for i, n in enumerate(names)])


def _singles(h, planes, b_max, b_min, wk, mse):
    return [h.encode_quadtree(p, b_max, b_min, wk, mse) for p in planes]


def _decodes(h, streams, max_iters=50):
    return [h.decode_quadtree(s, max_iters) for s in streams]


def _same_decode(h, streams, max_iters=50):
    img, avg, it = h.decode_quadtree_batch(streams, max_iters)
    for i, (oimg, oavg, oit) in enumerate(_decodes(h, streams, max_iters)):
        assert (img[i] == oimg).all() and it[i] == oit and avg[i].tobytes() == np.float32(oavg).tobytes(), (i, max_iters)
    return img, avg, it


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("b_max,b_min", PAIRS)
@pytest.mark.parametrize("wk", [0, 2, 20])
def test_mixed_batch_matches_single_calls(h, rgb, b_max, b_min, wk):
    planes = _batch(MIX, rgb)
    leaves = set()
    for mse in MSES:
        got = h.encode_quadtree_batch(planes, b_max, b_min, wk, mse)
        want = _singles(h, planes, b_max, b_min, wk, mse)
        assert got == want, mse
        leaves.update(struct.unpack(">i", s[28:32])[0] for s in got)
        if mse == 25.0:
            _same_decode(h, got)
    if b_min < b_max:  # from no splits to all splits
        assert len(leaves) > 2


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("n", [1, 2, 5, 64])
@pytest.mark.parametrize("wk", [0, 2])
def test_batch_sizes(h, fic, rgb, n, wk):
    names = [MIX[i % len(MIX)] for i in range(n)]
    planes = _batch(names, rgb)
    got = h.encode_quadtree_batch(planes, 16, 8, wk, 25.0)
    t = h.timings()
    assert got == _singles(h, planes, 16, 8, wk, 25.0)
    if wk == 0 and n >= 4:
        assert t.engine == fic.FIC_ENGINE_UMMA  # the tcgen05 group search at the finest level
    if wk == 2:
        assert t.engine == fic.FIC_ENGINE_FUSED
    _same_decode(h, got)


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("engine,wk", [("DIRECT", 0), ("DIRECT", 2), ("FUSED", 2), ("UMMA", 0)])
def test_forced_engines(h, fic, rgb, engine, wk):
    h.set_engine(getattr(fic, "FIC_ENGINE_" + engine))
    planes = _batch(MIX, rgb)
    for b_max, b_min in [(16, 8), (16, 4)]:
        got = h.encode_quadtree_batch(planes, b_max, b_min, wk, 25.0)
        assert h.timings().engine == getattr(fic, "FIC_ENGINE_" + engine)
        assert got == _singles(h, planes, b_max, b_min, wk, 25.0)


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_two_tensor_core_groups(h, fic, rgb):
    # 260 whole-pool images of 128^2: B = 8 runs the tcgen05 group search, at most 256 images a group
    planes = np.stack([_image(MIX[i % 5], rgb, 128, i) for i in range(260)])
    got = h.encode_quadtree_batch(planes, 16, 8, 0, 25.0)
    assert h.timings().engine == fic.FIC_ENGINE_UMMA
    assert got == _singles(h, planes, 16, 8, 0, 25.0)
    _same_decode(h, got[:7] + got[-7:])


def test_streams_match_the_oracle(h):
    from oracle import quadtree, quadtree_rgb

    quadtree.build()
    quadtree_rgb.build()
    for rgb, enc, dec in [(False, quadtree.encode_quadtree, quadtree.decode_quadtree),
                          (True, quadtree_rgb.encode_quadtree_rgb, quadtree_rgb.decode_quadtree_rgb)]:
        planes = _batch(["lena", "ties", "binary"], rgb)
        got = h.encode_quadtree_batch(planes, 16, 4, 2, 25.0)
        for p, s in zip(planes, got):
            assert s == enc(p, 16, 4, 2, 25.0, nthreads=16)
        img, avg, it = h.decode_quadtree_batch(got)
        for i, s in enumerate(got):
            oimg, oavg, oit = dec(s)
            assert (img[i] == oimg).all() and it[i] == oit and avg[i].tobytes() == np.float32(oavg).tobytes()


def _never_converges(s, rgb):
    """Stream s with every leaf set to a = -10 and a large offset: its pixels flip between 0 and 255 every sweep."""
    n = struct.unpack(">i", s[28:32])[0]
    W, b_max = struct.unpack(">i", s[4:8])[0], struct.unpack(">i", s[20:24])[0]
    ntop = (W // b_max) * (struct.unpack(">i", s[8:12])[0] // b_max)
    off = 32 + ntop + (-ntop % 4)
    S = 5 if rgb else 3
    leaves = np.frombuffer(s, ">i4", count=S * n, offset=off).reshape(n, S).copy()
    if rgb:
        leaves[:, 1] = -10_000_000
        leaves[:, 2:4] = 100_000_000
        leaves[:, 4] = 1000
    else:
        leaves[:, 1] = -1000
        leaves[:, 2] = 1000
    return s[:off] + leaves.astype(">i4").tobytes()


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_decodes_converge_at_different_sweeps(h, rgb):
    planes = _batch(["flat", "noise", "lena", "structured", "noise"], rgb)
    streams = h.encode_quadtree_batch(planes, 16, 4, 2, 25.0)
    streams[4] = _never_converges(streams[4], rgb)
    for max_iters in (1, 8, 9, 50):
        img, avg, it = _same_decode(h, streams, max_iters)
        if max_iters == 50:
            assert it[4] == 50 and len(set(it.tolist())) > 1


def _raw_encode(fic, h, planes, rgb, b_max, b_min, wk, mse, stride, n=None, null=None):
    L = fic._lib.load()
    n = planes.shape[0] if n is None else n
    buf = np.zeros(max(planes.shape[0] * stride, 1), np.uint8)
    sizes = np.zeros(planes.shape[0], np.uintp)
    args = [planes.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p), sizes.ctypes.data_as(C.c_void_p)]
    if null is not None:
        args[null] = None
    mode = fic.FIC_MODE_RGB_QT if rgb else fic.FIC_MODE_GREY_QT
    rc = L.fic_encode_quadtree_batch(h._h, mode, args[0], n, planes.shape[-1], planes.shape[-2], b_max, b_min, wk, mse,
                                     args[1], stride, args[2])
    return rc, buf, sizes


def _raw_decode(fic, h, mode, streams, stride=None):
    L = fic._lib.load()
    stride = stride or max(len(s) for s in streams)
    buf = np.zeros(len(streams) * stride, np.uint8)
    for i, s in enumerate(streams):
        buf[i * stride:i * stride + len(s)] = np.frombuffer(s, np.uint8)
    nb = np.array([len(s) for s in streams], np.uintp)
    out = np.zeros((len(streams), 3, 256, 256), np.uint8)
    rc = L.fic_decode_quadtree_batch(h._h, mode, len(streams), buf.ctypes.data_as(C.c_void_p), stride,
                                     nb.ctypes.data_as(C.c_void_p), 50, out.ctypes.data_as(C.c_void_p), None, None)
    return rc, L.fic_last_error(h._h).decode()


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_stride(h, fic, rgb):
    planes = _batch(MIX, rgb)
    want = _singles(h, planes, 16, 4, 2, 25.0)
    longest = max(len(s) for s in want)
    rc, buf, sizes = _raw_encode(fic, h, planes, rgb, 16, 4, 2, 25.0, longest - 1)
    assert rc == fic._lib.FIC_E_ARG and sizes.tolist() == [len(s) for s in want]
    rc, buf, sizes = _raw_encode(fic, h, planes, rgb, 16, 4, 2, 25.0, longest)
    assert rc == fic._lib.FIC_OK
    assert [buf[i * longest:i * longest + int(sizes[i])].tobytes() for i in range(5)] == want


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_rejections(h, fic, rgb):
    E_ARG, E_STREAM = fic._lib.FIC_E_ARG, fic._lib.FIC_E_STREAM
    mode = fic.FIC_MODE_RGB_QT if rgb else fic.FIC_MODE_GREY_QT
    planes = _batch(MIX, rgb)
    stride = 1 << 20
    assert _raw_encode(fic, h, planes, rgb, 16, 4, 2, 25.0, stride, n=0)[0] == E_ARG
    assert _raw_encode(fic, h, planes, rgb, 16, 4, 2, float("nan"), stride)[0] == E_ARG
    for k in range(3):
        assert _raw_encode(fic, h, planes, rgb, 16, 4, 2, 25.0, stride, null=k)[0] == E_ARG
    streams = h.encode_quadtree_batch(planes, 16, 4, 2, 25.0)
    assert _raw_decode(fic, h, mode, streams)[0] == fic._lib.FIC_OK
    # mixed geometry at image 3 (other levels, then another window)
    other = h.encode_quadtree_batch(planes[3:4], 16, 8, 2, 25.0)[0]
    rc, msg = _raw_decode(fic, h, mode, streams[:3] + [other] + streams[4:])
    assert rc == E_STREAM and "image 3" in msg
    other = h.encode_quadtree_batch(planes[3:4], 16, 4, 3, 25.0)[0]
    assert _raw_decode(fic, h, mode, streams[:3] + [other] + streams[4:])[0] == E_STREAM
    # a stream of the other mode at image 2
    alt = _batch(MIX[:1], not rgb)
    other = h.encode_quadtree_batch(alt, 16, 4, 2, 25.0)[0]
    rc, msg = _raw_decode(fic, h, mode, streams[:2] + [other] + streams[3:])
    assert rc == E_STREAM and "image 2" in msg
    # a truncated stream at image 4
    rc, msg = _raw_decode(fic, h, mode, streams[:4] + [streams[4][:-1]])
    assert rc == E_STREAM and "image 4" in msg
    # an out-of-pool leaf at image 1: caught by the device
    ntop = 256
    bad = bytearray(streams[1])
    bad[32 + ntop:36 + ntop] = struct.pack(">i", 1 << 24)
    rc, msg = _raw_decode(fic, h, mode, streams[:1] + [bytes(bad)] + streams[2:])
    assert rc == E_STREAM and "image 1" in msg and "pool" in msg
    # NULL arrays, n = 0, a mode that is not a quadtree mode
    L = fic._lib.load()
    buf = np.zeros(16, np.uint8)
    nb = np.zeros(1, np.uintp)
    p = buf.ctypes.data_as(C.c_void_p)
    assert L.fic_decode_quadtree_batch(h._h, mode, 0, p, 16, nb.ctypes.data_as(C.c_void_p), 50, p, None, None) == E_ARG
    assert L.fic_decode_quadtree_batch(h._h, mode, 1, None, 16, nb.ctypes.data_as(C.c_void_p), 50, p, None, None) == E_ARG
    assert L.fic_decode_quadtree_batch(h._h, mode, 1, p, 16, None, 50, p, None, None) == E_ARG
    assert L.fic_decode_quadtree_batch(h._h, mode, 1, p, 16, nb.ctypes.data_as(C.c_void_p), 50, None, None, None) == E_ARG
    assert L.fic_decode_quadtree_batch(h._h, fic.FIC_MODE_GREY, 1, p, 16, nb.ctypes.data_as(C.c_void_p), 50, p, None, None) == E_ARG


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("wk", [0, 2])
def test_launches_do_not_grow_with_the_batch(h, rgb, wk):
    launches = []
    for n in (8, 64):
        planes = np.stack([_image(MIX[i % 5], rgb, 256, i) for i in range(n)])
        h.encode_quadtree_batch(planes, 16, 8, wk, 25.0)
        launches.append(h.timings().launches)
    assert launches[0] == launches[1]
    s = h.encode_quadtree(_image("lena", rgb), 16, 8, wk, 25.0)
    h.decode_quadtree(s)
    single = h.timings().launches
    h.decode_quadtree_batch([s] * 16)
    assert h.timings().launches == single
