"""The RGB quadtree extension (FIC_MODE_RGB_QT) on the GPU: streams and decodes bit-identical to the CPU oracle, the
degenerate trees against the fixed-block RGB entries and the reference's unknown.run, the CUDA-core engine against AUTO,
a 2048^2 full pool against per-level GPU encodes, random trees with saturating leaves, and the rejections."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

from conftest import GOLD
from test_gpu_ext_decode import _levels, _same, _wk_l, qt_leaves, random_flags

pytestmark = pytest.mark.gpu

MSES = [-1.0, 0.0, 4.0, 25.0, 100.0, np.inf]
I32_MAX = 2**31 - 1


def _structured_rgb(W, H, seed):
    from fractal_image_compression_b200 import synth

    return np.stack([synth.structured(W, H, seed + k) for k in range(3)])


def _lena():
    return np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1).copy()


def _planes(name):
    from fractal_image_compression_b200 import synth

    if name == "lena":
        return _lena()
    if name == "structured512":
        return _structured_rgb(512, 512, 7)
    if name == "noise512":
        return np.stack([synth.noise(512, 512, 9 + k) for k in range(3)])
    if name == "structured512x256":
        return _structured_rgb(512, 256, 11)
    if name == "grey_as_rgb":
        g = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
        return np.stack([g, g, g])
    if name == "binary":  # per-channel 0 / 255: at B = 16 the reference's float RGB covariance rounds
        return np.stack([((synth.noise(128, 128, 13 + k) >> 7) * 255).astype(np.uint8) for k in range(3)])
    if name == "flat":
        return np.stack([np.full((128, 128), v, np.uint8) for v in (77, 140, 3)])
    if name == "ties":  # a few repeated 8 x 8 tiles: many equal scores
        t = np.stack([synth.noise(8, 8, 17 + k) for k in range(3)])
        return np.tile(np.concatenate([t, t[:, ::-1]], 1), (1, 8, 16))
    raise KeyError(name)


@pytest.fixture(scope="module")
def fic():
    import fractal_image_compression_b200 as f

    return f


@pytest.fixture(scope="module")
def h(fic):
    hh = fic.Handle(0)
    yield hh
    hh.close()


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree_rgb

    quadtree_rgb.build()
    return quadtree_rgb


CASES = [("lena", 16, 8, 2), ("lena", 16, 4, 0), ("lena", 8, 4, 4), ("structured512", 16, 8, 0), ("noise512", 16, 4, 3),
         ("structured512x256", 16, 4, 3), ("grey_as_rgb", 16, 4, 2), ("binary", 16, 8, 5), ("flat", 16, 4, 0),
         ("ties", 16, 4, 0)]


@pytest.mark.parametrize("name,b_max,b_min,wk", CASES)
def test_stream_and_decode_match_oracle(h, name, b_max, b_min, wk, qt):
    planes = _planes(name)
    for mse in MSES:
        got = h.encode_quadtree(planes, b_max, b_min, wk, mse)
        want = qt.encode_quadtree_rgb(planes, b_max, b_min, wk, mse, nthreads=16)
        assert got == want, (name, mse)
        img, avg, it = h.decode_quadtree(got)
        assert img.shape == planes.shape
        _same((img, avg, it), qt.decode_quadtree_rgb(want))


def test_decode_1024_matches_oracle(h, qt):
    planes = _structured_rgb(1024, 1024, 21)
    for b_max, b_min, mse in [(16, 4, 25.0), (16, 8, 4.0)]:
        s = h.encode_quadtree(planes, b_max, b_min, 2, mse)
        _same(h.decode_quadtree(s), qt.decode_quadtree_rgb(s))


def _leaves(s):
    W, H, b_max, n = struct.unpack(">i", s[4:8])[0], struct.unpack(">i", s[8:12])[0], struct.unpack(">i", s[20:24])[0], \
        struct.unpack(">i", s[28:32])[0]
    ntop = (W // b_max) * (H // b_max)
    return np.frombuffer(s, ">i4", count=5 * n, offset=32 + ntop + (-ntop % 4)).reshape(n, 5).astype(np.int32), ntop


@pytest.mark.parametrize("b_max,b_min,wk", [(16, 8, 2), (16, 4, 0), (8, 4, 0)])
def test_degenerate_trees(h, b_max, b_min, wk):
    planes = _lena()
    full = lambda B: wk or 2 * (256 // B) - 3  # noqa: E731
    _, q_max = h.encode_u8(planes, b_max, full(b_max))
    _, q_min = h.encode_u8(planes, b_min, full(b_min))
    s = h.encode_quadtree(planes, b_max, b_min, wk, np.inf)
    leaves, ntop = _leaves(s)
    assert (leaves == q_max).all()
    leaves, _ = _leaves(h.encode_quadtree(planes, b_max, b_min, wk, -1.0))
    assert sorted(map(tuple, leaves.tolist())) == sorted(map(tuple, q_min.tolist()))
    img, avg, it = h.decode_quadtree(s)
    fimg, favg, fit = h.decode_u8(q_max, 256, 256, b_max, full(b_max), True)
    assert (img == fimg).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == np.float32(favg).tobytes()


def test_unknown_run_pin(h, oracle, qt):
    """LenaColored at (8, 4), wk 2, never split: the leaves are the reference's own stream, and the decode is its decode."""
    ref = open(os.path.join(GOLD, "unknown_run.bin"), "rb").read()
    s = h.encode_quadtree(_lena(), 8, 4, 2, np.inf)
    assert struct.unpack(">8i", s[:32]) == (4, 256, 256, 0, 2, 8, 4, 1024)
    assert s[32:32 + 1024] == bytes(1024) and s[32 + 1024:] == ref[20:]
    img, avg, it = h.decode_quadtree(s)
    fimg, favg, fit = oracle.decode(ref)
    assert (img == qt.argb_to_planes(fimg)).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == np.float32(favg).tobytes()


def test_direct_engine_gives_the_same_stream(h, fic):
    planes = _lena()
    want = [h.encode_quadtree(planes, 16, 4, wk, 25.0) for wk in (2, 0)]
    h.set_engine(fic.FIC_ENGINE_DIRECT)
    try:
        assert [h.encode_quadtree(planes, 16, 4, wk, 25.0) for wk in (2, 0)] == want
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)


def test_2048_full_pool_against_level_encodes(h):
    planes = _structured_rgb(2048, 2048, 5)
    wk = dpw = 2 * 128 - 3
    q16 = h.encode_u8(planes, 16, wk)[1]
    q8 = h.encode_u8(planes, 8, 2 * 256 - 3)[1]
    ntop = len(q16)
    # every flag from a numpy recomputation of E of the 16 x 16 codes on the source's RGB decimation (the fourth tap
    # re-reads p01, FC:945-947; no x + 1 >= H slip on a square image)
    p = planes.astype(np.int64)
    dec = (p[:, 0::2, 0::2] + p[:, 0::2, 1::2] + 2 * p[:, 1::2, 0::2]) // 4
    c = q16[:, 0].astype(np.float32)
    # the whole pool: the window origin is 0 (generateKernel clamps it), so the codebook index is c itself
    idx = np.trunc(c / np.float32(wk)).astype(np.int64) * dpw + np.trunc(np.fmod(c, np.float32(wk))).astype(np.int64)
    a = q16[:, 1].astype(np.float32) / np.float32(1000000)
    bs = [q16[:, 2].astype(np.float32) / np.float32(100000), q16[:, 3].astype(np.float32) / np.float32(100000),
          q16[:, 4].astype(np.float32)]
    r, col = (idx // dpw) * 4, (idx % dpw) * 4
    ii = np.arange(16)
    E = np.zeros(ntop, np.int64)
    for ch in range(3):
        dblk = dec[ch][(r[:, None, None] + ii[None, :, None]), (col[:, None, None] + ii[None, None, :])]
        v = np.clip(np.trunc(a[:, None, None] * dblk.astype(np.float32) + bs[ch][:, None, None]), 0, 255).astype(np.int64)
        src = p[ch].reshape(128, 16, 128, 16).transpose(0, 2, 1, 3).reshape(-1, 16, 16)
        E += ((v - src) ** 2).sum(axis=(1, 2))
    # a threshold inside the range of E, so that the tree mixes both levels
    mse = float(np.median(E)) / 768.0
    s = h.encode_quadtree(planes, 16, 8, 0, mse)
    t = h.timings()
    assert t.launches > 0 and t.search_evals > 0
    leaves, _ = _leaves(s)
    flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
    assert ((flags & 1) == (E.astype(np.float64) > mse * 768.0)).all()
    assert 0 < (flags & 1).sum() < ntop
    assert not (flags & ~np.uint8(1)).any()
    # every leaf: the level encode's code of that range
    k = 0
    for t_ in range(ntop):
        if not flags[t_] & 1:
            assert (leaves[k] == q16[t_]).all()
            k += 1
            continue
        y, x = divmod(t_, 128)
        for kk in range(4):
            assert (leaves[k] == q8[(2 * y + (kk >> 1)) * 256 + 2 * x + (kk & 1)]).all()
            k += 1
    assert k == len(leaves)


# ---------------------------------------------------------------- decoder on random trees

def rgb_stream(W, H, b_max, b_min, wk, flags, codes):
    """A FIC_MODE_RGB_QT stream: header 4, W, H, 0, wk, b_max, b_min, n_leaves; the flag bytes, zero-padded to a multiple
    of 4; 20 big-endian bytes per leaf."""
    flags = np.asarray(flags, np.uint8)
    codes = np.asarray(codes, np.int64).astype(np.int32)
    return (struct.pack(">8i", 4, W, H, 0, wk, b_max, b_min, len(codes)) + flags.tobytes() + bytes(-len(flags) % 4) +
            codes.astype(">i4").tobytes())


def random_rgb_codes(rng, W, b_max, wk, leaves, extreme=False):
    """Random leaf codes: c inside the leaf's level window, a * 1e6 in [-1.2e6, 1.2e6], bR, bG * 1e5 in [-1e7, 3e7],
    bB in [-100, 300], one eighth flat; with `extreme` one leaf in sixteen takes a and the b's = +-(2^31 - 1)."""
    n = len(leaves)
    wkl = np.array([_wk_l(W, b_max >> L, wk) for L, _ in leaves], np.int64)
    c = np.empty((n, 5), np.int64)
    c[:, 0] = (rng.random(n) * wkl * wkl).astype(np.int64)
    c[:, 1] = rng.integers(-1200000, 1200001, n)
    c[:, 2:4] = rng.integers(-10000000, 30000001, (n, 2))
    c[:, 4] = rng.integers(-100, 301, n)
    c[rng.permutation(n)[: n // 8], 1] = 0
    if extreme:
        sel = rng.permutation(n)[: max(n // 16, 4)]
        c[sel, 1:] = rng.choice([-I32_MAX, I32_MAX], (len(sel), 4))
    return c


def test_stream_builder_matches_the_encoder(fic, h, qt):
    planes = _lena()
    for b_max, b_min, wk in [(16, 4, 2), (16, 8, 0), (8, 4, 3), (16, 16, 2)]:
        s = h.encode_quadtree(planes, b_max, b_min, wk, 25.0)
        ntop = (256 // b_max) ** 2
        flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
        codes, _ = _leaves(s)
        assert len(qt_leaves(256, 256, b_max, b_min, flags)) == len(codes)
        assert rgb_stream(256, 256, b_max, b_min, wk, flags, codes) == s
        assert fic.quadtree_stream_info(s) == (256, 256, b_max, b_min, wk, len(codes))


PAIRS = [(16, 16), (8, 8), (16, 8), (8, 4), (16, 4)]
# top blocks (across, down) and window: 81, 42 and 15 top blocks (1, 2, 3 mod 4), whole pool and small windows
QT_SHAPES = [(9, 9, 0), (9, 9, 2), (7, 6, 5), (6, 7, 3), (3, 5, 3), (5, 3, 2)]


@pytest.mark.parametrize("b_max,b_min", PAIRS)
@pytest.mark.parametrize("tx,ty,wk", QT_SHAPES)
def test_random_trees(h, qt, b_max, b_min, tx, ty, wk):
    W, H = tx * b_max, ty * b_max
    rng = np.random.default_rng(b_max * 1000 + b_min * 100 + tx * 10 + ty + wk)
    for extreme in (False, True):
        flags = random_flags(rng, tx * ty, _levels(b_max, b_min))
        codes = random_rgb_codes(rng, W, b_max, wk, qt_leaves(W, H, b_max, b_min, flags), extreme)
        s = rgb_stream(W, H, b_max, b_min, wk, flags, codes)
        for max_iters in (50, 2, 17):
            _same(h.decode_quadtree(s, max_iters), qt.decode_quadtree_rgb(s, max_iters))


@pytest.mark.parametrize("W,H,b_max,b_min,wk", [(2304, 2048, 16, 4, 3)])  # above 4 MB of planes: one output copy at the end
def test_large_random_tree(h, qt, W, H, b_max, b_min, wk):
    rng = np.random.default_rng(W + b_min)
    flags = random_flags(rng, (W // b_max) * (H // b_max), _levels(b_max, b_min))
    codes = random_rgb_codes(rng, W, b_max, wk, qt_leaves(W, H, b_max, b_min, flags), extreme=True)
    s = rgb_stream(W, H, b_max, b_min, wk, flags, codes)
    for max_iters in (50, 9):
        _same(h.decode_quadtree(s, max_iters), qt.decode_quadtree_rgb(s, max_iters))


def _refused(fic, h, qt, s):
    with pytest.raises(fic.FicError) as e:
        h.decode_quadtree(s)
    assert e.value.code == fic._lib.FIC_E_STREAM
    with pytest.raises(fic.FicError) as e:
        fic.quadtree_stream_info(s)
    assert e.value.code == fic._lib.FIC_E_STREAM
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(s)


@pytest.mark.parametrize("b_max,b_min", [(16, 4), (16, 8), (8, 4), (16, 16)])
@pytest.mark.parametrize("tx,ty,wk", [(9, 7, 3), (5, 5, 0)])
def test_pool_edge(fic, h, qt, b_max, b_min, tx, ty, wk):
    """The last leaf (the bottom-right block of the finest level, whose window is clamped to the pool's corner) at the
    last pool block decodes like the oracle; one past it is refused, by the host parser and by the device check."""
    W, H = tx * b_max, ty * b_max
    nl = _levels(b_max, b_min)
    rng = np.random.default_rng(tx + b_max + b_min)
    flags = random_flags(rng, tx * ty, nl)
    flags[-1] = {1: 0, 2: 1, 3: 1 | (2 << 3)}[nl]
    leaves = qt_leaves(W, H, b_max, b_min, flags)
    codes = random_rgb_codes(rng, W, b_max, wk, leaves)
    L_last, j_last = leaves[-1]
    B = b_max >> L_last
    assert L_last == nl - 1 and j_last == (W // B) * (H // B) - 1
    wkl = _wk_l(W, B, wk)
    codes[-1, 0] = wkl * wkl - 1
    s = rgb_stream(W, H, b_max, b_min, wk, flags, codes)
    assert fic.quadtree_stream_info(s)[5] == len(leaves)
    _same(h.decode_quadtree(s), qt.decode_quadtree_rgb(s))
    codes[-1, 0] = wkl * wkl
    bad = rgb_stream(W, H, b_max, b_min, wk, flags, codes)
    _refused(fic, h, qt, bad)
    out = np.zeros((3, H, W), np.uint8)
    rc = fic._lib.load().fic_decode_quadtree_rgb(h._h, np.frombuffer(bad, np.uint8).ctypes.data_as(C.c_void_p), len(bad),
                                                 50, out.ctypes.data_as(C.c_void_p), None, None)
    assert rc == fic._lib.FIC_E_STREAM


# ---------------------------------------------------------------- rejections

def test_rejections(h, fic):
    L = fic._lib.load()
    planes = _lena()
    ap = planes.ctypes.data_as(C.c_void_p)
    cap = L.fic_quadtree_rgb_stream_bound(256, 256, 16, 4)
    assert cap == 32 + 256 + 20 * 64 * 64
    buf = np.zeros(cap, np.uint8)
    n = C.c_size_t(0)

    def enc(W, H, bmax, bmin, wk, mse, capacity=cap):
        return L.fic_encode_quadtree_rgb(h._h, ap, W, H, bmax, bmin, wk, mse, buf.ctypes.data_as(C.c_void_p), capacity, C.byref(n))

    assert enc(256, 256, 32, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 4, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 8, 16, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 2, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(248, 256, 16, 4, 2, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 128, 16, 4, 0, 4.0) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 4, 2, float("nan")) == fic._lib.FIC_E_ARG
    assert L.fic_encode_quadtree_rgb(h._h, None, 256, 256, 16, 4, 2, 4.0, buf.ctypes.data_as(C.c_void_p), cap, C.byref(n)) == fic._lib.FIC_E_ARG
    assert enc(256, 256, 16, 4, 2, 25.0) == fic._lib.FIC_OK
    t = h.timings()
    assert t.launches > 0 and t.search_evals > 0 and t.total_ms > 0
    need = n.value
    assert enc(256, 256, 16, 4, 2, 25.0, need - 1) == fic._lib.FIC_E_ARG and n.value == need
    s = buf[:need].tobytes()
    assert fic.quadtree_stream_info(s) == (256, 256, 16, 4, 2, struct.unpack(">i", s[28:32])[0])
    out = np.zeros((3, 256, 256), np.uint8)
    sb = np.frombuffer(s, np.uint8)
    assert L.fic_decode_quadtree_rgb(h._h, sb.ctypes.data_as(C.c_void_p), len(s), 0, out.ctypes.data_as(C.c_void_p), None, None) == fic._lib.FIC_E_ARG

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
    bad = np.frombuffer(bytes(bad), np.uint8)
    rc = L.fic_decode_quadtree_rgb(h._h, bad.ctypes.data_as(C.c_void_p), len(bad), 50, out.ctypes.data_as(C.c_void_p), None, None)
    assert rc == fic._lib.FIC_E_STREAM

    # cross-mode: the grey entries refuse an RGB stream and the RGB entries a grey one, with FIC_E_STREAM
    grey = h.encode_quadtree(planes[0], 16, 4, 2, 25.0)
    gb = np.frombuffer(grey, np.uint8)
    v = [C.c_int() for _ in range(5)]
    cnt = C.c_int64()
    assert L.fic_quadtree_stream_info(sb.ctypes.data_as(C.c_void_p), len(s), *[C.byref(x) for x in v], C.byref(cnt)) == fic._lib.FIC_E_STREAM
    assert L.fic_quadtree_rgb_stream_info(gb.ctypes.data_as(C.c_void_p), len(grey), *[C.byref(x) for x in v], C.byref(cnt)) == fic._lib.FIC_E_STREAM
    assert L.fic_quadtree_rgb_stream_info(sb.ctypes.data_as(C.c_void_p), len(s), *[C.byref(x) for x in v], C.byref(cnt)) == fic._lib.FIC_OK
    big = np.zeros((3, 256, 256), np.uint8)
    assert L.fic_decode_quadtree(h._h, sb.ctypes.data_as(C.c_void_p), len(s), 50, big.ctypes.data_as(C.c_void_p), None, None) == fic._lib.FIC_E_STREAM
    assert not big.any()
    assert L.fic_decode_quadtree_rgb(h._h, gb.ctypes.data_as(C.c_void_p), len(grey), 50, big.ctypes.data_as(C.c_void_p), None, None) == fic._lib.FIC_E_STREAM
    assert not big.any()
    # the fixed-block header parser refuses an RGB quadtree stream (blockgroesse 0)
    off = C.c_size_t()
    assert L.fic_stream_read_header(sb.ctypes.data_as(C.c_void_p), len(s), *[C.byref(x) for x in v], C.byref(off)) == fic._lib.FIC_E_STREAM
    # a fixed-block entry that takes a mode rejects FIC_MODE_RGB_QT through its geometry check
    q = np.zeros((1024, 5), np.int32)
    assert L.fic_decode_u8(h._h, fic.FIC_MODE_RGB_QT, 256, 256, 8, 2, q.ctypes.data_as(C.c_void_p), 50,
                           big.ctypes.data_as(C.c_void_p), None, None) == fic._lib.FIC_E_ARG
