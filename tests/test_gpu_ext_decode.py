"""The two extension decoders on inputs our own encoder never writes, against the CPU oracle: the isometry decoder
(FIC_MODE_GREY_ISO) on random codes and out-of-range isometry indices, the quadtree decoder (FIC_MODE_GREY_QT) on random
trees with random and saturating leaves, and the quadtree encoder at its split threshold and on padded shapes.  A decode
matches when the pixels, the avgError bits and the sweep count are the oracle's."""
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ISO = 2  # FIC_MODE_GREY_ISO
I32_MAX = 2**31 - 1


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
def oracle():
    from oracle import oracle as O

    O.build()
    return O


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree

    quadtree.build()
    return quadtree


def _red(argb):
    return ((argb.view(np.uint32) >> 16) & 0xFF).astype(np.uint8)


def _same(got, want):
    """(image, avgError, sweeps) of a GPU decode against the oracle's; images as ARGB ints or 8-bit planes."""
    img, avg, it = got
    oimg, oavg, oit = want
    if img.dtype == np.uint8 and oimg.dtype != np.uint8:
        oimg = _red(oimg)
    assert it == oit, (it, oit)
    assert np.float32(avg).tobytes() == np.float32(oavg).tobytes(), (avg, oavg)
    assert (img == oimg).all(), int((img != oimg).sum())


# ---------------------------------------------------------------- isometry decoder on random codes

def _iso_codes(rng, W, H, B, wk):
    """Random window-local indices, a * 100 in [-120, 120], b in [-100, 300], one eighth of the blocks flat, and every
    isometry 0..7 on the same number of blocks (+- 1)."""
    nr = (W // B) * (H // B)
    q = np.empty((nr, 4), np.int32)
    q[:, 0] = rng.integers(0, wk * wk, nr)
    q[:, 1] = rng.integers(-120, 121, nr)
    q[:, 2] = rng.integers(-100, 301, nr)
    q[:, 3] = rng.permutation(np.arange(nr) % 8)
    q[rng.permutation(nr)[: nr // 8], 1] = 0
    assert set(q[:, 3].tolist()) == set(range(8))
    return q


def _oscillating(rng, c):
    """Contrast -3 .. -1.5 about the mid grey: every sweep flips the image between dark and bright, so the decode never
    converges and the sum of squared changes passes 2^24."""
    a = rng.integers(-300, -150, len(c))
    c[:, 1] = a
    c[:, 2] = (128 * (100 - a)) // 100 + rng.integers(-20, 21, len(c))
    return c


def _full(W, B):
    return 2 * W // B - 3


ISO_SHAPES = ([(128, 128, B, wk) for B in (4, 8, 16) for wk in (2, 3, 5, _full(128, B))] +
              [(272, 144, B, 5) for B in (4, 8, 16)] + [(144, 272, B, 3) for B in (4, 8, 16)] +
              [(264, 136, 8, 5),    # W % 16 == 8
               (100, 60, 4, 3)])    # W % 8 != 0


@pytest.mark.parametrize("W,H,B,wk", ISO_SHAPES)
def test_iso_random_codes(fic, h, oracle, W, H, B, wk):
    rng = np.random.default_rng(W * 7 + H * 3 + B * 11 + wk)
    q = _iso_codes(rng, W, H, B, wk)
    stream = fic.stream_write(q, W, H, B, wk, ISO)
    want = oracle.decode(stream)
    _same(h.decode(q, W, H, B, wk, ISO), want)
    _same(h.decode_u8(q, W, H, B, wk, ISO), want)


@pytest.mark.parametrize("W,H,B,wk", [(128, 128, 4, 3), (128, 128, 8, _full(128, 8)), (128, 128, 16, 2), (144, 272, 8, 3),
                                      (100, 60, 4, 2)])
def test_iso_batch_random_codes(fic, h, oracle, W, H, B, wk):
    """fic_decode_batch with three images and three carried-in avgErrors, each image against the oracle."""
    rng = np.random.default_rng(B * 101 + wk + W)
    q = np.stack([_iso_codes(rng, W, H, B, wk) for _ in range(3)])
    carries = np.array([0.0, 0.5863342, 3.5e7], np.float32)
    img, avg, it = h.decode_batch(q, W, H, B, wk, ISO, avg_error=carries.copy())
    for i in range(3):
        want = oracle.decode(fic.stream_write(q[i], W, H, B, wk, ISO), avg_error_in=float(carries[i]))
        _same((img[i], avg[i], it[i]), want)


@pytest.mark.parametrize("max_iters", [1, 2, 8, 9, 50])
def test_iso_iteration_limits(fic, h, oracle, max_iters):
    """Sweeps are enqueued eight at a time; every limit around the batch boundary must stop where a sweep-by-sweep
    loop with that limit stops, on a converging stream (the oracle's own encode) and on one that never converges."""
    from conftest import GOLD
    import os

    plane = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    lena = fic.synth.grey_to_argb(plane)
    enc = oracle.write_data(oracle.encode(lena, 8, 3, iso=True, nthreads=8), 256, 256, 8, 3, iso=True)
    rng = np.random.default_rng(5)
    rnd = _oscillating(rng, _iso_codes(rng, 128, 128, 4, 5))
    for stream in (enc, fic.stream_write(rnd, 128, 128, 4, 5, ISO)):
        mode, W, H, B, wk, q = fic.stream_read(stream)
        assert mode == ISO
        for carry in (0.0, 0.25):
            want = oracle.decode(stream, avg_error_in=carry, max_iters=max_iters)
            _same(h.decode(q, W, H, B, wk, ISO, avg_error=carry, max_iters=max_iters), want)
    assert oracle.decode(enc)[2] < 50 and oracle.decode(fic.stream_write(rnd, 128, 128, 4, 5, ISO))[2] == 50


def test_iso_above_2_24_pixels(fic, h, oracle):
    """4096 x 4104 > 2^24 pixels with isometries: every sweep replays the float running sum, over the per-pixel
    changes of the isometry gather."""
    W, H, B, wk = 4096, 4104, 8, 2
    _, q = h.encode(fic.synth.grey_to_argb(fic.synth.structured(W, H, 3)), B, wk, rgb=ISO)
    assert len(np.unique(q[:, 3])) == 8
    want = oracle.decode(fic.stream_write(q, W, H, B, wk, ISO))
    assert want[2] > 1
    _same(h.decode_u8(q, W, H, B, wk, ISO), want)


OUT_OF_RANGE = [8, 15, -1, -8, 2**24 + 1, 2**25 + 3, 2**31 - 7, I32_MAX, -2**31]


@pytest.mark.parametrize("k", OUT_OF_RANGE)
def test_iso_index_out_of_range(fic, h, oracle, k):
    """An isometry index outside 0..7 is read like every other stream field, through float (FC:372-374), then cast
    and reduced mod 8: 2^24 + 1 reads as 2^24 (isometry 0), 2^31 - 7 saturates to 2^31 - 1 (isometry 7)."""
    W, H, B, wk = 64, 48, 8, 3
    q = _iso_codes(np.random.default_rng(k & 0xFFFF), W, H, B, wk)
    q[:, 3] = k
    stream = fic.stream_write(q, W, H, B, wk, ISO)
    want = oracle.decode(stream)
    _same(h.decode(q, W, H, B, wk, ISO), want)
    _same(h.decode_u8(q, W, H, B, wk, ISO), want)
    # the index must act as the isometry the float read gives
    q2 = q.copy()
    q2[:, 3] = int(np.int32(np.clip(np.float64(np.float32(k)), -2**31, I32_MAX))) & 7
    _same(h.decode(q2, W, H, B, wk, ISO), want)


@pytest.mark.parametrize("B", [4, 8, 16])
def test_iso_index_out_of_range_mixed(fic, h, oracle, B):
    W, H, wk = 96, 64, 2
    rng = np.random.default_rng(B)
    q = np.stack([_iso_codes(rng, W, H, B, wk) for _ in range(3)])
    q[:, :, 3] = np.array(OUT_OF_RANGE + list(range(8)), np.int64)[rng.integers(0, len(OUT_OF_RANGE) + 8, q.shape[:2])]
    for i in range(3):
        _same(h.decode(q[i], W, H, B, wk, ISO), oracle.decode(fic.stream_write(q[i], W, H, B, wk, ISO)))
    img, avg, it = h.decode_batch(q, W, H, B, wk, ISO)
    for i in range(3):
        _same((img[i], avg[i], it[i]), oracle.decode(fic.stream_write(q[i], W, H, B, wk, ISO)))


# ---------------------------------------------------------------- quadtree decoder on random trees

def _wk_l(W, B, wk):
    """The window of level B: wk, or (wk == 0) the level's whole pool."""
    return wk if wk else 2 * (W // B) - 3


def _levels(b_max, b_min):
    return {16: 1, 8: 2, 4: 3}[b_min] - {16: 0, 8: 1}[b_max]


def qt_leaves(W, H, b_max, b_min, flags):
    """(level, range index) of every leaf in stream order: depth first, children in raster order."""
    rpw = [W // (b_max >> L) for L in range(3)]
    out = []
    for t, f in enumerate(flags):
        if not f & 1:
            out.append((0, t))
            continue
        for k in range(4):
            j1 = (2 * (t // rpw[0]) + (k >> 1)) * rpw[1] + 2 * (t % rpw[0]) + (k & 1)
            if not (f >> (1 + k)) & 1:
                out.append((1, j1))
                continue
            for k2 in range(4):
                out.append((2, (2 * (j1 // rpw[1]) + (k2 >> 1)) * rpw[2] + 2 * (j1 % rpw[1]) + (k2 & 1)))
    return out


def qt_stream(W, H, b_max, b_min, wk, flags, codes):
    """A FIC_MODE_GREY_QT stream: header 3, W, H, 0, wk, b_max, b_min, n_leaves; one flag byte per top block, zero-padded
    to a multiple of 4; 12 big-endian bytes per leaf."""
    flags = np.asarray(flags, np.uint8)
    codes = np.asarray(codes, np.int64).astype(np.int32)
    pad = -len(flags) % 4
    return (struct.pack(">8i", 3, W, H, 0, wk, b_max, b_min, len(codes)) + flags.tobytes() + bytes(pad) +
            codes.astype(">i4").tobytes())


def random_flags(rng, ntop, nl):
    """Legal flags in which an unsplit top, a split top with unsplit children and (three levels) every child split
    all occur."""
    if nl == 1:
        return np.zeros(ntop, np.uint8)
    f = (rng.random(ntop) < 0.6).astype(np.uint8)
    if nl == 3:
        f |= (rng.random((ntop, 4)) < 0.5).astype(np.uint8).dot(np.array([2, 4, 8, 16], np.uint8)).astype(np.uint8) * f
    f[:3] = [0, 1, 0x1F if nl == 3 else 1]
    return f


def random_codes(rng, W, b_max, wk, leaves, extreme=False):
    """Random leaf codes: c inside the leaf's level window, a * 100 in [-120, 120], b in [-100, 300], one eighth flat;
    with `extreme` one leaf in sixteen takes a, b = +-(2^31 - 1)."""
    n = len(leaves)
    wkl = np.array([_wk_l(W, b_max >> L, wk) for L, _ in leaves], np.int64)
    c = np.empty((n, 3), np.int64)
    c[:, 0] = (rng.random(n) * wkl * wkl).astype(np.int64)
    c[:, 1] = rng.integers(-120, 121, n)
    c[:, 2] = rng.integers(-100, 301, n)
    c[rng.permutation(n)[: n // 8], 1] = 0
    if extreme:
        sel = rng.permutation(n)[: max(n // 16, 4)]
        c[sel, 1:] = rng.choice([-I32_MAX, I32_MAX], (len(sel), 2))
    return c


def random_tree(rng, W, H, b_max, b_min, wk, extreme=False):
    flags = random_flags(rng, (W // b_max) * (H // b_max), _levels(b_max, b_min))
    leaves = qt_leaves(W, H, b_max, b_min, flags)
    return flags, leaves, random_codes(rng, W, b_max, wk, leaves, extreme)


def test_stream_builder_matches_the_encoder(fic, h, qt):
    """The builder writes the encoder's stream from its flags and leaves, and the parser reads back what it wrote."""
    from conftest import GOLD
    import os

    plane = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    for b_max, b_min, wk in [(16, 4, 2), (16, 8, 0), (8, 4, 3), (16, 16, 2)]:
        s = h.encode_quadtree(plane, b_max, b_min, wk, 25.0)
        ntop = (256 // b_max) ** 2
        flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
        n = struct.unpack(">i", s[28:32])[0]
        codes = np.frombuffer(s, ">i4", count=3 * n, offset=32 + ntop + (-ntop % 4)).reshape(n, 3)
        assert len(qt_leaves(256, 256, b_max, b_min, flags)) == n
        assert qt_stream(256, 256, b_max, b_min, wk, flags, codes) == s
    rng = np.random.default_rng(1)
    for W, H, b_max, b_min, wk in [(48, 80, 16, 4, 3), (112, 96, 16, 8, 5), (72, 72, 8, 4, 0), (144, 144, 16, 16, 2)]:
        flags, leaves, codes = random_tree(rng, W, H, b_max, b_min, wk, extreme=True)
        s = qt_stream(W, H, b_max, b_min, wk, flags, codes)
        assert fic.quadtree_stream_info(s) == (W, H, b_max, b_min, wk, len(leaves))
        qt.decode_quadtree(s, 2)   # the oracle accepts it


PAIRS = [(16, 16), (8, 8), (16, 8), (8, 4), (16, 4)]
# top blocks (across, down) and window: 81, 42 and 15 top blocks (1, 2, 3 mod 4), whole pool and small windows
QT_SHAPES = [(9, 9, 0), (9, 9, 2), (7, 6, 5), (6, 7, 3), (3, 5, 3), (5, 3, 2)]


@pytest.mark.parametrize("b_max,b_min", PAIRS)
@pytest.mark.parametrize("tx,ty,wk", QT_SHAPES)
def test_qt_random_trees(fic, h, qt, b_max, b_min, tx, ty, wk):
    W, H = tx * b_max, ty * b_max
    rng = np.random.default_rng(b_max * 1000 + b_min * 100 + tx * 10 + ty + wk)
    for extreme in (False, True):
        flags, leaves, codes = random_tree(rng, W, H, b_max, b_min, wk, extreme)
        s = qt_stream(W, H, b_max, b_min, wk, flags, codes)
        for max_iters in (50, 2):
            _same(h.decode_quadtree(s, max_iters), qt.decode_quadtree(s, max_iters))


@pytest.mark.parametrize("max_iters", [1, 2, 7, 8, 9, 16, 17, 50])
def test_qt_iteration_limits(fic, h, qt, max_iters):
    from conftest import GOLD
    import os

    plane = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    conv = h.encode_quadtree(plane, 16, 4, 2, 25.0)
    assert qt.decode_quadtree(conv)[2] < 50
    rng = np.random.default_rng(3)
    flags, _, codes = random_tree(rng, 160, 96, 16, 4, 3)
    rnd = qt_stream(160, 96, 16, 4, 3, flags, _oscillating(rng, codes))
    assert qt.decode_quadtree(rnd)[2] == 50
    for s in (conv, rnd):
        _same(h.decode_quadtree(s, max_iters), qt.decode_quadtree(s, max_iters))


@pytest.mark.parametrize("W,H,b_max,b_min,wk", [(1456, 1456, 16, 4, 2),   # 8281 top blocks: more than 256 warps of flags
                                                (2304, 2048, 16, 4, 3),   # above 4 Mpixel: the output is copied once at the end
                                                (2304, 2048, 8, 8, 2)])
def test_qt_large_random_trees(fic, h, qt, W, H, b_max, b_min, wk):
    flags, leaves, codes = random_tree(np.random.default_rng(W + b_min), W, H, b_max, b_min, wk, extreme=True)
    s = qt_stream(W, H, b_max, b_min, wk, flags, codes)
    for max_iters in (50, 9):
        _same(h.decode_quadtree(s, max_iters), qt.decode_quadtree(s, max_iters))


def _refused(fic, h, qt, s):
    with pytest.raises(fic.FicError) as e:
        h.decode_quadtree(s)
    assert e.value.code == fic._lib.FIC_E_STREAM
    with pytest.raises(fic.FicError) as e:
        fic.quadtree_stream_info(s)
    assert e.value.code == fic._lib.FIC_E_STREAM
    with pytest.raises(ValueError):
        qt.decode_quadtree(s)


@pytest.mark.parametrize("b_max,b_min", [(16, 4), (16, 8), (8, 4), (16, 16)])
@pytest.mark.parametrize("tx,ty,wk", [(9, 7, 3), (5, 5, 0)])
def test_qt_pool_edge(fic, h, qt, b_max, b_min, tx, ty, wk):
    """Leaves in the last range row and column of their level, where the window is clamped to the pool's corner:
    c = wk_L^2 - 1 is the last pool block, c = wk_L^2 lies below the pool.  A negative c that the window arithmetic
    maps back into the pool decodes like the oracle; one that leaves it (the first range block) is refused."""
    W, H = tx * b_max, ty * b_max
    nl = _levels(b_max, b_min)
    rng = np.random.default_rng(tx + b_max + b_min)
    flags = random_flags(rng, tx * ty, nl)
    flags[-1] = {1: 0, 2: 1, 3: 1 | (2 << 3)}[nl]   # the last top block: unsplit / split / its last child split too
    flags[0] = 0
    leaves = qt_leaves(W, H, b_max, b_min, flags)
    codes = random_codes(rng, W, b_max, wk, leaves)
    # the last leaf is the bottom-right block of the finest level (a b_min leaf under a split child on three levels);
    # the first leaf is top block 0, whose window sits at the pool's origin
    L_last, j_last = leaves[-1]
    B = b_max >> L_last
    assert L_last == nl - 1 and j_last == (W // B) * (H // B) - 1 and leaves[0] == (0, 0)
    wkl = _wk_l(W, B, wk)
    dpw, dph = 2 * (W // B) - 3, 2 * (H // B) - 3

    def in_pool(c, dy, dx):
        """The window arithmetic of calculateIndices (float division and remainder) for window origin (dy, dx)."""
        yd = int(np.trunc(np.float32(c) / np.float32(wkl)))
        xd = int(np.trunc(np.fmod(np.float32(c), np.float32(wkl))))
        return 0 <= xd + dx + (yd + dy) * dpw < dpw * dph

    def stream(c_last, c_first=None):
        c = codes.copy()
        c[-1, 0] = c_last
        if c_first is not None:
            c[0, 0] = c_first
        return qt_stream(W, H, b_max, b_min, wk, flags, c)

    inside = 0
    for c_last in (wkl * wkl - 1, -1, -wkl - 1, -(wkl * wkl - 1), -2 * wkl):
        s = stream(c_last)
        if in_pool(c_last, dph - wkl, dpw - wkl):   # the last range block's window is clamped to the pool's corner
            inside += 1
            assert fic.quadtree_stream_info(s)[5] == len(leaves)
            _same(h.decode_quadtree(s), qt.decode_quadtree(s))
        else:
            _refused(fic, h, qt, s)
    # the last pool block, and (a window smaller than the pool) at least one negative c; the whole pool as the window
    # has its origin at 0, where every negative c falls outside
    assert inside >= (2 if wk else 1)
    assert not in_pool(wkl * wkl, dph - wkl, dpw - wkl)
    _refused(fic, h, qt, stream(wkl * wkl))
    _refused(fic, h, qt, stream(wkl * wkl - 1, c_first=-1))


# ---------------------------------------------------------------- quadtree encode at the split threshold

def collage_errors(oracle, plane, W, H, B, wk, q):
    """E of every range block at block size B: the squared difference between the source and one decode step of its
    quantised code {c, a * 100, b}, read from the source's decimated plane (the oracle's scale_image)."""
    from conftest import to_argb_grey

    dec = _red(oracle.scale_image(to_argb_grey(plane))).astype(np.int64)
    rpw, rph = W // B, H // B
    dpw, dph = 2 * rpw - 3, 2 * rph - 3
    nr = rpw * rph
    dy, dx = np.empty(nr, np.int64), np.empty(nr, np.int64)
    for j in range(nr):
        x, y = (j % rpw) * B, (j // rpw) * B
        dy[j], dx[j] = oracle.generate_kernel(dpw, dph, oracle.domain_block_index(x, y, rpw, rph, dpw, B), wk)
    c = q[:, 0].astype(np.float32)
    yd = np.trunc(c / np.float32(wk)).astype(np.int64)
    xd = np.trunc(np.fmod(c, np.float32(wk))).astype(np.int64)
    idx = xd + dx + (yd + dy) * dpw
    assert ((idx >= 0) & (idx < dpw * dph)).all()
    a = q[:, 1].astype(np.float32) / np.float32(100)
    b = q[:, 2].astype(np.float32)
    r, col = (idx // dpw) * (B // 4), (idx % dpw) * (B // 4)
    ii = np.arange(B)
    dblk = dec[r[:, None, None] + ii[None, :, None], col[:, None, None] + ii[None, None, :]].astype(np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.clip(np.trunc(a[:, None, None] * dblk + b[:, None, None]), 0, 255).astype(np.int64)
    src = plane.astype(np.int64).reshape(rph, B, rpw, B).transpose(0, 2, 1, 3).reshape(-1, B, B)
    return ((v - src) ** 2).sum(axis=(1, 2))


def _qt_plane(fic, name):
    from conftest import GOLD
    import os

    if name == "lena":
        return np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    if name == "binary":
        return ((fic.synth.noise(128, 128, 13) >> 7) * 255).astype(np.uint8)
    t = fic.synth.noise(8, 8, 17)   # ties: a few repeated 8 x 8 tiles
    return np.tile(np.concatenate([t, t[::-1]], 0), (8, 16))


@pytest.mark.parametrize("name", ["lena", "ties", "binary"])
@pytest.mark.parametrize("b_min", [8, 4])
def test_qt_split_threshold(fic, h, oracle, qt, name, b_min):
    """max_mse = E_j / B^2 exactly (B^2 is a power of two) and one ulp either side: a block splits iff E > max_mse B^2,
    strictly, on the GPU and in the oracle."""
    plane = _qt_plane(fic, name)
    H, W = plane.shape
    wk = 4
    levels = [16 >> L for L in range({8: 2, 4: 3}[b_min])]
    E = [collage_errors(oracle, plane, W, H, B, wk, h.encode_u8(plane, B, wk)[1]) for B in levels]
    rng = np.random.default_rng(len(name) + b_min)
    for L in range(len(levels) - 1):
        B = levels[L]
        e = np.unique(E[L])
        picks = {int(e[0]), int(e[-1]), int(e[len(e) // 2]), int(rng.choice(e))}
        for ej in sorted(picks):
            exact = ej / float(B * B)
            assert exact * (B * B) == ej
            for mse in (exact, np.nextafter(exact, np.inf), np.nextafter(exact, -np.inf)):
                s = h.encode_quadtree(plane, 16, b_min, wk, float(mse))
                assert s == qt.encode_quadtree(plane, 16, b_min, wk, float(mse), nthreads=8), (ej, mse)
                ntop = (W // 16) * (H // 16)
                flags = np.frombuffer(s, np.uint8, count=ntop, offset=32)
                split0 = E[0].astype(np.float64) > mse * 256.0
                assert ((flags & 1) == split0).all()
                if len(levels) == 3:
                    split1 = (E[1].astype(np.float64) > mse * 64.0).reshape(H // 8, W // 8)
                    kids = np.stack([split1[0::2, 0::2], split1[0::2, 1::2], split1[1::2, 0::2], split1[1::2, 1::2]], -1)
                    want = (kids.reshape(-1, 4) & split0[:, None]).astype(np.uint8).dot(np.array([2, 4, 8, 16]))
                    assert ((flags & 0x1E) == want).all()
                else:
                    assert not (flags & 0x1E).any()
                if L == 0:   # the blocks at the threshold: kept at E_j / B^2 and above, split one ulp below
                    assert split0[E[0] == ej].all() == (mse < exact) and split0[E[0] == ej].any() == (mse < exact)


@pytest.mark.parametrize("W,H,b_max,b_min,wk", [(144, 144, 16, 4, 0), (112, 96, 16, 8, 5), (48, 80, 16, 4, 3), (72, 72, 8, 4, 0),
                                                (56, 48, 8, 4, 2), (24, 40, 8, 4, 3), (1456, 1456, 16, 4, 2),
                                                (2304, 2048, 16, 8, 2)])
def test_qt_encode_padded_shapes(fic, h, qt, W, H, b_max, b_min, wk):
    plane = fic.synth.structured(W, H, W + H)
    for mse in (-1.0, 10.0, 40.0):
        assert h.encode_quadtree(plane, b_max, b_min, wk, mse) == qt.encode_quadtree(plane, b_max, b_min, wk, mse, nthreads=8)
