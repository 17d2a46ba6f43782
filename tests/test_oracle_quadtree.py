"""The quadtree extension (FIC_MODE_GREY_QT) in the CPU oracle: its stream restated in numpy from the oracle's per-level
codes (collage error, split rule, assembly), its decoder restated in numpy, and the degenerate trees (no split: the
b_max codes; every split: the b_min codes) against the fixed-block stream and decoder."""
import os
import struct

import numpy as np
import pytest

from conftest import to_argb_grey

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [(16, 8), (16, 4), (8, 4)]
F32 = np.float32


def _synth():
    import importlib.util

    spec = importlib.util.spec_from_file_location("fic_synth", os.path.join(ROOT, "fractal-image-compression_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _images():
    s = _synth()
    lena = np.fromfile(os.path.join(ROOT, "tests", "golden", "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    lena64 = np.fromfile(os.path.join(ROOT, "tests", "golden", "lena64.u8"), np.uint8).reshape(64, 64)
    return {"lena256_wk2": (lena, 2), "lena64_full": (lena64, 0), "structured128_wk4": (s.structured(128, 128, 3), 4),
            "noise64_full": (s.noise(64, 64, 5), 0)}


IMAGES = _images()


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree

    quadtree.build()
    return quadtree


def _codes(oracle, plane, B, wk, cache={}):
    """writeData ints [NR][3] of the oracle's grey encode at B (wk 0: the whole pool)."""
    key = (plane.tobytes(), B, wk)
    if key not in cache:
        H, W = plane.shape
        wkl = wk or 2 * (W // B) - 3
        s = oracle.write_data(oracle.encode(to_argb_grey(plane), B, wkl, nthreads=8), W, H, B, wkl)
        cache[key] = np.frombuffer(s[20:], ">i4").reshape(-1, 3).astype(np.int64)
    return cache[key]


def _decimate(img):
    """FC:970-1007 on a grey plane (the fourth tap is 128 where x + 1 >= H)."""
    H, W = img.shape
    p = img.astype(np.int64)
    p11 = p[1::2, 1::2].copy()
    p11[:, np.arange(0, W, 2) + 1 >= H] = 128
    return ((p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p11) // 4).astype(np.int64)


def _domain(oracle, W, H, B, wk, j, c):
    """Codebook row and column (decimated pixels) of range j's code index c: calculateIndices, FC:853-893."""
    rpw, rph = W // B, H // B
    dpw, dph = 2 * rpw - 3, 2 * rph - 3
    di = oracle.domain_block_index((j % rpw) * B, (j // rpw) * B, rpw, rph, dpw, B)
    dy, dx = oracle.generate_kernel(dpw, dph, di, wk)
    cf = F32(c)
    yd, xd = int(np.trunc(cf / F32(wk))), int(np.trunc(np.fmod(cf, F32(wk))))
    idx = xd + dx + (yd + dy) * dpw
    assert 0 <= idx < dpw * dph
    return (idx // dpw) * (B // 4), (idx % dpw) * (B // 4)


def _px(a, b, d):
    return np.clip(np.trunc(F32(a) * d.astype(F32) + F32(b)), 0, 255).astype(np.int64)


def _collage_errors(oracle, plane, B, wk, q):
    H, W = plane.shape
    dec = _decimate(plane)
    wkl = wk or 2 * (W // B) - 3
    src = plane.astype(np.int64)
    E = np.zeros(len(q), np.int64)
    for j, (c, qa, qb) in enumerate(q):
        r, col = _domain(oracle, W, H, B, wkl, j, c)
        v = _px(F32(qa) / F32(100), F32(qb), dec[r:r + B, col:col + B])
        y, x = (j // (W // B)) * B, (j % (W // B)) * B
        E[j] = ((v - src[y:y + B, x:x + B]) ** 2).sum()
    return E


def _numpy_stream(oracle, plane, b_max, b_min, wk, max_mse):
    H, W = plane.shape
    Bs = [b_max >> L for L in range(4) if (b_max >> L) >= b_min]
    q = [_codes(oracle, plane, B, wk) for B in Bs]
    E = [_collage_errors(oracle, plane, B, wk, q[L]) for L, B in enumerate(Bs)]

    def split(L, j):
        return L < len(Bs) - 1 and float(E[L][j]) > max_mse * float(Bs[L] * Bs[L])

    def child(L, j, k):
        rpw, rpw1 = W // Bs[L], W // Bs[L + 1]
        return (2 * (j // rpw) + (k >> 1)) * rpw1 + 2 * (j % rpw) + (k & 1)

    flags, leaves = [], []

    def emit(L, j):
        if split(L, j):
            for k in range(4):
                emit(L + 1, child(L, j, k))
        else:
            leaves.append(q[L][j])

    for t in range((W // b_max) * (H // b_max)):
        f = 0
        if split(0, t):
            f = 1 | sum(2 << k for k in range(4) if split(1, child(0, t, k)))
        flags.append(f)
        emit(0, t)
    flags += [0] * (-len(flags) % 4)
    head = struct.pack(">8i", 3, W, H, 0, wk, b_max, b_min, len(leaves))
    return head + bytes(flags) + np.asarray(leaves, ">i4").tobytes()


def _numpy_decode(oracle, stream, max_iters=50):
    _, W, H, _, wk, b_max, b_min, n = struct.unpack(">8i", stream[:32])
    ntop = (W // b_max) * (H // b_max)
    flags = stream[32:32 + ntop]
    codes = np.frombuffer(stream, ">i4", count=3 * n, offset=32 + ntop + (-ntop % 4)).reshape(n, 3)
    leaves = []  # (B, y, x, row, col, a, b)

    def add(B, j):
        c, qa, qb = codes[len(leaves)]
        r, col = _domain(oracle, W, H, B, wk or 2 * (W // B) - 3, j, c)
        leaves.append((B, (j // (W // B)) * B, (j % (W // B)) * B, r, col, F32(qa) / F32(100), F32(qb)))

    for t, f in enumerate(flags):
        if not f & 1:
            add(b_max, t)
            continue
        for k in range(4):
            j1 = (2 * (t // (W // b_max)) + (k >> 1)) * (2 * W // b_max) + 2 * (t % (W // b_max)) + (k & 1)
            if not (f >> (1 + k)) & 1:
                add(b_max // 2, j1)
                continue
            r1 = W // (b_max // 2)
            for k2 in range(4):
                add(b_max // 4, (2 * (j1 // r1) + (k2 >> 1)) * (2 * r1) + 2 * (j1 % r1) + (k2 & 1))
    img = np.full((H, W), 128, np.int64)
    avg, it = F32(0), 0
    for it in range(1, max_iters + 1):
        dec = _decimate(img)
        new = img.copy()
        for B, y, x, r, col, a, b in leaves:
            new[y:y + B, x:x + B] = _px(a, b, dec[r:r + B, col:col + B])
        S = int(((new - img) ** 2).sum())
        img = new
        avg = F32(S) / F32(W * H)
        if avg < 1:
            break
    return img.astype(np.uint8), avg, it


@pytest.mark.parametrize("name", sorted(IMAGES))
@pytest.mark.parametrize("pair", PAIRS)
@pytest.mark.parametrize("max_mse", [0.0, 4.0, 25.0, 100.0])
def test_stream_matches_numpy_restatement(oracle, name, pair, max_mse, qt):
    plane, wk = IMAGES[name]
    got = qt.encode_quadtree(plane, pair[0], pair[1], wk, max_mse, nthreads=8)
    assert got == _numpy_stream(oracle, plane, pair[0], pair[1], wk, max_mse)


@pytest.mark.parametrize("pair", PAIRS)
def test_no_split_is_the_b_max_stream(oracle, pair, qt):
    plane, wk = IMAGES["lena256_wk2"]
    s = qt.encode_quadtree(plane, pair[0], pair[1], wk, np.inf)
    q = _codes(oracle, plane, pair[0], wk)
    ntop = len(q)
    assert struct.unpack(">8i", s[:32]) == (3, 256, 256, 0, wk, pair[0], pair[1], ntop)
    assert s[32:32 + ntop] == bytes(ntop)
    assert s[32 + ntop + (-ntop % 4):] == np.asarray(q, ">i4").tobytes()


@pytest.mark.parametrize("pair", PAIRS)
def test_every_split_is_the_b_min_codes_in_z_order(oracle, pair, qt):
    plane, wk = IMAGES["lena64_full"]
    b_max, b_min = pair
    s = qt.encode_quadtree(plane, b_max, b_min, wk, -1.0)
    q = _codes(oracle, plane, b_min, wk)
    r = b_max // b_min
    rpw = 64 // b_min
    order = []  # per top block, its b_min blocks in Z order (depth first, children in raster order)
    for ty in range(64 // b_max):
        for tx in range(64 // b_max):
            zs = sorted(range(r * r), key=lambda k: [((k // r) >> l & 1) * 2 + ((k % r) >> l & 1) for l in range(3, -1, -1)])
            order += [(ty * r + k // r) * rpw + tx * r + k % r for k in zs]
    assert s[32 + (-(64 // b_max) ** 2 % 4) + (64 // b_max) ** 2:] == np.asarray(q[order], ">i4").tobytes()


@pytest.mark.parametrize("size,name,pair,max_mse", [
    (64, "lena64_full", (16, 4), 25.0), (64, "noise64_full", (8, 4), 100.0), (64, "lena64_full", (16, 8), 4.0),
    (128, "structured128_wk4", (16, 4), 4.0), (128, "structured128_wk4", (8, 4), 100.0)])
def test_decoder_matches_numpy_restatement(oracle, size, name, pair, max_mse, qt):
    plane, wk = IMAGES[name]
    s = qt.encode_quadtree(plane, pair[0], pair[1], wk, max_mse, nthreads=8)
    img, avg, it = qt.decode_quadtree(s)
    nimg, navg, nit = _numpy_decode(oracle, s)
    assert img.shape == (size, size)
    assert (img == nimg).all() and it == nit and avg.tobytes() == navg.tobytes()


@pytest.mark.parametrize("name", ["lena256_wk2", "lena64_full", "noise64_full"])
def test_no_split_decodes_like_the_fixed_stream(oracle, name, qt):
    plane, wk = IMAGES[name]
    H, W = plane.shape
    s = qt.encode_quadtree(plane, 8, 4, wk, np.inf)
    wkl = wk or 2 * (W // 8) - 3
    fixed = struct.pack(">5i", 0, W, H, 8, wkl) + np.asarray(_codes(oracle, plane, 8, wk), ">i4").tobytes()
    img, avg, it = qt.decode_quadtree(s)
    fimg, favg, fit = oracle.decode(fixed)
    assert (img == (fimg & 0xFF)).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == favg.tobytes()


def test_malformed_streams_are_refused(oracle, qt):
    plane, wk = IMAGES["lena64_full"]
    s = qt.encode_quadtree(plane, 16, 4, wk, 25.0)
    ntop = 16
    with pytest.raises(ValueError):
        qt.decode_quadtree(s[:-1])
    bad = bytearray(s)
    bad[32] = 0x02  # a child split without its parent
    with pytest.raises(ValueError):
        qt.decode_quadtree(bytes(bad))
    bad = bytearray(s)
    bad[28:32] = struct.pack(">i", struct.unpack(">i", s[28:32])[0] + 1)
    with pytest.raises(ValueError):
        qt.decode_quadtree(bytes(bad))
    bad = bytearray(s)
    bad[32 + ntop:32 + ntop + 4] = struct.pack(">i", 1 << 20)
    with pytest.raises(ValueError):
        qt.decode_quadtree(bytes(bad))
    with pytest.raises(ValueError):
        qt.encode_quadtree(plane, 16, 4, wk, float("nan"))
