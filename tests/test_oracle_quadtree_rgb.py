"""The RGB quadtree extension (FIC_MODE_RGB_QT) in the CPU oracle: its stream restated in numpy from the oracle's per-level
RGB codes (RGB decimation with its x + 1 >= H slip, collage error over three channels, split rule, assembly), its decoder
restated in numpy, the degenerate trees, and the reference's own stream: an RGB tree that never splits at b_max = 8,
wk = 2 on LenaColored carries exactly the codes of unknown.run."""
import os
import struct

import numpy as np
import pytest

from conftest import GOLD, to_argb_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAIRS = [(16, 8), (16, 4), (8, 4)]
F32 = np.float32


def _synth():
    import importlib.util

    spec = importlib.util.spec_from_file_location("fic_synth", os.path.join(ROOT, "fractal-image-compression_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _structured_rgb(W, H, seed):
    s = _synth()
    return np.stack([s.structured(W, H, seed + k) for k in range(3)])


def _images():
    lena = np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1).copy()
    return {"lena256_wk2": (lena, 2), "lena64_full": (lena[:, ::4, ::4].copy(), 0),
            "structured128_wk4": (_structured_rgb(128, 128, 3), 4), "landscape128x64_wk3": (_structured_rgb(128, 64, 11), 3)}


IMAGES = _images()


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree_rgb

    quadtree_rgb.build()
    return quadtree_rgb


def _argb(planes):
    return to_argb_rgb(planes.transpose(1, 2, 0))


def _codes(oracle, planes, B, wk, cache={}):
    """writeData ints [NR][5] of the oracle's RGB encode at B (wk 0: the whole pool)."""
    key = (planes.tobytes(), planes.shape, B, wk)
    if key not in cache:
        _, H, W = planes.shape
        wkl = wk or 2 * (W // B) - 3
        s = oracle.write_data(oracle.encode(_argb(planes), B, wkl, rgb=True, nthreads=8), W, H, B, wkl, rgb=True)
        cache[key] = np.frombuffer(s[20:], ">i4").reshape(-1, 5).astype(np.int64)
    return cache[key]


def _decimate_rgb(img):
    """FC:901-962 on [3, H, W] planes: (p00 + p10 + 2 * p01) / 4 per channel, the fourth tap 128 where x + 1 >= H."""
    _, H, W = img.shape
    p = img.astype(np.int64)
    fourth = p[:, 1::2, 0::2].copy()
    fourth[:, :, np.arange(0, W, 2) + 1 >= H] = 128
    return (p[:, 0::2, 0::2] + p[:, 0::2, 1::2] + p[:, 1::2, 0::2] + fourth) // 4


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


def _dequant(code):
    """FC:446-450: a = qa / 1e6f, bR = qbR / 1e5f, bG = qbG / 1e5f, bB = qbB (unscaled)."""
    _, qa, qr, qg, qb = code
    return F32(qa) / F32(1000000), [F32(qr) / F32(100000), F32(qg) / F32(100000), F32(qb)]


def _px(a, b, d):
    """[3, B, B] decoded pixels of domain planes d: per channel clamp((int)(a * d + b_c))."""
    return np.stack([np.clip(np.trunc(a * d[c].astype(F32) + b[c]), 0, 255) for c in range(3)]).astype(np.int64)


def _collage_errors(oracle, planes, B, wk, q, cache={}):
    key = (planes.tobytes(), planes.shape, B, wk)
    if key not in cache:
        _, H, W = planes.shape
        dec = _decimate_rgb(planes)
        wkl = wk or 2 * (W // B) - 3
        src = planes.astype(np.int64)
        E = np.zeros(len(q), np.int64)
        for j, code in enumerate(q):
            r, col = _domain(oracle, W, H, B, wkl, j, code[0])
            a, b = _dequant(code)
            y, x = (j // (W // B)) * B, (j % (W // B)) * B
            E[j] = ((_px(a, b, dec[:, r:r + B, col:col + B]) - src[:, y:y + B, x:x + B]) ** 2).sum()
        cache[key] = E
    return cache[key]


def _numpy_stream(oracle, planes, b_max, b_min, wk, max_mse):
    _, H, W = planes.shape
    Bs = [b_max >> L for L in range(4) if (b_max >> L) >= b_min]
    q = [_codes(oracle, planes, B, wk) for B in Bs]
    E = [_collage_errors(oracle, planes, B, wk, q[L]) for L, B in enumerate(Bs)]

    def split(L, j):
        return L < len(Bs) - 1 and float(E[L][j]) > max_mse * float(3 * Bs[L] * Bs[L])

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
    head = struct.pack(">8i", 4, W, H, 0, wk, b_max, b_min, len(leaves))
    return head + bytes(flags) + np.asarray(leaves, ">i4").tobytes()


def _numpy_decode(oracle, stream, max_iters=50):
    _, W, H, _, wk, b_max, b_min, n = struct.unpack(">8i", stream[:32])
    ntop = (W // b_max) * (H // b_max)
    flags = stream[32:32 + ntop]
    codes = np.frombuffer(stream, ">i4", count=5 * n, offset=32 + ntop + (-ntop % 4)).reshape(n, 5).astype(np.int64)
    leaves = []  # (B, y, x, row, col, a, b)

    def add(B, j):
        code = codes[len(leaves)]
        r, col = _domain(oracle, W, H, B, wk or 2 * (W // B) - 3, j, code[0])
        leaves.append((B, (j // (W // B)) * B, (j % (W // B)) * B, r, col) + _dequant(code))

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
    img = np.full((3, H, W), 128, np.int64)
    avg, it = F32(0), 0
    for it in range(1, max_iters + 1):
        dec = _decimate_rgb(img)
        new = img.copy()
        for B, y, x, r, col, a, b in leaves:
            new[:, y:y + B, x:x + B] = _px(a, b, dec[:, r:r + B, col:col + B])
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
    planes, wk = IMAGES[name]
    got = qt.encode_quadtree_rgb(planes, pair[0], pair[1], wk, max_mse, nthreads=8)
    assert got == _numpy_stream(oracle, planes, pair[0], pair[1], wk, max_mse)


@pytest.mark.parametrize("name,pair,max_mse", [
    ("lena64_full", (16, 4), 25.0), ("lena64_full", (16, 8), 4.0), ("structured128_wk4", (16, 4), 4.0),
    ("structured128_wk4", (8, 4), 100.0), ("landscape128x64_wk3", (16, 4), 25.0)])
def test_decoder_matches_numpy_restatement(oracle, name, pair, max_mse, qt):
    planes, wk = IMAGES[name]
    s = qt.encode_quadtree_rgb(planes, pair[0], pair[1], wk, max_mse, nthreads=8)
    img, avg, it = qt.decode_quadtree_rgb(s)
    nimg, navg, nit = _numpy_decode(oracle, s)
    assert img.shape == planes.shape
    assert (img == nimg).all() and it == nit and avg.tobytes() == navg.tobytes()


def test_unknown_run_pin(oracle, qt):
    """LenaColored at (8, 4), wk 2, never split: the leaves are the reference's own stream unknown.run."""
    planes, _ = IMAGES["lena256_wk2"]
    ref = open(os.path.join(GOLD, "unknown_run.bin"), "rb").read()
    assert struct.unpack(">5i", ref[:20]) == (1, 256, 256, 8, 2)
    s = qt.encode_quadtree_rgb(planes, 8, 4, 2, np.inf, nthreads=8)
    assert struct.unpack(">8i", s[:32]) == (4, 256, 256, 0, 2, 8, 4, 1024)
    assert s[32:32 + 1024] == bytes(1024)
    assert s[32 + 1024:] == ref[20:]
    img, avg, it = qt.decode_quadtree_rgb(s)
    fimg, favg, fit = oracle.decode(ref)
    assert (img == qt.argb_to_planes(fimg)).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == np.float32(favg).tobytes()


@pytest.mark.parametrize("name", ["lena64_full", "structured128_wk4", "landscape128x64_wk3"])
def test_no_split_decodes_like_the_fixed_stream(oracle, name, qt):
    planes, wk = IMAGES[name]
    _, H, W = planes.shape
    s = qt.encode_quadtree_rgb(planes, 16, 8, wk, np.inf)
    wkl = wk or 2 * (W // 16) - 3
    q = _codes(oracle, planes, 16, wk)
    assert s[32 + len(q) + (-len(q) % 4):] == np.asarray(q, ">i4").tobytes()
    fixed = struct.pack(">5i", 1, W, H, 16, wkl) + np.asarray(q, ">i4").tobytes()
    img, avg, it = qt.decode_quadtree_rgb(s)
    fimg, favg, fit = oracle.decode(fixed)
    assert (img == qt.argb_to_planes(fimg)).all() and it == fit
    if favg < 1:
        assert avg.tobytes() == np.float32(favg).tobytes()


@pytest.mark.parametrize("pair", PAIRS)
def test_every_split_is_the_b_min_codes_in_z_order(oracle, pair, qt):
    planes, wk = IMAGES["lena64_full"]
    b_max, b_min = pair
    s = qt.encode_quadtree_rgb(planes, b_max, b_min, wk, -1.0)
    q = _codes(oracle, planes, b_min, wk)
    r = b_max // b_min
    rpw = 64 // b_min
    order = []  # per top block, its b_min blocks in Z order (depth first, children in raster order)
    for ty in range(64 // b_max):
        for tx in range(64 // b_max):
            zs = sorted(range(r * r), key=lambda k: [((k // r) >> l & 1) * 2 + ((k % r) >> l & 1) for l in range(3, -1, -1)])
            order += [(ty * r + k // r) * rpw + tx * r + k % r for k in zs]
    ntop = (64 // b_max) ** 2
    assert s[32 + ntop + (-ntop % 4):] == np.asarray(q[order], ">i4").tobytes()


def test_malformed_streams_are_refused(qt):
    from oracle import quadtree as grey_qt

    planes, wk = IMAGES["lena64_full"]
    s = qt.encode_quadtree_rgb(planes, 16, 4, wk, 25.0)
    ntop = 16
    qt.decode_quadtree_rgb(s)
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(s[:-1])
    bad = bytearray(s)
    bad[32] = 0x02  # a child split without its parent
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(bytes(bad))
    bad = bytearray(s)
    bad[28:32] = struct.pack(">i", struct.unpack(">i", s[28:32])[0] + 1)
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(bytes(bad))
    bad = bytearray(s)
    bad[32 + ntop:32 + ntop + 4] = struct.pack(">i", 1 << 20)
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(bytes(bad))
    with pytest.raises(ValueError):
        qt.encode_quadtree_rgb(planes, 16, 4, wk, float("nan"))
    # each decoder refuses the other mode's streams
    grey = grey_qt.encode_quadtree(planes[0], 16, 4, wk, 25.0)
    grey_qt.decode_quadtree(grey)
    with pytest.raises(ValueError):
        qt.decode_quadtree_rgb(grey)
    with pytest.raises(ValueError):
        grey_qt.decode_quadtree(s)
