"""Batch entries (fic_encode_batch[_u8], fic_decode_batch[_u8]) against a loop of single calls on the same handle:
every image's float bits, codes, decoded pixels, avgError bits and iteration count must be what the single entry
gives for that image alone (with that image's carry-in for the decoder)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLD, to_argb_grey, to_argb_rgb

pytestmark = pytest.mark.gpu

GREY, RGB, ISO = 0, 1, 2


@pytest.fixture(scope="module")
def fic():
    import fractal_image_compression_b200 as f

    return f


@pytest.fixture(scope="module")
def bh(fic):
    h = fic.Handle(0)
    yield h
    h.close()


@pytest.fixture
def h(fic, bh):
    bh.set_engine(fic.FIC_ENGINE_AUTO)
    yield bh
    bh.set_engine(fic.FIC_ENGINE_AUTO)


def bits_equal(a, b):
    """Float bits equal, except that any NaN equals any NaN (the 0/0 of a flat winner, FC:634, is only cast to int)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a.view(np.uint32)[~na] == b.view(np.uint32)[~nb]).all()


def grey_images(W, H, n, seed=1):
    """Structured and noise content with distinct seeds, ARGB ints [n, H, W]."""
    from fractal_image_compression_b200 import synth

    out = [synth.structured(W, H, seed + i) if i % 2 == 0 else synth.noise(W, H, seed + i) for i in range(n)]
    return np.stack([to_argb_grey(p) for p in out])


def rgb_images(W, H, n, seed=1):
    from fractal_image_compression_b200 import synth

    out = []
    for i in range(n):
        s = seed + 7 * i
        make = synth.structured if i % 2 == 0 else synth.noise
        out.append(to_argb_rgb(np.stack([make(W, H, s), make(W, H, s + 1), synth.structured(W, H, s + 2)], -1)))
    return np.stack(out)


def planes_of(argb, rgb):
    u = argb.view(np.uint32)
    if rgb:
        return np.ascontiguousarray(np.stack([(u >> 16) & 0xFF, (u >> 8) & 0xFF, u & 0xFF], 1).astype(np.uint8))
    return ((u >> 16) & 0xFF).astype(np.uint8)


def check_encode(h, imgs, B, wk, mode, u8=True):
    info, q = h.encode_batch(imgs, B, wk, mode)
    n, H, W = imgs.shape
    t = h.timings()
    S = (3, 5, 4)[mode]
    assert t.search_evals == n * (W // B) * (H // B) * wk * wk * (8 if mode == ISO else 1)
    for i in range(n):
        si, sq = h.encode(imgs[i], B, wk, mode)
        assert bits_equal(info[i], si), f"image {i}: info"
        assert (q[i] == sq).all(), f"image {i}: qcodes"
    assert info.shape == (n, (W // B) * (H // B), S)
    if u8:
        ui, uq = h.encode_batch_u8(planes_of(imgs, mode == RGB), B, wk, mode)
        assert bits_equal(ui, info) and (uq == q).all()
    return info, q


# ---------------------------------------------------------------- encode

@pytest.mark.parametrize("mode", [GREY, RGB])
@pytest.mark.parametrize("B", [4, 8, 16])
@pytest.mark.parametrize("wk", [1, 2, 16])
def test_encode_batch_grid(h, mode, B, wk):
    W, H = 256, 192  # 16 x 16 windows fit at every block size (B = 16: 29 x 21 domain blocks)
    imgs = (rgb_images if mode == RGB else grey_images)(W, H, 3, seed=B * 31 + wk)
    check_encode(h, imgs, B, wk, mode)


@pytest.mark.parametrize("mode", [GREY, RGB])
def test_encode_batch_landscape(h, mode):
    # 96 x 64: the reference's `x + 1 >= height` tap (FC:993, FC:940) slips into the image on landscape images
    imgs = (rgb_images if mode == RGB else grey_images)(96, 64, 3, seed=5)
    check_encode(h, imgs, 8, 2, mode)


def test_encode_batch_lena(fic, h, lena_grey, lena_colored):
    check_encode(h, np.stack([lena_grey] * 3), 8, 2, GREY)
    ref = open(os.path.join(GOLD, "unknown_run.bin"), "rb").read()  # the reference's own output for LenaColored
    _, q = check_encode(h, np.stack([lena_colored] * 3), 8, 2, RGB)
    for i in range(3):
        assert fic.stream_write(q[i], 256, 256, 8, 2, rgb=True) == ref


def test_encode_batch_mixed_content(h):
    W = H = 128
    flat = to_argb_grey(np.full((H, W), 77, np.uint8))
    binary = to_argb_grey(((np.arange(W * H).reshape(H, W) * 2654435761 >> 7) & 1).astype(np.uint8) * 255)
    noise = grey_images(W, H, 2, seed=9)[1]
    zero = to_argb_grey(np.zeros((H, W), np.uint8))
    imgs = np.stack([flat, binary, noise, zero, binary])
    for B, wk in [(8, 2), (4, 4), (16, 3)]:
        check_encode(h, imgs, B, wk, GREY)
    check_encode(h, np.stack([to_argb_rgb(np.stack([planes_of(x, False)] * 3, -1)) for x in imgs]), 8, 2, RGB)


@pytest.mark.parametrize("n", [1, 2, 3, 257])
def test_encode_batch_sizes(h, n):
    check_encode(h, grey_images(64, 64, n, seed=n), 8, 2, GREY, u8=(n != 257))


def test_encode_batch_fallback_engines(fic, h):
    # wk > 16, the whole pool: per-image engine inside the batch call
    imgs = grey_images(128, 128, 3, seed=3)
    check_encode(h, imgs, 8, 29, GREY)
    # the isometry extension
    check_encode(h, grey_images(64, 64, 3, seed=4), 8, 2, ISO)
    # forced engines
    h.set_engine(fic.FIC_ENGINE_DIRECT)
    check_encode(h, imgs, 8, 2, GREY)
    check_encode(h, rgb_images(64, 64, 2, seed=6), 4, 3, RGB)
    h.set_engine(fic.FIC_ENGINE_UMMA)
    check_encode(h, imgs, 8, 29, GREY)


def test_encode_batch_timings(fic, h):
    imgs = grey_images(256, 256, 8)
    h.encode_batch(imgs, 8, 2, GREY)
    t = h.timings()
    assert t.engine == fic.FIC_ENGINE_FUSED and t.launches == 1 and t.total_ms > 0


def test_encode_batch_against_oracle(h, oracle):
    imgs = grey_images(64, 64, 3, seed=11)
    info, _ = h.encode_batch(imgs, 8, 2, GREY)
    for i in range(3):
        assert bits_equal(info[i], oracle.encode(imgs[i], 8, 2))
    imgs = rgb_images(64, 64, 2, seed=12)
    info, _ = h.encode_batch(imgs, 4, 3, RGB)
    for i in range(2):
        assert bits_equal(info[i], oracle.encode(imgs[i], 4, 3, rgb=True))


# ---------------------------------------------------------------- decode

def check_decode(h, q, W, H, B, wk, mode, carries=None, max_iters=50):
    n = q.shape[0]
    img, avg, it = h.decode_batch(q, W, H, B, wk, mode, avg_error=carries, max_iters=max_iters)
    assert avg.dtype == np.float32 and it.dtype == np.int32 and img.shape == (n, H, W)
    for i in range(n):
        c = 0.0 if carries is None else float(np.float32(carries[i]))
        si, sa, sit = h.decode(q[i], W, H, B, wk, mode, avg_error=c, max_iters=max_iters)
        assert (img[i] == si).all(), f"image {i}: pixels"
        assert np.float32(avg[i]).view(np.uint32) == np.float32(sa).view(np.uint32), f"image {i}: avgError"
        assert it[i] == sit, f"image {i}: iterations"
    pl, pavg, pit = h.decode_batch_u8(q, W, H, B, wk, mode, avg_error=carries, max_iters=max_iters)
    assert (pl == planes_of(img, mode == RGB)).all()
    assert (pavg.view(np.uint32) == avg.view(np.uint32)).all() and (pit == it).all()
    return img, avg, it


def codes_of(h, imgs, B, wk, mode):
    return h.encode_batch(imgs, B, wk, mode)[1]


def test_decode_batch_convergence_differs(h, lena_grey):
    W = H = 256
    flat = to_argb_grey(np.full((H, W), 200, np.uint8))
    imgs = np.concatenate([np.stack([lena_grey, flat]), grey_images(W, H, 4, seed=21)])
    q = codes_of(h, imgs, 8, 2, GREY)
    _, _, it = check_decode(h, q, W, H, 8, 2, GREY)
    assert len(set(it.tolist())) > 1  # some images stop earlier and stay frozen while the others sweep on


@pytest.mark.parametrize("max_iters", [1, 3, 9, 50])
def test_decode_batch_max_iters(h, max_iters):
    imgs = grey_images(128, 128, 5, seed=max_iters)
    q = codes_of(h, imgs, 8, 2, GREY)
    check_decode(h, q, 128, 128, 8, 2, GREY, max_iters=max_iters)
    qr = codes_of(h, rgb_images(128, 64, 3, seed=max_iters), 8, 2, RGB)
    check_decode(h, qr, 128, 64, 8, 2, RGB, max_iters=max_iters)


def test_decode_batch_carries(h, lena_grey):
    q = codes_of(h, np.stack([lena_grey] * 3 + list(grey_images(256, 256, 3, seed=31))), 8, 2, GREY)
    carries = np.array([0.0, 0.7711792, 3.5e7, 3.5e7, 0.0, 0.7711792], np.float32)  # non-zero carries bail and re-run
    check_decode(h, q, 256, 256, 8, 2, GREY, carries=carries)
    check_decode(h, q, 256, 256, 8, 2, GREY, carries=carries, max_iters=2)


@pytest.mark.parametrize("W,H,B,mode", [(64, 64, 4, GREY), (72, 64, 8, GREY), (72, 48, 8, RGB), (64, 64, 4, RGB)])
def test_decode_batch_per_image_geometries(h, W, H, B, mode):
    # B = 4 and W % 16 != 0 have no one-launch decoder: the whole batch runs image by image
    imgs = (rgb_images if mode == RGB else grey_images)(W, H, 3, seed=W + B)
    check_decode(h, codes_of(h, imgs, B, 2, mode), W, H, B, 2, mode, carries=np.array([0, 0.5, 0], np.float32))


def test_decode_batch_isometry(h):
    q = codes_of(h, grey_images(64, 64, 3, seed=41), 8, 2, ISO)
    check_decode(h, q, 64, 64, 8, 2, ISO)


def test_decode_batch_lena64(fic, h, lena64):
    for fname, B in [("lena64_b8_full.run", 8), ("lena64_b4_full.run", 4)]:
        s = open(os.path.join(GOLD, fname), "rb").read()
        rgb, W, H, B, wk, q = fic.stream_read(s)
        check_decode(h, np.stack([q] * 3), W, H, B, wk, rgb)


def test_decode_batch_lena_oracle(fic, h, oracle):
    s = open(os.path.join(GOLD, "lena_grey_b8_wk2.run"), "rb").read()
    rgb, W, H, B, wk, q = fic.stream_read(s)
    carries = np.array([0.0, 0.5863342, 0.0], np.float32)
    img, avg, it = check_decode(h, np.stack([q] * 3), W, H, B, wk, rgb, carries=carries)
    for i in range(3):
        oimg, oavg, oit = oracle.decode(s, avg_error_in=float(carries[i]))
        assert (img[i] == oimg).all() and avg[i].view(np.uint32) == np.float32(oavg).view(np.uint32) and it[i] == oit


def test_decode_batch_unknown_run(fic, h, oracle):
    s = open(os.path.join(GOLD, "unknown_run.bin"), "rb").read()
    rgb, W, H, B, wk, q = fic.stream_read(s)
    img, avg, it = check_decode(h, np.stack([q] * 2), W, H, B, wk, rgb)
    oimg, oavg, oit = oracle.decode(s)
    assert (img[1] == oimg).all() and it[1] == oit


@pytest.mark.parametrize("mode", [GREY, RGB])
def test_decode_batch_random_codes(h, mode):
    rng = np.random.default_rng(7 + mode)
    W, H, B, wk = 128, 128, 8, 3
    nr, n = (W // B) * (H // B), 6
    S = 5 if mode == RGB else 3
    q = np.zeros((n, nr, S), np.int32)
    q[..., 0] = rng.integers(0, wk * wk, (n, nr))
    q[..., 1] = rng.integers(-120, 121, (n, nr))  # a in [-1.2, 1.2] (grey a * 100; RGB a * 100 too)
    q[..., 2:] = rng.integers(-200, 400, (n, nr, S - 2))
    if mode == RGB:
        q[..., 4] = rng.integers(-20, 20, (n, nr))
    check_decode(h, q, W, H, B, wk, mode)


def test_decode_batch_out_of_pool_names_image(fic, h):
    q = codes_of(h, grey_images(64, 64, 4, seed=51), 8, 2, GREY)
    q[2, 5, 0] = 1 << 20
    with pytest.raises(fic.FicError) as e:
        h.decode_batch(q, 64, 64, 8, 2, GREY)
    assert e.value.code == fic._lib.FIC_E_STREAM and "image 2" in str(e.value)
    q72 = codes_of(h, grey_images(72, 64, 3, seed=52), 8, 2, GREY)  # image-by-image geometry
    q72[1, 0, 0] = 1 << 20
    with pytest.raises(fic.FicError) as e:
        h.decode_batch(q72, 72, 64, 8, 2, GREY)
    assert e.value.code == fic._lib.FIC_E_STREAM and "image 1" in str(e.value)


def test_decode_batch_timings(h):
    imgs = np.stack([grey_images(256, 256, 1, seed=s)[0] for s in range(8)])  # structured content: converges
    q = codes_of(h, imgs, 8, 2, GREY)
    h.decode_batch(q, 256, 256, 8, 2, GREY)
    t = h.timings()
    assert t.launches == 1 and t.total_ms > 0


# ---------------------------------------------------------------- argument checks

def test_batch_rejections(fic, h):
    L, hh = h._L, h._h
    img = np.zeros((2, 64, 64), np.int32)
    info = np.zeros((2, 64, 3), np.float32)
    q = np.zeros((2, 64, 3), np.int32)
    out = np.zeros((2, 64, 64), np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    E = fic._lib.FIC_E_ARG
    assert L.fic_encode_batch(hh, GREY, p(img), 0, 64, 64, 8, 2, p(info), p(q)) == E
    assert L.fic_encode_batch(hh, GREY, None, 2, 64, 64, 8, 2, p(info), p(q)) == E
    assert L.fic_encode_batch(hh, GREY, p(img), 2, 64, 64, 8, 2, None, None) == E
    assert L.fic_encode_batch_u8(hh, GREY, None, 2, 64, 64, 8, 2, p(info), p(q)) == E
    assert L.fic_encode_batch(hh, 3, p(img), 2, 64, 64, 8, 2, p(info), p(q)) == E  # unknown mode
    assert L.fic_decode_batch(hh, GREY, 0, 64, 64, 8, 2, p(q), 50, p(out), None, None) == E
    assert L.fic_decode_batch(hh, GREY, 2, 64, 64, 8, 2, None, 50, p(out), None, None) == E
    assert L.fic_decode_batch(hh, GREY, 2, 64, 64, 8, 2, p(q), 50, None, None, None) == E
    assert L.fic_decode_batch(hh, GREY, 2, 64, 64, 8, 2, p(q), 0, p(out), None, None) == E
    assert L.fic_decode_batch_u8(hh, GREY, 2, 64, 64, 8, 2, p(q), 50, None, None, None) == E
    # the reference's own rejections (make_geom)
    for W, H, B, wk in [(64, 64, 2, 2), (64, 64, 5, 2), (60, 64, 8, 2), (64, 64, 8, 14), (64, 64, 8, 0), (8, 64, 8, 1)]:
        assert L.fic_encode_batch(hh, GREY, p(img), 2, W, H, B, wk, p(info), p(q)) == E
        assert L.fic_decode_batch(hh, GREY, 2, W, H, B, wk, p(q), 50, p(out), None, None) == E
    # the handle still works
    check_encode(h, grey_images(64, 64, 2), 8, 2, GREY, u8=False)
