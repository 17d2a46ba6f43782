"""Batches of full-pool images on the tcgen05 engine: a group of images is one block-diagonal tensor-core search (one
pool sort, one pack of either operand, one k_umma_search launch, one refine, one solve).  Every image's float bits and
codes must be what a single encode of that image gives, for every MMA kind, CTA-pair setting and mode the tensor path
has."""
import numpy as np
import pytest

from conftest import to_argb_grey, to_argb_rgb

pytestmark = pytest.mark.gpu

GREY, RGB, ISO = 0, 1, 2


@pytest.fixture(scope="module")
def fic():
    import fractal_image_compression_b200 as f

    return f


@pytest.fixture(scope="module")
def uh(fic):
    h = fic.Handle(0)
    yield h
    h.close()


@pytest.fixture
def h(fic, uh):
    yield uh
    uh.set_engine(fic.FIC_ENGINE_AUTO)
    uh.set_umma_kind(fic.FIC_UMMA_KIND_AUTO)
    uh.set_umma_pair(fic.FIC_UMMA_PAIR_AUTO)


def full_pool(W, B):
    return 2 * (W // B) - 3


def bits_equal(a, b):
    """Float bits equal, except that any NaN equals any NaN (the 0/0 of a flat winner, FC:634)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a.view(np.uint32)[~na] == b.view(np.uint32)[~nb]).all()


def grey_images(W, n, seed):
    from fractal_image_compression_b200 import synth

    return np.stack([to_argb_grey(synth.structured(W, W, seed + i) if i % 2 == 0 else synth.noise(W, W, seed + i))
                     for i in range(n)])


def rgb_images(W, n, seed):
    from fractal_image_compression_b200 import synth

    out = []
    for i in range(n):
        s = seed + 7 * i
        make = synth.structured if i % 2 == 0 else synth.noise
        out.append(to_argb_rgb(np.stack([make(W, W, s), make(W, W, s + 1), synth.structured(W, W, s + 2)], -1)))
    return np.stack(out)


def planes_of(argb, rgb):
    u = argb.view(np.uint32)
    if rgb:
        return np.ascontiguousarray(np.stack([(u >> 16) & 0xFF, (u >> 8) & 0xFF, u & 0xFF], 1).astype(np.uint8))
    return ((u >> 16) & 0xFF).astype(np.uint8)


def check(fic, h, imgs, B, mode, u8=True):
    """The batch on the tcgen05 engine, image by image against single encodes on the same handle."""
    n, H, W = imgs.shape
    wk = full_pool(W, B)
    info, q = h.encode_batch(imgs, B, wk, mode)
    t = h.timings()
    assert t.engine == fic.FIC_ENGINE_UMMA
    assert t.search_evals == n * (W // B) * (H // B) * wk * wk * (8 if mode == ISO else 1)
    for i in range(n):
        si, sq = h.encode(imgs[i], B, wk, mode)
        assert bits_equal(info[i], si), f"image {i}: info"
        assert (q[i] == sq).all(), f"image {i}: qcodes"
    if u8:
        ui, uq = h.encode_batch_u8(planes_of(imgs, mode == RGB), B, wk, mode)
        assert bits_equal(ui, info) and (uq == q).all()
    return info, q


GREY_CASES = [  # B, W, kind, pair: every kind / pair combination the grey tcgen05 kernels have
    (4, 64, "I8", "OFF"), (4, 64, "F16", "OFF"), (4, 64, "F16", "ON"),
    (8, 128, "I8", "OFF"), (8, 128, "F16", "OFF"), (8, 128, "F16", "ON"),
    (16, 256, "I8", "OFF"), (16, 256, "I8", "ON"),
]


@pytest.mark.parametrize("B,W,kind,pair", GREY_CASES)
def test_grey_kinds_and_pairs(fic, h, B, W, kind, pair):
    h.set_engine(fic.FIC_ENGINE_UMMA)
    h.set_umma_kind(getattr(fic, "FIC_UMMA_KIND_" + kind))
    h.set_umma_pair(getattr(fic, "FIC_UMMA_PAIR_" + pair))
    check(fic, h, grey_images(W, 4, seed=B * 13), B, GREY)
    assert h.umma_pair_used() == (pair == "ON")


@pytest.mark.parametrize("B,W", [(4, 64), (8, 128), (16, 256)])
@pytest.mark.parametrize("pair", ["OFF", "ON"])
def test_rgb(fic, h, B, W, pair):
    h.set_engine(fic.FIC_ENGINE_UMMA)
    h.set_umma_pair(getattr(fic, "FIC_UMMA_PAIR_" + pair))
    check(fic, h, rgb_images(W, 3, seed=B * 17), B, RGB)


def test_isometries(fic, h):
    h.set_engine(fic.FIC_ENGINE_UMMA)
    check(fic, h, grey_images(64, 5, seed=71), 8, ISO)


def test_auto_picks_tensor_groups(fic, h, oracle):
    # 256^2 at blockgroesse 8, full pool: a single image runs the CUDA-core search, a batch of 8 the tensor group
    imgs = grey_images(256, 8, seed=81)
    info, _ = check(fic, h, imgs, 8, GREY, u8=False)
    assert bits_equal(info[3], oracle.encode(imgs[3], 8, 61))
    rgb = rgb_images(256, 8, seed=82)
    info, _ = check(fic, h, rgb, 8, RGB, u8=False)
    assert bits_equal(info[5], oracle.encode(rgb[5], 8, 61, rgb=True))
    # below 4 images the tensor chain's fixed cost does not pay: the single call's CUDA-core search
    h.encode_batch(imgs[:3], 8, 61, GREY)
    assert h.timings().engine == fic.FIC_ENGINE_DIRECT
    # a full pool of 13 x 13 domains: the fused kernel, also for a whole group
    h.encode_batch(grey_images(64, 8, seed=83), 8, 13, GREY)
    assert h.timings().engine == fic.FIC_ENGINE_FUSED


def test_mixed_content(fic, h):
    W = 128
    flat = to_argb_grey(np.full((W, W), 77, np.uint8))  # vR = 0 rows, varD = 0 domains
    binary = to_argb_grey(((np.arange(W * W).reshape(W, W) * 2654435761 >> 7) & 1).astype(np.uint8) * 255)
    cells = to_argb_grey((((np.arange(W)[:, None] // 4 + np.arange(W)[None, :] // 4) * 2654435761 >> 9) & 1).astype(np.uint8) * 255)
    noise = grey_images(W, 2, seed=91)[1]
    yy, xx = np.mgrid[0:W, 0:W]
    periodic = to_argb_grey(((xx % 8) * 32 + (yy % 8) * 3).astype(np.uint8))  # every domain ties: flag lists overflow
    imgs = np.stack([flat, binary, noise, periodic, cells])
    h.set_engine(fic.FIC_ENGINE_UMMA)
    for B in (8, 16):
        check(fic, h, imgs, B, GREY)
    rgb = np.stack([to_argb_rgb(np.stack([planes_of(x, False), planes_of(y, False), planes_of(z, False)], -1))
                    for x, y, z in [(flat, binary, noise), (binary, cells, binary), (periodic, noise, cells), (cells, cells, flat)]])
    for B in (8, 16):
        check(fic, h, rgb, B, RGB)


@pytest.mark.parametrize("n", [1, 2, 257])
def test_group_sizes(fic, h, n):
    # 257 images: two groups (at most 256 images share one pool sort)
    h.set_engine(fic.FIC_ENGINE_UMMA)
    check(fic, h, grey_images(64, n, seed=n), 8, GREY, u8=(n != 257))


def test_chunked_units_across_images(fic, h):
    # 1024^2, B = 8: 32 super-blocks per image, so a batch of 2 splits the domain sweep into several units per row and
    # carries each row's bound between them
    h.set_engine(fic.FIC_ENGINE_UMMA)
    check(fic, h, grey_images(1024, 2, seed=101), 8, GREY, u8=False)


def test_tensor_equals_direct(fic, h):
    imgs = grey_images(128, 3, seed=111)
    h.set_engine(fic.FIC_ENGINE_UMMA)
    ti, tq = h.encode_batch(imgs, 8, 29, GREY)
    h.set_engine(fic.FIC_ENGINE_DIRECT)
    di, dq = h.encode_batch(imgs, 8, 29, GREY)
    assert h.timings().engine == fic.FIC_ENGINE_DIRECT
    assert bits_equal(ti, di) and (tq == dq).all()


def test_decode_lena_full_pool(fic, h, lena_grey):
    # BASELINE.md: LenaGrey at B = 8, widthKernel 61 decodes in 7 iterations to avgError 0.25120544
    h.set_engine(fic.FIC_ENGINE_UMMA)  # (AUTO gives groups of fewer than 4 images to the CUDA-core search)
    _, q = h.encode_batch(np.stack([lena_grey] * 3), 8, 61, GREY)
    assert h.timings().engine == fic.FIC_ENGINE_UMMA
    _, avg, it = h.decode_batch(q, 256, 256, 8, 61, GREY)
    assert (it == 7).all()
    assert (avg.view(np.uint32) == np.float32(0.25120544).view(np.uint32)).all()


def test_timings(fic, h):
    h.set_engine(fic.FIC_ENGINE_UMMA)
    launches = []
    for n in (2, 8):
        h.encode_batch(grey_images(128, n, seed=n), 8, 29, GREY)
        t = h.timings()
        assert t.engine == fic.FIC_ENGINE_UMMA
        assert t.pool_ms > 0 and t.search_ms > 0 and t.kernel_ms > 0 and t.solve_ms > 0 and t.total_ms >= t.search_ms
        launches.append(t.launches)
    assert launches[0] == launches[1]
