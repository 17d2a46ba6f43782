"""The quadtree encode to a byte budget in the CPU oracle, against its characterisation: the stream is the max_mse
oracle's stream at m*, it fits, and the stream at nextafter(m*, -inf) does not (or m* = -inf); m* is never -0.0; a
budget below the unsplit tree is rejected with that tree's size; size and m* are monotone in the budget.  Grey and RGB,
images with distinct, equal (flat) and repeated (tiled) collage errors."""
import math
import os

import numpy as np
import pytest

from conftest import GOLD

PAIRS = [(16, 8), (16, 4), (8, 4), (16, 16)]
SIZE_MAX = 2**64 - 1
MSES = [0.0, 5.0, 30.0, 100.0, 250.0, 1000.0]


def _grey_images():
    lena = np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)
    rng = np.random.default_rng(7)
    tile = rng.integers(0, 256, (16, 16), dtype=np.uint8)
    return {
        "lena": lena,
        "noise": rng.integers(0, 256, (64, 64), dtype=np.uint8),
        "flat": np.zeros((64, 64), np.uint8),  # every collage error is 0: m* = +0.0 between the two extreme trees
        "binary": (rng.integers(0, 2, (64, 64)) * 255).astype(np.uint8),
        "ties": np.tile(tile, (4, 4)),
    }


def _rgb_images():
    lena = np.fromfile(os.path.join(GOLD, "lena_colored_256.rgb"), np.uint8).reshape(256, 256, 3).transpose(2, 0, 1).copy()
    rng = np.random.default_rng(11)
    tile = rng.integers(0, 256, (3, 16, 16), dtype=np.uint8)
    return {
        "lena": lena,
        "noise": rng.integers(0, 256, (3, 64, 64), dtype=np.uint8),
        "flat": np.stack([np.full((64, 64), v, np.uint8) for v in (10, 128, 240)]),  # every error per pixel the same
        "binary": (rng.integers(0, 2, (3, 64, 64)) * 255).astype(np.uint8),
        "ties": np.tile(tile, (1, 4, 4)),
    }


GREY, RGB = _grey_images(), _rgb_images()
# wk 0 (every level's whole pool) on 64^2 images only: the CPU search of a 256^2 whole pool takes seconds per encode
CASES = [(rgb, name, pair, wk) for rgb in (False, True) for name in GREY for pair in PAIRS for wk in (0, 2)]


def case_id(c):
    rgb, name, pair, wk = c
    return f"{'rgb' if rgb else 'grey'}-{name}-{pair[0]}x{pair[1]}-wk{wk}"


def case_image(rgb, name, wk):
    img = (RGB if rgb else GREY)[name]
    if wk == 0 and img.shape[-1] > 64:
        img = img[..., ::4, ::4].copy()
    return img


def geometry(img, pair):
    """(unsplit tree's size, fully split tree's size, leaf bytes)."""
    H, W = img.shape[-2:]
    leaf = 20 if img.ndim == 3 else 12
    top = (W // pair[0]) * (H // pair[0])
    flags = (top + 3) & ~3
    return 32 + flags + leaf * top, 32 + flags + leaf * (W // pair[1]) * (H // pair[1]), leaf


def budgets_for(img, pair, sized):
    """Budgets of a case: the unsplit and fully split sizes, the sizes at MSES and +-1 byte and +- one leaf around them,
    the midpoints of the gaps between consecutive sizes wider than one split (inside a tie group), and SIZE_MAX.
    sized(m): the max_mse stream's size."""
    least, full, leaf = geometry(img, pair)
    sizes = sorted({sized(m) for m in MSES} | {least, full})
    out = {least, full, SIZE_MAX}
    for s in sizes:
        out |= {s - 1, s + 1, s - leaf, s + leaf, s - 3 * leaf, s + 3 * leaf, s}
    for a, b in zip(sizes, sizes[1:]):
        if b - a > 3 * leaf:
            out.add((a + b) // 2)
    return sorted(b for b in out if b >= least)


@pytest.fixture(scope="module")
def qb():
    from oracle import quadtree_budget

    quadtree_budget.build()
    return quadtree_budget


@pytest.fixture(scope="module")
def qt():
    from oracle import quadtree, quadtree_rgb

    return quadtree, quadtree_rgb


def max_mse_encoder(qt, rgb):
    quadtree, quadtree_rgb = qt
    return quadtree_rgb.encode_quadtree_rgb if rgb else quadtree.encode_quadtree


def budget_encoder(qb, rgb):
    return qb.encode_quadtree_rgb_budget if rgb else qb.encode_quadtree_budget


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_budget_matches_characterisation(qb, qt, case):
    rgb, name, pair, wk = case
    img = case_image(rgb, name, wk)
    enc, benc = max_mse_encoder(qt, rgb), budget_encoder(qb, rgb)
    cache = {}

    def at(m):  # keyed by the bits: -0.0 and +0.0 are distinct keys
        key = np.float64(m).tobytes()
        if key not in cache:
            cache[key] = enc(img, pair[0], pair[1], wk, m)
        return cache[key]

    least, full, _ = geometry(img, pair)
    assert len(at(math.inf)) == least and len(at(-math.inf)) == full
    with pytest.raises(qb.BudgetInfeasible) as e:
        benc(img, pair[0], pair[1], wk, least - 1)
    assert e.value.min_bytes == least
    prev_size, prev_m = 0, math.inf
    for b in budgets_for(img, pair, lambda m: len(at(m))):
        s, m = benc(img, pair[0], pair[1], wk, b)
        assert s == at(m), (b, m)
        assert len(s) <= b
        assert not (m == 0 and math.copysign(1, m) < 0), "m* must be +0.0"
        if m != -math.inf:
            assert len(at(float(np.nextafter(m, -np.inf)))) > b, (b, m)
        assert len(s) >= prev_size and m <= prev_m, (b, len(s), m)
        prev_size, prev_m = len(s), m
    s, m = benc(img, pair[0], pair[1], wk, SIZE_MAX)
    assert m == -math.inf and len(s) == full


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_flat_image_is_one_tie_group(qb, qt, rgb):
    """Every block of a flat image has the same collage error per pixel (zero on the black grey image): any budget between
    the unsplit and the fully split tree gives the unsplit tree, well under the budget, and one step below m* the fully
    split one."""
    img = (RGB if rgb else GREY)["flat"]
    least, full, _ = geometry(img, (16, 4))
    s, m = budget_encoder(qb, rgb)(img, 16, 4, 2, (least + full) // 2)
    assert len(s) == least
    assert len(max_mse_encoder(qt, rgb)(img, 16, 4, 2, float(np.nextafter(m, -np.inf)))) == full
    if not rgb:
        assert m == 0 and math.copysign(1, m) > 0
    s, m = budget_encoder(qb, rgb)(img, 16, 4, 2, full)
    assert len(s) == full and m == -math.inf
