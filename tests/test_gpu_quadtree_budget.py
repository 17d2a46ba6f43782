"""The quadtree encode to a byte budget on the GPU (fic_encode_quadtree_budget, fic_encode_quadtree_budget_batch): stream
and m* bits equal to the CPU oracle's across images, modes, level pairs, windows and budgets; the stream equal to the
max_mse encode's at m* on every engine; batches with per-image budgets equal to the single calls; the rejections; a
4096^2 whole-pool encode against the characterisation; and launch counts."""
import math

import numpy as np
import pytest

from test_oracle_quadtree_budget import CASES, SIZE_MAX, budgets_for, case_id, case_image, geometry

pytestmark = pytest.mark.gpu


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


def bits(m):
    return np.float64(m).tobytes()


def _images(rgb, n, W=64):
    from fractal_image_compression_b200 import synth

    out = []
    for i in range(n):
        kind = i % 4
        if kind == 0:
            g = [synth.structured(W, W, 5 + 3 * i + k) for k in range(3)]
        elif kind == 1:
            g = [synth.noise(W, W, 7 + 3 * i + k) for k in range(3)]
        elif kind == 2:
            g = [np.full((W, W), (40 * i + 50 * k) % 256, np.uint8) for k in range(3)]
        else:
            t = synth.noise(8, 8, 11 + i)
            g = [np.tile(t, (W // 8, W // 8)) for _ in range(3)]
        out.append(np.stack(g) if rgb else g[0])
    return np.stack(out)


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_matches_the_oracle(h, fic, case):
    from oracle import quadtree_budget as QB

    rgb, name, pair, wk = case
    img = case_image(rgb, name, wk)
    oenc = QB.encode_quadtree_rgb_budget if rgb else QB.encode_quadtree_budget
    least, _, _ = geometry(img, pair)
    with pytest.raises(fic.FicError) as e:
        h.encode_quadtree_budget(img, pair[0], pair[1], wk, least - 1)
    assert e.value.code == fic._lib.FIC_E_ARG
    for b in budgets_for(img, pair, lambda m: len(h.encode_quadtree(img, pair[0], pair[1], wk, m))):
        s, m = h.encode_quadtree_budget(img, pair[0], pair[1], wk, b)
        os_, om = oenc(img, pair[0], pair[1], wk, b)
        assert s == os_ and bits(m) == bits(om), (b, m, om)


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("engine,wk", [("DIRECT", 0), ("DIRECT", 2), ("FUSED", 2), ("UMMA", 0)])
def test_engines_match_the_max_mse_encode(h, fic, rgb, engine, wk):
    h.set_engine(getattr(fic, "FIC_ENGINE_" + engine))
    img = _images(rgb, 1, 128)[0]
    for b_max, b_min in [(16, 8), (16, 4), (8, 4)]:
        least, full, _ = geometry(img, (b_max, b_min))
        for b in (least, (2 * least + full) // 3, (least + 2 * full) // 3, full - 1):
            s, m = h.encode_quadtree_budget(img, b_max, b_min, wk, b)
            assert h.timings().engine == getattr(fic, "FIC_ENGINE_" + engine)
            assert len(s) <= b and s == h.encode_quadtree(img, b_max, b_min, wk, m)
            if m != -math.inf:
                assert len(h.encode_quadtree(img, b_max, b_min, wk, float(np.nextafter(m, -np.inf)))) > b


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("n,W,wk", [(1, 64, 2), (5, 64, 2), (64, 64, 0), (260, 128, 0)])
def test_batch_matches_single_calls(h, rgb, n, W, wk):
    # 260 whole-pool images of 128^2: the finest level runs as two tcgen05 group searches (at most 256 images a group)
    planes = _images(rgb, n, W)
    least, full, _ = geometry(planes[0], (16, 8))
    budgets = [least + (i * 997) % (full - least + 1) for i in range(n)]
    got, mse = h.encode_quadtree_budget_batch(planes, 16, 8, wk, budgets)
    assert mse.dtype == np.float64 and mse.shape == (n,)
    picks = range(n) if n <= 64 else list(range(6)) + list(range(n - 6, n))
    for i in picks:
        s, m = h.encode_quadtree_budget(planes[i], 16, 8, wk, budgets[i])
        assert got[i] == s and bits(mse[i]) == bits(m), i
    one, m1 = h.encode_quadtree_budget_batch(planes, 16, 8, wk, full)  # an int budget for every image
    assert all(len(s) == len(one[0]) for s in one) and (m1 == -math.inf).all()


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
def test_rejections(h, fic, rgb):
    import ctypes as C

    L = fic._lib.load()
    planes = _images(rgb, 5, 64)
    least, full, leaf = geometry(planes[0], (16, 4))
    mode = fic.FIC_MODE_RGB_QT if rgb else fic.FIC_MODE_GREY_QT
    a = np.ascontiguousarray(planes)
    stride = full
    buf = np.zeros(5 * stride, np.uint8)
    sizes = np.zeros(5, np.uintp)
    mse = np.zeros(5, np.float64)
    budgets = np.array([full, full, least - 1, least - 1, full], np.uintp)

    def call(n=5, md=mode, bud=budgets, st=stride, out=buf, sz=sizes, ms=mse):
        p = lambda x: None if x is None else x.ctypes.data_as(C.c_void_p)
        return L.fic_encode_quadtree_budget_batch(h._h, md, p(a), n, 64, 64, 16, 4, 2, p(bud), p(out), st, p(sz), p(ms))

    assert call() == fic._lib.FIC_E_ARG  # infeasible budgets fail the whole batch, naming the lowest
    assert "image 2" in L.fic_last_error(h._h).decode()
    assert (sizes == least).all() and (mse == np.inf).all()
    budgets[2:4] = full
    assert call(st=least) == fic._lib.FIC_E_ARG  # stride below the streams' sizes: every size reported
    need = sizes.copy()
    assert (need >= least).all() and need.max() > least
    assert call() == 0
    for bad in (dict(bud=None), dict(out=None), dict(sz=None), dict(ms=None), dict(n=0), dict(n=-1), dict(md=0), dict(md=5)):
        assert call(**bad) == fic._lib.FIC_E_ARG, bad
    # the single entry: capacity too small, a budget below the unsplit tree, NULL outputs, a bad mode
    one = np.ascontiguousarray(planes[0])
    n, m = C.c_size_t(0), C.c_double(0)
    out = np.zeros(full, np.uint8)
    p = lambda x: x.ctypes.data_as(C.c_void_p)
    assert L.fic_encode_quadtree_budget(h._h, mode, p(one), 64, 64, 16, 4, 2, full, p(out), least, C.byref(n), C.byref(m)) == fic._lib.FIC_E_ARG
    assert n.value > least
    assert L.fic_encode_quadtree_budget(h._h, mode, p(one), 64, 64, 16, 4, 2, least - 1, p(out), full, C.byref(n), C.byref(m)) == fic._lib.FIC_E_ARG
    assert n.value == least and m.value == math.inf
    assert L.fic_encode_quadtree_budget(h._h, mode, p(one), 64, 64, 16, 4, 2, full, p(out), full, None, C.byref(m)) == fic._lib.FIC_E_ARG
    assert L.fic_encode_quadtree_budget(h._h, mode, p(one), 64, 64, 16, 4, 2, full, p(out), full, C.byref(n), None) == fic._lib.FIC_E_ARG
    assert L.fic_encode_quadtree_budget(h._h, 1, p(one), 64, 64, 16, 4, 2, full, p(out), full, C.byref(n), C.byref(m)) == fic._lib.FIC_E_ARG
    s, mm = h.encode_quadtree_budget(one, 16, 4, 2, SIZE_MAX)
    assert len(s) == full and mm == -math.inf


def test_4096_whole_pool(h):
    from fractal_image_compression_b200 import synth

    img = synth.structured(4096, 4096, 3)
    least, full, _ = geometry(img, (16, 4))
    b = (least + full) // 2
    s, m = h.encode_quadtree_budget(img, 16, 4, 0, b)
    assert len(s) <= b and math.isfinite(m)
    assert s == h.encode_quadtree(img, 16, 4, 0, m)
    assert len(h.encode_quadtree(img, 16, 4, 0, float(np.nextafter(m, -np.inf)))) > b


@pytest.mark.parametrize("rgb", [False, True], ids=["grey", "rgb"])
@pytest.mark.parametrize("wk", [0, 2])
def test_launches(h, rgb, wk):
    counts = []
    for n in (8, 64):
        planes = _images(rgb, n, 64)
        h.encode_quadtree_batch(planes, 16, 4, wk, 25.0)
        base = h.timings().launches
        h.encode_quadtree_budget_batch(planes, 16, 4, wk, 4000)
        counts.append(h.timings().launches)
        assert counts[-1] <= base + 2, (n, counts[-1], base)
    assert counts[0] == counts[1]
