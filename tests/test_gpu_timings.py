"""What fic_get_timings reports for every encode entry: which stage fields are zero and which are positive, total_ms
against the stages, launches and search_evals -- for single host encodes (fused, direct, tcgen05), the device entry,
batches (fused, per-image direct, tcgen05 groups), the quadtree encode and a one-device multi handle."""
import os

import numpy as np
import pytest

from conftest import GOLD, to_argb_grey

pytestmark = pytest.mark.gpu

STAGES = ("h2d_ms", "pool_ms", "search_ms", "kernel_ms", "solve_ms", "d2h_ms")
EPS = 0.01  # ms: sums of event intervals that tile one span, each read at the events' resolution


@pytest.fixture(scope="module")
def h():
    import fractal_image_compression_b200 as fic

    hh = fic.Handle(0)
    yield hh
    hh.close()


@pytest.fixture(scope="module")
def l64():
    return np.fromfile(os.path.join(GOLD, "lena64.u8"), np.uint8).reshape(64, 64)


@pytest.fixture(scope="module")
def l256():
    return np.fromfile(os.path.join(GOLD, "lena_grey_256.u8"), np.uint8).reshape(256, 256)


def _positive(t, fields):
    for f in STAGES:
        v = getattr(t, f)
        assert (v > 0) if f in fields else (v == 0), (f, v)
    assert t.total_ms > 0 and t.total_ms >= t.search_ms and t.search_ms >= t.kernel_ms


def _nr(W, H, B):
    return (W // B) * (H // B)


def test_single_fused(fic, h, l64):
    h.set_engine(fic.FIC_ENGINE_AUTO)
    h.encode(to_argb_grey(l64), 8, 2, rgb=False)
    t = h.timings()
    assert t.engine == fic.FIC_ENGINE_FUSED and t.launches == 1  # the kernel reads the ARGB ints itself
    _positive(t, {"h2d_ms", "search_ms", "kernel_ms", "d2h_ms"})
    assert t.search_ms == t.kernel_ms
    assert abs(t.h2d_ms + t.search_ms + t.d2h_ms - t.total_ms) < EPS
    assert t.search_evals == _nr(64, 64, 8) * 2 * 2


@pytest.mark.parametrize("engine,wk", [("DIRECT", 2), ("UMMA", 13)])
def test_single_direct_umma(fic, h, l64, engine, wk):
    eng = getattr(fic, "FIC_ENGINE_" + engine)
    h.set_engine(eng)
    try:
        h.encode_u8(l64, 8, wk)
        tu = h.timings()
        h.encode(to_argb_grey(l64), 8, wk, rgb=False)
        t = h.timings()
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)
    for x in (tu, t):
        assert x.engine == eng
        _positive(x, set(STAGES))
        assert abs(x.h2d_ms + x.pool_ms + x.search_ms + x.solve_ms + x.d2h_ms - x.total_ms) < EPS
        assert x.search_evals == _nr(64, 64, 8) * wk * wk
    assert t.launches == tu.launches + 1  # the ARGB unpack


def test_single_iso_evals(fic, h, l64):
    h.encode(to_argb_grey(l64), 8, 2, rgb=fic.FIC_MODE_GREY_ISO)
    t = h.timings()
    assert t.engine == fic.FIC_ENGINE_DIRECT
    _positive(t, set(STAGES))
    assert t.search_evals == _nr(64, 64, 8) * 2 * 2 * 8


@pytest.mark.parametrize("engine,wk", [("DIRECT", 2), ("FUSED", 2), ("UMMA", 13)])
def test_planes_dev(fic, h, l64, engine, wk):
    import torch

    eng = getattr(fic, "FIC_ENGINE_" + engine)
    NR = _nr(64, 64, 8)
    d_p = torch.from_numpy(l64.copy()).cuda()
    d_i = torch.empty((NR, 3), dtype=torch.float32, device="cuda")
    d_q = torch.empty((NR, 3), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    h.set_engine(eng)
    try:
        h.encode_planes_dev(d_p.data_ptr(), 0, 64, 64, 8, wk, 0, NR, d_i.data_ptr(), d_q.data_ptr())
        h.sync()
        t = h.timings()
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)
    assert t.engine == eng and t.search_evals == NR * wk * wk and t.launches > 0
    assert t.kernel_ms > 0
    if engine == "FUSED":
        _positive(t, {"search_ms", "kernel_ms"})
        assert abs(t.search_ms - t.total_ms) < EPS
    else:
        _positive(t, {"pool_ms", "search_ms", "kernel_ms", "solve_ms"})
        assert abs(t.pool_ms + t.search_ms + t.solve_ms - t.total_ms) < EPS


def test_batch_fused_and_direct(fic, h, l64):
    imgs = np.stack([l64, l64[::-1], l64[:, ::-1]])
    h.set_engine(fic.FIC_ENGINE_AUTO)
    h.encode_batch_u8(imgs, 8, 2)
    t = h.timings()
    assert t.engine == fic.FIC_ENGINE_FUSED and t.launches == 1
    _positive(t, set())
    assert t.search_evals == 3 * _nr(64, 64, 8) * 4
    h.set_engine(fic.FIC_ENGINE_DIRECT)
    try:
        h.encode_u8(l64, 8, 2)
        single = h.timings().launches
        h.encode_batch_u8(imgs, 8, 2)
        t = h.timings()
        h.encode_batch(np.stack([to_argb_grey(p) for p in imgs]), 8, 2, rgb=False)
        ta = h.timings()
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)
    for x in (t, ta):
        assert x.engine == fic.FIC_ENGINE_DIRECT
        _positive(x, set())
        assert x.search_evals == 3 * _nr(64, 64, 8) * 4
    assert t.launches == 3 * single and ta.launches == 3 * (single + 1)


@pytest.mark.parametrize("n", [4, 257])  # one tcgen05 group; two (a group holds at most 256 images)
def test_batch_umma_groups(fic, h, l64, n):
    imgs = np.stack([np.roll(l64, i, 1) for i in range(n)])
    h.set_engine(fic.FIC_ENGINE_UMMA)
    try:
        h.encode_batch_u8(imgs, 8, 13)
        t = h.timings()
    finally:
        h.set_engine(fic.FIC_ENGINE_AUTO)
    assert t.engine == fic.FIC_ENGINE_UMMA and t.launches > 0
    _positive(t, {"pool_ms", "search_ms", "kernel_ms", "solve_ms"})
    assert t.total_ms >= t.pool_ms + t.search_ms + t.solve_ms - EPS
    assert t.search_evals == n * _nr(64, 64, 8) * 13 * 13


def _quadtree(fic, h, plane, b_max, b_min, wk):
    """(timings of the quadtree encode, summed launches and evals of its levels' single encodes, last level's engine)."""
    h.encode_quadtree(plane, b_max, b_min, wk, 25.0)
    t = h.timings()
    W = plane.shape[1]
    launches = evals = 0
    B = b_max
    while B >= b_min:
        wl = wk or 2 * W // B - 3
        h.encode_u8(plane, B, wl)
        s = h.timings()
        launches += s.launches
        evals += s.search_evals
        engine = s.engine
        B //= 2
    return t, launches, evals, engine


def test_quadtree(fic, h, l256):
    h.set_engine(fic.FIC_ENGINE_AUTO)
    extra = {}
    for b_max, b_min, wk, fused in [(16, 8, 2, True), (16, 8, 0, False), (16, 4, 2, True), (16, 4, 0, False)]:
        t, launches, evals, engine = _quadtree(fic, h, l256, b_max, b_min, wk)
        assert t.engine == engine and t.search_evals == evals
        assert (engine == fic.FIC_ENGINE_FUSED) == fused
        _positive(t, {"search_ms", "kernel_ms"} if fused else {"pool_ms", "search_ms", "kernel_ms", "solve_ms"})
        nl = {8: 2, 4: 3}[b_min]
        extra.setdefault(nl, set()).add(t.launches - launches)
    # one decimation, one collage kernel per level, decide, scan and scatter: depends on the number of levels only
    assert len(extra[2]) == 1 and len(extra[3]) == 1
    assert extra[3].pop() - extra[2].pop() == 1


@pytest.mark.parametrize("engine", ["AUTO", "DIRECT"])
def test_multi_one_device(fic, h, l64, engine):
    eng = getattr(fic, "FIC_ENGINE_" + engine)
    h.set_engine(eng)
    m = fic.MultiHandle([0])
    try:
        m.set_engine(eng)
        h.encode_u8(l64, 8, 2)
        s = h.timings()
        m.encode(l64, 8, 2)
        t0, tv = m.timings(0), m.timings()
    finally:
        m.close()
        h.set_engine(fic.FIC_ENGINE_AUTO)
    for t in (t0, tv):
        assert t.engine == s.engine and t.launches == s.launches and t.search_evals == s.search_evals
        _positive(t, {f for f in STAGES if getattr(s, f) > 0})
        assert t.h2d_ms > 0 and t.d2h_ms > 0
    assert [getattr(tv, f) for f in STAGES + ("total_ms",)] == [getattr(t0, f) for f in STAGES + ("total_ms",)]
