"""Feature_detector::detect on the device (dsdtm_detect / dsdtm_detect_batch, ref: src/Feature_detection.cpp:69-154) against the
oracle's detect_cells + detect_select, whose selection runs g++'s std::sort: the same corners in the same order, score bits equal.
Tiled scenes carry many tied scores above 20; there the device must take the literal-sort path and the stable-order selection
must differ, which shows the comparison can tell the two orders apart."""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from dsdtm_b200 import capi, synth as S

pytestmark = pytest.mark.gpu

CELL = 15


def _tiled(period, seed, w=640, h=480):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


def _want(img, cell=CELL, thr=5.0, occ=None, mask=None, circles=None, max_new=300, levels=5, stable=False):
    packed, offs, ws, hs = O.pyramid(img, levels)
    cells = O.detect_cells(packed, offs, ws, hs, cell, occ, thr)
    if max_new <= 0:
        return np.zeros(0, capi.CORNER_DT)
    m = np.full(img.shape, 255, np.uint8) if mask is None else mask.copy()
    for c in (circles if circles is not None else []):
        O.circle_fill(m, O.cvround(c["px"][0]), O.cvround(c["px"][1]), int(c["radius"]))
    if not stable:
        return O.detect_select(cells, m, cell, max_new)[0]
    out = []
    for i in np.argsort(-cells["score"], kind="stable"):
        c = cells[i]
        if c["score"] > 20 and m[c["y"], c["x"]] == 255:
            out.append(c)
            O.circle_fill(m, int(c["x"]), int(c["y"]), cell)
            if len(out) >= max_new:
                break
    return np.array(out, capi.CORNER_DT)


def _same(got, want):
    return (len(got) == len(want) and (got["x"] == want["x"]).all() and (got["y"] == want["y"]).all()
            and (got["level"] == want["level"]).all() and (got["score"].view(np.uint32) == want["score"].view(np.uint32)).all())


def _circles(pts, r=15):
    c = np.zeros(len(pts), capi.CIRCLE_DT)
    c["px"] = np.asarray(pts, np.float32)
    c["radius"] = r
    return c


def _holes(seed, w=640, h=480):
    rng = np.random.default_rng(seed)
    m = np.full((h, w), 255, np.uint8)
    for _ in range(12):
        x, y = rng.integers(0, w - 60), rng.integers(0, h - 60)
        m[y:y + rng.integers(5, 60), x:x + rng.integers(5, 60)] = rng.choice([0, 128, 254])
    return m


@pytest.mark.parametrize("thr", [5.0, 20.0])
@pytest.mark.parametrize("with_occ", [False, True])
def test_kinect_equals_std_sort_selection(ctx, scenario, thr, with_occ):
    img = scenario["ref_img"]
    ctx.upload(0, img)
    occ = (np.random.default_rng(3).random(ctx.n_cells) < 0.3).astype(np.uint8) if with_occ else None
    got, exact = ctx.detect(0, thr, occupied=occ)
    want = _want(img, thr=thr, occ=occ)
    assert len(want) > 100 and _same(got[0], want)
    assert not exact[0]
    if not with_occ and thr == 5.0:
        assert _same(got[0], scenario["corners"])


def test_euroc_test1_geometry(golden):
    img = golden["test1_fast"]["img"]
    c = capi.Context(dict(S.EUROC), levels=5, cell_size=30, max_feats=64, max_patches=64, max_frames=2, max_batch=2)
    try:
        c.upload(0, img)
        got, exact = c.detect(0, 5.0)
        want = _want(img, cell=30)
        assert len(want) > 50 and _same(got[0], want) and not exact[0]
    finally:
        c.close()


def test_prior_circles_and_mask_with_holes(ctx, scenario):
    img = scenario["ref_img"]
    ctx.upload(0, img)
    rng = np.random.default_rng(11)
    inside = rng.uniform([0, 0], [640, 480], (40, 2))
    border = [(0, 0), (639, 479), (0, 240), (639, 100), (320, 0), (200, 479), (10.5, 11.5), (-0.5, 300.5)]
    beyond = [(-5, 200), (-15, -15), (650, 240), (660, 490), (300, -14.6), (300, 494.4), (-100, -100), (1e6, 5)]
    circ = _circles(np.concatenate([inside, border, beyond]))
    mask = _holes(5)
    for m, cs in ((None, circ), (mask, None), (mask, circ)):
        got, exact = ctx.detect(0, 5.0, mask=m, circles=cs)
        assert _same(got[0], _want(img, mask=m, circles=cs)) and not exact[0]


@pytest.mark.parametrize("max_new", [1, 7, 300, 0, -4])
def test_max_new_caps_the_walk(ctx, scenario, max_new):
    img = scenario["ref_img"]
    ctx.upload(0, img)
    got, _ = ctx.detect(0, 5.0, max_new=max_new)
    want = _want(img, max_new=max_new)
    assert _same(got[0], want) and len(want) == max(max_new, 0)


@pytest.mark.parametrize("period", [15, 30, 45])
def test_tiled_scenes_take_the_literal_sort(ctx, period):
    img = _tiled(period, period)
    ctx.upload(0, img)
    got, exact = ctx.detect(0, 5.0)
    want = _want(img)
    assert exact[0] and _same(got[0], want)
    assert not _same(want, _want(img, stable=True)), "a stable sort selects the same features: the scene does not discriminate"
    mask = _holes(period)
    circ = _circles(np.random.default_rng(period).uniform([-20, -20], [660, 500], (30, 2)))
    got, exact = ctx.detect(0, 5.0, mask=mask, circles=circ, max_new=120)
    assert exact[0] and _same(got[0], _want(img, mask=mask, circles=circ, max_new=120))


def test_mixed_batch_equals_single_frames(ctx, scenario):
    imgs = [scenario["ref_img"], _tiled(15, 1), scenario["cur_img"], _tiled(45, 2), _tiled(30, 3)]
    n = len(imgs)
    for i, im in enumerate(imgs):
        ctx.upload(i, im)
    rng = np.random.default_rng(9)
    occ = (rng.random((n, ctx.n_cells)) < 0.2).astype(np.uint8)
    masks = np.stack([np.full((480, 640), 255, np.uint8)] + [_holes(20 + i) for i in range(1, n)])
    circles = [_circles(rng.uniform([-20, -20], [660, 500], (k, 2))) for k in (0, 25, 3, 40, 10)]
    max_new = np.array([300, 7, 1, 300, 0], np.int32)
    got, exact = ctx.detect(0, 5.0, occupied=occ, mask=masks, circles=circles, max_new=max_new, n=n)
    for i in range(n):
        one, ex1 = ctx.detect(i, 5.0, occupied=occ[i], mask=masks[i], circles=circles[i], max_new=int(max_new[i]))
        assert _same(got[i], one[0]) and exact[i] == ex1[0], i
        assert _same(got[i], _want(imgs[i], occ=occ[i], mask=masks[i], circles=circles[i], max_new=int(max_new[i]))), i
    assert exact[1] and exact[3] and not exact[0] and not exact[2]


def test_bad_arguments_return_e_arg(ctx):
    L, h = ctx.L, ctx.hp
    out = np.zeros(300, capi.CORNER_DT)
    n_out = np.zeros(9, np.int32)
    mn = np.full(9, 300, np.int32)
    circ = _circles([(100, 100)])
    nc = np.ones(9, np.int32)
    f = C.c_float(5.0)

    def batch(first=0, n=1, circles=None, cs=0, ncirc=None, max_new=mn, stride=300, o=out):
        return L.dsdtm_detect_batch(h, first, n, f, None, None, capi._p(circles), cs, capi._p(ncirc), capi._p(max_new), stride,
                                    capi._p(o), capi._p(n_out), None)
    assert batch() == 0
    assert batch(first=11, n=2) == -1                                    # slot out of range (max_frames 12)
    assert batch(n=9) == -1                                              # n > max_batch
    assert batch(stride=299) == -1                                       # max_new > out_stride
    assert batch(o=None) == -1                                           # NULL out
    for r in (-1, 65):
        bad = circ.copy(); bad["radius"] = r
        assert batch(circles=bad, cs=1, ncirc=nc) == -1                  # radius out of range
    assert batch(circles=circ, cs=1, ncirc=nc) == 0
    n1 = C.c_int(0)
    assert L.dsdtm_detect(h, 12, f, None, None, None, 0, 300, capi._p(out), C.byref(n1), None) == -1
    assert L.dsdtm_detect(h, 0, f, None, None, capi._p(circ), 1, 300, None, C.byref(n1), None) == -1
    big = dict(S.KINECT, width=800, height=600)
    c2 = capi.Context(big, levels=4, cell_size=15, max_feats=16, max_patches=16, max_frames=1, max_batch=1)
    try:                                                                 # 800 x 600 does not fit the 752 x 480 bitmap
        assert c2.L.dsdtm_detect(c2.hp, 0, f, None, None, None, 0, 300, capi._p(out), C.byref(n1), None) == -1
    finally:
        c2.close()
