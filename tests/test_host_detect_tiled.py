"""Feature_detector::detect through the C++ adapter on a frame that already carries features, as CraeteKeyframe calls it
(ref: src/Tracking.cpp:415-416): SearchLocalPoints has painted its circles into mImgMask, Set_Mask adds Min_dist circles around
the features with map points, and the mask goes to the device with the occupancy grid. The scene is tiled, so its scores tie
and the selection depends on std::sort's order of equal scores."""
import ctypes as C

import numpy as np
import pytest

import hostlib as HL
import oracle as O
from dsdtm_b200 import synth as S

CELL, MIN_DIST, LEVELS = 15, 15, 5


def _tiled(period, seed, w=640, h=480):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


def _points(cam, px, depth=2.0):
    fx, fy, cx, cy = (float(np.float32(cam[k])) for k in ("fx", "fy", "cx", "cy"))
    return np.stack([(px[:, 0] - cx) / fx * depth, (px[:, 1] - cy) / fy * depth, np.full(len(px), depth)], 1)


@pytest.mark.gpu
def test_detect_on_tiled_frame_with_existing_features(built):
    cam = dict(S.KINECT)
    img = _tiled(30, 30)
    cam_h = HL.configure(cam, cell=CELL, max_fts=300, min_dist=MIN_DIST)
    g0 = HL.HFrame(cam_h, img, S.IDENTITY)
    n0 = g0.detect(5.0)
    px0, _, _ = g0.features()
    g0.attach_points(_points(cam, px0.astype(np.float64)), np.ones(n0, np.uint8))
    kf_h = HL.lib().hs_keyframe_new(g0.h)

    cur = HL.HFrame(cam_h, img, S.IDENTITY)
    nrep = C.c_int(0)
    m = HL.lib().hs_search_local_points(cam_h, cur.h, kf_h, None, C.byref(nrep))
    assert m > 20, m
    mask = cur.mask()                                     # SearchLocalPoints' CellSize circles
    assert (mask == 0).any()
    px, lv, _ = cur.features()
    has = (np.arange(m) % 2 == 0).astype(np.uint8)
    cur.attach_points(_points(cam, px.astype(np.float64)), has)

    n = cur.detect(5.0, use_existing=True)
    got_px, got_lv, _ = cur.features()

    # the oracle: Set_ExistingFeatures' occupancy, Set_Mask's Min_dist circles, detect_cells + detect_select (std::sort)
    rows, cols = O.grid_dims(640, 480, CELL)
    occ = np.zeros(rows * cols, np.uint8)
    for x, y in px:
        occ[int(np.float32(y) / np.float32(CELL)) * cols + int(np.float32(x) / np.float32(CELL))] = 1
    for (x, y), h in zip(px, has):
        if h:
            O.circle_fill(mask, O.cvround(x), O.cvround(y), MIN_DIST)
    packed, offs, ws, hs = O.pyramid(img, LEVELS)
    cells = O.detect_cells(packed, offs, ws, hs, CELL, occ, 5.0)
    sel = cells["score"][cells["score"] > 20]
    assert len(sel) > len(np.unique(sel))                 # tied scores: the literal-sort path
    want, _ = O.detect_select(cells, mask, CELL, 300, n_existing=m)
    assert n == m + len(want) and len(want) > 0
    assert (got_px[:m] == px).all()
    assert (got_px[m:, 0] == want["x"]).all() and (got_px[m:, 1] == want["y"]).all() and (got_lv[m:] == want["level"]).all()
    assert cur.mask().max() == 0                          # mImgMask.release() (ref: :153)
