"""The CPU reference of the key-frame half of the batched chain (tests/cpp/keyframe_chain_oracle.cpp) against the oracle's Python calls
composed as test_gpu_sequence.py composes them at its key frames: occupancy + CellSize and Min_dist circles -> detect_cells ->
detect_select (g++'s std::sort) -> undistort_points / feature_depth / unproject. Runs without a GPU."""
import numpy as np
import pytest

import helpers as H
import keyframe_chain as KC
import track_select as TS
from dsdtm_b200 import synth as S

LEVELS, SCALE = 5, 5000.0


def _tiled(period, seed, w, h):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


def _pair(cam, seed, n_match, tiled=False):
    """a rendered (or tiled) cur image, its 16-bit depth, a pose and n_match matches at sub-pixel positions; two of them sit where the
    occupancy index leaves the grid"""
    rng = np.random.default_rng(seed)
    w, h = cam["width"], cam["height"]
    pose = S.pose_from_xi(rng.uniform(-0.1, 0.1, 6))
    img, z = S.render(S.Scene(seed), cam, pose)
    if tiled:
        img = _tiled(15, seed, w, h)
    d16 = np.clip(np.rint(z * SCALE), 0, 65535).astype(np.uint16)
    m = np.zeros(200, TS.MATCH_DT)
    px = rng.uniform([8, 8], [w - 8, h - 8], (n_match, 2)).astype(np.float32)
    if n_match >= 4:
        px[0] = (5.25, -31.0)                                            # a negative row: linear index < 0
        px[1] = (w + 60.5, h - 0.5)                                      # column past the grid on the last row: index >= n_cells
    m["px"][:n_match] = px
    m["point"][:n_match] = np.arange(n_match)
    return img, d16, pose, m, px


CASES = {
    # name: (camera, dist, cell, min_dist, n_match, max_fts, tiled)
    "cell_lt_min_dist": ("KINECT", (0.0,) * 5, 15, 25, 120, 300, False),
    "cell_gt_min_dist": ("KINECT", (0.0,) * 5, 15, 10, 150, 300, False),
    "zero_matches": ("KINECT", (0.0,) * 5, 15, 15, 0, 300, False),
    "max_new_zero": ("KINECT", (0.0,) * 5, 15, 15, 150, 150, False),
    "max_new_negative": ("KINECT", (0.0,) * 5, 15, 15, 180, 100, False),
    "tiled": ("KINECT", (0.0,) * 5, 15, 15, 60, 300, True),
    "euroc": ("EUROC", KC.EUROC_DIST, 20, 15, 100, 300, False),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_cpp_reference_equals_python_composition(name):
    camn, dist, cell, min_dist, nm, max_fts, tiled = CASES[name]
    cam = dict(getattr(S, camn))
    oc = H.ocam(cam)
    imgs, d16s, poses, ms, pxs = [], [], [], [], []
    for k in range(3):                                                   # three pairs: depth, no depth, not wanted
        img, d16, pose, m, px = _pair(cam, 100 + 7 * k + len(name), nm, tiled)
        imgs.append(img); d16s.append(d16); poses.append(pose); ms.append(m); pxs.append(px)
    want = np.array([1, 1, 0], np.uint8)
    has = np.array([1, 0, 1], np.int32)
    got = KC.keyframe_chain(oc, LEVELS, cell, min_dist, max_fts, 5.0, dist, SCALE, np.stack(imgs), np.stack(ms), np.full(3, nm, np.int32),
                            np.stack(poses), np.stack(d16s), has, want, n_threads=2)
    for i in range(2):
        new, lf, skipped, tied = KC.compose(oc, LEVELS, cell, min_dist, max_fts, 5.0, dist, SCALE, imgs[i], pxs[i], poses[i],
                                      d16s[i] if has[i] else None)
        k = int(got["n_new"][i])
        assert KC.same_corners(got["corners"][i][:k], new), (name, i)
        assert got["lifted"][i][:k].tobytes() == lf.tobytes(), (name, i)
        assert (got["corners"][i][k:].view(np.uint8) == 0).all() and (got["lifted"][i][k:].view(np.uint8) == 0).all()
        assert got["occ_skipped"][i] == skipped == (2 if nm >= 4 else 0)
        assert got["tied"][i] == tied
        if max_fts - nm <= 0:
            assert k == 0
        else:
            assert k > 0 and k <= max_fts - nm
        if has[i] and k:
            assert (lf["status"] == KC.LIFT_OK).mean() > 0.5             # no holes; undistortion moves border pixels off the image
        if not has[i]:
            assert (lf["status"] == KC.LIFT_NO_DEPTH).all()
    assert got["n_new"][2] == 0 and not got["tied"][2]
    if tiled:
        assert got["tied"][0] and got["tied"][1]                         # the tiled cur images take the literal sort


def test_min_dist_circles_change_the_selection():
    """The Set_Mask circles matter: with Min_dist larger than CellSize the selection differs from the one with CellSize circles only,
    so the comparison above can tell whether both circle sets were painted."""
    cam = dict(S.KINECT)
    oc = H.ocam(cam)
    img, d16, pose, m, px = _pair(cam, 5, 120)
    a = KC.compose(oc, LEVELS, 15, 15, 300, 5.0, (0.0,) * 5, SCALE, img, px, pose)
    b = KC.compose(oc, LEVELS, 15, 25, 300, 5.0, (0.0,) * 5, SCALE, img, px, pose)
    assert not KC.same_corners(a[0], b[0])
