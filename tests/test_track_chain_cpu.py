"""CPU suite for the tracked-pose chain (dsdtm_batch_run flags 7): the circle-span rule the selection kernel tests instead of a mask
bitmap, and the whole-chain driver built on the oracle (tests/cpp/track_chain_oracle.cpp) against the Python restatement of SearchLocalPoints' selection."""
import numpy as np
import pytest

import helpers as H
import oracle as O
import track_select as TS
from dsdtm_b200 import synth as S
from dsdtm_b200 import workload as W


def _span_mask(w, h, cx, cy, r):
    """pixels painted by cv::circle(c, r, -1) according to the span rule: |dy| <= r and |dx| <= span[|dy|]"""
    spans = W.circle_mask_offsets(r)
    half = np.full(2 * r + 1, -1)
    for dy, hw in spans.items():
        half[dy + r] = hw
    Y, X = np.mgrid[0:h, 0:w]
    dy = Y - cy
    inside = np.abs(dy) <= r
    hw = np.where(inside, half[np.clip(dy + r, 0, 2 * r)], -1)
    return inside & (np.abs(X - cx) <= hw)


@pytest.mark.parametrize("w", [640, 752])
@pytest.mark.parametrize("r", [5, 15, 30])
def test_circle_span_rule_equals_cv_circle(w, r):
    """The selection kernel never paints a mask: a pixel is masked iff it lies within the row spans of an earlier circle. That rule
    must equal the pinned filled circle (orc_circle_fill, tests/golden/circle_cv2.npz) for centres inside, on and beyond every border
    (clipping at the border only removes pixels outside the image)."""
    h = 480
    spans = W.circle_mask_offsets(r)
    assert all(spans[dy] == spans[-dy] for dy in range(r + 1))           # the kernel's table is indexed by |dy|
    xs = [-r - 2, -r, -1, 0, 1, r, w // 2, w - 1 - r, w - 1, w, w + r - 1, w + r + 3]
    ys = [-r - 2, -r, -1, 0, r, h // 2, h - 1 - r, h - 1, h, h + r + 3]
    for cx in xs:
        for cy in ys:
            img = np.full((h, w), 255, np.uint8)
            O.circle_fill(img, cx, cy, r, 0)
            assert ((img == 0) == _span_mask(w, h, cx, cy, r)).all(), (cx, cy)


@pytest.mark.parametrize("cam_name", ["KINECT", "EUROC"])
def test_oracle_track_selection_equals_replay(cam_name):
    """The whole-chain driver's selection (full-size mask, orc_circle_fill) equals the Python restatement of SearchLocalPoints over the
    same records, for found counts with many ties; its solve equals orc_pose_optimization on those matches from T_c2r * T_ref."""
    cam = dict(getattr(S, cam_name))
    oc = H.ocam(cam)
    b = TS.make_batch(cam, 3, 300, n_scenes=3, empty_pair=2)
    rng = np.random.default_rng(5)
    founds = [np.ones((3, 300), np.int32), rng.integers(1, 3, (3, 300)).astype(np.int32), rng.integers(-2, 40, (3, 300)).astype(np.int32)]
    for found in founds:
        o = TS.pair_batch_track(oc, 5, 15, b["ref_pyrs"], b["cur_imgs"], b["feats"], b["n_feats"], b["centers"], b["poses_ref"],
                               b["poses_in"], 5, 0, 8, 300, 2, 10, found=found, ba_iters=100, n_threads=3)
        assert o["n_matches"][2] == 0 and o["summaries"]["termination"][2] == O.BA_NO_RESIDUALS
        assert o["n_matches"][:2].min() > 50
        for i in range(3):
            want = TS.replay(o["reproj"][i], found[i], cam["width"], cam["height"], 15)
            TS.assert_matches_equal(o["matches"][i], int(o["n_matches"][i]), want)
            m = o["matches"][i][:o["n_matches"][i]]
            nm = np.array([O.feature_normal(oc, p) for p in m["px"]]).reshape(-1, 3)
            pw = b["feats"][i]["point_w"][m["point"]].reshape(-1, 3)
            start = O.se3_mul(o["poses_c2r"][i], b["poses_ref"][i])
            pose, res, summ = O.pose_optimization(nm, m["level"], pw, start)
            assert (pose == o["poses"][i]).all() and (res == o["res_norm"][i][:len(m)]).all()
            assert summ.tobytes() == o["summaries"][i].tobytes()
            assert (o["res_norm"][i][len(m):] == 0).all()
