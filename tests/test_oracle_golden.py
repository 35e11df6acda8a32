"""CPU suite: the oracle against the golden vectors (cv2 4.13, the reference's FAST library, the 167-corner KAT) and,
where a checkout of the reference is present, against oracle/_ref (the reference's own FAST sources)."""
import numpy as np
import pytest

import oracle as O


def test_pyrdown_matches_cv2_goldens(golden):
    g = golden["pyrdown_cv2"]
    i = 0
    while "in%d" % i in g:
        assert (O.pyrdown(g["in%d" % i]) == g["out%d" % i]).all(), i
        i += 1
    assert i == 7


def test_pyramid_chain_matches_cv2_on_test1(golden):
    g = golden["test1_fast"]
    packed, offs, ws, hs = O.pyramid(g["img"], 5)
    assert list(ws) == [752, 376, 188, 94, 47] and list(hs) == [480, 240, 120, 60, 30]   # SURVEY 3.5
    for l in range(1, 5):
        assert (O.pyr_level(packed, offs, ws, hs, l) == g["pyr%d" % l]).all(), l


def test_fast_kat_167_corners(golden):
    """ref: Thirdparty/fast/test/test.cpp:20,45,52 -- FAST-10 @75 on test1.png extracts 167 features."""
    g = golden["test1_fast"]
    xy = O.fast10_detect(g["img"], 75)
    assert len(xy) == 167
    assert (xy == g["xy75"]).all()


@pytest.mark.parametrize("barrier", [75, 20])
def test_fast_detect_score_nonmax_equal_reference_lists(golden, barrier):
    g = golden["test1_fast"]
    xy = O.fast10_detect(g["img"], barrier)
    assert xy.shape == g["xy%d" % barrier].shape and (xy == g["xy%d" % barrier]).all()
    sc = O.fast10_score(g["img"], xy)
    assert (sc == g["score%d" % barrier]).all() and sc.min() >= barrier
    keep = O.fast_nonmax(xy, sc)
    assert (keep == g["keep%d" % barrier]).all()
    if barrier == 20:
        assert len(xy) == 3787 and len(keep) == 843      # SURVEY App. C probe 2


@pytest.mark.skipif(not O.have_ref(), reason="oracle/_ref/libfast_ref.so needs the reference sources at BASELINE.json's reference_path (or DSDTM_REFERENCE)")
def test_fast_closed_form_equals_reference_library_on_adversarial_images():
    rng = np.random.default_rng(5)
    for t in range(24):
        h, w = int(rng.integers(7, 70)), int(rng.integers(7, 100))
        if t % 3 == 0:
            im = rng.integers(0, 256, (h, w), dtype=np.uint8)
        elif t % 3 == 1:
            im = (rng.integers(0, 2, (h, w)) * 255).astype(np.uint8)          # saturation + plateaus
        else:
            im = np.repeat(np.repeat(rng.integers(0, 256, (h // 3 + 1, w // 3 + 1), dtype=np.uint8), 3, 0), 3, 1)[:h, :w].copy()
        for b in (20, 1, 100):
            a = O.fast10_detect(im, b)
            for sse in (True, False):
                r = O.ref_fast10_detect(im, b, sse)
                assert len(a) == len(r) and (a == r).all(), (h, w, b, sse)
            if len(a):
                s = O.fast10_score(im, a)
                assert (s == O.ref_fast10_score(im, a, b)).all()
                assert (O.fast_nonmax(a, s) == O.ref_fast_nonmax(a, s)).all()


def test_circle_fill_matches_cv2_goldens(golden):
    g = golden["circle_cv2"]
    H, W = g["shape"]
    for (cx, cy, r), bits in zip(g["cases"], g["masks"]):
        m = np.full((H, W), 255, np.uint8)
        O.circle_fill(m, cx, cy, r, 0)
        want = np.unpackbits(bits)[:H * W].reshape(H, W).astype(bool)
        assert ((m == 0) == want).all(), (cx, cy, r)


def test_cvround_is_half_to_even():
    assert [O.cvround(v) for v in (0.5, 1.5, 2.5, -0.5, -1.5, 2.4999, 2.5001)] == [0, 2, 2, 0, -2, 2, 3]


def test_shitomasi_border_and_symmetry():
    rng = np.random.default_rng(2)
    im = rng.integers(0, 256, (40, 50), dtype=np.uint8)
    assert O.shitomasi(im, 4, 20) == 0.0 and O.shitomasi(im, 45, 20) == 0.0      # x_min < 1 / x_max >= cols-1
    assert O.shitomasi(im, 5, 5) > 0.0
    assert O.shitomasi(np.full((40, 50), 9, np.uint8), 20, 20) == 0.0


def test_detect_selection_respects_mask_and_limit(scenario):
    packed, offs, ws, hs = scenario["ref_pyr"]
    cells = O.detect_cells(packed, offs, ws, hs, 15, None, 5.0)
    mask = np.full((480, 640), 255, np.uint8)
    feats, sorted_cells = O.detect_select(cells, mask, 15, 300)
    assert len(feats) == 300 and (np.diff(sorted_cells["score"]) <= 0).all()
    assert (feats["score"] > 20).all()
    # every selected feature is > CellSize away (cv::circle disc) from every earlier one
    for i in range(1, 40):
        d2 = (feats["x"][:i] - feats["x"][i]) ** 2 + (feats["y"][:i] - feats["y"][i]) ** 2
        assert d2.min() > 15 * 15 - 30
    # occupied cells are skipped (ref: src/Feature_detection.cpp:100)
    occ = np.zeros(len(cells), np.uint8); occ[::2] = 1
    c2 = O.detect_cells(packed, offs, ws, hs, 15, occ, 5.0)
    assert (c2["score"][::2] == np.float32(5.0)).all() and (c2[1::2] == cells[1::2]).all()


def test_sparse_align_converges_to_ground_truth(scenario):
    import helpers as H
    from dsdtm_b200 import synth as S
    packed, offs, ws, hs = scenario["ref_pyr"]
    for (ml, it) in ((4, 30), (5, 8)):
        pose, n, log = O.sparse_align(H.ocam(scenario["cam"]), packed, scenario["cur_pyr"][0], offs, ws, hs, scenario["feats"],
                                      scenario["ref_center"], S.IDENTITY, ml, 0, it)
        e0 = S.pose_dist(S.IDENTITY, scenario["T_c2r"])
        e1 = S.pose_dist(pose, scenario["T_c2r"])
        assert e1[0] < 0.02 * e0[0] and e1[1] < 0.02 * e0[1] and n > 250
        assert log[0]["level"] == ml - 1 and log[-1]["level"] == 0
        # Q6/revert rule: a reverted iteration is always the last one of its level
        for a, b in zip(log[:-1], log[1:]):
            if a["flags"] & 2:
                assert b["level"] == a["level"] - 1 and b["iter"] == 0


def test_sparse_align_no_visible_feature_gives_nan_chi2_and_keeps_pose(scenario):
    import helpers as H
    from dsdtm_b200 import synth as S
    packed, offs, ws, hs = scenario["ref_pyr"]
    far = S.pose_from_xi([50.0, 0, 0, 0, 0, 0])     # everything projects outside the image
    pose, n, log = O.sparse_align(H.ocam(scenario["cam"]), packed, scenario["cur_pyr"][0], offs, ws, hs, scenario["feats"],
                                  scenario["ref_center"], far, 2, 0, 5)
    assert n == 0 and np.isnan(log[0]["chi2"]) and np.allclose(pose, far)


def test_align2d_recovers_subpixel_truth(scenario):
    """test_Feature_alignment recipe (ref: Test/test_Feature_alignment.cpp:56-81): truth (130.2,120.3), offset (1.1,0.8)."""
    import helpers as H
    packed, offs, ws, hs = scenario["cur_pyr"]
    img = O.pyr_level(packed, offs, ws, hs, 0)
    levels, patches, truth, start = H.make_patches(scenario["cur_pyr"], 50, 11, max_level=0, pert=1.2)
    errs = []
    for i in range(50):
        p, conv, nit = O.align2d(img, patches[i], 10, start[i])
        if conv:
            errs.append(np.linalg.norm(p - truth[i]))
    assert len(errs) >= 45 and np.median(errs) < 0.05


def test_warp_affine_integer_division_quirk(scenario):
    """Q3: for search level >= 1 the sampling grid collapses to the reference pixel -> constant patch."""
    packed, offs, ws, hs = scenario["ref_pyr"]
    img = O.pyr_level(packed, offs, ws, hs, 0)
    p0 = O.warp_affine(np.eye(2), img, (100.0, 90.0), 0, 0)
    assert (p0.reshape(10, 10) == img[85:95, 95:105]).all()          # identity warp, integer position: x,y in [-5,4]
    p1 = O.warp_affine(np.eye(2) * 2.0, img, (100.0, 90.0), 0, 1)
    assert (p1 == img[90, 100]).all()


def test_se3_group_axioms():
    from dsdtm_b200 import synth as S
    rng = np.random.default_rng(0)
    for _ in range(5):
        x = rng.uniform(-0.3, 0.3, 6)
        a = O.se3_exp(x)
        assert np.allclose(a, S.pose_from_xi(x), atol=1e-12)
        assert np.allclose(O.se3_mul(a, O.se3_inv(a)), S.IDENTITY, atol=1e-12)
        p = rng.uniform(-1, 1, 3)
        assert np.allclose(O.se3_act(a, p), S.pose_act(a, p), atol=1e-12)


def test_undistort_points_matches_cv2_golden(golden):
    """SURVEY 8f-3: the restatement of cv::undistortPoints as called by Frame::UndistortFeatures (ref: src/Frame.cpp:121-122)
    against cv2 4.13 on the reference's own distortion sets (tests/golden/make_golden_ingest.py)."""
    g = golden["undistort_cv2"]
    for name in ("euroc", "default", "zero", "strong"):
        K, D, src, dst = g[name + "_K"], g[name + "_D"], g[name + "_src"], g[name + "_dst"]
        w, h = (int(v) for v in g[name + "_wh"])
        cam = O.make_cam(w, h, float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2]), float(K[0, 0]))
        got = O.undistort_points(cam, D, src)
        bad = int((got.view(np.uint32) != dst.view(np.uint32)).sum())
        assert bad == 0, (name, bad, np.abs(got - dst).max())
    z = g["zero_src"]
    assert np.abs(g["zero_dst"] - z).max() < 1e-4        # zero distortion: identity up to the float round trip


def test_depth_lookup_and_convert_restatements():
    """ref: src/Tracking.cpp:56 (convertTo CV_32F, 1/scale) and src/Frame.cpp:200-224 (Get_FeatureDetph)."""
    rng = np.random.default_rng(5)
    d16 = rng.integers(0, 65536, (48, 64)).astype(np.uint16)
    for scale in (5000.0, 1000.0, 1.0):
        want = d16.astype(np.float32) * np.float32(np.float32(1.0) / np.float32(scale))
        assert (O.depth_convert(d16, scale) == want).all()
    d = np.zeros((10, 12), np.float32)
    d[5, 4] = 2.5            # left neighbour of (5,5) in image coords is (x=4,y=5)
    d[4, 5] = 3.5            # upper neighbour
    assert O.feature_depth(d, (5.2, 4.6)) == 2.5     # cvRound -> (5,5); centre 0 -> (-1,0) first
    d[5, 4] = 0
    assert O.feature_depth(d, (5.0, 5.0)) == 3.5     # then (0,-1)
    d[4, 5] = 0
    assert O.feature_depth(d, (5.0, 5.0)) == -1.0
    d[5, 5] = 1.25
    assert O.feature_depth(d, (5.49, 4.51)) == 1.25
    assert O.feature_depth(d, (0.0, 0.0)) == -1.0    # neighbours outside the image count as 0


def test_clahe_matches_cv2_golden(golden):
    """cv::createCLAHE(clip, tiles)->apply (the preprocessing of the reference's test drivers, Test/test_Feature_detection.cpp:85-86)
    against cv2 4.13 on deterministic numpy inputs (tests/golden/make_golden_ingest.py)."""
    import helpers as H
    g = golden["clahe_cv2"]
    for name, h, w, clip, tiles in H.CLAHE_CASES:
        img = H.clahe_input(name, h, w)
        assert (O.clahe(img, clip, tiles) == g[name]).all(), name


def test_se3_exp_matches_the_matrix_exponential_scipy_computes():
    """An anchor outside this repository for the Sophus restatement (SE3::exp, translation-first twist; SE3 * SE3; SE3 * point):
    scipy.linalg.expm of the 4x4 twist matrix and plain matrix products."""
    from scipy.linalg import expm
    from scipy.spatial.transform import Rotation as Rot
    rng = np.random.default_rng(3)

    def mat(p):
        M = np.eye(4)
        M[:3, :3] = Rot.from_quat(np.r_[p[1:4], p[0]]).as_matrix(); M[:3, 3] = p[4:]
        return M
    for scale in (1e-12, 1e-6, 0.3, 2.5):
        for _ in range(4):
            x = rng.uniform(-scale, scale, 6)
            W = np.array([[0, -x[5], x[4]], [x[5], 0, -x[3]], [-x[4], x[3], 0]])
            T = np.zeros((4, 4)); T[:3, :3] = W; T[:3, 3] = x[:3]
            a = O.se3_exp(x)
            assert np.allclose(mat(a), expm(T), atol=1e-12)
            b = O.se3_exp(rng.uniform(-0.5, 0.5, 6))
            assert np.allclose(mat(O.se3_mul(a, b)), mat(a) @ mat(b), atol=1e-12)
            assert np.allclose(mat(O.se3_inv(a)) @ mat(a), np.eye(4), atol=1e-12)
            p = rng.uniform(-2, 2, 3)
            assert np.allclose(O.se3_act(a, p), (mat(a) @ np.r_[p, 1.0])[:3], atol=1e-12)


def test_pose_parameterisation_round_trip_and_plus_against_scipy():
    """PoseLocalParameterization (ref: include/Optimizer.h:220-236) as the oracle's PoseOptimization uses it: with no residual the
    solve hands back exp(log(R)) of the start pose (SO3::log / SO3::exp round trip); one capped iteration moves the pose by a left
    multiplication -- checked through scipy's rotation vectors."""
    from scipy.spatial.transform import Rotation as Rot
    rng = np.random.default_rng(4)
    for _ in range(10):
        w = rng.uniform(-1, 1, 3); w *= rng.uniform(0.0, 3.0) / np.linalg.norm(w)      # rotation angles up to 3 rad
        q = Rot.from_rotvec(w).as_quat()
        pose = np.r_[q[3], q[:3], rng.uniform(-1, 1, 3)]
        out, res, sm = O.pose_optimization(np.zeros((0, 3)), np.zeros(0, np.int32), np.zeros((0, 3)), pose)
        assert sm["termination"] == O.BA_NO_RESIDUALS and len(res) == 0
        same = np.abs(out - pose).max() < 1e-14 or np.abs(out[:4] + pose[:4]).max() < 1e-14      # q and -q are the same rotation
        assert same and np.abs(out[4:] - pose[4:]).max() == 0
