"""Pins oracle/dsdtm_oracle.cpp to the reference's OWN source for the floating-point rows of SURVEY.md 8(a) (a5-a16, f-1, f-3).

oracle/_ref/libdsdtm_ref.so = <reference>/src/{Sprase_ImageAlign,Feature_alignment,Feature_detection,Camera,Frame,MapPoint,
Keyframe,Map,Config}.cpp + Thirdparty/fast, compiled UNMODIFIED (recipe: oracle/Makefile, target ref_dsdtm) against the stand-in
third-party headers of tests/ref_shim. Every test below feeds the reference's classes and the oracle the same inputs.

What "equal" means here:
* everything the reference writes coefficient by coefficient in its own source (patches, Jacobians, H, Jres, chi2, the GN loop's
  control flow, bilinear weights, integer decisions, sort / mask / grid logic) is asserted BIT-EQUAL;
* what happens inside Eigen / Sophus calls (LDLT, SE3::exp, quaternion products, norms) is the stand-in's restatement; the default
  build associates reductions left to right like the oracle, and the `_tree` build (Eigen's fixed-size unroller order) is checked to
  move results only in the last bits -- i.e. the comparison does not hinge on that unpinnable choice.
These tests need the library built from a checkout of the reference (at BASELINE.json's reference_path, or DSDTM_REFERENCE) and skip without it; part of the
values they establish travel as tests/golden/refpin.npz (see test_ref_golden.py)."""
import numpy as np
import pytest

import helpers as H
import oracle as O
from dsdtm_b200 import synth as S
from oracle import refpin as RP
from oracle_seq import CELL, LEVELS, OMap, OracleFrame, _oracle_search_multi, _oracle_sparse_align, _trajectory

RP.build()
pytestmark = pytest.mark.skipif(not RP.available(), reason="oracle/_ref/libdsdtm_ref.so needs the reference sources at %s (or DSDTM_REFERENCE)" % RP.REFERENCE)

CFGS = [(4, 0, 30), (5, 0, 8), (5, 2, 8), (3, 1, 4)]        # BASELINE configs[0] ctor, production ctor, truncated variants


@pytest.fixture(scope="module")
def kin():
    return RP.Ref(dict(S.KINECT), levels=5)


@pytest.fixture(scope="module")
def kin_tree():
    return RP.Ref(dict(S.KINECT), tree=True, levels=5)


def _load_pair(R, sc, pose_cur_start):
    """ref frame with the scenario's features + map points, cur frame at a start pose."""
    R.reset()
    ref = R.frame(sc["ref_img"], sc["T_ref"])
    cur = R.frame(sc["cur_img"], pose_cur_start)
    kf = R.keyframe(ref)
    for f in sc["feats"]:
        k = R.add_feature(ref, f["px"], f["level"], True)          # Frame::Add_Feature computes mNormal (ref: src/Frame.cpp:83-92)
        R.set_mappoint(ref, k, R.mappoint(f["point_w"], kf))
    return ref, cur


# ---------------------------------------------------------------------------------------------- a1, a5, a6
def test_pyramid_and_feature_normals(kin):
    sc = H.make_scenario(3)
    ref, cur = _load_pair(kin, sc, sc["T_ref"])
    packed, offs, ws, hs = sc["ref_pyr"]
    for l in range(5):
        assert (kin.frame_level(ref, l) == O.pyr_level(packed, offs, ws, hs, l)).all()
    f = kin.features(ref)
    assert (f["normal"] == sc["feats"]["normal"]).all()            # float Pixel2Camera widened, then normalize() (Q8)
    assert (f["initial"] == 1).all()


def test_shitomasi_bits(kin):
    rng = np.random.default_rng(5)
    img = S.make_pair(11)["ref_img"]
    pts = np.c_[rng.integers(0, 640, 400), rng.integers(0, 480, 400)]
    pts = np.r_[pts, [[4, 4], [5, 5], [635, 475], [634, 474], [0, 0], [639, 479], [5, 100], [100, 5]]]   # the border rule of ref :171
    for u, v in pts:
        a = np.float32(kin.shitomasi(img, u, v)); b = np.float32(O.shitomasi(img, u, v))
        assert a.view(np.uint32) == b.view(np.uint32), (u, v, a, b)


@pytest.mark.parametrize("camname,seed", [("KINECT", 20260101), ("KINECT", 8), ("EUROC", 100)])
def test_detect_equals_reference(camname, seed):
    cam = dict(getattr(S, camname))
    R = RP.Ref(cam, levels=5)
    pr = S.make_pair(seed, cam)
    fr = R.frame(pr["ref_img"], S.IDENTITY)
    n = R.detect(fr, 5.0, True)
    f = R.features(fr)
    oc, _ = H.detect_oracle(pr["ref_img"], 5, 15, 300)
    assert n == len(oc) and n > 200
    assert (f["px"][:, 0] == oc["x"]).all() and (f["px"][:, 1] == oc["y"]).all() and (f["level"] == oc["level"]).all()
    assert kin_mask_released(R, fr)


def kin_mask_released(R, fr):
    return R.mask(fr) is None                                       # detect ends with mImgMask.release() (ref: :153)


# ---------------------------------------------------------------------------------------------- a7-a10
@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("seed", [20260101, 4])
def test_sparse_align_run_is_bit_equal(kin, cfg, seed):
    sc = H.make_scenario(seed)
    oc = H.ocam(sc["cam"])
    packed, offs, ws, hs = sc["ref_pyr"]
    ref, cur = _load_pair(kin, sc, sc["T_ref"])
    pr, nr = kin.sparse_align_run(cur, ref, *cfg)
    po, no, log = O.sparse_align(oc, packed, sc["cur_pyr"][0], offs, ws, hs, sc["feats"], sc["ref_center"], S.IDENTITY, *cfg)
    assert nr == no and (pr == po).all(), (np.abs(pr - po).max(), nr, no)
    e = S.pose_dist(pr, sc["T_c2r"])
    assert len(log) >= cfg[0] - cfg[1] and (cfg[1] > 0 or (e[0] < 3e-4 and e[1] < 1e-3))   # the truncated variants stop above level 0


def test_sparse_align_run_with_moved_reference_and_start_offsets(kin, kin_tree):
    """Non-identity reference pose (exercises mT_c2r = cur * ref^-1 and Set_Pose(mT_c2r * ref), ref: :43,57), perturbed start poses,
    features without map points / with a zero point / near the border (the visibility rules of ref :83-100)."""
    rng = np.random.default_rng(17)
    T_ref = S.pose_from_xi(np.r_[0.3, -0.2, 0.1, 0.05, -0.04, 0.08])
    for seed in (31, 32):
        pr = S.make_pair(seed, S.KINECT, ref_pose=T_ref)
        corners, pyr = H.detect_oracle(pr["ref_img"], 5, 15, 300)
        feats = H.ref_feats_from_corners(S.KINECT, corners, pr["ref_points"])
        feats["initial"][::17] = 0                                  # features that never got a map point
        feats["point_w"][5] = 0.0                                   # isZero(0) rule
        center = O.se3_inv(pr["T_ref"])[4:]
        start = O.se3_mul(S.pose_from_xi(rng.uniform(-0.004, 0.004, 6)), pr["T_ref"])
        for R in (kin, kin_tree):
            R.reset()
            ref = R.frame(pr["ref_img"], pr["T_ref"]); cur = R.frame(pr["cur_img"], start)
            kf = R.keyframe(ref)
            for f in feats:
                k = R.add_feature(ref, f["px"], f["level"], True)
                if f["initial"]:
                    R.set_mappoint(ref, k, R.mappoint(f["point_w"], kf))
            p_ref, c_ref = R.frame_pose(ref)
            assert (c_ref == center).all()                          # Frame::Set_Pose -> mOw (ref: src/Frame.cpp:167-174)
            pr_out, nr = R.sparse_align_run(cur, ref, 5, 0, 8)
            T0 = O.se3_mul(start, O.se3_inv(pr["T_ref"]))
            po, no, log = O.sparse_align(H.ocam(S.KINECT), pyr[0], O.pyramid(pr["cur_img"], 5)[0], pyr[1], pyr[2], pyr[3], feats, center, T0, 5, 0, 8)
            want = O.se3_mul(po, pr["T_ref"])
            if R is kin:
                assert nr == no and (pr_out == want).all(), np.abs(pr_out - want).max()
            else:   # Eigen's unroller order inside norm()/dot(): last bits only
                assert nr == no and np.abs(pr_out - want).max() < 1e-12
            d = S.pose_dist(pr_out, pr["T_cur"])
            assert d[0] < 3e-4 and d[1] < 1e-3


def test_sparse_align_refined_positions_and_extreme_bytes_are_bit_equal(kin):
    """The inputs of tests/test_gpu_align.py::test_sparse_align_subnormal_byte_encoding_keeps_full_precision, against the REFERENCE: features at
    refined (arbitrary float) positions -- the case inside Tracking, where the last frame's features come out of Align2D -- on images of
    saturated 0 / 255 blocks, from a start pose with arbitrary fractions. The bilinear weights are then general doubles at every level."""
    sc = H.make_scenario(11, trans=0.015, rot_deg=0.4)
    rng = np.random.default_rng(5)
    hard = {}
    for k in ("ref_img", "cur_img"):
        img = sc[k].copy()
        img[(img > 150)] = 255
        img[(img < 90)] = 0
        hard[k] = img
    feats = sc["feats"].copy()
    feats["px"] = (feats["px"] + rng.uniform(0.0, 1.0, feats["px"].shape)).astype(np.float32)
    oc = H.ocam(sc["cam"])
    for f in feats:
        f["normal"] = O.feature_normal(oc, f["px"])                  # what Frame::Add_Feature derives from the pixel (ref: src/Frame.cpp:83-92)
    start_c2r = S.pose_from_xi(rng.uniform(-0.003, 0.003, 6))
    start = O.se3_mul(start_c2r, sc["T_ref"])
    kin.reset()
    ref = kin.frame(hard["ref_img"], sc["T_ref"]); cur = kin.frame(hard["cur_img"], start)
    kf = kin.keyframe(ref)
    for f in feats:
        k = kin.add_feature(ref, f["px"], f["level"], True)
        kin.set_mappoint(ref, k, kin.mappoint(f["point_w"], kf))
    pr, nr = kin.sparse_align_run(cur, ref, 4, 0, 30)
    ref_pyr = O.pyramid(hard["ref_img"], 5); cur_pyr = O.pyramid(hard["cur_img"], 5)
    T0 = O.se3_mul(start, O.se3_inv(sc["T_ref"]))
    po, no, log = O.sparse_align(oc, ref_pyr[0], cur_pyr[0], ref_pyr[1], ref_pyr[2], ref_pyr[3], feats, sc["ref_center"], T0, 4, 0, 30)
    want = O.se3_mul(po, sc["T_ref"])
    assert nr == no and (pr == want).all(), (np.abs(pr - want).max(), nr, no)
    assert len(log) >= 8


def test_sparse_align_too_few_features_returns_zero(kin):
    sc = H.make_scenario(3, max_fts=40)                             # Camera.Min_fts = 50 (ref: src/Sprase_ImageAlign.cpp:34-38)
    ref, cur = _load_pair(kin, sc, sc["T_ref"])
    before, _ = kin.frame_pose(cur)
    p, n = kin.sparse_align_run(cur, ref, 5, 0, 8)
    assert n == 0 and (p == before).all()


@pytest.mark.parametrize("level", [0, 2, 4])
def test_linearization_matches_first_oracle_iteration(kin, level):
    """GetJocabianMat + one ComputeResiduals of the reference at the start pose, against the oracle's first logged iteration of the
    same level: chi2 bit-equal, and x = ldlt(H) b bit-equal when the reference's H, b go through the oracle's LDLT."""
    sc = H.make_scenario(12)
    oc = H.ocam(sc["cam"])
    packed, offs, ws, hs = sc["ref_pyr"]
    ref, cur = _load_pair(kin, sc, sc["T_ref"])
    T0 = S.pose_from_xi([0.002, -0.001, 0.003, 0.001, -0.002, 0.0015])
    lin = kin.sparse_align_linearize(cur, ref, level, T0)
    po, no, log = O.sparse_align(oc, packed, sc["cur_pyr"][0], offs, ws, hs, sc["feats"], sc["ref_center"], T0, level + 1, level, 1)
    assert len(log) == 1 and log[0]["level"] == level
    assert lin["n_pts"] == log[0]["n_pts"] == no
    assert lin["chi2"] == log[0]["chi2"]
    assert (O.ldlt6_solve(lin["H"], lin["b"]) == log[0]["x"]).all()
    assert np.allclose(lin["H"], lin["H"].T, rtol=0, atol=0)        # J J^T accumulated entry by entry: exactly symmetric
    # the staged quantities have the documented shapes / values: 16 bilinear samples per feature inside [0, 255]
    assert lin["patch"].shape == (lin["n"], 16) and lin["patch"].min() >= 0 and lin["patch"].max() <= 255
    assert lin["jac"].shape == (lin["n"] * 16, 6)


# ---------------------------------------------------------------------------------------------- a14-a16
def test_align2d_bits(kin):
    sc = H.make_scenario(6)
    levels, patches, truth, start = H.make_patches(sc["cur_pyr"], 300, 3, max_level=2)
    packed, offs, ws, hs = sc["cur_pyr"]
    n_conv = 0
    for iters in (3, 10):
        for i in range(300):
            img = O.pyr_level(packed, offs, ws, hs, int(levels[i]))
            p8 = O.patch_no_border(patches[i])
            pr, cr = kin.align2d(img, patches[i], p8, iters, start[i])
            po, co, _ = O.align2d(img, patches[i], iters, start[i])
            assert cr == co and (pr == po).all(), (i, iters, pr, po)
            n_conv += cr
    assert n_conv > 400
    # the recipe of ref Test/test_Feature_alignment.cpp:56-81: offset (+1.1, +0.8), 3 iterations
    img = O.pyr_level(packed, offs, ws, hs, 0)
    lv, pt, tr, _ = H.make_patches(sc["cur_pyr"], 1, 9, max_level=0)
    pr, cr = kin.align2d(img, pt[0], O.patch_no_border(pt[0]), 3, tr[0] + (1.1, 0.8))
    po, co, _ = O.align2d(img, pt[0], 3, tr[0] + (1.1, 0.8))
    assert (pr == po).all() and cr == co and np.abs(pr - tr[0]).max() < 0.1


def test_align2d_edge_rules(kin):
    """Q4: `>` in the bounds test lets u_r == cols-4 through (reads one column past the edge); NaN start; constant patch
    (singular H -> inf/NaN update -> not converged)."""
    sc = H.make_scenario(6)
    packed, offs, ws, hs = sc["cur_pyr"]
    img = O.pyr_level(packed, offs, ws, hs, 1)
    h, w = img.shape
    _, pt, _, _ = H.make_patches(sc["cur_pyr"], 1, 4, max_level=0)
    flat = np.full(100, 77, np.uint8)
    for patch, px in [(pt[0], (3.9, 50.0)), (pt[0], (50.0, 3.2)), (pt[0], (w - 3.5, 60.0)), (pt[0], (w - 4.0 + 0.25, 60.0)),
                      (pt[0], (60.0, h - 4.0 + 0.5)), (pt[0], (np.nan, 50.0)), (flat, (80.0, 60.0)), (pt[0], (w - 4.5, h - 4.5))]:
        if px[0] == px[0] and (int(np.floor(px[0])) == w - 4 or int(np.floor(px[1])) == h - 4):
            continue   # the 1-past-the-edge read is memory the reference does not own: defined only for the oracle / kernel (zeros)
        pr, cr = kin.align2d(img, patch, O.patch_no_border(patch), 10, px)
        po, co, _ = O.align2d(img, patch, 10, px)
        assert cr == co and ((pr == po) | ((pr != pr) & (po != po))).all(), (px, pr, po)


def test_warp_affine_and_search_level_bits(kin):
    rng = np.random.default_rng(8)
    sc = H.make_scenario(6)
    packed, offs, ws, hs = sc["ref_pyr"]
    for t in range(200):
        L0 = int(rng.integers(0, 3))
        img = O.pyr_level(packed, offs, ws, hs, L0)
        h, w = img.shape
        A = np.eye(2) * rng.uniform(0.6, 3.2) + rng.normal(0, 0.2, (2, 2))
        px = np.array([rng.uniform(0, w - 1), rng.uniform(0, h - 1)], np.float32) * np.float32(1 << L0)
        if t % 9 == 0:
            px = np.array([rng.uniform(0, 3) * (1 << L0), rng.uniform(0, h - 1) * (1 << L0)], np.float32)       # patch leaves the image: zeros
        SL = kin.best_search_level(A, 2)
        assert SL == O.best_search_level(A, 2)
        for sl in {SL, 0, 1}:                                       # Q3: integer 1/(1<<L) == 0 for L >= 1 -> constant patch
            a = kin.warp_affine(A, img, px, L0, sl); b = O.warp_affine(A, img, px, L0, sl)
            assert (a == b).all(), (t, sl)
            if sl >= 1:
                assert len(set(a.tolist())) == 1


def test_solve_affine_find_match_and_closest_obs(kin):
    """SolveAffineMatrix / FindMatchDirect / Get_ClosetObs on a two-key-frame map (ref: src/Feature_alignment.cpp:128-190,
    src/MapPoint.cpp:133-174)."""
    cam = dict(S.KINECT)
    oc = H.ocam(cam)
    scene = S.Scene(91)
    poses = _trajectory(6, seed=9)
    poses[3] = S.pose_mul(S.pose_from_xi([0.25, 0.02, 0.0, 0.0, 0.12, 0.0]), poses[3])      # a second key frame seen from the side
    kin.reset()
    kfs, frames, of = [], [], []
    for k in (0, 3):
        img, _, pts = S.render(scene, cam, poses[k], want_points=True)
        fr = kin.frame(img, poses[k])
        corners, _ = H.detect_oracle(img, 5, 15, 200)
        F = H.ref_feats_from_corners(cam, corners, pts)
        for f in F:
            kin.add_feature(fr, f["px"], f["level"], True)
        kfs.append(kin.keyframe(fr)); frames.append(fr)
        o = OracleFrame(img, poses[k]); o.feats = F; of.append(o)
    # map points of key frame 0, observed by key frame 0 and (nominally) by feature i of key frame 1
    mps = []
    for i, f in enumerate(of[0].feats):
        mp = kin.mappoint(f["point_w"], kfs[0])
        kin.add_observation(mp, kfs[0], i); kin.kf_feature_set_mappoint(kfs[0], i, mp)
        if i < len(of[1].feats):
            kin.add_observation(mp, kfs[1], i)
        mps.append(mp)
    for i, f in enumerate(of[1].feats):                             # the features of key frame 1 need a map point of their own for :167
        mp = kin.mappoint(f["point_w"], kfs[1]); kin.kf_feature_set_mappoint(kfs[1], i, mp)
    chosen = set()
    n_ok = 0
    # two current frames: one next to key frame 0, one next to the sideways key frame 1
    for pose_cur in (poses[5], S.pose_mul(S.pose_from_xi([0.01, 0.0, 0.0, 0.0, 0.004, 0.0]), poses[3])):
        imgc, _ = S.render(scene, cam, pose_cur)
        cur = kin.frame(imgc, pose_cur)
        ocur = OracleFrame(imgc, pose_cur)
        cur_center = O.se3_inv(pose_cur)[4:]
        for i, mp in enumerate(mps):
            P = of[0].feats[i]["point_w"]
            centers = [O.se3_inv(of[0].pose)[4:]] + ([O.se3_inv(of[1].pose)[4:]] if i < len(of[1].feats) else [])
            ok_o, best = O.closest_obs(cur_center, P, np.array(centers))
            ok_r, kf_r, fi_r = kin.closest_obs(mp, cur)
            # std::map<KeyFrame*, size_t> iterates in ADDRESS order; the cosines differ, so the winner does not depend on it
            assert ok_r == ok_o and kf_r == kfs[best] and fi_r == i
            chosen.add(best)
            kf = of[best]; f = kf.feats[i]
            T_c2r = O.se3_mul(pose_cur, O.se3_inv(kf.pose))
            A_o = O.solve_affine(oc, O.se3_inv(kf.pose)[4:], f["point_w"], f["normal"], f["px"], int(f["level"]), T_c2r)
            A_r = kin.solve_affine(kfs[best], cur, i, mp)
            assert (A_r == A_o).all(), (i, A_r - A_o)
            # FindMatchDirect from the reprojected position
            px0 = kin.world2pixel(cur, P)
            ok, pxo, cell = O.reproject_point(oc, pose_cur, P, 15, 43)
            assert (px0 == pxo).all()
            okr, pr, lr = kin.find_match_direct(mp, cur, px0)
            # oracle chain
            L0 = int(f["level"])
            rpx = f["px"] / np.float32(1 << L0)
            inimg = O.is_in_image(oc, rpx[0], rpx[1], 5, L0)
            if not ok_o or not inimg:
                assert not okr
                continue
            SL = O.best_search_level(A_o, LEVELS - 3)
            packed, offs, ws, hs = kf.pyr
            patch = O.warp_affine(A_o, O.pyr_level(packed, offs, ws, hs, L0), f["px"], L0, SL)
            p, conv, _ = O.align2d(O.pyr_level(ocur.pyr[0], offs, ws, hs, SL), patch, 10, px0 / (1 << SL))
            q = p * (1 << SL)
            assert okr == conv and lr == SL and ((pr == q) | ((pr != pr) & (q != q))).all(), (i, pr, p)   # Q3: search level >= 1 ends in NaN on both sides
            n_ok += conv
    assert chosen == {0, 1} and n_ok > 100


def test_is_in_image_and_nan(kin):
    """Camera::IsInImage (ref: src/Camera.cpp:187-193): cvRound of the float pixel; NaN rounds to INT_MIN and fails the test."""
    oc = H.ocam(S.KINECT)
    rng = np.random.default_rng(3)
    for _ in range(2000):
        x, y = rng.uniform(-20, 660), rng.uniform(-20, 500)
        b, l = int(rng.integers(0, 9)), int(rng.integers(0, 3))
        assert kin.is_in_image(x, y, b, l) == O.is_in_image(oc, x, y, b, l)
    for x, y in [(0.5, 0.5), (1.5, 2.5), (639.5, 10), (638.5, 10), (7.5, 8.5), (8.5, 7.5), (631.5, 471.5), (np.nan, 5.0), (5.0, np.nan), (np.inf, 5.0), (-np.inf, 5.0), (3e9, 5)]:
        for b in (0, 1, 8):
            assert kin.is_in_image(x, y, b, 0) == O.is_in_image(oc, x, y, b, 0), (x, y, b)
    assert not kin.is_in_image(np.nan, np.nan, 0, 0)


# ---------------------------------------------------------------------------------------------- f-3
def test_keyframe_ingest_helpers():
    """Frame::UndistortFeatures / Get_FeatureDetph / UnProject / isVisible / World2Pixel (ref: src/Frame.cpp:94-157,200-224,300-323)."""
    cam = dict(S.EUROC)
    dist = (-0.28340811, 0.07395907, 0.00019359, 1.76187114e-05, 0.0)      # ref: Config/EuRoc.yaml:15-19
    R = RP.Ref(cam, levels=5, dist=dist)
    oc = H.ocam(cam)
    pr = S.make_pair(41, cam)
    depth = pr["ref_depth"].astype(np.float32)
    depth[::7, ::5] = 0.0                                           # holes: the 4-neighbourhood fallback
    pose = S.pose_from_xi([0.2, -0.1, 0.05, 0.03, -0.02, 0.04])
    fr = R.frame(pr["ref_img"], pose, depth=depth)
    rng = np.random.default_rng(1)
    px = np.c_[rng.uniform(2, 749, 300), rng.uniform(2, 477, 300)].astype(np.float32)
    px[:40] = np.floor(px[:40]) + np.float32(0.5)                   # ties of cvRound (round half to even)
    for p in px:
        R.add_feature(fr, p, 0, False)
    R.undistort_features(fr)
    f = R.features(fr)
    und = O.undistort_points(oc, dist, px)
    assert (f["px"] == und).all()
    for i in range(300):
        assert (f["normal"][i] == O.feature_normal(oc, und[i])).all()
        d = R.feature_depth(fr, px[i])
        assert d == O.feature_depth(depth, px[i])
        if d > 0:
            assert (R.unproject(fr, px[i], d) == O.unproject(oc, pose, px[i], d)).all()
    pts = rng.normal(0, 2.0, (500, 3)) + (0, 0, 2.0)
    for P in pts:
        q = O.se3_act(pose, P)
        okr = R.is_visible(fr, P, 0)
        if q[2] < 0.0:
            assert not okr
            continue
        ok, pxo, _ = O.reproject_point(oc, pose, P, 15, 51)
        assert (R.world2pixel(fr, P) == pxo).all()
        assert okr == O.is_in_image(oc, np.float32(pxo[0]), np.float32(pxo[1]), 0, 0)


# ---------------------------------------------------------------------------------------------- the SE3 stand-in vs the oracle's
def test_se3_standin_agrees_with_oracle(kin, kin_tree):
    rng = np.random.default_rng(0)
    for t in range(300):
        x = rng.normal(0, 1, 6) * (10.0 ** rng.uniform(-12, 0))
        if t % 20 == 0:
            x[3:] = 0
        a = O.se3_exp(x)
        assert (kin.se3_exp(x) == a).all()
        assert np.abs(kin_tree.se3_exp(x) - a).max() < 1e-15
        b = O.se3_exp(rng.normal(0, 0.3, 6))
        assert (kin.se3_mul(a, b) == O.se3_mul(a, b)).all() and (kin.se3_inv(a) == O.se3_inv(a)).all()


# ---------------------------------------------------------------------------------------------- the whole front-end loop
def test_sequence_against_reference_classes(kin):
    """BASELINE configs[3] at test scale through the reference's OWN classes: Frame ctor (pyramid), Sprase_ImgAlign::Run against the
    last frame, Feature_Alignment::ResetGrid / ReprojectPoint / SearchLocalPoints over a growing key-frame map (with
    MapPoint::Get_ClosetObs, IncreaseFound, the cv::circle mask), and Tracking::CraeteKeyframe's Set_ExistingFeatures + detect on a frame
    that carries matches -- against the oracle-side model that the GPU sequence tests compare the CUDA path with
    (tests/oracle_seq.py). Everything is bit-equal: poses, match order, refined pixels, levels, found counters, new corners."""
    cam = dict(S.KINECT)
    oc = H.ocam(cam)
    scene = S.Scene(91)
    n_frames, kf_at = 9, 4
    poses = _trajectory(n_frames, seed=9)
    cfg = (5, 0, 8)
    R = kin
    R.reset()
    omap = OMap()

    img0, _, pts0 = S.render(scene, cam, poses[0], want_points=True)
    r0 = R.frame(img0, poses[0]); o0 = OracleFrame(img0, poses[0])
    assert R.detect(r0, 5.0, True) == 300
    corners, _ = H.detect_oracle(img0, LEVELS, CELL, 300)
    f0 = R.features(r0)
    assert (f0["px"][:, 0] == corners["x"]).all() and (f0["px"][:, 1] == corners["y"]).all()
    R.undistort_features(r0)                                        # zero distortion: normals from the (unchanged) pixels (ref: src/Initializer.cpp:46)
    o0.feats = H.ref_feats_from_corners(cam, corners, pts0)
    f0 = R.features(r0)
    assert (f0["px"] == o0.feats["px"]).all() and (f0["normal"] == o0.feats["normal"]).all()
    rkf = [R.keyframe(r0)]
    o0.feat_mp = [omap.new_mp(o0.feats[i]["point_w"]) for i in range(len(corners))]
    rmp = {}
    for i, mp in enumerate(o0.feat_mp):
        omap.mp_obs[mp].append((0, i))
        rmp[mp] = R.mappoint(o0.feats[i]["point_w"], rkf[0])
        R.set_mappoint(r0, i, rmp[mp]); R.add_observation(rmp[mp], rkf[0], i); R.increase_found(rmp[mp], 1)
    omap.kfs.append(o0)
    inv_rmp = {v: k for k, v in rmp.items()}

    r_last, o_last = r0, o0
    n_matches = []
    for k in range(1, n_frames):
        img, _, pts = S.render(scene, cam, poses[k], want_points=True)
        r_cur = R.frame(img, R.frame_pose(r_last)[0]); o_cur = OracleFrame(img, o_last.pose)
        pose_r, n_r = R.sparse_align_run(r_cur, r_last, *cfg)
        pose_o, n_o = _oracle_sparse_align(oc, o_cur, o_last, cfg)
        o_cur.pose = pose_o
        assert n_r == n_o and (pose_r == pose_o).all(), (k, np.abs(pose_r - pose_o).max())
        # TrackWithLocalMap -> UpdateLocalMap: every map point of every local key frame once (ref: src/Tracking.cpp:283-303)
        R.reset_grid()
        seen = set()
        for q in range(len(omap.kfs)):
            for mp in omap.kfs[q].feat_mp:
                if mp >= 0 and mp not in seen:
                    seen.add(mp); R.reproject_point(r_cur, rmp[mp])
        R.search_local_points(r_cur)
        want = _oracle_search_multi(oc, cam, o_cur, omap, list(range(len(omap.kfs))))
        f = R.features(r_cur)
        ids = [inv_rmp[m] for m in R.frame_mappoints(r_cur)]
        assert len(want) == len(f["px"]) == len(ids) and len(want) > 100, (k, len(want), len(f["px"]))
        for (mp, p, SL, _), gp, gl, gid in zip(want, f["px"], f["level"], ids):
            assert gid == mp and gl == SL and (p == gp).all(), (k, mp, p, gp)
        n_matches.append(len(want))
        F = np.zeros(len(want), O.REF_FEAT_DT)
        for j, (mp, p, SL, _) in enumerate(want):
            omap.mp_found[mp] += 1
            assert R.found(rmp[mp]) == omap.mp_found[mp]
            F[j]["px"] = p; F[j]["level"] = SL; F[j]["initial"] = 1
            F[j]["normal"] = O.feature_normal(oc, p); F[j]["point_w"] = omap.mp_point[mp]
        assert (f["normal"] == F["normal"]).all()                   # Feature ctor + Add_Feature(tbNormal = true) (ref: src/Feature_alignment.cpp:108-113)
        o_cur.feats = F
        o_cur.feat_mp = [w_[0] for w_ in want]
        if k >= kf_at + 1:
            assert len({w_[3] for w_ in want}) == 2

        if k == kf_at:
            n_old = len(want)
            R.set_existing_from_frame(r_cur)
            n_all = R.detect(r_cur, 5.0, True)
            f2 = R.features(r_cur)
            packed, offs, ws, hs = o_cur.pyr
            rows_, cols_ = O.grid_dims(cam["width"], cam["height"], CELL)
            occ = np.zeros(rows_ * cols_, np.uint8)
            for p in F["px"]:
                occ[int(p[1] / np.float32(CELL)) * cols_ + int(p[0] / np.float32(CELL))] = 1
            cells = O.detect_cells(packed, offs, ws, hs, CELL, occ, 5.0)
            # SearchLocalPoints has already painted CellSize circles; Set_Mask adds Min_dist circles at features with map points
            mask = np.full((cam["height"], cam["width"]), 255, np.uint8)
            for p in F["px"]:
                O.circle_fill(mask, O.cvround(p[0]), O.cvround(p[1]), CELL, 0)
            for p in F["px"]:
                O.circle_fill(mask, O.cvround(p[0]), O.cvround(p[1]), 15, 0)
            new_c, _ = O.detect_select(cells, mask, CELL, 300, n_existing=n_old)
            assert n_all == n_old + len(new_c) and n_all > n_old
            assert (f2["px"][n_old:, 0] == new_c["x"]).all() and (f2["px"][n_old:, 1] == new_c["y"]).all() and (f2["level"][n_old:] == new_c["level"]).all()
            R.undistort_features(r_cur)                             # normals of the new features (ref: src/Tracking.cpp:417)
            Fn = H.ref_feats_from_corners(cam, new_c, pts)
            f3 = R.features(r_cur)
            assert (f3["normal"][n_old:] == Fn["normal"]).all() and (f3["px"][:n_old] == F["px"]).all()
            o_cur.feats = np.concatenate([o_cur.feats, Fn])
            new_ids = [omap.new_mp(Fn[i]["point_w"]) for i in range(len(new_c))]
            o_cur.feat_mp = o_cur.feat_mp + new_ids
            kfi = len(omap.kfs)
            rkf.append(R.keyframe(r_cur))
            for i, mp in enumerate(o_cur.feat_mp):
                omap.mp_obs[mp].append((kfi, i))
                if mp not in rmp:
                    rmp[mp] = R.mappoint(omap.mp_point[mp], rkf[kfi]); inv_rmp[rmp[mp]] = mp
                    R.set_mappoint(r_cur, i, rmp[mp]); R.increase_found(rmp[mp], 1)
                R.add_observation(rmp[mp], rkf[kfi], i)
            omap.kfs.append(o_cur)
        r_last, o_last = r_cur, o_cur
    assert min(n_matches) > 100


# ---------------------------------------------------------------------------------------------- f-1, the caller's half
def test_update_local_map_against_reference_tracking(kin):
    """Tracking::GetCloseKeyFrames + Tracking::UpdateLocalMap of the reference (src/Tracking.cpp:257-345, compiled unmodified; the
    private members are reached by lifting access control in the wrapper's translation unit only) on a 14-key-frame map: visible
    flags, distances (bit-equal), the ten nearest in order, then SearchLocalPoints on the grid UpdateLocalMap filled -- against
    orc_close_keyframes and the oracle-side search model with the same key-frame order."""
    cam = dict(S.KINECT)
    oc = H.ocam(cam)
    scene = S.Scene(91)
    R = kin
    R.reset()
    R.tracking_create()
    rng = np.random.default_rng(4)
    omap = OMap()
    n_kf = 14
    kf_poses = []
    for k in range(n_kf):
        xi = np.r_[rng.uniform(-0.5, 0.5), rng.uniform(-0.3, 0.3), rng.uniform(-0.1, 0.1), np.deg2rad(rng.uniform(-6, 6, 3))]
        if k in (5, 9):
            xi[:3] += (4.0, 3.0, 0.0)                               # far away: sees another part of the scene
        kf_poses.append(S.pose_from_xi(xi))
    rkf, rmp = [], {}
    pt_begin, pt_count, kf_t, pts_all = [], [], [], []
    for k, pose in enumerate(kf_poses):
        img, _, pts = S.render(scene, cam, pose, want_points=True)
        fr = R.frame(img, pose)
        o = OracleFrame(img, pose)
        corners, _ = H.detect_oracle(img, LEVELS, CELL, 80)
        o.feats = H.ref_feats_from_corners(cam, corners, pts)
        for f in o.feats:
            R.add_feature(fr, f["px"], f["level"], True)
        rkf.append(R.keyframe(fr))
        o.feat_mp = []
        rows = []
        for i, f in enumerate(o.feats):
            if i % 13 == 5:                                         # a feature without a map point: NULL in KeyFrame::mvMapPoints
                o.feat_mp.append(-1); rows.append(np.zeros(3)); continue
            P = np.zeros(3) if i % 29 == 7 else f["point_w"]        # a map point at the origin: the isZero(0) rule
            mp = omap.new_mp(P)
            omap.mp_obs[mp].append((k, i))
            omap.mp_found[mp] = 1 + (i * 7 + k) % 4                 # uneven found counters: the per-cell sort matters
            rmp[mp] = R.mappoint(P, rkf[k])
            R.kf_feature_set_mappoint(rkf[k], i, rmp[mp]); R.keyframe_add_mappoint(rkf[k], i, rmp[mp]); R.add_observation(rmp[mp], rkf[k], i)
            R.increase_found(rmp[mp], omap.mp_found[mp])
            o.feat_mp.append(mp); rows.append(P)
        if len(o.feats) == 0:
            rows = []
        omap.kfs.append(o)
        pt_begin.append(sum(pt_count)); pt_count.append(len(rows)); kf_t.append(pose[4:]); pts_all += rows
    inv_rmp = {v: k for k, v in rmp.items()}
    pose_cur = S.pose_from_xi([0.05, -0.02, 0.01, 0.01, -0.02, 0.005])
    imgc, _ = S.render(scene, cam, pose_cur)
    cur = R.frame(imgc, pose_cur)
    ocur = OracleFrame(imgc, pose_cur)

    ids, dist = R.close_keyframes(cur)
    vis, odist, local = O.close_keyframes(oc, pose_cur, pt_begin, pt_count, np.array(kf_t), np.array(pts_all), 10)
    assert sorted(ids.tolist()) == np.nonzero(vis)[0].tolist() and 10 < len(ids) < n_kf        # Map iterates a std::set<KeyFrame*>: address order
    assert 5 not in ids and 9 not in ids                            # the two far key frames share no visible point
    for k, d in zip(ids, dist):
        assert d == odist[k]
    loc, n_local_pts = R.update_local_map(cur)
    ds = [odist[k] for k in loc]
    assert len(loc) == 10 and ds == sorted(ds) and set(loc.tolist()) == set(local.tolist())
    assert len(set(ds)) == len(ds) and (loc == local).all()         # no ties in this map: the order is the oracle's
    R.tracking_search_local_points()
    want = _oracle_search_multi(oc, cam, ocur, omap, loc.tolist())
    f = R.features(cur)
    got_ids = [inv_rmp[m] for m in R.frame_mappoints(cur)]
    assert len(want) == len(got_ids) and len(want) > 60, (len(want), len(got_ids))
    for (mp, p, SL, _), gp, gl, gid in zip(want, f["px"], f["level"], got_ids):
        assert gid == mp and gl == SL and (p == gp).all()
    # the number of local map points = points that landed in the image (ref: src/Tracking.cpp:299-301)
    n_in = 0
    seen = set()
    for q in loc:
        for mp in omap.kfs[q].feat_mp:
            if mp >= 0 and mp not in seen:
                seen.add(mp)
                n_in += O.reproject_point(oc, pose_cur, omap.mp_point[mp], CELL, 43)[0]
    assert n_local_pts == n_in
