"""GPU suite for the key frame behind the tracked pose: dsdtm_batch_run(flags 15) = pyramid -> Run -> the refinement chain ->
SearchLocalPoints' selection -> PoseOptimization -> Tracking::CraeteKeyframe's detection and depth lift (ref: src/Tracking.cpp:412-464),
all on the device, against the CPU reference tests/cpp/keyframe_chain_oracle.cpp, the single-frame entry points and the analytic scene."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import keyframe_chain as KC
import track_select as TS
from dsdtm_b200 import synth as S

pytestmark = pytest.mark.gpu

PPP, CELL, MIN_DIST, MAX_FTS, SCALE = 300, 15, 10, 300, 5000.0
EMPTY, TILED = 5, 6                    # the pair with no map points, the pair whose cur image is a tiled pattern
E_ARG, E_STATE = -1, -4


def _tiled(period, seed, w, h):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


def _stage(c, b, dist, want=None, max_fts=MAX_FTS, depth=True):
    n = b["n"]
    ref_slots = 2 * np.arange(n, dtype=np.int32); cur_slots = ref_slots + 1
    c.batch_stage(ref_slots, cur_slots, b["feats"], b["n_feats"], b["centers"], b["poses_in"], 5, 0, 8, None, None, None, 10)
    c.batch_stage_map(b["poses_ref"], b["ppp"], 2, 10)
    c.batch_stage_track(None, 100)
    c.batch_stage_keyframe(np.arange(n, dtype=np.int32) if depth else None, want, 5.0, MIN_DIST, max_fts, dist, SCALE)


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def setup(request, built):
    from dsdtm_b200 import capi
    cam = dict(getattr(S, request.param))
    b = TS.make_batch(cam, 8, PPP, n_scenes=4, empty_pair=EMPTY)
    b["cur_imgs"][TILED] = _tiled(15, 3, cam["width"], cam["height"])
    n = b["n"]
    c = capi.Context(cam, levels=5, cell_size=CELL, max_feats=PPP, max_patches=PPP, max_frames=2 * n, max_batch=n)
    c.set_option("depth_slots", n)
    d16, pts = [], []
    for i in range(n):
        pr = b["prs"][i % len(b["prs"])]
        c.upload(2 * i, pr["ref_img"]); c.upload(2 * i + 1, b["cur_imgs"][i])
        _, z, p = S.render(pr["scene"], cam, pr["T_cur"], want_points=True)
        d16.append(np.clip(np.rint(z * SCALE), 0, 65535).astype(np.uint16)); pts.append(p)
        c.depth_upload(i, d16[-1])
    b["d16"] = np.stack(d16); b["pts"] = pts
    b["dist"] = KC.EUROC_DIST if request.param == "EUROC" else (0.0,) * 5
    yield c, b
    c.close()


def _reference(c, b, dist, max_fts=MAX_FTS):
    poses, nm, m, _, _ = c.batch_fetch_track()
    return KC.keyframe_chain(H.ocam(b["cam"]), 5, CELL, MIN_DIST, max_fts, 5.0, dist, SCALE, b["cur_imgs"], m, nm, poses, b["d16"]), nm, m, poses


def _assert_lifted_close(got, want):
    """test_gpu_ingest's bar: undistorted px bit-equal, depth and status exact, normals and points within 1e-12"""
    assert got["px"].tobytes() == want["px"].tobytes()
    assert got["depth"].tobytes() == want["depth"].tobytes() and (got["status"] == want["status"]).all()
    assert np.abs(got["normal"] - want["normal"]).max(initial=0) <= 1e-12
    assert np.abs(got["point_w"] - want["point_w"]).max(initial=0) <= 1e-12


def test_corners_and_lift_equal_the_cpu_reference(setup):
    """corners (x, y, level, score bits, order) and exact_path equal the CPU reference run on the same run's matches and poses; the tiled
    pair takes the literal sort; the lifted records meet test_gpu_ingest's bar against the oracle"""
    c, b = setup
    _stage(c, b, b["dist"])
    c.batch_run(15)
    nn, cr, lf, ex = c.batch_fetch_keyframe()
    o, nm, _, _ = _reference(c, b, b["dist"])
    assert (nn == o["n_new"]).all() and (ex == o["tied"]).all()
    for i in range(b["n"]):
        k = int(nn[i])
        assert KC.same_corners(cr[i][:k], o["corners"][i][:k]), i
        _assert_lifted_close(lf[i][:k], o["lifted"][i][:k])
        assert (cr[i][k:].view(np.uint8) == 0).all() and (lf[i][k:].view(np.uint8) == 0).all()
    assert ex[TILED] and nm[EMPTY] == 0 and nn[EMPTY] > 0 and nn.min() > 0
    print("occupancy indices outside the grid:", int(o["occ_skipped"].sum()), "of", int(nm.sum()), "matches")


def test_equals_single_frame_entry_points(setup):
    """corners bit-equal to dsdtm_detect fed host-built occupancy + CellSize and Min_dist circles; lifted records bit-equal to
    dsdtm_keyframe_lift with the fetched pose"""
    from dsdtm_b200 import capi
    c, b = setup
    _stage(c, b, b["dist"])
    c.batch_run(15)
    poses, nm, m, _, _ = c.batch_fetch_track()
    nn, cr, lf, ex = c.batch_fetch_keyframe()
    for i in range(b["n"]):
        k = int(nm[i])
        px = m[i]["px"][:k]
        occ = np.zeros(c.n_cells, np.uint8)
        for q in px:
            idx = int(q[1] / np.float32(CELL)) * c.grid_cols + int(q[0] / np.float32(CELL))
            if 0 <= idx < c.n_cells:
                occ[idx] = 1
        circ = np.zeros(2 * k, capi.CIRCLE_DT)
        circ["px"][:k] = px; circ["radius"][:k] = CELL
        circ["px"][k:] = px; circ["radius"][k:] = MIN_DIST
        one, ex1 = c.detect(2 * i + 1, 5.0, occupied=occ, circles=circ, max_new=MAX_FTS - k)
        assert KC.same_corners(cr[i][:nn[i]], one[0]) and ex[i] == ex1[0], i
        if nn[i]:
            xy = np.stack([cr[i]["x"][:nn[i]], cr[i]["y"][:nn[i]]], 1).astype(np.float32)
            assert lf[i][:nn[i]].tobytes() == c.keyframe_lift(i, poses[i], b["dist"], SCALE, xy).tobytes(), i


def test_world_points_match_the_scene(setup):
    """without distortion, the lifted points of the tracked pairs lie on the rendered scene within 16-bit depth quantisation (the pair with
    no map points is not tracked: Run has nothing to align, so its pose is not the pose the depth was rendered at)"""
    c, b = setup
    _stage(c, b, (0.0,) * 5)
    c.batch_run(15)
    nn, cr, lf, _ = c.batch_fetch_keyframe()
    worst = 0.0
    for i in range(b["n"]):
        if i in (TILED, EMPTY):
            continue
        k = int(nn[i])
        assert (lf[i]["status"][:k] == KC.LIFT_OK).all()
        want = b["pts"][i][np.rint(lf[i]["px"][:k, 1]).astype(int), np.rint(lf[i]["px"][:k, 0]).astype(int)]
        worst = max(worst, np.abs(lf[i]["point_w"][:k] - want).max())
    assert worst < 2e-3, worst


def test_flags_15_leaves_flags_7_unchanged(setup):
    """poses, matches, res_norm and summaries bit-equal between flags 7 and 15, flags-3 records too; replays are stable; a
    dsdtm_detect_batch call between two replays does not change the next replay"""
    c, b = setup
    _stage(c, b, b["dist"])
    c.batch_run(3)
    rep3 = c.batch_fetch_map().tobytes()
    c.batch_run(7)
    t7 = [a.tobytes() for a in c.batch_fetch_track()]
    c.batch_run(15)
    assert [a.tobytes() for a in c.batch_fetch_track()] == t7 and c.batch_fetch_map().tobytes() == rep3
    kf = [a.tobytes() for a in c.batch_fetch_keyframe()]
    c.batch_run(15)
    assert [a.tobytes() for a in c.batch_fetch_keyframe()] == kf
    occ = np.ones((3, c.n_cells), np.uint8); occ[:, ::3] = 0
    c.detect(1, 20.0, occupied=occ, mask=np.zeros((3, c.height, c.width), np.uint8) + 255, max_new=[5, 50, 500], n=3)
    c.batch_run(15)
    assert [a.tobytes() for a in c.batch_fetch_keyframe()] == kf
    assert [a.tobytes() for a in c.batch_fetch_track()] == t7
    c.batch_run(7)
    assert [a.tobytes() for a in c.batch_fetch_track()] == t7
    c.batch_run(3)
    assert c.batch_fetch_map().tobytes() == rep3


def test_want_mask_and_max_fts(setup):
    """unwanted pairs return no corners and zero rows; wanted pairs equal the all-wanted run; max_fts <= n_matches selects nothing"""
    c, b = setup
    n = b["n"]
    _stage(c, b, b["dist"])
    c.batch_run(15)
    full = c.batch_fetch_keyframe()
    want = (np.arange(n) % 3 == 1).astype(np.uint8)
    _stage(c, b, b["dist"], want=want)
    c.batch_run(15)
    nn, cr, lf, ex = c.batch_fetch_keyframe()
    for i in range(n):
        if want[i]:
            assert nn[i] == full[0][i] and cr[i].tobytes() == full[1][i].tobytes() and lf[i].tobytes() == full[2][i].tobytes()
            assert ex[i] == full[3][i]
        else:
            assert nn[i] == 0 and not ex[i] and (cr[i].view(np.uint8) == 0).all() and (lf[i].view(np.uint8) == 0).all()
    _stage(c, b, b["dist"], want=np.zeros(n, np.uint8))
    c.batch_run(15)
    assert (c.batch_fetch_keyframe()[0] == 0).all()
    _, nm, _, _, _ = c.batch_fetch_track()
    cap = int(np.median(nm))
    _stage(c, b, b["dist"], max_fts=cap)
    c.batch_run(15)
    nn, cr, lf, ex = c.batch_fetch_keyframe()
    o, _, _, _ = _reference(c, b, b["dist"], max_fts=cap)
    assert (nn == o["n_new"]).all() and (nn[nm >= cap] == 0).all() and (nn[nm < cap] > 0).all()
    for i in range(n):
        assert KC.same_corners(cr[i][:nn[i]], o["corners"][i][:nn[i]]), i


def _raw_stage(c, ds=None, want=None, min_dist=MIN_DIST, max_fts=MAX_FTS, dist=(0.0,) * 5):
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    return c.L.dsdtm_batch_stage_keyframe(c.hp, p(None if ds is None else np.ascontiguousarray(ds, np.int32)),
                                          p(None if want is None else np.ascontiguousarray(want, np.uint8)), C.c_float(5.0), int(min_dist),
                                          int(max_fts), p(np.ascontiguousarray(dist, np.float32)), C.c_float(SCALE))


def _trivial_batch(c):
    from dsdtm_b200 import capi
    c.batch_stage([0], [0], np.zeros((1, 1), capi.REF_FEAT_DT), [0], np.zeros((1, 3)), S.IDENTITY[None], 4, 0, 8)
    c.batch_stage_map(S.IDENTITY[None], 1, 2, 10)


def test_state_and_argument_errors(setup, built):
    from dsdtm_b200 import capi
    c, b = setup
    n = b["n"]
    _stage(c, b, b["dist"])
    for bad in ([n] + [0] * (n - 1), [-2] + [0] * (n - 1)):              # past option depth_slots, below -1
        assert _raw_stage(c, ds=bad) == E_ARG
    assert _raw_stage(c, max_fts=0) == E_ARG and _raw_stage(c, max_fts=513) == E_ARG
    assert _raw_stage(c, min_dist=65) == E_ARG and _raw_stage(c, min_dist=-1) == E_ARG
    assert _raw_stage(c, ds=-np.ones(n)) == 0 and _raw_stage(c, ds=np.arange(n), want=np.ones(n)) == 0
    assert c.L.dsdtm_batch_run(c.hp, 8 | 2 | 1) == E_STATE                 # bit 3 without bit 2
    c.batch_stage_track(None, 100)                                       # drops the key-frame staging
    assert c.L.dsdtm_batch_run(c.hp, 15) == E_STATE
    with pytest.raises(capi.DsdtmError):
        c.batch_fetch_keyframe()
    c.batch_stage_map(b["poses_ref"], PPP, 2, 10)
    assert _raw_stage(c) == E_STATE                                      # stage_track first
    c2 = capi.Context(b["cam"], levels=5, cell_size=CELL, max_feats=16, max_patches=16, max_frames=2, max_batch=1)
    try:
        _trivial_batch(c2)
        assert _raw_stage(c2) == E_STATE
        c2.batch_stage_track(None, 10)
        assert _raw_stage(c2, ds=[0]) == E_ARG                           # a depth slot before the depth pool exists
        assert _raw_stage(c2, ds=[-1]) == 0
    finally:
        c2.close()
    big = dict(b["cam"], width=800, height=600)
    c3 = capi.Context(big, levels=4, cell_size=CELL, max_feats=16, max_patches=16, max_frames=1, max_batch=1)
    try:
        _trivial_batch(c3)
        c3.batch_stage_track(None, 10)
        assert _raw_stage(c3) == E_ARG                                   # 800 x 600 does not fit the selection bitmap
    finally:
        c3.close()
