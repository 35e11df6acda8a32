"""GPU suite for the tracked-pose chain: dsdtm_batch_run(flags | 2 | 4) = pyramid -> Run -> the refinement chain -> SearchLocalPoints'
selection -> PoseOptimization, all on the device (ref: src/Tracking.cpp:219-236)."""
import numpy as np
import pytest

import helpers as H
import oracle as O
import track_select as TS
from dsdtm_b200 import synth as S

pytestmark = pytest.mark.gpu

PPP = 300


def _stage(c, b, found=None, max_iters=100):
    n = b["n"]
    ref_slots = 2 * np.arange(n, dtype=np.int32); cur_slots = ref_slots + 1
    c.batch_stage(ref_slots, cur_slots, b["feats"], b["n_feats"], b["centers"], b["poses_in"], 5, 0, 8, None, None, None, 10)
    c.batch_stage_map(b["poses_ref"], b["ppp"], 2, 10)
    c.batch_stage_track(found, max_iters)


def _context(b):
    from dsdtm_b200 import capi
    n, ppp = b["n"], b["ppp"]
    c = capi.Context(b["cam"], levels=5, cell_size=15, max_feats=ppp, max_patches=ppp, max_frames=2 * n, max_batch=n)
    for i in range(n):
        c.upload(2 * i, b["prs"][i % len(b["prs"])]["ref_img"]); c.upload(2 * i + 1, b["cur_imgs"][i])
    return c


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def setup(request, built):
    b = TS.make_batch(dict(getattr(S, request.param)), 8, PPP, n_scenes=4, empty_pair=5)
    c = _context(b)
    yield c, b
    c.close()


def _founds(n, ppp):
    rng = np.random.default_rng(11)
    return {"null": None, "random": rng.integers(1, 60, (n, ppp)).astype(np.int32),
            "tied": rng.integers(1, 3, (n, ppp)).astype(np.int32)}


def test_selection_is_bit_exact_against_the_replay(setup):
    """the flags-7 matches equal the greedy replay over the records batch_fetch_map returns from the same run: point, float px bits,
    level and order; NULL, random and heavily tied found counts"""
    c, b = setup
    w, h = b["cam"]["width"], b["cam"]["height"]
    for name, found in _founds(b["n"], PPP).items():
        _stage(c, b, found)
        c.batch_run(7)
        rep = c.batch_fetch_map()
        _, nm, m, res, _ = c.batch_fetch_track()
        f = np.ones((b["n"], PPP), np.int32) if found is None else found
        for i in range(b["n"]):
            TS.assert_matches_equal(m[i], int(nm[i]), TS.replay(rep[i], f[i], w, h, 15))
            assert (m[i][nm[i]:].view(np.uint8) == 0).all() and (res[i][nm[i]:] == 0).all()
        assert nm[5] == 0 and nm.max() > 50, name


def test_handoff_equals_pose_optimize_batch(setup):
    """final poses, res_norm and summaries are bit-equal to dsdtm_pose_optimize_batch on host-built observations (Frame::Add_Feature's
    bearing through the oracle, the staged points, the match levels) from O.se3_mul(T_c2r, T_ref), same n_pairs; the zero-match pair
    ends NO_RESIDUALS with the pose the solver gives for no observations"""
    from dsdtm_b200 import capi
    c, b = setup
    oc = H.ocam(b["cam"])
    _stage(c, b)
    c.batch_run(7)
    poses_c2r, _, _, _ = c.batch_fetch()
    poses, nm, m, res, summ = c.batch_fetch_track()
    n = b["n"]
    obs = np.zeros((n, 200), capi.BA_OBS_DT)
    starts = np.zeros((n, 7))
    for i in range(n):
        for k in range(nm[i]):
            obs[i, k]["normal"] = O.feature_normal(oc, m[i, k]["px"])
            obs[i, k]["point_w"] = b["feats"][i, m[i, k]["point"]]["point_w"]
            obs[i, k]["level"] = m[i, k]["level"]
        starts[i] = O.se3_mul(poses_c2r[i], b["poses_ref"][i])
    p2, r2, s2 = c.pose_optimize_batch(obs, nm, starts, 100)
    assert poses.tobytes() == p2.tobytes() and summ.tobytes() == s2.tobytes()
    for i in range(n):
        assert res[i][:nm[i]].tobytes() == r2[i][:nm[i]].tobytes()
    assert nm[5] == 0 and summ["termination"][5] == capi.BA_NO_RESIDUALS
    p0, _, _ = c.pose_optimize_batch(np.zeros((n, 200), capi.BA_OBS_DT), np.zeros(n, np.int32), starts, 100)
    assert poses[5].tobytes() == p0[5].tobytes()


def test_whole_chain_against_the_oracle(setup):
    """the oracle's whole chain (tests/cpp/track_chain_oracle.cpp): match lists equal (points, levels), px within 1e-3, final pose within 1e-5 rad / m, termination and
    iteration counts equal"""
    c, b = setup
    oc = H.ocam(b["cam"])
    found = _founds(b["n"], PPP)["tied"]
    _stage(c, b, found)
    c.batch_run(7)
    poses, nm, m, _, summ = c.batch_fetch_track()
    o = TS.pair_batch_track(oc, 5, 15, b["ref_pyrs"], b["cur_imgs"], b["feats"], b["n_feats"], b["centers"], b["poses_ref"], b["poses_in"],
                           5, 0, 8, PPP, 2, 10, found=found, ba_iters=100, n_threads=4)
    assert (nm == o["n_matches"]).all()
    for i in range(b["n"]):
        k = nm[i]
        assert (m[i]["point"][:k] == o["matches"][i]["point"][:k]).all() and (m[i]["level"][:k] == o["matches"][i]["level"][:k]).all()
        assert k == 0 or np.abs(m[i]["px"][:k] - o["matches"][i]["px"][:k]).max() <= 1e-3
        d = S.pose_dist(o["poses"][i], poses[i])
        assert d[0] < 1e-5 and d[1] < 1e-5, (i, d)
    assert (summ["termination"] == o["summaries"]["termination"]).all()
    assert (summ["iterations"] == o["summaries"]["iterations"]).all()


def test_two_hundred_match_cap(built):
    """512 staged features on a textured scene: the uncapped replay finds more than 200 matches, the device stops at exactly 200 and its
    list equals the capped replay"""
    cam = dict(S.KINECT)
    b = TS.make_batch(cam, 2, 512, seed0=71, n_scenes=2, trans=0.01, rot_deg=0.3)
    c = _context(b)
    try:
        _stage(c, b)
        c.batch_run(7)
        rep = c.batch_fetch_map()
        _, nm, m, _, summ = c.batch_fetch_track()
        ones = np.ones(512, np.int32)
        for i in range(2):
            assert len(TS.replay(rep[i], ones, cam["width"], cam["height"], 15, cap=None)) > 200
            TS.assert_matches_equal(m[i], int(nm[i]), TS.replay(rep[i], ones, cam["width"], cam["height"], 15))
            assert nm[i] == 200 and summ["n_obs"][i] == 200
    finally:
        c.close()


def test_graph_state(setup):
    """flags-7 replays give identical bytes; the flags-3 records are unchanged by running flags 7; a larger dsdtm_pose_optimize_batch
    call between two replays (it regrows its own buffers) does not disturb the captured step; bit 2 without stage_track or bit 1 raises"""
    from dsdtm_b200 import capi
    c, b = setup
    n = b["n"]
    _stage(c, b)
    c.batch_run(3)
    rep3 = c.batch_fetch_map().tobytes()
    c.batch_run(7)
    first = [a.tobytes() for a in c.batch_fetch_track()]
    assert c.batch_fetch_map().tobytes() == rep3
    c.batch_run(7)
    assert [a.tobytes() for a in c.batch_fetch_track()] == first
    pr = H.make_ba_problem(4, n=300)
    big = 4 * n
    obs = np.tile(H.ba_obs_records(pr, capi.BA_OBS_DT), (big, 1))
    c.pose_optimize_batch(obs, np.full(big, 300, np.int32), np.tile(pr["pose_in"], (big, 1)))
    c.batch_run(7)
    assert [a.tobytes() for a in c.batch_fetch_track()] == first
    c.batch_run(3)
    assert c.batch_fetch_map().tobytes() == rep3
    with pytest.raises(capi.DsdtmError):
        c.batch_run(5)                                                   # bit 2 without bit 1
    c.batch_stage_map(b["poses_ref"], PPP, 2, 10)                        # drops the track staging
    with pytest.raises(capi.DsdtmError):
        c.batch_run(7)
    with pytest.raises(capi.DsdtmError):
        c.batch_fetch_track()
