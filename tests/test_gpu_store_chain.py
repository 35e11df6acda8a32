"""GPU suite for the batched chain on the map store (dsdtm_batch_stage_store): every frame's local map is UpdateLocalMap's nearest key
frames of a real multi-key-frame map (tests/store_map.py), not its reference frame seen as one key frame. The single-frame
dsdtm_store_track, which tests/test_gpu_sequence.py holds to the reference's literal loop, is the yardstick of the records."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import oracle as O
import store_map as SM
import track_select as TS
from dsdtm_b200 import capi, synth as S

pytestmark = pytest.mark.gpu

N_SCENES, N_KFS, FRAMES_PER_SCENE = 4, 8, 2
N = N_SCENES * FRAMES_PER_SCENE
CPF = 2048
MAX_LOCAL = 6
CUR0 = N_SCENES * N_KFS                       # cur slots follow the key-frame slots


def _context(cam, max_batch=N, max_patches=CPF, extra_slots=0):
    return capi.Context(cam, levels=5, cell_size=15, max_feats=320, max_patches=max_patches, max_frames=CUR0 + N + extra_slots,
                        max_batch=max_batch)


def _frames(rs, maps, frames):
    """host arrays of the batch frames [(scene, frame index)]: pair i tracks cur slot CUR0 + i against its scene's last key frame"""
    n = len(frames)
    feats = np.zeros((n, 320), capi.REF_FEAT_DT); nf = np.zeros(n, np.int32)
    centers = np.zeros((n, 3)); poses_ref = np.zeros((n, 7)); ref_slots = np.zeros(n, np.int32)
    for i, (s, _) in enumerate(frames):
        feats[i], nf[i] = SM.ref_feats(maps[s], 320)
        last = maps[s]["kfs"][-1]
        centers[i] = last["center"]; poses_ref[i] = last["pose"]; ref_slots[i] = last["slot"]
    return dict(frames=frames, feats=feats, n_feats=nf, centers=centers, poses_ref=poses_ref, ref_slots=ref_slots,
                cur_slots=CUR0 + np.arange(n, dtype=np.int32), imgs=[rs[s]["frames"][f]["img"] for s, f in frames])


def _stage(c, fr, kf_range=None, max_local=MAX_LOCAL, cpf=CPF, found=None, track=True):
    n = len(fr["frames"])
    for i in range(n):
        c.upload(int(fr["cur_slots"][i]), fr["imgs"][i])
    c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], np.tile(S.IDENTITY, (n, 1)), 5, 0, 8)
    c.batch_stage_store(fr["poses_ref"], kf_range, max_local, 2, 10, cpf)
    if track:
        c.batch_stage_track(found, 100)


def _prior(c, fr):
    poses_c2r, _, _, _ = c.batch_fetch()
    pose = [O.se3_mul(poses_c2r[i], fr["poses_ref"][i]) for i in range(len(poses_c2r))]
    return pose, [O.se3_inv(p)[4:] for p in pose]


def _assert_frame_equals_store_track(c, i, pose, center, loc, nl, rec, nc, max_local=MAX_LOCAL, cur_slot=None):
    local, ref = c.store_track(int(CUR0 + i if cur_slot is None else cur_slot), pose, center, max_local, 2, 10, cap=8192)
    ref = ref[np.argsort(ref["order"], kind="stable")]
    assert int(nl[i]) == len(local) and (loc[i][:nl[i]] == local).all() and (loc[i][nl[i]:] == -1).all()
    assert int(nc[i]) == len(ref)
    got = rec[i][:nc[i]]
    assert (np.diff(got["order"]) > 0).all()                     # records come back in ReprojectPoint order
    assert got.tobytes() == ref.tobytes(), i                     # every field, refined px bits included
    return ref


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def setup(request, built):
    cam = dict(getattr(S, request.param))
    rs = SM.render_scenes(cam, [3100 + 17 * k for k in range(N_SCENES)], N_KFS, FRAMES_PER_SCENE)
    c = _context(cam)
    maps = [SM.build_map(c, cam, rs[s], s * N_KFS) for s in range(N_SCENES)]
    offs = SM.load_maps(c, maps)
    fr = _frames(rs, maps, [(s, f) for f in range(FRAMES_PER_SCENE) for s in range(N_SCENES)])
    ranges = np.array([[offs[s][0], offs[s][0] + N_KFS] for s, _ in fr["frames"]], np.int32)
    yield dict(cam=cam, c=c, rs=rs, maps=maps, offs=offs, fr=fr, ranges=ranges)
    c.close()


def test_maps_have_shared_points_bad_points_and_pointless_features(setup):
    """the built maps carry what the tracker's maps carry: points observed by several key frames, bad points, features without a point"""
    for m in setup["maps"]:
        mp = np.concatenate([kf["feats"]["mp"] for kf in m["kfs"]])
        obs = np.bincount(mp[mp >= 0], minlength=len(m["pw"]))
        assert (obs >= 3).sum() > 50 and (mp < 0).any() and m["bad"].any()


def test_records_equal_store_track(setup):
    """every row of the store (kf_range NULL): per frame, local rows, n_local and the records are bit-equal to dsdtm_store_track on the
    same store with that frame's prior pose, keyed by order; the local maps hold several key frames and several hundred candidates"""
    c, fr = setup["c"], setup["fr"]
    _stage(c, fr, None, track=False)
    c.batch_run(3)
    loc, nl, rec, nc = c.batch_fetch_store()
    pose, center = _prior(c, fr)
    for i in range(N):
        _assert_frame_equals_store_track(c, i, pose[i], center[i], loc, nl, rec, nc)
    assert nl.min() >= 3 and nc.min() > 200 and (rec[:, 0]["r"]["flags"] & capi.LM_CONVERGED).any()
    assert (rec.view(np.uint8).reshape(N, -1)[:, nc.max() * capi.STORE_CAND_DT.itemsize:] == 0).all()


def test_partitions_equal_single_scene_contexts(setup):
    """K scenes' maps in one store with per-frame ranges give each frame exactly the outputs of a context holding only its scene's map
    (records, local rows, matches, poses, residuals, summaries), after mapping store rows; local rows never leave the range"""
    c, fr, maps, offs, cam = setup["c"], setup["fr"], setup["maps"], setup["offs"], setup["cam"]
    _stage(c, fr, setup["ranges"])
    c.batch_run(7)
    loc, nl, rec, nc = c.batch_fetch_store()
    poses, nm, m, res, summ = c.batch_fetch_track()
    for s in range(N_SCENES):
        k0, p0 = offs[s]
        idx = [i for i, (sc, _) in enumerate(fr["frames"]) if sc == s]
        for i in idx:
            assert ((loc[i][:nl[i]] >= k0) & (loc[i][:nl[i]] < k0 + N_KFS)).all()
        c2 = _context(cam)
        try:
            SM.load_maps(c2, [maps[s]])
            sub = {k: (v[idx] if isinstance(v, np.ndarray) else [v[i] for i in idx]) for k, v in fr.items()}
            sub["cur_slots"] = fr["cur_slots"][idx]
            _stage(c2, sub, None)
            c2.batch_run(7)
            loc2, nl2, rec2, nc2 = c2.batch_fetch_store()
            poses2, nm2, m2, res2, summ2 = c2.batch_fetch_track()
        finally:
            c2.close()
        feat0 = sum(len(kf["feats"]) for mm in maps[:s] for kf in mm["kfs"])
        for q, i in enumerate(idx):
            assert nl[i] == nl2[q] and (loc[i][:nl[i]] - k0 == loc2[q][:nl2[q]]).all()
            assert nc[i] == nc2[q]
            a, b = rec[i][:nc[i]].copy(), rec2[q][:nc2[q]]
            a["mp"] -= p0
            a["r"]["obs"][a["r"]["obs"] >= 0] -= feat0
            assert a.tobytes() == b.tobytes(), (s, i)
            assert nm[i] == nm2[q] and nm[i] > 20
            mm = m[i].copy(); mm["point"][:nm[i]] -= p0
            assert mm.tobytes() == m2[q].tobytes()
            assert poses[i].tobytes() == poses2[q].tobytes() and res[i].tobytes() == res2[q].tobytes()
            assert summ[i].tobytes() == summ2[q].tobytes()


def _founds(n_pts):
    rng = np.random.default_rng(23)
    return {"null": None, "random": rng.integers(1, 60, n_pts).astype(np.int32), "tied": rng.integers(1, 3, n_pts).astype(np.int32)}


def test_selection_and_pose_against_restatements(setup):
    """matches equal tests/track_select.py's restatement over the fetched records with NULL, random and tied found counts per store
    point; poses, residual norms and summaries are bit-equal to dsdtm_pose_optimize_batch on host-built observations (the store's
    points) from the prior pose"""
    c, fr, cam = setup["c"], setup["fr"], setup["cam"]
    oc = H.ocam(cam)
    n_pts = sum(len(mm["pw"]) for mm in setup["maps"])
    pw = np.concatenate([mm["pw"] for mm in setup["maps"]])
    for name, found in _founds(n_pts).items():
        _stage(c, fr, setup["ranges"], found=found)
        c.batch_run(7)
        _, _, rec, nc = c.batch_fetch_store()
        poses, nm, m, res, summ = c.batch_fetch_track()
        f = np.ones(n_pts, np.int32) if found is None else found
        obs = np.zeros((N, 200), capi.BA_OBS_DT)
        for i in range(N):
            r = rec[i][:nc[i]]
            want = [(int(r["mp"][j]), p, lv) for j, p, lv in TS.replay(r["r"], f[r["mp"]], cam["width"], cam["height"], 15)]
            TS.assert_matches_equal(m[i], int(nm[i]), want)
            assert (m[i][nm[i]:].view(np.uint8) == 0).all() and (res[i][nm[i]:] == 0).all()
            for k in range(nm[i]):
                obs[i, k]["normal"] = O.feature_normal(oc, m[i, k]["px"])
                obs[i, k]["point_w"] = pw[m[i, k]["point"]]
                obs[i, k]["level"] = m[i, k]["level"]
        pose, _ = _prior(c, fr)
        p2, r2, s2 = c.pose_optimize_batch(obs, nm, np.array(pose), 100)
        assert poses.tobytes() == p2.tobytes() and summ.tobytes() == s2.tobytes(), name
        for i in range(N):
            assert res[i][:nm[i]].tobytes() == r2[i][:nm[i]].tobytes()
        assert nm.min() > 20, name


def test_two_hundred_match_cap(setup):
    """a frame whose selection reaches 200 matches stops there, and its list equals the capped restatement"""
    c, fr, cam = setup["c"], setup["fr"], setup["cam"]
    _stage(c, fr, setup["ranges"], max_local=N_KFS)
    c.batch_run(7)
    _, _, rec, nc = c.batch_fetch_store()
    _, nm, m, _, _ = c.batch_fetch_track()
    capped = 0
    for i in range(N):
        r = rec[i][:nc[i]]
        full = TS.replay(r["r"], np.ones(nc[i], np.int32), cam["width"], cam["height"], 15, cap=None)
        TS.assert_matches_equal(m[i], int(nm[i]), [(int(r["mp"][j]), p, lv) for j, p, lv in full[:200]])
        capped += len(full) > 200
    assert capped > 0 and nm.max() == 200


def _assert_step_follows_store(c, fr, pw, cam):
    """the outputs of the last flags-7 run: records equal dsdtm_store_track on the store as it is now, matches equal the restatement
    (found 1 everywhere), and poses equal dsdtm_pose_optimize_batch on host-built observations with the store's current points pw"""
    loc, nl, rec, nc = c.batch_fetch_store()
    poses, nm, m, res, summ = c.batch_fetch_track()
    pose, center = _prior(c, fr)
    oc = H.ocam(cam)
    obs = np.zeros((N, 200), capi.BA_OBS_DT)
    for i in range(N):
        _assert_frame_equals_store_track(c, i, pose[i], center[i], loc, nl, rec, nc)
        r = rec[i][:nc[i]]
        want = [(int(r["mp"][j]), p, lv) for j, p, lv in TS.replay(r["r"], np.ones(nc[i], np.int32), cam["width"], cam["height"], 15)]
        TS.assert_matches_equal(m[i], int(nm[i]), want)
        for k in range(nm[i]):
            obs[i, k]["normal"] = O.feature_normal(oc, m[i, k]["px"]); obs[i, k]["point_w"] = pw[m[i, k]["point"]]
            obs[i, k]["level"] = m[i, k]["level"]
    p2, _, s2 = c.pose_optimize_batch(obs, nm, np.array(pose), 100)
    assert poses.tobytes() == p2.tobytes() and summ.tobytes() == s2.tobytes()
    return rec, nc


def test_replays_are_stable_and_follow_store_changes(setup, built):
    """replays are byte-stable; each store change between two replays of the SAME captured flags-7 step -- store_update_points (a bad
    point, a moved point), store_set_points (appended points), store_append_keyframe, store_set_keyframe -- reaches the next replay: it
    equals dsdtm_store_track, the selection restatement and dsdtm_pose_optimize_batch on the changed map; a flags-7 stage_map run after a
    store-mode run equals the same run on a fresh context"""
    cam, maps, fr, rs = setup["cam"], setup["maps"], setup["fr"], setup["rs"]
    c = _context(cam, extra_slots=1)
    try:
        SM.load_maps(c, maps)
        _stage(c, fr, None)
        c.batch_run(7)
        first = c.batch_fetch_store(), c.batch_fetch_track()
        c.batch_run(7)
        again = c.batch_fetch_store(), c.batch_fetch_track()
        for a, b in zip(first[0] + first[1], again[0] + again[1]):
            assert a.tobytes() == b.tobytes()
        # change the map between replays of the step captured above
        pw = np.concatenate([mm["pw"] for mm in maps])
        loc, nl, rec, nc = first[0]
        pts = rec[0][:nc[0]]["mp"]
        prev = rec.tobytes()

        def replay_and_check():
            nonlocal prev
            c.batch_run(7)
            r, _ = _assert_step_follows_store(c, fr, pw, cam)
            changed = r.tobytes() != prev
            prev = r.tobytes()
            return changed
        c.store_update_points([int(pts[0]), int(pts[5])], None, [1, 1])
        assert replay_and_check()
        pw[int(pts[7])] += np.array([0.01, -0.005, 0.002])
        c.store_update_points([int(pts[7])], pw[int(pts[7])][None], None)
        assert replay_and_check()
        # appended points (the point table is reallocated past its capacity) observed by an appended key frame
        extra = pw[:5000] + np.array([0.0, 0.0, 0.001])
        p0 = c.store_points
        c.store_set_points(p0, extra)
        pw = np.concatenate([pw, extra])
        last = maps[0]["kfs"][-1]
        F = last["feats"].copy()
        F["mp"][F["mp"] >= 0] += p0
        c.upload(CUR0 + N, maps[0]["imgs"][-1])
        c.store_append_keyframe(CUR0 + N, S.pose_mul(S.pose_from_xi(np.r_[0.004, 0, 0, 0, 0.002, 0]), last["pose"]), last["center"], F)
        assert replay_and_check()
        k = int(loc[1][0])
        moved = S.pose_mul(S.pose_from_xi(np.r_[0.0, 0.003, 0, 0.001, 0, 0]), maps[0]["kfs"][0]["pose"])
        c.store_set_keyframe(k, maps[0]["kfs"][0]["slot"], moved, S.pose_inv(moved)[4:])
        assert replay_and_check()
        # the one-key-frame mode after a store-mode run equals a fresh context
        b = TS.make_batch(dict(cam), 4, 300, n_scenes=2)

        def run_map(ctx):
            for i in range(4):
                ctx.upload(2 * i, b["prs"][i % 2]["ref_img"]); ctx.upload(2 * i + 1, b["cur_imgs"][i])
            ctx.batch_stage(2 * np.arange(4, dtype=np.int32), 2 * np.arange(4, dtype=np.int32) + 1, b["feats"], b["n_feats"], b["centers"],
                            b["poses_in"], 5, 0, 8)
            ctx.batch_stage_map(b["poses_ref"], 300, 2, 10)
            ctx.batch_stage_track(None, 100)
            ctx.batch_run(7)
            return ctx.batch_fetch_map(), ctx.batch_fetch_track()
        got = run_map(c)
        c2 = _context(cam)
        try:
            want = run_map(c2)
        finally:
            c2.close()
        assert got[0].tobytes() == want[0].tobytes()
        for a, b_ in zip(got[1], want[1]):
            assert a.tobytes() == b_.tobytes()
    finally:
        c.close()


def test_overflow_frame_and_others_unchanged(setup):
    """with cands_per_frame below one frame's candidate count, that frame keeps its first records in order, gets n_matches -1, its
    prior pose and no key frame; every other frame's records, matches and pose equal the run with room for all"""
    c, fr = setup["c"], setup["fr"]
    _stage(c, fr, setup["ranges"])
    c.batch_run(7)
    _, _, rec, nc = c.batch_fetch_store()
    full = c.batch_fetch_track()
    small = int(np.sort(nc)[-1]) - 1
    assert small >= int(np.sort(nc)[-2])                         # exactly one frame overflows
    i_over = int(np.argmax(nc))
    _stage(c, fr, setup["ranges"], cpf=small)
    c.batch_stage_keyframe(None, None, 5.0, 15, 300, (0.0,) * 5, 5000.0)
    c.batch_run(15)
    _, _, rec2, nc2 = c.batch_fetch_store()
    poses, nm, m, res, summ = c.batch_fetch_track()
    n_new, _, _, _ = c.batch_fetch_keyframe()
    pose, _ = _prior(c, fr)
    assert (nc2 == nc).all() and nm[i_over] == -1 and poses[i_over].tobytes() == pose[i_over].tobytes()
    assert n_new[i_over] == 0 and (m[i_over].view(np.uint8) == 0).all()
    assert rec2[i_over].tobytes() == rec[i_over][:small].tobytes()
    for i in range(N):
        if i == i_over:
            continue
        assert rec2[i][:nc[i]].tobytes() == rec[i][:nc[i]].tobytes()
        assert nm[i] == full[1][i] and m[i].tobytes() == full[2][i].tobytes() and poses[i].tobytes() == full[0][i].tobytes()
        assert n_new[i] > 0


def test_range_beyond_one_thousand_key_frames(setup, built):
    """1100 cheap key frames (a few features each, observing scene 0's points) behind one map: the prelude's one CTA covers the range and
    the records equal dsdtm_store_track, which takes its three-kernel path there"""
    cam, maps, fr = setup["cam"], setup["maps"], setup["fr"]
    c = _context(cam)
    try:
        SM.load_maps(c, [maps[0]])
        rng = np.random.default_rng(5)
        last = maps[0]["kfs"][-1]
        good = np.flatnonzero(maps[0]["bad"] == 0)
        for k in range(1100):
            F = last["feats"][rng.choice(len(last["feats"]), 4, replace=False)].copy()
            F["mp"] = rng.choice(good, 4, replace=False); F["is_obs"] = 1
            T = S.pose_mul(S.pose_from_xi(rng.uniform(-0.3, 0.3, 6) * np.r_[1, 1, 1, 0.2, 0.2, 0.2]), last["pose"])
            c.store_append_keyframe(last["slot"], T, S.pose_inv(T)[4:], F)
        idx = [i for i, (s, _) in enumerate(fr["frames"]) if s == 0]
        sub = {k: (v[idx] if isinstance(v, np.ndarray) else [v[i] for i in idx]) for k, v in fr.items()}
        sub["cur_slots"] = fr["cur_slots"][idx]
        _stage(c, sub, None, max_local=10, track=False)
        c.batch_run(3)
        loc, nl, rec, nc = c.batch_fetch_store()
        pose, center = _prior(c, sub)
        for q, i in enumerate(idx):
            _assert_frame_equals_store_track(c, q, pose[q], center[q], loc, nl, rec, nc, max_local=10, cur_slot=int(sub["cur_slots"][q]))
        assert (loc[:, :nl.min()] >= N_KFS).any()
    finally:
        c.close()


def test_errors_enqueue_nothing(setup, built):
    """every DSDTM_E_ARG and DSDTM_E_STATE of the store staging, and a run after the store lost the staged rows, return before anything
    is enqueued"""
    cam, maps, fr = setup["cam"], setup["maps"], setup["fr"]
    c = _context(cam)
    L, h = c.L, c.hp
    pr = np.ascontiguousarray(fr["poses_ref"])
    p = pr.ctypes.data_as(C.c_void_p)
    try:
        assert L.dsdtm_batch_stage_store(h, p, None, 10, 2, 10, 64) == -4            # no dsdtm_batch_stage
        for i in range(N):
            c.upload(int(fr["cur_slots"][i]), fr["imgs"][i])
        c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], np.tile(S.IDENTITY, (N, 1)), 5, 0, 8)
        assert L.dsdtm_batch_stage_store(h, p, None, 10, 2, 10, 64) == -1            # empty store
        SM.load_maps(c, maps)
        n0 = c.launch_count()
        bad_range = np.tile(np.array([[0, N_SCENES * N_KFS + 1]], np.int32), (N, 1))
        neg_range = np.tile(np.array([[3, 2]], np.int32), (N, 1))
        for args in [(bad_range, 10, 2, 10, 64), (neg_range, 10, 2, 10, 64), (None, 0, 2, 10, 64), (None, 17, 2, 10, 64),
                     (None, 10, 2, 10, 0), (None, 10, 2, 10, CPF + 1), (None, 10, 5, 10, 64), (None, 10, 2, -1, 64)]:
            r = args[0]
            assert L.dsdtm_batch_stage_store(h, p, None if r is None else r.ctypes.data_as(C.c_void_p), *args[1:]) == -1, args[1:]
        assert L.dsdtm_batch_fetch_store(h, None, None, None, None) == -4
        assert L.dsdtm_batch_run(h, 3) == -4                                         # nothing staged for bit 1
        assert c.launch_count() == n0
        ranges = np.ascontiguousarray(setup["ranges"])
        c.batch_stage_store(fr["poses_ref"], ranges, 10, 2, 10, 64)
        before = c.launch_count()
        c.store_clear()
        assert L.dsdtm_batch_run(h, 3) == -4                                         # the store lost the staged rows
        assert c.launch_count() == before
    finally:
        c.close()


def test_keyframes_in_store_mode(setup, built):
    """flags 15 on the store-backed chain, with the camera's distortion (EuRoC: Config/EuRoc.yaml) and rendered depth: the corners and
    lifted records equal dsdtm_detect_batch and dsdtm_keyframe_lift fed occupancy and circles built on the host from the fetched matches
    and poses; the frame whose candidates overflowed gets no key frame"""
    import keyframe_chain as KC
    cam, maps, fr, rs = setup["cam"], setup["maps"], setup["fr"], setup["rs"]
    dist = KC.EUROC_DIST if cam["width"] == S.EUROC["width"] else (0.0,) * 5
    c = _context(cam)
    try:
        c.set_option("depth_slots", N)
        SM.load_maps(c, maps)
        for i, (s, f) in enumerate(fr["frames"]):
            c.depth_upload(i, rs[s]["frames"][f]["d16"])
        _stage(c, fr, setup["ranges"], track=False)
        c.batch_run(3)
        nc = c.batch_fetch_store()[3]
        cpf = int(np.sort(nc)[-1]) - 1                           # one frame overflows
        _stage(c, fr, setup["ranges"], cpf=cpf)
        c.batch_stage_keyframe(np.arange(N, dtype=np.int32), None, 5.0, 10, 300, dist, 5000.0)
        c.batch_run(15)
        poses, nm, m, _, _ = c.batch_fetch_track()
        n_new, cr, lf, ex = c.batch_fetch_keyframe()
        assert (nm < 0).sum() == 1 and n_new[nm < 0][0] == 0
        occ = np.zeros((N, c.n_cells), np.uint8)
        circles, max_new = [], np.zeros(N, np.int32)
        for i in range(N):
            cs = np.zeros(2 * max(nm[i], 0), capi.CIRCLE_DT)
            for k in range(max(nm[i], 0)):
                px = m[i, k]["px"]
                cell = int(px[1] / np.float32(15)) * c.grid_cols + int(px[0] / np.float32(15))
                if 0 <= cell < c.n_cells:
                    occ[i, cell] = 1
                cs[2 * k]["px"] = px; cs[2 * k]["radius"] = 15; cs[2 * k + 1]["px"] = px; cs[2 * k + 1]["radius"] = 10
            circles.append(cs)
            max_new[i] = 300 - nm[i] if nm[i] >= 0 else 0
        got, exact = c.detect(CUR0, 5.0, occupied=occ, circles=circles, max_new=max_new, n=N)
        assert (exact == ex).all()
        for i in range(N):
            assert n_new[i] == len(got[i]) and cr[i][:n_new[i]].tobytes() == got[i].tobytes(), i
            if n_new[i]:
                px = np.stack([got[i]["x"], got[i]["y"]], 1).astype(np.float32)
                want = c.keyframe_lift(i, poses[i], dist, 5000.0, px)
                assert lf[i][:n_new[i]].tobytes() == want.tobytes(), i
                assert (lf[i][:n_new[i]]["status"] == capi.LIFT_OK).any()
        assert (n_new[nm >= 0] > 0).all()
    finally:
        c.close()


def test_sample_against_the_oracle_chain(setup):
    """the oracle's own chain on a sample of frames, sharing no code with the device path: O.close_keyframes for GetCloseKeyFrames and
    the ranking, tests/oracle_seq.py's OMap and _oracle_search_multi for UpdateLocalMap + SearchLocalPoints (found 1), then the oracle's
    PoseOptimization. Local key frames and match lists (points, levels) equal, px within 1e-3, poses within 1e-5 with the same
    termination"""
    import oracle_seq as OS
    c, fr, cam, maps, offs = setup["c"], setup["fr"], setup["cam"], setup["maps"], setup["offs"]
    oc = H.ocam(cam)
    _stage(c, fr, setup["ranges"], max_local=MAX_LOCAL)
    c.batch_run(7)
    loc, nl, _, _ = c.batch_fetch_store()
    poses, nm, m, _, summ = c.batch_fetch_track()
    pose, _ = _prior(c, fr)
    for i in (0, N_SCENES + 1):
        s = fr["frames"][i][0]
        mp_map, (k0, p0) = maps[s], offs[s]
        kfs = mp_map["kfs"]
        pw = mp_map["pw"]
        rows = [np.where((kf["feats"]["mp"] >= 0)[:, None], pw[np.maximum(kf["feats"]["mp"], 0)], 0.0) for kf in kfs]
        counts = np.array([len(r) for r in rows], np.int32)
        _, _, local = O.close_keyframes(oc, pose[i], np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int32), counts,
                                        np.stack([kf["pose"][4:] for kf in kfs]), np.concatenate(rows), MAX_LOCAL)
        assert (loc[i][:nl[i]] - k0).tolist() == local.tolist()
        om = OS.OMap()
        for p in pw:
            om.new_mp(p)
        for q in reversed(range(len(kfs))):                      # observations newest first, as the store's chains are walked
            for j, mpj in enumerate(kfs[q]["feats"]["mp"]):
                if mpj >= 0:
                    om.mp_obs[mpj].append((q, j))
        for q, kf in enumerate(kfs):
            of = OS.OracleFrame(mp_map["imgs"][q], kf["pose"])
            F = np.zeros(len(kf["feats"]), O.REF_FEAT_DT)
            F["px"] = kf["feats"]["px"]; F["level"] = kf["feats"]["level"]; F["normal"] = kf["feats"]["normal"]; F["initial"] = 1
            has = kf["feats"]["mp"] >= 0
            F["point_w"][has] = pw[kf["feats"]["mp"][has]]
            of.feats = F
            of.feat_mp = np.where(has & (mp_map["bad"][np.maximum(kf["feats"]["mp"], 0)] == 0), kf["feats"]["mp"], -1)
            om.kfs.append(of)
        cur = OS.OracleFrame(fr["imgs"][i], pose[i])
        out = OS._oracle_search_multi(oc, cam, cur, om, [int(q) for q in local])
        assert nm[i] == len(out)
        assert (m[i]["point"][:nm[i]] - p0).tolist() == [o[0] for o in out]
        assert m[i]["level"][:nm[i]].tolist() == [o[2] for o in out]
        assert np.abs(m[i]["px"][:nm[i]] - np.array([o[1] for o in out])).max() <= 1e-3
        normals = np.array([O.feature_normal(oc, o[1]) for o in out])
        po, _, os_ = O.pose_optimization(normals, np.array([o[2] for o in out], np.int32), pw[[o[0] for o in out]], pose[i], 100)
        d = S.pose_dist(po, poses[i])
        assert d[0] < 1e-5 and d[1] < 1e-5, d
        assert int(os_["termination"]) == int(summ[i]["termination"])


@pytest.mark.slow
def test_scale_4096_frames(setup, built):
    """4096 frames (the 8 base frames tiled, replicas from perturbed start poses, one cur slot each) on the store with every row: whole-
    batch properties on every frame, and on a spread sample of 100 frames the records equal dsdtm_store_track, the matches the
    restatement and the poses dsdtm_pose_optimize_batch (one warp per frame pinned on both sides, option pose_opt_solo_max 0)"""
    cam, maps, fr = setup["cam"], setup["maps"], setup["fr"]
    B = 4096
    c = capi.Context(cam, levels=5, cell_size=15, max_feats=320, max_patches=CPF, max_frames=CUR0 + B, max_batch=B)
    try:
        c.set_option("pose_opt_solo_max", 0)
        SM.load_maps(c, maps)
        base = np.arange(B) % N
        rng = np.random.default_rng(4242)
        start = np.concatenate([rng.uniform(-0.004, 0.004, (B, 3)), rng.uniform(-0.002, 0.002, (B, 3))], 1)
        poses_in = np.stack([S.IDENTITY if g < N else S.pose_from_xi(start[g]) for g in range(B)])
        for g0 in range(0, B, 64):
            c.upload_batch(CUR0 + g0, np.stack([fr["imgs"][base[g]] for g in range(g0, min(g0 + 64, B))]))
        cur_slots = (CUR0 + np.arange(B)).astype(np.int32)
        c.batch_stage(fr["ref_slots"][base], cur_slots, fr["feats"][base], fr["n_feats"][base], fr["centers"][base], poses_in, 5, 0, 8)
        c.batch_stage_store(fr["poses_ref"][base], None, MAX_LOCAL, 2, 10, CPF)
        c.batch_stage_track(None, 100)
        c.batch_run(7)
        loc, nl, rec, nc = c.batch_fetch_store()
        poses, nm, m, res, summ = c.batch_fetch_track()
        poses_c2r, _, _, _ = c.batch_fetch()
        n_kfs = N_SCENES * N_KFS
        assert (nc <= CPF).all() and (nc > 200).all() and (nl >= 1).all() and (nl <= MAX_LOCAL).all()
        assert ((nm >= 20) & (nm <= 200)).all()
        for g in range(B):
            assert ((loc[g][:nl[g]] >= 0) & (loc[g][:nl[g]] < n_kfs)).all() and (loc[g][nl[g]:] == -1).all()
            assert (np.diff(rec[g][:nc[g]]["order"]) > 0).all()
        sample = np.unique(np.linspace(0, B - 1, 100).astype(int))
        pose = [O.se3_mul(poses_c2r[g], fr["poses_ref"][base[g]]) for g in sample]
        pw = np.concatenate([mm["pw"] for mm in maps])
        oc = H.ocam(cam)
        obs = np.zeros((len(sample), 200), capi.BA_OBS_DT)
        for q, g in enumerate(sample):
            _assert_frame_equals_store_track(c, g, pose[q], O.se3_inv(pose[q])[4:], loc, nl, rec, nc)
            r = rec[g][:nc[g]]
            want = [(int(r["mp"][j]), p, lv) for j, p, lv in TS.replay(r["r"], np.ones(nc[g], np.int32), cam["width"], cam["height"], 15)]
            TS.assert_matches_equal(m[g], int(nm[g]), want)
            for k in range(nm[g]):
                obs[q, k]["normal"] = O.feature_normal(oc, m[g, k]["px"]); obs[q, k]["point_w"] = pw[m[g, k]["point"]]
                obs[q, k]["level"] = m[g, k]["level"]
        p2, r2, s2 = c.pose_optimize_batch(obs, nm[sample], np.array(pose), 100)
        assert poses[sample].tobytes() == p2.tobytes() and summ[sample].tobytes() == s2.tobytes()
        for q, g in enumerate(sample):
            assert res[g][:nm[g]].tobytes() == r2[q][:nm[g]].tobytes()
    finally:
        c.close()
