"""GPU suite for dsdtm_batch_commit_store: the batched chain's write-back into the map store (found counts, bad flags, the key frames
of flags 15 with their new points and observation chains) on the device. Its yardsticks are the calls a caller makes without it --
dsdtm_store_set_points, dsdtm_store_append_keyframe per key frame in frame order, dsdtm_store_update_points, dsdtm_store_set_found -- and
tests/store_commit.py's numpy model, which also covers key frames filling reserved rows. Maps come from tests/store_map.py."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import oracle as O
import store_commit as SCM
import store_map as SM
from dsdtm_b200 import capi, synth as S

pytestmark = pytest.mark.gpu

N_SCENES, N_KFS, FRAMES_PER_SCENE = 4, 6, 2
N = N_SCENES * FRAMES_PER_SCENE
CPF = 2048
MAX_LOCAL = 6
CUR0 = N_SCENES * N_KFS


def _context(cam, max_batch=N, extra_slots=0):
    c = capi.Context(cam, levels=5, cell_size=15, max_feats=320, max_patches=CPF, max_frames=CUR0 + N + extra_slots, max_batch=max_batch)
    c.set_option("depth_slots", N)
    return c


def _frames(rs, maps, frames):
    n = len(frames)
    feats = np.zeros((n, 320), capi.REF_FEAT_DT); nf = np.zeros(n, np.int32)
    centers = np.zeros((n, 3)); poses_ref = np.zeros((n, 7)); ref_slots = np.zeros(n, np.int32)
    for i, (s, _) in enumerate(frames):
        feats[i], nf[i] = SM.ref_feats(maps[s], 320)
        last = maps[s]["kfs"][-1]
        centers[i] = last["center"]; poses_ref[i] = last["pose"]; ref_slots[i] = last["slot"]
    return dict(frames=frames, feats=feats, n_feats=nf, centers=centers, poses_ref=poses_ref, ref_slots=ref_slots,
                cur_slots=CUR0 + np.arange(n, dtype=np.int32), imgs=[rs[s]["frames"][f]["img"] for s, f in frames],
                d16=[rs[s]["frames"][f]["d16"] for s, f in frames])


def _load(c, setup, reserve=0):
    """the scenes' maps tiled into c's store, `reserve` empty key frames after each scene's rows (inside its range). Returns the ranges
    per frame and the reserved rows per scene."""
    c.store_clear()
    rows, reserved = [], []
    for m in setup["maps"]:
        k0 = c.store_keyframes
        SM.load_maps(c, [m], clear=False)
        reserved.append([c.store_append_keyframe(0, S.IDENTITY, np.zeros(3), np.zeros(0, capi.STORE_FEAT_DT)) for _ in range(reserve)])
        rows.append((k0, c.store_keyframes))
    for i, d in enumerate(setup["fr"]["d16"]):
        c.depth_upload(i, d)
    return np.array([rows[s] for s, _ in setup["fr"]["frames"]], np.int32), reserved


def _step(c, fr, ranges, flags=15, want=None, cpf=CPF, live=True, found=None):
    n = len(fr["frames"])
    for i in range(n):
        c.upload(int(fr["cur_slots"][i]), fr["imgs"][i])
    c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], np.tile(S.IDENTITY, (n, 1)), 5, 0, 8)
    c.batch_stage_store(fr["poses_ref"], ranges, MAX_LOCAL, 2, 10, cpf)
    if live:
        c.batch_stage_track_live(100)
    else:
        c.batch_stage_track(found, 100)
    if flags & 8:
        c.batch_stage_keyframe(np.arange(n, dtype=np.int32), want, 5.0, 15, 300, (0.0,) * 5, 5000.0)
    c.batch_run(flags)
    return SCM.step_outputs(c, fr["cur_slots"], want, keyframes=bool(flags & 8))


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def setup(request, built):
    cam = dict(getattr(S, request.param))
    rs = SM.render_scenes(cam, [5200 + 31 * k for k in range(N_SCENES)], N_KFS, FRAMES_PER_SCENE)
    c = _context(cam)
    try:
        maps = [SM.build_map(c, cam, rs[s], s * N_KFS) for s in range(N_SCENES)]
    finally:
        c.close()
    fr = _frames(rs, maps, [(s, f) for f in range(FRAMES_PER_SCENE) for s in range(N_SCENES)])
    n_pts = sum(len(m["pw"]) for m in maps)
    found = np.random.default_rng(7).integers(1, 9, n_pts).astype(np.int32)
    st = dict(cam=cam, rs=rs, maps=maps, fr=fr, found=found)
    # the want mask: wanted, unwanted, and one wanted frame whose candidates overflow (n_matches -1)
    c = _context(cam)
    try:
        ranges, _ = _load(c, st)
        o = _step(c, fr, ranges, flags=7)
        nc = c.batch_fetch_store()[3]
    finally:
        c.close()
    # the outlier threshold (LocalBAthreshhold / Camera.f in the tracker): the upper quartile of this step's residual norms, so that the
    # commits below see inliers and outliers
    res = np.concatenate([o["res"][i][:o["nm"][i]] for i in range(N)])
    st["thr"] = np.float32(np.quantile(res, 0.75))
    st["cpf"] = int(np.sort(nc)[-1]) - 1
    st["i_over"] = int(np.argmax(nc))
    want = np.ones(N, bool); want[[1, 6]] = False; want[st["i_over"]] = True
    st["want"] = want
    yield st


def _pair(setup, reserve=0):
    """two contexts holding the same tiled maps and the same found counts (set through store_set_found)"""
    cs = [_context(setup["cam"]) for _ in range(2)]
    for c in cs:
        ranges, reserved = _load(c, setup, reserve)
        c.store_set_found(np.arange(len(setup["found"])), setup["found"])
    return cs, ranges, reserved


def test_commit_equals_host_path(setup):
    """kf_rows NULL: the device commit after a flags-15 step (wanted, unwanted and one overflowed frame) leaves the store byte-equal to
    the existing calls made on the host from the fetched outputs, and to the numpy model; the per-frame outputs agree; two key frames of
    the commit observe a common point, linked newest first"""
    THR = setup["thr"]
    cam, fr = setup["cam"], setup["fr"]
    (a, b), ranges, _ = _pair(setup)
    try:
        oa = _step(a, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        ob = _step(b, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        for k in ("poses", "nm", "m", "res", "n_new", "corners", "lifted"):
            assert oa[k].tobytes() == ob[k].tobytes(), k
        assert oa["nm"][setup["i_over"]] == -1 and (oa["nm"] >= 0).sum() == N - 1
        pre = a.store_fetch()
        l0 = a.launch_count()
        got = a.batch_commit_store(THR)
        assert a.launch_count() == l0 + 4
        want = SCM.host_commit(b, cam, ob, THR)
        ea, eb = a.store_fetch(), b.store_fetch()
        SCM.assert_stores_equal(ea, eb)
        mdl, mout = SCM.model(pre, cam, oa, THR)
        SCM.assert_stores_equal(ea, mdl)
        for x, y, z in zip(got, want, mout):
            assert (x == y).all() and (x == z).all()
        assert (a.store_keyframes, a.store_points) == (b.store_keyframes, b.store_points)
        kf_frames = np.flatnonzero(got[0] >= 0)
        assert set(kf_frames) == set(np.flatnonzero(setup["want"] & (oa["nm"] >= 0))) and len(kf_frames) >= N - 3
        assert (got[2][kf_frames] > 0).all()
        # shared points across key frames of this commit: the chain lists the newer key frame first
        K, F, P, found = ea
        new = F[len(pre[1]):]
        obs_kf = new["is_obs"][new["is_obs"] > 0] - 1
        mp = new["mp"][new["is_obs"] > 0]
        shared = [p for p in np.unique(mp) if len(np.unique(obs_kf[mp == p])) > 1]
        assert shared
        for p in shared[:20]:
            g = int(P["last_obs"][p]); seen = []
            while g >= len(pre[1]):
                seen.append(g); g = int(F["next_obs"][g])
            assert seen == sorted(seen, reverse=True) and len(seen) >= 2
            assert g == int(pre[2]["last_obs"][p])
        # counts moved both ways, and some outliers were erased
        touched = np.unique(np.concatenate([oa["m"][i]["point"][:oa["nm"][i]] for i in range(N) if oa["nm"][i] >= 0]))
        d = found[touched] - pre[3][touched]
        assert (d == 1).any() and (d == 0).any()                 # inliers counted, outliers erased
    finally:
        a.close(); b.close()


def test_reserved_rows_equal_model_and_do_not_change_records(setup):
    """key frames fill the empty rows each scene reserved inside its range: the store equals the numpy model byte for byte (the model
    itself equals the host path in append mode, above); the empty rows inside the ranges change no record, match or pose of a flags-15
    step compared with the same ranges without them"""
    THR = setup["thr"]
    cam, fr = setup["cam"], setup["fr"]
    (a, b), ranges, reserved = _pair(setup, reserve=FRAMES_PER_SCENE)
    try:
        oa = _step(a, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        c = _context(cam)
        try:
            r0, _ = _load(c, setup)
            c.store_set_found(np.arange(len(setup["found"])), setup["found"])
            oc = _step(c, fr, r0, want=setup["want"], cpf=setup["cpf"])
            loc_c, nl_c, rec_c, nc_c = c.batch_fetch_store()
        finally:
            c.close()
        loc_a, nl_a, rec_a, nc_a = a.batch_fetch_store()
        assert rec_a.tobytes() == rec_c.tobytes() and (nl_a == nl_c).all() and (nc_a == nc_c).all()
        shift = {int(r0[i][0]): int(ranges[i][0]) - int(r0[i][0]) for i in range(N)}
        for i in range(N):
            assert (loc_a[i][:nl_a[i]] - shift[int(r0[i][0])] == loc_c[i][:nl_c[i]]).all()
        for k in ("poses", "nm", "m", "res", "n_new", "corners", "lifted"):
            assert oa[k].tobytes() == oc[k].tobytes(), k
        rows = np.array([reserved[s][f] for s, f in fr["frames"]], np.int32)
        pre = a.store_fetch()
        got = a.batch_commit_store(THR, rows)
        mdl, mout = SCM.model(pre, cam, oa, THR, rows)
        SCM.assert_stores_equal(a.store_fetch(), mdl)
        for x, z in zip(got, mout):
            assert (x == z).all()
        assert a.store_keyframes == len(pre[0])
        kf = got[0] >= 0
        assert (got[0][kf] == rows[kf]).all() and (kf == (setup["want"] & (oa["nm"] >= 0))).all()
    finally:
        a.close(); b.close()


def test_next_step_sees_the_commit(setup):
    """after the commit, a step staged with live found counts on the committed store gives records, matches, poses and key frames byte-
    equal to the same step on the host-built store staged with the host-side counts"""
    THR = setup["thr"]
    cam, fr = setup["cam"], setup["fr"]
    (a, b), ranges, _ = _pair(setup)
    try:
        oa = _step(a, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        ob = _step(b, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        a.batch_commit_store(THR)
        SCM.host_commit(b, cam, ob, THR)
        grown = np.array([[r[0], a.store_keyframes] for r in ranges], np.int32)   # every scene also sees the new key frames
        oa2 = _step(a, fr, grown, live=True)
        found_b = b.store_fetch()[3]
        ob2 = _step(b, fr, grown, live=False, found=found_b)
        for k in ("poses", "nm", "m", "res", "n_new", "corners", "lifted"):
            assert oa2[k].tobytes() == ob2[k].tobytes(), k
        ra, rb = a.batch_fetch_store(), b.batch_fetch_store()
        for x, y in zip(ra, rb):
            assert x.tobytes() == y.tobytes()
        assert (ra[1] > MAX_LOCAL // 2).all()
        assert any(oa2["m"][i]["point"][:oa2["nm"][i]].max() >= len(setup["found"]) for i in range(N) if oa2["nm"][i] > 0)
    finally:
        a.close(); b.close()


def test_short_sequence_stays_equal_and_follows_the_oracle(setup):
    """four steps, a key frame every other step (flags 15, 7, 15, 7) into rows each scene reserved inside its range, each step's
    reference frame the last key frame of its frame (chosen here on the host), each step's cur frames in fresh slots (the key frames
    keep theirs): after every commit the device store equals the numpy model, and the frames of the last step match the oracle's chain
    (UpdateLocalMap + SearchLocalPoints on an OMap holding the store's map and found counts as that step saw them, the oracle's
    PoseOptimization)"""
    THR = setup["thr"]
    import oracle_seq as OS
    cam, fr0 = setup["cam"], setup["fr"]
    steps = 4
    c = _context(cam, extra_slots=(steps - 1) * N)
    try:
        ranges, reserved = _load(c, setup, reserve=FRAMES_PER_SCENE * (steps // 2))
        c.store_set_found(np.arange(len(setup["found"])), setup["found"])
        fr = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in fr0.items()}
        for step in range(steps):
            flags = 15 if step % 2 == 0 else 7
            fr["cur_slots"] = (CUR0 + step * N + np.arange(N)).astype(np.int32)
            o = _step(c, fr, ranges, flags=flags)
            rows = np.array([reserved[s][(step // 2) * FRAMES_PER_SCENE + f] for s, f in fr["frames"]], np.int32)
            pre = c.store_fetch()
            got = c.batch_commit_store(THR, rows)
            mdl, mout = SCM.model(pre, cam, o, THR, rows if flags & 8 else None)
            SCM.assert_stores_equal(c.store_fetch(), mdl)
            for x, z in zip(got, mout):
                assert (x == z).all(), step
            if flags & 8:
                assert (got[0] >= 0).sum() == (o["nm"] >= 0).sum() > N // 2
                K, F, P, _ = c.store_fetch()
                for i in np.flatnonzero(got[0] >= 0):             # the key frame becomes the frame's next reference frame
                    r = int(got[0][i])
                    Fk = F[K["feat_begin"][r]:K["feat_begin"][r] + K["feat_count"][r]]
                    q = min(len(Fk), 320)
                    ref = np.zeros(320, capi.REF_FEAT_DT)
                    has = Fk["mp"][:q] >= 0
                    ref["px"][:q] = Fk["px"][:q]; ref["level"][:q] = Fk["level"][:q]; ref["normal"][:q] = Fk["normal"][:q]
                    ref["initial"][:q] = has; ref["point_w"][:q][has] = P["point_w"][Fk["mp"][:q][has]]
                    fr["feats"][i], fr["n_feats"][i] = ref, q
                    fr["centers"][i], fr["poses_ref"][i], fr["ref_slots"][i] = K["center"][r], K["pose_c2w"][r], K["slot"][r]
        # the oracle's chain for two frames of the last step, on the map and counts that step saw (the store before its commit)
        oc = H.ocam(cam)
        K, F, P, found = pre
        loc, nl, _, _ = c.batch_fetch_store()
        poses, nm, m, _, summ = c.batch_fetch_track()
        poses_c2r, _, _, _ = c.batch_fetch()
        for i in (0, N_SCENES + 1):
            pose = O.se3_mul(poses_c2r[i], fr["poses_ref"][i])
            k0, k1 = int(ranges[i][0]), int(ranges[i][1])
            om = OS.OMap()
            for p in P["point_w"]:
                om.new_mp(p)
            om.mp_found = [int(v) for v in found]
            for q in range(k0, k1):
                Fk = F[K["feat_begin"][q]:K["feat_begin"][q] + K["feat_count"][q]]
                of = OS.OracleFrame(c.download_level(int(K["slot"][q]), 0), K["pose_c2w"][q])
                R = np.zeros(len(Fk), O.REF_FEAT_DT)
                R["px"] = Fk["px"]; R["level"] = Fk["level"]; R["normal"] = Fk["normal"]; R["initial"] = 1
                has = Fk["mp"] >= 0
                R["point_w"][has] = P["point_w"][Fk["mp"][has]]
                of.feats = R
                of.feat_mp = np.where(has & (P["bad"][np.maximum(Fk["mp"], 0)] == 0), Fk["mp"], -1)
                om.kfs.append(of)
            for p in np.unique(F["mp"][F["is_obs"] > 0]):              # observations newest first: the store's chain order
                g = int(P["last_obs"][p])
                while g >= 0:
                    kr = int(F["is_obs"][g]) - 1
                    if k0 <= kr < k1:
                        om.mp_obs[p].append((kr - k0, g - int(K["feat_begin"][kr])))
                    g = int(F["next_obs"][g])
            out = OS._oracle_search_multi(oc, cam, OS.OracleFrame(fr["imgs"][i], pose), om, [int(x) - k0 for x in loc[i][:nl[i]]])
            assert nm[i] == len(out) and nm[i] > 20
            assert m[i]["point"][:nm[i]].tolist() == [o_[0] for o_ in out]
            po, _, os_ = O.pose_optimization(np.array([O.feature_normal(oc, o_[1]) for o_ in out]), np.array([o_[2] for o_ in out], np.int32),
                                             P["point_w"][[o_[0] for o_ in out]], pose, 100)
            d = S.pose_dist(po, poses[i])
            assert d[0] < 1e-5 and d[1] < 1e-5, d
            assert int(os_["termination"]) == int(summ[i]["termination"])
    finally:
        c.close()


def test_erase_found_and_bad(setup):
    """the rule as written, with counts of 0 and -1 staged through store_set_found between the run and the commit (the commit applies
    the step to the counts it finds): +1 per match, -1 per outlier (res_norm > threshold, strict), bad when the count ends <= 0; a point
    flagged bad between the run and the commit is not decremented. Every staged point is a match of the step, and the values are checked
    literally, not only against the model"""
    THR = setup["thr"]
    cam, fr = setup["cam"], setup["fr"]
    (a, b), ranges, _ = _pair(setup)
    try:
        o = _step(a, fr, ranges, flags=7)
        pts = [(int(o["m"][i]["point"][k]), o["res"][i][k]) for i in range(N) for k in range(o["nm"][i])]
        count = {}
        for p, _ in pts:
            count[p] = count.get(p, 0) + 1
        once_out = [p for p, r in pts if r > np.float64(THR) and count[p] == 1][:2]
        once_in = [p for p, r in pts if r <= np.float64(THR) and count[p] == 1][:2]
        assert len(once_out) == 2 and len(once_in) == 2
        ids = np.array(once_out + once_in, np.int32)
        staged = np.array([0, 0, -1, 0], np.int32)
        a.store_set_found(ids, staged)
        a.store_update_points(ids[1:2], None, [1])                  # bad before the commit starts: not decremented
        pre = a.store_fetch()
        a.batch_commit_store(THR)
        post = a.store_fetch()
        mdl, _ = SCM.model(pre, cam, o, THR)
        SCM.assert_stores_equal(post, mdl)
        P, f = post[2], post[3]
        # outlier from 0: 0 + 1 - 1 = 0, bad; outlier already bad: 0 + 1, stays bad; inlier from -1: 0, bad; inlier from 0: 1, not bad
        assert f[ids].tolist() == [0, 1, 0, 1]
        assert P["bad"][ids].tolist() == [1, 1, 1, 0]
        assert (pre[2]["bad"][ids] == [0, 1, 0, 0]).all()
    finally:
        a.close(); b.close()


def test_keyframes_sharing_points_chain_newest_first(setup):
    """four frames of one map in one flags-15 commit (scene 0's two frames, each from two start poses): points observed by all four new
    key frames are linked newest first above their old chains, and the whole store equals the host path and the model"""
    THR = setup["thr"]
    cam, fr0 = setup["cam"], setup["fr"]
    idx = [0, N_SCENES, 0, N_SCENES]                             # scene 0's two frames, twice each
    fr = {k: (v[idx] if isinstance(v, np.ndarray) else [v[i] for i in idx]) for k, v in fr0.items()}
    fr["frames"] = [fr0["frames"][i] for i in idx]
    fr["cur_slots"] = (CUR0 + np.arange(4)).astype(np.int32)
    (a, b), ranges, _ = _pair(setup)
    try:
        rng = np.random.default_rng(11)
        start = np.stack([S.IDENTITY] + [S.pose_from_xi(np.r_[rng.uniform(-0.003, 0.003, 3), rng.uniform(-0.002, 0.002, 3)])
                                         for _ in range(3)])
        outs = []
        for c in (a, b):
            for i in range(4):
                c.depth_upload(i, fr["d16"][i])
                c.upload(int(fr["cur_slots"][i]), fr["imgs"][i])
            c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], start, 5, 0, 8)
            c.batch_stage_store(fr["poses_ref"], np.tile(ranges[0], (4, 1)), MAX_LOCAL, 2, 10, CPF)
            c.batch_stage_track_live(100)
            c.batch_stage_keyframe(np.arange(4, dtype=np.int32), None, 5.0, 15, 300, (0.0,) * 5, 5000.0)
            c.batch_run(15)
            outs.append(SCM.step_outputs(c, fr["cur_slots"]))
        assert (outs[0]["nm"] > 0).all()
        pre = a.store_fetch()
        a.batch_commit_store(THR)
        SCM.host_commit(b, cam, outs[1], THR)
        post = a.store_fetch()
        SCM.assert_stores_equal(post, b.store_fetch())
        SCM.assert_stores_equal(post, SCM.model(pre, cam, outs[0], THR)[0])
        K, F, P, _ = post
        f0 = len(pre[1])
        depth = {}
        for p in np.unique(F["mp"][f0:][F["is_obs"][f0:] > 0]):
            g, seen = int(P["last_obs"][p]), []
            while g >= f0:
                seen.append(g); g = int(F["next_obs"][g])
            assert seen == sorted(seen, reverse=True) and g == (int(pre[2]["last_obs"][p]) if p < len(pre[2]) else -1)
            depth[len(seen)] = depth.get(len(seen), 0) + 1
        assert depth.get(4, 0) > 0, depth                       # four-long lists: the merge sort's inner merges run
    finally:
        a.close(); b.close()


def test_errors_leave_the_store_unchanged(setup):
    """every argument and state error returns its code with nothing changed (store_fetch before and after)"""
    THR = setup["thr"]
    cam, fr = setup["cam"], setup["fr"]
    c = _context(cam)
    L, h = c.L, c.hp
    try:
        ranges, reserved = _load(c, setup, reserve=FRAMES_PER_SCENE)
        before = c.store_fetch()

        def commit(rows=None, thr=THR):
            r = None if rows is None else np.ascontiguousarray(rows, np.int32)
            return L.dsdtm_batch_commit_store(h, C.c_float(thr), None if r is None else r.ctypes.data_as(C.c_void_p), None, None, None)

        def same():
            SCM.assert_stores_equal(c.store_fetch(), before)
        assert commit() == -4; same()                                             # nothing run
        _step(c, fr, ranges, flags=3)
        assert commit() == -4; same()                                             # flags 3
        rows = np.array([reserved[s][f] for s, f in fr["frames"]], np.int32)
        _step(c, fr, ranges, want=setup["want"], cpf=setup["cpf"])
        for bad_rows in (np.where(np.arange(N) == 0, 0, rows), np.where(np.arange(N) == 2, rows[0], rows),
                         np.where(np.arange(N) == 3, c.store_keyframes, rows), np.where(np.arange(N) == 4, -1, rows)):
            assert commit(bad_rows) == -1; same()                                 # not empty / twice / outside / negative
        assert commit(rows, np.float32("nan")) == -1; same()
        n0 = c.launch_count()
        assert commit(np.where(setup["want"], rows, 0)) == 0                     # unwanted frames' entries are ignored
        assert c.launch_count() == n0 + 4
        after = c.store_fetch()
        assert commit(rows) == -4                                                 # a second commit
        SCM.assert_stores_equal(c.store_fetch(), after)
        # the one-key-frame mode (flags 7 after dsdtm_batch_stage_map) has no store to commit to
        n = len(fr["frames"])
        c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], np.tile(S.IDENTITY, (n, 1)), 5, 0, 8)
        c.batch_stage_map(fr["poses_ref"], 100, 2, 10)
        c.batch_stage_track(None, 100)
        c.batch_run(7)
        assert commit() == -4
        SCM.assert_stores_equal(c.store_fetch(), after)
        assert L.dsdtm_batch_stage_track_live(h, 100) == -4
        # a store cleared after the run: the step's matches name rows that are gone
        _step(c, fr, ranges, flags=7)
        c.store_clear()
        assert commit() == -4
    finally:
        c.close()


@pytest.mark.slow
def test_scale_4096_frames(setup):
    """4096 frames (the base frames tiled over 512 copies of the scenes' maps, two frames per map copy, from perturbed start poses) with
    flags 15 and every eighth frame unwanted: the device commit equals the host path on the whole store"""
    THR = setup["thr"]
    cam, fr, maps = setup["cam"], setup["fr"], setup["maps"]
    B, copies = 4096, 4096 // N
    cs = [capi.Context(cam, levels=5, cell_size=15, max_feats=320, max_patches=CPF, max_frames=CUR0 + B, max_batch=B) for _ in range(2)]
    try:
        base = np.arange(B) % N
        rng = np.random.default_rng(99)
        start = np.concatenate([rng.uniform(-0.003, 0.003, (B, 3)), rng.uniform(-0.002, 0.002, (B, 3))], 1)
        poses_in = np.stack([S.IDENTITY if g < N else S.pose_from_xi(start[g]) for g in range(B)])
        want = (np.arange(B) % 8) != 5
        outs = []
        for c in cs:
            c.set_option("depth_slots", B)
            offs = SM.load_maps(c, [maps[q % N_SCENES] for q in range(copies * N_SCENES)])
            ranges = np.zeros((B, 2), np.int32)
            for g in range(B):
                k0 = offs[(g // N) * N_SCENES + fr["frames"][base[g]][0]][0]     # copy g // N of the frame's scene map
                ranges[g] = (k0, k0 + N_KFS)
            for g0 in range(0, B, 64):
                c.upload_batch(CUR0 + g0, np.stack([fr["imgs"][base[g]] for g in range(g0, min(g0 + 64, B))]))
                for g in range(g0, min(g0 + 64, B)):
                    c.depth_upload(g, fr["d16"][base[g]])
            cur = (CUR0 + np.arange(B)).astype(np.int32)
            c.batch_stage(fr["ref_slots"][base], cur, fr["feats"][base], fr["n_feats"][base], fr["centers"][base], poses_in, 5, 0, 8)
            c.batch_stage_store(fr["poses_ref"][base], ranges, MAX_LOCAL, 2, 10, CPF)
            c.batch_stage_track_live(100)
            c.batch_stage_keyframe(np.arange(B, dtype=np.int32), want, 5.0, 15, 300, (0.0,) * 5, 5000.0)
            c.batch_run(15)
            outs.append(SCM.step_outputs(c, cur, want))
        for k in ("poses", "nm", "m", "res", "n_new", "lifted"):
            assert outs[0][k].tobytes() == outs[1][k].tobytes(), k
        got = cs[0].batch_commit_store(THR)
        want_rows = SCM.host_commit(cs[1], cam, outs[1], THR)
        SCM.assert_stores_equal(cs[0].store_fetch(), cs[1].store_fetch())
        for x, y in zip(got, want_rows):
            assert (x == y).all()
        assert (got[0] >= 0).sum() == (want & (outs[0]["nm"] >= 0)).sum() > 3000
    finally:
        for c in cs:
            c.close()
