"""GPU suite for sequences on the device: dsdtm_batch_upload_step -> dsdtm_batch_run -> dsdtm_batch_commit_store -> dsdtm_batch_advance,
each step's frames becoming the next step's reference frames (TrackWithLastFrame). Its yardstick is the host-driven loop -- fetch, the next
reference frame built on the host (tests/sequence_chain.py), restaging, one upload per frame -- and the oracle's chain. Maps come from
tests/store_map.py, one map copy per sequence, with rows reserved inside each copy's range for the key frames the sequence adds."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import oracle as O
import oracle_seq as OS
import sequence_chain as SC
import store_commit as SCM
import store_map as SM
from dsdtm_b200 import capi, synth as S

pytestmark = pytest.mark.gpu

N_SCENES, N_KFS, SEQ_PER_SCENE, STEPS = 4, 6, 2, 8
N = N_SCENES * SEQ_PER_SCENE
CPF, MAX_LOCAL, FEAT_STRIDE = 2048, 6, 320
CUR0 = N_SCENES * N_KFS
THR = np.float32(0.004)                                      # LocalBAthreshhold / Camera.f, in normalised image units
DIST = {"KINECT": (0.0,) * 5, "EUROC": (-0.283408, 0.0739591, 0.00019359, 1.76187e-05, 0.0)}


def _context(cam, steps=STEPS, n=N):
    c = capi.Context(cam, levels=5, cell_size=15, max_feats=FEAT_STRIDE, max_patches=CPF, max_frames=CUR0 + (steps + 2) * n, max_batch=n)
    c.set_option("depth_slots", n)
    return c


def _scenes(cam, steps, n_scenes=N_SCENES):
    rs = SC.render_sequences(cam, [6100 + 37 * k for k in range(n_scenes)], N_KFS, SEQ_PER_SCENE, steps)
    c = _context(cam, steps, n_scenes * SEQ_PER_SCENE)
    try:
        maps = [SM.build_map(c, cam, rs[s], s * N_KFS) for s in range(n_scenes)]
    finally:
        c.close()
    return rs, maps


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def setup(request, built):
    cam = dict(getattr(S, request.param))
    rs, maps = _scenes(cam, STEPS)
    return dict(cam=cam, rs=rs, maps=maps, dist=DIST[request.param], n_scenes=N_SCENES)


def _frames(st):
    """frame i = sequence (i // n_scenes) % SEQ_PER_SCENE of scene i % n_scenes, on its own map copy i; st["tile"] (default 1) repeats
    the n_scenes x SEQ_PER_SCENE sequences that many times"""
    n_sc = st["n_scenes"]
    return [(i % n_sc, i // n_sc) for i in range(n_sc * SEQ_PER_SCENE)] * st.get("tile", 1)


def _load(c, st, reserve):
    """one map copy per frame, `reserve` empty key frames after each copy's rows (inside its range). -> ranges, reserved rows per frame"""
    c.store_clear()
    ranges, reserved = [], []
    for s, _ in _frames(st):
        k0 = c.store_keyframes
        SM.load_maps(c, [st["maps"][s]], clear=False)
        reserved.append([c.store_append_keyframe(0, S.IDENTITY, np.zeros(3), np.zeros(0, capi.STORE_FEAT_DT)) for _ in range(reserve)])
        ranges.append((k0, c.store_keyframes))
    c.depth_upload(0, st["rs"][0]["seqs"][0][0]["d16"])         # the depth pool exists before the key-frame half names its slots
    return np.array(ranges, np.int32), reserved


def _first(st, n):
    fr = dict(ref_slots=np.zeros(n, np.int32), cur_slots=(CUR0 + np.arange(n)).astype(np.int32), feats=np.zeros((n, FEAT_STRIDE), capi.REF_FEAT_DT),
              n_feats=np.zeros(n, np.int32), centers=np.zeros((n, 3)), poses_ref=np.zeros((n, 7)), poses_in=np.tile(S.IDENTITY, (n, 1)))
    for i, (s, _) in enumerate(_frames(st)):
        m = st["maps"][s]
        fr["feats"][i], fr["n_feats"][i] = SM.ref_feats(m, FEAT_STRIDE)
        last = m["kfs"][-1]
        fr["centers"][i] = last["center"]; fr["poses_ref"][i] = last["pose"]; fr["ref_slots"][i] = last["slot"]
    return fr


def _images(st, k):
    cache = st.setdefault("images", {})
    if k not in cache:
        cache.clear()                                            # one step's images at a time (3.8 GB at 4096 frames)
        fs = [st["rs"][s]["seqs"][q][k] for s, q in _frames(st)]
        cache[k] = (np.stack([f["img"] for f in fs]), np.stack([f["d16"] for f in fs]))
    return cache[k]


def _stage(c, st, fr, ranges, want, cpf=CPF, feat_stride=FEAT_STRIDE):
    n = len(fr["ref_slots"])
    c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"][:, :feat_stride], fr["n_feats"], fr["centers"], fr["poses_in"], 5, 0, 8)
    c.batch_stage_store(fr["poses_ref"], ranges, MAX_LOCAL, 2, 10, cpf)
    c.batch_stage_track_live(100)
    c.batch_stage_keyframe(np.arange(n, dtype=np.int32), want, 5.0, 15, 300, st["dist"], 5000.0)


def _outputs(c, cur_slots, want, flags):
    o = SCM.step_outputs(c, cur_slots, want, keyframes=bool(flags & 8))
    o["n_tracked"] = c.batch_fetch()[1]
    return o


def _next_cur(k, n, reverse=False):
    """the cur slots of step k + 1: block k + 1 of the pool, in frame order or reversed (then dsdtm_batch_upload_step copies frame by
    frame instead of in one strided copy)"""
    j = np.arange(n)
    return (CUR0 + (k + 1) * n + (n - 1 - j if reverse else j)).astype(np.int32)


def _host_step(c, st, fr, ranges, want, flags, rows, k, cpf=CPF, hold=None, next_cur=None):
    """today's loop: one upload per frame, restaging, run, fetch, commit, the next reference frame built on the host"""
    imgs, d16 = _images(st, k)
    for i in range(len(imgs)):
        c.upload(int(fr["cur_slots"][i]), imgs[i])
        c.depth_upload(i, d16[i])
    _stage(c, st, fr, ranges, want, cpf)
    c.batch_run(flags)
    o = _outputs(c, fr["cur_slots"], want, flags)
    c.batch_commit_store(THR, rows if flags & 8 else None)
    nxt = _next_cur(k, len(imgs)) if next_cur is None else next_cur
    nx, status = SC.next_ref(st["cam"], fr, o, c.store_fetch()[2]["point_w"], nxt, hold, keyframes=bool(flags & 8))
    return o, nx, status


def _device_step(c, st, want, want_next, flags, rows, k, hold=None, next_cur=None):
    """upload_step -> run -> commit -> advance; want = the mask the run reads (the staged one, or the last want_next)"""
    imgs, d16 = _images(st, k)
    c.batch_upload_step(imgs, d16)
    c.batch_run(flags)
    o = _outputs(c, c.batch_fetch_ref()["cur_slots"], want, flags)
    c.batch_commit_store(THR, rows if flags & 8 else None)
    status = c.batch_advance(_next_cur(k, len(imgs)) if next_cur is None else next_cur, hold, want_next)
    return o, status


def _wants(steps, n, seed=5):
    rng = np.random.default_rng(seed)
    return [rng.random(n) < 0.7 for _ in range(steps + 1)]


def _rows(reserved, step_kf):
    return np.array([r[step_kf] for r in reserved], np.int32)


def test_equals_host_driven_loop(setup):
    """8 steps, flags 15 / 7 alternating, the want mask changing every step: after every step the staged inputs (batch_fetch_ref), the
    step's outputs and the whole store are byte-equal between the device chain and the host-driven loop"""
    st = setup
    wants = _wants(STEPS, N)
    a, b = _context(st["cam"]), _context(st["cam"])
    try:
        ranges, reserved = _load(a, st, STEPS // 2)
        _load(b, st, STEPS // 2)
        fr = _first(st, N)
        _stage(a, st, fr, ranges, wants[0])
        for k in range(STEPS):
            flags = 15 if k % 2 == 0 else 7
            rows = _rows(reserved, k // 2)
            nxt = _next_cur(k, N, reverse=k % 3 == 1)            # every third step's cur slots are not contiguous
            ob, fr, sb = _host_step(b, st, fr, ranges, wants[k], flags, rows, k, next_cur=nxt)
            oa, sa = _device_step(a, st, wants[k], wants[k + 1], flags, rows, k, next_cur=nxt)
            for key in ob:
                if isinstance(ob[key], np.ndarray):
                    assert oa[key].tobytes() == ob[key].tobytes(), (k, key)
            SCM.assert_stores_equal(a.store_fetch(), b.store_fetch())
            assert (sa == sb).all(), k
            SC.assert_ref_equal(a.batch_fetch_ref(), fr)
            if flags & 8:
                assert (sa == capi.ADV_KEYFRAME).sum() == (wants[k] & (ob["nm"] >= 0)).sum() > 0
            assert (ob["nm"] > 20).sum() >= N // 2, k
        # the host loop's own staging of the next step reads back what the host built
        _stage(b, st, fr, ranges, wants[STEPS])
        SC.assert_ref_equal(b.batch_fetch_ref(), a.batch_fetch_ref())
    finally:
        a.close(); b.close()


def test_follows_the_oracle(setup):
    """two frames of the last of four steps (flags 15, 7, 15, 7): sparse alignment against the last frame, UpdateLocalMap +
    SearchLocalPoints on an OMap of the store as that step saw it, and PoseOptimization, each against the oracle"""
    st = setup
    cam = st["cam"]
    steps = 4
    c = _context(cam)
    try:
        ranges, reserved = _load(c, st, steps // 2)
        fr = _first(st, N)
        _stage(c, st, fr, ranges, None)
        for k in range(steps):
            flags = 15 if k % 2 == 0 else 7
            if k == steps - 1:
                ref = fr                                         # the last frame as the host builds it (tests/sequence_chain.py)
                pre = c.store_fetch()
                ref_imgs = _images(st, k - 1)[0].copy()
                imgs = _images(st, k)[0].copy()
            o, _ = _device_step(c, st, None, None, flags, _rows(reserved, k // 2), k)
            fr, _ = SC.next_ref(cam, fr, o, c.store_fetch()[2]["point_w"], _next_cur(k, N), keyframes=bool(flags & 8))
        oc = H.ocam(cam)
        K, F, P, found = pre
        # the outputs of the last run are still the context's (advance rewrites only the staged inputs)
        loc, nl, _, _ = c.batch_fetch_store()
        poses, nm, m, _, summ = c.batch_fetch_track()
        poses_c2r, n_tracked, _, _ = c.batch_fetch()
        for i in (0, N_SCENES + 1):
            rf = OS.OracleFrame(ref_imgs[i], ref["poses_ref"][i])
            rf.feats = ref["feats"][i][:ref["n_feats"][i]].astype(O.REF_FEAT_DT)
            po, n_o = OS._oracle_sparse_align(oc, OS.OracleFrame(imgs[i], ref["poses_ref"][i]), rf, (5, 0, 8))
            pose = O.se3_mul(poses_c2r[i], ref["poses_ref"][i])
            d = S.pose_dist(po, pose)
            assert d[0] < 1e-5 and d[1] < 1e-5 and n_o == n_tracked[i], (d, n_o, n_tracked[i])
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
            for p in np.unique(F["mp"][F["is_obs"] > 0]):
                g = int(P["last_obs"][p])
                while g >= 0:
                    kr = int(F["is_obs"][g]) - 1
                    if k0 <= kr < k1:
                        om.mp_obs[p].append((kr - k0, g - int(K["feat_begin"][kr])))
                    g = int(F["next_obs"][g])
            out = OS._oracle_search_multi(oc, cam, OS.OracleFrame(imgs[i], pose), om, [int(x) - k0 for x in loc[i][:nl[i]]])
            assert nm[i] == len(out) and nm[i] > 20
            assert m[i]["point"][:nm[i]].tolist() == [o_[0] for o_ in out]
            po, _, os_ = O.pose_optimization(np.array([O.feature_normal(oc, o_[1]) for o_ in out]), np.array([o_[2] for o_ in out], np.int32),
                                             P["point_w"][[o_[0] for o_ in out]], pose, 100)
            d = S.pose_dist(po, poses[i])
            assert d[0] < 1e-5 and d[1] < 1e-5, d
            assert int(os_["termination"]) == int(summ[i]["termination"])
    finally:
        c.close()


def test_tracks_the_trajectory(built):
    """kinect, 8 sequences x 16 steps, a key frame every 4th step: every tracked pose is within 1e-3 / 3e-3 of the rendered trajectory,
    no frame is held and every frame keeps at least 100 matches"""
    cam, steps = dict(S.KINECT), 16
    rs, maps = _scenes(cam, steps)
    st = dict(cam=cam, rs=rs, maps=maps, dist=DIST["KINECT"], n_scenes=N_SCENES)
    c = _context(cam, steps)
    try:
        ranges, reserved = _load(c, st, steps // 4)
        _stage(c, st, _first(st, N), ranges, None)
        for k in range(steps):
            flags = 15 if k % 4 == 3 else 7
            o, status = _device_step(c, st, None, None, flags, _rows(reserved, k // 4), k)
            assert (status <= capi.ADV_KEYFRAME).all() and (o["nm"] >= 100).all(), (k, status, o["nm"])
            for i, (s, q) in enumerate(_frames(st)):
                e = S.pose_dist(o["poses"][i], rs[s]["seqs"][q][k]["pose"])
                assert e[0] < 1e-3 and e[1] < 3e-3, (k, i, e)
    finally:
        c.close()


def test_hold_and_want_next(setup):
    """a frame whose candidates overflow and a frame the caller holds keep their reference byte for byte (only the cur slot moves), the
    other frames equal a run without the hold, and the held frame tracks at the next step; want_next changes what the next flags-15 step
    detects and nothing else"""
    st = setup
    cam = st["cam"]
    probe = _context(cam)
    try:
        ranges, _ = _load(probe, st, 1)
        _stage(probe, st, _first(st, N), ranges, None)
        probe.upload_batch(CUR0, _images(st, 0)[0])
        probe.batch_run(7)
        nc = probe.batch_fetch_store()[3]
    finally:
        probe.close()
    cpf, i_over = int(nc.max()) - 1, int(np.argmax(nc))
    i_hold = (i_over + 1) % N
    hold = np.arange(N) == i_hold
    a, b = _context(cam), _context(cam)
    try:
        for c in (a, b):
            ranges, reserved = _load(c, st, 1)
            _stage(c, st, _first(st, N), ranges, None, cpf)
        r0 = a.batch_fetch_ref()
        oa, sa = _device_step(a, st, None, None, 7, None, 0, hold=hold)
        ob, sb = _device_step(b, st, None, None, 7, None, 0)
        assert sa[i_over] == sb[i_over] == capi.ADV_HELD_OVERFLOW and oa["nm"][i_over] == -1
        assert sa[i_hold] == capi.ADV_HELD_CALLER and sb[i_hold] == capi.ADV_ADVANCED
        ra, rb = a.batch_fetch_ref(), b.batch_fetch_ref()
        for i in (i_over, i_hold):
            for key in ("ref_slots", "feats", "n_feats", "centers", "poses_ref", "poses_in"):
                assert ra[key][i].tobytes() == r0[key][i].tobytes(), (i, key)
            assert ra["cur_slots"][i] == _next_cur(0, N)[i]
        other = ~hold
        for key in ra:
            assert ra[key][other].tobytes() == rb[key][other].tobytes(), key
        # the next step: the held frame tracks against its old reference; the two contexts pass different want_next masks
        want = np.ones(N, bool); want[::2] = False
        oa, _ = _device_step(a, st, None, np.ones(N, bool), 7, None, 1)
        _device_step(b, st, None, want, 7, None, 1)
        assert oa["nm"][i_hold] > 20 and oa["n_tracked"][i_hold] > 20
        rows = _rows(reserved, 0)
        oa, _ = _device_step(a, st, np.ones(N, bool), None, 15, rows, 2)
        ob, _ = _device_step(b, st, want, None, 15, rows, 2)
        for key in ("poses", "nm", "m", "res", "n_tracked"):
            assert oa[key][other].tobytes() == ob[key][other].tobytes(), key
        tracked = other & (ob["nm"] >= 0)
        assert (ob["n_new"][~want] == 0).all() and (ob["n_new"][want & tracked] == oa["n_new"][want & tracked]).all()
        assert (oa["n_new"][~want & tracked] > 0).any()
    finally:
        a.close(); b.close()


def test_replays(setup):
    """six flags-7 steps with advance capture once; a want_next change keeps the flags-7 capture; a replay after advance equals the same
    step on a freshly staged context; each advance is one launch; a commit that writes key frames makes the next flags-7 run and the next
    flags-15 run capture again, a commit without key frames does not"""
    st = setup
    cam = st["cam"]
    a = _context(cam)
    try:
        ranges, reserved = _load(a, st, 1)
        _stage(a, st, _first(st, N), ranges, None)
        g0 = a.graph_captures()
        for k in range(6):
            imgs, d16 = _images(st, k)
            a.batch_upload_step(imgs, d16)
            a.batch_run(7)
            a.batch_commit_store(THR)
            l0 = a.launch_count()
            a.batch_advance(_next_cur(k, N), None, (np.arange(N) % 3 != k % 3) if k == 4 else None)
            assert a.launch_count() == l0 + 1
        assert a.graph_captures() == g0 + 1
        # the same step on a fresh context staged from what the advance left
        ref, (K, F, P, found) = a.batch_fetch_ref(), a.store_fetch()
        b = _context(cam)
        try:
            _load(b, st, 1)
            b.store_set_found(np.arange(len(found)), found)
            b.store_update_points(np.arange(len(P)), None, P["bad"])
            SCM.assert_stores_equal(b.store_fetch(), (K, F, P, found))
            fr = {k: ref[k] for k in ref}
            imgs, d16 = _images(st, 6)
            for i in range(N):
                b.upload(int(fr["cur_slots"][i]), imgs[i])
                r = int(fr["ref_slots"][i])
                if r >= CUR0:                                 # slot CUR0 + j * N + i holds the cur frame of step j
                    b.upload(r, _images(st, (r - CUR0) // N)[0][(r - CUR0) % N])
            _stage(b, st, fr, ranges, np.arange(N) % 3 != 1)
            b.batch_run(7)
            ob = _outputs(b, fr["cur_slots"], None, 7)
        finally:
            b.close()
        a.batch_upload_step(imgs, d16)
        a.batch_run(7)
        assert a.graph_captures() == g0 + 1
        oa = _outputs(a, fr["cur_slots"], None, 7)
        for key in ("poses", "nm", "m", "res", "n_tracked"):
            assert oa[key].tobytes() == ob[key].tobytes(), key
        a.batch_commit_store(THR)
        a.batch_advance(_next_cur(6, N))
        a.batch_upload_step(*_images(st, 7))
        a.batch_run(15)                                          # the first flags-15 run of the context
        assert a.graph_captures() == g0 + 2
        kf = a.batch_commit_store(THR, _rows(reserved, 0))[0]   # writes key frames: the captured steps are dropped
        assert (kf >= 0).sum() > 0
        a.batch_advance(_next_cur(7, N))
        a.batch_upload_step(*_images(st, 7))                     # the same images again: the frames track against themselves
        a.batch_run(7)
        assert a.graph_captures() == g0 + 3                      # flags 7 captured again
        a.batch_commit_store(THR)                                # no key frame: the captures stay
        a.batch_advance(_next_cur(8, N))
        a.batch_upload_step(*_images(st, 7))
        a.batch_run(7)
        assert a.graph_captures() == g0 + 3
        a.batch_run(15)
        assert a.graph_captures() == g0 + 4                      # flags 15 captured again after the key-frame commit
    finally:
        a.close()


def test_errors_leave_everything_unchanged(setup):
    """every state and argument error of dsdtm_batch_advance and dsdtm_batch_upload_step returns its code with the staged inputs, the
    store and the captures unchanged; a valid advance still follows"""
    st = setup
    cam = st["cam"]
    c = _context(cam)
    L, h = c.L, c.hp
    try:
        assert L.dsdtm_batch_upload_step(h, _images(st, 0)[0].ctypes.data_as(C.c_void_p), None) == -4      # nothing staged
        ranges, reserved = _load(c, st, 1)
        fr = _first(st, N)
        c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], fr["poses_in"], 5, 0, 8)
        c.batch_stage_store(fr["poses_ref"], ranges, MAX_LOCAL, 2, 10, CPF)
        c.batch_stage_track_live(100)
        d16 = _images(st, 0)[1]
        assert L.dsdtm_batch_upload_step(h, _images(st, 0)[0].ctypes.data_as(C.c_void_p), d16.ctypes.data_as(C.c_void_p)) == -4  # no depth slots

        def adv(nxt, hold=None, want=None):
            nx = np.ascontiguousarray(nxt, np.int32)
            p = lambda x: None if x is None else np.ascontiguousarray(x, np.uint8).ctypes.data_as(C.c_void_p)
            return L.dsdtm_batch_advance(h, nx.ctypes.data_as(C.c_void_p), p(hold), p(want), None)

        def snap():
            return c.batch_fetch_ref(), c.store_fetch(), c.graph_captures(), c.launch_count()

        def same(s0):
            s1 = snap()
            SC.assert_ref_equal(s1[0], s0[0])
            SCM.assert_stores_equal(s1[1], s0[1])
            assert s1[2:] == s0[2:]
        nxt = _next_cur(0, N)
        s0 = snap()
        assert adv(nxt) == -4; same(s0)                                           # no run
        c.batch_upload_step(_images(st, 0)[0])
        c.batch_run(3)
        s0 = snap()
        assert adv(nxt) == -4; same(s0)                                           # flags 3: nothing to commit
        c.batch_run(7)
        s0 = snap()
        assert adv(nxt) == -4; same(s0)                                           # no commit
        c.batch_commit_store(THR)
        s0 = snap()
        assert adv(nxt, want=np.ones(N)) == -4; same(s0)                          # want_next without the key-frame half
        kf_slot = int(st["maps"][0]["kfs"][0]["slot"])
        for bad in (np.where(np.arange(N) == 0, -1, nxt), np.where(np.arange(N) == 1, c.prm.max_frames, nxt),
                    np.where(np.arange(N) == 2, nxt[3], nxt), np.where(np.arange(N) == 4, kf_slot, nxt),
                    np.where(np.arange(N) == 5, CUR0, nxt)):                      # outside / twice / a key frame's / a reference slot after
            assert adv(bad) == -1; same(s0)
        held = np.arange(N) == 0
        assert adv(np.where(held, CUR0 + 1, nxt), hold=held) == -1; same(s0)     # frame 1's cur slot becomes its reference slot
        assert adv(np.where(held, CUR0, nxt), hold=held) == 0                    # frame 0's own old cur slot is free when it is held
        s0 = snap()
        assert adv(nxt + N) == -4; same(s0)                                       # a second advance
        # a feature stride below DSDTM_TRACK_MAX_MATCHES
        c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"][:, :150], np.minimum(fr["n_feats"], 150), fr["centers"], fr["poses_in"], 5, 0, 8)
        c.batch_stage_store(fr["poses_ref"], ranges, MAX_LOCAL, 2, 10, CPF)
        c.batch_stage_track_live(100)
        c.batch_run(7)
        c.batch_commit_store(THR)
        s0 = snap()
        assert adv(nxt) == -1; same(s0)
        # the one-key-frame mode has no store to advance on
        c.batch_stage(fr["ref_slots"], fr["cur_slots"], fr["feats"], fr["n_feats"], fr["centers"], fr["poses_in"], 5, 0, 8)
        c.batch_stage_map(fr["poses_ref"], 100, 2, 10)
        c.batch_stage_track(None, 100)
        c.batch_run(7)
        s0 = snap()
        assert adv(nxt) == -4; same(s0)
    finally:
        c.close()


@pytest.mark.slow
def test_scale_4096_frames_equals_host_driven_loop(built):
    """kinect, 4096 sequences (the 8 rendered sequences tiled over 4096 map copies) x 4 steps, flags 15 / 7, the want mask changing every
    step, every step's cur slots reversed (the upload copies frame by frame): after every step the staged inputs, the step's outputs, the
    advance status and the whole store are byte-equal between the device chain and the host-driven loop"""
    cam, steps, n = dict(S.KINECT), 4, 4096
    rs, maps = _scenes(cam, steps)
    st = dict(cam=cam, rs=rs, maps=maps, dist=DIST["KINECT"], n_scenes=N_SCENES, tile=n // N)
    wants = _wants(steps, n, seed=9)
    a, b = _context(cam, steps, n), _context(cam, steps, n)
    try:
        ranges, reserved = _load(a, st, steps // 2)
        _load(b, st, steps // 2)
        fr = _first(st, n)
        _stage(a, st, fr, ranges, wants[0])
        for k in range(steps):
            flags = 15 if k % 2 == 0 else 7
            rows = _rows(reserved, k // 2)
            nxt = _next_cur(k, n, reverse=True)
            ob, fr, sb = _host_step(b, st, fr, ranges, wants[k], flags, rows, k, next_cur=nxt)
            oa, sa = _device_step(a, st, wants[k], wants[k + 1], flags, rows, k, next_cur=nxt)
            for key in ob:
                if isinstance(ob[key], np.ndarray):
                    assert oa[key].tobytes() == ob[key].tobytes(), (k, key)
            SCM.assert_stores_equal(a.store_fetch(), b.store_fetch())
            assert (sa == sb).all(), k
            SC.assert_ref_equal(a.batch_fetch_ref(), fr)
            assert (ob["nm"] > 20).sum() > n // 2, k
            if flags & 8:
                assert (sa == capi.ADV_KEYFRAME).sum() == (wants[k] & (ob["nm"] >= 0)).sum() > n // 2
    finally:
        a.close(); b.close()
