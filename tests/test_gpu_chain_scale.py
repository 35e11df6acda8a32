"""GPU suite of the batched chain at the size it is benchmarked at: dsdtm_batch_run flags 15 (pyramid -> Run -> the refinement chain ->
SearchLocalPoints' selection -> PoseOptimization -> CraeteKeyframe's detection and depth lift) on 4096 pairs of the bench workload
(workload.render_scenes / assemble_batch / upload_frames with the constants of scripts/keyframe_chain_bench.py), against the CPU
references tests/cpp/track_chain_oracle.cpp and tests/cpp/keyframe_chain_oracle.cpp. At 4096 pairs the step runs other kernels and
launch shapes than the 8-pair suites do: PoseOptimization's sweep kernel (the solo kernel only up to the SM count), the throughput
width of sparse alignment, a partial last CTA of track_select_kernel, FAST and the lift at grid rows far past 8. Also here: the
profiling mode against the graph replay and its launch tally, and batches at and past DSDTM_MAX_BATCH_FRAMES (the frame index of the
pyramid, FAST, CLAHE and lift launches is a grid y / z coordinate)."""
import ctypes as C
import os

import numpy as np
import pytest

import helpers as H
import keyframe_chain as KC
import oracle as O
import track_select as TS
from dsdtm_b200 import synth as S
from dsdtm_b200 import workload as W

pytestmark = [pytest.mark.gpu, pytest.mark.slow]

LEVELS, N_FEATS, FEAT_STRIDE, SA, A2D_ITERS, BA_ITERS = 5, 300, 320, (4, 0, 30), 10, 100
CELL, MIN_DIST, MAX_FTS, THR, SCALE = 15, 15, 300, 5.0, 5000.0
PAIRS, SCENES, STARTS = 4096, 8, 8
POSE_TOL, PX_TOL = 1e-5, 1e-3
E_ARG, E_STATE = -1, -4
THREADS = os.cpu_count() or 4
# select CTA boundaries (4 pairs per CTA), the solo / sweep switch at 148 SMs, the throughput width from 592 pairs, the halves, the tail
EDGES = (0, 1, 3, 4, 5, 147, 148, 149, 591, 592, 2047, 2048, 4092, 4093, 4094, 4095)
TRACK = ("poses", "nm", "m", "res", "summ")
KEYFRAME = ("nn", "cr", "lf", "ex")
# launches per stage of one step: the pyramid's count depends on the geometry (EuRoC builds its two small levels in one launch)
PYRAMID_LAUNCHES = {"KINECT": 4, "EUROC": 3}


@pytest.fixture(scope="module", params=["KINECT", "EUROC"])
def chain(request, built):
    from dsdtm_b200 import capi
    cam = dict(getattr(S, request.param))
    ctx = capi.Context(cam, levels=LEVELS, cell_size=CELL, max_feats=FEAT_STRIDE, max_patches=N_FEATS, max_frames=2 * PAIRS, max_batch=PAIRS)
    try:
        ctx.set_option("depth_slots", SCENES)
        scenes = W.render_scenes(SCENES, cam, procs=1)
        b = W.build_batch(ctx, cam, PAIRS, n_scenes=SCENES, n_feats=N_FEATS, feat_stride=FEAT_STRIDE, patches_per_pair=N_FEATS, scenes=scenes)
        d16 = []
        for s, sc in enumerate(scenes):                                     # depth per scene, rendered at the cur pose
            _, z = S.render(S.Scene(sc["seed"]), cam, S.pose_mul(sc["T_c2r"], sc["T_ref"]))
            d16.append(np.clip(np.rint(z * SCALE), 0, 65535).astype(np.uint16))
            ctx.depth_upload(s, d16[-1])
        b.update(name=request.param, cam=cam, oc=H.ocam(cam), d16=np.stack(d16),
                 dist=KC.EUROC_DIST if request.param == "EUROC" else (0.0,) * 5,
                 ref_pyrs=np.stack([O.pyramid(sc["ref_img"], LEVELS)[0] for sc in scenes]),
                 cur_imgs=np.stack([sc["cur_img"] for sc in scenes]))
        # replica classes: pair g = scene g % 8 from start pose (g // 8) % 8, so class g % 64; every class has a member in each of the
        # 64 blocks of 64 pairs (CTA starts, the solo / sweep switch, the tail)
        rng = np.random.default_rng(4096)
        starts = np.stack([S.IDENTITY] + [S.pose_from_xi(np.r_[rng.uniform(-0.004, 0.004, 3), rng.uniform(-0.002, 0.002, 3)])
                                          for _ in range(STARTS - 1)])
        g = np.arange(PAIRS)
        b["cls"] = g % SCENES + SCENES * ((g // SCENES) % STARTS)
        b["poses_replica"] = starts[(g // SCENES) % STARTS]
        yield ctx, b
    finally:
        ctx.close()


def _stage(ctx, b, idx=None, poses=None, want=None):
    """pairs idx of the batch (all, in order, by default) as one staged step; depth slot = the pair's scene"""
    idx = np.arange(PAIRS) if idx is None else np.asarray(idx)
    poses = b["poses_in"] if poses is None else poses
    ctx.batch_stage(b["ref_slots"][idx], b["cur_slots"][idx], b["feats"][idx], b["n_feats"][idx], b["centers"][idx], poses[idx], *SA,
                    None, None, None, A2D_ITERS)
    ctx.batch_stage_map(b["poses_ref"][idx], N_FEATS, LEVELS - 3, A2D_ITERS)
    ctx.batch_stage_track(None, BA_ITERS)
    ctx.batch_stage_keyframe((idx % SCENES).astype(np.int32), want, THR, MIN_DIST, MAX_FTS, b["dist"], SCALE)


def _run(ctx, flags=15):
    ctx.batch_run(flags)
    out = dict(zip(TRACK, ctx.batch_fetch_track()))
    out.update(zip(KEYFRAME, ctx.batch_fetch_keyframe()))
    return out


def _rows(a):
    """one byte row per pair (bit comparisons, NaN included)"""
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).reshape(len(a), -1)


def _zero_past(a, k):
    """rows of a (n, K) record array at or past k[i] are zero bytes"""
    b = np.ascontiguousarray(a).view(np.uint8).reshape(a.shape[0], a.shape[1], -1)
    return not b[np.arange(a.shape[1])[None, :] >= np.asarray(k)[:, None]].any()


def _whole_batch(out):
    nm, nn = out["nm"], out["nn"]
    assert nm.min() >= 0 and nm.max() <= 200 and nm.max() > 50
    assert nn.min() >= 0 and nn.max() <= MAX_FTS and nn.max() > 0
    assert _zero_past(out["m"], nm) and _zero_past(out["res"], nm)
    assert _zero_past(out["cr"], nn) and _zero_past(out["lf"], nn)
    live = np.arange(MAX_FTS)[None, :] < nn[:, None]
    assert np.isin(out["lf"]["status"][live], (KC.LIFT_OK, KC.LIFT_NO_DEPTH)).all()


def _assert_lifted_close(got, want):
    """test_gpu_ingest's bar: undistorted px and depth bit-equal, status equal, normals and points within 1e-12"""
    assert got["px"].tobytes() == want["px"].tobytes()
    assert got["depth"].tobytes() == want["depth"].tobytes() and (got["status"] == want["status"]).all()
    assert np.abs(got["normal"] - want["normal"]).max(initial=0) <= 1e-12
    assert np.abs(got["point_w"] - want["point_w"]).max(initial=0) <= 1e-12


def _check_references(b, out, idx, poses_in):
    """pairs idx (rows idx of out) against the oracle's whole tracked-pose chain and against the CPU key-frame reference fed this run's
    matches and poses. Returns the worst pose difference (rad, m) and the worst lifted-point difference."""
    idx = np.asarray(idx)
    s = idx % SCENES
    o = TS.pair_batch_track(b["oc"], LEVELS, CELL, b["ref_pyrs"][s], b["cur_imgs"][s], b["feats"][idx].astype(O.REF_FEAT_DT), b["n_feats"][idx], b["centers"][idx],
                            b["poses_ref"][idx], poses_in[idx], *SA, N_FEATS, LEVELS - 3, A2D_ITERS, ba_iters=BA_ITERS, n_threads=THREADS)
    nm, m, poses, summ = out["nm"][idx], out["m"][idx], out["poses"][idx], out["summ"][idx]
    assert (nm == o["n_matches"]).all(), idx[nm != o["n_matches"]]
    worst = np.zeros(3)
    for k, i in enumerate(idx):
        n = nm[k]
        assert (m[k]["point"][:n] == o["matches"][k]["point"][:n]).all() and (m[k]["level"][:n] == o["matches"][k]["level"][:n]).all(), i
        assert n == 0 or np.abs(m[k]["px"][:n] - o["matches"][k]["px"][:n]).max() <= PX_TOL, i
        d = S.pose_dist(o["poses"][k], poses[k])
        assert d[0] < POSE_TOL and d[1] < POSE_TOL, (i, d)
        worst[:2] = np.maximum(worst[:2], d)
    bad = (summ["termination"] != o["summaries"]["termination"]) | (summ["iterations"] != o["summaries"]["iterations"])
    assert not bad.any(), idx[bad]
    r = KC.keyframe_chain(b["oc"], LEVELS, CELL, MIN_DIST, MAX_FTS, THR, b["dist"], SCALE, b["cur_imgs"][s], m, nm, poses, b["d16"][s],
                          n_threads=THREADS)
    nn, cr, lf, ex = out["nn"][idx], out["cr"][idx], out["lf"][idx], out["ex"][idx]
    assert (nn == r["n_new"]).all() and (ex == r["tied"]).all(), idx[(nn != r["n_new"]) | (ex != r["tied"])]
    for k, i in enumerate(idx):
        q = nn[k]
        assert KC.same_corners(cr[k][:q], r["corners"][k][:q]), i
        _assert_lifted_close(lf[k][:q], r["lifted"][k][:q])
        worst[2] = max(worst[2], float(np.abs(lf[k]["point_w"][:q] - r["lifted"][k]["point_w"][:q]).max(initial=0)))
    return worst


def test_production_size_against_the_references(chain):
    """flags 15 at 4096 pairs: a spread sample of 100 pairs (the edges of every launch shape + seeded random pairs) against both
    references at the 8-pair suites' bars; on every pair: at most 200 matches, zero rows past n_matches and n_new, valid lift statuses"""
    ctx, b = chain
    _stage(ctx, b)
    out = _run(ctx)
    _whole_batch(out)
    rng = np.random.default_rng(100)
    idx = np.sort(np.r_[EDGES, rng.choice(np.setdiff1d(np.arange(PAIRS), EDGES), 100 - len(EDGES), replace=False)])
    worst = _check_references(b, out, idx, b["poses_in"])
    print("%s: %d pairs against the references; worst pose difference %.3g rad / %.3g m, worst lifted point %.3g m"
          % (b["name"], len(idx), worst[0], worst[1], worst[2]))


def test_replica_classes_cover_every_pair(chain):
    """8 scenes x 8 start poses tiled over 4096 pairs: every pair's flags-15 outputs are bit-equal to its class representative (poses,
    matches, res_norm, summaries, corners, lifted records, exact_path), and the 64 representatives match both references"""
    ctx, b = chain
    _stage(ctx, b, poses=b["poses_replica"])
    out = _run(ctx)
    _whole_batch(out)
    cls = b["cls"]
    reps = np.array([np.flatnonzero(cls == c)[0] for c in range(SCENES * STARTS)])
    for f in TRACK + KEYFRAME:
        r = _rows(out[f])
        bad = (r != r[reps[cls]]).any(1)
        assert not bad.any(), (f, np.flatnonzero(bad)[:16])
    worst = _check_references(b, out, reps, b["poses_replica"])
    print("%s: 64 class representatives against the references; worst pose difference %.3g rad / %.3g m, worst lifted point %.3g m"
          % (b["name"], worst[0], worst[1], worst[2]))


def _assert_rows_equal(got, want, what):
    for f in TRACK + KEYFRAME:
        bad = (_rows(got[f]) != _rows(want[f])).any(1)
        assert not bad.any(), (what, f, np.flatnonzero(bad)[:16])


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_batch_size_and_position_do_not_change_a_pair(chain):
    """with the kernel choices pinned (sparse alignment 3 warps per pair, PoseOptimization's sweep kernel at every size) a pair's
    flags-15 outputs are bit-equal whether it runs in a batch of 1, 3, 5, 148, 149, 593, 4093 (a partial select CTA) or 4096 pairs,
    and in reversed order; a replay after changing pose_opt_solo_max runs the kernel the option names. With the defaults, a batch of
    as many pairs as the GPU has SMs (148 on a B200: the solo kernel, sparse alignment one CTA per SM) and one pair more (the sweep
    kernel, a narrower sparse-alignment width) agree: matches and corners bit-equal, poses and lifted points within 1e-9, the same
    decisions; both sizes match the references (the two sparse-alignment widths round differently)."""
    ctx, b = chain
    sm = _sm_count()
    ctx.set_option("sa_warps_per_pair", 3)
    ctx.set_option("pose_opt_solo_max", 0)
    try:
        _stage(ctx, b)
        full = _run(ctx)
        for n in (1, 3, 5, 148, 149, 593, 4093):
            _stage(ctx, b, idx=np.arange(n))
            _assert_rows_equal(_run(ctx), {f: full[f][:n] for f in full}, n)
        rev = np.arange(PAIRS)[::-1]
        _stage(ctx, b, idx=rev)
        _assert_rows_equal(_run(ctx), {f: full[f][rev] for f in full}, "reversed")
        _stage(ctx, b, idx=np.arange(sm + 1))
        _run(ctx)                                                           # the step is captured with the sweep kernel
        ctx.set_option("pose_opt_solo_max", sm + 1)                         # no re-staging: the next replay must not reuse that graph
        replay = _run(ctx)
        _stage(ctx, b, idx=np.arange(sm + 1))
        _assert_rows_equal(replay, _run(ctx), "replay after pose_opt_solo_max")
        print("%s: %d SMs; solo and sweep poses bit-equal on %d of %d pairs" % (
            b["name"], sm, int((_rows(replay["poses"]) == _rows(full["poses"][:sm + 1])).all(1).sum()), sm + 1))
    finally:
        ctx.set_option("sa_warps_per_pair", 0)
        ctx.set_option("pose_opt_solo_max", -1)
    _stage(ctx, b, idx=np.arange(sm))
    solo = _run(ctx)
    _stage(ctx, b, idx=np.arange(sm + 1))
    sweep = _run(ctx)
    edges = np.array([i for i in EDGES if i <= sm])
    _check_references(b, solo, edges[edges < sm], b["poses_in"])
    _check_references(b, sweep, edges, b["poses_in"])
    sweep = {f: v[:sm] for f, v in sweep.items()}
    for f in ("nm", "m", "nn", "cr", "ex"):
        assert (_rows(solo[f]) == _rows(sweep[f])).all(), f
    for k in ("termination", "iterations", "n_successful", "n_obs"):
        assert (solo["summ"][k] == sweep["summ"][k]).all(), k
    assert (solo["lf"]["status"] == sweep["lf"]["status"]).all()
    assert np.abs(solo["poses"] - sweep["poses"]).max() <= 1e-9
    assert np.abs(solo["lf"]["point_w"] - sweep["lf"]["point_w"]).max() <= 1e-9


def test_sparse_want_masks(chain):
    """about one pair in eight wanted (seeded, plus the first and the last pair): wanted rows bit-equal to the all-wanted run, unwanted
    rows zero, the tracked half unchanged; with no pair wanted, no corners and the flags-7 outputs unchanged"""
    ctx, b = chain
    _stage(ctx, b)
    full = _run(ctx)
    want = (np.random.default_rng(8).random(PAIRS) < 0.125).astype(np.uint8)
    want[0] = want[-1] = 1
    w = want.astype(bool)
    _stage(ctx, b, want=want)
    out = _run(ctx)
    for f in TRACK:
        assert (_rows(out[f]) == _rows(full[f])).all(), f
    for f in KEYFRAME:
        assert (_rows(out[f])[w] == _rows(full[f])[w]).all(), f
        assert not _rows(out[f])[~w].any(), f
    _stage(ctx, b, want=np.zeros(PAIRS, np.uint8))
    out = _run(ctx)
    for f in TRACK:
        assert (_rows(out[f]) == _rows(full[f])).all(), f
    for f in KEYFRAME:
        assert not _rows(out[f]).any(), f


def _fetch(ctx, flags):
    out = [a for a in ctx.batch_fetch() if a is not None]
    if flags & 2:
        out.append(ctx.batch_fetch_map())
    if flags & 4:
        out += list(ctx.batch_fetch_track())
    if flags & 8:
        out += list(ctx.batch_fetch_keyframe())
    return [a.tobytes() for a in out]


def _expected_launches(name, flags, wanted=True):
    e = {"pyramid": PYRAMID_LAUNCHES[name], "sparse_align": 1}
    if flags & 2:
        e.update(local_map=2, warp_affine=1, align2d=2)
    if flags & 4:
        e.update(local_map=3, pose_opt=1)
    if flags & 8:
        e.update(fast=3 if wanted else 2, ingest=1)
    return e


def test_profiling_mode_equals_the_graph(chain):
    """dsdtm_profile(ctx, 1) launches the step directly instead of replaying its graph: for flags 1, 3, 7 and 15 (and 15 with no pair
    wanted) the fetched outputs are byte-identical to the graph replay's, every stage the flags imply reports its launches, and the
    per-stage total equals the dsdtm_launch_count delta of the profiled step and of a graph replay"""
    ctx, b = chain
    for flags, want in ((1, None), (3, None), (7, None), (15, None), (15, np.zeros(PAIRS, np.uint8))):
        _stage(ctx, b, want=want)
        ctx.batch_run(flags)                                                # captures the graph
        l0 = ctx.launch_count()
        ctx.batch_run(flags)
        ctx.sync()
        graph_launches = ctx.launch_count() - l0
        graph = _fetch(ctx, flags)
        ctx.profile(True)
        try:
            ctx.profile_get(reset=True)
            l0 = ctx.launch_count()
            ctx.batch_run(flags)
            stages = ctx.profile_get(reset=True)
            profiled_launches = ctx.launch_count() - l0
        finally:
            ctx.profile(False)
        assert _fetch(ctx, flags) == graph, flags
        per_stage = {k: v[1] for k, v in stages.items() if v[1]}
        assert per_stage == _expected_launches(b["name"], flags, want is None), (flags, per_stage)
        assert all(stages[k][0] > 0 for k in per_stage), (flags, stages)
        assert sum(per_stage.values()) == profiled_launches == graph_launches, (flags, per_stage, profiled_launches, graph_launches)


# ---------------------------------------------------------------------------------------------- batches at the grid limit
TINY = dict(width=64, height=48, fx=60.0, fy=60.0, cx=31.5, cy=23.5, f=60.0)
TINY_LEVELS = 3
LIMIT = 65535                                                               # DSDTM_MAX_BATCH_FRAMES
PROBES = (0, 32767, 65534)
CLAHE_TILES = (8, 6)


@pytest.fixture(scope="module")
def tiny(built):
    """a 64 x 48 camera with 3 levels: 65536 frame slots cost about 300 MB"""
    from dsdtm_b200 import capi
    c = capi.Context(TINY, levels=TINY_LEVELS, cell_size=CELL, max_feats=1, max_patches=1, max_frames=LIMIT + 1, max_batch=LIMIT + 1)
    try:
        rng = np.random.default_rng(LIMIT)
        imgs = np.repeat(np.repeat(rng.integers(0, 256, (LIMIT + 1, 24, 32), dtype=np.uint8), 2, 1), 2, 2)   # 2x2 blocks: corners survive
        yield c, imgs
    finally:
        c.close()


def _assert_pyramid(c, slot, img):
    packed, offs, ws, hs = O.pyramid(img, TINY_LEVELS)
    for l in range(TINY_LEVELS):
        assert (c.download_level(slot, l) == O.pyr_level(packed, offs, ws, hs, l)).all(), (slot, l)


def _cells_equal(a, b):
    return all((a[k] == b[k]).all() for k in ("x", "y", "level")) and (a["score"].view(np.uint32) == b["score"].view(np.uint32)).all()


def test_batches_of_65535_frames(tiny):
    """n = DSDTM_MAX_BATCH_FRAMES: the batched pyramid with each pyramid_kernel (bulk and strip: frame = blockIdx.y; tile: blockIdx.z),
    fast_cells, detect and the CLAHE upload equal the oracle on the first, the middle and the last frame"""
    c, imgs = tiny
    n = LIMIT
    zero = [np.zeros((c.hs[l], c.ws[l]), np.uint8) for l in range(TINY_LEVELS)]
    for k in (0, 1, 2):
        c.set_option("pyramid_kernel", k)
        for i in PROBES:                                                    # a stale pyramid from the previous kernel cannot pass
            for l in range(1, TINY_LEVELS):
                c.upload_level(i, l, zero[l])
        c.upload_batch(0, imgs[:n])
        for i in PROBES:
            _assert_pyramid(c, i, imgs[i])
    c.set_option("pyramid_kernel", 0)
    cells = c.fast_cells(0, 20, 5.0, n=n)
    det, _ = c.detect(0, 5.0, max_new=20, n=n)
    for i in PROBES:
        packed, offs, ws, hs = O.pyramid(imgs[i], TINY_LEVELS)
        want = O.detect_cells(packed, offs, ws, hs, CELL, None, 5.0)
        assert _cells_equal(cells[i], want), i
        sel, _ = O.detect_select(want, np.full((TINY["height"], TINY["width"]), 255, np.uint8), CELL, 20)
        assert len(sel) > 0 and _cells_equal(det[i], sel), i
    eq = c.upload_clahe(0, imgs[:n], 3.0, CLAHE_TILES)
    for i in PROBES:
        want = O.clahe(imgs[i], 3.0, CLAHE_TILES)
        assert (eq[i] == want).all(), i
        _assert_pyramid(c, i, want)


def test_batches_past_the_limit_are_refused(tiny):
    """n = DSDTM_MAX_BATCH_FRAMES + 1 (within max_frames and max_batch): every batched entry whose launches put the frame or pair index
    in gridDim.y / z returns DSDTM_E_ARG naming the limit, before anything is enqueued (the slots keep their content, nothing is
    staged); the context then gives correct results"""
    c, imgs = tiny
    from dsdtm_b200 import capi
    n = LIMIT + 1
    c.upload_batch(0, imgs[1:3])                                            # slot 0 holds frame 1; the refused calls would write frame 0
    before = [c.download_level(0, l).copy() for l in range(TINY_LEVELS)]
    p = capi._p
    L, hp = c.L, c.hp
    slots = np.arange(n, dtype=np.int32)
    feats = np.zeros((n, 1), capi.REF_FEAT_DT)
    nf = np.zeros(n, np.int32)
    centers = np.zeros((n, 3))
    poses = np.tile(S.IDENTITY, (n, 1))
    cells = np.zeros(n * c.n_cells, capi.CORNER_DT)
    max_new = np.full(n, 4, np.int32)
    corners = np.zeros((n, 4), capi.CORNER_DT)
    n_out = np.zeros(n, np.int32)
    poses_out = np.zeros((n, 7))
    n_tracked = np.zeros(n, np.int32)
    reproj = np.zeros(n, capi.REPROJ_DT)
    calls = {
        "dsdtm_frames_upload_pyramid": lambda: L.dsdtm_frames_upload_pyramid(hp, 0, n, p(imgs)),
        "dsdtm_frames_build_pyramid": lambda: L.dsdtm_frames_build_pyramid(hp, 0, n),
        "dsdtm_fast_cells_batch": lambda: L.dsdtm_fast_cells_batch(hp, 0, n, 20, C.c_float(5.0), None, p(cells)),
        "dsdtm_detect_batch": lambda: L.dsdtm_detect_batch(hp, 0, n, C.c_float(5.0), None, None, None, 0, None, p(max_new), 4, p(corners),
                                                           p(n_out), None),
        "dsdtm_frames_upload_clahe_pyramid": lambda: L.dsdtm_frames_upload_clahe_pyramid(hp, 0, n, p(imgs), C.c_double(3.0), CLAHE_TILES[0],
                                                                                         CLAHE_TILES[1], None),
        "dsdtm_batch_stage": lambda: L.dsdtm_batch_stage(hp, n, p(slots), p(slots), p(feats), 1, p(nf), p(centers), p(poses), 2, 0, 10,
                                                         None, None, None, 0, 10),
        "dsdtm_pair_batch_e2e": lambda: L.dsdtm_pair_batch_e2e(hp, n, p(imgs), p(slots), p(slots), p(feats), 1, p(nf), p(centers), p(poses),
                                                               2, 0, 10, None, None, None, 0, 10, p(poses_out), p(n_tracked), None, None),
        "dsdtm_track_batch_e2e": lambda: L.dsdtm_track_batch_e2e(hp, n, p(imgs), p(slots), p(slots), p(feats), 1, p(nf), p(centers), p(poses),
                                                                 p(poses), 2, 0, 10, 1, 0, 10, p(poses_out), p(n_tracked), p(reproj)),
    }
    for name, call in calls.items():
        assert call() == E_ARG, name
        assert b"DSDTM_MAX_BATCH_FRAMES" in L.dsdtm_last_error(hp), (name, L.dsdtm_last_error(hp))
    c.sync()
    for l in range(TINY_LEVELS):
        assert (c.download_level(0, l) == before[l]).all(), l
    assert L.dsdtm_batch_run(hp, 0) == E_STATE                              # the refused dsdtm_batch_stage staged nothing
    c.upload_batch(0, imgs[:3])
    for i in range(3):
        _assert_pyramid(c, i, imgs[i])
    packed, offs, ws, hs = O.pyramid(imgs[2], TINY_LEVELS)
    assert _cells_equal(c.fast_cells(0, 20, 5.0, n=3)[2], O.detect_cells(packed, offs, ws, hs, CELL, None, 5.0))
