"""Multi-key-frame maps for the map store, built the way the tracker builds them, and tiled into one store for the batched chain.

A scene's map grows along a short rendered trajectory: key frame 0 is `detect` plus the rendered world points of its corners; every
later key frame first tracks against the map built so far (dsdtm_store_track at the key frame's true pose, then SearchLocalPoints'
selection restated in tests/track_select.py), so its matches observe existing points -- shared points with several observations --
and then detects new corners around them, whose rendered points are new map points. Some new corners get no map point and some new
points are flagged bad. Everything the map holds is kept on the host, so the same map can be loaded into any context, alone or tiled
with other scenes' maps at other row offsets."""
import multiprocessing as mp
import os

import numpy as np

import track_select as TS
from dsdtm_b200 import capi, synth as S
from dsdtm_b200.workload import feature_normals

MAX_FTS = 300
MIN_DIST = 15


def _render_scene(args):
    seed, cam, n_kfs, n_frames = args
    rng = np.random.default_rng(seed + 99)
    scene = S.Scene(seed)
    T = S.IDENTITY.copy()
    kfs = []
    for k in range(n_kfs):
        if k:
            T = S.pose_mul(S.random_motion(rng, 0.03, 0.8), T)
        img, _, pts = S.render(scene, cam, T, want_points=True)
        kfs.append(dict(pose=T.copy(), img=img, pts=pts))
    frames = []
    for _ in range(n_frames):
        Tc = S.pose_mul(S.random_motion(rng, 0.02, 0.5), T)
        img, z = S.render(scene, cam, Tc)
        frames.append(dict(pose=Tc, img=img, d16=np.clip(np.rint(z * 5000.0), 0, 65535).astype(np.uint16)))
    return dict(seed=seed, kfs=kfs, frames=frames)


def render_scenes(cam, seeds, n_kfs, n_frames):
    """renders the key frames (n_kfs: one count, or one per seed) and n_frames later frames of every seed's scene on a process pool"""
    args = [(s, cam, n_kfs if isinstance(n_kfs, int) else n_kfs[i], n_frames) for i, s in enumerate(seeds)]
    procs = min(len(args), max(1, (os.cpu_count() or 2) // 2), 16)
    if procs <= 1:
        return [_render_scene(a) for a in args]
    with mp.get_context("spawn").Pool(procs) as pool:
        return pool.map(_render_scene, args)


def build_map(ctx, cam, rs, slot0, cell_size=15, max_search_level=2):
    """Builds the map of one rendered scene in ctx's (cleared) store, key frame k in slot slot0 + k. Returns the host description:
    dict(pw, bad, kfs = [dict(slot, pose, center, feats STORE_FEAT_DT)], imgs)."""
    ctx.store_clear()
    pw, bad, kfs = [], [], []
    for k, kf in enumerate(rs["kfs"]):
        slot = slot0 + k
        ctx.upload(slot, kf["img"])
        center = S.pose_inv(kf["pose"])[4:]
        feats = []
        circles = []
        if k:
            _, rec = ctx.store_track(slot, kf["pose"], center, 10, max_search_level, 10, cap=8192)
            rec = rec[np.argsort(rec["order"], kind="stable")]
            for j, p, lv in TS.replay(rec["r"], np.ones(len(rec), np.int32), cam["width"], cam["height"], cell_size):
                feats.append((int(rec["mp"][j]), lv, p, 1))
                circles += [(p, cell_size), (p, MIN_DIST)]
        circ = np.zeros(len(circles), capi.CIRCLE_DT)
        for i, (p, r) in enumerate(circles):
            circ[i]["px"] = p; circ[i]["radius"] = r
        new, _ = ctx.detect(slot, 5.0, circles=circ if len(circ) else None, max_new=max(MAX_FTS - len(feats), 1))
        new = new[0][:max(MAX_FTS - len(feats), 0)]
        for i, c in enumerate(new):
            p = np.array([c["x"], c["y"]], np.float32)
            if i % 9 == 4:                                       # a feature without a map point
                feats.append((-1, int(c["level"]), p, 0))
                continue
            feats.append((len(pw), int(c["level"]), p, 1))
            pw.append(kf["pts"][c["y"], c["x"]]); bad.append(1 if len(pw) % 13 == 0 else 0)
        n_old = ctx.store_points
        if len(pw) > n_old:
            ctx.store_set_points(n_old, np.array(pw[n_old:]), np.array(bad[n_old:], np.int32))
        F = np.zeros(len(feats), capi.STORE_FEAT_DT)
        for i, (m, lv, p, obs) in enumerate(feats):
            F[i]["mp"] = m; F[i]["level"] = lv; F[i]["px"] = p; F[i]["is_obs"] = obs
        F["normal"] = feature_normals(cam, F["px"].astype(np.float32))
        ctx.store_append_keyframe(slot, kf["pose"], center, F)
        kfs.append(dict(slot=slot, pose=kf["pose"], center=center, feats=F))
    return dict(pw=np.array(pw), bad=np.array(bad, np.int32), kfs=kfs, imgs=[kf["img"] for kf in rs["kfs"]])


def load_maps(ctx, maps, clear=True):
    """Tiles the host maps into ctx's store (images into their slots). Returns per map (first key-frame row, first point row)."""
    if clear:
        ctx.store_clear()
    offs = []
    for m in maps:
        k0, p0 = ctx.store_keyframes, ctx.store_points
        ctx.store_set_points(p0, m["pw"], m["bad"])
        for kf, img in zip(m["kfs"], m["imgs"]):
            ctx.upload(kf["slot"], img)
            F = kf["feats"].copy()
            F["mp"][F["mp"] >= 0] += p0
            ctx.store_append_keyframe(kf["slot"], kf["pose"], kf["center"], F)
        offs.append((k0, p0))
    return offs


def ref_feats(m, stride):
    """the last key frame's features with map points as the sparse alignment's reference features"""
    F = m["kfs"][-1]["feats"]
    out = np.zeros(stride, capi.REF_FEAT_DT)
    n = min(len(F), stride)
    out["px"][:n] = F["px"][:n]; out["level"][:n] = F["level"][:n]; out["normal"][:n] = F["normal"][:n]
    has = F["mp"][:n] >= 0
    out["initial"][:n] = has
    out["point_w"][:n][has] = m["pw"][F["mp"][:n][has]]
    return out, n
