"""Host side of the device sequence chain (dsdtm_batch_advance): the next step's reference frame built on the host from a step's fetched
outputs, with the rules dsdtm_batch_advance documents, and rendered trajectories to run sequences on.

A scene's map is built as tests/store_map.py builds it; each of its sequences then renders consecutive frames along its own trajectory,
S.random_motion chained from the last key frame's pose, with depth at scale 5000."""
import multiprocessing as mp
import os

import numpy as np

import oracle as O
from dsdtm_b200 import capi, synth as S
from dsdtm_b200.workload import feature_normals


def _render(args):
    seed, cam, n_kfs, n_seq, n_steps = args
    rng = np.random.default_rng(seed + 99)
    scene = S.Scene(seed)
    T = S.IDENTITY.copy()
    kfs = []
    for k in range(n_kfs):
        if k:
            T = S.pose_mul(S.random_motion(rng, 0.03, 0.8), T)
        img, _, pts = S.render(scene, cam, T, want_points=True)
        kfs.append(dict(pose=T.copy(), img=img, pts=pts))
    seqs = []
    for q in range(n_seq):
        Tc, frames = T.copy(), []
        for _ in range(n_steps):
            Tc = S.pose_mul(S.random_motion(rng, 0.01, 0.3), Tc)
            img, z = S.render(scene, cam, Tc)
            frames.append(dict(pose=Tc.copy(), img=img, d16=np.clip(np.rint(z * 5000.0), 0, 65535).astype(np.uint16)))
        seqs.append(frames)
    return dict(seed=seed, kfs=kfs, seqs=seqs)


def render_sequences(cam, seeds, n_kfs, n_seq, n_steps):
    """per seed: the key frames of its map (n_kfs: one count or one per seed) and n_seq trajectories of n_steps frames each"""
    args = [(s, cam, n_kfs if isinstance(n_kfs, int) else n_kfs[i], n_seq, n_steps) for i, s in enumerate(seeds)]
    procs = min(len(args), max(1, (os.cpu_count() or 2) // 2), 16)
    if procs <= 1:
        return [_render(a) for a in args]
    with mp.get_context("spawn").Pool(procs) as pool:
        return pool.map(_render, args)


def next_ref(cam, staged, out, points_w, next_cur, hold=None, keyframes=False):
    """The staged arrays of the next step, built on the host from this step's staged arrays (dict as batch_fetch_ref returns) and fetched
    outputs (tests/store_commit.py's step_outputs; want = the run's want mask), with the store's point positions after the commit. Frames
    with n_matches -1 or hold[i] keep everything but their cur slot. Returns (arrays, status)."""
    n = len(out["nm"])
    nx = {k: v.copy() for k, v in staged.items()}
    stride = nx["feats"].shape[1]
    status = np.zeros(n, np.uint8)
    for i in range(n):
        nx["cur_slots"][i] = next_cur[i]
        k = int(out["nm"][i])
        if k < 0:
            status[i] = capi.ADV_HELD_OVERFLOW
            continue
        if hold is not None and hold[i]:
            status[i] = capi.ADV_HELD_CALLER
            continue
        kf = keyframes and bool(out["want"][i])
        status[i] = capi.ADV_KEYFRAME if kf else capi.ADV_ADVANCED
        R = np.zeros(stride, capi.REF_FEAT_DT)
        mt = out["m"][i][:k]
        R["px"][:k] = mt["px"]; R["level"][:k] = mt["level"]; R["initial"][:k] = 1
        if k:
            R["normal"][:k] = feature_normals(cam, mt["px"].astype(np.float32))   # the bearing PoseOptimization used
            R["point_w"][:k] = points_w[mt["point"]]
        nf = k
        if kf:
            nn = int(out["n_new"][i])
            lf = out["lifted"][i][:nn]
            ok = lf["status"] == capi.LIFT_OK
            R["px"][k:k + nn] = lf["px"]; R["level"][k:k + nn] = out["corners"][i][:nn]["level"]; R["initial"][k:k + nn] = ok
            R["normal"][k:k + nn] = lf["normal"]
            R["point_w"][k:k + nn] = np.where(ok[:, None], lf["point_w"], 0.0)
            nf += nn
        pose = out["poses"][i]
        nx["feats"][i], nx["n_feats"][i] = R, nf
        nx["ref_slots"][i] = staged["cur_slots"][i]
        nx["poses_ref"][i] = pose
        nx["centers"][i] = O.se3_inv(pose)[4:]
        nx["poses_in"][i] = S.IDENTITY
    return nx, status


def assert_ref_equal(a, b):
    for k in ("ref_slots", "cur_slots", "feats", "n_feats", "centers", "poses_ref", "poses_in"):
        assert a[k].tobytes() == b[k].tobytes(), k
