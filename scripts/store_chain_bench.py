"""The batched chain on the map store (dsdtm_batch_stage_store) against the one-key-frame local map (dsdtm_batch_stage_map), on the same
frames: 8 rendered scenes, each with a map of 8 to 10 key frames built by tests/store_map.py (detect, store_track + SearchLocalPoints'
selection, new corners with new points), tiled into one store with per-frame key-frame ranges; 4096 frames per camera (kinect 640x480
and EuRoC 752x480), frame g tracking a cur image of scene g % 8 against that scene's last key frame (Sprase_ImgAlign(4,0,30), Align2D 10
iterations, PoseOptimization 100 iterations, UpdateLocalMap's ten nearest key frames). Replicas start from perturbed poses, as in the
bench workload. Flags 3 and 7 of both modes run on two contexts and are alternated step by step in one process (CUDA events,
dsdtm_last_run_ms); the per-stage split comes from a separate profiling run. Reports ms per step, frames per second, local key frames,
candidates and matches per frame. The GPU name and power limit are read in the same run (nvidia-smi query only). Writes one JSON file."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LEVELS, FEAT_STRIDE, SA, A2D_ITERS, BA_ITERS, MAX_LOCAL = 5, 320, (4, 0, 30), 10, 100, 10
N_SCENES, FRAMES_PER_SCENE = 8, 2


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def run_cam(name, frames, steps, cpf):
    import store_map as SM
    from dsdtm_b200 import capi, synth as S
    cam = dict(getattr(S, name))
    n_kfs = [8 + s % 3 for s in range(N_SCENES)]
    kf_slot0 = np.concatenate([[0], np.cumsum(n_kfs)])
    cur0 = int(kf_slot0[-1])
    rs = SM.render_scenes(cam, [5200 + 31 * s for s in range(N_SCENES)], n_kfs, FRAMES_PER_SCENE)
    mk = lambda: capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=cpf, max_frames=cur0 + frames,
                              max_batch=frames)
    cs, cm = mk(), mk()
    try:
        maps = [SM.build_map(cs, cam, rs[s], int(kf_slot0[s])) for s in range(N_SCENES)]
        offs = SM.load_maps(cs, maps)
        for s in range(N_SCENES):
            for kf, img in zip(maps[s]["kfs"], maps[s]["imgs"]):
                cm.upload(kf["slot"], img)
        scene = np.arange(frames) % N_SCENES
        which = (np.arange(frames) // N_SCENES) % FRAMES_PER_SCENE
        feats = np.zeros((frames, FEAT_STRIDE), capi.REF_FEAT_DT); nf = np.zeros(frames, np.int32)
        per = [SM.ref_feats(m, FEAT_STRIDE) for m in maps]
        for g in range(frames):
            feats[g], nf[g] = per[scene[g]]
        last = [m["kfs"][-1] for m in maps]
        centers = np.stack([last[s]["center"] for s in scene]); poses_ref = np.stack([last[s]["pose"] for s in scene])
        ref_slots = np.array([last[s]["slot"] for s in scene], np.int32)
        cur_slots = (cur0 + np.arange(frames)).astype(np.int32)
        rng = np.random.default_rng(4242)
        start = np.concatenate([rng.uniform(-0.004, 0.004, (frames, 3)), rng.uniform(-0.002, 0.002, (frames, 3))], 1)
        poses_in = np.stack([S.IDENTITY if g < N_SCENES * FRAMES_PER_SCENE else S.pose_from_xi(start[g]) for g in range(frames)])
        ranges = np.array([[offs[s][0], offs[s][0] + n_kfs[s]] for s in scene], np.int32)
        for c in (cs, cm):
            for g0 in range(0, frames, 64):
                c.upload_batch(cur0 + g0, np.stack([rs[scene[g]]["frames"][which[g]]["img"] for g in range(g0, min(g0 + 64, frames))]))
        ppp = int(nf.max())

        def stage(flags_track):
            for c in (cs, cm):
                c.batch_stage(ref_slots, cur_slots, feats, nf, centers, poses_in, *SA, None, None, None, A2D_ITERS)
            cs.batch_stage_store(poses_ref, ranges, MAX_LOCAL, LEVELS - 3, A2D_ITERS, cpf)
            cm.batch_stage_map(poses_ref, ppp, LEVELS - 3, A2D_ITERS)
            if flags_track:
                cs.batch_stage_track(None, BA_ITERS); cm.batch_stage_track(None, BA_ITERS)

        out = {}
        for flags in (3, 7):
            stage(flags == 7)
            for c in (cs, cm, cs, cm):
                c.batch_run(flags)
                c.sync()
            ms = {"store": [], "one_kf": []}
            for _ in range(steps):
                for key, c in (("store", cs), ("one_kf", cm)):          # alternated: both see the same box state
                    c.batch_run(flags)
                    c.batch_fetch()
                    ms[key].append(c.last_run_ms())
            loc, nl, rec, nc = cs.batch_fetch_store()
            rep = cm.batch_fetch_map()
            res = {}
            for key in ms:
                med = float(np.median(ms[key]))
                res[key] = {"ms_per_step": med, "ms_min": float(np.min(ms[key])), "frames_per_s": frames / (med * 1e-3)}
            res["store"].update(mean_local_keyframes=float(nl.mean()), mean_candidates=float(nc.mean()), max_candidates=int(nc.max()),
                                overflow_frames=int((nc > cpf).sum()))
            res["one_kf"].update(mean_candidates=float(((rep["flags"] & capi.LM_IN_IMAGE) != 0).sum(1).mean()))
            if flags == 7:
                _, nm_s, _, _, _ = cs.batch_fetch_track()
                _, nm_m, _, _, _ = cm.batch_fetch_track()
                res["store"]["mean_matches"] = float(nm_s[nm_s >= 0].mean()); res["one_kf"]["mean_matches"] = float(nm_m.mean())
            for key, c in (("store", cs), ("one_kf", cm)):
                c.profile(True); c.profile_get(reset=True)
                for _ in range(steps):
                    c.batch_run(flags)
                st = c.profile_get(reset=True)
                c.profile(False)
                res[key]["stage_ms_per_step"] = {k: round(v[0] / steps, 4) for k, v in st.items() if v[1]}
            out["flags%d" % flags] = res
        return {"camera": name, "width": cam["width"], "height": cam["height"], "frames": frames, "steps": steps,
                "cands_per_frame": cpf, "keyframes_per_map": n_kfs, "points_per_map": [int(len(m["pw"])) for m in maps], "results": out}
    finally:
        cs.close(); cm.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--cpf", type=int, default=2048)
    ap.add_argument("--cams", default="KINECT,EUROC")
    ap.add_argument("--out", default="store_chain_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    res = {"gpu": gpu_info(),
           "workload": "%d frames over %d scenes (maps of 8-10 key frames, tests/store_map.py), Sprase_ImgAlign%s, Align2D %d it, "
                       "PoseOptimization %d it, max_local %d, cands_per_frame %d" % (a.frames, N_SCENES, SA, A2D_ITERS, BA_ITERS, MAX_LOCAL, a.cpf),
           "cams": [run_cam(c, a.frames, a.steps, a.cpf) for c in a.cams.split(",")]}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
