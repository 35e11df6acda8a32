"""dsdtm_batch_commit_store on 4096 kinect frames: 8 rendered scenes with maps of 8 to 10 key frames (tests/store_map.py), tiled `copies`
times into one store so that each map copy serves frames_per_map frames (the sweep layout), frame g tracking a cur image of scene g % 8
(rendered depth in its own depth slot) against that scene's last key frame with flags 15 (Sprase_ImgAlign(4,0,30), Align2D 10 iterations, PoseOptimization 100 iterations, ten
local key frames, live found counts). Reports, with the GPU name and power limit read in the same run (nvidia-smi query only):
  - the commit (host wall clock of the call, which ends in its one synchronisation; and CUDA events around it) with every frame, one in
    eight and no frame wanted;
  - the same commit through the host path: fetch_track + fetch_keyframe, then dsdtm_store_set_points, one dsdtm_store_append_keyframe per
    key frame, dsdtm_store_update_points and dsdtm_store_set_found (tests/store_commit.py's host_commit);
  - a whole step of a sequence: staging (which drops the captured graph), run with capture, fetch of the poses, commit.
Every timed commit follows its own run of the step; the store grows by each commit's key frames (outside the frames' ranges, so the
records do not change; the found counts do). Writes one JSON file."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LEVELS, FEAT_STRIDE, SA, A2D_ITERS, BA_ITERS, MAX_LOCAL, CPF = 5, 320, (4, 0, 30), 10, 100, 10, 2048
N_SCENES = 8
THR = np.float32(0.0)                          # set from the data (see main)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def main():
    global THR
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--frames-per-map", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="store_commit_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import store_commit as SCM
    import store_map as SM
    from dsdtm_b200 import capi, synth as S
    cam = dict(S.KINECT)
    frames = a.frames
    copies = max(1, frames // (N_SCENES * a.frames_per_map))
    n_kfs = [8 + s % 3 for s in range(N_SCENES)]
    kf_slot0 = np.concatenate([[0], np.cumsum(n_kfs)])
    cur0 = int(kf_slot0[-1])
    rs = SM.render_scenes(cam, [5200 + 31 * s for s in range(N_SCENES)], n_kfs, 2)
    mk = lambda: capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=CPF, max_frames=cur0 + frames, max_batch=frames)
    c, h = mk(), mk()
    try:
        maps = [SM.build_map(c, cam, rs[s], int(kf_slot0[s])) for s in range(N_SCENES)]
        scene = np.arange(frames) % N_SCENES
        which = (np.arange(frames) // N_SCENES) % 2
        copy = (np.arange(frames) // N_SCENES) % copies
        feats = np.zeros((frames, FEAT_STRIDE), capi.REF_FEAT_DT); nf = np.zeros(frames, np.int32)
        per = [SM.ref_feats(m, FEAT_STRIDE) for m in maps]
        for q in range(frames):
            feats[q], nf[q] = per[scene[q]]
        last = [m["kfs"][-1] for m in maps]
        centers = np.stack([last[s]["center"] for s in scene]); poses_ref = np.stack([last[s]["pose"] for s in scene])
        ref_slots = np.array([last[s]["slot"] for s in scene], np.int32)
        cur_slots = (cur0 + np.arange(frames)).astype(np.int32)
        rng = np.random.default_rng(4242)
        start = np.concatenate([rng.uniform(-0.004, 0.004, (frames, 3)), rng.uniform(-0.002, 0.002, (frames, 3))], 1)
        poses_in = np.stack([S.IDENTITY if q < 2 * N_SCENES else S.pose_from_xi(start[q]) for q in range(frames)])
        t0 = time.perf_counter()
        for ctx in (c, h):
            ctx.set_option("depth_slots", frames)
            for q in range(frames):
                ctx.depth_upload(q, rs[scene[q]]["frames"][which[q]]["d16"])
            offs = SM.load_maps(ctx, [maps[s] for _ in range(copies) for s in range(N_SCENES)])
            for g0 in range(0, frames, 64):
                ctx.upload_batch(cur0 + g0, np.stack([rs[scene[q]]["frames"][which[q]]["img"] for q in range(g0, min(g0 + 64, frames))]))
        load_s = time.perf_counter() - t0
        ranges = np.array([[offs[copy[q] * N_SCENES + scene[q]][0], offs[copy[q] * N_SCENES + scene[q]][0] + n_kfs[scene[q]]] for q in range(frames)],
                          np.int32)

        def stage(ctx, want):
            ctx.batch_stage(ref_slots, cur_slots, feats, nf, centers, poses_in, *SA, None, None, None, A2D_ITERS)
            ctx.batch_stage_store(poses_ref, ranges, MAX_LOCAL, LEVELS - 3, A2D_ITERS, CPF)
            ctx.batch_stage_track_live(BA_ITERS)
            ctx.batch_stage_keyframe(np.arange(frames, dtype=np.int32), want, 5.0, 15, 300, (0.0,) * 5, 5000.0)

        wants = {"all": np.ones(frames, bool), "one_in_8": (np.arange(frames) % 8) == 0, "none": np.zeros(frames, bool)}
        # the outlier threshold: the upper quartile of a first step's residual norms, so that the commits erase as well as count
        stage(c, wants["none"])
        c.batch_run(15)
        _, nm0, _, res0, _ = c.batch_fetch_track()
        THR = np.float32(np.quantile(np.concatenate([res0[q][:nm0[q]] for q in range(frames) if nm0[q] > 0]), 0.75))
        res = {"gpu": gpu_info(), "frames": frames, "outlier_threshold": float(THR), "map_copies": copies * N_SCENES, "frames_per_map": a.frames_per_map,
               "keyframes_per_map": n_kfs, "points_per_map": [int(len(m["pw"])) for m in maps], "load_s": load_s, "commit": {}}
        for name, want in wants.items():
            stage(c, want)
            wall, ev, step_ms, kfs, rows = [], [], [], [], []
            for r in range(a.reps + 1):
                c.batch_run(15)
                c.batch_fetch()
                step_ms.append(c.last_run_ms())
                nk0, nf0, _ = c.store_size()
                c.timer_start()
                t0 = time.perf_counter()
                out = c.batch_commit_store(THR)
                t1 = time.perf_counter()
                e = c.timer_stop()
                nk1, nf1, _ = c.store_size()
                if r:                                          # the first commit also grows the tables' capacity
                    wall.append((t1 - t0) * 1e3); ev.append(e); kfs.append(nk1 - nk0); rows.append(nf1 - nf0)
            res["commit"][name] = {"wall_ms_median": float(np.median(wall)), "wall_ms_min": float(np.min(wall)), "event_ms_median": float(np.median(ev)),
                                   "keyframes": int(np.median(kfs)), "feature_rows": int(np.median(rows)),
                                   "flags15_run_ms_median": float(np.median(step_ms))}
        # the host path on the second context, every frame and one in eight wanted: the caller keeps bad flags and found counts on the
        # host (read here from the store, untimed), fetches the step's outputs and makes the store calls
        res["host_path"] = {}
        for name in ("all", "one_in_8"):
            stage(h, wants[name])
            fetch, calls, kf = [], [], []
            for r in range(a.reps):
                h.batch_run(15)
                h.sync()
                _, _, P, found = h.store_fetch()
                t0 = time.perf_counter()
                out = SCM.step_outputs(h, cur_slots, wants[name])
                t1 = time.perf_counter()
                SCM.host_commit(h, cam, out, THR, state=(P["bad"], found))
                t2 = time.perf_counter()
                fetch.append((t1 - t0) * 1e3); calls.append((t2 - t1) * 1e3); kf.append(int((wants[name] & (out["nm"] >= 0)).sum()))
            res["host_path"][name] = {"fetch_ms_median": float(np.median(fetch)), "store_calls_ms_median": float(np.median(calls)),
                                      "total_ms_median": float(np.median(np.add(fetch, calls))), "total_ms_min": float(np.min(np.add(fetch, calls))),
                                      "keyframes": int(np.median(kf)), "reps": a.reps}
        # whole steps of a sequence: stage + run (captured anew) + poses + commit
        step = []
        for r in range(a.reps + 1):
            t0 = time.perf_counter()
            stage(c, wants["one_in_8"])
            c.batch_run(15)
            c.batch_fetch_track()
            c.batch_commit_store(THR)
            if r:
                step.append((time.perf_counter() - t0) * 1e3)
        res["sequence_step_ms"] = {"median": float(np.median(step)), "min": float(np.min(step)), "want": "one_in_8"}
        res["gpu_after"] = gpu_info()
    finally:
        c.close(); h.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
