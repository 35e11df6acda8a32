"""The key frame behind the tracked pose (dsdtm_batch_run flags 15 = flags 7 followed by Tracking::CraeteKeyframe's detection and depth
lift) against flags 7 alone, on the bench workload: 4096 independent 640x480 kinect pairs (workload.build_batch, 300 features,
Sprase_ImgAlign(4,0,30), Align2D 10 iterations, PoseOptimization 100 iterations) and the same on the 752x480 EuRoC geometry, with a 16-bit
depth image per scene (rendered at the cur pose, scale 5000). For every pair wanted, one pair in eight wanted and none wanted: ms per step of
both flag sets alternated in one process (CUDA events, dsdtm_last_run_ms), key frames per second, and the stage split of the profiling
mode; the literal-sort count and new corners per key frame; and the CPU reference of the key-frame half (tests/cpp/keyframe_chain_oracle.cpp)
on all host threads for a sample, on the same run's matches and poses, with the parity figures beside it. The GPU name and power limit are
read in the same run (nvidia-smi query only). Writes one JSON file (--out)."""
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

LEVELS, N_FEATS, FEAT_STRIDE, SA, A2D_ITERS, BA_ITERS = 5, 300, 320, (4, 0, 30), 10, 100
CELL, MIN_DIST, MAX_FTS, THR, SCALE = 15, 15, 300, 5.0, 5000.0
DIST = (0.0, 0.0, 0.0, 0.0, 0.0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def run_cam(name, pairs, steps, sample, scenes):
    import keyframe_chain as KC
    import oracle as O
    from dsdtm_b200 import capi, synth as S, workload as W
    cam = dict(getattr(S, name))
    ctx = capi.Context(cam, levels=LEVELS, cell_size=CELL, max_feats=FEAT_STRIDE, max_patches=N_FEATS, max_frames=2 * pairs + 2, max_batch=pairs)
    try:
        ctx.set_option("depth_slots", scenes)
        batch = W.build_batch(ctx, cam, pairs, n_scenes=scenes, n_feats=N_FEATS, feat_stride=FEAT_STRIDE, patches_per_pair=N_FEATS)
        k = batch["n_scenes"]
        d16 = []
        for s, sc in enumerate(batch["scenes"]):
            _, z = S.render(S.Scene(sc["seed"]), cam, S.pose_mul(sc["T_c2r"], sc["T_ref"]))
            d16.append(np.clip(np.rint(z * SCALE), 0, 65535).astype(np.uint16))
            ctx.depth_upload(s, d16[-1])
        depth_slots = (np.arange(pairs) % k).astype(np.int32)

        def stage(want):
            ctx.batch_stage(batch["ref_slots"], batch["cur_slots"], batch["feats"], batch["n_feats"], batch["centers"], batch["poses_in"], *SA,
                            None, None, None, A2D_ITERS)
            ctx.batch_stage_map(batch["poses_ref"], N_FEATS, LEVELS - 3, A2D_ITERS)
            ctx.batch_stage_track(None, BA_ITERS)
            ctx.batch_stage_keyframe(depth_slots, want, THR, MIN_DIST, MAX_FTS, DIST, SCALE)

        modes = {"all": np.ones(pairs, np.uint8), "one_in_8": (np.arange(pairs) % 8 == 0).astype(np.uint8), "none": np.zeros(pairs, np.uint8)}
        out = {}
        for mode, want in modes.items():
            stage(want)
            for flags in (7, 15, 7, 15):
                ctx.batch_run(flags)
            ctx.sync()
            ms = {7: [], 15: []}
            for _ in range(steps):
                for flags in (7, 15):                  # alternated: both see the same box state
                    ctx.batch_run(flags)
                    ctx.batch_fetch()
                    ms[flags].append(ctx.last_run_ms())
            nn, _, _, ex = ctx.batch_fetch_keyframe()
            stages = {}
            for flags in (7, 15):
                ctx.profile(True); ctx.profile_get(reset=True)
                for _ in range(steps):
                    ctx.batch_run(flags)
                st = ctx.profile_get(reset=True)
                ctx.profile(False)
                stages[flags] = {kk: round(v[0] / steps, 4) for kk, v in st.items() if v[1]}
            m7, m15 = float(np.median(ms[7])), float(np.median(ms[15]))
            nw = int(want.sum())
            out[mode] = {"wanted_pairs": nw,
                         "ms_per_step": {"flags7": m7, "flags15": m15, "flags7_min": float(np.min(ms[7])), "flags15_min": float(np.min(ms[15])),
                                         "added_by_keyframe": m15 - m7},
                         "keyframes_per_s": nw / (m15 * 1e-3) if nw else 0.0,
                         "stage_ms_per_step": {"flags7": stages[7], "flags15": stages[15]},
                         "literal_path_pairs": int(ex.sum()),
                         "mean_new_corners_per_keyframe": float(nn[want.astype(bool)].mean()) if nw else 0.0}
        # the CPU reference on a sample of the all-wanted run, all host threads
        stage(modes["all"])
        ctx.batch_run(15)
        poses, nm, m, _, _ = ctx.batch_fetch_track()
        nn, cr, lf, ex = ctx.batch_fetch_keyframe()
        oc = O.make_cam(cam["width"], cam["height"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["f"])
        cur = np.stack([batch["scenes"][i % k]["cur_img"] for i in range(sample)])
        dd = np.stack([d16[i % k] for i in range(sample)])
        threads = os.cpu_count() or 1
        args = (oc, LEVELS, CELL, MIN_DIST, MAX_FTS, THR, DIST, SCALE, cur, m[:sample], nm[:sample], poses[:sample], dd)
        KC.keyframe_chain(*args, n_threads=threads)
        t0 = time.perf_counter()
        o = KC.keyframe_chain(*args, n_threads=threads)
        cpu_s = time.perf_counter() - t0
        same = sum(int(nn[i]) == int(o["n_new"][i]) and KC.same_corners(cr[i][:nn[i]], o["corners"][i][:nn[i]]) for i in range(sample))
        dpt = max(float(np.abs(lf[i]["point_w"][:nn[i]] - o["lifted"][i]["point_w"][:nn[i]]).max(initial=0)) for i in range(sample))
        return {"camera": name, "width": cam["width"], "height": cam["height"], "pairs": pairs, "steps": steps, "modes": out,
                "mean_matches_per_pair": float(np.mean(nm)),
                "occupancy_indices_outside_grid": int(sum(((k_ < 0) | (k_ >= ctx.n_cells)).sum() for k_ in (
                    (m[i]["px"][:nm[i], 1] / np.float32(CELL)).astype(np.int64) * ctx.grid_cols
                    + (m[i]["px"][:nm[i], 0] / np.float32(CELL)).astype(np.int64) for i in range(pairs)))),
                "cpu_reference": {"sample_pairs": sample, "threads": threads, "seconds": cpu_s, "keyframes_per_s": sample / cpu_s,
                                  "corner_lists_equal": int(same), "exact_path_equal": int((ex[:sample] == o["tied"]).sum()),
                                  "max_point_diff": dpt}}
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--sample", type=int, default=256)
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--cams", default="KINECT,EUROC")
    ap.add_argument("--out", default="keyframe_chain_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    res = {"gpu": gpu_info(),
           "workload": "workload.build_batch: %d pairs, %d features, Sprase_ImgAlign%s, Align2D %d it, PoseOptimization %d it; key frame: "
                       "detection_threshold %.1f, Min_dist %d, Max_fts %d, 16-bit depth per scene (scale %.0f), no distortion"
                       % (a.pairs, N_FEATS, SA, A2D_ITERS, BA_ITERS, THR, MIN_DIST, MAX_FTS, SCALE),
           "cams": [run_cam(c, a.pairs, a.steps, a.sample, a.scenes) for c in a.cams.split(",")]}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
