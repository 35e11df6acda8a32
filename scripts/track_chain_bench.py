"""The tracked-pose chain (dsdtm_batch_run flags 7 = pyramid -> Sprase_ImgAlign::Run -> refinement chain -> SearchLocalPoints'
selection -> PoseOptimization) against the chain without the last two stages (flags 3), on the bench workload: 4096 independent
640x480 kinect pairs (workload.build_batch, 300 features, Sprase_ImgAlign(4,0,30), Align2D 10 iterations) and the same on the 752x480
EuRoC geometry. Per camera: ms per step of both flag sets alternated in one process (CUDA events, dsdtm_last_run_ms), the stage split
of the profiling mode, frames tracked per second, mean matches and LM iterations per pair, the one-pair latency of the flags-7 graph,
and the oracle's whole chain (tests/cpp/track_chain_oracle.cpp) on all host threads for a sample with the parity figures beside it. The GPU name
and power limit are read in the same run (nvidia-smi query only). Writes one JSON file (--out)."""
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


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def run_cam(name, pairs, steps, sample, scenes):
    import oracle as O
    import track_select as TS
    from dsdtm_b200 import capi, synth as S, workload as W
    cam = dict(getattr(S, name))
    ctx = capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=N_FEATS, max_frames=2 * pairs + 2, max_batch=pairs)
    try:
        batch = W.build_batch(ctx, cam, pairs, n_scenes=scenes, n_feats=N_FEATS, feat_stride=FEAT_STRIDE, patches_per_pair=N_FEATS)

        def stage(n):
            ctx.batch_stage(batch["ref_slots"][:n], batch["cur_slots"][:n], batch["feats"][:n], batch["n_feats"][:n], batch["centers"][:n],
                            batch["poses_in"][:n], *SA, None, None, None, A2D_ITERS)
            ctx.batch_stage_map(batch["poses_ref"][:n], N_FEATS, LEVELS - 3, A2D_ITERS)
            ctx.batch_stage_track(None, BA_ITERS)

        stage(pairs)
        for flags in (3, 7, 3, 7):
            ctx.batch_run(flags)
        ctx.sync()
        ms = {3: [], 7: []}
        for _ in range(steps):
            for flags in (3, 7):                       # alternated: both see the same box state
                ctx.batch_run(flags)
                ctx.batch_fetch()
                ms[flags].append(ctx.last_run_ms())
        poses, nm, m, res, summ = ctx.batch_fetch_track()
        poses_c2r, _, _, _ = ctx.batch_fetch()
        stages = {}
        for flags in (3, 7):
            ctx.profile(True); ctx.profile_get(reset=True)
            for _ in range(steps):
                ctx.batch_run(flags)
            st = ctx.profile_get(reset=True)
            ctx.profile(False)
            stages[flags] = {k: round(v[0] / steps, 4) for k, v in st.items() if v[1]}
        # one pair: the flags-7 graph replayed
        stage(1)
        for _ in range(5):
            ctx.batch_run(7)
        ctx.batch_fetch_track()
        lat = []
        for _ in range(50):
            ctx.batch_run(7)
            ctx.batch_fetch_track()
            lat.append(ctx.last_run_ms())
        # the oracle's whole chain on a sample of the same pairs, all host threads
        k = batch["n_scenes"]
        ref_pyrs = np.stack([O.pyramid(batch["scenes"][i % k]["ref_img"], LEVELS)[0] for i in range(sample)])
        cur_imgs = np.stack([batch["scenes"][i % k]["cur_img"] for i in range(sample)])
        oc = O.make_cam(cam["width"], cam["height"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["f"])
        threads = os.cpu_count() or 1
        args = (oc, LEVELS, 15, ref_pyrs, cur_imgs, batch["feats"][:sample].astype(O.REF_FEAT_DT), batch["n_feats"][:sample],
                batch["centers"][:sample], batch["poses_ref"][:sample], batch["poses_in"][:sample], *SA, N_FEATS, LEVELS - 3, A2D_ITERS)
        TS.pair_batch_track(*args, ba_iters=BA_ITERS, n_threads=threads)
        t0 = time.perf_counter()
        o = TS.pair_batch_track(*args, ba_iters=BA_ITERS, n_threads=threads)
        cpu_s = time.perf_counter() - t0
        same = [int(nm[i]) == int(o["n_matches"][i]) and (m[i]["point"][:nm[i]] == o["matches"][i]["point"][:nm[i]]).all()
                and (m[i]["level"][:nm[i]] == o["matches"][i]["level"][:nm[i]]).all() for i in range(sample)]
        dpose = np.array([S.pose_dist(o["poses"][i], poses[i]) for i in range(sample)])
        m3, m7 = float(np.median(ms[3])), float(np.median(ms[7]))
        return {
            "camera": name, "width": cam["width"], "height": cam["height"], "pairs": pairs, "steps": steps,
            "ms_per_step": {"flags3": m3, "flags7": m7, "flags3_min": float(np.min(ms[3])), "flags7_min": float(np.min(ms[7])),
                            "added_by_select_and_pose_opt": m7 - m3},
            "frames_tracked_per_s": pairs / (m7 * 1e-3),
            "stage_ms_per_step": {"flags3": stages[3], "flags7": stages[7]},
            "mean_matches_per_pair": float(np.mean(nm)), "pairs_at_200_matches": int((nm == 200).sum()),
            "mean_lm_iterations_per_pair": float(np.mean(summ["iterations"])),
            "terminations": {str(t): int((summ["termination"] == t).sum()) for t in np.unique(summ["termination"])},
            "one_pair_flags7_graph_us": {"median": 1e3 * float(np.median(lat)), "min": 1e3 * float(np.min(lat))},
            "oracle_chain": {"sample_pairs": sample, "threads": threads, "seconds": cpu_s, "pairs_per_s": sample / cpu_s,
                             "match_lists_equal": int(sum(same)), "max_pose_diff_rad": float(dpose[:, 0].max()),
                             "max_pose_diff_m": float(dpose[:, 1].max())},
        }
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--sample", type=int, default=256)
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--cams", default="KINECT,EUROC")
    ap.add_argument("--out", default="track_chain_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    res = {"gpu": gpu_info(), "workload": "workload.build_batch: %d pairs, %d features, Sprase_ImgAlign%s, Align2D %d it, PoseOptimization %d it"
           % (a.pairs, N_FEATS, SA, A2D_ITERS, BA_ITERS), "cams": [run_cam(c, a.pairs, a.steps, a.sample, a.scenes) for c in a.cams.split(",")]}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
