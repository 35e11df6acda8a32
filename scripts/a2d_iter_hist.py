"""Align2D iteration statistics of the bench batch, on the CPU: the per-patch iteration histogram (oracle.align2d's count of
executed Gauss-Newton iterations) and the lane utilisation when 2 or 4 consecutive patches share a warp, which then runs until
the slowest of them is done. Patches are grouped in their batch order; unused entries (level < 0) take 0 iterations.

    python scripts/a2d_iter_hist.py [--out FILE]
"""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import bench
import oracle as O
from dsdtm_b200 import synth as S, workload as W


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=4096)
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--out")
    a = ap.parse_args()
    cam = dict(S.KINECT)
    scenes = W.render_scenes(a.scenes, cam, seed0=W.BASE_SEED)
    batch = bench.host_batch_with_oracle_detector(cam, scenes, a.scenes, W.BASE_SEED)
    # pair g uses scene g % k and the scene's patches and start positions unchanged, so the scene's counts repeat over the batch
    nit = np.zeros((a.scenes, bench.N_FEATS), np.int64)
    for s, sc in enumerate(scenes):
        packed, offs, ws, hs = O.pyramid(sc["cur_img"], bench.LEVELS)
        for j in range(bench.N_FEATS):
            L = int(batch["patch_level"][s, j])
            if L >= 0:
                img = O.pyr_level(packed, offs, ws, hs, L)
                nit[s, j] = O.align2d(img, batch["patches"][s, j], bench.ALIGN2D_ITERS, batch["patch_px"][s, j])[2]
    per_pair = nit[np.arange(a.pairs) % a.scenes]                       # batch order: pair-major, 300 patches per pair
    flat = per_pair.reshape(-1)
    used = (batch["patch_level"][np.arange(a.pairs) % a.scenes] >= 0).reshape(-1)
    res = {"pairs": a.pairs, "patches": int(flat.size), "used_patches": int(used.sum()),
           "histogram_used": {int(k): int(((flat == k) & used).sum()) for k in range(bench.ALIGN2D_ITERS + 1)},
           "mean_iters_used": float(flat[used].mean()), "group": {}}
    for g in (2, 4):
        m = flat.reshape(-1, g).max(1)
        res["group"][g] = {"warp_iters_per_patch": float(m.sum() / flat.size), "lane_utilisation": float(flat.sum() / (g * m.sum())),
                           "histogram_group_max": {int(k): int((m == k).sum()) for k in range(bench.ALIGN2D_ITERS + 1)}}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
