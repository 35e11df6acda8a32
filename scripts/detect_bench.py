"""Key-frame detection on the device (dsdtm_detect_batch = FAST + per-cell best + sort + mask-circle selection, one submission)
against dsdtm_fast_cells_batch alone (the cells, with the sort and the selection left to the host), alternated in one process, on
4096 640x480 kinect frames and 4096 752x480 EuRoC frames (workload.render_scenes, ref and cur images cycled), and on 4096 tiled
frames (a random 15x15, 30x30 or 45x45 block repeated), where every frame ties scores above 20 and takes the literal std::sort
path. Also: the one-frame latency of dsdtm_detect with and without the 307 KB mask upload, and the CPU baseline: the oracle's
detect_cells + detect_select on all host threads. Host wall time per call (ends in the call's synchronisation) and device time
(profiling mode, DSDTM_STAGE_FAST) are both reported. The GPU name and power limit are read in the same run (nvidia-smi query
only). Writes one JSON file (--out)."""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LEVELS, CELL, THR, MAX_NEW = 5, 15, 5.0, 300


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def tiled(period, seed, w, h):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


def oracle_detect(img):
    import oracle as O
    packed, offs, ws, hs = O.pyramid(img, LEVELS)
    cells = O.detect_cells(packed, offs, ws, hs, CELL, None, THR)
    return O.detect_select(cells, np.full(img.shape, 255, np.uint8), CELL, MAX_NEW)[0]


def same(a, b):
    return len(a) == len(b) and all((a[k] == b[k]).all() for k in ("x", "y", "level")) and (a["score"].view(np.uint32) == b["score"].view(np.uint32)).all()


def run_set(name, cam, imgs, frames, steps, sample):
    from dsdtm_b200 import capi
    ctx = capi.Context(cam, levels=LEVELS, cell_size=CELL, max_feats=16, max_patches=16, max_frames=frames, max_batch=frames)
    try:
        k = len(imgs)
        for i0 in range(0, frames, 64):
            n = min(64, frames - i0)
            ctx.upload_batch(i0, np.stack([imgs[(i0 + j) % k] for j in range(n)]))
        for _ in range(2):
            ctx.detect(0, THR, max_new=MAX_NEW, n=frames)
            ctx.fast_cells(0, 20, THR, n=frames)
        wall = {"detect_batch": [], "fast_cells_batch": []}
        for _ in range(steps):                                   # alternated: both see the same box state
            t0 = time.perf_counter()
            got, exact = ctx.detect(0, THR, max_new=MAX_NEW, n=frames)
            t1 = time.perf_counter()
            ctx.fast_cells(0, 20, THR, n=frames)
            t2 = time.perf_counter()
            wall["detect_batch"].append(t1 - t0); wall["fast_cells_batch"].append(t2 - t1)
        dev = {}
        for key, fn in (("detect_batch", lambda: ctx.detect(0, THR, max_new=MAX_NEW, n=frames)), ("fast_cells_batch", lambda: ctx.fast_cells(0, 20, THR, n=frames))):
            ctx.profile(True); ctx.profile_get(reset=True)
            for _ in range(steps):
                fn()
            dev[key] = ctx.profile_get(reset=True)["fast"][0] / steps
            ctx.profile(False)
        # parity on a sample (frame i holds imgs[i % k])
        idx = np.linspace(0, frames - 1, sample).astype(int)
        equal = sum(same(got[i], oracle_detect(imgs[i % k])) for i in idx)
        # one frame: dsdtm_detect with and without a mask image
        mask = np.full((cam["height"], cam["width"]), 255, np.uint8)
        occ = np.zeros(ctx.n_cells, np.uint8)
        lat = {}
        for key, kw in (("no_mask_us", {}), ("with_mask_and_occupancy_us", {"mask": mask, "occupied": occ})):
            for _ in range(10):
                ctx.detect(0, THR, max_new=MAX_NEW, **kw)
            ts = []
            for _ in range(200):
                t0 = time.perf_counter()
                ctx.detect(0, THR, max_new=MAX_NEW, **kw)
                ts.append(time.perf_counter() - t0)
            lat[key] = {"median": 1e6 * float(np.median(ts)), "min": 1e6 * float(np.min(ts))}
        md, mf = float(np.median(wall["detect_batch"])), float(np.median(wall["fast_cells_batch"]))
        return {
            "set": name, "width": cam["width"], "height": cam["height"], "frames": frames, "distinct_images": k, "steps": steps,
            "wall_ms_per_call": {"detect_batch": 1e3 * md, "fast_cells_batch": 1e3 * mf},
            "frames_per_s": {"detect_batch": frames / md, "fast_cells_batch": frames / mf},
            "device_ms_per_call": dev,
            "exact_path_frames": int(exact.sum()), "mean_selected": float(np.mean([len(g) for g in got])),
            "oracle_parity": {"sample": int(sample), "equal": int(equal)},
            "one_frame_detect": lat,
        }
    finally:
        ctx.close()


def cpu_baseline(imgs, n):
    threads = os.cpu_count() or 1
    work = [imgs[i % len(imgs)] for i in range(n)]
    with ThreadPoolExecutor(threads) as ex:                       # ctypes releases the GIL inside the oracle's calls
        list(ex.map(oracle_detect, work[:threads]))
        t0 = time.perf_counter()
        list(ex.map(oracle_detect, work))
        s = time.perf_counter() - t0
    return {"frames": n, "threads": threads, "seconds": s, "frames_per_s": n / s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--scenes", type=int, default=8)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--cpu-frames", type=int, default=512)
    ap.add_argument("--out", default="detect_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    from dsdtm_b200 import synth as S, workload as W
    res = {"gpu": gpu_info(), "workload": "threshold %.1f, CellSize %d, %d levels, max_new %d, no occupancy, no mask (batch)" % (THR, CELL, LEVELS, MAX_NEW),
           "sets": [], "cpu_baseline": {}}
    for name in ("KINECT", "EUROC"):
        cam = dict(getattr(S, name))
        scenes = W.render_scenes(a.scenes, cam)
        imgs = [sc[k] for sc in scenes for k in ("ref_img", "cur_img")]
        res["sets"].append(run_set(name, cam, imgs, a.frames, a.steps, a.sample))
        res["cpu_baseline"][name] = cpu_baseline(imgs, a.cpu_frames)
        if name == "KINECT":
            timgs = [tiled(p, 100 * p + s, cam["width"], cam["height"]) for p in (15, 30, 45) for s in range(4)]
            res["sets"].append(run_set("KINECT_TILED", cam, timgs, a.frames, a.steps, a.sample))
            res["cpu_baseline"]["KINECT_TILED"] = cpu_baseline(timgs, a.cpu_frames)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
