"""Sequences on the device (dsdtm_batch_upload_step -> dsdtm_batch_run -> dsdtm_batch_commit_store -> dsdtm_batch_advance) against the
host-driven loop (one upload per frame, fetch, the next reference frame built on the host by tests/sequence_chain.py, restaging, run,
commit), alternated step by step on two contexts holding the same store.

Workload: 4096 kinect sequences. 8 rendered scenes (maps of 8 to 10 key frames, tests/store_map.py), each with one rendered trajectory of
`steps` frames (S.random_motion chained from the last key frame's pose, depth at scale 5000), tiled into 4096 map copies, one per sequence,
each with steps / 8 empty key-frame rows reserved inside its range. Every step runs flags 15: sequence g wants a key frame at steps k with
(k + g) % 8 == 7, so 512 frames are wanted per step and each sequence adds a key frame every 8th step (Sprase_ImgAlign(4,0,30), Align2D
10 iterations, PoseOptimization 100 iterations, ten local key frames, live found counts). The images and depth of a step go up every step
(pinned buffers): 4096 x 640 x 480 bytes of image and twice that of depth. A second phase of --track-steps flags-7 steps (no key frame
wanted) shows the replayed step. Reports per step: ms (median, min, max), frames tracked per second, the upload / run / commit / advance
split, graph captures per step and the share of steps that replayed, with the GPU name and power limit read in the same run. Writes one
JSON file."""
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
N_SCENES, POOL = 8, 7                           # slots per sequence: its key frames' (steps / 8), its reference and its cur frame
THR = np.float32(0.004)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi: %s)" % q.stderr.strip()


def stats(v):
    return {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--track-steps", type=int, default=8)
    ap.add_argument("--out", default="sequence_chain_bench.json")
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import sequence_chain as SC
    import store_commit as SCM
    import store_map as SM
    from dsdtm_b200 import capi, synth as S
    cam = dict(S.KINECT)
    n, steps, total = a.frames, a.steps, a.steps + a.track_steps
    n_kfs = [8 + s % 3 for s in range(N_SCENES)]
    kf_slot0 = np.concatenate([[0], np.cumsum(n_kfs)])
    cur0 = int(kf_slot0[-1])
    t0 = time.perf_counter()
    rs = SC.render_sequences(cam, [5200 + 31 * s for s in range(N_SCENES)], n_kfs, 1, total)
    render_s = time.perf_counter() - t0
    scene = np.arange(n) % N_SCENES
    reserve = (steps + 7) // 8
    mk = lambda: capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=CPF, max_frames=cur0 + POOL * n, max_batch=n)
    ca, cb = mk(), mk()
    try:
        maps = [SM.build_map(ca, cam, rs[s], int(kf_slot0[s])) for s in range(N_SCENES)]
        t0 = time.perf_counter()
        ranges, reserved = np.zeros((n, 2), np.int32), []
        for ctx in (ca, cb):
            ctx.set_option("depth_slots", n)
            ctx.store_clear()
            reserved = []
            for q in range(n):
                k0 = ctx.store_keyframes
                SM.load_maps(ctx, [maps[scene[q]]], clear=False)
                reserved.append([ctx.store_append_keyframe(0, S.IDENTITY, np.zeros(3), np.zeros(0, capi.STORE_FEAT_DT)) for _ in range(reserve)])
                ranges[q] = (k0, ctx.store_keyframes)
            ctx.depth_upload(0, rs[0]["seqs"][0][0]["d16"])       # the depth pool exists before the key-frame half names its slots
        load_s = time.perf_counter() - t0
        per = [SM.ref_feats(m, FEAT_STRIDE) for m in maps]
        last = [m["kfs"][-1] for m in maps]
        fr = dict(ref_slots=np.array([last[s]["slot"] for s in scene], np.int32), cur_slots=(cur0 + POOL * np.arange(n)).astype(np.int32),
                  feats=np.stack([per[s][0] for s in scene]), n_feats=np.array([per[s][1] for s in scene], np.int32),
                  centers=np.stack([last[s]["center"] for s in scene]), poses_ref=np.stack([last[s]["pose"] for s in scene]),
                  poses_in=np.tile(S.IDENTITY, (n, 1)))
        imgs = capi.pinned_empty((n, cam["height"], cam["width"]), np.uint8)
        d16 = capi.pinned_empty((n, cam["height"], cam["width"]), np.uint16)

        def want_at(k):
            return ((k + np.arange(n)) % 8 == 7) if k < steps else np.zeros(n, bool)

        def stage(ctx, f, want):
            ctx.batch_stage(f["ref_slots"], f["cur_slots"], f["feats"], f["n_feats"], f["centers"], f["poses_in"], *SA, None, None, None, A2D_ITERS)
            ctx.batch_stage_store(f["poses_ref"], ranges, MAX_LOCAL, LEVELS - 3, A2D_ITERS, CPF)
            ctx.batch_stage_track_live(BA_ITERS)
            ctx.batch_stage_keyframe(np.arange(n, dtype=np.int32), want, 5.0, 15, 300, (0.0,) * 5, 5000.0)

        # slots: sequence q owns cur0 + POOL * q + [0, POOL); the next cur slot is the first that holds none of its key frames, its
        # reference after the advance or its cur frame now
        kf_slots = [set() for _ in range(n)]
        n_kf = np.zeros(n, np.int32)

        def next_slots(cur, ref_next):
            out = np.empty(n, np.int32)
            for q in range(n):
                busy = kf_slots[q] | {int(ref_next[q]), int(cur[q])}
                out[q] = next(cur0 + POOL * q + j for j in range(POOL) if cur0 + POOL * q + j not in busy)
            return out

        stage(ca, fr, want_at(0))
        res = {"gpu": gpu_info(), "frames": n, "steps": steps, "track_steps": a.track_steps, "keyframes_per_map": n_kfs,
               "render_s": render_s, "load_s": load_s, "device": [], "host": []}
        for k in range(total):
            flags = 15 if k < steps else 7
            for q in range(n):
                f = rs[scene[q]]["seqs"][0][k]
                imgs[q] = f["img"]; d16[q] = f["d16"]
            want, want_next = want_at(k), want_at(k + 1)
            rows = np.array([reserved[q][min(n_kf[q], reserve - 1)] for q in range(n)], np.int32)
            # (a) the device chain
            g0 = ca.graph_captures()
            t = [time.perf_counter()]
            ca.batch_upload_step(imgs, d16); t.append(time.perf_counter())
            ca.batch_run(flags); ca.sync(); t.append(time.perf_counter())
            ca.batch_commit_store(THR, rows if flags & 8 else None); t.append(time.perf_counter())
            cur = fr["cur_slots"].copy()
            _, nm, _, _, _ = ca.batch_fetch_track()                         # untimed: the slot bookkeeping of this script
            adv_ref = np.where((nm >= 0), cur, fr["ref_slots"])
            nxt = next_slots(cur, adv_ref)
            t.append(time.perf_counter())
            status = ca.batch_advance(nxt, None, want_next if k + 1 < total else None); t.append(time.perf_counter())
            d = np.diff(t) * 1e3
            res["device"].append({"step": k, "flags": flags, "upload_ms": d[0], "run_ms": d[1], "commit_ms": d[2], "advance_ms": d[4],
                                  "total_ms": d[0] + d[1] + d[2] + d[4], "captures": ca.graph_captures() - g0,
                                  "keyframes": int((status == capi.ADV_KEYFRAME).sum()), "held": int((status >= capi.ADV_HELD_OVERFLOW).sum())})
            # (b) the host-driven loop
            t0 = time.perf_counter()
            for q in range(n):
                cb.upload(int(fr["cur_slots"][q]), imgs[q])
                cb.depth_upload(q, d16[q])
            stage(cb, fr, want)
            cb.batch_run(flags)
            o = SCM.step_outputs(cb, fr["cur_slots"], want, keyframes=bool(flags & 8))
            cb.batch_commit_store(THR, rows if flags & 8 else None)
            nx, sb = SC.next_ref(cam, fr, o, cb.store_fetch()[2]["point_w"], nxt, keyframes=bool(flags & 8))
            res["host"].append({"step": k, "flags": flags, "total_ms": (time.perf_counter() - t0) * 1e3})
            same = bool((sb == status).all())
            ra = ca.batch_fetch_ref()
            same &= all(ra[key].tobytes() == nx[key].tobytes() for key in ra)
            res["device"][-1]["equal_to_host"] = same
            for q in np.flatnonzero(status == capi.ADV_KEYFRAME):
                kf_slots[q].add(int(cur[q])); n_kf[q] += 1
            fr = nx
            print(json.dumps({"device": res["device"][-1], "host": res["host"][-1]}), flush=True)
        for arm in ("device", "host"):
            for name, sel in (("keyframe_steps", lambda r: r["flags"] == 15), ("track_steps", lambda r: r["flags"] == 7)):
                rows_ = [r for r in res[arm] if sel(r)][1:]                   # the first step of a phase also grows capacities
                if not rows_:
                    continue
                tot = [r["total_ms"] for r in rows_]
                s = {"total_ms": stats(tot), "frames_per_s": float(n / (np.median(tot) * 1e-3)), "steps": len(rows_)}
                if arm == "device":
                    for key in ("upload_ms", "run_ms", "commit_ms", "advance_ms"):
                        s[key] = stats([r[key] for r in rows_])
                    s["captures_per_step"] = float(np.mean([r["captures"] for r in rows_]))
                    s["replayed_share"] = float(np.mean([r["captures"] == 0 for r in rows_]))
                    s["all_equal_to_host"] = all(r["equal_to_host"] for r in rows_)
                res.setdefault("summary", {}).setdefault(arm, {})[name] = s
        res["gpu_after"] = gpu_info()
    finally:
        ca.close(); cb.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res.get("summary"), indent=1))


if __name__ == "__main__":
    main()
