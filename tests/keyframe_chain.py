"""The key-frame half of the batched chain on the CPU (Tracking::CraeteKeyframe, ref: src/Tracking.cpp:412-464, after the tracked pose):
tests/cpp/keyframe_chain_oracle.cpp compiled with the oracle's sources, and the same steps composed in Python from the oracle's calls --
O.detect_cells + O.detect_select + O.undistort_points / feature_depth / unproject, the composition test_gpu_sequence.py uses at its key
frames. Shared by the CPU and GPU tests of dsdtm_batch_run flags 15."""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle as O
import track_select as TS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIFTED_DT = np.dtype([("px", "<f4", 2), ("depth", "<f4"), ("status", "<i4"), ("normal", "<f8", 3), ("point_w", "<f8", 3)])
LIFT_OK, LIFT_NO_DEPTH = 1, 2
EUROC_DIST = (-0.28368365, 0.07451284, -0.00010473, -3.55590700e-05, 0.0)      # ref: Config/EuRoc.yaml:16-20
_lib = None


def _kf():
    global _lib
    if _lib is None:
        d = os.path.join(ROOT, "tests", "cpp", "_build")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libkeyframe_chain_oracle.so")
        srcs = [os.path.join(ROOT, "tests", "cpp", "keyframe_chain_oracle.cpp"), os.path.join(ROOT, "oracle", "dsdtm_oracle.cpp")]
        deps = srcs + [os.path.join(ROOT, "oracle", "dsdtm_oracle.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
            subprocess.check_call(["g++", "-O3", "-std=c++17", "-ffp-contract=off", "-fPIC", "-pthread", "-shared"] + srcs + ["-o", so])
        _lib = C.CDLL(so)
    return _lib


def keyframe_chain(cam, levels, cell_size, min_dist, max_fts, thr, dist, depth_scale, cur_imgs, matches, n_matches, poses, depth16=None,
                   has_depth=None, want=None, n_threads=4):
    """The C++ reference for n pairs. matches: (n, 200) MATCH_DT; poses: (n, 7) c2w after PoseOptimization; depth16: (n, h, w) uint16 or
    None. Returns dict(n_new, corners (n, max_fts) CORNER_DT, lifted (n, max_fts) LIFTED_DT, tied (n,) bool, occ_skipped (n,))."""
    p = O._p
    n = len(n_matches)
    out = dict(n_new=np.zeros(n, np.int32), corners=np.zeros((n, max_fts), O.CORNER_DT), lifted=np.zeros((n, max_fts), LIFTED_DT),
               tied=np.zeros(n, np.uint8), occ_skipped=np.zeros(n, np.int32))
    d16 = None if depth16 is None else np.ascontiguousarray(depth16, np.uint16)
    hd = None if has_depth is None else np.ascontiguousarray(has_depth, np.int32)
    wt = None if want is None else np.ascontiguousarray(want, np.uint8)
    _kf().orc_keyframe_chain(C.byref(cam), int(levels), int(cell_size), int(min_dist), int(max_fts), C.c_float(thr),
                             p(np.ascontiguousarray(dist, np.float32)), C.c_float(depth_scale), n, p(O.u8(cur_imgs)),
                             p(np.ascontiguousarray(matches, TS.MATCH_DT)), p(np.ascontiguousarray(n_matches, np.int32)),
                             p(np.ascontiguousarray(poses, np.float64)), p(d16), p(hd), p(wt), int(n_threads), p(out["n_new"]),
                             p(out["corners"]), p(out["lifted"]), p(out["tied"]), p(out["occ_skipped"]))
    out["tied"] = out["tied"].astype(bool)
    return out


def compose(cam, levels, cell_size, min_dist, max_fts, thr, dist, depth_scale, cur_img, px, pose, depth16=None):
    """One pair through the oracle's Python calls. px: (m, 2) float32 match positions. Returns (corners CORNER_DT, lifted LIFTED_DT,
    occupancy indices skipped, tied: two cells above 20 share a score, so the selection depends on std::sort's order of ties)."""
    h, w = cur_img.shape
    rows, cols = O.grid_dims(w, h, cell_size)
    occ = np.zeros(rows * cols, np.uint8)
    skipped = 0
    for q in px:
        k = int(q[1] / np.float32(cell_size)) * cols + int(q[0] / np.float32(cell_size))
        if 0 <= k < rows * cols:
            occ[k] = 1
        else:
            skipped += 1
    mask = np.full((h, w), 255, np.uint8)
    for r in (cell_size, min_dist):
        for q in px:
            O.circle_fill(mask, O.cvround(q[0]), O.cvround(q[1]), r, 0)
    if max_fts - len(px) <= 0:
        return np.zeros(0, O.CORNER_DT), np.zeros(0, LIFTED_DT), skipped, False
    packed, offs, ws, hs = O.pyramid(cur_img, levels)
    cells = O.detect_cells(packed, offs, ws, hs, cell_size, occ, thr)
    above = cells["score"][cells["score"] > 20]
    tied = len(np.unique(above)) < len(above)
    new, _ = O.detect_select(cells, mask, cell_size, max_fts, n_existing=len(px))
    lf = np.zeros(len(new), LIFTED_DT)
    if len(new):
        und = O.undistort_points(cam, dist, np.stack([new["x"], new["y"]], 1).astype(np.float32))
        df = None if depth16 is None else O.depth_convert(depth16, depth_scale)
        for i in range(len(new)):
            lf[i]["px"] = und[i]
            lf[i]["normal"] = O.feature_normal(cam, und[i])
            z = -1.0 if df is None else O.feature_depth(df, und[i])
            lf[i]["depth"] = z
            lf[i]["status"] = LIFT_NO_DEPTH
            if z >= 0:
                lf[i]["point_w"] = O.unproject(cam, pose, und[i], z)
                lf[i]["status"] = LIFT_OK
    return new, lf, skipped, tied


def same_corners(got, want):
    """x, y, level and score bits, in order"""
    return (len(got) == len(want) and (got["x"] == want["x"]).all() and (got["y"] == want["y"]).all()
            and (got["level"] == want["level"]).all() and (got["score"].view(np.uint32) == want["score"].view(np.uint32)).all())
