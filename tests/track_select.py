"""Python restatement of SearchLocalPoints' greedy selection (ref: src/Feature_alignment.cpp:71-121) over the records of the batched
refinement chain -- the rules of tests/oracle_seq.py's _oracle_search and of the host replay Feature_Alignment::SearchFused -- on a
full-size mask painted with the pinned circle (oracle circle_fill). Shared by the CPU and GPU tests of the tracked-pose chain."""
import ctypes as C
import os
import subprocess

import numpy as np

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MATCH_DT = np.dtype([("point", "<i4"), ("px", "<f4", 2), ("level", "<i4")])
_chain_lib = None

GATES = 2 | 4          # OBS_OK | REF_OK
CONVERGED = 8


def replay(reproj, found, width, height, cell_size, cap=200):
    """reproj: one pair's REPROJ records (index = feature j = ReprojectPoint order); found: per-record found counts.
    Returns the matches in match order as a list of (point j, float32 px[2], level)."""
    cells = {}
    for j in range(len(reproj)):
        if reproj[j]["cell"] >= 0:
            cells.setdefault(int(reproj[j]["cell"]), []).append(j)
    mask = np.full((height, width), 255, np.uint8)
    out = []
    for k in sorted(cells):
        for j in sorted(cells[k], key=lambda q: -int(found[q])):            # stable, like std::list::sort
            r = reproj[j]
            if mask[O.cvround(np.float32(r["px_proj"][1])), O.cvround(np.float32(r["px_proj"][0]))] != 255:
                continue
            if (r["flags"] & GATES) != GATES or r["level"] < 0 or not (r["flags"] & CONVERGED):
                continue
            p = r["px"].astype(np.float32)
            out.append((j, p, int(r["level"])))
            O.circle_fill(mask, O.cvround(p[0]), O.cvround(p[1]), cell_size, 0)
            break
        if cap is not None and len(out) >= cap:
            break
    return out


def assert_matches_equal(got, n_got, want):
    """device / oracle MATCH records (first n_got valid) == replay list: point, float px bits, level, order"""
    assert n_got == len(want)
    for m, (j, p, lv) in zip(got[:n_got], want):
        assert int(m["point"]) == j and int(m["level"]) == lv
        assert m["px"].view(np.uint32).tolist() == p.view(np.uint32).tolist()


def make_batch(cam, n, ppp, seed0=61, n_scenes=3, empty_pair=None, trans=0.03, rot_deg=0.8):
    """n frame pairs over n_scenes rendered scenes (every other one at a non-identity reference pose), ppp reference features per pair
    detected on the oracle. empty_pair: index of a pair whose features carry no map point (no candidates, no matches)."""
    import helpers as H
    from dsdtm_b200 import synth as S
    T_ref = S.pose_from_xi(np.r_[0.2, -0.1, 0.05, 0.03, -0.02, 0.04])
    prs = [S.make_pair(seed0 + k, cam, trans=trans, rot_deg=rot_deg, ref_pose=(T_ref if k % 2 else None)) for k in range(n_scenes)]
    det = [H.detect_oracle(pr["ref_img"], 5, 15, ppp) for pr in prs]
    feats = np.zeros((n, ppp), O.REF_FEAT_DT); nf = np.zeros(n, np.int32); centers = np.zeros((n, 3))
    poses_ref = np.zeros((n, 7)); poses_in = np.tile(S.IDENTITY, (n, 1))
    ref_pyrs, cur_imgs = [], []
    for i in range(n):
        pr = prs[i % n_scenes]
        corners, pyr = det[i % n_scenes]
        F = H.ref_feats_from_corners(cam, corners, pr["ref_points"])
        if i == empty_pair:
            F["initial"] = 0
        nf[i] = len(F); feats[i, :nf[i]] = F; centers[i] = O.se3_inv(pr["T_ref"])[4:]; poses_ref[i] = pr["T_ref"]
        ref_pyrs.append(pyr[0]); cur_imgs.append(pr["cur_img"])
    return dict(cam=cam, n=n, ppp=ppp, prs=prs, feats=feats, n_feats=nf, centers=centers, poses_ref=poses_ref, poses_in=poses_in,
                ref_pyrs=np.stack(ref_pyrs), cur_imgs=np.stack(cur_imgs))


def _chain():
    """tests/cpp/track_chain_oracle.cpp compiled with the oracle's sources (oracle flags: -O3, no FMA contraction, threads)"""
    global _chain_lib
    if _chain_lib is None:
        d = os.path.join(ROOT, "tests", "cpp", "_build")
        os.makedirs(d, exist_ok=True)
        so = os.path.join(d, "libtrack_chain_oracle.so")
        srcs = [os.path.join(ROOT, "tests", "cpp", "track_chain_oracle.cpp"), os.path.join(ROOT, "oracle", "dsdtm_oracle.cpp")]
        deps = srcs + [os.path.join(ROOT, "oracle", "dsdtm_oracle.h")]
        if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
            subprocess.check_call(["g++", "-O3", "-std=c++17", "-ffp-contract=off", "-fPIC", "-pthread", "-shared"] + srcs + ["-o", so])
        _chain_lib = C.CDLL(so)
    return _chain_lib


def pair_batch_track(cam, levels, cell_size, ref_pyrs, cur_imgs, feats, n_feats, ref_centers, poses_ref, poses_in, max_level, min_level,
                     max_iters, points_per_pair, max_search_level, align_iters, found=None, ba_iters=100, n_threads=4):
    """The oracle's whole tracked-pose chain: pair_batch_map + SearchLocalPoints' selection + PoseOptimization per pair.
    Returns dict(poses_c2r, n_tracked, reproj, poses (c2w after PoseOptimization), n_matches, matches (n, 200), res_norm (n, 200),
    summaries)."""
    n_pairs = len(n_feats)
    feats = np.ascontiguousarray(feats, O.REF_FEAT_DT)
    fpp = feats.size // n_pairs
    p = O._p
    poses_out = np.empty((n_pairs, 7)); n_tracked = np.empty(n_pairs, np.int32)
    rep = np.zeros((n_pairs, points_per_pair), O.REPROJ_DT)
    poses_trk = np.empty((n_pairs, 7)); nm = np.zeros(n_pairs, np.int32)
    matches = np.zeros((n_pairs, 200), MATCH_DT); res = np.zeros((n_pairs, 200)); summ = np.zeros(n_pairs, O.BA_SUMMARY_DT)
    f = None if found is None else np.ascontiguousarray(found, np.int32).reshape(n_pairs, points_per_pair)
    _chain().orc_pair_batch_track(C.byref(cam), int(levels), int(cell_size), p(O.u8(ref_pyrs)), p(O.u8(cur_imgs)), n_pairs, p(feats), fpp,
                                  p(np.ascontiguousarray(n_feats, np.int32)), p(np.ascontiguousarray(ref_centers, np.float64)),
                                  p(np.ascontiguousarray(poses_ref, np.float64)), p(np.ascontiguousarray(poses_in, np.float64)),
                                  int(max_level), int(min_level), int(max_iters), int(points_per_pair), int(max_search_level),
                                  int(align_iters), p(f), int(ba_iters), int(n_threads), p(poses_out), p(n_tracked), p(rep), p(poses_trk),
                                  p(nm), p(matches), p(res), p(summ))
    return dict(poses_c2r=poses_out, n_tracked=n_tracked, reproj=rep, poses=poses_trk, n_matches=nm, matches=matches, res_norm=res,
                summaries=summ)
