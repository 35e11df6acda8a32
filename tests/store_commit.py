"""What dsdtm_batch_commit_store does to the map store, twice over, from a store-mode step's fetched outputs:

- `host_commit` makes the calls a caller makes without it: dsdtm_store_set_points for the new points, dsdtm_store_append_keyframe per
  key frame in frame order, dsdtm_store_update_points for the bad flags and dsdtm_store_set_found for the counts;
- `model` builds the expected tables in numpy from the store as it was before the commit (dsdtm_store_fetch), in either row mode --
  appended key frames, or key frames filling reserved empty rows, which no existing call can do.

The found rule (MapPoint::IncreaseFound on every match, EraseFound on every match whose residual norm is above the threshold unless its
point was bad when the commit started, bad when the count ends <= 0) is evaluated once, in `found_update`, for both."""
import numpy as np

import oracle as O
from dsdtm_b200 import capi
from dsdtm_b200.workload import feature_normals


def step_outputs(c, cur_slots, want=None, keyframes=True):
    """the fetched outputs of the last flags-7/15 store-mode run that the commit reads"""
    poses, nm, m, res, _ = c.batch_fetch_track()
    out = dict(poses=poses, nm=nm, m=m, res=res, cur_slots=np.asarray(cur_slots, np.int32), keyframes=keyframes,
               want=np.ones(len(nm), bool) if want is None else np.asarray(want, bool))
    if keyframes:
        out["n_new"], out["corners"], out["lifted"], _ = c.batch_fetch_keyframe()
    return out


def found_update(found, bad, out, thr):
    """-> (new counts, ids of the matched points, bad flags of those points after the commit)"""
    found = found.copy()
    thr = np.float64(np.float32(thr))
    ids = []
    for i in range(len(out["nm"])):
        k = int(out["nm"][i])
        if k < 0:
            continue
        p = out["m"][i]["point"][:k]
        np.add.at(found, p, 1)
        erase = (out["res"][i][:k] > thr) & (bad[p] == 0)
        np.add.at(found, p[erase], -1)
        ids.append(p)
    ids = np.unique(np.concatenate(ids)) if ids else np.zeros(0, np.int32)
    return found, ids, np.where(found[ids] <= 0, 1, bad[ids]).astype(np.int32)


def keyframe_rows(cam, out):
    """per key frame (frame order): (frame, STORE_FEAT_DT rows with is_obs as the caller passes it, new point positions)"""
    kfs = []
    if not out["keyframes"]:
        return kfs
    for i in range(len(out["nm"])):
        k = int(out["nm"][i])
        if k < 0 or not out["want"][i]:
            continue
        nn = int(out["n_new"][i])
        F = np.zeros(k + nn, capi.STORE_FEAT_DT)
        mt = out["m"][i][:k]
        F["mp"][:k] = mt["point"]; F["level"][:k] = mt["level"]; F["px"][:k] = mt["px"]; F["is_obs"][:k] = 1
        if k:
            F["normal"][:k] = feature_normals(cam, mt["px"].astype(np.float32))
        lf = out["lifted"][i][:nn]
        F["level"][k:] = out["corners"][i][:nn]["level"]; F["px"][k:] = lf["px"]; F["normal"][k:] = lf["normal"]
        ok = lf["status"] == capi.LIFT_OK
        F["mp"][k:] = -1
        F["is_obs"][k:] = ok
        kfs.append((i, F, ok, lf["point_w"][ok]))
    return kfs


def host_commit(c, cam, out, thr, state=None):
    """the commit through the existing calls on context c (append mode). state = (bad flags, found counts) of every point as the caller
    keeps them; None reads them from the store. Returns per frame (kf_row, point_first, n_points)."""
    if state is None:
        _, _, P, found = c.store_fetch()
        state = (P["bad"], found)
    n = len(out["nm"])
    row, pf, npt = np.full(n, -1, np.int32), np.full(n, -1, np.int32), np.zeros(n, np.int32)
    found, ids, bad = found_update(state[1], state[0], out, thr)
    for i, F, ok, pw in keyframe_rows(cam, out):
        p0 = c.store_points
        if len(pw):
            c.store_set_points(p0, pw)
        mp = F["mp"]
        k = int(out["nm"][i])
        mp[k:][ok] = p0 + np.arange(len(pw), dtype=np.int32)
        pose = out["poses"][i]
        row[i] = c.store_append_keyframe(int(out["cur_slots"][i]), pose, O.se3_inv(pose)[4:], F)
        pf[i], npt[i] = p0, len(pw)
    if len(ids):
        c.store_update_points(ids, None, bad)
        c.store_set_found(ids, found[ids])
    return row, pf, npt


def model(pre, cam, out, thr, kf_rows=None):
    """the store after the commit, built from pre = store_fetch() before it: (K, F, P, found) and per frame (kf_row, point_first,
    n_points). kf_rows: reserved empty key-frame rows per frame, or None (append)."""
    K, F, P, found = (a.copy() for a in pre)
    n = len(out["nm"])
    row, pf, npt = np.full(n, -1, np.int32), np.full(n, -1, np.int32), np.zeros(n, np.int32)
    found, ids, bad = found_update(found, P["bad"], out, thr)
    P["bad"][ids] = bad
    feats, pts, kfs_new, f_found = [F], [P], [K], [found]
    n_f, n_p, n_k = len(F), len(P), len(K)
    last = {}                                                   # point -> newest observing feature row of this commit
    for i, Fk, ok, pw in keyframe_rows(cam, out):
        k = int(out["nm"][i])
        Fk = Fk.copy()
        Fk["mp"][k:][ok] = n_p + np.arange(len(pw), dtype=np.int32)
        r = int(kf_rows[i]) if kf_rows is not None else n_k
        Fk["is_obs"] = np.where(Fk["is_obs"] != 0, r + 1, 0)
        Np = np.zeros(len(pw), capi.STORE_POINT_DT)
        Np["point_w"] = pw; Np["last_obs"] = -1
        pts.append(Np); f_found.append(np.ones(len(pw), np.int32))
        for j in range(len(Fk)):
            if Fk["is_obs"][j]:
                p = int(Fk["mp"][j])
                Fk["next_obs"][j] = last.get(p, int(P["last_obs"][p]) if p < len(P) else -1)
                last[p] = n_f + j
            else:
                Fk["next_obs"][j] = -1
        kr = np.zeros(1, capi.STORE_KF_DT)
        pose = out["poses"][i]
        kr["slot"] = out["cur_slots"][i]; kr["feat_begin"] = n_f; kr["feat_count"] = len(Fk)
        kr["pose_c2w"] = pose; kr["center"] = O.se3_inv(pose)[4:]
        if kf_rows is None:
            kfs_new.append(kr); n_k += 1
        else:
            kfs_new[0][r] = kr[0]
        feats.append(Fk)
        row[i], pf[i], npt[i] = r, n_p, len(pw)
        n_f += len(Fk); n_p += len(pw)
    K, F, P, found = np.concatenate(kfs_new), np.concatenate(feats), np.concatenate(pts), np.concatenate(f_found)
    for p, g in last.items():
        P["last_obs"][p] = g
    return (K, F, P, found), (row, pf, npt)


def assert_stores_equal(a, b):
    for x, y, name in zip(a, b, ("key frames", "features", "points", "found")):
        assert len(x) == len(y), (name, len(x), len(y))
        assert x.tobytes() == y.tobytes(), name
