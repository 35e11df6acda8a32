"""TEST INFRASTRUCTURE -- ctypes loader for oracle/_ref/libdsdtm_ref.so: the reference's OWN hot-path translation units
(<reference>/src/{Sprase_ImageAlign,Feature_alignment,Feature_detection,Camera,Frame,MapPoint,Keyframe,Map,Config}.cpp and
Thirdparty/fast), compiled unmodified against the stand-in third-party headers of tests/ref_shim by `make -C oracle ref_dsdtm`,
driven through oracle/ref_dsdtm_wrap.cpp.

Only tests/ (and the golden generator tests/golden/make_golden_refpin.py) import this module. It exists to pin
oracle/dsdtm_oracle.cpp to the reference's source for the floating-point rows of SURVEY.md 8(a).
"""
import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = {False: os.path.join(_HERE, "_ref", "libdsdtm_ref.so"), True: os.path.join(_HERE, "_ref", "libdsdtm_ref_tree.so")}


def _reference_root():
    """A checkout of the original DSDTM sources (github.com/gaochq/DSDTM): DSDTM_REFERENCE, else the location BASELINE.json
    records as reference_path. Without a checkout there the pin tests skip."""
    if os.environ.get("DSDTM_REFERENCE"):
        return os.environ["DSDTM_REFERENCE"]
    try:
        with open(os.path.join(os.path.dirname(_HERE), "BASELINE.json")) as f:
            return json.load(f).get("reference_path") or ""
    except (OSError, ValueError):
        return ""


REFERENCE = _reference_root()


def available(tree=False):
    return os.path.exists(_LIBS[tree])


def build(force=False):
    """Only possible where REFERENCE holds a checkout of the reference."""
    if REFERENCE and os.path.isdir(os.path.join(REFERENCE, "src")) and (force or not (available(False) and available(True))):
        subprocess.check_call(["make", "-C", _HERE, "ref_dsdtm", "REF=" + REFERENCE], stdout=subprocess.DEVNULL)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, np.float64)


def write_config(cam, levels=5, cell=15, max_fts=300, min_fts=50, min_dist=15, max_tkfts=200, dist=(0, 0, 0, 0, 0)):
    """The keys the hot-path classes read (ref: src/Camera.cpp:34-49, src/Frame.cpp:51-52, src/Feature_detection.cpp:13-17,
    src/Feature_alignment.cpp:24-28, src/Sprase_ImageAlign.cpp:14), in the flat YAML layout of the reference's Config/*.yaml."""
    kv = {"Camera.f": cam["f"], "Camera.fx": cam["fx"], "Camera.fy": cam["fy"], "Camera.cx": cam["cx"], "Camera.cy": cam["cy"],
          "Camera.k1": dist[0], "Camera.k2": dist[1], "Camera.p1": dist[2], "Camera.p2": dist[3], "Camera.k3": dist[4],
          "Camera.width": cam["width"], "Camera.height": cam["height"], "Camera.MaxPyraLevels": levels, "Camera.MinPyraLevels": 0,
          "Camera.CellSize": cell, "Camera.Max_fts": max_fts, "Camera.Min_fts": min_fts, "Camera.Min_dist": min_dist,
          "Camera.Max_tkfts": max_tkfts,
          # read by the Tracking constructor (ref: src/Tracking.cpp:20-29); values of Config/kinect.yaml
          "Camera.depth_scale": 1000.0, "Optimization.MaxIter": 8, "KeyFrame.min_rot": 0.08, "KeyFrame.min_trans": 0.08,
          "KeyFrame.min_features": 25, "KeyFrame.min_dist": 0.12}
    fd, path = tempfile.mkstemp(suffix=".yaml", prefix="dsdtm_refpin_")
    with os.fdopen(fd, "w") as f:
        f.write("%YAML:1.0\n---\n")
        for k, v in kv.items():
            f.write("%s: %s\n" % (k, repr(float(v)) if isinstance(v, float) else v))
    return path


class Ref:
    """One loaded copy of the reference library, initialised for one camera / parameter set."""

    def __init__(self, cam, tree=False, **params):
        if not available(tree):
            raise RuntimeError("oracle/_ref/libdsdtm_ref.so is not built (needs the reference sources at %s: make -C oracle ref_dsdtm)" % (REFERENCE or "DSDTM_REFERENCE"))
        # the library keeps its objects (Config singleton, camera, frames, map) in globals: every Ref gets a private copy of the
        # shared object so that two parameter sets can be alive at once
        import shutil
        fd, self._so = tempfile.mkstemp(suffix=".so", prefix="dsdtm_ref_")
        os.close(fd)
        shutil.copyfile(_LIBS[tree], self._so)
        self.L = C.CDLL(self._so)
        os.unlink(self._so)          # stays mapped
        L = self.L
        L.ref_shitomasi.restype = C.c_float
        L.ref_frame_feature_depth.restype = C.c_float
        L.ref_frame_feature_depth.argtypes = [C.c_int, C.c_float, C.c_float]
        L.ref_frame_add_feature.argtypes = [C.c_int, C.c_float, C.c_float, C.c_int, C.c_int]
        L.ref_frame_unproject.argtypes = [C.c_int, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.ref_is_in_image.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int]
        L.ref_detect.argtypes = [C.c_int, C.c_double, C.c_int]
        L.ref_warp_affine.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p]
        self.cam = dict(cam)
        self.params = params
        path = write_config(cam, **params)
        try:
            if L.ref_init(path.encode()) != 0:
                raise RuntimeError("ref_init failed")
        finally:
            os.unlink(path)

    def reset(self):
        self.L.ref_reset_objects()

    # ---- frames
    def frame(self, img, pose_c2w, depth=None):
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape
        d = np.ascontiguousarray(depth, np.float32) if depth is not None else None
        return self.L.ref_frame_create(_p(img), w, h, _p(d), _p(_f64(pose_c2w)))

    def frame_level(self, fr, level):
        w = C.c_int(); h = C.c_int()
        self.L.ref_frame_level(fr, level, None, C.byref(w), C.byref(h))
        out = np.empty((h.value, w.value), np.uint8)
        self.L.ref_frame_level(fr, level, _p(out), C.byref(w), C.byref(h))
        return out

    def frame_set_pose(self, fr, pose):
        self.L.ref_frame_set_pose(fr, _p(_f64(pose)))

    def frame_pose(self, fr):
        p = np.empty(7); c = np.empty(3)
        self.L.ref_frame_get_pose(fr, _p(p), _p(c))
        return p, c

    def add_feature(self, fr, px, level, with_normal=True):
        return self.L.ref_frame_add_feature(fr, float(np.float32(px[0])), float(np.float32(px[1])), int(level), int(with_normal))

    def set_normal(self, fr, idx, n):
        self.L.ref_feature_set_normal(fr, idx, _p(_f64(n)))

    def set_mappoint(self, fr, idx, mp):
        self.L.ref_feature_set_mappoint(fr, idx, mp)

    def features(self, fr):
        n = self.L.ref_frame_feature_count(fr)
        px = np.empty((n, 2), np.float32); lv = np.empty(n, np.int32); nm = np.empty((n, 3)); mp = np.empty(n, np.int32)
        ini = np.empty(n, np.int32)
        self.L.ref_frame_features(fr, _p(px), _p(lv), _p(nm), _p(mp), _p(ini))
        return dict(px=px, level=lv, normal=nm, mp=mp, initial=ini)

    def frame_mappoints(self, fr, cap=4096):
        mp = np.empty(cap, np.int32)
        n = self.L.ref_frame_mappoints(fr, _p(mp), cap)
        return mp[:n].copy()

    def mask(self, fr):
        out = np.empty((self.cam["height"], self.cam["width"]), np.uint8)
        return out if self.L.ref_frame_mask(fr, _p(out)) else None

    def undistort_features(self, fr):
        self.L.ref_frame_undistort_features(fr)

    def feature_depth(self, fr, px):
        return float(self.L.ref_frame_feature_depth(fr, float(np.float32(px[0])), float(np.float32(px[1]))))

    def unproject(self, fr, px, d):
        out = np.empty(3)
        self.L.ref_frame_unproject(fr, float(np.float32(px[0])), float(np.float32(px[1])), float(np.float32(d)), _p(out))
        return out

    def is_visible(self, fr, p, boundary=0):
        return bool(self.L.ref_frame_is_visible(fr, _p(_f64(p)), int(boundary)))

    def world2pixel(self, fr, p):
        out = np.empty(2)
        self.L.ref_frame_world2pixel(fr, _p(_f64(p)), _p(out))
        return out

    def is_in_image(self, x, y, boundary, level=0):
        return bool(self.L.ref_is_in_image(float(np.float32(x)), float(np.float32(y)), int(boundary), int(level)))

    # ---- map
    def keyframe(self, fr):
        return self.L.ref_keyframe_create(fr)

    def mappoint(self, pos, kf):
        return self.L.ref_mappoint_create(_p(_f64(pos)), kf)

    def add_observation(self, mp, kf, feat_idx):
        self.L.ref_mappoint_add_observation(mp, kf, feat_idx)

    def increase_found(self, mp, n=1):
        self.L.ref_mappoint_increase_found(mp, n)

    def found(self, mp):
        return self.L.ref_mappoint_found(mp)

    def set_outlier(self, mp, bad=True):
        self.L.ref_mappoint_set_outlier(mp, int(bad))

    def kf_feature_set_mappoint(self, kf, idx, mp):
        self.L.ref_keyframe_feature_set_mappoint(kf, idx, mp)

    def closest_obs(self, mp, fr):
        kf = C.c_int(-1); fi = C.c_int(-1)
        ok = self.L.ref_mappoint_closest_obs(mp, fr, C.byref(kf), C.byref(fi))
        return bool(ok), kf.value, fi.value

    # ---- detection
    def shitomasi(self, img, u, v):
        img = np.ascontiguousarray(img, np.uint8)
        return float(self.L.ref_shitomasi(_p(img), img.shape[1], img.shape[0], int(u), int(v)))

    def set_existing(self, px):
        px = np.ascontiguousarray(px, np.float32).reshape(-1, 2)
        self.L.ref_detector_set_existing(_p(px), len(px))

    def set_existing_from_frame(self, fr):
        self.L.ref_detector_set_existing_from_frame(fr)

    def detect(self, fr, thr=5.0, first=True):
        return self.L.ref_detect(fr, float(thr), int(first))

    # ---- sparse alignment
    def sparse_align_run(self, cur, ref, max_level, min_level, max_iters):
        out = np.empty(7)
        n = self.L.ref_sparse_align_run(cur, ref, max_level, min_level, max_iters, _p(out))
        return out, n

    def sparse_align_linearize(self, cur, ref, level, pose_c2r, cap=1024):
        patch = np.empty((cap, 16)); jac = np.empty((cap * 16, 6)); pts = np.empty((cap, 3))
        H = np.empty((6, 6)); b = np.empty(6); chi2 = C.c_double(0); npts = C.c_int(0)
        n = self.L.ref_sparse_align_linearize(cur, ref, level, _p(_f64(pose_c2r)), cap, _p(patch), _p(jac), _p(pts), _p(H), _p(b),
                                              C.byref(chi2), C.byref(npts))
        assert n >= 0
        return dict(n=n, patch=patch[:n].copy(), jac=jac[:n * 16].copy(), pts=pts[:n].copy(), H=H, b=b, chi2=chi2.value, n_pts=npts.value)

    # ---- feature alignment
    def align2d(self, img, patch10, patch8, iters, px):
        img = np.ascontiguousarray(img, np.uint8)
        p = _f64(px).copy()
        ok = self.L.ref_align2d(_p(img), img.shape[1], img.shape[0], _p(np.ascontiguousarray(patch10, np.uint8)),
                                _p(np.ascontiguousarray(patch8, np.uint8)), int(iters), _p(p))
        return p, bool(ok)

    def best_search_level(self, A, max_level):
        return self.L.ref_best_search_level(_p(_f64(A).reshape(-1)), int(max_level))

    def warp_affine(self, A, img, px, ref_level, search_level):
        img = np.ascontiguousarray(img, np.uint8)
        out = np.empty(100, np.uint8)
        self.L.ref_warp_affine(_p(_f64(A).reshape(-1)), _p(img), img.shape[1], img.shape[0], float(np.float32(px[0])), float(np.float32(px[1])),
                               int(ref_level), int(search_level), _p(out))
        return out

    def solve_affine(self, kf, cur, feat_idx, mp):
        A = np.empty(4)
        self.L.ref_solve_affine(kf, cur, feat_idx, mp, _p(A))
        return A.reshape(2, 2)

    def find_match_direct(self, mp, cur, px):
        p = _f64(px).copy(); lv = C.c_int(0)
        ok = self.L.ref_find_match_direct(mp, cur, _p(p), C.byref(lv))
        return bool(ok), p, lv.value

    def reset_grid(self):
        self.L.ref_fa_reset_grid()

    def reproject_point(self, cur, mp):
        return bool(self.L.ref_fa_reproject_point(cur, mp))

    def search_local_points(self, cur):
        self.L.ref_fa_search_local_points(cur)

    # ---- Tracking (caller side of f-1)
    def tracking_create(self):
        self.L.ref_tracking_create()

    def keyframe_add_mappoint(self, kf, idx, mp):
        self.L.ref_keyframe_add_mappoint(kf, idx, mp)

    def close_keyframes(self, fr, cap=4096):
        ids = np.empty(cap, np.int32); d = np.empty(cap)
        n = self.L.ref_tracking_close_keyframes(fr, _p(ids), _p(d), cap)
        return ids[:n].copy(), d[:n].copy()

    def update_local_map(self, fr, cap=64):
        ids = np.empty(cap, np.int32); npts = C.c_int(0)
        n = self.L.ref_tracking_update_local_map(fr, _p(ids), cap, C.byref(npts))
        return ids[:n].copy(), npts.value

    def tracking_search_local_points(self):
        self.L.ref_tracking_search_local_points()

    # ---- SE3 stand-in
    def se3_exp(self, x):
        out = np.empty(7); self.L.ref_se3_exp(_p(_f64(x)), _p(out)); return out

    def se3_mul(self, a, b):
        out = np.empty(7); self.L.ref_se3_mul(_p(_f64(a)), _p(_f64(b)), _p(out)); return out

    def se3_inv(self, a):
        out = np.empty(7); self.L.ref_se3_inv(_p(_f64(a)), _p(out)); return out
