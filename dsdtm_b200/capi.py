"""ctypes binding of include/dsdtm_gpu.h (libdsdtm_gpu.so). Harness-side only: tests, bench.py and smoke() call the
CUDA path through this C-ABI exactly as the C++ adapters in dsdtm_b200/host do. There is NO CPU fallback: if the library
is missing or no CUDA device is present, everything here raises."""
import ctypes as C
import os

import numpy as np

from . import build as _build

STAGES = ("pyramid", "fast", "sparse_align", "align2d", "warp_affine", "cand_prep", "local_map", "ingest", "pose_opt")

CORNER_DT = np.dtype([("x", "<i4"), ("y", "<i4"), ("level", "<i4"), ("score", "<f4")])
REF_FEAT_DT = np.dtype([("px", "<f4", 2), ("level", "<i4"), ("initial", "<i4"),
                        ("normal", "<f8", 3), ("point_w", "<f8", 3)])
ITER_LOG_DT = np.dtype([("level", "<i4"), ("iter", "<i4"), ("n_pts", "<i4"), ("flags", "<i4"),
                        ("chi2", "<f8"), ("x", "<f8", 6)])
CANDIDATE_DT = np.dtype([("ref_slot", "<i4"), ("ref_level", "<i4"), ("ref_px", "<f4", 2), ("ref_normal", "<f8", 3),
                         ("ref_point_w", "<f8", 3), ("kf_center", "<f8", 3), ("pose_c2r", "<f8", 7), ("px", "<f8", 2)])
assert CANDIDATE_DT.itemsize == 160
KF_VIEW_DT = np.dtype([("slot", "<i4"), ("reserved", "<i4"), ("center", "<f8", 3), ("pose_c2w", "<f8", 7)])
OBS_DT = np.dtype([("kf", "<i4"), ("level", "<i4"), ("px", "<f4", 2), ("normal", "<f8", 3), ("point_w", "<f8", 3)])
MAP_POINT_DT = np.dtype([("point_w", "<f8", 3), ("obs_begin", "<i4"), ("obs_count", "<i4")])
REPROJ_DT = np.dtype([("px_proj", "<f8", 2), ("px", "<f8", 2), ("cell", "<i4"), ("obs", "<i4"), ("flags", "<i4"), ("level", "<i4")])
assert KF_VIEW_DT.itemsize == 88 and OBS_DT.itemsize == 64 and MAP_POINT_DT.itemsize == 32 and REPROJ_DT.itemsize == 48
LM_IN_IMAGE, LM_OBS_OK, LM_REF_OK, LM_CONVERGED = 1, 2, 4, 8
LIFTED_DT = np.dtype([("px", "<f4", 2), ("depth", "<f4"), ("status", "<i4"), ("normal", "<f8", 3), ("point_w", "<f8", 3)])
assert LIFTED_DT.itemsize == 64
LIFT_SKIPPED, LIFT_OK, LIFT_NO_DEPTH = 0, 1, 2
MAP_KF_DT = np.dtype([("pt_begin", "<i4"), ("pt_count", "<i4"), ("t", "<f8", 3)])
assert MAP_KF_DT.itemsize == 32
BA_OBS_DT = np.dtype([("normal", "<f8", 3), ("point_w", "<f8", 3), ("level", "<i4"), ("reserved", "<i4")])
BA_SUMMARY_DT = np.dtype([("iterations", "<i4"), ("termination", "<i4"), ("n_successful", "<i4"), ("n_obs", "<i4"),
                          ("initial_cost", "<f8"), ("final_cost", "<f8")])
assert BA_OBS_DT.itemsize == 56 and BA_SUMMARY_DT.itemsize == 32
BA_FUNCTION_TOL, BA_PARAMETER_TOL, BA_GRADIENT_TOL, BA_NO_CONVERGENCE, BA_FAILURE, BA_MIN_RADIUS, BA_NO_RESIDUALS = range(7)
BA_MAX_OBS = 4096
MATCH_DT = np.dtype([("point", "<i4"), ("px", "<f4", 2), ("level", "<i4")])
assert MATCH_DT.itemsize == 16
TRACK_MAX_MATCHES = 200
ADV_ADVANCED, ADV_KEYFRAME, ADV_HELD_OVERFLOW, ADV_HELD_CALLER = 0, 1, 2, 3   # dsdtm_batch_advance's per-frame status
CIRCLE_DT = np.dtype([("px", "<f4", 2), ("radius", "<i4"), ("reserved", "<i4")])
assert CIRCLE_DT.itemsize == 16
# device-resident map store (dsdtm_store_*)
STORE_KF_DT = np.dtype([("slot", "<i4"), ("feat_begin", "<i4"), ("feat_count", "<i4"), ("reserved", "<i4"), ("pose_c2w", "<f8", 7),
                        ("center", "<f8", 3)])
STORE_FEAT_DT = np.dtype([("mp", "<i4"), ("level", "<i4"), ("px", "<f4", 2), ("normal", "<f8", 3), ("is_obs", "<i4"), ("next_obs", "<i4")])
STORE_POINT_DT = np.dtype([("point_w", "<f8", 3), ("bad", "<i4"), ("last_obs", "<i4")])
STORE_CAND_DT = np.dtype([("mp", "<i4"), ("order", "<i4"), ("r", REPROJ_DT)])
assert STORE_KF_DT.itemsize == 96 and STORE_FEAT_DT.itemsize == 48 and STORE_POINT_DT.itemsize == 32 and STORE_CAND_DT.itemsize == 56
# dsdtm_batch_run flags: 1 = rebuild the cur pyramids, 2 = the refinement chain (batch_stage_map), 4 (with 2) = SearchLocalPoints'
# selection + PoseOptimization behind it (batch_stage_track): flags 7 ends in the tracked pose of every pair; 8 (with 4) = the key frame
# behind the tracked pose (batch_stage_keyframe): flags 15 ends in the new corners and their lifted records
RUN_PYRAMID, RUN_CHAIN, RUN_TRACK, RUN_KEYFRAME = 1, 2, 4, 8


class Cam(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("fx", C.c_float), ("fy", C.c_float),
                ("cx", C.c_float), ("cy", C.c_float), ("f", C.c_float)]


class TrackIn(C.Structure):
    _fields_ = [("ref_slot", C.c_int32), ("cur_slot", C.c_int32), ("img", C.c_void_p), ("stride", C.c_int32),
                ("feats", C.c_void_p), ("n_feats", C.c_int32), ("ref_center", C.c_double * 3), ("pose_ref_c2w", C.c_double * 7),
                ("pose_c2r_in", C.c_double * 7), ("max_level", C.c_int32), ("min_level", C.c_int32), ("max_iters", C.c_int32),
                ("kfs", C.c_void_p), ("n_kfs", C.c_int32), ("obs", C.c_void_p), ("n_obs", C.c_int32), ("pts", C.c_void_p), ("n_pts", C.c_int32),
                ("max_search_level", C.c_int32), ("align_iters", C.c_int32)]


class TrackOut(C.Structure):
    _fields_ = [("pose_c2r", C.c_double * 7), ("pose_cur_c2w", C.c_double * 7), ("cur_center", C.c_double * 3), ("n_tracked", C.c_int32),
                ("reserved", C.c_int32)]


class Params(C.Structure):
    _fields_ = [("levels", C.c_int), ("cell_size", C.c_int), ("max_feats", C.c_int), ("max_patches", C.c_int),
                ("max_frames", C.c_int), ("max_batch", C.c_int)]


class DsdtmError(RuntimeError):
    pass


_lib = None

# every symbol include/dsdtm_gpu.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "dsdtm_abi_version", "dsdtm_create", "dsdtm_create_error", "dsdtm_destroy", "dsdtm_last_error", "dsdtm_sync",
    "dsdtm_level_info", "dsdtm_frame_stride", "dsdtm_host_alloc", "dsdtm_host_free", "dsdtm_launch_count",
    "dsdtm_profile", "dsdtm_profile_get", "dsdtm_frame_upload_pyramid", "dsdtm_frames_upload_pyramid",
    "dsdtm_frames_build_pyramid", "dsdtm_frame_download_level", "dsdtm_fast_cells", "dsdtm_fast_cells_batch",
    "dsdtm_fast_score_map", "dsdtm_grid_dims", "dsdtm_sparse_align", "dsdtm_sparse_align_batch",
    "dsdtm_align2d_batch", "dsdtm_warp_affine_batch", "dsdtm_batch_stage", "dsdtm_batch_run", "dsdtm_batch_fetch",
    "dsdtm_pair_batch_e2e", "dsdtm_last_run_ms", "dsdtm_timer_start", "dsdtm_timer_stop", "dsdtm_set_option", "dsdtm_feature_align_batch",
    "dsdtm_local_map_align_batch", "dsdtm_depth_upload", "dsdtm_depth_convert_f32", "dsdtm_keyframe_lift",
    "dsdtm_frame_upload_pyramid_host", "dsdtm_frames_upload_clahe_pyramid", "dsdtm_track_frame",
    "dsdtm_pose_optimize", "dsdtm_pose_optimize_batch", "dsdtm_map_table_upload", "dsdtm_close_keyframes", "dsdtm_probe_fp64", "dsdtm_frame_upload_pyramid_async", "dsdtm_track_frame_store", "dsdtm_store_set_points", "dsdtm_store_update_points", "dsdtm_store_append_keyframe", "dsdtm_store_set_keyframe", "dsdtm_store_clear", "dsdtm_store_track", "dsdtm_frame_upload_level", "dsdtm_batch_stage_map", "dsdtm_batch_fetch_map", "dsdtm_track_batch_e2e",
    "dsdtm_batch_stage_track", "dsdtm_batch_fetch_track", "dsdtm_detect", "dsdtm_detect_batch",
    "dsdtm_batch_stage_keyframe", "dsdtm_batch_fetch_keyframe", "dsdtm_batch_stage_store", "dsdtm_batch_fetch_store",
    "dsdtm_batch_advance", "dsdtm_batch_upload_step", "dsdtm_batch_fetch_ref", "dsdtm_graph_captures",
    "dsdtm_store_set_found", "dsdtm_store_size", "dsdtm_store_fetch", "dsdtm_batch_stage_track_live", "dsdtm_batch_commit_store",
]


def lib_path():
    return _build.LIB


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB):
        raise DsdtmError("libdsdtm_gpu.so is not built (run __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(_build.LIB)
    L.dsdtm_create.restype = C.c_void_p
    L.dsdtm_create.argtypes = [C.c_int, C.POINTER(Cam), C.POINTER(Params)]
    L.dsdtm_create_error.restype = C.c_char_p
    L.dsdtm_last_error.restype = C.c_char_p
    L.dsdtm_last_error.argtypes = [C.c_void_p]
    L.dsdtm_destroy.argtypes = [C.c_void_p]
    L.dsdtm_frame_stride.restype = C.c_size_t
    L.dsdtm_frame_stride.argtypes = [C.c_void_p]
    L.dsdtm_host_alloc.restype = C.c_void_p
    L.dsdtm_host_alloc.argtypes = [C.c_size_t]
    L.dsdtm_host_free.argtypes = [C.c_void_p]
    L.dsdtm_launch_count.restype = C.c_longlong
    L.dsdtm_launch_count.argtypes = [C.c_void_p]
    L.dsdtm_graph_captures.restype = C.c_longlong
    L.dsdtm_graph_captures.argtypes = [C.c_void_p]
    L.dsdtm_last_run_ms.restype = C.c_float
    L.dsdtm_last_run_ms.argtypes = [C.c_void_p]
    L.dsdtm_timer_stop.restype = C.c_float
    L.dsdtm_timer_stop.argtypes = [C.c_void_p]
    L.dsdtm_timer_start.argtypes = [C.c_void_p]
    _lib = L
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def pinned_empty(shape, dtype):
    """numpy array backed by pinned host memory (cudaMallocHost). Keep the returned array alive while in use."""
    L = load()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    ptr = L.dsdtm_host_alloc(max(n, 1))
    if not ptr:
        raise DsdtmError("cudaMallocHost failed")
    buf = (C.c_uint8 * max(n, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.ctypes.data] = ptr
    return arr


_PINNED = {}


class Context:
    def __init__(self, cam, levels=5, cell_size=15, max_feats=320, max_patches=320, max_frames=8, max_batch=1, device=0):
        L = load()
        self.L = L
        self.cam = Cam(cam["width"], cam["height"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["f"])
        self.prm = Params(levels, cell_size, max_feats, max_patches, max_frames, max_batch)
        self.h = L.dsdtm_create(device, C.byref(self.cam), C.byref(self.prm))
        if not self.h:
            raise DsdtmError("dsdtm_create failed: %s" % L.dsdtm_create_error().decode())
        self.levels = levels
        self.ws, self.hs, self.offs = [], [], []
        for l in range(levels):
            w, h, o = C.c_int(), C.c_int(), C.c_size_t()
            self._ck(L.dsdtm_level_info(C.c_void_p(self.h), l, C.byref(w), C.byref(h), C.byref(o)))
            self.ws.append(w.value); self.hs.append(h.value); self.offs.append(o.value)
        r, c_ = C.c_int(), C.c_int()
        L.dsdtm_grid_dims(C.c_void_p(self.h), C.byref(r), C.byref(c_))
        self.grid_rows, self.grid_cols = r.value, c_.value
        self.n_cells = r.value * c_.value
        self.width, self.height = cam["width"], cam["height"]
        self.store_points = self.store_keyframes = 0       # rows of the map store, as the store_* calls below leave them

    def _ck(self, rc):
        if rc != 0:
            raise DsdtmError("dsdtm error %d: %s" % (rc, self.L.dsdtm_last_error(C.c_void_p(self.h)).decode()))

    def close(self):
        if self.h:
            self.L.dsdtm_destroy(C.c_void_p(self.h))
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def hp(self):
        return C.c_void_p(self.h)

    def sync(self):
        self._ck(self.L.dsdtm_sync(self.hp))

    def launch_count(self):
        return int(self.L.dsdtm_launch_count(self.hp))

    def graph_captures(self):
        """CUDA graphs batch_run has captured on this context: a run that replays a captured step adds nothing"""
        return int(self.L.dsdtm_graph_captures(self.hp))

    def set_option(self, key, value):
        self._ck(self.L.dsdtm_set_option(self.hp, key.encode(), int(value)))

    def probe_fp64(self):
        """-> (TFLOP/s of dependency-free DFMA streams, DFMA warp instructions per clock and SM at the nominal max clock)"""
        t = C.c_double(0); w = C.c_double(0)
        self._ck(self.L.dsdtm_probe_fp64(self.hp, C.byref(t), C.byref(w)))
        return t.value, w.value

    def profile(self, on):
        self._ck(self.L.dsdtm_profile(self.hp, int(on)))

    def profile_get(self, reset=True):
        ms = (C.c_float * len(STAGES))()
        n = (C.c_int * len(STAGES))()
        self._ck(self.L.dsdtm_profile_get(self.hp, ms, n, int(reset)))
        return {s: (float(ms[i]), int(n[i])) for i, s in enumerate(STAGES)}

    # ---- pyramid
    def upload(self, slot, img):
        img = np.ascontiguousarray(img, np.uint8)
        assert img.shape == (self.height, self.width)
        self._ck(self.L.dsdtm_frame_upload_pyramid(self.hp, int(slot), _p(img), img.shape[1]))

    def upload_async(self, slot, img):
        """dsdtm_frame_upload_pyramid_async: queued on the context's stream, no synchronisation (later calls are ordered after it)"""
        img = np.ascontiguousarray(img, np.uint8)
        assert img.shape == (self.height, self.width)
        self._ck(self.L.dsdtm_frame_upload_pyramid_async(self.hp, int(slot), _p(img), img.shape[1]))

    def upload_level(self, slot, level, img):
        img = np.ascontiguousarray(img, np.uint8)
        assert img.shape == (self.hs[level], self.ws[level])
        self._ck(self.L.dsdtm_frame_upload_level(self.hp, int(slot), int(level), _p(img), img.shape[1]))

    def upload_with_levels(self, slot, img):
        """upload + pyramid + host copies of levels 1.. in one call -> list of level images (level 0 is img itself)"""
        img = np.ascontiguousarray(img, np.uint8)
        assert img.shape == (self.height, self.width)
        offs = self.offs
        last = self.levels - 1
        tail = offs[last] + self.ws[last] * self.hs[last] - offs[1]
        buf = np.empty(tail, np.uint8)
        self._ck(self.L.dsdtm_frame_upload_pyramid_host(self.hp, int(slot), _p(img), img.shape[1], _p(buf)))
        return [img] + [buf[offs[l] - offs[1]: offs[l] - offs[1] + self.ws[l] * self.hs[l]].reshape(self.hs[l], self.ws[l]) for l in range(1, self.levels)]

    def upload_clahe(self, first_slot, imgs, clip_limit=3.0, tiles=(8, 8), fetch=True):
        """CLAHE + pyramid for n raw images -> the equalised level-0 images (n, h, w) when fetch"""
        imgs = np.ascontiguousarray(imgs, np.uint8)
        if imgs.ndim == 2:
            imgs = imgs[None]
        assert imgs.shape[1:] == (self.height, self.width)
        out = np.empty_like(imgs) if fetch else None
        self._ck(self.L.dsdtm_frames_upload_clahe_pyramid(self.hp, int(first_slot), len(imgs), _p(imgs), C.c_double(clip_limit),
                                                          int(tiles[0]), int(tiles[1]), _p(out)))
        return out

    def upload_batch(self, first_slot, imgs):
        imgs = np.ascontiguousarray(imgs, np.uint8)
        assert imgs.shape[1:] == (self.height, self.width)
        self._ck(self.L.dsdtm_frames_upload_pyramid(self.hp, int(first_slot), imgs.shape[0], _p(imgs)))

    def build_pyramid(self, first_slot, n):
        self._ck(self.L.dsdtm_frames_build_pyramid(self.hp, int(first_slot), int(n)))

    def download_level(self, slot, level):
        out = np.empty((self.hs[level], self.ws[level]), np.uint8)
        self._ck(self.L.dsdtm_frame_download_level(self.hp, int(slot), int(level), _p(out)))
        return out

    # ---- FAST
    def fast_cells(self, slot, barrier=20, seed_score=5.0, occupied=None, n=1):
        cells = np.zeros(n * self.n_cells, CORNER_DT)
        occ = np.ascontiguousarray(occupied, np.uint8) if occupied is not None else None
        self._ck(self.L.dsdtm_fast_cells_batch(self.hp, int(slot), int(n), int(barrier), C.c_float(seed_score), _p(occ), _p(cells)))
        return cells if n == 1 else cells.reshape(n, self.n_cells)

    def detect(self, slot, threshold=5.0, occupied=None, mask=None, circles=None, max_new=300, n=1):
        """Feature_detector::detect for the n slots slot..slot+n-1 (dsdtm_detect for n == 1, dsdtm_detect_batch otherwise).
        occupied: (n, n_cells) or None; mask: (n, h, w) uint8 or None; circles: one CIRCLE_DT array per frame (a list) or, for
        n == 1, one array; max_new: an int or one per frame. Returns (list of CORNER_DT arrays in Add_Feature order, exact-path
        flags (n,) bool)."""
        mn = np.broadcast_to(np.asarray(max_new, np.int32), (n,)).copy()
        occ = None if occupied is None else np.ascontiguousarray(occupied, np.uint8).reshape(n, self.n_cells)
        msk = None if mask is None else np.ascontiguousarray(mask, np.uint8).reshape(n, self.height, self.width)
        if circles is not None and n == 1 and not isinstance(circles, (list, tuple)):
            circles = [circles]
        exact = np.zeros(n, np.uint8)
        if n == 1:
            c = None if circles is None else np.ascontiguousarray(circles[0], CIRCLE_DT)
            out = np.zeros(max(int(mn[0]), 1), CORNER_DT)
            n_out = C.c_int(0)
            self._ck(self.L.dsdtm_detect(self.hp, int(slot), C.c_float(threshold), _p(occ), _p(msk), _p(c), 0 if c is None else len(c),
                                         int(mn[0]), _p(out), C.byref(n_out), _p(exact)))
            return [out[:n_out.value].copy()], exact.astype(bool)
        stride = max(int(mn.max()), 1)
        out = np.zeros((n, stride), CORNER_DT)
        n_out = np.zeros(n, np.int32)
        circ = nc = None
        cs = 0
        if circles is not None:
            nc = np.array([len(c) for c in circles], np.int32)
            cs = max(int(nc.max()), 1)
            circ = np.zeros((n, cs), CIRCLE_DT)
            for i, c in enumerate(circles):
                circ[i, :len(c)] = c
        self._ck(self.L.dsdtm_detect_batch(self.hp, int(slot), int(n), C.c_float(threshold), _p(occ), _p(msk), _p(circ), cs, _p(nc),
                                           _p(mn), stride, _p(out), _p(n_out), _p(exact)))
        return [out[i, :n_out[i]].copy() for i in range(n)], exact.astype(bool)

    def fast_score_map(self, slot, level, barrier=20):
        s = np.empty((self.hs[level], self.ws[level]), np.uint8)
        m = np.empty_like(s)
        self._ck(self.L.dsdtm_fast_score_map(self.hp, int(slot), int(level), int(barrier), _p(s), _p(m)))
        return s, m

    # ---- sparse align
    def sparse_align(self, ref_slot, cur_slot, feats, ref_center, pose_in, max_level, min_level, max_iters, log_cap=256):
        feats = np.ascontiguousarray(feats, REF_FEAT_DT)
        pose_out = np.empty(7)
        n_tracked = C.c_int(0)
        log = np.zeros(log_cap, ITER_LOG_DT)
        n_log = C.c_int(0)
        self._ck(self.L.dsdtm_sparse_align(self.hp, int(ref_slot), int(cur_slot), _p(feats), len(feats),
                                           _p(np.ascontiguousarray(ref_center, np.float64)),
                                           _p(np.ascontiguousarray(pose_in, np.float64)), int(max_level), int(min_level),
                                           int(max_iters), _p(pose_out), C.byref(n_tracked), _p(log), log_cap, C.byref(n_log)))
        return pose_out, n_tracked.value, log[:min(n_log.value, log_cap)].copy()

    def sparse_align_batch(self, ref_slots, cur_slots, feats, n_feats, ref_centers, poses_in, max_level, min_level, max_iters,
                           log_cap=0):
        n = len(ref_slots)
        feats = np.ascontiguousarray(feats, REF_FEAT_DT).reshape(n, -1)
        poses_out = np.empty((n, 7)); n_tracked = np.empty(n, np.int32)
        log = np.zeros((n, max(log_cap, 1)), ITER_LOG_DT) if log_cap else None
        n_log = np.zeros(n, np.int32)
        self._ck(self.L.dsdtm_sparse_align_batch(
            self.hp, n, _p(np.ascontiguousarray(ref_slots, np.int32)), _p(np.ascontiguousarray(cur_slots, np.int32)), _p(feats),
            feats.shape[1], _p(np.ascontiguousarray(n_feats, np.int32)), _p(np.ascontiguousarray(ref_centers, np.float64)),
            _p(np.ascontiguousarray(poses_in, np.float64)), int(max_level), int(min_level), int(max_iters), _p(poses_out),
            _p(n_tracked), _p(log), int(log_cap), _p(n_log)))
        return poses_out, n_tracked, log, n_log

    # ---- feature alignment
    def align2d(self, cur_slot, levels, patches10, px, max_iters=10):
        levels = np.ascontiguousarray(levels, np.int32)
        patches10 = np.ascontiguousarray(patches10, np.uint8).reshape(len(levels), 100)
        px = np.array(px, np.float64).reshape(len(levels), 2)
        conv = np.zeros(len(levels), np.uint8)
        self._ck(self.L.dsdtm_align2d_batch(self.hp, int(cur_slot), _p(levels), _p(patches10), _p(px), len(levels), int(max_iters), _p(conv)))
        return px, conv.astype(bool)

    def warp_affine(self, ref_slots, A, ref_px, ref_levels, search_levels):
        n = len(ref_slots)
        out = np.empty((n, 100), np.uint8)
        self._ck(self.L.dsdtm_warp_affine_batch(
            self.hp, _p(np.ascontiguousarray(ref_slots, np.int32)), _p(np.ascontiguousarray(A, np.float64).reshape(n, 4)),
            _p(np.ascontiguousarray(ref_px, np.float32).reshape(n, 2)), _p(np.ascontiguousarray(ref_levels, np.int32)),
            _p(np.ascontiguousarray(search_levels, np.int32)), n, _p(out)))
        return out

    def feature_align_batch(self, cur_slot, cands, max_search_level, max_iters=10, want_A=False):
        cands = np.ascontiguousarray(cands, CANDIDATE_DT)
        n = len(cands)
        px = np.empty((n, 2)); lv = np.empty(n, np.int32); conv = np.zeros(n, np.uint8)
        A = np.empty((n, 2, 2)) if want_A else None
        self._ck(self.L.dsdtm_feature_align_batch(self.hp, int(cur_slot), _p(cands), n, int(max_search_level), int(max_iters),
                                                  _p(px), _p(lv), _p(conv), _p(A)))
        return px, lv, conv.astype(bool), A

    def local_map_align_batch(self, cur_slot, pose_cur_c2w, cur_center, kfs, obs, pts, max_search_level, max_iters=10):
        kfs = np.ascontiguousarray(kfs, KF_VIEW_DT); obs = np.ascontiguousarray(obs, OBS_DT); pts = np.ascontiguousarray(pts, MAP_POINT_DT)
        out = np.zeros(len(pts), REPROJ_DT)
        self._ck(self.L.dsdtm_local_map_align_batch(
            self.hp, int(cur_slot), _p(np.ascontiguousarray(pose_cur_c2w, np.float64)), _p(np.ascontiguousarray(cur_center, np.float64)),
            _p(kfs), len(kfs), _p(obs), len(obs), _p(pts), len(pts), int(max_search_level), int(max_iters), _p(out)))
        return out

    # ---- keyframe ingest (f-3 / f-4)
    def depth_upload(self, depth_slot, depth_u16):
        d = np.ascontiguousarray(depth_u16, np.uint16)
        assert d.shape == (self.height, self.width)
        self._ck(self.L.dsdtm_depth_upload(self.hp, int(depth_slot), _p(d), 0))

    def depth_convert_f32(self, first_depth_slot, n, depth_scale, fetch=True):
        out = np.empty((n, self.height, self.width), np.float32) if fetch else None
        self._ck(self.L.dsdtm_depth_convert_f32(self.hp, int(first_depth_slot), int(n), C.c_float(depth_scale), _p(out)))
        return out

    def keyframe_lift(self, depth_slot, pose_c2w, dist, depth_scale, px_in, initial=None):
        px = np.ascontiguousarray(px_in, np.float32).reshape(-1, 2)
        ini = None if initial is None else np.ascontiguousarray(initial, np.uint8)
        out = np.zeros(len(px), LIFTED_DT)
        self._ck(self.L.dsdtm_keyframe_lift(self.hp, int(depth_slot), _p(np.ascontiguousarray(pose_c2w, np.float64)),
                                            _p(np.ascontiguousarray(dist, np.float32)), C.c_float(depth_scale), _p(px), _p(ini), len(px), _p(out)))
        return out

    def map_table_upload(self, first_kf, kfs, first_point, points_w):
        """dsdtm_map_table_upload: (re)write key-frame rows from first_kf and point rows from first_point."""
        kfs = np.ascontiguousarray(kfs, MAP_KF_DT).reshape(-1)
        pts = np.ascontiguousarray(points_w, np.float64).reshape(-1, 3)
        self._ck(self.L.dsdtm_map_table_upload(self.hp, int(first_kf), len(kfs), _p(kfs), int(first_point), len(pts), _p(pts)))

    def close_keyframes(self, pose_cur_c2w, n_kfs, max_local=10):
        """dsdtm_close_keyframes -> (visible u8[n_kfs], dist f64[n_kfs], local key-frame rows in rank order)"""
        vis = np.zeros(n_kfs, np.uint8); dist = np.zeros(n_kfs); local = np.zeros(max(max_local, 1), np.int32); n = C.c_int32(0)
        self._ck(self.L.dsdtm_close_keyframes(self.hp, _p(np.ascontiguousarray(pose_cur_c2w, np.float64)), int(n_kfs), int(max_local),
                                              _p(vis), _p(dist), _p(local), C.byref(n)))
        return vis, dist, local[:n.value].copy()

    def pose_optimize_batch(self, obs, n_obs, poses_in, max_iters=100, want_res=True):
        """dsdtm_pose_optimize_batch: obs = (n_frames, obs_stride) BA_OBS_DT, n_obs per frame, poses (n_frames, 7).
        Returns (poses_out, res_norm or None, summaries)."""
        obs = np.ascontiguousarray(obs, BA_OBS_DT)
        n_obs = np.ascontiguousarray(n_obs, np.int32).reshape(-1)
        nf = len(n_obs)
        obs = obs.reshape(nf, -1) if nf else obs.reshape(0, 0)
        poses_in = np.ascontiguousarray(poses_in, np.float64).reshape(nf, 7)
        out = np.zeros((nf, 7)); summ = np.zeros(nf, BA_SUMMARY_DT)
        res = np.zeros(obs.shape, np.float64) if want_res else None
        self._ck(self.L.dsdtm_pose_optimize_batch(self.hp, nf, _p(obs), int(obs.shape[1]), _p(n_obs), _p(poses_in), int(max_iters), _p(out),
                                                  _p(res), _p(summ)))
        return out, res, summ

    def pose_optimize(self, obs, pose_in, max_iters=100):
        """dsdtm_pose_optimize (Optimizer::PoseOptimization of one frame). Returns (pose_out, res_norm, summary record)."""
        obs = np.ascontiguousarray(obs, BA_OBS_DT).reshape(-1)
        pose_in = np.ascontiguousarray(pose_in, np.float64).reshape(7)
        out = np.zeros(7); res = np.zeros(len(obs)); summ = np.zeros(1, BA_SUMMARY_DT)
        self._ck(self.L.dsdtm_pose_optimize(self.hp, _p(obs), len(obs), _p(pose_in), int(max_iters), _p(out), _p(res), _p(summ)))
        return out, res, summ[0]

    def track_frame(self, ref_slot, cur_slot, img, feats, ref_center, pose_ref_c2w, pose_c2r_in, sa_cfg, kfs, obs, pts, max_search_level,
                    align_iters=10):
        """dsdtm_track_frame: upload + pyramid + sparse align + pose composition + local-map alignment in one call.
        Returns (TrackOut fields as dict, REPROJ_DT array)."""
        img = np.ascontiguousarray(img, np.uint8); feats = np.ascontiguousarray(feats, REF_FEAT_DT)
        kfs = np.ascontiguousarray(kfs, KF_VIEW_DT); obs = np.ascontiguousarray(obs, OBS_DT); pts = np.ascontiguousarray(pts, MAP_POINT_DT)
        ti = TrackIn()
        ti.ref_slot, ti.cur_slot, ti.img, ti.stride = int(ref_slot), int(cur_slot), img.ctypes.data, img.shape[1]
        ti.feats, ti.n_feats = feats.ctypes.data, len(feats)
        ti.ref_center[:] = [float(v) for v in ref_center]; ti.pose_ref_c2w[:] = [float(v) for v in pose_ref_c2w]
        ti.pose_c2r_in[:] = [float(v) for v in pose_c2r_in]
        ti.max_level, ti.min_level, ti.max_iters = (int(v) for v in sa_cfg)
        ti.kfs, ti.n_kfs, ti.obs, ti.n_obs, ti.pts, ti.n_pts = kfs.ctypes.data, len(kfs), obs.ctypes.data, len(obs), pts.ctypes.data, len(pts)
        ti.max_search_level, ti.align_iters = int(max_search_level), int(align_iters)
        to = TrackOut()
        rep = np.zeros(len(pts), REPROJ_DT)
        self._keep = (img, feats, kfs, obs, pts)
        self._ck(self.L.dsdtm_track_frame(self.hp, C.byref(ti), C.byref(to), _p(rep)))
        return dict(pose_c2r=np.array(to.pose_c2r[:]), pose_cur_c2w=np.array(to.pose_cur_c2w[:]), cur_center=np.array(to.cur_center[:]),
                    n_tracked=int(to.n_tracked)), rep

    # ---- device-resident map store
    def store_clear(self):
        self._ck(self.L.dsdtm_store_clear(self.hp))
        self.store_points = self.store_keyframes = 0

    def store_set_points(self, first, points_w, bad=None):
        """dsdtm_store_set_points: append (first == current size) or rewrite point rows [first, first + n)"""
        pw = np.ascontiguousarray(points_w, np.float64).reshape(-1, 3)
        b = None if bad is None else np.ascontiguousarray(bad, np.int32).reshape(len(pw))
        self._ck(self.L.dsdtm_store_set_points(self.hp, int(first), len(pw), _p(pw), _p(b)))
        self.store_points = max(self.store_points, int(first) + len(pw))

    def store_update_points(self, ids, points_w=None, bad=None):
        """dsdtm_store_update_points: scattered positions (None = keep) and bad flags (None = keep)"""
        ids = np.ascontiguousarray(ids, np.int32).reshape(-1)
        pw = None if points_w is None else np.ascontiguousarray(points_w, np.float64).reshape(len(ids), 3)
        b = None if bad is None else np.ascontiguousarray(bad, np.int32).reshape(len(ids))
        self._ck(self.L.dsdtm_store_update_points(self.hp, _p(ids), len(ids), _p(pw), _p(b)))

    def store_append_keyframe(self, slot, pose_c2w, center, feats):
        """dsdtm_store_append_keyframe: feats = STORE_FEAT_DT rows (mp, level, px, normal, is_obs). Returns the key frame's row."""
        kf = np.zeros(1, STORE_KF_DT)
        kf["slot"] = slot; kf["pose_c2w"] = pose_c2w; kf["center"] = center
        fs = np.ascontiguousarray(feats, STORE_FEAT_DT).reshape(-1)
        row = C.c_int32(0)
        self._ck(self.L.dsdtm_store_append_keyframe(self.hp, _p(kf), _p(fs), len(fs), C.byref(row)))
        self.store_keyframes = row.value + 1
        return row.value

    def store_set_keyframe(self, row, slot, pose_c2w, center):
        self._ck(self.L.dsdtm_store_set_keyframe(self.hp, int(row), int(slot), _p(np.ascontiguousarray(pose_c2w, np.float64)),
                                                  _p(np.ascontiguousarray(center, np.float64))))

    def store_set_found(self, ids, found):
        """dsdtm_store_set_found: MapPoint::mnFound of the point rows ids (appended points start at 1)"""
        ids = np.ascontiguousarray(ids, np.int32).reshape(-1)
        f = np.ascontiguousarray(found, np.int32).reshape(len(ids))
        self._ck(self.L.dsdtm_store_set_found(self.hp, _p(ids), len(ids), _p(f)))

    def store_size(self):
        """-> (key frames, features, points): the rows of the store's tables"""
        k, f, p = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        self._ck(self.L.dsdtm_store_size(self.hp, C.byref(k), C.byref(f), C.byref(p)))
        return k.value, f.value, p.value

    def store_fetch(self, kfs=None, feats=None, points=None):
        """dsdtm_store_fetch: kfs / feats / points = (first, n) row ranges, None = the whole table. Returns (STORE_KF_DT, STORE_FEAT_DT,
        STORE_POINT_DT, found int32) as the library holds them: is_obs = observing key-frame row + 1, next_obs / last_obs the chains."""
        nk, nf, npt = self.store_size()
        (k0, kn), (f0, fn), (p0, pn) = kfs or (0, nk), feats or (0, nf), points or (0, npt)
        K = np.zeros(kn, STORE_KF_DT); F = np.zeros(fn, STORE_FEAT_DT); P = np.zeros(pn, STORE_POINT_DT); fd = np.zeros(pn, np.int32)
        self._ck(self.L.dsdtm_store_fetch(self.hp, int(k0), int(kn), _p(K), int(f0), int(fn), _p(F), int(p0), int(pn), _p(P), _p(fd)))
        return K, F, P, fd

    def store_track(self, cur_slot, pose_cur_c2w, cur_center, max_local=10, max_search_level=2, align_iters=10, cap=4096):
        """dsdtm_store_track -> (local key-frame rows in rank order, STORE_CAND_DT records in arrival order). More than cap candidates
        raises."""
        local = np.zeros(16, np.int32); nl = C.c_int32(0); out = np.zeros(cap, STORE_CAND_DT); n = C.c_int32(0)
        self._ck(self.L.dsdtm_store_track(self.hp, int(cur_slot), _p(np.ascontiguousarray(pose_cur_c2w, np.float64)),
                                          _p(np.ascontiguousarray(cur_center, np.float64)), int(max_local), int(max_search_level),
                                          int(align_iters), _p(local), C.byref(nl), _p(out), int(cap), C.byref(n)))
        return local[:nl.value].copy(), out[:n.value].copy()

    # ---- batched front end
    def batch_stage(self, ref_slots, cur_slots, feats, n_feats, ref_centers, poses_in, max_level, min_level, max_iters,
                    patches10=None, patch_px=None, patch_level=None, align_iters=10):
        n = len(ref_slots)
        feats = np.ascontiguousarray(feats, REF_FEAT_DT).reshape(n, -1)
        ppp = 0 if patch_level is None else np.asarray(patch_level).reshape(n, -1).shape[1]
        self._n = n; self._ppp = ppp; self._store_cpf = None; self._feat_stride = feats.shape[1]
        self._ck(self.L.dsdtm_batch_stage(
            self.hp, n, _p(np.ascontiguousarray(ref_slots, np.int32)), _p(np.ascontiguousarray(cur_slots, np.int32)), _p(feats),
            feats.shape[1], _p(np.ascontiguousarray(n_feats, np.int32)), _p(np.ascontiguousarray(ref_centers, np.float64)),
            _p(np.ascontiguousarray(poses_in, np.float64)), int(max_level), int(min_level), int(max_iters),
            _p(np.ascontiguousarray(patches10, np.uint8)) if ppp else None,
            _p(np.ascontiguousarray(patch_px, np.float64)) if ppp else None,
            _p(np.ascontiguousarray(patch_level, np.int32)) if ppp else None, ppp, int(align_iters)))

    def batch_stage_map(self, poses_ref_c2w, points_per_pair, max_search_level, align_iters=10):
        """after batch_stage: the refinement chain's inputs (reference poses); batch_run(flags | 2) then runs the chain"""
        pr = np.ascontiguousarray(poses_ref_c2w, np.float64).reshape(self._n, 7)
        self._map_ppp = int(points_per_pair); self._store_cpf = None
        self._ck(self.L.dsdtm_batch_stage_map(self.hp, _p(pr), int(points_per_pair), int(max_search_level), int(align_iters)))

    def batch_stage_store(self, poses_ref_c2w, kf_range=None, max_local=10, max_search_level=2, align_iters=10, cands_per_frame=1024):
        """after batch_stage: the store-backed local map (dsdtm_batch_stage_store); kf_range = (n_pairs, 2) key-frame rows [begin, end)
        or None (every row); batch_run(flags | 2) then runs UpdateLocalMap per frame on the map store"""
        pr = np.ascontiguousarray(poses_ref_c2w, np.float64).reshape(self._n, 7)
        kr = None if kf_range is None else np.ascontiguousarray(kf_range, np.int32).reshape(self._n, 2)
        self._ck(self.L.dsdtm_batch_stage_store(self.hp, _p(pr), _p(kr), int(max_local), int(max_search_level), int(align_iters),
                                                int(cands_per_frame)))
        self._store_cpf = int(cands_per_frame)

    def batch_fetch_store(self):
        """-> (local rows (n, 16), n_local (n,), records (n, cands_per_frame) STORE_CAND_DT in order, n_cand (n,) true counts)"""
        n, F = self._n, self._store_cpf
        loc = np.empty((n, 16), np.int32); nl = np.empty(n, np.int32); rec = np.empty((n, F), STORE_CAND_DT); nc = np.empty(n, np.int32)
        self._ck(self.L.dsdtm_batch_fetch_store(self.hp, _p(loc), _p(nl), _p(rec), _p(nc)))
        return loc, nl, rec, nc

    def batch_fetch_map(self):
        out = np.zeros((self._n, self._map_ppp), REPROJ_DT)
        self._ck(self.L.dsdtm_batch_fetch_map(self.hp, _p(out)))
        return out

    def batch_stage_track(self, found=None, max_iters=100):
        """after batch_stage_map: found = (n_pairs, points_per_pair) MapPoint::mnFound counts (None = all 1), max_iters = PoseOptimization's
        cap; batch_run(7) then ends in the tracked poses"""
        f = None if found is None else np.ascontiguousarray(found, np.int32).reshape(-1)
        if f is not None and getattr(self, "_store_cpf", None) is None:
            f = f.reshape(self._n, self._map_ppp)
        elif f is not None and len(f) != self.store_points:     # store mode: one count per store point row
            raise DsdtmError("batch_stage_track: found has %d entries, the map store %d points" % (len(f), self.store_points))
        self._ck(self.L.dsdtm_batch_stage_track(self.hp, _p(f), int(max_iters)))

    def batch_stage_track_live(self, max_iters=100):
        """after batch_stage_store: as batch_stage_track, but the selection reads the store's own found counts at every run"""
        self._ck(self.L.dsdtm_batch_stage_track_live(self.hp, int(max_iters)))

    def batch_commit_store(self, outlier_threshold, kf_rows=None):
        """dsdtm_batch_commit_store after a store-mode batch_run(7 or 15): found counts, bad flags and (flags 15) the key frames of the
        wanted frames into the store. kf_rows = (n_pairs,) reserved empty key-frame rows or None (append). Returns (kf_row, point_first,
        n_points) per frame and updates store_points / store_keyframes."""
        n = self._n
        kr = None if kf_rows is None else np.ascontiguousarray(kf_rows, np.int32).reshape(n)
        row = np.empty(n, np.int32); pf = np.empty(n, np.int32); npt = np.empty(n, np.int32)
        self._ck(self.L.dsdtm_batch_commit_store(self.hp, C.c_float(outlier_threshold), _p(kr), _p(row), _p(pf), _p(npt)))
        self.store_keyframes, _, self.store_points = self.store_size()
        return row, pf, npt

    def batch_advance(self, next_cur_slots, hold=None, want_next=None):
        """dsdtm_batch_advance after batch_commit_store: every frame that is not held becomes its own next reference frame on the device,
        every frame's cur slot moves to next_cur_slots. hold / want_next = (n_pairs,) bools or None. Returns the (n_pairs,) ADV_* status."""
        n = self._n
        nc = np.ascontiguousarray(next_cur_slots, np.int32).reshape(n)
        hd = None if hold is None else np.ascontiguousarray(hold, np.uint8).reshape(n)
        wt = None if want_next is None else np.ascontiguousarray(want_next, np.uint8).reshape(n)
        st = np.empty(n, np.uint8)
        self._ck(self.L.dsdtm_batch_advance(self.hp, _p(nc), _p(hd), _p(wt), _p(st)))
        return st

    def batch_upload_step(self, imgs, depth=None):
        """dsdtm_batch_upload_step: (n_pairs, height, width) uint8 images into the staged cur slots and, optionally, (n_pairs, height, width)
        uint16 depth images into the staged depth slots; batch_run(flags | 1) builds the pyramids"""
        n = self._n
        im = np.ascontiguousarray(imgs, np.uint8).reshape(n, self.height, self.width)
        d = None if depth is None else np.ascontiguousarray(depth, np.uint16).reshape(n, self.height, self.width)
        self._ck(self.L.dsdtm_batch_upload_step(self.hp, _p(im), _p(d)))

    def batch_fetch_ref(self):
        """-> dict(ref_slots, cur_slots, feats (n, feat_stride) REF_FEAT_DT, n_feats, centers (n, 3), poses_ref (n, 7), poses_in (n, 7)):
        the staged per-frame inputs as the next batch_run reads them"""
        n, fs = self._n, self._feat_stride
        r = dict(ref_slots=np.empty(n, np.int32), cur_slots=np.empty(n, np.int32), feats=np.empty((n, fs), REF_FEAT_DT),
                 n_feats=np.empty(n, np.int32), centers=np.empty((n, 3)), poses_ref=np.empty((n, 7)), poses_in=np.empty((n, 7)))
        self._ck(self.L.dsdtm_batch_fetch_ref(self.hp, *(_p(r[k]) for k in ("ref_slots", "cur_slots", "feats", "n_feats", "centers",
                                                                            "poses_ref", "poses_in"))))
        return r

    def batch_fetch_track(self):
        """-> (poses c2w after PoseOptimization (n, 7), n_matches (n,), matches (n, 200) MATCH_DT, res_norm (n, 200), summaries (n,)
        BA_SUMMARY_DT); rows past n_matches[i] are zero"""
        n, K = self._n, TRACK_MAX_MATCHES
        poses = np.empty((n, 7)); nm = np.empty(n, np.int32); m = np.empty((n, K), MATCH_DT); res = np.empty((n, K))
        summ = np.empty(n, BA_SUMMARY_DT)
        self._ck(self.L.dsdtm_batch_fetch_track(self.hp, _p(poses), _p(nm), _p(m), _p(res), _p(summ)))
        return poses, nm, m, res, summ

    def batch_stage_keyframe(self, depth_slots=None, want=None, detection_threshold=5.0, min_dist=15, max_fts=300,
                             dist=(0.0, 0.0, 0.0, 0.0, 0.0), depth_scale=5000.0):
        """after batch_stage_track: Tracking::CraeteKeyframe behind the tracked pose. depth_slots = (n_pairs,) depth slots (-1 = no depth;
        None = none), want = (n_pairs,) bools (None = every pair); batch_run(15) then ends in the key frames"""
        ds = None if depth_slots is None else np.ascontiguousarray(depth_slots, np.int32).reshape(self._n)
        wt = None if want is None else np.ascontiguousarray(want, np.uint8).reshape(self._n)
        self._kf_max_fts = int(max_fts)
        self._ck(self.L.dsdtm_batch_stage_keyframe(self.hp, _p(ds), _p(wt), C.c_float(detection_threshold), int(min_dist), int(max_fts),
                                                   _p(np.ascontiguousarray(dist, np.float32)), C.c_float(depth_scale)))

    def batch_fetch_keyframe(self):
        """-> (n_new (n,), corners (n, max_fts) CORNER_DT, lifted (n, max_fts) LIFTED_DT, exact_path (n,) bool); rows past n_new[i] are
        zero"""
        n, F = self._n, self._kf_max_fts
        nn = np.empty(n, np.int32); cr = np.empty((n, F), CORNER_DT); lf = np.empty((n, F), LIFTED_DT); ex = np.empty(n, np.uint8)
        self._ck(self.L.dsdtm_batch_fetch_keyframe(self.hp, _p(nn), _p(cr), _p(lf), _p(ex)))
        return nn, cr, lf, ex.astype(bool)

    def track_batch_e2e(self, cur_imgs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_ref, poses_in, max_level, min_level,
                        max_iters, points_per_pair, max_search_level, align_iters, out):
        """All arrays contiguous with the right dtype (pinned for async copies); out = dict(poses, n_tracked, reproj)."""
        n = len(ref_slots)
        self._ck(self.L.dsdtm_track_batch_e2e(
            self.hp, n, _p(cur_imgs), _p(ref_slots), _p(cur_slots), _p(feats), int(feat_stride), _p(n_feats), _p(ref_centers), _p(poses_ref),
            _p(poses_in), int(max_level), int(min_level), int(max_iters), int(points_per_pair), int(max_search_level), int(align_iters),
            _p(out["poses"]), _p(out["n_tracked"]), _p(out["reproj"])))

    def batch_run(self, flags=0):
        self._ck(self.L.dsdtm_batch_run(self.hp, int(flags)))

    def batch_fetch(self):
        n, ppp = self._n, self._ppp
        poses = np.empty((n, 7)); nt = np.empty(n, np.int32)
        px = np.empty((n, ppp, 2)) if ppp else None
        conv = np.empty((n, ppp), np.uint8) if ppp else None
        self._ck(self.L.dsdtm_batch_fetch(self.hp, _p(poses), _p(nt), _p(px), _p(conv)))
        return poses, nt, px, conv

    def timer_start(self):
        self._ck(self.L.dsdtm_timer_start(self.hp))

    def timer_stop(self):
        ms = float(self.L.dsdtm_timer_stop(self.hp))
        if ms < 0:
            self._ck(-2)
        return ms

    def last_run_ms(self):
        return float(self.L.dsdtm_last_run_ms(self.hp))

    def pair_batch_e2e(self, cur_imgs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_in, max_level,
                       min_level, max_iters, patches10, patch_px, patch_level, ppp, align_iters, out):
        """All arrays must already be contiguous with the right dtype (pinned for async copies); out = dict of result arrays."""
        n = len(ref_slots)
        self._ck(self.L.dsdtm_pair_batch_e2e(
            self.hp, n, _p(cur_imgs), _p(ref_slots), _p(cur_slots), _p(feats), int(feat_stride), _p(n_feats), _p(ref_centers),
            _p(poses_in), int(max_level), int(min_level), int(max_iters), _p(patches10), _p(patch_px), _p(patch_level), int(ppp),
            int(align_iters), _p(out["poses"]), _p(out["n_tracked"]), _p(out.get("px")), _p(out.get("conv"))))
