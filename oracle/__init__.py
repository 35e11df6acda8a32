"""TEST INFRASTRUCTURE -- ctypes loader for the CPU oracle (oracle/dsdtm_oracle.cpp) and, when built,
the reference's own FAST library (oracle/_ref/libfast_ref.so).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import this
package. Nothing under dsdtm_b200/ does. See dsdtm_oracle.h for the pinning status of each function.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "_build", "liboracle.so")
_REF = os.path.join(_HERE, "_ref", "libfast_ref.so")


def build(force=False):
    """Compile the oracle (and oracle/_ref where refpin.REFERENCE holds a checkout of the reference). Building is not using."""
    src = os.path.join(_HERE, "dsdtm_oracle.cpp")
    stale = (not os.path.exists(_LIB)) or os.path.getmtime(_LIB) < max(
        os.path.getmtime(src), os.path.getmtime(os.path.join(_HERE, "dsdtm_oracle.h")))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "_build/liboracle.so"], stdout=subprocess.DEVNULL)
    from . import refpin
    if refpin.REFERENCE and os.path.isdir(os.path.join(refpin.REFERENCE, "Thirdparty", "fast", "src")) and (force or not os.path.exists(_REF)):
        subprocess.check_call(["make", "-C", _HERE, "ref", "REF=" + refpin.REFERENCE], stdout=subprocess.DEVNULL)
    # the reference's own hot-path translation units against the stand-in headers of tests/ref_shim (oracle/refpin.py)
    refpin.build(force)


class Cam(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("fx", C.c_float), ("fy", C.c_float),
                ("cx", C.c_float), ("cy", C.c_float), ("f", C.c_float)]


CORNER_DT = np.dtype([("x", "<i4"), ("y", "<i4"), ("level", "<i4"), ("score", "<f4")])
REF_FEAT_DT = np.dtype([("px", "<f4", 2), ("level", "<i4"), ("initial", "<i4"),
                        ("normal", "<f8", 3), ("point_w", "<f8", 3)])
ITER_LOG_DT = np.dtype([("level", "<i4"), ("iter", "<i4"), ("n_pts", "<i4"), ("flags", "<i4"),
                        ("chi2", "<f8"), ("x", "<f8", 6)])
assert REF_FEAT_DT.itemsize == 64 and ITER_LOG_DT.itemsize == 72 and CORNER_DT.itemsize == 16

_lib = None
_ref = None


def _p(a, t=C.c_void_p):
    return a.ctypes.data_as(t) if a is not None else None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB)
        _lib.orc_shitomasi.restype = C.c_float
        _lib.orc_cvround.argtypes = [C.c_double]
        _lib.orc_feature_depth.restype = C.c_float
        _lib.orc_is_in_image.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_int]
        _lib.orc_depth_convert.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_void_p]
        _lib.orc_unproject.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
    return _lib


def have_ref():
    return os.path.exists(_REF)


def ref():
    global _ref
    if _ref is None:
        _ref = C.CDLL(_REF)
    return _ref


def make_cam(width, height, fx, fy, cx, cy, f):
    return Cam(width, height, fx, fy, cx, cy, f)


def u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


# ---------------------------------------------------------------- pyramid
def pyrdown(img):
    img = u8(img)
    h, w = img.shape
    out = np.empty(((h + 1) // 2, (w + 1) // 2), np.uint8)
    lib().orc_pyrdown_u8(_p(img), w, h, w, _p(out))
    return out


def level_dims(w, h, levels):
    ws, hs = [w], [h]
    for _ in range(1, levels):
        ws.append((ws[-1] + 1) // 2)
        hs.append((hs[-1] + 1) // 2)
    offs = np.concatenate([[0], np.cumsum([a * b for a, b in zip(ws, hs)])]).astype(np.int32)
    return np.array(ws, np.int32), np.array(hs, np.int32), offs[:-1].copy(), int(offs[-1])


def pyramid(img, levels):
    """returns (packed u8 buffer, offs, ws, hs)"""
    img = u8(img)
    h, w = img.shape
    ws, hs, offs, total = level_dims(w, h, levels)
    out = np.empty(total, np.uint8)
    o = np.empty(levels, np.int32); ww = np.empty(levels, np.int32); hh = np.empty(levels, np.int32)
    lib().orc_pyramid(_p(img), w, h, levels, _p(out), _p(o), _p(ww), _p(hh))
    assert (o == offs).all() and (ww == ws).all() and (hh == hs).all()
    return out, offs, ws, hs


def pyr_level(packed, offs, ws, hs, l):
    return packed[offs[l]:offs[l] + ws[l] * hs[l]].reshape(hs[l], ws[l])


# ---------------------------------------------------------------- FAST
def fast10_detect(img, barrier):
    img = u8(img)
    h, w = img.shape
    xy = np.empty((w * h, 2), np.int16)
    n = lib().orc_fast10_detect(_p(img), w, h, w, int(barrier), _p(xy), w * h)
    return xy[:n].copy()


def fast10_score(img, xy):
    img = u8(img)
    xy = np.ascontiguousarray(xy, np.int16)
    s = np.empty(len(xy), np.int32)
    lib().orc_fast10_score(_p(img), img.shape[1], _p(xy), len(xy), _p(s))
    return s


def fast_nonmax(xy, scores):
    xy = np.ascontiguousarray(xy, np.int16)
    scores = np.ascontiguousarray(scores, np.int32)
    keep = np.empty(len(xy), np.int32)
    m = lib().orc_fast_nonmax_3x3(_p(xy), _p(scores), len(xy), _p(keep))
    return keep[:m].copy()


def ref_fast10_detect(img, barrier, sse2=True):
    img = u8(img)
    h, w = img.shape
    xy = np.empty((w * h, 2), np.int16)
    n = ref().fastref_detect10(_p(img), w, h, w, int(barrier), int(sse2), _p(xy), w * h)
    return xy[:n].copy()


def ref_fast10_score(img, xy, threshold):
    img = u8(img)
    xy = np.ascontiguousarray(xy, np.int16)
    s = np.empty(len(xy), np.int32)
    ref().fastref_score10(_p(img), img.shape[1], _p(xy), len(xy), int(threshold), _p(s))
    return s


def ref_fast_nonmax(xy, scores):
    xy = np.ascontiguousarray(xy, np.int16)
    scores = np.ascontiguousarray(scores, np.int32)
    keep = np.empty(len(xy), np.int32)
    m = ref().fastref_nonmax(_p(xy), _p(scores), len(xy), _p(keep))
    return keep[:m].copy()


def shitomasi(img, u, v):
    img = u8(img)
    return float(lib().orc_shitomasi(_p(img), img.shape[1], img.shape[0], img.shape[1], int(u), int(v)))


def grid_dims(w, h, cell):
    return -(-h // cell), -(-w // cell)


def detect_cells(packed, offs, ws, hs, cell, occupied=None, thr=5.0):
    levels = len(ws)
    rows, cols = grid_dims(int(ws[0]), int(hs[0]), cell)
    cells = np.zeros(rows * cols, CORNER_DT)
    occ = u8(occupied) if occupied is not None else None
    lib().orc_detect_cells(_p(packed), _p(offs), _p(ws), _p(hs), levels, int(ws[0]), int(hs[0]), int(cell),
                           _p(occ), C.c_double(thr), _p(cells))
    return cells


def detect_select(cells, mask, cell, max_fts, n_existing=0):
    """cells sorted in place (copy returned), mask painted in place. returns (features, sorted_cells)"""
    cells = cells.copy()
    h, w = mask.shape
    assert mask.dtype == np.uint8 and mask.flags.c_contiguous
    out = np.zeros(len(cells), CORNER_DT)
    n = lib().orc_detect_select(_p(cells), len(cells), _p(mask), w, h, int(cell), int(max_fts), int(n_existing), _p(out))
    return out[:n].copy(), cells


def circle_fill(img, cx, cy, r, color=0):
    assert img.dtype == np.uint8 and img.flags.c_contiguous
    h, w = img.shape
    lib().orc_circle_fill(_p(img), w, h, w, int(cx), int(cy), int(r), int(color))


def cvround(v):
    return int(lib().orc_cvround(float(v)))


# ---------------------------------------------------------------- sparse alignment
def sparse_align(cam, ref_pyr, cur_pyr, offs, ws, hs, feats, ref_center, pose_in, max_level, min_level, max_iters,
                 log_cap=512):
    feats = np.ascontiguousarray(feats, REF_FEAT_DT)
    ref_center = np.ascontiguousarray(ref_center, np.float64)
    pose_in = np.ascontiguousarray(pose_in, np.float64)
    pose_out = np.empty(7, np.float64)
    log = np.zeros(log_cap, ITER_LOG_DT)
    n_log = C.c_int(0)
    n = lib().orc_sparse_align(C.byref(cam), _p(ref_pyr), _p(cur_pyr), _p(offs), _p(ws), _p(hs), _p(feats), len(feats),
                               _p(ref_center), _p(pose_in), int(max_level), int(min_level), int(max_iters),
                               _p(pose_out), _p(log), log_cap, C.byref(n_log))
    return pose_out, int(n), log[:min(n_log.value, log_cap)].copy()


# ---------------------------------------------------------------- feature alignment
def solve_affine(cam, kf_center, ref_point_w, ref_normal, ref_px, ref_level, pose_c2r):
    A = np.empty(4, np.float64)
    lib().orc_solve_affine(C.byref(cam), _p(np.ascontiguousarray(kf_center, np.float64)),
                           _p(np.ascontiguousarray(ref_point_w, np.float64)),
                           _p(np.ascontiguousarray(ref_normal, np.float64)),
                           _p(np.ascontiguousarray(ref_px, np.float32)), int(ref_level),
                           _p(np.ascontiguousarray(pose_c2r, np.float64)), _p(A))
    return A.reshape(2, 2)


def best_search_level(A, max_level):
    return int(lib().orc_best_search_level(_p(np.ascontiguousarray(A, np.float64).reshape(-1)), int(max_level)))


def warp_affine(A, ref_img, ref_px, ref_level, search_level):
    ref_img = u8(ref_img)
    h, w = ref_img.shape
    out = np.empty(100, np.uint8)
    lib().orc_warp_affine(_p(np.ascontiguousarray(A, np.float64).reshape(-1)), _p(ref_img), w, h, w,
                          _p(np.ascontiguousarray(ref_px, np.float32)), int(ref_level), int(search_level), _p(out))
    return out


def patch_no_border(p10):
    p10 = u8(p10).reshape(-1)
    out = np.empty(64, np.uint8)
    lib().orc_patch_no_border(_p(p10), _p(out))
    return out


def align2d(cur_img, patch10, max_iters, px):
    cur_img = u8(cur_img)
    h, w = cur_img.shape
    p10 = u8(patch10).reshape(-1)
    p8 = patch_no_border(p10)
    p = np.array(px, np.float64)
    nit = C.c_int(0)
    conv = lib().orc_align2d(_p(cur_img), w, h, w, _p(p10), _p(p8), int(max_iters), _p(p), C.byref(nit))
    return p, bool(conv), nit.value


# ---------------------------------------------------------------- SE3
def ldlt6_solve(H, b):
    x = np.empty(6)
    lib().orc_ldlt6_solve(_p(np.ascontiguousarray(H, np.float64).reshape(-1)), _p(np.ascontiguousarray(b, np.float64)), _p(x))
    return x


def se3_exp(x):
    out = np.empty(7); lib().orc_se3_exp(_p(np.ascontiguousarray(x, np.float64)), _p(out)); return out


def se3_mul(a, b):
    out = np.empty(7)
    lib().orc_se3_mul(_p(np.ascontiguousarray(a, np.float64)), _p(np.ascontiguousarray(b, np.float64)), _p(out))
    return out


def se3_inv(a):
    out = np.empty(7); lib().orc_se3_inv(_p(np.ascontiguousarray(a, np.float64)), _p(out)); return out


def se3_act(a, p):
    out = np.empty(3)
    lib().orc_se3_act(_p(np.ascontiguousarray(a, np.float64)), _p(np.ascontiguousarray(p, np.float64)), _p(out))
    return out


def feature_normal(cam, px):
    out = np.empty(3)
    lib().orc_feature_normal(C.byref(cam), _p(np.ascontiguousarray(px, np.float32)), _p(out))
    return out


def is_in_image(cam, x, y, boundary, level=0):
    return bool(lib().orc_is_in_image(C.byref(cam), float(np.float32(x)), float(np.float32(y)), int(boundary), int(level)))


def reproject_point(cam, pose_cur_c2w, point_w, cell_size, grid_cols):
    """-> (in_image, px[2], cell or -1)"""
    px = np.empty(2); cell = C.c_int(-1)
    ok = lib().orc_reproject_point(C.byref(cam), _p(np.ascontiguousarray(pose_cur_c2w, np.float64)), _p(np.ascontiguousarray(point_w, np.float64)),
                                   int(cell_size), int(grid_cols), _p(px), C.byref(cell))
    return bool(ok), px, (cell.value if ok else -1)


def closest_obs(cur_center, point_w, kf_centers):
    """-> (returned bool, index of the chosen observation or -1)"""
    kc = np.ascontiguousarray(kf_centers, np.float64).reshape(-1, 3)
    best = C.c_int(-1)
    ok = lib().orc_closest_obs(_p(np.ascontiguousarray(cur_center, np.float64)), _p(np.ascontiguousarray(point_w, np.float64)),
                               _p(kc), len(kc), C.byref(best))
    return bool(ok), best.value


def undistort_points(cam, dist, src):
    src = np.ascontiguousarray(src, np.float32).reshape(-1, 2)
    dst = np.empty_like(src)
    lib().orc_undistort_points(C.byref(cam), _p(np.ascontiguousarray(dist, np.float32)), _p(src), len(src), _p(dst))
    return dst


def depth_convert(depth_u16, depth_scale):
    d = np.ascontiguousarray(depth_u16, np.uint16)
    out = np.empty(d.shape, np.float32)
    lib().orc_depth_convert(_p(d), d.size, float(np.float32(depth_scale)), _p(out))
    return out


def feature_depth(depth_f32, px):
    d = np.ascontiguousarray(depth_f32, np.float32)
    return float(lib().orc_feature_depth(_p(d), d.shape[1], d.shape[0], _p(np.ascontiguousarray(px, np.float32))))


def unproject(cam, pose_c2w, px, d):
    out = np.empty(3)
    lib().orc_unproject(C.byref(cam), _p(np.ascontiguousarray(pose_c2w, np.float64)), _p(np.ascontiguousarray(px, np.float32)),
                        float(np.float32(d)), _p(out))
    return out


def clahe(img, clip_limit=3.0, tiles=(8, 8)):
    """cv::createCLAHE(clip_limit, tiles)->apply(img) for sizes divisible by the tile grid."""
    a = u8(img)
    h, w = a.shape
    assert w % tiles[0] == 0 and h % tiles[1] == 0
    out = np.empty_like(a)
    f = lib().orc_clahe
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_void_p]
    f(_p(a), w, h, float(clip_limit), int(tiles[0]), int(tiles[1]), _p(out))
    return out


def pair_batch(cam, levels, ref_pyrs, cur_imgs, feats, n_feats, ref_centers, poses_in, max_level, min_level,
               max_iters, patches10, patch_px, patch_level, align_iters, n_threads):
    """CPU restatement of one bench 'step' over n_pairs pairs (pyramid(cur) + Run + Align2D per patch)."""
    n_pairs = len(n_feats)
    feats = np.ascontiguousarray(feats, REF_FEAT_DT)
    fpp = feats.size // n_pairs
    ppp = patch_level.size // n_pairs
    poses_out = np.empty((n_pairs, 7)); n_tracked = np.empty(n_pairs, np.int32)
    px_out = np.empty((n_pairs, ppp, 2)); conv = np.empty((n_pairs, ppp), np.uint8)
    lib().orc_pair_batch(C.byref(cam), int(levels), _p(u8(ref_pyrs)), _p(u8(cur_imgs)), n_pairs, _p(feats), fpp,
                         _p(np.ascontiguousarray(n_feats, np.int32)), _p(np.ascontiguousarray(ref_centers, np.float64)),
                         _p(np.ascontiguousarray(poses_in, np.float64)), int(max_level), int(min_level), int(max_iters),
                         _p(u8(patches10)), _p(np.ascontiguousarray(patch_px, np.float64)),
                         _p(np.ascontiguousarray(patch_level, np.int32)), ppp, int(align_iters), int(n_threads),
                         _p(poses_out), _p(n_tracked), _p(px_out), _p(conv))
    return poses_out, n_tracked, px_out, conv


REPROJ_DT = np.dtype([("px_proj", "<f8", 2), ("px", "<f8", 2), ("cell", "<i4"), ("obs", "<i4"), ("flags", "<i4"), ("level", "<i4")])


def pair_batch_map(cam, levels, cell_size, ref_pyrs, cur_imgs, feats, n_feats, ref_centers, poses_ref, poses_in, max_level, min_level,
                   max_iters, points_per_pair, max_search_level, align_iters, n_threads):
    """CPU restatement of one bench step with the reference's refinement chain (pyramid(cur) + Run + per-feature FindMatchDirect)."""
    n_pairs = len(n_feats)
    feats = np.ascontiguousarray(feats, REF_FEAT_DT)
    fpp = feats.size // n_pairs
    poses_out = np.empty((n_pairs, 7)); n_tracked = np.empty(n_pairs, np.int32)
    rep = np.zeros((n_pairs, points_per_pair), REPROJ_DT)
    lib().orc_pair_batch_map(C.byref(cam), int(levels), int(cell_size), _p(u8(ref_pyrs)), _p(u8(cur_imgs)), n_pairs, _p(feats), fpp,
                             _p(np.ascontiguousarray(n_feats, np.int32)), _p(np.ascontiguousarray(ref_centers, np.float64)),
                             _p(np.ascontiguousarray(poses_ref, np.float64)), _p(np.ascontiguousarray(poses_in, np.float64)),
                             int(max_level), int(min_level), int(max_iters), int(points_per_pair), int(max_search_level), int(align_iters),
                             int(n_threads), _p(poses_out), _p(n_tracked), _p(rep))
    return poses_out, n_tracked, rep


BA_SUMMARY_DT = np.dtype([("iterations", "<i4"), ("termination", "<i4"), ("n_successful", "<i4"), ("pad", "<i4"),
                          ("initial_cost", "<f8"), ("final_cost", "<f8")])
BA_FUNCTION_TOL, BA_PARAMETER_TOL, BA_GRADIENT_TOL, BA_NO_CONVERGENCE, BA_FAILURE, BA_MIN_RADIUS, BA_NO_RESIDUALS = range(7)


def pose_optimization(normals, levels, points_w, pose_in, max_iters=100):
    """Optimizer::PoseOptimization (ceres::Solve restated). Returns (pose_out[7], res_norm[n], summary record)."""
    nm = np.ascontiguousarray(normals, np.float64).reshape(-1, 3)
    lv = np.ascontiguousarray(levels, np.int32).reshape(-1)
    pw = np.ascontiguousarray(points_w, np.float64).reshape(-1, 3)
    assert len(nm) == len(lv) == len(pw)
    out = np.zeros(7); res = np.zeros(len(lv)); summ = np.zeros(1, BA_SUMMARY_DT)
    f = lib().orc_pose_optimization
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    f(len(lv), _p(nm), _p(lv), _p(pw), _p(np.ascontiguousarray(pose_in, np.float64)), int(max_iters), _p(out), _p(res), _p(summ))
    return out, res, summ[0]


def close_keyframes(cam, pose_cur_c2w, pt_begin, pt_count, kf_t, points_w, max_local=10):
    """Tracking::GetCloseKeyFrames + UpdateLocalMap's ranking -> (visible, dist, local rows)."""
    pb = np.ascontiguousarray(pt_begin, np.int32); pc = np.ascontiguousarray(pt_count, np.int32)
    kt = np.ascontiguousarray(kf_t, np.float64).reshape(-1, 3); pw = np.ascontiguousarray(points_w, np.float64).reshape(-1, 3)
    n = len(pb)
    vis = np.zeros(n, np.uint8); dist = np.zeros(n); local = np.zeros(max(max_local, 1), np.int32)
    f = lib().orc_close_keyframes
    f.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    k = f(C.byref(cam), _p(np.ascontiguousarray(pose_cur_c2w, np.float64)), _p(pb), _p(pc), _p(kt), n, _p(pw), int(max_local), _p(vis), _p(dist), _p(local))
    return vis, dist, local[:k].copy()
