"""CPU suite for the device's restatement of libstdc++'s std::sort (dsdtm_b200/csrc/std_sort.cuh, compiled for the host -- the
very source detect_select_kernel runs when scores tie): on the corner record and the score-descending comparator of
Feature_detector::detect it must leave every element where g++'s std::sort does. The cell index rides in the record, so equal
scores in a different order fail the comparison."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CORNER_DT = np.dtype([("x", "<i4"), ("y", "<i4"), ("level", "<i4"), ("score", "<f4")])


@pytest.fixture(scope="module")
def sorts():
    d = os.path.join(ROOT, "tests", "cpp", "_build")
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, "libstd_sort_host.so")
    src = os.path.join(ROOT, "tests", "cpp", "std_sort_host.cpp")
    deps = [src, os.path.join(ROOT, "dsdtm_b200", "csrc", "std_sort.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", src, "-o", so])
    lib = C.CDLL(so)
    lib.prod_sort_corners.argtypes = [C.c_void_p, C.c_long]
    lib.ref_sort_corners.argtypes = [C.c_void_p, C.c_long]

    def run(scores):
        c = np.zeros(len(scores), CORNER_DT)
        c["x"] = np.arange(len(scores))
        c["score"] = scores
        a, b = c.copy(), c.copy()
        lib.prod_sort_corners(a.ctypes.data, len(a))
        lib.ref_sort_corners(b.ctypes.data, len(b))
        return a, b
    return run


def _median_of_three_killer(n):
    """Musser's median-of-three killer. Against libstdc++'s pivot (median of first + 1, mid, last - 1) it makes enough lopsided
    partitions that the depth limit is reached: n = 1376 takes the heap-sort fallback 4 times, n = 5000 18 times."""
    k = n // 2
    a = np.zeros(n, np.float32)
    for i in range(1, k + 1):
        if i % 2:
            a[i - 1] = i
            a[i] = k + i
        a[k + i - 1] = 2 * i
    return -a            # the comparator sorts descending


def _inputs():
    rng = np.random.default_rng(7)
    out = []
    for n in (0, 1, 2, 15, 16, 17, 33, 416, 1376, 5000):
        out += [("random", rng.random(n, np.float32) * 100), ("equal", np.full(n, 42.0, np.float32)),
                ("two", rng.integers(0, 2, n).astype(np.float32) + 21), ("few", rng.integers(0, 5, n).astype(np.float32) * 10),
                ("ascending", np.arange(n, dtype=np.float32)), ("descending", np.arange(n, dtype=np.float32)[::-1].copy()),
                ("organ", np.concatenate([np.arange(n // 2), np.arange(n - n // 2)[::-1]]).astype(np.float32))]
    out += [("killer", _median_of_three_killer(n)) for n in (64, 1376, 5000)]
    return out


@pytest.mark.parametrize("name,scores", _inputs(), ids=lambda v: v if isinstance(v, str) else str(len(v)))
def test_std_sort_restatement_matches_gxx_permutation(sorts, name, scores):
    a, b = sorts(scores)
    assert (a["x"] == b["x"]).all(), name


def test_killer_reaches_the_heap_sort_fallback(sorts):
    """The killer sequence must really exercise __partial_sort: a quicksort-only restatement (no depth limit) would not
    match g++ there, and the order of equal keys after the fallback is not that of a stable sort."""
    s = _median_of_three_killer(1376)
    s = np.round(s / 8)              # ties inside the heap-sorted ranges
    a, b = sorts(s.astype(np.float32))
    assert (a["x"] == b["x"]).all()
    stable = np.argsort(-s, kind="stable")
    assert not (a["x"] == stable).all()


def _tiled(period, seed, w=640, h=480):
    rng = np.random.default_rng(seed)
    block = rng.integers(0, 256, (period, period)).astype(np.uint8)
    return np.tile(block, (-(-h // period), -(-w // period)))[:h, :w].copy()


@pytest.mark.parametrize("period", [15, 30, 45])
def test_tiled_scene_cells_sort_like_gxx(sorts, period):
    img = _tiled(period, period)
    packed, offs, ws, hs = O.pyramid(img, 5)
    cells = O.detect_cells(packed, offs, ws, hs, 15, None, 5.0)
    a, b = sorts(cells["score"])
    assert (a["x"] == b["x"]).all()
    sel = cells["score"][cells["score"] > 20]
    assert len(sel) > len(np.unique(sel)), "the tiled scene must carry tied scores above 20"
