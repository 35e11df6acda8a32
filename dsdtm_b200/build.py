"""In-tree build of the sm_100a CUDA library (dsdtm_b200/lib/libdsdtm_gpu.so) with nvcc.

The built .so is git-ignored but travels to the GPU box with the gpurun snapshot. Rebuilds only when a source is newer.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# DSDTM_GPU_LIB: measurement scripts load a prebuilt experiment library (scripts/sa_build_variants.py) instead of the default build
LIB = os.environ.get("DSDTM_GPU_LIB") or os.path.join(LIBDIR, "libdsdtm_gpu.so")
SOURCES = ["capi.cu", "pyramid.cu", "fast.cu", "sparse_align.cu", "align2d.cu", "local_map.cu", "ingest.cu", "clahe.cu", "pose_opt.cu", "select.cu", "detect_select.cu", "keyframe.cu", "store_commit.cu", "sequence_advance.cu", "probe.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--fmad=true", "-Xptxas", "-v"]


def extra_flags():
    """DSDTM_NVCC_FLAGS lets experiments add -D switches (e.g. on the GPU box) without editing sources."""
    return os.environ.get("DSDTM_NVCC_FLAGS", "").split()


def nvcc():
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found: the CUDA library cannot be built (there is no CPU fallback)")
    return p


def _headers():
    """Every header a translation unit may include: a change to any of them rebuilds every object (the context struct is
    shared by all of them; a stale object with an old layout corrupts memory silently)."""
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + [os.path.join(ROOT, "include", "dsdtm_gpu.h")]


def _deps():
    return [os.path.join(CSRC, s) for s in SOURCES] + _headers()


STAMP = os.path.join(LIBDIR, "flags.stamp")


def _flag_key():
    return " ".join(NVCC_FLAGS + extra_flags())


def _stamp_matches():
    """The flags the objects in lib/ were compiled with. An experiment built with DSDTM_NVCC_FLAGS must never be mistaken for the
    default build by a later plain build() (the library is newer than every source in that case)."""
    try:
        with open(STAMP) as f:
            return f.read() == _flag_key()
    except OSError:
        return False


def stale():
    if os.environ.get("DSDTM_GPU_LIB"):
        return False                      # an explicitly named library is taken as it is
    if not os.path.exists(LIB) or not _stamp_matches():
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    if not _stamp_matches():
        force = True                      # other flags: every object is rebuilt
    objs = []
    log = []
    for s in SOURCES:
        o = os.path.join(LIBDIR, s.replace(".cu", ".o"))
        src = os.path.join(CSRC, s)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(p) for p in [src] + _headers()):
            cmd = [nvcc()] + NVCC_FLAGS + extra_flags() + ["-c", src, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            log.append(r.stderr)
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc failed for %s" % s)
        objs.append(o)
    cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(LIBDIR, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    with open(STAMP, "w") as f:
        f.write(_flag_key())
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(LIB)
