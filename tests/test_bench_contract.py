"""The JSON contract of bench.py's reference arm (`--impl reference`: the oracle port of the path on the host cores, rank 0 only)
for both camera geometries, and `--dump-outputs` of both arms: repeatable on the CPU, and the CUDA arm's outputs equal to the
reference arm's on the same batch (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra, env=None):
    e = dict(os.environ); e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-sample", "8", "--scenes", "2"] + extra, capture_output=True, text=True, env=e, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


@pytest.mark.parametrize("cam,size", [("kinect", "640x480"), ("euroc", "752x480")])
def test_reference_arm_line(built, cam, size):
    lines = _run(["--cam", cam])
    assert len(lines) == 1                                              # ONE JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frame_pairs/s" and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert size in d["metric"] and size in d["config"]["workload"] and d["config"]["camera"] == cam
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None and d["dtype"] == "f64"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "8 pairs" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly(built):
    # under torchrun only rank 0 runs the CPU arm; the other ranks print nothing and exit 0
    lines = _run([], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert lines == []


DUMPED = {"pair_index": (np.float64, ()), "poses": (np.float64, (7,)), "n_tracked": (np.float64, ()),
          "patch_px": (np.float64, (300, 2)), "patch_converged": (np.float32, (300,))}


def _load_dump(d, n=None):
    """the files of one --dump-outputs DIR; n: every pair of an n-pair batch was written"""
    assert sorted(os.listdir(d)) == sorted(k + ".npy" for k in DUMPED)
    out = {k: np.load(os.path.join(d, k + ".npy")) for k in DUMPED}
    for k, (dt, shape) in DUMPED.items():
        assert out[k].dtype == dt and out[k].shape == (len(out["pair_index"]),) + shape, k
    if n is not None:
        assert (out["pair_index"] == np.arange(n)).all()
    return out


def test_reference_arm_dumps_the_same_outputs_every_run(built, tmp_path):
    runs = []
    for r in range(2):
        d = str(tmp_path / ("run%d" % r))
        lines = _run(["--steps", "2", "--dump-outputs", d])
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
        runs.append(_load_dump(d, 8))
    for k in DUMPED:
        assert (runs[0][k] == runs[1][k]).all(), k
    assert runs[0]["patch_converged"].sum() > 0 and (runs[0]["n_tracked"] > 0).all()


def test_dump_above_the_size_limit_is_a_fixed_sample_of_pairs(tmp_path):
    import bench
    n = 12000                                                       # 12000 pairs x 6072 bytes > 64 MB
    rng = np.random.default_rng(3)
    poses = rng.normal(size=(n, 7)); nt = rng.integers(0, 301, n).astype(np.int32)
    px = rng.normal(size=(n, 300, 2)); conv = rng.integers(0, 2, (n, 300)).astype(np.uint8)
    got = []
    for r in range(2):
        d = str(tmp_path / ("run%d" % r))
        bench.dump_outputs(d, poses, nt, px, conv)
        assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= bench.DUMP_LIMIT
        got.append(_load_dump(d))
    idx = got[0]["pair_index"].astype(np.int64)
    assert 10000 < len(idx) < n and (np.diff(idx) > 0).all() and idx[-1] < n
    assert (got[0]["pair_index"] == got[1]["pair_index"]).all()
    assert (got[0]["poses"] == poses[idx]).all() and (got[0]["n_tracked"] == nt[idx]).all()
    assert (got[0]["patch_px"] == px[idx]).all() and (got[0]["patch_converged"] == conv[idx]).all()


@pytest.mark.gpu
def test_gpu_arm_dump_matches_the_reference_arm(built, tmp_path):
    """--dump-outputs of the CUDA path against the reference arm's on the same batch (north_star tolerances)."""
    n = 32
    g, c = str(tmp_path / "gpu"), str(tmp_path / "cpu")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--pairs", str(n), "--scenes", "2",
                          "--no-cpu", "--no-strong", "--dump-outputs", g], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    _run(["--pairs", str(n), "--cpu-sample", str(n), "--dump-outputs", c])
    a, b = _load_dump(g, n), _load_dump(c, n)
    from dsdtm_b200 import synth as S
    for i in range(n):
        d = S.pose_dist(a["poses"][i], b["poses"][i])
        assert d[0] < 1e-5 and d[1] < 1e-5, (i, d)
    assert (a["n_tracked"] == b["n_tracked"]).all()
    # a flag may differ only where |d|^2 straddles the convergence threshold within fp32 rounding (test_gpu_align.py)
    assert (a["patch_converged"] != b["patch_converged"]).mean() < 1e-3
    ok = (a["patch_converged"] == 1) & (b["patch_converged"] == 1)
    assert ok.sum() > n * 100 and np.abs(a["patch_px"][ok] - b["patch_px"][ok]).max() <= 1e-3


def test_roofline_inputs_of_the_gpu_arm_are_committed():
    """bench.py's `roofline` for the dominant kernel reads the newest committed ncu capture (profiles/*_traffic.json): the FP64-pipe
    instruction count and the DRAM traffic per pair must be there and plausible, or the bench line silently loses its roofline."""
    import bench
    p = bench.traffic_file()
    assert os.path.exists(p), p
    fpi = bench.fp64_insts_per_pair("sparse_align_kernel")
    tr = bench.measured_traffic("sparse_align_kernel", 4096)
    assert fpi is not None and 5e4 < fpi < 2e5                      # ~78 k FP64 warp instructions per pair
    assert tr is not None and 1e9 < tr < 5e9                        # ~2.3 GB per launch of 4096 pairs
    s = bench.ncu_summary("sparse_align_kernel")
    assert "fp64_pipe_pct" in s and "source" in s
