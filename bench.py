#!/usr/bin/env python
"""bench.py -- the tracking front end's hot path on batches of independent synthetic frame pairs.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one batch of B frame pairs per GPU, all inputs resident in HBM:
    pyramid(cur frame) -> Sprase_ImgAlign (levels max_level-1..0, Gauss-Newton on SE3) -> Align2D of the pair's patches.
`value` = frame pairs / s over all ranks (max-over-ranks device time, CUDA events on the launching stream).
`e2e`   = the same metric through the C-ABI call with HOST (pinned) buffers: H2D of the cur images + per-pair inputs and
          D2H of the results inside the timed region.
The reference arm (--impl reference) times the CPU restatement of the reference (oracle/, kind "port": the reference itself
needs OpenCV/Eigen/Sophus/Ceres and cannot be built here) on all host threads.
--dump-outputs DIR writes what the timed path returned in its last step for rank 0's batch (poses, tracked counts, refined patch positions and
flags, float32 / float64 .npy) for comparing two builds on the same seeded inputs.
No pair shards across GPUs: N > 1 = N independent replicas of the batch (weak scaling), no collective on the data path.
Extra keys on the same line: `refine_chain` = the step with the reference's own refinement chain (reprojection -> closest observation ->
affine -> warp -> Align2D on the device) instead of host patches; `strong_scaling` = BASELINE configs[4] as written: ONE batch of 4096
EuRoC 752x480 pairs partitioned over the ranks (contiguous blocks, SURVEY 8e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "sparse-align frame pairs/sec (640x480, 300 feats)"
UNIT = "frame_pairs/s"
ALIGN_CFG = dict(max_level=4, min_level=0, max_iters=30)      # Test/test_SpraseImg_alignment.cpp:110 -> Sprase_ImgAlign(4, 0, 30)
LEVELS = 5                                                      # Camera.MaxPyraLevels (Config/kinect.yaml:66)
ALIGN2D_ITERS = 10                                              # src/Feature_alignment.cpp:152
N_FEATS = 300
FEAT_STRIDE = 320


def make_config(cam_name, cam, B):
    """The `config` object: identical in the GPU arm and in the reference arm (the driver compares them)."""
    w, h = cam["width"], cam["height"]
    pyr = 0
    for _ in range(LEVELS):
        pyr += w * h
        w, h = (w + 1) // 2, (h + 1) // 2
    return {"workload": "%s: %d independent %dx%d %s frame pairs per GPU, %d FAST/Shi-Tomasi features, 5-level pyramid(cur) + "
                        "Sprase_ImgAlign(4,0,30) + Align2D(%d patches, 10 it)"
                        % ("configs[4] sweep" if cam_name == "euroc" else "configs[0] shape batched", B, cam["width"], cam["height"], cam_name, N_FEATS, N_FEATS),
            "camera": cam_name, "pairs_per_gpu": B, "features": N_FEATS, "levels": LEVELS, "sparse_align": ALIGN_CFG, "align2d_iters": ALIGN2D_ITERS,
            "l2": "inputs larger than L2 (%.0f MB of pyramids per step)" % (2 * B * pyr / 1e6)}


def shard(n_total, world, rank):
    """Contiguous block partition of n_total independent units over `world` ranks (SURVEY 8e)."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed regions: NVML polled every 2 ms from a thread (the C-ABI calls release the GIL),
    filtered to the wall-clock window of a region afterwards. Falls back to `nvidia-smi -lms 20` when NVML cannot be loaded."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.samples = []            # (t, sm_mhz, max_mhz, set(reasons))
        self.p = None
        self.nvml = None
        self.how = None
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.how = "NVML, 2 ms period"
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.how = "nvidia-smi -lms 20"
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _poll(self):
        N = self.nvml
        bits = (("hw_slowdown", getattr(N, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                ("hw_thermal_slowdown", getattr(N, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                ("sw_thermal_slowdown", getattr(N, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                ("sw_power_cap", getattr(N, "nvmlClocksEventReasonSwPowerCap", 0x4)))
        reasons_fn = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(N, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                mhz = float(N.nvmlDeviceGetClockInfo(self.h, N.NVML_CLOCK_SM))
                mask = int(reasons_fn(self.h))
                self.samples.append((time.perf_counter(), mhz, self.max_mhz, {n for n, b in bits if mask & b}))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for line in self.p.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                sm, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.samples.append((time.perf_counter(), sm, mx, {n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")}))

    def wait_first(self, timeout=5.0):
        t0 = time.perf_counter()
        while (self.p or self.nvml) and not self.samples and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def stop(self):
        self._stop.set()
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=2)
            except Exception:
                self.p.kill()

    def summary(self, t0, t1):
        if not (self.p or self.nvml):
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["neither NVML nor nvidia-smi available"], "samples": 0}
        sel = [x for x in self.samples if t0 <= x[0] <= t1 + 0.03]
        reasons = set()
        for x in sel:
            reasons |= x[3]
        return {"sm_mhz": float(np.median([x[1] for x in sel])) if sel else None, "sm_max_mhz": max(x[2] for x in sel) if sel else None,
                "reasons": sorted(reasons), "samples": len(sel), "sampler": self.how}


def bind_to_gpu_numa(index):
    """Pin this rank to the CPUs of its GPU's NUMA node BEFORE any pinned host buffer is allocated (cudaHostAlloc places pages by the
    calling thread's policy = local node): with 4-8 ranks on one box the H2D streams otherwise share one socket's memory controllers and
    cross the inter-socket link (r1: e2e efficiency 0.43 at 8 GPUs)."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=10).stdout.strip().lower()
        if bus.count(":") == 2 and len(bus.split(":")[0]) == 8:
            bus = bus[4:]                                   # 00000000:1b:00.0 -> 0000:1b:00.0
        d = "/sys/bus/pci/devices/" + bus
        node = int(open(d + "/numa_node").read().strip())
        cpus = set()
        for part in open(d + "/local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if node >= 0 and cpus:
            os.sched_setaffinity(0, cpus)
            return {"node": node, "cpus": len(cpus), "bound": True}
        return {"node": node, "cpus": len(os.sched_getaffinity(0)), "bound": False}
    except Exception as e:                                   # no sysfs / single-node box: nothing to bind
        return {"node": None, "cpus": len(os.sched_getaffinity(0)), "bound": False, "note": str(e)[:80]}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_file():
    """the newest committed ncu --set full capture of the dominant kernel"""
    for name in ("r2e_traffic.json", "r2d_traffic.json", "r2b_traffic.json", "r2_traffic.json", "r1_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            return p
    return os.path.join(ROOT, "profiles", "r2_traffic.json")


def fp64_insts_per_pair(kernel):
    """smsp__inst_executed_pipe_fp64.sum (warp instructions on the FP64 pipe) per pair from the committed capture, or None"""
    p = traffic_file()
    if not os.path.exists(p):
        return None
    t = json.load(open(p)).get(kernel) or {}
    return t.get("fp64_warp_insts_per_pair")


def ncu_summary(kernel):
    """Pipe / issue figures of `kernel` from the committed ncu --set full capture (profiles/r1_traffic.json); {} if absent."""
    p = traffic_file()
    if not os.path.exists(p):
        return {}
    t = json.load(open(p)).get(kernel) or {}
    return {k: t[k] for k in ("issue_slots_busy_pct", "fp64_pipe_pct", "dram_throughput_pct", "l1tex_hit_pct", "l2_hit_pct", "warp_instructions", "fp64_warp_insts_per_pair", "source") if k in t}


def measured_traffic(kernel, pairs):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture
    (profiles/r1_traffic.json, taken at 4096 pairs), scaled per pair. None if the capture is absent."""
    p = traffic_file()
    if not os.path.exists(p):
        return None
    t = json.load(open(p)).get(kernel)
    return None if not t else float(t["bytes_per_pair"]) * pairs


DUMP_LIMIT = 64 << 20


def dump_outputs(d, poses, n_tracked, px, conv):
    """--dump-outputs: what the timed path returned for its last step, one float array per output as DIR/<name>.npy, so that two
    builds can be compared output for output on the same seeded inputs. Above DUMP_LIMIT bytes a fixed seeded sample of the pairs is
    written; pair_index.npy names the pairs either way."""
    n = len(poses)
    per_pair = 8 * (1 + 7 + 1 + px[0].size) + 4 * conv[0].size
    idx = np.arange(n)
    if n * per_pair > DUMP_LIMIT - 4096:                       # 4 KB for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, (DUMP_LIMIT - 4096) // per_pair, replace=False))
    os.makedirs(d, exist_ok=True)
    out = {"pair_index": idx.astype(np.float64), "poses": poses[idx], "n_tracked": n_tracked[idx].astype(np.float64),
           "patch_px": px[idx], "patch_converged": conv[idx].astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a))


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dsdtm_b200 import capi, synth as S, workload as W

    rank, world, local = dist_setup(args.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    full_affinity = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cam = dict(S.EUROC if args.cam == "euroc" else S.KINECT)
    B = args.pairs
    ctx = capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=N_FEATS, max_frames=2 * B + 2, max_batch=B,
                       device=local)
    t0 = time.time()
    # scene rendering is CPU work outside the timed regions: share the host cores between the ranks of the box
    render_procs = max(1, min(args.scenes, (os.cpu_count() or 2) // (2 * world)))
    scenes = W.render_scenes(args.scenes, cam, seed0=W.BASE_SEED + 1000 * rank, procs=render_procs)
    batch = W.build_batch(ctx, cam, B, n_scenes=args.scenes, n_feats=N_FEATS, feat_stride=FEAT_STRIDE, patches_per_pair=N_FEATS,
                          seed0=W.BASE_SEED + 1000 * rank, scenes=scenes)
    prep_s = time.time() - t0
    ppp = batch["patches_per_pair"]
    ctx.batch_stage(batch["ref_slots"], batch["cur_slots"], batch["feats"], batch["n_feats"], batch["centers"], batch["poses_in"],
                    ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"], batch["patch_px"],
                    batch["patch_level"], ALIGN2D_ITERS)

    def restage():
        # single-call entry points reuse the staging buffers: stage the batch again before batch_run
        ctx.batch_stage(batch["ref_slots"], batch["cur_slots"], batch["feats"], batch["n_feats"], batch["centers"], batch["poses_in"],
                        ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"], batch["patch_px"],
                        batch["patch_level"], ALIGN2D_ITERS)

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # ---------------- device-resident steps (value)
    clocks = ClockSampler(local)
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        ctx.batch_run(1)
    ctx.sync()
    poses, n_tracked, px, conv = ctx.batch_fetch()
    # sanity: converged to the ground-truth motion (checked on every rank; parity proper lives in tests/)
    err = np.array([S.pose_dist(poses[i], batch["truth"][i]) for i in range(min(B, 64))])
    if not (np.median(err[:, 0]) < 5e-4 and np.median(err[:, 1]) < 1e-3):
        raise SystemExit("bench.py: alignment did not converge to the synthetic ground truth: %s" % np.median(err, 0))
    barrier()
    l0 = ctx.launch_count()
    clocks.wait_first()
    tw0 = time.perf_counter()
    ctx.timer_start()
    for _ in range(args.steps):
        ctx.batch_run(1)
    dev_ms = ctx.timer_stop()
    tw1 = time.perf_counter()
    launches = ctx.launch_count() - l0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *ctx.batch_fetch())
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    ms_per_step = max_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ---------------- per-stage device times (profiling pass, outside the timed region; events per stage)
    ctx.profile(True)
    ctx.profile_get(reset=True)
    for _ in range(args.steps):
        ctx.batch_run(1)
    stages = ctx.profile_get(reset=True)
    ctx.profile(False)
    sa_ms = stages["sparse_align"][0] / max(stages["sparse_align"][1], 1)
    pyr_ms = stages["pyramid"][0] / args.steps
    a2d_ms = stages["align2d"][0] / max(stages["align2d"][1], 1)
    # iterations actually executed (for the algorithmic byte count)
    _, _, log, nlog = ctx.sparse_align_batch(batch["ref_slots"][:min(B, 64)], batch["cur_slots"][:min(B, 64)], batch["feats"][:min(B, 64)],
                                             batch["n_feats"][:min(B, 64)], batch["centers"][:min(B, 64)], batch["poses_in"][:min(B, 64)],
                                             ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], log_cap=128)
    iters = float(np.mean(nlog))
    n_levels = ALIGN_CFG["max_level"] - ALIGN_CFG["min_level"]
    restage()
    hbm_peak, peak_src = peaks()
    fp64_tflops, dfma_per_clk_sm = ctx.probe_fp64()          # measured live: dependency-free DFMA streams on this GPU
    sa_bytes = B * (int(np.mean(batch["n_feats"])) * (64 + 49 * n_levels + 25 * iters) + 112)
    g = ctx
    pyr_bytes = B * sum(g.ws[l - 1] * g.hs[l - 1] + g.ws[l] * g.hs[l] for l in range(1, LEVELS))
    # FAST stage (keyframes only, not part of the step): timed separately over the ref frames for its roofline
    nfast = min(B, 256)
    ctx.profile(True); ctx.profile_get(reset=True)
    cells_tmp = np.zeros(nfast * ctx.n_cells, capi.CORNER_DT)
    fast_ms = None
    try:
        # consecutive slots 0..nfast-1 hold ref/cur frames alternately: all are valid pyramids
        for _ in range(3):
            ctx._ck(ctx.L.dsdtm_fast_cells_batch(ctx.hp, 0, nfast, 20, capi.C.c_float(5.0), None, capi._p(cells_tmp)))
        st = ctx.profile_get(reset=True)
        fast_ms = st["fast"][0] / max(st["fast"][1], 1)
    finally:
        ctx.profile(False)
    fast_bytes = nfast * (sum(g.ws[l] * g.hs[l] for l in range(LEVELS)) + ctx.n_cells * 16)

    # ---------------- the step with the reference's own refinement chain (VERDICT r1 item 7): patches are NOT host inputs; every
    # reference feature with a map point is reprojected through the aligned pose, gated, affine-warped from the reference frame and
    # refined by Align2D on the device (dsdtm_batch_stage_map / dsdtm_batch_run(flags | 2)) -- dsdtm_track_frame, batched
    ctx.batch_stage_map(batch["poses_ref"], N_FEATS, LEVELS - 3, ALIGN2D_ITERS)
    for _ in range(max(args.warmup, 3)):
        ctx.batch_run(3)
    ctx.sync()
    rep = ctx.batch_fetch_map()
    chain_conv = float(((rep["flags"] & capi.LM_CONVERGED) != 0).sum() / max(int(batch["n_feats"].sum()), 1))
    if chain_conv < 0.5:
        raise SystemExit("bench.py: refinement chain converged on %.0f %% of the features only" % (100 * chain_conv))
    barrier()
    lc0 = ctx.launch_count()
    ctx.timer_start()
    for _ in range(args.steps):
        ctx.batch_run(3)
    chain_ms = ctx.timer_stop()
    chain_launches = ctx.launch_count() - lc0
    barrier()
    tc = torch.tensor([chain_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    chain_ms_per_step = float(tc.item()) / args.steps
    ctx.profile(True); ctx.profile_get(reset=True)
    for _ in range(args.steps):
        ctx.batch_run(3)
    cst = ctx.profile_get(reset=True)
    ctx.profile(False)
    chain_stages = {k_: cst[k_][0] / args.steps for k_ in ("pyramid", "sparse_align", "local_map", "warp_affine", "align2d")}

    # ---------------- single-pair latency (BASELINE target: < 200 us sparse alignment + feature refinement per 640x480 frame)
    def stage_n(n):
        ctx.batch_stage(batch["ref_slots"][:n], batch["cur_slots"][:n], batch["feats"][:n], batch["n_feats"][:n], batch["centers"][:n],
                        batch["poses_in"][:n], ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"][:n],
                        batch["patch_px"][:n], batch["patch_level"][:n], ALIGN2D_ITERS)
    stage_n(1)
    for _ in range(5):
        ctx.batch_run(1)
    ctx.sync()
    reps = 50
    ctx.timer_start()
    for _ in range(reps):
        ctx.batch_run(1)                      # CUDA-graph replay of pyramid + sparse align + align2d for ONE pair
    lat_ms = ctx.timer_stop() / reps
    ctx.profile(True); ctx.profile_get(reset=True)
    for _ in range(reps):
        ctx.batch_run(1)
    lst = ctx.profile_get(reset=True)
    ctx.profile(False)
    latency = {"frame_us": lat_ms * 1e3, "sparse_align_us": lst["sparse_align"][0] / reps * 1e3, "align2d_us": lst["align2d"][0] / reps * 1e3,
               "pyramid_us": lst["pyramid"][0] / reps * 1e3, "sparse_plus_refine_us": (lst["sparse_align"][0] + lst["align2d"][0]) / reps * 1e3,
               "note": "one pair, 300 features + 300 patches; frame_us = graph replay of all 6 kernels (events on the launching stream); "
                       "per-stage numbers from direct launches with an event pair per stage"}
    # the same frame through the single-pair C-ABI calls an adapter makes (host buffers, synchronous, host wall clock; the
    # ctypes argument marshalling is hoisted out of the loop so that the number is what a C++ caller pays):
    # dsdtm_frame_upload_pyramid (H2D 300 KB + pyramid) -> dsdtm_sparse_align -> dsdtm_align2d_batch
    C_ = capi.C
    nf0 = int(batch["n_feats"][0])
    img0 = np.ascontiguousarray(batch["scenes"][0]["cur_img"])
    rs0, cs0 = int(batch["ref_slots"][0]), int(batch["cur_slots"][0])
    f0 = np.ascontiguousarray(batch["feats"][0][:nf0]); cen0 = np.ascontiguousarray(batch["centers"][0]); pose0 = np.ascontiguousarray(batch["poses_in"][0])
    lv0 = np.ascontiguousarray(batch["patch_level"][0], np.int32); pt0 = np.ascontiguousarray(batch["patches"][0], np.uint8)
    px0 = np.ascontiguousarray(batch["patch_px"][0], np.float64); pxio = px0.copy()
    po0 = np.empty(7); ntr0 = C_.c_int(0); nlog0 = C_.c_int(0); conv0 = np.zeros(len(lv0), np.uint8)
    P_ = lambda arr: arr.ctypes.data_as(C_.c_void_p)
    calls = (("upload_pyramid_us", ctx.L.dsdtm_frame_upload_pyramid, (ctx.hp, cs0, P_(img0), img0.shape[1])),
             ("sparse_align_call_us", ctx.L.dsdtm_sparse_align, (ctx.hp, rs0, cs0, P_(f0), nf0, P_(cen0), P_(pose0), ALIGN_CFG["max_level"], ALIGN_CFG["min_level"],
                                                                  ALIGN_CFG["max_iters"], P_(po0), C_.byref(ntr0), None, 0, C_.byref(nlog0))),
             ("align2d_call_us", ctx.L.dsdtm_align2d_batch, (ctx.hp, cs0, P_(lv0), P_(pt0), P_(pxio), len(lv0), ALIGN2D_ITERS, P_(conv0))))
    capi_lat = {}
    for name, fn, cargs in calls:
        tsum = 0.0
        for it in range(reps + 5):
            pxio[...] = px0
            t0 = time.perf_counter()
            rc = fn(*cargs)
            if it >= 5:
                tsum += time.perf_counter() - t0
            if rc != 0:
                raise RuntimeError("%s failed: %s" % (name, ctx.L.dsdtm_last_error(ctx.hp)))
        capi_lat[name] = tsum / reps * 1e6
    capi_lat["sparse_plus_refine_call_us"] = capi_lat["sparse_align_call_us"] + capi_lat["align2d_call_us"]
    # the whole front end of one frame as ONE call with one synchronisation (dsdtm_track_frame): upload + pyramid + sparse alignment +
    # device-side pose composition + reprojection / closest observation / affine warp / Align2D of the key frame's 300 map points
    T_ref0 = np.ascontiguousarray(batch["scenes"][0]["T_ref"], np.float64)
    kfs0 = np.zeros(1, capi.KF_VIEW_DT); kfs0[0]["slot"] = rs0; kfs0[0]["pose_c2w"] = T_ref0; kfs0[0]["center"] = cen0
    obs0 = np.zeros(nf0, capi.OBS_DT); pts0 = np.zeros(nf0, capi.MAP_POINT_DT)
    obs0["kf"] = 0; obs0["level"] = f0["level"]; obs0["px"] = f0["px"]; obs0["normal"] = f0["normal"]; obs0["point_w"] = f0["point_w"]
    pts0["point_w"] = f0["point_w"]; pts0["obs_begin"] = np.arange(nf0); pts0["obs_count"] = 1
    ti = capi.TrackIn(); to = capi.TrackOut(); rep0 = np.zeros(nf0, capi.REPROJ_DT)
    ti.ref_slot, ti.cur_slot, ti.img, ti.stride = rs0, cs0, img0.ctypes.data, img0.shape[1]
    ti.feats, ti.n_feats = f0.ctypes.data, nf0
    ti.ref_center[:] = [float(v) for v in cen0]; ti.pose_ref_c2w[:] = [float(v) for v in T_ref0]; ti.pose_c2r_in[:] = [float(v) for v in pose0]
    ti.max_level, ti.min_level, ti.max_iters = ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"]
    ti.kfs, ti.n_kfs, ti.obs, ti.n_obs, ti.pts, ti.n_pts = kfs0.ctypes.data, 1, obs0.ctypes.data, nf0, pts0.ctypes.data, nf0
    ti.max_search_level, ti.align_iters = LEVELS - 3, ALIGN2D_ITERS
    tsum = 0.0
    for it in range(reps + 5):
        t0 = time.perf_counter()
        rc = ctx.L.dsdtm_track_frame(ctx.hp, C_.byref(ti), C_.byref(to), P_(rep0))
        if it >= 5:
            tsum += time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError("dsdtm_track_frame failed: %s" % ctx.L.dsdtm_last_error(ctx.hp))
    capi_lat["track_frame_call_us"] = tsum / reps * 1e6
    capi_lat["track_frame_matches"] = int(((rep0["flags"] & capi.LM_CONVERGED) != 0).sum())
    capi_lat["note"] = ("one frame through the three synchronous single-pair C-ABI calls with pageable host buffers, host wall clock "
                        "(H2D of inputs, kernel, D2H of results and the stream synchronisation inside each call)")
    latency["capi"] = capi_lat
    restage()

    # ---------------- keyframe ingest (SURVEY 8f-3 / 8f-4), not part of the step: depth convertTo (HBM-bound) and the per-feature lift
    ingest = None
    try:
        nd = 1024                                   # 1.9 GB of traffic per launch: well past L2
        ctx.set_option("depth_slots", nd)
        rng_d = np.random.default_rng(1)
        d16 = rng_d.integers(0, 65536, (cam["height"], cam["width"])).astype(np.uint16)
        for k_ in range(nd):
            ctx.depth_upload(k_, np.roll(d16, k_, axis=0) if k_ < 8 else d16)
        ctx.profile(True); ctx.profile_get(reset=True)
        for _ in range(5):
            ctx.depth_convert_f32(0, nd, 5000.0, fetch=False)
        st = ctx.profile_get(reset=True)
        conv_ms = st["ingest"][0] / max(st["ingest"][1], 1)
        px_l = np.stack([rng_d.integers(3, cam["width"] - 3, N_FEATS), rng_d.integers(3, cam["height"] - 3, N_FEATS)], 1).astype(np.float32)
        dist_l = (-0.28368365, 0.07451284, -0.00010473, -3.55590700e-05, 0.0)
        for _ in range(5):
            ctx.keyframe_lift(0, batch["poses_in"][0], dist_l, 5000.0, px_l)
        ctx.profile_get(reset=True)
        t0 = time.perf_counter()
        for _ in range(reps):
            ctx.keyframe_lift(0, batch["poses_in"][0], dist_l, 5000.0, px_l)
        lift_wall_us = (time.perf_counter() - t0) / reps * 1e6
        st = ctx.profile_get(reset=True)
        ctx.profile(False)
        conv_bytes = nd * cam["height"] * cam["width"] * 6
        ingest = {"depth_convert": {"ms_per_launch": conv_ms, "frames": nd, "algorithmic_bytes": conv_bytes, "GBps": conv_bytes / (conv_ms * 1e-3) / 1e9,
                                    "frac_hbm": conv_bytes / (conv_ms * 1e-3) / 1e9 / hbm_peak},
                  "keyframe_lift": {"features": N_FEATS, "kernel_us": st["ingest"][0] / max(st["ingest"][1], 1) * 1e3, "call_us": lift_wall_us,
                                    "note": "undistort + normal + depth lookup + UnProject for one keyframe; call_us = C-ABI call with host buffers"}}
    finally:
        ctx.profile(False)
    restage()

    # ---------------- pose refinement after matching (SURVEY 8f-2: Optimizer::PoseOptimization), not part of the step
    pose_opt = None
    if rank == 0:
        try:
            nf_po = min(B, 4096)
            base_po = [W.make_ba_problem(300 + i, n=N_FEATS, max_level=i % 4) for i in range(16)]
            rec = []
            for pr in base_po:
                o = np.zeros(N_FEATS, capi.BA_OBS_DT)
                o["normal"] = pr["normals"]; o["point_w"] = pr["points_w"]; o["level"] = pr["levels"]
                rec.append(o)
            obs_po = np.stack([rec[i % 16] for i in range(nf_po)])
            nobs_po = np.full(nf_po, N_FEATS, np.int32)
            poses_po = np.stack([base_po[i % 16]["pose_in"] for i in range(nf_po)])
            ctx.pose_optimize_batch(obs_po, nobs_po, poses_po)
            ctx.profile(True); ctx.profile_get(reset=True)
            for _ in range(5):
                _, _, sm_po = ctx.pose_optimize_batch(obs_po, nobs_po, poses_po, want_res=False)
            st = ctx.profile_get(reset=True)
            po_ms = st["pose_opt"][0] / max(st["pose_opt"][1], 1)
            for _ in range(5):
                ctx.pose_optimize(obs_po[0], poses_po[0])
            ctx.profile_get(reset=True)
            t0 = time.perf_counter()
            for _ in range(reps):
                _, _, s1_po = ctx.pose_optimize(obs_po[0], poses_po[0])
            po_call_us = (time.perf_counter() - t0) / reps * 1e6
            st = ctx.profile_get(reset=True)
            import oracle as O_po                                   # cpu_baseline leg: the oracle port, one thread, bounded sample
            t0 = time.perf_counter()
            for i in range(16):
                O_po.pose_optimization(base_po[i]["normals"], base_po[i]["levels"], base_po[i]["points_w"], base_po[i]["pose_in"])
            po_cpu_us = (time.perf_counter() - t0) / 16 * 1e6
            pose_opt = {"ms_per_launch": po_ms, "frames": nf_po, "observations": N_FEATS, "frames_per_s": nf_po / (po_ms * 1e-3),
                        "lm_iterations_per_frame": float(sm_po["iterations"].mean()),
                        "one_frame": {"kernel_us": st["pose_opt"][0] / max(st["pose_opt"][1], 1) * 1e3, "call_us": po_call_us,
                                      "lm_iterations": int(s1_po["iterations"])},
                        "cpu_port_us_per_frame": po_cpu_us,
                        "note": "motion-only BA over 300 matches per frame (ceres::Solve configuration of the reference restated): sweep = one warp "
                                "per frame, one frame = a CTA of eight warps; latency-bound dependent chain, not part of the step; cpu = oracle port, "
                                "1 thread, 16 frames"}
        finally:
            ctx.profile(False)

    # ---------------- end-to-end through the C-ABI with host buffers
    h, w = cam["height"], cam["width"]
    pin = capi.pinned_empty
    cur_imgs = pin((B, h, w), np.uint8)
    for i in range(B):
        cur_imgs[i] = batch["scenes"][i % batch["n_scenes"]]["cur_img"]
    hb = dict(ref_slots=pin((B,), np.int32), cur_slots=pin((B,), np.int32), feats=pin((B, FEAT_STRIDE), capi.REF_FEAT_DT),
              n_feats=pin((B,), np.int32), centers=pin((B, 3), np.float64), poses_in=pin((B, 7), np.float64),
              patches=pin((B, ppp, 100), np.uint8), patch_px=pin((B, ppp, 2), np.float64), patch_level=pin((B, ppp), np.int32))
    for k_, src in (("ref_slots", batch["ref_slots"]), ("cur_slots", batch["cur_slots"]), ("feats", batch["feats"]), ("n_feats", batch["n_feats"]),
                    ("centers", batch["centers"]), ("poses_in", batch["poses_in"]), ("patches", batch["patches"]), ("patch_px", batch["patch_px"]),
                    ("patch_level", batch["patch_level"])):
        hb[k_][...] = src
    out = dict(poses=pin((B, 7), np.float64), n_tracked=pin((B,), np.int32), px=pin((B, ppp, 2), np.float64), conv=pin((B, ppp), np.uint8))

    def e2e_step():
        ctx.pair_batch_e2e(cur_imgs, hb["ref_slots"], hb["cur_slots"], hb["feats"], FEAT_STRIDE, hb["n_feats"], hb["centers"], hb["poses_in"],
                           ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], hb["patches"], hb["patch_px"],
                           hb["patch_level"], ppp, ALIGN2D_ITERS, out)

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    if not np.array_equal(out["poses"], poses):
        raise SystemExit("bench.py: e2e results differ from the device-resident run")
    barrier()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    e2e_wall = time.perf_counter() - t1
    clocks.stop()
    clk = clocks.summary(tw0, tw1)
    clk["window"] = "device-resident timed region"
    if clk["samples"] < 3:       # short region: widen to the e2e timed region as well, and say so
        clk = clocks.summary(tw0, t1 + e2e_wall)
        clk["window"] = "device-resident + e2e timed regions"
    clk["e2e_region"] = clocks.summary(t1, t1 + e2e_wall)     # the same sampler over the e2e timed region alone
    barrier()
    t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t.item())
    h2d = int(cur_imgs.nbytes + sum(hb[k_].nbytes for k_ in hb))
    d2h = int(sum(out[k_].nbytes for k_ in out))

    # ---------------- the chain variant end to end: per pair only the cur image, the reference features and four small arrays go up
    hb["poses_ref"] = pin((B, 7), np.float64); hb["poses_ref"][...] = batch["poses_ref"]
    cout = dict(poses=pin((B, 7), np.float64), n_tracked=pin((B,), np.int32), reproj=pin((B, N_FEATS), capi.REPROJ_DT))

    def chain_e2e_step():
        ctx.track_batch_e2e(cur_imgs, hb["ref_slots"], hb["cur_slots"], hb["feats"], FEAT_STRIDE, hb["n_feats"], hb["centers"], hb["poses_ref"],
                            hb["poses_in"], ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], N_FEATS, LEVELS - 3,
                            ALIGN2D_ITERS, cout)

    for _ in range(max(args.warmup, 3)):
        chain_e2e_step()
    if cout["reproj"].tobytes() != rep.tobytes():
        raise SystemExit("bench.py: chain e2e results differ from the device-resident run")
    barrier()
    t2 = time.perf_counter()
    for _ in range(args.steps):
        chain_e2e_step()
    chain_e2e_wall = time.perf_counter() - t2
    barrier()
    tce = torch.tensor([chain_e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tce, op=dist.ReduceOp.MAX)
    chain_h2d = int(cur_imgs.nbytes + sum(hb[k_].nbytes for k_ in ("ref_slots", "cur_slots", "feats", "n_feats", "centers", "poses_in", "poses_ref")))
    chain_d2h = int(sum(cout[k_].nbytes for k_ in cout))
    refine_chain = {
        "value": world * B / (chain_ms_per_step * 1e-3), "unit": UNIT, "ms_per_step": chain_ms_per_step, "gpu_launches": int(chain_launches),
        "stages_ms_per_step": chain_stages, "converged_fraction": chain_conv,
        "e2e": {"value": world * B * args.steps / float(tce.item()), "unit": UNIT, "h2d_bytes_per_step": chain_h2d, "d2h_bytes_per_step": chain_d2h,
                "ms_per_step": float(tce.item()) * 1e3 / args.steps},
        "workload": "pyramid(cur) -> Sprase_ImgAlign(4,0,30) -> cur.Set_Pose -> ReprojectPoint + Get_ClosetObs + IsInImage gates -> SolveAffineMatrix + "
                    "GetBestSearchLevel -> WarpAffine -> Align2DGaussNewton(10) for the %d map points of the pair's reference key frame "
                    "(ref: src/Tracking.cpp:219-224,257-313; src/Feature_alignment.cpp:54-69,128-158), all on the device" % N_FEATS}

    # ---------------- CLAHE ingest stage (SURVEY 8f-4; overwrites frame slots, therefore after everything that uses them)
    if ingest is not None and rank == 0:
        try:
            ncl = min(B, 512)
            raw = cur_imgs[:ncl]
            ctx.profile(True); ctx.profile_get(reset=True)
            for _ in range(3):
                ctx.upload_clahe(0, raw, 3.0, (8, 8), fetch=False)
            st = ctx.profile_get(reset=True)
            cl_ms = st["ingest"][0] / 3.0
            cl_bytes = ncl * cam["height"] * cam["width"] * 3
            ingest["clahe"] = {"ms_per_call": cl_ms, "frames": ncl, "algorithmic_bytes": cl_bytes, "GBps": cl_bytes / (cl_ms * 1e-3) / 1e9,
                               "frac_hbm": cl_bytes / (cl_ms * 1e-3) / 1e9 / hbm_peak,
                               "note": "createCLAHE(3.0, 8x8): histogram/LUT kernel + apply kernel, two reads + one write per pixel"}
        finally:
            ctx.profile(False)

    # ---------------- CPU baseline beside it (rank 0, N = 1 only): the oracle port on a bounded sample, all host threads
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        os.sched_setaffinity(0, full_affinity)          # the CPU baseline uses every host core, not only the GPU's NUMA node
        cpu = cpu_baseline(batch, cam, sample=min(B, args.cpu_sample))
        # the checker beside the number: CPU port and CUDA path agree on the sampled pairs (tolerances of tests/)
        cp = cpu.pop("_poses")
        d = np.array([S.pose_dist(cp[i], poses[i]) for i in range(len(cp))])
        cpu["max_pose_diff_vs_gpu"] = [float(d[:, 0].max()), float(d[:, 1].max())]
        ccpu = cpu_baseline(batch, cam, sample=min(B, args.cpu_sample), chain=True)
        crep = ccpu.pop("_reproj"); ccpu.pop("_poses")
        nchk = len(crep)
        same = bool((crep["flags"] == rep[:nchk]["flags"]).all() and (crep["level"] == rep[:nchk]["level"]).all())
        okc = (crep["flags"] & capi.LM_CONVERGED) != 0
        ccpu["decisions_equal_gpu"] = same
        ccpu["max_px_diff_vs_gpu"] = float(np.abs(crep["px"][okc] - rep[:nchk]["px"][okc]).max()) if okc.any() else None
        refine_chain["cpu_baseline"] = ccpu

    ctx.close()
    strong = None
    if not args.no_strong:
        bind_to_gpu_numa(local)                         # (the CPU baseline above ran on every core)
        strong = run_strong(args, torch, dist, rank, world, local)

    if rank == 0:
        sa_gbs = sa_bytes / (sa_ms * 1e-3) / 1e9
        traffic = measured_traffic("sparse_align_kernel", B) if args.cam == "kinect" else None
        fpi = fp64_insts_per_pair("sparse_align_kernel") if args.cam == "kinect" else None
        # The dominant kernel is an fp64 Gauss-Newton chain: its pipe is the FP64 pipe, its memory side is far from the HBM roof.
        # achieved = warp instructions on the FP64 pipe (ncu smsp__inst_executed_pipe_fp64.sum of the committed capture, per pair) x 32 lanes
        # x 2 flop / measured kernel time; peak = the DFMA rate dsdtm_probe_fp64 measured on this GPU in this run.
        fp64_achieved = (fpi * B * 64.0 / (sa_ms * 1e-3) / 1e12) if fpi else None
        roofline = {"kernel": "sparse_align_kernel", "bound": "fp64", "achieved": fp64_achieved, "peak": fp64_tflops, "unit": "TFLOP/s",
                    "frac": (fp64_achieved / fp64_tflops) if fp64_achieved else None, "traffic": traffic,
                    "peak_source": "measured live: dsdtm_probe_fp64 (16 independent DFMA chains per thread, 8 CTAs of 256 threads per SM, best of 4); "
                                   "%.2f DFMA warp instructions per clock and SM at the nominal max clock" % dfma_per_clk_sm,
                    "ms_per_launch": sa_ms, "fp64_warp_insts_per_launch": (fpi * B) if fpi else None,
                    "hbm": {"achieved": sa_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": sa_gbs / hbm_peak, "traffic": traffic,
                            "algorithmic_bytes_per_launch": sa_bytes, "sector_waste": (traffic / sa_bytes) if traffic else None,
                            "peak_source": peak_src},
                    "ncu": ncu_summary("sparse_align_kernel") if args.cam == "kinect" else None,   # the committed capture is the 640x480 step
                    "note": "dependent Gauss-Newton chain on the FP64 pipe: latency/issue-bound (profiles/r2_sparse_align.md: a round of the feature "
                            "pass is a 3.4-4.5 k-cycle dependent chain at 2.9 warps per scheduler); the HBM side is reported under `hbm` (DRAM traffic "
                            "= 32-byte sectors for 5- and 7-byte window rows); see stages for the HBM-bound kernels"}
        line = {
            "metric": METRIC.replace("640x480", "%dx%d" % (cam["width"], cam["height"])), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic: %d ray-cast relief scenes tiled to %d pairs/GPU with per-pair start poses; every pair has its own frames, "
                    "features and patches in HBM" % (batch["n_scenes"], B),
            "config": make_config(args.cam, cam, B),
            "us_per_pair": ms_per_step * 1e3 / B,
            "gn_iterations_per_pair": iters,
            "latency": latency,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": float(t.item()) * 1e3 / args.steps, "timer": "host wall clock around the C-ABI call"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": roofline,
            "stages": {
                "pyramid": {"ms_per_step": pyr_ms, "GBps": pyr_bytes / (pyr_ms * 1e-3) / 1e9, "frac_hbm": pyr_bytes / (pyr_ms * 1e-3) / 1e9 / hbm_peak,
                            "algorithmic_bytes": pyr_bytes},
                "sparse_align": {"ms_per_step": sa_ms, "us_per_pair_per_sm": sa_ms * 1e3 * 148 / B},
                "align2d": {"ms_per_step": a2d_ms},
                "fast_cells": {"ms_per_launch": fast_ms, "frames": nfast, "GBps": fast_bytes / (fast_ms * 1e-3) / 1e9 if fast_ms else None,
                               "frac_hbm": fast_bytes / (fast_ms * 1e-3) / 1e9 / hbm_peak if fast_ms else None, "algorithmic_bytes": fast_bytes,
                               "note": "keyframe-only stage, not part of the step"},
                "ingest": ingest,
                "pose_opt": pose_opt},
            "cpu_baseline": cpu,
            "refine_chain": refine_chain,
            "strong_scaling": strong,
            "numa": numa,
            "prep_s": prep_s,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_strong(args, torch, dist, rank, world, local):
    """BASELINE configs[4] as written (SURVEY 8e): ONE batch of `--total-pairs` EuRoC 752x480 pairs, partitioned into contiguous blocks
    over the ranks (shard()); every rank builds the same global batch description (same seeds) and owns its block. Strong scaling:
    value = total pairs / max-over-ranks time of a step. No collective on the data path."""
    from dsdtm_b200 import capi, synth as S, workload as W
    total = args.total_pairs
    lo, hi = shard(total, world, rank)
    n = hi - lo
    cam = dict(S.EUROC)
    ctx = capi.Context(cam, levels=LEVELS, cell_size=15, max_feats=FEAT_STRIDE, max_patches=N_FEATS, max_frames=2 * n + 2, max_batch=max(n, 1), device=local)
    nsc = min(args.scenes, 8)
    scenes = W.render_scenes(nsc, cam, seed0=W.BASE_SEED + 500000, procs=max(1, min(nsc, (os.cpu_count() or 2) // (2 * world))))
    batch = W.build_batch(ctx, cam, total, n_feats=N_FEATS, feat_stride=FEAT_STRIDE, patches_per_pair=N_FEATS, seed0=W.BASE_SEED + 500000,
                          scenes=scenes, lo=lo, hi=hi)
    ppp = batch["patches_per_pair"]

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def allmax(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ctx.batch_stage(batch["ref_slots"], batch["cur_slots"], batch["feats"], batch["n_feats"], batch["centers"], batch["poses_in"],
                    ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"], batch["patch_px"],
                    batch["patch_level"], ALIGN2D_ITERS)
    for _ in range(max(args.warmup, 3)):
        ctx.batch_run(1)
    poses, nt, px, conv = ctx.batch_fetch()
    err = np.array([S.pose_dist(poses[i], batch["truth"][i]) for i in range(min(n, 64))])
    if n and not (np.median(err[:, 0]) < 5e-4 and np.median(err[:, 1]) < 1e-3):
        raise SystemExit("bench.py: strong-scaling batch did not converge to the synthetic ground truth: %s" % np.median(err, 0))
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        ctx.batch_run(1)
    ms = allmax(ctx.timer_stop()) / args.steps
    ctx.profile(True); ctx.profile_get(reset=True)
    for _ in range(args.steps):
        ctx.batch_run(1)
    st = ctx.profile_get(reset=True)
    ctx.profile(False)
    # end to end with host buffers
    h, w = cam["height"], cam["width"]
    pin = capi.pinned_empty
    cur_imgs = pin((n, h, w), np.uint8)
    k = batch["n_scenes"]
    for i in range(n):
        cur_imgs[i] = batch["scenes"][(lo + i) % k]["cur_img"]
    hb = dict(ref_slots=pin((n,), np.int32), cur_slots=pin((n,), np.int32), feats=pin((n, FEAT_STRIDE), capi.REF_FEAT_DT),
              n_feats=pin((n,), np.int32), centers=pin((n, 3), np.float64), poses_in=pin((n, 7), np.float64),
              patches=pin((n, ppp, 100), np.uint8), patch_px=pin((n, ppp, 2), np.float64), patch_level=pin((n, ppp), np.int32))
    for k_, src in (("ref_slots", batch["ref_slots"]), ("cur_slots", batch["cur_slots"]), ("feats", batch["feats"]), ("n_feats", batch["n_feats"]),
                    ("centers", batch["centers"]), ("poses_in", batch["poses_in"]), ("patches", batch["patches"]), ("patch_px", batch["patch_px"]),
                    ("patch_level", batch["patch_level"])):
        hb[k_][...] = src
    out = dict(poses=pin((n, 7), np.float64), n_tracked=pin((n,), np.int32), px=pin((n, ppp, 2), np.float64), conv=pin((n, ppp), np.uint8))

    def e2e_step():
        ctx.pair_batch_e2e(cur_imgs, hb["ref_slots"], hb["cur_slots"], hb["feats"], FEAT_STRIDE, hb["n_feats"], hb["centers"], hb["poses_in"],
                           ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], hb["patches"], hb["patch_px"],
                           hb["patch_level"], ppp, ALIGN2D_ITERS, out)

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    if not np.array_equal(out["poses"], poses):
        raise SystemExit("bench.py: strong-scaling e2e results differ from the device-resident run")
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    wall = allmax(time.perf_counter() - t0)
    barrier()
    g = ctx
    pyr_bytes = n * sum(g.ws[l - 1] * g.hs[l - 1] + g.ws[l] * g.hs[l] for l in range(1, LEVELS))
    hbm_peak, _ = peaks()
    pyr_ms = st["pyramid"][0] / args.steps
    res = {"config": "BASELINE configs[4]: %d independent 752x480 EuRoC pairs partitioned over %d GPU(s) in contiguous blocks" % (total, world),
           "scaling": "strong", "total_pairs": total, "pairs_per_gpu": n, "value": total / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
           "e2e": {"value": total * args.steps / wall, "unit": UNIT, "ms_per_step": wall * 1e3 / args.steps,
                   "h2d_bytes_per_step_per_gpu": int(cur_imgs.nbytes + sum(hb[k_].nbytes for k_ in hb)),
                   "d2h_bytes_per_step_per_gpu": int(sum(out[k_].nbytes for k_ in out))},
           "stages_ms_per_step_rank0": {"pyramid": pyr_ms, "sparse_align": st["sparse_align"][0] / args.steps, "align2d": st["align2d"][0] / args.steps},
           "pyramid_frac_hbm_rank0": (pyr_bytes / (pyr_ms * 1e-3) / 1e9 / hbm_peak) if pyr_ms > 0 else None,
           "resident_ctas_note": "%d pairs per GPU against %d resident sparse-alignment CTAs (4 per SM)" % (n, 4 * 148)}
    ctx.close()
    return res


def cpu_baseline(batch, cam, sample, threads=None, reps=1, chain=False):
    """The oracle (CPU restatement of the reference, kind 'port') on `sample` pairs of the same workload, all host threads.
    chain: the step with the reference's refinement chain (orc_pair_batch_map) instead of host patches."""
    import oracle as O
    from dsdtm_b200 import synth as S
    threads = threads or (os.cpu_count() or 1)
    oc = O.make_cam(cam["width"], cam["height"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["f"])
    k = batch["n_scenes"]
    ref_pyr = [O.pyramid(sc["ref_img"], LEVELS)[0] for sc in batch["scenes"]]
    pyr_bytes = len(ref_pyr[0])
    n = sample
    ref_pyrs = np.empty((n, pyr_bytes), np.uint8)
    cur_imgs = np.empty((n, cam["height"], cam["width"]), np.uint8)
    lo = batch.get("lo", 0)
    for i in range(n):
        ref_pyrs[i] = ref_pyr[(lo + i) % k]
        cur_imgs[i] = batch["scenes"][(lo + i) % k]["cur_img"]
    feats = batch["feats"][:n].astype(O.REF_FEAT_DT)
    if chain:
        args = (oc, LEVELS, 15, ref_pyrs, cur_imgs, feats, batch["n_feats"][:n], batch["centers"][:n], batch["poses_ref"][:n], batch["poses_in"][:n],
                ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], N_FEATS, LEVELS - 3, ALIGN2D_ITERS, threads)
        fn = O.pair_batch_map
        what = "pyramid(cur)+sparse align+reproject/affine/warp/align2d of %d map points" % N_FEATS
    else:
        args = (oc, LEVELS, ref_pyrs, cur_imgs, feats, batch["n_feats"][:n], batch["centers"][:n], batch["poses_in"][:n],
                ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"][:n], batch["patch_px"][:n],
                batch["patch_level"][:n], ALIGN2D_ITERS, threads)
        fn = O.pair_batch
        what = "pyramid(cur)+sparse align+align2d"
    fn(*args)     # warm-up (page in, thread start)
    t0 = time.perf_counter()
    for _ in range(reps):
        res = fn(*args)
    dt = (time.perf_counter() - t0) / reps
    out = {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
           "sample": "%d pairs of the same workload (%s), %d std::threads, %.2f s" % (n, what, threads, dt),
           "us_per_pair_per_core": dt / n * threads * 1e6, "_poses": res[0]}
    if chain:
        out["_reproj"] = res[2]
    return out


def host_batch_with_oracle_detector(cam, scenes, n_pairs, seed0):
    """The SAME batch the GPU arm stages (dsdtm_b200.workload: same scenes, same selection code, same per-pair start poses, centres and
    patches), with the per-cell corner records coming from the oracle's detector instead of dsdtm_fast_cells -- the two are bit-equal
    (tests/test_gpu_pyramid_fast.py, tests/test_ref_pin.py), so the reference arm needs no GPU to build the GPU arm's inputs."""
    import oracle as O
    from dsdtm_b200 import workload as W
    per_scene = []
    for sc in scenes:
        packed, offs, ws, hs = O.pyramid(sc["ref_img"], LEVELS)
        oc = O.detect_cells(packed, offs, ws, hs, 15, None, 5.0)
        cells = np.zeros(len(oc), W.CORNER_DT)
        for f in ("x", "y", "level", "score"):
            cells[f] = oc[f]
        per_scene.append(W.scene_inputs(sc, cam, cells, 15, N_FEATS, FEAT_STRIDE, N_FEATS))
    return W.assemble_batch(scenes, per_scene, n_pairs, FEAT_STRIDE, N_FEATS, seed0)


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port) on the box's host cores, same config / metric / unit."""
    rank, world, local = dist_setup(args.gpus)
    if rank != 0:
        return
    from dsdtm_b200 import synth as S, workload as W
    import oracle as O
    cam = dict(S.EUROC if args.cam == "euroc" else S.KINECT)
    threads = os.cpu_count() or 1
    sample = args.cpu_sample
    # the GPU arm's own batch (same scenes, features, start poses, centres, patches: host_batch_with_oracle_detector), bounded to the
    # first `sample` pairs per step
    scenes = W.render_scenes(args.scenes, cam, seed0=W.BASE_SEED)
    batch = host_batch_with_oracle_detector(cam, scenes, args.pairs, W.BASE_SEED)
    k = len(scenes)
    ref_pyr = [O.pyramid(sc["ref_img"], LEVELS)[0] for sc in scenes]
    ref_pyrs = np.empty((sample, len(ref_pyr[0])), np.uint8); cur_imgs = np.empty((sample, cam["height"], cam["width"]), np.uint8)
    for i in range(sample):
        ref_pyrs[i] = ref_pyr[i % k]; cur_imgs[i] = scenes[i % k]["cur_img"]
    oc = O.make_cam(cam["width"], cam["height"], cam["fx"], cam["fy"], cam["cx"], cam["cy"], cam["f"])
    a = (oc, LEVELS, ref_pyrs, cur_imgs, batch["feats"][:sample].astype(O.REF_FEAT_DT), batch["n_feats"][:sample], batch["centers"][:sample],
         batch["poses_in"][:sample], ALIGN_CFG["max_level"], ALIGN_CFG["min_level"], ALIGN_CFG["max_iters"], batch["patches"][:sample],
         batch["patch_px"][:sample], batch["patch_level"][:sample], ALIGN2D_ITERS, threads)
    for _ in range(max(args.warmup, 1)):
        O.pair_batch(*a)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = O.pair_batch(*a)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res)
    value = sample * args.steps / dt
    line = {"impl": "reference", "metric": METRIC.replace("640x480", "%dx%d" % (cam["width"], cam["height"])), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 1),
            "ms_per_step": dt * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic: %d ray-cast relief scenes tiled to %d pairs (the GPU arm's batch); each CPU step runs the first %d of them (bounded sample)" % (k, args.pairs, sample),
            "config": make_config(args.cam, cam, args.pairs),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "%d pairs per step, %d std::threads (the reference needs OpenCV/Eigen/Sophus/Ceres: not buildable here; "
                                       "oracle/ restates it line by line)" % (sample, threads)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=4096, help="frame pairs per GPU per step")
    ap.add_argument("--scenes", type=int, default=16, help="distinct ray-cast scenes (tiled to --pairs)")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="pairs in the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--total-pairs", type=int, default=4096, help="strong-scaling extra (configs[4]): EuRoC pairs partitioned over the ranks")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling extra")
    ap.add_argument("--cam", default="kinect", choices=["kinect", "euroc"],
                    help="kinect = 640x480 (the metric's configuration, default); euroc = 752x480, BASELINE configs[4]'s sweep geometry")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's outputs of its last step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
