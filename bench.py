#!/usr/bin/env python
"""bench.py -- 4K frames/s of the marker pipeline (undistort + gamma -> detectMarkers(APRILTAG) -> pose -> vehicle distances).

    python bench.py --gpus N --steps K --warmup W          # our arm (one rank per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N ...          # reference arm: cv2 on the host cores, rank 0 only
    python bench.py --workload preprocess64|dense-apriltag|dense-classic   # BASELINE.json configs[1] / configs[4]

Default workload = BASELINE.json configs[2] (N = 1) / configs[3] (N > 1): ONE STEP = THE WHOLE 1800-frame synthetic
3840x2160 sequence, resident in HBM (44.8 GB), through the public sequence API (shard.run_sequence):
    batched GPU pipeline (undistort + gamma + gray -> detectMarkers -> estimatePoseSingleMarkers) per rank
    -> per-frame results gathered on rank 0 -> native sequence post-pass (marker-length recurrence, gating, second exact
    pose pass, vehicle distances) -> the CSV text of aruco_detect.py:146-185, to its last row.
For N > 1 the SAME sequence is frame-sharded: strong scaling, the gather and the post-pass on rank 0 are inside the timed
region, no collective on the pipeline's streams: contiguous blocks (shard.shard_bounds), one gather and one post-pass at the end.
--stream: the frames are dealt out in rounds (shard.round_plan; round k = N consecutive batches, one per rank) and the post-pass is
STREAMED (shard.run_sequence_streamed): the results of round k travel to rank 0 on a side stream and are post-processed there
(worker thread) while all ranks compute round k + 1.  Built for sequences that arrive over time; for a resident sequence it was
measured and is slower than the plain run (1 GPU: 54.2 against 54.0 ms per 1800 frames; 8 GPUs: 12.7 against 10.3 ms).
Timed region: barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks.
`value`        : frames resident in HBM -> last CSV row (every step streams 44.8 GB, far beyond the 126 MB L2).
`pipeline_only`: the same frames through the GPU pipeline alone (no gather / post-pass): what `roofline` explains.
`e2e`          : frames in pinned HOST memory: H2D of every batch, pipeline, post-pass, CSV inside the timed region.
`roofline`     : dominant kernel by device time (per-kernel CUDA events recorded inside libapse_b200 on the launching
                 stream), algorithmic bytes per launch from SURVEY.md 8(d) / DESIGN.md, peak from MEASURED_PEAKS.json.
`cpu_baseline` : the reference's own cv2 call chain (aruco_detect.py:250-269,592-601) on the host cores, bounded sample,
                 1 thread and all threads, median and best per frame (BASELINE.md section 3).
--dump-outputs DIR: what the last timed step returned to its caller (rank 0), one DIR/<name>.npy per array (dump_outputs).
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

W, H = 3840, 2160
FRAME_BYTES = W * H * 3
SEQUENCE_FRAMES = 1800            # BASELINE.json configs[2], configs[3]
# algorithmic bytes per 4K frame (SURVEY.md 8(d), restated in DESIGN.md); keys = kernel ids of libapse_b200
ALG_BYTES = {
    "k_preprocess_fused": 33_177_600,   # read BGR 24 883 200 + write gray 8 294 400
    "k_preprocess_bgr": 58_060_800,     # configs[1]: additionally writes the corrected BGR frame
    "k_tile_minmax": 8_294_400,          # read gray (tile arrays negligible)
    "k_threshold": 16_588_800,           # read gray + write ternary
    "k_ccl_local": 41_472_000,           # read ternary + write labels (u32)
    "k_ccl_merge": 0, "k_ccl_flatten": 41_472_000, "k_emit_points": 41_472_000,
    "k_adaptive_threshold": 16_588_800,  # per window: read gray + write binary
    "pipeline": 132_710_400,
    "classic_window": 91_238_400,        # per threshold window of the classic path (SURVEY.md 8(d))
}
# the library times its launches per kernel ID; what the IDs that can dominate stand for
KERNEL_NOTES = {
    "k_preprocess_fused": "kernel id of the preprocess launches: k_preprocess_tma<MODE 1> (bounds pass of the sparse evaluation: every pixel "
                          "remapped through TMA-staged tiles and bounded) when no gray output is asked for, k_preprocess_tma<MODE 0> "
                          "(dense colour chain) otherwise",
    "k_sparse_exact": "exact colour chain on the tiles the bounds pass could not rule out",
}
METRIC = "4K frames/s (undistort+ArUco detect+pose)"
DUMP_BYTES = 64_000_000           # --dump-outputs: at most this much in all


def load_camera():
    cam = json.load(open(os.path.join(ROOT, "tests", "golden", "cam_params.json")))
    return np.array(cam["mtx"]), np.array(cam["dist"]).ravel()


def dictionary():
    from apse_uav_b200 import aruco
    return aruco.getPredefinedDictionary(aruco.DICT_4X4_50)


def base_frames(n, seed=1000):
    """n distinct sparse frames (ids 1,2,3 vehicles + 4 host), seeded; host numpy uint8 [n,H,W,3]."""
    from tools import synth
    d = dictionary()
    return np.stack([synth.make_frame(d.bytesList, seed + i, W, H, ids=(1, 2, 3, 4), side_range=(50, 90)) for i in range(n)])


def base_sequence(n, seed=2000):
    """n consecutive frames of a slowly drifting sparse sequence (tools.synth.make_sequence): the track gating of
    aruco_detect.py:613 passes from frame to frame, so the distance stage has work in every frame."""
    from tools import synth
    return np.stack(list(synth.make_sequence(dictionary().bytesList, seed, n)))


def dense_frames(n, seed=77):
    from tools import synth
    d = dictionary()
    return np.stack([synth.make_dense_frame(d.bytesList, seed + i, W, H) for i in range(n)])


def sequence_plan(n_frames, n_base):
    """Frame k of the synthetic sequence = base frame p(k) (ping-pong through the rendered drift sequence, so consecutive
    frames stay consecutive) cyclically translated by a slow Lissajous walk (dy, dx): every frame has different pixels, the
    markers move a few pixels per frame.  The same plan on every rank: the sequence does not depend on the world size."""
    period = max(1, 2 * n_base - 2)
    plan = []
    for k in range(n_frames):
        p = k % period
        p = p if p < n_base else period - p
        dx = int(round(90 * np.sin(2 * np.pi * k / 611.0)))
        dy = int(round(60 * np.sin(2 * np.pi * k / 419.0)))
        plan.append((p, dy, dx))
    return plan


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons DURING the timed region, read in-process through NVML (nvidia-ml-py); spawning
    nvidia-smi inside the timed region stalls CUDA launches, so it is only the fallback for a single sample."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.nv, self.handle = index, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _reasons(self):
        nv = self.nv
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        out = []
        for name, attr in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            bit = getattr(nv, attr, None)
            if bit is not None and mask & bit:
                out.append(name)
        return out

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            try:
                self.samples.append((float(self.nv.nvmlDeviceGetClockInfo(self.handle, self.nv.NVML_CLOCK_SM)), self._reasons()))
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": "nvml unavailable"}
        sm = [s[0] for s in self.samples]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": self.max_sm, "reasons": sorted({r for s in self.samples for r in s[1]}),
                "samples": len(sm), "source": "nvml, 50 ms period, during the timed region"}


# ---------------------------------------------------------------------------------------------------------------
class CpuReference:
    """The reference's cv2 call chain (aruco_detect.py:250-269,592-601 through the 4.13 compat shim)."""

    def __init__(self, threads, frames, classic=None):
        import cv2
        from oracle import cv2_compat as C
        self.cv2, self.C, self.threads = cv2, C, threads
        self.K, self.D = load_camera()
        cv2.setNumThreads(threads)
        self.mapx, self.mapy = cv2.initUndistortRectifyMap(self.K, self.D, None, self.K, (W, H), 5)
        self.lut, self.params = C.gamma_lut(), C.reference_parameters()
        if classic is not None:   # configs[4]: the classic candidate path with one threshold-window sweep
            self.params.cornerRefinementMethod = 0
            self.params.adaptiveThreshWinSizeMin, self.params.adaptiveThreshWinSizeMax, self.params.adaptiveThreshWinSizeStep = classic
        self.frames = frames
        self.markers = 0
        self.run(1)  # warm-up

    def run(self, n, times=None):
        for i in range(n):
            t0 = time.perf_counter()
            r = self.C.reference_chain(self.frames[i % len(self.frames)], self.mapx, self.mapy, self.lut, self.params,
                                       self.K, self.D)
            if times is not None:
                times.append(time.perf_counter() - t0)
            self.markers += 0 if r["ids"] is None else len(r["ids"])

    def info(self, n):
        return {"kind": "reference", "cores": self.threads,
                "sample": f"{n} synthetic 4K frames through cv2 {self.cv2.__version__} (remap+RGB2LAB+LUT+LAB2RGB+BGR2GRAY+"
                          f"ArucoDetector+solvePnP per marker), cv2.setNumThreads({self.threads})"}


def cpu_baseline(frames, n_frames, classic=None):
    """BASELINE.md section 3: the reference chain with 1 thread and with all host threads, 3 warm-up + n timed frames each,
    median and best per frame.  `value` = frames/s of the all-thread run over its whole sample."""
    all_threads = os.cpu_count() or 1
    out = {"unit": "frames/s", "kind": "reference"}
    try:
        for label, threads, n in (("one_thread", 1, max(4, n_frames // 3)), ("all_threads", all_threads, n_frames)):
            ref = CpuReference(threads, frames, classic)
            ref.run(3)
            times = []
            t0 = time.perf_counter()
            ref.run(n, times)
            dt = time.perf_counter() - t0
            out[label] = {"threads": threads, "frames": n, "frames_per_s": n / dt, "median_ms_per_frame": 1e3 * float(np.median(times)),
                          "best_ms_per_frame": 1e3 * float(np.min(times))}
            info = ref.info(n)
        out.update(value=out["all_threads"]["frames_per_s"], cores=all_threads,
                   sample=info["sample"] + f"; plus {out['one_thread']['frames']} frames with 1 thread")
    except ImportError:
        fps, info = port_fps(max(2, n_frames // 8), frames)
        out.update(value=fps, cores=info["cores"], kind=info["kind"], sample=info["sample"])
    return out


def port_fps(n_frames, frames):
    from oracle import oracle as O
    from apse_uav_b200 import aruco
    import __graft_entry__ as G
    K, D = load_camera()
    d = dictionary()
    p = G.reference_parameters(aruco)
    lut = G.gamma_lut()
    mx, my = O.init_undistort_map(K, D, W, H)
    t0 = time.perf_counter()
    for i in range(n_frames):
        _, gray = O.preprocess(frames[i % len(frames)], mx, my, lut)
        c, ids, _ = O.detect_markers_apriltag(gray, d.raw, p)
        O.estimate_pose_single_markers(c, 0.55, K, D)
    dt = time.perf_counter() - t0
    return n_frames / dt, {"kind": "port", "cores": 1, "sample": f"{n_frames} synthetic 4K frames through the C oracle (1 thread)"}


def workload_config(args, frames_per_step, world):
    if args.workload == "sequence":
        return {"workload": "configs[2] (1 GPU) / configs[3] (frame-sharded): full pipeline undistort+gamma -> detectMarkers("
                            "CORNER_REFINE_APRILTAG, DICT_4X4_50, parameters of aruco_detect.py:190-203) -> "
                            "estimatePoseSingleMarkers -> marker-length recurrence + vehicle distances -> CSV rows, on a synthetic "
                            "3840x2160 sequence (ids 1-4, sigma-3 noise, slow drift)",
                "frames_per_step": frames_per_step, "frame": [W, H, 3], "sequence_frames": args.sequence_frames,
                "step": "one step = the whole sequence, first enqueue to last CSV row",
                "l2": "every step streams the whole HBM-resident sequence (44.8 GB at 1800 frames; L2 is 126 MB)",
                "batch": args.batch, "streams_per_gpu": args.streams,
                "parallelism": (f"same sequence frame-sharded x{world} in rounds of {world} batches (round-robin), no collective on the "
                                "pipeline's streams; per-round results sent to rank 0 on a side stream, sequential post-pass streamed "
                                "behind the pipeline" if args.stream else
                                f"same sequence frame-sharded x{world} (contiguous blocks), no collective on the hot path; "
                                "per-frame results gathered on rank 0 for the sequential post-pass")}
    if args.workload == "preprocess64":
        return {"workload": "configs[1]: undistort (cam_params.json) + gamma correction (+ gray) on a batch of 64 synthetic 4K frames, "
                            "corrected BGR and gray written", "frames_per_step": frames_per_step, "frame": [W, H, 3],
                "l2": "each step reads 1.59 GB and writes 2.12 GB (L2 is 126 MB)", "parallelism": f"independent batches x{world}"}
    return {"workload": f"configs[4] ({args.workload}): dense stress frames (~200 rotated / perspective / partially occluded markers, "
                        "sigma-4 noise), " + ("APRILTAG candidate path" if args.workload == "dense-apriltag" else
                                              "classic candidate path, adaptiveThreshWinSize sweep " + str(args.classic_windows)),
            "frames_per_step": frames_per_step, "frame": [W, H, 3],
            "l2": "each step reads frames_per_step x 24.9 MB of distinct frames (>= 0.4 GB; L2 is 126 MB)",
            "parallelism": f"independent batches x{world}"}


def run_reference(args, rank):
    """Reference arm: the reference's own cv2 chain on the host cores (rank 0 only), each step a bounded sample of the workload."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    per_step = max(1, args.ref_frames_per_step)
    classic = None
    if args.workload == "dense-classic":
        classic = tuple(args.classic_windows)
    frames = dense_frames(min(4, per_step)) if args.workload.startswith("dense") else base_sequence(min(4, per_step))
    try:
        ref = CpuReference(threads, frames, classic)
        if args.workload == "dense-apriltag":
            pass
        runner, info = ref.run, ref.info(args.steps * per_step)
    except ImportError:
        runner, info = (lambda n: port_fps(n, frames)), {"kind": "port", "cores": 1, "sample": "C oracle, 1 thread"}
    for _ in range(args.warmup):
        runner(per_step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        runner(per_step)
    dt = time.perf_counter() - t0
    fps = args.steps * per_step / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.workload == "sequence" else "weak", "vs_baseline": None,
            "dtype": "u8/f64", "data": "synthetic",
            "config": workload_config(args, per_step, args.gpus),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": info["cores"], "kind": info["kind"],
                             "sample": f"{args.steps} steps x {per_step} frames (bounded sample of the workload; per-frame metric; the reference's "
                                       "distance stage, < 1 ms of Python per frame, is left out in its favour); " + info["sample"]},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def latest_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per frame of the latest `ncu --set full` capture of this kernel"""
    try:
        import glob
        tfile = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))[-1]
        tj = json.load(open(tfile))
        if kernel in tj:
            return tj[kernel]["dram_bytes_per_frame"], f"profiles/{os.path.basename(tfile)} (ncu --set full capture, bytes per frame x frames per launch)"
    except Exception:
        pass
    return None, None


def roofline_of(ktimes, frames_timed, alg_override=None):
    """Dominant kernel by accumulated device time of the per-kernel timing pass."""
    peak, peak_src = peaks()
    if not ktimes:
        return {"kernel": "none", "bound": "hbm", "achieved": 0.0, "peak": peak, "unit": "GB/s", "frac": 0.0, "traffic": None}
    name, (kms, kcount) = max(ktimes.items(), key=lambda kv: kv[1][0])
    frames_per_launch = frames_timed / max(kcount, 1)
    per_frame = (alg_override or {}).get(name, ALG_BYTES.get(name, ALG_BYTES["pipeline"]))
    alg = per_frame * frames_per_launch
    achieved = alg / (kms / max(kcount, 1) / 1e3) / 1e9 if kms > 0 else 0.0
    ksum = sum(v[0] for v in ktimes.values())
    tpf, tsrc = latest_traffic(name)
    return {"kernel": name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": None if tpf is None else tpf * frames_per_launch, "peak_source": peak_src, "traffic_source": tsrc,
            "share_of_kernel_time": kms / ksum if ksum else None, "algorithmic_bytes_per_frame": per_frame,
            "algorithmic_bytes_per_launch": alg, "frames_per_launch": frames_per_launch, "launches": kcount,
            "avg_ms": kms / max(kcount, 1),
            "kernel_note": KERNEL_NOTES.get(name)}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes every array of `arrays` (name -> numpy array or torch tensor) as out_dir/<name>.npy.  Integers of
    up to 16 bits and float32 are written as float32, everything else as float64 (exact either way).  An array larger than
    its equal share of DUMP_BYTES is flattened and written at a fixed sample of its indices (seed 0, sorted), the same sample
    in every run with the same arguments."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 128                  # 128: the .npy header
    for name, a in arrays.items():
        t = torch.from_numpy(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a
        dtype = torch.float32 if t.element_size() <= 2 or t.dtype == torch.float32 else torch.float64
        cap = share // (4 if dtype == torch.float32 else 8)
        if t.numel() > cap:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), cap))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.to(dtype).cpu().numpy())


def collect_ktimes(engines):
    ktimes = {}
    for e in engines:
        for k, (kms_, kc_) in e.timing_collect(reset=True).items():
            a_, b_ = ktimes.get(k, (0.0, 0))
            ktimes[k] = (a_ + kms_, b_ + kc_)
    return ktimes


class Ctx:
    """Per-rank plumbing shared by the workloads."""

    def __init__(self, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        self.torch, self.dist, self.args, self.rank, self.world, self.local_rank = torch, dist, args, rank, world, local_rank
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        """barrier | e0 | fn(i) for i in range(steps) | e1 | barrier -> milliseconds between the events (this rank)"""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        e1.synchronize()
        wall = 1e3 * (time.perf_counter() - t0)
        self.barrier()
        return e0.elapsed_time(e1), wall

    def reduce(self, values, op="max"):
        torch = self.torch
        t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(v) for v in t]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def make_pipeline(args, local_rank, params=None, max_batch=None, max_markers=None):
    import apse_uav_b200 as A
    from apse_uav_b200 import aruco
    import __graft_entry__ as G
    K, D = load_camera()
    p = params if params is not None else G.reference_parameters(aruco)
    return A.Pipeline(K, D, (W, H), G.gamma_lut(), dictionary(), p, max_batch=max_batch or args.batch, device=local_rank,
                      max_markers=max_markers or args.max_markers, streams=args.streams, ring=4)


# ---------------------------------------------------------------------------------------------------------------
def run_sequence_workload(args, rank, world, local_rank):
    from apse_uav_b200 import shard, sequence
    c = Ctx(args, rank, world, local_rank)
    torch = c.torch
    dev = c.dev
    pipe = make_pipeline(args, local_rank)
    n_seq = args.sequence_frames
    # ---- this rank's frames of the synthetic sequence, resident in HBM.  Streamed run (default for N > 1): the sequence is dealt out in
    # rounds (shard.round_plan: round k = world consecutive batches, rank r takes the r-th), so that rank 0 runs the sequential
    # post-pass of round k while all ranks compute round k + 1; --no-stream: contiguous blocks, post-pass after the gather
    if args.stream:
        rounds = shard.round_plan(n_seq, world, args.batch, tail=args.tail_frames)
        local_idx = [g for rnd in rounds for g in range(*rnd[rank])]
    else:
        rounds = None
        local_idx = list(range(*shard.shard_bounds(n_seq, world)[rank]))
    n_local = len(local_idx)
    base = torch.from_numpy(base_sequence(args.base_frames)).to(dev)
    plan = sequence_plan(n_seq, args.base_frames)
    frames = torch.empty((n_local, H, W, 3), dtype=torch.uint8, device=dev)
    for j, g in enumerate(local_idx):
        p, dy, dx = plan[g]
        frames[j] = torch.roll(base[p], shifts=(dy, dx), dims=(0, 1))
    torch.cuda.synchronize()
    state = {}

    def step(_i):
        if args.stream:
            rows = shard.run_sequence_streamed(pipe, frames, rounds, rank, world, as_rows=True)
        else:
            rows = shard.run_sequence(pipe, frames, rank, world, as_rows=True)
        if rank == 0:
            state["rows"] = rows
            state["csv"] = sequence.rows_to_csv(rows)          # the text aruco_detect.py:131-185 writes, to its last row

    def step_pipeline(_i):
        state["det"] = pipe.run_sequence(frames)

    for i in range(args.warmup):
        step(i)
    sampler = ClockSampler(local_rank)
    if not os.environ.get("APSE_BENCH_NOSAMPLER"):
        sampler.start()
    l0 = pipe.launches
    ms, wall_ms = c.timed(step, args.steps)
    launches = pipe.launches - l0
    sampler.stop_flag = True
    if rank == 0 and args.dump_outputs:   # the CSV row fields (the CSV text is rendered from them)
        dump_outputs(args.dump_outputs, {f: state["rows"][f] for f in state["rows"].dtype.names})
    # ---- the GPU pipeline alone on the same frames (no gather, no post-pass)
    step_pipeline(0)
    ms_pipe, _ = c.timed(step_pipeline, args.steps)
    markers = int(state["det"]["n"].sum().item())
    # ---- post-pass alone (rank 0; everything after the pipeline of a one-GPU run), for the split in the report
    post_ms = None
    stream_check = None
    if world == 1:
        if args.stream:   # the streamed rows are the rows of the plain run (gather at the end, one post-pass)
            stream_check = bool(sequence.rows_to_csv(shard.run_sequence(pipe, frames, 0, 1, as_rows=True)) == state["csv"])
        det = state["det"]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            sequence.rows_to_csv(sequence.postpass_device(pipe.engine, det))
        post_ms = 1e3 * (time.perf_counter() - t0) / 3

    # ---- per-kernel pass: one batch at a time on ONE stream with every launch bracketed by CUDA events inside the library
    # (apse_timing_*), so that a kernel's event pair measures that kernel alone (in the passes above kernels of different
    # streams share the SMs and their durations overlap)
    n_kt = min(n_local, args.batch * max(1, min(args.kernel_batches, n_local // max(1, args.batch))))
    for e in pipe.engines:
        e.timing(True)
    pipe.run_batch(frames[:min(args.batch, n_local)], serial=True)
    collect_ktimes(pipe.engines)

    def step_kt(_i):
        for b in range(0, n_kt, args.batch):
            pipe.run_batch(frames[b:b + args.batch], serial=True)
    ms_instrumented, _ = c.timed(step_kt, 1)
    ktimes = collect_ktimes(pipe.engines)
    for e in pipe.engines:
        e.timing(False)

    # ---- e2e: the sequence in pinned HOST memory -> H2D per batch -> pipeline -> post-pass -> CSV, all inside the timed region.
    # A ring of pinned batches holds the first frames of this rank's block and is reused cyclically (pinning the whole
    # 44.8 GB sequence would not leave the host usable); every batch is copied H2D again in every step.
    n_ring = max(1, min(args.host_ring, (n_local + args.batch - 1) // args.batch))
    host = [torch.empty((args.batch, H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(n_ring)]
    for j in range(n_ring):
        b = min(args.batch, n_local - j * args.batch)
        host[j][:b].copy_(frames[j * args.batch:j * args.batch + b])
        if b < args.batch:
            host[j][b:].copy_(frames[:args.batch - b])
    n_e2e = n_local if args.e2e_frames <= 0 else min(n_local, max(args.batch, args.e2e_frames // world))

    def host_batches():
        left, k = n_e2e, 0
        while left > 0:
            b = min(args.batch, left)
            yield host[k % n_ring][:b]
            left -= b
            k += 1

    def step_e2e(_i):
        rows = shard.run_sequence_host(pipe, host_batches(), n_e2e, rank, world, as_rows=True)
        if rank == 0:
            state["csv_e2e"] = sequence.rows_to_csv(rows)

    step_e2e(0)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_ms, _ = c.timed(step_e2e, e2e_steps)
    d2h = n_e2e * (4 + 4 + args.max_markers * (4 + 32 + 24 + 24))    # n, status, ids, corners, rvec, tvec per frame

    ms, ms_pipe, e2e_ms = c.reduce([ms, ms_pipe, e2e_ms], "max")
    launches, markers = (int(v) for v in c.reduce([launches, markers], "sum"))
    if rank == 0:
        peak, _ = peaks()
        value = args.steps * n_seq / (ms / 1e3)
        pipe_value = args.steps * n_seq / (ms_pipe / 1e3)
        e2e_value = e2e_steps * n_e2e * world / (e2e_ms / 1e3)
        csv_lines = state["csv"].count("\n")
        rows = state["rows"]
        roof = roofline_of(ktimes, n_kt)
        roof["bound_note"] = ("HBM is the roofline SURVEY.md 8(d) prescribes; see profiles/ for what limits the kernel itself")
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8/i32 pixels, f64 line fits and pose", "data": "synthetic",
            "config": workload_config(args, n_seq, world),
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": n_e2e * world * FRAME_BYTES,
                    "d2h_bytes_per_step": int(d2h * world), "steps": e2e_steps, "frames_per_step": n_e2e * world,
                    "note": "pinned host frames -> H2D per batch (copy stream, double-buffered) -> pipeline -> gather -> post-pass -> CSV text"},
            "gpu_launches": int(launches),
            "markers_found": markers,
            "csv": {"rows": int(len(rows)), "lines": int(csv_lines), "bytes": len(state["csv"]),
                    "frames_with_host_marker": int((rows["detected"][:, 3] == 1).sum()),
                    "distance_values": int((rows["detected"][:, :3] == 1).sum())},
            "wall_ms_per_step": wall_ms / args.steps,
            "pipeline_only": {"value": pipe_value, "unit": "frames/s", "ms_per_step": ms_pipe / args.steps,
                              "note": "GPU pipeline alone (undistort+gamma+gray -> detect -> pose), no gather / post-pass / CSV"},
            "postpass_ms_per_step": post_ms,
            "postpass": ({"mode": "streamed", "rounds": len(rounds), "frames_in_last_round": sum(b - a for a, b in rounds[-1]) if rounds else 0,
                          "equals_unstreamed_csv": stream_check,
                          "note": "post-pass of round k on rank 0 while all ranks compute round k+1 (shard.run_sequence_streamed); "
                                  "postpass_ms_per_step = the same post-pass run in one piece after the pipeline"}
                         if args.stream else {"mode": "after the gather"}),
            "pipeline_roofline": {"algorithmic_bytes_per_frame": ALG_BYTES["pipeline"],
                                  "achieved_gbs_per_gpu": ALG_BYTES["pipeline"] * pipe_value / world / 1e9,
                                  "frac_of_hbm_peak": ALG_BYTES["pipeline"] * pipe_value / world / 1e9 / peak,
                                  "whole_step_frac_of_hbm_peak": ALG_BYTES["pipeline"] * value / world / 1e9 / peak},
            "roofline": roof,
            "kernel_ms_per_frame": {k: v[0] / n_kt for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0])},
            "kernel_timing_pass": {"frames": n_kt, "ms": ms_instrumented,
                                   "note": "batches repeated on one stream (sub-batches serialised) with a CUDA event pair "
                                           "around every launch; the headline passes overlap sub-batches on several streams"},
            "clocks": sampler.summary(),
        }
        if world == 1 and args.cpu_frames > 0:
            line["cpu_baseline"] = cpu_baseline(base_sequence(4), args.cpu_frames)
        print(json.dumps(line), flush=True)
    c.close()


# ---------------------------------------------------------------------------------------------------------------
def run_preprocess_workload(args, rank, world, local_rank):
    """configs[1]: undistort + gamma correction of a batch of 64 frames, corrected BGR + gray written."""
    c = Ctx(args, rank, world, local_rank)
    torch, dev = c.torch, c.dev
    from apse_uav_b200.engine import Engine
    import __graft_entry__ as G
    K, D = load_camera()
    B = 64
    e = Engine(local_rank, W, H, B)
    e.set_camera(K, D, W, H)
    e.set_lut(G.gamma_lut())
    base = torch.from_numpy(base_frames(args.base_frames, seed=1000 + 97 * rank)).to(dev)
    n_slices = 3
    seq = torch.empty((n_slices, B, H, W, 3), dtype=torch.uint8, device=dev)
    g = torch.Generator().manual_seed(7 + rank)
    for s in range(n_slices):
        for j in range(B):
            dx, dy = (int(v) for v in torch.randint(-40, 41, (2,), generator=g))
            seq[s, j] = torch.roll(base[(s * B + j) % len(base)], shifts=(dy, dx), dims=(0, 1))
    out = {}

    def step(i):
        out["bgr"], out["gray"] = e.preprocess(seq[i % n_slices], want_bgr=True)

    for i in range(args.warmup):
        step(i)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = e.launches
    ms, _ = c.timed(step, args.steps)
    launches = e.launches - l0
    sampler.stop_flag = True
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    e.timing(True)
    step(0)
    e.timing_collect(reset=True)
    c.timed(step, args.steps)
    ktimes = collect_ktimes([e])
    e.timing(False)
    # e2e: pinned host batch in, corrected frames + gray back to the host
    hin = torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory()
    hin.copy_(seq[0])
    hout = torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory()
    hgray = torch.empty((B, H, W), dtype=torch.uint8).pin_memory()
    stage = torch.empty_like(seq[0])

    def step_e2e(_i):
        stage.copy_(hin, non_blocking=True)
        b, gr = e.preprocess(stage, want_bgr=True)
        hout.copy_(b, non_blocking=True)
        hgray.copy_(gr, non_blocking=True)

    step_e2e(0)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_ms, _ = c.timed(step_e2e, e2e_steps)
    ms, e2e_ms = c.reduce([ms, e2e_ms], "max")
    launches, = (int(v) for v in c.reduce([launches], "sum"))
    if rank == 0:
        value = args.steps * B * world / (ms / 1e3)
        roof = roofline_of(ktimes, args.steps * B, {"k_preprocess_fused": ALG_BYTES["k_preprocess_bgr"]})
        line = {"metric": "4K frames/s (undistort+gamma correction)", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8 pixels, Q5/Q15 fixed point", "data": "synthetic", "config": workload_config(args, B, world),
                "e2e": {"value": e2e_steps * B * world / (e2e_ms / 1e3), "unit": "frames/s", "h2d_bytes_per_step": B * FRAME_BYTES,
                        "d2h_bytes_per_step": B * (FRAME_BYTES + W * H), "steps": e2e_steps},
                "gpu_launches": launches, "roofline": roof, "clocks": sampler.summary()}
        if world == 1 and args.cpu_frames > 0:
            line["cpu_baseline"] = cpu_preprocess_baseline(base_frames(2), max(4, args.cpu_frames // 2))
        print(json.dumps(line), flush=True)
    c.close()


def cpu_preprocess_baseline(frames, n):
    """aruco_detect.py:250-259,592 on the host cores (cv2): remap + RGB2LAB + LUT + LAB2RGB + BGR2GRAY."""
    try:
        import cv2
        from oracle import cv2_compat as C
    except ImportError:
        return {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "cv2 unavailable"}
    K, D = load_camera()
    threads = os.cpu_count() or 1
    cv2.setNumThreads(threads)
    mapx, mapy = cv2.initUndistortRectifyMap(K, D, None, K, (W, H), 5)
    lut = C.gamma_lut()

    def one(f):
        f = cv2.remap(f, mapx, mapy, cv2.INTER_LINEAR)
        lab = cv2.cvtColor(f, cv2.COLOR_RGB2LAB)
        lab[..., 0] = cv2.LUT(lab[..., 0], lut)
        f = cv2.cvtColor(lab, cv2.COLOR_LAB2RGB)
        return f, cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
    one(frames[0])
    t0 = time.perf_counter()
    for i in range(n):
        one(frames[i % len(frames)])
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": "frames/s", "cores": threads, "kind": "reference",
            "sample": f"{n} synthetic 4K frames through cv2 {cv2.__version__} remap+RGB2LAB+LUT+LAB2RGB+BGR2GRAY, cv2.setNumThreads({threads})"}


# ---------------------------------------------------------------------------------------------------------------
def run_dense_workload(args, rank, world, local_rank):
    """configs[4]: dense stress frames through the APRILTAG path or the classic path with a threshold-window sweep."""
    from apse_uav_b200 import aruco
    import apse_uav_b200 as A
    import __graft_entry__ as G
    c = Ctx(args, rank, world, local_rank)
    torch, dev = c.torch, c.dev
    params = G.reference_parameters(aruco)
    classic = args.workload == "dense-classic"
    nwin = 0
    if classic:
        params.cornerRefinementMethod = aruco.CORNER_REFINE_NONE
        params.adaptiveThreshWinSizeMin, params.adaptiveThreshWinSizeMax, params.adaptiveThreshWinSizeStep = args.classic_windows
        nwin = len(range(args.classic_windows[0], args.classic_windows[1] + 1, args.classic_windows[2]))
    B = args.dense_batch
    pipe = make_pipeline(args, local_rank, params=params, max_batch=B, max_markers=512)
    base = torch.from_numpy(dense_frames(args.base_frames, seed=77 + 13 * rank)).to(dev)
    n_slices = 3
    seq = torch.empty((n_slices, B, H, W, 3), dtype=torch.uint8, device=dev)
    g = torch.Generator().manual_seed(11 + rank)
    for s in range(n_slices):
        for j in range(B):
            dx, dy = (int(v) for v in torch.randint(-30, 31, (2,), generator=g))
            seq[s, j] = torch.roll(base[(s * B + j) % len(base)], shifts=(dy, dx), dims=(0, 1))
    state = {}

    def step(i):
        state["det"] = pipe.run_batch(seq[i % n_slices])

    for i in range(args.warmup):
        step(i)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = pipe.launches
    ms, _ = c.timed(step, args.steps)
    launches = pipe.launches - l0
    sampler.stop_flag = True
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, state["det"])
    markers = int(state["det"]["n"].sum().item())
    for e in pipe.engines:
        e.timing(True)
    pipe.run_batch(seq[0], serial=True)
    collect_ktimes(pipe.engines)
    c.timed(lambda i: pipe.run_batch(seq[i % n_slices], serial=True), args.steps)
    ktimes = collect_ktimes(pipe.engines)
    for e in pipe.engines:
        e.timing(False)
    host = torch.empty((B, H, W, 3), dtype=torch.uint8).pin_memory()
    host.copy_(seq[0])

    def step_e2e(_i):
        for out in pipe.run_host_stream([host]):
            state["host"] = out

    step_e2e(0)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_ms, _ = c.timed(step_e2e, e2e_steps)
    ms, e2e_ms = c.reduce([ms, e2e_ms], "max")
    launches, markers = (int(v) for v in c.reduce([launches, markers], "sum"))
    if rank == 0:
        peak, _ = peaks()
        value = args.steps * B * world / (ms / 1e3)
        alg_frame = ALG_BYTES["k_preprocess_fused"] + nwin * ALG_BYTES["classic_window"] if classic else ALG_BYTES["pipeline"]
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8/i32 pixels, f64 line fits and pose", "data": "synthetic", "config": workload_config(args, B, world),
                "e2e": {"value": e2e_steps * B * world / (e2e_ms / 1e3), "unit": "frames/s", "h2d_bytes_per_step": B * FRAME_BYTES,
                        "d2h_bytes_per_step": int(sum(v.nbytes for v in state["host"].values())), "steps": e2e_steps},
                "gpu_launches": launches, "markers_found_last_step": markers, "markers_per_frame": markers / (B * world),
                "pipeline_roofline": {"algorithmic_bytes_per_frame": alg_frame, "achieved_gbs_per_gpu": alg_frame * value / world / 1e9,
                                      "frac_of_hbm_peak": alg_frame * value / world / 1e9 / peak},
                "roofline": roofline_of(ktimes, args.steps * B),
                "kernel_ms_per_frame": {k: v[0] / (args.steps * B) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0])},
                "clocks": sampler.summary()}
        if world == 1 and args.cpu_frames > 0:
            line["cpu_baseline"] = cpu_baseline(dense_frames(2), max(4, args.cpu_frames // 4), tuple(args.classic_windows) if classic else None)
        print(json.dumps(line), flush=True)
    c.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps; one step = the whole sequence (default workload)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-stream", dest="stream", action="store_false", default=None,
                    help="sequence workload: contiguous blocks, one gather and one post-pass after the pipeline (the default)")
    ap.add_argument("--stream", dest="stream", action="store_true",
                    help="sequence workload: frames dealt out in rounds, post-pass streamed behind the pipeline")
    ap.add_argument("--tail-frames", type=int, default=8, help="streamed sequence: frames per rank in the short last round")
    ap.add_argument("--workload", default="sequence", choices=["sequence", "preprocess64", "dense-apriltag", "dense-classic"])
    ap.add_argument("--sequence-frames", type=int, default=SEQUENCE_FRAMES, help="frames of the sequence (configs[2]: 1800)")
    ap.add_argument("--batch", type=int, default=60, help="frames per pipeline batch")
    ap.add_argument("--base-frames", type=int, default=12, help="distinct seeded frames rendered on the host")
    ap.add_argument("--max-markers", type=int, default=64)
    ap.add_argument("--streams", type=int, default=3, help="CUDA streams (sub-batches in flight) per GPU")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per e2e step over all ranks (0 = the whole sequence)")
    ap.add_argument("--host-ring", type=int, default=3, help="pinned host batches reused cyclically by the e2e pass")
    ap.add_argument("--kernel-batches", type=int, default=4, help="batches of the per-kernel timing pass")
    ap.add_argument("--cpu-frames", type=int, default=24, help="frames of the bounded all-thread CPU baseline sample (0 = skip)")
    ap.add_argument("--ref-frames-per-step", type=int, default=2)
    ap.add_argument("--dense-batch", type=int, default=24)
    ap.add_argument("--classic-windows", type=int, nargs=3, default=[3, 23, 10], metavar=("MIN", "MAX", "STEP"))
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    if args.stream is None:
        # the plain run (contiguous blocks, one gather, one post-pass) is the default: streaming the post-pass behind the pipeline
        # was measured and loses -- 1 GPU 54.2 against 54.0 ms per 1800 frames, 8 GPUs 12.7 against 10.3 ms (per-round packing and
        # gathers, the short last round's latency, the worker thread sharing the interpreter with the enqueueing thread)
        args.stream = False
    {"sequence": run_sequence_workload, "preprocess64": run_preprocess_workload,
     "dense-apriltag": run_dense_workload, "dense-classic": run_dense_workload}[args.workload](args, rank, world, local_rank)


if __name__ == "__main__":
    main()
