"""End-to-end frames/s of the benchmark's 1800-frame 4K sequence from pinned HOST memory, fed as NV12 (a video decoder's output,
12.4 MB per frame, converted on the GPU by k_yuv420_to_bgr) against the same pixels fed as BGR (24.9 MB per frame, converted on
the host by cv2.cvtColor beforehand).  One e2e step = host ring -> H2D per batch -> pipeline -> gather -> post-pass -> CSV text
(shard.run_sequence_host), as bench.py's `e2e`.  The two arms alternate in one process and are repeated, so the spread is
visible; both see identical pixels, so their CSV texts must be equal (asserted).

    python tools/bench_yuv.py [--gpus N] [--repeats 3] [--out profiles/r03_yuv_e2e_n1.json]

Also reported: the H2D bytes per step of each arm, the conversion kernel's device time per 4K frame (apse_timing, a batch of
--batch frames converted alone on one stream) and its achieved GB/s (12.4 MB read + 24.9 MB written per frame) against the HBM
peak of bench.peaks(), and the card name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402

W, H = bench.W, bench.H
NV12_BYTES = W * H * 3 // 2
BGR_BYTES = W * H * 3


def card_info(local_rank):
    """name and power limit (W) of this rank's GPU, read now (NVML, else nvidia-smi --query-gpu)"""
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    phys = int(visible.split(",")[local_rank]) if visible and visible.split(",")[local_rank].isdigit() else local_rank
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        name = pynvml.nvmlDeviceGetName(h)
        return {"name": name.decode() if isinstance(name, bytes) else name,
                "power_limit_w": pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0, "source": "nvml"}
    except Exception:
        out = subprocess.run(["nvidia-smi", f"--id={phys}", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True).stdout.strip()
        name, _, pl = out.rpartition(",")
        return {"name": name.strip(), "power_limit_w": float(pl), "source": "nvidia-smi --query-gpu"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--repeats", type=int, default=3, help="timed (NV12, BGR) pairs, order alternating")
    ap.add_argument("--sequence-frames", type=int, default=bench.SEQUENCE_FRAMES)
    ap.add_argument("--batch", type=int, default=60)
    ap.add_argument("--base-frames", type=int, default=12)
    ap.add_argument("--max-markers", type=int, default=64)
    ap.add_argument("--streams", type=int, default=3)
    ap.add_argument("--host-ring", type=int, default=3, help="pinned host batches reused cyclically (as bench.py's e2e)")
    ap.add_argument("--kernel-launches", type=int, default=20)
    ap.add_argument("--out", help="also write the JSON line here (rank 0)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29543", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))

    import cv2
    from apse_uav_b200 import shard, sequence
    from tools import synth
    c = bench.Ctx(args, rank, world, local_rank)
    torch = c.torch
    pipe = bench.make_pipeline(args, local_rank)
    n_seq = args.sequence_frames
    lo, hi = shard.shard_bounds(n_seq, world)[rank]
    n_local = hi - lo
    base = bench.base_sequence(args.base_frames)
    plan = bench.sequence_plan(n_seq, args.base_frames)
    # the ring: the first frames of this rank's block, converted to NV12 once on the host; the BGR arm gets cv2's conversion of
    # exactly those NV12 frames, so both arms carry the same pixels
    n_ring = max(1, min(args.host_ring, (n_local + args.batch - 1) // args.batch))
    ring = {"nv12": [torch.empty((args.batch, H * 3 // 2, W), dtype=torch.uint8).pin_memory() for _ in range(n_ring)],
            "bgr": [torch.empty((args.batch, H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(n_ring)]}
    for j in range(n_ring):
        for i in range(args.batch):
            p, dy, dx = plan[lo + (j * args.batch + i) % n_local]
            nv12 = synth.bgr_to_yuv420(np.roll(base[p], (dy, dx), axis=(0, 1)), "nv12")
            ring["nv12"][j][i].copy_(torch.from_numpy(nv12))
            ring["bgr"][j][i].copy_(torch.from_numpy(cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12)))
    state = {}

    def host_batches(arm):
        left, k = n_local, 0
        while left > 0:
            b = min(args.batch, left)
            yield ring[arm][k % n_ring][:b]
            left -= b
            k += 1

    def step(arm):
        rows = shard.run_sequence_host(pipe, host_batches(arm), n_local, rank, world, as_rows=True,
                                       layout="nv12" if arm == "nv12" else None)
        if rank == 0:
            state[arm] = sequence.rows_to_csv(rows)

    for arm in ("nv12", "bgr"):   # warm-up of both arms
        step(arm)
    ms = {"nv12": [], "bgr": []}
    for r in range(args.repeats):
        for arm in (("nv12", "bgr") if r % 2 == 0 else ("bgr", "nv12")):
            t, _ = c.timed(lambda _i, a=arm: step(a), 1)
            ms[arm].append(c.reduce([t], "max")[0])
    csv_equal = state.get("nv12") == state.get("bgr") if rank == 0 else None
    if rank == 0:
        assert csv_equal, "the NV12 and BGR arms wrote different CSV texts"

    # the conversion kernel alone: one batch converted on one stream, every launch bracketed by CUDA events in the library
    e = pipe.engine
    src = ring["nv12"][0].to(e.tdev)
    dst = torch.empty((args.batch, H, W, 3), dtype=torch.uint8, device=e.tdev)
    e.cvt_yuv420(src, "nv12", out=dst)
    e.timing_collect(reset=True)
    e.timing(True)
    for _ in range(args.kernel_launches):
        e.cvt_yuv420(src, "nv12", out=dst)
    kt = e.timing_collect(reset=True).get("k_yuv420_to_bgr", (0.0, 0))
    e.timing(False)
    k_ms_frame = kt[0] / max(1, kt[1]) / args.batch
    k_ms_frame = c.reduce([k_ms_frame], "max")[0]
    card = card_info(local_rank)

    if rank == 0:
        peak, peak_src = bench.peaks()
        fps = {a: [n_seq / (t / 1e3) for t in v] for a, v in ms.items()}
        gbs = (NV12_BYTES + BGR_BYTES) / (k_ms_frame / 1e3) / 1e9 if k_ms_frame > 0 else 0.0
        line = {
            "metric": "e2e 4K frames/s from pinned host memory, NV12 vs BGR input", "n_gpus": world,
            "frames_per_step": n_seq, "batch": args.batch, "streams": args.streams, "repeats": args.repeats,
            "nv12": {"fps": fps["nv12"], "fps_median": float(np.median(fps["nv12"])), "ms_per_step": ms["nv12"],
                     "h2d_bytes_per_step": n_seq * NV12_BYTES},
            "bgr": {"fps": fps["bgr"], "fps_median": float(np.median(fps["bgr"])), "ms_per_step": ms["bgr"],
                    "h2d_bytes_per_step": n_seq * BGR_BYTES},
            "speedup_median": float(np.median(fps["nv12"]) / np.median(fps["bgr"])),
            "csv_equal": bool(csv_equal), "csv_rows": state["nv12"].count("\n") - 1,
            "yuv2bgr_kernel": {"ms_per_frame": k_ms_frame, "bytes_per_frame": NV12_BYTES + BGR_BYTES, "achieved_gbs": gbs,
                               "hbm_peak_gbs": peak, "peak_source": peak_src, "frac_of_peak": gbs / peak,
                               "launches": int(kt[1]), "frames_per_launch": args.batch,
                               "note": "apse_timing (CUDA events around each launch), batch converted alone on one stream, max over ranks"},
            "card": card,
            "note": "one step = the whole sequence: pinned host ring -> H2D per batch (copy stream) [-> NV12 to BGR on the device] "
                    "-> pipeline -> gather -> post-pass -> CSV text; arms alternate in one process; time = max over ranks",
        }
        txt = json.dumps(line)
        print(txt, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(txt + "\n")
    c.close()


if __name__ == "__main__":
    main()
