"""Frame-wise sharding of a sequence across GPUs (one process + one Pipeline per GPU, no collective on the hot
path; SURVEY.md section 8e) and the two-pass handling of the only cross-frame coupling, the marker-length
recurrence of aruco_detect.py:306-308,601,623,641.

Pass 1 (parallel, per rank): preprocess + detect + pose with the nominal marker length on the rank's block of frames.
Gather  (after the hot path): the per-frame results (~5 KB per frame) go to rank 0 as tensors (dist.gather).
Scan    (rank 0, sequential, native: sequence.py / csrc/sequence.cu): the marker logic over frames in order with tvec scaled
        by L_k / L_nominal (tvec is linear in the marker length), which yields the marker length L_k each frame's pose must use.
Pass 2 (rank 0, one batched launch): exact pose of every frame with its L_k, the final scan, one launch for all
        projection jobs (vehicle outlines, LED strip), CSV rows.
The *_python functions below are the per-frame Python mirror of the same flow (postpass.SequencePostPass); the tests check the
native path against them.
"""
from __future__ import annotations

import numpy as np

from .postpass import SequencePostPass, MARKER_LENGTH_ORG, csv_line


def shard_bounds(n_frames: int, world: int):
    """Contiguous blocks: rank r gets frames [lo, hi)."""
    return [(n_frames * r // world, n_frames * (r + 1) // world) for r in range(world)]


def pack_results(host, lo):
    """Per-frame records from Pipeline.to_host output."""
    recs = []
    for i in range(len(host["n"])):
        n = int(host["n"][i])
        recs.append(dict(frame=lo + i, ids=host["ids"][i, :n].copy(), corners=host["corners"][i, :n].copy(),
                         rvec=host["rvec"][i, :n].copy(), tvec=host["tvec"][i, :n].copy()))
    return recs


def gather_records(local, rank=0, world=1, group=None):
    """All ranks' records on rank 0, ordered by frame (small python objects; works on gloo and nccl groups)."""
    if world == 1:
        return sorted(local, key=lambda r: r["frame"])
    import torch.distributed as dist
    out = [None] * world if rank == 0 else None
    dist.gather_object(local, out, dst=0, group=group)
    if rank != 0:
        return None
    return sorted([r for part in out for r in part], key=lambda r: r["frame"])


def scan_marker_lengths(records, project, start_frame=1):
    """First sequential scan: poses were computed with MARKER_LENGTH_ORG; rescale tvec by L_k / L_nominal."""
    pp = SequencePostPass(project, start_frame=start_frame)
    lengths = []
    for r in records:
        L = pp.marker_length
        lengths.append(L)
        pp.step(start_frame + r["frame"], r["ids"] if len(r["ids"]) else None, r["corners"], r["rvec"],
                r["tvec"] * (L / MARKER_LENGTH_ORG))
    return lengths


def exact_pose(records, lengths, pose_fn):
    """Second pass: pose_fn(corners (n,4,2) f32, marker_len (n,) f32) -> (rvec (n,3), tvec (n,3)) in ONE batched call."""
    counts = [len(r["ids"]) for r in records]
    if sum(counts) == 0:
        return records
    corners = np.concatenate([r["corners"].reshape(-1, 4, 2) for r in records if len(r["ids"])]).astype(np.float32)
    ml = np.concatenate([np.full(c, L, np.float32) for c, L in zip(counts, lengths) if c])
    rv, tv = pose_fn(corners, ml)
    out, o = [], 0
    for r, c in zip(records, counts):
        out.append(dict(r, rvec=rv[o:o + c], tvec=tv[o:o + c]))
        o += c
    return out


def final_scan(records, project, start_frame=1, led_mean_for_frame=None, led_sums_for_frame=None):
    pp = SequencePostPass(project, start_frame=start_frame)
    rows = []
    for r in records:
        if led_mean_for_frame is not None:
            pp.led_mean = led_mean_for_frame(r["frame"])
        if led_sums_for_frame is not None:
            pp.led_sums = led_sums_for_frame(r["frame"])
        rows.append(pp.step(start_frame + r["frame"], r["ids"] if len(r["ids"]) else None, r["corners"], r["rvec"], r["tvec"]))
    return rows


def gather_detections(det, n_local, rank=0, world=1, group=None):
    """Per-frame results of every rank's block on rank 0, in frame order, as one dict of tensors (device tensors over
    NCCL, CPU tensors over gloo).  This is the only data-path exchange of a frame-sharded run: two collectives -- the block
    sizes and the number of marker slots in use, then ONE packed byte buffer per rank holding only those slots
    (8 + 84 bytes per frame and used slot instead of 5.4 KB per frame)."""
    keys = ("n", "ids", "corners", "rvec", "tvec", "status")
    if world == 1:
        return {k: det[k] for k in keys}, [n_local]
    import torch
    import torch.distributed as dist
    dev = det["n"].device
    M = int(det["ids"].shape[1])
    hdr = torch.zeros(2, dtype=torch.int64, device=dev)
    hdr[0] = n_local
    if n_local:
        hdr[1] = det["n"][:n_local].max()
    all_hdr = torch.empty((world, 2), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(all_hdr, hdr, group=group) if dev.type == "cuda" else dist.all_gather(list(all_hdr.unbind(0)), hdr, group=group)
    all_hdr = all_hdr.cpu()
    sizes = [int(v) for v in all_hdr[:, 0]]
    cap, m = max(max(sizes), 1), max(1, min(M, int(all_hdr[:, 1].max())))
    # packed layout of one rank: n [cap] i32 | status [cap] i32 | ids [cap, m] i32 | corners [cap, m, 8] f32 | rvec [cap, m, 3] f64 | tvec
    fields = (("n", torch.int32, ()), ("status", torch.int32, ()), ("ids", torch.int32, (m,)), ("corners", torch.float32, (m, 4, 2)),
              ("rvec", torch.float64, (m, 3)), ("tvec", torch.float64, (m, 3)))
    sizes_b = [cap * int(np.prod(shape, dtype=np.int64)) * torch.empty((), dtype=dt).element_size() for _, dt, shape in fields]
    offs = np.concatenate([[0], np.cumsum([(b + 15) // 16 * 16 for b in sizes_b])]).astype(np.int64)   # 16-byte aligned fields
    buf = torch.zeros(int(offs[-1]), dtype=torch.uint8, device=dev)
    for (k, dt, shape), o, sb in zip(fields, offs, sizes_b):
        dst = buf[int(o):int(o) + sb].view(dt).reshape((cap,) + shape)
        src = det[k][:n_local]
        dst[:n_local] = src[:, :m] if len(shape) else src
    parts = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
    dist.gather(buf, parts, dst=0, group=group)
    if rank != 0:
        return None, sizes
    out = {}
    for (k, dt, shape), o, sb in zip(fields, offs, sizes_b):
        out[k] = torch.cat([p_[int(o):int(o) + sb].view(dt).reshape((cap,) + shape)[:sz] for p_, sz in zip(parts, sizes)], 0)
    return out, sizes


def _exchange_led_jobs(engine, gray, frame0, rank, world, group):
    """LED read-out of a frame-sharded run (aruco_detect.py:338-373 needs the gray pixels of the frame, which live on the
    rank that processed it): rank 0 broadcasts the job list, every rank evaluates the LED jobs of its own frames, rank 0
    collects the results.  A few hundred KB per sequence, after the hot path."""
    import torch
    import torch.distributed as dist
    from . import sequence
    from ._lib import SEQ_JOB_DTYPE, SEQ_RESULT_DTYPE
    dev = engine.tdev

    def exchange(jobs, results):
        cnt = torch.tensor([len(jobs) if rank == 0 else 0], dtype=torch.int64, device=dev)
        dist.broadcast(cnt, 0, group=group)
        nj = int(cnt.item())
        if nj == 0:
            return results
        buf = torch.empty(nj * np.dtype(SEQ_JOB_DTYPE).itemsize, dtype=torch.uint8, device=dev)
        if rank == 0:
            buf.copy_(torch.from_numpy(np.ascontiguousarray(jobs).view(np.uint8).reshape(-1)))
        dist.broadcast(buf, 0, group=group)
        if rank != 0:
            jobs_l = buf.cpu().numpy().view(SEQ_JOB_DTYPE)
            led = jobs_l["kind"] == 0
            res_l = np.zeros(nj, SEQ_RESULT_DTYPE)
            if led.any():
                res_l[led] = sequence.run_jobs(engine, jobs_l[led], gray=gray, frame0=frame0)
        else:
            res_l = results
        rt = torch.from_numpy(np.ascontiguousarray(res_l).view(np.uint8).reshape(-1).copy()).to(dev)
        parts = [torch.empty_like(rt) for _ in range(world)] if rank == 0 else None
        dist.gather(rt, parts, dst=0, group=group)
        if rank == 0:
            merged = results.copy()
            for p_ in parts[1:]:
                r = p_.cpu().numpy().view(SEQ_RESULT_DTYPE)
                take = (r["valid"] == 1) & (merged["valid"] == 0)
                merged[take] = r[take]
            return merged
        return None
    return exchange


def run_sequence(pipe, frames, rank=0, world=1, group=None, start_frame=1, leds=False, leds_threshold=None, as_rows=False):
    """aruco_detect.py:571-810 for a frame-sharded sequence.  frames: this rank's contiguous block ([n_local,H,W,3] uint8 CUDA
    tensor); the blocks of ranks 0..world-1 concatenate to the sequence.  Returns on rank 0 the list of CSV row dicts
    (as_rows=True: the native row array, for sequence.rows_to_csv) and None elsewhere.
    Pipeline of one run: batched GPU pipeline per rank (nominal marker length) -> gather of the per-frame results on rank 0
    -> native post-pass (sequence.postpass_device: scan, one exact-pose launch, scan, one projection-job launch).
    leds=True: the corrected gray frames stay on the device of the rank that produced them and the LED strip of the host
    vehicle (:338-373) is read there."""
    e = pipe.engine
    torch = e.torch
    n_local = int(frames.shape[0])
    w, h = pipe.size
    gray = torch.empty((n_local, h, w), dtype=torch.uint8, device=e.tdev) if leds and n_local else None
    if n_local:
        det = pipe.run_sequence(frames, gray_out=gray)
    else:
        det = e.alloc_detections(0, pipe.max_markers, False, pose=True)
    return _finish_sequence(pipe, det, gray, n_local, rank, world, group, start_frame, leds, leds_threshold, as_rows)


def run_sequence_host(pipe, host_batches, n_local, rank=0, world=1, group=None, start_frame=1, leds=False, leds_threshold=None,
                      as_rows=False):
    """run_sequence for frames that live in (pinned) HOST memory: host_batches yields this rank's block as uint8 tensors
    [b,H,W,3] with b <= pipe.max_batch, n_local frames in total.  Two device staging buffers and a copy stream: the H2D copy
    of batch k+1 runs under the kernels of batch k; everything after the pipeline is the same as run_sequence."""
    e = pipe.engine
    torch = e.torch
    dev = e.tdev
    w, h = pipe.size
    gray = torch.empty((n_local, h, w), dtype=torch.uint8, device=dev) if leds and n_local else None
    det = e.alloc_detections(n_local, pipe.max_markers, False, pose=True)
    main = torch.cuda.current_stream(dev)
    if not hasattr(pipe, "_copy_stream"):
        pipe._copy_stream = torch.cuda.Stream(device=dev)
        pipe._stage = [torch.empty((pipe.max_batch, h, w, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
    cs, stage = pipe._copy_stream, pipe._stage
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    free = [None, None]                      # completion events of the batch that last read staging buffer i
    filled = main.record_event()
    for st in pipe.streams:
        st.wait_event(filled)
    cs.wait_event(filled)
    pending, lo = [], 0
    for k, hb in enumerate(host_batches):
        b = int(hb.shape[0])
        buf = k % 2
        for ev in free[buf] or ():
            cs.wait_event(ev)
        with torch.cuda.stream(cs):
            stage[buf][:b].copy_(hb, non_blocking=True)
            ready[buf].record(cs)
        main.wait_event(ready[buf])
        sl = {key: v[lo:lo + b] for key, v in det.items()}
        r = pipe.run_batch(stage[buf][:b], sync=False, input_ready=False, gray_out=None if gray is None else gray[lo:lo + b], out=sl)
        done = list(r.get("_done", ()))
        if not done:
            done = [main.record_event()]
        free[buf] = done
        pending.extend(done)
        lo += b
    if lo != n_local:
        raise ValueError(f"host_batches held {lo} frames, expected {n_local}")
    for ev in pending:
        main.wait_event(ev)
    return _finish_sequence(pipe, det, gray, n_local, rank, world, group, start_frame, leds, leds_threshold, as_rows)


def _finish_sequence(pipe, det, gray, n_local, rank, world, group, start_frame, leds, leds_threshold, as_rows):
    from . import sequence
    e = pipe.engine
    torch = e.torch
    all_det, sizes = gather_detections(det, n_local, rank, world, group)
    frame0 = sum(sizes[:rank])
    exchange = _exchange_led_jobs(e, gray, frame0, rank, world, group) if (leds and world > 1) else None
    if rank != 0:
        if exchange is not None:
            exchange(None, None)
        return None
    bad = torch.nonzero(all_det["status"]).flatten()
    if bad.numel():
        from ._lib import ApseError
        raise ApseError(int(all_det["status"][bad[0]]), f"work-buffer capacity exceeded in frames {bad.tolist()[:8]}")
    rows = sequence.postpass_device(e, all_det, start_frame=start_frame, leds=leds, leds_threshold=leds_threshold, gray=gray,
                                    frame0=0, exchange=exchange)
    return rows if as_rows else sequence.rows_to_dicts(rows)


def round_plan(n_frames: int, world: int, batch: int, tail: int = 0):
    """Round-robin sharding for a streamed run: the sequence is cut into rounds of at most world * batch consecutive frames and
    every round into `world` consecutive parts (rank r takes part r), all as equal as possible.  Round k is complete as soon as
    every rank has finished its k-th batch, so rank 0 can run the sequential post-pass of round k while all ranks work on round
    k + 1 -- with contiguous blocks (shard_bounds) nothing could start before the very end.  tail > 0: a last, short round of
    about `tail` frames per rank keeps the part of the post-pass that nothing overlaps small.
    Returns [[(lo, hi) for each rank] for each round]."""
    world, batch = max(1, int(world)), max(1, int(batch))
    cuts = [0]
    tail_frames = min(n_frames, max(0, int(tail)) * world)
    if tail_frames and n_frames - tail_frames < world * batch:
        tail_frames = 0
    body = n_frames - tail_frames
    nr = max(1, -(-body // (world * batch))) if body else 0
    for k in range(nr):
        cuts.append((body * (k + 1)) // nr)
    if tail_frames:
        cuts.append(n_frames)
    return [[(a + lo, a + hi) for lo, hi in shard_bounds(b - a, world)] for a, b in zip(cuts[:-1], cuts[1:])]


def _packed_fields(torch, cap, m):
    """Layout of the packed per-round results of one rank: n | status | ids | corners | rvec | tvec, 16-byte aligned fields."""
    fields = (("n", torch.int32, ()), ("status", torch.int32, ()), ("ids", torch.int32, (m,)), ("corners", torch.float32, (m, 4, 2)),
              ("rvec", torch.float64, (m, 3)), ("tvec", torch.float64, (m, 3)))
    sizes_b = [cap * int(np.prod(shape, dtype=np.int64)) * torch.empty((), dtype=dt).element_size() for _, dt, shape in fields]
    offs = np.concatenate([[0], np.cumsum([(b + 15) // 16 * 16 for b in sizes_b])]).astype(np.int64)
    return fields, sizes_b, offs


def run_sequence_streamed(pipe, frames, plan, rank=0, world=1, group=None, start_frame=1, as_rows=False, chunk_frames=240):
    """aruco_detect.py:571-810 for a sequence sharded by round_plan, with the post-pass streamed behind the pipeline.
    frames: this rank's parts of all rounds, concatenated ([n_local,H,W,3] uint8 CUDA tensor); plan: round_plan(...) of the whole
    sequence (the same on every rank).  Per round every rank enqueues its batch (no host synchronisation), packs the batch's
    results on a side stream and -- world > 1 -- sends them to rank 0 (one NCCL gather per round, off the pipeline's streams);
    rank 0 copies the round to pinned memory and a worker thread feeds every completed round to a sequence.SequenceStream
    (both scans, exact poses, projection jobs for those frames) while the calling thread keeps enqueueing.  What is left after
    the last batch is the post-pass of the last round.  Rows equal run_sequence's (tests/test_gpu_pipeline.py).  No LED read-out (run_sequence)."""
    from . import sequence
    from ._lib import ApseError
    e = pipe.engine
    torch = e.torch
    dev = e.tdev
    M = pipe.max_markers
    nr = len(plan)
    cap = max(1, max((hi - lo for rnd in plan for lo, hi in rnd), default=0))
    if cap > pipe.max_batch:
        raise ApseError(-1, f"round_plan parts of {cap} frames exceed the pipeline's max_batch {pipe.max_batch}")
    fields, sizes_b, offs = _packed_fields(torch, cap, M)
    nbytes = int(offs[-1])
    n_local = sum(rnd[rank][1] - rnd[rank][0] for rnd in plan)
    if int(frames.shape[0]) != n_local:
        raise ValueError(f"rank {rank} holds {int(frames.shape[0])} frames, the plan gives it {n_local}")
    key = (nr, world, nbytes, n_local)
    st = getattr(pipe, "_stream_bufs", None)
    if st is None or st["key"] != key:
        st = pipe._stream_bufs = dict(key=key, comm=torch.cuda.Stream(device=dev, priority=-1),
                                      send=torch.zeros((nr, nbytes), dtype=torch.uint8, device=dev),
                                      recv=torch.zeros((nr, world, nbytes), dtype=torch.uint8, device=dev) if rank == 0 else None,
                                      pin=torch.zeros((nr, world, nbytes), dtype=torch.uint8).pin_memory() if rank == 0 else None,
                                      det=e.alloc_detections(max(n_local, 1), M, False, pose=True))
        torch.cuda.current_stream(dev).synchronize()
    comm, det = st["comm"], st["det"]
    cur = torch.cuda.current_stream(dev)
    filled = cur.record_event()
    for s_ in pipe.streams or ():
        s_.wait_event(filled)
    comm.wait_event(filled)
    seq = sequence.SequenceStream(e, start_frame) if rank == 0 else None
    arrived = []          # rank 0: (round, event) of rounds whose results are on their way to pinned memory
    done_upto = 0

    def process(upto):
        # rounds [done_upto, upto) are in pinned memory: one push
        nonlocal done_upto
        if upto <= done_upto:
            return
        host = st["pin"].numpy()
        parts = {k: [] for k, _, _ in fields}
        dev_c, dev_n = [], []
        for r in range(done_upto, upto):
            for q in range(world):
                sz = plan[r][q][1] - plan[r][q][0]
                if sz == 0:
                    continue
                for (k, dt, shape), o, sb in zip(fields, offs, sizes_b):
                    parts[k].append(host[r, q, int(o):int(o) + sb].view(sequence._NP[dt]).reshape((cap,) + shape)[:sz])
                    if k in ("corners", "n"):
                        (dev_c if k == "corners" else dev_n).append(st["recv"][r, q, int(o):int(o) + sb].view(dt).reshape((cap,) + shape)[:sz])
        if not parts["n"]:
            done_upto = upto
            return
        h = {k: (v[0] if len(v) == 1 else np.concatenate(v)) for k, v in parts.items()}
        bad = np.nonzero(h["status"])[0]
        if len(bad):
            raise ApseError(int(h["status"][bad[0]]), f"work-buffer capacity exceeded in frames {(seq.frames + bad[:8]).tolist()}")
        with torch.cuda.stream(seq.stream):
            seq.stream.wait_event(arrived[upto - 1][1])
            cd = dev_c[0].contiguous() if len(dev_c) == 1 else torch.cat(dev_c, 0)
            nd = dev_n[0].contiguous() if len(dev_n) == 1 else torch.cat(dev_n, 0)
        seq.push(h["n"], h["ids"], h["corners"], h["rvec"], h["tvec"], cd, nd)
        done_upto = upto

    # rank 0: the post-pass runs on a worker thread of its own (every push blocks on two small device round trips; on the
    # enqueueing thread each of them lets the pipeline's launch queue run dry: 57.4 against 54.2 ms per 1800 frames on one GPU).
    # The worker waits for the rounds in order and pushes them once chunk_frames frames have piled up; event / stream
    # synchronisation and the ctypes calls release the interpreter lock.  Waiting by polling with short sleeps was tried and is
    # much worse (67 - 105 ms: every wake-up takes the lock away from the enqueueing thread).
    import queue
    import threading
    todo = queue.Queue()
    failure = []

    def worker():
        try:
            torch.cuda.set_device(dev)
            for _ in range(nr):
                r_, ev_ = todo.get()
                if ev_ is None:
                    return
                ev_.synchronize()   # releases the interpreter lock (so do the ctypes calls of the push)
                pending = sum(hi_ - lo_ for rr in range(done_upto, r_ + 1) for lo_, hi_ in plan[rr])
                if pending >= chunk_frames or r_ + 1 >= nr - 1:   # the last two rounds go one by one: nothing hides the very last push
                    process(r_ + 1)
        except BaseException as exc:   # re-raised on the calling thread
            failure.append(exc)

    th = None
    if rank == 0 and nr:
        th = threading.Thread(target=worker, name="apse-postpass", daemon=True)
        th.start()
    try:
        lo = 0
        for r in range(nr):
            a, b = plan[r][rank]
            sz = b - a
            done = []
            if sz:
                sl = {k: v[lo:lo + sz] for k, v in det.items()}
                res = pipe.run_batch(frames[lo:lo + sz], sync=False, input_ready=False, out=sl)
                done = list(res.get("_done", ())) or [cur.record_event()]
            with torch.cuda.stream(comm):
                for ev in done:
                    comm.wait_event(ev)
                buf = st["send"][r] if world > 1 or rank != 0 else st["recv"][r, 0]
                if sz:
                    for (k, dt, shape), o, sb in zip(fields, offs, sizes_b):
                        buf[int(o):int(o) + sb].view(dt).reshape((cap,) + shape)[:sz] = det[k][lo:lo + sz]
                if world > 1:
                    import torch.distributed as dist
                    dist.gather(buf, list(st["recv"][r].unbind(0)) if rank == 0 else None, dst=0, group=group)
                if rank == 0:
                    st["pin"][r].copy_(st["recv"][r], non_blocking=True)
                    arrived.append((r, comm.record_event()))
                    if th is not None:
                        todo.put(arrived[-1])
            lo += sz   # (after a failure of the worker the remaining rounds are still enqueued: the other ranks wait in their gathers)
    except BaseException:
        if th is not None:
            todo.put((nr, None))
        raise
    finally:
        if th is not None:
            th.join()
    if failure:
        raise failure[0]
    if rank != 0:
        comm.synchronize()
        return None
    rows = seq.result()
    return rows if as_rows else sequence.rows_to_dicts(rows)


def run_sequence_python(pipe, frames, start_frame=1, leds=False):
    """Single-process run with the per-frame Python mirror of the reference's loop (postpass.SequencePostPass) instead of the
    native post-pass: every cv2.projectPoints of the reference becomes one kernel launch.  Kept for the parity tests (the
    native rows must equal these) -- orders of magnitude slower per frame than run_sequence."""
    n_local = int(frames.shape[0])
    det = pipe.run(frames, want_gray=leds)
    gray = det.pop("gray") if leds else None
    host = pipe.to_host(det)
    records = gather_records(pack_results(host, 0))
    e = pipe.engine
    project = lambda obj, rvec, tvec: e.project_points(obj, rvec, tvec).cpu().numpy()

    def pose_fn(corners, ml):
        rv, tv = e.pose(corners, ml)
        return rv.cpu().numpy(), tv.cpu().numpy()

    lengths = scan_marker_lengths(records, project, start_frame)
    records = exact_pose(records, lengths, pose_fn)
    led_fn = None
    if gray is not None:
        led_fn = lambda frame: (lambda xy: e.patch_sums(gray, [(frame, int(x), int(y)) for x, y in xy], half=2))
    return final_scan(records, project, start_frame, led_sums_for_frame=led_fn)


def rows_to_csv(rows):
    from .postpass import CSV_HEADER
    return "\n".join([CSV_HEADER] + [csv_line(r) for r in rows]) + "\n"
