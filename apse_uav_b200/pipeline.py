"""Batched, device-resident marker pipeline: the per-frame work of aruco_detect.py:589-601
(preprocessFrame -> BGR2GRAY -> detectMarkers -> estimatePoseSingleMarkers) for many frames at once.

Frames are independent up to the pose scale (SURVEY.md section 0.5), so a sequence is processed in batches on
one GPU and sharded frame-wise across GPUs (shard.py); the sequential marker-length / gating / distance logic of
aruco_detect.py:598-782 runs afterwards on the host over the small per-frame results (postpass.py).
"""
from __future__ import annotations

import numpy as np

from .engine import Engine
from ._lib import ApseError


class Pipeline:
    """`streams` > 1 splits every batch into that many sub-batches, each with its own context (scratch), and runs the
    two halves of the pipeline on different CUDA streams: the fused preprocess kernel (issue / bandwidth bound, fills the
    whole GPU) of all sub-batches goes to ONE normal-priority stream, the candidate / decode / pose chain (many short,
    latency-bound kernels) of sub-batch s to high-priority stream s.  The chain of sub-batch k therefore runs under the
    preprocess of sub-batch k+1 (also across consecutive run_batch calls when `sync=False`)."""

    def __init__(self, camera_matrix, dist_coeffs, size, lut, dictionary, params, max_batch=16, device=0,
                 max_markers=64, marker_length=0.55, streams=1, ring=4):
        w, h = int(size[0]), int(size[1])
        streams = max(1, min(int(streams), max_batch))
        self.sub_batch = (max_batch + streams - 1) // streams
        bl = np.ascontiguousarray(dictionary.bytesList, np.uint8)
        self.engines = []
        for _ in range(streams):
            e = Engine(device, w, h, self.sub_batch)
            e.set_camera(camera_matrix, dist_coeffs, w, h)
            e.set_lut(lut)
            e.set_dictionary(bl.reshape(bl.shape[0], -1), dictionary.markerSize, dictionary.maxCorrectionBits)
            e.set_params(params)
            self.engines.append(e)
        self.engine = self.engines[0]
        torch = self.engine.torch
        dev = self.engine.tdev
        self.streams, self.pre_stream, self._gray, self._done = [], None, [], []
        self._ring, self._ring_size, self._ring_pos = {}, max(2, int(ring)), 0   # result buffers of run_batch(sync=False)
        if streams > 1:
            # consecutive preprocess launches are independent (different frames, different contexts): rotating over
            # several streams lets the next launch fill the SMs while the last wave of the previous one drains, and lets the
            # short flag / exact kernels of one sub-batch run beside the bounds pass of the next (measured per 1800 frames:
            # 1 stream 52.7 ms, 2: 47.7, 3: 45.6, 4: 45.7, 6: 45.9)
            self.pre_streams = [torch.cuda.Stream(device=dev, priority=0) for _ in range(3)]
            self.pre_stream = self.pre_streams[0]
            self._pre_pos = 0
            self.streams = [torch.cuda.Stream(device=dev, priority=-1) for _ in range(streams)]
            # two gray buffers per engine (the library keeps two tile-extrema buffers to match): the preprocess of the next
            # use of engine s may run while the chain of the previous use still reads its gray / extrema; chains of one
            # engine are ordered by their stream, and a buffer is rewritten only after the chain two uses back has finished
            self._gray = [[torch.empty((self.sub_batch, h, w), dtype=torch.uint8, device=dev) for _ in range(2)] for _ in range(streams)]
            self._done = [[None, None] for _ in range(streams)]   # completion event of the chain that last used (engine s, buffer p)
            self._use = [0] * streams
        self.max_batch, self.max_markers, self.marker_length = max_batch, max_markers, float(marker_length)
        self.size = (w, h)

    @property
    def launches(self):
        return sum(e.launches for e in self.engines)

    def close(self):
        for e in self.engines:
            e.close()

    def _run_on(self, e, frames, out, want_gray, marker_length, gray_out=None):
        gray = gray_out
        if want_gray and gray is None:
            gray = e.torch.empty(frames.shape[:3], dtype=e.torch.uint8, device=e.tdev)
        e.process_frames(frames, out, marker_length, gray=gray)   # one library call: K1t -> candidates -> decode -> pose
        return gray

    def run_batch(self, frames, want_gray=False, want_rejected=False, marker_length=None, serial=False, sync=True,
                  input_ready=False, gray_out=None, out=None):
        """frames: [B,H,W,3] uint8 CUDA tensor, B <= max_batch.  Returns dict of device tensors.
        serial=True      runs the sub-batches one after the other on the current stream (clean per-kernel timing).
        sync=False       does not make the current stream wait for the result: call Pipeline.wait(det) (or to_host)
                         before touching it; lets consecutive batches overlap (multi-stream mode only).  The result
                         tensors come from a ring of `ring` preallocated sets (no allocation, no fill kernel on the hot
                         path): a result stays valid until `ring` further run_batch(sync=False) calls.
        input_ready=True the frames are already complete in device memory (no ordering against the current stream).
        gray_out         [B,H,W] uint8 CUDA tensor (e.g. a slice of a sequence-long buffer): the corrected gray frames are
                         written there instead of the pipeline's scratch (LED read-out, aruco_detect.py:338-373, needs them
                         after the poses are known); nothing is allocated, so batches still overlap with sync=False.
        out              dict of result tensors to write into (slices of a sequence-long set from alloc_detections(pose=True))
                         instead of the ring / a fresh allocation."""
        e = self.engine
        torch = e.torch
        B = frames.shape[0]
        if B > self.max_batch:
            raise ApseError(-1, f"batch {B} exceeds max_batch {self.max_batch}")
        ml = self.marker_length if marker_length is None else marker_length
        if gray_out is not None:
            if tuple(gray_out.shape) != tuple(frames.shape[:3]) or gray_out.dtype != torch.uint8 or not gray_out.is_contiguous():
                raise ApseError(-1, "gray_out must be a contiguous uint8 tensor of shape [B,H,W]")
            want_gray = False
        overlap = bool(self.streams) and B > 1 and not serial and not sync and not want_gray
        if out is not None:
            det = dict(out)
        elif overlap:
            key = (B, bool(want_rejected))
            if key not in self._ring:
                self._ring[key] = [e.alloc_detections(B, self.max_markers, want_rejected, pose=True) for _ in range(self._ring_size)]
                torch.cuda.current_stream(e.tdev).synchronize()
            det = dict(self._ring[key][self._ring_pos % self._ring_size])
            self._ring_pos += 1
        else:
            det = e.alloc_detections(B, self.max_markers, want_rejected, pose=True)
        if not self.streams or B <= 1:
            gray = self._run_on(e, frames, det, want_gray, ml, gray_out)
        elif serial:
            grays = []
            for s, eng in enumerate(self.engines):
                lo, hi = s * self.sub_batch, min(B, (s + 1) * self.sub_batch)
                if lo >= hi:
                    break
                sl = {k: v[lo:hi] for k, v in det.items()}
                mls = ml[lo:hi] if isinstance(ml, torch.Tensor) else ml
                grays.append(self._run_on(eng, frames[lo:hi], sl, want_gray, mls, None if gray_out is None else gray_out[lo:hi]))
            gray = torch.cat(grays, 0) if want_gray else None
        else:
            cur = torch.cuda.current_stream(e.tdev)
            alloc = None
            if not overlap and out is None:
                alloc = cur.record_event()          # output tensors are zero-filled on the current stream
            ready = None
            if not input_ready:
                ready = alloc if alloc is not None else cur.record_event()
            done, grays = [], []
            for s, (eng, st) in enumerate(zip(self.engines, self.streams)):
                lo, hi = s * self.sub_batch, min(B, (s + 1) * self.sub_batch)
                if lo >= hi:
                    break
                pre = self.pre_streams[self._pre_pos % len(self.pre_streams)]
                self._pre_pos += 1
                if ready is not None:
                    pre.wait_event(ready)
                par = self._use[s] & 1
                self._use[s] += 1
                if gray_out is not None:
                    g = gray_out[lo:hi]
                elif want_gray:
                    g = torch.empty((hi - lo,) + frames.shape[1:3], dtype=torch.uint8, device=e.tdev)
                else:
                    g = self._gray[s][par][:hi - lo]
                if self._done[s][par] is not None:
                    pre.wait_event(self._done[s][par])   # this gray / extrema buffer pair of engine s is free again
                # the pipeline's own gray buffers are scratch of the chain that follows: sparse evaluation; a caller who
                # asked for the gray frames gets all of them
                eng.preprocess_tiles(frames[lo:hi], g, stream=pre, sparse=(gray_out is None and not want_gray))
                ev = pre.record_event()
                st.wait_event(ev)
                if alloc is not None:
                    st.wait_event(alloc)
                sl = {k: v[lo:hi] for k, v in det.items()}
                mls = ml[lo:hi] if isinstance(ml, torch.Tensor) else ml
                with torch.cuda.stream(st):   # (a per-frame marker-length tensor is staged on the chain's stream)
                    eng.detect_pose_frames(g, sl, mls, stream=st)
                self._done[s][par] = st.record_event()
                done.append(self._done[s][par])
                grays.append(g)
            if overlap:
                det["_done"] = done
            else:
                for ev in done:
                    cur.wait_event(ev)
            # (after the waits: the gray sub-batches are written on the preprocess streams, which the current stream has only
            # now been ordered behind through the chains' completion events)
            gray = torch.cat(grays, 0) if want_gray else None
        if want_gray:
            det["gray"] = gray
        return det

    @staticmethod
    def wait(det):
        """Make the current stream wait for a result returned by run_batch(sync=False)."""
        import torch
        evs = det.pop("_done", None)
        if evs:
            cur = torch.cuda.current_stream(det["n"].device)
            for ev in evs:
                cur.wait_event(ev)
        return det

    def run_sequence(self, frames, gray_out=None, want_rejected=False, marker_length=None):
        """A whole HBM-resident sequence [n,H,W,3] through the pipeline, batch after batch without host synchronisation
        (the chain of batch k runs under the preprocess of batch k+1); results of all n frames in one set of device tensors.
        gray_out: [n,H,W] uint8 CUDA tensor that receives the corrected gray frames (LED read-out), or None."""
        e = self.engine
        torch = e.torch
        n = int(frames.shape[0])
        det = e.alloc_detections(n, self.max_markers, want_rejected, pose=True)
        cur = torch.cuda.current_stream(e.tdev)
        filled = cur.record_event()   # the fills of alloc_detections run on the current stream; the chains write on their own
        for st in self.streams:
            st.wait_event(filled)
        pending = []
        for lo in range(0, n, self.max_batch):
            hi = min(n, lo + self.max_batch)
            sl = {k: v[lo:hi] for k, v in det.items()}
            r = self.run_batch(frames[lo:hi], want_rejected=want_rejected, marker_length=marker_length, sync=False, input_ready=False,
                               gray_out=None if gray_out is None else gray_out[lo:hi], out=sl)
            pending.extend(r.get("_done", ()))
        for ev in pending:
            cur.wait_event(ev)
        return det

    def run(self, frames, **kw):
        """Any number of frames, processed in batches of max_batch; results concatenated on the device."""
        torch = self.engine.torch
        outs = [self.run_batch(frames[i:i + self.max_batch], **kw) for i in range(0, frames.shape[0], self.max_batch)]
        if len(outs) == 1:
            return outs[0]
        if "_done" in outs[0]:
            for o in outs:
                self.wait(o)
        return {k: torch.cat([o[k] for o in outs], 0) for k in outs[0]}

    def run_host_stream(self, host_batches, **kw):
        """End-to-end path for frames that live in (pinned) host memory: yields one host result dict per batch.
        Two device staging buffers and a copy stream: the H2D copy of batch k+1 runs while batch k is processed and
        its detections are read back, so a sequence is bounded by the slower of PCIe and the kernels, not their sum."""
        torch = self.engine.torch
        dev = self.engine.tdev
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=dev)
            w, h = self.size
            self._stage = [torch.empty((self.max_batch, h, w, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
        cs, stage = self._copy_stream, self._stage
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        it = iter(host_batches)
        cur = next(it, None)
        if cur is None:
            return
        cs.wait_stream(main)
        with torch.cuda.stream(cs):
            stage[0][:len(cur)].copy_(cur, non_blocking=True)
            ready[0].record(cs)
        k = 0
        while cur is not None:
            nxt = next(it, None)
            if nxt is not None:
                if k >= 1:
                    cs.wait_event(done[(k + 1) % 2])   # the other buffer was the input of batch k-1
                with torch.cuda.stream(cs):
                    stage[(k + 1) % 2][:len(nxt)].copy_(nxt, non_blocking=True)
                    ready[(k + 1) % 2].record(cs)
            main.wait_event(ready[k % 2])
            det = self.run_batch(stage[k % 2][:len(cur)], **kw)
            done[k % 2].record(main)
            yield self.to_host(det)
            cur, k = nxt, k + 1

    @staticmethod
    def to_host(det):
        """Gather the small per-frame results to the host as numpy arrays (the only D2H traffic of the pipeline)."""
        Pipeline.wait(det)
        out = {k: v.cpu().numpy() for k, v in det.items() if k != "gray"}
        bad = np.nonzero(out["status"])[0]
        if len(bad):
            raise ApseError(int(out["status"][bad[0]]), f"work-buffer capacity exceeded in frames {bad.tolist()[:8]}")
        return out
