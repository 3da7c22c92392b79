"""detect -> NMS -> associate as one pipelined object: what ``tracker/track.py:138-179`` does per frame
(model forward, non_max_suppression + scale_coords, tracker.update), for B sequences at once.

CUDA streams keep the B200 busy across frames:
  copy    : pinned host frames -> device, then the uint8 ingest kernel (letterbox + RGB + /255 + ReOrg + 16-bit NHWC)
  detect  : the 107 tcgen05 convs + glue of the forward (one CUDA graph per detector), back to back
  nms     : Detect decode fused with NMS (second graph)
  track   : [camera-motion estimate] + fused ByteTrack / SORT / BoT-SORT step on the NMS output, then D2H of the track rows
With ONE detector the ingest and the NMS share the detect stream (its input, head and output buffers are single).  With TWO twin
detectors (same weights, same plans, own buffers; frames alternate between them) frame t+1 is ingested and frame t-1 is
post-processed while frame t's forward runs: the detect stream never idles between forward graphs.  Cross-frame hazards (the input
staging, the stem input, the head maps and the NMS output of each detector) are guarded by events.  ``step()`` returns the tracks of
the PREVIOUS call (one frame of latency, same results); ``flush()`` returns the last ones.
"""
import gc

import torch

from . import _lib as L


class TrackingPipeline:
    def __init__(self, detector, engine, out_rows=512, gmc=None):
        """detector: a ``DetectorW6`` or a pair of twins (see above).
        gmc: a ``b200track.gmc.GmcEstimator`` for the source-frame size (BoT-SORT with camera-motion compensation, reference
        botsort.py:380-382): the warp of every sequence is estimated on the GPU from the uint8 frames and the NMS output and fed
        to the tracker step without leaving the device."""
        self.dets = list(detector) if isinstance(detector, (list, tuple)) else [detector]
        if len(self.dets) not in (1, 2):
            raise L.B2TError("TrackingPipeline takes one detector or two twins")
        self.det, self.eng, self.gmc = self.dets[0], engine, gmc
        det = self.det
        for d in self.dets:
            # the fused tracker kernel indexes the NMS output as [sequence][dmax][6]: the objects must agree on the layout
            if engine.S != d.B or engine.dmax != d.max_det or (d.B, d.H, d.W) != (det.B, det.H, det.W):
                raise L.B2TError("TrackEngine(n_seq=%d, dmax=%d) does not match DetectorW6(batch=%d, max_det=%d)" % (engine.S, engine.dmax, d.B, d.max_det))
        if gmc is not None and gmc.S != det.B:
            raise L.B2TError("GmcEstimator(n_seq=%d) does not match DetectorW6(batch=%d)" % (gmc.S, det.B))
        dev = det.dev
        self.dev = dev
        self.twin = len(self.dets) == 2
        self.s_copy, self.s_det, self.s_trk = (torch.cuda.Stream(device=dev) for _ in range(3))
        self.s_nms = torch.cuda.Stream(device=dev) if self.twin else self.s_det
        B = det.B
        self.t_out = torch.zeros((B, out_rows, L.OUT_COLS), dtype=torch.float64, device=dev)
        self.t_stat = torch.zeros((B, L.STAT_WORDS), dtype=torch.int32, device=dev)
        self.h_out = [torch.zeros((B, out_rows, L.OUT_COLS), dtype=torch.float64).pin_memory() for _ in range(2)]
        self.h_stat = [torch.zeros((B, L.STAT_WORDS), dtype=torch.int32).pin_memory() for _ in range(2)]
        nd = len(self.dets)
        ev = lambda: [torch.cuda.Event() for _ in range(nd)]                 # noqa: E731
        self.ev_src_free = ev()      # the ingest kernel has consumed det.src_u8 / det.img
        self.ev_in_ready = ev()      # the stem input of the detector is written
        self.ev_fwd_done = ev()      # the forward graph has finished (stem input consumed, head maps written)
        self.ev_nms_done = ev()      # det.out / det.out_count are written (head maps consumed)
        self.ev_out_free = ev()      # the tracker step has consumed det.out
        self.ev_trk_done = [torch.cuda.Event(), torch.cuda.Event()]
        self.g_fwd, self.g_nms = [None] * nd, [None] * nd
        self.n = 0
        self._capture()

    def _capture(self):
        # Collect dead objects first: an unreachable detector (its op closures hold it in a reference cycle) is otherwise freed by
        # whichever garbage collection happens to run next -- possibly inside a capture below, where its plans' cudaFree would
        # invalidate the graph.  torch.cuda.graph no longer collects on entry.
        gc.collect()
        torch.cuda.synchronize()
        for i, det in enumerate(self.dets):
            with torch.cuda.stream(self.s_det):
                det._forward_launches(); det._nms_launch(True)                    # warm-up (also sets kernel attributes)
                torch.cuda.synchronize()
                self.g_fwd[i] = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.g_fwd[i], stream=self.s_det):
                    for fn, _, name in det.ops[1:]:                               # ops[0] is the ReOrg that reads det.img
                        fn()
                self.g_nms[i] = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.g_nms[i], stream=self.s_det):
                    det._nms_launch(True)
            torch.cuda.synchronize()
            self.ev_src_free[i].record(self.s_copy)
            self.ev_fwd_done[i].record(self.s_det)
            self.ev_nms_done[i].record(self.s_nms)
            self.ev_out_free[i].record(self.s_trk)
        torch.cuda.synchronize()

    def step(self, frames, warps=None):
        """frames: one frame per sequence, pinned host tensor (copied on the copy stream) or device tensor, either
          * uint8 BGR (B, h, w, 3) as cv2.imread returns them -- the letterbox / RGB / 255 / ReOrg / fp16 conversion runs on the device
            (b2t_letterbox_reorg; call ``det.set_source_frames((h, w))`` once before, on every twin), 3 bytes per pixel over PCIe, or
          * float32 (B, 3, H, W) in [0, 1], the tensor the reference's dataloader produces.
        Returns (rows, stat) of the previous frame as pinned host tensors, or None on the first call."""
        eng = self.eng
        k = self.n & 1
        i = k if self.twin else 0
        det = self.dets[i]
        u8 = frames.dtype == torch.uint8
        if u8 and (getattr(det, "src_u8", None) is None or tuple(frames.shape) != tuple(det.src_u8.shape)):
            raise L.B2TError("uint8 frames of shape %s: call det.set_source_frames((h, w)) first" % (tuple(frames.shape),))
        # ---- input: copy once the previous ingest of this detector has read the staging buffer; the ingest kernel follows on the same
        # stream as soon as the detector's previous forward has consumed the stem input (twin mode) / on the detect stream (single)
        s_in = self.s_copy if self.twin else self.s_det
        with torch.cuda.stream(self.s_copy):
            self.s_copy.wait_event(self.ev_src_free[i])
            (det.src_u8 if u8 else det.img).copy_(frames, non_blocking=True)
            if not self.twin:
                self.ev_in_ready[i].record(self.s_copy)
        with torch.cuda.stream(s_in):
            if self.twin:
                s_in.wait_event(self.ev_fwd_done[i])
                if self.gmc is not None:
                    s_in.wait_event(self.ev_out_free[i])                       # the estimate of two frames ago has read this slot's planes
            else:
                s_in.wait_event(self.ev_in_ready[i])
            if u8:
                det.ingest_u8_launch()                                         # letterbox + RGB + /255 + ReOrg + 16-bit NHWC
                if self.gmc is not None:
                    self.gmc.prepare(det.src_u8, k)                            # gray / FAST scores / smoothed image while the frame buffer is valid
            else:
                det.ops[0][0]()                                                # ReOrg + 16-bit NHWC of the float tensor
            self.ev_src_free[i].record(s_in)
            if self.twin:
                self.ev_in_ready[i].record(s_in)
        # ---- detect
        with torch.cuda.stream(self.s_det):
            if self.twin:
                self.s_det.wait_event(self.ev_in_ready[i])
                self.s_det.wait_event(self.ev_nms_done[i])                     # this detector's head maps have been post-processed
            self.g_fwd[i].replay()
            self.ev_fwd_done[i].record(self.s_det)
        with torch.cuda.stream(self.s_nms):
            if self.twin:
                self.s_nms.wait_event(self.ev_fwd_done[i])
            self.s_nms.wait_event(self.ev_out_free[i])                         # the tracker step has read this detector's det.out
            self.g_nms[i].replay()
            self.ev_nms_done[i].record(self.s_nms)
        # ---- associate + read back
        with torch.cuda.stream(self.s_trk):
            self.s_trk.wait_event(self.ev_nms_done[i])
            if self.gmc is not None and u8:
                # key points outside the boxes of the high-score detections (botsort.py:380), matching, RANSAC -> warps on the device
                w23, _ = self.gmc.estimate_prepared(k, det.out, det.out_count, det_thresh=float(eng.cfg.conf_thresh))
                warps = w23.view(eng.S, 6)
            eng.step_device(det.out, det.out_count, self.t_out, self.t_stat, warps=warps)
            self.ev_out_free[i].record(self.s_trk)
            self.h_out[k].copy_(self.t_out, non_blocking=True)
            self.h_stat[k].copy_(self.t_stat, non_blocking=True)
            self.ev_trk_done[k].record(self.s_trk)
        self.n += 1
        if self.n == 1:
            return None
        return self._collect(1 - k)

    def _collect(self, k):
        self.ev_trk_done[k].synchronize()
        err = int(self.h_stat[k][:, L.STAT_ERR].max())
        if err:
            raise L.B2TError("tracker capacity error bits 0x%x (slots / detections / edges / output rows)" % err)
        return self.h_out[k], self.h_stat[k]

    def flush(self):
        """Tracks of the last submitted frame."""
        if self.n == 0:
            return None
        return self._collect((self.n - 1) & 1)
