"""Host side of the fused tracker: device memory, pinned staging and launches.

PyTorch is used for what it is good at here -- owning device memory, pinned host buffers and the
CUDA stream; all arithmetic happens in libb200track.so (csrc/b2t_step.cuh).  One ``TrackEngine``
advances ``n_seq`` independent video sequences per call, one CTA per sequence.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L


def _dev_ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class TrackEngine:
    def __init__(self, kind="bytetrack", n_seq=1, dtype="f64", cap=1024, dmax=1024, ecap=None, kalman_format=None,
                 conf_thresh=0.2, iou_thresh=0.5, track_buffer=30, frame_rate=30, use_gmc=True, device="cuda:0"):
        if not torch.cuda.is_available():
            raise L.B2TError("TrackEngine needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = L.load()
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if kind == "c_biou":
            # C-BIoU has no Kalman filter (the format is never read) and runs in float64 only, like the reference's buffered IoU
            kalman_format, dtype = "default", "f64"
        if kalman_format is None:
            kalman_format = "botsort" if kind == "botsort" else "default"      # track.py:68-69
        self.kind, self.kalman_format = kind, kalman_format
        self.dtype = L.F64 if dtype in ("f64", "float64", L.F64) and dtype != L.F32 else L.F32
        if ecap is None:
            ecap = 128 * max(cap, dmax)       # sub-threshold (track, detection) pairs per association: 2 MB of spill per sequence
        self.S, self.cap, self.dmax, self.ecap = n_seq, cap, dmax, ecap
        self.cfg = L.TrackerConfig(kind=L.KIND_BY_NAME[kind], dtype=self.dtype, fmt=L.FMT_BY_NAME[kalman_format],
                                   n_seq=n_seq, cap=cap, dmax=dmax, ecap=ecap, use_gmc=int(bool(use_gmc)),
                                   track_buffer=int(track_buffer), conf_thresh=float(conf_thresh),
                                   iou_thresh=float(iou_thresh), frame_rate=float(frame_rate))
        nbytes = self.lib.b2t_tracker_state_bytes(C.byref(self.cfg))
        if nbytes == 0:
            raise L.B2TError((self.lib.b2t_last_error() or b"").decode())
        with torch.cuda.device(self.device):
            self.state_mem = torch.zeros(nbytes + 256, dtype=torch.uint8, device=self.device)
            base = self.state_mem.data_ptr()
            self._state_ptr = base + ((-base) % 256)
            self.handle = C.c_void_p()
            L.check(self.lib, self.lib.b2t_tracker_create(C.byref(self.cfg), C.c_void_p(self._state_ptr),
                                                          self._stream(), C.byref(self.handle)))
        # pinned host staging (the e2e path copies these every step)
        self.h_dets = torch.zeros((n_seq, dmax, 6), dtype=torch.float32).pin_memory()
        self.h_count = torch.zeros(n_seq, dtype=torch.int32).pin_memory()
        self.h_warps = torch.zeros((n_seq, 6), dtype=torch.float64).pin_memory()
        self.h_idbase = torch.zeros(n_seq, dtype=torch.int32).pin_memory()
        self.h_out = torch.zeros((n_seq, cap, L.OUT_COLS), dtype=torch.float64).pin_memory()
        self.h_stat = torch.zeros((n_seq, L.STAT_WORDS), dtype=torch.int32).pin_memory()
        self.np_dets, self.np_count = self.h_dets.numpy(), self.h_count.numpy()
        self.np_warps, self.np_idbase = self.h_warps.numpy(), self.h_idbase.numpy()
        self.np_out, self.np_stat = self.h_out.numpy(), self.h_stat.numpy()
        self.out_rows = cap
        self.h2d_bytes_per_step = self.h_dets.numel() * 4 + self.h_count.numel() * 4
        self.d2h_bytes_per_step = 0

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.b2t_tracker_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def reset(self):
        L.check(self.lib, self.lib.b2t_tracker_reset(self.handle, self._stream()))

    def set_out_rows(self, rows):
        """Rows of output copied back per sequence per step (<= cap)."""
        self.out_rows = int(min(max(rows, 1), self.cap))

    # ---- host-buffer path: what a caller with NumPy / CPU detections uses (and what e2e times)
    def load_dets(self, dets_list):
        """Fill the pinned staging buffers from per-sequence (n_i, 6) float32 arrays."""
        for s, a in enumerate(dets_list):
            a = np.asarray(a, dtype=np.float32).reshape(-1, 6)
            n = a.shape[0]
            if n > self.dmax:
                raise L.B2TError("sequence %d: %d detections > dmax=%d" % (s, n, self.dmax))
            self.np_dets[s, :n] = a
            self.np_count[s] = n

    def step_host(self, warps=None, id_base=None, predict_only=False):
        """H2D copy of the staged detections, one fused launch, D2H of tracks + stats, sync."""
        w = ib = None
        if warps is not None:
            self.np_warps[:] = np.asarray(warps, dtype=np.float64).reshape(self.S, 6)
            w = C.c_void_p(self.h_warps.data_ptr())
        if id_base is not None:
            self.np_idbase[:] = np.asarray(id_base, dtype=np.int32)
            ib = C.c_void_p(self.h_idbase.data_ptr())
        with torch.cuda.device(self.device):
            rc = self.lib.b2t_tracker_step_host(self.handle, C.c_void_p(self.h_dets.data_ptr()),
                                                C.c_void_p(self.h_count.data_ptr()), w, ib,
                                                C.c_void_p(self.h_out.data_ptr()), self.out_rows,
                                                C.c_void_p(self.h_stat.data_ptr()), int(predict_only), self._stream())
        L.check(self.lib, rc)
        self.d2h_bytes_per_step = self.S * (self.out_rows * L.OUT_COLS * 8 + L.STAT_WORDS * 4)
        return self.results()

    def step_cuda_dets(self, dets_list, warps=None, id_base=None):
        """Detections that already live on THIS device (the NMS output tracker/track.py:151 hands to tracker.update): no host round
        trip of the boxes.  dets_list: per sequence an (n_i, 6) float32 CUDA tensor.  The rows are copied device-to-device into the
        kernel's [sequence][dmax][6] layout, the counts / id base / warps (a few bytes) go up from pinned memory, the fused kernel
        runs, track rows + stats come back asynchronously and ONE stream synchronisation ends the call (the API returns Python
        objects).  Same results as step(); 24 B + 24 KB... less traffic and one sync instead of three."""
        if not hasattr(self, "d_dets"):
            self.d_dets = torch.zeros((self.S, self.dmax, 6), dtype=torch.float32, device=self.device)
            self.d_count = torch.zeros(self.S, dtype=torch.int32, device=self.device)
            self.d_idbase = torch.zeros(self.S, dtype=torch.int32, device=self.device)
            self.d_warps = torch.zeros((self.S, 6), dtype=torch.float64, device=self.device)
            self.d_out = torch.zeros((self.S, self.cap, L.OUT_COLS), dtype=torch.float64, device=self.device)
            self.d_stat = torch.zeros((self.S, L.STAT_WORDS), dtype=torch.int32, device=self.device)
        for s, d in enumerate(dets_list):
            n = int(d.shape[0])
            if n > self.dmax:
                raise L.B2TError("sequence %d: %d detections > dmax=%d" % (s, n, self.dmax))
            if d.device != self.device:
                raise L.B2TError("step_cuda_dets: detections live on %s, the engine on %s" % (d.device, self.device))
            if n:
                self.d_dets[s, :n].copy_(d.detach().reshape(n, 6).to(torch.float32), non_blocking=True)
            self.np_count[s] = n
        self.d_count.copy_(self.h_count, non_blocking=True)
        w = ib = None
        if warps is not None:
            self.np_warps[:] = np.asarray(warps, dtype=np.float64).reshape(self.S, 6)
            self.d_warps.copy_(self.h_warps, non_blocking=True)
            w = self.d_warps
        if id_base is not None:
            self.np_idbase[:] = np.asarray(id_base, dtype=np.int32)
            self.d_idbase.copy_(self.h_idbase, non_blocking=True)
            ib = self.d_idbase
        rows = self.out_rows
        out = self.d_out[:, :rows] if rows == self.cap else self.d_out.view(-1)[: self.S * rows * L.OUT_COLS].view(self.S, rows, L.OUT_COLS)
        self.step_device(self.d_dets, self.d_count, out, self.d_stat, warps=w, id_base=ib)
        self.h_out.view(-1)[: self.S * rows * L.OUT_COLS].copy_(out.reshape(-1), non_blocking=True)
        self.h_stat.copy_(self.d_stat, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        err = int(self.np_stat[:, L.STAT_ERR].max())
        if err:
            raise L.B2TError("b2t_tracker_step: capacity exceeded (cap / dmax / ecap / out rows), stat[STAT_ERR] = 0x%x" % err)
        return self.results()

    def results(self):
        out = self.np_out.reshape(-1)[: self.S * self.out_rows * L.OUT_COLS].reshape(self.S, self.out_rows, L.OUT_COLS)
        return [out[s, : self.np_stat[s, L.STAT_NOUT]] for s in range(self.S)]

    def step(self, dets_list, warps=None, id_base=None, predict_only=False):
        if not predict_only:
            self.load_dets(dets_list)
        return self.step_host(warps, id_base, predict_only)

    # ---- device-pointer path: detections already resident (detector output), no sync
    def step_device(self, dets, det_count, out, stat, warps=None, id_base=None, predict_only=False):
        """dets (S,dmax,6) f32, det_count (S) i32, out (S,rows,8) f64, stat (S,64) i32: contiguous CUDA tensors on this engine's
        device.  The kernel indexes them as raw [sequence][dmax][6] / [sequence][rows][8] arrays: the layout is checked here."""
        def _chk(t, shape, dtype, what):
            if t is None:
                return
            if tuple(t.shape) != shape or t.dtype != dtype or not t.is_cuda or not t.is_contiguous() or t.device != self.device:
                raise L.B2TError("step_device: %s must be a contiguous %s CUDA tensor of shape %s on %s, got %s %s on %s" %
                                 (what, dtype, shape, self.device, tuple(t.shape), t.dtype, t.device))
        _chk(dets, (self.S, self.dmax, 6), torch.float32, "dets")
        _chk(det_count, (self.S,), torch.int32, "det_count")
        if out.dim() != 3 or out.shape[0] != self.S or out.shape[2] != L.OUT_COLS:
            raise L.B2TError("step_device: out must be (%d, rows, %d), got %s" % (self.S, L.OUT_COLS, tuple(out.shape)))
        _chk(out, (self.S, int(out.shape[1]), L.OUT_COLS), torch.float64, "out")
        _chk(stat, (self.S, L.STAT_WORDS), torch.int32, "stat")
        _chk(warps, (self.S, 6), torch.float64, "warps")
        _chk(id_base, (self.S,), torch.int32, "id_base")
        with torch.cuda.device(self.device):
            rc = self.lib.b2t_tracker_step(self.handle, _dev_ptr(dets), _dev_ptr(det_count), _dev_ptr(warps),
                                           _dev_ptr(id_base), _dev_ptr(out), int(out.shape[1]), _dev_ptr(stat),
                                           int(predict_only), self._stream())
        L.check(self.lib, rc)

    def read_list(self, seq, which="tracked"):
        """(n, 13) float64 rows of the sequence's tracked / lost list in the reference's list order: id, tlwh, cls, score, slot,
        state, is_activated, tracklet_len, start_frame, frame_id (b2t_tracker_read_list)."""
        rows = np.zeros((self.cap, 13))
        n = C.c_int(0)
        with torch.cuda.device(self.device):
            rc = self.lib.b2t_tracker_read_list(self.handle, int(seq), 0 if which == "tracked" else 1, rows.ctypes.data_as(C.c_void_p), self.cap,
                                                C.byref(n), self._stream())
        L.check(self.lib, rc)
        return rows[:n.value].copy()

    def read_slot(self, seq, slot):
        """The slot's 72-double record as (mean[8], cov[8, 8]): the Kalman state, or for kind c_biou the record documented in
        csrc/b2t_cbiou.cuh (see cbiou_record)."""
        mean = np.zeros(8); cov = np.zeros((8, 8))
        with torch.cuda.device(self.device):
            rc = self.lib.b2t_tracker_read_slot(self.handle, int(seq), int(slot), mean.ctypes.data_as(C.c_void_p),
                                                cov.ctypes.data_as(C.c_void_p), self._stream())
        L.check(self.lib, rc)
        return mean, cov

    def cbiou_record(self, seq, slot):
        """Kind c_biou: the slot's record as a dict -- history (n, 4) tlwh oldest first, motion_state1 / motion_state2 (4,) tlwh,
        time_since_update -- float32 boxes as the reference keeps them."""
        mean, cov = self.read_slot(seq, slot)
        r = np.concatenate([mean, cov.reshape(-1)])
        n = int(r[0])
        return dict(history=r[8:8 + 4 * n].reshape(n, 4).astype(np.float32), motion_state1=r[32:36].astype(np.float32),
                    motion_state2=r[36:40].astype(np.float32), time_since_update=int(r[1]))


# ------------------------------------------------------------------ op-level helpers (device tensors)
def _tdt(dtype):
    return torch.float64 if dtype == L.F64 else torch.float32


class Ops:
    """Thin wrappers over the op-level C ABI for CUDA tensors (used by the drop-in modules)."""

    def __init__(self, device="cuda:0"):
        if not torch.cuda.is_available():
            raise L.B2TError("libb200track ops need a CUDA device; there is no CPU fallback")
        self.lib = L.load()
        self.device = torch.device(device)

    def _s(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def dev(self, a, dtype):
        return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(self.device, non_blocking=False).contiguous()

    def kalman_initiate(self, dtype, fmt, meas):
        k = meas.shape[0]
        mean = torch.empty((k, 8), dtype=_tdt(dtype), device=self.device)
        cov = torch.empty((k, 8, 8), dtype=_tdt(dtype), device=self.device)
        L.check(self.lib, self.lib.b2t_kalman_initiate(dtype, fmt, _dev_ptr(meas), _dev_ptr(mean), _dev_ptr(cov), k, self._s()))
        return mean, cov

    def kalman_predict(self, dtype, fmt, mean, cov, flags=None, q_f32=False):
        L.check(self.lib, self.lib.b2t_kalman_predict(dtype, fmt, _dev_ptr(mean), _dev_ptr(cov), _dev_ptr(flags),
                                                      mean.shape[0], int(q_f32), self._s()))

    def kalman_project(self, dtype, fmt, mean, cov, flags=None, conf=None):
        n = mean.shape[0]
        pm = torch.empty((n, 4), dtype=_tdt(dtype), device=self.device)
        ps = torch.empty((n, 4, 4), dtype=_tdt(dtype), device=self.device)
        L.check(self.lib, self.lib.b2t_kalman_project(dtype, fmt, _dev_ptr(mean), _dev_ptr(cov), _dev_ptr(flags),
                                                      _dev_ptr(conf), _dev_ptr(pm), _dev_ptr(ps), n, self._s()))
        return pm, ps

    def kalman_update(self, dtype, fmt, mean, cov, meas, idx=None, conf=None, flags=None):
        L.check(self.lib, self.lib.b2t_kalman_update(dtype, fmt, _dev_ptr(mean), _dev_ptr(cov), _dev_ptr(idx), _dev_ptr(meas),
                                                     _dev_ptr(conf), _dev_ptr(flags), meas.shape[0], self._s()))

    def kalman_gating(self, dtype, fmt, mean, cov, meas, only_position=False, metric=0):
        m = meas.shape[0]
        out = torch.empty(m, dtype=_tdt(dtype), device=self.device)
        L.check(self.lib, self.lib.b2t_kalman_gating(dtype, fmt, _dev_ptr(mean), _dev_ptr(cov), _dev_ptr(meas), m,
                                                     int(only_position), int(metric), _dev_ptr(out), self._s()))
        return out

    def gmc_apply(self, dtype, mean, cov, warp):
        w6 = (C.c_double * 6)(*np.asarray(warp, dtype=np.float64).reshape(-1)[:6])
        L.check(self.lib, self.lib.b2t_gmc_apply(dtype, _dev_ptr(mean), _dev_ptr(cov), mean.shape[0], w6, self._s()))

    def iou_cost(self, dtype, a, b, as_distance=True, out=None):
        """a (B,n,4) / (n,4), b (B,m,4) / (m,4) CUDA tensors -> cost (B,n,m) / (n,m)."""
        batched = a.dim() == 3
        a3, b3 = (a, b) if batched else (a[None], b[None])
        bsz, n, m = a3.shape[0], a3.shape[1], b3.shape[1]
        if out is None:
            out = torch.empty((bsz, n, m), dtype=_tdt(dtype), device=self.device)
        L.check(self.lib, self.lib.b2t_iou_cost(dtype, _dev_ptr(a3), n, _dev_ptr(b3), m, _dev_ptr(out), max(m, 1), bsz,
                                                int(as_distance), self._s()))
        return out if batched else out[0]

    def lap_workspace(self, dtype, n, m, batch=1):
        nbytes = self.lib.b2t_lap_workspace_bytes(dtype, n, m, batch)
        return torch.empty(nbytes + 256, dtype=torch.uint8, device=self.device)

    def lap_solve(self, dtype, cost, thresh, workspace=None):
        batched = cost.dim() == 3
        c3 = cost if batched else cost[None]
        bsz, n, m = c3.shape
        x = torch.empty((bsz, n), dtype=torch.int32, device=self.device)
        y = torch.empty((bsz, m), dtype=torch.int32, device=self.device)
        if workspace is None:
            workspace = self.lap_workspace(dtype, n, m, bsz)
        L.check(self.lib, self.lib.b2t_lap_solve(dtype, _dev_ptr(c3), n, m, max(m, 1), float(thresh), _dev_ptr(x), _dev_ptr(y),
                                                 _dev_ptr(workspace), workspace.numel(), bsz, self._s()))
        return (x, y) if batched else (x[0], y[0])


_ops = None


def ops():
    global _ops
    if _ops is None:
        _ops = Ops()
    return _ops
