"""Drop-in for the reference's ``tracker/c_biou_tracker.py``: ``C_BIoUTracker(opts, frame_rate=30)`` with
``update(det_results, ori_img) -> list of tracks`` (reference :218-353), executed as one fused kernel per frame
(csrc/b2t_cbiou.cuh, kind = c_biou, float64).

C-BIoU (cascaded buffered IoU) has no Kalman filter: a track keeps its last matched boxes and two "motion states", boxes
enlarged by the buffer scales b1 = 0.3 and b2 = 0.5 and extrapolated over missed frames; a frame is three IoU associations on
those buffered boxes followed by ByteTrack's list algebra.  ``opts.kalman_format`` is never read.  Lost tracks are never pruned
(as in the reference): ``opts.b2t_cap`` (default 1024 slots) bounds the tracked + lost tracks of a whole sequence, and running out
raises ``B2TError`` instead of dropping tracks.

``C_BIoUSTrack`` is also a complete stand-alone track (NumPy float32 state) for code that drives tracks one by one.
"""
import numpy as np

import _b2t_path  # noqa: F401
from basetrack import (TrackState, BaseTrack, BaseTracker, _TrackView,  # noqa: F401
                       joint_stracks, sub_stracks, remove_duplicate_stracks)
from b200track import _lib as L

_B1, _B2, _N = 0.3, 0.5, 5


def _buffer(tlwh, b):
    """Box enlarged by b of its size on every side, clipped at 0, in float32 (get_buffer_bbox, :48-62)."""
    t = np.asarray(tlwh, dtype=np.float32)
    grow = np.array([np.float32(-b) * t[2], np.float32(-b) * t[3], np.float32(2 * b) * t[2], np.float32(2 * b) * t[3]], np.float32)
    return np.maximum(np.float32(0), t + grow)


class C_BIoUSTrack(BaseTrack):
    def __init__(self, cls, tlwh, score):
        super().__init__()
        self.cls = cls
        self._tlwh = np.asarray(tlwh, dtype=np.float32)
        self.score = score
        self.is_activated = False
        self.tracklet_len = 0
        self.track_id = None
        self.start_frame = None
        self.frame_id = None
        self.time_since_update = 0
        self.b1, self.b2, self.n = _B1, _B2, _N
        self.origin_bbox_buffer = [self._tlwh]          # the last matched boxes, oldest first, at most n + 1
        self.buffer_bbox1 = self.get_buffer_bbox(level=1)
        self.buffer_bbox2 = self.get_buffer_bbox(level=2)
        self.motion_state1 = self.buffer_bbox1.copy()
        self.motion_state2 = self.buffer_bbox2.copy()

    def get_buffer_bbox(self, level=1, bbox=None):
        assert level in (1, 2), 'level must be 1 or 2'
        return _buffer(self._tlwh if bbox is None else bbox, self.b1 if level == 1 else self.b2)

    @property
    def tlwh(self):
        return np.array(self.origin_bbox_buffer[-1], dtype=np.float32)

    @property
    def tlbr(self):
        return self.tlwh2tlbr(self.tlwh)

    def _push(self, box):
        if len(self.origin_bbox_buffer) > self.n:
            self.origin_bbox_buffer.pop(0)
        self.origin_bbox_buffer.append(box)

    def activate(self, frame_id):
        self.track_id = BaseTrack.next_id()
        self.state = TrackState.Tracked
        if frame_id == 1:
            self.is_activated = True
        self.frame_id = frame_id
        self.start_frame = frame_id

    def re_activate(self, new_track, frame_id, new_id=False):
        # time_since_update is kept on purpose, as the reference does: the next update() extrapolates with it
        self.tracklet_len = 0
        self.state = TrackState.Tracked
        self.is_activated = True
        self.frame_id = frame_id
        if new_id:
            self.track_id = self.next_id()
        self.score = new_track.score
        self._tlwh = new_track._tlwh
        self._push(self._tlwh)
        self.buffer_bbox1 = self.get_buffer_bbox(level=1)
        self.buffer_bbox2 = self.get_buffer_bbox(level=2)
        self.motion_state1 = self.buffer_bbox1.copy()
        self.motion_state2 = self.buffer_bbox2.copy()

    def update(self, new_track, frame_id):
        self.frame_id = frame_id
        self.tracklet_len += 1
        box = new_track.tlwh
        self._tlwh = box
        self.score = new_track.score
        self._push(box)
        src = box
        if self.time_since_update and len(self.origin_bbox_buffer) >= self.n:
            last, first = self.origin_bbox_buffer[-1], self.origin_bbox_buffer[0]
            src = last + np.float32(self.time_since_update / self.n) * (last - first)
        self.motion_state1 = self.get_buffer_bbox(level=1, bbox=src)
        self.motion_state2 = self.get_buffer_bbox(level=2, bbox=src)
        self.state = TrackState.Tracked
        self.is_activated = True
        self.time_since_update = 0

    @staticmethod
    def tlbr2tlwh(tlbr):
        r = np.asarray(tlbr).copy()
        r[..., 2:] -= r[..., :2]
        return r

    @staticmethod
    def tlwh2tlbr(tlwh):
        r = np.asarray(tlwh).copy()
        r[..., 2:] += r[..., :2]
        return r

    @staticmethod
    def xywh2tlwh(xywh):
        r = np.asarray(xywh).copy()
        r[..., :2] -= r[..., 2:] // 2
        return r

    @staticmethod
    def xywh2tlbr(xywh):
        r = C_BIoUSTrack.xywh2tlwh(xywh)
        r[..., 2:] = r[..., :2] + r[..., 2:]
        return np.maximum(0.0, r)


class _CBIoUView(_TrackView):
    """A track of the fused C-BIoU kernel.  ``tlwh`` is the last matched detection box; ``motion_state1 / 2``, ``time_since_update``
    (and, for returned tracks, ``tracklet_len`` / ``start_frame``) are read from the slot on first access, in the frame the track
    was returned; ``buffer_bbox1 / 2`` are computed here from ``tlwh``."""

    def __init__(self, engine, seq, row, frame_id, extra=None):
        self._lazy = {}
        super().__init__(engine, seq, row, 'default', frame_id, extra=extra)
        if extra is None:                                   # output rows carry no list metadata
            self._lazy.pop('tracklet_len', None)
            self._lazy.pop('start_frame', None)

    def _check_frame(self):
        if self._engine.np_stat[self._seq, L.STAT_FRAME] != self._view_frame:
            raise RuntimeError("track %d: the slot was not read at frame %d and the tracker has moved on: read it in the frame the "
                               "track was returned" % (self.track_id, self._view_frame))

    def _record(self):
        if 'record' not in self._lazy:
            self._check_frame()
            self._lazy['record'] = self._engine.cbiou_record(self._seq, self._slot)
        return self._lazy['record']

    def _meta(self, name):
        if name not in self._lazy:
            self._check_frame()
            row = next(r for r in self._engine.read_list(self._seq, 'tracked') if int(r[7]) == self._slot)
            self._lazy['tracklet_len'], self._lazy['start_frame'] = int(row[10]), int(row[11])
        return self._lazy[name]

    tracklet_len = property(lambda self: self._meta('tracklet_len'), lambda self, v: self._lazy.__setitem__('tracklet_len', v))
    start_frame = property(lambda self: self._meta('start_frame'), lambda self, v: self._lazy.__setitem__('start_frame', v))
    time_since_update = property(lambda self: self._record()['time_since_update'], lambda self, v: None)
    motion_state1 = property(lambda self: self._record()['motion_state1'].copy())
    motion_state2 = property(lambda self: self._record()['motion_state2'].copy())
    buffer_bbox1 = property(lambda self: _buffer(self.tlwh, _B1))
    buffer_bbox2 = property(lambda self: _buffer(self.tlwh, _B2))
    kalman = None

    @property
    def tlwh(self):
        return self._row[1:5].astype(np.float32)

    @property
    def tlbr(self):
        return C_BIoUSTrack.tlwh2tlbr(self.tlwh)


class C_BIoUTracker(BaseTracker):
    """``update`` == reference c_biou_tracker.py:218-353, executed by the fused kernel (kind c_biou, float64)."""
    _kind = 'c_biou'

    def __init__(self, opts, frame_rate=30, *args, **kwargs):
        super().__init__(opts, frame_rate, *args, **kwargs)
        self.kalman = None

    def _get_engine(self):
        if self._engine is None:
            from b200track.engine import TrackEngine
            kw = dict(self._engine_kw, dtype='f64')
            self._engine = TrackEngine(kind='c_biou', n_seq=1, conf_thresh=self.opts.conf_thresh, track_buffer=self.opts.track_buffer,
                                       frame_rate=self._frame_rate, use_gmc=False, **kw)
        return self._engine

    def _views(self, which):
        rows = self._engine.read_list(0, which)
        return [_CBIoUView(self._engine, 0, r, self.frame_id, extra=r[8:13]) for r in rows]

    def update(self, det_results, ori_img):
        self._step(det_results, ori_img)
        self._last = [_CBIoUView(v._engine, 0, v._row, self.frame_id) for v in self._last]
        return list(self._last)

    def update_without_detection(self, det_results, ori_img):
        # the reference inherits BaseTracker.update_without_detection (basetrack.py:489-537), which predicts every confirmed and lost
        # track with STrack.multi_predict(kalman=None) and fails as soon as one exists
        raise NotImplementedError("C_BIoUTracker.update_without_detection: C-BIoU has no Kalman filter to predict with")
