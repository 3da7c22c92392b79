"""Oracle: the C-BIoU tracker of the reference (``C_BIoUTracker.update``, tracker/c_biou_tracker.py:218-353).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Restates, on slot-indexed records and index lists (the layout the CUDA kernel
csrc/b2t_cbiou.cuh uses), the cascaded buffered-IoU tracker: no Kalman filter, three IoU associations on buffered boxes, then
ByteTrack's list algebra.  Box arithmetic is float32 with every operation rounded, as NumPy 2 does it on the reference's float32
arrays; the IoU is the float64 "+1" IoU of oracle/iou.py.  The quirks are kept on purpose: ``re_activate`` does not reset
``time_since_update``; lost tracks are never pruned; ``cls`` is never updated.  Pinned against the reference class itself run
through oracle/refshim.py (tests/golden/loop_c_biou.npz).
"""
import numpy as np

from .iou import iou_distance_tlbr
from .lapjv import linear_assignment
from .trackers import IdCounter, NEW, TRACKED, LOST, REMOVED  # noqa: F401

F32 = np.float32
B1, B2, N_HIST = 0.3, 0.5, 5


def buffered(tlwh, b):
    """get_buffer_bbox (:48-62): max(0, tlwh + [-b w, -b h, 2b w, 2b h]) in float32."""
    t = np.asarray(tlwh, dtype=F32)
    nb, b2 = F32(-b), F32(2 * b)
    r = np.array([t[0] + nb * t[2], t[1] + nb * t[3], t[2] + b2 * t[2], t[3] + b2 * t[3]], dtype=F32)
    return np.maximum(F32(0), r)


def tlwh_to_tlbr(tlwh):
    r = np.asarray(tlwh, dtype=F32).copy()
    r[2:] += r[:2]
    return r


class _Trk:
    __slots__ = ("tid", "state", "activated", "tracklet_len", "start_frame", "frame_id", "cls", "score", "hist", "ms1", "ms2",
                 "tsu", "removed_at")


class CBIoUOracle:
    def __init__(self, conf_thresh=0.2, track_buffer=30, frame_rate=30, ids=None):
        self.det_thresh = conf_thresh                                   # basetrack.py:354
        self.max_time_lost = int(frame_rate / 30.0 * track_buffer)     # basetrack.py:355-356
        self.ids = ids if ids is not None else IdCounter()
        self.frame_id = 0
        self.trk = {}
        self._next_slot = 0
        self.tracked, self.lost = [], []
        self.removed_ids = set()

    # ------------------------------------------------------------------ track life cycle
    def _append(self, t, box):
        if len(t.hist) > N_HIST:
            t.hist.pop(0)
        t.hist.append(box)

    def _update(self, s, box, score, f):                    # C_BIoUSTrack.update, :114-152
        t = self.trk[s]
        t.frame_id = f
        t.tracklet_len += 1
        t.score = score
        self._append(t, box)
        src = box
        if t.tsu and len(t.hist) >= N_HIST:
            o = t.hist
            src = o[-1] + F32(t.tsu / N_HIST) * (o[-1] - o[0])
        t.ms1, t.ms2 = buffered(src, B1), buffered(src, B2)
        t.state, t.activated = TRACKED, True
        t.tsu = 0

    def _re_activate(self, s, box, score, f):               # C_BIoUSTrack.re_activate, :89-112 (keeps tsu)
        t = self.trk[s]
        t.tracklet_len = 0
        t.state, t.activated = TRACKED, True
        t.frame_id = f
        t.score = score
        self._append(t, box)
        t.ms1, t.ms2 = buffered(box, B1), buffered(box, B2)

    def _birth(self, box, score, cls, f):                   # C_BIoUSTrack.__init__ + activate, :18-46, :76-87
        t = _Trk()
        t.tid = self.ids.next_id()
        t.state = TRACKED
        t.activated = f == 1
        t.tracklet_len = 0
        t.start_frame = t.frame_id = f
        t.cls, t.score = cls, score
        t.hist = [box]
        t.ms1, t.ms2 = buffered(box, B1), buffered(box, B2)
        t.tsu = 0
        t.removed_at = None
        s = self._next_slot
        self._next_slot += 1
        self.trk[s] = t
        return s

    def _ms_tlbr(self, slots, level):
        out = np.zeros((len(slots), 4), dtype=np.float64)
        for k, s in enumerate(slots):
            t = self.trk[s]
            out[k] = tlwh_to_tlbr(t.ms1 if level == 1 else t.ms2)
        return out

    # ------------------------------------------------------------------ one frame
    def update(self, dets):
        trk = self.trk
        self.frame_id += 1
        f = self.frame_id
        dets = np.asarray(dets, dtype=np.float32).reshape(-1, 6)
        keep = np.nonzero(dets[:, 4] > F32(self.det_thresh))[0]                  # :238
        tlwh = dets[:, :4].copy()
        tlwh[:, 2:] -= tlwh[:, :2]                                              # tlbr2tlwh, float32
        sc = dets[:, 4]
        buf1 = np.array([tlwh_to_tlbr(buffered(tlwh[d], B1)) for d in range(len(dets))], np.float64).reshape(-1, 4)
        buf2 = np.array([tlwh_to_tlbr(buffered(tlwh[d], B2)) for d in range(len(dets))], np.float64).reshape(-1, 4)

        unconfirmed = [s for s in self.tracked if not trk[s].activated]
        confirmed = [s for s in self.tracked if trk[s].activated]
        have = {trk[s].tid for s in confirmed}
        pool = confirmed + [s for s in self.lost if trk[s].tid not in have]      # joint_stracks
        refind, births, lost_now, removed_now = [], [], [], []

        # stage 1: pool motion_state1 x level-1 buffers, 0.9
        m0, ut0, ud0 = linear_assignment(iou_distance_tlbr(self._ms_tlbr(pool, 1), buf1[keep]), 0.9)
        for it, idt in m0:
            s, d = pool[it], keep[idt]
            if trk[s].state == TRACKED:
                self._update(s, tlwh[d], sc[d], f)
            else:
                self._re_activate(s, tlwh[d], sc[d], f)
                refind.append(s)
        u_tracks0 = [pool[i] for i in ut0 if trk[pool[i]].state == TRACKED]
        u_dets0 = [keep[i] for i in ud0]

        # stage 2: Tracked leftovers, motion_state2 x level-2 buffers, 0.5
        m1, ut1, ud1 = linear_assignment(iou_distance_tlbr(self._ms_tlbr(u_tracks0, 2), buf2[u_dets0].reshape(-1, 4)), 0.5)
        for it, idt in m1:
            self._update(u_tracks0[it], tlwh[u_dets0[idt]], sc[u_dets0[idt]], f)
        u_tracks1 = [u_tracks0[i] for i in ut1]
        u_dets1 = [u_dets0[i] for i in ud1]

        # stage 3': unconfirmed, motion_state1 x level-1 buffers, 0.7
        m2, ut2, ud2 = linear_assignment(iou_distance_tlbr(self._ms_tlbr(unconfirmed, 1), buf1[u_dets1].reshape(-1, 4)), 0.7)
        for it, idt in m2:
            self._update(unconfirmed[it], tlwh[u_dets1[idt]], sc[u_dets1[idt]], f)
        for it in ut2:
            trk[unconfirmed[it]].state = REMOVED
            removed_now.append(unconfirmed[it])
        for i in ud2:
            d = u_dets1[i]
            if sc[d] > F32(self.det_thresh + 0.1):
                births.append(self._birth(tlwh[d], sc[d], dets[d, 5], f))

        # step 4: only tracks that were Tracked at frame start; the lost list is never pruned
        for s in u_tracks1:
            t = trk[s]
            if f - t.frame_id > self.max_time_lost:
                t.state = REMOVED
                removed_now.append(s)
            else:
                t.state = LOST
                t.tsu = f - t.frame_id
                lost_now.append(s)

        active = self._finish(lost_now, removed_now, births, refind)
        return [(trk[s].tid, np.asarray(trk[s].hist[-1], np.float64), float(trk[s].cls), float(trk[s].score)) for s in active]

    def _finish(self, lost_now, removed_now, births, refind):
        trk = self.trk
        tracked = [s for s in self.tracked if trk[s].state == TRACKED]
        have = {trk[s].tid for s in tracked}
        for s in births + refind:                           # joint_stracks x2
            if trk[s].tid not in have:
                have.add(trk[s].tid)
                tracked.append(s)
        lost, seen = [], set()
        for s in self.lost:                                 # sub_stracks(lost, tracked)
            tid = trk[s].tid
            if tid not in seen:
                seen.add(tid)
                if tid not in have:
                    lost.append(s)
        lost = lost + lost_now
        out, seen = [], set()
        for s in lost:                                      # sub_stracks(lost, removed list of earlier frames)
            tid = trk[s].tid
            if tid not in seen:
                seen.add(tid)
                if tid not in self.removed_ids:
                    out.append(s)
        lost = out
        for s in removed_now:
            self.removed_ids.add(trk[s].tid)
        if tracked and lost:                                # remove_duplicate_stracks on the last original boxes
            a = np.array([tlwh_to_tlbr(trk[s].hist[-1]) for s in tracked], np.float64)
            b = np.array([tlwh_to_tlbr(trk[s].hist[-1]) for s in lost], np.float64)
            pd = iou_distance_tlbr(a, b)
            dupa, dupb = set(), set()
            for p, q in zip(*np.where(pd < 0.15)):
                tp = trk[tracked[p]].frame_id - trk[tracked[p]].start_frame
                tq = trk[lost[q]].frame_id - trk[lost[q]].start_frame
                if tp > tq:
                    dupb.add(q)
                else:
                    dupa.add(p)
            tracked = [s for i, s in enumerate(tracked) if i not in dupa]
            lost = [s for i, s in enumerate(lost) if i not in dupb]
        self.tracked, self.lost = tracked, lost
        live = set(tracked) | set(lost)
        for s in list(trk):
            if s not in live:
                del trk[s]
        return [s for s in tracked if trk[s].activated]

    def record(self, slot):
        """The slot's state the way b2t_tracker_read_slot reports it for C-BIoU (csrc/b2t_cbiou.cuh)."""
        t = self.trk[slot]
        return dict(history=np.array(t.hist, np.float32), motion_state1=t.ms1, motion_state2=t.ms2, time_since_update=t.tsu)
