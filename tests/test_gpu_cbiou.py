"""-m gpu: the fused C-BIoU kernel (csrc/b2t_cbiou.cuh) on the B200 against the reference goldens (tests/golden/loop_c_biou.npz) and
the oracle (oracle/cbiou.py); the drop-in ``C_BIoUTracker`` in the reference driver's per-frame body (tracker/track.py:138-179); and
``TrackingPipeline`` with a c_biou engine."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from b200track import _lib as L  # noqa: E402
from b200track.synth import make_stream, make_vanish_stream  # noqa: E402
from oracle import cbiou as CB  # noqa: E402
from oracle.trackers import IdCounter  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "yolov7-tracker_b200")
GOLDEN = os.path.join(ROOT, "tests", "golden", "loop_c_biou.npz")


def _engine(**kw):
    from b200track.engine import TrackEngine
    return TrackEngine("c_biou", device="cuda:0", **kw)


@pytest.mark.parametrize("case", ["small", "c3", "vanish"])
def test_gpu_cbiou_matches_reference_golden(case):
    g = np.load(GOLDEN)
    seed, n_obj, n_frames = [int(v) for v in g[case + "_cfg"]]
    frames = make_vanish_stream(seed, n_frames) if case == "vanish" else make_stream(seed, n_frames, n_obj)[0]
    eng = _engine(cap=1024, dmax=1024)
    assert eng.dtype == L.F64
    off = np.concatenate([[0], np.cumsum(g[case + "_count"])])
    rec_frames = [int(v) for v in g[case + "_rec_frames"]]
    roff = np.concatenate([[0], np.cumsum(g[case + "_rec_count"])])
    for i, f in enumerate(frames):
        r = eng.step([f])[0]
        sl = slice(off[i], off[i + 1])
        assert np.array_equal(r[:, 0].astype(np.int64), g[case + "_ids"][sl]), "track ids differ at frame %d" % (i + 1)
        assert np.array_equal(r[:, 1:5], g[case + "_tlwh"][sl].astype(np.float64)), "boxes differ at frame %d" % (i + 1)
        assert np.array_equal(r[:, 5].astype(np.float32), g[case + "_cls"][sl])
        assert eng.np_stat[0, L.STAT_NTRACKED] == g[case + "_ntracked"][i] and eng.np_stat[0, L.STAT_NLOST] == g[case + "_nlost"][i]
        if i in rec_frames:
            k = rec_frames.index(i)
            rs = slice(roff[k], roff[k + 1])
            rows = eng.read_list(0, "tracked")
            assert np.array_equal(rows[:, 0].astype(np.int64), g[case + "_rec_ids"][rs])
            recs = [eng.cbiou_record(0, s) for s in rows[:, 7]]
            assert np.array_equal(np.array([x["motion_state1"] for x in recs]).reshape(-1, 4), g[case + "_rec_ms1"][rs])
            assert np.array_equal(np.array([x["motion_state2"] for x in recs]).reshape(-1, 4), g[case + "_rec_ms2"][rs])
            assert [x["time_since_update"] for x in recs] == g[case + "_rec_tsu"][rs].tolist()


def test_gpu_cbiou_four_sequences_one_launch():
    streams = [make_stream(100 + s, 40, 60 + 40 * s)[0] for s in range(3)] + [make_vanish_stream(104, 40)]
    eng = _engine(n_seq=4, cap=512, dmax=512)
    orcs = [CB.CBIoUOracle() for _ in range(4)]
    for i in range(40):
        res = eng.step([st[i] for st in streams])
        for s in range(4):
            e = orcs[s].update(streams[s][i])
            assert [int(v) for v in res[s][:, 0]] == [x[0] for x in e], "seq %d frame %d" % (s, i + 1)
            if e:
                assert np.array_equal(res[s][:, 1:5], np.array([x[1] for x in e]))


def test_gpu_cbiou_crowded_scene():
    frames, _ = make_stream(77, 8, 300, img=700)
    eng = _engine(cap=1024, dmax=512, ecap=131072)
    orc = CB.CBIoUOracle()
    most = 0
    for i, f in enumerate(frames):
        r = eng.step([f])[0]
        e = orc.update(f)
        assert [int(v) for v in r[:, 0]] == [x[0] for x in e], "frame %d" % (i + 1)
        if e:
            assert np.array_equal(r[:, 1:5], np.array([x[1] for x in e]))
        most = max(most, int(eng.np_stat[0, 15]))
    assert most > 8000, most


def test_gpu_cbiou_capacity_error():
    frames = make_vanish_stream(13, 90)
    eng = _engine(cap=64, dmax=64)
    with pytest.raises(L.B2TError, match="capacity"):
        for f in frames:
            eng.step([f])
    assert eng.np_stat[0, L.STAT_ERR] & 1


def _dropin_imports():
    names = ("models", "utils", "basetrack", "bytetrack", "botsort", "matching", "kalman_filter", "c_biou_tracker")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k in names or k.startswith(("models.", "utils."))}
    sys.path.insert(0, os.path.join(PKG, "tracker"))
    sys.path.insert(1, PKG)
    return names, saved


def _restore(names, saved):
    sys.path.remove(os.path.join(PKG, "tracker")); sys.path.remove(PKG)
    for k in list(sys.modules):
        if k in names or k.startswith(("models.", "utils.")):
            sys.modules.pop(k)
    sys.modules.update(saved)


class Opts:
    conf_thresh = 0.2; track_buffer = 30; kalman_format = "naive"; img_size = 256; iou_thresh = 0.5
    reid_model_path = ""; dhn_path = ""; gamma = 0.1; tracker = "c_biou"; min_area = 0.0


def test_gpu_cbiou_dropin_in_the_driver_loop():
    """The body of track.py:138-179 with the drop-in C_BIoUTracker over two sequences that share BaseTrack._count; CUDA-tensor
    detections (the NMS output) and NumPy detections give the same tracks."""
    names, saved = _dropin_imports()
    try:
        from basetrack import BaseTrack
        from c_biou_tracker import C_BIoUTracker
        opts = Opts()
        seqs = {"a": make_stream(31, 30, 50)[0], "b": make_vanish_stream(32, 30)}
        img0 = np.zeros((8, 8, 3), np.uint8)
        BaseTrack._count = 0
        ids = IdCounter()
        for name, frames in seqs.items():
            trk_gpu = C_BIoUTracker(opts, frame_rate=30, gamma=opts.gamma)     # track.py:132 ('naive' is accepted: never read)
            orc = CB.CBIoUOracle(ids=ids)
            for frame_id, dets in enumerate(frames, 1):
                cur = trk_gpu.update(torch.from_numpy(dets).cuda(), img0)     # track.py:151
                cur_tlwh, cur_id, cur_cls = [], [], []
                for t in cur:                                                   # track.py:160-171
                    bbox = t.tlwh
                    if bbox[2] * bbox[3] > opts.min_area:
                        cur_tlwh.append(bbox); cur_id.append(t.track_id); cur_cls.append(t.cls)
                exp = orc.update(dets)
                assert cur_id == [e[0] for e in exp], "%s frame %d" % (name, frame_id)
                if exp:
                    assert np.array_equal(np.array(cur_tlwh, np.float64), np.array([e[1] for e in exp]))
                for t, s in zip(cur, [s for s in orc.tracked if orc.trk[s].activated]):
                    assert np.array_equal(t.motion_state1, orc.trk[s].ms1) and np.array_equal(t.motion_state2, orc.trk[s].ms2)
                    assert t.time_since_update == orc.trk[s].tsu and t.tracklet_len == orc.trk[s].tracklet_len
                    assert t.start_frame == orc.trk[s].start_frame and t.frame_id == frame_id
                    assert np.array_equal(t.buffer_bbox1, CB.buffered(orc.trk[s].hist[-1], 0.3))
                assert [t.track_id for t in trk_gpu.lost_stracks] == [orc.trk[s].tid for s in orc.lost]
            assert BaseTrack._count == ids.count
        assert ids.count > 0
        # CUDA tensor input == NumPy input
        BaseTrack._count = 0
        ta, tb = C_BIoUTracker(opts), C_BIoUTracker(opts)
        for dets in seqs["a"]:
            c0 = BaseTrack._count
            ra = [(t.track_id, t.tlwh.tolist()) for t in ta.update(torch.from_numpy(dets).cuda(), img0)]
            c1 = BaseTrack._count
            BaseTrack._count = c0
            rb = [(t.track_id, t.tlwh.tolist()) for t in tb.update(dets, img0)]
            assert ra == rb and BaseTrack._count == c1
        with pytest.raises(NotImplementedError):
            ta.update_without_detection(None, img0)
    finally:
        _restore(names, saved)


def test_gpu_cbiou_tracking_pipeline():
    """TrackingPipeline (ingest -> detector -> NMS -> tracker step, all on the device, one frame of latency) with a c_biou engine
    returns, frame by frame, the rows of the straight sequence: the same detector's detect() output fed to a c_biou engine."""
    from b200track.detector import DetectorW6
    from b200track.engine import TrackEngine
    from b200track.pipeline import TrackingPipeline
    from b200track.w6 import calibrated_state_dict
    sd = calibrated_state_dict(0, 256, "cuda")
    g = torch.Generator().manual_seed(3)
    base = torch.rand((2, 3, 256, 256), generator=g)
    frames = [torch.roll(base, shifts=(2 * k, 3 * k), dims=(2, 3)).contiguous().pin_memory() for k in range(6)]
    # straight sequence (its objects stay alive until the end of the test)
    det_ref = DetectorW6(sd, batch=2, img_size=256, use_graph=False, autotune=False)
    eng_ref = TrackEngine("c_biou", n_seq=2, cap=512, dmax=det_ref.max_det, device="cuda:0")
    want = []
    for f in frames:
        out, cnt = det_ref.detect(f.cuda(), post=True)
        torch.cuda.synchronize()
        want.append([r.copy() for r in eng_ref.step_cuda_dets([out[s, : int(cnt[s])] for s in range(2)])])
    # pipeline
    det = DetectorW6(sd, batch=2, img_size=256, use_graph=False, autotune=False)
    eng = TrackEngine("c_biou", n_seq=2, cap=512, dmax=det.max_det, device="cuda:0")
    pipe = TrackingPipeline(det, eng, out_rows=512)
    got = []
    for f in frames:
        r = pipe.step(f)
        if r is not None:
            got.append([r[0][s, :int(r[1][s, L.STAT_NOUT])].numpy().copy() for s in range(2)])
    r = pipe.flush()
    got.append([r[0][s, :int(r[1][s, L.STAT_NOUT])].numpy().copy() for s in range(2)])
    assert len(got) == len(want) == 6
    for k, (a, b) in enumerate(zip(got, want)):
        for s in range(2):
            assert np.array_equal(a[s], b[s]), "frame %d sequence %d" % (k + 1, s)
    assert sum(len(w[s]) for w in want for s in range(2)) > 0
