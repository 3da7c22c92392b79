"""not-gpu: the fused C-BIoU kernel (csrc/b2t_cbiou.cuh) executed by the fiber simulator (tests/hostsim) against the reference
goldens (tests/golden/loop_c_biou.npz) and the oracle (oracle/cbiou.py): ids, float32 boxes, list lengths and the slot records."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "hostsim"))
from simlib import ptr, sim, SimTracker  # noqa: E402
from b200track import _lib as L  # noqa: E402
from b200track.synth import make_stream, make_vanish_stream  # noqa: E402
from oracle import cbiou as CB  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "loop_c_biou.npz")


def read_list(trk, which):
    rows = np.zeros((trk.cap, 13))
    n = C.c_int(0)
    L.check(sim(), sim().b2t_tracker_read_list(trk.h, 0, which, ptr(rows), trk.cap, C.byref(n), None))
    return rows[:n.value]


def read_record(trk, slot):
    mean, cov = np.zeros(8), np.zeros(64)
    L.check(sim(), sim().b2t_tracker_read_slot(trk.h, 0, int(slot), ptr(mean), ptr(cov), None))
    r = np.concatenate([mean, cov])
    n = int(r[0])
    return dict(history=r[8:8 + 4 * n].reshape(n, 4), motion_state1=r[32:36], motion_state2=r[36:40], time_since_update=int(r[1]))


@pytest.mark.parametrize("case,n_frames,cap", [("small", 120, 128), ("c3", 20, 1024), ("vanish", 90, 256)])
def test_cbiou_kernel_matches_reference_golden(case, n_frames, cap):
    g = np.load(GOLDEN)
    seed, n_obj, total = [int(v) for v in g[case + "_cfg"]]
    frames = make_vanish_stream(seed, total) if case == "vanish" else make_stream(seed, total, n_obj)[0]
    trk = SimTracker("c_biou", cap=cap, dmax=512, ecap=65536)
    off = np.concatenate([[0], np.cumsum(g[case + "_count"])])
    rec_frames = [int(v) for v in g[case + "_rec_frames"]]
    roff = np.concatenate([[0], np.cumsum(g[case + "_rec_count"])])
    for i in range(n_frames):
        r = trk.step([frames[i]])[0]
        sl = slice(off[i], off[i + 1])
        assert np.array_equal(r[:, 0].astype(np.int64), g[case + "_ids"][sl]), "track ids differ at frame %d" % (i + 1)
        assert np.array_equal(r[:, 5].astype(np.float32), g[case + "_cls"][sl])
        assert np.array_equal(r[:, 1:5], g[case + "_tlwh"][sl].astype(np.float64)), "boxes differ at frame %d" % (i + 1)
        assert trk.stat[0, L.STAT_NTRACKED] == g[case + "_ntracked"][i] and trk.stat[0, L.STAT_NLOST] == g[case + "_nlost"][i]
        if i in rec_frames:
            k = rec_frames.index(i)
            rs = slice(roff[k], roff[k + 1])
            rows = read_list(trk, 0)
            assert np.array_equal(rows[:, 0].astype(np.int64), g[case + "_rec_ids"][rs])
            recs = [read_record(trk, s) for s in rows[:, 7]]
            assert np.array_equal(np.array([x["motion_state1"] for x in recs]).reshape(-1, 4), g[case + "_rec_ms1"][rs].astype(np.float64))
            assert np.array_equal(np.array([x["motion_state2"] for x in recs]).reshape(-1, 4), g[case + "_rec_ms2"][rs].astype(np.float64))
            assert [x["time_since_update"] for x in recs] == g[case + "_rec_tsu"][rs].tolist()
            # read_list reports the last matched box
            assert np.array_equal(rows[:, 1:5], np.array([x["history"][-1] for x in recs]).reshape(-1, 4))


def test_cbiou_kernel_records_equal_oracle():
    frames = make_vanish_stream(5, 24)
    trk = SimTracker("c_biou", cap=128, dmax=128, ecap=4096)
    orc = CB.CBIoUOracle()
    for f in frames:
        r = trk.step([f])[0]
        e = orc.update(f)
        assert [int(v) for v in r[:, 0]] == [x[0] for x in e]
        for which, slots in ((0, orc.tracked), (1, orc.lost)):
            rows = read_list(trk, which)
            assert [int(v) for v in rows[:, 0]] == [orc.trk[s].tid for s in slots]
            for row, s in zip(rows, slots):
                got, exp = read_record(trk, row[7]), orc.record(s)
                assert np.array_equal(got["history"], exp["history"].astype(np.float64))
                assert np.array_equal(got["motion_state1"], exp["motion_state1"].astype(np.float64))
                assert np.array_equal(got["motion_state2"], exp["motion_state2"].astype(np.float64))
                assert got["time_since_update"] == exp["time_since_update"]
                assert row[10] == orc.trk[s].tracklet_len and row[12] == orc.trk[s].frame_id


def test_cbiou_crowded_scene_spills_edges():
    """300 objects in a 300 x 300 px area: the buffered boxes overlap far more than plain ones, so the first association has more
    sub-threshold pairs than the shared-memory edge mirror holds.  Ids and boxes must still equal the oracle's."""
    frames, _ = make_stream(77, 6, 300, img=700)
    trk = SimTracker("c_biou", cap=1024, dmax=512, ecap=131072)
    orc = CB.CBIoUOracle()
    most = 0
    for i, f in enumerate(frames):
        r = trk.step([f])[0]
        e = orc.update(f)
        assert trk.stat[0, L.STAT_ERR] == 0
        assert [int(v) for v in r[:, 0]] == [x[0] for x in e], "track ids differ at frame %d" % (i + 1)
        if len(e):
            assert np.array_equal(r[:, 1:5], np.array([x[1] for x in e]))
        most = max(most, int(trk.stat[0, 15]))            # stat word 15: sub-threshold pairs of the first association
    assert most > 8000, most


def test_cbiou_slot_overflow_is_an_error():
    """Lost tracks are never pruned: on the vanish stream 64 slots run out, and the step reports it instead of dropping tracks."""
    frames = make_vanish_stream(13, 90)
    trk = SimTracker("c_biou", cap=64, dmax=64, ecap=4096)
    with pytest.raises(L.B2TError, match="capacity"):
        for f in frames:
            trk.step([f])
    assert trk.stat[0, L.STAT_ERR] & 1                    # ERR_SLOTS
    with pytest.raises(L.B2TError, match="capacity"):     # sticky
        trk.step([frames[0]])


def test_cbiou_rejects_f32_and_predict_only():
    lib = sim()
    cfg = L.TrackerConfig(kind=L.CBIOU, dtype=L.F32, fmt=0, n_seq=1, cap=64, dmax=64, ecap=1024, use_gmc=0, track_buffer=30,
                          conf_thresh=0.2, iou_thresh=0.5, frame_rate=30)
    assert lib.b2t_tracker_state_bytes(C.byref(cfg)) == 0
    assert b"B2T_F64" in lib.b2t_last_error()
    trk = SimTracker("c_biou", cap=64, dmax=64, ecap=1024)
    with pytest.raises(L.B2TError, match="predict_only"):
        trk.step([np.zeros((0, 6), np.float32)], predict_only=True)
    trk.step([make_stream(1, 1, 10)[0][0]])               # the tracker is still usable


def test_cbiou_fits_the_default_engine_capacities():
    cfg = L.TrackerConfig(kind=L.CBIOU, dtype=L.F64, fmt=0, n_seq=1, cap=1024, dmax=1024, ecap=131072, use_gmc=0, track_buffer=30,
                          conf_thresh=0.2, iou_thresh=0.5, frame_rate=30)
    assert sim().b2t_tracker_state_bytes(C.byref(cfg)) > 0, sim().b2t_last_error()
