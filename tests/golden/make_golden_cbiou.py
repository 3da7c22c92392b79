"""Writes tests/golden/loop_c_biou.npz by running the UNMODIFIED reference ``C_BIoUTracker`` (tracker/c_biou_tracker.py).

Run where the reference tree exists (``python tests/golden/make_golden_cbiou.py``; B2T_REFERENCE_ROOT points elsewhere): the
output is committed because the GPU box has no reference.  The module is imported by ``load_c_biou`` below on top of the
modules oracle/refshim.py loads (np.float alias, lap / cython_bbox stand-ins); nothing in the reference is edited.

Streams: ``small`` and ``c3`` (the streams of loop_<kind>.npz) and ``vanish`` (b200track.synth.make_vanish_stream: objects that live a few frames
and disappear, so that the never-pruned lost list grows past max_time_lost).  Stored per frame: ids, cls, tlwh of the returned
tracks, len(tracked_stracks), len(lost_stracks); on the frames listed in <name>_rec_frames also the ids, motion states and
time_since_update of every track in tracked_stracks (list order).
"""
import importlib
import os
import sys

import numpy as np
import scipy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "yolov7-tracker_b200"))

from oracle import refshim                                   # noqa: E402
from b200track.synth import make_stream, make_vanish_stream, stream_digest      # noqa: E402

VERS = dict(numpy=np.__version__, scipy=scipy.__version__)

LOOPS = [  # (name, seed, n_obj, n_frames)
    ("small", 11, 40, 120),
    ("c3", 12, 300, 64),
    ("vanish", 13, 0, 90),
]


def stream(name, seed, n_obj, n_frames):
    if name == "vanish":
        return make_vanish_stream(seed, n_frames)
    return make_stream(seed, n_frames, n_obj)[0]


def load_c_biou():
    """The reference's tracker/c_biou_tracker.py module, importing the reference's own basetrack / matching (refshim.load())."""
    ns = refshim.load()
    saved = {k: sys.modules.get(k) for k in ("basetrack", "matching", "c_biou_tracker")}
    sys.modules["basetrack"], sys.modules["matching"] = ns.basetrack, ns.matching
    sys.modules.pop("c_biou_tracker", None)
    tracker_dir = os.path.join(refshim.REF_ROOT, "tracker")
    sys.path.insert(0, tracker_dir)
    try:
        return importlib.import_module("c_biou_tracker")
    finally:
        sys.path.remove(tracker_dir)
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def run_reference(mod, frames, rec_frames):
    mod.BaseTrack._count = 0
    trk = mod.C_BIoUTracker(refshim.Opts(kalman_format="default"))
    img = np.zeros((4, 4, 3), np.uint8)
    res, recs = [], []
    for i, f in enumerate(frames):
        cur = trk.update(f.copy(), img)
        res.append((np.array([t.track_id for t in cur], np.int32),
                    np.array([np.asarray(t.tlwh, np.float32) for t in cur], np.float32).reshape(-1, 4),
                    np.array([float(t.cls) for t in cur], np.float32),
                    len(trk.tracked_stracks), len(trk.lost_stracks)))
        if i in rec_frames:
            ts = trk.tracked_stracks
            recs.append((np.array([t.track_id for t in ts], np.int32),
                         np.array([t.motion_state1 for t in ts], np.float32).reshape(-1, 4),
                         np.array([t.motion_state2 for t in ts], np.float32).reshape(-1, 4),
                         np.array([t.time_since_update for t in ts], np.int32)))
    return res, recs


def main():
    mod = load_c_biou()
    out = {}
    for name, seed, n_obj, n_frames in LOOPS:
        frames = stream(name, seed, n_obj, n_frames)
        rec_frames = [i for i in range(n_frames) if i % 16 == 15 or i == n_frames - 1]
        res, recs = run_reference(mod, frames, rec_frames)
        out[name + "_digest"] = stream_digest(frames)
        out[name + "_cfg"] = np.array([seed, n_obj, n_frames])
        out[name + "_count"] = np.array([len(r[0]) for r in res], np.int32)
        out[name + "_ids"] = np.concatenate([r[0] for r in res])
        out[name + "_cls"] = np.concatenate([r[2] for r in res])
        out[name + "_tlwh"] = np.concatenate([r[1] for r in res])
        out[name + "_ntracked"] = np.array([r[3] for r in res], np.int32)
        out[name + "_nlost"] = np.array([r[4] for r in res], np.int32)
        out[name + "_rec_frames"] = np.array(rec_frames, np.int32)
        out[name + "_rec_count"] = np.array([len(r[0]) for r in recs], np.int32)
        out[name + "_rec_ids"] = np.concatenate([r[0] for r in recs])
        out[name + "_rec_ms1"] = np.concatenate([r[1] for r in recs])
        out[name + "_rec_ms2"] = np.concatenate([r[2] for r in recs])
        out[name + "_rec_tsu"] = np.concatenate([r[3] for r in recs])
        print("loop c_biou", name, "max id", out[name + "_ids"].max(), "last frame tracks", len(res[-1][0]),
              "tracked / lost at the end", res[-1][3], res[-1][4], "stale time_since_update", int((recs[-1][3] > 0).sum()))
    np.savez_compressed(os.path.join(HERE, "loop_c_biou.npz"), **out, **{"ver_" + k: v for k, v in VERS.items()})


if __name__ == "__main__":
    main()
