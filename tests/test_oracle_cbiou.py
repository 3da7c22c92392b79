"""not-gpu: the C-BIoU oracle (oracle/cbiou.py) against the reference's own C_BIoUTracker (tests/golden/loop_c_biou.npz), bit for
bit; the float32 buffered-box restatement; and the drop-in module's public names."""
import ast
import os

import numpy as np
import pytest

from b200track.synth import make_stream, make_vanish_stream, stream_digest
from oracle import cbiou as CB

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "loop_c_biou.npz")


def golden_frames(g, case):
    seed, n_obj, n_frames = [int(v) for v in g[case + "_cfg"]]
    frames = make_vanish_stream(seed, n_frames) if case == "vanish" else make_stream(seed, n_frames, n_obj)[0]
    assert stream_digest(frames) == str(g[case + "_digest"]), "stream generator drifted"
    return frames


@pytest.mark.parametrize("case", ["small", "c3", "vanish"])
def test_oracle_matches_reference_golden(case):
    g = np.load(GOLDEN)
    frames = golden_frames(g, case)
    orc = CB.CBIoUOracle()
    off = np.concatenate([[0], np.cumsum(g[case + "_count"])])
    rec_frames = [int(v) for v in g[case + "_rec_frames"]]
    roff = np.concatenate([[0], np.cumsum(g[case + "_rec_count"])])
    for i, f in enumerate(frames):
        res = orc.update(f)
        sl = slice(off[i], off[i + 1])
        assert [r[0] for r in res] == g[case + "_ids"][sl].tolist(), "ids differ at frame %d" % (i + 1)
        assert np.array_equal(np.array([r[2] for r in res], np.float32), g[case + "_cls"][sl])
        assert np.array_equal(np.array([r[1] for r in res]).reshape(-1, 4), g[case + "_tlwh"][sl].astype(np.float64))
        assert len(orc.tracked) == g[case + "_ntracked"][i] and len(orc.lost) == g[case + "_nlost"][i]
        if i in rec_frames:
            k = rec_frames.index(i)
            rs = slice(roff[k], roff[k + 1])
            assert [orc.trk[s].tid for s in orc.tracked] == g[case + "_rec_ids"][rs].tolist()
            assert np.array_equal(np.array([orc.trk[s].ms1 for s in orc.tracked]).reshape(-1, 4), g[case + "_rec_ms1"][rs])
            assert np.array_equal(np.array([orc.trk[s].ms2 for s in orc.tracked]).reshape(-1, 4), g[case + "_rec_ms2"][rs])
            assert [orc.trk[s].tsu for s in orc.tracked] == g[case + "_rec_tsu"][rs].tolist()


def test_golden_pins_the_quirks():
    g = np.load(GOLDEN)
    # re_activate keeps time_since_update: tracked tracks carry a stale value at the end of the C3 stream
    n = int(g["c3_rec_count"][-1])
    assert (g["c3_rec_tsu"][-n:] > 0).sum() > 0
    # lost tracks are never pruned: the vanish stream's lost list outgrows max_time_lost (30)
    assert g["vanish_nlost"][-1] > 30


def test_buffered_box_is_float32_numpy_arithmetic():
    rng = np.random.default_rng(3)
    t = np.concatenate([rng.uniform(-50, 1300, (2000, 2)), rng.uniform(0, 300, (2000, 2))], 1).astype(np.float32)
    for b in (0.3, 0.5):
        # the reference's expression (c_biou_tracker.py:59) evaluated by NumPy on float32 scalars
        exp = np.array([np.maximum(0.0, x + np.array([-b * x[2], -b * x[3], 2 * b * x[2], 2 * b * x[3]])) for x in t])
        got = np.array([CB.buffered(x, b) for x in t])
        assert got.dtype == np.float32 and np.array_equal(got, exp)


def test_dropin_exports_what_track_py_imports():
    src = open(os.path.join(ROOT, "yolov7-tracker_b200", "tracker", "c_biou_tracker.py")).read()
    tree = ast.parse(src)
    names = {n.name for n in tree.body if isinstance(n, (ast.ClassDef, ast.FunctionDef))}
    for n in tree.body:
        if isinstance(n, ast.ImportFrom):
            names |= {a.asname or a.name for a in n.names}
    assert {"C_BIoUSTrack", "C_BIoUTracker", "joint_stracks", "sub_stracks", "remove_duplicate_stracks"} <= names
    cls = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == "C_BIoUTracker")
    assert [b.id for b in cls.bases] == ["BaseTracker"]
