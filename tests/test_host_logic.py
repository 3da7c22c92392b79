"""not-gpu: host-side logic -- C-ABI export check (no compute), sharding over 2 gloo ranks, stream generator."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cabi_library_exports_every_declared_symbol():
    """libb200track.so (nvcc build) loads and exports everything include/b200track.h declares."""
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    lib_path = ge.build()
    lib = ctypes.CDLL(lib_path)
    hdr = open(os.path.join(ROOT, "include", "b200track.h")).read()
    declared = set(re.findall(r"\b(b2t_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"b2t_tracker_config"}
    assert len(declared) >= 20
    for name in sorted(declared):
        assert hasattr(lib, name), "missing export: " + name
    from b200track import _lib as L
    assert set(L.SIGNATURES) == declared
    L.declare(lib)
    assert lib.b2t_version() >= 100
    assert lib.b2t_tracker_out_cols() == L.OUT_COLS and lib.b2t_tracker_stat_words() == L.STAT_WORDS
    cfg = L.TrackerConfig(kind=1, dtype=1, fmt=0, n_seq=4, cap=1024, dmax=512, ecap=32768, use_gmc=0, track_buffer=30,
                          conf_thresh=0.2, iou_thresh=0.5, frame_rate=30.0)
    assert lib.b2t_tracker_state_bytes(ctypes.byref(cfg)) > 4 * 1024 * 576            # pure host arithmetic
    bad = L.TrackerConfig(kind=1, dtype=1, fmt=0, n_seq=1, cap=4096, dmax=1024, ecap=1, use_gmc=0, track_buffer=30,
                          conf_thresh=0.2, iou_thresh=0.5, frame_rate=30.0)
    assert lib.b2t_tracker_state_bytes(ctypes.byref(bad)) == 0 and b"shared memory" in lib.b2t_last_error()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "yolov7-tracker_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f + " imports the oracle"


def test_engine_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from b200track.engine import TrackEngine
    from b200track._lib import B2TError
    with pytest.raises(B2TError):
        TrackEngine("bytetrack")


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from b200track.sharding import shard_sequences, global_id_offsets, to_global_ids
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
births = [7, 11, 3, 20, 5]                       # births per sequence, 5 sequences
mine = shard_sequences(5, rank, 2)
off = global_id_offsets([births[s] for s in mine], mine, 5)
assert off.tolist() == [0, 7, 18, 21, 41], off
assert to_global_ids(2, 3, off) == 23
print("rank", rank, "ok")
dist.destroy_process_group()
'''


def test_global_id_offsets_two_gloo_ranks(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 1000)
    pkg = os.path.join(ROOT, "yolov7-tracker_b200")
    procs = [subprocess.Popen([sys.executable, str(script), pkg, port, str(r)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
             for r in range(2)]
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out.decode()


def test_sharded_tracking_equals_sequential_reference_ids():
    """Oracle-level statement of 8e: per-sequence local counters + offsets == one global counter."""
    from oracle import trackers as T
    from b200track.synth import make_stream
    import torch
    from b200track.sharding import global_id_offsets
    streams = [make_stream(900 + s, 12, 25)[0] for s in range(3)]
    shared = T.IdCounter()
    seq_ref = []
    for s in range(3):                                   # the reference: sequences one after another, one counter
        trk = T.TrackerOracle("bytetrack", ids=shared)
        seq_ref.append([[o[0] for o in trk.update(f)] for f in streams[s]])
    local, births = [], []
    for s in range(3):                                   # sharded: independent counters
        trk = T.TrackerOracle("bytetrack")
        local.append([[o[0] for o in trk.update(f)] for f in streams[s]])
        births.append(trk.ids.count)
    off = global_id_offsets(torch.tensor(births), [0, 1, 2], 3)
    for s in range(3):
        assert [[i + int(off[s]) for i in fr] for fr in local[s]] == seq_ref[s]


def test_stream_generator_contract():
    from b200track.synth import make_stream, pack_frames
    frames, warps = make_stream(1, 5, 50, warp_sigma=2.0)
    for f in frames:
        assert f.dtype == np.float32 and f.shape[1] == 6
        assert np.all(np.diff(f[:, 4]) <= 0)                              # NMS order: descending score (q13)
        assert np.all(f[:, :4] == np.round(f[:, :4])) and np.all(f[:, 2] - f[:, 0] >= 4)   # q9
    d, c = pack_frames(frames, 64)
    assert d.shape == (5, 64, 6) and c.tolist() == [len(f) for f in frames]
    assert warps.shape == (5, 2, 3)


def test_result_writer_matches_reference_format(tmp_path):
    """b200track.results against the files the reference's own save_results (tracker/track.py:247-273) wrote for the same rows
    (tests/golden/refchecks.npz), and against the documented line formats."""
    import numpy as np
    from b200track.results import format_rows, write_sequence
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden_refchecks import results_frames
    g = np.load(os.path.join(ROOT, "tests", "golden", "refchecks.npz"))
    frames = results_frames()
    for data_type in ("mot17", "default"):
        out = write_sequence(str(tmp_path / ("ours_%s" % data_type) / "seq.txt"), frames, data_type)
        assert open(out).read() == str(g["results_" + data_type])
        first = format_rows(1, frames[0][:1], data_type)[0]
        assert first.startswith("1,%d," % int(frames[0][0, 0])) and first.endswith("\n")
        assert first.count(",") == (9 if data_type == "mot17" else 6)


def test_header_is_plain_c():
    """include/b200track.h is the C-ABI contract: it must compile as C99 and as C++ on its own (no torch / CUDA types)."""
    import shutil
    import subprocess
    hdr = os.path.join(ROOT, "include", "b200track.h")
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    for cmd in (["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", hdr], ["g++", "-std=c++17", "-fsyntax-only", "-x", "c++", hdr]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    code = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)           # comments may cite torch / cudaStream_t, declarations may not
    assert "torch" not in code.lower() and "cudaStream_t" not in code and "#include <cuda" not in code
