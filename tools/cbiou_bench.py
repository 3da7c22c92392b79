"""C-BIoU vs ByteTrack on the fused per-frame kernel, same C3 streams, fp64, one process: prints one JSON line.

    python tools/cbiou_bench.py [--steps 100] [--warm 20] [--seqs 4,148]

For each batch size (sequences per launch) both engines advance the same seeded C3 streams (300 objects per sequence, the stream
of tests/golden/loop_c_biou.npz for sequence 0): a device-resident loop, the two kinds alternating step by step, an L2 flush
before every timed launch (outside the CUDA-event pair, as bench_sub.tracker_loop does).  The CPU arm times the per-frame update
of the C3 stream on one core: the reference's own C_BIoUTracker when the packed reference archive (oracle/_ref) carries
c_biou_tracker.py, otherwise the oracle's restatement (oracle/cbiou.py), labelled "port".
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "yolov7-tracker_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=20).stdout.strip()
        power = float(q.splitlines()[0])
    except Exception:
        power = None
    return name, power


def gpu_arm(n_seq, steps, warm, n_obj=300, seed0=12):
    import torch
    from b200track import _lib as L
    from b200track.engine import TrackEngine
    from b200track.synth import make_stream, pack_frames
    dev = torch.device("cuda:0")
    dmax, cap = 512, 1024
    n_frames = warm + steps
    packed = [pack_frames(make_stream(seed0 + s, n_frames, n_obj)[0], dmax) for s in range(n_seq)]
    d_dets = torch.from_numpy(np.stack([p[0] for p in packed], 1)).to(dev)
    d_cnt = torch.from_numpy(np.stack([p[1] for p in packed], 1)).to(dev)
    engs = {k: TrackEngine(k, n_seq=n_seq, dtype="f64", cap=cap, dmax=dmax, device=dev) for k in ("c_biou", "bytetrack")}
    outs = {k: torch.zeros((n_seq, cap, L.OUT_COLS), dtype=torch.float64, device=dev) for k in engs}
    stats = {k: torch.zeros((n_frames, n_seq, L.STAT_WORDS), dtype=torch.int32, device=dev) for k in engs}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)] for k in engs}
    for f in range(n_frames):
        for k, eng in engs.items():
            timed = f >= warm
            if timed:
                flush.zero_()
                ev[k][f - warm][0].record()
            eng.step_device(d_dets[f], d_cnt[f], outs[k], stats[k][f])
            if timed:
                ev[k][f - warm][1].record()
    torch.cuda.synchronize()
    res = {}
    for k in engs:
        ms = np.array([a.elapsed_time(b) for a, b in ev[k]])
        st = stats[k][warm:].cpu().numpy()
        assert int(st[:, :, L.STAT_ERR].max()) == 0, "%s: capacity error" % k
        res[k] = {"us_per_step_median": round(1e3 * float(np.median(ms)), 2), "us_per_step_p90": round(1e3 * float(np.percentile(ms, 90)), 2),
                  "frames_per_s": round(n_seq * steps / (ms.sum() / 1e3), 1), "tracked_mean": round(float(st[:, :, L.STAT_NTRACKED].mean()), 1),
                  "lost_mean": round(float(st[:, :, L.STAT_NLOST].mean()), 1)}
    res["c_biou_over_bytetrack"] = round(res["c_biou"]["us_per_step_median"] / res["bytetrack"]["us_per_step_median"], 3)
    return res


def cpu_arm(frames):
    from oracle import build_ref, refshim
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        src = build_ref.unpack(tmp)
        if src and os.path.exists(os.path.join(src, "tracker", "c_biou_tracker.py")):
            sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
            import make_golden_cbiou as MG
            refshim.use_root(src)
            mod = MG.load_c_biou()
            trk = mod.C_BIoUTracker(refshim.Opts())
            img = np.zeros((4, 4, 3), np.uint8)
            step, label = (lambda d: trk.update(d.copy(), img)), "reference"
        else:
            from oracle.cbiou import CBIoUOracle
            orc = CBIoUOracle()
            step, label = orc.update, "port"
        t = []
        for d in frames:
            t0 = time.perf_counter()
            step(d)
            t.append(time.perf_counter() - t0)
    t = np.array(t[8:])
    return {"impl": label, "ms_per_frame_median": round(1e3 * float(np.median(t)), 2), "frames": len(t)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warm", type=int, default=20)
    ap.add_argument("--seqs", default="4,148")
    a = ap.parse_args()
    from b200track.synth import make_stream
    name, power = gpu_identity()
    out = {"bench": "cbiou_vs_bytetrack", "gpu": name, "power_limit_W": power, "dtype": "f64", "stream": "C3 (300 objects, seed 12 + sequence)",
           "steps": a.steps, "gpu_arm": {}}
    for s in [int(v) for v in a.seqs.split(",")]:
        out["gpu_arm"]["seqs_%d" % s] = gpu_arm(s, a.steps, a.warm)
    out["cpu_arm"] = cpu_arm(make_stream(12, 64, 300)[0])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
