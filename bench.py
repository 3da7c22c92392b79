"""bench.py -- end-to-end tracked frames/s (detect + NMS + associate) of the B200-native path, and the CPU reference arm.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload pipeline|tracker] [--dump-outputs DIR]

Default workload "pipeline" (bench_pipeline.py) = the BASELINE.json metric: YOLOv7-w6 1280 x 1280, batch 8 -> decode + NMS ->
ByteTrack, one uint8 frame per sequence per step; its JSON line also carries BASELINE configs C1 / C3 / C4 / C5, C4 end to end with the
camera-motion warp estimated on the GPU, and the camera-motion / ReID kernels alone as ``config.sub_benchmarks`` (bench_sub.py).  ``--workload tracker`` = the association path alone (config C3) as its own line.
Sequences are independent units: under torchrun every rank owns its own sequences (weak scaling), there is no data-path
collective; one tiny all-gather of per-sequence birth counts gives the global track-id offsets (SURVEY.md section 8e).
``--impl reference`` = the reference's own CPU implementation on the host cores (bench_reference.py), rank 0 only.

Printed JSON (rank 0, one line):
  value         frames/s with the inputs already resident in HBM
  e2e           frames/s through the public API with HOST buffers: pinned H2D of the step's inputs + D2H of the tracks, every step
  roofline      the dominant kernel against MEASURED_PEAKS.json
  cpu_baseline  the reference's CPU path on a bounded sample (N = 1 only)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

if os.environ.get("OMP_NUM_THREADS", "") in ("", "1") and os.environ.get("RANK", "0") == "0":
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm (rank 0 only: --impl reference, and the cpu_baseline leg of
    # the default run) is meant to use the host's cores, and OpenMP / MKL read the variable when torch is imported -- so set it
    # before that import, to the cores this process may actually run on (affinity-aware: os.cpu_count() over-reports on a
    # shared host and oversubscribed torch-cpu convolutions ran 10x slower in round 1's SCALE run).
    try:
        _n = len(os.sched_getaffinity(0))
    except Exception:
        _n = os.cpu_count() or 1
    _n = str(max(1, min(32, _n)))
    os.environ["OMP_NUM_THREADS"] = _n
    os.environ["MKL_NUM_THREADS"] = _n

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "yolov7-tracker_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "tracked_frames_per_sec"
N_OBJ = 300
STREAM_WARM = 60          # frames run before anything is timed: reach the ~250 live + ~45 lost steady state


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU DURING the timed region: NVML in-process (a query costs ~50 us, so a
    0.3 s region still gets dozens of samples), nvidia-smi subprocess as the fallback when NVML cannot be loaded."""
    _REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self._stop_evt = index, threading.Event()
        self.sm, self.mx, self.reasons, self.n = [], [], set(), 0
        self.source = "nvml"
        try:
            import pynvml
            pynvml.nvmlInit()
            try:                                   # CUDA ordinal -> physical GPU (CUDA_VISIBLE_DEVICES may renumber)
                import torch
                self._h = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(index).uuid))
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nv = pynvml
        except Exception:
            self._nv, self.source = None, "nvidia-smi"

    def _poll_nvml(self):
        nv, h = self._nv, self._h
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
        bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        for nm, bit in self._REASONS:
            if bits & bit:
                self.reasons.add(nm)
        self.n += 1

    def _poll_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [c.strip() for c in out.split(",")]
        if len(r) >= 6:
            self.sm.append(float(r[0])); self.mx.append(float(r[1]))
            for k, (nm, _) in enumerate(self._REASONS):
                if r[2 + k].lower().startswith("active"):
                    self.reasons.add(nm)
            self.n += 1

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self._nv is not None:
                    self._poll_nvml()
                else:
                    self._poll_smi()
            except Exception:
                if self._nv is not None:        # NVML query failed: fall back to the CLI for the rest of the run
                    self._nv, self.source = None, "nvidia-smi"
            self._stop_evt.wait(0.01 if self._nv is not None else 0.2)

    def summary(self):
        self._stop_evt.set()
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": self.n, "source": self.source}


def _tracker_traffic(n_seq):
    """DRAM bytes per launch of track_step_kernel from the committed ncu --set full capture (taken at 4 sequences)."""
    try:
        names = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.endswith("_track_step_traffic.json"))
        tj = json.load(open(os.path.join(ROOT, "profiles", names[-1])))
        return (tj["dram_bytes_read"] + tj["dram_bytes_write"]) if n_seq == 4 else None
    except Exception:
        return None


def algorithmic_bytes(stat_rows, esize):
    """SURVEY.md section 8(d) per-unit figures x the units of this launch: predict 144 values/track
    (72 read + 72 written), update 148 values/matched track, IoU + LAP one write + one read of every
    n x m cost matrix (associations 1-3), dedup one n x m IoU matrix."""
    from b200track import _lib as L
    total = 0
    for st in stat_rows:
        pool, hi, lo, m0 = int(st[L.STAT_NPOOL]), int(st[L.STAT_NHI]), int(st[L.STAT_NLO]), int(st[L.STAT_NMATCH0])
        ntr, nlost = int(st[L.STAT_NTRACKED]), int(st[L.STAT_NLOST])
        total += pool * 144 * esize + m0 * 148 * esize
        total += 2 * pool * hi * esize + 2 * max(pool - m0, 0) * lo * esize + ntr * nlost * esize
    return total


def run_reference_arm(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path -- the reference is pure
    Python and cannot travel to the GPU box, so this is the oracle port of it (oracle/trackers.py,
    checked bit-for-bit against the reference in tests/golden), single thread like the reference."""
    if rank != 0:
        return
    from oracle import trackers as T
    from b200track.synth import make_stream
    S = args.seqs
    n_frames = STREAM_WARM + args.warmup + args.steps
    streams = [make_stream(3000 + s, n_frames, N_OBJ)[0] for s in range(S)]
    trk = [T.TrackerOracle(args.tracker) for _ in range(S)]
    for f in range(STREAM_WARM + args.warmup):
        for s in range(S):
            trk[s].update(streams[s][f])
    t0 = time.perf_counter()
    for f in range(STREAM_WARM + args.warmup, n_frames):
        for s in range(S):
            trk[s].update(streams[s][f])
    dt = time.perf_counter() - t0
    fps = S * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "C3: %s full loop, %d dets/frame, %d-seq synthetic 1280x1280 stream (tracker only)" % (args.tracker, N_OBJ, S)},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": 1, "kind": "port",
                             "sample": "%d frames x %d sequences after %d warm-up frames" % (args.steps, S, STREAM_WARM + args.warmup)},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 100 pipeline, 1500 tracker-only; 20 and 200 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--seqs", type=int, default=4)
    ap.add_argument("--tracker", default="bytetrack")
    ap.add_argument("--dtype", default="f64")
    ap.add_argument("--cpu-sample-frames", type=int, default=60)
    ap.add_argument("--workload", default="pipeline", choices=["pipeline", "tracker"],
                    help="pipeline: YOLOv7-w6 detect + NMS + ByteTrack (BASELINE metric); tracker: association only (config C3)")
    ap.add_argument("--batch", type=int, default=8, help="pipeline: frames per step = sequences per GPU")
    ap.add_argument("--img", type=int, default=1280)
    ap.add_argument("--no-sub", action="store_true", help="pipeline: skip config.sub_benchmarks (C3 / C4 / C5)")
    ap.add_argument("--quick-sub", action="store_true", help="pipeline: shorter sub-benchmarks")
    ap.add_argument("--no-cpu", action="store_true", help="pipeline: skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def track_outputs(rows, stat):
    """What a tracker step returns, for dump_outputs: the track rows, with the rows past each sequence's count (stale buffer
    contents) zeroed, and the result counters (the stat words from STAT_PHASE0 on are clock-cycle counts, not results)."""
    from b200track import _lib as L
    rows, stat = np.array(rows, dtype=np.float64), np.asarray(stat)
    for s, n in enumerate(stat[:, L.STAT_NOUT]):
        rows[s, int(n):] = 0
    return {"tracks": rows, "stat": stat[:, :L.STAT_PHASE0]}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float64: the inputs are seeded, so two builds run with the same arguments
    can be compared output for output.  The leading axis of every array is the sequence; when all of them would take more than
    DUMP_BYTES, the same fixed, seeded sample of sequences is written from each, and its indices as sequence_index.npy."""
    arrays = {name: np.asarray(a, dtype=np.float64) for name, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    keep = DUMP_BYTES // (sum(a[0].nbytes for a in arrays.values()) + 8)
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {name: a[idx] for name, a in arrays.items()}
        arrays["sequence_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def main():
    args = parse_args()
    if args.steps is None:
        args.steps = (20 if args.impl == "reference" else 100) if args.workload == "pipeline" else (200 if args.impl == "reference" else 1500)
    if args.workload == "pipeline":
        import bench_pipeline
        return bench_pipeline.run(args)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from b200track import _lib as L
    from b200track.engine import TrackEngine
    from b200track.synth import make_stream, pack_frames

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()

    S, K, W = args.seqs, args.steps, args.warmup
    n_frames = STREAM_WARM + max(W + K, args.cpu_sample_frames)
    dmax = 512
    streams = [make_stream(3000 + rank * S + s, n_frames, N_OBJ)[0] for s in range(S)]
    packed = [pack_frames(st, dmax) for st in streams]
    dets_all = np.stack([p[0] for p in packed], 1)           # (F, S, dmax, 6)
    cnt_all = np.stack([p[1] for p in packed], 1)            # (F, S)
    esize = 8 if args.dtype == "f64" else 4

    def fresh_engine():
        eng = TrackEngine(args.tracker, n_seq=S, dtype=args.dtype, cap=1024, dmax=dmax, device=dev)
        eng.set_out_rows(512)
        return eng

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)      # > 126 MB L2

    # ---------------- device-resident arm: detections already in HBM
    eng = fresh_engine()
    d_dets = torch.from_numpy(dets_all).to(dev)
    d_cnt = torch.from_numpy(cnt_all).to(dev)
    d_out = torch.zeros((S, 512, L.OUT_COLS), dtype=torch.float64, device=dev)
    d_stat = torch.zeros((n_frames, S, L.STAT_WORDS), dtype=torch.int32, device=dev)
    for f in range(STREAM_WARM + W):
        eng.step_device(d_dets[f], d_cnt[f], d_out, d_stat[f])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    torch.cuda.profiler.start()
    launches0 = lib.b2t_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for k in range(K):
        f = STREAM_WARM + W + k
        flush.zero_()                                        # L2 flush between timed iterations (outside the event pair)
        ev[k][0].record()
        eng.step_device(d_dets[f], d_cnt[f], d_out, d_stat[f])
        ev[k][1].record()
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_wall0
    launches = lib.b2t_launch_count() - launches0
    dev_ms = np.array([a.elapsed_time(b) for a, b in ev])
    step_ms = float(dev_ms.sum())
    stat_host = d_stat[STREAM_WARM + W:STREAM_WARM + W + K].cpu().numpy()     # the K timed steps (d_stat may hold more rows)
    last_outputs = track_outputs(d_out.cpu().numpy(), stat_host[-1])          # what the last timed step returned
    err = int(stat_host[:, :, L.STAT_ERR].max())
    assert err == 0, "tracker capacity error %d" % err
    algo_bytes = sum(algorithmic_bytes(stat_host[k], esize) for k in range(K)) / K
    births_local = torch.tensor([int(stat_host[-1, s, L.STAT_NEXT_ID]) for s in range(S)], dtype=torch.int64, device=dev)

    # ---------------- e2e arm: host buffers through b2t_tracker_step_host, every step
    eng2 = fresh_engine()
    for f in range(STREAM_WARM + W):
        eng2.np_dets[:] = dets_all[f]; eng2.np_count[:] = cnt_all[f]
        eng2.step_host()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for k in range(K):
        f = STREAM_WARM + W + k
        eng2.np_dets[:] = dets_all[f]; eng2.np_count[:] = cnt_all[f]      # the caller's frame lands in pinned memory
        eng2.step_host()                                                   # H2D + kernel + D2H + sync
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    torch.cuda.profiler.stop()
    clocks = sampler.summary()
    # same stream, same inputs: both arms must agree on the final ids
    ids_a = d_out[:, :, 0].cpu().numpy()
    res_b = eng2.results()
    for s in range(S):
        nb = len(res_b[s])
        assert np.array_equal(ids_a[s, :nb], res_b[s][:, 0]), "device-resident and host-buffer arms disagree"

    # ---------------- scale-out over sequences on one GPU: one CTA per sequence, 148 SMs
    sweep = {}
    if rank == 0 and world == 1:
        for S2 in (148,):
            engs = TrackEngine(args.tracker, n_seq=S2, dtype=args.dtype, cap=1024, dmax=dmax, device=dev)
            dd = torch.from_numpy(np.ascontiguousarray(np.tile(dets_all[:STREAM_WARM + 40], (1, (S2 + S - 1) // S, 1, 1))[:, :S2])).to(dev)
            dc = torch.from_numpy(np.ascontiguousarray(np.tile(cnt_all[:STREAM_WARM + 40], (1, (S2 + S - 1) // S))[:, :S2])).to(dev)
            do = torch.zeros((S2, 512, L.OUT_COLS), dtype=torch.float64, device=dev)
            ds = torch.zeros((S2, L.STAT_WORDS), dtype=torch.int32, device=dev)
            for f in range(STREAM_WARM):
                engs.step_device(dd[f], dc[f], do, ds)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for f in range(STREAM_WARM, STREAM_WARM + 40):
                engs.step_device(dd[f], dc[f], do, ds)
            b.record(); torch.cuda.synchronize()
            sweep["S=%d" % S2] = {"frames_per_s": S2 * 40 / (a.elapsed_time(b) / 1e3), "us_per_step": 1e3 * a.elapsed_time(b) / 40}
            del engs, dd, dc, do, ds

    # ---------------- max over ranks, global id bookkeeping
    t = torch.tensor([step_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gathered = [torch.zeros_like(births_local) for _ in range(world)]
        dist.all_gather(gathered, births_local)              # the ONLY collective: per-sequence birth counts
        id_offsets = torch.cumsum(torch.cat(gathered), 0) - torch.cat(gathered)
    else:
        id_offsets = torch.cumsum(births_local, 0) - births_local
    step_ms_max, e2e_ms_max = float(t[0]), float(t[1])

    if rank == 0:
        hbm, how = _peaks()
        total_frames = S * K * world
        value = total_frames / (step_ms_max / 1e3)
        e2e = total_frames / (e2e_ms_max / 1e3)
        kern_us = 1e3 * step_ms / K
        achieved = algo_bytes / (kern_us * 1e-6) / 1e9
        # CPU baseline: oracle port on a bounded sample of the same workload (rank 0, N=1 only)
        cpu = None
        if world == 1:
            from oracle import trackers as T
            orc = T.TrackerOracle(args.tracker)
            for f in range(STREAM_WARM):
                orc.update(streams[0][f])
            nsamp = args.cpu_sample_frames
            t0 = time.perf_counter()
            for f in range(STREAM_WARM, STREAM_WARM + nsamp):
                orc.update(streams[0][f])
            cdt = time.perf_counter() - t0
            cpu = {"value": nsamp / cdt, "unit": "frames/s", "cores": 1, "kind": "port",
                   "sample": "%d frames of sequence 0 after %d warm-up frames (oracle/trackers.py, NumPy+SciPy)" % (nsamp, STREAM_WARM)}
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": "C3: %s full loop, %d dets/frame, %d-seq synthetic 1280x1280 stream per GPU "
                                   "(association path only: --workload tracker)" % (args.tracker, N_OBJ, S),
                       "sequences_per_gpu": S, "frames_per_step": S, "l2": "flushed (256 MiB memset) between timed steps, outside the event pairs",
                       "stream_warmup_frames": STREAM_WARM, "global_id_offsets": [int(v) for v in id_offsets.cpu()][:8],
                       "sequence_sweep_device_resident": sweep},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(eng2.h2d_bytes_per_step),
                    "d2h_bytes_per_step": int(eng2.d2h_bytes_per_step), "ms_per_step": e2e_ms_max / K},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "track_step_kernel<%s>" % ("double" if esize == 8 else "float"),
                         "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": _tracker_traffic(S),
                         "peak_source": how, "algorithmic_bytes_per_launch": algo_bytes, "kernel_us": kern_us,
                         "note": "latency-bound: one CTA per sequence, %d CTAs per launch (SURVEY 8d: ~1 MB/frame/sequence)" % S},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "wall_s_device_arm": t_wall,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_outputs)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
