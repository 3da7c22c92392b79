"""bench_pipeline.py -- the BASELINE.json metric: end-to-end tracked frames/s, detect + NMS + associate.

One "step" = one 1280 x 1280 frame for each of the B sequences a rank owns (BASELINE config C2 + C3: YOLOv7-w6, batch 8,
detect + NMS, then ByteTrack on the <= 300 detections per frame):
    uint8 BGR frames (as cv2.imread / tracker_dataloader.py:64-79 produce them)
      -> letterbox + BGR->RGB + /255 + ReOrg + NHWC fp16 (one kernel) -> 96 tcgen05 conv launches (107 convs)
      -> Detect decode fused with NMS (+ scale_coords / clip / round)                                             [CUDA graphs]
      -> fused ByteTrack step (one CTA per sequence) on the device-resident detections.
value : the frames already resident in HBM (uint8), tracks read back.
e2e   : every step copies the B frames from pinned host memory (B x 4.9 MB of bytes) and reads the tracks back: the public
        TrackingPipeline.step() call with HOST buffers.
Inputs exceed L2 (>1 GB of activations per step), so there is no explicit flush.
The pipeline runs over two twin detectors (b200track/pipeline.py): only the forward graph is on the critical path.
config.sub_benchmarks carries BASELINE configs C1 (YOLOv7-tiny plumbing case), C3 (tracker only), C4 (BoT-SORT, 8 sequences; and end to end
with the GPU camera-motion estimate), C5 (IoU + LAP sweep), and the camera-motion / ReID kernels with the reference's host code beside them.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "yolov7-tracker_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "tracked_frames_per_sec"
POOL = 4


def _workload(args):
    return ("C2+C3: YOLOv7-w6 (seeded LSUV-calibrated random init) %dx%d batch %d detect+NMS (conf 0.01, iou 0.45, 300 dets cap) "
            "+ ByteTrack, one uint8 frame per sequence per step" % (args.img, args.img, args.batch))


def make_frames(batch, size, seed):
    """POOL uint8 BGR frame batches (batch, size, size, 3): one seeded noise image per sequence, shifted a little per frame."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (batch, size, size, 3), dtype=np.uint8)
    return [np.ascontiguousarray(np.roll(base, (2 * k, k), axis=(1, 2))) for k in range(POOL)]


def conv_traffic(n_conv):
    """DRAM bytes of the conv launches of one step from the newest committed ``ncu --set full`` capture of this command
    (profiles/*_conv_traffic.json, written by tools/summarize_profiles.py).  Returns (bytes per step, source, partial)."""
    try:
        pdir = os.path.join(ROOT, "profiles")
        for cand in sorted((f for f in os.listdir(pdir) if f.endswith("_conv_traffic.json")), reverse=True):
            tj = json.load(open(os.path.join(pdir, cand)))
            total = tj["dram_bytes_read"] + tj["dram_bytes_write"]
            if tj.get("launches") == n_conv:
                return total, "profiles/" + cand, None
            return None, None, {"launches": tj.get("launches"), "dram_bytes": total,
                                "algorithmic_bytes": tj.get("algorithmic_bytes_same_launches"), "source": "profiles/" + cand}
    except Exception:
        pass
    return None, None, None


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU path (bench_reference.py), one frame per step, rank 0 only."""
    if rank != 0:
        return
    import torch
    import bench_reference as BR
    from b200track.w6 import calibrated_state_dict
    sd = calibrated_state_dict(0, args.img, "cuda" if torch.cuda.is_available() else "cpu")
    sd = {k: v.cpu() for k, v in sd.items()}
    n = args.steps
    w = max(1, min(args.warmup, 2))
    r = BR.run_cpu_arm(sd, args.img, n, w)
    fps = r["value"]
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": n, "warmup": w,
            "ms_per_step": 1e3 / fps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": _workload(args) + " [CPU arm: one frame per step, batch 1 like tracker/track.py:138-179]",
                       "requested_steps": args.steps, "ms_per_frame": r["ms_per_frame"]},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run(args):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    B, K, W = args.batch, args.steps, max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist
    from bench import ClockSampler, track_outputs
    from b200track import _lib as L
    from b200track.detector import DetectorW6
    from b200track.engine import TrackEngine
    from b200track.pipeline import TrackingPipeline
    from b200track.w6 import calibrated_state_dict

    assert torch.cuda.is_available(), "bench needs a CUDA device: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    hbm_gbs = float(peaks.get("hbm_gbs", 6650.0))
    sd = calibrated_state_dict(0, args.img, dev)
    det = DetectorW6(sd, batch=B, img_size=args.img, device=dev, use_graph=True)
    det.set_source_frames((args.img, args.img))
    # a twin (same weights, same plans from the per-process tuning cache, own buffers: +1.2 GB): frames alternate between the two, so the
    # ingest of frame t+1 and the decode / NMS of frame t-1 run beside frame t's forward instead of between two forwards
    det2 = DetectorW6(sd, batch=B, img_size=args.img, device=dev, use_graph=True)
    det2.set_source_frames((args.img, args.img))
    eng = TrackEngine("bytetrack", n_seq=B, dtype="f64", cap=1024, dmax=det.max_det, device=dev)
    eng.set_out_rows(512)
    frames_np = make_frames(B, args.img, 1000 + rank)
    host_frames = [torch.from_numpy(f).pin_memory() for f in frames_np]
    dev_frames = [f.to(dev) for f in host_frames]
    pipe = TrackingPipeline([det, det2], eng, out_rows=512)

    for k in range(W + 4):
        pipe.step(dev_frames[k % POOL])
    pipe.flush()
    torch.cuda.synchronize()
    n_graph_kernels = len(det.ops) + 5                         # ingest + forward ops + fused decode/filter, bin scan, scatter, rank, greedy NMS

    def timed_device(steps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(pipe.s_copy)
        for k in range(steps):
            pipe.step(dev_frames[k % POOL])
        pipe.flush()
        e1.record(pipe.s_trk)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def timed_e2e(steps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for k in range(steps):
            pipe.step(host_frames[k % POOL])
        res = pipe.flush()
        torch.cuda.synchronize()
        return 1e3 * (time.perf_counter() - t0), res

    sampler = ClockSampler(local_rank); sampler.start()
    torch.cuda.profiler.start()                                  # ncu --profile-from-start off: only the timed region
    l0 = lib.b2t_launch_count()
    dev_ms = timed_device(K)                                     # ---- the K timed steps: frames resident in HBM
    tracker_launches = lib.b2t_launch_count() - l0
    e2e_ms, (h_out, h_stat) = timed_e2e(K)                       # ---- the K timed steps through the public API with HOST frames
    torch.cuda.profiler.stop()
    clocks = sampler.summary()
    stat = pipe.t_stat.cpu().numpy()
    assert int(stat[:, L.STAT_ERR].max()) == 0
    # ---- repeats: the timed region is ~0.4 s; two more runs of the same K steps show the run-to-run spread
    rep_dev = [dev_ms] + [timed_device(K) for _ in range(2)]
    rep_e2e = [e2e_ms] + [timed_e2e(K)[0] for _ in range(2)]
    last_outputs = track_outputs(*(t.numpy() for t in pipe.flush()))            # what the last timed step returned
    # phase cycles of the last track_step_kernel launch under the pipeline's own load (stat words 16..28, SM clocks; mean over sequences)
    phase_names = ["P0 dets", "P1 lists", "P2 predict", "P3 boxes", "P4 csr1", "P5 lap1", "P6 apply1", "P7 assoc2", "P8 assoc3", "P9 births",
                   "P10 lists", "P11 dedup", "P12 output"]
    phases = {nm: float(stat[:, L.STAT_PHASE0 + i].mean()) for i, nm in enumerate(phase_names)}
    sub = stat[:, L.STAT_SUB0:L.STAT_SUB0 + 16].astype(np.float64).mean(0)
    pool_sizes = {"pool_mean": float(stat[:, L.STAT_NPOOL].mean()), "lost_mean": float(stat[:, L.STAT_NLOST].mean()),
                  "edges_assoc1_mean": float(stat[:, 15].mean()), "rows_left_after_kernelisation_mean": float(stat[:, 12].mean()),
                  "searches_deferred_once_mean": float(stat[:, 13].mean()), "searches_deferred_twice_mean": float(stat[:, 14].mean()),
                  "lap1_sub_cycles": {"init": sub[8], "kernelize": sub[9], "compact": sub[10], "labels": sub[11], "solve": sub[12]}}
    n_tracks = [int(v) for v in h_stat[:, L.STAT_NOUT]]
    live = [int(v) for v in stat[:, L.STAT_NTRACKED]]
    births_per_frame = float(np.mean(stat[:, L.STAT_NBIRTH]))

    # ---- conv share of the step for the tensor roofline: the conv launches replayed back to back as one CUDA graph
    def graph_ms(fns, reps=5):
        s = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(s):
            for fn in fns:
                fn()
            torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph, stream=s):
                for fn in fns:
                    fn()
            gph.replay(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            for _ in range(reps):
                gph.replay()
            b.record(s)
            torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    n_conv = sum(1 for _, fl, _ in det.ops if fl > 0)
    conv_ms = graph_ms([fn for fn, fl, _ in det.ops if fl > 0])
    other_ms = graph_ms([fn for fn, fl, _ in det.ops[1:] if fl == 0])
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); det.ingest_u8_launch(); b.record(); torch.cuda.synchronize()
    ingest_ms = a.elapsed_time(b)
    a.record(); det._nms_launch(True); b.record(); torch.cuda.synchronize()
    nms_ms = a.elapsed_time(b)
    a.record(); eng.step_device(det.out, det.out_count, pipe.t_out, pipe.t_stat); b.record(); torch.cuda.synchronize()
    trk_ms = a.elapsed_time(b)
    ingest_bytes = B * args.img * args.img * 3 + B * (args.img // 2) * (args.img // 2) * 16 * 2      # uint8 frame read + 16-channel fp16 rows written

    t = torch.tensor([dev_ms, e2e_ms] + rep_dev + rep_e2e, dtype=torch.float64, device=dev)
    births = torch.tensor([int(v) for v in stat[:, L.STAT_NEXT_ID]], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        parts = [torch.zeros_like(births) for _ in range(world)]
        dist.all_gather(parts, births)                          # the only collective of the path: per-sequence birth counts (8e)
        allb = torch.cat(parts)
    else:
        allb = births
    offsets = (torch.cumsum(allb, 0) - allb)[:8].tolist()
    # ---- C4 end to end: the same detectors and the same frames feeding BoT-SORT, the camera-motion warp ESTIMATED on the GPU from the frames
    # (consecutive pool frames differ by a (+2, +1) roll: the estimator has a true shift to find), tracks read back every step.
    # (Textured frames were tried: the seeded random-init detector, calibrated on noise, passes ~all 102 000 anchors at conf 0.01 on them
    # and the NMS alone takes 18 ms -- tools/c4_diag.py -- so the noise frames of the headline are used.)
    c4_pipe = None
    if rank == 0 and not args.no_sub:
        from b200track.gmc import GmcEstimator
        tex = dev_frames
        eng_b = TrackEngine("botsort", n_seq=B, dtype="f64", cap=1152, dmax=det.max_det, device=dev)
        gmc = GmcEstimator(B, args.img, args.img, 2, max_kp=32768, device=dev)
        pipe_b = TrackingPipeline([det, det2], eng_b, out_rows=1152, gmc=gmc)
        for k in range(8):
            pipe_b.step(tex[k % POOL])
        pipe_b.flush(); torch.cuda.synchronize()
        nb = 40
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for k in range(nb):
            pipe_b.step(tex[(8 + k) % POOL])
        rows_b, stat_b = pipe_b.flush()
        b.record(); torch.cuda.synchronize()
        ms_b = a.elapsed_time(b) / nb
        gst = gmc.stat.cpu().numpy(); gw = gmc.warps.cpu().numpy()
        c4_pipe = {"frames_per_s": B * 1e3 / ms_b, "ms_per_step": ms_b, "steps": nb, "sequences": B,
                   "what": "the headline's uint8 frames resident in HBM -> ingest -> YOLOv7-w6 -> decode + NMS -> camera-motion estimate (FAST + ORB + 2-NN + RANSAC on the "
                           "GPU, boxes of the high-score detections masked) -> BoT-SORT step with that warp -> track rows on the host, every step",
                   "keypoints_mean": float(gst[:, 0].mean()), "ransac_inliers_mean": float(gst[:, 4].mean()),
                   "last_warp_translation_px": [float(gw[:, 0, 2].mean()), float(gw[:, 1, 2].mean())], "true_motion_px_between_pool_frames": [1, 2], "gmc_flags_seen": sorted(set(int(v) for v in gst[:, 5])),
                   "tracks_out_mean": float(np.mean([int(v) for v in stat_b[:, L.STAT_NOUT]]))}
        del pipe_b, eng_b, gmc
        torch.cuda.empty_cache()
    # ---- the other BASELINE configurations, same run (every rank takes its share of C4)
    import bench_sub
    sub = bench_sub.run_all(torch, dev, rank, world, hbm_gbs, quick=args.quick_sub) if not args.no_sub else {}
    if rank == 0 and c4_pipe is not None:
        sub["C4_pipeline_botsort_with_gpu_gmc"] = c4_pipe
    if rank == 0:
        frames = B * K * world
        value = frames / (float(t[0]) / 1e3)
        e2e = frames / (float(t[1]) / 1e3)
        conv_tflops = det.flops / (conv_ms * 1e-3) / 1e12
        traffic, traffic_src, traffic_partial = conv_traffic(n_conv)
        cpu = None
        if world == 1 and not args.no_cpu:
            import bench_reference as BR
            r = BR.run_cpu_arm({k: v.cpu() for k, v in sd.items()}, args.img, 4, 1)
            cpu = {"value": r["value"], "unit": "frames/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "ms_per_frame": r["ms_per_frame"]}
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": float(t[0]) / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16", "data": "synthetic",
            "config": {"workload": _workload(args), "sequences_per_gpu": B, "frames_per_step": B,
                       "l2": "inputs larger than L2 (39 MB of uint8 frames per step, >1 GB of activations per step); no explicit flush",
                       "pipelining": "4 streams over two twin detectors (same weights and plans, own buffers): H2D + uint8 ingest / forward (CUDA graphs, back to back) / decode + NMS / associate + D2H; frame t+1 is ingested and frame t-1 post-processed and associated while frame t's forward runs",
                       "precision": "fp16 activations and weights, fp32 accumulation (the reference's GPU half mode, detect.py:41); tracker fp64",
                       "tracks_out_per_sequence": n_tracks, "tracked_per_sequence": live, "births_per_frame_per_sequence": births_per_frame,
                       "association_load_note": ("the detector runs on seeded noise frames, so its 300 detections per frame are not temporally coherent: "
                                                 "the tracker sees ~%.0f births per frame instead of C3's ~250 persistent tracks (the C3 load is measured "
                                                 "separately in sub_benchmarks)" % births_per_frame),
                       "global_id_offsets": offsets,
                       "track_step_phase_cycles": phases, "track_step_load": pool_sizes,
                       "ms_breakdown_per_step": {"ingest_u8": ingest_ms, "conv": conv_ms, "glue": other_ms, "nms": nms_ms, "track_step": trk_ms},
                       "ingest": {"kernel": "letterbox_reorg_kernel", "bytes_per_step": ingest_bytes, "GBs": ingest_bytes / (ingest_ms * 1e-3) / 1e9,
                                  "frac_of_hbm": ingest_bytes / (ingest_ms * 1e-3) / 1e9 / hbm_gbs},
                       "repeats": {"note": "the same K timed steps run 3 times (max over ranks each): frames/s",
                                   "value": [frames / (float(v) / 1e3) for v in t[2:5]], "e2e": [frames / (float(v) / 1e3) for v in t[5:8]]},
                       "sub_benchmarks": sub},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(B * args.img * args.img * 3),
                    "d2h_bytes_per_step": int(h_out.numel() * 8 + h_stat.numel() * 4), "ms_per_step": float(t[1]) / K},
            "gpu_launches": int(K * n_graph_kernels + tracker_launches),
            "roofline": {"bound": "tensor", "kernel": "conv_bias_act_kernel (%d launches per step: the 107 convs of the graph, ELAN 1x1 pairs stacked)" % n_conv,
                         "achieved": conv_tflops, "peak": tf_peak, "unit": "TFLOP/s", "frac": conv_tflops / tf_peak, "traffic": traffic,
                         "traffic_unit": "bytes per step (all conv launches)", "traffic_source": traffic_src, "traffic_partial": traffic_partial,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (a kernel timed inside a long step)" if peaks else "fallback 1400 (sustained)",
                         "algorithmic_flops_per_step": det.flops, "conv_ms_per_step": conv_ms,
                         "note": "algorithmic 2 x MAC of the 107 convs (SURVEY 8d: 359.7 GFLOP/img; the 255-channel heads are counted at 255) x batch / "
                                 "CUDA-event time of the conv launches replayed back to back as one graph"},
            "cpu_baseline": cpu,
            "clocks": clocks,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            from bench import dump_outputs
            dump_outputs(args.dump_outputs, last_outputs)
    if world > 1:
        dist.destroy_process_group()
