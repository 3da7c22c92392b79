"""Seeded synthetic detection streams (SURVEY.md section 8d "Synthetic inputs").

There is no dataset and no detector checkpoint in the reference (weights/ has no YOLO
weights), so every tracker-side test, golden fixture and bench line is driven by these
streams.  A stream is what ``tracker/track.py:149`` hands to ``tracker.update``: per frame an
``(n, 6)`` float32 array ``[x1, y1, x2, y2, score, cls]`` with integer-rounded, clipped
coordinates (q9) sorted by descending score (q13: NMS output order).
"""
import hashlib

import numpy as np


def make_stream(seed, n_frames, n_obj=300, img=1280, miss=0.05, warp_sigma=0.0):
    """Returns (frames, warps): list of (n_i, 6) float32 arrays and a (n_frames, 2, 3) float64
    array of per-frame camera warps (identity rotation, N(0, warp_sigma) translation)."""
    rng = np.random.default_rng(seed)
    cx = rng.uniform(200, img - 200, n_obj)
    cy = rng.uniform(200, img - 200, n_obj)
    w = rng.uniform(20, 80, n_obj)
    h = rng.uniform(40, 160, n_obj)
    vx = rng.normal(0, 1, n_obj)
    vy = rng.normal(0, 1, n_obj)
    cls = rng.integers(0, 3, n_obj).astype(np.float32)
    frames = []
    warps = np.zeros((n_frames, 2, 3), dtype=np.float64)
    warps[:, 0, 0] = warps[:, 1, 1] = 1.0
    cam = np.zeros(2)
    for f in range(n_frames):
        cx += vx
        cy += vy
        # bounce on the borders so the population stays inside the frame
        bx = (cx < 60) | (cx > img - 60)
        by = (cy < 60) | (cy > img - 60)
        vx[bx] = -vx[bx]
        vy[by] = -vy[by]
        if warp_sigma > 0:
            t = rng.normal(0, warp_sigma, 2)
            warps[f, :, 2] = t
            cam += t
        jit = rng.normal(0, 1, (n_obj, 4))
        score = rng.uniform(0.05, 0.95, n_obj).astype(np.float32)
        keep = rng.uniform(0, 1, n_obj) >= miss
        x1 = cx - w / 2 + jit[:, 0] + cam[0]
        y1 = cy - h / 2 + jit[:, 1] + cam[1]
        x2 = cx + w / 2 + jit[:, 2] + cam[0]
        y2 = cy + h / 2 + jit[:, 3] + cam[1]
        box = np.stack([x1, y1, x2, y2], 1)
        box = np.round(np.clip(box, 0, img))
        ok = keep & ((box[:, 2] - box[:, 0]) >= 4) & ((box[:, 3] - box[:, 1]) >= 4)
        d = np.concatenate([box[ok], score[ok, None], cls[ok, None]], 1).astype(np.float32)
        order = np.argsort(-d[:, 4], kind="stable")
        frames.append(np.ascontiguousarray(d[order]))
    return frames, warps


def make_vanish_stream(seed, n_frames, per_frame=3, img=1280):
    """Seeded stream of short-lived objects: every frame starts `per_frame` new objects that move for 3..8 frames and vanish
    (C-BIoU never prunes its lost tracks, so this stream grows the lost list without bound).
    Per frame an (n, 6) float32 [x1, y1, x2, y2, score, cls] array, integer-rounded boxes, sorted by descending score."""
    rng = np.random.default_rng(seed)
    objs = []
    frames = []
    for f in range(n_frames):
        for _ in range(per_frame):
            cx, cy = rng.uniform(100, img - 100, 2)
            w, h = rng.uniform(20, 80), rng.uniform(40, 160)
            objs.append([cx, cy, w, h, rng.normal(0, 3), rng.normal(0, 3), f + int(rng.integers(3, 9)), float(rng.integers(0, 3))])
        rows = []
        for o in objs:
            if o[6] <= f:
                continue
            o[0] += o[4]; o[1] += o[5]
            box = np.round(np.clip([o[0] - o[2] / 2, o[1] - o[3] / 2, o[0] + o[2] / 2, o[1] + o[3] / 2] + rng.normal(0, 1, 4), 0, img))
            rows.append([*box, rng.uniform(0.3, 0.95), o[7]])
        objs = [o for o in objs if o[6] > f]
        d = np.array(rows, np.float32).reshape(-1, 6)
        frames.append(np.ascontiguousarray(d[np.argsort(-d[:, 4], kind="stable")]))
    return frames


def stream_digest(frames):
    """sha1 of the raw bytes: stored with golden fixtures to detect generator drift."""
    hsh = hashlib.sha1()
    for f in frames:
        hsh.update(np.ascontiguousarray(f, dtype=np.float32).tobytes())
    return hsh.hexdigest()


def pack_frames(frames, max_dets=None):
    """List of ragged (n_i,6) arrays -> (dets (F, D, 6) float32 zero padded, counts (F,) int32)."""
    d = max(len(f) for f in frames) if max_dets is None else max_dets
    out = np.zeros((len(frames), d, 6), dtype=np.float32)
    cnt = np.zeros(len(frames), dtype=np.int32)
    for i, f in enumerate(frames):
        n = min(len(f), d)
        out[i, :n] = f[:n]
        cnt[i] = n
    return out, cnt


def textured_frame(seed, height=720, width=1280, n_rect=400):
    """Seeded uint8 BGR frame with corners for the camera-motion estimator (SURVEY.md 8f row 1): smooth multi-scale noise plus
    random rectangles of random grey level and a little pixel noise.  NumPy only (the bench must not need OpenCV)."""
    rng = np.random.default_rng(seed)
    img = np.full((height, width), 128.0, dtype=np.float32)
    for s, a in ((64, 40.0), (16, 30.0), (4, 12.0)):
        n = rng.standard_normal((height // s + 2, width // s + 2)).astype(np.float32)
        up = np.kron(n, np.ones((s, s), dtype=np.float32))
        # box-smooth the blocks once so that the field is continuous
        up = (up[: height + s, : width + s][s // 2: s // 2 + height, s // 2: s // 2 + width] + up[:height, :width]) * 0.5
        img += a * up
    for _ in range(n_rect):
        x, y = int(rng.integers(0, width - 8)), int(rng.integers(0, height - 8))
        w, h = int(rng.integers(6, 60)), int(rng.integers(6, 60))
        img[y:y + h, x:x + w] += float(rng.uniform(-70, 70))
    img += rng.standard_normal((height, width)).astype(np.float32) * 2.0
    g = np.clip(img, 0, 255)
    bgr = np.stack([g * 0.9 + 10, g, g * 0.8 + 25], -1)
    return np.clip(bgr, 0, 255).astype(np.uint8)
