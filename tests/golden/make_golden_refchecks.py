"""Runs the UNMODIFIED reference (a checkout of JackWoo0831/Yolov7-tracker, path in B2T_REFERENCE_ROOT) once and stores what the
reference-comparing CPU tests compare against in tests/golden/refchecks.npz, so that those tests need nothing outside this repository:

  reid_*     tracker/reid_models/deepsort_reid.py: ``Extractor._preprocess`` on seeded crops (a seeded sample of its elements and
             per-crop sums), whether the extractor leaves its net in training mode, the state dict names of ``Net(reid=True)``,
             and that net on the seeded stand-in weights in eval mode, in training mode, and in eval mode after that
             training-mode call updated the BatchNorm buffers;
  w6train_*  models/yolo.py ``Model(cfg/training/yolov7-w6.yaml)`` (BatchNorm, auxiliary heads, IAuxDetect): its state dict's
             names and shapes and its Detect anchors, and, in eval mode on the seeded weights of ``training_state_dict`` below,
             a seeded sample of the output rows and the whole objectness column;
  tiny_*     ``Model(cfg/deploy/yolov7-tiny.yaml)`` (fused, eval) on ``b200track.tiny.seeded_state_dict(0)``: its state dict's names
             and shapes, a seeded sample of the output rows and the whole objectness column;
  gmc_H      tracker/botsort.py ``GMC(method='orb', downscale=2).apply`` over ``gmc_sequence()``;
  results_*  tracker/track.py ``save_results`` on ``results_frames()``, one file per data type.

    B2T_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden_refchecks.py
"""
import ast
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "yolov7-tracker_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

OUT = os.path.join(ROOT, "tests", "golden", "refchecks.npz")
REID_CROPS = (9, 5)                  # oracle.reid.seeded_crops(seed, n)
REID_SAMPLE = 8192                   # elements of the preprocessed batch kept
ROW_SAMPLE = 96                      # detector output rows kept per image


def sample_index(n, k, seed):
    """A fixed, seeded, sorted choice of k of n indices (all of them when k >= n)."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def stored_shapes(names, shapes):
    """{name: shape} from the two string arrays the generator stores for a reference state dict."""
    return {k: tuple(int(d) for d in v.split(",") if d) for k, v in zip(names.tolist(), shapes.tolist())}


def training_state_dict(shapes, anchors, seed=3):
    """A state dict with every name and shape of the reference's training graph (``shapes``: cfg/training/yolov7-w6.yaml).  The
    seeded deploy-graph weights (b200track.w6.seeded_state_dict(0)) are written in the training graph's format: every activated
    conv gets a BatchNorm with seeded statistics and the conv weight / BN bias that fold back to the deploy weights, the Detect head
    (index 122) gets seeded implicit ``ia`` / ``im`` tensors.  The names inference does not use (the auxiliary convs 118-121 and
    their BatchNorm, ``m2``) get seeded values, ``num_batches_tracked`` zero, and the Detect anchors the reference's own
    (``anchors``: {name: array})."""
    from b200track.w6 import conv_shapes, seeded_state_dict
    sd = seeded_state_dict(0)
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, cin, cout, k, s, act in conv_shapes():
        w, b = sd[name + ".weight"].float(), sd[name + ".bias"].float()
        if act:
            pre = name[:-len(".conv")]
            gamma = torch.rand(cout, generator=g) * 0.5 + 1.2
            var = torch.rand(cout, generator=g) * 0.5 + 0.75
            mu = torch.randn(cout, generator=g) * 0.1
            scale = gamma / torch.sqrt(var + 1e-3)
            out[name + ".weight"] = w / scale.view(-1, 1, 1, 1)
            out[pre + ".bn.weight"], out[pre + ".bn.bias"] = gamma, b + mu * scale
            out[pre + ".bn.running_mean"], out[pre + ".bn.running_var"] = mu, var
        else:
            j = int(name.rsplit(".", 1)[1])
            out["model.122.m.%d.weight" % j], out["model.122.m.%d.bias" % j] = w, b
            out["model.122.ia.%d.implicit" % j] = torch.randn((1, cin, 1, 1), generator=g) * 0.02
            out["model.122.im.%d.implicit" % j] = 1 + torch.randn((1, cout, 1, 1), generator=g) * 0.02
    assert set(out) <= set(shapes) and all(tuple(v.shape) == shapes[k] for k, v in out.items())
    for k, shape in shapes.items():
        if k in anchors:
            out[k] = torch.from_numpy(np.asarray(anchors[k]))
        elif k.endswith(".num_batches_tracked"):
            out[k] = torch.tensor(0)
        elif k not in out:
            out[k] = torch.rand(shape, generator=g) * 0.5 + 0.75
    return out


def w6train_image():
    return torch.rand((1, 3, 128, 128), generator=torch.Generator().manual_seed(3))


def tiny_image():
    return torch.rand((2, 3, 192, 256), generator=torch.Generator().manual_seed(5))


def gmc_sequence():
    """Four textured 720 x 1280 frames moved by seeded small rotations / scalings / shifts, and the detections that follow them."""
    import cv2
    from b200track.synth import textured_frame
    f = textured_frame(11, 720, 1280)
    dets = np.array([[200, 100, 420, 500, 0.9, 0], [700, 300, 900, 640, 0.7, 1]], np.float32)
    rng = np.random.default_rng(0)
    seq = []
    for k in range(4):
        seq.append((f, dets))
        true = (float(rng.uniform(-6, 6)), float(rng.uniform(-6, 6)))
        angle, scale = float(rng.uniform(-0.5, 0.5)), 1.0 + float(rng.uniform(-0.004, 0.004))
        h, w = f.shape[:2]
        M = cv2.getRotationMatrix2D((w / 2, h / 2), angle, scale)
        M[:, 2] += true
        f = cv2.warpAffine(f, M, (w, h), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT_101)
        dets = dets + np.array([true[0], true[1], true[0], true[1], 0, 0], np.float32)
    return seq


def results_frames():
    """Four frames of seeded track rows (id, x, y, w, h, class, ...) for the result writers."""
    rng = np.random.default_rng(3)
    frames = []
    for k in range(4):
        n = int(rng.integers(1, 6))
        rows = np.zeros((n, 8))
        rows[:, 0] = rng.integers(1, 500, n)
        rows[:, 1:5] = rng.uniform(0, 1280, (n, 4)).round(3)
        rows[:, 5] = rng.integers(0, 10, n)
        frames.append(rows)
    return frames


def _reid(ref, out):
    from oracle import reid as R
    sys.path.insert(0, os.path.join(ref, "tracker"))
    try:
        from reid_models import deepsort_reid as M
    finally:
        sys.path.remove(os.path.join(ref, "tracker"))
        for k in [k for k in sys.modules if k.startswith("reid_models")]:
            del sys.modules[k]
    crops = R.seeded_crops(*REID_CROPS)
    ext = M.Extractor(os.path.join(ref, "weights", "ckpt.t7"), use_cuda=False)
    x_ref = ext._preprocess(crops).numpy()
    idx = sample_index(x_ref.size, REID_SAMPLE, 1)
    out["reid_x_index"], out["reid_x_values"] = idx, x_ref.reshape(-1)[idx]
    out["reid_x_shape"], out["reid_x_sums"] = np.array(x_ref.shape), x_ref.astype(np.float64).sum(axis=(1, 2, 3))
    out["reid_extractor_training"] = np.array(bool(ext.net.training))
    x = R.preprocess(crops)
    net = M.Net(reid=True).eval()
    out["reid_net_keys"] = np.array(list(net.state_dict()))
    net.load_state_dict(R.seeded_state_dict(3), strict=False)
    with torch.no_grad():
        out["reid_eval"] = net(x).numpy()
        out["reid_train"] = net.train()(x).numpy()                # also updates the BatchNorm running buffers
        out["reid_eval_after"] = net.eval()(x).numpy()
    for k, v in net.state_dict().items():
        if k.endswith((".running_mean", ".running_var")):
            out["reid_after/" + k] = v.numpy()


def _detectors(out):
    from b200track import tiny
    from oracle import refshim
    model = refshim.load_detector_model("cfg/training/yolov7-w6.yaml", fuse=False)
    msd = model.state_dict()
    out["w6train_keys"] = np.array(list(msd))
    out["w6train_key_shapes"] = np.array([",".join(str(d) for d in v.shape) for v in msd.values()])
    anchors = {k: v.numpy() for k, v in msd.items() if k.endswith((".anchors", ".anchor_grid"))}
    out.update({"w6train_anchor/" + k: v for k, v in anchors.items()})
    model.load_state_dict(training_state_dict(stored_shapes(out["w6train_keys"], out["w6train_key_shapes"]), anchors), strict=True)
    with torch.no_grad():
        pred = model(w6train_image())[0][0].numpy()
    rows = sample_index(pred.shape[0], ROW_SAMPLE, 2)
    out["w6train_shape"], out["w6train_rows"], out["w6train_pred_rows"] = np.array((1,) + pred.shape), rows, pred[rows]
    out["w6train_obj"] = pred[:, 4]
    model = refshim.load_detector_model("cfg/deploy/yolov7-tiny.yaml")
    msd = model.state_dict()
    out["tiny_keys"] = np.array(list(msd))
    out["tiny_key_shapes"] = np.array([",".join(str(d) for d in v.shape) for v in msd.values()])
    model.load_state_dict(tiny.seeded_state_dict(0), strict=False)
    with torch.no_grad():
        pred = model(tiny_image())[0].numpy()
    rows = sample_index(pred.shape[1], ROW_SAMPLE, 3)
    out["tiny_shape"], out["tiny_rows"], out["tiny_pred_rows"] = np.array(pred.shape), rows, pred[:, rows]
    out["tiny_obj"] = pred[..., 4]


def _gmc(out):
    from oracle import refshim
    gmc = refshim.load().botsort.GMC(method='orb', downscale=2)
    out["gmc_H"] = np.stack([gmc.apply(f, d) for f, d in gmc_sequence()]).astype(np.float64)


def _results(ref, out):
    src = os.path.join(ref, "tracker", "track.py")
    fn = next(n for n in ast.parse(open(src).read()).body if isinstance(n, ast.FunctionDef) and n.name == "save_results")
    ns = {"os": os}
    exec(compile(ast.Module([fn], []), src, "exec"), ns)
    frames = results_frames()
    results = [(k + 1, [int(r[0]) for r in rows], [r[1:5] for r in rows], [r[5] for r in rows]) for k, rows in enumerate(frames)]
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for data_type in ("mot17", "default"):
                ns["save_results"](data_type, "seq", results, data_type=data_type)
                out["results_" + data_type] = np.array(open(os.path.join("tracker", "results", data_type, "seq.txt")).read())
        finally:
            os.chdir(cwd)


if __name__ == "__main__":
    from oracle import refshim
    if not refshim.available():
        sys.exit("set B2T_REFERENCE_ROOT to a checkout of the reference")
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    out = {}
    _reid(refshim.REF_ROOT, out)
    _detectors(out)
    _gmc(out)
    _results(refshim.REF_ROOT, out)
    np.savez_compressed(OUT, **out)
    print("wrote %s (%d KB): %s" % (OUT, os.path.getsize(OUT) // 1024, sorted(k for k in out if "/" not in k)))
