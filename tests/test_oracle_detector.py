"""not-gpu: the torch oracle of the detector against the committed outputs of the reference's own Model
(tests/golden/detector_w6.npz) -- pins both oracle/detector.py and the product's graph builder (w6_layers)."""
import os
import sys

import numpy as np
import torch

from b200track.w6 import ANCHORS, STRIDES, conv_shapes, layer_channels, seeded_state_dict, w6_layers
from oracle import detector as OD

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "detector_w6.npz")
REFCHECKS = os.path.join(os.path.dirname(__file__), "golden", "refchecks.npz")
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))


def test_graph_bookkeeping():
    layers = w6_layers()
    assert len(layers) == 119 and layers[-1][1] == "detect"
    ch = layer_channels(layers)
    assert ch[46] == 1024 and ch[47] == 512 and ch[83] == 128 and ch[117] == 1024 and ch[9] == 256 and ch[58] == 1536
    shapes = conv_shapes(layers)
    assert len(shapes) == 107                                    # SURVEY 8(a): 107 convs after fusion
    n_params = sum(ci * co * k * k + co for _, ci, co, k, s, _ in shapes)
    assert abs(n_params - 70.43e6) / 70.43e6 < 0.01              # 70.4 M parameters (SURVEY 8a)


def test_stackable_1x1_pairs_and_rowpack_layout():
    """Host logic of the detector planner: the 11 ELAN blocks each open with two 1x1 convs of the same input that are adjacent
    in the block's concat; the row-packed stem weight layout is k = kh*64 + kw*16 + c with a zero fourth pixel."""
    from b200track.w6 import stackable_pairs
    pairs = stackable_pairs()
    assert len(pairs) == 11 and pairs[0] == (3, 4) and (12, 13) in pairs and (50 + 2, 50 + 3) in pairs
    layers = w6_layers()
    for a, b in pairs:
        assert layers[a][1] == layers[b][1] == "conv" and layers[a][3] == layers[b][3] and layers[b][2] == -2
    from b200track.conv import pack_conv_weight_rowpack
    w = torch.arange(64 * 12 * 9, dtype=torch.float32).reshape(64, 12, 3, 3) / 4096.0
    pk = pack_conv_weight_rowpack(w).float().reshape(64, 3, 4, 16)
    assert torch.equal(pk[:, :, :3, :12], w.to(torch.bfloat16).float().permute(0, 2, 3, 1))
    assert bool((pk[:, :, 3] == 0).all()) and bool((pk[:, :, :, 12:] == 0).all())


def test_oracle_forward_and_nms_match_reference_golden():
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    g = np.load(GOLDEN)
    sd = seeded_state_dict(0)
    gen = torch.Generator().manual_seed(123)
    img = torch.rand((1, 3, 256, 256), generator=gen)
    with torch.no_grad():
        pred = OD.forward(w6_layers(), sd, img, ANCHORS, STRIDES)
    assert tuple(pred.shape) == tuple(g["pred_shape"])
    np.testing.assert_allclose(pred[0, g["rows"]].numpy(), g["pred_rows"], rtol=2e-3, atol=2e-3)
    assert int((pred[0, :, 4] > 0.01).sum()) == int(g["n_candidates"])
    dets = OD.non_max_suppression(pred, conf_thres=0.01)[0].numpy()
    ref = g["dets"]
    assert dets.shape == ref.shape
    assert np.array_equal(dets[:, 5], ref[:, 5])                 # classes and order: exact
    np.testing.assert_allclose(dets[:, :5], ref[:, :5], rtol=2e-3, atol=2e-2)


def test_fold_batchnorm_and_implicit_layers_math():
    """fold_reference_state_dict on a synthetic one-layer problem: Conv + BN(eval) and ia / m / im head == the folded convs."""
    import torch.nn.functional as F
    from b200track.w6 import conv_shapes, fold_reference_state_dict
    g = torch.Generator().manual_seed(1)
    sd = {}
    for name, cin, cout, k, s, act in conv_shapes():
        if act:
            sd[name + ".weight"] = torch.randn((cout, cin, k, k), generator=g) * 0.05
            pre = name[:-len(".conv")]
            sd[pre + ".bn.weight"] = torch.rand(cout, generator=g) + 0.5
            sd[pre + ".bn.bias"] = torch.randn(cout, generator=g) * 0.1
            sd[pre + ".bn.running_mean"] = torch.randn(cout, generator=g) * 0.1
            sd[pre + ".bn.running_var"] = torch.rand(cout, generator=g) + 0.2
        else:
            j = int(name.rsplit(".", 1)[1])
            sd["model.122.m.%d.weight" % j] = torch.randn((cout, cin, 1, 1), generator=g) * 0.05
            sd["model.122.m.%d.bias" % j] = torch.randn(cout, generator=g) * 0.1
            sd["model.122.m2.%d.weight" % j] = torch.zeros((cout, 8, 1, 1))
            sd["model.122.ia.%d.implicit" % j] = torch.randn((1, cin, 1, 1), generator=g) * 0.02
            sd["model.122.im.%d.implicit" % j] = 1 + torch.randn((1, cout, 1, 1), generator=g) * 0.02
    out = fold_reference_state_dict(sd)
    assert set(out) == {n + s for n, *_ in conv_shapes() for s in (".weight", ".bias")}
    name = "model.5.conv"                                             # a 3x3 Conv + BN
    x = torch.randn((1, 64, 9, 9), generator=g)
    pre = "model.5"
    ref = F.batch_norm(F.conv2d(x, sd[name + ".weight"], None, padding=1), sd[pre + ".bn.running_mean"], sd[pre + ".bn.running_var"],
                       sd[pre + ".bn.weight"], sd[pre + ".bn.bias"], False, 0.03, 1e-3)
    got = F.conv2d(x, out[name + ".weight"], out[name + ".bias"], padding=1)
    assert torch.allclose(got, ref, atol=1e-5)
    x = torch.randn((1, 256, 5, 5), generator=g)                      # head 0: m(ia + x) * im
    ref = F.conv2d(x + sd["model.122.ia.0.implicit"], sd["model.122.m.0.weight"], sd["model.122.m.0.bias"]) * sd["model.122.im.0.implicit"]
    got = F.conv2d(x, out["model.118.m.0.weight"], out["model.118.m.0.bias"])
    assert torch.allclose(got, ref, atol=1e-5)
    assert fold_reference_state_dict(out).keys() == out.keys()        # an already fused dict passes through


def test_fold_training_checkpoint_equals_reference_inference():
    """The reference's own TRAINING graph (cfg/training/yolov7-w6.yaml: Conv + BN, aux heads, IAuxDetect with implicit layers) on
    seeded weights for its whole state dict, with seeded BN statistics, evaluated by the reference in eval mode
    (tests/golden/refchecks.npz) == the oracle forward on the deploy-graph weights folded from that whole state dict."""
    from b200track.w6 import fold_reference_state_dict
    from make_golden_refchecks import stored_shapes, training_state_dict, w6train_image
    g = np.load(REFCHECKS)
    anchors = {k.split("/", 1)[1]: g[k] for k in g.files if k.startswith("w6train_anchor/")}
    sd = training_state_dict(stored_shapes(g["w6train_keys"], g["w6train_key_shapes"]), anchors)
    assert len(sd) == len(g["w6train_keys"]) and any(k.startswith("model.121.bn.") for k in sd) and any(".m2." in k for k in sd)
    folded = fold_reference_state_dict(sd)
    with torch.no_grad():
        got = OD.forward(w6_layers(), folded, w6train_image(), ANCHORS, STRIDES)
    assert tuple(got.shape) == tuple(g["w6train_shape"])
    np.testing.assert_allclose(got[0, g["w6train_rows"]].numpy(), g["w6train_pred_rows"], rtol=2e-3, atol=2e-3)
    np.testing.assert_allclose(got[0, :, 4].numpy(), g["w6train_obj"], rtol=2e-3, atol=2e-3)


def test_pickled_checkpoint_is_refused_and_converted(tmp_path):
    """The reference's checkpoints pickle the whole nn.Module (its models/experimental.py:83-106).  The drop-in attempt_load refuses
    such a file with a message that names tools/export_state_dict.py, and the converter, pointed at the package that defines the
    pickled classes (a stand-in ``models.yolo.Model`` under tmp_path), writes the module's floating-point state dict."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    (tmp_path / "models").mkdir()
    (tmp_path / "models" / "__init__.py").write_text("")
    (tmp_path / "models" / "yolo.py").write_text(
        "import torch\n\nclass Model(torch.nn.Module):\n    def __init__(self):\n        super().__init__()\n"
        "        self.conv = torch.nn.Conv2d(3, 8, 3)\n        self.bn = torch.nn.BatchNorm2d(8)\n")
    ckpt, expect, out = tmp_path / "pickled.pt", tmp_path / "expect.pt", tmp_path / "state.pt"
    make = ("import sys, torch\nsys.path.insert(0, %r)\nfrom models.yolo import Model\ntorch.manual_seed(3)\nm = Model()\n"
            "torch.save({'model': m, 'ema': None, 'epoch': -1}, %r)\ntorch.save(m.state_dict(), %r)\n" % (str(tmp_path), str(ckpt), str(expect)))
    r = subprocess.run([sys.executable, "-c", make], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    code = ("import sys; sys.path.insert(0, %r); from models.experimental import attempt_load\n"
            "try:\n    attempt_load(%r, map_location='cpu')\nexcept RuntimeError as e:\n    print('MSG', str(e))\n"
            % (os.path.join(root, "yolov7-tracker_b200"), str(ckpt)))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert "MSG" in r.stdout and "tools/export_state_dict.py" in r.stdout, r.stdout + r.stderr
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "export_state_dict.py"), "--reference", str(tmp_path),
                        "--weights", str(ckpt), "--out", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    got, ref = torch.load(str(out), weights_only=True), torch.load(str(expect), weights_only=True)
    assert set(got) == {k for k, v in ref.items() if v.is_floating_point()} and len(got) == 6
    assert all(torch.equal(got[k], ref[k]) for k in got)


def test_tiny_oracle_equals_reference_model():
    """YOLOv7-tiny (cfg/deploy/yolov7-tiny.yaml: LeakyReLU convs, MP / SP pools, three-level Detect): the oracle's restatement of the
    graph against the reference's own ``Model`` (fused, eval, CPU) on the same seeded weights (tests/golden/refchecks.npz)."""
    from b200track import tiny
    from make_golden_refchecks import stored_shapes, tiny_image
    g = np.load(REFCHECKS)
    sd = tiny.seeded_state_dict(0)
    msd = stored_shapes(g["tiny_keys"], g["tiny_key_shapes"])
    assert all(k in msd and msd[k] == tuple(v.shape) for k, v in sd.items()), [k for k in sd if k not in msd][:3]
    with torch.no_grad():
        got = OD.forward(tiny.tiny_layers(), sd, tiny_image(), tiny.ANCHORS, tiny.STRIDES, act="leaky", name_offset=-1).numpy()
    assert tuple(g["tiny_shape"]) == got.shape == (2, 3 * (24 * 32 + 12 * 16 + 6 * 8), 85)
    assert float(np.abs(got[:, g["tiny_rows"]] - g["tiny_pred_rows"]).max()) < 2e-3
    assert float(np.abs(got[..., 4] - g["tiny_obj"]).max()) < 1e-5
