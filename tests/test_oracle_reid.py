"""Pins oracle/reid.py (restatement of tracker/reid_models/deepsort_reid.py) against what the UNMODIFIED reference computed on the
same seeded crops and weights (tests/golden/refchecks.npz).  CPU tier."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "yolov7-tracker_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
from oracle import reid as R  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "refchecks.npz")


def test_restatement_equals_reference_net_and_preprocess():
    """Against tests/golden/refchecks.npz (tests/golden/make_golden_refchecks.py): the reference Extractor's _preprocess of the same
    seeded crops, and the reference's own Net on the seeded weights in eval mode, in training mode (the extractor's mode), and in
    eval mode after that training-mode call updated the BatchNorm buffers."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden_refchecks import REID_CROPS
    g = np.load(GOLDEN)
    crops = R.seeded_crops(*REID_CROPS)
    x = R.preprocess(crops)
    assert tuple(x.shape) == tuple(g["reid_x_shape"])
    xs = x.numpy()                                              # cv2.resize on float data, restated
    assert float(np.abs(xs.reshape(-1)[g["reid_x_index"]] - g["reid_x_values"]).max()) < 2e-6
    assert np.all(np.abs(xs.astype(np.float64).sum(axis=(1, 2, 3)) - g["reid_x_sums"]) < 2e-6 * xs[0].size)
    assert bool(g["reid_extractor_training"])                   # the quirk: the reference never switches its extractor to eval()
    seeded = R.seeded_state_dict(3)
    ref_keys = set(g["reid_net_keys"].tolist())
    assert not [k for k in ref_keys - set(seeded) if "classifier" not in k and "num_batches_tracked" not in k] and not set(seeded) - ref_keys
    with torch.no_grad():
        assert float(np.abs(R.forward(seeded, x, batch_stats=False).numpy() - g["reid_eval"]).max()) < 2e-5
        assert float(np.abs(R.forward(seeded, x, batch_stats=True).numpy() - g["reid_train"]).max()) < 2e-5
    sd_after = dict(seeded)
    sd_after.update({k.split("/", 1)[1]: torch.from_numpy(g[k]) for k in g.files if k.startswith("reid_after/")})
    with torch.no_grad():
        assert float(np.abs(R.forward(sd_after, x, batch_stats=False).numpy() - g["reid_eval_after"]).max()) < 2e-5


def test_seeded_network_is_well_conditioned():
    """The seeded stand-in weights give distinct, unit-norm features (the GPU parity test is meaningful on them)."""
    with torch.no_grad():
        f = R.forward(R.seeded_state_dict(3), R.preprocess(R.seeded_crops(1, 6)), batch_stats=True)
    assert torch.allclose(f.norm(dim=1), torch.ones(6), atol=1e-5)
    cos = (f @ f.T).numpy()
    assert np.all(cos[~np.eye(6, dtype=bool)] < 0.999)
