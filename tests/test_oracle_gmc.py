"""Pins oracle/gmc.py (the restatement of tracker/botsort.py:111-235, GMC method 'orb') stage by stage against the cv2 calls the
reference makes, and end to end against what the UNMODIFIED reference class computed (tests/golden).  CPU tier."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "yolov7-tracker_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

cv2 = pytest.importorskip("cv2")
from oracle import gmc as G                      # noqa: E402
from b200track.synth import textured_frame      # noqa: E402


def moved(frame, angle_deg, scale, tx, ty):
    h, w = frame.shape[:2]
    M = cv2.getRotationMatrix2D((w / 2, h / 2), angle_deg, scale)
    M[:, 2] += (tx, ty)
    return cv2.warpAffine(frame, M, (w, h), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT_101), M


@pytest.mark.parametrize("shape", [(360, 480), (362, 486), (375, 481)])
def test_gray_half_equals_cv2(shape):
    f = textured_frame(3, *shape)
    ref = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
    ref = cv2.resize(ref, (shape[1] // 2, shape[0] // 2))
    assert np.array_equal(G.gray_half(f, 2), ref)


def test_fast_keypoints_equal_cv2_with_mask():
    g = G.gray_half(textured_frame(4, 720, 960), 2)
    dets = np.array([[100, 80, 300, 400, 0.9, 0], [500, 200, 640, 700, 0.8, 1], [0, 0, 50, 60, 0.5, 0]], np.float32)
    mask = G.keypoint_mask(g.shape, dets, 2)
    kp = cv2.FastFeatureDetector_create(20).detect(g, mask)
    xs, ys, sc = G.fast_keypoints(g, mask)
    assert len(kp) > 500
    assert [(int(k.pt[0]), int(k.pt[1]), int(k.response)) for k in kp] == list(zip(xs.tolist(), ys.tolist(), sc.tolist()))


def test_orb_descriptors_equal_cv2():
    total = bad = 0
    for seed in (5, 6):
        g = G.gray_half(textured_frame(seed, 720, 960), 2)
        kp = cv2.FastFeatureDetector_create(20).detect(g, None)
        kp2, d = cv2.ORB_create().compute(g, kp)
        xs, ys, _ = G.fast_keypoints(g)
        keep = G.orb_filter_border(xs, ys, g.shape)
        xs, ys = xs[keep], ys[keep]
        assert [(int(k.pt[0]), int(k.pt[1])) for k in kp2] == list(zip(xs.tolist(), ys.tolist()))
        mine = G.orb_descriptors(g, xs, ys)
        total += d.size
        bad += int((mine != d).sum())
    # the float blur's rounding ties (a handful of pixels per million) are the only tolerated difference
    assert bad <= total * 1e-4, (bad, total)


def test_knn2_equals_bfmatcher():
    f0 = textured_frame(7, 720, 960)
    f1, _ = moved(f0, 0.6, 1.003, 4.2, -3.1)
    o = G.GMCOracle()
    _, xs0, ys0, d0 = o.stages(f0)
    _, xs1, ys1, d1 = o.stages(f1)
    knn = cv2.BFMatcher(cv2.NORM_HAMMING).knnMatch(d0, d1, 2)
    i1, b1, i2, b2 = G.knn2(d0, d1)
    assert all(m[0].trainIdx == i1[q] and m[0].distance == b1[q] and m[1].trainIdx == i2[q] and m[1].distance == b2[q] for q, m in enumerate(knn))


def test_estimate_equals_reference_class():
    """The whole recipe against the reference's own GMC(method='orb', downscale=2).apply over a short moving sequence with
    detections masked out (tests/golden/refchecks.npz): same key points, same matches -> the same cv2.estimateAffinePartial2D
    input -> the same matrix."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden_refchecks import gmc_sequence
    g = np.load(os.path.join(ROOT, "tests", "golden", "refchecks.npz"))
    orc = G.GMCOracle(estimator="cv2")
    own = G.GMCOracle(estimator="restated")
    for k, (f, dets) in enumerate(gmc_sequence()):
        Hr = g["gmc_H"][k]
        Ho = orc.apply(f, dets)
        Hw = own.apply(f, dets)
        np.testing.assert_allclose(Ho, Hr, rtol=0, atol=1e-9)
        if k:
            # the restated RANSAC (own sampling sequence) against OpenCV's: within the spread of its own random sampling
            assert np.abs(Hw[:, :2] - Hr[:, :2]).max() < 1e-3 and np.abs(Hw[:, 2] - Hr[:, 2]).max() < 0.25, (Hw, Hr)


def test_oracle_reproduces_committed_reference_golden():
    """tests/golden/gmc.npz = the matrices of the UNMODIFIED reference GMC class (tests/golden/make_golden_gmc.py): the restatement with
    cv2's estimator reproduces them exactly, with the restated RANSAC within OpenCV's sampling spread."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden_gmc import CASES, frames_and_dets
    g = np.load(os.path.join(ROOT, "tests", "golden", "gmc.npz"))
    for k, case in enumerate(CASES):
        frames, dets = frames_and_dets(case)
        orc = G.GMCOracle(estimator="both")
        for i, f in enumerate(frames):
            H = orc.apply(f, dets)
            np.testing.assert_allclose(H, g["H%d" % k][i], rtol=0, atol=1e-9)
            Hw = orc.last["H_restated"]
            # two RANSAC realisations on a few hundred points of a small frame: compared by where they send the frame's corners
            assert G.corner_displacement(Hw, H, case["h"], case["w"]) < 1.0
            if i:
                d = np.subtract(case["shifts"][i], case["shifts"][i - 1])           # (dy, dx) of this frame against the previous one
                assert abs(H[0, 2] - d[1]) < 1.0 and abs(H[1, 2] - d[0]) < 1.0              # (the rolled frame wraps around: the reference's own estimate is up to 0.7 px off)
