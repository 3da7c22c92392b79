"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's ReID extractor (SURVEY.md section 8f row 3).

Follows tracker/reid_models/deepsort_reid.py: ``Extractor._preprocess`` :134-146 (crop.astype(float32) / 255 -> cv2.resize to
64 x 128 -> ToTensor -> Normalize) restated in NumPy, ``Net.forward`` :92-106 with ``reid=True`` (+ ``BasicBlock.forward`` :41-49)
restated with torch.nn.functional on the checkpoint's tensors (BatchNorm in eval mode, unfolded, fp32).
tests/test_oracle_reid.py pins both against what the UNMODIFIED reference classes computed on seeded crops and seeded weights
(tests/golden/refchecks.npz, made by tests/golden/make_golden_refchecks.py).
"""
import numpy as np
import torch
import torch.nn.functional as F

MEAN = np.array([0.485, 0.456, 0.406], np.float32)
STD = np.array([0.229, 0.224, 0.225], np.float32)
STAGES = (("layer1", False), ("layer2", True), ("layer3", True), ("layer4", True))


def _taps(dst, src):
    scale = np.float64(1.0) / (np.float64(dst) / np.float64(src))          # cv::resize: scale = 1 / (dsize / ssize)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    lo, hi = s < 0, s >= src - 1
    f[lo] = 0; s[lo] = 0
    f[hi] = 0; s[hi] = src - 1
    return s, np.minimum(s + 1, src - 1), f


def preprocess(crops):
    """list of (h, w, 3) uint8 -> (n, 3, 128, 64) float32 tensor (:134-146)."""
    out = []
    for im in crops:
        a = im.astype(np.float32) / np.float32(255.0)
        h, w = a.shape[:2]
        x0, x1, fx = _taps(64, w)
        y0, y1, fy = _taps(128, h)
        fx = fx[None, :, None]; fy = fy[:, None, None]
        rows = a[:, x0] * (np.float32(1) - fx) + a[:, x1] * fx                                  # horizontal pass
        r = rows[y0] * (np.float32(1) - fy) + rows[y1] * fy                                     # vertical pass
        r = (r - MEAN) / STD                                                                     # Normalize on the channels as they come (B, G, R)
        out.append(torch.from_numpy(np.ascontiguousarray(r.transpose(2, 0, 1))))
    return torch.stack(out).float()


_TRAIN = [True]


def _bn(x, sd, p):
    if _TRAIN[0]:       # batch statistics (training-mode normalisation; the running buffers are left alone)
        return F.batch_norm(x, None, None, sd[p + ".weight"], sd[p + ".bias"], True, 0.0, 1e-5)
    return F.batch_norm(x, sd[p + ".running_mean"], sd[p + ".running_var"], sd[p + ".weight"], sd[p + ".bias"], False, 0.0, 1e-5)


def forward(sd, x, batch_stats=True):
    """Net(reid=True).forward on a float state dict.  batch_stats=True is what the reference's Extractor computes: it never calls
    ``net.eval()`` (:112-121), so every BatchNorm layer normalises with the statistics of the crops of THIS call (:148-153);
    batch_stats=False is eval mode (running statistics)."""
    _TRAIN[0] = bool(batch_stats)
    x = F.relu(_bn(F.conv2d(x, sd["conv.0.weight"], sd["conv.0.bias"], 1, 1), sd, "conv.1"))
    x = F.max_pool2d(x, 3, 2, 1)
    for name, down in STAGES:
        for blk in range(2):
            p = "%s.%d" % (name, blk)
            s = 2 if (down and blk == 0) else 1
            y = F.relu(_bn(F.conv2d(x, sd[p + ".conv1.weight"], None, s, 1), sd, p + ".bn1"))
            y = _bn(F.conv2d(y, sd[p + ".conv2.weight"], None, 1, 1), sd, p + ".bn2")
            if (p + ".downsample.0.weight") in sd:
                x = _bn(F.conv2d(x, sd[p + ".downsample.0.weight"], None, s, 0), sd, p + ".downsample.1")
            x = F.relu(x + y)
    x = F.avg_pool2d(x, (8, 4), 1).flatten(1)
    return x / x.norm(p=2, dim=1, keepdim=True)


def seeded_state_dict(seed=0):
    """A state dict with the keys and shapes of Net(reid=True): Kaiming-scaled conv weights, BatchNorm statistics away from the
    identity (so that folding is exercised).  The GPU tests cannot carry the 46 MB checkpoint."""
    g = torch.Generator().manual_seed(seed)
    sd = {}

    def conv(name, cout, cin, k, bias=False):
        sd[name + ".weight"] = torch.randn((cout, cin, k, k), generator=g) * (2.0 / (cin * k * k)) ** 0.5
        if bias:
            sd[name + ".bias"] = torch.randn(cout, generator=g) * 0.1

    def bn(name, c):
        sd[name + ".weight"] = 1.0 + 0.2 * torch.randn(c, generator=g)
        sd[name + ".bias"] = 0.1 * torch.randn(c, generator=g)
        sd[name + ".running_mean"] = 0.2 * torch.randn(c, generator=g)
        sd[name + ".running_var"] = 0.5 + torch.rand(c, generator=g)
    conv("conv.0", 64, 3, 3, bias=True); bn("conv.1", 64)
    cin = 64
    for name, cout, down in (("layer1", 64, False), ("layer2", 128, True), ("layer3", 256, True), ("layer4", 512, True)):
        for blk in range(2):
            p = "%s.%d" % (name, blk)
            c_in = cin if blk == 0 else cout
            conv(p + ".conv1", cout, c_in, 3); bn(p + ".bn1", cout)
            conv(p + ".conv2", cout, cout, 3); bn(p + ".bn2", cout)
            if blk == 0 and (down or c_in != cout):
                conv(p + ".downsample.0", cout, c_in, 1); bn(p + ".downsample.1", cout)
        cin = cout
    return sd


def seeded_crops(seed, n):
    rng = np.random.default_rng(seed)
    crops = []
    for _ in range(n):
        h, w = int(rng.integers(24, 220)), int(rng.integers(12, 120))
        base = rng.integers(0, 256, (h // 8 + 2, w // 8 + 2, 3)).astype(np.float32)
        im = np.kron(base, np.ones((8, 8, 1), np.float32))[:h, :w] + rng.normal(0, 12, (h, w, 3))
        crops.append(np.clip(im, 0, 255).astype(np.uint8))
    return crops
