"""Shared, seeded test cases (inputs only -- expected values come from the oracle / golden files)."""
import numpy as np

from detectron.pytorch_b200 import synthetic as S

# name -> dict(shape, scale, P, sr, n_rois)   small enough for the CPU oracle to finish in < 1 s
ROI_CASES = {
    "cfg1_small": dict(shape=(2, 8, 50, 68), scale=1.0 / 16, P=7, sr=2, n_rois=32),
    "adaptive": dict(shape=(2, 8, 50, 68), scale=1.0 / 16, P=7, sr=0, n_rois=32),
    "p14": dict(shape=(1, 6, 50, 68), scale=1.0 / 16, P=14, sr=2, n_rois=24),
    "odd_hw": dict(shape=(2, 5, 25, 42), scale=1.0 / 32, P=7, sr=2, n_rois=24),
    "sr3": dict(shape=(1, 4, 40, 40), scale=1.0 / 8, P=5, sr=3, n_rois=16),
}

PYRAMID_800x1333 = ((200, 336), (100, 168), (50, 84), (25, 42))        # (H, W) of FPN P2..P5 of an 800 x 1333 image

# Both sides of every dispatch limit of the quad-strip forward (roi_align_strip.cu, strip_geometry), as
# (N, H, W, R, PH, PW, sr).  Under B200_ROI_ALIGN_PATH=quad the single-map workspace size is the strip path's alone, so a
# non-zero size means the path takes the shape.  tests/test_abi.py pins which side of each limit these shapes are on;
# tests/test_gpu_geometry.py runs them on the GPU.
QUAD_LIMITS = {
    # limit: (accepted, rejected)
    "keys_batch": ((16, 64, 336, 64, 7, 7, 2), (17, 64, 336, 64, 7, 7, 2)),          # 16 images x 6 strips x 64 rows = 6144 CSR keys
    "keys_height": ((1, 1536, 100, 64, 7, 7, 2), (1, 1537, 100, 64, 7, 7, 2)),       # 4 strips x 1536 rows = 6144
    "columns": ((1, 4, 5384, 64, 7, 7, 2), (1, 4, 5385, 64, 7, 7, 2)),              # 96 strips of one image
    "rois": ((1, 50, 68, 65535, 7, 7, 2), (1, 50, 68, 65536, 7, 7, 2)),             # 16-bit RoI index of the fragment record
    "axis_square": ((1, 50, 68, 64, 16, 16, 2), (1, 50, 68, 64, 17, 17, 2)),        # P * sr <= 32
    "axis_pw": ((1, 50, 68, 64, 16, 3, 2), (1, 50, 68, 64, 3, 17, 2)),              # PH and PW are limited separately
}

NMS_SIZES = (1, 2, 63, 64, 65, 128, 129, 1000, 2000, 6000, 12000)


def roi_case(name):
    c = ROI_CASES[name]
    feats = S.make_features(c["shape"], seed=0)
    rois = S.make_rois(c["n_rois"], c["shape"], c["scale"], seed=0)
    rois = np.concatenate([rois, S.make_edge_rois(c["shape"], c["scale"])]).astype(np.float32)
    R = rois.shape[0]
    dy = np.random.RandomState(1).standard_normal((R, c["shape"][1], c["P"], c["P"])).astype(np.float32)
    return c, feats, rois, dy


def sample_index(size, seed, k=8192):
    """A fixed, seeded sample of k flat indices into an array of `size` elements: large outputs are stored under
    tests/golden/ as their values at these indices."""
    return np.sort(np.random.RandomState(seed).choice(size, k, replace=False))


def spread_cases():
    """name -> (shape, scale, P, sr, rois, dy seed): the backward run-to-run spread cases (BASELINE cfg2 and a pile-up)."""
    return {
        "cfg2": (S.CFG2["shape"], S.CFG2["scale"], S.CFG2["pooled"], S.CFG2["sampling_ratio"],
                 S.make_rois(S.CFG2["rois"], S.CFG2["shape"], S.CFG2["scale"]).astype(np.float32), 1),
        "pileup_1500": ((3, 40, 46, 70), 0.125, 7, 2,
                        S.make_rois(1500, (3, 40, 46, 70), 0.125, seed=6, min_size=64, max_size=500).astype(np.float32), 7),
    }


# (soft_nms, soft_method, bbox_vote, vote_scoring) settings of the test-time detection post-processing
DETECTION_SETTINGS = (
    (False, "linear", False, "ID"), (True, "linear", False, "ID"), (True, "gaussian", False, "ID"),
    (False, "linear", True, "ID"), (False, "linear", True, "IOU_AVG"), (True, "linear", True, "AVG"),
    (False, "linear", True, "TEMP_AVG"), (False, "linear", True, "QUASI_SUM"), (False, "linear", True, "GENERALIZED_AVG"),
)


def detection_case(seed, R=300, K=21):
    """Clustered proposals: 25 objects x 12 jittered copies, every class gets its own regressed box per proposal.
    Returns scores (R, K) and boxes (R, 4K), fp32."""
    rng = np.random.RandomState(seed)
    cx = np.repeat(rng.uniform(100, 1200, 25), 12)[:R]; cy = np.repeat(rng.uniform(100, 700, 25), 12)[:R]
    w = np.repeat(rng.uniform(40, 300, 25), 12)[:R]; h = np.repeat(rng.uniform(40, 300, 25), 12)[:R]
    boxes = np.zeros((R, 4 * K), np.float32)
    for j in range(K):
        jx = cx + rng.normal(0, 0.06, R) * w; jy = cy + rng.normal(0, 0.06, R) * h
        jw = w * (1 + rng.normal(0, 0.08, R)); jh = h * (1 + rng.normal(0, 0.08, R))
        boxes[:, 4 * j:4 * j + 4] = np.stack([jx - jw / 2, jy - jh / 2, jx + jw / 2, jy + jh / 2], 1)
    logits = rng.standard_normal((R, K)) * 2.0
    scores = (np.exp(logits) / np.exp(logits).sum(1, keepdims=True)).astype(np.float32)
    return scores, boxes


def crop_case(seed=0):
    shape = (2, 6, 30, 44)
    img = S.make_features(shape, seed=seed)
    grid = S.make_crop_grid(8, 7, 7, seed=seed)      # R = 8 -> 4 RoIs per image
    grid[0, 0, 0] = (-1.0, -1.0)                      # exact corners / borders
    grid[0, 0, 1] = (1.0, 1.0)
    grid[1, 3, 3] = (-1.5, 0.2)                       # outside
    grid[2, 2, 2] = (0.3, 1.7)
    go = np.random.RandomState(seed + 1).standard_normal((8, shape[1], 7, 7)).astype(np.float32)
    return img, grid.astype(np.float32), go


def nms_case(n, seed=0):
    return S.make_nms_boxes(n, seed=seed)


def nms_chain_case(n, shift=10.0, width=100.0):
    """Worst case of the block-parallel resolve: box i overlaps box i+1 above 0.7 but not box i+2, so the greedy
    result alternates keep / drop and every decision depends on the previous one (suppression chain of length n)."""
    import numpy as np
    x1 = np.arange(n, dtype=np.float32) * np.float32(shift)
    b = np.stack([x1, np.zeros(n, np.float32), x1 + np.float32(width), np.full(n, 50, np.float32),
                  np.linspace(1.0, 0.1, n).astype(np.float32)], axis=1)
    return b.astype(np.float32)


def nms_clustered_case(n, seed=0, copies=10):
    """Score-sorted proposals where near-duplicates are ADJACENT in the order (dense diagonal blocks)."""
    import numpy as np
    b = S.make_nms_boxes(n, seed=seed, copies=copies)
    rng = np.random.RandomState(seed + 1)
    seeds = b[rng.permutation(n)[: (n + copies - 1) // copies], :4]
    rep = np.repeat(seeds, copies, axis=0)[:n] + rng.normal(0, 2.0, (n, 4)).astype(np.float32)
    rep[:, 2:] = np.maximum(rep[:, 2:], rep[:, :2] + 1)
    return np.concatenate([rep, b[:, 4:5]], axis=1).astype(np.float32)
