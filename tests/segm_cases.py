"""Seeded inputs of the Mask R-CNN mask paste tests (lib/core/test.py:793-847 segm_results): expected values come from
oracle/segm.py and tests/golden/segm.npz (tests/golden/make_golden_segm.py)."""
import numpy as np


# Mask R-CNN mask paste (lib/core/test.py:793-847 segm_results): name -> (im_h, im_w, M, num_classes, class-specific)
SEGM_CASES = {
    "a": (800, 1199, 28, 81, True),        # e2e_mask_rcnn_R-50-FPN_1x at test scale, ~100 detections
    "b": (600, 800, 14, 21, False),        # class-agnostic mask head
    "c": (480, 640, 28, 5, True),          # edge boxes
    "d": (37, 53, 14, 4, True),            # small odd image, boxes spanning the full height: runs wrap across columns
    "e": (800, 1333, 28, 81, False),       # 1000 detections
}


def _soft_masks(rng, D, K, M):
    """Blob-shaped sigmoid masks with noise, (D, K, M, M) float32 in (0, 1)."""
    g = (np.arange(M, dtype=np.float64) + 0.5) / M
    cy = rng.uniform(0.2, 0.8, (D, K, 1, 1)); cx = rng.uniform(0.2, 0.8, (D, K, 1, 1))
    ry = rng.uniform(0.15, 0.6, (D, K, 1, 1)); rx = rng.uniform(0.15, 0.6, (D, K, 1, 1))
    r = np.sqrt(((g[None, None, :, None] - cy) / ry) ** 2 + ((g[None, None, None, :] - cx) / rx) ** 2)
    z = 6.0 * (1.0 - r) + rng.normal(0, 1.0, (D, K, M, M))
    return (1.0 / (1.0 + np.exp(-z))).astype(np.float32)


def segm_case(name):
    """Inputs of segm_results(cls_boxes, masks, ref_boxes, im_h, im_w): a dict with im_h, im_w, M, num_classes,
    cls_specific, cls_boxes (num_classes arrays (n_j, 5), class 0 empty), masks (D, num_classes or 1, M, M) float32 and
    ref_boxes (D, 4) float32, the boxes of cls_boxes[1:] stacked in class order (what the reference passes)."""
    im_h, im_w, M, K, cls_specific = SEGM_CASES[name]
    rng = np.random.RandomState(ord(name))
    if name in ("a", "b", "e"):
        D = {"a": 100, "b": 40, "e": 1000}[name]
        w = rng.uniform(8, 0.6 * im_w, D) * rng.uniform(0.2, 1.0, D) ** 2 + 2
        h = rng.uniform(8, 0.6 * im_h, D) * rng.uniform(0.2, 1.0, D) ** 2 + 2
        x1 = rng.uniform(0, im_w - 1, D); y1 = rng.uniform(0, im_h - 1, D)
        boxes = np.stack([x1, y1, np.minimum(x1 + w, im_w - 1), np.minimum(y1 + h, im_h - 1)], 1)
    elif name == "c":
        W, H = float(im_w), float(im_h)
        boxes = np.array([
            [-20.5, 100, 60.3, 180], [200, -30.2, 290, 40.7], [W - 50.2, 300, W + 15.6, 370], [400, H - 40.1, 470, H + 22.9],
            [-3.7, -2.2, 40.1, 33.3], [-0.4, 50, 20, 90],                        # negative corners: truncation toward zero
            [W + 100, 50, W + 150, 100], [50, H + 100, 120, H + 140],           # entirely right of / below the image
            [-W - 300, 10, -W - 250, 60],                                      # entirely left, farther than the image is wide
            [100.2, 100, 100.2, 160], [300, 200.6, 380, 200.1],                  # expanded w = 1, h <= 1
            [300, 300, 290, 340],                                              # x2 < x1
            [-50, -40, W + 60, H + 30],                                        # larger than the image
            [100, 200, 127.25, 227.25],                                        # expands to exactly M + 2 px: identity resize
            [150, 20, 162.75, 32.75],                                          # expands to (M + 2) / 2 px: cv2's 2x area path
            [0, 0, W - 1, H - 1], [W - 30, H - 30, W - 1, H - 1],
        ], np.float64)
    else:
        boxes = np.array([[-3, -15, 10, im_h + 14], [20.5, -12.5, 27.3, im_h + 11.5], [40, -20, 60, im_h + 20],
                          [0, 0, im_w - 1, im_h - 1], [5, 5, 30, 20], [im_w - 9, -3, im_w + 4, im_h + 3]], np.float64)
    D = len(boxes)
    labels = np.sort(rng.randint(1, K, D))
    masks = _soft_masks(rng, D, K if cls_specific else 1, M)
    if name == "c":
        # values exactly at the threshold: the identity-resize box reads them unchanged (strict `>` keeps them 0)
        ch = labels[13] if cls_specific else 0
        masks[13, ch, ::2, :] = 0.5
        masks[13, ch, 1::4, :] = np.float32(0.5) + np.float32(2 ** -24)
        masks[14, labels[14] if cls_specific else 0, 3:9, 3:9] = 0.5
    boxes = boxes.astype(np.float32)
    scores = rng.uniform(0.05, 1.0, D).astype(np.float32)
    cls_boxes = [np.zeros((0, 5), np.float32)] + [np.concatenate([boxes[labels == j], scores[labels == j, None]], 1)
                                                  for j in range(1, K)]
    return dict(im_h=im_h, im_w=im_w, M=M, num_classes=K, cls_specific=cls_specific, cls_boxes=cls_boxes, masks=masks,
                ref_boxes=boxes)
