"""Numpy restatement of the reference's Mask R-CNN mask paste and RLE (lib/core/test.py:793-847 `segm_results`,
lib/utils/boxes.py:233-249 `expand_boxes`), without cv2 or pycocotools.  Test infrastructure: the CUDA kernels of
detectron/pytorch_b200/csrc/segm.cu are checked against this, and this against goldens recorded from the reference.

Per detection i (soft mask `masks[i, channel[i]]`, M x M, and reference box `ref_boxes[i]`):
  1. expand_boxes in float32 (numpy >= 2 promotion rules): half sizes `(x2 - x1) * .5`, centres `(x2 + x1) * .5`,
     half sizes times float32((M + 2) / M), corners `c -/+ half`; stored in float64 and truncated toward zero to int32;
  2. w = max(x2 - x1 + 1, 1), h likewise; the (M + 2)^2 zero-padded mask is resized to (h, w) exactly like
     cv2.resize(INTER_LINEAR) on float32 with IPP off (`axis_table`, `resize`);
  3. `> thresh` in float32, pasted into the clipped window [max(y1, 0), min(y2 + 1, im_h)) x [max(x1, 0),
     min(x2 + 1, im_w)) of an all-zero (im_h, im_w) uint8 image;
  4. COCO's uncompressed RLE of the column-major (Fortran-order) image: alternating run lengths, zeros first.

The window in step 3 is empty when a clipped bound crosses the other.  The reference slices with these bounds as Python
slice indices, so a box whose far edge lies at -2 or further left / above, or whose start lies beyond im_w / im_h by more
than its own width, makes it index from the other end or raise a broadcast error.  Boxes clipped to the image (which is
what the detection step produces), expanded by (M + 2) / M, never reach that.
"""
import numpy as np


def expand_boxes_int(ref_boxes, M):
    """(D, 4) float32 -> (D, 4) int32, the reference's expand_boxes followed by .astype(np.int32)."""
    b = np.asarray(ref_boxes, dtype=np.float32).reshape(-1, 4)
    w_half = (b[:, 2] - b[:, 0]) * np.float32(.5)
    h_half = (b[:, 3] - b[:, 1]) * np.float32(.5)
    x_c = (b[:, 2] + b[:, 0]) * np.float32(.5)
    y_c = (b[:, 3] + b[:, 1]) * np.float32(.5)
    s = np.float32((M + 2.0) / M)
    w_half = w_half * s
    h_half = h_half * s
    out = np.zeros(b.shape, np.float64)
    out[:, 0] = x_c - w_half
    out[:, 2] = x_c + w_half
    out[:, 1] = y_c - h_half
    out[:, 3] = y_c + h_half
    return out.astype(np.int32)


def axis_table(src, dst, clamp_weights=True):
    """cv2's INTER_LINEAR source indices and weights per destination index (one axis): (s0, s1, a0, a1).
    cv2 zeroes the fraction where the source index leaves [0, src - 1] on the horizontal axis only; on the vertical axis
    it clips the two row indices and keeps the fraction (clamp_weights=False)."""
    scale = 1.0 / (float(dst) / float(src))
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if clamp_weights:
        lo = s < 0
        s[lo] = 0; f[lo] = 0
        hi = s >= src - 1
        s[hi] = src - 1; f[hi] = 0
    return np.clip(s, 0, src - 1), np.clip(s + 1, 0, src - 1), (np.float32(1) - f).astype(np.float32), f


def resize(src, w, h):
    """cv2.resize(src, (w, h)) for a float32 2-D array, INTER_LINEAR, IPP off: horizontal pass then vertical pass,
    every product and sum rounded to float32 separately.  An exact 2x downscale on both axes is cv2's area-fast path
    instead: ((a + b) + (c + d)) * 0.25 over each 2 x 2 block in its 4-wide vector loop (the first 4 * (w // 4)
    columns, which equals the linear result), (((a + b) + c) + d) * 0.25 in its scalar tail."""
    src = np.asarray(src, dtype=np.float32)
    sh, sw = src.shape
    if 2 * w == sw and 2 * h == sh:
        a, b, c, d = src[0::2, 0::2], src[0::2, 1::2], src[1::2, 0::2], src[1::2, 1::2]
        out = ((a + b) + (c + d)) * np.float32(.25)
        nv = 4 * (w // 4)
        out[:, nv:] = ((((a + b) + c) + d) * np.float32(.25))[:, nv:]
        return out
    xs0, xs1, xa0, xa1 = axis_table(sw, w)
    ys0, ys1, yb0, yb1 = axis_table(sh, h, clamp_weights=False)
    rows = src[:, xs0] * xa0 + src[:, xs1] * xa1                    # (sh, w) float32
    return rows[ys0, :] * yb0[:, None] + rows[ys1, :] * yb1[:, None]   # (h, w) float32


def paste_one(mask, box, im_h, im_w, thresh):
    """One detection: M x M soft mask, expanded int box -> (im_h, im_w) uint8."""
    M = mask.shape[0]
    padded = np.zeros((M + 2, M + 2), np.float32)
    padded[1:-1, 1:-1] = mask
    x1, y1, x2, y2 = (int(v) for v in box)
    w = max(x2 - x1 + 1, 1)
    h = max(y2 - y1 + 1, 1)
    binar = (resize(padded, w, h) > np.float32(thresh)).astype(np.uint8)
    im = np.zeros((im_h, im_w), np.uint8)
    x0, x1c = max(x1, 0), min(x2 + 1, im_w)
    y0, y1c = max(y1, 0), min(y2 + 1, im_h)
    if x0 < x1c and y0 < y1c:
        im[y0:y1c, x0:x1c] = binar[y0 - y1:y1c - y1, x0 - x1:x1c - x1]
    return im


def paste(masks, channels, ref_boxes, im_h, im_w, thresh=0.5):
    """masks (D, K, M, M) float32, channels (D,) -> (D, im_h, im_w) uint8 dense binary masks."""
    masks = np.asarray(masks, dtype=np.float32)
    D, M = masks.shape[0], masks.shape[-1]
    boxes = expand_boxes_int(ref_boxes, M)
    out = np.zeros((D, im_h, im_w), np.uint8)
    for i in range(D):
        out[i] = paste_one(masks[i, int(channels[i])], boxes[i], im_h, im_w, thresh)
    return out


def rle_runs(im):
    """COCO uncompressed RLE counts of one (H, W) binary image in column-major order: zeros first."""
    flat = np.asarray(im, dtype=np.uint8).ravel(order="F")
    change = np.flatnonzero(np.diff(np.concatenate([[0], flat])) != 0)       # positions where the value changes
    bounds = np.concatenate([[0], change, [flat.size]])
    return np.diff(bounds).astype(np.int64)


def segm_runs(masks, channels, ref_boxes, im_h, im_w, thresh=0.5):
    """Per detection RLE: (runs concatenated, counts per detection) and the dense masks."""
    dense = paste(masks, channels, ref_boxes, im_h, im_w, thresh)
    per = [rle_runs(m) for m in dense]
    runs = np.concatenate(per) if per else np.zeros((0,), np.int64)
    return runs, np.array([len(r) for r in per], np.int64), dense


def channels_for(cls_counts, cls_specific):
    """The reference's mask_ind walk: detections of class j (j = 1 .. K-1, in order) read channel j, or 0."""
    return np.concatenate([np.full(int(n), j if cls_specific else 0, np.int64) for j, n in enumerate(cls_counts, start=1)]
                          + [np.zeros((0,), np.int64)])
