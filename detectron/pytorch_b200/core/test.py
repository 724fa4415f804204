"""Test-time post-processing of the detection head on the device (SURVEY.md 8f N3).

Mirrors `box_results_with_nms_and_limit(scores, boxes)` of lib/core/test.py:732-790 (reference): per class j >= 1 keep the
detections with score > SCORE_THRESH, run NMS (or soft-NMS), optionally refine the kept boxes by box voting, then limit
the image to DETECTIONS_PER_IM detections over all classes.  The reference loops over the (80) classes on the host and
calls the Cython NMS once per class; here the per-class problems of an image go through ONE batched launch pair
(`b200_nms_batched`; soft-NMS: one warp per class in `b200_soft_nms_batched`; voting: `b200_box_voting_batched`), with one
host read of the kept counts.

Configuration: pass the reference's `cfg` object (read at call time like the reference: cfg.MODEL.NUM_CLASSES,
cfg.TEST.SCORE_THRESH / NMS / SOFT_NMS.* / BBOX_VOTE.* / DETECTIONS_PER_IM) or the same values as keyword arguments.
Inputs and outputs are numpy arrays like the reference's; CUDA tensors are accepted and skip the upload.

Flavour note (as for the proposal NMS): the device NMS keeps the reference CUDA kernel's `IoU > thresh` test, the Cython
routine the reference calls here uses `>=`; they differ only on pairs whose IoU equals the threshold to the last bit.
Soft-NMS follows lib/utils/cython_nms.pyx:98-203 step for step (same greedy order, same drop rule).
"""
import numpy as np
import torch

from .. import ops

_SOFT_METHODS = {"hard": 0, "linear": 1, "gaussian": 2}
_VOTE_SCORING = {"ID": 0, "AVG": 1, "IOU_AVG": 2, "TEMP_AVG": 3, "GENERALIZED_AVG": 4, "QUASI_SUM": 5}


def _params(cfg, kw):
    if cfg is not None:
        t = cfg.TEST
        p = dict(num_classes=cfg.MODEL.NUM_CLASSES, score_thresh=t.SCORE_THRESH, nms=t.NMS, detections_per_im=t.DETECTIONS_PER_IM,
                 soft_nms=t.SOFT_NMS.ENABLED, soft_sigma=t.SOFT_NMS.SIGMA, soft_method=t.SOFT_NMS.METHOD,
                 bbox_vote=t.BBOX_VOTE.ENABLED, vote_th=t.BBOX_VOTE.VOTE_TH, vote_scoring=t.BBOX_VOTE.SCORING_METHOD)
    else:
        p = dict(num_classes=None, score_thresh=0.05, nms=0.5, detections_per_im=100, soft_nms=False, soft_sigma=0.5,
                 soft_method="linear", bbox_vote=False, vote_th=0.8, vote_scoring="ID")       # lib/core/config.py:262-330
    p.update(kw)
    return p


def box_results_with_nms_and_limit(scores, boxes, cfg=None, **kw):
    """scores (R, K), boxes (R, 4K) -> (scores (D,), boxes (D, 4), cls_boxes list of K arrays (n_j, 5)), like the reference."""
    p = _params(cfg, kw)
    dev = torch.device("cuda", torch.cuda.current_device())
    S = scores if torch.is_tensor(scores) else torch.from_numpy(np.ascontiguousarray(scores, dtype=np.float32))
    B = boxes if torch.is_tensor(boxes) else torch.from_numpy(np.ascontiguousarray(boxes, dtype=np.float32))
    S = S.to(dev, dtype=torch.float32); B = B.to(dev, dtype=torch.float32)
    K = int(p["num_classes"] or S.size(1))
    cls_boxes = [[] for _ in range(K)]
    # candidates of every class, in the reference's order (ascending detection index), one host read for the counts
    mask = S[:, 1:K] > float(p["score_thresh"])                       # (R, K-1)
    counts = mask.sum(dim=0).cpu().numpy().astype(np.int64)            # per class
    cls_idx, det_idx = torch.nonzero(mask.t(), as_tuple=True)          # grouped by class, ascending detection index inside
    j_of = cls_idx + 1
    sc = S[det_idx, j_of]
    bx = B.view(B.size(0), -1, 4)[det_idx, j_of]
    dets = torch.cat([bx, sc[:, None]], dim=1).contiguous()            # (sum counts, 5), class-major
    offs = np.concatenate([[0], np.cumsum(counts)])
    live = [j for j in range(K - 1) if counts[j] > 0]
    kept = {}
    if live:
        if p["soft_nms"]:
            out, inds, n_out = ops.soft_nms_batched(dets, [int(c) for c in counts], sigma=float(p["soft_sigma"]), overlap_thresh=float(p["nms"]),
                                                    score_thresh=0.0001, method=_SOFT_METHODS.get(p["soft_method"], 0))
            n_out = n_out.cpu().numpy()
            for j in live:
                kept[j] = out[offs[j]:offs[j] + int(n_out[j])]
        else:
            # score-sorted copies per class (stable), batched NMS, back to ascending original order like cython_nms.nms
            order = torch.empty_like(det_idx)
            for j in live:                                             # tiny per-class sorts; keys are (class, -score)
                seg = slice(int(offs[j]), int(offs[j + 1]))
                order[seg] = torch.sort(sc[seg], descending=True, stable=True)[1] + int(offs[j])
            sorted_dets = dets[order]
            keep, num = ops.nms_batched_chunked(sorted_dets, [int(c) for c in counts], float(p["nms"]))
            num = num.cpu().numpy()
            for j in live:
                k = keep[offs[j]:offs[j] + int(num[j])].long() + int(offs[j])      # positions in the sorted copy
                orig = torch.sort(order[k])[0]                                       # ascending original index
                kept[j] = dets[orig]
        if p["bbox_vote"]:
            top_counts = [int(kept[j].size(0)) if j in kept else 0 for j in range(K - 1)]
            top = torch.cat([kept[j] for j in live], dim=0) if live else dets[:0]
            voted = ops.box_voting_batched(top, top_counts, dets, [int(c) for c in counts], float(p["vote_th"]),
                                           _VOTE_SCORING[p["vote_scoring"]], 1.0)
            o = 0
            for j in live:
                kept[j] = voted[o:o + top_counts[j]]; o += top_counts[j]
    for j in range(1, K):
        cls_boxes[j] = kept[j - 1].cpu().numpy() if (j - 1) in kept else np.zeros((0, 5), dtype=np.float32)
    # limit to max_per_image detections over all classes (host, like the reference: a sort of <= a few thousand scores)
    dpi = int(p["detections_per_im"])
    if dpi > 0:
        image_scores = np.hstack([cls_boxes[j][:, -1] for j in range(1, K)]) if K > 1 else np.zeros((0,), np.float32)
        if len(image_scores) > dpi:
            image_thresh = np.sort(image_scores)[-dpi]
            for j in range(1, K):
                keep = np.where(cls_boxes[j][:, -1] >= image_thresh)[0]
                cls_boxes[j] = cls_boxes[j][keep, :]
    im_results = np.vstack([cls_boxes[j] for j in range(1, K)]) if K > 1 else np.zeros((0, 5), np.float32)
    return im_results[:, -1], im_results[:, :-1], cls_boxes


def _segm_params(cfg, kw):
    if cfg is not None:
        p = dict(num_classes=cfg.MODEL.NUM_CLASSES, resolution=cfg.MRCNN.RESOLUTION, cls_specific_mask=cfg.MRCNN.CLS_SPECIFIC_MASK,
                 thresh_binarize=cfg.MRCNN.THRESH_BINARIZE)
    else:
        p = dict(num_classes=None, resolution=None, cls_specific_mask=True, thresh_binarize=0.5)     # lib/core/config.py MRCNN
    p.update(kw)
    return p


def _coco_mask():
    """pycocotools.mask, or None when it is not installed (a module without a file is a stand-in, not pycocotools)."""
    try:
        import pycocotools.mask as mask_util
    except ImportError:
        return None
    return mask_util if getattr(mask_util, "__file__", None) else None


def segm_results(cls_boxes, masks, ref_boxes, im_h, im_w, cfg=None, **kw):
    """Mask R-CNN masks -> COCO RLEs, like lib/core/test.py:793-847: a list of num_classes lists (class 0 empty) with one
    RLE dict per detection of cls_boxes[j], in order.

    masks (D, K or 1, M, M) and ref_boxes (D, 4) may be numpy arrays or CUDA tensors (a tensor straight from the mask
    head skips the upload).  Detection i of class j reads channel j when masks are class-specific, channel 0 otherwise.
    Configuration: the reference's `cfg` (MODEL.NUM_CLASSES, MRCNN.RESOLUTION, MRCNN.CLS_SPECIFIC_MASK,
    MRCNN.THRESH_BINARIZE) or the keyword arguments num_classes, resolution, cls_specific_mask, thresh_binarize.

    The binary masks are computed on the device (ops.segm_rle) with cv2.resize's INTER_LINEAR arithmetic as cv2 runs it
    with IPP disabled.  Flavour note: the default cv2 build routes this resize through IPP, whose results differ by up to
    ~2e-6; after thresholding that changes a pixel only when the resized value lies that close to the threshold (none
    in this project's golden cases, 3 of 29.8 M pixels in a wider probe).
    With pycocotools importable each RLE is exactly the reference's dict: `{'size': [im_h, im_w], 'counts': str}`
    (pycocotools' compressed string).  Without it the dict is COCO's uncompressed RLE, `{'size': [im_h, im_w],
    'counts': [run lengths]}`: column-major runs alternating from a run of zeros, which pycocotools' frPyObjects and
    COCO.annToRLE accept.
    """
    p = _segm_params(cfg, kw)
    K = int(p["num_classes"] or len(cls_boxes))
    counts = [int(np.asarray(cls_boxes[j]).shape[0]) for j in range(1, K)]
    D = sum(counts)
    if int(masks.shape[0]) != D:
        raise ValueError("masks hold %d detections, cls_boxes %d" % (int(masks.shape[0]), D))
    cls_segms = [[] for _ in range(K)]
    if D == 0:
        return cls_segms
    M = int(p["resolution"] or masks.shape[-1])
    if tuple(masks.shape[-2:]) != (M, M):
        raise ValueError("masks are %s, expected M = %d" % (tuple(masks.shape[-2:]), M))
    dev = torch.device("cuda", torch.cuda.current_device())
    Mk = masks if torch.is_tensor(masks) else torch.from_numpy(np.ascontiguousarray(masks, dtype=np.float32))
    B = ref_boxes if torch.is_tensor(ref_boxes) else torch.from_numpy(np.ascontiguousarray(ref_boxes, dtype=np.float32))
    Mk = Mk.to(dev, dtype=torch.float32).reshape(D, -1, M, M)
    B = B.to(dev, dtype=torch.float32).reshape(D, 4)
    chan = None
    if p["cls_specific_mask"]:
        chan = np.repeat(np.arange(1, K, dtype=np.int32), counts)
    runs, n_runs = ops.segm_rle(Mk, chan, B, im_h, im_w, float(p["thresh_binarize"]))
    mask_util = _coco_mask()
    runs = runs.tolist()
    size = [int(im_h), int(im_w)]
    o = 0
    i = 0
    for j in range(1, K):
        segms = []
        for _ in range(counts[j - 1]):
            rle = {"size": list(size), "counts": runs[o:o + int(n_runs[i])]}
            if mask_util is not None:
                rle = mask_util.frPyObjects(rle, size[0], size[1])
                rle["counts"] = rle["counts"].decode("ascii")
            segms.append(rle)
            o += int(n_runs[i]); i += 1
        cls_segms[j] = segms
    return cls_segms
