"""Golden vectors for the Mask R-CNN mask paste (lib/core/test.py:793-847 segm_results), produced by the UNMODIFIED
reference function imported from oracle/_ref/reflib (python oracle/make_reflib.py).  Runs on CPU with cv2:

    python tests/golden/make_golden_segm.py [OUT_DIR]      # -> segm.npz

Inputs are tests/segm_cases.py segm_case(name) for cases a-d (case e, 1000 detections, is checked against oracle/segm.py
only).  pycocotools' `encode` is replaced from outside by a recorder that keeps the Fortran-order image the reference
hands it, stored as COCO uncompressed RLE.  Every case runs twice: with cv2's IPP disabled (the arithmetic the device
reproduces) and with cv2's default.  Per case and setting the file holds `<case>/<ipp>/runs` (all run lengths, detection
after detection) and `<case>/<ipp>/counts` (runs per detection), <ipp> = off | on.  `<case>/flips` lists (detection, y,
x, IPP-off value) of every pixel where the two binarisations differ, and `<case>/flip_values` the IPP-off resized value
there (float32, recomputed with cv2.resize, IPP off).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refmodel          # noqa: E402
from oracle import segm as oseg      # noqa: E402
from tests.segm_cases import segm_case   # noqa: E402

CASES = ("a", "b", "c", "d")


def main(out_dir):
    import cv2
    cfg = refmodel.setup(use_b200_ops=False)
    import core.test as ref_test
    recorded = []

    def encode(arr):
        assert arr.flags.f_contiguous and arr.dtype == np.uint8 and arr.ndim == 3
        recorded.append(np.array(arr[:, :, 0]))
        return [{"size": [arr.shape[0], arr.shape[1]], "counts": b""}]

    ref_test.mask_util.encode = encode
    ipp0 = cv2.ipp.useIPP()
    gold = {}
    try:
        for name in CASES:
            c = segm_case(name)
            cfg.MODEL.NUM_CLASSES = c["num_classes"]
            cfg.MRCNN.RESOLUTION = c["M"]
            cfg.MRCNN.CLS_SPECIFIC_MASK = c["cls_specific"]
            cfg.MRCNN.THRESH_BINARIZE = 0.5
            dense = {}
            for ipp in ("off", "on"):
                cv2.ipp.setUseIPP(ipp == "on")
                del recorded[:]
                segms = ref_test.segm_results(c["cls_boxes"], c["masks"], c["ref_boxes"], c["im_h"], c["im_w"])
                assert len(segms) == c["num_classes"] and segms[0] == []
                assert sum(len(s) for s in segms) == len(recorded) == len(c["ref_boxes"])
                per = [oseg.rle_runs(m) for m in recorded]
                gold["%s/%s/runs" % (name, ipp)] = np.concatenate(per).astype(np.int32)
                gold["%s/%s/counts" % (name, ipp)] = np.array([len(r) for r in per], np.int64)
                dense[ipp] = np.stack(recorded)
            flips = np.argwhere(dense["on"] != dense["off"])
            ch = oseg.channels_for([len(b) for b in c["cls_boxes"][1:]], c["cls_specific"])
            boxes = oseg.expand_boxes_int(c["ref_boxes"], c["M"])
            cv2.ipp.setUseIPP(False)
            vals = []
            for i, y, x in flips:
                M = c["M"]
                padded = np.zeros((M + 2, M + 2), np.float32)
                padded[1:-1, 1:-1] = c["masks"][i, ch[i]]
                bx1, by1, bx2, by2 = (int(v) for v in boxes[i])
                r = cv2.resize(padded, (max(bx2 - bx1 + 1, 1), max(by2 - by1 + 1, 1)))
                vals.append(r[y - by1, x - bx1])
            gold[name + "/flips"] = np.concatenate([flips, dense["off"][tuple(flips.T)][:, None]], 1).astype(np.int32).reshape(-1, 4)
            gold[name + "/flip_values"] = np.array(vals, np.float32)
            print(name, "detections", len(boxes), "runs", len(gold[name + "/off/runs"]), "IPP flips", len(flips))
    finally:
        cv2.ipp.setUseIPP(ipp0)
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "segm.npz"), **gold)
    print("written", os.path.join(out_dir, "segm.npz"), len(gold), "arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
