"""Golden vectors for test-time detection post-processing (SURVEY.md 8f N3), produced by the UNMODIFIED reference code:
lib/core/test.py box_results_with_nms_and_limit with its own utils.boxes and the Cython routines built from its .pyx,
imported from oracle/_ref/reflib (python oracle/make_reflib.py).  Runs on CPU:

    python tests/golden/make_golden_detections.py [OUT_DIR]      # -> detections.npz

Inputs are tests/cases.py detection_case(seed); for every seed and setting of cases.DETECTION_SETTINGS the file holds
the reference's scores / boxes and its per-class results for classes 1..20, concatenated (`<seed>_<setting>/cls`, (n, 5))
with the count of each class (`<seed>_<setting>/cls_counts`).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import refmodel          # noqa: E402
from tests import cases              # noqa: E402

SEEDS = (0, 1)


def main(out_dir):
    cfg = refmodel.setup(use_b200_ops=False)
    import core.test as ref_test
    cfg.MODEL.NUM_CLASSES = 21
    cfg.TEST.SCORE_THRESH = 0.05; cfg.TEST.NMS = 0.5; cfg.TEST.DETECTIONS_PER_IM = 100; cfg.TEST.BBOX_VOTE.VOTE_TH = 0.8
    gold = {"soft_nms_sigma": np.float64(cfg.TEST.SOFT_NMS.SIGMA)}
    for seed in SEEDS:
        scores, boxes = cases.detection_case(seed)
        for i, (soft, method, vote, scoring) in enumerate(cases.DETECTION_SETTINGS):
            cfg.TEST.SOFT_NMS.ENABLED = soft; cfg.TEST.SOFT_NMS.METHOD = method
            cfg.TEST.BBOX_VOTE.ENABLED = vote; cfg.TEST.BBOX_VOTE.SCORING_METHOD = scoring
            rs, rb, rc = ref_test.box_results_with_nms_and_limit(scores, boxes)
            key = "%d_%d" % (seed, i)
            gold[key + "/scores"] = np.asarray(rs)
            gold[key + "/boxes"] = np.asarray(rb)
            assert len(rc) == 21
            per_class = [np.asarray(rc[j]).reshape(-1, 5) for j in range(1, 21)]
            gold[key + "/cls"] = np.concatenate(per_class)
            gold[key + "/cls_counts"] = np.array([len(a) for a in per_class], np.int64)
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "detections.npz"), **gold)
    print("written", os.path.join(out_dir, "detections.npz"), len(gold), "arrays")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
