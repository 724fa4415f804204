"""SURVEY.md 8f N3: test-time detection post-processing on the device (per-class NMS in one batched launch pair, soft-NMS,
box voting, the per-image limit) against the REFERENCE'S OWN functions -- lib/core/test.py:732-790, lib/utils/boxes.py and
the Cython routines built from its .pyx.  Their results on the seeded inputs of tests/cases.py are stored in
tests/golden/detections.npz (tests/golden/make_golden_detections.py runs the unmodified reference on CPU)."""
import os

import numpy as np
import pytest

from tests import cases

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "detections.npz")


@pytest.mark.gpu
def test_box_results_with_nms_and_limit_matches_the_reference():
    from detectron.pytorch_b200.core.test import box_results_with_nms_and_limit as ours
    g = np.load(GOLDEN)
    checked = 0
    for seed in (0, 1):
        scores, boxes = cases.detection_case(seed)
        for i, (soft, method, vote, scoring) in enumerate(cases.DETECTION_SETTINGS):
            key = "%d_%d" % (seed, i)
            os_, ob, oc = ours(scores, boxes, num_classes=21, score_thresh=0.05, nms=0.5, detections_per_im=100, soft_nms=soft,
                               soft_sigma=float(g["soft_nms_sigma"]), soft_method=method, bbox_vote=vote, vote_th=0.8,
                               vote_scoring=scoring)
            assert len(oc) == 21
            ref_cls = np.split(g[key + "/cls"], np.cumsum(g[key + "/cls_counts"])[:-1])
            for j in range(1, 21):
                a, b = ref_cls[j - 1], np.asarray(oc[j]).reshape(-1, 5)
                assert a.shape == b.shape, (seed, soft, method, vote, scoring, j, a.shape, b.shape)
                if vote:      # numpy averages in float32 pairwise order; ours accumulates in fp64
                    np.testing.assert_allclose(b, a, rtol=1e-4, atol=2e-3)
                elif soft and method == "gaussian":
                    np.testing.assert_allclose(b, a, rtol=1e-6, atol=1e-6)
                else:
                    assert np.array_equal(a, b), (seed, soft, method, j)
            assert g[key + "/scores"].shape == os_.shape and g[key + "/boxes"].shape == ob.shape
            checked += 1
    assert checked == 18


def test_detection_batches_validate_on_the_host():
    import ctypes
    from detectron.pytorch_b200 import _lib
    lib = _lib.load()
    counts = (ctypes.c_int * 2)(3, 4)
    assert lib.b200_soft_nms_batched(None, ctypes.cast(counts, ctypes.c_void_p), 2, ctypes.c_float(0.5), ctypes.c_float(0.3),
                                     ctypes.c_float(0.001), 1, None, None, None) == -1
    assert lib.b200_box_voting_batched(None, ctypes.cast(counts, ctypes.c_void_p), None, ctypes.cast(counts, ctypes.c_void_p), 2,
                                       ctypes.c_float(0.8), 9, ctypes.c_float(1.0), None, None) == -1
