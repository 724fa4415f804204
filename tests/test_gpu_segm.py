"""GPU: the Mask R-CNN mask paste and RLE on the device (csrc/segm.cu, core.test.segm_results) against the reference's own
segm_results with cv2's IPP off (tests/golden/segm.npz) and the numpy restatement oracle/segm.py."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import segm as oseg
from tests.segm_cases import segm_case

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "segm.npz")
GOLDEN_CASES = ("a", "b", "c", "d")


def _cfg(c):
    return SimpleNamespace(MODEL=SimpleNamespace(NUM_CLASSES=c["num_classes"]),
                           MRCNN=SimpleNamespace(RESOLUTION=c["M"], CLS_SPECIFIC_MASK=c["cls_specific"], THRESH_BINARIZE=0.5))


def _channels(c):
    return oseg.channels_for([len(b) for b in c["cls_boxes"][1:]], c["cls_specific"])


def _golden_runs(g, name):
    return np.split(g[name + "/off/runs"], np.cumsum(g[name + "/off/counts"])[:-1])


def _rles_to_runs(segms, K):
    out = []
    for j in range(1, K):
        for rle in segms[j]:
            out.append(np.asarray(rle["counts"], np.int64))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN_CASES)
@pytest.mark.parametrize("inputs", ("numpy", "cuda"))
@pytest.mark.parametrize("config", ("cfg", "kw"))
def test_segm_results_matches_the_reference(name, inputs, config):
    import torch
    from detectron.pytorch_b200.core import test as T
    c = segm_case(name)
    g = np.load(GOLDEN)
    masks, boxes = c["masks"], c["ref_boxes"]
    if inputs == "cuda":
        masks, boxes = torch.from_numpy(masks).cuda(), torch.from_numpy(boxes).cuda()
    if config == "cfg":
        segms = T.segm_results(c["cls_boxes"], masks, boxes, c["im_h"], c["im_w"], cfg=_cfg(c))
    else:
        segms = T.segm_results(c["cls_boxes"], masks, boxes, c["im_h"], c["im_w"], num_classes=c["num_classes"],
                               resolution=c["M"], cls_specific_mask=c["cls_specific"], thresh_binarize=0.5)
    K = c["num_classes"]
    assert len(segms) == K and segms[0] == []
    assert [len(s) for s in segms[1:]] == [len(b) for b in c["cls_boxes"][1:]]
    gold = _golden_runs(g, name)
    if T._coco_mask() is None:
        for rle in (r for s in segms[1:] for r in s):
            assert rle["size"] == [c["im_h"], c["im_w"]]
        ours = _rles_to_runs(segms, K)
        assert len(ours) == len(gold)
        for i, (a, b) in enumerate(zip(ours, gold)):
            np.testing.assert_array_equal(a, b, err_msg="%s detection %d" % (name, i))
    else:
        mask_util = T._coco_mask()
        dense = oseg.paste(c["masks"], _channels(c), c["ref_boxes"], c["im_h"], c["im_w"])
        flat = [r for s in segms[1:] for r in s]
        for i, rle in enumerate(flat):
            assert isinstance(rle["counts"], str)
            np.testing.assert_array_equal(mask_util.decode(rle), dense[i], err_msg="%s detection %d" % (name, i))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("a", "b", "c", "d", "e"))
def test_dense_paste_and_rle_match_the_oracle(name):
    import torch
    from detectron.pytorch_b200 import ops
    c = segm_case(name)
    ch = _channels(c)
    H, W = c["im_h"], c["im_w"]
    masks, boxes = torch.from_numpy(c["masks"]).cuda(), torch.from_numpy(c["ref_boxes"]).cuda()
    runs, counts = ops.segm_rle(masks, ch if c["cls_specific"] else None, boxes, H, W, 0.5)
    assert runs.dtype == np.int32 and counts.shape == (len(ch),)
    per = np.split(runs, np.cumsum(counts)[:-1])
    exp_boxes = oseg.expand_boxes_int(c["ref_boxes"], c["M"])
    step = 100
    for d0 in range(0, len(ch), step):
        d1 = min(d0 + step, len(ch))
        dense = ops.segm_paste(masks[d0:d1], ch[d0:d1] if c["cls_specific"] else None, boxes[d0:d1], H, W, 0.5).cpu().numpy()
        for i in range(d0, d1):
            ref = oseg.paste_one(c["masks"][i, ch[i]], exp_boxes[i], H, W, 0.5)
            np.testing.assert_array_equal(dense[i - d0], ref, err_msg="%s detection %d" % (name, i))
            np.testing.assert_array_equal(per[i], oseg.rle_runs(ref), err_msg="%s detection %d" % (name, i))
            assert per[i].sum() == H * W and per[i][1::2].sum() == dense[i - d0].sum()


@pytest.mark.gpu
def test_launch_count_does_not_depend_on_the_detection_count():
    import torch
    from detectron.pytorch_b200 import _lib, ops
    c = segm_case("e")
    masks, boxes = torch.from_numpy(c["masks"]).cuda(), torch.from_numpy(c["ref_boxes"]).cuda()
    H, W = c["im_h"], c["im_w"]
    used = {}
    for D in (0, 10, 1000):
        n0 = _lib.launch_count()
        ops.segm_rle(masks[:D], None, boxes[:D], H, W)
        n1 = _lib.launch_count()
        ops.segm_paste(masks[:D], None, boxes[:D], H, W)
        used[D] = (n1 - n0, _lib.launch_count() - n1)
    torch.cuda.synchronize()
    assert used[0] == (0, 0)
    assert used[10] == used[1000] == (3, 1)


@pytest.mark.gpu
def test_results_on_a_side_stream():
    import torch
    from detectron.pytorch_b200 import ops
    c = segm_case("a")
    ch = _channels(c)
    g = np.load(GOLDEN)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        masks, boxes = torch.from_numpy(c["masks"]).cuda(), torch.from_numpy(c["ref_boxes"]).cuda()
        runs, counts = ops.segm_rle(masks, ch, boxes, c["im_h"], c["im_w"])
        dense = ops.segm_paste(masks, ch, boxes, c["im_h"], c["im_w"])
        host = dense.cpu().numpy()
    np.testing.assert_array_equal(counts, g["a/off/counts"])
    np.testing.assert_array_equal(runs, g["a/off/runs"])
    for i in (0, 17, 99):
        np.testing.assert_array_equal(oseg.rle_runs(host[i]), _golden_runs(g, "a")[i])


@pytest.mark.gpu
def test_pycocotools_decode_equals_the_dense_mask():
    from detectron.pytorch_b200.core import test as T
    mask_util = T._coco_mask()
    if mask_util is None:
        pytest.skip("pycocotools not installed")
    c = segm_case("d")
    segms = T.segm_results(c["cls_boxes"], c["masks"], c["ref_boxes"], c["im_h"], c["im_w"], cfg=_cfg(c))
    dense = oseg.paste(c["masks"], _channels(c), c["ref_boxes"], c["im_h"], c["im_w"])
    flat = [r for s in segms[1:] for r in s]
    for i, rle in enumerate(flat):
        np.testing.assert_array_equal(mask_util.decode(rle), dense[i])
