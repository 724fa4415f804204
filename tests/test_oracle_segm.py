"""CPU: the numpy restatement of the Mask R-CNN mask paste (oracle/segm.py) against the reference's own segm_results
(lib/core/test.py:793-847, recorded in tests/golden/segm.npz by tests/golden/make_golden_segm.py) and against cv2, the
RLE invariants on every case of tests/segm_cases.py, and argument validation of the b200_segm_* entry points."""
import os

import numpy as np
import pytest

from oracle import segm as oseg
from tests.segm_cases import segm_case

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "segm.npz")
GOLDEN_CASES = ("a", "b", "c", "d")


def _oracle(name):
    c = segm_case(name)
    ch = oseg.channels_for([len(b) for b in c["cls_boxes"][1:]], c["cls_specific"])
    return c, ch, oseg.segm_runs(c["masks"], ch, c["ref_boxes"], c["im_h"], c["im_w"])


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_equals_reference_with_ipp_off(name):
    g = np.load(GOLDEN)
    _, _, (runs, counts, _) = _oracle(name)
    np.testing.assert_array_equal(counts, g[name + "/off/counts"])
    gr = np.split(g[name + "/off/runs"], np.cumsum(g[name + "/off/counts"])[:-1])
    ours = np.split(runs, np.cumsum(counts)[:-1])
    for i, (a, b) in enumerate(zip(ours, gr)):
        np.testing.assert_array_equal(a, b, err_msg="detection %d" % i)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_ipp_flips_are_few_and_at_the_threshold(name):
    g = np.load(GOLDEN)
    flips, vals = g[name + "/flips"], g[name + "/flip_values"]
    assert len(flips) == len(vals) <= 10
    assert np.all(np.abs(vals.astype(np.float64) - 0.5) <= 2e-6)
    assert np.all(flips[:, 3] == (vals > np.float32(0.5)))      # stored IPP-off value is the binarised resize
    same = (g[name + "/on/counts"].shape == g[name + "/off/counts"].shape and
            np.array_equal(g[name + "/on/runs"], g[name + "/off/runs"]))
    assert same == (len(flips) == 0)


@pytest.mark.parametrize("name", ("a", "b", "c", "d"))
def test_rle_invariants(name):
    c, _, (runs, counts, dense) = _oracle(name)
    H, W = c["im_h"], c["im_w"]
    for i, r in enumerate(np.split(runs, np.cumsum(counts)[:-1])):
        assert r.sum() == H * W
        assert np.all(r[1:] > 0) and r[0] >= 0                   # alternate: only the leading zero run may be empty
        assert r[1::2].sum() == dense[i].sum()
        np.testing.assert_array_equal(np.repeat(np.arange(len(r)) % 2, r).astype(np.uint8), dense[i].ravel(order="F"))


def test_edge_case_geometry():
    """The edge boxes of case c land where the reference's arithmetic puts them."""
    c = segm_case("c")
    b = oseg.expand_boxes_int(c["ref_boxes"], c["M"])
    x1, y1, x2, y2 = c["ref_boxes"][4]
    s = np.float32((c["M"] + 2.0) / c["M"])
    ex = (x2 + x1) * np.float32(.5) - (x2 - x1) * np.float32(.5) * s
    ey = (y2 + y1) * np.float32(.5) - (y2 - y1) * np.float32(.5) * s
    assert ex < -1 and ey < -1 and ex != np.floor(ex)
    assert (b[4, 0], b[4, 1]) == (np.trunc(ex), np.trunc(ey))                  # truncation toward zero
    assert b[9, 2] - b[9, 0] + 1 <= 1 and b[10, 3] - b[10, 1] + 1 <= 1
    assert b[11, 2] < b[11, 0]
    assert tuple(b[13, 2:] - b[13, :2] + 1) == (30, 30) and tuple(b[14, 2:] - b[14, :2] + 1) == (15, 15)
    _, _, (_, counts, dense) = _oracle("c")
    assert np.all(dense[6:9].sum(axis=(1, 2)) == 0) and np.all(counts[6:9] == 1)   # entirely outside
    assert dense[12].sum() > 0                                                     # larger than the image


def test_case_d_runs_wrap_across_columns():
    c, _, (runs, counts, dense) = _oracle("d")
    wraps = 0
    for i in range(len(counts)):
        col = dense[i]
        wraps += int(np.sum(col[-1, :-1] & col[0, 1:]))
    assert wraps > 0


def test_resize_equals_cv2_without_ipp():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.RandomState(7)
    ipp = cv2.ipp.useIPP()
    try:
        cv2.ipp.setUseIPP(False)
        for M in (14, 28):
            src = rng.rand(M + 2, M + 2).astype(np.float32)
            sizes = [(1, 1), (M + 2, M + 2), ((M + 2) // 2, (M + 2) // 2), (1, 1000), (1500, 1)]
            sizes += [(int(rng.randint(1, 1501)), int(rng.randint(1, 1001))) for _ in range(24)]
            for w, h in sizes:
                a, b = cv2.resize(src, (w, h)), oseg.resize(src, w, h)
                np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32), err_msg="M %d, %d x %d" % (M, w, h))
    finally:
        cv2.ipp.setUseIPP(ipp)
    assert cv2.ipp.useIPP() == ipp


def test_case_e_is_consistent():
    c = segm_case("e")
    assert c["masks"].shape == (1000, 1, 28, 28) and c["ref_boxes"].shape == (1000, 4)
    assert sum(len(b) for b in c["cls_boxes"][1:]) == 1000


def test_segm_entry_points_reject_bad_arguments():
    from detectron.pytorch_b200 import _lib
    lib = _lib.load()
    EINVAL = -1
    P = 1 << 20                                # never dereferenced: validation fails first
    for fn, tail in ((lib.b200_segm_paste, [P]), (lib.b200_segm_rle_count, [P]), (lib.b200_segm_rle_emit, [P, P])):
        ok = [P, None, P, 4, 81, 28, 800, 1199, 0.5]
        bad = [
            [P, None, P, -1, 81, 28, 800, 1199, 0.5],      # negative count
            [P, None, P, 4, 0, 28, 800, 1199, 0.5],        # no channel
            [P, None, P, 4, 81, 0, 800, 1199, 0.5],        # resolution 0
            [P, None, P, 4, 81, 127, 800, 1199, 0.5],      # resolution above the limit
            [P, None, P, 4, 81, 28, 0, 1199, 0.5],         # empty image
            [P, None, P, 4, 81, 28, 800, -5, 0.5],
            [P, None, P, 4, 81, 28, 800, 32769, 0.5],      # wider than the limit
            [P, None, P, 4, 81, 28, 65536, 32768, 0.5],    # 2^31 pixels
            [None, None, P, 4, 81, 28, 800, 1199, 0.5],    # null masks
            [P, None, None, 4, 81, 28, 800, 1199, 0.5],    # null boxes
        ]
        for args in bad:
            assert fn(*(args + tail + [None])) == EINVAL, (fn.__name__, args)
        for k in range(len(tail)):
            t = list(tail); t[k] = None
            assert fn(*(ok + t + [None])) == EINVAL, (fn.__name__, "null output / offsets")
