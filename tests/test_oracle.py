"""CPU-only: pin the oracle (oracle/roi_ops_oracle.c).

  * index / weight logic  vs  torchvision.ops.roi_align(aligned=False), roi_pool, F.grid_sample  (independent code)
  * the fused (GPU-rounding) variant  vs  golden outputs of the REFERENCE's own CUDA kernels
    (tests/golden/*.npz, produced on a B200 by tests/golden/make_golden.py from oracle/_ref)
  * internal consistency: backward == adjoint of forward, NMS vs a pure-Python greedy loop.
"""
import os

import numpy as np
import pytest
import torch
import torchvision

from detectron.pytorch_b200 import synthetic as S
from oracle import cpu as O
from tests import cases

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _golden(name):
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        pytest.skip("golden file %s not generated yet" % name)
    return np.load(path)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_unfused_equals_torchvision(name):
    c, f, r, _ = cases.roi_case(name)
    O.set_fused(False)
    try:
        out = O.roi_align_forward(f, r, c["P"], c["P"], c["scale"], c["sr"])
    finally:
        O.set_fused(True)
    tv = torchvision.ops.roi_align(torch.from_numpy(f), torch.from_numpy(r), (c["P"], c["P"]), c["scale"], c["sr"],
                                   aligned=False).numpy()
    assert np.array_equal(out, tv)          # bit-exact


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_fused_close_to_torchvision(name):
    c, f, r, _ = cases.roi_case(name)
    out = O.roi_align_forward(f, r, c["P"], c["P"], c["scale"], c["sr"])
    tv = torchvision.ops.roi_align(torch.from_numpy(f), torch.from_numpy(r), (c["P"], c["P"]), c["scale"], c["sr"],
                                   aligned=False).numpy()
    # FMA contraction moves sample coordinates by <= 1 ulp: a few 1e-5 at |feature| ~ 4
    np.testing.assert_allclose(out, tv, rtol=0, atol=1e-4)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_backward_is_adjoint(name):
    c, f, r, dy = cases.roi_case(name)
    out = O.roi_align_forward(f, r, c["P"], c["P"], c["scale"], c["sr"])
    dx = O.roi_align_backward(dy, r, c["shape"], c["P"], c["P"], c["scale"], c["sr"], acc64=True)
    lhs = float(np.sum(out.astype(np.float64) * dy))
    rhs = float(np.sum(dx.astype(np.float64) * f))
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))
    dx32 = O.roi_align_backward(dy, r, c["shape"], c["P"], c["P"], c["scale"], c["sr"])
    np.testing.assert_allclose(dx32, dx, rtol=1e-5, atol=1e-5)   # fp32 summation-order noise scales with |dx|


def test_roi_align_backward_vs_torchvision_autograd():
    c, f, r, dy = cases.roi_case("cfg1_small")
    ft = torch.from_numpy(f).requires_grad_(True)
    o = torchvision.ops.roi_align(ft, torch.from_numpy(r), (c["P"], c["P"]), c["scale"], c["sr"], aligned=False)
    o.backward(torch.from_numpy(dy))
    dx = O.roi_align_backward(dy, r, c["shape"], c["P"], c["P"], c["scale"], c["sr"], acc64=True)
    np.testing.assert_allclose(dx, ft.grad.numpy(), rtol=0, atol=2e-4)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_pool_equals_torchvision(name):
    c, f, r, _ = cases.roi_case(name)
    out, argmax = O.roi_pool_forward(f, r, c["P"], c["P"], c["scale"])
    tv = torchvision.ops.roi_pool(torch.from_numpy(f), torch.from_numpy(r), (c["P"], c["P"]), c["scale"]).numpy()
    assert np.array_equal(out, tv)
    flat = f.reshape(-1)
    sel = argmax >= 0
    assert np.array_equal(flat[argmax[sel]], out[sel])
    assert np.all(out[~sel] == 0)


def test_roi_pool_backward_matches_scatter():
    c, f, r, dy = cases.roi_case("cfg1_small")
    out, argmax = O.roi_pool_forward(f, r, c["P"], c["P"], c["scale"])
    dx = O.roi_pool_backward(dy, argmax, r, c["shape"], c["P"], c["P"], c["scale"])
    # a plain scatter-add of dy at argmax is an upper bound of what the reference credits; it only
    # differs where the reference's feasibility test drops a contribution
    scat = np.zeros(f.size, np.float64)
    np.add.at(scat, argmax[argmax >= 0], dy[argmax >= 0].astype(np.float64))
    diff = np.abs(dx.reshape(-1) - scat)
    assert np.mean(diff > 1e-4) < 0.01


def test_roi_crop_equals_grid_sample():
    img, grid, go = cases.crop_case()
    out = O.roi_crop_forward(img, grid)
    N = img.shape[0]
    per = grid.shape[0] // N
    rep = torch.from_numpy(img).repeat_interleave(per, 0)
    gxy = torch.from_numpy(grid[..., ::-1].copy())
    tv = torch.nn.functional.grid_sample(rep, gxy, mode="bilinear", padding_mode="zeros", align_corners=True).numpy()
    np.testing.assert_allclose(out, tv, rtol=0, atol=2e-5)
    # image gradient
    rep_t = torch.from_numpy(img).clone().requires_grad_(True)
    o = torch.nn.functional.grid_sample(rep_t.repeat_interleave(per, 0), gxy, mode="bilinear", padding_mode="zeros",
                                        align_corners=True)
    o.backward(torch.from_numpy(go))
    gi = O.roi_crop_backward(go, grid, img.shape, acc64=True)
    np.testing.assert_allclose(gi, rep_t.grad.numpy(), rtol=0, atol=1e-4)


# Non-square pooled grids (PH, PW, sr): every kernel keeps separate PH / PW index arithmetic, and so must the oracle that
# checks them -- a swap of the two sizes shows up as a wrong shape or as different values here.
NON_SQUARE = [(7, 14, 2), (14, 7, 2), (3, 9, 1), (16, 5, 2), (1, 31, 1), (5, 3, 0)]


def non_square_case(PH, PW, seed=0):
    shape, scale = (2, 5, 38, 52), 1.0 / 8
    f = S.make_features(shape, seed=seed)
    r = np.concatenate([S.make_rois(28, shape, scale, seed=seed, min_size=8, max_size=400),
                        S.make_edge_rois(shape, scale)]).astype(np.float32)
    dy = np.random.RandomState(seed + 1).standard_normal((r.shape[0], shape[1], PH, PW)).astype(np.float32)
    return shape, scale, f, r, dy


@pytest.mark.parametrize("PH,PW,sr", NON_SQUARE)
def test_roi_align_non_square_vs_torchvision(PH, PW, sr):
    shape, scale, f, r, dy = non_square_case(PH, PW)
    tv = torchvision.ops.roi_align(torch.from_numpy(f), torch.from_numpy(r), (PH, PW), scale, sr, aligned=False).numpy()
    O.set_fused(False)
    try:
        out = O.roi_align_forward(f, r, PH, PW, scale, sr)
    finally:
        O.set_fused(True)
    assert out.shape == (r.shape[0], shape[1], PH, PW)
    assert np.array_equal(out, tv)                                         # bit-exact unfused
    np.testing.assert_allclose(O.roi_align_forward(f, r, PH, PW, scale, sr), tv, rtol=0, atol=1e-4)
    # backward vs torchvision's autograd in float64 (same sample positions: the RoIs are exact in float32)
    ft = torch.from_numpy(f.astype(np.float64)).requires_grad_(True)
    o = torchvision.ops.roi_align(ft, torch.from_numpy(r.astype(np.float64)), (PH, PW), scale, sr, aligned=False)
    o.backward(torch.from_numpy(dy.astype(np.float64)))
    dx = O.roi_align_backward(dy, r, shape, PH, PW, scale, sr, acc64=True)
    np.testing.assert_allclose(dx, ft.grad.numpy(), rtol=0, atol=1e-4)
    # the transposed grid is a different operation: a kernel that swaps PH and PW cannot pass both
    if PH != PW:
        tv_t = torchvision.ops.roi_align(torch.from_numpy(f), torch.from_numpy(r), (PW, PH), scale, sr, aligned=False).numpy()
        assert not np.allclose(tv_t, np.swapaxes(out, 2, 3), atol=1e-3)


@pytest.mark.parametrize("PH,PW", [(PH, PW) for PH, PW, _ in NON_SQUARE])
def test_roi_pool_non_square_vs_torchvision(PH, PW):
    shape, scale, f, r, dy = non_square_case(PH, PW)
    out, argmax = O.roi_pool_forward(f, r, PH, PW, scale)
    tv = torchvision.ops.roi_pool(torch.from_numpy(f), torch.from_numpy(r), (PH, PW), scale).numpy()
    assert out.shape == (r.shape[0], shape[1], PH, PW)
    assert np.array_equal(out, tv)
    sel = argmax >= 0
    assert np.array_equal(f.reshape(-1)[argmax[sel]], out[sel])
    assert np.all(out[~sel] == 0)
    # backward: where the reference's feasibility test keeps every contribution, the gradient is a scatter of dy at argmax
    dx = O.roi_pool_backward(dy, argmax, r, shape, PH, PW, scale)
    scat = np.zeros(f.size, np.float64)
    np.add.at(scat, argmax[sel], dy[sel].astype(np.float64))
    assert np.mean(np.abs(dx.reshape(-1) - scat) > 1e-4) < 0.01


def _py_greedy_nms(b, thresh):
    keep, removed = [], np.zeros(len(b), bool)
    f32 = np.float32
    for i in range(len(b)):
        if removed[i]:
            continue
        keep.append(i)
        a = b[i]
        Sa = f32(f32(f32(a[2] - a[0]) + f32(1)) * f32(f32(a[3] - a[1]) + f32(1)))
        for j in range(i + 1, len(b)):
            if removed[j]:
                continue
            c = b[j]
            w = max(f32(f32(min(a[2], c[2]) - max(a[0], c[0])) + f32(1)), f32(0))
            h = max(f32(f32(min(a[3], c[3]) - max(a[1], c[1])) + f32(1)), f32(0))
            inter = f32(w * h)
            bw = f32(f32(c[2] - c[0]) + f32(1)); bh = f32(f32(c[3] - c[1]) + f32(1))
            t = f32(np.float64(bw) * np.float64(bh) + np.float64(Sa))      # fma: single rounding of the exact product+sum
            den = f32(t - inter)
            if f32(inter / den) > f32(thresh):
                removed[j] = True
    return np.asarray(keep, np.int32)


@pytest.mark.parametrize("n", [1, 2, 63, 64, 65, 300])
def test_nms_cuda_semantics_vs_python(n):
    b = cases.nms_case(n)
    k = O.nms_cuda(b, 0.7)
    assert np.array_equal(k, _py_greedy_nms(b, 0.7))
    assert np.all(np.diff(k) > 0) and k[0] == 0


def test_nms_mask_consistent_with_scan():
    b = cases.nms_case(200)
    mask = O.nms_cuda_mask(b, 0.7)
    cb = mask.shape[1]
    remv = np.zeros(cb, np.uint64)
    keep = []
    for i in range(200):
        if not (int(remv[i // 64]) >> (i % 64)) & 1:
            keep.append(i)
            remv[i // 64:] |= mask[i, i // 64:]
    assert np.array_equal(np.asarray(keep, np.int32), O.nms_cuda(b, 0.7))


def test_nms_empty_and_flavours():
    assert len(O.nms_cuda(np.zeros((0, 5), np.float32), 0.7)) == 0
    b = cases.nms_case(1000)
    # the cython flavour (>=, unfused) agrees with the CUDA flavour on generic data ...
    assert np.array_equal(O.nms_cuda(b, 0.7), O.nms_cython(b, 0.7).astype(np.int32))
    # ... but not at an exact-threshold tie: IoU == 0.5 is suppressed by cython (>=) only
    t = np.array([[0, 0, 9, 19, 0.9], [0, 0, 9, 9, 0.8]], np.float32)      # inter 100, union 200
    assert list(O.nms_cuda(t, 0.5)) == [0, 1]
    assert list(O.nms_cython(t, 0.5)) == [0]


# ---- golden vectors from the reference's own CUDA kernels (generated on a B200) ----------------
@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_oracle_matches_reference_kernel_golden_roi_align(name):
    g = _golden("roi_align_xfrom_" + name)
    c, f, r, dy = cases.roi_case(name)
    out = O.roi_align_forward(f, r, c["P"], c["P"], c["scale"], c["sr"])
    assert np.array_equal(out, g["out"])                     # bit-exact with the reference kernel
    dx = O.roi_align_backward(dy, r, c["shape"], c["P"], c["P"], c["scale"], c["sr"], acc64=True)
    np.testing.assert_allclose(dx, g["dx"], rtol=1e-5, atol=1e-5)   # reference uses fp32 atomics (order noise)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_oracle_matches_reference_kernel_golden_legacy_and_pool(name):
    g = _golden("legacy_pool_" + name)
    c, f, r, dy = cases.roi_case(name)
    out = O.roi_align_legacy_forward(f, r, c["P"], c["P"], c["scale"])
    assert np.array_equal(out, g["legacy_out"])
    dx = O.roi_align_legacy_backward(dy, r, c["shape"], c["P"], c["P"], c["scale"], acc64=True)
    np.testing.assert_allclose(dx, g["legacy_dx"], rtol=1e-5, atol=1e-5)
    po, am = O.roi_pool_forward(f, r, c["P"], c["P"], c["scale"])
    assert np.array_equal(po, g["pool_out"]) and np.array_equal(am, g["pool_argmax"])
    pdx = O.roi_pool_backward(dy, am, r, c["shape"], c["P"], c["P"], c["scale"])
    assert np.array_equal(pdx, g["pool_dx"])                 # deterministic gather: bit-exact


def test_oracle_matches_reference_kernel_golden_crop():
    g = _golden("roi_crop")
    img, grid, go = cases.crop_case()
    assert np.array_equal(O.roi_crop_forward(img, grid), g["out"])
    np.testing.assert_allclose(O.roi_crop_backward(go, grid, img.shape, acc64=True), g["grad_img"], rtol=1e-5, atol=1e-5)
    assert not np.any(g["grad_grid"])                        # the reference CUDA kernel never writes it


@pytest.mark.parametrize("n", cases.NMS_SIZES)
def test_oracle_matches_reference_kernel_golden_nms(n):
    g = _golden("nms")
    keep = O.nms_cuda(cases.nms_case(n), 0.7)
    assert np.array_equal(keep, g["keep_%d" % n])
