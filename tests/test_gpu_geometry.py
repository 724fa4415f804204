"""GPU tests of the RoI ops away from the square grids and ordinary shapes the rest of the suite uses:
  * non-square pooled grids (PH != PW) through every RoIAlign forward path and every backward path, legacy RoIAlign, RoIPool,
    RoIAlignAvg / RoIAlignMax, the reference-named launchers and the FPN pyramid call;
  * both sides of each dispatch limit of the quad-strip forward (tests/cases.py QUAD_LIMITS;
    tests/test_abi.py pins which side of each limit its shapes are on);
  * the quad-strip prepass with more RoIs than resident CTAs (several RoIs per CTA before its grid barrier);
  * the FPN pyramid call at batch sizes whose strip geometry no longer fits (the per-level loop must take over).

The CPU oracle (oracle/roi_ops_oracle.c) is the reference throughout.  Tolerances are those of tests/test_gpu_parity.py:
forward bit-exact on the generic path, 1e-6 with a floor on the fraction of bit-exact elements on the fast paths, gradients
within 1e-5 of the fp64-accumulated oracle.  Launch-counter deltas prove which path ran: quad-strip forward 2 (prep + main),
stream 3 (count + fill + main), tiled 2, generic 1; NHWC and gather backward 2, scalar-atomic backward 1.
"""
import ctypes

import numpy as np
import pytest
import torch

from detectron.pytorch_b200 import _lib, synthetic as S
from detectron.pytorch_b200.model.roi_align.functions.roi_align import RoIAlignFunction as LegacyRoIAlignFunction
from detectron.pytorch_b200.model.roi_pooling.functions.roi_pool import RoIPoolFunction
from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align import RoIAlignFunction
from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align_fpn import RoIAlignFPNFunction
from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.modules.roi_align import RoIAlignAvg, RoIAlignMax
from oracle import cpu as O
from tests.cases import PYRAMID_800x1333, QUAD_LIMITS

pytestmark = pytest.mark.gpu
GRAD_TOL = dict(rtol=1e-5, atol=1e-5)
FWD_LAUNCHES = {"generic": 1, "tiled": 2, "stream": 3, "quad": 2}
BWD_LAUNCHES = {"generic": 1, "nhwc": 2, "rows": 2}
EXACT_FLOOR = {"tiled": 0.5, "stream": 0.9, "quad": 0.9}


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_fwd_matches(out, ref, path):
    """generic: bit-exact.  Fast paths: |a - b| <= 1e-6 + 1e-6 |b| (bins whose samples are summed as two or four partial sums)
    and most elements bit-exact."""
    if path == "generic":
        assert np.array_equal(out, ref)
    else:
        np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
        assert np.mean(out == ref) > EXACT_FLOOR[path]


@pytest.fixture
def roi_path(lib_option):
    """set(fwd, bwd): force the RoIAlign forward and backward dispatch for one test (restored afterwards)."""
    def set_paths(fwd=None, bwd=None):
        lib_option("B200_ROI_ALIGN_PATH", fwd)
        lib_option("B200_ROI_ALIGN_BWD_PATH", bwd)
    return set_paths


def with_bad_batch(r, row, N):
    """RoI `row` gets an out-of-range batch index: its output rows are zeros and it contributes no gradient.  Returns the
    RoIs to run and the RoIs the oracle sees (batch 0) -- the caller zeroes that row of the oracle's output / dY."""
    r = r.copy(); r[row, 0] = N + 3
    rr = r.copy(); rr[row, 0] = 0
    return r, rr


# ------------------------------------------------------------------------------------ non-square RoIAlign
# (PH, PW, sr): the table's grids at the quad-strip axis limit, mask-head halves, single rows / columns
NON_SQUARE = [(7, 14, 2), (14, 7, 2), (2, 7, 2), (14, 7, 1), (3, 9, 1), (16, 5, 2), (16, 3, 2), (3, 16, 2), (1, 31, 1), (31, 1, 1)]
# forward path -> the backward it is paired with (all three backward paths appear)
FWD_BWD = {"generic": "generic", "tiled": "nhwc", "stream": "generic", "quad": "nhwc"}


@pytest.mark.parametrize("fwd", sorted(FWD_BWD))
@pytest.mark.parametrize("PH,PW,sr", NON_SQUARE)
def test_roi_align_non_square_every_path(PH, PW, sr, fwd, roi_path):
    bwd = FWD_BWD[fwd]
    roi_path(fwd, bwd)
    shape, s = (2, 8, 46, 70), 1.0 / 8
    lib = _lib.load()
    f = S.make_features(shape, seed=PH * 32 + PW)
    r = np.concatenate([S.make_rois(60, shape, s, seed=PW, min_size=8, max_size=256), S.make_edge_rois(shape, s)]).astype(np.float32)
    r, rr = with_bad_batch(r, 5, shape[0])
    R = r.shape[0]
    dy = np.random.RandomState(sr).standard_normal((R, shape[1], PH, PW)).astype(np.float32)
    ref = O.roi_align_forward(f, rr, PH, PW, s, sr); ref[5] = 0
    dyr = dy.copy(); dyr[5] = 0
    ref_dx = O.roi_align_backward(dyr, rr, shape, PH, PW, s, sr, acc64=True)

    # every grid here is inside every fast path's limits (P * sr <= 32 per axis, sr in {1, 2})
    assert (lib.b200_roi_align_workspace_bytes(shape[0], R, shape[2], shape[3], PH, PW, sr) > 0) == (fwd != "generic")
    assert (lib.b200_roi_align_backward_workspace_bytes(shape[0], R, shape[1], shape[2], shape[3], PH, PW, sr) > 0) == (bwd != "generic")
    F = dev(f).requires_grad_(True)
    before = _lib.launch_count()
    out = RoIAlignFunction(PH, PW, s, sr)(F, dev(r))
    assert _lib.launch_count() - before == FWD_LAUNCHES[fwd]
    assert tuple(out.shape) == (R, shape[1], PH, PW)
    before = _lib.launch_count()
    out.backward(dev(dy))
    assert _lib.launch_count() - before == BWD_LAUNCHES[bwd]
    assert_fwd_matches(out.detach().cpu().numpy(), ref, fwd)
    np.testing.assert_allclose(F.grad.cpu().numpy(), ref_dx, **GRAD_TOL)


# (PH, PW, sr, C): the row-stationary gather backward takes PW in {7, 14} and any PH; C % 128 == 0 selects 4 channels per lane
ROWS_GRIDS = [(14, 7, 2, 64), (3, 7, 2, 128), (16, 7, 2, 64), (5, 14, 2, 64), (14, 7, 1, 128), (2, 14, 1, 64)]


@pytest.mark.parametrize("PH,PW,sr,C", ROWS_GRIDS)
def test_roi_align_backward_rows_non_square(PH, PW, sr, C, roi_path):
    roi_path("quad", "rows")
    shape, s = (2, C, 30, 45), 1.0 / 8
    f = S.make_features(shape, seed=1)
    r = np.concatenate([S.make_rois(40, shape, s, seed=PH, min_size=8, max_size=300), S.make_edge_rois(shape, s)]).astype(np.float32)
    r, rr = with_bad_batch(r, 3, shape[0])
    R = r.shape[0]
    dy = np.random.RandomState(PW).standard_normal((R, C, PH, PW)).astype(np.float32)
    dyr = dy.copy(); dyr[3] = 0
    # the workspace is the gather path's (the scalar-atomic kernel needs none): the gather path is the one that runs
    assert _lib.load().b200_roi_align_backward_workspace_bytes(shape[0], R, C, shape[2], shape[3], PH, PW, sr) > 0
    F = dev(f).requires_grad_(True)
    out = RoIAlignFunction(PH, PW, s, sr)(F, dev(r))
    before = _lib.launch_count()
    out.backward(dev(dy))
    assert _lib.launch_count() - before == BWD_LAUNCHES["rows"]
    ref = O.roi_align_forward(f, rr, PH, PW, s, sr); ref[3] = 0
    assert_fwd_matches(out.detach().cpu().numpy(), ref, "quad")
    np.testing.assert_allclose(F.grad.cpu().numpy(), O.roi_align_backward(dyr, rr, shape, PH, PW, s, sr, acc64=True), **GRAD_TOL)


def test_roi_align_auto_dispatch_sends_non_square_grid_through_gather_backward(lib_option):
    """PH = 14, PW = 7 at a shape where the automatic backward choice is the gather path (enough taps, enough rows)."""
    shape, s, PH, PW, sr = (1, 256, 150, 136), 1.0 / 4, 14, 7, 2
    R = 200
    lib = _lib.load()
    auto = lib.b200_roi_align_backward_workspace_bytes(shape[0], R, shape[1], shape[2], shape[3], PH, PW, sr)
    lib_option("B200_ROI_ALIGN_BWD_PATH", "rows")
    assert auto > 0 and auto == lib.b200_roi_align_backward_workspace_bytes(shape[0], R, shape[1], shape[2], shape[3], PH, PW, sr)
    lib_option("B200_ROI_ALIGN_BWD_PATH", None)
    f = S.make_features(shape, seed=3)
    r = S.make_rois(R, shape, s, seed=4).astype(np.float32)
    dy = np.random.RandomState(5).standard_normal((R, shape[1], PH, PW)).astype(np.float32)
    F = dev(f).requires_grad_(True)
    out = RoIAlignFunction(PH, PW, s, sr)(F, dev(r))
    before = _lib.launch_count()
    out.backward(dev(dy))
    assert _lib.launch_count() - before == BWD_LAUNCHES["rows"]
    np.testing.assert_allclose(out.detach().cpu().numpy(), O.roi_align_forward(f, r, PH, PW, s, sr), rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(F.grad.cpu().numpy(), O.roi_align_backward(dy, r, shape, PH, PW, s, sr, acc64=True), **GRAD_TOL)


# ------------------------------------------------------------------------- non-square legacy RoIAlign, RoIPool
# legacy RoIAlign places PH x PW samples on the lattice corners, bin size = extent / (P - 1): PH = 1 is all NaN, as in the reference
@pytest.mark.parametrize("PH,PW", [(7, 14), (14, 7), (3, 9), (2, 31), (31, 2), (16, 5)])
def test_legacy_roi_align_and_roi_pool_non_square(PH, PW):
    shape, s = (2, 6, 40, 52), 1.0 / 8
    f = S.make_features(shape, seed=2)
    r = np.concatenate([S.make_rois(30, shape, s, seed=PH, min_size=8, max_size=300), S.make_edge_rois(shape, s)]).astype(np.float32)
    dy = np.random.RandomState(PW).standard_normal((r.shape[0], shape[1], PH, PW)).astype(np.float32)
    F = dev(f).requires_grad_(True)
    out = LegacyRoIAlignFunction(PH, PW, s)(F, dev(r))
    out.backward(dev(dy))
    assert np.array_equal(out.detach().cpu().numpy(), O.roi_align_legacy_forward(f, r, PH, PW, s))
    np.testing.assert_allclose(F.grad.cpu().numpy(), O.roi_align_legacy_backward(dy, r, shape, PH, PW, s, acc64=True), **GRAD_TOL)
    fn = RoIPoolFunction(PH, PW, s)
    Fp = dev(f).requires_grad_(True)
    pout = fn(Fp, dev(r))
    pout.backward(dev(dy))
    o_out, o_arg = O.roi_pool_forward(f, r, PH, PW, s)
    assert np.array_equal(pout.detach().cpu().numpy(), o_out)
    assert np.array_equal(fn.argmax.cpu().numpy(), o_arg)
    assert np.array_equal(Fp.grad.cpu().numpy(), O.roi_pool_backward(dy, o_arg, r, shape, PH, PW, s))


@pytest.mark.parametrize("PH,PW", [(7, 3), (3, 7)])
def test_roi_align_avg_max_non_square(PH, PW, lib_option):
    """RoIAlignAvg / RoIAlignMax align at (PH + 1) x (PW + 1) and pool 2 x 2 with stride 1."""
    lib_option("B200_ROI_ALIGN_PATH", "generic")
    shape, s = (2, 8, 50, 68), 1.0 / 16
    f = S.make_features(shape, seed=0)
    r = np.concatenate([S.make_rois(32, shape, s, seed=0), S.make_edge_rois(shape, s)]).astype(np.float32)
    base = torch.from_numpy(O.roi_align_forward(f, r, PH + 1, PW + 1, s, 2))
    avg = RoIAlignAvg(PH, PW, s, 2)(dev(f), dev(r)).cpu()
    mx = RoIAlignMax(PH, PW, s, 2)(dev(f), dev(r)).cpu()
    assert tuple(mx.shape) == (r.shape[0], shape[1], PH, PW)
    assert torch.equal(mx, torch.nn.functional.max_pool2d(base, 2, 1))
    torch.testing.assert_close(avg, torch.nn.functional.avg_pool2d(base, 2, 1), rtol=1e-6, atol=1e-6)


def test_reference_named_launchers_non_square():
    """ROIAlign* / ROIPool* of the compatibility libraries with aligned_height = 7, aligned_width = 14 (and the transpose)."""
    from detectron.pytorch_b200 import build as B
    lib = ctypes.CDLL(B.compat_lib_path("libb200_ref_launchers.so"))
    leg = ctypes.CDLL(B.compat_lib_path("libb200_ref_launchers_legacy.so"))
    shape, s, sr = (2, 8, 50, 68), 1.0 / 16, 2
    N, C, H, W = shape
    f = S.make_features(shape, seed=0)
    r = np.concatenate([S.make_rois(32, shape, s, seed=0), S.make_edge_rois(shape, s)]).astype(np.float32)
    R = r.shape[0]
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    F, Rt = dev(f), dev(r)
    for PH, PW in ((7, 14), (14, 7)):
        dy = np.random.RandomState(PH).standard_normal((R, C, PH, PW)).astype(np.float32)
        DY = dev(dy)
        out = torch.empty((R, C, PH, PW), device="cuda")
        assert lib.ROIAlignForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, PH, PW, sr, vp(Rt), vp(out), st) == 1
        assert np.array_equal(out.cpu().numpy(), O.roi_align_forward(f, r, PH, PW, s, sr))
        dx = torch.empty(shape, device="cuda")
        assert lib.ROIAlignBackwardLaucher(vp(DY), ctypes.c_float(s), N, R, H, W, C, PH, PW, sr, vp(Rt), vp(dx), st) == 1
        np.testing.assert_allclose(dx.cpu().numpy(), O.roi_align_backward(dy, r, shape, PH, PW, s, sr, acc64=True), **GRAD_TOL)
        lout = torch.empty((R, C, PH, PW), device="cuda")
        assert leg.ROIAlignForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, PH, PW, vp(Rt), vp(lout), st) == 1
        assert np.array_equal(lout.cpu().numpy(), O.roi_align_legacy_forward(f, r, PH, PW, s))
        pout = torch.empty((R, C, PH, PW), device="cuda"); arg = torch.empty((R, C, PH, PW), dtype=torch.int32, device="cuda")
        assert lib.ROIPoolForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, PH, PW, vp(Rt), vp(pout), vp(arg), st) == 1
        o_out, o_arg = O.roi_pool_forward(f, r, PH, PW, s)
        assert np.array_equal(pout.cpu().numpy(), o_out) and np.array_equal(arg.cpu().numpy(), o_arg)
        pdx = torch.empty(shape, device="cuda")
        assert lib.ROIPoolBackwardLaucher(vp(DY), ctypes.c_float(s), N, R, H, W, C, PH, PW, vp(Rt), vp(pdx), vp(arg), st) == 1
        assert np.array_equal(pdx.cpu().numpy(), O.roi_pool_backward(dy, o_arg, r, shape, PH, PW, s))


# ---------------------------------------------------------------------------------------------- FPN
def fpn_case(shapes, counts, seed, min_size=16, max_size=300):
    scales = [1.0 / 2 ** (l + 2) for l in range(len(shapes))]
    feats = [S.make_features(sh, seed=seed + i) for i, sh in enumerate(shapes)]
    rois = [S.make_rois(c, sh, sc, seed=seed + 10 + i, min_size=min_size * 2 ** i, max_size=max_size * 2 ** i).astype(np.float32)
            if c else np.zeros((0, 5), np.float32) for i, (c, sh, sc) in enumerate(zip(counts, shapes, scales))]
    restore = np.random.RandomState(seed).permutation(sum(counts)).astype(np.int32)
    return scales, feats, rois, restore


def fpn_oracle(feats, rois, restore, PH, PW, scales, sr):
    parts = [O.roi_align_forward(f, r, PH, PW, sc, sr) for f, r, sc in zip(feats, rois, scales) if len(r)]
    return np.concatenate(parts, axis=0)[restore]


@pytest.mark.parametrize("PH,PW", [(7, 14), (14, 7)])
def test_roi_align_fpn_non_square(PH, PW):
    """RoIAlignFPNFunction(PH, PW, ...) against the per-level oracle in restored order, forward and backward; one pyramid
    call (prep + main: every level has W % 4 == 0) with an empty level."""
    shapes = [(2, 32, 48, 64), (2, 32, 24, 32), (2, 32, 12, 16), (2, 32, 6, 8)]
    counts = [150, 40, 0, 9]
    scales, feats, rois, restore = fpn_case(shapes, counts, seed=PH)
    total = sum(counts)
    dy = np.random.RandomState(PW).standard_normal((total, 32, PH, PW)).astype(np.float32)
    F = [dev(f).requires_grad_(True) for f in feats]
    before = _lib.launch_count()
    out = RoIAlignFPNFunction(PH, PW, scales, 2)(F, [dev(r) for r in rois], restore)
    assert _lib.launch_count() - before == 2
    out.backward(dev(dy))
    got = out.detach().cpu().numpy()
    assert got.shape == (total, 32, PH, PW)
    ref = fpn_oracle(feats, rois, restore, PH, PW, scales, 2)
    np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-6)
    assert np.mean(got == ref) > 0.9
    inv = np.empty_like(restore); inv[restore] = np.arange(total, dtype=np.int32)
    off = 0
    for Fl, f, r, sc, c in zip(F, feats, rois, scales, counts):
        if c:                                          # level l's RoIs own rows inv[off:off + c] of the restored output
            ref_dx = O.roi_align_backward(dy[inv[off:off + c]], r, f.shape, PH, PW, sc, 2, acc64=True)
            np.testing.assert_allclose(Fl.grad.cpu().numpy(), ref_dx, **GRAD_TOL)
        else:
            assert torch.count_nonzero(Fl.grad) == 0
        off += c


@pytest.mark.parametrize("path", ["auto", "stream"])
@pytest.mark.parametrize("N", [5, 6, 8])
def test_roi_align_fpn_batch_beyond_strip_geometry(N, path, lib_option):
    """The 800 x 1333 pyramid (P2..P5) at batch 5 fits the quad-strip geometry (one pyramid call: P2..P4 by TMA, P5 by cp.async
    producers, two launches each); at batch 6 and 8 it has too many strip rows, so RoIAlignFPNFunction must fall back to the
    per-level loop -- also when the forward is forced onto the streaming path, which the pyramid call does not have."""
    if path == "stream":
        lib_option("B200_ROI_ALIGN_PATH", "stream")
    C = 8
    shapes = [(N, C) + hw for hw in PYRAMID_800x1333]
    counts = [300, 200, 100, 40]
    scales, feats, rois, restore = fpn_case(shapes, counts, seed=N)
    before = _lib.launch_count()
    out = RoIAlignFPNFunction(7, 7, scales, 2)([dev(f) for f in feats], [dev(r) for r in rois], restore).cpu().numpy()
    launches = _lib.launch_count() - before
    fused = path == "auto" and N <= 5
    hs = (ctypes.c_int * 4)(*[h for h, _ in PYRAMID_800x1333]); ws = (ctypes.c_int * 4)(*[w for _, w in PYRAMID_800x1333])
    assert (_lib.load().b200_roi_align_fpn_workspace_bytes(4, ctypes.cast(hs, ctypes.c_void_p), ctypes.cast(ws, ctypes.c_void_p),
                                                           N, sum(counts), 7, 7, 2) > 0) == fused
    if fused:
        assert launches == 4
    elif path == "auto":
        assert launches == 4                           # per level: too little work for the fast paths, one generic launch each
    ref = fpn_oracle(feats, rois, restore, 7, 7, scales, 2)
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
    assert np.mean(out == ref) > 0.9


# --------------------------------------------------------------------------------- quad-strip dispatch limits
def limit_rois(N, H, W, R, seed):
    """R RoIs on an (N, ., H, W) map at scale 1/4 (boxes of 2..48 cells), plus the edge RoIs when there is room."""
    shape = (N, 1, H, W)
    r = S.make_rois(R, shape, 0.25, seed=seed, min_size=8, max_size=192).astype(np.float32)
    if R >= 64:
        e = S.make_edge_rois(shape, 0.25)
        r[:len(e)] = e
    return r


@pytest.mark.parametrize("side", ["accepted", "rejected"])
@pytest.mark.parametrize("limit", sorted(QUAD_LIMITS))
def test_quad_strip_limits_both_sides(limit, side, lib_option):
    """Under B200_ROI_ALIGN_PATH=quad: the last shape each limit admits runs the quad-strip kernels (2 launches) and matches the
    oracle; the first shape it rejects falls back to the generic kernel (1 launch) and is bit-exact."""
    lib_option("B200_ROI_ALIGN_PATH", "quad")
    N, H, W, R, PH, PW, sr = QUAD_LIMITS[limit][0 if side == "accepted" else 1]
    C, s = 4, 0.25
    f = S.make_features((N, C, H, W), seed=7)
    r = limit_rois(N, H, W, R, seed=8)
    before = _lib.launch_count()
    out = RoIAlignFunction(PH, PW, s, sr)(dev(f), dev(r)).cpu().numpy()
    assert _lib.launch_count() - before == (2 if side == "accepted" else 1)
    ref = O.roi_align_forward(f, r, PH, PW, s, sr)
    assert_fwd_matches(out, ref, "quad" if side == "accepted" else "generic")


def test_quad_strip_prepass_more_rois_than_resident_ctas(lib_option):
    """8000 RoIs on a BASELINE-cfg2-sized map: the prepass grid is capped at the resident CTAs (<= 16 per SM x 148 SMs), so
    each CTA walks several RoIs before the grid barrier.  Matches the oracle and is bit-identical run to run."""
    lib_option("B200_ROI_ALIGN_PATH", "quad")
    shape, s, P, sr = (1, 32, 200, 272), 0.25, 7, 2
    f = S.make_features(shape, seed=9)
    r = S.make_rois(8000, shape, s, seed=10).astype(np.float32)
    F, Rt = dev(f), dev(r)
    before = _lib.launch_count()
    out = RoIAlignFunction(P, P, s, sr)(F, Rt)
    assert _lib.launch_count() - before == 2
    out2 = RoIAlignFunction(P, P, s, sr)(F, Rt)
    assert torch.equal(out, out2)
    assert_fwd_matches(out.cpu().numpy(), O.roi_align_forward(f, r, P, P, s, sr), "quad")
