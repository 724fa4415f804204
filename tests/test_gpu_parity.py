"""GPU parity tests (run with `-m gpu` on the B200 box): the sm_100a kernels, called through the
C ABI via the reference-shaped Python surface, against
  (1) the CPU oracle (oracle/roi_ops_oracle.c) on the same seeded inputs,
  (2) the reference's own CUDA kernels, through their outputs on the same inputs stored under tests/golden/
      (tests/golden/make_golden*.py run the reference; full-size outputs are stored as fixed, seeded samples),
and, at BASELINE.json's full sizes, through size-independent properties.

Tolerances: RoIAlign/legacy/crop forward, RoIPool fwd+bwd and NMS keep indices are BIT-EXACT
(integer / identically-rounded fp32 work).  Gradients that the reference accumulates with fp32
atomics are compared with |a-b| <= 1e-5 + 1e-5*|b| (north_star's 1e-5 fp32; summation order is
undefined in the reference itself).
"""
import os

import numpy as np
import pytest
import torch

from detectron.pytorch_b200 import _lib, synthetic as S
from detectron.pytorch_b200.model.nms.nms_gpu import nms_gpu
from detectron.pytorch_b200.model.nms.nms_wrapper import nms as nms_wrapper
from detectron.pytorch_b200.model.roi_align.functions.roi_align import RoIAlignFunction as LegacyRoIAlignFunction
from detectron.pytorch_b200.model.roi_crop.functions.roi_crop import RoICropFunction
from detectron.pytorch_b200.model.roi_pooling.functions.roi_pool import RoIPoolFunction
from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align import RoIAlignFunction
from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.modules.roi_align import RoIAlignAvg, RoIAlignMax
from oracle import cpu as O
from tests import cases

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
GRAD_TOL = dict(rtol=1e-5, atol=1e-5)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(params=["generic", "tiled", "tiled-rows", "stream", "quad"])
def fwd_path(request, lib_option):
    """Force the RoIAlign forward AND backward dispatch (b200_roi_ops_set_option):
    generic = RoI-centric kernels (scalar atomics in the backward), tiled = feature-map-stationary
    forward + vector-reduction (NHWC scratch) backward, tiled-rows = same forward + row-stationary gather
    backward (falls back to the scalar-atomic kernel for shapes it does not cover), stream = cp.async streaming-strip
    forward (falls back to the generic kernel for shapes it does not cover) + the default backward, quad = the quad-strip
    forward (roi_align_strip.cu, the default fast path; same fallback) + the default backward."""
    lib_option("B200_ROI_ALIGN_PATH", {"generic": "generic", "tiled": "tiled", "tiled-rows": "tiled", "stream": "stream", "quad": "quad"}[request.param])
    lib_option("B200_ROI_ALIGN_BWD_PATH", {"generic": "generic", "tiled": "nhwc", "tiled-rows": "rows", "stream": "auto", "quad": "auto"}[request.param])
    return request.param


def golden(name):
    return np.load(os.path.join(GOLDEN, name))


def sampled(a, g, key):
    """a's values at the sample the golden file `g` stores for `key` (tests/golden/make_golden_full_size.py)."""
    return a.reshape(-1)[cases.sample_index(a.size, int(g[key + "_seed"]))]


def run_fwd_bwd(fn, f, r, dy):
    F = dev(f).requires_grad_(True)
    out = fn(F, dev(r))
    out.backward(dev(dy))
    return out.detach().cpu().numpy(), F.grad.cpu().numpy()


def test_roi_crop_through_affine_grid_gen_matches_grid_sample():
    """The RoICrop pooling mode as model_builder.py:280-288 chains it: affine_grid_gen -> (y, x) swap -> RoICropFunction.
    For boxes inside the map this is bilinear grid sampling with corner alignment; torch's grid_sample is an independent
    implementation of the same arithmetic."""
    from detectron.pytorch_b200.utils.net import affine_grid_gen
    feat = dev(S.make_features((1, 6, 30, 44), seed=4))
    rois = torch.tensor([[0, 16.0, 32.0, 300.0, 200.0], [0, 100.0, 50.0, 600.0, 400.0], [0, 0.0, 0.0, 688.0, 464.0]]).cuda()
    grid_xy = affine_grid_gen(rois, feat.shape[2:], 7)
    grid_yx = torch.stack([grid_xy[:, :, :, 1], grid_xy[:, :, :, 0]], 3).contiguous()
    out = RoICropFunction()(feat, grid_yx)
    ref = torch.nn.functional.grid_sample(feat.expand(3, -1, -1, -1), grid_xy, mode="bilinear", padding_mode="zeros", align_corners=True)
    torch.testing.assert_close(out, ref, rtol=1e-5, atol=1e-5)


# ---------------------------------------------------------------------------------------- RoIAlign
def assert_fwd_matches(out, ref, path):
    """generic path: bit-exact.  tiled path: bit-exact except bins whose samples straddle two tiles,
    which add <= 4 partial means in a different association (~1 ulp): |a-b| <= 1e-6 + 1e-6*|b|.
    stream path: bit-exact except the rare bins whose samples cannot be resident together (two partial sums)."""
    if path in ("stream", "quad"):
        np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
        assert np.mean(out == ref) > 0.9
    elif path.startswith("tiled"):
        np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
        assert np.mean(out == ref) > 0.5
    else:
        assert np.array_equal(out, ref)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_vs_oracle(name, fwd_path):
    c, f, r, dy = cases.roi_case(name)
    P, s, sr = c["P"], c["scale"], c["sr"]
    out, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    assert_fwd_matches(out, O.roi_align_forward(f, r, P, P, s, sr), fwd_path)
    np.testing.assert_allclose(dx, O.roi_align_backward(dy, r, c["shape"], P, P, s, sr, acc64=True), **GRAD_TOL)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_vs_reference_kernel(name, fwd_path):
    """Against the reference kernel's own forward and backward on these inputs (tests/golden/make_golden.py)."""
    c, f, r, dy = cases.roi_case(name)
    P, s, sr = c["P"], c["scale"], c["sr"]
    out, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    g = golden("roi_align_xfrom_%s.npz" % name)
    ref_out, ref_dx = g["out"], g["dx"]
    assert_fwd_matches(out, ref_out, fwd_path)
    np.testing.assert_allclose(dx, ref_dx, **GRAD_TOL)


@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_roi_align_vs_golden(name, fwd_path):
    path = os.path.join(GOLDEN, "roi_align_xfrom_%s.npz" % name)
    if not os.path.exists(path):
        pytest.skip("golden not generated")
    g = np.load(path)
    c, f, r, dy = cases.roi_case(name)
    out, dx = run_fwd_bwd(RoIAlignFunction(c["P"], c["P"], c["scale"], c["sr"]), f, r, dy)
    assert_fwd_matches(out, g["out"], fwd_path)
    np.testing.assert_allclose(dx, g["dx"], **GRAD_TOL)


def test_roi_align_baseline_cfg1_and_cfg2_full_size(fwd_path):
    """BASELINE.json configs 1 and 2 at full size: forward bit-exact vs the oracle; backward within
    1e-5; plus size-independent properties (adjointness, linearity, dX support); and against a fixed, seeded sample of the
    reference kernel's own outputs (tests/golden/make_golden_full_size.py)."""
    for name, cfg in (("cfg1", S.CFG1), ("cfg2", S.CFG2)):
        P, s, sr = cfg["pooled"], cfg["scale"], cfg["sampling_ratio"]
        f = S.make_features(cfg["shape"]); r = S.make_rois(cfg["rois"], cfg["shape"], s)
        dy = np.random.RandomState(1).standard_normal((cfg["rois"], cfg["shape"][1], P, P)).astype(np.float32)
        out, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
        assert_fwd_matches(out, O.roi_align_forward(f, r, P, P, s, sr), fwd_path)
        ref_dx = O.roi_align_backward(dy, r, cfg["shape"], P, P, s, sr, acc64=True)
        np.testing.assert_allclose(dx, ref_dx, **GRAD_TOL)
        # <out, dy> == <dx, f>
        lhs = float(np.sum(out.astype(np.float64) * dy)); rhs = float(np.sum(dx.astype(np.float64) * f))
        assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))
        # cells no tap touches get exactly zero gradient
        assert np.count_nonzero(np.abs(dx).sum(axis=(0, 1))) <= O.roi_align_touched_cells(r, cfg["shape"][0], cfg["shape"][2],
                                                                                            cfg["shape"][3], P, P, s, sr)
        g = golden("roi_align_ref_%s.npz" % name)
        assert_fwd_matches(sampled(out, g, "out"), g["out"], fwd_path)
        # the reference kernel's own dX at full size (atomic order differs run to run: same tolerance as against the oracle)
        np.testing.assert_allclose(sampled(dx, g, "dx"), g["dx"], **GRAD_TOL)


def test_backward_tolerance_is_derived_from_the_reference_kernels_own_spread():
    """VERDICT r1 item 6: the 1e-5 (and, for the 1500-RoI pile-up case, 2e-5) gradient tolerances are not taken on faith.
    The reference's ROIAlignBackward accumulates with fp32 atomicAdd in an order the hardware picks, so (1) two runs of the
    reference kernel on the same inputs differ from each other, and (2) each run is off the fp64 oracle by the fp32
    accumulation error.  Both were measured on a B200 at BASELINE cfg2 (full size) and on the pile-up case over four runs
    of the reference kernel and are stored with a fixed, seeded sample of its first run's dX
    (tests/golden/make_golden_full_size.py).  Our gather backward (fixed order per launch) must be no further from the fp64
    oracle than the reference kernel is, and it is compared with the reference kernel's dX directly within both
    accumulation errors."""
    import json
    g = golden("roi_align_ref_spread.npz")
    report = {}
    for name, (shape, s, P, sr, r, seed) in cases.spread_cases().items():
        dy = np.random.RandomState(seed).standard_normal((r.shape[0], shape[1], P, P)).astype(np.float32)
        ref64 = O.roi_align_backward(dy, r, shape, P, P, s, sr, acc64=True)
        spread = float(g[name + "/run_to_run_max_abs"])
        ref_err = float(g[name + "/vs_fp64_max_abs"])
        ours = ops_backward(dy, r, shape, P, s, sr)
        ours2 = ops_backward(dy, r, shape, P, s, sr)
        our_err = float(np.max(np.abs(ours - ref64)))
        vs_ref = float(np.max(np.abs(sampled(ours, g, name + "/dx") - g[name + "/dx"])))
        scale = float(np.max(np.abs(ref64)))
        report[name] = dict(reference_run_to_run_max_abs=spread, reference_vs_fp64_max_abs=ref_err, ours_vs_fp64_max_abs=our_err,
                            ours_vs_reference_sample_max_abs=vs_ref, ours_run_to_run_max_abs=float(np.max(np.abs(ours - ours2))),
                            max_abs_gradient=scale)
        assert our_err <= 1.25 * ref_err + 1e-7, "our backward is further from the fp64 oracle than the reference kernel itself"
        assert vs_ref <= ref_err + our_err + 1e-7
        # the tolerance used across this file, |a - b| <= 1e-5 + 1e-5 |b| (2e-5 absolute in the pile-up test), must cover the
        # reference kernel's own error against the same oracle -- otherwise the reference would fail its own parity test
        np.testing.assert_allclose(ours, ref64, rtol=1e-5, atol=2e-5 if name == "pileup_1500" else 1e-5)
    print(json.dumps(report))


def ops_backward(dy, r, shape, P, s, sr):
    from detectron.pytorch_b200 import ops
    return ops.roi_align_backward(dev(dy), dev(r), shape, P, P, s, sr).cpu().numpy()


def test_roi_align_backward_rows_path_many_rows_unranked(lib_option):
    """N * H > 1024: the main kernel skips the heaviest-first row order (items are handed out in natural order)."""
    lib_option("B200_ROI_ALIGN_BWD_PATH", "rows")
    shape, s, P, sr = (6, 64, 180, 40), 1.0 / 8, 7, 2
    r = S.make_rois(300, shape, s, seed=9).astype(np.float32)
    dy = np.random.RandomState(4).standard_normal((r.shape[0], shape[1], P, P)).astype(np.float32)
    f = S.make_features(shape, seed=2)
    assert _lib.load().b200_roi_align_backward_workspace_bytes(shape[0], r.shape[0], shape[1], shape[2], shape[3], P, P, sr) > 0
    _, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    np.testing.assert_allclose(dx, O.roi_align_backward(dy, r, shape, P, P, s, sr, acc64=True), **GRAD_TOL)


ROWS_CASES = {
    # name: (shape, scale, P, sr, n_rois)  -- shapes the row-stationary backward covers (C % 64 == 0, P in {7, 14}, sr in {1, 2})
    "c64_odd_w": ((2, 64, 25, 45), 1.0 / 16, 7, 2, 40),
    "c128_sr1": ((1, 128, 30, 33), 1.0 / 8, 7, 1, 24),
    "c128_cpl4": ((3, 128, 20, 70), 1.0 / 16, 7, 2, 48),
    "p14_sr2": ((1, 64, 28, 40), 1.0 / 8, 14, 2, 16),
    "p14_sr1": ((2, 64, 16, 31), 1.0 / 16, 14, 1, 16),
    "w_lt_32": ((1, 64, 12, 9), 1.0 / 32, 7, 2, 12),
}


@pytest.mark.parametrize("name", sorted(ROWS_CASES))
@pytest.mark.parametrize("cpl", ["2", "4"])
def test_roi_align_backward_rows_path(name, cpl, lib_option):
    """Row-stationary gather backward vs the oracle (fp64 accumulation): edge RoIs (outside the map, degenerate,
    bad batch index), partial x-tiles, several images, both channel-per-lane variants."""
    lib_option("B200_ROI_ALIGN_BWD_PATH", "rows")
    lib_option("B200_ROI_ALIGN_BWD_CPL", cpl)
    shape, s, P, sr, n = ROWS_CASES[name]
    assert _lib.load().b200_roi_align_backward_workspace_bytes(shape[0], n, shape[1], shape[2], shape[3], P, P, sr) > 0
    r = np.concatenate([S.make_rois(n, shape, s, seed=2), S.make_edge_rois(shape, s)]).astype(np.float32)
    dy = np.random.RandomState(3).standard_normal((r.shape[0], shape[1], P, P)).astype(np.float32)
    f = S.make_features(shape, seed=1)
    out, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    ref_dx = O.roi_align_backward(dy, r, shape, P, P, s, sr, acc64=True)
    np.testing.assert_allclose(dx, ref_dx, **GRAD_TOL)
    assert np.array_equal(dx == 0, ref_dx == 0) or np.count_nonzero((dx == 0) != (ref_dx == 0)) < dx.size * 1e-4
    # run-to-run: no atomics in this path, but the unit order inside a row comes from a counting sort with atomics
    _, dx2 = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    np.testing.assert_allclose(dx2, dx, **GRAD_TOL)


def test_roi_align_backward_rows_path_row_overflow(lib_option):
    """400 tiny RoIs piled onto the same few rows of a tall map: the per-row unit lists (capacity = 8x the mean row
    population) run over and the shared overflow list is exercised."""
    lib_option("B200_ROI_ALIGN_BWD_PATH", "rows")
    shape, s, P, sr = (1, 64, 200, 40), 1.0 / 4, 7, 2
    rng = np.random.RandomState(5)
    n = 400
    x1 = rng.uniform(0, 120, n); y1 = rng.uniform(396, 404, n)
    r = np.stack([np.zeros(n), x1, y1, x1 + rng.uniform(2, 30, n), y1 + rng.uniform(0.5, 3, n)], axis=1).astype(np.float32)
    dy = rng.standard_normal((n, shape[1], P, P)).astype(np.float32)
    f = S.make_features(shape, seed=1)
    _, dx = run_fwd_bwd(RoIAlignFunction(P, P, s, sr), f, r, dy)
    # thousands of addends per cell: fp32 accumulation (ours, and the reference's atomicAdd alike) is only good to
    # ~n * eps * sum|terms| against the fp64 oracle, hence the wider tolerance of this stress case
    np.testing.assert_allclose(dx, O.roi_align_backward(dy, r, shape, P, P, s, sr, acc64=True), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("bwd", ["auto", "nhwc", "generic"])
def test_roi_align_fpn_equals_per_level_loop_cat_and_restore(bwd, lib_option):
    """SURVEY 8f N2: RoIAlignFPNFunction == the reference flow (per-level RoIAlign, torch.cat, gather by the restore
    index; model_builder.py:264-303), forward and backward, with an empty level, fast-path and generic-path levels."""
    from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align_fpn import RoIAlignFPNFunction
    if bwd != "auto":
        lib_option("B200_ROI_ALIGN_BWD_PATH", bwd)
    rng = np.random.RandomState(11)
    shapes = [(2, 64, 48, 64), (2, 64, 24, 32), (2, 64, 12, 16), (2, 64, 6, 8)]
    scales = [1.0 / 4, 1.0 / 8, 1.0 / 16, 1.0 / 32]
    counts = [150, 40, 0, 9]
    P, sr = 7, 2
    feats = [S.make_features(sh, seed=20 + i) for i, sh in enumerate(shapes)]
    rois = [S.make_rois(c, sh, sc, seed=30 + i).astype(np.float32) if c else np.zeros((0, 5), np.float32)
            for i, (c, sh, sc) in enumerate(zip(counts, shapes, scales))]
    total = sum(counts)
    restore = rng.permutation(total).astype(np.int32)
    dy = rng.standard_normal((total, 64, P, P)).astype(np.float32)

    F1 = [dev(f).requires_grad_(True) for f in feats]
    outs = [RoIAlignFunction(P, P, sc, sr)(f, dev(r)) for f, r, sc in zip(F1, rois, scales) if len(r)]
    ref = torch.cat(outs, dim=0)[torch.from_numpy(restore.astype(np.int64)).cuda()]
    ref.backward(dev(dy))

    F2 = [dev(f).requires_grad_(True) for f in feats]
    out = RoIAlignFPNFunction(P, P, scales, sr)(F2, [dev(r) for r in rois], restore)
    out.backward(dev(dy))

    torch.testing.assert_close(out, ref, rtol=1e-6, atol=1e-6)
    assert float((out == ref).float().mean()) > 0.9
    for a, b, c in zip(F2, F1, counts):
        if c:
            np.testing.assert_allclose(a.grad.cpu().numpy(), b.grad.cpu().numpy(), **GRAD_TOL)
        else:
            assert a.grad is not None and torch.count_nonzero(a.grad) == 0


def test_roi_align_fpn_single_launch_sequence_bit_exact():
    """SURVEY 8f N2, second step: the whole pyramid in ONE launch sequence (count + fill + one streaming kernel over the strip
    columns of every level) -- bit-identical to the per-level calls, 3 kernel launches instead of 3 per level."""
    from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align_fpn import RoIAlignFPNFunction
    rng = np.random.RandomState(12)
    shapes = [(2, 96, 200, 336), (2, 96, 100, 168), (2, 96, 50, 84), (2, 96, 25, 42)]
    scales = [1.0 / 4, 1.0 / 8, 1.0 / 16, 1.0 / 32]
    counts = [400, 350, 120, 6]
    for P in (7, 14):
        feats = [S.make_features(sh, seed=40 + i) for i, sh in enumerate(shapes)]
        rois = [S.make_rois(c, sh, sc, seed=50 + i, min_size=16 * 2 ** i, max_size=140 * 2 ** i).astype(np.float32)
                for i, (c, sh, sc) in enumerate(zip(counts, shapes, scales))]
        total = sum(counts)
        restore = rng.permutation(total).astype(np.int32)
        F = [dev(f) for f in feats]
        before = _lib.launch_count()
        out = RoIAlignFPNFunction(P, P, scales, 2)(F, [dev(r) for r in rois], restore)
        assert _lib.launch_count() - before == 4          # prep + main for P2..P4 (TMA-staged) and again for P5 (W = 42: cp.async producers)
        ref = np.concatenate([O.roi_align_forward(f, r, P, P, sc, 2) for f, r, sc in zip(feats, rois, scales)])[restore]
        got = out.cpu().numpy()
        np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-6)
        assert np.mean(got == ref) > 0.999


def test_roi_align_forward_linearity_and_determinism(fwd_path):
    cfg = S.CFG2
    P, s, sr = cfg["pooled"], cfg["scale"], cfg["sampling_ratio"]
    F1 = dev(S.make_features(cfg["shape"], seed=3)); F2 = dev(S.make_features(cfg["shape"], seed=4))
    R = dev(S.make_rois(cfg["rois"], cfg["shape"], s, seed=5))
    fn = RoIAlignFunction(P, P, s, sr)
    a, b, ab = fn(F1, R), fn(F2, R), fn(F1 + F2, R)
    torch.testing.assert_close(ab, a + b, rtol=1e-5, atol=1e-5)
    if fwd_path in ("generic", "stream", "quad"):                  # stream: at most two partial sums per element -> order-independent
        assert torch.equal(fn(F1, R), a)                   # run-to-run bit-identical
        assert torch.equal(fn(2 * F1, R), 2 * a)           # scaling by a power of two is exact
    else:                                                  # bins split over 4 tiles add 3 partials atomically
        torch.testing.assert_close(fn(F1, R), a, rtol=1e-6, atol=1e-6)
        assert (fn(F1, R) == a).float().mean() > 0.95


def test_roi_align_many_rois_multi_image_partial_channels(fwd_path):
    """> 512 RoIs hitting one tile (chunked RoI list), N = 3 with mixed batch indices, C not a multiple
    of 32, an out-of-range batch index (defined result: zeros), P = 14 mask-head geometry."""
    shape = (3, 40, 46, 70)
    f = S.make_features(shape, seed=5)
    r = S.make_rois(1500, shape, 0.125, seed=6, min_size=64, max_size=500)
    r[7, 0] = 5.0                       # batch index out of range
    for P, sr in ((7, 2), (14, 2), (3, 1), (6, 4), (5, 3)):
        dy = np.random.RandomState(P).standard_normal((1500, 40, P, P)).astype(np.float32)
        out, dx = run_fwd_bwd(RoIAlignFunction(P, P, 0.125, sr), f, r, dy)
        rr = r.copy(); rr[7, 0] = 0
        ref = O.roi_align_forward(f, rr, P, P, 0.125, sr)
        ref[7] = 0
        assert_fwd_matches(out, ref, fwd_path)
        dyr = dy.copy(); dyr[7] = 0          # the RoI with the bad batch index contributes nothing
        np.testing.assert_allclose(dx, O.roi_align_backward(dyr, rr, shape, P, P, 0.125, sr, acc64=True), rtol=1e-5, atol=2e-5)
    # C = 6 (not a multiple of 4): the vector path must fall back to scalar reductions per channel
    shape6 = (2, 6, 30, 34)
    f6 = S.make_features(shape6, seed=8); r6 = S.make_rois(64, shape6, 0.25, seed=9)
    dy6 = np.random.RandomState(3).standard_normal((64, 6, 7, 7)).astype(np.float32)
    out6, dx6 = run_fwd_bwd(RoIAlignFunction(7, 7, 0.25, 2), f6, r6, dy6)
    assert_fwd_matches(out6, O.roi_align_forward(f6, r6, 7, 7, 0.25, 2), fwd_path)
    np.testing.assert_allclose(dx6, O.roi_align_backward(dy6, r6, shape6, 7, 7, 0.25, 2, acc64=True), **GRAD_TOL)


STREAM_CASES = {
    # name: (shape, scale, P, sr, n_rois, min_size, max_size) -- shapes the streaming-strip forward covers (sr in {1, 2})
    "c40_n2": ((2, 40, 60, 100), 1.0 / 8, 7, 2, 200, 32, 512),       # C not a multiple of 32, two strips, two images
    "p14": ((1, 64, 50, 84), 1.0 / 16, 14, 2, 60, 64, 600),           # mask-head geometry, one strip
    "sr1": ((3, 32, 40, 68), 1.0 / 16, 7, 1, 80, 32, 512),
    "wide": ((1, 32, 50, 336), 1.0 / 4, 7, 2, 150, 16, 1300),         # six strips; whole-width boxes -> x-split bins
    "tall": ((1, 32, 400, 64), 1.0 / 4, 7, 2, 100, 16, 1590),         # whole-height boxes -> y-split bins (span > ring depth)
    "c256": ((1, 256, 64, 96), 1.0 / 8, 7, 2, 128, 32, 512),          # 8 channel groups
    "odd_w": ((2, 48, 25, 42), 1.0 / 32, 7, 2, 60, 64, 900),          # FPN P5: W = 42 (168-byte pitch), partial channel group
    "narrow": ((1, 32, 30, 9), 1.0 / 32, 7, 2, 12, 32, 300),          # W < 32: one partial chunk
}


STRIP_LAUNCHES = {"stream": 3, "quad": 2}       # count + fill + main / prep + main (memsets are not counted)


@pytest.mark.parametrize("path", ["stream", "quad"])
@pytest.mark.parametrize("name", sorted(STREAM_CASES))
def test_roi_align_stream_path(name, path, lib_option):
    """Streaming-strip forward (cp.async + mbarrier ring) vs the oracle: every bin whose samples fit the strip halo / the ring is computed by one
    lane in the reference's order -> bit-exact; bins cut into two partial sums (huge boxes) agree to 1e-6.  The launch
    counter proves the streaming kernels ran (count + fill + main, or prep + main for the quad-strip generation) and not a fallback."""
    lib_option("B200_ROI_ALIGN_PATH", path)
    shape, s, P, sr, n, lo, hi = STREAM_CASES[name]
    f = S.make_features(shape, seed=3)
    r = np.concatenate([S.make_rois(n, shape, s, seed=4, min_size=lo, max_size=hi), S.make_edge_rois(shape, s)]).astype(np.float32)
    r[5, 0] = shape[0] + 2                      # batch index out of range: defined result, zeros
    rr = r.copy(); rr[5, 0] = 0
    ref = O.roi_align_forward(f, rr, P, P, s, sr); ref[5] = 0
    before = _lib.launch_count()
    out = RoIAlignFunction(P, P, s, sr)(dev(f), dev(r)).cpu().numpy()
    assert _lib.launch_count() - before == STRIP_LAUNCHES[path]
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
    per_roi_exact = (out == ref).reshape(out.shape[0], -1).all(axis=1)
    # the quad-strip generation keeps 8 halo columns (9 in the first one): in the "wide" case (boxes up to 325 cells) more bins are cut in two
    assert per_roi_exact[:n].mean() > (0.9 if (path, name) != ("quad", "wide") else 0.6), "bins of ordinary RoIs must be bit-exact"
    out2 = RoIAlignFunction(P, P, s, sr)(dev(f), dev(r)).cpu().numpy()
    assert np.array_equal(out, out2)              # deterministic, split bins included


@pytest.mark.parametrize("path", ["stream", "quad"])
def test_roi_align_stream_cfg2_bit_exact(path, lib_option):
    """BASELINE cfg2 through the streaming path: no bin needs a split at this geometry except a handful -> the result is
    bit-identical to the reference kernel's (and to the oracle) on > 99.9 % of the elements, 1e-6 on the rest."""
    lib_option("B200_ROI_ALIGN_PATH", path)
    cfg = S.CFG2
    P, s, sr = cfg["pooled"], cfg["scale"], cfg["sampling_ratio"]
    f = S.make_features(cfg["shape"]); r = S.make_rois(cfg["rois"], cfg["shape"], s)
    before = _lib.launch_count()
    out = RoIAlignFunction(P, P, s, sr)(dev(f), dev(r)).cpu().numpy()
    assert _lib.launch_count() - before == STRIP_LAUNCHES[path]
    ref = O.roi_align_forward(f, r, P, P, s, sr)
    np.testing.assert_allclose(out, ref, rtol=1e-6, atol=1e-6)
    assert np.mean(out == ref) > 0.999
    g = golden("roi_align_ref_cfg2.npz")                  # a fixed, seeded sample of the reference kernel's output
    assert np.mean(sampled(out, g, "out") == g["out"]) > 0.999


def test_roi_align_empty_and_degenerate():
    F = dev(S.make_features((1, 4, 10, 12)))
    fn = RoIAlignFunction(7, 7, 0.25, 2)
    out = fn(F, torch.zeros((0, 5), device="cuda"))
    assert tuple(out.shape) == (0, 4, 7, 7)
    Fg = F.clone().requires_grad_(True)
    o = fn(Fg, torch.zeros((0, 5), device="cuda"))
    o.sum().backward()
    assert torch.count_nonzero(Fg.grad) == 0              # dX fully defined (zeros) with no RoIs
    with pytest.raises(NotImplementedError):
        fn(F.cpu(), torch.zeros((1, 5)))


def test_roi_align_avg_max_modules():
    c, f, r, _ = cases.roi_case("cfg1_small")
    base = O.roi_align_forward(f, r, 8, 8, c["scale"], 2)
    avg = RoIAlignAvg(7, 7, c["scale"], 2)(dev(f), dev(r)).cpu()
    mx = RoIAlignMax(7, 7, c["scale"], 2)(dev(f), dev(r)).cpu()
    tb = torch.from_numpy(base)
    assert torch.equal(mx, torch.nn.functional.max_pool2d(tb, 2, 1))
    torch.testing.assert_close(avg, torch.nn.functional.avg_pool2d(tb, 2, 1), rtol=1e-6, atol=1e-6)


# ---------------------------------------------------------------------------- legacy RoIAlign, RoIPool
@pytest.mark.parametrize("name", sorted(cases.ROI_CASES))
def test_legacy_and_pool_vs_oracle_and_reference(name):
    c, f, r, dy = cases.roi_case(name)
    P, s = c["P"], c["scale"]
    out, dx = run_fwd_bwd(LegacyRoIAlignFunction(P, P, s), f, r, dy)
    assert np.array_equal(out, O.roi_align_legacy_forward(f, r, P, P, s))
    np.testing.assert_allclose(dx, O.roi_align_legacy_backward(dy, r, c["shape"], P, P, s, acc64=True), **GRAD_TOL)
    fn = RoIPoolFunction(P, P, s)
    pout, pdx = run_fwd_bwd(fn, f, r, dy)
    o_out, o_arg = O.roi_pool_forward(f, r, P, P, s)
    assert np.array_equal(pout, o_out) and np.array_equal(fn.argmax.cpu().numpy(), o_arg)
    assert np.array_equal(pdx, O.roi_pool_backward(dy, o_arg, r, c["shape"], P, P, s))
    g = golden("legacy_pool_%s.npz" % name)               # the reference kernels' outputs (tests/golden/make_golden.py)
    assert np.array_equal(out, g["legacy_out"]) and np.array_equal(pout, g["pool_out"])
    np.testing.assert_allclose(dx, g["legacy_dx"], **GRAD_TOL)
    assert np.array_equal(o_arg, g["pool_argmax"])
    assert np.array_equal(pdx, g["pool_dx"])


def test_pool_many_rois_chunked_list():
    """> 512 overlapping RoIs on one tile exercises the chunked RoI list of the backward."""
    shape = (1, 3, 20, 24)
    f = S.make_features(shape)
    r = S.make_rois(1400, shape, 0.25, seed=2, min_size=40, max_size=96)
    fn = RoIPoolFunction(3, 3, 0.25)
    dy = np.random.RandomState(1).standard_normal((1400, 3, 3, 3)).astype(np.float32)
    pout, pdx = run_fwd_bwd(fn, f, r, dy)
    o_out, o_arg = O.roi_pool_forward(f, r, 3, 3, 0.25)
    assert np.array_equal(pout, o_out)
    assert np.array_equal(pdx, O.roi_pool_backward(dy, o_arg, r, shape, 3, 3, 0.25))


# ---------------------------------------------------------------------------------------- RoICrop
def test_roi_crop_vs_oracle_reference_golden():
    img, grid, go = cases.crop_case()
    I = dev(img).requires_grad_(True); Gd = dev(grid).requires_grad_(True)
    out = RoICropFunction()(I, Gd)
    out.backward(dev(go))
    o = out.detach().cpu().numpy(); gi = I.grad.cpu().numpy()
    assert np.array_equal(o, O.roi_crop_forward(img, grid))
    np.testing.assert_allclose(gi, O.roi_crop_backward(go, grid, img.shape, acc64=True), **GRAD_TOL)
    assert torch.count_nonzero(Gd.grad) == 0
    g = golden("roi_crop.npz")                            # the reference kernels' outputs (tests/golden/make_golden.py)
    assert np.array_equal(o, g["out"])
    np.testing.assert_allclose(gi, g["grad_img"], **GRAD_TOL)
    assert np.count_nonzero(g["grad_grid"]) == 0


@pytest.mark.parametrize("shape,R", [((2, 32, 20, 24), 40), ((4, 256, 13, 17), 64), ((1, 48, 16, 16), 24)])
def test_roi_crop_backward_vector_reduction_path(shape, R, lib_option):
    """RoICrop image gradient through the channel-innermost scratch image (red.global.add.v4.f32, roi_crop.cu): against the fp64
    oracle and against the scalar-atomic kernel (B200_ROI_ALIGN_BWD_PATH=generic), samples partly outside the image included."""
    from detectron.pytorch_b200 import ops
    img = S.make_features(shape, seed=7)
    grid = S.make_crop_grid(R, 7, 7, seed=8).astype(np.float32)
    grid[0, 0, 0] = (-1.0, -1.0); grid[1, 3, 3] = (-1.5, 0.2); grid[2, 6, 6] = (1.0, 1.0)
    go = np.random.RandomState(9).standard_normal((R, shape[1], 7, 7)).astype(np.float32)
    before = _lib.launch_count()
    gi, gg = ops.roi_crop_backward(dev(go), dev(grid), shape)
    assert _lib.launch_count() - before == 2                     # scatter + transpose (the scalar path counts 1)
    ref = O.roi_crop_backward(go, grid, shape, acc64=True)
    np.testing.assert_allclose(gi.cpu().numpy(), ref, **GRAD_TOL)
    assert torch.count_nonzero(gg) == 0
    lib_option("B200_ROI_ALIGN_BWD_PATH", "generic")
    before = _lib.launch_count()
    gi2, _ = ops.roi_crop_backward(dev(go), dev(grid), shape)
    assert _lib.launch_count() - before == 1
    np.testing.assert_allclose(gi.cpu().numpy(), gi2.cpu().numpy(), **GRAD_TOL)


# -------------------------------------------------------------------------------------------- NMS
@pytest.mark.parametrize("n", cases.NMS_SIZES)
def test_nms_bit_exact(n):
    b = cases.nms_case(n)
    keep = nms_gpu(dev(b), 0.7)
    assert keep.dtype == torch.int32 and keep.dim() == 2 and keep.size(1) == 1 and keep.is_cuda
    k = keep.cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, 0.7))
    assert np.array_equal(k, golden("nms.npz")["keep_%d" % n])      # the reference kernel's keep list (tests/golden/make_golden.py)


@pytest.mark.parametrize("thresh", [0.3, 0.5, 0.9])
def test_nms_thresholds_and_properties(thresh):
    b = cases.nms_case(3000, seed=7)
    k = nms_gpu(dev(b), thresh).cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, thresh))
    assert k[0] == 0 and np.all(np.diff(k) > 0)            # sorted, best box always kept
    k2 = nms_gpu(dev(b[k]), thresh).cpu().numpy().reshape(-1)
    assert np.array_equal(k2, np.arange(len(k)))            # idempotent


@pytest.mark.parametrize("n", [8000, 12000, 15000])
def test_nms_large_inputs(n):
    # 8000: near-diagonal reach 3; 12000: reach 2; 15000: words do not fit shared memory -> unpipelined scan
    b = cases.nms_case(n, seed=3)
    k = nms_gpu(dev(b), 0.7).cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, 0.7))


def test_nms_simple_scan_matches(lib_option):
    lib_option("B200_NMS_SCAN", "simple")
    b = cases.nms_case(3000, seed=11)
    k = nms_gpu(dev(b), 0.7).cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, 0.7))


@pytest.mark.parametrize("n", [63, 64, 65, 1000, 4097])
def test_nms_suppression_chain(n):
    b = cases.nms_chain_case(n)             # every decision depends on the previous one: 64 resolve rounds per block
    k = nms_gpu(dev(b), 0.7).cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, 0.7))
    assert np.array_equal(k, np.arange(0, n, 2))


@pytest.mark.parametrize("n,thresh", [(3000, 0.7), (6000, 0.5), (777, 0.3)])
def test_nms_clustered_order(n, thresh):
    b = cases.nms_clustered_case(n, seed=n)
    k = nms_gpu(dev(b), thresh).cpu().numpy().reshape(-1)
    assert np.array_equal(k, O.nms_cuda(b, thresh))


def test_nms_edge_cases():
    assert nms_wrapper(torch.zeros((0, 5), device="cuda"), 0.7) == []
    one = dev(np.array([[0, 0, 10, 10, 0.5]], np.float32))
    assert nms_gpu(one, 0.7).cpu().numpy().tolist() == [[0]]
    dup = dev(np.tile(np.array([[5, 5, 50, 60, 0.9]], np.float32), (130, 1)))
    assert nms_gpu(dup, 0.7).cpu().numpy().tolist() == [[0]]          # all duplicates collapse
    # degenerate boxes: zero-area union -> 0/0 = NaN -> never suppressed (reference semantics)
    deg = np.array([[10, 10, 9, 9, 0.9], [10, 10, 9, 9, 0.8], [0, 0, 5, 5, 0.7]], np.float32)
    assert np.array_equal(nms_gpu(dev(deg), 0.7).cpu().numpy().reshape(-1), O.nms_cuda(deg, 0.7))
    # extra columns are ignored, like boxes_dim in the reference
    b6 = np.concatenate([cases.nms_case(500), np.ones((500, 1), np.float32)], axis=1)
    assert np.array_equal(nms_gpu(dev(b6), 0.7).cpu().numpy().reshape(-1), O.nms_cuda(b6[:, :5], 0.7))


def test_nms_batched_equals_per_problem_calls():
    """b200_nms_batched: the (image, level) proposal sets of one step in one pair of launches -- per problem bit-identical
    to b200_nms / the oracle: sizes across the scan's REACH classes, an empty problem, a one-box problem, a dense chain."""
    from detectron.pytorch_b200 import ops
    probs = [cases.nms_case(1000, seed=1), cases.nms_case(2000, seed=2), np.zeros((0, 5), np.float32), cases.nms_chain_case(130),
             cases.nms_case(1, seed=3), cases.nms_clustered_case(777, seed=5), cases.nms_case(6000, seed=4), cases.nms_case(65, seed=6)]
    counts = [len(b) for b in probs]
    keep, num = ops.nms_batched_raw(dev(np.concatenate(probs)), counts, 0.7)
    keep = keep.cpu().numpy(); num = num.cpu().numpy()
    off = 0
    for b, c, k in zip(probs, counts, num):
        ref = O.nms_cuda(b, 0.7) if c else np.zeros((0,), np.int64)
        assert k == len(ref)
        assert np.array_equal(keep[off:off + k], ref)
        off += c
    # ten FPN-like problems (5 levels x 2 images): same answers as ten separate calls
    ten = [cases.nms_case(n, seed=20 + i) for i, n in enumerate([1000, 1000, 1000, 1000, 1000, 1000, 1000, 1000, 525, 525])]
    keep, num = ops.nms_batched_raw(dev(np.concatenate(ten)), [len(b) for b in ten], 0.7)
    keep = keep.cpu().numpy(); num = num.cpu().numpy(); off = 0
    for b, k in zip(ten, num):
        single = nms_gpu(dev(b), 0.7).cpu().numpy().reshape(-1)
        assert np.array_equal(keep[off:off + k], single)
        off += len(b)
    with pytest.raises(ValueError):
        ops.nms_batched_raw(dev(probs[0]), [10, 20], 0.7)


def test_generate_proposals_batched_levels_equal_per_level_calls():
    """generate_proposals_batched (all FPN levels x images through ONE batched NMS and one host read) returns exactly what
    the per-level op calls return, and those equal the numpy restatement of the reference op."""
    from detectron.pytorch_b200.modeling.generate_proposals import GenerateProposalsOp, generate_proposals_batched
    from oracle import proposals as OP
    rng = np.random.RandomState(3)
    N, A = 2, 3
    ops_l, probs_l, preds_l, refs = [], [], [], []
    im_info = np.array([[320, 480, 1.5], [300, 400, 1.25]], dtype=np.float32)
    for lvl, (H, W) in zip((2, 3, 4), ((80, 120), (40, 60), (20, 30))):
        stride = 2 ** lvl
        anchors = np.round((rng.uniform(-1, 1, (A, 4)) * 4 * stride + np.array([-3, -3, 3, 3]) * stride) * 2) / 2
        scores = ((rng.permutation(N * A * H * W).astype(np.float32) + 0.5) / (N * A * H * W)).reshape(N, A, H, W)
        deltas = (rng.standard_normal((N, 4 * A, H, W)) * 0.4).astype(np.float32)
        mode = dict(RPN_PRE_NMS_TOP_N=600, RPN_POST_NMS_TOP_N=200, RPN_NMS_THRESH=0.7, RPN_MIN_SIZE=0)
        ops_l.append(GenerateProposalsOp(anchors, 1.0 / stride, train=mode, test=mode))
        probs_l.append(dev(scores)); preds_l.append(dev(deltas))
        refs.append(OP.generate_proposals(scores, deltas, im_info, anchors, float(stride), 600, 200, 0.7, 0))
    fused = generate_proposals_batched(ops_l, probs_l, preds_l, torch.from_numpy(im_info))
    for (rois, probs), op, p, d, (rr, pp) in zip(fused, ops_l, probs_l, preds_l, refs):
        r1, p1 = op(p, d, torch.from_numpy(im_info))
        assert np.array_equal(rois, r1) and np.array_equal(probs, p1)
        assert rois.shape == rr.shape
        np.testing.assert_allclose(rois, rr, rtol=0, atol=1e-3)
        assert np.array_equal(probs, pp)
    with pytest.raises(ValueError):                       # the op is bound to its anchor count (ADVICE r1)
        ops_l[0](probs_l[0][:, :2], preds_l[0], torch.from_numpy(im_info))


def test_reference_named_launchers_compute():
    """The compatibility libraries (include/b200_ref_launchers.h): the reference's launcher names and argument lists, called
    the way the reference's *_cuda.c glue calls them (raw device pointers, current stream), against the oracle."""
    import ctypes
    from detectron.pytorch_b200 import build as B
    lib = ctypes.CDLL(B.compat_lib_path("libb200_ref_launchers.so"))
    leg = ctypes.CDLL(B.compat_lib_path("libb200_ref_launchers_legacy.so"))
    c, f, r, dy = cases.roi_case("cfg1_small")
    P, s, sr = c["P"], c["scale"], c["sr"]
    N, C, H, W = c["shape"]
    R = r.shape[0]
    F, Rt, DY = dev(f), dev(r), dev(dy)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    out = torch.empty((R, C, P, P), device="cuda")
    assert lib.ROIAlignForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, P, P, sr, vp(Rt), vp(out), st) == 1
    assert np.array_equal(out.cpu().numpy(), O.roi_align_forward(f, r, P, P, s, sr))
    dx = torch.empty(c["shape"], device="cuda")
    assert lib.ROIAlignBackwardLaucher(vp(DY), ctypes.c_float(s), N, R, H, W, C, P, P, sr, vp(Rt), vp(dx), st) == 1
    np.testing.assert_allclose(dx.cpu().numpy(), O.roi_align_backward(dy, r, c["shape"], P, P, s, sr, acc64=True), **GRAD_TOL)
    lout = torch.empty((R, C, P, P), device="cuda")
    assert leg.ROIAlignForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, P, P, vp(Rt), vp(lout), st) == 1
    assert np.array_equal(lout.cpu().numpy(), O.roi_align_legacy_forward(f, r, P, P, s))
    pout = torch.empty((R, C, P, P), device="cuda"); arg = torch.empty((R, C, P, P), dtype=torch.int32, device="cuda")
    assert lib.ROIPoolForwardLaucher(vp(F), ctypes.c_float(s), R, H, W, C, P, P, vp(Rt), vp(pout), vp(arg), st) == 1
    o_out, o_arg = O.roi_pool_forward(f, r, P, P, s)
    assert np.array_equal(pout.cpu().numpy(), o_out) and np.array_equal(arg.cpu().numpy(), o_arg)
    pdx = torch.empty(c["shape"], device="cuda")
    assert lib.ROIPoolBackwardLaucher(vp(DY), ctypes.c_float(s), N, R, H, W, C, P, P, vp(Rt), vp(pdx), vp(arg), st) == 1
    assert np.array_equal(pdx.cpu().numpy(), O.roi_pool_backward(dy, o_arg, r, c["shape"], P, P, s))
    img, grid, go = cases.crop_case()
    IM, GR = dev(img), dev(grid)
    B_, Cc, ih, iw = img.shape
    ob, oh, ow = grid.shape[0], grid.shape[1], grid.shape[2]
    cout = torch.empty((ob, Cc, oh, ow), device="cuda")
    assert lib.BilinearSamplerBHWD_updateOutput_cuda_kernel(Cc, ow, oh, ob, Cc, ih, iw, B_, vp(IM), Cc * ih * iw, ih * iw, iw, 1,
                                                            vp(GR), oh * ow * 2, 1, ow * 2, 2, vp(cout), Cc * oh * ow, oh * ow, ow, 1, st) == 1
    assert np.array_equal(cout.cpu().numpy(), O.roi_crop_forward(img, grid))
    b = cases.nms_case(1000)
    Bx = dev(b)
    keep = torch.empty((1000,), dtype=torch.int32, device="cuda"); num = torch.zeros((1,), dtype=torch.int32, device="cuda")
    lib.nms_cuda_compute.restype = None
    torch.cuda.synchronize()                                  # the launcher runs on the legacy default stream, like the reference
    lib.nms_cuda_compute(vp(keep), vp(num), vp(Bx), 1000, 5, ctypes.c_float(0.7))
    torch.cuda.synchronize()
    k = int(num.item())
    assert np.array_equal(keep[:k].cpu().numpy(), O.nms_cuda(b, 0.7))


def test_ops_honour_current_stream_and_noncontiguous_input():
    c, f, r, _ = cases.roi_case("cfg1_small")
    F = dev(np.transpose(f, (0, 1, 3, 2))).transpose(2, 3)   # non-contiguous view of the same values
    assert not F.is_contiguous()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        out = RoIAlignFunction(7, 7, c["scale"], 2)(F, dev(r))
    s.synchronize()
    assert np.array_equal(out.cpu().numpy(), O.roi_align_forward(f, r, 7, 7, c["scale"], 2))


# ------------------------------------------------------------------------------ proposal layer (SURVEY 8f N1)
def _golden_proposals():
    g = np.load(os.path.join(GOLDEN, "proposals.npz"))
    return g, sorted({k.split("/")[0] for k in g.files if k.endswith("/params")})


@pytest.mark.parametrize("name", ["all_candidates", "c4_test", "fpn_p5_train", "min_size"])
def test_generate_proposals_matches_the_reference_op(name):
    """Device proposal layer vs the output of the reference's own GenerateProposalsOp (golden vectors generated on CPU
    by tests/golden/make_golden_proposals.py from the unmodified reference code)."""
    from detectron.pytorch_b200.modeling.generate_proposals import GenerateProposalsOp
    G, _ = _golden_proposals()
    g = {k.split("/", 1)[1]: G[k] for k in G.files if k.startswith(name + "/")}
    stride, pre, post, thresh, min_size = g["params"]
    mode = dict(RPN_PRE_NMS_TOP_N=int(pre), RPN_POST_NMS_TOP_N=int(post), RPN_NMS_THRESH=float(thresh), RPN_MIN_SIZE=float(min_size))
    op = GenerateProposalsOp(g["anchors"], 1.0 / float(stride), train=mode, test=mode)
    rois, probs = op(dev(g["scores"]), dev(g["deltas"]), torch.from_numpy(g["im_info"]))
    assert rois.shape == g["rois"].shape and probs.shape == g["probs"].shape
    assert np.array_equal(probs, g["probs"])                       # same candidates survive, in the same order
    assert np.array_equal(rois[:, 0], g["rois"][:, 0])
    np.testing.assert_allclose(rois, g["rois"], rtol=0, atol=1e-4)
    assert np.mean(rois == g["rois"]) > 0.999                      # double-precision exp: CUDA vs numpy agree to the last float32 bit almost everywhere


def test_generate_proposals_realistic_level_vs_oracle():
    """FPN P2-sized level (3 x 200 x 336 = 201 600 anchors, top 2000 -> NMS 0.7 -> 1000) against oracle/proposals.py."""
    from detectron.pytorch_b200.modeling.generate_proposals import GenerateProposalsOp
    from oracle import proposals as OP
    rng = np.random.RandomState(3)
    N, A, H, W, stride = 2, 3, 200, 336, 4
    anchors = np.array([[-22., -10., 25., 13.], [-14., -14., 17., 17.], [-10., -22., 13., 25.]])     # 32 px, ratios 0.5 / 1 / 2
    scores = ((rng.permutation(N * A * H * W).astype(np.float32) + 0.5) / (N * A * H * W)).reshape(N, A, H, W)
    deltas = (rng.standard_normal((N, 4 * A, H, W)) * 0.5).astype(np.float32)
    im_info = np.array([[800, 1333, 1.5], [800, 1216, 1.3]], dtype=np.float32)
    mode = dict(RPN_PRE_NMS_TOP_N=2000, RPN_POST_NMS_TOP_N=1000, RPN_NMS_THRESH=0.7, RPN_MIN_SIZE=0)
    op = GenerateProposalsOp(anchors, 1.0 / stride, train=mode, test=mode)
    rois, probs = op(dev(scores), dev(deltas), torch.from_numpy(im_info))
    ref_rois, ref_probs = OP.generate_proposals(scores, deltas, im_info, anchors, float(stride), 2000, 1000, 0.7, 0)
    assert rois.shape == ref_rois.shape
    assert np.array_equal(probs, ref_probs)
    np.testing.assert_allclose(rois, ref_rois, rtol=0, atol=1e-4)


def test_rpn_heads_to_box_head_chain_on_device():
    """SURVEY 8f N1 + N2 end to end: per-level device proposals -> collect -> distribute -> RoIAlignFPNFunction, all on
    CUDA tensors, against the oracle chain (oracle/proposals.py -> oracle/fpn.py -> per-level RoIAlign oracle + restore)."""
    from detectron.pytorch_b200.modeling.collect_and_distribute_fpn_rpn_proposals import collect, distribute
    from detectron.pytorch_b200.modeling.generate_proposals import GenerateProposalsOp
    from detectron.pytorch_b200.modeling.roi_xfrom.roi_align.functions.roi_align_fpn import RoIAlignFPNFunction
    from oracle import fpn as OF
    from oracle import proposals as OP
    rng = np.random.RandomState(21)
    N, A, C, P, sr = 2, 3, 64, 7, 2
    sizes = {2: (48, 64), 3: (24, 32), 4: (12, 16), 5: (6, 8)}
    im_info = np.array([[192, 256, 1.0], [180, 240, 1.2]], dtype=np.float32)
    mode = dict(RPN_PRE_NMS_TOP_N=300, RPN_POST_NMS_TOP_N=100, RPN_NMS_THRESH=0.7, RPN_MIN_SIZE=0)
    lvl_rois, lvl_probs, ref_rois, ref_probs, feats = [], [], [], [], {}
    for lvl, (H, W) in sizes.items():
        stride = 2 ** lvl
        base = 8.0 * stride
        anchors = np.array([[-base * .7 + .5, -base * .35 + .5, base * .7 - .5, base * .35 - .5], [-base / 2 + .5, -base / 2 + .5, base / 2 - .5, base / 2 - .5],
                            [-base * .35 + .5, -base * .7 + .5, base * .35 - .5, base * .7 - .5]])
        scores = ((rng.permutation(N * A * H * W).astype(np.float32) + 0.5) / (N * A * H * W)).reshape(N, A, H, W)
        deltas = (rng.standard_normal((N, 4 * A, H, W)) * 0.3).astype(np.float32)
        op = GenerateProposalsOp(anchors, 1.0 / stride, train=mode, test=mode, return_tensors=True)
        r, p = op(dev(scores), dev(deltas), torch.from_numpy(im_info))
        lvl_rois.append(r); lvl_probs.append(p)
        rr, pp = OP.generate_proposals(scores, deltas, im_info, anchors, float(stride), 300, 100, 0.7, 0)
        ref_rois.append(rr); ref_probs.append(pp)
        feats[lvl] = S.make_features((N, C, H, W), seed=lvl)
    top = 250
    rois = collect(lvl_rois, lvl_probs, top)
    blobs = distribute(rois, 2, 5)
    r_ref = OF.collect(ref_rois, ref_probs, top)
    b_ref = OF.distribute(r_ref, 2, 5)
    assert np.array_equal(blobs["rois_idx_restore_int32"].cpu().numpy(), b_ref["rois_idx_restore_int32"])
    np.testing.assert_allclose(rois.cpu().numpy(), r_ref, rtol=0, atol=1e-4)
    levels = [2, 3, 4, 5]
    scales = [1.0 / 2 ** l for l in levels]
    out = RoIAlignFPNFunction(P, P, scales, sr)([dev(feats[l]) for l in levels], [blobs["rois_fpn%d" % l].contiguous() for l in levels],
                                                blobs["rois_idx_restore_int32"])
    ref_parts = [O.roi_align_forward(feats[l], b_ref["rois_fpn%d" % l], P, P, sc, sr) for l, sc in zip(levels, scales) if len(b_ref["rois_fpn%d" % l])]
    ref_out = np.concatenate(ref_parts, axis=0)[b_ref["rois_idx_restore_int32"]]
    assert out.shape == ref_out.shape
    np.testing.assert_allclose(out.cpu().numpy(), ref_out, rtol=1e-4, atol=1e-4)       # RoI coordinates agree to 1e-4 px
