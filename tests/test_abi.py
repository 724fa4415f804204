"""CPU-only: the C-ABI library builds for sm_100a, loads, exports every symbol include/*.h declares,
and validates its arguments before touching CUDA (no compute calls here: there is no GPU)."""
import ctypes
import os
import re

import pytest

from detectron.pytorch_b200 import _lib, build
from tests import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200_roi_ops.h")).read()
    return sorted(set(re.findall(r"B200_API[^;(]*?\b(b200_\w+)\s*\(", text)))


def test_library_builds_and_exports_header_symbols():
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    declared = _declared_symbols()
    assert len(declared) >= 13
    for name in declared:
        assert hasattr(lib, name), "header declares %s but the library does not export it" % name
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared       # python binding covers exactly the header


def test_reference_named_launchers_are_exported():
    """SURVEY 8b: the reference's own launcher names with the reference's argument lists (include/b200_ref_launchers.h),
    so that lib/.../src/*_cuda.c links unchanged.  Two libraries because the two RoIAlign flavours share their names."""
    build.build()
    text = open(os.path.join(ROOT, "include", "b200_ref_launchers.h")).read()
    body = text[text.index("#ifndef B200_REF_LEGACY_ROI_ALIGN"):]
    main_part, legacy_part = body[:body.rindex("#else")], body[body.rindex("#else"):]
    names = lambda t: sorted(set(re.findall(r"B200_REF_API\s+\w+\s+(\w+)\s*\(", t)))
    lib = ctypes.CDLL(build.compat_lib_path("libb200_ref_launchers.so"))
    assert names(main_part) == ["BilinearSamplerBHWD_updateGradInput_cuda_kernel", "BilinearSamplerBHWD_updateOutput_cuda_kernel",
                                "ROIAlignBackwardLaucher", "ROIAlignForwardLaucher", "ROIPoolBackwardLaucher", "ROIPoolForwardLaucher",
                                "nms_cuda_compute"]
    for n in names(main_part):
        assert hasattr(lib, n), n
    leg = ctypes.CDLL(build.compat_lib_path("libb200_ref_launchers_legacy.so"))
    assert names(legacy_part) == ["ROIAlignBackwardLaucher", "ROIAlignForwardLaucher"]
    for n in names(legacy_part):
        assert hasattr(leg, n), n
    # argument errors come back as 0 (the reference's glue treats 0 as failure), before any CUDA call
    lib.ROIAlignForwardLaucher.restype = ctypes.c_int
    assert lib.ROIAlignForwardLaucher(None, ctypes.c_float(0.25), 4, 0, 10, 3, 7, 7, 2, None, None, None) == 0
    # non-dense strides are refused by the RoICrop launchers
    assert lib.BilinearSamplerBHWD_updateOutput_cuda_kernel(3, 7, 7, 2, 3, 10, 10, 1, None, 300, 100, 10, 2, None, 98, 1, 14, 2,
                                                            None, 147, 49, 7, 1, None) == 0


def test_sm100a_cubin_embedded():
    import subprocess
    path = build.build()
    out = subprocess.run(["cuobjdump", "-lelf", path], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True).stdout
    assert "sm_100a" in out


def test_argument_validation_without_gpu():
    lib = _lib.load()
    assert lib.b200_roi_ops_abi_version() == 3
    EINVAL = -1
    # negative / zero dimensions and null pointers are rejected before any CUDA call
    assert lib.b200_roi_align_forward(None, 0.25, 1, 4, 0, 10, 3, 7, 7, 2, None, None, None) == EINVAL
    assert lib.b200_roi_align_forward(None, 0.25, 1, 4, 10, 10, 3, 7, 7, 2, None, None, None) == EINVAL
    assert lib.b200_roi_align_backward(None, 0.25, 1, 4, 10, 10, 3, 7, 7, 2, None, None, None) == EINVAL
    assert lib.b200_roi_pool_forward(None, 0.25, 1, 4, 10, 10, 3, -7, 7, None, None, None, None) == EINVAL
    assert lib.b200_roi_crop_forward(None, None, 1, 3, 10, 10, 2, 7, 7, None, None) == EINVAL
    assert lib.b200_nms(None, 10, 5, 0.7, None, None, None, 0, None) == EINVAL
    assert b"invalid argument" in lib.b200_roi_ops_strerror(EINVAL)
    assert lib.b200_roi_ops_strerror(0) == b"success"
    # workspace sizing is pure host arithmetic: n rows x ceil(n/64) 64-bit words
    assert lib.b200_nms_workspace_bytes(6000) == (6000 * 94 + 94 * 64) * 8      # mask words + transposed diagonal words
    assert lib.b200_nms_workspace_bytes(0) > 0
    assert lib.b200_nms_workspace_bytes(64) == (64 + 64) * 8


def test_workspace_sizing_is_host_arithmetic(lib_option):
    lib = _lib.load()
    # forward fast path: per-RoI tables + per-tile work lists; 0 when the parameters are outside the fast path
    w = lib.b200_roi_align_workspace_bytes(1, 512, 200, 272, 7, 7, 2)
    assert w > 512 * (32 + 28 * 16) and w % 256 == 0
    assert lib.b200_roi_align_workspace_bytes(1, 512, 200, 272, 7, 7, 0) == 0          # adaptive sampling -> generic kernel
    assert lib.b200_roi_align_workspace_bytes(1, 512, 200, 272, 40, 40, 2) == 0        # P * sr > 32 per axis
    assert lib.b200_roi_align_workspace_bytes(1, 0, 200, 272, 7, 7, 2) == 0
    # backward, row-stationary gather path: tables + per-row unit lists + a channel-innermost copy of dY
    wb = lib.b200_roi_align_backward_workspace_bytes(1, 512, 256, 200, 272, 7, 7, 2)
    assert 512 * 256 * 49 * 4 < wb < 512 * 256 * 49 * 4 + (4 << 20) and wb % 256 == 0
    lib_option("B200_ROI_ALIGN_BWD_PATH", "nhwc")     # vector-reduction path: one channel-innermost scratch image of dX
    assert lib.b200_roi_align_backward_workspace_bytes(1, 512, 256, 200, 272, 7, 7, 2) == 256 * 200 * 272 * 4
    lib_option("B200_ROI_ALIGN_BWD_PATH", "generic")
    assert lib.b200_roi_align_backward_workspace_bytes(1, 512, 256, 200, 272, 7, 7, 2) == 0
    lib_option("B200_ROI_ALIGN_BWD_PATH", None)
    assert lib.b200_roi_ops_set_option(b"NO_SUCH_SWITCH", b"x") == -1
    assert lib.b200_roi_align_backward_workspace_bytes(0, 512, 256, 200, 272, 7, 7, 2) == 0
    assert lib.b200_roi_align_backward_workspace_bytes(1, 512, 252, 200, 272, 7, 7, 2) == 252 * 200 * 272 * 4     # C % 64 != 0 -> NHWC path
    assert lib.b200_roi_align_backward_workspace_bytes(1, 8, 256, 200, 272, 7, 7, 2) == 0      # tiny gather volume -> scalar atomics
    # batched NMS: sum over problems of (mask words + transposed diagonal words), host arithmetic on a host array
    counts = (ctypes.c_int * 3)(6000, 0, 64)
    assert lib.b200_nms_batched_workspace_bytes(ctypes.cast(counts, ctypes.c_void_p), 3) == ((6000 * 94 + 94 * 64) + (64 + 64)) * 8 + 256
    assert lib.b200_nms_batched_workspace_bytes(ctypes.cast(counts, ctypes.c_void_p), 0) == 0
    assert lib.b200_nms_batched(None, ctypes.cast(counts, ctypes.c_void_p), 3, 5, ctypes.c_float(0.7), None, None, None, 0, None) == -1
    # NULL workspace is legal for the _ws entry points (generic kernels run); bad dims are still rejected first
    assert lib.b200_roi_align_forward_ws(None, 0.25, 1, 4, 10, 10, 3, 0, 7, 2, None, None, None, 0, None) == -1
    assert lib.b200_roi_align_backward_ws(None, 0.25, 1, 4, 10, -1, 3, 7, 7, 2, None, None, None, 0, None) == -1


def test_round2_entry_points_validate_arguments_without_gpu():
    """Top-k, RoI targets, FPN forward: argument errors are reported before any CUDA call; workspace sizing is host arithmetic."""
    lib = _lib.load()
    EINVAL = -1
    assert lib.b200_topk_batched_workspace_bytes(10) == 10 * 3 * 2048 * 4
    assert lib.b200_topk_batched_workspace_bytes(0) == 0 and lib.b200_topk_batched_workspace_bytes(65) == 0
    assert lib.b200_topk_batched(None, None, None, None, 3, None, None, None, 0, None) == EINVAL
    assert lib.b200_bbox_overlaps(None, 5, None, 4, None, None) == EINVAL
    assert lib.b200_bbox_overlaps(None, 0, None, 4, None, None) == 0                       # nothing to do
    assert lib.b200_roi_assign(None, 3, None, None, 0, None, None, None, None) == EINVAL
    assert lib.b200_roi_select(None, 5, ctypes.c_float(0.5), ctypes.c_float(0.5), ctypes.c_float(0.0), None, None, None, None) == EINVAL
    w4 = (ctypes.c_float * 4)(10, 10, 5, 5)
    assert lib.b200_fast_rcnn_targets(None, None, None, None, None, 4, 5, ctypes.cast(w4, ctypes.c_void_p), 81, 0, ctypes.c_float(1.0),
                                      ctypes.c_float(0.0), None, None, None, None, None, None) == EINVAL      # num_fg > num_keep
    # FPN workspace: the whole pyramid of an 800 x 1333 image (P5 is 25 x 42: staged by cp.async, P2..P4 by TMA)
    H = (ctypes.c_int * 4)(200, 100, 50, 25); W = (ctypes.c_int * 4)(336, 168, 84, 42)
    wf = lib.b200_roi_align_fpn_workspace_bytes(4, ctypes.cast(H, ctypes.c_void_p), ctypes.cast(W, ctypes.c_void_p), 2, 1000, 7, 7, 2)
    assert wf > 1000 * 28 * 16 and wf % 256 == 0
    assert lib.b200_roi_align_forward_fpn(7, None, None, None, None, None, 2, 1000, 256, 7, 7, 2, None, None, None, None, 0, None) == EINVAL
    # single-map workspace covers the quad-strip path's tables, CSR records and temporary records
    w = lib.b200_roi_align_workspace_bytes(1, 512, 200, 272, 7, 7, 2)
    assert w >= 512 * 28 * 16 + 512 * 196 * 24


def fpn_workspace_bytes(lib, levels, N, R, PH, PW, sr):
    H = (ctypes.c_int * len(levels))(*[h for h, _ in levels]); W = (ctypes.c_int * len(levels))(*[w for _, w in levels])
    return lib.b200_roi_align_fpn_workspace_bytes(len(levels), ctypes.cast(H, ctypes.c_void_p), ctypes.cast(W, ctypes.c_void_p),
                                                  N, R, PH, PW, sr)


@pytest.mark.parametrize("P,sr", [(7, 1), (7, 2), (14, 1), (14, 2), ((7, 14), 2)])
def test_fpn_workspace_is_zero_exactly_when_the_pyramid_call_cannot_run(P, sr, lib_option):
    """b200_roi_align_forward_fpn runs the quad-strip path only, so the size must be the strip path's alone: non-zero while the
    pyramid fits the strip geometry (batch 1..5 of 800 x 1333 images), 0 from batch 6 on (too many strip columns / rows) and
    whenever the forward is forced onto a path the pyramid call does not have.  A non-zero size there makes
    RoIAlignFPNFunction call a forward that returns B200_ROI_EWORKSPACE instead of looping over the levels."""
    lib = _lib.load()
    PH, PW = P if isinstance(P, tuple) else (P, P)
    sizes = [fpn_workspace_bytes(lib, cases.PYRAMID_800x1333, N, 1000, PH, PW, sr) for N in range(1, 9)]
    assert all(s > 0 and s % 256 == 0 for s in sizes[:5]), sizes
    assert sizes[5:] == [0, 0, 0], sizes
    # forcing the quad-strip path changes nothing; forcing any other forward path, or the per-level loop, switches the call off
    lib_option("B200_ROI_ALIGN_PATH", "quad")
    assert fpn_workspace_bytes(lib, cases.PYRAMID_800x1333, 1, 1000, PH, PW, sr) == sizes[0]
    assert fpn_workspace_bytes(lib, cases.PYRAMID_800x1333, 6, 1000, PH, PW, sr) == 0
    for path in ("stream", "generic", "tiled"):
        lib_option("B200_ROI_ALIGN_PATH", path)
        assert [fpn_workspace_bytes(lib, cases.PYRAMID_800x1333, N, 1000, PH, PW, sr) for N in (1, 5, 8)] == [0, 0, 0], path
    lib_option("B200_ROI_ALIGN_PATH", None)
    lib_option("B200_FPN_PATH", "levels")
    assert fpn_workspace_bytes(lib, cases.PYRAMID_800x1333, 1, 1000, PH, PW, sr) == 0


@pytest.mark.parametrize("limit", sorted(cases.QUAD_LIMITS))
def test_quad_strip_dispatch_limits(limit, lib_option):
    lib = _lib.load()
    lib_option("B200_ROI_ALIGN_PATH", "quad")
    ok, bad = cases.QUAD_LIMITS[limit]
    N, H, W, R, PH, PW, sr = ok
    assert lib.b200_roi_align_workspace_bytes(N, R, H, W, PH, PW, sr) > 0
    N, H, W, R, PH, PW, sr = bad
    assert lib.b200_roi_align_workspace_bytes(N, R, H, W, PH, PW, sr) == 0
    if limit == "axis_pw":                                       # the transposed grid of each side lands on the same side
        assert lib.b200_roi_align_workspace_bytes(1, 64, 50, 68, 3, 16, 2) > 0
        assert lib.b200_roi_align_workspace_bytes(1, 64, 50, 68, 17, 3, 2) == 0


def test_product_package_never_imports_oracle():
    pkg = os.path.join(ROOT, "detectron")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), fn
                assert "liboracle" not in text and "oracle/_ref" not in text, fn
