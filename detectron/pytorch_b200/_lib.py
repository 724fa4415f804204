"""ctypes binding of libb200_roi_ops.so -- the C ABI declared in include/b200_roi_ops.h.

This is the ONLY compute backend of the package: there is no CPU or PyTorch fallback.  If the
shared library is missing and cannot be built (no nvcc), every op raises ImportError loudly.
"""
import ctypes
import os
import threading

from . import build as _build

_c_float_p = ctypes.c_void_p      # raw device pointers are passed as integers
_stream_t = ctypes.c_void_p

_lock = threading.Lock()
_lib = None

_SIGNATURES = {
    "b200_roi_ops_abi_version": (ctypes.c_int, []),
    "b200_roi_ops_strerror": (ctypes.c_char_p, [ctypes.c_int]),
    "b200_roi_ops_launch_count": (ctypes.c_ulonglong, []),
    "b200_roi_ops_set_option": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_char_p]),
    "b200_roi_ops_debug_timing_buffer": (None, [ctypes.c_void_p]),
    # (bottom, scale, N, R, H, W, C, PH, PW, sr, rois, top, stream)
    "b200_roi_align_forward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 8 + [_c_float_p, _c_float_p, _stream_t]),
    "b200_roi_align_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 7),
    # (bottom, scale, N, R, H, W, C, PH, PW, sr, rois, top, workspace, workspace_bytes, stream)
    "b200_roi_align_forward_ws": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 8 +
                                  [_c_float_p, _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    "b200_roi_align_backward_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 8),
    "b200_roi_align_backward_ws": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 8 +
                                   [_c_float_p, _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    "b200_roi_align_backward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 8 + [_c_float_p, _c_float_p, _stream_t]),
    # (bottom, scale, N, R, H, W, C, PH, PW, sr, rois, top_rows, top, workspace, workspace_bytes, stream)
    "b200_roi_align_forward_indexed": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 8 +
                                       [_c_float_p, ctypes.c_void_p, _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    # (top_diff, top_rows, scale, N, R, H, W, C, PH, PW, sr, rois, bottom_diff, workspace, workspace_bytes, stream)
    "b200_roi_align_backward_indexed": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, ctypes.c_float] + [ctypes.c_int] * 8 +
                                        [_c_float_p, _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    # (bottom, scale, N, R, H, W, C, PH, PW, rois, top, stream)
    "b200_roi_align_legacy_forward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, _stream_t]),
    "b200_roi_align_legacy_backward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, _stream_t]),
    # (bottom, scale, N, R, H, W, C, PH, PW, rois, top, argmax, stream)
    "b200_roi_pool_forward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, ctypes.c_void_p, _stream_t]),
    "b200_roi_pool_backward": (ctypes.c_int, [_c_float_p, ctypes.c_float] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, ctypes.c_void_p, _stream_t]),
    # (image, grids, N, C, H, W, R, oh, ow, output, stream)
    "b200_roi_crop_forward": (ctypes.c_int, [_c_float_p, _c_float_p] + [ctypes.c_int] * 7 + [_c_float_p, _stream_t]),
    # (grad_output, grids, N, C, H, W, R, oh, ow, grad_image, grad_grids, stream)
    "b200_roi_crop_backward": (ctypes.c_int, [_c_float_p, _c_float_p] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, _stream_t]),
    "b200_roi_crop_backward_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int] * 7),
    # (grad_output, grids, N, C, H, W, R, oh, ow, grad_image, grad_grids, workspace, workspace_bytes, stream)
    "b200_roi_crop_backward_ws": (ctypes.c_int, [_c_float_p, _c_float_p] + [ctypes.c_int] * 7 + [_c_float_p, _c_float_p, ctypes.c_void_p,
                                                                                              ctypes.c_size_t, _stream_t]),
    # (deltas, anchors, order, scores, k, A, H, W, stride, im_h, im_w, min_size, dets, valid, stream)
    "b200_proposal_decode": (ctypes.c_int, [_c_float_p, _c_float_p, ctypes.c_void_p, _c_float_p] + [ctypes.c_int] * 4 +
                             [ctypes.c_float] * 4 + [_c_float_p, ctypes.c_void_p, _stream_t]),
    "b200_nms_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int]),
    # (boxes, n, dim, thresh, keep_out, num_out, workspace, workspace_bytes, stream)
    "b200_nms": (ctypes.c_int, [_c_float_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                                ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    # (L, heights_host, widths_host, N, R, PH, PW, sr)
    "b200_roi_align_fpn_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5),
    # (L, bottoms_host, heights_host, widths_host, scales_host, roi_begin_host, N, R, C, PH, PW, sr, rois, top_rows, top, ws, ws_bytes, stream)
    "b200_roi_align_forward_fpn": (ctypes.c_int, [ctypes.c_int] + [ctypes.c_void_p] * 5 + [ctypes.c_int] * 6 +
                                   [_c_float_p, ctypes.c_void_p, _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    "b200_nms_batched_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int]),
    # (boxes, counts_host, P, dim, thresh, keep_out, num_out, workspace, workspace_bytes, stream)
    "b200_nms_batched": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    # (dets, counts_host, P, sigma, Nt, score_thresh, method, inds_out, num_out, stream)
    "b200_soft_nms_batched": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                                             ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, _stream_t]),
    # (top, top_counts_host, all, all_counts_host, P, thresh, scoring, beta, out, stream)
    "b200_box_voting_batched": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, _c_float_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float,
                                               ctypes.c_int, ctypes.c_float, _c_float_p, _stream_t]),
    "b200_topk_batched_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int]),
    # (score_ptrs_host, A_host, HW_host, k_host, P, order_out, scores_out, workspace, workspace_bytes, stream)
    "b200_topk_batched": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                         _c_float_p, ctypes.c_void_p, ctypes.c_size_t, _stream_t]),
    # (boxes, N, query, K, out, stream)
    "b200_bbox_overlaps": (ctypes.c_int, [_c_float_p, ctypes.c_int, _c_float_p, ctypes.c_int, _c_float_p, _stream_t]),
    # (boxes, N, gt, gt_classes, G, max_overlaps, argmax, max_classes, stream)
    "b200_roi_assign": (ctypes.c_int, [_c_float_p, ctypes.c_int, _c_float_p, ctypes.c_void_p, ctypes.c_int, _c_float_p, ctypes.c_void_p,
                                       ctypes.c_void_p, _stream_t]),
    # (max_overlaps, N, fg, bg_hi, bg_lo, fg_inds, bg_inds, counts, stream)
    "b200_roi_select": (ctypes.c_int, [_c_float_p, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p, _stream_t]),
    # (boxes, gt, argmax, max_classes, keep, n, n_fg, weights4_host, reg_classes, agnostic, im_scale, batch_idx, labels, rois, targets, inside, outside, stream)
    "b200_fast_rcnn_targets": (ctypes.c_int, [_c_float_p, _c_float_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                              ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                              ctypes.c_void_p, _c_float_p, _c_float_p, _c_float_p, _c_float_p, _stream_t]),
    # (masks, mask_channel, ref_boxes, D, K, M, im_h, im_w, thresh, out, stream)
    "b200_segm_paste": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, _c_float_p] + [ctypes.c_int] * 5 + [ctypes.c_float, ctypes.c_void_p,
                                                                                                         _stream_t]),
    # (masks, mask_channel, ref_boxes, D, K, M, im_h, im_w, thresh, offsets_out, stream)
    "b200_segm_rle_count": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, _c_float_p] + [ctypes.c_int] * 5 + [ctypes.c_float,
                                                                                                             ctypes.c_void_p, _stream_t]),
    # (masks, mask_channel, ref_boxes, D, K, M, im_h, im_w, thresh, offsets, runs_out, stream)
    "b200_segm_rle_emit": (ctypes.c_int, [_c_float_p, ctypes.c_void_p, _c_float_p] + [ctypes.c_int] * 5 + [ctypes.c_float, ctypes.c_void_p,
                                                                                                            ctypes.c_void_p, _stream_t]),
}

EXPORTED_SYMBOLS = tuple(sorted(_SIGNATURES))


def lib_path():
    return _build.LIB_PATH


def load():
    """Load (building in-tree first if needed) libb200_roi_ops.so and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(_build.LIB_PATH):
            try:
                _build.build()
            except Exception as exc:  # noqa: BLE001
                raise ImportError(
                    "detectron.pytorch_b200: libb200_roi_ops.so is missing and could not be built (%s). "
                    "There is no CPU/PyTorch fallback for these ops; run `python -m detectron.pytorch_b200.build`." % exc)
        lib = ctypes.CDLL(_build.LIB_PATH)
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here == header/library mismatch: fail loudly
            fn.restype = restype
            fn.argtypes = argtypes
        if lib.b200_roi_ops_abi_version() != 3:
            raise ImportError("libb200_roi_ops.so ABI version mismatch")
        _lib = lib
    return _lib


def check(status, what):
    if status != 0:
        msg = load().b200_roi_ops_strerror(status)
        raise RuntimeError("%s failed: %s (status %d)" % (what, msg.decode() if msg else "?", status))


def launch_count():
    return int(load().b200_roi_ops_launch_count())


def set_option(name, value=None):
    """Path-selection switch (see b200_roi_ops_set_option in include/b200_roi_ops.h); value None restores the default."""
    check(load().b200_roi_ops_set_option(name.encode(), None if value is None else str(value).encode()), "b200_roi_ops_set_option")
