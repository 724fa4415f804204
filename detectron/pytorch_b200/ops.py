"""torch.autograd.Function front-ends over the C ABI (new-style, static) + functional helpers.

These are what the reference-shaped shims in `model/` and `modeling/` delegate to.  Every op
  * requires CUDA fp32 tensors (the reference raises NotImplementedError / asserts for CPU input),
  * makes its inputs contiguous (the reference passed raw pointers and silently assumed it),
  * launches on torch's current stream of the tensor's device,
  * allocates outputs with torch.empty (the kernels define every output element; the reference
    needed `.zero_()` passes, functions/roi_align.py:23,39-40).
"""
import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda_f32(t, name):
    if not t.is_cuda:
        raise NotImplementedError("%s must be a CUDA tensor (the reference has no CPU path for this op)" % name)
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, t.dtype))


def _rois_ok(rois):
    if rois.dim() != 2 or rois.size(1) != 5:
        raise ValueError("rois must be (R, 5) = [batch_idx, x1, y1, x2, y2], got %s" % (tuple(rois.shape),))


# ------------------------------------------------------------------------------------------------
# RoIAlign (Caffe2-exact, sampling_ratio)
# ------------------------------------------------------------------------------------------------
def roi_align_forward(features, rois, aligned_height, aligned_width, spatial_scale, sampling_ratio):
    _need_cuda_f32(features, "features"); _need_cuda_f32(rois, "rois"); _rois_ok(rois)
    features = features.contiguous(); rois = rois.contiguous()
    N, C, H, W = features.shape
    R = rois.size(0)
    out = torch.empty((R, C, aligned_height, aligned_width), dtype=torch.float32, device=features.device)
    lib = _lib.load()
    ws_bytes = int(lib.b200_roi_align_workspace_bytes(N, R, H, W, aligned_height, aligned_width, sampling_ratio))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=features.device) if ws_bytes else None   # caching allocator, stream-ordered
    with torch.cuda.device(features.device):
        _lib.check(lib.b200_roi_align_forward_ws(features.data_ptr(), spatial_scale, N, R, H, W, C, aligned_height,
                                                 aligned_width, sampling_ratio, rois.data_ptr(), out.data_ptr(),
                                                 ws.data_ptr() if ws is not None else None, ws_bytes, _stream()),
                   "b200_roi_align_forward_ws")
    return out


def roi_align_backward(grad_output, rois, feature_size, aligned_height, aligned_width, spatial_scale, sampling_ratio):
    _need_cuda_f32(grad_output, "grad_output")
    grad_output = grad_output.contiguous(); rois = rois.contiguous()
    N, C, H, W = feature_size
    grad_input = torch.empty((N, C, H, W), dtype=torch.float32, device=grad_output.device)
    lib = _lib.load()
    ws_bytes = int(lib.b200_roi_align_backward_workspace_bytes(N, rois.size(0), C, H, W, aligned_height, aligned_width,
                                                              sampling_ratio)) if rois.size(0) > 0 else 0
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=grad_output.device) if ws_bytes else None
    with torch.cuda.device(grad_output.device):
        _lib.check(lib.b200_roi_align_backward_ws(grad_output.data_ptr(), spatial_scale, N, rois.size(0), H, W, C,
                                                  aligned_height, aligned_width, sampling_ratio, rois.data_ptr(),
                                                  grad_input.data_ptr(), ws.data_ptr() if ws is not None else None,
                                                  ws_bytes, _stream()),
                   "b200_roi_align_backward_ws")
    return grad_input


class _RoIAlign(Function):
    @staticmethod
    def forward(ctx, features, rois, aligned_height, aligned_width, spatial_scale, sampling_ratio):
        ctx.args = (int(aligned_height), int(aligned_width), float(spatial_scale), int(sampling_ratio))
        ctx.feature_size = tuple(features.shape)
        ctx.save_for_backward(rois)
        return roi_align_forward(features, rois, *ctx.args)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        (rois,) = ctx.saved_tensors
        assert grad_output.is_cuda
        return roi_align_backward(grad_output, rois, ctx.feature_size, *ctx.args), None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# RoIAlign over an FPN pyramid, results written in restored order (SURVEY.md 8f N2)
# ------------------------------------------------------------------------------------------------
class _RoIAlignFPN(Function):
    """One autograd node for the reference's per-level loop + torch.cat + `xform_shuffled[restore_bl]`
    (lib/modeling/model_builder.py:264-303): level l's RoI r is row offset_l + r of the concatenated tensor, which the
    gather moves to every output row j with restore[j] == offset_l + r.  `restore` is a permutation, so each RoI has
    exactly one destination row, and the per-level kernels write it directly (b200_roi_align_forward_indexed); the
    backward reads the gradient rows of the shared tensor in place (b200_roi_align_backward_indexed)."""

    @staticmethod
    def forward(ctx, restore, aligned_height, aligned_width, sampling_ratio, scales, num_levels, *tensors):
        feats, rois = tensors[:num_levels], tensors[num_levels:]
        P = (int(aligned_height), int(aligned_width)); sr = int(sampling_ratio)
        dev = feats[0].device
        counts = [int(r.size(0)) for r in rois]
        total = sum(counts)
        if restore.numel() != total:
            raise ValueError("restore index has %d entries for %d RoIs" % (restore.numel(), total))
        C = feats[0].size(1)
        if restore.is_cuda:
            inv = torch.empty((total,), dtype=torch.int32, device=dev)
            inv[restore.to(dtype=torch.long)] = torch.arange(total, dtype=torch.int32, device=dev)
        else:                                       # the reference's restore index is a host array: invert it there
            inv_h = torch.empty((total,), dtype=torch.int32)
            inv_h[restore.to(dtype=torch.long)] = torch.arange(total, dtype=torch.int32)
            inv = inv_h.to(dev, non_blocking=False)
        out = torch.empty((total, C, P[0], P[1]), dtype=torch.float32, device=dev)
        lib = _lib.load()
        for f, r in zip(feats, rois):
            _need_cuda_f32(f, "features"); _need_cuda_f32(r, "rois"); _rois_ok(r)
            if f.size(1) != C or f.size(0) != feats[0].size(0):
                raise ValueError("every pyramid level must have the same batch size and number of channels")
        kept = [r.contiguous() for r in rois]
        done = False
        if total > 0:
            # one launch sequence over the whole pyramid: levels without RoIs drop out, the rest go level-major
            import ctypes
            live = [l for l in range(num_levels) if counts[l] > 0]
            fl = [feats[l].contiguous() for l in live]
            Lc = len(live)
            N = int(fl[0].size(0))
            hs = (ctypes.c_int * Lc)(*[int(f.size(2)) for f in fl]); wd = (ctypes.c_int * Lc)(*[int(f.size(3)) for f in fl])
            ws_bytes = int(lib.b200_roi_align_fpn_workspace_bytes(Lc, ctypes.cast(hs, ctypes.c_void_p), ctypes.cast(wd, ctypes.c_void_p), N,
                                                                  total, P[0], P[1], sr))
            if ws_bytes > 0:
                ptrs = (ctypes.c_void_p * Lc)(*[f.data_ptr() for f in fl])
                scs = (ctypes.c_float * Lc)(*[float(scales[l]) for l in live])
                begins, acc = [], 0
                for l in live:
                    begins.append(acc); acc += counts[l]
                begins.append(acc)
                bg = (ctypes.c_int * (Lc + 1))(*begins)
                all_rois = torch.cat([kept[l] for l in live], dim=0) if Lc > 1 else kept[live[0]]
                # inv is indexed by the position in the FULL level-major order; empty levels contribute nothing, so it is the same order
                ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
                with torch.cuda.device(dev):
                    _lib.check(lib.b200_roi_align_forward_fpn(Lc, ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(hs, ctypes.c_void_p),
                                                              ctypes.cast(wd, ctypes.c_void_p), ctypes.cast(scs, ctypes.c_void_p),
                                                              ctypes.cast(bg, ctypes.c_void_p), N, total, C, P[0], P[1], sr,
                                                              all_rois.data_ptr(), inv.data_ptr(), out.data_ptr(), ws.data_ptr(), ws_bytes,
                                                              _stream()), "b200_roi_align_forward_fpn")
                done = True
        off = 0
        with torch.cuda.device(dev):
            for f, r, sc, n_l in zip(feats, kept, scales, counts):
                if n_l and not done:
                    f = f.contiguous()
                    N, _, H, W = f.shape
                    ws_bytes = int(lib.b200_roi_align_workspace_bytes(N, n_l, H, W, P[0], P[1], sr))
                    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
                    rows = inv[off:off + n_l]
                    _lib.check(lib.b200_roi_align_forward_indexed(f.data_ptr(), float(sc), N, n_l, H, W, C, P[0], P[1], sr,
                                                                  r.data_ptr(), rows.data_ptr(), out.data_ptr(),
                                                                  ws.data_ptr() if ws is not None else None, ws_bytes, _stream()),
                               "b200_roi_align_forward_indexed")
                off += n_l
        ctx.meta = (P, sr, [float(sc) for sc in scales], counts, [tuple(f.shape) for f in feats], num_levels)
        ctx.save_for_backward(inv, *kept)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        P, sr, scales, counts, shapes, num_levels = ctx.meta
        inv, rois = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        assert grad_output.is_cuda
        grad_output = grad_output.contiguous()
        dev = grad_output.device
        lib = _lib.load()
        grads = []
        off = 0
        with torch.cuda.device(dev):
            for r, sc, n_l, shape in zip(rois, scales, counts, shapes):
                N, C, H, W = shape
                if n_l == 0:
                    grads.append(torch.zeros(shape, dtype=torch.float32, device=dev))
                    continue
                g = torch.empty(shape, dtype=torch.float32, device=dev)
                ws_bytes = int(lib.b200_roi_align_backward_workspace_bytes(N, n_l, C, H, W, P[0], P[1], sr))
                ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
                rows = inv[off:off + n_l]
                _lib.check(lib.b200_roi_align_backward_indexed(grad_output.data_ptr(), rows.data_ptr(), sc, N, n_l, H, W, C,
                                                               P[0], P[1], sr, r.data_ptr(), g.data_ptr(),
                                                               ws.data_ptr() if ws is not None else None, ws_bytes, _stream()),
                           "b200_roi_align_backward_indexed")
                grads.append(g)
                off += n_l
        return (None, None, None, None, None, None) + tuple(grads) + (None,) * num_levels


def roi_align_fpn(features, rois, restore, aligned_height, aligned_width, spatial_scales, sampling_ratio):
    """features: list of (N, C, H_l, W_l) CUDA tensors; rois: list of (R_l, 5) CUDA tensors (same order); restore: the
    reference's `*_idx_restore_int32` (any integer tensor / array of length sum R_l); spatial_scales: one per level.
    Returns (sum R_l, C, PH, PW) in restored order == torch.cat([RoIAlign_l(...)])[restore]."""
    if len(features) != len(rois) or len(features) != len(spatial_scales):
        raise ValueError("features, rois and spatial_scales must have one entry per pyramid level")
    restore = torch.as_tensor(restore)
    return _RoIAlignFPN.apply(restore, aligned_height, aligned_width, sampling_ratio, tuple(spatial_scales), len(features),
                              *features, *rois)


# ------------------------------------------------------------------------------------------------
# RoIAlign (legacy, lattice-corner samples)
# ------------------------------------------------------------------------------------------------
def roi_align_legacy_forward(features, rois, aligned_height, aligned_width, spatial_scale):
    _need_cuda_f32(features, "features"); _need_cuda_f32(rois, "rois"); _rois_ok(rois)
    features = features.contiguous(); rois = rois.contiguous()
    N, C, H, W = features.shape
    R = rois.size(0)
    out = torch.empty((R, C, aligned_height, aligned_width), dtype=torch.float32, device=features.device)
    with torch.cuda.device(features.device):
        _lib.check(_lib.load().b200_roi_align_legacy_forward(features.data_ptr(), spatial_scale, N, R, H, W, C,
                                                             aligned_height, aligned_width, rois.data_ptr(),
                                                             out.data_ptr(), _stream()),
                   "b200_roi_align_legacy_forward")
    return out


def roi_align_legacy_backward(grad_output, rois, feature_size, aligned_height, aligned_width, spatial_scale):
    _need_cuda_f32(grad_output, "grad_output")
    grad_output = grad_output.contiguous(); rois = rois.contiguous()
    N, C, H, W = feature_size
    grad_input = torch.empty((N, C, H, W), dtype=torch.float32, device=grad_output.device)
    with torch.cuda.device(grad_output.device):
        _lib.check(_lib.load().b200_roi_align_legacy_backward(grad_output.data_ptr(), spatial_scale, N, rois.size(0), H, W, C,
                                                              aligned_height, aligned_width, rois.data_ptr(),
                                                              grad_input.data_ptr(), _stream()),
                   "b200_roi_align_legacy_backward")
    return grad_input


class _RoIAlignLegacy(Function):
    @staticmethod
    def forward(ctx, features, rois, aligned_height, aligned_width, spatial_scale):
        ctx.args = (int(aligned_height), int(aligned_width), float(spatial_scale))
        ctx.feature_size = tuple(features.shape)
        ctx.save_for_backward(rois)
        return roi_align_legacy_forward(features, rois, *ctx.args)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        (rois,) = ctx.saved_tensors
        assert grad_output.is_cuda
        return roi_align_legacy_backward(grad_output, rois, ctx.feature_size, *ctx.args), None, None, None, None


# ------------------------------------------------------------------------------------------------
# RoIPool
# ------------------------------------------------------------------------------------------------
def roi_pool_forward(features, rois, pooled_height, pooled_width, spatial_scale):
    _need_cuda_f32(features, "features"); _need_cuda_f32(rois, "rois"); _rois_ok(rois)
    features = features.contiguous(); rois = rois.contiguous()
    N, C, H, W = features.shape
    R = rois.size(0)
    out = torch.empty((R, C, pooled_height, pooled_width), dtype=torch.float32, device=features.device)
    argmax = torch.empty((R, C, pooled_height, pooled_width), dtype=torch.int32, device=features.device)
    with torch.cuda.device(features.device):
        _lib.check(_lib.load().b200_roi_pool_forward(features.data_ptr(), spatial_scale, N, R, H, W, C, pooled_height,
                                                     pooled_width, rois.data_ptr(), out.data_ptr(), argmax.data_ptr(),
                                                     _stream()),
                   "b200_roi_pool_forward")
    return out, argmax


def roi_pool_backward(grad_output, argmax, rois, feature_size, pooled_height, pooled_width, spatial_scale):
    _need_cuda_f32(grad_output, "grad_output")
    grad_output = grad_output.contiguous(); rois = rois.contiguous(); argmax = argmax.contiguous()
    N, C, H, W = feature_size
    grad_input = torch.empty((N, C, H, W), dtype=torch.float32, device=grad_output.device)
    with torch.cuda.device(grad_output.device):
        _lib.check(_lib.load().b200_roi_pool_backward(grad_output.data_ptr(), spatial_scale, N, rois.size(0), H, W, C,
                                                      pooled_height, pooled_width, rois.data_ptr(), grad_input.data_ptr(),
                                                      argmax.data_ptr(), _stream()),
                   "b200_roi_pool_backward")
    return grad_input


class _RoIPool(Function):
    @staticmethod
    def forward(ctx, features, rois, pooled_height, pooled_width, spatial_scale):
        ctx.args = (int(pooled_height), int(pooled_width), float(spatial_scale))
        ctx.feature_size = tuple(features.shape)
        out, argmax = roi_pool_forward(features, rois, *ctx.args)
        ctx.save_for_backward(rois, argmax)
        ctx.mark_non_differentiable(argmax)
        return out, argmax

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output, _grad_argmax):
        rois, argmax = ctx.saved_tensors
        assert grad_output.is_cuda
        return roi_pool_backward(grad_output, argmax, rois, ctx.feature_size, *ctx.args), None, None, None, None


# ------------------------------------------------------------------------------------------------
# RoICrop
# ------------------------------------------------------------------------------------------------
def roi_crop_forward(input1, input2):
    _need_cuda_f32(input1, "input1"); _need_cuda_f32(input2, "input2")
    if input2.dim() != 4 or input2.size(3) != 2:
        raise ValueError("input2 (grid) must be (R, h, w, 2) in (y, x) order, got %s" % (tuple(input2.shape),))
    assert input1.get_device() == input2.get_device(), "input1 and input2 must on the same device"
    input1 = input1.contiguous(); input2 = input2.contiguous()
    N, C, H, W = input1.shape
    R, oh, ow, _ = input2.shape
    out = torch.empty((R, C, oh, ow), dtype=torch.float32, device=input1.device)
    with torch.cuda.device(input1.device):
        _lib.check(_lib.load().b200_roi_crop_forward(input1.data_ptr(), input2.data_ptr(), N, C, H, W, R, oh, ow,
                                                     out.data_ptr(), _stream()),
                   "b200_roi_crop_forward")
    return out


def roi_crop_backward(grad_output, input2, input1_size):
    _need_cuda_f32(grad_output, "grad_output")
    grad_output = grad_output.contiguous(); input2 = input2.contiguous()
    N, C, H, W = input1_size
    R, oh, ow, _ = input2.shape
    grad_input1 = torch.empty((N, C, H, W), dtype=torch.float32, device=grad_output.device)
    grad_input2 = torch.empty_like(input2)
    lib = _lib.load()
    ws_bytes = int(lib.b200_roi_crop_backward_workspace_bytes(N, C, H, W, R, oh, ow))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=grad_output.device) if ws_bytes else None
    with torch.cuda.device(grad_output.device):
        _lib.check(lib.b200_roi_crop_backward_ws(grad_output.data_ptr(), input2.data_ptr(), N, C, H, W, R, oh, ow,
                                                 grad_input1.data_ptr(), grad_input2.data_ptr(),
                                                 ws.data_ptr() if ws is not None else None, ws_bytes, _stream()),
                   "b200_roi_crop_backward_ws")
    return grad_input1, grad_input2


class _RoICrop(Function):
    @staticmethod
    def forward(ctx, input1, input2):
        ctx.input1_size = tuple(input1.shape)
        ctx.save_for_backward(input2)
        return roi_crop_forward(input1, input2)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        (input2,) = ctx.saved_tensors
        assert grad_output.is_cuda
        return roi_crop_backward(grad_output, input2, ctx.input1_size)


# ------------------------------------------------------------------------------------------------
# NMS
# ------------------------------------------------------------------------------------------------
TOPK_MAX_K = 16384
TOPK_MAX_PROBLEMS = 64


def topk_batched_raw(score_maps, ks):
    """Top-k of several (A, H, W) float32 CUDA score maps in one batched call (b200_topk_batched: radix select + in-CTA sort,
    no host read).  ks: host ints, k_p <= min(A*H*W, 16384); <= 64 problems.  Returns (order int64 (sum k,), scores float32
    (sum k,)): problem p's slice holds, best first, the indices into its (H, W, A) flattening and the scores."""
    import ctypes
    P = len(score_maps)
    if P < 1 or P > TOPK_MAX_PROBLEMS or len(ks) != P:
        raise ValueError("topk_batched_raw: 1..64 problems with one k each")
    maps = []
    for m in score_maps:
        _need_cuda_f32(m, "score map")
        if m.dim() != 3:
            raise ValueError("score maps must be (A, H, W), got %s" % (tuple(m.shape),))
        maps.append(m.contiguous())
    ks = [int(k) for k in ks]
    dev = maps[0].device
    total = sum(ks)
    order = torch.empty((max(total, 1),), dtype=torch.int64, device=dev)
    scores = torch.empty((max(total, 1),), dtype=torch.float32, device=dev)
    lib = _lib.load()
    ptrs = (ctypes.c_void_p * P)(*[m.data_ptr() for m in maps])
    A = (ctypes.c_int * P)(*[m.size(0) for m in maps])
    HW = (ctypes.c_int * P)(*[m.size(1) * m.size(2) for m in maps])
    K = (ctypes.c_int * P)(*ks)
    ws_bytes = int(lib.b200_topk_batched_workspace_bytes(P))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.b200_topk_batched(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(A, ctypes.c_void_p), ctypes.cast(HW, ctypes.c_void_p),
                                         ctypes.cast(K, ctypes.c_void_p), P, order.data_ptr(), scores.data_ptr(), ws.data_ptr(), ws_bytes,
                                         _stream()), "b200_topk_batched")
    return order[:total], scores[:total]


def nms_batched_raw(dets, counts, thresh):
    """`len(counts)` independent NMS problems in one pair of launches.  dets: (sum(counts), >=4) rows of the problems back to
    back, each problem score-sorted; counts: host ints.  Returns (keep int32 (sum(counts),), num_out int32 (P,)) on the
    device: problem p's kept indices (relative to its first row) sit at keep[offset_p : offset_p + num_out[p]]."""
    import ctypes
    _need_cuda_f32(dets, "dets")
    if dets.dim() != 2 or dets.size(1) < 4:
        raise ValueError("dets must be (N, >=4) = [x1, y1, x2, y2, score], got %s" % (tuple(dets.shape),))
    counts = [int(c) for c in counts]
    if sum(counts) != dets.size(0) or not counts:
        raise ValueError("counts %s do not add up to %d rows" % (counts, dets.size(0)))
    dets = dets.contiguous()
    lib = _lib.load()
    P = len(counts)
    c_arr = (ctypes.c_int * P)(*counts)
    keep = torch.empty((max(dets.size(0), 1),), dtype=torch.int32, device=dets.device)
    num_out = torch.empty((P,), dtype=torch.int32, device=dets.device)
    ws_bytes = int(lib.b200_nms_batched_workspace_bytes(ctypes.cast(c_arr, ctypes.c_void_p), P))
    if ws_bytes == 0:
        raise ValueError("b200_nms_batched: 1..64 problems expected, got %d" % P)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dets.device)
    with torch.cuda.device(dets.device):
        _lib.check(lib.b200_nms_batched(dets.data_ptr(), ctypes.cast(c_arr, ctypes.c_void_p), P, dets.size(1), float(thresh), keep.data_ptr(),
                                        num_out.data_ptr(), ws.data_ptr(), ws_bytes, _stream()), "b200_nms_batched")
    return keep, num_out


def nms_batched_chunked(dets, counts, thresh):
    """nms_batched_raw for any number of problems (b200_nms_batched takes up to 64 per call): same return layout."""
    counts = [int(c) for c in counts]
    if len(counts) <= 64:
        return nms_batched_raw(dets, counts, thresh)
    keeps, nums, off = [], [], 0
    for c0 in range(0, len(counts), 64):
        chunk = counts[c0:c0 + 64]
        n = sum(chunk)
        if n == 0:
            keeps.append(torch.empty((0,), dtype=torch.int32, device=dets.device))
            nums.append(torch.zeros((len(chunk),), dtype=torch.int32, device=dets.device))
        else:
            k, m = nms_batched_raw(dets[off:off + n], chunk, thresh)
            keeps.append(k[:n]); nums.append(m)
        off += n
    return torch.cat(keeps), torch.cat(nums)


def soft_nms_batched(dets, counts, sigma=0.5, overlap_thresh=0.3, score_thresh=0.001, method=1):
    """Soft-NMS (lib/utils/cython_nms.pyx:98-203) on `len(counts)` problems stored back to back in dets (sum(counts), 5).
    Returns (dets_out, inds, num_out): problem p's survivors are dets_out[off_p : off_p + num_out[p]] (decayed scores, the
    reference's output order), inds their original row indices within the problem."""
    import ctypes
    _need_cuda_f32(dets, "dets")
    counts = [int(c) for c in counts]
    if dets.dim() != 2 or dets.size(1) != 5 or sum(counts) != dets.size(0):
        raise ValueError("dets must be (sum(counts), 5)")
    lib = _lib.load()
    out = dets.contiguous().clone()
    P = len(counts)
    inds = torch.empty((max(out.size(0), 1),), dtype=torch.int32, device=dets.device)
    num_out = torch.empty((P,), dtype=torch.int32, device=dets.device)
    offs = 0
    for c0 in range(0, P, 128):
        chunk = counts[c0:c0 + 128]
        n = sum(chunk)
        c_arr = (ctypes.c_int * len(chunk))(*chunk)
        with torch.cuda.device(dets.device):
            _lib.check(lib.b200_soft_nms_batched(out.data_ptr() + offs * 20, ctypes.cast(c_arr, ctypes.c_void_p), len(chunk), float(sigma),
                                                 float(overlap_thresh), float(score_thresh), int(method), inds.data_ptr() + offs * 4,
                                                 num_out.data_ptr() + c0 * 4, _stream()), "b200_soft_nms_batched")
        offs += n
    return out, inds, num_out


def box_voting_batched(top_dets, top_counts, all_dets, all_counts, thresh, scoring=0, beta=1.0):
    """Box voting (lib/utils/boxes.py:268-317) for `len(top_counts)` class problems; returns the refined top_dets."""
    import ctypes
    _need_cuda_f32(top_dets, "top_dets"); _need_cuda_f32(all_dets, "all_dets")
    top_counts = [int(c) for c in top_counts]; all_counts = [int(c) for c in all_counts]
    if len(top_counts) != len(all_counts) or sum(top_counts) != top_dets.size(0) or sum(all_counts) != all_dets.size(0):
        raise ValueError("counts do not match the detection tensors")
    lib = _lib.load()
    top_dets = top_dets.contiguous(); all_dets = all_dets.contiguous()
    out = torch.empty_like(top_dets)
    to = ao = 0
    for c0 in range(0, len(top_counts), 128):
        tc, ac = top_counts[c0:c0 + 128], all_counts[c0:c0 + 128]
        t_arr = (ctypes.c_int * len(tc))(*tc); a_arr = (ctypes.c_int * len(ac))(*ac)
        with torch.cuda.device(top_dets.device):
            _lib.check(lib.b200_box_voting_batched(top_dets.data_ptr() + to * 20, ctypes.cast(t_arr, ctypes.c_void_p),
                                                   all_dets.data_ptr() + ao * 20, ctypes.cast(a_arr, ctypes.c_void_p), len(tc), float(thresh),
                                                   int(scoring), float(beta), out.data_ptr() + to * 20, _stream()), "b200_box_voting_batched")
        to += sum(tc); ao += sum(ac)
    return out


def nms_raw(dets, thresh):
    """Returns (keep int32 (N,), num_out int32 (1,)) on the device, no host sync."""
    _need_cuda_f32(dets, "dets")
    if dets.dim() != 2 or dets.size(1) < 4:
        raise ValueError("dets must be (N, >=4) = [x1, y1, x2, y2, score], got %s" % (tuple(dets.shape),))
    dets = dets.contiguous()
    n, dim = dets.shape
    lib = _lib.load()
    keep = torch.empty((max(n, 1),), dtype=torch.int32, device=dets.device)
    num_out = torch.empty((1,), dtype=torch.int32, device=dets.device)
    ws_bytes = int(lib.b200_nms_workspace_bytes(n))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dets.device)
    with torch.cuda.device(dets.device):
        _lib.check(lib.b200_nms(dets.data_ptr(), n, dim, float(thresh), keep.data_ptr(), num_out.data_ptr(),
                                ws.data_ptr(), ws_bytes, _stream()),
                   "b200_nms")
    return keep, num_out


# ------------------------------------------------------------------------------------------------
# Test-time mask paste (lib/core/test.py:793-847 segm_results)
# ------------------------------------------------------------------------------------------------
def _segm_args(masks, mask_channel, ref_boxes, im_h, im_w):
    _need_cuda_f32(masks, "masks"); _need_cuda_f32(ref_boxes, "ref_boxes")
    if masks.dim() != 4 or masks.size(2) != masks.size(3):
        raise ValueError("masks must be (D, K, M, M), got %s" % (tuple(masks.shape),))
    D = masks.size(0)
    if tuple(ref_boxes.shape) != (D, 4):
        raise ValueError("ref_boxes must be (D, 4) = [x1, y1, x2, y2], got %s" % (tuple(ref_boxes.shape),))
    if mask_channel is None:
        chan = None
    else:
        chan = torch.as_tensor(mask_channel, dtype=torch.int32, device=masks.device).reshape(-1).contiguous()
        if chan.numel() != D:
            raise ValueError("mask_channel must hold one channel per detection (%d), got %d" % (D, chan.numel()))
    return masks.contiguous(), chan, ref_boxes.contiguous(), D, masks.size(1), masks.size(2), int(im_h), int(im_w)


def segm_paste(masks, mask_channel, ref_boxes, im_h, im_w, thresh=0.5):
    """Dense binary masks (D, im_h, im_w) uint8 on the device: detection i's soft mask masks[i, mask_channel[i]]
    (None: channel 0) resized to its (M + 2) / M-expanded box like cv2.resize with IPP off, `> thresh`, pasted into the
    image (lib/core/test.py:806-833)."""
    masks, chan, boxes, D, K, M, im_h, im_w = _segm_args(masks, mask_channel, ref_boxes, im_h, im_w)
    out = torch.empty((D, im_h, im_w), dtype=torch.uint8, device=masks.device)
    with torch.cuda.device(masks.device):
        _lib.check(_lib.load().b200_segm_paste(masks.data_ptr(), chan.data_ptr() if chan is not None else None, boxes.data_ptr(), D, K, M,
                                               im_h, im_w, float(thresh), out.data_ptr(), _stream()), "b200_segm_paste")
    return out


def segm_rle(masks, mask_channel, ref_boxes, im_h, im_w, thresh=0.5):
    """COCO uncompressed RLE of the masks segm_paste would produce, without materialising them.  Returns host numpy
    arrays (runs int32, counts int64): detection i's run lengths are runs[sum(counts[:i]) : sum(counts[:i + 1])],
    column-major, alternating from a run of zeros.  One host read of the counts, one copy of all runs."""
    import numpy as np
    masks, chan, boxes, D, K, M, im_h, im_w = _segm_args(masks, mask_channel, ref_boxes, im_h, im_w)
    if D == 0:
        return np.zeros((0,), np.int32), np.zeros((0,), np.int64)
    lib = _lib.load()
    args = (masks.data_ptr(), chan.data_ptr() if chan is not None else None, boxes.data_ptr(), D, K, M, im_h, im_w, float(thresh))
    offsets = torch.empty((D + 1,), dtype=torch.int64, device=masks.device)
    with torch.cuda.device(masks.device):
        _lib.check(lib.b200_segm_rle_count(*args, offsets.data_ptr(), _stream()), "b200_segm_rle_count")
        offs = offsets.cpu().numpy()
        runs = torch.empty((max(int(offs[-1]), 1),), dtype=torch.int32, device=masks.device)
        _lib.check(lib.b200_segm_rle_emit(*args, offsets.data_ptr(), runs.data_ptr(), _stream()), "b200_segm_rle_emit")
        runs_h = runs[:int(offs[-1])].cpu().numpy()
    return runs_h, np.diff(offs).astype(np.int64)
