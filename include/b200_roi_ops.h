/*
 * b200_roi_ops.h -- C ABI of libb200_roi_ops.so: hand-written sm_100a CUDA replacements for the
 * per-image detection hot path of roytseng-tw/Detectron.pytorch (RoIAlign fwd/bwd in both
 * flavours, RoIPool, RoICrop, proposal NMS).
 *
 * The boundary mirrors the raw-pointer `extern "C"` launchers that sit under the reference's
 * cffi/THC glue (the layer its `_ext` modules bind): plain device pointers, ints and floats, a
 * CUDA stream, no torch types.  Each entry point cites the reference launcher it replaces
 * (paths relative to the reference repository root).
 *
 * Conventions (all entry points)
 *   - every pointer is a DEVICE pointer to dense, row-major ("contiguous") memory;
 *   - features / gradients are fp32 NCHW; rois are fp32 (R,5) = [batch_idx, x1, y1, x2, y2] in
 *     image pixels; boxes for NMS are fp32 (N,dim>=4) = [x1, y1, x2, y2, ...];
 *   - work is enqueued on `stream` (pass torch's current stream); calls never synchronise unless
 *     stated, keep no reference to caller memory after the enqueued work finishes, and are
 *     re-entrant per device;
 *   - outputs need NOT be pre-zeroed by the caller (the reference required `.zero_()`,
 *     functions/roi_align.py:23,39-40): every call fully defines its output;
 *   - return value: 0 = success; > 0 = a cudaError_t raised by the launch; < 0 = argument error
 *     (B200_ROI_EINVAL, B200_ROI_EWORKSPACE).  The reference instead returned 1/0 and called
 *     exit(-1) on a launch error (roi_align_kernel.cu:135-139); the Python layer turns a non-zero
 *     status into RuntimeError.
 */
#ifndef B200_ROI_OPS_H_
#define B200_ROI_OPS_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* b200_stream_t; /* == cudaStream_t */

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

#define B200_ROI_OK 0
#define B200_ROI_EINVAL (-1)
#define B200_ROI_EWORKSPACE (-2)

/* ABI version of this header (bumped on any signature change). */
B200_API int b200_roi_ops_abi_version(void);
/* Human-readable message for a status returned by any entry point. */
B200_API const char* b200_roi_ops_strerror(int status);

/* ---- RoIAlign, Caffe2/Detectron-exact variant (sampling_ratio) ---------------------------------
 * replaces ROIAlignForwardLaucher / ROIAlignBackwardLaucher,
 *   lib/modeling/roi_xfrom/roi_align/src/roi_align_kernel.cu:123-142, 272-290
 *   (declared lib/modeling/roi_xfrom/roi_align/src/roi_align_kernel.h:13-27; bound through
 *    roi_align_forward_cuda / roi_align_backward_cuda, src/roi_align_cuda.c:7-40, 42-76).
 * Same argument meaning and order; `batch_size` is added to the forward (the reference only passed
 * it to the backward) so that batch indices can be range-checked by the planner.
 * top: (R, C, aligned_height, aligned_width).  bottom_diff: (batch_size, C, H, W), fully written. */
B200_API int b200_roi_align_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                           int height, int width, int channels, int aligned_height, int aligned_width,
                           int sampling_ratio, const float* bottom_rois, float* top_data,
                           b200_stream_t stream);
B200_API int b200_roi_align_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois,
                            int height, int width, int channels, int aligned_height, int aligned_width,
                            int sampling_ratio, const float* bottom_rois, float* bottom_diff,
                            b200_stream_t stream);

/* Workspace variant of the forward: the feature-map-stationary fast path needs
 * b200_roi_align_workspace_bytes(batch_size, num_rois, height, width, aligned_height, aligned_width,
 * sampling_ratio) bytes of device scratch (per-RoI sample tables + per-tile RoI lists; 256-byte
 * aligned; 0 = fast path not applicable to these parameters).  The Python layer takes it from torch's caching allocator.  The plain
 * b200_roi_align_forward obtains the same scratch with cudaMallocAsync/cudaFreeAsync on `stream`.
 * With workspace == NULL (or too small) the shape-generic kernel runs.  Results are identical
 * either way up to ~1 ulp on bins whose samples straddle two tiles. */
B200_API size_t b200_roi_align_workspace_bytes(int batch_size, int num_rois, int height, int width,
                                               int aligned_height, int aligned_width, int sampling_ratio);
B200_API int b200_roi_align_forward_ws(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                              int height, int width, int channels, int aligned_height, int aligned_width,
                              int sampling_ratio, const float* bottom_rois, float* top_data,
                              void* workspace, size_t workspace_bytes, b200_stream_t stream);

/* Workspace variant of the backward.  The fast paths need device scratch:
 *   - row-stationary gather path (no atomics): per-RoI tables, row-bucketed unit lists and a channel-innermost
 *     copy of dY (~ sizeof dY);
 *   - vector-reduction path: a channel-innermost scratch image of dX (= sizeof dX).
 * b200_roi_align_backward_workspace_bytes(...) returns what the path chosen for these parameters needs (0: the
 * scalar-atomic kernel runs and needs none).  NULL / too small -> the scalar-atomic kernel runs.  The plain
 * b200_roi_align_backward obtains the scratch with cudaMallocAsync/cudaFreeAsync on `stream`. */
B200_API size_t b200_roi_align_backward_workspace_bytes(int batch_size, int num_rois, int channels, int height, int width,
                                                        int aligned_height, int aligned_width, int sampling_ratio);
B200_API int b200_roi_align_backward_ws(const float* top_diff, float spatial_scale, int batch_size, int num_rois,
                               int height, int width, int channels, int aligned_height, int aligned_width,
                               int sampling_ratio, const float* bottom_rois, float* bottom_diff,
                               void* workspace, size_t workspace_bytes, b200_stream_t stream);

/* Indexed variants (SURVEY.md 8f N2: the FPN per-level loop + torch.cat + restore gather of
 * Generalized_RCNN.roi_feature_transform, lib/modeling/model_builder.py:264-303): RoI r reads / writes row
 * top_rows[r] of top_data / top_diff instead of row r, so the pooled features of every pyramid level land directly
 * in the restored order of one shared output tensor (and the backward picks its gradient rows out of the shared
 * tensor) -- no concatenated intermediate, no gather pass.  top_rows == NULL is the identity (= the _ws variants).
 * The forward writes exactly the rows named by top_rows; the caller sizes top_data. */
B200_API int b200_roi_align_forward_indexed(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                                   int height, int width, int channels, int aligned_height, int aligned_width,
                                   int sampling_ratio, const float* bottom_rois, const int* top_rows, float* top_data,
                                   void* workspace, size_t workspace_bytes, b200_stream_t stream);
B200_API int b200_roi_align_backward_indexed(const float* top_diff, const int* top_rows, float spatial_scale, int batch_size,
                                    int num_rois, int height, int width, int channels, int aligned_height,
                                    int aligned_width, int sampling_ratio, const float* bottom_rois, float* bottom_diff,
                                    void* workspace, size_t workspace_bytes, b200_stream_t stream);

/* ---- RoIAlign, legacy variant (one bilinear sample per lattice corner, fp64 interpolation) -----
 * replaces ROIAlignForwardLaucher / ROIAlignBackwardLaucher,
 *   lib/model/roi_align/src/roi_align_kernel.cu:73-91, 145-162 (header roi_align_kernel.h). */
B200_API int b200_roi_align_legacy_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                                  int height, int width, int channels, int aligned_height, int aligned_width,
                                  const float* bottom_rois, float* top_data, b200_stream_t stream);
B200_API int b200_roi_align_legacy_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois,
                                   int height, int width, int channels, int aligned_height, int aligned_width,
                                   const float* bottom_rois, float* bottom_diff, b200_stream_t stream);

/* ---- RoIPool -----------------------------------------------------------------------------------
 * replaces ROIPoolForwardLaucher / ROIPoolBackwardLaucher,
 *   lib/model/roi_pooling/src/roi_pooling_kernel.cu:95-125, 205-234 (header roi_pooling_kernel.h:8-18).
 * argmax_data: int32 (R, C, PH, PW), flat index into the WHOLE bottom tensor or -1; may be NULL in
 * the forward.  The backward is deterministic and bit-identical to the reference's gather. */
B200_API int b200_roi_pool_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                          int height, int width, int channels, int pooled_height, int pooled_width,
                          const float* bottom_rois, float* top_data, int* argmax_data, b200_stream_t stream);
B200_API int b200_roi_pool_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois,
                           int height, int width, int channels, int pooled_height, int pooled_width,
                           const float* bottom_rois, float* bottom_diff, const int* argmax_data,
                           b200_stream_t stream);

/* ---- RoICrop (bilinear sampler from an explicit grid) -----------------------------------------
 * replaces BilinearSamplerBHWD_updateOutput_cuda_kernel / _updateGradInput_cuda_kernel,
 *   lib/model/roi_crop/src/roi_crop_cuda_kernel.cu:201-255, 257-326 (header roi_crop_cuda_kernel.h:6-32).
 * image: (N, C, H, W); grids: (R, out_h, out_w, 2) with channel 0 = y, channel 1 = x in [-1, 1];
 * output: (R, C, out_h, out_w).  RoI b samples image b / (R / N) (kernel :64, :217).  Dense tensors
 * only (the reference took explicit strides; the Python layer makes inputs contiguous).
 * grad_grids (same shape as grids) is zero-filled when non-NULL: the reference CUDA kernel never
 * stores the grid gradient (:111-194), so the observable result is zeros. */
B200_API int b200_roi_crop_forward(const float* image, const float* grids, int batch_size, int channels, int height,
                          int width, int num_rois, int out_height, int out_width, float* output,
                          b200_stream_t stream);
B200_API int b200_roi_crop_backward(const float* grad_output, const float* grids, int batch_size, int channels,
                           int height, int width, int num_rois, int out_height, int out_width,
                           float* grad_image, float* grad_grids, b200_stream_t stream);
/* Same with caller-supplied scratch (the Python layer takes it from torch's caching allocator): when the image gradient goes
 * through the channel-innermost scratch image (vector reductions; C % 4 == 0 and enough taps) it needs
 * b200_roi_crop_backward_workspace_bytes() bytes -- 0 when the scalar-atomic kernel is used.  b200_roi_crop_backward obtains
 * the scratch with cudaMallocAsync / cudaFreeAsync on `stream`. */
B200_API size_t b200_roi_crop_backward_workspace_bytes(int batch_size, int channels, int height, int width, int num_rois,
                                                       int out_height, int out_width);
B200_API int b200_roi_crop_backward_ws(const float* grad_output, const float* grids, int batch_size, int channels, int height,
                                       int width, int num_rois, int out_height, int out_width, float* grad_image,
                                       float* grad_grids, void* workspace, size_t workspace_bytes, b200_stream_t stream);

/* ---- proposal NMS ------------------------------------------------------------------------------
 * replaces nms_cuda_compute, lib/model/nms/src/nms_cuda_kernel.cu:87-161 (header nms_cuda_kernel.h:5-6;
 * bound through nms_cuda, src/nms_cuda.c:8-19).
 * boxes_dev: (boxes_num, boxes_dim) fp32, ALREADY sorted by score (the function never sorts).
 * keep_out_dev: int32[boxes_num], receives the kept row indices in ascending order;
 * num_out_dev: int32[1], receives their count.  Unlike the reference (cudaMalloc/cudaFree, four
 * blocking memcpys, host-side greedy scan, legacy default stream) everything runs on `stream` with
 * no host round trip; scratch comes from the caller: `workspace` must hold at least
 * b200_nms_workspace_bytes(boxes_num) bytes (256-byte aligned). */
B200_API size_t b200_nms_workspace_bytes(int boxes_num);
B200_API int b200_nms(const float* boxes_dev, int boxes_num, int boxes_dim, float nms_overlap_thresh,
             int* keep_out_dev, int* num_out_dev, void* workspace, size_t workspace_bytes,
             b200_stream_t stream);

/* ---- RoIAlign over a feature pyramid in ONE launch sequence (SURVEY.md 8f N2) -------------------------------------
 * replaces the per-level loop + torch.cat + gather of Generalized_RCNN.roi_feature_transform,
 * lib/modeling/model_builder.py:264-303: `num_levels` feature maps (same batch size and channel count, any H x W), the
 * RoIs of all levels stored level-major in bottom_rois (level l owns rows level_roi_begin_host[l] .. [l + 1]), and
 * top_rows[r] = the row of top_data RoI r is written to (the inverse of the reference's restore permutation; NULL:
 * identity).  The four *_host arrays and bottom_data_host (device pointers of the maps) are HOST arrays read during the
 * call.  The quad-strip kernels walk the strip columns of every level; results are bit-identical to per-level
 * b200_roi_align_forward calls.  This call has no fallback: b200_roi_align_fpn_workspace_bytes(...) is the quad-strip
 * path's size alone, and it is 0 exactly when that path cannot run (sampling_ratio outside {1, 2}, PH or PW times
 * sampling_ratio above 32, more than 96 strip columns or more than 6144 rows summed over them (all levels and images),
 * more than 65535 RoIs, B200_ROI_ALIGN_PATH forced to generic / tiled / stream, B200_FPN_PATH=levels).  Then loop over
 * b200_roi_align_forward_indexed instead; b200_roi_align_forward_fpn returns B200_ROI_EWORKSPACE. */
B200_API size_t b200_roi_align_fpn_workspace_bytes(int num_levels, const int* heights_host, const int* widths_host,
                                                   int batch_size, int num_rois, int aligned_height, int aligned_width,
                                                   int sampling_ratio);
B200_API int b200_roi_align_forward_fpn(int num_levels, const float* const* bottom_data_host, const int* heights_host,
                                        const int* widths_host, const float* spatial_scales_host,
                                        const int* level_roi_begin_host, int batch_size, int num_rois, int channels,
                                        int aligned_height, int aligned_width, int sampling_ratio,
                                        const float* bottom_rois, const int* top_rows, float* top_data, void* workspace,
                                        size_t workspace_bytes, b200_stream_t stream);

/* Several independent NMS problems in ONE pair of launches (mask kernel over all problems' tiles, one scan CTA per
 * problem): the (image, FPN level) proposal sets of one step (lib/modeling/generate_proposals.py:91-99 runs them one
 * after the other on the host).  Problem p has counts_host[p] score-sorted rows, stored back to back in boxes_dev;
 * its kept indices (relative to its own first row) go to keep_out_dev + (sum of the counts before p), their number to
 * num_out_dev[p].  counts_host is a HOST array (the counts are launch geometry); 1 <= num_problems <= 64 and every
 * count <= ~13 800 (the pipelined scan's shared-memory limit), else B200_ROI_EINVAL -- loop over b200_nms then.
 * Results per problem are bit-identical to b200_nms. */
B200_API size_t b200_nms_batched_workspace_bytes(const int* counts_host, int num_problems);
B200_API int b200_nms_batched(const float* boxes_dev, const int* counts_host, int num_problems, int boxes_dim,
                              float nms_overlap_thresh, int* keep_out_dev, int* num_out_dev, void* workspace,
                              size_t workspace_bytes, b200_stream_t stream);

/* ---- test-time detection post-processing (SURVEY.md 8f N3) ------------------------------------------------------
 * The per-class problems of lib/core/test.py:732-790 (box_results_with_nms_and_limit), batched like b200_nms_batched:
 * problem p = the detections of one class, counts_host[p] rows of [x1, y1, x2, y2, score] stored back to back
 * (1 <= num_problems <= 128).  Classic NMS goes through b200_nms_batched.
 * b200_soft_nms_batched: lib/utils/cython_nms.pyx:98-203 step for step (method 1 linear, 2 gaussian, else hard), IN PLACE:
 *   afterwards problem p's first num_out_dev[p] rows are its surviving detections with decayed scores, in the
 *   reference's output order, and inds_out_dev holds their original row indices (relative to the problem).
 * b200_box_voting_batched: lib/utils/boxes.py:268-317; top_dets (the NMS survivors) are replaced in out_dev by the
 *   score-weighted average of all_dets rows with IoU >= thresh (cython_bbox.bbox_overlaps convention); scoring_method
 *   0 ID, 1 AVG, 2 IOU_AVG, 3 TEMP_AVG, 4 GENERALIZED_AVG, 5 QUASI_SUM. */
B200_API int b200_soft_nms_batched(float* dets_dev, const int* counts_host, int num_problems, float sigma, float overlap_thresh,
                                   float score_thresh, int method, int* inds_out_dev, int* num_out_dev, b200_stream_t stream);
B200_API int b200_box_voting_batched(const float* top_dets_dev, const int* top_counts_host, const float* all_dets_dev,
                                     const int* all_counts_host, int num_problems, float thresh, int scoring_method, float beta,
                                     float* out_dev, b200_stream_t stream);

/* ---- test-time mask paste (N3, masks) ----------------------------------------------------------------------------
 * replaces the per-detection host loop of segm_results, lib/core/test.py:793-847, with expand_boxes,
 * lib/utils/boxes.py:233-249 (cv2.resize + threshold + paste + pycocotools RLE encode).
 * Detection i: soft mask = channel mask_channel[i] of masks (num_dets, num_channels, resolution, resolution) fp32
 * (mask_channel: int32 device array, NULL = channel 0 for every detection; a channel outside [0, num_channels) gives an
 * empty mask); ref_boxes (num_dets, 4) fp32 (x1, y1, x2, y2) in image pixels.  The box is expanded by
 * (resolution + 2) / resolution in float32 and truncated to int32, the zero-padded mask is resized to it exactly like
 * cv2.resize(INTER_LINEAR) on float32 with IPP disabled, binarised with `value > thresh` and pasted into the box's window
 * clipped to the im_h x im_w image.  Limits: resolution <= 126, im_w <= 32768, im_h * im_w < 2^31, else B200_ROI_EINVAL.
 * b200_segm_paste      masks_out (num_dets, im_h, im_w) uint8, every byte written (1 inside the mask, 0 elsewhere).
 * b200_segm_rle_count  offsets_out: int64[num_dets + 1], the exclusive scan of the number of runs of each detection's
 *                      COCO uncompressed RLE (column-major image, run lengths alternating from a run of zeros, which
 *                      is 0 when pixel (0, 0) is set; they sum to im_h * im_w); offsets_out[num_dets] is the total.
 * b200_segm_rle_emit   runs_out: int32[offsets[num_dets]]; detection i's runs at runs_out + offsets[i].  `offsets` is
 *                      b200_segm_rle_count's output for the same arguments.
 * Each entry point launches a fixed number of kernels whatever num_dets is (paste 1, count 2, emit 1), none for
 * num_dets == 0. */
B200_API int b200_segm_paste(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets,
                             int num_channels, int resolution, int im_h, int im_w, float thresh, unsigned char* masks_out_dev,
                             b200_stream_t stream);
B200_API int b200_segm_rle_count(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets,
                                 int num_channels, int resolution, int im_h, int im_w, float thresh, long long* offsets_out_dev,
                                 b200_stream_t stream);
B200_API int b200_segm_rle_emit(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets,
                                int num_channels, int resolution, int im_h, int im_w, float thresh, const long long* offsets_dev,
                                int* runs_out_dev, b200_stream_t stream);

/* ---- introspection used by the benchmark / tests (no compute) ----------------------------------
 * Number of kernel launches the library has enqueued since load (all entry points). */
B200_API unsigned long long b200_roi_ops_launch_count(void);
/* Path-selection switches (A/B runs and tests): name is one of "B200_ROI_ALIGN_PATH" (auto|generic|tiled|stream|quad),
 * "B200_ROI_ALIGN_BWD_PATH" (auto|generic|nhwc|rows), "B200_ROI_ALIGN_BWD_CPL" (4|2), "B200_FWD_ZERO" (dense|bins),
 * "B200_NMS_SCAN" (resolver|simple), "B200_STREAM_STAGE" (tma|async|regs), "B200_STREAM_PHASES" (all|prepass: timing probe), "B200_STRIP_ROWCOST" (0..9),
 * "B200_STRIP_PDL" (1|0), "B200_FPN_PATH" (fused|levels);
 * value NULL or "" restores the default.  Each switch takes its initial value from the
 * environment variable of the same name, read once at first use -- no entry point calls getenv() on the hot path.
 * Returns 0, or B200_ROI_EINVAL for an unknown name. */
B200_API int b200_roi_ops_set_option(const char* name, const char* value);
/* Debug: register (or clear with NULL) a device buffer of 8 x uint64 into which the tiled RoIAlign forward
 * adds per-warp clock64 deltas [staging, compute, end-of-item wait, warp-items, RoI items, 8-bin groups, max compute]. */
B200_API void b200_roi_ops_debug_timing_buffer(void* device_u64x16);

/* ---- RPN proposal decode (SURVEY.md 8f N1: the GPU-resident proposal layer) --------------------------------
 * replaces the numpy block of GenerateProposalsOp.proposals_for_one_image, lib/modeling/generate_proposals.py:108-150
 * (gather by score order, utils.boxes.bbox_transform :157-196, clip_tiled_boxes :138-154, _filter_boxes :171-182),
 * for candidates that were selected and sorted on the device.  `order` holds indices into the (H, W, A)-flattened
 * score map, best first; row t of dets_out is (x1, y1, x2, y2, score) ready for b200_nms, or the degenerate box
 * (0, 0, -1, -1, score) with valid_out[t] = 0 when the size / centre filter rejects the candidate (such rows cannot
 * interact with any box in NMS; the caller drops them afterwards).  min_size is already multiplied by im_info[2]. */
B200_API int b200_proposal_decode(const float* bbox_deltas, const float* anchors, const long long* order, const float* scores,
                         int num_candidates, int num_anchors, int height, int width, float feat_stride, float im_height,
                         float im_width, float min_size, float* dets_out, int* valid_out, b200_stream_t stream);

/* ---- batched top-k of RPN score maps (SURVEY.md 8f N1) ----------------------------------------------------------
 * replaces np.argpartition + np.argsort of lib/modeling/generate_proposals.py:118-131 (and the torch.topk / torch.sort the
 * first device version used): problem p is one (A_p, H_p * W_p) float32 score map on the device, read where it lies;
 * order_out receives, best first, the k_p indices into its (H, W, A) flattening (what b200_proposal_decode takes as
 * `order`), scores_out the scores; problems are stored back to back.  <= 64 problems, k_p <= 16384 (else
 * B200_ROI_EWORKSPACE: the caller sorts by other means).  Equal scores come out in ascending index; which of several
 * scores EQUAL TO THE k-th are taken is deterministic (memory order), the reference leaves it unspecified.
 * Radix select (3 histogram launches, chunk-parallel) + one collect-and-sort launch; no host read. */
B200_API size_t b200_topk_batched_workspace_bytes(int num_problems);
B200_API int b200_topk_batched(const float* const* scores_dev_ptrs_host, const int* num_anchors_host, const int* num_cells_host,
                               const int* k_host, int num_problems, long long* order_out_dev, float* scores_out_dev, void* workspace,
                               size_t workspace_bytes, b200_stream_t stream);

/* ---- RoI label / regression-target generation on the device (SURVEY.md 8f N4) ---------------------------------
 * The per-image host work of the reference's training data path, for proposals that already live on the GPU.  Boxes are
 * float32 (x1, y1, x2, y2) rows in image pixels, exactly the roidb's `boxes`.
 * b200_bbox_overlaps    lib/utils/cython_bbox.pyx:32-73: (N, K) IoU with the +1 pixel convention, bit-exact float32.
 * b200_roi_assign       lib/datasets/json_dataset.py:429-463 + :514-531 without the (N, K) matrix: per box the best
 *                       ground-truth overlap (0 when none is positive), its index (first maximum; -1) and class (0).
 * b200_roi_select       lib/roi_data/fast_rcnn.py:138-151: ascending index lists of the foreground (>= fg_thresh) and
 *                       background ([bg_lo, bg_hi)) boxes, counts_out = {num_fg, num_bg}.
 * b200_fast_rcnn_targets  fast_rcnn.py:161-187 + :203-248 for the kept rows (the first num_fg are foreground): labels
 *                       (int32), rois (batch_idx, box * im_scale), regression targets (utils/boxes.py:199-230) expanded
 *                       to 4 * num_reg_classes columns, inside / outside weights.  bbox_reg_weights_host: 4 floats. */
B200_API int b200_bbox_overlaps(const float* boxes_dev, int num_boxes, const float* query_boxes_dev, int num_query,
                                float* overlaps_out_dev, b200_stream_t stream);
B200_API int b200_roi_assign(const float* boxes_dev, int num_boxes, const float* gt_boxes_dev, const int* gt_classes_dev, int num_gt,
                             float* max_overlaps_out_dev, int* argmax_out_dev, int* max_classes_out_dev, b200_stream_t stream);
B200_API int b200_roi_select(const float* max_overlaps_dev, int num_boxes, float fg_thresh, float bg_thresh_hi, float bg_thresh_lo,
                             int* fg_inds_out_dev, int* bg_inds_out_dev, int* counts_out_dev, b200_stream_t stream);
B200_API int b200_fast_rcnn_targets(const float* boxes_dev, const float* gt_boxes_dev, const int* argmax_dev, const int* max_classes_dev,
                                    const int* keep_inds_dev, int num_keep, int num_fg, const float* bbox_reg_weights_host,
                                    int num_reg_classes, int cls_agnostic, float im_scale, float batch_idx, int* labels_out_dev,
                                    float* rois_out_dev, float* bbox_targets_out_dev, float* inside_weights_out_dev,
                                    float* outside_weights_out_dev, b200_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200_ROI_OPS_H_ */
