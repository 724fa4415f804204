// api.cu -- the extern "C" boundary of libb200_roi_ops.so (see include/b200_roi_ops.h).
// Argument validation + dispatch only; kernels live in the per-op translation units.
#include "common.cuh"
#include <mutex>
#include <stdlib.h>
#include <string.h>

namespace b200 {
unsigned long long g_launch_count = 0;

static const char* const kOptionNames[kNumOptions] = {"B200_ROI_ALIGN_PATH", "B200_ROI_ALIGN_BWD_PATH", "B200_ROI_ALIGN_BWD_CPL",
                                                      "B200_FWD_ZERO", "B200_NMS_SCAN", "B200_STREAM_STAGE", "B200_STREAM_PHASES",
                                                      "B200_FPN_PATH", "B200_STRIP_ROWCOST", "B200_STRIP_PDL", "B200_BWD_TRCH"};
static int g_options[kNumOptions];
static std::once_flag g_options_once;

static void options_init() {
    for (int i = 0; i < kNumOptions; ++i) {
        const char* e = getenv(kOptionNames[i]);
        __atomic_store_n(&g_options[i], e ? (int)(unsigned char)e[0] : 0, __ATOMIC_RELAXED);
    }
}

int option_get(Option which) {
    std::call_once(g_options_once, options_init);
    return __atomic_load_n(&g_options[which], __ATOMIC_RELAXED);
}

static int option_set(const char* name, const char* value) {
    std::call_once(g_options_once, options_init);
    if (!name) return B200_ROI_EINVAL;
    for (int i = 0; i < kNumOptions; ++i)
        if (strcmp(name, kOptionNames[i]) == 0) {
            __atomic_store_n(&g_options[i], value ? (int)(unsigned char)value[0] : 0, __ATOMIC_RELAXED);
            return B200_ROI_OK;
        }
    return B200_ROI_EINVAL;
}

int roi_align_forward_generic(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, cudaStream_t);
int roi_align_backward_generic(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, cudaStream_t);
int roi_align_legacy_forward(const float*, float, int, int, int, int, int, int, int, const float*, float*, cudaStream_t);
int roi_align_legacy_backward(const float*, float, int, int, int, int, int, int, int, const float*, float*, cudaStream_t);
int roi_pool_forward(const float*, float, int, int, int, int, int, int, int, const float*, float*, int*, cudaStream_t);
int roi_pool_backward(const float*, float, int, int, int, int, int, int, int, const float*, float*, const int*, cudaStream_t);
int roi_crop_forward(const float*, const float*, int, int, int, int, int, int, int, float*, cudaStream_t);
int roi_crop_backward(const float*, const float*, int, int, int, int, int, int, int, float*, float*, void*, size_t, cudaStream_t);
size_t roi_crop_backward_workspace_bytes(int, int, int, int, int, int, int);
size_t nms_workspace_bytes(int);
int proposal_decode(const float*, const float*, const long long*, const float*, int, int, int, int, float, float, float, float, float*, int*, cudaStream_t);
size_t roi_align_tiled_workspace_bytes(int, int, int, int, int, int, int);
void roi_align_tiled_set_timing_buffer(unsigned long long*);
void nms_set_timing_buffer(unsigned long long*);
void roi_align_stream_set_debug_buffer(unsigned long long*);
int roi_align_forward_tiled(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, void*, size_t, cudaStream_t);
size_t roi_align_stream_workspace_bytes(int, int, int, int, int, int, int);
int roi_align_forward_stream(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, void*, size_t, cudaStream_t);
size_t roi_align_strip_workspace_bytes(int, int, int, int, int, int, int);
size_t roi_align_strip_fpn_workspace_bytes(int, const int*, const int*, int, int, int, int, int);
int roi_align_forward_strip_fpn(int, const float* const*, const int*, const int*, const float*, const int*, int, int, int, int, int, int,
                                const float*, float*, const int*, void*, size_t, cudaStream_t);
int roi_align_forward_strip(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, void*, size_t, cudaStream_t);
void roi_align_strip_set_debug_buffer(unsigned long long*);

size_t topk_batched_workspace_bytes(int);
int topk_batched(const float* const*, const int*, const int*, const int*, int, long long*, float*, void*, size_t, cudaStream_t);
int bbox_overlaps(const float*, int, const float*, int, float*, cudaStream_t);
int roi_assign(const float*, int, const float*, const int*, int, float*, int*, int*, cudaStream_t);
int roi_select(const float*, int, float, float, float, int*, int*, int*, cudaStream_t);
int fast_rcnn_targets(const float*, const float*, const int*, const int*, const int*, int, int, const float*, int, int, float, float, int*,
                      float*, float*, float*, float*, cudaStream_t);

// B200_ROI_ALIGN_PATH=generic|tiled|stream|auto (default auto) -- test/benchmark override of the forward dispatch
//   0 auto: quad-strip path -> streaming-strip path -> tiled path -> generic, each when it applies
//   1 generic only; 2 tiled (-> generic); 3 stream (-> generic); 4 quad strip (-> generic)
static int forward_path_mode() {
    const int e = option_get(kOptFwdPath);
    if (e == 'g') return 1;
    if (e == 't') return 2;
    if (e == 's') return 3;
    if (e == 'q') return 4;
    return 0;
}

static size_t forward_workspace_bytes(int mode, int N, int R, int H, int W, int PH, int PW, int sr) {
    if (mode == 1) return 0;
    const size_t a = (mode == 3 || mode == 0) ? roi_align_stream_workspace_bytes(N, R, H, W, PH, PW, sr) : 0;
    const size_t b = (mode == 2 || mode == 0) ? roi_align_tiled_workspace_bytes(N, R, H, W, PH, PW, sr) : 0;
    const size_t c = (mode == 4 || mode == 0) ? roi_align_strip_workspace_bytes(N, R, H, W, PH, PW, sr) : 0;
    const size_t ab = a > b ? a : b;
    return ab > c ? ab : c;
}

static bool tiled_pays_off(int R, int C, int H, int W, int PH, int PW) {
    // the fast paths stream the whole map and pay a ~15 us prepass; they win once the gather volume dwarfs both
    // (measured r03e: BASELINE cfg1, 0.4 M outputs, 32 us through the streaming path vs ~10 us generic)
    const long long outputs = (long long)R * C * PH * PW;
    return outputs >= 1500000LL && (long long)H * W >= 1024;
}
int nms(const float*, int, int, float, int*, int*, void*, size_t, cudaStream_t);
size_t nms_batched_workspace_bytes(const int*, int);
int soft_nms_batched(float*, const int*, int, float, float, float, int, int*, int*, cudaStream_t);
int box_voting_batched(const float*, const int*, const float*, const int*, int, float, int, float, float*, cudaStream_t);
int nms_batched(const float*, const int*, int, int, float, int*, int*, void*, size_t, cudaStream_t);
bool segm_args_ok(int, int, int, int, int);
int segm_paste(const float*, const int*, const float*, int, int, int, int, int, float, unsigned char*, cudaStream_t);
int segm_rle_count(const float*, const int*, const float*, int, int, int, int, int, float, long long*, cudaStream_t);
int segm_rle_emit(const float*, const int*, const float*, int, int, int, int, int, float, const long long*, int*, cudaStream_t);
size_t roi_align_bwd_nhwc_workspace_bytes(int, int, int, int);
int roi_align_backward_nhwc(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, void*, size_t, cudaStream_t);

size_t roi_align_bwd_rows_workspace_bytes(int, int, int, int, int, int, int, int);
int roi_align_backward_rows(const float*, float, int, int, int, int, int, int, int, int, const float*, float*, const int*, void*, size_t, cudaStream_t);

// B200_ROI_ALIGN_BWD_PATH=generic|nhwc|rows|auto
static int backward_path_mode() {
    const int e = option_get(kOptBwdPath);
    if (e == 'g') return 1;
    if (e == 'n') return 2;
    if (e == 'r') return 3;
    return 0;
}

static bool nhwc_pays_off(int N, int R, int C, int H, int W, int PH, int PW, int sr) {
    // fixed cost: zero + transpose the whole map; gain: 4x fewer L2 reduction ops
    if (sr < 1 || (C & 3)) return false;
    const long long taps = (long long)R * C * PH * PW * sr * sr * 4;
    return taps >= 2LL * N * C * H * W;
}

// 0: generic (scalar atomics), 2: NHWC vector reductions, 3: row-stationary gather
static int backward_path_choice(int N, int R, int C, int H, int W, int PH, int PW, int sr) {
    const int mode = backward_path_mode();
    if (mode == 1 || R <= 0) return 0;
    const bool pays = nhwc_pays_off(N, R, C, H, W, PH, PW, sr);
    bool rows_ok = roi_align_bwd_rows_workspace_bytes(N, R, C, H, W, PH, PW, sr) > 0;
    if (rows_ok && mode != 3) {
        // The gather path's parallelism is (image rows) x (32-cell tiles) x (128-channel blocks) warp items, each walking
        // every unit of its row: few rows with many RoIs (FPN P4 / P5 with a thousand boxes, measured r03e: 315 us / 1 ms)
        // leave most of the 1776 resident warps idle behind a few very long items.
        const long long items = (long long)N * H * ((W + 31) / 32) * ((C + 127) / 128);
        const long long units_per_row = 2LL * R * PH * (sr > 0 ? sr : 1) / ((long long)N * H);
        if (items < 1200 || units_per_row > 160) rows_ok = false;
        if (PW != 7) rows_ok = false;       // 14 x 14 (mask head): 675 us through the gather path vs 530 us reference at P2, R = 256 (r03f)
    }
    if (mode == 3) return rows_ok ? 3 : 0;
    if (mode == 2) return 2;
    if (rows_ok && pays) return 3;
    return pays ? 2 : 0;
}

static inline bool bad_dims(int N, int R, int H, int W, int C, int PH, int PW) {
    return N < 0 || R < 0 || H <= 0 || W <= 0 || C < 0 || PH <= 0 || PW <= 0;
}
}  // namespace b200

using namespace b200;

extern "C" {

int b200_roi_ops_abi_version(void) { return 3; }

const char* b200_roi_ops_strerror(int status) {
    if (status == B200_ROI_OK) return "success";
    if (status == B200_ROI_EINVAL) return "b200_roi_ops: invalid argument (null pointer, negative or zero dimension)";
    if (status == B200_ROI_EWORKSPACE) return "b200_roi_ops: workspace missing or smaller than b200_nms_workspace_bytes()";
    if (status > 0) return cudaGetErrorString((cudaError_t)status);
    return "b200_roi_ops: unknown status";
}

unsigned long long b200_roi_ops_launch_count(void) { return g_launch_count; }

int b200_roi_ops_set_option(const char* name, const char* value) { return option_set(name, value); }

void b200_roi_ops_debug_timing_buffer(void* device_u64x16) {
    roi_align_tiled_set_timing_buffer((unsigned long long*)device_u64x16);
    nms_set_timing_buffer((unsigned long long*)device_u64x16);
    roi_align_stream_set_debug_buffer((unsigned long long*)device_u64x16);      // -DB200_STREAM_DEBUG builds only
    roi_align_strip_set_debug_buffer((unsigned long long*)device_u64x16);       // watchdog records of the quad-strip path
}

size_t b200_roi_align_workspace_bytes(int batch_size, int num_rois, int height, int width, int aligned_height,
                                      int aligned_width, int sampling_ratio) {
    if (batch_size <= 0 || num_rois <= 0 || height <= 0 || width <= 0 || aligned_height <= 0 || aligned_width <= 0) return 0;
    return forward_workspace_bytes(forward_path_mode(), batch_size, num_rois, height, width, aligned_height, aligned_width, sampling_ratio);
}

int b200_roi_align_forward_ws(const float* bottom_data, float spatial_scale, int batch_size, int num_rois, int height,
                              int width, int channels, int aligned_height, int aligned_width, int sampling_ratio,
                              const float* bottom_rois, float* top_data, void* workspace, size_t workspace_bytes,
                              b200_stream_t stream) {
    return b200_roi_align_forward_indexed(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                          aligned_height, aligned_width, sampling_ratio, bottom_rois, nullptr, top_data,
                                          workspace, workspace_bytes, stream);
}

int b200_roi_align_forward_indexed(const float* bottom_data, float spatial_scale, int batch_size, int num_rois, int height,
                                   int width, int channels, int aligned_height, int aligned_width, int sampling_ratio,
                                   const float* bottom_rois, const int* top_rows, float* top_data, void* workspace,
                                   size_t workspace_bytes, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if (num_rois > 0 && channels > 0 && (!bottom_data || !bottom_rois || !top_data)) return B200_ROI_EINVAL;
    const int mode = forward_path_mode();
    const bool pays = tiled_pays_off(num_rois, channels, height, width, aligned_height, aligned_width);
    if (workspace != nullptr && (mode == 4 || (mode == 0 && pays))) {
        const int rc = roi_align_forward_strip(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                               aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, top_rows,
                                               workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != 1000) return rc;
    }
    if (workspace != nullptr && (mode == 3 || (mode == 0 && pays))) {
        const int rc = roi_align_forward_stream(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                                aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, top_rows,
                                                workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != 1000) return rc;
    }
    if (workspace != nullptr && (mode == 2 || (mode == 0 && pays))) {
        const int rc = roi_align_forward_tiled(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                               aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, top_rows,
                                               workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != 1000) return rc;
    }
    return roi_align_forward_generic(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                     aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, top_rows,
                                     (cudaStream_t)stream);
}

int b200_roi_align_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois, int height,
                           int width, int channels, int aligned_height, int aligned_width, int sampling_ratio,
                           const float* bottom_rois, float* top_data, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if (num_rois > 0 && channels > 0 && (!bottom_data || !bottom_rois || !top_data)) return B200_ROI_EINVAL;
    const int mode = forward_path_mode();
    const size_t wsb = (num_rois > 0) ? forward_workspace_bytes(mode, batch_size, num_rois, height, width, aligned_height, aligned_width,
                                                                sampling_ratio) : 0;
    if (wsb > 0 && (mode >= 2 || tiled_pays_off(num_rois, channels, height, width, aligned_height, aligned_width))) {
        void* ws = nullptr;
        if (cudaMallocAsync(&ws, wsb, (cudaStream_t)stream) == cudaSuccess) {
            const int rc = b200_roi_align_forward_ws(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                                     aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, ws,
                                                     wsb, stream);
            cudaFreeAsync(ws, (cudaStream_t)stream);
            return rc;
        }
        (void)cudaGetLastError();
    }
    return roi_align_forward_generic(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                     aligned_height, aligned_width, sampling_ratio, bottom_rois, top_data, nullptr,
                                     (cudaStream_t)stream);
}

size_t b200_roi_align_backward_workspace_bytes(int batch_size, int num_rois, int channels, int height, int width,
                                               int aligned_height, int aligned_width, int sampling_ratio) {
    if (batch_size <= 0 || num_rois <= 0 || channels <= 0 || height <= 0 || width <= 0 || aligned_height <= 0 || aligned_width <= 0) return 0;
    const int path = backward_path_choice(batch_size, num_rois, channels, height, width, aligned_height, aligned_width, sampling_ratio);
    if (path == 3) return roi_align_bwd_rows_workspace_bytes(batch_size, num_rois, channels, height, width, aligned_height, aligned_width, sampling_ratio);
    if (path == 2) return roi_align_bwd_nhwc_workspace_bytes(batch_size, channels, height, width);
    return 0;
}

int b200_roi_align_backward_ws(const float* top_diff, float spatial_scale, int batch_size, int num_rois, int height,
                               int width, int channels, int aligned_height, int aligned_width, int sampling_ratio,
                               const float* bottom_rois, float* bottom_diff, void* workspace, size_t workspace_bytes,
                               b200_stream_t stream) {
    return b200_roi_align_backward_indexed(top_diff, nullptr, spatial_scale, batch_size, num_rois, height, width, channels,
                                           aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff, workspace,
                                           workspace_bytes, stream);
}

int b200_roi_align_backward_indexed(const float* top_diff, const int* top_rows, float spatial_scale, int batch_size,
                                    int num_rois, int height, int width, int channels, int aligned_height, int aligned_width,
                                    int sampling_ratio, const float* bottom_rois, float* bottom_diff, void* workspace,
                                    size_t workspace_bytes, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!bottom_diff || (num_rois > 0 && (!top_diff || !bottom_rois))) return B200_ROI_EINVAL;
    int path = (workspace != nullptr) ? backward_path_choice(batch_size, num_rois, channels, height, width, aligned_height, aligned_width, sampling_ratio) : 0;
    if (path == 3) {
        const int rc = roi_align_backward_rows(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                               aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff,
                                               top_rows, workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != 1000) return rc;
        path = 2;                                   // workspace too small for the gather path: try the NHWC one
    }
    if (path == 2) {
        const int rc = roi_align_backward_nhwc(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                               aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff,
                                               top_rows, workspace, workspace_bytes, (cudaStream_t)stream);
        if (rc != 1000) return rc;
    }
    return roi_align_backward_generic(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                      aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff, top_rows,
                                      (cudaStream_t)stream);
}

int b200_roi_align_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois, int height,
                            int width, int channels, int aligned_height, int aligned_width, int sampling_ratio,
                            const float* bottom_rois, float* bottom_diff, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!bottom_diff || (num_rois > 0 && (!top_diff || !bottom_rois))) return B200_ROI_EINVAL;
    const size_t wsb = b200_roi_align_backward_workspace_bytes(batch_size, num_rois, channels, height, width, aligned_height,
                                                               aligned_width, sampling_ratio);
    if (wsb > 0) {
        void* ws = nullptr;
        if (cudaMallocAsync(&ws, wsb, (cudaStream_t)stream) == cudaSuccess) {
            const int rc = b200_roi_align_backward_ws(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                                      aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff,
                                                      ws, wsb, stream);
            cudaFreeAsync(ws, (cudaStream_t)stream);
            return rc;
        }
        (void)cudaGetLastError();
    }
    return roi_align_backward_generic(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                      aligned_height, aligned_width, sampling_ratio, bottom_rois, bottom_diff, nullptr,
                                      (cudaStream_t)stream);
}

int b200_proposal_decode(const float* bbox_deltas, const float* anchors, const long long* order, const float* scores,
                         int num_candidates, int num_anchors, int height, int width, float feat_stride, float im_height,
                         float im_width, float min_size, float* dets_out, int* valid_out, b200_stream_t stream) {
    if (num_candidates < 0 || num_anchors <= 0 || height <= 0 || width <= 0) return B200_ROI_EINVAL;
    if (num_candidates > 0 && (!bbox_deltas || !anchors || !order || !scores || !dets_out || !valid_out)) return B200_ROI_EINVAL;
    return proposal_decode(bbox_deltas, anchors, order, scores, num_candidates, num_anchors, height, width, feat_stride,
                           im_height, im_width, min_size, dets_out, valid_out, (cudaStream_t)stream);
}

int b200_roi_align_legacy_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois,
                                  int height, int width, int channels, int aligned_height, int aligned_width,
                                  const float* bottom_rois, float* top_data, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if (num_rois > 0 && channels > 0 && (!bottom_data || !bottom_rois || !top_data)) return B200_ROI_EINVAL;
    return roi_align_legacy_forward(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels,
                                    aligned_height, aligned_width, bottom_rois, top_data, (cudaStream_t)stream);
}

int b200_roi_align_legacy_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois,
                                   int height, int width, int channels, int aligned_height, int aligned_width,
                                   const float* bottom_rois, float* bottom_diff, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, aligned_height, aligned_width)) return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!bottom_diff || (num_rois > 0 && (!top_diff || !bottom_rois))) return B200_ROI_EINVAL;
    return roi_align_legacy_backward(top_diff, spatial_scale, batch_size, num_rois, height, width, channels,
                                     aligned_height, aligned_width, bottom_rois, bottom_diff, (cudaStream_t)stream);
}

int b200_roi_pool_forward(const float* bottom_data, float spatial_scale, int batch_size, int num_rois, int height,
                          int width, int channels, int pooled_height, int pooled_width, const float* bottom_rois,
                          float* top_data, int* argmax_data, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, pooled_height, pooled_width)) return B200_ROI_EINVAL;
    if (num_rois > 0 && channels > 0 && (!bottom_data || !bottom_rois || !top_data)) return B200_ROI_EINVAL;
    return roi_pool_forward(bottom_data, spatial_scale, batch_size, num_rois, height, width, channels, pooled_height,
                            pooled_width, bottom_rois, top_data, argmax_data, (cudaStream_t)stream);
}

int b200_roi_pool_backward(const float* top_diff, float spatial_scale, int batch_size, int num_rois, int height,
                           int width, int channels, int pooled_height, int pooled_width, const float* bottom_rois,
                           float* bottom_diff, const int* argmax_data, b200_stream_t stream) {
    if (bad_dims(batch_size, num_rois, height, width, channels, pooled_height, pooled_width)) return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!bottom_diff || (num_rois > 0 && (!top_diff || !bottom_rois || !argmax_data))) return B200_ROI_EINVAL;
    return roi_pool_backward(top_diff, spatial_scale, batch_size, num_rois, height, width, channels, pooled_height,
                             pooled_width, bottom_rois, bottom_diff, argmax_data, (cudaStream_t)stream);
}

int b200_roi_crop_forward(const float* image, const float* grids, int batch_size, int channels, int height, int width,
                          int num_rois, int out_height, int out_width, float* output, b200_stream_t stream) {
    if (batch_size < 0 || channels < 0 || height <= 0 || width <= 0 || num_rois < 0 || out_height < 0 || out_width < 0)
        return B200_ROI_EINVAL;
    if ((size_t)num_rois * out_height * out_width * channels > 0 && (!image || !grids || !output)) return B200_ROI_EINVAL;
    return roi_crop_forward(image, grids, batch_size, channels, height, width, num_rois, out_height, out_width, output,
                            (cudaStream_t)stream);
}

int b200_roi_crop_backward(const float* grad_output, const float* grids, int batch_size, int channels, int height,
                           int width, int num_rois, int out_height, int out_width, float* grad_image,
                           float* grad_grids, b200_stream_t stream) {
    if (batch_size < 0 || channels < 0 || height <= 0 || width <= 0 || num_rois < 0 || out_height < 0 || out_width < 0)
        return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!grad_image) return B200_ROI_EINVAL;
    if ((size_t)num_rois * out_height * out_width > 0 && (!grad_output || !grids)) return B200_ROI_EINVAL;
    return roi_crop_backward(grad_output, grids, batch_size, channels, height, width, num_rois, out_height, out_width,
                             grad_image, grad_grids, nullptr, 0, (cudaStream_t)stream);
}

size_t b200_roi_crop_backward_workspace_bytes(int batch_size, int channels, int height, int width, int num_rois, int out_height,
                                              int out_width) {
    if (batch_size <= 0 || channels <= 0 || height <= 0 || width <= 0 || num_rois <= 0 || out_height <= 0 || out_width <= 0) return 0;
    return roi_crop_backward_workspace_bytes(batch_size, channels, height, width, num_rois, out_height, out_width);
}

int b200_roi_crop_backward_ws(const float* grad_output, const float* grids, int batch_size, int channels, int height, int width,
                              int num_rois, int out_height, int out_width, float* grad_image, float* grad_grids, void* workspace,
                              size_t workspace_bytes, b200_stream_t stream) {
    if (batch_size < 0 || channels < 0 || height <= 0 || width <= 0 || num_rois < 0 || out_height < 0 || out_width < 0)
        return B200_ROI_EINVAL;
    if ((size_t)batch_size * channels == 0) return B200_ROI_OK;
    if (!grad_image) return B200_ROI_EINVAL;
    if ((size_t)num_rois * out_height * out_width > 0 && (!grad_output || !grids)) return B200_ROI_EINVAL;
    return roi_crop_backward(grad_output, grids, batch_size, channels, height, width, num_rois, out_height, out_width,
                             grad_image, grad_grids, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t b200_nms_workspace_bytes(int boxes_num) { return nms_workspace_bytes(boxes_num); }

int b200_nms(const float* boxes_dev, int boxes_num, int boxes_dim, float nms_overlap_thresh, int* keep_out_dev,
             int* num_out_dev, void* workspace, size_t workspace_bytes, b200_stream_t stream) {
    if (!num_out_dev || (boxes_num > 0 && (!boxes_dev || !keep_out_dev))) return B200_ROI_EINVAL;
    return nms(boxes_dev, boxes_num, boxes_dim, nms_overlap_thresh, keep_out_dev, num_out_dev, workspace,
               workspace_bytes, (cudaStream_t)stream);
}

// The pyramid call runs the quad-strip path only, so its size is the only one that counts: 0 (the caller loops over the
// levels) whenever that path would reject the geometry or the forward is forced onto another path.
size_t b200_roi_align_fpn_workspace_bytes(int num_levels, const int* heights_host, const int* widths_host, int batch_size, int num_rois,
                                          int aligned_height, int aligned_width, int sampling_ratio) {
    const int mode = forward_path_mode();
    if (num_levels < 1 || !heights_host || !widths_host || batch_size <= 0 || num_rois <= 0 || (mode != 0 && mode != 4) ||
        option_get(kOptFpnPath) == 'l')
        return 0;
    return roi_align_strip_fpn_workspace_bytes(num_levels, heights_host, widths_host, batch_size, num_rois, aligned_height, aligned_width,
                                               sampling_ratio);
}

int b200_roi_align_forward_fpn(int num_levels, const float* const* bottom_data_host, const int* heights_host, const int* widths_host,
                               const float* spatial_scales_host, const int* level_roi_begin_host, int batch_size, int num_rois,
                               int channels, int aligned_height, int aligned_width, int sampling_ratio, const float* bottom_rois,
                               const int* top_rows, float* top_data, void* workspace, size_t workspace_bytes, b200_stream_t stream) {
    if (num_levels < 1 || num_levels > 6 || !bottom_data_host || !heights_host || !widths_host || !spatial_scales_host || !level_roi_begin_host)
        return B200_ROI_EINVAL;
    if (batch_size <= 0 || num_rois <= 0 || channels <= 0 || aligned_height <= 0 || aligned_width <= 0 || !bottom_rois || !top_data)
        return B200_ROI_EINVAL;
    if (level_roi_begin_host[0] != 0 || level_roi_begin_host[num_levels] != num_rois) return B200_ROI_EINVAL;
    for (int l = 0; l < num_levels; ++l)
        if (!bottom_data_host[l] || level_roi_begin_host[l + 1] < level_roi_begin_host[l]) return B200_ROI_EINVAL;
    int rc = 1000;
    const int mode = forward_path_mode();
    if ((mode == 0 || mode == 4) && option_get(kOptFpnPath) != 'l') {
        // Levels that TMA can stage (W % 4 == 0, 16-byte aligned base) and levels that need the cp.async producers (FPN P5 of an
        // 800 x 1333 image: W = 42) go to separate launch sequences: runs of consecutive levels of the same kind, each over its
        // own contiguous range of the level-major RoIs.  The workspace is reused (stream order).
        const int bins = aligned_height * aligned_width;
        int l0 = 0;
        rc = B200_ROI_OK;
        while (l0 < num_levels && rc == B200_ROI_OK) {
            auto tma_ok = [&](int l) { return (widths_host[l] & 3) == 0 && ((uintptr_t)bottom_data_host[l] & 15u) == 0; };
            int l1 = l0 + 1;
            while (l1 < num_levels && tma_ok(l1) == tma_ok(l0)) ++l1;
            const int r0 = level_roi_begin_host[l0], r1 = level_roi_begin_host[l1];
            if (r1 > r0) {
                int begin[8];
                for (int l = l0; l <= l1; ++l) begin[l - l0] = level_roi_begin_host[l] - r0;
                rc = roi_align_forward_strip_fpn(l1 - l0, bottom_data_host + l0, heights_host + l0, widths_host + l0, spatial_scales_host + l0,
                                                 begin, batch_size, r1 - r0, channels, aligned_height, aligned_width, sampling_ratio,
                                                 bottom_rois + (size_t)5 * r0, top_rows ? top_data : top_data + (size_t)r0 * channels * bins,
                                                 top_rows ? top_rows + r0 : nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
            }
            l0 = l1;
        }
        if (rc != B200_ROI_OK && rc != 1000) return rc;
    }
    return rc == 1000 ? B200_ROI_EWORKSPACE : rc;
}

size_t b200_nms_batched_workspace_bytes(const int* counts_host, int num_problems) {
    if (!counts_host) return 0;
    return nms_batched_workspace_bytes(counts_host, num_problems);
}

int b200_nms_batched(const float* boxes_dev, const int* counts_host, int num_problems, int boxes_dim, float nms_overlap_thresh,
                     int* keep_out_dev, int* num_out_dev, void* workspace, size_t workspace_bytes, b200_stream_t stream) {
    if (!counts_host || num_problems < 1 || !num_out_dev) return B200_ROI_EINVAL;
    long long total = 0;
    for (int p = 0; p < num_problems && p < 64; ++p) total += counts_host[p] > 0 ? counts_host[p] : 0;
    if (total > 0 && (!boxes_dev || !keep_out_dev)) return B200_ROI_EINVAL;
    const int rc = nms_batched(boxes_dev, counts_host, num_problems, boxes_dim, nms_overlap_thresh, keep_out_dev, num_out_dev, workspace,
                               workspace_bytes, (cudaStream_t)stream);
    return rc == 1000 ? B200_ROI_EINVAL : rc;
}

int b200_soft_nms_batched(float* dets_dev, const int* counts_host, int num_problems, float sigma, float overlap_thresh,
                          float score_thresh, int method, int* inds_out_dev, int* num_out_dev, b200_stream_t stream) {
    if (!counts_host || num_problems < 1 || !num_out_dev) return B200_ROI_EINVAL;
    long long total = 0;
    for (int p = 0; p < num_problems && p < 128; ++p) total += counts_host[p] > 0 ? counts_host[p] : 0;
    if (total > 0 && (!dets_dev || !inds_out_dev)) return B200_ROI_EINVAL;
    return soft_nms_batched(dets_dev, counts_host, num_problems, sigma, overlap_thresh, score_thresh, method, inds_out_dev, num_out_dev,
                            (cudaStream_t)stream);
}

int b200_box_voting_batched(const float* top_dets_dev, const int* top_counts_host, const float* all_dets_dev, const int* all_counts_host,
                            int num_problems, float thresh, int scoring_method, float beta, float* out_dev, b200_stream_t stream) {
    if (!top_counts_host || !all_counts_host || num_problems < 1) return B200_ROI_EINVAL;
    long long total = 0;
    for (int p = 0; p < num_problems && p < 128; ++p) total += top_counts_host[p] > 0 ? top_counts_host[p] : 0;
    if (total > 0 && (!top_dets_dev || !all_dets_dev || !out_dev)) return B200_ROI_EINVAL;
    if (scoring_method < 0 || scoring_method > 5) return B200_ROI_EINVAL;
    return box_voting_batched(top_dets_dev, top_counts_host, all_dets_dev, all_counts_host, num_problems, thresh, scoring_method, beta, out_dev,
                              (cudaStream_t)stream);
}

size_t b200_topk_batched_workspace_bytes(int num_problems) { return topk_batched_workspace_bytes(num_problems); }

int b200_topk_batched(const float* const* scores_dev_ptrs_host, const int* num_anchors_host, const int* num_cells_host, const int* k_host,
                      int num_problems, long long* order_out_dev, float* scores_out_dev, void* workspace, size_t workspace_bytes,
                      b200_stream_t stream) {
    if (num_problems < 1 || !scores_dev_ptrs_host || !num_anchors_host || !num_cells_host || !k_host) return B200_ROI_EINVAL;
    long long total = 0;
    for (int p = 0; p < num_problems && p < 64; ++p) {
        if (!scores_dev_ptrs_host[p] || k_host[p] < 0) return B200_ROI_EINVAL;
        total += k_host[p];
    }
    if (total > 0 && (!order_out_dev || !scores_out_dev)) return B200_ROI_EINVAL;
    const int rc = topk_batched(scores_dev_ptrs_host, num_anchors_host, num_cells_host, k_host, num_problems, order_out_dev, scores_out_dev,
                                workspace, workspace_bytes, (cudaStream_t)stream);
    return rc == 1000 ? B200_ROI_EWORKSPACE : rc;
}

int b200_bbox_overlaps(const float* boxes_dev, int num_boxes, const float* query_boxes_dev, int num_query, float* overlaps_out_dev,
                       b200_stream_t stream) {
    if (num_boxes < 0 || num_query < 0) return B200_ROI_EINVAL;
    if ((long long)num_boxes * num_query > 0 && (!boxes_dev || !query_boxes_dev || !overlaps_out_dev)) return B200_ROI_EINVAL;
    return bbox_overlaps(boxes_dev, num_boxes, query_boxes_dev, num_query, overlaps_out_dev, (cudaStream_t)stream);
}

int b200_roi_assign(const float* boxes_dev, int num_boxes, const float* gt_boxes_dev, const int* gt_classes_dev, int num_gt,
                    float* max_overlaps_out_dev, int* argmax_out_dev, int* max_classes_out_dev, b200_stream_t stream) {
    if (num_boxes < 0 || num_gt < 0) return B200_ROI_EINVAL;
    if (num_boxes > 0 && (!boxes_dev || !max_overlaps_out_dev || !argmax_out_dev || !max_classes_out_dev)) return B200_ROI_EINVAL;
    if (num_boxes > 0 && num_gt > 0 && (!gt_boxes_dev || !gt_classes_dev)) return B200_ROI_EINVAL;
    return roi_assign(boxes_dev, num_boxes, gt_boxes_dev, gt_classes_dev, num_gt, max_overlaps_out_dev, argmax_out_dev, max_classes_out_dev,
                      (cudaStream_t)stream);
}

int b200_roi_select(const float* max_overlaps_dev, int num_boxes, float fg_thresh, float bg_thresh_hi, float bg_thresh_lo,
                    int* fg_inds_out_dev, int* bg_inds_out_dev, int* counts_out_dev, b200_stream_t stream) {
    if (num_boxes < 0 || !counts_out_dev) return B200_ROI_EINVAL;
    if (num_boxes > 0 && (!max_overlaps_dev || !fg_inds_out_dev || !bg_inds_out_dev)) return B200_ROI_EINVAL;
    return roi_select(max_overlaps_dev, num_boxes, fg_thresh, bg_thresh_hi, bg_thresh_lo, fg_inds_out_dev, bg_inds_out_dev, counts_out_dev,
                      (cudaStream_t)stream);
}

int b200_fast_rcnn_targets(const float* boxes_dev, const float* gt_boxes_dev, const int* argmax_dev, const int* max_classes_dev,
                           const int* keep_inds_dev, int num_keep, int num_fg, const float* bbox_reg_weights_host, int num_reg_classes,
                           int cls_agnostic, float im_scale, float batch_idx, int* labels_out_dev, float* rois_out_dev,
                           float* bbox_targets_out_dev, float* inside_weights_out_dev, float* outside_weights_out_dev,
                           b200_stream_t stream) {
    if (num_keep < 0 || num_fg < 0 || num_fg > num_keep || num_reg_classes < 1 || !bbox_reg_weights_host) return B200_ROI_EINVAL;
    if (num_keep > 0 && (!boxes_dev || !argmax_dev || !max_classes_dev || !keep_inds_dev || !labels_out_dev || !rois_out_dev ||
                         !bbox_targets_out_dev || !inside_weights_out_dev || !outside_weights_out_dev))
        return B200_ROI_EINVAL;
    return fast_rcnn_targets(boxes_dev, gt_boxes_dev, argmax_dev, max_classes_dev, keep_inds_dev, num_keep, num_fg, bbox_reg_weights_host,
                             num_reg_classes, cls_agnostic, im_scale, batch_idx, labels_out_dev, rois_out_dev, bbox_targets_out_dev,
                             inside_weights_out_dev, outside_weights_out_dev, (cudaStream_t)stream);
}

// test-time mask paste (N3, masks): lib/core/test.py:793-847, lib/utils/boxes.py:233-249 (expand_boxes)
int b200_segm_paste(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets, int num_channels,
                    int resolution, int im_h, int im_w, float thresh, unsigned char* masks_out_dev, b200_stream_t stream) {
    if (!segm_args_ok(num_dets, num_channels, resolution, im_h, im_w)) return B200_ROI_EINVAL;
    if (num_dets > 0 && (!masks_dev || !ref_boxes_dev || !masks_out_dev)) return B200_ROI_EINVAL;
    return segm_paste(masks_dev, mask_channel_dev, ref_boxes_dev, num_dets, num_channels, resolution, im_h, im_w, thresh, masks_out_dev,
                      (cudaStream_t)stream);
}

int b200_segm_rle_count(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets, int num_channels,
                        int resolution, int im_h, int im_w, float thresh, long long* offsets_out_dev, b200_stream_t stream) {
    if (!segm_args_ok(num_dets, num_channels, resolution, im_h, im_w)) return B200_ROI_EINVAL;
    if (num_dets > 0 && (!masks_dev || !ref_boxes_dev || !offsets_out_dev)) return B200_ROI_EINVAL;
    return segm_rle_count(masks_dev, mask_channel_dev, ref_boxes_dev, num_dets, num_channels, resolution, im_h, im_w, thresh,
                          offsets_out_dev, (cudaStream_t)stream);
}

int b200_segm_rle_emit(const float* masks_dev, const int* mask_channel_dev, const float* ref_boxes_dev, int num_dets, int num_channels,
                       int resolution, int im_h, int im_w, float thresh, const long long* offsets_dev, int* runs_out_dev,
                       b200_stream_t stream) {
    if (!segm_args_ok(num_dets, num_channels, resolution, im_h, im_w)) return B200_ROI_EINVAL;
    if (num_dets > 0 && (!masks_dev || !ref_boxes_dev || !offsets_dev || !runs_out_dev)) return B200_ROI_EINVAL;
    return segm_rle_emit(masks_dev, mask_channel_dev, ref_boxes_dev, num_dets, num_channels, resolution, im_h, im_w, thresh, offsets_dev,
                         runs_out_dev, (cudaStream_t)stream);
}

}  // extern "C"
