// segm.cu -- test-time mask paste of Mask R-CNN (SURVEY.md 8f N3, masks): lib/core/test.py:793-847 `segm_results` with
// lib/utils/boxes.py:233-249 `expand_boxes` (reference).  Per detection the M x M soft mask, zero-padded to M + 2, is
// resized to its expanded integer box exactly like cv2.resize(INTER_LINEAR) on float32 with IPP off, thresholded with
// `>` and pasted into the clipped window of an all-zero im_h x im_w image.  Two products:
//   segm_paste_kernel   the dense (D, im_h, im_w) uint8 images, grid (row band, detection);
//   segm_rle_kernel     COCO's uncompressed RLE of each column-major image without materialising it: one CTA per
//                       detection walks the window's columns; a count pass + device scan gives every detection's offset,
//                       an emit pass writes the run lengths there.
// All rounding follows cv2's scalar code: products and sums rounded separately (_rn intrinsics, no FMA contraction).
#include "common.cuh"

namespace b200 {

namespace {
constexpr int kSegmThreads = 256;
constexpr int kPasteTile = 128;       // columns of horizontally resized rows staged per pass of the paste kernel
constexpr int kPasteBandBytes = 16384;
constexpr int kSegmMaxRes = 126;      // (M + 2) rows of staged floats must fit shared memory
constexpr int kSegmMaxWidth = 32768;

struct SegmGeom {
    int bx1, by1;           // expanded integer box corner (destination pixel (0, 0) of the resize)
    int w, h;               // resize destination size
    int x0, x1, y0, y1;     // clipped window [y0, y1) x [x0, x1); empty when x0 >= x1 or y0 >= y1
    bool area2;             // cv2 takes its area-fast path: exact 2x downscale on both axes
};

__device__ __forceinline__ SegmGeom segm_geom(const float* __restrict__ box, float scale, int M, int im_h, int im_w) {
    // expand_boxes in float32, then float64 storage and .astype(np.int32) (truncation toward zero)
    const float bx1 = box[0], by1 = box[1], bx2 = box[2], by2 = box[3];
    const float w_half = __fmul_rn(__fmul_rn(__fsub_rn(bx2, bx1), .5f), scale);
    const float h_half = __fmul_rn(__fmul_rn(__fsub_rn(by2, by1), .5f), scale);
    const float x_c = __fmul_rn(__fadd_rn(bx2, bx1), .5f), y_c = __fmul_rn(__fadd_rn(by2, by1), .5f);
    const long long ex1 = (int)__fsub_rn(x_c, w_half), ex2 = (int)__fadd_rn(x_c, w_half);
    const long long ey1 = (int)__fsub_rn(y_c, h_half), ey2 = (int)__fadd_rn(y_c, h_half);
    SegmGeom g;
    g.bx1 = (int)ex1; g.by1 = (int)ey1;
    const long long w = ex2 - ex1 + 1, h = ey2 - ey1 + 1;
    g.w = (int)(w < 1 ? 1 : (w > 0x7fffffffLL ? 0x7fffffffLL : w));
    g.h = (int)(h < 1 ? 1 : (h > 0x7fffffffLL ? 0x7fffffffLL : h));
    g.x0 = (int)(ex1 > 0 ? ex1 : 0); g.x1 = (int)(ex2 + 1 < im_w ? ex2 + 1 : im_w);
    g.y0 = (int)(ey1 > 0 ? ey1 : 0); g.y1 = (int)(ey2 + 1 < im_h ? ey2 + 1 : im_h);
    if (g.x1 < g.x0) g.x1 = g.x0;
    if (g.y1 < g.y0) g.y1 = g.y0;
    g.area2 = (2LL * g.w == M + 2) && (2LL * g.h == M + 2);
    return g;
}

// One axis of cv2's INTER_LINEAR table: fx = (float)((d + 0.5) * scale - 0.5), sx = floor(fx), fx -= sx, weights
// (1 - fx, fx).  Horizontally cv2 zeroes fx where sx leaves [0, src - 1]; vertically it only clips the two row indices.
struct SegmTap {
    int s0, s1;
    float a0, a1;
};

__device__ __forceinline__ SegmTap segm_tap(int d, int src, double scale, bool clamp_weights) {
    float f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    int s = (int)floorf(f);
    f = __fsub_rn(f, (float)s);
    if (clamp_weights) {
        if (s < 0) { s = 0; f = 0.f; }
        if (s >= src - 1) { s = src - 1; f = 0.f; }
    }
    SegmTap t;
    t.s0 = min(max(s, 0), src - 1);
    t.s1 = min(max(s + 1, 0), src - 1);
    t.a0 = __fsub_rn(1.f, f);
    t.a1 = f;
    return t;
}

__device__ __forceinline__ double segm_scale(int dst, int src) { return __ddiv_rn(1.0, __ddiv_rn((double)dst, (double)src)); }

// zero-padded source: padded (s, t) = mask (s - 1, t - 1) inside, 0 on the one-pixel border
__device__ __forceinline__ float segm_src(const float* __restrict__ S, int M, int s, int t) {
    return (s >= 1 && s <= M && t >= 1 && t <= M) ? __ldg(S + (s - 1) * M + (t - 1)) : 0.f;
}

__device__ __forceinline__ float segm_hpass(const float* __restrict__ S, int M, int s, const SegmTap& tx) {
    return __fadd_rn(__fmul_rn(segm_src(S, M, s, tx.s0), tx.a0), __fmul_rn(segm_src(S, M, s, tx.s1), tx.a1));
}

__device__ __forceinline__ float segm_vpass(float r0, float r1, const SegmTap& ty) {
    return __fadd_rn(__fmul_rn(r0, ty.a0), __fmul_rn(r1, ty.a1));
}

// cv2's area-fast 2x downscale (resizeAreaFast_): ((a + b) + (c + d)) * 0.25 in its 4-wide vector loop over the first
// 4 * (w / 4) destination columns, (((a + b) + c) + d) * 0.25 in the scalar tail.
__device__ __forceinline__ float segm_area2(const float* __restrict__ S, int M, int w, int dy, int dx) {
    const float a = segm_src(S, M, 2 * dy, 2 * dx), b = segm_src(S, M, 2 * dy, 2 * dx + 1);
    const float c = segm_src(S, M, 2 * dy + 1, 2 * dx), d = segm_src(S, M, 2 * dy + 1, 2 * dx + 1);
    const float sum = (dx < (w & ~3)) ? __fadd_rn(__fadd_rn(a, b), __fadd_rn(c, d)) : __fadd_rn(__fadd_rn(__fadd_rn(a, b), c), d);
    return __fmul_rn(sum, .25f);
}

__device__ __forceinline__ const float* segm_mask(const float* masks, const int* chan, int d, int K, int M) {
    const int c = chan ? chan[d] : 0;
    if (c < 0 || c >= K) return nullptr;                       // out-of-range channel: empty mask, no out-of-bounds read
    return masks + ((size_t)d * K + c) * M * M;
}

// ---- dense paste --------------------------------------------------------------------------------------------------
// CTA (band, d) owns rows [band * band_rows, +band_rows) of image d: it binarises the window part of those rows into a
// shared byte image of the band (zeros elsewhere), then copies the band to global memory with 16-byte stores.  The
// window columns go in tiles of kPasteTile: the horizontally resized source rows the band needs are staged once per
// tile ((M + 2) x kPasteTile floats at most) and every output row of the tile reads them.
__global__ void __launch_bounds__(kSegmThreads)
segm_paste_kernel(const float* __restrict__ masks, const int* __restrict__ chan, const float* __restrict__ boxes, int K, int M,
                  int im_h, int im_w, float thresh, float scale, int band_rows, unsigned char* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem[];
    float* rt = reinterpret_cast<float*>(smem);                                   // [(M + 2)][kPasteTile]
    SegmTap* xt = reinterpret_cast<SegmTap*>(rt + (M + 2) * kPasteTile);          // [kPasteTile]
    SegmTap* yt = xt + kPasteTile;                                                // [band_rows]
    unsigned char* bin = reinterpret_cast<unsigned char*>(yt + band_rows);        // [band_rows * im_w]
    const int d = blockIdx.y, tid = threadIdx.x;
    const int ya = blockIdx.x * band_rows, yb = min(ya + band_rows, im_h);
    const int nbytes = (yb - ya) * im_w;
    const SegmGeom g = segm_geom(boxes + 4 * d, scale, M, im_h, im_w);
    const float* S = segm_mask(masks, chan, d, K, M);
    for (int i = tid; i < nbytes; i += kSegmThreads) bin[i] = 0;
    const int ry0 = max(ya, g.y0), ry1 = min(yb, g.y1);
    const int src = M + 2;
    if (S && ry0 < ry1 && g.x0 < g.x1) {
        const double sx = segm_scale(g.w, src), sy = segm_scale(g.h, src);
        for (int r = tid; r < ry1 - ry0; r += kSegmThreads) yt[r] = segm_tap(ry0 + r - g.by1, src, sy, false);
        __syncthreads();
        const int slo = yt[0].s0, shi = yt[ry1 - ry0 - 1].s1;             // source rows this band reads (monotone taps)
        for (int cx = g.x0; cx < g.x1; cx += kPasteTile) {
            const int ncols = min(kPasteTile, g.x1 - cx);
            if (!g.area2) {
                for (int c = tid; c < ncols; c += kSegmThreads) xt[c] = segm_tap(cx + c - g.bx1, src, sx, true);
                __syncthreads();
                for (int i = tid; i < (shi - slo + 1) * ncols; i += kSegmThreads) {
                    const int s = slo + i / ncols, c = i % ncols;
                    rt[(s - slo) * kPasteTile + c] = segm_hpass(S, M, s, xt[c]);
                }
                __syncthreads();
            }
            for (int i = tid; i < (ry1 - ry0) * ncols; i += kSegmThreads) {
                const int r = i / ncols, c = i % ncols;
                float v;
                if (g.area2) {
                    v = segm_area2(S, M, g.w, ry0 + r - g.by1, cx + c - g.bx1);
                } else {
                    const SegmTap ty = yt[r];
                    v = segm_vpass(rt[(ty.s0 - slo) * kPasteTile + c], rt[(ty.s1 - slo) * kPasteTile + c], ty);
                }
                bin[(ry0 + r - ya) * im_w + cx + c] = v > thresh ? 1 : 0;
            }
            __syncthreads();
        }
    }
    __syncthreads();
    // the band is one contiguous byte range of the output: byte stores up to 16-byte alignment, then 16-byte stores
    unsigned char* dst = out + ((size_t)d * im_h + ya) * im_w;
    const int head = min(nbytes, (int)((16 - ((uintptr_t)dst & 15)) & 15));
    const int nvec = (nbytes - head) >> 4;
    for (int i = tid; i < head; i += kSegmThreads) dst[i] = bin[i];
    for (int i = tid; i < nvec; i += kSegmThreads) {
        const unsigned char* b = bin + head + 16 * i;
        uint32_t wv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
            wv[k] = (uint32_t)b[4 * k] | ((uint32_t)b[4 * k + 1] << 8) | ((uint32_t)b[4 * k + 2] << 16) | ((uint32_t)b[4 * k + 3] << 24);
        reinterpret_cast<uint4*>(dst + head)[i] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
    }
    for (int i = head + 16 * nvec + tid; i < nbytes; i += kSegmThreads) dst[i] = bin[i];
}

// ---- column-major RLE ---------------------------------------------------------------------------------------------
// The image is zero outside the window, so the value changes of its column-major sequence (with a virtual 0 before
// pixel 0) all lie on window columns: inside a column, at the window's top (against 0, or against the bottom pixel of
// the column to the left when the window spans every row and so the sequence runs on from column to column), and after
// its last row (unless the next column continues it or the image ends).  Runs = changes + 1: change k at flat position
// p_k closes run k = p_k - p_{k-1} (p_{-1} = 0), the last run ends at im_h * im_w.
// One CTA per detection, one thread per window column of a kSegmThreads-wide tile; the horizontally resized source
// rows of the tile are staged in shared memory.  kEmit = false counts, kEmit = true writes the runs at their offset.

// block-wide exclusive scan of (sum a, max b), kSegmThreads threads; returns the totals through *tot_a, *tot_b
__device__ __forceinline__ void segm_block_scan(int a, int b, int* excl_a, int* excl_b, int* tot_a, int* tot_b, int* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int ia = a, ib = b;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib = max(ib, tb); }
    }
    if (lane == 31) { sh[warp] = ia; sh[32 + warp] = ib; }
    __syncthreads();
    if (warp == 0) {
        int wa = lane < kSegmThreads / 32 ? sh[lane] : 0, wb = lane < kSegmThreads / 32 ? sh[32 + lane] : -1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int ta = __shfl_up_sync(0xffffffffu, wa, o), tb = __shfl_up_sync(0xffffffffu, wb, o);
            if (lane >= o) { wa += ta; wb = max(wb, tb); }
        }
        sh[64 + lane] = wa; sh[96 + lane] = wb;                        // inclusive over warps
    }
    __syncthreads();
    const int pa = warp > 0 ? sh[64 + warp - 1] : 0, pb = warp > 0 ? sh[96 + warp - 1] : -1;
    *excl_a = pa + ia - a;
    const int eb = __shfl_up_sync(0xffffffffu, ib, 1);
    *excl_b = max(pb, lane > 0 ? eb : -1);
    *tot_a = sh[64 + kSegmThreads / 32 - 1];
    *tot_b = sh[96 + kSegmThreads / 32 - 1];
    __syncthreads();
}

template <bool kEmit>
__global__ void __launch_bounds__(kSegmThreads)
segm_rle_kernel(const float* __restrict__ masks, const int* __restrict__ chan, const float* __restrict__ boxes, int K, int M,
                int im_h, int im_w, float thresh, float scale, long long* __restrict__ offsets, int* __restrict__ runs) {
    extern __shared__ __align__(16) unsigned char smem[];
    float* rt = reinterpret_cast<float*>(smem);                          // [(M + 2)][kSegmThreads]
    __shared__ unsigned char lastv[kSegmThreads];
    __shared__ int scan_sh[128];
    const int d = blockIdx.x, tid = threadIdx.x;
    const SegmGeom g = segm_geom(boxes + 4 * d, scale, M, im_h, im_w);
    const float* S = segm_mask(masks, chan, d, K, M);
    const int src = M + 2;
    const bool live = S && g.x0 < g.x1 && g.y0 < g.y1;
    const bool wrap = g.y0 == 0 && g.y1 == im_h;
    const int total = im_h * im_w;
    int* out = kEmit ? runs + offsets[d] : nullptr;
    int carry_n = 0, carry_pos = 0;                                     // changes so far, position of the last one
    int carry_last = 0;                                                 // bottom value of the column left of the tile
    const double sx = segm_scale(g.w, src), sy = segm_scale(g.h, src);
    for (int cx = g.x0; live && cx < g.x1; cx += kSegmThreads) {
        const int x = cx + tid;
        const bool col = x < g.x1;
        SegmTap tx;
        if (col && !g.area2) {
            tx = segm_tap(x - g.bx1, src, sx, true);
            for (int s = 0; s < src; ++s) rt[s * kSegmThreads + tid] = segm_hpass(S, M, s, tx);
        }
        auto value = [&](int y) -> int {
            const int dy = y - g.by1;
            float v;
            if (g.area2) {
                v = segm_area2(S, M, g.w, dy, x - g.bx1);
            } else {
                const SegmTap ty = segm_tap(dy, src, sy, false);
                v = segm_vpass(rt[ty.s0 * kSegmThreads + tid], rt[ty.s1 * kSegmThreads + tid], ty);
            }
            return v > thresh ? 1 : 0;
        };
        if (col) lastv[tid] = (unsigned char)value(g.y1 - 1);
        __syncthreads();
        const int start = (wrap && x > g.x0) ? (tid > 0 ? lastv[tid - 1] : carry_last) : 0;
        const bool close_end = !(wrap && x + 1 < g.x1) && !(g.y1 == im_h && x == im_w - 1);
        int n = 0, last = -1;
        if (col) {
            int prev = start;
            const int base = x * im_h;
            for (int y = g.y0; y < g.y1; ++y) {
                const int v = value(y);
                if (v != prev) { ++n; last = base + y; }
                prev = v;
            }
            if (prev && close_end) { ++n; last = base + g.y1; }
        }
        if (!kEmit) {
            int ea, eb, ta, tb;
            segm_block_scan(n, last, &ea, &eb, &ta, &tb, scan_sh);
            carry_n += ta;
        } else {
            int ea, eb, ta, tb;
            segm_block_scan(n, last, &ea, &eb, &ta, &tb, scan_sh);
            if (col && n > 0) {
                int k = carry_n + ea;
                int prevpos = max(carry_pos, eb);
                int prev = start;
                const int base = x * im_h;
                for (int y = g.y0; y < g.y1; ++y) {
                    const int v = value(y);
                    if (v != prev) { out[k++] = base + y - prevpos; prevpos = base + y; }
                    prev = v;
                }
                if (prev && close_end) out[k] = base + g.y1 - prevpos;
            }
            carry_n += ta;
            carry_pos = max(carry_pos, tb);
        }
        carry_last = lastv[min(kSegmThreads, g.x1 - cx) - 1];
        __syncthreads();
    }
    if (tid == 0) {
        if (kEmit) out[carry_n] = total - carry_pos;
        else offsets[d + 1] = carry_n + 1;
    }
}

// offsets[1 .. D] hold the per-detection run counts; turn them into the exclusive offsets (offsets[0] = 0) in place.
__global__ void __launch_bounds__(1024) segm_scan_kernel(long long* __restrict__ offsets, int D) {
    __shared__ long long warp_sum[32];
    __shared__ long long carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { carry = 0; offsets[0] = 0; }
    __syncthreads();
    for (int c0 = 0; c0 < D; c0 += 1024) {
        const int i = c0 + tid;
        long long v = i < D ? offsets[i + 1] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, v, o);
            if (lane >= o) v += t;
        }
        if (lane == 31) warp_sum[warp] = v;
        __syncthreads();
        if (warp == 0) {
            long long w = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_sum[lane] = w;
        }
        __syncthreads();
        const long long incl = carry + (warp > 0 ? warp_sum[warp - 1] : 0) + v;
        if (i < D) offsets[i + 1] = incl;
        __syncthreads();
        if (tid == 1023) carry = incl;
        __syncthreads();
    }
}

int segm_band_rows(int im_w) { return max(1, min(32, kPasteBandBytes / im_w)); }

size_t segm_paste_smem(int M, int im_w) {
    const int band = segm_band_rows(im_w);
    return (size_t)(M + 2) * kPasteTile * 4 + (size_t)(kPasteTile + band) * sizeof(SegmTap) + (size_t)band * im_w;
}

size_t segm_rle_smem(int M) { return (size_t)(M + 2) * kSegmThreads * 4; }

template <typename Kernel>
int segm_smem_attr(Kernel k, size_t bytes) {
    if (bytes <= 48 * 1024) return 0;
    return (int)cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

float segm_scale_f(int M) { return (float)((M + 2.0) / M); }
}  // namespace

bool segm_args_ok(int D, int K, int M, int im_h, int im_w) {
    return D >= 0 && K >= 1 && M >= 1 && M <= kSegmMaxRes && im_h >= 1 && im_w >= 1 && im_w <= kSegmMaxWidth &&
           (long long)im_h * im_w <= 0x7fffffffLL;
}

int segm_paste(const float* masks, const int* chan, const float* boxes, int D, int K, int M, int im_h, int im_w, float thresh,
               unsigned char* out, cudaStream_t stream) {
    if (D == 0) return B200_ROI_OK;
    const size_t smem = segm_paste_smem(M, im_w);
    if (int rc = segm_smem_attr(segm_paste_kernel, smem)) return rc;
    const int band = segm_band_rows(im_w);
    dim3 grid((im_h + band - 1) / band, D);
    segm_paste_kernel<<<grid, kSegmThreads, smem, stream>>>(masks, chan, boxes, K, M, im_h, im_w, thresh, segm_scale_f(M), band, out);
    return finish_launch();
}

int segm_rle_count(const float* masks, const int* chan, const float* boxes, int D, int K, int M, int im_h, int im_w, float thresh,
                   long long* offsets, cudaStream_t stream) {
    if (D == 0) return B200_ROI_OK;
    const size_t smem = segm_rle_smem(M);
    if (int rc = segm_smem_attr(segm_rle_kernel<false>, smem)) return rc;
    segm_rle_kernel<false><<<D, kSegmThreads, smem, stream>>>(masks, chan, boxes, K, M, im_h, im_w, thresh, segm_scale_f(M), offsets, nullptr);
    segm_scan_kernel<<<1, 1024, 0, stream>>>(offsets, D);
    return finish_launch(2);
}

int segm_rle_emit(const float* masks, const int* chan, const float* boxes, int D, int K, int M, int im_h, int im_w, float thresh,
                  const long long* offsets, int* runs, cudaStream_t stream) {
    if (D == 0) return B200_ROI_OK;
    const size_t smem = segm_rle_smem(M);
    if (int rc = segm_smem_attr(segm_rle_kernel<true>, smem)) return rc;
    segm_rle_kernel<true><<<D, kSegmThreads, smem, stream>>>(masks, chan, boxes, K, M, im_h, im_w, thresh, segm_scale_f(M),
                                                             const_cast<long long*>(offsets), runs);
    return finish_launch();
}

}  // namespace b200
