// resize.cu -- bilinear resize (cv2.resize INTER_LINEAR on uint8: utils/transform.py:167-179,
// modules/preprocessor.py:136-143) and the YOLO input transform behind modules/yolo.py:112
// (Ultralytics LetterBox -> BGR2RGB -> HWC2CHW -> /255 -> half), batched over cameras.
//
// The interpolation is OpenCV's 11-bit fixed-point scheme (pixel_math.cuh: linear_coef /
// linear_vblend), so the uint8 result is bit-identical to cv2.
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace bv {

template <int CN>
__global__ void __launch_bounds__(256) resize_kernel(const uint8_t *__restrict__ src, int sh, int sw,
                                                     uint8_t *__restrict__ dst, int dh, int dw, double scale_x,
                                                     double scale_y, size_t total) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int x = (int)(i % dw);
        const size_t t = i / dw;
        const int y = (int)(t % dh);
        const size_t f = t / dh;
        const LinCoef cx = linear_coef(x, sw, scale_x, true);
        const LinCoef cy = linear_coef(y, sh, scale_y, false);
        const uint8_t *s0 = src + (f * sh + cy.i0) * (size_t)sw * CN;
        const uint8_t *s1 = src + (f * sh + cy.i1) * (size_t)sw * CN;
        uint8_t *d = dst + i * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c) {
            const int h0 = s0[cx.i0 * CN + c] * cx.w0 + s0[cx.i1 * CN + c] * cx.w1;
            const int h1 = s1[cx.i0 * CN + c] * cx.w0 + s1[cx.i1 * CN + c] * cx.w1;
            d[c] = (uint8_t)linear_vblend(h0, h1, cy.w0, cy.w1);
        }
    }
}

struct LetterboxImg {
    const uint8_t *src;
    int sh, sw;          // source size
    int uh, uw;          // un-padded (resized) size
    int top, left;       // padding offsets
    double scale_x, scale_y;
};

template <bool FP16>
__global__ void __launch_bounds__(256) letterbox_kernel(const LetterboxImg *__restrict__ imgs, void *__restrict__ out, int oh,
                                                        int ow, int pad) {
    const LetterboxImg im = imgs[blockIdx.z];
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    if (x >= ow) return;
    int b = pad, g = pad, r = pad;
    const int ux = x - im.left, uy = y - im.top;
    if (ux >= 0 && ux < im.uw && uy >= 0 && uy < im.uh) {
        if (im.uw == im.sw && im.uh == im.sh) {
            const uint8_t *p = im.src + ((size_t)uy * im.sw + ux) * 3;
            b = p[0];
            g = p[1];
            r = p[2];
        } else {
            const LinCoef cx = linear_coef(ux, im.sw, im.scale_x, true);
            const LinCoef cy = linear_coef(uy, im.sh, im.scale_y, false);
            const uint8_t *s0 = im.src + (size_t)cy.i0 * im.sw * 3;
            const uint8_t *s1 = im.src + (size_t)cy.i1 * im.sw * 3;
            int v[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const int h0 = s0[cx.i0 * 3 + c] * cx.w0 + s0[cx.i1 * 3 + c] * cx.w1;
                const int h1 = s1[cx.i0 * 3 + c] * cx.w0 + s1[cx.i1 * 3 + c] * cx.w1;
                v[c] = linear_vblend(h0, h1, cy.w0, cy.w1);
            }
            b = v[0];
            g = v[1];
            r = v[2];
        }
    }
    // BGR -> RGB, HWC -> CHW, /255 (float32 division, then one rounding to half: what torch does
    // for `im.half() / 255`)
    const size_t plane = (size_t)oh * ow;
    const size_t o = (size_t)blockIdx.z * 3 * plane + (size_t)y * ow + x;
    const float fr = __fdiv_rn((float)r, 255.f), fg = __fdiv_rn((float)g, 255.f), fb = __fdiv_rn((float)b, 255.f);
    if (FP16) {
        __half *q = reinterpret_cast<__half *>(out);
        q[o] = __float2half_rn(fr);
        q[o + plane] = __float2half_rn(fg);
        q[o + 2 * plane] = __float2half_rn(fb);
    } else {
        float *q = reinterpret_cast<float *>(out);
        q[o] = fr;
        q[o + plane] = fg;
        q[o + 2 * plane] = fb;
    }
}


// ----------------------------------------------------------------------------------------------
// Letterbox with TMA-staged source rows.  A work item is one output row of one image: the two
// source rows that row interpolates between (2 x W x 3 bytes, e.g. 13 KB at 2208 px) are pulled
// into shared memory by a single elected thread with cp.async.bulk (the TMA engine; SASS: UBLKCP)
// signalling an mbarrier, so HBM sees two long sequential bursts per block instead of 12 scattered
// byte loads per output pixel; all threads then gather their taps from shared memory.
// Rows whose byte size or address is not 16-byte aligned are staged with ordinary loads instead.
// ----------------------------------------------------------------------------------------------
constexpr int kLbMaxRowBytes = 11520;  // up to 3840 px wide sources (4 stages x 2 rows = 92 KB of shared memory)

// horizontal taps of one output column
struct LbCoef {
    short o0, o1;  // byte offsets of the two taps inside a source row; o0 < 0: padding column
    short w0, w1;
};

__device__ __forceinline__ LbCoef lb_coef(const LetterboxImg &im, bool identity, int x) {
    LbCoef c;
    const int ux = x - im.left;
    if (ux < 0 || ux >= im.uw) {
        c.o0 = c.o1 = -1;
        c.w0 = c.w1 = 0;
    } else if (identity) {
        c.o0 = c.o1 = (short)(ux * 3);
        c.w0 = 2048;
        c.w1 = 0;
    } else {
        const LinCoef cx = linear_coef(ux, im.sw, im.scale_x, true);
        c.o0 = (short)(cx.i0 * 3);
        c.o1 = (short)(cx.i1 * 3);
        c.w0 = (short)cx.w0;
        c.w1 = (short)cx.w1;
    }
    return c;
}

struct LbItem {
    LetterboxImg im;
    int img, y, uy;
    bool inside_y, identity, tma_ok;
    uint32_t row_bytes;
    LinCoef cy;
    const uint8_t *g0, *g1;
};

__device__ __forceinline__ LbItem lb_item(const LetterboxImg *__restrict__ imgs, int item, int oh) {
    LbItem t;
    t.img = item / oh;
    t.y = item - t.img * oh;
    t.im = imgs[t.img];
    t.uy = t.y - t.im.top;
    t.inside_y = t.uy >= 0 && t.uy < t.im.uh;
    t.identity = t.im.uw == t.im.sw && t.im.uh == t.im.sh;
    t.row_bytes = (uint32_t)t.im.sw * 3u;
    t.cy.i0 = t.cy.i1 = t.uy;
    t.cy.w0 = 2048;
    t.cy.w1 = 0;
    if (t.inside_y && !t.identity) t.cy = linear_coef(t.uy, t.im.sh, t.im.scale_y, false);
    t.g0 = t.g1 = t.im.src;
    t.tma_ok = false;
    if (t.inside_y) {
        t.g0 = t.im.src + (size_t)t.cy.i0 * t.row_bytes;
        t.g1 = t.im.src + (size_t)t.cy.i1 * t.row_bytes;
        t.tma_ok = (t.row_bytes % 16u == 0) && ((reinterpret_cast<uintptr_t>(t.g0) & 15) == 0) &&
                   ((reinterpret_cast<uintptr_t>(t.g1) & 15) == 0);
    }
    return t;
}

// The horizontal taps depend on (image, output column) only: worked out once per call (float64
// coordinate arithmetic, ~40 instructions) instead of once per output pixel.
__global__ void __launch_bounds__(256) letterbox_coef_kernel(const LetterboxImg *__restrict__ imgs, LbCoef *__restrict__ coefs, int ow,
                                                             int total) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int img = i / ow, x = i - img * ow;
    const LetterboxImg im = imgs[img];
    coefs[i] = lb_coef(im, im.uw == im.sw && im.uh == im.sh, x);
}

__device__ __forceinline__ LbCoef coef_from_words(uint32_t a, uint32_t b) {
    LbCoef c;
    c.o0 = (short)(a & 0xFFFFu);
    c.o1 = (short)(a >> 16);
    c.w0 = (short)(b & 0xFFFFu);
    c.w1 = (short)(b >> 16);
    return c;
}

// Persistent, warp-specialised blocks: warp 8 is the producer -- one lane works out the next item
// (which image, which two source rows) and hands the copy to the TMA engine as soon as a stage is
// free; warps 0-7 only ever wait for a filled stage, interpolate one output row out of it and
// release it.  kLbStages rows-pairs are in flight per block, so neither the descriptor arithmetic
// nor the HBM latency of a row sits on the consumers' critical path.
constexpr int kLbStages = 2;  // per block; 5-6 blocks per SM keep ~12 row pairs in flight per SM
constexpr int kLbConsumers = 256;
constexpr int kLbMaxImgs = 256;
constexpr int kLbSmemImgs = 64;

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kLbConsumers) : "memory"); }

template <bool FP16>
__global__ void __launch_bounds__(kLbConsumers + 32) letterbox_tma_kernel(const LetterboxImg *__restrict__ imgs, int n_imgs,
                                                                         const LbCoef *__restrict__ coefs, void *__restrict__ out,
                                                                         int oh, int ow, int pad, int n_items, int row_stride) {
    extern __shared__ __align__(128) uint8_t lb_rows[];  // [kLbStages][2][row_stride], then LbCoef[ow] of the current image
    __shared__ __align__(8) uint64_t full[kLbStages], empty[kLbStages];
    __shared__ float norm[256];  // v / 255 in float32 (IEEE division once per value instead of per pixel)
    __shared__ LbItem sitem[kLbStages];
    __shared__ LetterboxImg simgs[kLbSmemImgs];  // descriptors of the first images (3 KB); larger batches read the rest from L2
    for (int k = threadIdx.x; k < 256; k += blockDim.x) norm[k] = __fdiv_rn((float)k, 255.f);
    for (int k = threadIdx.x; k < n_imgs && k < kLbSmemImgs; k += blockDim.x) simgs[k] = imgs[k];
    if (threadIdx.x == 0) {
        for (int s = 0; s < kLbStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kLbConsumers / 32);
        }
    }
    __syncthreads();
    // a block takes a contiguous range of output rows: almost always inside one image, whose
    // horizontal taps then sit in shared memory for the whole range
    const int per_block = (n_items + gridDim.x - 1) / gridDim.x;
    const int item_begin = blockIdx.x * per_block, item_end = min(n_items, item_begin + per_block);
    if (threadIdx.x >= kLbConsumers) {
        // ---- producer ----
        if (threadIdx.x != kLbConsumers) return;
        int k = 0;
        for (int item = item_begin; item < item_end; ++item, ++k) {
            const int stage = k % kLbStages, round = k / kLbStages;
            if (round > 0) mbar_wait(&empty[stage], (uint32_t)(round - 1) & 1u);
            const LbItem t = lb_item(n_imgs <= kLbSmemImgs ? simgs : imgs, item, oh);
            sitem[stage] = t;
            if (t.inside_y && t.tma_ok) {
                uint8_t *r0 = lb_rows + (size_t)(stage * 2) * row_stride;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                mbar_expect_tx(&full[stage], t.identity ? t.row_bytes : 2u * t.row_bytes);
                bulk_g2s(r0, t.g0, t.row_bytes, &full[stage]);
                if (!t.identity) bulk_g2s(r0 + row_stride, t.g1, t.row_bytes, &full[stage]);
            } else {
                mbar_arrive(&full[stage]);  // nothing to copy (padding row), or the consumers load it themselves
            }
        }
        return;
    }
    // ---- consumers ----
    const size_t plane = (size_t)oh * ow;
    const bool wide_rows = (ow % 8 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    LbCoef *scoef = reinterpret_cast<LbCoef *>(lb_rows + (size_t)kLbStages * 2 * row_stride);
    int coef_img = -1;
    int k = 0;
    for (int item = item_begin; item < item_end; ++item, ++k) {
        const int stage = k % kLbStages, round = k / kLbStages;
        const int img_now = item / oh;
        if (img_now != coef_img) {  // block-uniform; the loads overlap the wait for the first row of the image
            if (coef_img >= 0) consumer_sync();  // everyone is done with the previous image's taps
            for (int x = threadIdx.x; x < ow; x += kLbConsumers) scoef[x] = coefs[(size_t)img_now * ow + x];
            coef_img = img_now;
            consumer_sync();
        }
        mbar_wait(&full[stage], (uint32_t)round & 1u);
        const LbItem &t = sitem[stage];
        uint8_t *w0 = lb_rows + (size_t)(stage * 2) * row_stride;
        if (t.inside_y && !t.tma_ok) {  // unaligned source rows: ordinary loads (block-uniform branch)
            for (uint32_t q = threadIdx.x; q < t.row_bytes; q += kLbConsumers) {
                w0[q] = t.g0[q];
                if (!t.identity) w0[row_stride + q] = t.g1[q];
            }
            consumer_sync();
        }
        const size_t obase = (size_t)t.img * 3 * plane + (size_t)t.y * ow;
        if (!t.inside_y) {
            // padding row (44 % of the rows of a 16:9 camera): three constant rows, 16-byte stores
            const float pv = norm[pad & 255];
            if (wide_rows) {
                if (FP16) {
                    const uint32_t h2 = (uint32_t)__half_as_ushort(__float2half_rn(pv)) * 0x10001u;
                    const uint4 v = make_uint4(h2, h2, h2, h2);
                    const int per_plane = ow / 8;
                    for (int q = threadIdx.x; q < 3 * per_plane; q += kLbConsumers) {
                        const int c = q / per_plane, i = q - c * per_plane;
                        st_stream(reinterpret_cast<uint4 *>(reinterpret_cast<__half *>(out) + obase + c * plane) + i, v);
                    }
                } else {
                    const uint32_t fv = __float_as_uint(pv);
                    const uint4 v = make_uint4(fv, fv, fv, fv);
                    const int per_plane = ow / 4;
                    for (int q = threadIdx.x; q < 3 * per_plane; q += kLbConsumers) {
                        const int c = q / per_plane, i = q - c * per_plane;
                        st_stream(reinterpret_cast<uint4 *>(reinterpret_cast<float *>(out) + obase + c * plane) + i, v);
                    }
                }
            } else {
                for (int q = threadIdx.x; q < 3 * ow; q += kLbConsumers) {
                    const int c = q / ow, x = q - c * ow;
                    if (FP16)
                        reinterpret_cast<__half *>(out)[obase + c * plane + x] = __float2half_rn(pv);
                    else
                        reinterpret_cast<float *>(out)[obase + c * plane + x] = pv;
                }
            }
        } else {
            const uint8_t *r0 = w0;
            const uint8_t *r1 = t.identity ? w0 : w0 + row_stride;  // single staged row; weights (2048, 0) copy it exactly
            const int cw0 = t.cy.w0, cw1 = t.cy.w1;
            // adjacent lanes take adjacent output pixels: their taps are ~10 bytes apart in the staged row,
            // the mapping with the fewest shared-memory bank conflicts short of re-striding the row
            for (int x = threadIdx.x; x < ow; x += kLbConsumers) {
                const uint2 q = *reinterpret_cast<const uint2 *>(scoef + x);
                const LbCoef cx = coef_from_words(q.x, q.y);
                int v[3] = {pad, pad, pad};
                if (cx.o0 >= 0) {
                    if ((cx.o1 == cx.o0 + 3 || cx.w1 == 0) && cx.w0 >= 0 && cx.w1 >= 0) {
                        // the two taps are 6 adjacent bytes (or the right one has weight 0): three aligned words per
                        // staged row, a funnel shift to the tap's byte offset, one byte-permute + one 2-way dot
                        // product per channel (weights as int16 pairs, pixels as bytes)
                        const uint32_t wpack = (uint32_t)(uint16_t)cx.w0 | ((uint32_t)(uint16_t)cx.w1 << 16);
                        const int a = cx.o0 & ~3;
                        const uint32_t sh = 8u * (uint32_t)(cx.o0 & 3);
                        int h[2][3];  // unsigned dot product: weights are 0..2048, pixels 0..255
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const uint32_t *q = reinterpret_cast<const uint32_t *>((j ? r1 : r0) + a);
                            const uint32_t q0 = q[0], q1 = q[1], q2 = q[2];
                            const uint32_t lo = __funnelshift_r(q0, q1, sh), hi = __funnelshift_r(q1, q2, sh);  // bytes o0..o0+7
                            h[j][0] = (int)__dp2a_lo(wpack, __byte_perm(lo, hi, 0x4430), 0u);  // (byte 0, byte 3)
                            h[j][1] = (int)__dp2a_lo(wpack, __byte_perm(lo, hi, 0x4441), 0u);  // (byte 1, byte 4)
                            h[j][2] = (int)__dp2a_lo(wpack, __byte_perm(lo, hi, 0x4452), 0u);  // (byte 2, byte 5)
                        }
#pragma unroll
                        for (int c = 0; c < 3; ++c) v[c] = linear_vblend(h[0][c], h[1][c], cw0, cw1);
                    } else {
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const int h0 = r0[cx.o0 + c] * cx.w0 + r0[cx.o1 + c] * cx.w1;
                            const int h1 = r1[cx.o0 + c] * cx.w0 + r1[cx.o1 + c] * cx.w1;
                            v[c] = linear_vblend(h0, h1, cw0, cw1);
                        }
                    }
                }
                const float fr = norm[v[2]], fg = norm[v[1]], fb = norm[v[0]];
                if (FP16) {
                    __half *o = reinterpret_cast<__half *>(out) + obase + x;
                    o[0] = __float2half_rn(fr);
                    o[plane] = __float2half_rn(fg);
                    o[2 * plane] = __float2half_rn(fb);
                } else {
                    float *o = reinterpret_cast<float *>(out) + obase + x;
                    o[0] = fr;
                    o[plane] = fg;
                    o[2 * plane] = fb;
                }
            }
        }
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(&empty[stage]);  // this warp is done with the stage
    }
}

}  // namespace bv

using namespace bv;

extern "C" int bv_resize_linear(bv_ctx *ctx, const uint8_t *src_dev, int src_h, int src_w, uint8_t *dst_dev, int dst_h,
                                int dst_w, int channels, int batch) {
    BV_REQUIRE(ctx && src_dev && dst_dev, "null argument");
    BV_REQUIRE(src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0 && batch > 0, "sizes must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t total = (size_t)batch * dst_h * dst_w;
    const double sx = (double)src_w / dst_w, sy = (double)src_h / dst_h;
    const int grid = grid_for(ctx, total, 256, 8);
    if (channels == 3)
        BV_LAUNCH(ctx, resize_kernel<3>, grid, 256, 0, src_dev, src_h, src_w, dst_dev, dst_h, dst_w, sx, sy, total);
    else
        BV_LAUNCH(ctx, resize_kernel<1>, grid, 256, 0, src_dev, src_h, src_w, dst_dev, dst_h, dst_w, sx, sy, total);
    return BV_OK;
}

extern "C" int bv_letterbox(bv_ctx *ctx, const uint8_t *const *srcs_host, const int32_t *heights_host,
                            const int32_t *widths_host, int n, void *out_dev, int out_h, int out_w, int pad_value,
                            int out_fp16) {
    BV_REQUIRE(ctx && srcs_host && heights_host && widths_host && out_dev, "null argument");
    BV_REQUIRE(n > 0 && n <= 65535 && out_h > 0 && out_w > 0 && out_h <= 65535, "bad batch or output size");
    BV_CUDA(cudaSetDevice(ctx->device));
    // cv2.copyMakeBorder saturates the border value to uint8; the kernels index a 256-entry table with it
    pad_value = pad_value < 0 ? 0 : (pad_value > 255 ? 255 : pad_value);
    static thread_local LetterboxImg descs[256];
    memset(descs, 0, sizeof(LetterboxImg) * (size_t)(n > 0 && n <= 256 ? n : 0));  // padding bytes compare equal
    BV_REQUIRE(n <= 256, "at most 256 images per call");
    for (int i = 0; i < n; ++i) {
        const int h = heights_host[i], w = widths_host[i];
        BV_REQUIRE(srcs_host[i] && h > 0 && w > 0, "bad source image");
        // Ultralytics LetterBox(auto=False, scaleup=True, center=True); python round() is
        // round-half-even == nearbyint in the default rounding mode
        const double r = fmin((double)out_h / h, (double)out_w / w);
        const int uw = (int)nearbyint(w * r), uh = (int)nearbyint(h * r);
        const double dw = (out_w - uw) / 2.0, dh = (out_h - uh) / 2.0;
        LetterboxImg &d = descs[i];
        d.src = srcs_host[i];
        d.sh = h;
        d.sw = w;
        d.uh = uh;
        d.uw = uw;
        d.top = (int)nearbyint(dh - 0.1);
        d.left = (int)nearbyint(dw - 0.1);
        d.scale_x = (double)w / uw;
        d.scale_y = (double)h / uh;
        BV_REQUIRE(uw > 0 && uh > 0, "degenerate letterbox size");
    }
    const size_t lb_bytes = sizeof(LetterboxImg) * kLbMaxImgs + sizeof(LbCoef) * (size_t)n * out_w + 16;
    const bool regrown = ctx->scratch_bytes[SCR_LETTERBOX] < lb_bytes;
    BV_TRY(ensure_scratch(ctx, SCR_LETTERBOX, lb_bytes));
    LetterboxImg *d_descs = (LetterboxImg *)ctx->scratch[SCR_LETTERBOX];
    // the same cameras frame after frame: descriptors and tap table are already on the device
    if (!ctx->lb_cache) ctx->lb_cache = calloc(1, sizeof(LetterboxImg) * kLbMaxImgs);
    const bool same = !regrown && ctx->lb_cache && ctx->lb_cache_n == n && ctx->lb_cache_ow == out_w && ctx->lb_cache_oh == out_h &&
                      memcmp(ctx->lb_cache, descs, sizeof(LetterboxImg) * n) == 0;
    if (!same) {
        BV_CUDA(cudaMemcpyAsync(d_descs, descs, sizeof(LetterboxImg) * n, cudaMemcpyHostToDevice, ctx->stream));
        ctx->lb_cache_n = 0;  // the tap table is rebuilt below (or unused by the gather kernel)
    }
    bool fits = true;  // the staged kernel holds two source rows and the tap table in shared memory
    for (int i = 0; i < n; ++i) fits = fits && (size_t)widths_host[i] * 3 <= (size_t)kLbMaxRowBytes;
    static const bool use_tma = getenv("BV_LETTERBOX_GATHER") == nullptr;
    int max_w = 0;
    for (int i = 0; i < n; ++i) max_w = widths_host[i] > max_w ? widths_host[i] : max_w;
    const int row_stride = (max_w * 3 + 127) & ~127;
    const size_t smem = (size_t)kLbStages * 2 * row_stride + sizeof(LbCoef) * (size_t)out_w;
    if (fits && use_tma && smem > (size_t)ctx->lb_smem_set) {
        // the tap table grows with out_w: past the device's opt-in shared memory (out_w of ~24 000 on a
        // B200) the gather kernel, which needs none, takes the call
        int optin = 0;
        BV_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
        cudaFuncAttributes fa16, fa32;
        BV_CUDA(cudaFuncGetAttributes(&fa16, letterbox_tma_kernel<true>));
        BV_CUDA(cudaFuncGetAttributes(&fa32, letterbox_tma_kernel<false>));
        const size_t static_smem = fa16.sharedSizeBytes > fa32.sharedSizeBytes ? fa16.sharedSizeBytes : fa32.sharedSizeBytes;
        if (smem + static_smem > (size_t)optin) {
            fits = false;
        } else {
            BV_CUDA(cudaFuncSetAttribute(letterbox_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            BV_CUDA(cudaFuncSetAttribute(letterbox_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            ctx->lb_smem_set = (int)smem;
        }
    }
    if (fits && use_tma) {
        const int n_items = out_h * n;
        // persistent blocks: as many as fit next to each other (dynamic rows + ~14 KB of static tables)
        int per_sm = (int)((208 * 1024) / (smem + 6 * 1024));
        per_sm = per_sm < 1 ? 1 : (per_sm > 6 ? 6 : per_sm);
        int grid = ctx->sm_count * per_sm;
        if (grid > n_items) grid = n_items;
        LbCoef *d_coefs = (LbCoef *)(d_descs + kLbMaxImgs);
        if (!same) {
            BV_LAUNCH(ctx, letterbox_coef_kernel, (n * out_w + 255) / 256, 256, 0, d_descs, d_coefs, out_w, n * out_w);
            if (ctx->lb_cache) {
                memcpy(ctx->lb_cache, descs, sizeof(LetterboxImg) * n);
                ctx->lb_cache_n = n;
                ctx->lb_cache_ow = out_w;
                ctx->lb_cache_oh = out_h;
            }
        }
        if (out_fp16)
            BV_LAUNCH(ctx, letterbox_tma_kernel<true>, grid, kLbConsumers + 32, smem, d_descs, n, d_coefs, out_dev, out_h, out_w,
                      pad_value, n_items, row_stride);
        else
            BV_LAUNCH(ctx, letterbox_tma_kernel<false>, grid, kLbConsumers + 32, smem, d_descs, n, d_coefs, out_dev, out_h, out_w,
                      pad_value, n_items, row_stride);
        return BV_OK;
    }
    dim3 grid((out_w + 255) / 256, out_h, n);
    if (out_fp16)
        BV_LAUNCH(ctx, letterbox_kernel<true>, grid, 256, 0, d_descs, out_dev, out_h, out_w, pad_value);
    else
        BV_LAUNCH(ctx, letterbox_kernel<false>, grid, 256, 0, d_descs, out_dev, out_h, out_w, pad_value);
    return BV_OK;
}
