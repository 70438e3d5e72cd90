// canny.cu -- cv2.Canny(src, threshold1, threshold2, apertureSize, L2gradient) on uint8 grey or BGR frames, bit-exact
// against OpenCV 4.13.0 (oracle/canny_np.py restates the rules; DESIGN.md section 2 lists them).
//
//   canny_nms_kernel   one block per 64 x 16 tile: the source tile plus a halo of aperture/2 + 1 pixels (replicated at
//                      the frame's edges) goes to shared memory; dx, dy and the magnitude of the selected channel are
//                      computed on the tile plus a one-pixel ring (magnitude 0 outside the frame); non-maximum
//                      suppression and the two thresholds give the candidate and strong bits, one __ballot_sync word per
//                      warp and 32 pixels of a row, in the morph.cuh layout.  The magnitude never leaves the SM.
//   hysteresis         8-connected union-find of the candidate bits (union_bits: ccl.cu's init + merge kernels);
//                      canny_seed_kernel marks the root of every run that holds a strong pixel in a per-frame bitmap;
//                      canny_write_kernel writes 255 on every candidate run whose root is marked, 0 elsewhere.
//
// The union-find stays inside each frame (per-frame parent arrays, no merge across a frame's first row), so the frames
// of a batch never interact.  A long candidate chain costs union operations, not rounds: there is no iterative
// dilation.  HBM traffic: the source (C B/px) read once, 1/4 B/px of bits, the parent entries of candidate runs, and the
// 1 B/px output.
#include <math.h>

#include "morph.cuh"

namespace bv {

namespace {

constexpr int kTileW = 64;  // two bit words per tile row
constexpr int kTileH = 16;
constexpr int kThreads = 256;
// tan(22.5 deg) in 15-bit fixed point, as cv2's Canny rounds it
constexpr int kTG22 = (int)(0.4142135623730950488016887242097 * (1 << 15) + 0.5);

// the separable Sobel kernel of an aperture: binomial smoothing row and derivative row
__host__ __device__ constexpr int sobel_smooth(int ap, int i) {
    return ap == 3 ? (i == 1 ? 2 : 1)
         : ap == 5 ? (i == 2 ? 6 : (i == 1 || i == 3) ? 4 : 1)
                   : (i == 3 ? 20 : (i == 2 || i == 4) ? 15 : (i == 1 || i == 5) ? 6 : 1);
}
__host__ __device__ constexpr int sobel_deriv(int ap, int i) {
    return ap == 3 ? i - 1
         : ap == 5 ? (i == 0 ? -1 : i == 1 ? -2 : i == 2 ? 0 : i == 3 ? 2 : 1)
                   : (i == 0 ? -1 : i == 1 ? -4 : i == 2 ? -5 : i == 3 ? 0 : i == 4 ? 5 : i == 5 ? 4 : 1);
}

// s / 16 rounded half to even: cv2's CV_16S Sobel with scale 1/16 (aperture 7) rounds the exact float quotient with cvRound
__device__ __forceinline__ int div16_half_even(int s) {
    const int q = s >> 4, r = s & 15;
    return q + ((r > 8) | ((r == 8) & (q & 1)));
}

}  // namespace

template <int AP, int CH, bool L2>
__global__ void __launch_bounds__(kThreads) canny_nms_kernel(const uint8_t *__restrict__ src, uint32_t *__restrict__ cand,
                                                             uint32_t *__restrict__ strong, int height, int width, int wpr,
                                                             int tiles_x, uint32_t tiles_per_frame, uint32_t n_tiles, int low,
                                                             int high) {
    constexpr int R = AP / 2 + 1;                         // source halo: Sobel radius + the magnitude ring
    constexpr int SW = kTileW + 2 * R, SH = kTileH + 2 * R;
    constexpr int GW = kTileW + 2, GH = kTileH + 2;         // tile + ring of gradients
    constexpr int ROW_BYTES = SW * CH;
    __shared__ uint8_t s_src[SH * ROW_BYTES];
    __shared__ int s_mag[GH * GW];
    __shared__ uint32_t s_dxy[GH * GW];                    // dx (low 16 bits), dy (high 16 bits) of the selected channel
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const uint32_t f = t / tiles_per_frame;
        const uint32_t rem = t - f * tiles_per_frame;
        const int y0 = (int)(rem / (uint32_t)tiles_x) * kTileH;
        const int x0 = (int)(rem % (uint32_t)tiles_x) * kTileW;
        const uint8_t *fsrc = src + (size_t)f * height * width * CH;
        __syncthreads();  // the previous tile's readers are done with shared memory
        for (int i = threadIdx.x; i < SH * ROW_BYTES; i += kThreads) {
            const int sy = i / ROW_BYTES, b = i - sy * ROW_BYTES;
            const int sx = b / CH, c = b - sx * CH;
            const int y = min(max(y0 - R + sy, 0), height - 1);   // BORDER_REPLICATE
            const int x = min(max(x0 - R + sx, 0), width - 1);
            s_src[i] = fsrc[((size_t)y * width + x) * CH + c];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < GH * GW; i += kThreads) {
            const int gy = i / GW, gx = i - gy * GW;
            const int y = y0 - 1 + gy, x = x0 - 1 + gx;
            int m = 0;
            uint32_t dxy = 0;
            if (y >= 0 && y < height && x >= 0 && x < width) {
#pragma unroll
                for (int c = 0; c < CH; ++c) {
                    int dx = 0, dy = 0;
#pragma unroll
                    for (int j = 0; j < AP; ++j) {
                        const uint8_t *row = s_src + (gy + j) * ROW_BYTES + gx * CH + c;
                        int rd = 0, rs = 0;
#pragma unroll
                        for (int k = 0; k < AP; ++k) {
                            const int v = row[k * CH];
                            rd += sobel_deriv(AP, k) * v;
                            rs += sobel_smooth(AP, k) * v;
                        }
                        dx += sobel_smooth(AP, j) * rd;
                        dy += sobel_deriv(AP, j) * rs;
                    }
                    if (AP == 7) {
                        dx = div16_half_even(dx);
                        dy = div16_half_even(dy);
                    }
                    const int mc = L2 ? dx * dx + dy * dy : abs(dx) + abs(dy);
                    if (c == 0 || mc > m) {  // the first channel wins a tie
                        m = mc;
                        dxy = ((uint32_t)dx & 0xFFFFu) | ((uint32_t)dy << 16);
                    }
                }
            }
            s_mag[i] = m;
            s_dxy[i] = dxy;
        }
        __syncthreads();
        // one warp = 32 pixels of one tile row = one bit word
        for (int seg = warp; seg < kTileH * (kTileW / 32); seg += kThreads / 32) {
            const int ty = seg / (kTileW / 32), tw = seg - ty * (kTileW / 32);
            const int y = y0 + ty, x = x0 + tw * 32 + lane;
            bool is_cand = false, is_strong = false;
            if (y < height && x < width) {
                const int gi = (ty + 1) * GW + tw * 32 + lane + 1;
                const int m = s_mag[gi];
                if (m > low) {
                    const uint32_t dxy = s_dxy[gi];
                    const int dx = (int)(int16_t)(dxy & 0xFFFFu), dy = (int)(int16_t)(dxy >> 16);
                    const int ax = abs(dx), ay = abs(dy);
                    const int tg22x = ax * kTG22;
                    const int tg67x = tg22x + (ax << 16);
                    const int ay15 = ay << 15;
                    bool keep;
                    if (ay15 < tg22x) {                      // horizontal gradient
                        keep = m > s_mag[gi - 1] && m >= s_mag[gi + 1];
                    } else if (ay15 > tg67x) {               // vertical
                        keep = m > s_mag[gi - GW] && m >= s_mag[gi + GW];
                    } else {                                 // diagonal
                        const int s = ((dx ^ dy) < 0) ? -1 : 1;
                        keep = m > s_mag[gi - GW - s] && m > s_mag[gi + GW + s];
                    }
                    is_cand = keep;
                    is_strong = keep && m > high;
                }
            }
            const uint32_t cw = __ballot_sync(0xFFFFFFFFu, is_cand);
            const uint32_t sw = __ballot_sync(0xFFFFFFFFu, is_strong);
            const int wx = x0 / 32 + tw;
            if (lane == 0 && y < height && wx < wpr) {
                const size_t wi = ((size_t)f * height + y) * wpr + wx;
                cand[wi] = cw;
                strong[wi] = sw;
            }
        }
    }
}

// every candidate run holding a strong pixel marks its component's root in the frame's bitmap (bit = pixel index)
__global__ void __launch_bounds__(256) canny_seed_kernel(const uint32_t *__restrict__ cand, const uint32_t *__restrict__ strong,
                                                         const int *__restrict__ parent, uint32_t *__restrict__ roots,
                                                         int height, int width, int wpr, uint32_t total_words,
                                                         uint32_t root_words) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        uint32_t s = strong[i];
        if (!s) continue;
        const uint32_t c = cand[i];  // strong bits are candidate bits
        const WordPos wp = word_pos(i, wpr, height);
        const uint32_t f = (wp.row - wp.y) / (uint32_t)height;
        const int *fp = parent + (size_t)(wp.row - wp.y) * width;
        while (s) {
            const int st = run_start(c, __ffs(s) - 1);
            s &= ~run_mask(c, st);  // one root look-up per run
            const int r = find_root(fp, wp.y * width + wp.wx * 32 + st);
            atomicOr(&roots[(size_t)f * root_words + (r >> 5)], 1u << (r & 31));
        }
    }
}

// dst = 255 on the candidate runs whose root is marked, 0 elsewhere; every byte of the frame is written
__global__ void __launch_bounds__(256) canny_write_kernel(const uint32_t *__restrict__ cand, const int *__restrict__ parent,
                                                          const uint32_t *__restrict__ roots, uint8_t *__restrict__ dst,
                                                          int height, int width, int wpr, uint32_t total_words,
                                                          uint32_t root_words) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const WordPos wp = word_pos(i, wpr, height);
        uint32_t rest = cand[i], out = 0;
        if (rest) {
            const uint32_t *fr = roots + (size_t)((wp.row - wp.y) / (uint32_t)height) * root_words;
            const int *fp = parent + (size_t)(wp.row - wp.y) * width;
            while (rest) {
                const int st = __ffs(rest) - 1;
                const uint32_t run = run_mask(rest, st);
                rest &= ~run;
                const int r = find_root(fp, wp.y * width + wp.wx * 32 + st);
                if ((fr[r >> 5] >> (r & 31)) & 1u) out |= run;
            }
        }
        store_mask_word(dst + (size_t)wp.row * width + (size_t)wp.wx * 32, min(32, width - wp.wx * 32), out);
    }
}

// cvFloor on x86-64: INT_MIN for NaN and for anything that does not fit in int32
static int cv_floor(double v) {
    const double f = floor(v);
    return (f >= -2147483648.0 && f < 2147483648.0) ? (int)f : INT32_MIN;
}

template <int AP, int CH, bool L2>
static int launch_nms(bv_ctx *ctx, const uint8_t *src, uint32_t *cand, uint32_t *strong, int batch, int height, int width,
                      int low, int high) {
    const int tiles_x = (width + kTileW - 1) / kTileW;
    const uint32_t tiles_per_frame = (uint32_t)tiles_x * (uint32_t)((height + kTileH - 1) / kTileH);
    const uint32_t n_tiles = tiles_per_frame * (uint32_t)batch;  // <= the word count, < 2^31
    const uint32_t cap = (uint32_t)ctx->sm_count * 8;
    const int grid = (int)(n_tiles < cap ? n_tiles : cap);
    BV_LAUNCH(ctx, (canny_nms_kernel<AP, CH, L2>), grid, kThreads, 0, src, cand, strong, height, width, words_per_row(width),
              tiles_x, tiles_per_frame, n_tiles, low, high);
    return BV_OK;
}

template <int AP>
static int launch_nms_ap(bv_ctx *ctx, const uint8_t *src, uint32_t *cand, uint32_t *strong, int batch, int height, int width,
                         int channels, bool l2, int low, int high) {
    if (channels == 1)
        return l2 ? launch_nms<AP, 1, true>(ctx, src, cand, strong, batch, height, width, low, high)
                  : launch_nms<AP, 1, false>(ctx, src, cand, strong, batch, height, width, low, high);
    return l2 ? launch_nms<AP, 3, true>(ctx, src, cand, strong, batch, height, width, low, high)
              : launch_nms<AP, 3, false>(ctx, src, cand, strong, batch, height, width, low, high);
}

}  // namespace bv

using namespace bv;

extern "C" int bv_canny(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width, int channels,
                        double threshold1, double threshold2, int aperture_size, int l2_gradient) {
    BV_REQUIRE(ctx && src_dev && dst_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_REQUIRE(aperture_size == 3 || aperture_size == 5 || aperture_size == 7, "aperture_size must be 3, 5 or 7");
    const size_t px = (size_t)batch * height * width;
    const uintptr_t s0 = (uintptr_t)src_dev, d0 = (uintptr_t)dst_dev;
    BV_REQUIRE(d0 + px <= s0 || s0 + px * channels <= d0, "src and dst overlap: in-place Canny is not supported");
    const int wpr = words_per_row(width);
    const size_t total_words = (size_t)batch * height * wpr;
    BV_REQUIRE((size_t)height * width < (1ull << 31) && total_words < (1ull << 31),
               "frame or batch too large for 32-bit indices");
    BV_CUDA(cudaSetDevice(ctx->device));

    // thresholds as cv2.Canny reads them (oracle/canny_np.py: thresholds)
    double lo = threshold1, hi = threshold2;
    if (lo > hi) {
        const double t = lo;
        lo = hi;
        hi = t;
    }
    if (aperture_size == 7) {  // cv2 scales the aperture-7 Sobel by 1/16 and the thresholds with it
        lo /= 16.0;
        hi /= 16.0;
    }
    if (l2_gradient) {
        lo = lo < 32767.0 ? lo : 32767.0;  // std::min(32767.0, t): NaN becomes 32767
        hi = hi < 32767.0 ? hi : 32767.0;
        if (lo > 0) lo *= lo;
        if (hi > 0) hi *= hi;
    }
    const int low = cv_floor(lo), high = cv_floor(hi);

    const uint32_t root_words = (uint32_t)(((size_t)height * width + 31) / 32);
    BV_TRY(ensure_scratch(ctx, SCR_BITS_A, total_words * 8));
    BV_TRY(ensure_scratch(ctx, SCR_BITS_B, (size_t)batch * root_words * 4));
    uint32_t *cand = (uint32_t *)ctx->scratch[SCR_BITS_A];
    uint32_t *strong = cand + total_words;
    uint32_t *roots = (uint32_t *)ctx->scratch[SCR_BITS_B];
    LabelScratch ls;
    BV_TRY(label_scratch(ctx, batch, height, width, &ls));

    const bool l2 = l2_gradient != 0;
    if (aperture_size == 3)
        BV_TRY(launch_nms_ap<3>(ctx, src_dev, cand, strong, batch, height, width, channels, l2, low, high));
    else if (aperture_size == 5)
        BV_TRY(launch_nms_ap<5>(ctx, src_dev, cand, strong, batch, height, width, channels, l2, low, high));
    else
        BV_TRY(launch_nms_ap<7>(ctx, src_dev, cand, strong, batch, height, width, channels, l2, low, high));
    BV_TRY(union_bits(ctx, cand, batch, height, width, ls));
    BV_CUDA(cudaMemsetAsync(roots, 0, (size_t)batch * root_words * 4, ctx->stream));
    const int gw = grid_for(ctx, total_words, 256, 8);
    BV_LAUNCH(ctx, canny_seed_kernel, gw, 256, 0, cand, strong, ls.parent, roots, height, width, wpr, (uint32_t)total_words,
              root_words);
    BV_LAUNCH(ctx, canny_write_kernel, gw, 256, 0, cand, ls.parent, roots, dst_dev, height, width, wpr,
              (uint32_t)total_words, root_words);
    return BV_OK;
}
