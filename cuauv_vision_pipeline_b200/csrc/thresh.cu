// thresh.cu -- cv2.threshold with THRESH_OTSU / THRESH_TRIANGLE and cv2.adaptiveThreshold on uint8 frames, matching
// OpenCV 4.13.0 (oracle/threshold_np.py restates the rules; include/b200vision.h and DESIGN.md section 2 list them).
//
//   thresh_hist_kernel          16 bytes per thread into a block histogram in shared memory; the lanes of a warp that
//                               hold the same value add once (__match_any_sync), so a constant frame does not serialise
//                               32 atomics on one bin.  Non-zero bins are added to the frame's global histogram.
//   thresh_search_kernel        one thread per frame: cv2's Otsu or Triangle loop over the 256 bins (double, or float32
//                               for Triangle, every operation rounded on its own), the threshold written to thresh_dev.
//   thresh_apply_kernel         cv2.threshold's 8-bit rule with each frame's threshold read on the device: op1_apply,
//                               the same arithmetic as bv_threshold.
//   adapt_prefix_kernel         MEAN_C: one block per row, the row's inclusive prefix sums (uint32) in scratch.
//   adapt_mean_cols_kernel      MEAN_C: one thread per column and strip of rows.  A row's window sum is two prefix
//                               reads plus the replicated edge pixels counted explicitly; the column window slides down
//                               the strip.  Strips are as tall as the window where that leaves enough blocks to fill
//                               the device (a pixel then costs O(1) in k), shorter where it does not.  The mean and the
//                               compare are fused.
//   adapt_gauss_rows_kernel     GAUSSIAN_C: float32 row filter of a 256-pixel segment and its halo staged in shared
//                               memory, taps in tap order, into a float32 plane.
//   adapt_gauss_cols_kernel     GAUSSIAN_C: the column filter of that plane fused with cvRound and the compare.
#include <math.h>

#include <vector>

#include "common.cuh"
#include "pointwise.cuh"

namespace bv {

namespace {

constexpr int kHistThreads = 256;
constexpr int kSearchThreads = 64;
constexpr int kApplyThreads = 256;
constexpr int kRowThreads = 256;
constexpr int kColThreads = 128;
constexpr int kMinStrip = 32;  // rows of a MEAN_C column strip, at least

// cvRound of a double as OpenCV computes it on x86-64: half to even, INT_MIN where the value has no int32
int cv_round(double v) {
    const double r = nearbyint(v);
    return (r >= -2147483648.0 && r <= 2147483647.0) ? (int)r : INT32_MIN;
}

int saturate_u8(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }

bool disjoint(const void *a, size_t na, const void *b, size_t nb) {
    const uintptr_t pa = (uintptr_t)a, pb = (uintptr_t)b;
    return pa + na <= pb || pb + nb <= pa;
}

}  // namespace

__global__ void __launch_bounds__(kHistThreads) thresh_hist_kernel(const uint8_t *__restrict__ src, uint32_t frame_px,
                                                                   int *__restrict__ hist) {
    __shared__ int s_hist[256];
    const int f = blockIdx.y;
    for (int i = threadIdx.x; i < 256; i += kHistThreads) s_hist[i] = 0;
    __syncthreads();
    const uint8_t *fsrc = src + (size_t)f * frame_px;
    const bool vec = aligned16(fsrc);
    const uint32_t n_vec = (frame_px + 15) / 16;
    const int lane = threadIdx.x & 31;
    for (uint32_t v0 = blockIdx.x * kHistThreads; v0 < n_vec; v0 += gridDim.x * kHistThreads) {
        const uint32_t v = v0 + threadIdx.x;  // the whole block iterates together: __match_any_sync sees every lane
        const uint32_t p0 = v * 16;
        uint32_t w[4] = {0, 0, 0, 0};
        int nb = 0;
        if (v < n_vec) {
            if (vec && p0 + 16 <= frame_px) {
                const uint4 q = ld_stream(reinterpret_cast<const uint4 *>(fsrc + p0));
                w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
                nb = 16;
            } else {
                for (; nb < 16 && p0 + nb < frame_px; ++nb) w[nb >> 2] |= (uint32_t)fsrc[p0 + nb] << (8 * (nb & 3));
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int b = i < nb ? (int)BV_GETB(w, i) : 256;  // 256: no byte here
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, b);
            if (b < 256 && lane == __ffs(peers) - 1) atomicAdd(&s_hist[b], __popc(peers));
        }
    }
    __syncthreads();
    int *fh = hist + (size_t)f * 256;
    for (int i = threadIdx.x; i < 256; i += kHistThreads)
        if (s_hist[i]) atomicAdd(&fh[i], s_hist[i]);
}

// cv2's getThreshVal_Otsu on 8 bits, every double operation rounded on its own
__device__ double otsu_threshold(const int *h, uint32_t frame_px) {
    const double eps = 1.1920928955078125e-07;  // FLT_EPSILON
    const double scale = __ddiv_rn(1.0, (double)frame_px);
    double mu = 0;
    for (int i = 0; i < 256; ++i) mu = __dadd_rn(mu, __dmul_rn((double)i, (double)h[i]));  // exact: integers < 2^53
    mu = __dmul_rn(mu, scale);
    double mu1 = 0, q1 = 0, max_sigma = 0, max_val = 0;
    for (int i = 0; i < 256; ++i) {
        const double p = __dmul_rn((double)h[i], scale);
        mu1 = __dmul_rn(mu1, q1);
        q1 = __dadd_rn(q1, p);
        const double q2 = __dadd_rn(1.0, -q1);
        if (fmin(q1, q2) < eps || fmax(q1, q2) > __dadd_rn(1.0, -eps)) continue;
        mu1 = __ddiv_rn(__dadd_rn(mu1, __dmul_rn((double)i, p)), q1);
        const double mu2 = __ddiv_rn(__dadd_rn(mu, -__dmul_rn(q1, mu1)), q2);
        const double d = __dadd_rn(mu1, -mu2);
        const double sigma = __dmul_rn(__dmul_rn(__dmul_rn(q1, q2), d), d);
        if (sigma > max_sigma) {
            max_sigma = sigma;
            max_val = i;
        }
    }
    return max_val;
}

// cv2's getThreshVal_Triangle_8u: integer bounds and peak, float32 distance search, no FMA
__device__ double triangle_threshold(const int *h) {
    int left = 0, right = 0, peak = 0, max = 0;
    for (int i = 0; i < 256; ++i)
        if (h[i] > 0) {
            left = i;
            break;
        }
    if (left > 0) --left;
    for (int i = 255; i > 0; --i)
        if (h[i] > 0) {
            right = i;
            break;
        }
    if (right < 255) ++right;
    for (int i = 0; i < 256; ++i)
        if (h[i] > max) {
            max = h[i];
            peak = i;
        }
    const bool flipped = peak - left < right - peak;
    if (flipped) {
        left = 255 - right;
        peak = 255 - peak;
    }
    int thresh = left;
    const float a = (float)max, b = (float)(left - peak);
    float dist = 0;
    for (int i = left + 1; i <= peak; ++i) {
        const float t = __fadd_rn(__fmul_rn(a, (float)i), __fmul_rn(b, (float)h[flipped ? 255 - i : i]));
        if (t > dist) {
            dist = t;
            thresh = i;
        }
    }
    --thresh;
    return flipped ? 255 - thresh : thresh;
}

__global__ void __launch_bounds__(kSearchThreads) thresh_search_kernel(const int *__restrict__ hist, int batch,
                                                                       uint32_t frame_px, int method,
                                                                       double *__restrict__ thresh) {
    const int f = blockIdx.x * kSearchThreads + threadIdx.x;
    if (f >= batch) return;
    const int *h = hist + (size_t)f * 256;
    thresh[f] = method == BV_THRESH_OTSU ? otsu_threshold(h, frame_px) : triangle_threshold(h);
}

// src and dst may be the same buffer: every byte is read once, by the thread that writes it
template <bool VEC>
__global__ void __launch_bounds__(kApplyThreads) thresh_apply_kernel(const uint8_t *src, uint8_t *dst, uint32_t frame_px,
                                                                     const double *__restrict__ thresh, int maxval,
                                                                     int type) {
    const int f = blockIdx.y;
    // cv2.threshold on 8 bits, as bv_threshold: thresh floored, clamped for TRUNC
    Op1Params prm{(int)floor(thresh[f]), maxval, type};
    if (type == BV_THRESH_TRUNC) prm.a = prm.a < 0 ? 0 : (prm.a > 255 ? 255 : prm.a);
    const uint8_t *fsrc = src + (size_t)f * frame_px;
    uint8_t *fdst = dst + (size_t)f * frame_px;
    const uint32_t stride = gridDim.x * kApplyThreads;
    if (VEC) {
        for (uint32_t g = blockIdx.x * kApplyThreads + threadIdx.x; g < frame_px / 16; g += stride) {
            const uint4 v = reinterpret_cast<const uint4 *>(fsrc)[g];
            const uint32_t in[4] = {v.x, v.y, v.z, v.w};
            uint32_t out[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 16; ++j) BV_PUTB(out, j, op1_apply(OP1_THRESH, prm, BV_GETB(in, j), nullptr));
            reinterpret_cast<uint4 *>(fdst)[g] = make_uint4(out[0], out[1], out[2], out[3]);
        }
    }
    const uint32_t first = VEC ? frame_px / 16 * 16 : 0;
    for (uint32_t i = first + blockIdx.x * kApplyThreads + threadIdx.x; i < frame_px; i += stride)
        fdst[i] = (uint8_t)op1_apply(OP1_THRESH, prm, fsrc[i], nullptr);
}

// the adaptive compare: cv2's 768-entry table, src - mean > -idelta (BINARY) or <= -idelta (BINARY_INV)
__device__ __forceinline__ uint8_t adapt_out(int x, int mean, int neg_delta, bool inv, int maxval) {
    return ((x - mean > neg_delta) != inv) ? (uint8_t)maxval : (uint8_t)0;
}

__global__ void __launch_bounds__(kRowThreads) adapt_prefix_kernel(const uint8_t *__restrict__ src, int width,
                                                                   uint32_t *__restrict__ prefix) {
    __shared__ uint32_t s_warp[kRowThreads / 32];
    const size_t row = blockIdx.x;
    const uint8_t *rsrc = src + row * width;
    uint32_t *rp = prefix + row * (width + 1);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) rp[0] = 0;
    uint32_t carry = 0;
    for (int x0 = 0; x0 < width; x0 += kRowThreads) {
        const int x = x0 + threadIdx.x;
        const uint32_t v = x < width ? rsrc[x] : 0;
        uint32_t incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        uint32_t before = carry, total = carry;
        for (int w = 0; w < kRowThreads / 32; ++w) {
            if (w < warp) before += s_warp[w];
            total += s_warp[w];
        }
        if (x < width) rp[x + 1] = before + incl;
        carry = total;
        __syncthreads();  // s_warp is rewritten by the next chunk
    }
}

__global__ void __launch_bounds__(kColThreads) adapt_mean_cols_kernel(const uint8_t *__restrict__ src,
                                                                      const uint32_t *__restrict__ prefix,
                                                                      uint8_t *__restrict__ dst, int height, int width,
                                                                      int radius, int strip, int strips, int col_blocks,
                                                                      float scale, double dscale, int neg_delta, int inv,
                                                                      int maxval) {
    const int cb = blockIdx.x % col_blocks;
    const int s = (blockIdx.x / col_blocks) % strips;
    const size_t f = blockIdx.x / ((size_t)col_blocks * strips);
    const int x = cb * kColThreads + threadIdx.x;
    if (x >= width) return;
    const uint8_t *fsrc = src + f * height * width;
    const uint32_t *fp = prefix + f * height * (width + 1);
    uint8_t *fdst = dst + f * height * width;
    // the row window [x - radius, x + radius]: the columns inside the frame through the prefix sums, the replicated
    // first and last pixels counted explicitly
    const int lo = x - radius < 0 ? 0 : x - radius;
    const int hi = x + radius > width - 1 ? width : x + radius + 1;
    const uint32_t el = radius > x ? (uint32_t)(radius - x) : 0u;
    const uint32_t er = x + radius > width - 1 ? (uint32_t)(x + radius - (width - 1)) : 0u;
    auto row_sum = [&](int y) {
        const uint32_t *p = fp + (size_t)y * (width + 1);
        uint32_t v = __ldg(p + hi) - __ldg(p + lo);
        if (el) v += el * fsrc[(size_t)y * width];
        if (er) v += er * fsrc[(size_t)y * width + width - 1];
        return v;
    };
    const int y0 = s * strip, y1 = y0 + strip < height ? y0 + strip : height;
    // the column window of row y0, rows replicated past the top and bottom
    uint32_t sum = 0;
    const int a = y0 - radius < 0 ? 0 : y0 - radius, b = y0 + radius > height - 1 ? height - 1 : y0 + radius;
    for (int y = a; y <= b; ++y) sum += row_sum(y);
    if (radius > y0) sum += (uint32_t)(radius - y0) * row_sum(0);
    if (y0 + radius > height - 1) sum += (uint32_t)(y0 + radius - (height - 1)) * row_sum(height - 1);
    for (int y = y0; y < y1; ++y) {
        // cv2.boxFilter's 8-bit sum: int32 scaled in float32 up to k^2 = 2^23, double above (dscale != 0)
        const int mean = dscale != 0 ? __double2int_rn(__dmul_rn((double)sum, dscale))
                                     : __float2int_rn(__fmul_rn(__uint2float_rn(sum), scale));
        const size_t i = (size_t)y * width + x;
        fdst[i] = adapt_out(fsrc[i], mean > 255 ? 255 : mean, neg_delta, inv, maxval);
        if (y + 1 < y1) {
            const int add = y + 1 + radius > height - 1 ? height - 1 : y + 1 + radius;
            const int sub = y - radius < 0 ? 0 : y - radius;
            sum += row_sum(add) - row_sum(sub);
        }
    }
}

__global__ void __launch_bounds__(kRowThreads) adapt_gauss_rows_kernel(const uint8_t *__restrict__ src,
                                                                       const float *__restrict__ taps, int ksize,
                                                                       int width, int segs, float *__restrict__ plane) {
    extern __shared__ float s_mem[];
    float *s_taps = s_mem, *s_px = s_mem + ksize;
    const size_t row = blockIdx.x / segs;
    const int x0 = (int)(blockIdx.x % segs) * kRowThreads;
    const int radius = ksize / 2;
    const uint8_t *rsrc = src + row * width;
    for (int j = threadIdx.x; j < ksize; j += kRowThreads) s_taps[j] = taps[j];
    for (int j = threadIdx.x; j < kRowThreads + ksize - 1; j += kRowThreads) {
        int xx = x0 - radius + j;
        xx = xx < 0 ? 0 : xx > width - 1 ? width - 1 : xx;
        s_px[j] = (float)rsrc[xx];
    }
    __syncthreads();
    const int x = x0 + threadIdx.x;
    if (x >= width) return;
    float acc = 0.f;
    for (int j = 0; j < ksize; ++j) acc = __fadd_rn(acc, __fmul_rn(s_taps[j], s_px[threadIdx.x + j]));
    plane[row * width + x] = acc;
}

__global__ void __launch_bounds__(kColThreads) adapt_gauss_cols_kernel(const uint8_t *__restrict__ src,
                                                                       const float *__restrict__ plane,
                                                                       const float *__restrict__ taps, int ksize,
                                                                       int height, int width, int col_blocks,
                                                                       uint8_t *__restrict__ dst, int neg_delta, int inv,
                                                                       int maxval) {
    extern __shared__ float s_taps[];
    for (int j = threadIdx.x; j < ksize; j += kColThreads) s_taps[j] = taps[j];
    __syncthreads();
    const size_t row = blockIdx.x / col_blocks;  // frame * height + y
    const int x = (int)(blockIdx.x % col_blocks) * kColThreads + threadIdx.x;
    if (x >= width) return;
    const int y = (int)(row % height);
    const float *fp = plane + (row - y) * width + x;
    const int radius = ksize / 2;
    float acc = 0.f;
    for (int j = 0; j < ksize; ++j) {
        int yy = y - radius + j;
        yy = yy < 0 ? 0 : yy > height - 1 ? height - 1 : yy;
        acc = __fadd_rn(acc, __fmul_rn(s_taps[j], __ldg(fp + (size_t)yy * width)));
    }
    int mean = __float2int_rn(acc);
    mean = mean < 0 ? 0 : mean > 255 ? 255 : mean;
    const size_t i = row * width + x;
    dst[i] = adapt_out(src[i], mean, neg_delta, inv, maxval);
}

}  // namespace bv

using namespace bv;

extern "C" int bv_threshold_auto(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                                 double maxval, int type, int method, double *thresh_dev) {
    BV_REQUIRE(ctx && src_dev && dst_dev && thresh_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(batch <= 65535, "batch must not exceed 65535");
    const size_t frame_px = (size_t)height * width;
    BV_REQUIRE(frame_px < (1ull << 31), "frame too large for 32-bit counts");
    BV_REQUIRE(method == BV_THRESH_OTSU || method == BV_THRESH_TRIANGLE, "method must be OTSU or TRIANGLE");
    BV_REQUIRE(type >= BV_THRESH_BINARY && type <= BV_THRESH_TOZERO_INV, "unknown threshold type");
    BV_REQUIRE(isfinite(maxval), "maxval must be finite");
    const size_t bytes = (size_t)batch * frame_px, tbytes = (size_t)batch * sizeof(double);
    BV_REQUIRE(src_dev == dst_dev || disjoint(src_dev, bytes, dst_dev, bytes), "src and dst overlap without being equal");
    BV_REQUIRE(disjoint(src_dev, bytes, thresh_dev, tbytes) && disjoint(dst_dev, bytes, thresh_dev, tbytes),
               "thresh overlaps src or dst");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_scratch(ctx, SCR_THRESH_SMALL, (size_t)batch * 256 * sizeof(int)));
    int *hist = (int *)ctx->scratch[SCR_THRESH_SMALL];
    BV_CUDA(cudaMemsetAsync(hist, 0, (size_t)batch * 256 * sizeof(int), ctx->stream));
    const size_t n_vec = (frame_px + 15) / 16;
    const int gh = grid_for(ctx, n_vec * batch, kHistThreads, 8);
    BV_LAUNCH(ctx, thresh_hist_kernel, dim3((gh + batch - 1) / batch, batch), kHistThreads, 0, src_dev,
              (uint32_t)frame_px, hist);
    BV_LAUNCH(ctx, thresh_search_kernel, (batch + kSearchThreads - 1) / kSearchThreads, kSearchThreads, 0, hist, batch,
              (uint32_t)frame_px, method, thresh_dev);
    // cv2.threshold's 8-bit maxval: cvRound, saturated (TRUNC takes the threshold instead, in the kernel)
    const int imax = saturate_u8(cv_round(maxval));
    const bool vec = host_aligned16(src_dev) && host_aligned16(dst_dev) && frame_px % 16 == 0;
    const int ga = grid_for(ctx, (vec ? n_vec : frame_px) * batch, kApplyThreads, 8);
    const dim3 grid((ga + batch - 1) / batch, batch);
    if (vec)
        BV_LAUNCH(ctx, thresh_apply_kernel<true>, grid, kApplyThreads, 0, src_dev, dst_dev, (uint32_t)frame_px,
                  thresh_dev, imax, type);
    else
        BV_LAUNCH(ctx, thresh_apply_kernel<false>, grid, kApplyThreads, 0, src_dev, dst_dev, (uint32_t)frame_px,
                  thresh_dev, imax, type);
    return BV_OK;
}

// cv2.getGaussianKernel(k, 0, CV_32F) as OpenCV 4.x builds it (getGaussianKernelBitExact, double arithmetic): its
// dyadic table for k <= 9; above, sigma = fma(k, 0.15, 0.35), the half-kernel exp(x^2 * (-0.125 / sigma^2)) at the
// doubled offsets x = 1 - k, 3 - k, .., their sum doubled plus the centre's 1, each tap times 1 / sum
static std::vector<float> gaussian_taps(int k) {
    static const float small[5][9] = {
        {1.f},
        {0.25f, 0.5f, 0.25f},
        {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f},
        {0.03125f, 0.109375f, 0.21875f, 0.28125f, 0.21875f, 0.109375f, 0.03125f},
        {4 / 256.f, 13 / 256.f, 30 / 256.f, 51 / 256.f, 60 / 256.f, 51 / 256.f, 30 / 256.f, 13 / 256.f, 4 / 256.f}};
    std::vector<float> t(k);
    if (k <= 9) {
        for (int i = 0; i < k; ++i) t[i] = small[k >> 1][i];
        return t;
    }
    const double sigma = fma((double)k, 0.15, 0.35);
    const double scale2 = -0.125 / (sigma * sigma);
    const int half = (k - 1) / 2;
    std::vector<double> v(half);
    double sum = 0;
    for (int i = 0; i < half; ++i) {
        const int x = 1 - k + 2 * i;
        v[i] = exp((double)(x * x) * scale2);
        sum += v[i];
    }
    sum = sum * 2 + 1;
    const double mul = 1. / sum;
    for (int i = 0; i < half; ++i) t[i] = t[k - 1 - i] = (float)(v[i] * mul);
    t[half] = (float)mul;
    return t;
}

extern "C" int bv_adaptive_threshold(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height,
                                     int width, double max_value, int method, int type, int block_size, double c) {
    BV_REQUIRE(ctx && src_dev && dst_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(block_size % 2 == 1 && block_size > 1, "block_size must be odd and above 1");
    BV_REQUIRE(block_size <= BV_ADAPTIVE_MAX_BLOCK, "block_size above BV_ADAPTIVE_MAX_BLOCK");
    BV_REQUIRE(method == BV_ADAPTIVE_THRESH_MEAN_C || method == BV_ADAPTIVE_THRESH_GAUSSIAN_C, "unknown adaptive method");
    BV_REQUIRE(type == BV_THRESH_BINARY || type == BV_THRESH_BINARY_INV, "type must be BINARY or BINARY_INV");
    BV_REQUIRE(isfinite(max_value) && isfinite(c), "max_value and c must be finite");
    BV_REQUIRE(fabs(c) < 2147483647.0, "|c| has no int32 ceiling / floor");
    const size_t frame_px = (size_t)height * width, bytes = (size_t)batch * frame_px;
    BV_REQUIRE(frame_px < (1ull << 31), "frame too large for 32-bit indices");
    BV_REQUIRE(disjoint(src_dev, bytes, dst_dev, bytes), "src and dst overlap");
    BV_CUDA(cudaSetDevice(ctx->device));

    // cv2's table: idelta = ceil(c) (BINARY) or floor(c) (BINARY_INV); src - mean lies in [-255, 255], so -idelta
    // clamped to [-256, 256] compares the same
    const double idelta = type == BV_THRESH_BINARY ? ceil(c) : floor(c);
    const int neg_delta = -idelta > 256 ? 256 : -idelta < -256 ? -256 : (int)-idelta;
    const int imax = max_value < 0 ? 0 : saturate_u8(cv_round(max_value));
    const int inv = type == BV_THRESH_BINARY_INV;
    const int radius = block_size / 2;
    const size_t rows = (size_t)batch * height;
    const int col_blocks = (width + kColThreads - 1) / kColThreads;

    if (method == BV_ADAPTIVE_THRESH_MEAN_C) {
        BV_TRY(ensure_scratch(ctx, SCR_THRESH_PLANE, rows * (width + 1) * sizeof(uint32_t)));
        uint32_t *prefix = (uint32_t *)ctx->scratch[SCR_THRESH_PLANE];
        // strips as tall as the window (capped by the frame), so the window's first sum costs no more than the strip's
        // sliding steps; halved (down to kMinStrip rows) while the launch would leave the SMs short of blocks: a
        // strip's rows are sequential, so a few tall strips leave most of the device idle
        int strip = block_size < height ? block_size : height;
        strip = strip < kMinStrip ? kMinStrip : strip;
        while (strip > kMinStrip && (size_t)batch * col_blocks * ((height + strip - 1) / strip) < 4 * (size_t)ctx->sm_count)
            strip = strip / 2 < kMinStrip ? kMinStrip : strip / 2;
        const int strips = (height + strip - 1) / strip;
        const size_t blocks = (size_t)batch * strips * col_blocks;
        BV_REQUIRE(rows <= 0x7FFFFFFFu && blocks <= 0x7FFFFFFFu, "too many rows for one launch");
        const double area = (double)block_size * block_size;
        const float scale = (float)(1. / area);
        const double dscale = area > (double)(1 << 23) ? 1. / area : 0.;
        BV_LAUNCH(ctx, adapt_prefix_kernel, (unsigned)rows, kRowThreads, 0, src_dev, width, prefix);
        BV_LAUNCH(ctx, adapt_mean_cols_kernel, (unsigned)blocks, kColThreads, 0, src_dev, prefix, dst_dev, height, width,
                  radius, strip, strips, col_blocks, scale, dscale, neg_delta, inv, imax);
        return BV_OK;
    }

    const std::vector<float> taps = gaussian_taps(block_size);
    const int segs = (width + kRowThreads - 1) / kRowThreads;
    BV_REQUIRE(rows * segs <= 0x7FFFFFFFu && rows * col_blocks <= 0x7FFFFFFFu, "too many rows for one launch");
    BV_TRY(ensure_scratch(ctx, SCR_THRESH_SMALL, (size_t)block_size * sizeof(float)));
    BV_TRY(ensure_scratch(ctx, SCR_THRESH_PLANE, bytes * sizeof(float)));
    float *d_taps = (float *)ctx->scratch[SCR_THRESH_SMALL];
    float *plane = (float *)ctx->scratch[SCR_THRESH_PLANE];
    BV_CUDA(cudaMemcpyAsync(d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    const size_t row_smem = (size_t)(2 * block_size - 1 + kRowThreads) * sizeof(float);
    BV_LAUNCH(ctx, adapt_gauss_rows_kernel, (unsigned)(rows * segs), kRowThreads, row_smem, src_dev, d_taps, block_size,
              width, segs, plane);
    BV_LAUNCH(ctx, adapt_gauss_cols_kernel, (unsigned)(rows * col_blocks), kColThreads, (size_t)block_size * sizeof(float),
              src_dev, plane, d_taps, block_size, height, width, col_blocks, dst_dev, neg_delta, inv, imax);
    return BV_OK;
}
