// filter.cu -- the tuner-gated geometric / smoothing steps of the reference's preprocessor:
//
//   cv2.GaussianBlur(mat, (2k+1, 2k+1), 0)                         modules/preprocessor.py:110-114
//   cv2.warpAffine(mat, getRotationMatrix2D(...), BORDER_REPLICATE) modules/preprocessor.py:130-135
//   cv2.warpAffine(mat, [[1,0,tx],[0,1,ty]])  (BORDER_CONSTANT 0)   modules/preprocessor.py:144-149
//
// Both reproduce OpenCV 4.x's 8-bit fixed-point arithmetic bit for bit (pinned against cv2 4.13.0,
// oracle/spec_np.py::gaussian_blur_8u / warp_affine_8u):
//
// GaussianBlur, uint8: the float64 kernel (tables for sizes <= 9, else exp(-x^2 / 2 sigma^2) with
//   sigma = 0.3((n-1)/2 - 1) + 0.8, normalised) is converted to 8.8 fixed point by error diffusion
//   from the outside in, the centre tap taking what is left of 256; the horizontal pass accumulates
//   tap * pixel in 16 bits (8.8), the vertical pass tap * that in 32 bits (16.16), the result is
//   (v + 2^15) >> 16; borders are BORDER_REFLECT_101.
// warpAffine, uint8, INTER_LINEAR: the matrix is inverted in double; source coordinates are
//   fixed point with 10 fractional bits, X = round(M0 x 1024) + round((M1 y + M2) 1024) + 16,
//   reduced to 5 fractional bits; the four bilinear weights come from a 32x32 table of int16
//   (float32 products scaled by 2^15, rounded, largest/smallest entry adjusted so that they sum
//   to 2^15); result (sum + 2^14) >> 15.  Taps outside the image replicate the edge
//   (BORDER_REPLICATE) or take the border value (BORDER_CONSTANT).
#include <limits.h>
#include <math.h>

#include "common.cuh"

namespace bv {

// ----------------------------------------------------------------------------------------------
// Gaussian blur: a block stages a tile plus halo (reflected at the image border) in shared memory,
// runs the horizontal pass into a 16-bit tile and the vertical pass out of it.
// ----------------------------------------------------------------------------------------------
constexpr int kBlurMaxTaps = 201;   // the reference's tuner reaches 2 * 100 + 1 (modules/preprocessor.py:25,110-114)
constexpr int kBlurTileW = 64, kBlurTileH = 32;
struct BlurTaps {
    int nx, ny;
    uint16_t kx[kBlurMaxTaps], ky[kBlurMaxTaps];
};

__device__ __forceinline__ int reflect101(int p, int len) {
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

// Threads are laid out (byte column, row): no index division inside the passes; NT > 0 unrolls the tap loops
// for the common small kernels (3, 5, 7 taps), NT = 0 is the generic form.
template <int CN, int NT>
__global__ void __launch_bounds__(256) gaussian_blur_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int height,
                                                            int width, BlurTaps taps) {
    extern __shared__ __align__(16) uint8_t blur_smem[];
    const int nx = NT > 0 ? NT : taps.nx, ny = NT > 0 ? NT : taps.ny;
    const int rx = nx / 2, ry = ny / 2;
    const int raw_w = (kBlurTileW + 2 * rx) * CN;         // bytes per staged row
    const int raw_h = kBlurTileH + 2 * ry;
    constexpr int hz_w = kBlurTileW * CN;                 // 16-bit values per row of the horizontal result
    uint8_t *raw = blur_smem;
    uint16_t *hz = reinterpret_cast<uint16_t *>(blur_smem + ((raw_w * raw_h + 15) & ~15));
    const int x0 = blockIdx.x * kBlurTileW, y0 = blockIdx.y * kBlurTileH;
    const size_t frame_off = (size_t)blockIdx.z * height * width * CN;
    const uint8_t *f = src + frame_off;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 byte-columns x 4 rows per step
    // stage rows y0-ry .. y0+TH+ry-1, columns x0-rx .. x0+TW+rx-1, reflected (BORDER_REFLECT_101)
    for (int b = tx; b < raw_w; b += 64) {
        const int px = b / CN, c = b - px * CN;
        const int sx = reflect101(x0 - rx + px, width);
        for (int r = ty; r < raw_h; r += 4) {
            const int sy = reflect101(y0 - ry + r, height);
            raw[r * raw_w + b] = f[((size_t)sy * width + sx) * CN + c];
        }
    }
    __syncthreads();
    // horizontal pass: hz[r][b] = sum_k kx[k] * raw[r][b + k*CN]      (8.8 in 16 bits)
    for (int b = tx; b < hz_w; b += 64)
        for (int r = ty; r < raw_h; r += 4) {
            const uint8_t *p = raw + r * raw_w + b;
            uint32_t acc = 0;
            if (NT > 0) {
#pragma unroll
                for (int k = 0; k < (NT > 0 ? NT : 1); ++k) acc += (uint32_t)taps.kx[k] * p[k * CN];
            } else {
                for (int k = 0; k < nx; ++k) acc += (uint32_t)taps.kx[k] * p[k * CN];
            }
            hz[r * hz_w + b] = (uint16_t)(acc > 0xFFFFu ? 0xFFFFu : acc);  // ufixedpoint16 saturates (never reached: taps sum to 256)
        }
    __syncthreads();
    // vertical pass
    for (int b = tx; b < hz_w; b += 64) {
        const int x = x0 + b / CN;
        if (x >= width) continue;
        for (int r = ty; r < kBlurTileH; r += 4) {
            const int y = y0 + r;
            if (y >= height) break;
            const uint16_t *p = hz + r * hz_w + b;
            uint32_t acc = 0;
            if (NT > 0) {
#pragma unroll
                for (int k = 0; k < (NT > 0 ? NT : 1); ++k) acc += (uint32_t)taps.ky[k] * p[k * hz_w];
            } else {
                for (int k = 0; k < ny; ++k) acc += (uint32_t)taps.ky[k] * p[k * hz_w];
            }
            const uint32_t v = (acc + (1u << 15)) >> 16;
            dst[frame_off + ((size_t)y * width + x0) * CN + b] = (uint8_t)(v > 255u ? 255u : v);
        }
    }
}

// ----------------------------------------------------------------------------------------------
// Large kernels (the tile + halo no longer fits shared memory): the same two passes with the 16-bit horizontal
// result in a global scratch image.  One thread per output byte; the taps sit in shared memory.
// ----------------------------------------------------------------------------------------------
template <int CN>
__global__ void __launch_bounds__(256) blur_rows16_kernel(const uint8_t *__restrict__ src, uint16_t *__restrict__ hz, int height,
                                                          int width, BlurTaps taps) {
    __shared__ uint16_t k[kBlurMaxTaps];
    for (int i = threadIdx.x; i < taps.nx; i += blockDim.x) k[i] = taps.kx[i];
    __syncthreads();
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= width) return;
    const size_t row = ((size_t)blockIdx.z * height + y) * width;
    const int rx = taps.nx / 2;
    uint32_t acc[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) acc[c] = 0;
    for (int t = 0; t < taps.nx; ++t) {
        const uint8_t *p = src + (row + reflect101(x - rx + t, width)) * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c) acc[c] += (uint32_t)k[t] * p[c];
    }
#pragma unroll
    for (int c = 0; c < CN; ++c) hz[(row + x) * CN + c] = (uint16_t)(acc[c] > 0xFFFFu ? 0xFFFFu : acc[c]);
}

template <int CN>
__global__ void __launch_bounds__(256) blur_cols16_kernel(const uint16_t *__restrict__ hz, uint8_t *__restrict__ dst, int height,
                                                          int width, BlurTaps taps) {
    __shared__ uint16_t k[kBlurMaxTaps];
    for (int i = threadIdx.x; i < taps.ny; i += blockDim.x) k[i] = taps.ky[i];
    __syncthreads();
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= width) return;
    const size_t frame = (size_t)blockIdx.z * height * width;
    const int ry = taps.ny / 2;
    uint32_t acc[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) acc[c] = 0;
    for (int t = 0; t < taps.ny; ++t) {
        const uint16_t *p = hz + (frame + (size_t)reflect101(y - ry + t, height) * width + x) * CN;
#pragma unroll
        for (int c = 0; c < CN; ++c) acc[c] += (uint32_t)k[t] * p[c];
    }
#pragma unroll
    for (int c = 0; c < CN; ++c) {
        const uint32_t v = (acc[c] + (1u << 15)) >> 16;
        dst[(frame + (size_t)y * width + x) * CN + c] = (uint8_t)(v > 255u ? 255u : v);
    }
}

// ----------------------------------------------------------------------------------------------
// The common kernels (3, 5, 7 taps; rows a multiple of 4 bytes): the image row is handled as a byte
// stream, a thread owns 4 consecutive output bytes.  Rows are staged with aligned 32-bit loads
// (byte-wise only where the reflected border is involved), the horizontal taps are cut out of the few
// staged words that hold them (all offsets are compile-time), the 16-bit horizontal results move as
// 8-byte vectors, and the result leaves as one 32-bit store.
// ----------------------------------------------------------------------------------------------
constexpr int kFastTileWords = 64;   // 256 bytes of a row per block
constexpr int kFastTileH = 32;

template <int CN, int NT>
__global__ void __launch_bounds__(256) gaussian_blur_fast_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int height,
                                                                 int width, BlurTaps taps) {
    constexpr int R = NT / 2;                 // taps each side
    constexpr int HB = R * CN;                // halo in bytes
    constexpr int HBW = (HB + 3) / 4;         // ... in whole words
    constexpr int PAD = 4 * HBW - HB;         // bytes between the staged row's start and the first tap of byte 0
    constexpr int RAW_W = kFastTileWords + 2 * HBW;
    constexpr int RAW_H = kFastTileH + 2 * R;
    constexpr int SPAN = 4 + (NT - 1) * CN;   // bytes the taps of 4 adjacent outputs cover
    constexpr int NW = (PAD + SPAN + 3) / 4;  // words that hold them
    __shared__ uint32_t raw[RAW_H][RAW_W];
    __shared__ __align__(8) uint16_t hz[RAW_H][kFastTileWords * 4];
    const int row_bytes = width * CN;
    const int x0b = blockIdx.x * kFastTileWords * 4, y0 = blockIdx.y * kFastTileH;
    const size_t frame_off = (size_t)blockIdx.z * height * row_bytes;
    const uint8_t *f = src + frame_off;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    // ---- stage
    for (int w = tx; w < RAW_W; w += 64) {
        const int gb = x0b - 4 * HBW + 4 * w;  // byte offset of this word in the image row
        const bool inside = gb >= 0 && gb + 4 <= row_bytes;
        int sxb[4];
        if (!inside) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int b = gb + j;
                const int px = b >= 0 ? b / CN : -((-b + CN - 1) / CN);  // floor
                const int c = b - px * CN;
                sxb[j] = reflect101(px, width) * CN + c;
            }
        }
        for (int r = ty; r < RAW_H; r += 4) {
            const uint8_t *row = f + (size_t)reflect101(y0 - R + r, height) * row_bytes;
            uint32_t v;
            if (inside)
                v = __ldg(reinterpret_cast<const uint32_t *>(row + gb));
            else
                v = (uint32_t)row[sxb[0]] | ((uint32_t)row[sxb[1]] << 8) | ((uint32_t)row[sxb[2]] << 16) | ((uint32_t)row[sxb[3]] << 24);
            raw[r][w] = v;
        }
    }
    __syncthreads();
    // ---- horizontal pass: 4 outputs per thread and row
    uint32_t kx[NT], ky[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) {
        kx[k] = taps.kx[k];
        ky[k] = taps.ky[k];
    }
    for (int r = ty; r < RAW_H; r += 4) {
        uint32_t wd[NW];
#pragma unroll
        for (int q = 0; q < NW; ++q) wd[q] = raw[r][tx + q];
        uint32_t acc[4] = {0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int k = 0; k < NT; ++k) {
                constexpr int dummy = 0;
                (void)dummy;
                const int bi = PAD + j + k * CN;  // compile-time after unrolling
                acc[j] += kx[k] * ((wd[bi >> 2] >> (8 * (bi & 3))) & 0xFFu);
            }
        // 8.8 values never exceed 255 * 256: no saturation needed (taps sum to 256)
        *reinterpret_cast<uint2 *>(&hz[r][4 * tx]) = make_uint2(acc[0] | (acc[1] << 16), acc[2] | (acc[3] << 16));
    }
    __syncthreads();
    // ---- vertical pass
    const int ob = x0b + 4 * tx;  // first output byte of this thread in the row
    if (ob >= row_bytes) return;
    for (int r = ty; r < kFastTileH; r += 4) {
        const int y = y0 + r;
        if (y >= height) break;
        uint32_t acc[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < NT; ++k) {
            const uint2 h = *reinterpret_cast<const uint2 *>(&hz[r + k][4 * tx]);
            acc[0] += ky[k] * (h.x & 0xFFFFu);
            acc[1] += ky[k] * (h.x >> 16);
            acc[2] += ky[k] * (h.y & 0xFFFFu);
            acc[3] += ky[k] * (h.y >> 16);
        }
        uint32_t o = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t v = (acc[j] + (1u << 15)) >> 16;
            o |= (v > 255u ? 255u : v) << (8 * j);
        }
        uint8_t *out = dst + frame_off + (size_t)y * row_bytes + ob;
        if (ob + 4 <= row_bytes) {
            *reinterpret_cast<uint32_t *>(out) = o;
        } else {
            for (int j = 0; ob + j < row_bytes; ++j) out[j] = (uint8_t)(o >> (8 * j));
        }
    }
}

// OpenCV's getGaussianKernelBitExact + getGaussianKernelFixedPoint_ED for 8.8 fixed point
static int gaussian_taps_fixed(int n, double sigma, uint16_t *out) {
    static const double small[5][9] = {{1.},
                                       {0.25, 0.5, 0.25},
                                       {0.0625, 0.25, 0.375, 0.25, 0.0625},
                                       {0.03125, 0.109375, 0.21875, 0.28125, 0.21875, 0.109375, 0.03125},
                                       {4. / 256, 13. / 256, 30. / 256, 51. / 256, 60. / 256, 51. / 256, 30. / 256, 13. / 256, 4. / 256}};
    double k[kBlurMaxTaps];
    if (sigma <= 0 && n <= 9) {
        for (int i = 0; i < n; ++i) k[i] = small[n / 2][i];
    } else {
        const double s = sigma > 0 ? sigma : ((n - 1) * 0.5 - 1) * 0.3 + 0.8;
        const double scale2 = -0.5 / (s * s);
        double sum = 0;
        for (int i = 0; i < n; ++i) {
            const double x = i - (n - 1) * 0.5;
            k[i] = exp(scale2 * x * x);
            sum += k[i];
        }
        for (int i = 0; i < n; ++i) k[i] /= sum;
    }
    const int h = n / 2;
    double err = 0;
    long acc = 0;
    for (int i = 0; i < h; ++i) {
        const double adj = k[i] * 256.0 + err;
        const long v = (long)nearbyint(adj);  // cvRound: round half to even
        err = adj - (double)v;
        if (v < 0 || v > 256) return BV_ERR_INVALID;
        out[i] = out[n - 1 - i] = (uint16_t)v;
        acc += v;
    }
    const long centre = 256 - 2 * acc;
    if (centre < 0) return BV_ERR_INVALID;
    out[h] = (uint16_t)centre;
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// warpAffine
// ----------------------------------------------------------------------------------------------
struct WarpParams {
    double m[6];  // inverted matrix (destination -> source)
    int border_constant;
    int border_value[4];
};

// cvRound / saturate_cast<int> of OpenCV on x86-64 (cvtsd2si, cvtss2si): round half to even; NaN, +-inf and every value
// whose rounded result lies outside int32 give INT_MIN ("integer indefinite"), on either side.
__device__ __forceinline__ int sat_round_int(double v) {
    const double r = rint(v);
    return r >= -2147483648.0 && r <= 2147483647.0 ? (int)r : INT_MIN;
}

__device__ __forceinline__ int sat_round_int(float v) {
    const float r = rintf(v);
    return r >= -2147483648.f && r < 2147483648.f ? (int)r : INT_MIN;
}

__device__ __forceinline__ short sat_short(int v) { return (short)(v < -32768 ? -32768 : (v > 32767 ? 32767 : v)); }

// The fixed-point coordinate terms depend on the column (adelta, bdelta) or on the row (X0, Y0) only: OpenCV
// tabulates them per call, and so does this kernel's small prologue launch (coords = [adelta | bdelta | X0 | Y0]).
__global__ void __launch_bounds__(256) warp_coords_kernel(int *__restrict__ coords, int dst_w, int dst_h, WarpParams wp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const double scale = 1024.;  // AB_SCALE = 1 << AB_BITS, AB_BITS = 10
    const int round_delta = 1024 / 32 / 2;
    if (i < dst_w) {
        coords[i] = sat_round_int(__dmul_rn(__dmul_rn(wp.m[0], (double)i), scale));
        coords[dst_w + i] = sat_round_int(__dmul_rn(__dmul_rn(wp.m[3], (double)i), scale));
    }
    if (i < dst_h) {
        coords[2 * dst_w + i] = sat_round_int(__dmul_rn(__dadd_rn(__dmul_rn(wp.m[1], (double)i), wp.m[2]), scale)) + round_delta;
        coords[2 * dst_w + dst_h + i] = sat_round_int(__dmul_rn(__dadd_rn(__dmul_rn(wp.m[4], (double)i), wp.m[5]), scale)) + round_delta;
    }
}

// remapBilinear of OpenCV on uint8: taps (sx, sy) .. (sx + 1, sy + 1), weights from the 32 x 32 x 4 int16 table entry `frac`
// (= fy * 32 + fx), (sum + 2^14) >> 15; outside taps take the border value (constant) or the nearest pixel (replicate).
template <int CN>
__device__ __forceinline__ void bilinear_sample(const uint8_t *__restrict__ f, size_t frame_bytes, bool words_ok, int height, int width,
                                                int sx, int sy, int frac, const short *__restrict__ tab, const WarpParams &wp,
                                                uint8_t *__restrict__ o) {
    const short *w = tab + 4 * frac;
    const int w00 = w[0], w01 = w[1], w10 = w[2], w11 = w[3];
    // interior pixels (all four taps inside the image): the two taps of a row are 2*CN adjacent bytes; fetch them with
    // aligned 32-bit loads and a funnel shift instead of one load per byte
    if (words_ok && sx >= 0 && sy >= 0 && sx + 1 < width && sy + 1 < height) {
        const size_t off0 = ((size_t)sy * width + sx) * CN, off1 = off0 + (size_t)width * CN;
        if (off1 + 12 <= frame_bytes) {
            uint32_t lo[2], hi[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const size_t off = j ? off1 : off0;
                const uint32_t *a = reinterpret_cast<const uint32_t *>(f + (off & ~(size_t)3));
                const uint32_t w0 = __ldg(a), w1 = __ldg(a + 1), w2 = CN == 3 ? __ldg(a + 2) : 0u;
                const uint32_t sh = 8u * (uint32_t)(off & 3);
                lo[j] = __funnelshift_r(w0, w1, sh);   // bytes off .. off+3
                hi[j] = __funnelshift_r(w1, w2, sh);   // bytes off+4 .. off+7
            }
#pragma unroll
            for (int c = 0; c < CN; ++c) {
                int v[2][2];
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    v[j][0] = (int)((lo[j] >> (8 * c)) & 0xFFu);
                    const int b1 = CN + c;  // byte index of the right tap's channel c
                    v[j][1] = (int)(((b1 < 4 ? lo[j] >> (8 * b1) : hi[j] >> (8 * (b1 - 4)))) & 0xFFu);
                }
                const int s_ = v[0][0] * w00 + v[0][1] * w01 + v[1][0] * w10 + v[1][1] * w11;
                o[c] = (uint8_t)sat_u8((s_ + (1 << 14)) >> 15);
            }
            return;
        }
    }
    const int xs[2] = {sx, sx + 1}, ys[2] = {sy, sy + 1};
    const uint8_t *p[2][2];
    bool inside[2][2];
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            inside[j][i] = xs[i] >= 0 && xs[i] < width && ys[j] >= 0 && ys[j] < height;
            const int cx = min(max(xs[i], 0), width - 1), cy = min(max(ys[j], 0), height - 1);
            p[j][i] = f + ((size_t)cy * width + cx) * CN;
        }
#pragma unroll
    for (int c = 0; c < CN; ++c) {
        int v[2][2];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int i = 0; i < 2; ++i) v[j][i] = (wp.border_constant && !inside[j][i]) ? wp.border_value[c] : (int)p[j][i][c];
        const int s_ = v[0][0] * w00 + v[0][1] * w01 + v[1][0] * w10 + v[1][1] * w11;
        o[c] = (uint8_t)sat_u8((s_ + (1 << 14)) >> 15);
    }
}

template <int CN>
__global__ void __launch_bounds__(256) warp_affine_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int height,
                                                          int width, int dst_h, int dst_w, WarpParams wp,
                                                          const short *__restrict__ tab, const int *__restrict__ coords) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dst_w) return;
    const size_t frame_bytes = (size_t)height * width * CN;
    const uint8_t *f = src + (size_t)blockIdx.z * frame_bytes;
    const bool words_ok = (reinterpret_cast<uintptr_t>(f) & 3) == 0;  // block-uniform
    uint8_t *o = dst + ((size_t)blockIdx.z * dst_h * dst_w + (size_t)y * dst_w + x) * CN;
    constexpr int AB_BITS = 10, INTER_BITS = 5, TAB = 32;
    const int adelta = __ldg(coords + x), bdelta = __ldg(coords + dst_w + x);
    const int X0 = __ldg(coords + 2 * dst_w + y), Y0 = __ldg(coords + 2 * dst_w + dst_h + y);
    const int X = (X0 + adelta) >> (AB_BITS - INTER_BITS), Y = (Y0 + bdelta) >> (AB_BITS - INTER_BITS);
    const int sx = sat_short(X >> INTER_BITS), sy = sat_short(Y >> INTER_BITS);  // saturate_cast<short>
    bilinear_sample<CN>(f, frame_bytes, words_ok, height, width, sx, sy, (Y & (TAB - 1)) * TAB + (X & (TAB - 1)), tab, wp, o);
}

// cv2.remap(INTER_LINEAR) on uint8.  FIXED: map1 = int16 (x, y) pairs, map2 = uint16 fy * 32 + fx (CV_16SC2 + CV_16UC1).
// Otherwise map1 / map2 are float32 x / y planes, converted the way RemapInvoker converts them block by block:
// cvRound(x * 32) in float32 (NaN, +-inf and |x * 32| >= 2^31 give INT_MIN, so such a tap lands on the left / top border),
// integer part saturated to short, the two 5-bit fractions.
template <int CN, bool FIXED>
__global__ void __launch_bounds__(256) remap_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int height, int width,
                                                    int dst_h, int dst_w, const void *__restrict__ map1, const void *__restrict__ map2,
                                                    WarpParams wp, const short *__restrict__ tab) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dst_w) return;
    const size_t frame_bytes = (size_t)height * width * CN;
    const uint8_t *f = src + (size_t)blockIdx.z * frame_bytes;
    const bool words_ok = (reinterpret_cast<uintptr_t>(f) & 3) == 0;  // block-uniform
    uint8_t *o = dst + ((size_t)blockIdx.z * dst_h * dst_w + (size_t)y * dst_w + x) * CN;
    const size_t i = (size_t)y * dst_w + x;
    int sx, sy, frac;
    if (FIXED) {
        const short2 xy = __ldg(static_cast<const short2 *>(map1) + i);
        sx = xy.x;
        sy = xy.y;
        frac = __ldg(static_cast<const unsigned short *>(map2) + i) & 1023;
    } else {
        const int X = sat_round_int(__fmul_rn(__ldg(static_cast<const float *>(map1) + i), 32.f));
        const int Y = sat_round_int(__fmul_rn(__ldg(static_cast<const float *>(map2) + i), 32.f));
        sx = sat_short(X >> 5);  // saturate_cast<short>
        sy = sat_short(Y >> 5);
        frac = (Y & 31) * 32 + (X & 31);
    }
    bilinear_sample<CN>(f, frame_bytes, words_ok, height, width, sx, sy, frac, tab, wp, o);
}

// cv2.initUndistortRectifyMap: for every destination pixel the normalised ray through the new camera (and rotation),
// the radial / tangential distortion polynomial, the source pixel through the original camera.  All in float64 with
// every product and sum rounded separately, in the order of oracle/spec_np.py::init_undistort_rectify_map (which matches
// cv2 bit for bit on the reference's camera files).  Writes float32 maps (CV_32FC1) and / or the fixed-point pair that
// cv2.undistort builds straight from the doubles (CV_16SC2 + CV_16UC1).
struct UndistortParams {
    double ir[9];       // inverse of (new camera matrix x rotation)
    double k[8];        // k1 k2 p1 p2 k3 k4 k5 k6
    double fx, fy, cx, cy;
};

__global__ void __launch_bounds__(256) undistort_maps_kernel(UndistortParams p, int width, int height, float *__restrict__ mapx,
                                                             float *__restrict__ mapy, short2 *__restrict__ xy,
                                                             unsigned short *__restrict__ frac) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= width) return;
#define MUL(a, b) __dmul_rn((a), (b))
#define ADD(a, b) __dadd_rn((a), (b))
    const double u = (double)j, v = (double)i;
    const double X = ADD(MUL(p.ir[0], u), ADD(MUL(p.ir[1], v), p.ir[2]));
    const double Y = ADD(MUL(p.ir[3], u), ADD(MUL(p.ir[4], v), p.ir[5]));
    const double W = ADD(MUL(p.ir[6], u), ADD(MUL(p.ir[7], v), p.ir[8]));
    const double x = __ddiv_rn(X, W), y = __ddiv_rn(Y, W);
    const double x2 = MUL(x, x), y2 = MUL(y, y);
    const double r2 = ADD(x2, y2), _2xy = MUL(MUL(2.0, x), y);
    const double k1 = p.k[0], k2 = p.k[1], p1 = p.k[2], p2 = p.k[3], k3 = p.k[4], k4 = p.k[5], k5 = p.k[6], k6 = p.k[7];
    const double num = ADD(1.0, MUL(ADD(MUL(ADD(MUL(k3, r2), k2), r2), k1), r2));
    const double den = ADD(1.0, MUL(ADD(MUL(ADD(MUL(k6, r2), k5), r2), k4), r2));
    const double kr = __ddiv_rn(num, den);
    const double xd = ADD(ADD(MUL(x, kr), MUL(p1, _2xy)), MUL(p2, ADD(r2, MUL(2.0, x2))));
    const double yd = ADD(ADD(MUL(y, kr), MUL(p1, ADD(r2, MUL(2.0, y2)))), MUL(p2, _2xy));
    const double us = ADD(MUL(p.fx, xd), p.cx), vs = ADD(MUL(p.fy, yd), p.cy);
#undef MUL
#undef ADD
    const size_t o = (size_t)i * width + j;
    if (mapx) {
        mapx[o] = (float)us;
        mapy[o] = (float)vs;
    }
    if (xy) {
        const int iu = sat_round_int(us * 32.0), iv = sat_round_int(vs * 32.0);  // saturate_cast<int>(u * INTER_TAB_SIZE)
        xy[o] = make_short2(sat_short(iu >> 5), sat_short(iv >> 5));  // saturate_cast<short>
        frac[o] = (unsigned short)((iv & 31) * 32 + (iu & 31));
    }
}

// OpenCV's BilinearTab_i (initInterTab2D(INTER_LINEAR, fixpt = true)): 32 x 32 x 4 int16
static void build_bilinear_tab(short *tab) {
    float t1[32][2];
    for (int i = 0; i < 32; ++i) {
        const float x = (float)i * (1.f / 32.f);
        t1[i][0] = 1.f - x;
        t1[i][1] = x;
    }
    for (int i = 0; i < 32; ++i)
        for (int j = 0; j < 32; ++j) {
            short *it = tab + (i * 32 + j) * 4;
            int isum = 0;
            for (int k1 = 0; k1 < 2; ++k1)
                for (int k2 = 0; k2 < 2; ++k2) {
                    const float v = t1[i][k1] * t1[j][k2];
                    long r = lrintf(v * 32768.f);
                    r = r < -32768 ? -32768 : (r > 32767 ? 32767 : r);
                    it[k1 * 2 + k2] = (short)r;
                    isum += (int)r;
                }
            if (isum != 32768) {
                // Only the entry (fy, fx) = (0, 0) gets here: 1.0 * 2^15 saturates to 32767.  OpenCV's
                // fix-up searches the "central" 2x2 block of a ksize x ksize kernel, which for ksize = 2
                // starts at the LAST tap (and runs past the entry into zeros), so the missing 1 lands on
                // the bottom-right tap: {32767, 0, 0, 1}.  The pixel value is the same either way:
                // (32767 p00 + p11 + 2^14) >> 15 == p00.
                it[3] = (short)(it[3] - (isum - 32768));
            }
        }
}

// ---- white_balance_bgr_blur (utils/color.py:381-391): a / b planes shifted by their local box mean -----------------
// cv2.blur of a float32 plane (BORDER_REPLICATE) sums in double (exact here: the values are integers 0..255) and
// returns float(sum * (1.0 / (k*k))).  Pass 1 keeps the horizontal window sums of a and b, pass 2 adds them down the
// column, forms `a - (mean - 128)` in float32 as numpy does and casts like numpy's astype(uint8): truncate, wrap mod 256.
__global__ void __launch_bounds__(256) box_rows_ab_kernel(const uint8_t *__restrict__ lab, uint2 *__restrict__ sums,
                                                         int height, int width, int radius) {
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= width) return;
    const size_t row = ((size_t)blockIdx.z * height + blockIdx.y) * width;
    const uint8_t *p = lab + row * 3;
    unsigned sa = 0, sb = 0;
    for (int d = -radius; d <= radius; ++d) {
        const int xx = min(max(x + d, 0), width - 1);
        sa += p[xx * 3 + 1];
        sb += p[xx * 3 + 2];
    }
    sums[row + x] = make_uint2(sa, sb);
}

__device__ __forceinline__ uint8_t numpy_f32_to_u8(float v) { return (uint8_t)((int)v & 255); }

__global__ void __launch_bounds__(256) box_cols_shift_kernel(const uint8_t *__restrict__ lab, const uint2 *__restrict__ sums,
                                                            uint8_t *__restrict__ out, int height, int width, int radius,
                                                            double scale) {
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= width) return;
    const int y = blockIdx.y;
    const size_t frame = (size_t)blockIdx.z * height * width;
    unsigned sa = 0, sb = 0;
    for (int d = -radius; d <= radius; ++d) {
        const int yy = min(max(y + d, 0), height - 1);
        const uint2 s = sums[frame + (size_t)yy * width + x];
        sa += s.x;
        sb += s.y;
    }
    const size_t i = (frame + (size_t)y * width + x) * 3;
    const float ma = (float)((double)sa * scale), mb = (float)((double)sb * scale);
    out[i] = lab[i];
    out[i + 1] = numpy_f32_to_u8(__fsub_rn((float)lab[i + 1], __fsub_rn(ma, 128.f)));
    out[i + 2] = numpy_f32_to_u8(__fsub_rn((float)lab[i + 2], __fsub_rn(mb, 128.f)));
}

static int ensure_bilinear_tab(bv_ctx *ctx) {
    if (!ctx->d_bilinear_tab) {
        short tab[32 * 32 * 4];
        build_bilinear_tab(tab);
        BV_CUDA(cudaMalloc(&ctx->d_bilinear_tab, sizeof(tab)));
        BV_CUDA(cudaMemcpyAsync(ctx->d_bilinear_tab, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
        BV_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return BV_OK;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_gaussian_blur(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                                int channels, int ksize_x, int ksize_y, double sigma_x, double sigma_y) {
    BV_REQUIRE(ctx && src_dev && dst_dev, "null argument");
    BV_REQUIRE(src_dev != dst_dev, "in-place blur is not supported");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_REQUIRE(ksize_x >= 1 && ksize_y >= 1 && (ksize_x & 1) && (ksize_y & 1) && ksize_x <= kBlurMaxTaps && ksize_y <= kBlurMaxTaps,
               "kernel sizes must be odd and in 1..201");
    BV_REQUIRE(batch <= 65535, "batch too large");
    BV_CUDA(cudaSetDevice(ctx->device));
    if (sigma_y <= 0) sigma_y = sigma_x;  // cv2: sigmaY = sigmaX when not given
    BlurTaps taps;
    memset(&taps, 0, sizeof(taps));
    taps.nx = ksize_x;
    taps.ny = ksize_y;
    if (gaussian_taps_fixed(ksize_x, sigma_x, taps.kx) != BV_OK || gaussian_taps_fixed(ksize_y, sigma_y, taps.ky) != BV_OK) {
        set_error("bv_gaussian_blur: kernel cannot be represented in 8.8 fixed point");
        return BV_ERR_INVALID;
    }
    const int rx = ksize_x / 2, ry = ksize_y / 2;
    const size_t raw = (size_t)(kBlurTileW + 2 * rx) * channels * (kBlurTileH + 2 * ry);
    const size_t smem = ((raw + 15) & ~(size_t)15) + (size_t)kBlurTileW * channels * (kBlurTileH + 2 * ry) * 2;
    if (smem > 200 * 1024) {  // large kernels: 16-bit horizontal result through a global scratch image
        BV_REQUIRE(height <= 65535, "image too tall");
        BV_TRY(ensure_scratch(ctx, SCR_MORPH_TMP, (size_t)batch * height * width * channels * sizeof(uint16_t)));
        uint16_t *hz = (uint16_t *)ctx->scratch[SCR_MORPH_TMP];
        // only 3-channel images get here: the largest 1-channel tile (201 x 201 taps) needs 90 944 bytes
        dim3 g((width + 255) / 256, height, batch);
        BV_LAUNCH(ctx, blur_rows16_kernel<3>, g, 256, 0, src_dev, hz, height, width, taps);
        BV_LAUNCH(ctx, blur_cols16_kernel<3>, g, 256, 0, hz, dst_dev, height, width, taps);
        return BV_OK;
    }
    dim3 grid((width + kBlurTileW - 1) / kBlurTileW, (height + kBlurTileH - 1) / kBlurTileH, batch);
#define BV_BLUR(CN, NT)                                                                                                          \
    do {                                                                                                                         \
        if (smem > 48 * 1024)                                                                                                    \
            BV_CUDA(cudaFuncSetAttribute(gaussian_blur_kernel<CN, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        BV_LAUNCH(ctx, (gaussian_blur_kernel<CN, NT>), grid, 256, smem, src_dev, dst_dev, height, width, taps);                  \
    } while (0)
    const int nt = (ksize_x == ksize_y && (ksize_x == 3 || ksize_x == 5 || ksize_x == 7)) ? ksize_x : 0;
    // word-wide path: rows (and so every frame) start 4-byte aligned
    if (nt && ((size_t)width * channels) % 4 == 0 && (reinterpret_cast<uintptr_t>(src_dev) & 3) == 0 &&
        (reinterpret_cast<uintptr_t>(dst_dev) & 3) == 0) {
        dim3 fgrid((unsigned)(((size_t)width * channels + kFastTileWords * 4 - 1) / (kFastTileWords * 4)),
                   (height + kFastTileH - 1) / kFastTileH, batch);
#define BV_BLURF(CN, NT) BV_LAUNCH(ctx, (gaussian_blur_fast_kernel<CN, NT>), fgrid, 256, 0, src_dev, dst_dev, height, width, taps)
        if (channels == 3) {
            if (nt == 3) BV_BLURF(3, 3); else if (nt == 5) BV_BLURF(3, 5); else BV_BLURF(3, 7);
        } else {
            if (nt == 3) BV_BLURF(1, 3); else if (nt == 5) BV_BLURF(1, 5); else BV_BLURF(1, 7);
        }
#undef BV_BLURF
        return BV_OK;
    }
    if (channels == 3) {
        if (nt == 3) BV_BLUR(3, 3); else if (nt == 5) BV_BLUR(3, 5); else if (nt == 7) BV_BLUR(3, 7); else BV_BLUR(3, 0);
    } else {
        if (nt == 3) BV_BLUR(1, 3); else if (nt == 5) BV_BLUR(1, 5); else if (nt == 7) BV_BLUR(1, 7); else BV_BLUR(1, 0);
    }
#undef BV_BLUR
    return BV_OK;
}

extern "C" int bv_warp_affine(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                              int channels, int dst_height, int dst_width, const double *m_host, int border_mode,
                              const uint8_t *border_value_host) {
    BV_REQUIRE(ctx && src_dev && dst_dev && m_host, "null argument");
    BV_REQUIRE(src_dev != dst_dev, "in-place warp is not supported");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0 && dst_height > 0 && dst_width > 0, "sizes must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_REQUIRE(border_mode == BV_BORDER_CONSTANT || border_mode == BV_BORDER_REPLICATE, "border mode must be constant or replicate");
    BV_REQUIRE(height <= 32767 && width <= 32767 && batch <= 65535 && dst_height <= 65535, "image too large");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_bilinear_tab(ctx));
    WarpParams wp;
    memset(&wp, 0, sizeof(wp));
    // cv::warpAffine without WARP_INVERSE_MAP: invert the 2x3 matrix in double
    double M[6];
    for (int i = 0; i < 6; ++i) M[i] = m_host[i];
    double D = M[0] * M[4] - M[1] * M[3];
    D = D != 0 ? 1. / D : 0;
    const double A11 = M[4] * D, A22 = M[0] * D;
    M[0] = A11;
    M[1] *= -D;
    M[3] *= -D;
    M[4] = A22;
    const double b1 = -M[0] * M[2] - M[1] * M[5];
    const double b2 = -M[3] * M[2] - M[4] * M[5];
    M[2] = b1;
    M[5] = b2;
    for (int i = 0; i < 6; ++i) wp.m[i] = M[i];
    wp.border_constant = border_mode == BV_BORDER_CONSTANT;
    for (int c = 0; c < channels; ++c) wp.border_value[c] = border_value_host ? border_value_host[c] : 0;
    BV_TRY(ensure_scratch(ctx, SCR_WARP, sizeof(int) * 2 * ((size_t)dst_width + dst_height)));
    int *coords = (int *)ctx->scratch[SCR_WARP];
    const int longest = dst_width > dst_height ? dst_width : dst_height;
    BV_LAUNCH(ctx, warp_coords_kernel, (longest + 255) / 256, 256, 0, coords, dst_width, dst_height, wp);
    dim3 grid((dst_width + 255) / 256, dst_height, batch);
    if (channels == 3)
        BV_LAUNCH(ctx, warp_affine_kernel<3>, grid, 256, 0, src_dev, dst_dev, height, width, dst_height, dst_width, wp,
                  ctx->d_bilinear_tab, coords);
    else
        BV_LAUNCH(ctx, warp_affine_kernel<1>, grid, 256, 0, src_dev, dst_dev, height, width, dst_height, dst_width, wp,
                  ctx->d_bilinear_tab, coords);
    return BV_OK;
}

extern "C" int bv_lab_shift_local_mean(bv_ctx *ctx, const uint8_t *lab_dev, uint8_t *dst_dev, int batch, int height, int width,
                                       int ksize) {
    BV_REQUIRE(ctx && lab_dev && dst_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(ksize >= 1 && (ksize & 1) && ksize <= 4095, "ksize must be odd and in 1..4095");  // 255 k^2 < 2^32
    BV_REQUIRE(batch <= 65535 && height <= 65535, "image too large");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_scratch(ctx, SCR_WARP, sizeof(uint2) * (size_t)batch * height * width));
    uint2 *sums = (uint2 *)ctx->scratch[SCR_WARP];
    dim3 grid((width + 255) / 256, height, batch);
    BV_LAUNCH(ctx, box_rows_ab_kernel, grid, 256, 0, lab_dev, sums, height, width, ksize / 2);
    BV_LAUNCH(ctx, box_cols_shift_kernel, grid, 256, 0, lab_dev, sums, dst_dev, height, width, ksize / 2,
              1.0 / ((double)ksize * ksize));
    return BV_OK;
}

extern "C" int bv_remap(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width, int channels,
                        int dst_height, int dst_width, const void *map1_dev, const void *map2_dev, int map_format, int border_mode,
                        const uint8_t *border_value_host) {
    BV_REQUIRE(ctx && src_dev && dst_dev && map1_dev && map2_dev, "null argument");
    BV_REQUIRE(src_dev != dst_dev, "in-place remap is not supported");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0 && dst_height > 0 && dst_width > 0, "sizes must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_REQUIRE(map_format == BV_MAP_F32 || map_format == BV_MAP_FIXED, "map format must be BV_MAP_F32 or BV_MAP_FIXED");
    BV_REQUIRE(border_mode == BV_BORDER_CONSTANT || border_mode == BV_BORDER_REPLICATE, "border mode must be constant or replicate");
    BV_REQUIRE(height <= 32767 && width <= 32767 && batch <= 65535 && dst_height <= 65535, "image too large");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_bilinear_tab(ctx));
    WarpParams wp;
    memset(&wp, 0, sizeof(wp));
    wp.border_constant = border_mode == BV_BORDER_CONSTANT;
    for (int c = 0; c < channels; ++c) wp.border_value[c] = border_value_host ? border_value_host[c] : 0;
    dim3 grid((dst_width + 255) / 256, dst_height, batch);
#define BV_REMAP(CN, FX)                                                                                                    \
    BV_LAUNCH(ctx, (remap_kernel<CN, FX>), grid, 256, 0, src_dev, dst_dev, height, width, dst_height, dst_width, map1_dev, \
              map2_dev, wp, ctx->d_bilinear_tab)
    if (channels == 3) {
        if (map_format == BV_MAP_FIXED) BV_REMAP(3, true); else BV_REMAP(3, false);
    } else {
        if (map_format == BV_MAP_FIXED) BV_REMAP(1, true); else BV_REMAP(1, false);
    }
#undef BV_REMAP
    return BV_OK;
}

extern "C" int bv_undistort_maps(bv_ctx *ctx, const double *camera_matrix_host, const double *dist_coeffs_host, int n_dist,
                                 const double *inv_new_camera_rot_host, int width, int height, float *mapx_dev, float *mapy_dev,
                                 int16_t *map_xy_dev, uint16_t *map_frac_dev) {
    BV_REQUIRE(ctx && camera_matrix_host && inv_new_camera_rot_host, "null argument");
    BV_REQUIRE(n_dist == 0 || dist_coeffs_host, "null argument");
    BV_REQUIRE(n_dist == 0 || n_dist == 4 || n_dist == 5 || n_dist == 8, "4, 5 or 8 distortion coefficients (k1 k2 p1 p2 [k3 [k4 k5 k6]])");
    BV_REQUIRE(width > 0 && height > 0 && height <= 65535, "sizes must be positive");
    BV_REQUIRE((mapx_dev && mapy_dev) || (map_xy_dev && map_frac_dev), "no output map given");
    BV_REQUIRE((mapx_dev == nullptr) == (mapy_dev == nullptr) && (map_xy_dev == nullptr) == (map_frac_dev == nullptr),
               "maps come in pairs");
    BV_CUDA(cudaSetDevice(ctx->device));
    UndistortParams p;
    memset(&p, 0, sizeof(p));
    for (int i = 0; i < 9; ++i) p.ir[i] = inv_new_camera_rot_host[i];
    for (int i = 0; i < n_dist; ++i) p.k[i] = dist_coeffs_host[i];
    p.fx = camera_matrix_host[0];
    p.fy = camera_matrix_host[4];
    p.cx = camera_matrix_host[2];
    p.cy = camera_matrix_host[5];
    dim3 grid((width + 255) / 256, height);
    BV_LAUNCH(ctx, undistort_maps_kernel, grid, 256, 0, p, width, height, mapx_dev, mapy_dev, reinterpret_cast<short2 *>(map_xy_dev),
              map_frac_dev);
    return BV_OK;
}
