// cvt.cu -- pointwise kernels: colour conversion (+ channel split), inRange, threshold, LUT, and
// the fused convert+inRange.  Replaces cv2.cvtColor / cv2.split / cv2.inRange / cv2.threshold at
// the reference call sites utils/color.py:11-32,105-201, modules/bins.py:13-16,
// modules/preprocessor.py:56-109.
//
// Data layout: flat interleaved uint8.  A thread owns 16 consecutive pixels = 48 bytes in (three
// 128-bit loads), and writes 48 bytes (3-channel result), 16 bytes (1-channel result) and/or
// 3 x 16 bytes (split planes) with 128-bit stores.  HBM-bound by design: 3 B/px in, 1..6 B/px out.
#include "common.cuh"
#include "convert.cuh"
#include "pointwise.cuh"

namespace bv {

// ----------------------------------------------------------------------------------------------
// cvt: src(3ch) -> dst (3ch or 1ch) and/or split planes
// ----------------------------------------------------------------------------------------------
template <int CODE, bool HAS_DST, bool HAS_PLANES, bool VEC>
__global__ void __launch_bounds__(256) cvt_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                  uint8_t *__restrict__ p0, uint8_t *__restrict__ p1,
                                                  uint8_t *__restrict__ p2, size_t npx, int width,
                                                  const uint16_t *__restrict__ g_gamma,
                                                  const uint16_t *__restrict__ g_cbrt) {
    __shared__ SmemTabs tabs;
    init_tabs<CODE>(tabs, g_gamma, g_cbrt);
    const int vec_end = width - (width % 32);
    const size_t ngroups = npx / 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    if (VEC) {
        for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
            Px16 in;
            load_px16<false>(src, g, in);
            int x = CvtTraits<CODE>::kNeedsX ? (int)((g * 16) % (size_t)width) : 0;
            Px16 out;
            uint32_t q0[4] = {0, 0, 0, 0}, q1[4] = {0, 0, 0, 0}, q2[4] = {0, 0, 0, 0};
#pragma unroll
            for (int k = 0; k < 12; ++k) out.w[k] = 0;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                int o0, o1, o2;
                convert_px<CODE>(BV_GETB(in.w, 3 * j), BV_GETB(in.w, 3 * j + 1), BV_GETB(in.w, 3 * j + 2),
                                 x < vec_end, tabs, o0, o1, o2);
                if (CvtTraits<CODE>::kNeedsX) {
                    if (++x == width) x = 0;
                }
                if (HAS_DST && !CvtTraits<CODE>::kOneChannel) {
                    BV_PUTB(out.w, 3 * j, o0);
                    BV_PUTB(out.w, 3 * j + 1, o1);
                    BV_PUTB(out.w, 3 * j + 2, o2);
                }
                if (HAS_PLANES || CvtTraits<CODE>::kOneChannel) BV_PUTB(q0, j, o0);
                if (HAS_PLANES) {
                    BV_PUTB(q1, j, o1);
                    BV_PUTB(q2, j, o2);
                }
            }
            if (HAS_DST) {
                if (CvtTraits<CODE>::kOneChannel)
                    st_stream(reinterpret_cast<uint4 *>(dst) + g, make_uint4(q0[0], q0[1], q0[2], q0[3]));
                else
                    store_px16(dst, g, out);
            }
            if (HAS_PLANES) {
                st_stream(reinterpret_cast<uint4 *>(p0) + g, make_uint4(q0[0], q0[1], q0[2], q0[3]));
                if (!CvtTraits<CODE>::kOneChannel) {
                    st_stream(reinterpret_cast<uint4 *>(p1) + g, make_uint4(q1[0], q1[1], q1[2], q1[3]));
                    st_stream(reinterpret_cast<uint4 *>(p2) + g, make_uint4(q2[0], q2[1], q2[2], q2[3]));
                }
            }
        }
    }
    // scalar path: the < 16 trailing pixels (VEC) or everything (unaligned buffers)
    const size_t first = VEC ? ngroups * 16 : 0;
    for (size_t p = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        const int x = CvtTraits<CODE>::kNeedsX ? (int)(p % (size_t)width) : 0;
        int o0, o1, o2;
        convert_px<CODE>(src[3 * p], src[3 * p + 1], src[3 * p + 2], x < vec_end, tabs, o0, o1, o2);
        if (HAS_DST) {
            if (CvtTraits<CODE>::kOneChannel) {
                dst[p] = (uint8_t)o0;
            } else {
                dst[3 * p] = (uint8_t)o0;
                dst[3 * p + 1] = (uint8_t)o1;
                dst[3 * p + 2] = (uint8_t)o2;
            }
        }
        if (HAS_PLANES) {
            p0[p] = (uint8_t)o0;
            if (!CvtTraits<CODE>::kOneChannel) {
                p1[p] = (uint8_t)o1;
                p2[p] = (uint8_t)o2;
            }
        }
    }
}

__global__ void __launch_bounds__(256) gray2bgr_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                       size_t npx) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        const uint8_t v = src[p];
        dst[3 * p] = v;
        dst[3 * p + 1] = v;
        dst[3 * p + 2] = v;
    }
}

// ----------------------------------------------------------------------------------------------
// fused convert + inRange -> uint8 mask (0/255).  CODE = -1 thresholds the source itself
// (plain 3-channel cv2.inRange).
// ----------------------------------------------------------------------------------------------
template <int CODE, bool VEC>
__global__ void __launch_bounds__(256) cvt_inrange_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ mask,
                                                          size_t npx, int width, Bounds3 bd,
                                                          const uint16_t *__restrict__ g_gamma,
                                                          const uint16_t *__restrict__ g_cbrt) {
    __shared__ SmemTabs tabs;
    init_tabs<CODE>(tabs, g_gamma, g_cbrt);
    const int vec_end = width - (width % 32);
    const size_t ngroups = npx / 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    constexpr bool one = CvtTraits<CODE>::kOneChannel;
    if (VEC) {
        for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
            Px16 in;
            load_px16<false>(src, g, in);
            int x = CvtTraits<CODE>::kNeedsX ? (int)((g * 16) % (size_t)width) : 0;
            uint32_t q[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                int o0, o1, o2;
                convert_px<CODE>(BV_GETB(in.w, 3 * j), BV_GETB(in.w, 3 * j + 1), BV_GETB(in.w, 3 * j + 2),
                                 x < vec_end, tabs, o0, o1, o2);
                if (CvtTraits<CODE>::kNeedsX) {
                    if (++x == width) x = 0;
                }
                bool in_r = o0 >= bd.lo[0] && o0 <= bd.hi[0];
                if (!one) in_r = in_r && o1 >= bd.lo[1] && o1 <= bd.hi[1] && o2 >= bd.lo[2] && o2 <= bd.hi[2];
                BV_PUTB(q, j, in_r ? 255u : 0u);
            }
            st_stream(reinterpret_cast<uint4 *>(mask) + g, make_uint4(q[0], q[1], q[2], q[3]));
        }
    }
    const size_t first = VEC ? ngroups * 16 : 0;
    for (size_t p = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        const int x = CvtTraits<CODE>::kNeedsX ? (int)(p % (size_t)width) : 0;
        int o0, o1, o2;
        convert_px<CODE>(src[3 * p], src[3 * p + 1], src[3 * p + 2], x < vec_end, tabs, o0, o1, o2);
        bool in_r = o0 >= bd.lo[0] && o0 <= bd.hi[0];
        if (!one) in_r = in_r && o1 >= bd.lo[1] && o1 <= bd.hi[1] && o2 >= bd.lo[2] && o2 <= bd.hi[2];
        mask[p] = in_r ? 255 : 0;
    }
}

// ----------------------------------------------------------------------------------------------
// 1-channel pointwise: inRange, threshold, LUT (16 bytes per thread)
// ----------------------------------------------------------------------------------------------
template <int OP, bool VEC>
__global__ void __launch_bounds__(256) op1_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, size_t n,
                                                  Op1Params prm, const uint8_t *__restrict__ g_lut) {
    __shared__ uint8_t lut[256];
    if (OP == OP1_LUT) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = g_lut[i];
        __syncthreads();
    }
    const size_t nvec = n / 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    if (VEC) {
        for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < nvec; g += stride) {
            const uint4 v = ld_stream(reinterpret_cast<const uint4 *>(src) + g);
            const uint32_t in[4] = {v.x, v.y, v.z, v.w};
            uint32_t out[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 16; ++j) BV_PUTB(out, j, op1_apply(OP, prm, BV_GETB(in, j), lut));
            st_stream(reinterpret_cast<uint4 *>(dst) + g, make_uint4(out[0], out[1], out[2], out[3]));
        }
    }
    const size_t first = VEC ? nvec * 16 : 0;
    for (size_t i = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        dst[i] = (uint8_t)op1_apply(OP, prm, src[i], lut);
}

// 3-channel LUT (per-channel tables), 16 px per thread
template <bool VEC>
__global__ void __launch_bounds__(256) lut3_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, size_t npx,
                                                   const uint8_t *__restrict__ g_lut) {
    __shared__ uint8_t lut[768];
    for (int i = threadIdx.x; i < 768; i += blockDim.x) lut[i] = g_lut[i];
    __syncthreads();
    const size_t ngroups = npx / 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    if (VEC) {
        for (size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
            Px16 in, out;
            load_px16<false>(src, g, in);
#pragma unroll
            for (int k = 0; k < 12; ++k) out.w[k] = 0;
#pragma unroll
            for (int k = 0; k < 48; ++k) BV_PUTB(out.w, k, lut[(k % 3) * 256 + BV_GETB(in.w, k)]);
            store_px16(dst, g, out);
        }
    }
    const size_t first = VEC ? ngroups * 48 : 0;
    for (size_t i = first + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx * 3; i += stride)
        dst[i] = lut[(i % 3) * 256 + src[i]];
}

// ----------------------------------------------------------------------------------------------
// weighted colour distance (utils/color.py:66-103).  Arithmetic as numpy 2.x evaluates the
// reference's expression: the square is float32, the weight is a float64 scalar, so each channel's
// update is dists = float32(double(dists) + w * double(float32 square)).
// ----------------------------------------------------------------------------------------------
struct ColorDistParams {
    float color[3];
    double weight[3];
    int use[3];
    float max_dist;  // inclusive upper bound on dists (already squared), as float32 like cv2.inRange
};

__global__ void __launch_bounds__(256) color_distance_kernel(const uint8_t *__restrict__ p0, const uint8_t *__restrict__ p1,
                                                             const uint8_t *__restrict__ p2, uint8_t *__restrict__ mask,
                                                             uint8_t *__restrict__ dist, float *__restrict__ dists_f32, size_t n,
                                                             ColorDistParams prm) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint8_t v[3] = {p0[i], p1[i], p2[i]};
        float d = 0.f;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (!prm.use[c]) continue;
            const float t = __fsub_rn((float)v[c], prm.color[c]);
            const float sq = __fmul_rn(t, t);
            d = (float)__dadd_rn((double)d, __dmul_rn(prm.weight[c], (double)sq));
        }
        if (mask) mask[i] = (d >= 0.f && d <= prm.max_dist) ? 255 : 0;
        if (dist) dist[i] = (uint8_t)(((int)__fsqrt_rn(d)) & 0xFF);  // np.uint8(np.sqrt(.)): truncate, wrap
        if (dists_f32) dists_f32[i] = d;
    }
}

// ----------------------------------------------------------------------------------------------
// k-th smallest of a float32 array (the order statistics np.percentile interpolates between,
// utils/color.py:98-99): radix select over the order-preserving integer image of the floats,
// 8 bits per pass, each pass one 256-bin histogram of the elements that match the prefix so far.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t float_key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(256) select_hist_kernel(const float *__restrict__ v, size_t n, uint32_t prefix, uint32_t prefix_mask,
                                                          int shift, uint32_t *__restrict__ hist) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t k = float_key(v[i]);
        if ((k & prefix_mask) == prefix) atomicAdd(&h[(k >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

// BGR -> Luv: 8 table nodes per pixel gathered from the 287 KB node table (L2 resident); a debug
// split-post of the preprocessor (modules/preprocessor.py:76-80), not a throughput path.
__global__ void __launch_bounds__(256) bgr2luv_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                      uint8_t *__restrict__ p0, uint8_t *__restrict__ p1, uint8_t *__restrict__ p2,
                                                      size_t npx, const int16_t *__restrict__ tab) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += stride) {
        int L, u, v;
        bgr2luv(src[3 * i], src[3 * i + 1], src[3 * i + 2], tab, L, u, v);
        if (dst) {
            dst[3 * i] = (uint8_t)L;
            dst[3 * i + 1] = (uint8_t)u;
            dst[3 * i + 2] = (uint8_t)v;
        }
        if (p0) {
            p0[i] = (uint8_t)L;
            p1[i] = (uint8_t)u;
            p2[i] = (uint8_t)v;
        }
    }
}

static int launch_luv(bv_ctx *ctx, const uint8_t *src, uint8_t *dst, uint8_t *const *planes, size_t npx) {
    if (!ctx->d_luv_tab) {
        static int16_t tab[kLuvNodes * 4];
        static bool built = false;
        if (!built) {
            luv_build_table(tab);
            built = true;
        }
        BV_CUDA(cudaMalloc(&ctx->d_luv_tab, sizeof(tab)));
        BV_CUDA(cudaMemcpyAsync(ctx->d_luv_tab, tab, sizeof(tab), cudaMemcpyHostToDevice, ctx->stream));
        BV_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    BV_LAUNCH(ctx, bgr2luv_kernel, grid_for(ctx, npx, 256, 8), 256, 0, src, dst, planes ? planes[0] : nullptr,
              planes ? planes[1] : nullptr, planes ? planes[2] : nullptr, npx, ctx->d_luv_tab);
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// host dispatch
// ----------------------------------------------------------------------------------------------
template <int CODE>
static int launch_cvt(bv_ctx *ctx, const uint8_t *src, uint8_t *dst, uint8_t *const *planes, size_t npx, int width) {
    const bool has_dst = dst != nullptr, has_pl = planes != nullptr;
    bool vec = host_aligned16(src) && (!has_dst || host_aligned16(dst));
    if (has_pl) vec = vec && host_aligned16(planes[0]) && (CvtTraits<CODE>::kOneChannel || (host_aligned16(planes[1]) && host_aligned16(planes[2])));
    uint8_t *p0 = has_pl ? planes[0] : nullptr;
    uint8_t *p1 = has_pl && !CvtTraits<CODE>::kOneChannel ? planes[1] : nullptr;
    uint8_t *p2 = has_pl && !CvtTraits<CODE>::kOneChannel ? planes[2] : nullptr;
    const int grid = grid_for(ctx, vec ? (npx + 15) / 16 : npx, 256, 8);
#define BV_CVT_CASE(D, P, V)                                                                                    \
    BV_LAUNCH(ctx, (cvt_kernel<CODE, D, P, V>), grid, 256, 0, src, dst, p0, p1, p2, npx, width, ctx->d_lab_gamma, \
              ctx->d_lab_cbrt)
    if (has_dst && has_pl) {
        if (vec) BV_CVT_CASE(true, true, true); else BV_CVT_CASE(true, true, false);
    } else if (has_dst) {
        if (vec) BV_CVT_CASE(true, false, true); else BV_CVT_CASE(true, false, false);
    } else {
        if (vec) BV_CVT_CASE(false, true, true); else BV_CVT_CASE(false, true, false);
    }
#undef BV_CVT_CASE
    return BV_OK;
}

template <int CODE>
static int launch_cvt_inrange(bv_ctx *ctx, const uint8_t *src, uint8_t *mask, size_t npx, int width, const Bounds3 &bd) {
    const bool vec = host_aligned16(src) && host_aligned16(mask);
    const int grid = grid_for(ctx, vec ? (npx + 15) / 16 : npx, 256, 8);
    if (vec)
        BV_LAUNCH(ctx, (cvt_inrange_kernel<CODE, true>), grid, 256, 0, src, mask, npx, width, bd, ctx->d_lab_gamma,
                  ctx->d_lab_cbrt);
    else
        BV_LAUNCH(ctx, (cvt_inrange_kernel<CODE, false>), grid, 256, 0, src, mask, npx, width, bd, ctx->d_lab_gamma,
                  ctx->d_lab_cbrt);
    return BV_OK;
}

int cvt_in_range_impl(bv_ctx *ctx, const uint8_t *src, uint8_t *mask, size_t npx, int width, int code,
                      const uint8_t *lo, const uint8_t *hi) {
    Bounds3 bd;
    for (int k = 0; k < 3; ++k) {
        bd.lo[k] = lo[k];
        bd.hi[k] = hi[k];
    }
    switch (code) {
        case -1: return launch_cvt_inrange<-1>(ctx, src, mask, npx, width, bd);
        case BV_BGR2HSV: return launch_cvt_inrange<BV_BGR2HSV>(ctx, src, mask, npx, width, bd);
        case BV_BGR2LAB: return launch_cvt_inrange<BV_BGR2LAB>(ctx, src, mask, npx, width, bd);
        case BV_BGR2GRAY: return launch_cvt_inrange<BV_BGR2GRAY>(ctx, src, mask, npx, width, bd);
        case BV_BGR2YCRCB: return launch_cvt_inrange<BV_BGR2YCRCB>(ctx, src, mask, npx, width, bd);
        case BV_HSV2BGR: return launch_cvt_inrange<BV_HSV2BGR>(ctx, src, mask, npx, width, bd);
        case BV_BGR2HLS: return launch_cvt_inrange<BV_BGR2HLS>(ctx, src, mask, npx, width, bd);
        case BV_BGR2RGB: return launch_cvt_inrange<BV_BGR2RGB>(ctx, src, mask, npx, width, bd);
        case BV_LAB2BGR: return launch_cvt_inrange<BV_LAB2BGR>(ctx, src, mask, npx, width, bd);
        default: set_error("bv_cvt_in_range: unknown conversion code %d", code); return BV_ERR_INVALID;
    }
}

}  // namespace bv

using namespace bv;

extern "C" int bv_cvt_color(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, uint8_t *const *planes_dev,
                            int batch, int height, int width, int code) {
    BV_REQUIRE(ctx && src_dev, "null context or source");
    BV_REQUIRE(dst_dev || planes_dev, "need dst_dev or planes_dev");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t npx = (size_t)batch * height * width;
    switch (code) {
        case BV_BGR2HSV: return launch_cvt<BV_BGR2HSV>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2LAB: return launch_cvt<BV_BGR2LAB>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2GRAY: return launch_cvt<BV_BGR2GRAY>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2YCRCB: return launch_cvt<BV_BGR2YCRCB>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_HSV2BGR: return launch_cvt<BV_HSV2BGR>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2HLS: return launch_cvt<BV_BGR2HLS>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2RGB: return launch_cvt<BV_BGR2RGB>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_LAB2BGR: return launch_cvt<BV_LAB2BGR>(ctx, src_dev, dst_dev, planes_dev, npx, width);
        case BV_BGR2LUV: return launch_luv(ctx, src_dev, dst_dev, planes_dev, npx);
        case BV_GRAY2BGR: {
            BV_REQUIRE(dst_dev && !planes_dev, "GRAY2BGR writes dst_dev only");
            BV_LAUNCH(ctx, gray2bgr_kernel, grid_for(ctx, npx, 256, 8), 256, 0, src_dev, dst_dev, npx);
            return BV_OK;
        }
        default: set_error("bv_cvt_color: unknown conversion code %d", code); return BV_ERR_INVALID;
    }
}

extern "C" int bv_cvt_in_range(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *mask_dev, int batch, int height,
                               int width, int code, const uint8_t *lo_host, const uint8_t *hi_host) {
    BV_REQUIRE(ctx && src_dev && mask_dev && lo_host && hi_host, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_CUDA(cudaSetDevice(ctx->device));
    return cvt_in_range_impl(ctx, src_dev, mask_dev, (size_t)batch * height * width, width, code, lo_host, hi_host);
}

extern "C" int bv_in_range(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *mask_dev, int batch, int height, int width,
                           int channels, const uint8_t *lo_host, const uint8_t *hi_host) {
    BV_REQUIRE(ctx && src_dev && mask_dev && lo_host && hi_host, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t npx = (size_t)batch * height * width;
    if (channels == 3) return cvt_in_range_impl(ctx, src_dev, mask_dev, npx, width, -1, lo_host, hi_host);
    Op1Params prm{lo_host[0], hi_host[0], 0};
    const bool vec = host_aligned16(src_dev) && host_aligned16(mask_dev);
    const int grid = grid_for(ctx, vec ? (npx + 15) / 16 : npx, 256, 8);
    if (vec)
        BV_LAUNCH(ctx, (op1_kernel<OP1_INRANGE, true>), grid, 256, 0, src_dev, mask_dev, npx, prm, nullptr);
    else
        BV_LAUNCH(ctx, (op1_kernel<OP1_INRANGE, false>), grid, 256, 0, src_dev, mask_dev, npx, prm, nullptr);
    return BV_OK;
}

extern "C" int bv_threshold(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n, int thresh, int maxval,
                            int type) {
    BV_REQUIRE(ctx && src_dev && dst_dev, "null argument");
    BV_REQUIRE(type >= BV_THRESH_BINARY && type <= BV_THRESH_TOZERO_INV, "unknown threshold type");
    BV_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return BV_OK;
    // cv2.threshold on 8-bit: thresh is floored and clamped, maxval saturated (imgproc thresh.cpp)
    Op1Params prm{thresh, maxval < 0 ? 0 : (maxval > 255 ? 255 : maxval), type};
    if (type == BV_THRESH_TRUNC) prm.a = thresh < 0 ? 0 : (thresh > 255 ? 255 : thresh);
    const bool vec = host_aligned16(src_dev) && host_aligned16(dst_dev);
    const int grid = grid_for(ctx, vec ? (n + 15) / 16 : n, 256, 8);
    if (vec)
        BV_LAUNCH(ctx, (op1_kernel<OP1_THRESH, true>), grid, 256, 0, src_dev, dst_dev, n, prm, nullptr);
    else
        BV_LAUNCH(ctx, (op1_kernel<OP1_THRESH, false>), grid, 256, 0, src_dev, dst_dev, n, prm, nullptr);
    return BV_OK;
}

static int color_distance_launch(bv_ctx *ctx, const uint8_t *const *planes_dev, size_t n, const double *color_host,
                                 const double *weights_host, const int32_t *use_host, double max_dist_sq, uint8_t *mask_dev,
                                 uint8_t *dist_dev, float *dists_f32_dev) {
    BV_REQUIRE(ctx && planes_dev && planes_dev[0] && planes_dev[1] && planes_dev[2] && color_host && weights_host && use_host,
               "null argument");
    BV_REQUIRE(mask_dev || dist_dev || dists_f32_dev, "need an output");
    BV_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return BV_OK;
    ColorDistParams prm;
    for (int c = 0; c < 3; ++c) {
        prm.color[c] = (float)color_host[c];
        prm.weight[c] = weights_host[c];
        prm.use[c] = use_host[c];
    }
    prm.max_dist = (float)max_dist_sq;
    BV_LAUNCH(ctx, color_distance_kernel, grid_for(ctx, n, 256, 8), 256, 0, planes_dev[0], planes_dev[1], planes_dev[2],
              mask_dev, dist_dev, dists_f32_dev, n, prm);
    return BV_OK;
}

extern "C" int bv_color_distance(bv_ctx *ctx, const uint8_t *const *planes_dev, size_t n, const double *color_host,
                                 const double *weights_host, const int32_t *use_host, double max_dist_sq,
                                 uint8_t *mask_dev, uint8_t *dist_dev) {
    return color_distance_launch(ctx, planes_dev, n, color_host, weights_host, use_host, max_dist_sq, mask_dev, dist_dev, nullptr);
}

extern "C" int bv_color_distance_f32(bv_ctx *ctx, const uint8_t *const *planes_dev, size_t n, const double *color_host,
                                     const double *weights_host, const int32_t *use_host, float *dists_dev) {
    BV_REQUIRE(dists_dev, "null argument");
    return color_distance_launch(ctx, planes_dev, n, color_host, weights_host, use_host, 0.0, nullptr, nullptr, dists_dev);
}

namespace bv {
int select_kth_f32(bv_ctx *ctx, const float *values_dev, size_t n, size_t k, float *value_host) {
    BV_TRY(ensure_scratch(ctx, SCR_MORPH_SE, 256 * sizeof(uint32_t)));
    uint32_t *d_hist = (uint32_t *)ctx->scratch[SCR_MORPH_SE];
    uint32_t prefix = 0, mask = 0, hist[256];
    size_t rank = k;  // rank of the wanted element among those matching the prefix
    for (int shift = 24; shift >= 0; shift -= 8) {
        BV_CUDA(cudaMemsetAsync(d_hist, 0, sizeof(hist), ctx->stream));
        BV_LAUNCH(ctx, select_hist_kernel, grid_for(ctx, n, 256, 8), 256, 0, values_dev, n, prefix, mask, shift, d_hist);
        BV_CUDA(cudaMemcpyAsync(hist, d_hist, sizeof(hist), cudaMemcpyDeviceToHost, ctx->stream));
        BV_CUDA(cudaStreamSynchronize(ctx->stream));
        int b = 0;
        for (; b < 256; ++b) {
            if (rank < hist[b]) break;
            rank -= hist[b];
        }
        if (b == 256) {
            set_error("bv_select_kth_f32: inconsistent histogram (NaN input?)");
            return BV_ERR_INVALID;
        }
        prefix |= (uint32_t)b << shift;
        mask |= 0xFFu << shift;
    }
    const uint32_t u = (prefix & 0x80000000u) ? (prefix & 0x7FFFFFFFu) : ~prefix;
    memcpy(value_host, &u, sizeof(float));
    return BV_OK;
}
}  // namespace bv

extern "C" int bv_select_kth_f32(bv_ctx *ctx, const float *values_dev, size_t n, size_t k, float *value_host) {
    BV_REQUIRE(ctx && values_dev && value_host, "null argument");
    BV_REQUIRE(n > 0 && k < n, "k must be below n");
    BV_CUDA(cudaSetDevice(ctx->device));
    return bv::select_kth_f32(ctx, values_dev, n, k, value_host);
}


extern "C" int bv_apply_lut(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, size_t n_pixels, int channels,
                            const uint8_t *lut_host) {
    BV_REQUIRE(ctx && src_dev && dst_dev && lut_host, "null argument");
    BV_REQUIRE(channels == 1 || channels == 3, "channels must be 1 or 3");
    BV_CUDA(cudaSetDevice(ctx->device));
    if (n_pixels == 0) return BV_OK;
    BV_TRY(ensure_scratch(ctx, SCR_MORPH_SE, 768));
    uint8_t *d_lut = (uint8_t *)ctx->scratch[SCR_MORPH_SE];
    BV_CUDA(cudaMemcpyAsync(d_lut, lut_host, (size_t)channels * 256, cudaMemcpyHostToDevice, ctx->stream));
    const bool vec = host_aligned16(src_dev) && host_aligned16(dst_dev);
    Op1Params prm{0, 0, 0};
    if (channels == 1) {
        const int grid = grid_for(ctx, vec ? (n_pixels + 15) / 16 : n_pixels, 256, 8);
        if (vec)
            BV_LAUNCH(ctx, (op1_kernel<OP1_LUT, true>), grid, 256, 0, src_dev, dst_dev, n_pixels, prm, d_lut);
        else
            BV_LAUNCH(ctx, (op1_kernel<OP1_LUT, false>), grid, 256, 0, src_dev, dst_dev, n_pixels, prm, d_lut);
    } else {
        const int grid = grid_for(ctx, vec ? (n_pixels + 15) / 16 : n_pixels * 3, 256, 8);
        if (vec)
            BV_LAUNCH(ctx, lut3_kernel<true>, grid, 256, 0, src_dev, dst_dev, n_pixels, d_lut);
        else
            BV_LAUNCH(ctx, lut3_kernel<false>, grid, 256, 0, src_dev, dst_dev, n_pixels, d_lut);
    }
    return BV_OK;
}
