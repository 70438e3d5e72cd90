// pixel_math.cuh -- per-pixel arithmetic of the hot path, written once as __host__ __device__
// functions.  The CUDA kernels are the product; the host instantiation exists only so that
// tests/hostmath (a test-only shared object, never loaded by the package) can sweep all 2^24
// colours against cv2 in a container without a GPU.
//
// Every function reproduces, bit for bit, what OpenCV 4.x computes for 8-bit images at the
// reference's call sites (utils/color.py:11-32, modules/bins.py:13, color_balance.cpp:654,693);
// the algorithms are restated in oracle/spec_np.py and SURVEY.md Appendix A.
#pragma once
#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define BV_HD __host__ __device__ __forceinline__
#else
#define BV_HD inline
#endif

// float32 operations with explicit rounding: on the device the intrinsics forbid contraction into
// FMA irrespective of compiler flags; on the host build with -ffp-contract=off.
#if defined(__CUDA_ARCH__)
#define BV_FMUL(a, b) __fmul_rn((a), (b))
#define BV_FADD(a, b) __fadd_rn((a), (b))
#define BV_FSUB(a, b) __fsub_rn((a), (b))
#define BV_FDIV(a, b) __fdiv_rn((a), (b))
#define BV_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#define BV_F2I_RZ(x) __float2int_rz(x)
#define BV_F2I_RN(x) __float2int_rn(x)
#define BV_FLOOR(x) floorf(x)
#else
#define BV_FMUL(a, b) ((float)(a) * (float)(b))
#define BV_FADD(a, b) ((float)(a) + (float)(b))
#define BV_FSUB(a, b) ((float)(a) - (float)(b))
#define BV_FDIV(a, b) ((float)(a) / (float)(b))
#define BV_FMA(a, b, c) fmaf((a), (b), (c))
#define BV_F2I_RZ(x) ((int)(x))
#define BV_F2I_RN(x) ((int)nearbyintf(x))
#define BV_FLOOR(x) floorf(x)
#endif

namespace bv {

BV_HD int imin(int a, int b) { return a < b ? a : b; }
BV_HD int imax(int a, int b) { return a > b ? a : b; }
BV_HD int sat_u8(int x) { return x < 0 ? 0 : (x > 255 ? 255 : x); }

// ------------------------------------------------------------------------------------------
// BGR -> HSV, 8-bit, H in [0,180).  sdiv[i] = rint((255<<12)/i), hdiv[i] = rint((180<<12)/(6i)),
// both 0 at i = 0 (OpenCV RGB2HSV_b, hsv_shift = 12).  Neither quotient ever lands on a tie, so
// the rounded division is (2n + i) / (2i) in integers.
// ------------------------------------------------------------------------------------------
constexpr int kHsvShift = 12;
BV_HD int hsv_sdiv(int i) { return i ? (2 * (255 << kHsvShift) + i) / (2 * i) : 0; }
BV_HD int hsv_hdiv(int i) { return i ? (2 * (180 << kHsvShift) + 6 * i) / (12 * i) : 0; }

// sdiv/hdiv: 256-entry int tables (shared memory on the device).
BV_HD void bgr2hsv(int b, int g, int r, const int *sdiv, const int *hdiv, int &h, int &s, int &v) {
    v = imax(imax(b, g), r);
    const int vmin = imin(imin(b, g), r);
    const int diff = v - vmin;
    // branch-free selection (test order r, then g, then b as OpenCV does): a warp never diverges here
    const int hr = g - b, hg = b - r + 2 * diff, hb = r - g + 4 * diff;
    int hh = (v == g) ? hg : hb;
    hh = (v == r) ? hr : hh;
    s = (diff * sdiv[v] + (1 << (kHsvShift - 1))) >> kHsvShift;
    hh = (hh * hdiv[diff] + (1 << (kHsvShift - 1))) >> kHsvShift;  // arithmetic shift
    h = hh + ((hh >> 31) & 180);                                    // hh < 0: += 180
}

#if defined(__CUDACC__)
// The two table entries computed instead of looked up: rint(num / d) for d in 0..255 with num = 255 << 12 (sdiv) or
// (180 << 12) / 6 (hdiv), through the reciprocal unit (MUFU.RCP, a pipe this path does not otherwise use) so that the
// shared-memory instruction path, which bounds the histogram passes (DESIGN.md 4b), loses two look-ups per pixel.
// Exact: num / d = k + r / d with an integer remainder r, never a tie (pixel_math.cuh above), so the quotient is at least
// 1 / (2d) away from the nearest rounding boundary, while the computed value is off by at most
// num / d * (2^-23 [rcp.approx, 1 ulp] + 2^-24 [the multiply]) <= 0.19 / d.  d = 0 gives 1 / 0 = +inf, whose sum with the
// magic constant keeps an all-zero low mantissa: 0, as the tables define.  rcp_tables_check_kernel (balance.cu) compares
// all 2 x 256 values with the integer formulas on the device when a context is created; bv_create fails on a mismatch.
__device__ __forceinline__ int rint_quotient_rcp(float num, int d) {
    const float df = __fsub_rn(__uint_as_float(0x4B000000u | (uint32_t)d), 8388608.f);   // float(d) without the conversion unit
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(df));
    const float q = __fmul_rn(num, r);
    return (int)(__float_as_uint(__fadd_rn(q, 12582912.f)) & 0x3FFFFFu);                 // 2^23 + 2^22: rint in the low mantissa bits
}

__device__ __forceinline__ void bgr2hsv_rcp(int b, int g, int r, int &h, int &s, int &v) {
    v = __vimax3_s32(b, g, r);               // one VIMNMX3 each (the nested two-input form compiles to two for the minimum)
    const int vmin = __vimin3_s32(b, g, r);
    const int diff = v - vmin;
    const int hr = g - b, hg = b - r + 2 * diff, hb = r - g + 4 * diff;
    int hh = (v == g) ? hg : hb;
    hh = (v == r) ? hr : hh;
    const int sd = rint_quotient_rcp((float)(255 << kHsvShift), v);
    const int hd = rint_quotient_rcp((float)((180 << kHsvShift) / 6), diff);
    s = (diff * sd + (1 << (kHsvShift - 1))) >> kHsvShift;
    hh = (hh * hd + (1 << (kHsvShift - 1))) >> kHsvShift;
    // hh < 0: += 180.  hh lies in [-180, 180], so as unsigned numbers the smaller of hh and hh + 180 is the answer
    // (a negative hh is huge): one add + one unsigned min instead of shift + and + add
    h = (int)umin((unsigned)hh, (unsigned)(hh + 180));
}
#endif

// ------------------------------------------------------------------------------------------
// HSV -> BGR, 8-bit, float32.  As cv2 4.13.0 computes it (measured over every H<180,S,V): the
// bracket is a single-rounding multiply-add; whole 32-pixel groups of a row ("vector path")
// truncate x*255, the remaining width%32 pixels of each row round to nearest even.
// ------------------------------------------------------------------------------------------
// Branch-free form.  Of the four OpenCV table values {v, v(1-s), v*fma(-s,f,1), v*fma(-s,1-f,1)}
// a pixel only ever uses three: max = v, min = v(1-s) and ONE mid value (f in odd sectors, 1-f in
// even ones).  The sector then merely permutes (max, mid, min) over (b, g, r), which is a single
// byte-permute of the packed result.  For s == 0 all three collapse to v exactly (1-0 = 1,
// fma(-0,f,1) = 1), so OpenCV's special case needs no branch.  Returns b | g<<8 | r<<16.
BV_HD uint32_t byte_perm3(uint32_t w, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(w, 0u, sel);
#else
    uint32_t out = 0;
    for (int k = 0; k < 4; ++k) {
        const uint32_t n = (sel >> (4 * k)) & 0xF;
        const uint32_t byte = n < 4 ? (w >> (8 * n)) & 0xFF : 0u;
        out |= byte << (8 * k);
    }
    return out;
#endif
}

// kHueBelow180: the caller guarantees H < 180 (a hue this library computed itself), so the sector is < 6.
template <bool kHueBelow180 = false>
BV_HD uint32_t hsv2bgr_packed(int H, int S, int V, bool vector_path) {
    const float hscale = 6.f / 180.f;
    const float inv255 = 1.f / 255.f;
#if defined(__CUDA_ARCH__)
    // Same float32 operations as below, with the int <-> float conversions done on the FMA / ALU pipes instead of the
    // conversion unit (7 of them per pixel otherwise): a byte n ORed into the mantissa of 2^23 is the float 2^23 + n, and
    // fma(2^23 + n, c, -2^23 c) rounds n*c once, exactly like fmul(float(n), c) (2^23 c is exact); adding 2^23 with
    // round-toward-zero leaves floor(x) in the low mantissa bits for 0 <= x < 2^23.
    const float kTwo23 = 8388608.f;
    const float h = __fmaf_rn(__uint_as_float(0x4B000000u | (uint32_t)H), hscale, -kTwo23 * hscale);
    const float s = __fmaf_rn(__uint_as_float(0x4B000000u | (uint32_t)S), inv255, -kTwo23 * inv255);
    const float v = __fmaf_rn(__uint_as_float(0x4B000000u | (uint32_t)V), inv255, -kTwo23 * inv255);
    const float hfloor = __fadd_rz(h, kTwo23);
    int sector = (int)(__float_as_uint(hfloor) & 15u);  // h <= 255 * 6/180 = 8.5
    const float f = BV_FSUB(h, __fsub_rn(hfloor, kTwo23));
#else
    const float h = BV_FMUL((float)H, hscale);
    const float s = BV_FMUL((float)S, inv255);
    const float v = BV_FMUL((float)V, inv255);
    int sector = (int)h;  // h >= 0: truncation == floor
    const float f = BV_FSUB(h, (float)sector);
#endif
    if (!kHueBelow180 && sector >= 6) sector -= 6;  // H >= 180 is out of contract; stay inside the table
    const float fm = (sector & 1) ? f : BV_FSUB(1.f, f);
    const float ymax = BV_FMUL(v, 255.f);
    const float ymin = BV_FMUL(BV_FMUL(v, BV_FSUB(1.f, s)), 255.f);
    const float ymid = BV_FMUL(BV_FMUL(v, BV_FMA(-s, fm, 1.f)), 255.f);
    uint32_t w;
    if (vector_path) {  // values lie in [0, 255]: no saturation needed
#if defined(__CUDA_ARCH__)
        // truncated values sit in byte 0 of the three sums; byte 2 of a float in [2^23, 2^23 + 256) is zero
        const uint32_t amax = __float_as_uint(__fadd_rz(ymax, kTwo23));
        const uint32_t amid = __float_as_uint(__fadd_rz(ymid, kTwo23));
        const uint32_t amin = __float_as_uint(__fadd_rz(ymin, kTwo23));
        w = __byte_perm(__byte_perm(amax, amid, 0x2240), amin, 0x3410);
#else
        w = (uint32_t)BV_F2I_RZ(ymax) | ((uint32_t)BV_F2I_RZ(ymid) << 8) | ((uint32_t)BV_F2I_RZ(ymin) << 16);
#endif
    } else {
        w = (uint32_t)sat_u8(BV_F2I_RN(ymax)) | ((uint32_t)sat_u8(BV_F2I_RN(ymid)) << 8) |
            ((uint32_t)sat_u8(BV_F2I_RN(ymin)) << 16);
    }
    // selector nibbles (r,g,b) -> index into (max=0, mid=1, min=2), one 10-bit field per sector:
    // s0 r=max g=mid b=min | s1 g=max r=mid b=min | s2 g=max b=mid r=min
    // s3 b=max g=mid r=min | s4 b=max r=mid g=min | s5 r=max b=mid g=min
    const unsigned long long kSel = 0x012ull | (0x102ull << 10) | (0x201ull << 20) | (0x210ull << 30) |
                                    (0x120ull << 40) | (0x021ull << 50);
    const uint32_t sel = (uint32_t)(kSel >> (10 * sector)) & 0x3FFu;
    return byte_perm3(w, sel | 0x4000u);  // byte 3 <- zero
}

BV_HD void hsv2bgr(int H, int S, int V, bool vector_path, int &b, int &g, int &r) {
    const uint32_t p = hsv2bgr_packed(H, S, V, vector_path);
    b = (int)(p & 0xFF);
    g = (int)((p >> 8) & 0xFF);
    r = (int)(p >> 16);
}

// ------------------------------------------------------------------------------------------
// BGR -> Lab, 8-bit, fixed point (OpenCV RGB2Lab_b): gamma table (256 x u16), cube-root table
// (3072 x u16); the tables themselves are generated on the host in float32 (lab_tables.cpp).
// ------------------------------------------------------------------------------------------
constexpr int kLabGammaSize = 256;
constexpr int kLabCbrtSize = 3072;
BV_HD int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

BV_HD void bgr2lab(int b, int g, int r, const uint16_t *gtab, const uint16_t *ctab, int &L, int &a, int &bb) {
    const int B = gtab[b], G = gtab[g], R = gtab[r];
    const int fX = ctab[descale(R * 1777 + G * 1541 + B * 778, 12)];
    const int fY = ctab[descale(R * 871 + G * 2929 + B * 296, 12)];
    const int fZ = ctab[descale(R * 73 + G * 448 + B * 3575, 12)];
    // OpenCV saturates these three; over all 2^24 inputs they stay inside L 0..255, a 42..226, b 20..223 on their own
    // (tests/test_hostmath.py compares every colour with cv2), so the clamps are left out
    L = descale(296 * fY - 1336934, 15);
    a = descale(500 * (fX - fY) + (128 << 15), 15);
    bb = descale(200 * (fY - fZ) + (128 << 15), 15);
}

// ------------------------------------------------------------------------------------------
// Lab -> BGR, 8-bit, fixed point (OpenCV Lab2RGBinteger, utils/color.py:27-29 lab_to_bgr): L selects
// (y, fy) from a 256 x 2 table in 2^14 fixed point; a and b offset fy to fx and fz; x and z are the
// cubes (or the linear toe) of those; one 3x3 matrix in 12-bit coefficients; inverse sRGB gamma through
// a 4096-entry table.  0 mismatches against cv2 over all 2^24 inputs (tests/test_hostmath.py).
// ------------------------------------------------------------------------------------------
constexpr int kLabInvGammaSize = 4096;
BV_HD int lab_f_to_xz(int i) {  // abToXZ_b of OpenCV, computed instead of tabulated; i in [-8145, 28718]
    if (i <= 3390) return (i * 108) / 841 - (((1 << 14) * 16 / 116) * 108) / 841;   // C division: toward zero
    return ((i * i) >> 14) * i >> 14;                                                  // i > 0 here
}

BV_HD void lab2bgr(int L, int a, int bb, const uint16_t *yf, const uint8_t *inv_gamma, int &b, int &g, int &r) {
    const int y = yf[2 * L], ify = yf[2 * L + 1];
    const int adiv = ((5 * a * 53687 + (1 << 7)) >> 13) - 128 * (1 << 14) / 500;
    const int bdiv = ((bb * 41943 + (1 << 4)) >> 9) - 128 * (1 << 14) / 200 + 1;
    const int x = lab_f_to_xz(ify + adiv), z = lab_f_to_xz(ify - bdiv);
    int ro = descale(12615 * x - 6296 * y - 2223 * z, 14);
    int go = descale(-3773 * x + 7684 * y + 185 * z, 14);
    int bo = descale(217 * x - 836 * y + 4715 * z, 14);
    ro = imax(0, imin(kLabInvGammaSize - 1, ro));
    go = imax(0, imin(kLabInvGammaSize - 1, go));
    bo = imax(0, imin(kLabInvGammaSize - 1, bo));
    b = inv_gamma[bo];
    g = inv_gamma[go];
    r = inv_gamma[ro];
}

// ------------------------------------------------------------------------------------------
// BGR -> Luv, 8-bit (OpenCV RGB2Luvinterpolate, utils/color.py:30 bgr_to_luv): trilinear interpolation
// in a 33^3 table of int16 (L, u, v) nodes in 2^14 fixed point, 4-bit weights per axis.
// PARITY: the interpolation is OpenCV's; the node table is rebuilt from the published float32 formulas
// with the host libm (powf, cbrtf), whereas OpenCV fills it with its softfloat pow / cubeRoot, so single
// nodes differ by 1 (685 of the 2^24 colours then differ by 1 LSB).  luv_fix.inc holds the 94 node values
// that a fit against cv2 4.13.0 over all 2^24 colours corrects; with them 9 colours remain off by 1 LSB in v
// and none by more (stated tolerance, tests/test_hostmath.py).
// ------------------------------------------------------------------------------------------
constexpr int kLuvDim = 33;
constexpr int kLuvNodes = kLuvDim * kLuvDim * kLuvDim;
#include "luv_fix.inc"

// node (p, q, r) = (R, G, B) index, 4 int16 per node: L, u, v, 0.  Host only: plain float32 expressions, one
// rounding per operation (x86-64 baseline has no fused multiply-add for the compiler to contract into).
#if defined(__CUDACC__)
__host__
#endif
inline void luv_build_table(int16_t *tab) {
    float gl[kLuvDim];
    for (int i = 0; i < kLuvDim; ++i) {
        const float x = (float)i / (float)(kLuvDim - 1);
        const float base = (x + 0.055f) * (float)(1 / 1.055);
        gl[i] = x <= 0.04045f ? x * (float)(1 / 12.92) : powf(base, 2.4f);
    }
    const float C[3][3] = {{0.412453f, 0.357580f, 0.180423f}, {0.212671f, 0.715160f, 0.072169f}, {0.019334f, 0.119193f, 0.950227f}};
    const double wx = 0.950456, wy = 1.0, wz = 1.088754;
    const float un = (float)(4 * wx / (wx + 15 * wy + 3 * wz)), vn = (float)(9 * wy / (wx + 15 * wy + 3 * wz));
    const float eps = 1.1920928955078125e-07f, lthresh = (float)(216. / 24389.), lscale = (float)(24389. / 27.);
    for (int p = 0; p < kLuvDim; ++p)
        for (int q = 0; q < kLuvDim; ++q)
            for (int r = 0; r < kLuvDim; ++r) {
                const float R = gl[p], G = gl[q], B = gl[r];
                volatile float t0, t1, t2;  // volatile: every product and sum is rounded to float32 on its own
                t0 = R * C[0][0]; t1 = G * C[0][1]; t2 = B * C[0][2]; t0 = t0 + t1; const float X = t0 + t2;
                t0 = R * C[1][0]; t1 = G * C[1][1]; t2 = B * C[1][2]; t0 = t0 + t1; const float Y = t0 + t2;
                t0 = R * C[2][0]; t1 = G * C[2][1]; t2 = B * C[2][2]; t0 = t0 + t1; const float Z = t0 + t2;
                float L;
                if (Y < lthresh) {
                    L = Y * lscale;
                } else {
                    t0 = cbrtf(Y) * 116.f;
                    L = t0 - 16.f;
                }
                t0 = 15.f * Y; t1 = 3.f * Z; t0 = X + t0; t0 = t0 + t1;
                float den = t0;
                if (den < eps) den = eps;
                const float d = 1.f / den;
                t0 = L * 13.f;
                t1 = 4.f * X; t1 = t1 * d; t1 = t1 - un; const float u = t0 * t1;
                t2 = 9.f * Y; t2 = t2 * d; t2 = t2 - vn; const float v = t0 * t2;
                int16_t *n = tab + ((size_t)(p * kLuvDim + q) * kLuvDim + r) * 4;
                t0 = 16384.f * L; t0 = t0 / 100.f; n[0] = (int16_t)nearbyintf(t0);
                t0 = u - -134.f; t0 = 16384.f * t0; t0 = t0 / 354.f; n[1] = (int16_t)nearbyintf(t0);
                t0 = v - -140.f; t0 = 16384.f * t0; t0 = t0 / 262.f; n[2] = (int16_t)nearbyintf(t0);
                n[3] = 0;
            }
    for (size_t k = 0; k < sizeof(kLuvNodeFix) / sizeof(kLuvNodeFix[0]); ++k) tab[kLuvNodeFix[k].index] = kLuvNodeFix[k].value;
}

// tab: kLuvNodes x 4 int16 (8 bytes per node)
BV_HD void bgr2luv(int b, int g, int r, const int16_t *tab, int &L, int &u, int &v) {
    const int cx = r * 64, cy = g * 64, cz = b * 64;                  // 8-bit -> 14-bit
    const int tx = cx >> 9, ty = cy >> 9, tz = cz >> 9;               // cell
    const int x = (cx >> 5) & 15, y = (cy >> 5) & 15, z = (cz >> 5) & 15;  // 4-bit position inside the cell
    int a0 = 0, a1 = 0, a2 = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
    for (int k = 0; k < 8; ++k) {
        const int dx = k >> 2, dy = (k >> 1) & 1, dz = k & 1;
        const int w = (dx ? x : 16 - x) * (dy ? y : 16 - y) * (dz ? z : 16 - z);
        // a zero weight may point one node past the table edge: clamp the index, the product vanishes
        const int px = tx + dx > kLuvDim - 1 ? kLuvDim - 1 : tx + dx, py = ty + dy > kLuvDim - 1 ? kLuvDim - 1 : ty + dy,
                  pz = tz + dz > kLuvDim - 1 ? kLuvDim - 1 : tz + dz;
        const int16_t *n = tab + ((size_t)(px * kLuvDim + py) * kLuvDim + pz) * 4;
#if defined(__CUDA_ARCH__)
        // a node is 4 int16 (L, u, v, pad) = one aligned 8-byte load instead of three 2-byte ones
        const uint2 q = __ldg(reinterpret_cast<const uint2 *>(n));
        a0 += (int)(short)(q.x & 0xFFFFu) * w;
        a1 += ((int)q.x >> 16) * w;
        a2 += (int)(short)(q.y & 0xFFFFu) * w;
#else
        a0 += n[0] * w;
        a1 += n[1] * w;
        a2 += n[2] * w;
#endif
    }
    L = sat_u8(descale(a0, 12) / 64);
    u = sat_u8(descale(a1, 12) / 64);
    v = sat_u8(descale(a2, 12) / 64);
}

// ------------------------------------------------------------------------------------------
// BGR -> GRAY (15-bit coefficients) and BGR -> YCrCb (14-bit), 8-bit.
// ------------------------------------------------------------------------------------------
BV_HD int bgr2gray(int b, int g, int r) { return (b * 3735 + g * 19235 + r * 9798 + 16384) >> 15; }

BV_HD void bgr2ycrcb(int b, int g, int r, int &y, int &cr, int &cb) {
    y = (b * 1868 + g * 9617 + r * 4899 + 8192) >> 14;
    cr = sat_u8(((r - y) * 11682 + (128 << 14) + 8192) >> 14);
    cb = sat_u8(((b - y) * 9241 + (128 << 14) + 8192) >> 14);
}

// ------------------------------------------------------------------------------------------
// BGR -> HLS, 8-bit, float32 (OpenCV RGB2HLS_f on scaled input, then rint).  `fused` selects the
// vector formulation (multiply-add in the hue term) cv2 uses for whole 32-px groups of a row.
// ------------------------------------------------------------------------------------------
BV_HD void bgr2hls(int bi, int gi, int ri, bool fused, int &H, int &L, int &S) {
    const float inv255 = 1.f / 255.f;
    const float b = BV_FMUL((float)bi, inv255), g = BV_FMUL((float)gi, inv255), r = BV_FMUL((float)ri, inv255);
    const float vmax = fmaxf(fmaxf(b, g), r), vmin = fminf(fminf(b, g), r);
    const float diff = BV_FSUB(vmax, vmin);
    const float sm = BV_FADD(vmax, vmin);
    const float l = BV_FMUL(sm, 0.5f);
    float h = 0.f, s = 0.f;
    if (diff > 1.1920928955078125e-07f) {  // FLT_EPSILON
        s = l < 0.5f ? BV_FDIV(diff, sm) : BV_FDIV(diff, BV_FSUB(2.f, sm));
        const float k = BV_FDIV(60.f, diff);
        bool wrapped = false;
        if (vmax == r) {
            h = BV_FMUL(BV_FSUB(g, b), k);
            // cv2's vector path wraps a negative hue with the product still unrounded: fma(g - b, k, 360) (measured: the three
            // colours of all 2^24 where (g - b) k + 360 is a rounding tie, e.g. BGR (244, 211, 255), need the single rounding)
            if (fused && h < 0.f) {
                h = BV_FMA(BV_FSUB(g, b), k, 360.f);
                wrapped = true;
            }
        } else if (vmax == g) {
            h = fused ? BV_FMA(BV_FSUB(b, r), k, 120.f) : BV_FADD(BV_FMUL(BV_FSUB(b, r), k), 120.f);
        } else {
            h = fused ? BV_FMA(BV_FSUB(r, g), k, 240.f) : BV_FADD(BV_FMUL(BV_FSUB(r, g), k), 240.f);
        }
        if (!wrapped && h < 0.f) h = BV_FADD(h, 360.f);
    }
    H = sat_u8(BV_F2I_RN(BV_FMUL(h, 0.5f)));
    L = sat_u8(BV_F2I_RN(BV_FMUL(l, 255.f)));
    S = sat_u8(BV_F2I_RN(BV_FMUL(s, 255.f)));
}

// ------------------------------------------------------------------------------------------
// cv2.resize INTER_LINEAR, 8-bit: 11-bit fixed-point coefficients (OpenCV resize.cpp,
// HResizeLinear / VResizeLinear for uchar).  One axis at a time.
// ------------------------------------------------------------------------------------------
struct LinCoef {
    int i0, i1;  // clamped source indices
    int w0, w1;  // int16 weights, nominally summing to 2048
};

BV_HD LinCoef linear_coef(int d, int src, double scale, bool horizontal) {
    float f = (float)(((double)d + 0.5) * scale - 0.5);
    int s = (int)BV_FLOOR(f);
    f = BV_FSUB(f, (float)s);
    if (horizontal) {
        if (s < 0) { f = 0.f; s = 0; }
        if (s >= src - 1) { f = 0.f; s = src - 1; }
    }
    LinCoef c;
    int w1 = BV_F2I_RN(BV_FMUL(f, 2048.f));
    int w0 = BV_F2I_RN(BV_FMUL(BV_FSUB(1.f, f), 2048.f));
    c.w1 = w1 < -32768 ? -32768 : (w1 > 32767 ? 32767 : w1);
    c.w0 = w0 < -32768 ? -32768 : (w0 > 32767 ? 32767 : w0);
    c.i0 = s < 0 ? 0 : (s > src - 1 ? src - 1 : s);
    c.i1 = s + 1 < 0 ? 0 : (s + 1 > src - 1 ? src - 1 : s + 1);
    return c;
}

// vertical blend of two horizontally interpolated int32 rows
BV_HD int linear_vblend(int h0, int h1, int b0, int b1) {
    return sat_u8((((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2);
}

}  // namespace bv
