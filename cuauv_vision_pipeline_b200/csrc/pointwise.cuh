// pointwise.cuh -- the 1-channel pointwise rules of cvt.cu's op1_kernel (inRange, threshold, LUT), shared with the
// per-frame automatic thresholds of thresh.cu so that both apply cv2.threshold's five types with the same arithmetic.
#pragma once
#include "common.cuh"

namespace bv {

enum Op1 { OP1_INRANGE = 0, OP1_THRESH = 1, OP1_LUT = 2 };

struct Op1Params {
    int a, b, type;  // inRange: lo, hi;  threshold: thresh, maxval, type
};

#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t op1_apply(int op, const Op1Params &p, uint32_t x, const uint8_t *lut) {
    if (op == OP1_INRANGE) return ((int)x >= p.a && (int)x <= p.b) ? 255u : 0u;
    if (op == OP1_LUT) return lut[x];
    const bool above = (int)x > p.a;
    switch (p.type) {
        case BV_THRESH_BINARY: return above ? (uint32_t)p.b : 0u;
        case BV_THRESH_BINARY_INV: return above ? 0u : (uint32_t)p.b;
        case BV_THRESH_TRUNC: return above ? (uint32_t)p.a : x;
        case BV_THRESH_TOZERO: return above ? x : 0u;
        default: return above ? 0u : x;
    }
}
#endif

}  // namespace bv
