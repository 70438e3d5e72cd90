// morph.cuh -- internal interface of the morphology / bit-mask kernels (morph.cu).
#pragma once
#include "common.cuh"

namespace bv {

// Bit-packed binary image: per frame `height` rows of `words_per_row(width)` uint32; bit i of
// word w is pixel x = 32*w + i; bits at x >= width are always 0.
inline int words_per_row(int width) { return (width + 31) / 32; }
inline size_t bits_frame_words(int height, int width) { return (size_t)height * words_per_row(width); }

// uint8 mask (non-zero = set) -> bits, and bits -> uint8 0/255
int mask_to_bits(bv_ctx *ctx, const uint8_t *mask, uint32_t *bits, int batch, int height, int width);
int bits_to_mask(bv_ctx *ctx, const uint32_t *bits, uint8_t *mask, int batch, int height, int width);

// One bv_morph_op with a kw x kh rectangle (anchor = centre) on bit-packed images.  `bits` holds
// the input and receives the result; `tmp`, `tmp2` and `tmp3` are same-sized scratch images.  Extents
// over 31 px take several passes; iterations < 1 is the identity, except for GRADIENT (all zero, as cv2).
int morph_bits_rect(bv_ctx *ctx, uint32_t *bits, uint32_t *tmp, uint32_t *tmp2, uint32_t *tmp3, int batch, int height,
                    int width, int op, int kw, int kh, int iterations);

// The whole list of steps in one launch (tile + halo in shared memory), writing the final bits
// (dst_bits, may be null, must differ from bits) and/or the uint8 mask (may be null).  *done = false
// when the chain does not qualify; nothing was launched then.
int morph_bits_chain(bv_ctx *ctx, const uint32_t *bits, uint32_t *dst_bits, uint8_t *mask, int batch, int height, int width,
                     int n_steps, const int *ops, const int *kws, const int *khs, const int *iters, bool *done);

// ---- labelling (ccl.cu) ----
struct LabelScratch {
    int *parent;      // union-find parents, one int per pixel of the batch
    int *row_count;   // roots per row
    int *row_off;     // exclusive scan of row_count per frame
    int *n_fallback;  // blob counts when the caller does not want them
};
int label_scratch(bv_ctx *ctx, int batch, int height, int width, LabelScratch *ls);
int label_bits(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int batch, int height, int width, bv_blob *blobs,
               int max_blobs, int32_t *n_blobs);
int label_bits_slice(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int f0, int nf, int height, int width, bv_blob *blobs,
                     int max_blobs, int32_t *n_blobs, const LabelScratch &ls);
// The union-find steps of the labelling alone (init + 8-connected merge) into ls.parent: afterwards find_root(frame's
// parent, node) of the first pixel of any run of set bits inside a word (a node) is the component's first pixel in
// raster order.  No count, scan or rank.  The caller has checked the 32-bit limits label_bits enforces.
int union_bits(bv_ctx *ctx, const uint32_t *bits, int batch, int height, int width, const LabelScratch &ls);

#if defined(__CUDACC__)
// ---- device helpers of the union-find (ccl.cu, canny.cu) ----
// `parent` is one frame's array; node ids are pixel indices y * width + x of run starts
__device__ __forceinline__ int find_root(const int *parent, int a) {
    int p = parent[a];
    while (p != a) {
        a = p;
        p = parent[a];
    }
    return a;
}

// first bit of the run of ones containing bit `pos` of w (w has bit pos set)
__device__ __forceinline__ int run_start(uint32_t w, int pos) {
    const uint32_t zeros_below = ~w & ((pos == 0) ? 0u : (0xFFFFFFFFu >> (32 - pos)));
    return zeros_below ? 32 - __clz(zeros_below) : 0;
}

// bits s..e of the run of ones of w that starts at bit s
__device__ __forceinline__ uint32_t run_mask(uint32_t w, int s) {
    const int len = __ffs(~(w >> s)) - 1;  // -1: the run reaches bit 31 (s == 0 and w all ones)
    const int e = (len < 0) ? 31 : s + len - 1;
    return ((e == 31) ? 0xFFFFFFFFu : ((2u << e) - 1u)) & ~((1u << s) - 1u);
}

struct WordPos {
    int wx, y;
    uint32_t row;  // frame * height + y
};

// 32-bit index math throughout the word-indexed kernels (64-bit div/mod costs ~10x; the host
// refuses batches of 2^31 words or more)
__device__ __forceinline__ WordPos word_pos(uint32_t i, int wpr, int height) {
    WordPos p;
    p.wx = (int)(i % (uint32_t)wpr);
    p.row = i / (uint32_t)wpr;
    p.y = (int)(p.row % (uint32_t)height);
    return p;
}

// the n (<= 32) pixels of one bit word as uint8 0/255 at p: two streaming 16-byte stores for a whole, aligned word
__device__ __forceinline__ void store_mask_word(uint8_t *p, int n, uint32_t w) {
    if (n == 32 && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        uint32_t v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t nib = (w >> (4 * k)) & 0xF;
            v[k] = ((nib & 1) * 0xFFu) | (((nib >> 1) & 1) * 0xFF00u) | (((nib >> 2) & 1) * 0xFF0000u) |
                   (((nib >> 3) & 1) * 0xFF000000u);
        }
        st_stream(reinterpret_cast<uint4 *>(p), make_uint4(v[0], v[1], v[2], v[3]));
        st_stream(reinterpret_cast<uint4 *>(p) + 1, make_uint4(v[4], v[5], v[6], v[7]));
    } else {
        for (int k = 0; k < n; ++k) p[k] = ((w >> k) & 1) ? 255 : 0;
    }
}
#endif  // __CUDACC__

}  // namespace bv
