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

}  // namespace bv
