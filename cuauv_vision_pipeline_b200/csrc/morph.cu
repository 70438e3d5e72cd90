// morph.cu -- flat-structuring-element morphology.  Replaces cv2.erode / cv2.dilate /
// cv2.morphologyEx at utils/transform.py:80-164, modules/bins.py:24, modules/red_buoy.py:33-34
// and modules/preprocessor.py:120-129.
//
// Semantics (cv2, verified in SURVEY.md A.5): erode = min over the SE support with out-of-image
// taps ignored (+inf border), dilate = max over the same taps dst(x,y) = max src(x+i-ax, y+j-ay)
// (cv2 4.13.0 does not mirror the SE: probed with even and asymmetric kernels) with out-of-image
// taps ignored (0 border); anchor = centre (kw/2, kh/2); OPEN/CLOSE/GRADIENT with `iterations=n` apply n
// erosions then n dilations (resp. the reverse, resp. the difference).
//
// Two implementations:
//   * binary masks, bit-packed 32 px per word: a 5x5 erosion is 4 funnel-shift/AND pairs per row
//     and an AND across 5 rows per 32 pixels; the whole mask of a 2208x1242 frame is 343 KB and
//     lives in L2.  Used by the fused stage (stage.cu).
//   * grey / multi-channel uint8 with an arbitrary SE given as horizontal runs (bv_morph).
#include <mutex>
#include <unordered_map>

#include "morph.cuh"

namespace bv {

// ----------------------------------------------------------------------------------------------
// uint8 mask <-> bits
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_to_bits_kernel(const uint8_t *__restrict__ mask, uint32_t *__restrict__ bits,
                                                           int height, int width, int wpr, uint32_t total_words) {
    const uint32_t stride = gridDim.x * blockDim.x;  // 32-bit index math: 64-bit div/mod costs ~10x
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const int wx = (int)(i % (uint32_t)wpr);
        const uint32_t row = i / (uint32_t)wpr;  // frame * height + y
        const uint8_t *p = mask + (size_t)row * width + (size_t)wx * 32;
        const int n = min(32, width - wx * 32);
        uint32_t w = 0;
        if (n == 32 && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p));
            const uint4 b = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
            const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int k = 0; k < 32; ++k)
                if (BV_GETB(v, k)) w |= 1u << k;
        } else {
            for (int k = 0; k < n; ++k)
                if (p[k]) w |= 1u << k;
        }
        bits[i] = w;
    }
}

__global__ void __launch_bounds__(256) bits_to_mask_kernel(const uint32_t *__restrict__ bits, uint8_t *__restrict__ mask,
                                                           int height, int width, int wpr, uint32_t total_words) {
    const uint32_t stride = gridDim.x * blockDim.x;  // 32-bit index math: 64-bit div/mod costs ~10x
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const int wx = (int)(i % (uint32_t)wpr);
        const uint32_t row = i / (uint32_t)wpr;
        store_mask_word(mask + (size_t)row * width + (size_t)wx * 32, min(32, width - wx * 32), bits[i]);
    }
}

static int check_words(size_t total) {
    if (total >= (1ull << 31)) {
        set_error("bit-packed batch too large (%zu words): split the batch", total);
        return BV_ERR_INVALID;
    }
    return BV_OK;
}

int mask_to_bits(bv_ctx *ctx, const uint8_t *mask, uint32_t *bits, int batch, int height, int width) {
    const int wpr = words_per_row(width);
    const size_t total = (size_t)batch * height * wpr;
    BV_TRY(check_words(total));
    BV_LAUNCH(ctx, mask_to_bits_kernel, grid_for(ctx, total, 256, 8), 256, 0, mask, bits, height, width, wpr, (uint32_t)total);
    return BV_OK;
}

int bits_to_mask(bv_ctx *ctx, const uint32_t *bits, uint8_t *mask, int batch, int height, int width) {
    const int wpr = words_per_row(width);
    const size_t total = (size_t)batch * height * wpr;
    BV_LAUNCH(ctx, bits_to_mask_kernel, grid_for(ctx, total, 256, 8), 256, 0, bits, mask, height, width, wpr, (uint32_t)total);
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// binary erode / dilate with a rectangle: taps x-L..x+R, y-U..y+D (each <= 31)
// ----------------------------------------------------------------------------------------------
template <bool ERODE>
__global__ void __launch_bounds__(256) morph_bits_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst,
                                                         int height, int width, int wpr, uint32_t total_words, int L, int R,
                                                         int U, int D) {
    const uint32_t stride = gridDim.x * blockDim.x;  // 32-bit index math: 64-bit div/mod costs ~10x
    const uint32_t neutral = ERODE ? 0xFFFFFFFFu : 0u;
    const int last = wpr - 1;
    const int tail = width - last * 32;  // valid bits in the last word of a row
    const uint32_t tail_mask = tail == 32 ? 0xFFFFFFFFu : ((1u << tail) - 1u);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const int wx = (int)(i % (uint32_t)wpr);
        const uint32_t row = i / (uint32_t)wpr;
        const int y = (int)(row % (uint32_t)height);
        const uint32_t *frame_row0 = src + (size_t)(row - y) * wpr;
        uint32_t acc = neutral;
        for (int yy = max(0, y - U); yy <= min(height - 1, y + D); ++yy) {
            const uint32_t *r = frame_row0 + (size_t)yy * wpr;
            uint32_t c = r[wx];
            uint32_t l = wx > 0 ? r[wx - 1] : neutral;
            uint32_t n = wx < last ? r[wx + 1] : neutral;
            if (ERODE) {  // pixels beyond the right image edge count as set
                if (wx == last) c |= ~tail_mask;
                if (wx + 1 == last) n |= ~tail_mask;
            }
            uint32_t h = c;
            for (int d = 1; d <= L; ++d) {  // tap x-d
                const uint32_t s = __funnelshift_l(l, c, d);
                h = ERODE ? (h & s) : (h | s);
            }
            for (int d = 1; d <= R; ++d) {  // tap x+d
                const uint32_t s = __funnelshift_r(c, n, d);
                h = ERODE ? (h & s) : (h | s);
            }
            acc = ERODE ? (acc & h) : (acc | h);
        }
        if (wx == last) acc &= tail_mask;
        dst[i] = acc;
    }
}

__global__ void __launch_bounds__(256) bits_andnot_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                                                          uint32_t *__restrict__ dst, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = a[i] & ~b[i];
}

// one erosion or dilation src -> dst (src != dst), extents already multiplied by the iteration count
static int morph_bits_basic(bv_ctx *ctx, const uint32_t *src, uint32_t *dst, uint32_t *tmp, int batch, int height,
                            int width, bool erode, int L, int R, int U, int D) {
    const int wpr = words_per_row(width);
    const size_t total = (size_t)batch * height * wpr;
    const int grid = grid_for(ctx, total, 256, 8);
    // extents above 31 are applied in several passes (erosions / dilations by rectangles compose);
    // pass k of P writes dst when (P - k) is even, tmp otherwise, so the last pass lands in dst.
    const int mx = max(max(L, R), max(U, D));
    const int passes = mx <= 31 ? 1 : (mx + 30) / 31;
    if (passes > 1 && !tmp) {
        set_error("binary morphology: structuring element too large for a single pass");
        return BV_ERR_UNSUPPORTED;
    }
    const uint32_t *cur = src;
    for (int k = 1; k <= passes; ++k) {
        const int l = L > 31 ? 31 : L, r = R > 31 ? 31 : R, u = U > 31 ? 31 : U, d = D > 31 ? 31 : D;
        L -= l; R -= r; U -= u; D -= d;
        uint32_t *out = ((passes - k) % 2 == 0) ? dst : tmp;
        if (erode)
            BV_LAUNCH(ctx, morph_bits_kernel<true>, grid, 256, 0, cur, out, height, width, wpr, (uint32_t)total, l, r, u, d);
        else
            BV_LAUNCH(ctx, morph_bits_kernel<false>, grid, 256, 0, cur, out, height, width, wpr, (uint32_t)total, l, r, u, d);
        cur = out;
    }
    return BV_OK;
}

// taps of a kw x kh rectangle applied `iterations` times, x-L .. x+R and y-U .. y+D, computed in 64 bits and clipped to the
// frame: a tap that lies a whole width or height away from every pixel never reads the image, so the clip changes nothing
static void rect_extents(int kw, int kh, int iterations, int height, int width, int &L, int &R, int &U, int &D) {
    const long long ax = kw / 2, ay = kh / 2, n = iterations;
    L = (int)min(ax * n, (long long)width - 1);
    R = (int)min((kw - 1 - ax) * n, (long long)width - 1);
    U = (int)min(ay * n, (long long)height - 1);
    D = (int)min((kh - 1 - ay) * n, (long long)height - 1);
}

int morph_bits_rect(bv_ctx *ctx, uint32_t *bits, uint32_t *tmp, uint32_t *tmp2, uint32_t *tmp3, int batch, int height,
                    int width, int op, int kw, int kh, int iterations) {
    const size_t total = (size_t)batch * height * words_per_row(width);
    // zero iterations or the identity element: dilate == erode == input, so the gradient is empty (cv2 4.13.0)
    if (iterations < 1 || (kw == 1 && kh == 1)) {
        if (op == BV_MORPH_GRADIENT) BV_CUDA(cudaMemsetAsync(bits, 0, total * 4, ctx->stream));
        return BV_OK;
    }
    // taps: x-L .. x+R, y-U .. y+D for erosion and dilation alike (cv2 does not mirror the element: probed, 4.13.0)
    int L, R, U, D;
    rect_extents(kw, kh, iterations, height, width, L, R, U, D);
    switch (op) {
        case BV_MORPH_ERODE:
            BV_TRY(morph_bits_basic(ctx, bits, tmp, tmp2, batch, height, width, true, L, R, U, D));
            BV_CUDA(cudaMemcpyAsync(bits, tmp, total * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            return BV_OK;
        case BV_MORPH_DILATE:
            BV_TRY(morph_bits_basic(ctx, bits, tmp, tmp2, batch, height, width, false, L, R, U, D));
            BV_CUDA(cudaMemcpyAsync(bits, tmp, total * 4, cudaMemcpyDeviceToDevice, ctx->stream));
            return BV_OK;
        case BV_MORPH_OPEN:
            BV_TRY(morph_bits_basic(ctx, bits, tmp, tmp2, batch, height, width, true, L, R, U, D));
            return morph_bits_basic(ctx, tmp, bits, tmp2, batch, height, width, false, L, R, U, D);
        case BV_MORPH_CLOSE:
            BV_TRY(morph_bits_basic(ctx, bits, tmp, tmp2, batch, height, width, false, L, R, U, D));
            return morph_bits_basic(ctx, tmp, bits, tmp2, batch, height, width, true, L, R, U, D);
        case BV_MORPH_GRADIENT:
            // bits (input), tmp (dilated), tmp2 (eroded); tmp3 is the ping-pong image of either basic's passes
            BV_TRY(morph_bits_basic(ctx, bits, tmp, tmp3, batch, height, width, false, L, R, U, D));
            BV_TRY(morph_bits_basic(ctx, bits, tmp2, tmp3, batch, height, width, true, L, R, U, D));
            BV_LAUNCH(ctx, bits_andnot_kernel, grid_for(ctx, total, 256, 8), 256, 0, tmp, tmp2, bits, total);
            return BV_OK;
        default: set_error("unknown morphology op %d", op); return BV_ERR_INVALID;
    }
}

// ----------------------------------------------------------------------------------------------
// A whole chain of binary erosions / dilations (OPEN = erode, dilate; CLOSE = dilate, erode; ...)
// in ONE launch: a block stages a tile of 32 output rows plus the halo rows the chain needs in
// shared memory (bits: a 2208-px row is 276 bytes; 32 warps, one row each per round), runs every step there as a horizontal pass
// (funnel shifts) and a vertical pass, and writes the final bits and/or the uint8 0/255 mask.
// Replaces one launch per elementary step plus the bits -> bytes expansion, each of which went
// through L2 with 15 dependent loads per word.
// ----------------------------------------------------------------------------------------------
constexpr int kChainMaxOps = 8;
constexpr int kChainThreads = 1024;  // 32 warps, one shared-memory row each per round
struct MorphChain {
    int n;
    int halo_up, halo_down;  // sum of the vertical extents
    struct {
        int erode, L, R, U, D;
    } op[kChainMaxOps];
};

// horizontal erosion / dilation of one word by taps x-L .. x+R (L, R <= 31); the common small
// symmetric extents are fully unrolled
template <bool ERODE>
__device__ __forceinline__ uint32_t hpass_word(uint32_t l, uint32_t c, uint32_t n, int L, int R) {
    uint32_t h = c;
#define BV_TAP_L(d) { const uint32_t s_ = __funnelshift_l(l, c, (d)); h = ERODE ? (h & s_) : (h | s_); }
#define BV_TAP_R(d) { const uint32_t s_ = __funnelshift_r(c, n, (d)); h = ERODE ? (h & s_) : (h | s_); }
    if (L == R && L <= 3) {
        if (L >= 1) { BV_TAP_L(1) BV_TAP_R(1) }
        if (L >= 2) { BV_TAP_L(2) BV_TAP_R(2) }
        if (L >= 3) { BV_TAP_L(3) BV_TAP_R(3) }
    } else {
        for (int d = 1; d <= L; ++d) BV_TAP_L(d)
        for (int d = 1; d <= R; ++d) BV_TAP_R(d)
    }
#undef BV_TAP_L
#undef BV_TAP_R
    return h;
}

// 4 mask bits -> 4 bytes of 0x00 / 0xFF
__device__ __forceinline__ uint32_t nibble_to_bytes(uint32_t nib) { return ((nib * 0x00204081u) & 0x01010101u) * 0xFFu; }

template <bool ERODE>
__device__ __forceinline__ void chain_step(uint32_t *A, uint32_t *B, int rows, int wpr, int ybase, int height, int L, int R,
                                           int U, int D, uint32_t tail_mask) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int last = wpr - 1;
    const uint32_t neutral = ERODE ? 0xFFFFFFFFu : 0u;
    // horizontal pass A -> B (taps x-L .. x+R)
    for (int r = warp; r < rows; r += nwarps) {
        const uint32_t *a = A + r * wpr;
        for (int wx = lane; wx < wpr; wx += 32) {
            uint32_t c = a[wx];
            const uint32_t l = wx > 0 ? a[wx - 1] : neutral;
            uint32_t n = wx < last ? a[wx + 1] : neutral;
            if (ERODE) {  // pixels beyond the right image edge count as set
                if (wx == last) c |= ~tail_mask;
                if (wx + 1 == last) n |= ~tail_mask;
            }
            B[r * wpr + wx] = hpass_word<ERODE>(l, c, n, L, R);
        }
    }
    __syncthreads();
    // vertical pass B -> A (rows y-U .. y+D; rows outside the image are ignored)
    for (int r = warp; r < rows; r += nwarps) {
        const int y = ybase + r;
        if (y < 0 || y >= height) continue;
        // rows the tile does not hold only feed halo rows that are discarded before the output
        const int r0 = max(max(0, y - U) - ybase, 0), r1 = min(min(height - 1, y + D) - ybase, rows - 1);
        for (int wx = lane; wx < wpr; wx += 32) {
            uint32_t acc = neutral;
            for (int rr = r0; rr <= r1; ++rr) {
                const uint32_t v = B[rr * wpr + wx];
                acc = ERODE ? (acc & v) : (acc | v);
            }
            if (wx == last) acc &= tail_mask;
            A[r * wpr + wx] = acc;
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kChainThreads) morph_chain_kernel(const uint32_t *__restrict__ src,
                                                                    uint32_t *__restrict__ dst_bits, uint8_t *__restrict__ mask,
                                                                    int height, int width, int wpr, int tiles_per_frame,
                                                                    int tile_rows, MorphChain ch) {
    extern __shared__ uint32_t chain_smem[];
    const int frame = blockIdx.x / tiles_per_frame, tile = blockIdx.x - frame * tiles_per_frame;
    const int rows = tile_rows + ch.halo_up + ch.halo_down;
    const int ybase = tile * tile_rows - ch.halo_up;  // image row of shared-memory row 0
    uint32_t *A = chain_smem, *B = chain_smem + rows * wpr;
    const uint32_t *fsrc = src + (size_t)frame * height * wpr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int r = warp; r < rows; r += nwarps) {
        const int y = ybase + r;
        const bool inside = y >= 0 && y < height;
        for (int wx = lane; wx < wpr; wx += 32) A[r * wpr + wx] = inside ? __ldg(fsrc + (size_t)y * wpr + wx) : 0u;
    }
    __syncthreads();
    const int last = wpr - 1;
    const int tail = width - last * 32;
    const uint32_t tail_mask = tail == 32 ? 0xFFFFFFFFu : ((1u << tail) - 1u);
    for (int k = 0; k < ch.n; ++k) {
        if (ch.op[k].erode)
            chain_step<true>(A, B, rows, wpr, ybase, height, ch.op[k].L, ch.op[k].R, ch.op[k].U, ch.op[k].D, tail_mask);
        else
            chain_step<false>(A, B, rows, wpr, ybase, height, ch.op[k].L, ch.op[k].R, ch.op[k].U, ch.op[k].D, tail_mask);
    }
    // output rows
    const int y_first = tile * tile_rows;
    const int n_rows = min(tile_rows, height - y_first);
    const bool wide_ok = (width % 16 == 0) && ((reinterpret_cast<uintptr_t>(mask) & 15) == 0);
    for (int r = warp; r < n_rows; r += nwarps) {
        const size_t row = (size_t)frame * height + y_first + r;
        for (int wx = lane; wx < wpr; wx += 32) {
            const uint32_t w = A[(r + ch.halo_up) * wpr + wx];
            if (dst_bits) dst_bits[row * wpr + wx] = w;
            if (mask) {
                uint8_t *p = mask + row * width + (size_t)wx * 32;
                const int n = min(32, width - wx * 32);
                if (n == 32 && wide_ok) {
                    uint32_t v[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) v[q] = nibble_to_bytes((w >> (4 * q)) & 0xFu);
                    st_stream(reinterpret_cast<uint4 *>(p), make_uint4(v[0], v[1], v[2], v[3]));
                    st_stream(reinterpret_cast<uint4 *>(p) + 1, make_uint4(v[4], v[5], v[6], v[7]));
                } else {
                    for (int q = 0; q < n; ++q) p[q] = ((w >> q) & 1) ? 255 : 0;
                }
            }
        }
    }
}

// ----------------------------------------------------------------------------------------------
// The same chain without shared memory or block barriers, for the shapes the modules use (square 3x3 / 5x5 elements,
// 1, 2 or 4 elementary steps: ERODE / DILATE / OPEN / CLOSE / OPEN+CLOSE, rows of at most 128 words = 4096 px).
// One WARP walks down a strip of rows; lane l keeps words l, l+32, l+64, l+96 of the current row in registers, gets
// the neighbouring words for the horizontal taps by shuffle, and every step keeps its last 2R horizontally processed
// rows in a register ring for the vertical taps -- a software pipeline in which step s emits row y - (s+1) R when row y
// comes in.  A strip re-reads 2 N R rows of halo above and below; strips are cut so that every SM gets ~8 warps.
// (The tile kernel above spends its time in 4 N block-wide barriers per 24 output rows with 1024-thread blocks, 5 active
// lanes in the third column round of a 69-word row, and 1.4 blocks per SM: 19 us per 4-frame launch at 2208x1242; this
// form: see profiles/r02_morph_variants.log.)
// ----------------------------------------------------------------------------------------------
template <int R, bool ERODE>
__device__ __forceinline__ uint32_t hpass_sq(uint32_t l, uint32_t c, uint32_t n) {
    uint32_t h = c;
#pragma unroll
    for (int d = 1; d <= R; ++d) {
        const uint32_t a = __funnelshift_l(l, c, d), b = __funnelshift_r(c, n, d);
        h = ERODE ? (h & a & b) : (h | a | b);
    }
    return h;
}

template <int R, int N, int K>
__global__ void __launch_bounds__(256) morph_roll_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst_bits,
                                                         uint8_t *__restrict__ mask, int batch, int height, int width, int wpr,
                                                         int strips, int strip_rows, uint32_t erode_bits) {
    const int lane = threadIdx.x & 31;
    const int job = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (job >= batch * strips) return;
    const int frame = job / strips, strip = job - frame * strips;
    const int y0 = strip * strip_rows, y1 = min(height, y0 + strip_rows);
    const uint32_t *fsrc = src + (size_t)frame * height * wpr;
    const int last = wpr - 1;
    const int tail = width - last * 32;
    const uint32_t tail_mask = tail == 32 ? 0xFFFFFFFFu : ((1u << tail) - 1u);
    const bool wide_ok = (width % 16 == 0) && ((reinterpret_cast<uintptr_t>(mask) & 15) == 0);
    uint32_t ring[N][2 * R][K];
#pragma unroll
    for (int s = 0; s < N; ++s)
#pragma unroll
        for (int j = 0; j < 2 * R; ++j)
#pragma unroll
            for (int k = 0; k < K; ++k) ring[s][j][k] = 0u;
    const int prev_lane = (lane + 31) & 31, next_lane = (lane + 1) & 31;
    // the next row's words are requested before the current row goes through the chain
    uint32_t nxt[K];
    const int y_begin = y0 - N * R, y_end = y1 + N * R;
    auto load_row = [&](int y, uint32_t (&v)[K]) {
        const bool inside = y >= 0 && y < height;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int wi = 32 * k + lane;
            v[k] = (inside && wi < wpr) ? __ldg(fsrc + (size_t)y * wpr + wi) : 0u;
        }
    };
    load_row(y_begin, nxt);
    for (int y = y_begin; y < y_end; ++y) {
        uint32_t cur[K];
#pragma unroll
        for (int k = 0; k < K; ++k) cur[k] = nxt[k];
        if (y + 1 < y_end) load_row(y + 1, nxt);
#pragma unroll
        for (int s = 0; s < N; ++s) {
            const bool erode = (erode_bits >> s) & 1u;
            const uint32_t neutral = erode ? 0xFFFFFFFFu : 0u;
            const int row = y - s * R;                         // index of the row `cur` holds for this step
            const bool inside = row >= 0 && row < height;      // rows outside the image do not take part in this step
            uint32_t v[K], rl[K], rr[K], h[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int wi = 32 * k + lane;
                v[k] = (inside && wi < wpr) ? cur[k] : neutral;
                if (erode && wi == last) v[k] |= ~tail_mask;   // pixels beyond the right edge count as set
                rl[k] = __shfl_sync(0xFFFFFFFFu, v[k], prev_lane);
                rr[k] = __shfl_sync(0xFFFFFFFFu, v[k], next_lane);
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint32_t l = lane == 0 ? (k > 0 ? rl[k > 0 ? k - 1 : 0] : neutral) : rl[k];
                const uint32_t n = lane == 31 ? (k < K - 1 ? rr[k < K - 1 ? k + 1 : k] : neutral) : rr[k];
                h[k] = erode ? hpass_sq<R, true>(l, v[k], n) : hpass_sq<R, false>(l, v[k], n);
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                uint32_t acc = h[k];
#pragma unroll
                for (int j = 0; j < 2 * R; ++j) acc = erode ? (acc & ring[s][j][k]) : (acc | ring[s][j][k]);
#pragma unroll
                for (int j = 0; j + 1 < 2 * R; ++j) ring[s][j][k] = ring[s][j + 1][k];
                ring[s][2 * R - 1][k] = h[k];
                cur[k] = (32 * k + lane == last) ? (acc & tail_mask) : acc;   // row `row - R` of this step's output
            }
        }
        const int o = y - N * R;
        if (o < y0 || o >= y1) continue;
        const size_t out_row = (size_t)frame * height + o;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int wi = 32 * k + lane;
            if (wi >= wpr) continue;
            const uint32_t w = cur[k];
            if (dst_bits) dst_bits[out_row * wpr + wi] = w;
            if (mask) {
                uint8_t *p = mask + out_row * width + (size_t)wi * 32;
                const int n = min(32, width - wi * 32);
                if (n == 32 && wide_ok) {
                    uint32_t q[8];
#pragma unroll
                    for (int t = 0; t < 8; ++t) q[t] = nibble_to_bytes((w >> (4 * t)) & 0xFu);
                    st_stream(reinterpret_cast<uint4 *>(p), make_uint4(q[0], q[1], q[2], q[3]));
                    st_stream(reinterpret_cast<uint4 *>(p) + 1, make_uint4(q[4], q[5], q[6], q[7]));
                } else {
                    for (int t = 0; t < n; ++t) p[t] = ((w >> t) & 1) ? 255 : 0;
                }
            }
        }
    }
}

template <int R, int N>
static int launch_roll(bv_ctx *ctx, const uint32_t *bits, uint32_t *dst_bits, uint8_t *mask, int batch, int height, int width,
                       int wpr, uint32_t erode_bits) {
    // warps per SM (BV_OPT_MORPH_WARPS, default 8), at least 4 output rows per strip (the halo of 2 N R rows is re-read
    // and re-computed by every strip: fewer, taller strips do less work but offer less parallelism)
    const int wps = ctx->opt[BV_OPT_MORPH_WARPS] > 0 ? ctx->opt[BV_OPT_MORPH_WARPS] : 8;
    int strips = (ctx->sm_count * wps + batch - 1) / batch;
    if (strips > (height + 3) / 4) strips = (height + 3) / 4;
    if (strips < 1) strips = 1;
    const int strip_rows = (height + strips - 1) / strips;
    strips = (height + strip_rows - 1) / strip_rows;
    const int jobs = batch * strips, grid = (jobs + 7) / 8;
    const int k = (wpr + 31) / 32;
#define BV_ROLL(KK) BV_LAUNCH(ctx, (morph_roll_kernel<R, N, KK>), grid, 256, 0, bits, dst_bits, mask, batch, height, width, wpr, strips, strip_rows, erode_bits)
    if (k == 1) BV_ROLL(1); else if (k == 2) BV_ROLL(2); else if (k == 3) BV_ROLL(3); else BV_ROLL(4);
#undef BV_ROLL
    return BV_OK;
}

// All steps as one chain, if they fit (erode / dilate / open / close with rectangles, horizontal
// extents <= 31 per elementary step, shared memory for tile + halos).  *done = false: use the
// step-by-step path.
int morph_bits_chain(bv_ctx *ctx, const uint32_t *bits, uint32_t *dst_bits, uint8_t *mask, int batch, int height, int width,
                     int n_steps, const int *ops, const int *kws, const int *khs, const int *iters, bool *done) {
    *done = false;
    MorphChain ch;
    memset(&ch, 0, sizeof(ch));
    for (int s = 0; s < n_steps; ++s) {
        if (ops[s] == BV_MORPH_GRADIENT) return BV_OK;   // three images: the step-by-step path (also at 0 iterations)
        if (iters[s] < 1 || (kws[s] == 1 && khs[s] == 1)) continue;  // identity
        const long long ax = kws[s] / 2, ay = khs[s] / 2, it = iters[s];
        if (ax * it > 31 || (kws[s] - 1 - ax) * it > 31) return BV_OK;
        const int L = (int)(ax * it), R = (int)((kws[s] - 1 - ax) * it);
        if (ay * it > 256 || (khs[s] - 1 - ay) * it > 256) return BV_OK;   // more than the 256 rows a tile may have
        const int U = (int)(ay * it), D = (int)((khs[s] - 1 - ay) * it);
        const int first_erode = (ops[s] == BV_MORPH_ERODE || ops[s] == BV_MORPH_OPEN) ? 1 : 0;
        const int n_el = (ops[s] == BV_MORPH_OPEN || ops[s] == BV_MORPH_CLOSE) ? 2 : 1;
        for (int e = 0; e < n_el; ++e) {
            if (ch.n == kChainMaxOps) return BV_OK;
            ch.op[ch.n].erode = e == 0 ? first_erode : !first_erode;
            ch.op[ch.n].L = L; ch.op[ch.n].R = R; ch.op[ch.n].U = U; ch.op[ch.n].D = D;
            // output row y of step k reads rows y-U .. y+D of step k-1
            ch.halo_up += U;
            ch.halo_down += D;
            ++ch.n;
        }
    }
    const int wpr = words_per_row(width);
    // register-rolling form: every step a square element of the same radius 1 or 2, 1 / 2 / 4 steps, rows <= 128 words
    if (ch.n >= 1 && wpr <= 128 && ctx->opt[BV_OPT_MORPH_VARIANT] == 0) {
        const int r = ch.op[0].L;
        bool square = r >= 1 && r <= 2;
        uint32_t erode_bits = 0;
        for (int i = 0; i < ch.n; ++i) {
            square = square && ch.op[i].L == r && ch.op[i].R == r && ch.op[i].U == r && ch.op[i].D == r;
            if (ch.op[i].erode) erode_bits |= 1u << i;
        }
        if (square && (ch.n == 1 || ch.n == 2 || ch.n == 4)) {
            int st;
            if (r == 1)
                st = ch.n == 1 ? launch_roll<1, 1>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits)
                   : ch.n == 2 ? launch_roll<1, 2>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits)
                               : launch_roll<1, 4>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits);
            else
                st = ch.n == 1 ? launch_roll<2, 1>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits)
                   : ch.n == 2 ? launch_roll<2, 2>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits)
                               : launch_roll<2, 4>(ctx, bits, dst_bits, mask, batch, height, width, wpr, erode_bits);
            BV_TRY(st);
            *done = true;
            return BV_OK;
        }
    }
    // shared-memory rows = a multiple of the 32 warps: 32 rows while the halo leaves at least half of
    // them as output rows, more otherwise
    const int halo = ch.halo_up + ch.halo_down;
    int rows = 32;
    while (rows - halo < rows / 2) rows += 32;
    const int tile_rows = rows - halo;
    const size_t smem = (size_t)2 * rows * wpr * sizeof(uint32_t);
    if (rows > 256 || smem > 200 * 1024) return BV_OK;
    if (smem > 48 * 1024) {
        // the opt-in is an attribute of the kernel on the device, shared by every context of the process: it is only ever
        // raised, so that a context's smaller launch cannot take away what another context's larger one relies on
        static std::mutex mu;
        static std::unordered_map<int, int> enabled;   // device -> bytes
        std::lock_guard<std::mutex> lock(mu);
        int &cur = enabled[ctx->device];
        if ((int)smem > cur) {
            BV_CUDA(cudaFuncSetAttribute(morph_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            cur = (int)smem;
        }
    }
    const int tiles = (height + tile_rows - 1) / tile_rows;
    BV_LAUNCH(ctx, morph_chain_kernel, batch * tiles, kChainThreads, smem, bits, dst_bits, mask, height, width, wpr, tiles,
              tile_rows, ch);
    *done = true;
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// grey morphology, arbitrary SE as horizontal runs
// ----------------------------------------------------------------------------------------------
constexpr int kMaxRuns = 256;
struct RunList {
    int n;
    short dy[kMaxRuns];
    int x0[kMaxRuns], x1[kMaxRuns];  // taps (x + x0 .. x + x1, y + dy); a rectangle's row run spans up to the frame width
};

template <bool ERODE>
__global__ void __launch_bounds__(256) morph_grey_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst,
                                                         int height, int width, int cn, size_t total, RunList runs) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t row_bytes = (size_t)width * cn;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const size_t row = i / row_bytes;  // frame * height + y
        const int xb = (int)(i - row * row_bytes);
        const int x = xb / cn, c = xb - x * cn;
        const int y = (int)(row % height);
        const uint8_t *frame = src + (row - y) * row_bytes;
        int v = ERODE ? 255 : 0;
        for (int r = 0; r < runs.n; ++r) {
            const int yy = y + runs.dy[r];
            if (yy < 0 || yy >= height) continue;
            const int xa = max(0, x + runs.x0[r]), xe = min(width - 1, x + runs.x1[r]);
            const uint8_t *p = frame + (size_t)yy * row_bytes + c;
            for (int xx = xa; xx <= xe; ++xx) {
                const int s = p[(size_t)xx * cn];
                v = ERODE ? min(v, s) : max(v, s);
            }
        }
        dst[i] = (uint8_t)v;
    }
}

__global__ void __launch_bounds__(256) sub_u8_kernel(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b,
                                                     uint8_t *__restrict__ dst, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = (int)a[i] - (int)b[i];
        dst[i] = (uint8_t)(d < 0 ? 0 : d);
    }
}

static int launch_grey(bv_ctx *ctx, const uint8_t *src, uint8_t *dst, int height, int width, int cn, size_t total,
                       bool erode, const RunList &runs) {
    const int grid = grid_for(ctx, total, 256, 8);
    if (erode)
        BV_LAUNCH(ctx, morph_grey_kernel<true>, grid, 256, 0, src, dst, height, width, cn, total, runs);
    else
        BV_LAUNCH(ctx, morph_grey_kernel<false>, grid, 256, 0, src, dst, height, width, cn, total, runs);
    return BV_OK;
}

struct SeInfo {
    bool rect;            // full rectangle: separable, iterations fold into the extents
    RunList erode_runs;   // taps for erosion
    RunList dilate_runs;  // taps for dilation (identical: cv2 does not mirror the SE)
    int kw, kh;
};

static int build_se(const uint8_t *se, int kw, int kh, SeInfo &info) {
    info.kw = kw;
    info.kh = kh;
    info.rect = true;
    for (int i = 0; i < kw * kh; ++i)
        if (!se[i]) info.rect = false;
    const int ax = kw / 2, ay = kh / 2;
    info.erode_runs.n = info.dilate_runs.n = 0;
    for (int j = 0; j < kh; ++j) {
        int i = 0;
        while (i < kw) {
            if (!se[j * kw + i]) {
                ++i;
                continue;
            }
            int e = i;
            while (e + 1 < kw && se[j * kw + e + 1]) ++e;
            if (info.erode_runs.n >= kMaxRuns) {
                set_error("bv_morph: structuring element has more than %d horizontal runs", kMaxRuns);
                return BV_ERR_UNSUPPORTED;
            }
            RunList &er = info.erode_runs;
            er.dy[er.n] = (short)(j - ay);
            er.x0[er.n] = (short)(i - ax);
            er.x1[er.n] = (short)(e - ax);
            er.n++;
            RunList &dr = info.dilate_runs;
            dr.dy[dr.n] = (short)(j - ay);
            dr.x0[dr.n] = (short)(i - ax);
            dr.x1[dr.n] = (short)(e - ax);
            dr.n++;
            i = e + 1;
        }
    }
    return BV_OK;
}

// n erosions (or dilations) src -> dst; src != dst; t1, t2 scratch images
static int grey_basic(bv_ctx *ctx, const uint8_t *src, uint8_t *dst, uint8_t *t1, uint8_t *t2, int batch, int height,
                      int width, int cn, bool erode, const SeInfo &se, int iterations) {
    const size_t total = (size_t)batch * height * width * cn;
    if (se.kw == 1 && se.kh == 1 && se.rect) {
        BV_CUDA(cudaMemcpyAsync(dst, src, total, cudaMemcpyDeviceToDevice, ctx->stream));
        return BV_OK;
    }
    if (se.rect) {
        // separable, and n iterations of a rectangle == one rectangle with n-fold extents, clipped to the frame
        int L, R, U, D;
        rect_extents(se.kw, se.kh, iterations, height, width, L, R, U, D);
        RunList h, v;
        h.n = 1;
        h.dy[0] = 0;
        h.x0[0] = -L;
        h.x1[0] = R;
        BV_TRY(launch_grey(ctx, src, t1, height, width, cn, total, erode, h));
        // the column taps y-U .. y+D in passes of at most kMaxRuns rows (U + D = sum of the passes' u + d): with out-of-image
        // taps ignored, erosions (dilations) by segments that contain their anchor compose into one by the summed segment.
        // Pass k of P writes dst when (P - k) is even, t2 otherwise, so the last pass lands in dst.
        const int passes = U + D == 0 ? 1 : (U + D + kMaxRuns - 2) / (kMaxRuns - 1);
        const uint8_t *cur = t1;
        for (int k = 1; k <= passes; ++k) {
            const int u = min(U, kMaxRuns - 1), d = min(D, kMaxRuns - 1 - u);
            U -= u;
            D -= d;
            v.n = u + d + 1;
            for (int j = 0; j < v.n; ++j) {
                v.dy[j] = (short)(j - u);
                v.x0[j] = v.x1[j] = 0;
            }
            uint8_t *out = ((passes - k) % 2 == 0) ? dst : t2;
            BV_TRY(launch_grey(ctx, cur, out, height, width, cn, total, erode, v));
            cur = out;
        }
        return BV_OK;
    }
    const RunList &runs = erode ? se.erode_runs : se.dilate_runs;
    const uint8_t *cur = src;
    for (int it = 0; it < iterations; ++it) {
        uint8_t *out = (it == iterations - 1) ? dst : (cur == t1 ? t2 : t1);
        BV_TRY(launch_grey(ctx, cur, out, height, width, cn, total, erode, runs));
        cur = out;
    }
    return BV_OK;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_morph(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                        int channels, int op, const uint8_t *se_host, int kw, int kh, int iterations) {
    BV_REQUIRE(ctx && src_dev && dst_dev && se_host, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(channels >= 1 && channels <= 4, "channels must be 1..4");
    BV_REQUIRE(kw >= 1 && kh >= 1 && kw <= 255 && kh <= 255, "structuring element size must be 1..255");
    BV_REQUIRE(op >= BV_MORPH_ERODE && op <= BV_MORPH_GRADIENT, "unknown morphology op");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t total = (size_t)batch * height * width * channels;
    if (iterations < 0) iterations = 1;   // cv2 reads a negative count as 1 (probed, 4.13.0)
    if (iterations == 0) {                 // cv2: the source unchanged, and for GRADIENT (dilate - erode of nothing) zeros
        if (op == BV_MORPH_GRADIENT)
            BV_CUDA(cudaMemsetAsync(dst_dev, 0, total, ctx->stream));
        else if (src_dev != dst_dev)
            BV_CUDA(cudaMemcpyAsync(dst_dev, src_dev, total, cudaMemcpyDeviceToDevice, ctx->stream));
        return BV_OK;
    }
    static thread_local SeInfo se;
    BV_TRY(build_se(se_host, kw, kh, se));
    BV_REQUIRE(se.erode_runs.n > 0, "structuring element is empty");
    BV_TRY(ensure_scratch(ctx, SCR_MORPH_TMP, total * 3));
    uint8_t *t0 = (uint8_t *)ctx->scratch[SCR_MORPH_TMP];
    uint8_t *t1 = t0 + total, *t2 = t1 + total;
    BV_TRY(ensure_scratch(ctx, SCR_MORPH_TMP2, total * 2));
    uint8_t *u0 = (uint8_t *)ctx->scratch[SCR_MORPH_TMP2];
    uint8_t *u1 = u0 + total;
    switch (op) {
        case BV_MORPH_ERODE:
        case BV_MORPH_DILATE: {
            const bool er = op == BV_MORPH_ERODE;
            if (src_dev == dst_dev) {
                BV_TRY(grey_basic(ctx, src_dev, t0, t1, t2, batch, height, width, channels, er, se, iterations));
                BV_CUDA(cudaMemcpyAsync(dst_dev, t0, total, cudaMemcpyDeviceToDevice, ctx->stream));
                return BV_OK;
            }
            return grey_basic(ctx, src_dev, dst_dev, t1, t2, batch, height, width, channels, er, se, iterations);
        }
        case BV_MORPH_OPEN:
        case BV_MORPH_CLOSE: {
            const bool first_erode = op == BV_MORPH_OPEN;
            BV_TRY(grey_basic(ctx, src_dev, t0, t1, t2, batch, height, width, channels, first_erode, se, iterations));
            return grey_basic(ctx, t0, dst_dev, t1, t2, batch, height, width, channels, !first_erode, se, iterations);
        }
        default: {  // gradient
            BV_TRY(grey_basic(ctx, src_dev, u0, t1, t2, batch, height, width, channels, false, se, iterations));
            BV_TRY(grey_basic(ctx, src_dev, u1, t1, t2, batch, height, width, channels, true, se, iterations));
            BV_LAUNCH(ctx, sub_u8_kernel, grid_for(ctx, total, 256, 8), 256, 0, u0, u1, dst_dev, total);
            return BV_OK;
        }
    }
}
