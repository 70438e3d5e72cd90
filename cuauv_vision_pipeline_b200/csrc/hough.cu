// hough.cu -- cv2.HoughLines / cv2.HoughLinesWithAccumulator (the standard transform) on uint8 frames, bit-exact against
// OpenCV 4.13.0 (oracle/hough_np.py restates the rules; include/b200vision.h and DESIGN.md section 2 list them).
//
//   hough_edges_kernel        16 bytes per thread (one 128-bit load where the frame is aligned): the (x, y) of every
//                             non-zero pixel, and its value with use_edgeval, appended to the frame's edge list through
//                             one atomic per block.  The order of the list does not matter: votes are integers.
//   hough_vote_kernel         one block per (slice of angles, chunk of the edge list, frame): whole accumulator rows of
//                             the slice in shared memory, shared-memory atomics for the votes, then every non-zero bin
//                             added to the global accumulator (RED).  Rows past the opt-in shared memory (numrho + 2
//                             above ~58 000) take hough_vote_global_kernel instead, with global atomics.
//   hough_peaks_kernel        one thread per bin: the local-maximum rule, and a unique 64-bit key (votes descending, flat
//                             index ascending) appended to the frame's list (one atomic per warp).
//   hough_sort_kernel         one block per frame: LSD radix sort of the keys over the key bits in use (8 bits a pass,
//                             stable ranks from __match_any_sync), then the first max_lines rows of (rho, theta, votes).
//
// Any sort of unique keys gives cv2's order, and integer votes added in any order give cv2's accumulator, so the result
// depends on no atomic order.  Trig tables are built on the host with libm, as cv2 builds them: CUDA's sin / cos are
// not glibc's.  Frames are independent; a batch whose scratch would pass kGroupBytes goes through in groups of frames.
#include <math.h>

#include <vector>

#include "common.cuh"

namespace bv {

namespace {

constexpr int kEdgeThreads = 256;
constexpr int kVoteThreads = 512;
constexpr int kVoteSmemTarget = 110 * 1024;  // two vote blocks per SM
constexpr int kPeakThreads = 256;
constexpr int kSortThreads = 1024;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kDigits = 256;
constexpr size_t kGroupBytes = size_t(1) << 30;  // accumulators, keys and edge lists of one group of frames

struct HoughGeom {
    int numangle, numrho, rowlen;  // rowlen = numrho + 2
    int shift;                     // (numrho - 1) / 2, C division
    uint32_t bins;                 // (numangle + 2) * rowlen
    uint32_t key_cap;              // peaks a frame can hold: at most every other bin of a row
};

__device__ __forceinline__ int vote_bin(float x, float y, float2 cs, int shift) {
    // cvRound(x * tabCos[n] + y * tabSin[n]): two products and a sum, each rounded to float32 (no FMA), half to even
    return __float2int_rn(__fadd_rn(__fmul_rn(x, cs.x), __fmul_rn(y, cs.y))) + shift;
}

}  // namespace

__global__ void __launch_bounds__(kEdgeThreads) hough_edges_kernel(const uint8_t *__restrict__ src, int width,
                                                                   uint32_t frame_px, uint32_t *__restrict__ edges,
                                                                   uint8_t *__restrict__ vals, int *__restrict__ n_edges) {
    __shared__ int s_warp[kEdgeThreads / 32];
    __shared__ int s_base;
    const int f = blockIdx.y;
    const uint8_t *fsrc = src + (size_t)f * frame_px;
    uint32_t *fedges = edges + (size_t)f * frame_px;
    uint8_t *fvals = vals ? vals + (size_t)f * frame_px : nullptr;
    const bool vec = aligned16(fsrc);
    const uint32_t n_vec = (frame_px + 15) / 16;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t v0 = blockIdx.x * kEdgeThreads; v0 < n_vec; v0 += gridDim.x * kEdgeThreads) {
        const uint32_t v = v0 + threadIdx.x;
        const uint32_t p0 = v * 16;
        uint32_t w[4] = {0, 0, 0, 0};
        if (v < n_vec) {
            if (vec && p0 + 16 <= frame_px) {
                const uint4 q = ld_stream(reinterpret_cast<const uint4 *>(fsrc + p0));
                w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
            } else {
                for (int i = 0; i < 16 && p0 + i < frame_px; ++i) w[i >> 2] |= (uint32_t)fsrc[p0 + i] << (8 * (i & 3));
            }
        }
        uint32_t mask = 0;  // bit i: byte i is non-zero
#pragma unroll
        for (int i = 0; i < 16; ++i) mask |= (uint32_t)(((w[i >> 2] >> (8 * (i & 3))) & 0xFFu) != 0) << i;
        const int cnt = __popc(mask);
        int incl = cnt;  // inclusive warp scan
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (threadIdx.x == 0) {
            int total = 0;
            for (int i = 0; i < kEdgeThreads / 32; ++i) {
                const int c = s_warp[i];
                s_warp[i] = total;
                total += c;
            }
            s_base = total ? atomicAdd(&n_edges[f], total) : 0;
        }
        __syncthreads();
        uint32_t pos = (uint32_t)(s_base + s_warp[warp] + incl - cnt);
        if (mask) {
            uint32_t y = p0 / (uint32_t)width, x = p0 - y * (uint32_t)width;
            for (int i = 0; i < 16; ++i) {
                if ((mask >> i) & 1u) {
                    fedges[pos] = (y << 16) | x;
                    if (fvals) fvals[pos] = (uint8_t)(w[i >> 2] >> (8 * (i & 3)));
                    ++pos;
                }
                if (++x == (uint32_t)width) {
                    x = 0;
                    ++y;
                }
            }
        }
        __syncthreads();  // s_warp and s_base are rewritten by the next round
    }
}

// a vote that falls outside its accumulator row lands where cv2's flat index puts it (a border bin or a neighbouring
// row), through a global atomic; one past the whole accumulator is dropped (cv2 would write out of bounds)
__device__ __forceinline__ void vote_far(int *facc, const HoughGeom &g, int n, int col, int val) {
    const long long flat = (long long)(n + 1) * g.rowlen + col;
    if (flat >= 0 && flat < (long long)g.bins) atomicAdd(&facc[flat], val);
}

__global__ void __launch_bounds__(kVoteThreads) hough_vote_kernel(const uint32_t *__restrict__ edges,
                                                                  const uint8_t *__restrict__ vals,
                                                                  const int *__restrict__ n_edges, uint32_t frame_px,
                                                                  const float2 *__restrict__ tab, HoughGeom g,
                                                                  int rows_per_block, int chunks, int *__restrict__ acc) {
    extern __shared__ int s_acc[];
    const int f = blockIdx.y;
    const int slice = blockIdx.x / chunks, chunk = blockIdx.x - slice * chunks;
    const int n0 = slice * rows_per_block;
    const int nrows = min(rows_per_block, g.numangle - n0);
    const int words = nrows * g.rowlen;
    int *facc = acc + (size_t)f * g.bins;
    for (int i = threadIdx.x; i < words; i += kVoteThreads) s_acc[i] = 0;
    __syncthreads();
    const uint32_t n = (uint32_t)n_edges[f];
    const uint32_t e0 = (uint32_t)((uint64_t)n * chunk / chunks), e1 = (uint32_t)((uint64_t)n * (chunk + 1) / chunks);
    const uint32_t *fedges = edges + (size_t)f * frame_px;
    const uint8_t *fvals = vals ? vals + (size_t)f * frame_px : nullptr;
    for (uint32_t e = e0 + threadIdx.x; e < e1; e += kVoteThreads) {
        const uint32_t xy = fedges[e];
        const float x = (float)(xy & 0xFFFFu), y = (float)(xy >> 16);
        const int val = fvals ? (int)fvals[e] : 1;
        for (int j = 0; j < nrows; ++j) {
            const int col = vote_bin(x, y, __ldg(&tab[n0 + j]), g.shift) + 1;
            if ((unsigned)col < (unsigned)g.rowlen)
                atomicAdd(&s_acc[j * g.rowlen + col], val);
            else
                vote_far(facc, g, n0 + j, col, val);
        }
    }
    __syncthreads();
    int *grows = facc + (size_t)(n0 + 1) * g.rowlen;
    for (int i = threadIdx.x; i < words; i += kVoteThreads) {
        const int v = s_acc[i];
        if (v) atomicAdd(&grows[i], v);  // result unused: RED
    }
}

// rows too wide for shared memory: every (edge, angle) pair votes with a global atomic
__global__ void __launch_bounds__(256) hough_vote_global_kernel(const uint32_t *__restrict__ edges,
                                                                const uint8_t *__restrict__ vals,
                                                                const int *__restrict__ n_edges, uint32_t frame_px,
                                                                const float2 *__restrict__ tab, HoughGeom g,
                                                                int *__restrict__ acc) {
    const int f = blockIdx.y;
    const uint64_t n = (uint64_t)n_edges[f];
    const uint64_t total = n * (uint64_t)g.numangle;
    const uint32_t *fedges = edges + (size_t)f * frame_px;
    const uint8_t *fvals = vals ? vals + (size_t)f * frame_px : nullptr;
    int *facc = acc + (size_t)f * g.bins;
    for (uint64_t i = blockIdx.x * 256ull + threadIdx.x; i < total; i += (uint64_t)gridDim.x * 256) {
        const int a = (int)(i / n);
        const uint32_t e = (uint32_t)(i - (uint64_t)a * n);  // consecutive threads: consecutive edges, one angle
        const uint32_t xy = fedges[e];
        const int val = fvals ? (int)fvals[e] : 1;
        const int col = vote_bin((float)(xy & 0xFFFFu), (float)(xy >> 16), __ldg(&tab[a]), g.shift) + 1;
        if ((unsigned)col < (unsigned)g.rowlen)
            atomicAdd(&facc[(size_t)(a + 1) * g.rowlen + col], val);
        else
            vote_far(facc, g, a, col, val);
    }
}

__global__ void __launch_bounds__(kPeakThreads) hough_peaks_kernel(const int *__restrict__ acc, HoughGeom g, int threshold,
                                                                   uint64_t *__restrict__ keys, int *__restrict__ n_peaks) {
    const int f = blockIdx.y;
    const int *facc = acc + (size_t)f * g.bins;
    const uint32_t interior = (uint32_t)g.numangle * (uint32_t)g.numrho;
    const int lane = threadIdx.x & 31;
    for (uint32_t i0 = blockIdx.x * kPeakThreads; i0 < interior; i0 += gridDim.x * kPeakThreads) {
        const uint32_t i = i0 + threadIdx.x;
        bool peak = false;
        int v = 0;
        uint32_t base = 0;
        if (i < interior) {
            const uint32_t n = i / (uint32_t)g.numrho, r = i - n * (uint32_t)g.numrho;
            base = (n + 1) * (uint32_t)g.rowlen + r + 1;
            v = facc[base];
            peak = v > threshold && v > facc[base - 1] && v >= facc[base + 1] && v > facc[base - g.rowlen] &&
                   v >= facc[base + g.rowlen];
        }
        const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, peak);
        if (!ballot) continue;
        int slot = 0;
        if (lane == __ffs(ballot) - 1) slot = atomicAdd(&n_peaks[f], __popc(ballot));
        slot = __shfl_sync(0xFFFFFFFFu, slot, __ffs(ballot) - 1);
        if (peak) {
            // votes descending, then flat index ascending: one ascending sort of unique keys gives cv2's order
            const uint32_t hi = 0x7FFFFFFFu - (uint32_t)v;
            keys[(size_t)f * g.key_cap + slot + __popc(ballot & ((1u << lane) - 1))] = ((uint64_t)hi << 32) | base;
        }
    }
}

__global__ void __launch_bounds__(kSortThreads) hough_sort_kernel(uint64_t *__restrict__ keys_a, uint64_t *__restrict__ keys_b,
                                                                  const int *__restrict__ n_peaks, HoughGeom g,
                                                                  int idx_bits, float rho, float theta, float min_theta,
                                                                  float *__restrict__ lines, int max_lines,
                                                                  int *__restrict__ n_lines) {
    __shared__ int s_wc[kSortWarps][kDigits];  // per tile: count, then exclusive prefix, of every digit in every warp
    __shared__ int s_base[kDigits];            // where each digit's next key goes
    __shared__ uint32_t s_lo[kSortWarps], s_hi[kSortWarps];
    const int f = blockIdx.x;
    const int n = n_peaks[f];
    if (threadIdx.x == 0) n_lines[f] = n;
    if (n == 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t *src = keys_a + (size_t)f * g.key_cap, *dst = keys_b + (size_t)f * g.key_cap;

    // the vote part of the keys spans [lo, hi]: only the bits of hi - lo and of the flat index are sorted on
    uint32_t lo = 0xFFFFFFFFu, hi = 0;
    for (int i = threadIdx.x; i < n; i += kSortThreads) {
        const uint32_t h = (uint32_t)(src[i] >> 32);
        lo = min(lo, h);
        hi = max(hi, h);
    }
    for (int d = 16; d; d >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, d));
        hi = max(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, d));
    }
    if (lane == 0) {
        s_lo[warp] = lo;
        s_hi[warp] = hi;
    }
    __syncthreads();
    lo = s_lo[0];
    hi = s_hi[0];
    for (int w = 1; w < kSortWarps; ++w) {
        lo = min(lo, s_lo[w]);
        hi = max(hi, s_hi[w]);
    }
    const int bits = idx_bits + (hi == lo ? 0 : 32 - __clz(hi - lo));
    auto sortable = [&](uint64_t k) { return ((uint64_t)((uint32_t)(k >> 32) - lo) << idx_bits) | (uint32_t)k; };

    for (int shift = 0; n > 1 && shift < bits; shift += 8) {
        if (threadIdx.x < kDigits) s_base[threadIdx.x] = 0;
        for (int i = threadIdx.x; i < kSortWarps * kDigits; i += kSortThreads) (&s_wc[0][0])[i] = 0;
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += kSortThreads) atomicAdd(&s_base[(sortable(src[i]) >> shift) & 255], 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            int run = 0;
            for (int d = 0; d < kDigits; ++d) {
                const int c = s_base[d];
                s_base[d] = run;
                run += c;
            }
        }
        __syncthreads();
        for (int t0 = 0; t0 < n; t0 += kSortThreads) {
            const int i = t0 + threadIdx.x;
            const bool valid = i < n;
            const uint64_t k = valid ? src[i] : 0;
            const int d = valid ? (int)((sortable(k) >> shift) & 255) : kDigits;  // the invalid tail is one group
            const uint32_t peers = __match_any_sync(0xFFFFFFFFu, d);
            const int rank = __popc(peers & ((1u << lane) - 1));
            if (valid && rank == 0) s_wc[warp][d] = __popc(peers);
            __syncthreads();
            int tile_count = 0;
            if (threadIdx.x < kDigits) {  // exclusive prefix over the warps, in warp order: the ranks stay stable
                for (int w = 0; w < kSortWarps; ++w) {
                    const int c = s_wc[w][threadIdx.x];
                    s_wc[w][threadIdx.x] = tile_count;
                    tile_count += c;
                }
            }
            __syncthreads();
            if (valid) dst[s_base[d] + s_wc[warp][d] + rank] = k;
            __syncthreads();
            if (threadIdx.x < kDigits) s_base[threadIdx.x] += tile_count;
            for (int j = threadIdx.x; j < kSortWarps * kDigits; j += kSortThreads) (&s_wc[0][0])[j] = 0;
            __syncthreads();
        }
        uint64_t *t = src;
        src = dst;
        dst = t;
    }

    const int m = min(n, max_lines);
    float *flines = lines + (size_t)f * max_lines * 3;
    for (int i = threadIdx.x; i < m; i += kSortThreads) {
        const uint64_t k = src[i];
        const int base = (int)(uint32_t)k;
        const int votes = (int)(0x7FFFFFFFu - (uint32_t)(k >> 32));
        const int a = base / g.rowlen - 1;
        const int r = base - (a + 1) * g.rowlen - 1;
        flines[3 * i + 0] = __fmul_rn((float)(r - g.shift), rho);
        flines[3 * i + 1] = __fadd_rn(min_theta, __fmul_rn((float)a, theta));
        flines[3 * i + 2] = (float)votes;
    }
}

static bool disjoint(const void *a, size_t na, const void *b, size_t nb) {
    const uintptr_t pa = (uintptr_t)a, pb = (uintptr_t)b;
    return !a || !b || na == 0 || nb == 0 || pa + na <= pb || pb + nb <= pa;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_hough_lines(bv_ctx *ctx, const uint8_t *src_dev, int batch, int height, int width, double rho,
                              double theta, int threshold, double min_theta, double max_theta, int use_edgeval,
                              float *lines_dev, int max_lines, int32_t *n_lines_dev) {
    BV_REQUIRE(ctx && src_dev && n_lines_dev && (lines_dev || max_lines == 0), "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(max_lines >= 0, "max_lines must not be negative");
    BV_REQUIRE(height <= 65535 && width <= 65535, "height and width must be below 65536");
    const size_t frame_px = (size_t)height * width;
    BV_REQUIRE(frame_px < (1ull << 31), "frame too large for 32-bit indices");
    BV_REQUIRE(!use_edgeval || 255.0 * (double)frame_px <= 2147483647.0,
               "use_edgeval: 255 * height * width votes would overflow int32");
    const float rho_f = (float)rho, theta_f = (float)theta;
    BV_REQUIRE(rho_f > 0 && theta_f > 0 && isfinite(rho_f) && isfinite(theta_f), "rho and theta must be positive and finite");
    BV_REQUIRE(isfinite(min_theta) && isfinite(max_theta), "min_theta and max_theta must be finite");
    BV_REQUIRE(min_theta <= max_theta, "min_theta must not exceed max_theta");
    const size_t src_bytes = (size_t)batch * frame_px, lines_bytes = (size_t)batch * max_lines * 3 * sizeof(float),
                 counts_bytes = (size_t)batch * sizeof(int32_t);
    BV_REQUIRE(disjoint(src_dev, src_bytes, lines_dev, lines_bytes) && disjoint(src_dev, src_bytes, n_lines_dev, counts_bytes) &&
                   disjoint(lines_dev, lines_bytes, n_lines_dev, counts_bytes),
               "src, lines and n_lines overlap");

    // rules 1-3: angle and rho counts as HoughLinesStandard sizes its accumulator
    const double na = floor((max_theta - min_theta) / (double)theta_f) + 1;
    BV_REQUIRE(na < 1e9, "too many angles for 32-bit indices");
    int numangle = (int)na;
    if (numangle > 1 && fabs(M_PI - (numangle - 1) * (double)theta_f) < (double)theta_f / 2) --numangle;
    const int numrho = (int)lrintf((float)(2 * (height + width) + 1) / rho_f);
    HoughGeom g;
    g.numangle = numangle;
    g.numrho = numrho;
    g.rowlen = numrho + 2;
    g.shift = (numrho - 1) / 2;
    const double bins = (double)(numangle + 2) * (double)(numrho + 2);
    BV_REQUIRE(bins < 2147483648.0, "accumulator too large for 32-bit indices");
    g.bins = (uint32_t)bins;
    g.key_cap = (uint32_t)numangle * (uint32_t)((numrho + 1) / 2);
    BV_CUDA(cudaSetDevice(ctx->device));

    // rule 4: the trig table, from the host's libm
    std::vector<float2> tab(numangle);
    const float irho = 1.0f / rho_f;
    float ang = (float)min_theta;
    for (int n = 0; n < numangle; ++n, ang += theta_f) {
        tab[n].x = (float)(cos((double)ang) * irho);
        tab[n].y = (float)(sin((double)ang) * irho);
    }

    const size_t per_frame = (size_t)g.bins * 4 + (size_t)g.key_cap * 16 + frame_px * (use_edgeval ? 5 : 4);
    int group = (int)(kGroupBytes / per_frame);
    group = group < 1 ? 1 : group > batch ? batch : group > 65535 ? 65535 : group;
    BV_TRY(ensure_scratch(ctx, SCR_HOUGH_TAB, (size_t)numangle * sizeof(float2) + 2 * (size_t)group * sizeof(int)));
    BV_TRY(ensure_scratch(ctx, SCR_HOUGH_ACC, (size_t)group * g.bins * 4));
    BV_TRY(ensure_scratch(ctx, SCR_HOUGH_KEYS, (size_t)group * g.key_cap * 16 + 16));
    BV_TRY(ensure_scratch(ctx, SCR_HOUGH_EDGES, (size_t)group * frame_px * (use_edgeval ? 5 : 4)));
    float2 *d_tab = (float2 *)ctx->scratch[SCR_HOUGH_TAB];
    int *n_edges = (int *)(d_tab + numangle), *n_peaks = n_edges + group;
    int *acc = (int *)ctx->scratch[SCR_HOUGH_ACC];
    uint64_t *keys_a = (uint64_t *)ctx->scratch[SCR_HOUGH_KEYS], *keys_b = keys_a + (size_t)group * g.key_cap;
    uint32_t *edges = (uint32_t *)ctx->scratch[SCR_HOUGH_EDGES];
    uint8_t *vals = use_edgeval ? (uint8_t *)(edges + (size_t)group * frame_px) : nullptr;
    BV_CUDA(cudaMemcpyAsync(d_tab, tab.data(), (size_t)numangle * sizeof(float2), cudaMemcpyHostToDevice, ctx->stream));

    // rows of the vote kernel: as many whole rows as fit two blocks an SM, or one row up to the opt-in limit
    int optin = 0;
    BV_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    const size_t row_bytes = (size_t)g.rowlen * 4;
    const bool smem_path = row_bytes <= (size_t)optin;
    int rows = (int)(kVoteSmemTarget / row_bytes);
    rows = rows < 1 ? 1 : rows > numangle ? numangle : rows;
    const int slices = (numangle + rows - 1) / rows;
    const size_t smem = (size_t)rows * row_bytes;
    if (smem_path && smem > 48 * 1024)
        BV_CUDA(cudaFuncSetAttribute(hough_vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int idx_bits = 32 - __builtin_clz(g.bins - 1);
    const uint32_t n_vec = (uint32_t)((frame_px + 15) / 16);

    for (int f0 = 0; f0 < batch; f0 += group) {
        const int gb = batch - f0 < group ? batch - f0 : group;
        BV_CUDA(cudaMemsetAsync(n_edges, 0, 2 * (size_t)group * sizeof(int), ctx->stream));
        BV_CUDA(cudaMemsetAsync(acc, 0, (size_t)gb * g.bins * 4, ctx->stream));
        const int ge = grid_for(ctx, (size_t)n_vec * gb, kEdgeThreads, 8);
        BV_LAUNCH(ctx, hough_edges_kernel, dim3((ge + gb - 1) / gb, gb), kEdgeThreads, 0, src_dev + (size_t)f0 * frame_px,
                  width, (uint32_t)frame_px, edges, vals, n_edges);
        if (smem_path) {
            // enough chunks of the edge list that every SM holds two blocks twice over
            const int want = ctx->sm_count * 4;
            int chunks = (want + slices * gb - 1) / (slices * gb);
            chunks = chunks > 64 ? 64 : chunks;
            BV_LAUNCH(ctx, hough_vote_kernel, dim3(slices * chunks, gb), kVoteThreads, smem, edges, vals, n_edges,
                      (uint32_t)frame_px, d_tab, g, rows, chunks, acc);
        } else {
            BV_LAUNCH(ctx, hough_vote_global_kernel, dim3((ctx->sm_count * 8 + gb - 1) / gb, gb), 256, 0, edges, vals,
                      n_edges, (uint32_t)frame_px, d_tab, g, acc);
        }
        if (g.key_cap) {
            const int gp = grid_for(ctx, (size_t)numangle * numrho * gb, kPeakThreads, 8);
            BV_LAUNCH(ctx, hough_peaks_kernel, dim3((gp + gb - 1) / gb, gb), kPeakThreads, 0, acc, g, threshold, keys_a,
                      n_peaks);
        }
        BV_LAUNCH(ctx, hough_sort_kernel, gb, kSortThreads, 0, keys_a, keys_b, n_peaks, g, idx_bits, rho_f, theta_f,
                  (float)min_theta, lines_dev + (size_t)f0 * max_lines * 3, max_lines, n_lines_dev + f0);
    }
    return BV_OK;
}
