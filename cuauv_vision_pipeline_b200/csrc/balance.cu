// balance.cu -- underwater colour balance on the device.  Replaces the reference's process_frame
// (utils/color_correction/color_balance.cpp:343-780) for every flag combination except the HSI
// branch (702-774); tilings (horizontal/vertical_blocks > 1) must divide the frame.
//
// The reference makes ~14 full passes over split planes on the CPU.  Here the whole algorithm is
// three streaming passes over the interleaved frame; the per-frame statistics run inside the last
// block of passes 1 and 2 ("last block done" ticket), so a frame costs three launches:
//
//   pass 1  hist_bgr    256-bin histograms of B, G, R                      (reads 3 B/px)
//   stats1  (last block of pass 1) percentile bounds (112-142), exact clipped means from the histogram (426-428),
//           dominant channel + gains in double (480-544), optional RGB contrast stretch
//           (546-645) -> ONE composed 256-entry table per channel
//   pass 2  hist_sv     table -> BGR2HSV -> histograms of S and V          (re-reads 3 B/px, L2)
//                       and keeps H,S,V (3 B/px) in an L2-resident scratch image
//   stats2  (last block of pass 2) S/V percentile bounds (671-681) -> stretch tables (683-686)
//   pass 3  final       H,S,V scratch -> S/V tables -> HSV2BGR -> [convert -> inRange]
//                       writes balanced BGR and/or converted image and/or mask
//           or mask_from_hsv (HSV inRange mask only): H,S,V scratch -> S/V tables -> one look-up
//                       in a 128 KB shared-memory table of hue intervals (see "hue-interval table")
//
// Because clipping, equalisation and the contrast stretch are all per-channel point operations
// that depend only on global statistics, they collapse into look-up tables computed once per frame;
// the exact integer channel sums come out of the histogram, so no extra reduction pass is needed.
// Frames are processed in chunks sized to stay L2-resident so that passes 2 and 3 do not touch HBM.
#include <stdlib.h>

#include "balance.cuh"
#include "convert.cuh"

namespace bv {

int hsi_run(bv_ctx *ctx, uint8_t *bgr, int batch, size_t npx);  // hsi.cu

constexpr int kBalThreads = 256;
constexpr int kBalWarps = kBalThreads / 32;

// constrain(val, 0, 255) of color_balance.cpp:13-23: clamp in double, truncate.  NaN (0 * inf when
// a channel mean is 0) is undefined behaviour in the reference; defined here as 0.
__device__ __forceinline__ int constrain255(double v) {
    if (v < 0.0) return 0;
    if (v > 255.0) return 255;
    if (v != v) return 0;
    return (int)v;
}

// `(unsigned char)double` as the compiled reference does it on x86-64 (truncate to int, keep the
// low byte); out-of-range input is undefined behaviour in the reference (634-640).
__device__ __forceinline__ int uchar_cast(double v) {
    if (v != v || v >= 2147483648.0 || v <= -2147483649.0) return 0;
    return ((int)v) & 0xFF;
}

// ----------------------------------------------------------------------------------------------
// Block-wide (256 threads) statistics of one finished 256-bin histogram; thread t owns bin t.
//   lo = first bin i with  sum_{j<=i} cnt[j] > low_bound     (percentile_min_max, 128-136)
//   hi = last  bin i with  sum_{j>=i} cnt[j] > high_bound    (137-145)
// which is exactly what the reference's subtract-as-you-go loops compute; with both bounds 0 they
// are the first / last non-empty bins (cv::minMaxLoc, 421-423).  Also the exact sum of the clipped
// channel, sum_i clamp(i, lo, hi) * cnt[i]  (the numerator of cv::mean, 426-428).
// ----------------------------------------------------------------------------------------------
// The statistics helpers below are run by the first 256 threads (8 whole warps) of a block, thread t owning bin t; they
// synchronise on named barrier 1 so that blocks of more than 256 threads can call them too.
__device__ __forceinline__ void stat_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

struct StatScratch {
    unsigned long long warp_sum[3][kBalWarps];
    uint32_t warp_cnt[3][kBalWarps];
    uint32_t cnt_lo[3][kBalWarps], cnt_hi[3][kBalWarps];
};

// N histograms at once (thread t owns bin t of each): the block-wide steps -- and their barriers --
// are shared by the channels, which keeps this tail of the histogram kernels short (one block works
// here while the rest of the machine waits for the tables).
template <int N>
__device__ void hist_stats_block(const uint32_t (&c)[N], size_t npx, long long low_bound, long long high_bound, StatScratch &sc,
                                 int (&lo)[N], int (&hi)[N], unsigned long long (&clipped_sum)[N]) {
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    uint32_t incl[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        incl[k] = c[k];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl[k], d);
            if (lane >= d) incl[k] += o;
        }
    }
    stat_sync();  // protects sc from the previous call
    if (lane == 31)
#pragma unroll
        for (int k = 0; k < N; ++k) sc.warp_cnt[k][wid] = incl[k];
    stat_sync();
#pragma unroll
    for (int k = 0; k < N; ++k) {
        uint32_t before = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w)
            if (w < wid) before += sc.warp_cnt[k][w];
        const long long prefix = (long long)before + incl[k];          // inclusive prefix sum
        const long long suffix = (long long)npx - prefix + c[k];        // inclusive suffix sum
        const uint32_t wl = __popc(__ballot_sync(0xFFFFFFFFu, prefix <= low_bound));
        const uint32_t wh = __popc(__ballot_sync(0xFFFFFFFFu, suffix > high_bound));
        if (lane == 0) {
            sc.cnt_lo[k][wid] = wl;
            sc.cnt_hi[k][wid] = wh;
        }
    }
    stat_sync();
    unsigned long long v[N];
#pragma unroll
    for (int k = 0; k < N; ++k) {
        int l = 0, h = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w) {
            l += (int)sc.cnt_lo[k][w];
            h += (int)sc.cnt_hi[k][w];
        }
        h -= 1;
        if (l > 255) l = 255;
        if (h < 0) h = 0;
        lo[k] = l;
        hi[k] = h;
        const int cl = t < l ? l : (t > h ? h : t);
        v[k] = (unsigned long long)cl * c[k];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v[k] += __shfl_down_sync(0xFFFFFFFFu, v[k], d);
        if (lane == 0) sc.warp_sum[k][wid] = v[k];
    }
    stat_sync();
#pragma unroll
    for (int k = 0; k < N; ++k) {
        unsigned long long tot = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w) tot += sc.warp_sum[k][w];
        clipped_sum[k] = tot;
    }
}

// float32 products truncated to int, exactly as color_balance.cpp:113-114
__device__ __forceinline__ void percentile_limits(size_t n, long long &low_bound, long long &high_bound) {
    low_bound = (int)__fmul_rn(0.002f, (float)n);
    high_bound = (int)(n - (size_t)(int)__fmul_rn(0.998f, (float)n));
}

// exact sum of a channel clipped to [lo, hi], from its histogram; thread t owns bin t
__device__ unsigned long long block_clipped_sum(uint32_t c, int lo, int hi, StatScratch &sc) {
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    const int cl = t < lo ? lo : (t > hi ? hi : t);
    unsigned long long v = (unsigned long long)cl * c;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, d);
    stat_sync();
    if (lane == 0) sc.warp_sum[0][wid] = v;
    stat_sync();
    unsigned long long tot = 0;
#pragma unroll
    for (int w = 0; w < kBalWarps; ++w) tot += sc.warp_sum[0][w];
    return tot;
}

// Run by the LAST block of a frame's pass 1: bounds, exact means, gains, composed tables -- one
// table set per tile (a single "tile" = the frame itself in the default 1x1 configuration).
__device__ void stats_bgr_block(BalFrame &F, size_t npx, const bv_balance_params &prm,
                                const double *__restrict__ pow_quarter, StatScratch &sc, BalTile *tiles, int n_tiles,
                                size_t tile_px) {
    __shared__ int s_lo[3], s_hi[3], s_dom;
    __shared__ double s_avg[3], s_local[3], s_gain[3], s_ratio[3];
    const int t = threadIdx.x;
    long long lb = 0, hb = 0;
    if (prm.rgb_extrema_clipping) percentile_limits(npx, lb, hb);
    {
        // written by other blocks' atomics: read at L2; the three loads are in flight together
        const uint32_t cnt[3] = {__ldcg(&F.hist_bgr[0][t]), __ldcg(&F.hist_bgr[1][t]), __ldcg(&F.hist_bgr[2][t])};
        int lo[3], hi[3];
        unsigned long long sum[3];
        hist_stats_block<3>(cnt, npx, lb, hb, sc, lo, hi, sum);
        if (t == 0)
            for (int c = 0; c < 3; ++c) {
                s_lo[c] = lo[c];
                s_hi[c] = hi[c];
                s_avg[c] = (double)sum[c] / (double)npx;
                s_local[c] = s_avg[c];  // a single tile is the frame itself: same histogram, same clipped sum
            }
    }
    stat_sync();
    if (t == 0) {
        const double b = s_avg[0], g = s_avg[1], r = s_avg[2];
        for (int c = 0; c < 3; ++c) {
            F.stats.bgr_min[c] = s_lo[c];
            F.stats.bgr_max[c] = s_hi[c];
            F.stats.bgr_avg[c] = s_avg[c];
        }
        F.stats.s_min = F.stats.v_min = 0;
        F.stats.s_max = F.stats.v_max = 255;
        F.stats.degenerate = 0;
        if (prm.rgb_contrast_correct) {
            // 560-627: order channels by the (pre-equalisation) means
            int mx, md, mn;
            if (r > g) {
                if (r > b) { mx = 2; if (g > b) { md = 1; mn = 0; } else { md = 0; mn = 1; } }
                else { mx = 0; md = 2; mn = 1; }
            } else {
                if (g > b) { mx = 1; if (r > b) { md = 2; mn = 0; } else { md = 0; mn = 2; } }
                else { mx = 0; md = 1; mn = 2; }
            }
            const double desired_max = (double)((s_hi[mn] + s_hi[md] + s_hi[mx]) / 3);   // 629: int division
            s_ratio[mn] = (desired_max - s_lo[mn]) / (double)(s_hi[mn] - s_lo[mn]);
            s_ratio[md] = (desired_max - 0.0) / (double)(s_hi[md] - s_lo[md]);
            s_ratio[mx] = ((double)s_hi[mx] - 0.0) / (double)(s_hi[mx] - s_lo[mx]);
        }
    }
    stat_sync();
    for (int tile = 0; tile < n_tiles; ++tile) {
        const uint32_t(*hist)[256] = tiles ? tiles[tile].hist : F.hist_bgr;
        uint8_t(*lut)[256] = tiles ? tiles[tile].lut : F.lut_bgr;
        if (tiles) {
            for (int c = 0; c < 3; ++c) {
                // local mean of the clipped tile (459-470; exact sum instead of the running mean)
                const unsigned long long sum = block_clipped_sum(__ldcg(&hist[c][t]), s_lo[c], s_hi[c], sc);
                if (t == 0) s_local[c] = (double)sum / (double)tile_px;
            }
        }
        stat_sync();
        if (t == 0) {
            double lb_ = s_local[0], lg_ = s_local[1], lr_ = s_local[2];
            // 474: unqualified abs() == int abs(int) in the compiled reference: the difference is
            // truncated toward zero first (see oracle/color_balance_np.py)
            if (abs((int)(lr_ - s_avg[2])) > s_avg[2] / 6 || abs((int)(lb_ - s_avg[0])) > s_avg[0] / 6 ||
                abs((int)(lg_ - s_avg[1])) > s_avg[1] / 6) {
                lb_ = s_avg[0];
                lg_ = s_avg[1];
                lr_ = s_avg[2];
            }
            int dom;
            // 480 / 501 / 522: red if strictly largest, else green if strictly largest, else blue
            if (lr_ > lg_ && lr_ > lb_) dom = 2;
            else if (lg_ > lr_ && lg_ > lb_) dom = 1;
            else dom = 0;
            const double loc[3] = {lb_, lg_, lr_};
            for (int c = 0; c < 3; ++c) s_gain[c] = (c == dom) ? 1.0 : loc[dom] / loc[c];
            s_dom = dom;
            if (tile == 0) F.stats.dominant = dom;
        }
        stat_sync();
        // every thread builds entry t of the three composed tables
        for (int c = 0; c < 3; ++c) {
            int x = t < s_lo[c] ? s_lo[c] : (t > s_hi[c] ? s_hi[c] : t);                 // clip_channel, 25-45
            if (prm.equalize_rgb && c != s_dom) {
                const double xd = (double)x;
                if (prm.adaptive_cast_correction)                                        // 489-491
                    x = constrain255(xd * (pow_quarter[x] * (s_gain[c] - 1.) + 1.));
                else                                                                     // 494-495
                    x = constrain255(xd * s_gain[c]);
            }
            if (prm.rgb_contrast_correct) x = uchar_cast((double)(x - s_lo[c]) * s_ratio[c]);  // 634-640
            lut[c][t] = (uint8_t)x;
        }
        stat_sync();
    }
}

// Run by the LAST block of a frame's pass 2: S/V percentile bounds and stretch tables (671-686).
__device__ void stats_sv_block(BalFrame &F, size_t npx, StatScratch &sc) {
    __shared__ int lo[2], hi[2];
    const int t = threadIdx.x;
    long long lb, hb;
    percentile_limits(npx, lb, hb);
    {
        const uint32_t cnt[2] = {__ldcg(&F.hist_sv[0][t]), __ldcg(&F.hist_sv[1][t])};
        int l[2], h[2];
        unsigned long long sum[2];
        hist_stats_block<2>(cnt, npx, lb, hb, sc, l, h, sum);
        if (t == 0)
            for (int c = 0; c < 2; ++c) {
                lo[c] = l[c];
                hi[c] = h[c];
            }
    }
    stat_sync();
    if (t == 0) {
        F.stats.s_min = lo[0];
        F.stats.s_max = hi[0];
        F.stats.v_min = lo[1];
        F.stats.v_max = hi[1];
        F.stats.degenerate = (lo[0] == hi[0] || lo[1] == hi[1]) ? 1 : 0;
    }
    for (int c = 0; c < 2; ++c) {
        const int x = t < lo[c] ? lo[c] : (t > hi[c] ? hi[c] : t);
        // int32, C division.  The reference divides by zero (SIGFPE) when hi == lo; defined as 0 here.
        const int d = hi[c] - lo[c];
        F.lut_sv[c][t] = (uint8_t)(d ? ((x - lo[c]) * 255) / d : 0);
    }
}

// "last block done": every block of a frame calls this after merging its histogram into HBM; the
// block that draws the final ticket sees all merges (fence + atomic) and does the statistics.
__device__ __forceinline__ bool last_block_of_frame(uint32_t *ticket, unsigned blocks_per_frame) {
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == blocks_per_frame - 1);
    __syncthreads();
    return is_last;
}

// ----------------------------------------------------------------------------------------------
// pass 1: BGR histograms.  One private 3x256 histogram per warp in shared memory, merged into
// the frame's histogram in HBM with one atomic per non-empty bin per block; the last block of a
// frame then computes the statistics and tables (no separate launch).
// ----------------------------------------------------------------------------------------------
// Shared-memory layout: 4 KB per warp (three 1 KB histograms + 1 KB unused), so that a counter's byte offset is
// (warp << 12) | (channel << 10) | (value << 2): the warp part is ORed into the mask that isolates the value (one LOP3) and the
// channel part is an immediate of the ATOMS, i.e. shift + and-or + ATOMS per sample instead of shift + and + add + ATOMS.
constexpr int kHistWarpWords = 1024;
template <bool VEC>
__global__ void __launch_bounds__(kBalThreads) hist_bgr_kernel(const uint8_t *__restrict__ src, BalFrame *__restrict__ st,
                                                               size_t npx, bv_balance_params prm,
                                                               const double *__restrict__ pow_quarter) {
    __shared__ uint32_t h[kBalWarps][kHistWarpWords];
    __shared__ StatScratch sc;
    for (int i = threadIdx.x; i < kBalWarps * kHistWarpWords; i += blockDim.x) (&h[0][0])[i] = 0;
    __syncthreads();
    const int frame = blockIdx.y;
    const uint8_t *f = src + (size_t)frame * npx * 3;
    unsigned char *hbytes = reinterpret_cast<unsigned char *>(&h[0][0]);
    const uint32_t woff = (threadIdx.x >> 5) << 12;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t ngroups = VEC ? npx / 16 : 0;
    // the next group's 48 bytes are requested before the current group's 48 atomics are issued, so
    // HBM latency overlaps the shared-memory atomics of the same warp
    size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    Px16 in, nxt;
    if (g < ngroups) load_px16<true>(f, g, in);
    for (; g < ngroups; g += stride) {
        if (g + stride < ngroups) load_px16<true>(f, g + stride, nxt);
#pragma unroll
        for (int k = 0; k < 48; ++k) {
            const uint32_t w = in.w[k >> 2];
            const int sh = 8 * (k & 3) - 2;   // value << 2, straight from its place in the word
            const uint32_t off = ((sh < 0 ? w << 2 : w >> sh) & 0x3FCu) | woff;
            atomicAdd(reinterpret_cast<uint32_t *>(hbytes + off + (k % 3) * 1024), 1u);
        }
        in = nxt;
    }
    uint32_t *hw = h[threadIdx.x >> 5];
    for (size_t p = ngroups * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        atomicAdd(&hw[f[3 * p]], 1u);
        atomicAdd(&hw[256 + f[3 * p + 1]], 1u);
        atomicAdd(&hw[512 + f[3 * p + 2]], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 768; i += blockDim.x) {
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w) s += h[w][i];
        if (s) atomicAdd(&st[frame].hist_bgr[0][0] + i, s);
    }
    if (last_block_of_frame(&st[frame].ticket[0], gridDim.x)) stats_bgr_block(st[frame], npx, prm, pow_quarter, sc, nullptr, 1, npx);
}

// insert the 24-bit packed pixel J (0..15) into the 12-word output buffer
template <int J>
__device__ __forceinline__ void put_px(uint32_t (&w)[12], uint32_t p) {
    constexpr int o = 3 * J, wi = o >> 2, sh = 8 * (o & 3);
    w[wi] |= p << sh;
    if constexpr (sh > 8) w[wi + 1] |= p >> (32 - sh);
}

// The three bytes of pixel J (clean values 0..255) go into the 48-byte output group: bytes are staged four at a time and a
// word is assembled with three byte-permutes when its last byte arrives (2.25 instructions per pixel; shifting and
// OR-ing the packed pixel into one or two words takes about four).
template <int Q>
__device__ __forceinline__ void put_byte(uint32_t (&w)[12], uint32_t (&st)[4], uint32_t v) {
    st[Q & 3] = v;
    if constexpr ((Q & 3) == 3)
        w[Q >> 2] = __byte_perm(__byte_perm(st[0], st[1], 0x1140u), __byte_perm(st[2], st[3], 0x1140u), 0x5410u);
}
template <int J>
__device__ __forceinline__ void put_px3(uint32_t (&w)[12], uint32_t (&st)[4], uint32_t c0, uint32_t c1, uint32_t c2) {
    put_byte<3 * J>(w, st, c0);
    put_byte<3 * J + 1>(w, st, c1);
    put_byte<3 * J + 2>(w, st, c2);
}

// pixels J..15 of a 16-pixel group of pass 2: tables -> BGR2HSV -> S and V counted, H,S,V packed
template <int J>
__device__ __forceinline__ void hsv_group(const Px16 &in, const uint8_t (*lut)[256], uint32_t (*hw)[256], Px16 &o,
                                          uint32_t (&stg)[4]) {
    if constexpr (J < 16) {
        int hh, ss, vv;
        bgr2hsv_rcp(lut[0][BV_GETB(in.w, 3 * J)], lut[1][BV_GETB(in.w, 3 * J + 1)], lut[2][BV_GETB(in.w, 3 * J + 2)], hh, ss, vv);
        atomicAdd(&hw[0][ss], 1u);
        atomicAdd(&hw[1][vv], 1u);
        put_px3<J>(o.w, stg, (uint32_t)hh, (uint32_t)ss, (uint32_t)vv);
        hsv_group<J + 1>(in, lut, hw, o, stg);
    }
}

// The H,S,V scratch lives for one pass: written by pass 2, read once by pass 3.  After a warp has consumed the 32 x 48
// bytes = 12 whole 128-byte lines of its 32 consecutive groups, lanes 0..11 tell L2 to drop those (still dirty) lines
// instead of writing them back to HBM (discard.global.L2; the bytes are indeterminate afterwards, and the next call's
// pass 2 rewrites them before anything reads them).  Requires the frame stride to be a multiple of 128 bytes and the
// warp's first group to be a multiple of 32, which the callers guarantee.
__device__ __forceinline__ void discard_scratch_lines(const uint8_t *frame_base, uint32_t first_group, uint32_t ngroups) {
    if (first_group + 32u > ngroups) return;  // warp-uniform: a partial last round (some lanes already left the loop) keeps its lines
    __syncwarp();                             // all 32 lanes are in this round and have stored what they computed from their loads
    const int lane = threadIdx.x & 31;
    if (lane < 12) {
        const uint8_t *line = frame_base + (size_t)first_group * 48u + (size_t)lane * 128u;
        asm volatile("discard.global.L2 [%0], 128;" ::"l"(line) : "memory");
    }
}

// ordinary (L2 write-back) 48-byte store: the scratch image is re-read by pass 3
__device__ __forceinline__ void store_px16_keep(uint8_t *base, size_t group, const Px16 &p) {
    uint4 *q = reinterpret_cast<uint4 *>(base) + group * 3;
    q[0] = make_uint4(p.w[0], p.w[1], p.w[2], p.w[3]);
    q[1] = make_uint4(p.w[4], p.w[5], p.w[6], p.w[7]);
    q[2] = make_uint4(p.w[8], p.w[9], p.w[10], p.w[11]);
}

// ----------------------------------------------------------------------------------------------
// pass 2: S and V histograms of the table-corrected frame (+ statistics in the last block)
// ----------------------------------------------------------------------------------------------
// The full H,S,V of every pixel is kept in `hsv` (frame stride hsv_stride bytes, 16-byte aligned):
// pass 3 starts from it instead of repeating the three table look-ups and the conversion.  Whole 16-pixel groups take
// sdiv / hdiv from the reciprocal unit instead of shared memory (pixel_math.cuh: rint_quotient_rcp); the scalar tail
// looks them up.
template <bool VEC>
__global__ void __launch_bounds__(kBalThreads) hist_sv_kernel(const uint8_t *__restrict__ src, BalFrame *__restrict__ st,
                                                              size_t npx, uint8_t *__restrict__ hsv, size_t hsv_stride) {
    __shared__ uint32_t h[kBalWarps][2][256];
    __shared__ uint8_t lut[3][256];
    __shared__ int sdiv[256], hdiv[256];
    __shared__ StatScratch sc;
    const int frame = blockIdx.y;
    for (int i = threadIdx.x; i < kBalWarps * 512; i += blockDim.x) (&h[0][0][0])[i] = 0;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sdiv[i] = hsv_sdiv(i);
        hdiv[i] = hsv_hdiv(i);
    }
    grid_dependency_wait();  // pass 1 (the tables of this frame) is complete from here on
    for (int i = threadIdx.x; i < 768; i += blockDim.x) (&lut[0][0])[i] = (&st[frame].lut_bgr[0][0])[i];
    __syncthreads();
    const uint8_t *f = src + (size_t)frame * npx * 3;
    uint32_t(*hw)[256] = h[threadIdx.x >> 5];
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t ngroups = VEC ? npx / 16 : 0;
    uint8_t *hf = hsv + (size_t)frame * hsv_stride;
    size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    Px16 in, nxt;
    if (g < ngroups) load_px16<true>(f, g, in);
    for (; g < ngroups; g += stride) {
        if (g + stride < ngroups) load_px16<true>(f, g + stride, nxt);  // prefetch, see pass 1
        Px16 o;
        uint32_t stg[4];
        hsv_group<0>(in, lut, hw, o, stg);
        store_px16_keep(hf, g, o);
        in = nxt;
    }
    for (size_t p = ngroups * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        int hh, ss, vv;
        bgr2hsv(lut[0][f[3 * p]], lut[1][f[3 * p + 1]], lut[2][f[3 * p + 2]], sdiv, hdiv, hh, ss, vv);
        atomicAdd(&hw[0][ss], 1u);
        atomicAdd(&hw[1][vv], 1u);
        hf[3 * p] = (uint8_t)hh;
        hf[3 * p + 1] = (uint8_t)ss;
        hf[3 * p + 2] = (uint8_t)vv;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 512; i += blockDim.x) {
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w) s += (&h[w][0][0])[i];
        if (s) atomicAdd(&st[frame].hist_sv[0][0] + i, s);
    }
    if (last_block_of_frame(&st[frame].ticket[1], gridDim.x)) stats_sv_block(st[frame], npx, sc);
}

// ----------------------------------------------------------------------------------------------
// pass 3: everything per pixel.  MODE 0: no balance (pure conversion); 1: BGR tables only
// (hsv_contrast_correct = 0); 2: tables + HSV stretch round trip from the BGR frame (tiled
// equalisation); 3: the input IS pass 2's H,S,V scratch image -> S/V tables -> HSV2BGR.
// CODE: conversion applied to the balanced pixel for the converted / mask outputs (-1: none).
// ----------------------------------------------------------------------------------------------
struct FinalSmem {
    uint8_t lut[3][256];
    uint8_t lut_sv[2][256];
    int sdiv[256], hdiv[256];
};

// returns the balanced pixel packed as b | g<<8 | r<<16
template <int MODE>
__device__ __forceinline__ uint32_t balance_px(uint32_t b, uint32_t g, uint32_t r, bool vec, const FinalSmem &fs) {
    if (MODE == 3) return hsv2bgr_packed<true>((int)b, fs.lut_sv[0][g], fs.lut_sv[1][r], vec);  // (b, g, r) hold (h, s, v) of pass 2
    if (MODE >= 1) {
        b = fs.lut[0][b];
        g = fs.lut[1][g];
        r = fs.lut[2][r];
    }
    if (MODE == 2) {
        int h, s, v;
        bgr2hsv((int)b, (int)g, (int)r, fs.sdiv, fs.hdiv, h, s, v);
        return hsv2bgr_packed<true>(h, fs.lut_sv[0][s], fs.lut_sv[1][v], vec);
    }
    return b | (g << 8) | (r << 16);
}

// one group of 16 pixels.  TRACK_X: the group touches the row tail (width % 32 columns), where
// cv2's scalar HSV2BGR / HLS rounding applies, or wraps to the next row.
template <int MODE, int CODE, bool TRACK_X, bool NEED_MASK, bool BAL, bool CVT, int J>
struct GroupBody {
    static __device__ __forceinline__ void run(const Px16 &in, int x, int width, int vec_end, const FinalSmem &fs,
                                               const SmemTabs &tabs, const RangeTest &bd, Px16 &ob, Px16 &oc, uint32_t (&q)[4],
                                               uint32_t &bits, uint32_t (&stg)[4]) {
        constexpr bool kOne = CvtTraits<CODE>::kOneChannel;
        const bool vec = TRACK_X ? (x < vec_end) : true;
        const uint32_t p = balance_px<MODE>(BV_GETB(in.w, 3 * J), BV_GETB(in.w, 3 * J + 1), BV_GETB(in.w, 3 * J + 2), vec, fs);
        if (BAL) put_px<J>(ob.w, p);   // packing the balanced pixel costs ~2.5 instructions: only when that output exists
        int o0, o1, o2;
        convert_px<CODE>((int)(p & 0xFF), (int)((p >> 8) & 0xFF), (int)(p >> 16), vec, tabs, o0, o1, o2);
        if (CVT) {   // the converted image is an output (a mask-only call skips assembling it)
            if (kOne) {
                BV_PUTB(q, J, o0);
            } else {
                put_px3<J>(oc.w, stg, (uint32_t)o0, (uint32_t)o1, (uint32_t)o2);
            }
        }
        if (NEED_MASK)
            if (in_range_px<CODE>(o0, o1, o2, bd)) bits |= 1u << J;
        if (TRACK_X) {
            if (++x == width) x = 0;
        }
        GroupBody<MODE, CODE, TRACK_X, NEED_MASK, BAL, CVT, J + 1>::run(in, x, width, vec_end, fs, tabs, bd, ob, oc, q, bits, stg);
    }
};
template <int MODE, int CODE, bool TRACK_X, bool NEED_MASK, bool BAL, bool CVT>
struct GroupBody<MODE, CODE, TRACK_X, NEED_MASK, BAL, CVT, 16> {
    static __device__ __forceinline__ void run(const Px16 &, int, int, int, const FinalSmem &, const SmemTabs &, const RangeTest &,
                                               Px16 &, Px16 &, uint32_t (&)[4], uint32_t &, uint32_t (&)[4]) {}
};

// BAL: the balanced image is an output (always when CODE == -1); without it the vector path skips packing it
template <int MODE, int CODE, bool VEC, bool NEED_MASK, bool BAL = true, bool CVT = true>
__global__ void __launch_bounds__(kBalThreads) final_kernel(const uint8_t *__restrict__ src, size_t src_stride,
                                                            const BalFrame *__restrict__ st, size_t npx, int width,
                                                            BalOutputs out, const uint16_t *__restrict__ g_gamma,
                                                            const uint16_t *__restrict__ g_cbrt) {
    __shared__ FinalSmem fs;
    __shared__ SmemTabs tabs;
    const int frame = blockIdx.y;
    if (MODE == 2) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            fs.sdiv[i] = hsv_sdiv(i);
            fs.hdiv[i] = hsv_hdiv(i);
        }
    }
    init_tabs<CODE>(tabs, g_gamma, g_cbrt);  // constant tables; ends with __syncthreads()
    grid_dependency_wait();                  // the previous pass (frame tables, H,S,V scratch) is complete from here on
    if (MODE == 1 || MODE == 2)
        for (int i = threadIdx.x; i < 768; i += blockDim.x) (&fs.lut[0][0])[i] = (&st[frame].lut_bgr[0][0])[i];
    if (MODE >= 2)
        for (int i = threadIdx.x; i < 512; i += blockDim.x) (&fs.lut_sv[0][0])[i] = (&st[frame].lut_sv[0][0])[i];
    __syncthreads();
    const size_t foff = (size_t)frame * npx;
    const uint8_t *f = src + (size_t)frame * src_stride;  // BGR frame, or pass 2's H,S,V scratch (MODE 3)
    const int vec_end = width - (width % 32);
    constexpr bool kOne = CvtTraits<CODE>::kOneChannel;
    constexpr bool kNeedX = (MODE >= 2) || CvtTraits<CODE>::kNeedsX;
    const RangeTest bd = make_range_test(out.lo, out.hi);
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t ngroups = VEC ? (uint32_t)(npx / 16) : 0u;  // npx < 2^31 (checked on the host)
    const uint32_t height = (uint32_t)(npx / (size_t)width);
    const int wp2 = ((width + 31) / 32) * 2;  // uint16 units per bit-packed row
    for (uint32_t g = blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
        Px16 in;
        load_px16<false>(f, g, in);
        uint32_t y = 0, x0 = 0;
        if (kNeedX || (NEED_MASK && out.mask_bits)) {
            const uint32_t p0 = g * 16u;
            y = p0 / (uint32_t)width;
            x0 = p0 - y * (uint32_t)width;
        }
        Px16 ob, oc;
        uint32_t q[4] = {0, 0, 0, 0};
        uint32_t bits = 0;
        uint32_t stg[4] = {0, 0, 0, 0};
#pragma unroll
        for (int k = 0; k < 12; ++k) ob.w[k] = oc.w[k] = 0;
        if (kNeedX && (int)x0 + 16 > vec_end)
            GroupBody<MODE, CODE, true, NEED_MASK, BAL, CVT, 0>::run(in, (int)x0, width, vec_end, fs, tabs, bd, ob, oc, q, bits, stg);
        else
            GroupBody<MODE, CODE, false, NEED_MASK, BAL, CVT, 0>::run(in, (int)x0, width, vec_end, fs, tabs, bd, ob, oc, q, bits, stg);
        if (BAL && out.balanced) store_px16(out.balanced + foff * 3, g, ob);
        if (CVT && out.converted) {
            if (kOne)
                st_stream(reinterpret_cast<uint4 *>(out.converted + foff) + g, make_uint4(q[0], q[1], q[2], q[3]));
            else
                store_px16(out.converted + foff * 3, g, oc);
        }
        if (NEED_MASK && out.mask) {
            uint32_t m[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t nib = (bits >> (4 * k)) & 0xF;
                // spread 4 bits to 4 bytes of 0x00 / 0xFF
                m[k] = ((nib & 1) * 0xFFu) | (((nib >> 1) & 1) * 0xFF00u) | (((nib >> 2) & 1) * 0xFF0000u) |
                       (((nib >> 3) & 1) * 0xFF000000u);
            }
            st_stream(reinterpret_cast<uint4 *>(out.mask + foff) + g, make_uint4(m[0], m[1], m[2], m[3]));
        }
        if (NEED_MASK && out.mask_bits)  // requires width % 16 == 0: a group never straddles rows
            out.mask_bits[((size_t)frame * height + y) * wp2 + (x0 >> 4)] = (uint16_t)bits;
        if (MODE == 3 && (src_stride & 127) == 0) discard_scratch_lines(f, g & ~31u, ngroups);
    }
    // scalar path: trailing pixels of each frame, or everything for unaligned / odd-sized frames
    for (size_t p = (size_t)ngroups * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npx; p += stride) {
        const int x = (int)(p % (size_t)width);
        const bool vec = x < vec_end;
        const uint32_t px = balance_px<MODE>(f[3 * p], f[3 * p + 1], f[3 * p + 2], vec, fs);
        const int b = (int)(px & 0xFF), gg = (int)((px >> 8) & 0xFF), r = (int)(px >> 16);
        if (out.balanced) {
            uint8_t *o = out.balanced + (foff + p) * 3;
            o[0] = (uint8_t)b;
            o[1] = (uint8_t)gg;
            o[2] = (uint8_t)r;
        }
        int o0, o1, o2;
        convert_px<CODE>(b, gg, r, vec, tabs, o0, o1, o2);
        if (out.converted) {
            if (kOne) {
                out.converted[foff + p] = (uint8_t)o0;
            } else {
                uint8_t *o = out.converted + (foff + p) * 3;
                o[0] = (uint8_t)o0;
                o[1] = (uint8_t)o1;
                o[2] = (uint8_t)o2;
            }
        }
        if (out.mask) out.mask[foff + p] = in_range_px<CODE>(o0, o1, o2, bd) ? 255 : 0;
    }
}

// ----------------------------------------------------------------------------------------------
// Hue-interval table: the HSV inRange mask of a balanced frame without the HSV -> BGR -> HSV
// round trip.
//
// With hsv_contrast_correct the balanced pixel is HSV2BGR(H, S', V') (color_balance.cpp:693) and
// modules/bins.py:13-16 immediately converts it back to HSV and thresholds it.  That composite
//     (H, S', V')  ->  HSV2BGR  ->  BGR2HSV  ->  inRange(lo, hi)
// does not depend on the frame, only on the bounds.  HSV2BGR yields max = trunc(v*255),
// min = trunc(v(1-s)*255) and a middle value that alone depends on H; so S2 and V2 of the round
// trip are functions of (S', V') and, for every (S', V'), the hues that pass are one cyclic
// interval of [0,180).  The table stores that interval for each of the 65536 (S', V') pairs as
// (first hue, span mod 256); a pixel passes iff ((H - first) & 255) <= span.  It is filled by the
// exact per-pixel arithmetic (all 180 x 65536 combinations) once per distinct bounds set, the
// build verifies the single-interval property for every pair (otherwise the generic pass 3 is
// used), and it lives in shared memory (128 KB, brought in with one TMA bulk copy per block).
// Valid for whole 32-pixel groups of a row only (cv2's vector HSV2BGR rounding): width % 32 == 0.
// ----------------------------------------------------------------------------------------------
constexpr int kIvlEntries = 65536;
constexpr uint32_t kIvlBytes = kIvlEntries * 2;
constexpr int kIvlEmpty = 200;  // first = 200, span = 0: no hue in [0,180) passes

__global__ void __launch_bounds__(256) ivl_build_kernel(uint16_t *__restrict__ table, int *__restrict__ bad, Bounds3 bd) {
    __shared__ int sdiv[256], hdiv[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        sdiv[i] = hsv_sdiv(i);
        hdiv[i] = hsv_hdiv(i);
    }
    __syncthreads();
    const RangeTest rt = make_range_test(bd.lo, bd.hi);
    const int lane = threadIdx.x & 31;
    const int pair = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // S' * 256 + V'
    const int S = pair >> 8, V = pair & 255;
    auto passes = [&](int H) {
        const uint32_t p = hsv2bgr_packed(H, S, V, true);
        int h2, s2, v2;
        bgr2hsv((int)(p & 0xFF), (int)((p >> 8) & 0xFF), (int)(p >> 16), sdiv, hdiv, h2, s2, v2);
        return in_range_px<BV_BGR2HSV>(h2, s2, v2, rt);
    };
    int n_in = 0, n_rise = 0, first = 0;
    for (int it = 0; it < 6; ++it) {
        const int H = it * 32 + lane;
        bool in = false, rise = false;
        if (H < 180) {
            in = passes(H);
            rise = in && !passes(H == 0 ? 179 : H - 1);
        }
        const uint32_t bi = __ballot_sync(0xFFFFFFFFu, in), br = __ballot_sync(0xFFFFFFFFu, rise);
        n_in += __popc(bi);
        n_rise += __popc(br);
        if (br) first = it * 32 + __ffs(br) - 1;
    }
    if (lane == 0) {
        int lo = kIvlEmpty, span = 0;
        if (n_in == 180) {
            lo = 0;
            span = 179;
        } else if (n_in > 0) {
            if (n_rise != 1) atomicOr(bad, 1);
            const int last = (first + n_in - 1) % 180;
            lo = first;
            span = (last - first) & 0xFF;
        }
        table[pair] = (uint16_t)(lo | (span << 8));
    }
}

struct IvlSmem {
    uint16_t tab[kIvlEntries];
    uint64_t bar;
};

// Per-frame composition of the S / V stretch tables into the interval table: entry (S, V) of frame f =
// table[(S'[S] << 8) | V'[V]], so that pass 3 indexes with the scratch image's own S and V bytes and needs ONE shared-memory
// look-up per pixel instead of three (the stretch tables are frame statistics, the interval table is not).  256 KB per
// 4-frame chunk, built in ~2 us behind pass 2 (programmatic dependent launch), read back by the TMA copy below.
__global__ void __launch_bounds__(1024) ivl_compose_kernel(const uint16_t *__restrict__ table, const BalFrame *__restrict__ st,
                                                           uint16_t *__restrict__ composed) {
    __shared__ uint8_t lsv[2][256];
    const int frame = blockIdx.y;
    grid_dependency_wait();  // pass 2 (the S / V tables of this frame) is complete from here on
    for (int i = threadIdx.x; i < 512; i += blockDim.x) (&lsv[0][0])[i] = (&st[frame].lut_sv[0][0])[i];
    __syncthreads();
    // entry index = (V << 8) | S: S and V are neighbouring bytes of the scratch image, so pass 3 takes the index out of the
    // packed words with one byte-permute
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < kIvlEntries; idx += gridDim.x * blockDim.x)
        composed[(size_t)frame * kIvlEntries + idx] = __ldg(table + (((uint32_t)lsv[0][idx & 255] << 8) | lsv[1][idx >> 8]));
}

// pass 3 of the fast path: H,S,V scratch -> S/V stretch tables -> hue interval -> mask
__global__ void __launch_bounds__(1024, 1) mask_from_hsv_kernel(const uint8_t *__restrict__ hsv, size_t hsv_stride,
                                                                const BalFrame *__restrict__ st,
                                                                const uint16_t *__restrict__ table, size_t npx, int width,
                                                                BalOutputs out) {
    extern __shared__ __align__(128) unsigned char ivl_raw[];
    IvlSmem &sm = *reinterpret_cast<IvlSmem *>(ivl_raw);
    const int frame = blockIdx.y;
    if (threadIdx.x == 0) {
        mbar_init(&sm.bar, 1);
        mbar_expect_tx(&sm.bar, kIvlBytes);
        const unsigned char *mine = reinterpret_cast<const unsigned char *>(table + (size_t)frame * kIvlEntries);  // this frame's composed table
        for (uint32_t o = 0; o < kIvlBytes; o += 32768u)
            bulk_g2s(reinterpret_cast<unsigned char *>(sm.tab) + o, mine + o, 32768u, &sm.bar);
    }
    const uint8_t *f = hsv + (size_t)frame * hsv_stride;
    const size_t foff = (size_t)frame * npx;
    const uint32_t stride = gridDim.x * blockDim.x, ngroups = (uint32_t)(npx / 16);
    const uint32_t height = (uint32_t)(npx / (size_t)width);
    const int wp2 = ((width + 31) / 32) * 2;
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    Px16 in, nxt;
    if (g < ngroups) load_px16<false>(f, g, in);   // the first group travels while the table is still on its way
    __syncthreads();
    mbar_wait(&sm.bar, 0);
    for (; g < ngroups; g += stride) {
        if (g + stride < ngroups) load_px16<false>(f, g + stride, nxt);  // prefetch the next group
        uint32_t bits = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const uint32_t h = BV_GETB(in.w, 3 * j);
            // bytes 3j+1 (S) and 3j+2 (V) as one little-endian 16-bit field = (V << 8) | S, possibly across two words
            const int o = 3 * j + 1, wi = o >> 2, bi = o & 3;
            uint32_t sv;
            if (bi < 3)   // both bytes in one word: one byte-permute (second operand = 0 supplies the zero bytes)
                sv = __byte_perm(in.w[wi], 0u, 0x4400u | (uint32_t)((bi + 1) << 4) | (uint32_t)bi);
            else          // S is the last byte of a word, V the first of the next (4 of the 16 pixels)
                sv = __funnelshift_r(in.w[wi], in.w[wi + 1 < 12 ? wi + 1 : wi], 24) & 0xFFFFu;
            const uint32_t e = sm.tab[sv];   // composed per frame: indexed by the raw S, V
            if (((h - (e & 0xFFu)) & 0xFFu) <= (e >> 8)) bits |= 1u << j;
        }
        if (out.mask) {
            uint32_t m[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t nib = (bits >> (4 * k)) & 0xF;
                m[k] = ((nib & 1) * 0xFFu) | (((nib >> 1) & 1) * 0xFF00u) | (((nib >> 2) & 1) * 0xFF0000u) |
                       (((nib >> 3) & 1) * 0xFF000000u);
            }
            st_stream(reinterpret_cast<uint4 *>(out.mask + foff) + g, make_uint4(m[0], m[1], m[2], m[3]));
        }
        if (out.mask_bits) {
            const uint32_t p0 = g * 16u, y = p0 / (uint32_t)width, x0 = p0 - y * (uint32_t)width;
            out.mask_bits[((size_t)frame * height + y) * wp2 + (x0 >> 4)] = (uint16_t)bits;
        }
        if ((hsv_stride & 127) == 0) discard_scratch_lines(f, g & ~31u, ngroups);
        in = nxt;
    }
}

// Table for these bounds, building it on first use (one build + one flag read-back per distinct
// bounds set; tuner changes are rare).  *table = nullptr when the fast path cannot be used.
static int ivl_table(bv_ctx *ctx, const uint8_t lo[3], const uint8_t hi[3], const uint16_t **table) {
    *table = nullptr;
    if (ctx->opt[BV_OPT_NO_HUE_TABLE] > 0) return BV_OK;
    uint8_t key[6] = {lo[0], lo[1], lo[2], hi[0], hi[1], hi[2]};
    for (int i = 0; i < BV_IVL_SLOTS; ++i)
        if (ctx->ivl[i].state && !memcmp(ctx->ivl[i].key, key, 6)) {
            if (ctx->ivl[i].state == 1) *table = ctx->ivl[i].table;
            return BV_OK;
        }
    const int slot = ctx->ivl_next;
    ctx->ivl_next = (slot + 1) % BV_IVL_SLOTS;
    if (ctx->ivl[slot].state) BV_CUDA(cudaStreamSynchronize(ctx->stream));  // the evicted table may still be in use
    if (!ctx->ivl[slot].table) BV_CUDA(cudaMalloc(&ctx->ivl[slot].table, kIvlBytes));
    if (!ctx->d_ivl_flag) BV_CUDA(cudaMalloc(&ctx->d_ivl_flag, sizeof(int)));
    ctx->ivl[slot].state = 0;
    BV_CUDA(cudaMemsetAsync(ctx->d_ivl_flag, 0, sizeof(int), ctx->stream));
    Bounds3 bd;
    for (int k = 0; k < 3; ++k) {
        bd.lo[k] = lo[k];
        bd.hi[k] = hi[k];
    }
    BV_LAUNCH(ctx, ivl_build_kernel, kIvlEntries / 8, 256, 0, ctx->ivl[slot].table, ctx->d_ivl_flag, bd);
    int bad = 0;
    BV_CUDA(cudaMemcpyAsync(&bad, ctx->d_ivl_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    BV_CUDA(cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->ivl[slot].key, key, 6);
    ctx->ivl[slot].state = bad ? 2 : 1;
    if (!bad) *table = ctx->ivl[slot].table;
    return BV_OK;
}

static int launch_mask_from_hsv(bv_ctx *ctx, const uint8_t *hsv, size_t hsv_stride, const BalFrame *st, int batch, size_t npx,
                                int width, const uint16_t *table, uint16_t *composed, const BalOutputs &out) {
    if (!ctx->ivl_attr_set) {  // per device
        BV_CUDA(cudaFuncSetAttribute(mask_from_hsv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IvlSmem)));
        ctx->ivl_attr_set = 1;
    }
    int bpf = (ctx->sm_count + batch - 1) / batch;  // one 1024-thread block per SM
    const size_t need = (npx / 16 + 1023) / 1024;
    if ((size_t)bpf > need) bpf = (int)(need ? need : 1);
    BV_LAUNCH_PDL(ctx, ivl_compose_kernel, dim3(8, batch), 1024, 0, table, st, composed);
    BV_LAUNCH(ctx, mask_from_hsv_kernel, dim3(bpf, batch), 1024, sizeof(IvlSmem), hsv, hsv_stride, st, composed, npx, width, out);
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// Tiled equalisation (P1): horizontal_blocks x vertical_blocks > 1.  One block works inside one
// tile (grid = blocks x tiles x frames), per pixel, with that tile's tables.  Same three passes.
// ----------------------------------------------------------------------------------------------
// 4 consecutive pixels = 3 aligned words (tile rows that start on a multiple of 4 pixels, 4-byte aligned frames)
__device__ __forceinline__ void unpack_px4(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t (&c)[4][3]) {
    c[0][0] = w0 & 0xFFu; c[0][1] = (w0 >> 8) & 0xFFu; c[0][2] = (w0 >> 16) & 0xFFu;
    c[1][0] = w0 >> 24;   c[1][1] = w1 & 0xFFu;        c[1][2] = (w1 >> 8) & 0xFFu;
    c[2][0] = (w1 >> 16) & 0xFFu; c[2][1] = w1 >> 24;  c[2][2] = w2 & 0xFFu;
    c[3][0] = (w2 >> 8) & 0xFFu;  c[3][1] = (w2 >> 16) & 0xFFu; c[3][2] = w2 >> 24;
}

template <int PASS, bool VEC4>
__global__ void __launch_bounds__(kBalThreads) hist_tiled_kernel(const uint8_t *__restrict__ src, BalFrame *__restrict__ st,
                                                                 BalTile *__restrict__ tiles, size_t npx, TileGeom tg,
                                                                 bv_balance_params prm, const double *__restrict__ pow_quarter) {
    __shared__ uint32_t h[kBalWarps][3][256];
    __shared__ uint8_t lut[3][256];
    __shared__ int sdiv[256], hdiv[256];
    __shared__ StatScratch sc;
    const int tile = blockIdx.y, frame = blockIdx.z, n_tiles = gridDim.y;
    BalTile &T = tiles[(size_t)frame * n_tiles + tile];
    for (int i = threadIdx.x; i < kBalWarps * 768; i += blockDim.x) (&h[0][0][0])[i] = 0;
    if (PASS == 2) {
        for (int i = threadIdx.x; i < 768; i += blockDim.x) (&lut[0][0])[i] = (&T.lut[0][0])[i];
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            sdiv[i] = hsv_sdiv(i);
            hdiv[i] = hsv_hdiv(i);
        }
    }
    __syncthreads();
    const uint8_t *f = src + (size_t)frame * npx * 3;
    uint32_t(*hw)[256] = h[threadIdx.x >> 5];
    const size_t tile_px = (size_t)tg.bw * tg.bh;
    // a warp takes whole rows of the tile, its lanes consecutive pixels of the row: no per-pixel index division
    const int ty = tile / tg.hb, tx = tile - ty * tg.hb;
    const int lane = threadIdx.x & 31, warps = gridDim.x * kBalWarps;
    if (VEC4) {
        // groups of 4 pixels, numbered row after row inside the tile, dealt out to all threads of the tile's blocks
        const unsigned gpr = (unsigned)tg.bw >> 2, n_groups = gpr * (unsigned)tg.bh;
        for (unsigned g = blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += gridDim.x * blockDim.x) {
            const unsigned yy = g / gpr, gx = g - yy * gpr;
            const uint32_t *rw = reinterpret_cast<const uint32_t *>(
                f + ((size_t)(ty * tg.bh + (int)yy) * tg.width + (size_t)tx * tg.bw + 4 * gx) * 3);
            uint32_t c[4][3];
            unpack_px4(__ldg(rw), __ldg(rw + 1), __ldg(rw + 2), c);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (PASS == 1) {
                    atomicAdd(&hw[0][c[k][0]], 1u);
                    atomicAdd(&hw[1][c[k][1]], 1u);
                    atomicAdd(&hw[2][c[k][2]], 1u);
                } else {
                    int hh, ss, vv;
                    bgr2hsv(lut[0][c[k][0]], lut[1][c[k][1]], lut[2][c[k][2]], sdiv, hdiv, hh, ss, vv);
                    atomicAdd(&hw[0][ss], 1u);
                    atomicAdd(&hw[1][vv], 1u);
                }
            }
        }
    }
    for (int yy = blockIdx.x * kBalWarps + (threadIdx.x >> 5); !VEC4 && yy < tg.bh; yy += warps) {
        const uint8_t *row = f + ((size_t)(ty * tg.bh + yy) * tg.width + (size_t)tx * tg.bw) * 3;
        for (int xx = lane; xx < tg.bw; xx += 32) {
            const uint8_t *px = row + 3 * xx;
            if (PASS == 1) {
                atomicAdd(&hw[0][px[0]], 1u);
                atomicAdd(&hw[1][px[1]], 1u);
                atomicAdd(&hw[2][px[2]], 1u);
            } else {
                int hh, ss, vv;
                bgr2hsv(lut[0][px[0]], lut[1][px[1]], lut[2][px[2]], sdiv, hdiv, hh, ss, vv);
                atomicAdd(&hw[0][ss], 1u);
                atomicAdd(&hw[1][vv], 1u);
            }
        }
    }
    __syncthreads();
    const int nbins = PASS == 1 ? 768 : 512;
    for (int i = threadIdx.x; i < nbins; i += blockDim.x) {
        uint32_t s = 0;
#pragma unroll
        for (int w = 0; w < kBalWarps; ++w) s += (&h[w][0][0])[i];
        if (!s) continue;
        if (PASS == 1) {
            atomicAdd(&T.hist[0][0] + i, s);
            atomicAdd(&st[frame].hist_bgr[0][0] + i, s);
        } else {
            atomicAdd(&st[frame].hist_sv[0][0] + i, s);
        }
    }
    if (last_block_of_frame(&st[frame].ticket[PASS - 1], gridDim.x * gridDim.y)) {
        if (PASS == 1)
            stats_bgr_block(st[frame], npx, prm, pow_quarter, sc, tiles + (size_t)frame * n_tiles, n_tiles, tile_px);
        else
            stats_sv_block(st[frame], npx, sc);
    }
}

template <int MODE, int CODE, bool VEC4>
__global__ void __launch_bounds__(kBalThreads) final_tiled_kernel(const uint8_t *__restrict__ src, const BalFrame *__restrict__ st,
                                                                  const BalTile *__restrict__ tiles, size_t npx, TileGeom tg,
                                                                  BalOutputs out, const uint16_t *__restrict__ g_gamma,
                                                                  const uint16_t *__restrict__ g_cbrt) {
    __shared__ FinalSmem fs;
    __shared__ SmemTabs tabs;
    const int tile = blockIdx.y, frame = blockIdx.z, n_tiles = gridDim.y;
    const BalTile &T = tiles[(size_t)frame * n_tiles + tile];
    for (int i = threadIdx.x; i < 768; i += blockDim.x) (&fs.lut[0][0])[i] = (&T.lut[0][0])[i];
    if (MODE == 2) {
        for (int i = threadIdx.x; i < 512; i += blockDim.x) (&fs.lut_sv[0][0])[i] = (&st[frame].lut_sv[0][0])[i];
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            fs.sdiv[i] = hsv_sdiv(i);
            fs.hdiv[i] = hsv_hdiv(i);
        }
    }
    init_tabs<CODE>(tabs, g_gamma, g_cbrt);
    const size_t foff = (size_t)frame * npx;
    const uint8_t *f = src + foff * 3;
    const int vec_end = tg.width - (tg.width % 32);
    constexpr bool kOne = CvtTraits<CODE>::kOneChannel;
    const RangeTest bd = make_range_test(out.lo, out.hi);
    __syncthreads();
    const int ty = tile / tg.hb, tx = tile - ty * tg.hb;
    const int lane = threadIdx.x & 31, warps = gridDim.x * kBalWarps;
    if constexpr (VEC4) {
        const unsigned gpr = (unsigned)tg.bw >> 2, n_groups = gpr * (unsigned)tg.bh;
        for (unsigned g = blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += gridDim.x * blockDim.x) {
            {
                const unsigned yy = g / gpr, gx = g - yy * gpr;
                const int x0 = tx * tg.bw + 4 * (int)gx;
                const size_t p = (size_t)(ty * tg.bh + (int)yy) * tg.width + x0;
                const uint32_t *rw = reinterpret_cast<const uint32_t *>(f + 3 * p);
                uint32_t c[4][3];
                unpack_px4(__ldg(rw), __ldg(rw + 1), __ldg(rw + 2), c);
                uint32_t bal[4], cv[4];
                uint32_t m = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool vec = x0 + k < vec_end;
                    bal[k] = balance_px<MODE>(c[k][0], c[k][1], c[k][2], vec, fs);
                    int o0, o1, o2;
                    convert_px<CODE>((int)(bal[k] & 0xFF), (int)((bal[k] >> 8) & 0xFF), (int)(bal[k] >> 16), vec, tabs, o0, o1, o2);
                    cv[k] = kOne ? (uint32_t)o0 : ((uint32_t)o0 | ((uint32_t)o1 << 8) | ((uint32_t)o2 << 16));
                    if (in_range_px<CODE>(o0, o1, o2, bd)) m |= 0xFFu << (8 * k);
                }
                if (out.balanced) {
                    uint32_t *o = reinterpret_cast<uint32_t *>(out.balanced + (foff + p) * 3);
                    o[0] = bal[0] | (bal[1] << 24);
                    o[1] = (bal[1] >> 8) | (bal[2] << 16);
                    o[2] = (bal[2] >> 16) | (bal[3] << 8);
                }
                if (out.converted) {
                    if (kOne) {
                        *reinterpret_cast<uint32_t *>(out.converted + foff + p) = cv[0] | (cv[1] << 8) | (cv[2] << 16) | (cv[3] << 24);
                    } else {
                        uint32_t *o = reinterpret_cast<uint32_t *>(out.converted + (foff + p) * 3);
                        o[0] = cv[0] | (cv[1] << 24);
                        o[1] = (cv[1] >> 8) | (cv[2] << 16);
                        o[2] = (cv[2] >> 16) | (cv[3] << 8);
                    }
                }
                if (out.mask) *reinterpret_cast<uint32_t *>(out.mask + foff + p) = m;
            }
        }
    } else {
    for (int yy = blockIdx.x * kBalWarps + (threadIdx.x >> 5); yy < tg.bh; yy += warps)
    for (int xx = lane; xx < tg.bw; xx += 32) {
        const int x = tx * tg.bw + xx;
        const size_t p = (size_t)(ty * tg.bh + yy) * tg.width + x;
        const bool vec = x < vec_end;
        const uint32_t px = balance_px<MODE>(f[3 * p], f[3 * p + 1], f[3 * p + 2], vec, fs);
        const int b = (int)(px & 0xFF), gg = (int)((px >> 8) & 0xFF), r = (int)(px >> 16);
        if (out.balanced) {
            uint8_t *o = out.balanced + (foff + p) * 3;
            o[0] = (uint8_t)b;
            o[1] = (uint8_t)gg;
            o[2] = (uint8_t)r;
        }
        int o0, o1, o2;
        convert_px<CODE>(b, gg, r, vec, tabs, o0, o1, o2);
        if (out.converted) {
            if (kOne) {
                out.converted[foff + p] = (uint8_t)o0;
            } else {
                uint8_t *o = out.converted + (foff + p) * 3;
                o[0] = (uint8_t)o0;
                o[1] = (uint8_t)o1;
                o[2] = (uint8_t)o2;
            }
        }
        if (out.mask) out.mask[foff + p] = in_range_px<CODE>(o0, o1, o2, bd) ? 255 : 0;
    }
}
}

template <int MODE>
static int dispatch_final_tiled(bv_ctx *ctx, const uint8_t *src, const BalFrame *st, const BalTile *tiles, dim3 grid,
                                size_t npx, const TileGeom &tg, int code, const BalOutputs &out, bool vec4) {
#define BV_FT(C)                                                                                                          \
    if (vec4)                                                                                                             \
        BV_LAUNCH(ctx, (final_tiled_kernel<MODE, C, true>), grid, kBalThreads, 0, src, st, tiles, npx, tg, out,           \
                  ctx->d_lab_gamma, ctx->d_lab_cbrt);                                                                     \
    else                                                                                                                  \
        BV_LAUNCH(ctx, (final_tiled_kernel<MODE, C, false>), grid, kBalThreads, 0, src, st, tiles, npx, tg, out,          \
                  ctx->d_lab_gamma, ctx->d_lab_cbrt);                                                                     \
    return BV_OK
    switch (code) {
        case -1: BV_FT(-1);
        case BV_BGR2HSV: BV_FT(BV_BGR2HSV);
        case BV_BGR2LAB: BV_FT(BV_BGR2LAB);
        case BV_BGR2GRAY: BV_FT(BV_BGR2GRAY);
        case BV_BGR2YCRCB: BV_FT(BV_BGR2YCRCB);
        case BV_BGR2HLS: BV_FT(BV_BGR2HLS);
        default: set_error("stage: conversion code %d is not available in the fused pass", code); return BV_ERR_INVALID;
    }
#undef BV_FT
}

static int balance_run_tiled(bv_ctx *ctx, const uint8_t *src, int batch, int height, int width, const bv_balance_params &prm,
                             int cvt_code, const BalOutputs &out, BalFrame *st) {
    const int hb = prm.horizontal_blocks, vb = prm.vertical_blocks;
    if (hb < 1 || vb < 1 || width % hb || height % vb) {
        // the reference walks off the end of the row for non-divisible tilings (color_balance.cpp:442-464)
        set_error("colour balance: horizontal/vertical_blocks must divide the frame (%dx%d into %dx%d tiles)", width, height, hb, vb);
        return BV_ERR_UNSUPPORTED;
    }
    const int n_tiles = hb * vb;
    if (n_tiles > 4096 || out.mask_bits) {
        set_error("colour balance: too many tiles, or bit-packed mask requested with tiling");
        return BV_ERR_UNSUPPORTED;
    }
    const size_t npx = (size_t)height * width;
    BV_TRY(ensure_scratch(ctx, SCR_BAL_TILES, sizeof(BalTile) * (size_t)batch * n_tiles));
    BalTile *tiles = (BalTile *)ctx->scratch[SCR_BAL_TILES];
    BV_CUDA(cudaMemsetAsync(tiles, 0, sizeof(BalTile) * (size_t)batch * n_tiles, ctx->stream));
    TileGeom tg{hb, vb, width / hb, height / vb, width, height};
    const size_t tile_px = (size_t)tg.bw * tg.bh;
    int bx = (int)((tile_px + kBalThreads * 16 - 1) / (kBalThreads * 16));
    const int cap = (ctx->sm_count * 8 + n_tiles * batch - 1) / (n_tiles * batch);
    if (bx > cap) bx = cap;
    if (bx < 1) bx = 1;
    dim3 grid(bx, n_tiles, batch);
    // word-wide path: every tile row starts on a multiple of 4 pixels and all buffers are 4-byte aligned
    auto aligned4 = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 3) == 0; };
    const bool vec4 = width % 4 == 0 && tg.bw % 4 == 0 && aligned4(src) && aligned4(out.balanced) && aligned4(out.converted) &&
                      aligned4(out.mask);
#define BV_HT(P)                                                                                                       \
    do {                                                                                                               \
        if (vec4)                                                                                                      \
            BV_LAUNCH(ctx, (hist_tiled_kernel<P, true>), grid, kBalThreads, 0, src, st, tiles, npx, tg, prm, ctx->d_pow_quarter); \
        else                                                                                                           \
            BV_LAUNCH(ctx, (hist_tiled_kernel<P, false>), grid, kBalThreads, 0, src, st, tiles, npx, tg, prm, ctx->d_pow_quarter); \
    } while (0)
    BV_HT(1);
    if (prm.hsv_contrast_correct) {
        BV_HT(2);
#undef BV_HT
        return dispatch_final_tiled<2>(ctx, src, st, tiles, grid, npx, tg, cvt_code, out, vec4);
    }
    return dispatch_final_tiled<1>(ctx, src, st, tiles, grid, npx, tg, cvt_code, out, vec4);
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
// Tuning knobs (bv_set_option / BV_* environment variables read at bv_create, see api.cu):
// blocks per SM of the histogram passes and of the final pass.  With side streams the passes of
// different chunks share the SMs, so each kernel takes a small persistent grid (2 blocks/SM); a
// lone chunk (single frame, or profiling) gets the whole machine.
static int hist_blocks_per_sm(const bv_ctx *ctx) { return ctx->opt[BV_OPT_HIST_BPS] > 0 ? ctx->opt[BV_OPT_HIST_BPS] : (ctx->overlapped ? 2 : 4); }
static int final_blocks_per_sm(const bv_ctx *ctx) { return ctx->opt[BV_OPT_FINAL_BPS] > 0 ? ctx->opt[BV_OPT_FINAL_BPS] : (ctx->overlapped ? 2 : 8); }

static bool vec_ok(const void *p, size_t npx, int batch, int bytes_per_px) {
    (void)bytes_per_px;
    return p == nullptr || (host_aligned16(p) && (npx % 16 == 0 || batch == 1));
}

template <int MODE, int CODE>
static int launch_final(bv_ctx *ctx, const uint8_t *src, size_t src_stride, const BalFrame *st, int batch, size_t npx,
                        int width, const BalOutputs &out, bool vec) {
    int bpf = (ctx->sm_count * final_blocks_per_sm(ctx) + batch - 1) / batch;
    const size_t need = (npx / 16 + kBalThreads - 1) / kBalThreads;
    if ((size_t)bpf > need) bpf = (int)(need ? need : 1);
    dim3 grid(bpf, batch);
    const bool need_mask = out.mask || out.mask_bits;
#define BV_FINAL(V, M)                                                                                              \
    BV_LAUNCH_PDL(ctx, (final_kernel<MODE, CODE, V, M>), grid, kBalThreads, 0, src, src_stride, st, npx, width, out, \
                  ctx->d_lab_gamma, ctx->d_lab_cbrt)
#define BV_FINAL_NOBAL(M)                                                                                                     \
    BV_LAUNCH_PDL(ctx, (final_kernel<MODE, CODE, true, M, false>), grid, kBalThreads, 0, src, src_stride, st, npx, width, out, \
                  ctx->d_lab_gamma, ctx->d_lab_cbrt)
    if (vec && CODE != -1 && !out.balanced && !out.converted && need_mask) {   // mask only (modules/bins.py, red_buoy.py)
        BV_LAUNCH_PDL(ctx, (final_kernel<MODE, CODE, true, true, false, false>), grid, kBalThreads, 0, src, src_stride, st, npx,
                      width, out, ctx->d_lab_gamma, ctx->d_lab_cbrt);
    } else if (vec && CODE != -1 && !out.balanced) {   // the common module case: only the converted image / the mask leave the pass
        if (need_mask) BV_FINAL_NOBAL(true); else BV_FINAL_NOBAL(false);
    } else if (vec) {
        if (need_mask) BV_FINAL(true, true); else BV_FINAL(true, false);
    } else {
        if (need_mask) BV_FINAL(false, true); else BV_FINAL(false, false);
    }
#undef BV_FINAL
#undef BV_FINAL_NOBAL
    return BV_OK;
}

template <int MODE>
static int dispatch_final(bv_ctx *ctx, const uint8_t *src, size_t src_stride, const BalFrame *st, int batch, size_t npx,
                          int width, int code, const BalOutputs &out, bool vec) {
    switch (code) {
        case -1: return launch_final<MODE, -1>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        case BV_BGR2HSV: return launch_final<MODE, BV_BGR2HSV>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        case BV_BGR2LAB: return launch_final<MODE, BV_BGR2LAB>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        case BV_BGR2GRAY: return launch_final<MODE, BV_BGR2GRAY>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        case BV_BGR2YCRCB: return launch_final<MODE, BV_BGR2YCRCB>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        case BV_BGR2HLS: return launch_final<MODE, BV_BGR2HLS>(ctx, src, src_stride, st, batch, npx, width, out, vec);
        default: set_error("stage: conversion code %d is not available in the fused pass", code); return BV_ERR_INVALID;
    }
}

static bool all_vec(const uint8_t *src, const BalOutputs &out, size_t npx, int batch) {
    return vec_ok(src, npx, batch, 3) && vec_ok(out.balanced, npx, batch, 3) && vec_ok(out.converted, npx, batch, 3) &&
           vec_ok(out.mask, npx, batch, 1);
}

// sdiv / hdiv through the reciprocal unit: compared once per context with the integer formulas, all 2 x 256 values
__global__ void rcp_tables_check_kernel(int *bad) {
    const int d = threadIdx.x;
    if (rint_quotient_rcp((float)(255 << kHsvShift), d) != hsv_sdiv(d) ||
        rint_quotient_rcp((float)((180 << kHsvShift) / 6), d) != hsv_hdiv(d))
        atomicOr(bad, 1);
}

int rcp_tables_check(bv_ctx *ctx) {   // called by bv_create: every BGR2HSV of the library relies on it
    if (!ctx->d_ivl_flag) BV_CUDA(cudaMalloc(&ctx->d_ivl_flag, sizeof(int)));
    BV_CUDA(cudaMemsetAsync(ctx->d_ivl_flag, 0, sizeof(int), ctx->stream));
    BV_LAUNCH(ctx, rcp_tables_check_kernel, 1, 256, 0, ctx->d_ivl_flag);
    int bad = 1;
    BV_CUDA(cudaMemcpyAsync(&bad, ctx->d_ivl_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    BV_CUDA(cudaStreamSynchronize(ctx->stream));
    if (bad) {
        set_error("bv_create: rcp.approx.f32 of this device does not reproduce OpenCV's sdiv / hdiv tables (library is built for sm_100a)");
        return BV_ERR_UNSUPPORTED;
    }
    return BV_OK;
}

int convert_run(bv_ctx *ctx, const uint8_t *src, int batch, int height, int width, int cvt_code, const BalOutputs &out) {
    const size_t npx = (size_t)height * width;
    const bool vec = all_vec(src, out, npx, batch);
    ctx->overlapped = 0;
    if (out.mask_bits && !(vec && width % 16 == 0)) {
        set_error("convert_run: bit-packed mask needs 16-byte aligned buffers and width %% 16 == 0");
        return BV_ERR_INVALID;
    }
    return dispatch_final<0>(ctx, src, npx * 3, nullptr, batch, npx, width, cvt_code, out, vec);
}

int balance_run(bv_ctx *ctx, const uint8_t *src, int batch, int height, int width, const bv_balance_params &prm,
                int cvt_code, const BalOutputs &out, bv_balance_stats *stats_host, const ChunkHook *after_chunk) {
    if (prm.hsi_contrast_correct) {
        // color_balance.cpp:702-774 runs after every other stage, on the balanced frame: produce that
        // frame with the remaining flags, correct it in place (hsi.cu), then convert / threshold it.
        const size_t npx_ = (size_t)height * width;
        uint8_t *bgr = out.balanced;
        if (!bgr) {
            BV_TRY(ensure_scratch(ctx, SCR_HSI_BGR, (size_t)batch * npx_ * 3));
            bgr = (uint8_t *)ctx->scratch[SCR_HSI_BGR];
        }
        bv_balance_params rest = prm;
        rest.hsi_contrast_correct = 0;
        BalOutputs first;
        memset(&first, 0, sizeof(first));
        first.balanced = bgr;
        for (int k = 0; k < 3; ++k) first.hi[k] = 255;
        BV_TRY(balance_run(ctx, src, batch, height, width, rest, -1, first, stats_host, nullptr));
        BV_TRY(hsi_run(ctx, bgr, batch, npx_));
        if (out.converted || out.mask || out.mask_bits) {
            BalOutputs second = out;
            second.balanced = nullptr;
            BV_TRY(convert_run(ctx, bgr, batch, height, width, cvt_code, second));
        }
        return BV_OK;
    }
    const bool tiled = prm.horizontal_blocks != 1 || prm.vertical_blocks != 1;
    const size_t npx = (size_t)height * width;
    if (npx >= (1ull << 31)) {
        set_error("colour balance: frame too large for 32-bit histogram counters");
        return BV_ERR_INVALID;
    }
    const bool vec = all_vec(src, out, npx, batch);
    if (out.mask_bits && !(vec && width % 16 == 0)) {
        set_error("balance_run: bit-packed mask needs 16-byte aligned buffers and width %% 16 == 0");
        return BV_ERR_INVALID;
    }
    BV_TRY(ensure_scratch(ctx, SCR_BAL_STATE, sizeof(BalFrame) * (size_t)batch));
    BalFrame *st = (BalFrame *)ctx->scratch[SCR_BAL_STATE];
    BV_CUDA(cudaMemsetAsync(st, 0, sizeof(BalFrame) * (size_t)batch, ctx->stream));
    if (tiled) {
        BV_TRY(balance_run_tiled(ctx, src, batch, height, width, prm, cvt_code, out, st));
        if (stats_host) {
            BV_CUDA(cudaMemcpy2DAsync(stats_host, sizeof(bv_balance_stats), &st[0].stats, sizeof(BalFrame),
                                      sizeof(bv_balance_stats), batch, cudaMemcpyDeviceToHost, ctx->stream));
            BV_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        return BV_OK;
    }

    // pass 2 leaves H,S,V of every pixel in a scratch image for pass 3 (frame stride padded to 16 bytes)
    const size_t hsv_stride = (npx * 3 + 127) & ~(size_t)127;   // whole 128-byte lines per frame (discard_scratch_lines)
    uint8_t *hsv = nullptr;
    const uint16_t *ivl = nullptr;
    uint16_t *ivl_frames = nullptr;
    if (prm.hsv_contrast_correct) {
        BV_TRY(ensure_scratch(ctx, SCR_BAL_HSV, hsv_stride * (size_t)batch));
        hsv = (uint8_t *)ctx->scratch[SCR_BAL_HSV];
        // HSV inRange mask as the only output, whole 32-pixel groups per row: hue-interval table
        if (cvt_code == BV_BGR2HSV && !out.balanced && !out.converted && (out.mask || out.mask_bits) && vec && npx % 16 == 0 &&
            width % 32 == 0)
            BV_TRY(ivl_table(ctx, out.lo, out.hi, &ivl));
        if (ivl) {  // one composed copy per frame of the batch
            BV_TRY(ensure_scratch(ctx, SCR_IVL_FRAMES, (size_t)batch * kIvlBytes));
            ivl_frames = (uint16_t *)ctx->scratch[SCR_IVL_FRAMES];
        }
    }

    // chunk the batch so that one chunk's input stays in L2 across the three passes; chunks are
    // independent and alternate over side streams so that their passes overlap on the SMs
    int chunk = (int)(l2_chunk_bytes(ctx) / (npx * 3));
    // large frames (4K: 25 MB each): a launch over a single frame is mostly ramp-up and tail, which costs more
    // than the L2 misses of a bigger chunk (tools/tune_c5.py: 16.9 k vs 15.8 k frames/s at 3840x2160 with 4 frames);
    // when the stage hangs morphology + labelling behind every chunk (after_chunk), a short call is better off with two
    // or three frames per chunk so that all side streams have one (tools/c3_overlap.py: 8 frames, 19.8 k vs 18.5 k frames/s)
    int min_chunk = 4;
    if (after_chunk) {
        const int per_stream = (batch + side_streams(ctx) - 1) / side_streams(ctx);
        min_chunk = per_stream < 2 ? 2 : (per_stream > 4 ? 4 : per_stream);
    }
    if (chunk < min_chunk && ctx->opt[BV_OPT_L2_CHUNK_MB] <= 0) chunk = min_chunk;
    // long calls: twice the L2-sized chunk while every side stream still gets one -- the fixed cost of a launch (ramp, the
    // blocks' histogram merge, the last block's statistics) is paid half as often, which is worth more than the L2 hits
    // it costs (tools/side_sweep.py, 32 frames per call: fused mask stage 84.9 k -> 90.0 k frames/s, C2 68.3 k -> 69.1 k)
    if (ctx->opt[BV_OPT_L2_CHUNK_MB] <= 0 && (size_t)(2 * chunk) * npx * 3 <= ((size_t)80 << 20) &&
        batch >= 2 * chunk * side_streams(ctx))
        chunk *= 2;
    BV_TRY(for_chunks_on_side_streams(ctx, batch, chunk, [&](int f0, int nf) -> int {
        const uint8_t *csrc = src + (size_t)f0 * npx * 3;
        BalFrame *cst = st + f0;
        uint8_t *chsv = hsv ? hsv + (size_t)f0 * hsv_stride : nullptr;
        int bpf = (ctx->sm_count * hist_blocks_per_sm(ctx) + nf - 1) / nf;
        const size_t need = (npx / 16 + kBalThreads - 1) / kBalThreads;
        if ((size_t)bpf > need) bpf = (int)(need ? need : 1);
        dim3 grid(bpf, nf);
        if (vec)
            BV_LAUNCH(ctx, hist_bgr_kernel<true>, grid, kBalThreads, 0, csrc, cst, npx, prm, ctx->d_pow_quarter);
        else
            BV_LAUNCH(ctx, hist_bgr_kernel<false>, grid, kBalThreads, 0, csrc, cst, npx, prm, ctx->d_pow_quarter);
        if (prm.hsv_contrast_correct) {
            if (vec)
                BV_LAUNCH_PDL(ctx, hist_sv_kernel<true>, grid, kBalThreads, 0, csrc, cst, npx, chsv, hsv_stride);
            else
                BV_LAUNCH_PDL(ctx, hist_sv_kernel<false>, grid, kBalThreads, 0, csrc, cst, npx, chsv, hsv_stride);
        }
        BalOutputs co = out;
        if (co.balanced) co.balanced += (size_t)f0 * npx * 3;
        if (co.converted) co.converted += (size_t)f0 * npx * (cvt_code == BV_BGR2GRAY ? 1 : 3);
        if (co.mask) co.mask += (size_t)f0 * npx;
        if (co.mask_bits) co.mask_bits += (size_t)f0 * height * (((width + 31) / 32) * 2);
        if (ivl)
            BV_TRY(launch_mask_from_hsv(ctx, chsv, hsv_stride, cst, nf, npx, width, ivl, ivl_frames + (size_t)f0 * kIvlEntries, co));
        else if (prm.hsv_contrast_correct)
            BV_TRY(dispatch_final<3>(ctx, chsv, hsv_stride, cst, nf, npx, width, cvt_code, co, vec));
        else
            BV_TRY(dispatch_final<1>(ctx, csrc, npx * 3, cst, nf, npx, width, cvt_code, co, vec));
        if (after_chunk) BV_TRY(after_chunk->fn(after_chunk->self, ctx, f0, nf));
        return BV_OK;
    }));
    if (stats_host) {
        BV_CUDA(cudaMemcpy2DAsync(stats_host, sizeof(bv_balance_stats), &st[0].stats, sizeof(BalFrame),
                                  sizeof(bv_balance_stats), batch, cudaMemcpyDeviceToHost, ctx->stream));
        BV_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    return BV_OK;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_color_balance(bv_ctx *ctx, const uint8_t *src_dev, uint8_t *dst_dev, int batch, int height, int width,
                                const bv_balance_params *params, bv_balance_stats *stats_host) {
    BV_REQUIRE(ctx && src_dev && dst_dev && params, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_CUDA(cudaSetDevice(ctx->device));
    BalOutputs out;
    memset(&out, 0, sizeof(out));
    out.balanced = dst_dev;
    for (int k = 0; k < 3; ++k) out.hi[k] = 255;
    return balance_run(ctx, src_dev, batch, height, width, *params, -1, out, stats_host);
}
