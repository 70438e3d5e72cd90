// ccl.cu -- 8-connected component labelling with per-blob raster moments, on bit-packed masks.
//
// Role in the reference: blob extraction after threshold + morphology, i.e. outer_contours +
// contour_centroid + contour_area (utils/feature.py:5-21,240-265; modules/bins.py:27,
// modules/red_buoy.py:38-44).  The reference uses cv2.findContours + polygon moments; the
// labelling form computed here has the declared oracle cv2.connectedComponentsWithStats(8) +
// cv2.moments(binaryImage=True) with labels in first-pixel raster order (SURVEY.md 8c).
//
// Algorithm (union-find over word runs):
//   nodes   = maximal runs of set bits inside one 32-px word; a node's id is the pixel index of its
//             first pixel, and `parent[]` is only ever touched at those sparse positions
//   init    parent[node] = node
//   merge   each word unions its runs with (a) the run ending at bit 31 of the word to the left,
//           (b) every run of the row above that touches the run's 3-neighbourhood, found with
//           bit tricks on a 34-bit window; unions link the larger root under the smaller with
//           atomicMin, so a component's root is its first pixel in raster order
//   count   compress every node to its root, count roots per row
//   scan    exclusive scan of the row counts per frame -> number of blobs
//   rank    roots receive 1, 2, 3... in raster order; stored negated in parent[root]
//   final   each word looks its runs' labels up, writes 32 int32 labels, and accumulates closed-form
//           run moments (sum of x^k over a run is a polynomial in its end points) with a warp
//           segmented reduction over equal labels, then one set of 64-bit atomics per segment
//
// HBM traffic: mask bits (1/8 B/px) are re-read from L2; the label image is written once (4 B/px);
// parent[] traffic is proportional to the number of runs, not pixels.
#include "morph.cuh"

namespace bv {

__device__ __forceinline__ int find_compress(int *parent, int a) {
    const int a0 = a;
    int p = parent[a];
    while (p != a) {
        a = p;
        p = parent[a];
    }
    if (a != a0) atomicMin(&parent[a0], a);
    return a;
}

__device__ void union_nodes(int *parent, int a, int b) {
    bool done;
    do {
        a = find_compress(parent, a);
        b = find_compress(parent, b);
        if (a < b) {
            const int old = atomicMin(&parent[b], a);
            done = (old == b);
            b = old;
        } else if (b < a) {
            const int old = atomicMin(&parent[a], b);
            done = (old == a);
            a = old;
        } else {
            done = true;
        }
    } while (!done);
}

__global__ void __launch_bounds__(256) ccl_init_kernel(const uint32_t *__restrict__ bits, int *__restrict__ parent,
                                                       int height, int width, int wpr, uint32_t total_words) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const uint32_t w = bits[i];
        if (!w) continue;
        const WordPos wp = word_pos(i, wpr, height);
        int *fp = parent + (size_t)(wp.row - wp.y) * width;  // this frame's parent array
        uint32_t starts = w & ~(w << 1);
        while (starts) {
            const int s = __ffs(starts) - 1;
            starts &= starts - 1;
            const int node = wp.y * width + wp.wx * 32 + s;
            fp[node] = node;
        }
    }
}

template <bool CONN8>
__global__ void __launch_bounds__(256) ccl_merge_kernel(const uint32_t *__restrict__ bits, int *__restrict__ parent,
                                                        int height, int width, int wpr, uint32_t total_words) {
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        const uint32_t w = bits[i];
        if (!w) continue;
        const WordPos wp = word_pos(i, wpr, height);
        int *fp = parent + (size_t)(wp.row - wp.y) * width;
        const int xbase = wp.wx * 32;
        // (a) continuation of the previous word's last run
        if ((w & 1u) && wp.wx > 0) {
            const uint32_t pw = bits[i - 1];
            if (pw >> 31) union_nodes(fp, wp.y * width + xbase, wp.y * width + xbase - 32 + run_start(pw, 31));
        }
        if (wp.y == 0) continue;
        // (b) row above, 34-bit window: bit k <-> x = xbase + k - 1
        const uint32_t up = bits[i - wpr];
        // 4-connectivity (background regions of an 8-connected foreground) has no diagonal contacts
        const uint32_t upl = (CONN8 && wp.wx > 0) ? bits[i - wpr - 1] : 0u;
        const uint32_t upr = (CONN8 && wp.wx < wpr - 1) ? bits[i - wpr + 1] : 0u;
        const unsigned long long U = ((unsigned long long)up << 1) | (unsigned long long)(upl >> 31) |
                                     ((unsigned long long)(upr & 1u) << 33);
        if (!U) continue;
        const int up_row = (wp.y - 1) * width;
        uint32_t starts = w & ~(w << 1);
        while (starts) {
            const int s = __ffs(starts) - 1;
            starts &= starts - 1;
            const uint32_t above_s = w >> s;                       // run from bit s
            const int len = __ffs(~above_s) - 1;                   // ~above_s != 0 unless run spans to bit 31
            const int e = (len < 0) ? 31 : s + len - 1;            // __ffs(0) = 0 -> len = -1
            // run occupies window bits s+1..e+1; its 8-neighbourhood above is s..e+2 (4-conn: s+1..e+1)
            const int nb = CONN8 ? e - s + 3 : e - s + 1;
            const unsigned long long dil = ((nb >= 64) ? ~0ull : ((1ull << nb) - 1ull)) << (CONN8 ? s : s + 1);
            unsigned long long T = U & dil;
            const int node = wp.y * width + xbase + s;
            while (T) {
                const int k = __ffsll((long long)T) - 1;           // first bit of a touching run
                // clear this touching run from T
                const unsigned long long from_k = T >> k;
                const int rl = __ffsll((long long)~from_k) - 1;    // length of ones starting at k (<= 34)
                T &= ~(((1ull << rl) - 1ull) << k);
                int other;
                if (k == 0)
                    other = up_row + xbase - 32 + run_start(upl, 31);
                else if (k == 33)
                    other = up_row + xbase + 32;                   // bit 0 of the next word starts a run
                else
                    other = up_row + xbase + run_start(up, k - 1);
                // a run of `up` reaching bit 0 may continue from the previous word; the horizontal
                // union (a) of the row above already ties those nodes together
                union_nodes(fp, node, other);
            }
        }
    }
}

// one warp per row: compress every node of the row to its root, count the roots
__global__ void __launch_bounds__(256) ccl_count_kernel(const uint32_t *__restrict__ bits, int *__restrict__ parent,
                                                        int *__restrict__ row_count, int height, int width, int wpr,
                                                        size_t total_rows) {
    const int lane = threadIdx.x & 31;
    const size_t warp0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t row = warp0; row < total_rows; row += nwarps) {
        const int y = (int)(row % height);
        int *fp = parent + (row - y) * (size_t)width;
        int cnt = 0;
        for (int wx = lane; wx < wpr; wx += 32) {
            const uint32_t w = bits[row * wpr + wx];
            uint32_t starts = w & ~(w << 1);
            while (starts) {
                const int s = __ffs(starts) - 1;
                starts &= starts - 1;
                const int node = y * width + wx * 32 + s;
                const int r = find_root(fp, node);
                if (r == node)
                    ++cnt;
                else
                    fp[node] = r;
            }
        }
        cnt = __reduce_add_sync(0xFFFFFFFFu, cnt);
        if (lane == 0) row_count[row] = cnt;
    }
}

// one block per frame: exclusive scan of the row counts; then the frame's blob table entries are cleared (the block knows
// the count it has just produced: no separate launch)
__global__ void __launch_bounds__(1024) ccl_scan_kernel(const int *__restrict__ row_count, int *__restrict__ row_off,
                                                        int *__restrict__ n_blobs, int height, bv_blob *__restrict__ blobs,
                                                        int max_blobs, int width) {
    __shared__ int warp_sums[32];
    __shared__ int carry;
    const int f = blockIdx.x;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < height; base += blockDim.x) {
        const int y = base + threadIdx.x;
        const int v = y < height ? row_count[(size_t)f * height + y] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) warp_sums[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            int ws = warp_sums[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int o = __shfl_up_sync(0xFFFFFFFFu, ws, d);
                if (lane >= d) ws += o;
            }
            warp_sums[lane] = ws;  // inclusive over warps
        }
        __syncthreads();
        const int before = carry + (wid ? warp_sums[wid - 1] : 0) + incl - v;
        if (y < height) row_off[(size_t)f * height + y] = before;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) n_blobs[f] = carry;
    if (blobs) {
        const int n = min(carry, max_blobs);   // carry is final: the loop ended with a barrier
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            bv_blob b;
            b.m00 = b.m10 = b.m01 = b.m20 = b.m11 = b.m02 = b.m30 = b.m21 = b.m12 = b.m03 = 0;
            b.x0 = width;
            b.y0 = height;
            b.x1 = -1;
            b.y1 = -1;
            blobs[(size_t)f * max_blobs + i] = b;
        }
    }
}

// bit `node` of frame f's frame-touching bitmap (bg_outer_kernel)
__device__ __forceinline__ bool is_outer(const uint32_t *outer, int height, int width, size_t f, int node) {
    const size_t words_per_frame = ((size_t)height * width + 31) / 32;
    return (outer[f * words_per_frame + (node >> 5)] >> (node & 31)) & 1u;
}

// one warp per row: number the roots of the row in raster order, store -(label) in parent[root].  SKIP_OUTER: roots
// marked in the frame-touching bitmap `outer` (bg_outer_kernel) are left alone and get no number (they keep parent[root]
// == root)
template <bool SKIP_OUTER>
__global__ void __launch_bounds__(256) ccl_rank_kernel(const uint32_t *__restrict__ bits, int *__restrict__ parent,
                                                       const int *__restrict__ row_off, int height, int width, int wpr,
                                                       size_t total_rows, int *__restrict__ root_px, int max_roots,
                                                       const uint32_t *__restrict__ outer) {
    const int lane = threadIdx.x & 31;
    const size_t warp0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t row = warp0; row < total_rows; row += nwarps) {
        const int y = (int)(row % height);
        int *fp = parent + (row - y) * (size_t)width;
        int *frame_roots = root_px ? root_px + ((row - y) / height) * (size_t)max_roots : nullptr;
        int next = row_off[row];  // labels handed out so far (0-based rank of the next root)
        for (int wbase = 0; wbase < wpr; wbase += 32) {
            const int wx = wbase + lane;
            const uint32_t w = wx < wpr ? bits[row * wpr + wx] : 0u;
            uint32_t starts = w & ~(w << 1);
            uint32_t roots = 0;
            for (uint32_t s_it = starts; s_it;) {
                const int s = __ffs(s_it) - 1;
                s_it &= s_it - 1;
                const int node = y * width + wx * 32 + s;
                if (fp[node] == node && !(SKIP_OUTER && is_outer(outer, height, width, (row - y) / height, node)))
                    roots |= 1u << s;
            }
            const int c = __popc(roots);
            int incl = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
                if (lane >= d) incl += o;
            }
            int rank = next + incl - c;
            while (roots) {
                const int s = __ffs(roots) - 1;
                roots &= roots - 1;
                fp[y * width + wx * 32 + s] = -(rank + 1);
                if (frame_roots && rank < max_roots) frame_roots[rank] = y * width + wx * 32 + s;
                ++rank;
            }
            next += __shfl_sync(0xFFFFFFFFu, incl, 31);
        }
    }
}

// sum_{x=a}^{b} x^k, k = 0..3, in closed form (exact in 64-bit for any image size that fits 32-bit pixel indices)
__device__ __forceinline__ void run_power_sums(int a, int b, int &n, int &s1, long long &s2, long long &s3) {
    const long long A = a, B = b, Am = A - 1;
    n = b - a + 1;
    s1 = (int)((A + B) * (long long)n / 2);            // <= 32 * 65535 per run
    // S2(k) = k(k+1)(2k+1)/6, S3(k) = (k(k+1)/2)^2
    s2 = B * (B + 1) * (2 * B + 1) / 6 - Am * (Am + 1) * (2 * Am + 1) / 6;
    const long long tb = B * (B + 1) / 2, ta = Am * (Am + 1) / 2;
    s3 = tb * tb - ta * ta;
}

// the ten raster moments of a set of pixels of ONE row y from the power sums of their x
__device__ __forceinline__ void row_moments(int n, int s1, long long s2, long long s3, int y, unsigned long long (&m)[10]) {
    const long long Y = y, N = n, S1 = s1;
    m[0] = (unsigned long long)N;                // m00
    m[1] = (unsigned long long)S1;               // m10
    m[2] = (unsigned long long)(Y * N);          // m01
    m[3] = (unsigned long long)s2;               // m20
    m[4] = (unsigned long long)(Y * S1);         // m11
    m[5] = (unsigned long long)(Y * Y * N);      // m02
    m[6] = (unsigned long long)s3;               // m30
    m[7] = (unsigned long long)(Y * s2);         // m21
    m[8] = (unsigned long long)(Y * Y * S1);     // m12
    m[9] = (unsigned long long)(Y * Y * Y * N);  // m03
}

// per-warp accumulator of the blob the warp currently "carries" (shared memory: no registers, no shuffles)
struct WarpAcc {
    unsigned long long m[10];
    int box[4];   // x0, y0, x1, y1
};

__device__ __forceinline__ void acc_reset(WarpAcc &a, int lane) {
    if (lane < 10) a.m[lane] = 0;
    else if (lane < 14) a.box[lane - 10] = (lane < 12) ? 0x7FFFFFFF : -1;
}

// all lanes of the warp: add the accumulator to its blob (one atomic per non-zero field) and clear it
__device__ __forceinline__ void acc_flush(WarpAcc &a, bv_blob *blobs, int max_blobs, long long key, int lane) {
    __syncwarp();
    if (key != 0) {
        bv_blob *b = &blobs[(size_t)(key >> 32) * max_blobs + ((int)(key & 0xFFFFFFFFll) - 1)];
        if (lane < 10) {
            const unsigned long long v = a.m[lane];
            if (v) atomicAdd(reinterpret_cast<unsigned long long *>(&b->m00) + lane, v);
        } else if (lane < 12) {
            atomicMin(&b->x0 + (lane - 10), a.box[lane - 10]);
        } else if (lane < 14) {
            atomicMax(&b->x0 + (lane - 10), a.box[lane - 10]);
        }
    }
    acc_reset(a, lane);
    __syncwarp();
}

// final: labels + moments.  All 32 lanes of a warp stay in the loop together (the segmented reduction uses full-warp
// shuffles).  A lane owns one 32-px word; its 32 labels are staged in a padded shared-memory tile (row = lane,
// bank-conflict-free) and the warp then writes the 32 words out row by row, so every store instruction covers 128
// contiguous bytes of the label image.
// Moments: the pixels a warp sees of one blob in one step lie on one row (the segment key contains the row), so only the
// four power sums of x (n, sum x, sum x^2, sum x^3) go through the segmented reduction -- 6 registers per shuffle level
// instead of the 20 of ten 64-bit moments -- and the segment head multiplies by the powers of y.  The blob with the most
// pixels in the step is "carried": its segments are added (shared-memory atomics) into the warp's accumulator and reach
// the table with one set of global atomics when another blob takes over or the kernel ends, so a blob that covers much
// of the frame costs a handful of atomic sets per WARP instead of one per 1024-pixel segment (they all hit the same
// addresses and serialise in L2).  Everything else goes to the table directly.
__global__ void __launch_bounds__(256, 4) ccl_final_kernel(const uint32_t *__restrict__ bits, const int *__restrict__ parent,
                                                           int *__restrict__ labels, bv_blob *__restrict__ blobs,
                                                           int max_blobs, int height, int width, int wpr,
                                                           uint32_t total_words) {
    __shared__ int tile[8][32][33];
    __shared__ WarpAcc accs[8];
    const int lane = threadIdx.x & 31;
    const bool full_words = (width & 31) == 0;
    int(*my_tile)[33] = tile[threadIdx.x >> 5];
    WarpAcc &acc = accs[threadIdx.x >> 5];
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t rounded = (total_words + 31u) / 32u * 32u;
    long long carry_key = 0;  // (frame << 32) | label of the blob this warp accumulates; warp-uniform
    acc_reset(acc, lane);
    __syncwarp();
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < rounded; i += stride) {
        const bool valid = i < total_words;
        const uint32_t w = valid ? bits[i] : 0u;
        const uint32_t warp_first = i - lane;  // word index owned by lane 0
        if (!__any_sync(0xFFFFFFFFu, w != 0)) {
            // empty warp (the common case on sparse masks): 4 KB of zeros, 128-bit coalesced stores
            if (!labels) continue;
            if (full_words && warp_first + 32 <= total_words) {
                int4 *base = reinterpret_cast<int4 *>(labels + (size_t)warp_first * 32);
#pragma unroll
                for (int k = 0; k < 8; ++k) base[k * 32 + lane] = make_int4(0, 0, 0, 0);
                continue;
            }
        }
        const WordPos wp = word_pos(valid ? i : 0, wpr, height);
        const uint32_t frame = (wp.row - wp.y) / (uint32_t)height;
        const int *fp = parent + (size_t)(wp.row - wp.y) * width;
        const int xbase = wp.wx * 32;
        uint32_t rest = w;
        int written = 0;  // pixels of this word already staged
        while (__any_sync(0xFFFFFFFFu, rest != 0)) {
            int lab = 0, n = 0, s1 = 0, xa = 0, xb = 0;
            long long s2 = 0, s3 = 0;
            if (rest) {
                const int s = __ffs(rest) - 1;
                const uint32_t from_s = rest >> s;
                const int len_raw = __ffs(~from_s) - 1;
                const int e = (len_raw < 0) ? 31 : s + len_raw - 1;
                rest &= (e == 31) ? 0u : ~((2u << e) - 1u);
                const int node = wp.y * width + xbase + s;
                const int v = fp[node];
                lab = v < 0 ? -v : -fp[v];
                if (labels) {
                    for (int x = written; x < s; ++x) my_tile[lane][x] = 0;
                    for (int x = s; x <= e; ++x) my_tile[lane][x] = lab;
                    written = e + 1;
                }
                xa = xbase + s;
                xb = xbase + e;
                if (blobs) run_power_sums(xa, xb, n, s1, s2, s3);
            }
            if (blobs) {
                // segmented reduction over consecutive lanes with the same (row, label)
                const long long key = lab ? ((long long)wp.row << 32) | (unsigned)lab : -(long long)lane - 1;
                const long long prev = __shfl_up_sync(0xFFFFFFFFu, key, 1);
                const bool head = lane == 0 || prev != key;
                const unsigned heads = __ballot_sync(0xFFFFFFFFu, head);
                const unsigned above = (lane == 31) ? 0u : (heads & ~((2u << lane) - 1u));
                const int seg_end = above ? __ffs(above) - 2 : 31;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const bool take = lane + d <= seg_end;
                    const int on = __shfl_down_sync(0xFFFFFFFFu, n, d), o1 = __shfl_down_sync(0xFFFFFFFFu, s1, d);
                    const long long o2 = __shfl_down_sync(0xFFFFFFFFu, s2, d), o3 = __shfl_down_sync(0xFFFFFFFFu, s3, d);
                    if (take) {
                        n += on;
                        s1 += o1;
                        s2 += o2;
                        s3 += o3;
                    }
                }
                const int x_last = __shfl_sync(0xFFFFFFFFu, xb, seg_end);   // lanes ascend in x inside a row
                const bool counted = head && lab && lab <= max_blobs;
                const long long fkey = ((long long)frame << 32) | (unsigned)lab;
                // the segment with the most pixels in this step designates the carried blob
                int best = counted ? n : 0;
                long long best_key = counted ? fkey : 0;
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    const int ob = __shfl_xor_sync(0xFFFFFFFFu, best, d);
                    const long long ok = __shfl_xor_sync(0xFFFFFFFFu, best_key, d);
                    if (ob > best || (ob == best && ok > best_key)) {
                        best = ob;
                        best_key = ok;
                    }
                }
                if (best_key != 0) {   // warp-uniform
                    if (best_key != carry_key) {
                        acc_flush(acc, blobs, max_blobs, carry_key, lane);
                        carry_key = best_key;
                    }
                    if (counted) {
                        unsigned long long m[10];
                        row_moments(n, s1, s2, s3, wp.y, m);
                        if (fkey == carry_key) {
#pragma unroll
                            for (int k = 0; k < 10; ++k) atomicAdd(&acc.m[k], m[k]);
                            atomicMin(&acc.box[0], xa);
                            atomicMin(&acc.box[1], wp.y);
                            atomicMax(&acc.box[2], x_last);
                            atomicMax(&acc.box[3], wp.y);
                        } else {
                            bv_blob *b = &blobs[frame * (size_t)max_blobs + (lab - 1)];
                            unsigned long long *bm = reinterpret_cast<unsigned long long *>(&b->m00);
#pragma unroll
                            for (int k = 0; k < 10; ++k) atomicAdd(bm + k, m[k]);
                            atomicMin(&b->x0, xa);
                            atomicMin(&b->y0, wp.y);
                            atomicMax(&b->x1, x_last);
                            atomicMax(&b->y1, wp.y);
                        }
                    }
                }
            }
        }
        if (labels) {
            for (int x = written; x < 32; ++x) my_tile[lane][x] = 0;
            __syncwarp();
            if (full_words) {  // width % 32 == 0: the label image is linear in the word index
                int *base = labels + (size_t)warp_first * 32;
                const int nk = min(32u, total_words - warp_first);
#pragma unroll 4
                for (int k = 0; k < nk; ++k) base[k * 32 + lane] = my_tile[k][lane];
            } else {
#pragma unroll 4
                for (int k = 0; k < 32; ++k) {
                    const uint32_t wi = warp_first + k;
                    if (wi >= total_words) break;
                    const int kwx = (int)(wi % (uint32_t)wpr);
                    const uint32_t krow = wi / (uint32_t)wpr;
                    const int x = kwx * 32 + lane;
                    if (x < width) labels[(size_t)krow * width + x] = my_tile[k][lane];
                }
            }
            __syncwarp();
        }
    }
    if (blobs) acc_flush(acc, blobs, max_blobs, carry_key, lane);
}

// node (pixel index of the run start) of the set pixel (y, x) in a bit image
__device__ __forceinline__ int node_of(const uint32_t *frame_bits, int wpr, int width, int y, int x) {
    const uint32_t w = frame_bits[(size_t)y * wpr + (x >> 5)];
    return y * width + (x & ~31) + run_start(w, x & 31);
}

// mark the background regions that touch the image frame: outer[root >> 5] |= 1 << (root & 31).  UNCOUNT: also take
// every newly marked root off its row's root count, so that the scan and rank steps number only the holes
template <bool UNCOUNT>
__global__ void __launch_bounds__(256) bg_outer_kernel(const uint32_t *__restrict__ inv, const int *__restrict__ parent,
                                                       uint32_t *__restrict__ outer, int height, int width, int wpr,
                                                       int batch, int *__restrict__ row_count) {
    const int per_frame = 2 * width + 2 * height;
    const size_t total = (size_t)per_frame * batch;
    const size_t words_per_frame = ((size_t)height * width + 31) / 32;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int f = (int)(i / per_frame);
        int k = (int)(i - (size_t)f * per_frame), x, y;
        if (k < width) { y = 0; x = k; }
        else if (k < 2 * width) { y = height - 1; x = k - width; }
        else if (k < 2 * width + height) { x = 0; y = k - 2 * width; }
        else { x = width - 1; y = k - 2 * width - height; }
        const uint32_t *fb = inv + (size_t)f * height * wpr;
        if (!((fb[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u)) continue;
        const int *fp = parent + (size_t)f * height * width;
        const int node = node_of(fb, wpr, width, y, x);
        const int p = fp[node];
        const int root = p;  // nodes were compressed to their root by ccl_count_kernel (roots point to themselves)
        const uint32_t old = atomicOr(&outer[(size_t)f * words_per_frame + (root >> 5)], 1u << (root & 31));
        if (UNCOUNT && !(old & (1u << (root & 31)))) atomicSub(&row_count[(size_t)f * height + root / width], 1);
    }
}

// Scratch of the labelling for a batch of `batch` frames; frames f0.. of the batch use the slices at f0 (label_scratch_slice),
// so that independent chunks of one batch can be labelled concurrently on different streams.
int label_scratch(bv_ctx *ctx, int batch, int height, int width, LabelScratch *ls) {
    const size_t total_rows = (size_t)batch * height;
    BV_TRY(ensure_scratch(ctx, SCR_CCL_PARENT, total_rows * width * sizeof(int)));
    BV_TRY(ensure_scratch(ctx, SCR_CCL_AUX, (total_rows * 2 + batch) * sizeof(int)));
    ls->parent = (int *)ctx->scratch[SCR_CCL_PARENT];
    ls->row_count = (int *)ctx->scratch[SCR_CCL_AUX];
    ls->row_off = ls->row_count + total_rows;
    ls->n_fallback = ls->row_off + total_rows;
    return BV_OK;
}

static LabelScratch label_scratch_slice(const LabelScratch &ls, int f0, int height, int width) {
    LabelScratch s;
    s.parent = ls.parent + (size_t)f0 * height * width;
    s.row_count = ls.row_count + (size_t)f0 * height;
    s.row_off = ls.row_off + (size_t)f0 * height;
    s.n_fallback = ls.n_fallback + f0;
    return s;
}

static int label_bits_ex(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int batch, int height, int width,
                         bv_blob *blobs, int max_blobs, int32_t *n_blobs, int *root_px, int max_roots, const LabelScratch &sc,
                         uint32_t *outer = nullptr);

int union_bits(bv_ctx *ctx, const uint32_t *bits, int batch, int height, int width, const LabelScratch &ls) {
    const int wpr = words_per_row(width);
    const size_t total_words = (size_t)batch * height * wpr;
    const int gw = grid_for(ctx, total_words, 256, 8);
    BV_LAUNCH(ctx, ccl_init_kernel, gw, 256, 0, bits, ls.parent, height, width, wpr, (uint32_t)total_words);
    BV_LAUNCH(ctx, ccl_merge_kernel<true>, gw, 256, 0, bits, ls.parent, height, width, wpr, (uint32_t)total_words);
    return BV_OK;
}

int label_bits(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int batch, int height, int width, bv_blob *blobs,
               int max_blobs, int32_t *n_blobs) {
    LabelScratch ls;
    BV_TRY(label_scratch(ctx, batch, height, width, &ls));
    return label_bits_ex(ctx, bits, labels, batch, height, width, blobs, max_blobs, n_blobs, nullptr, 0, ls);
}

// frames f0 .. f0 + nf - 1 of a batch whose scratch is `ls`; every pointer argument already points at frame f0
int label_bits_slice(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int f0, int nf, int height, int width, bv_blob *blobs,
                     int max_blobs, int32_t *n_blobs, const LabelScratch &ls) {
    return label_bits_ex(ctx, bits, labels, nf, height, width, blobs, max_blobs, n_blobs, nullptr, 0,
                         label_scratch_slice(ls, f0, height, width));
}

// Foreground (`outer` == NULL): 8-connected components of `bits`.  Background (`outer` != NULL): `bits` is the inverted
// mask and its regions are 4-connected (the background of an 8-connected foreground); the regions that touch the image
// frame are marked in the bitmap `outer` (batch x ceil(H*W / 32) words) and, when `root_px` is given, the other regions
// -- the holes -- are counted and numbered in raster order of their first pixel, frame-touching regions skipped.
static int label_bits_ex(bv_ctx *ctx, const uint32_t *bits, int32_t *labels, int batch, int height, int width,
                         bv_blob *blobs, int max_blobs, int32_t *n_blobs, int *root_px, int max_roots, const LabelScratch &sc,
                         uint32_t *outer) {
    const int wpr = words_per_row(width);
    const size_t total_words = (size_t)batch * height * wpr;
    const size_t total_rows = (size_t)batch * height;
    if ((size_t)height * width >= (1ull << 31) || total_words >= (1ull << 31)) {
        set_error("bv_label: frame or batch too large for 32-bit indices");
        return BV_ERR_INVALID;
    }
    int *parent = sc.parent;
    int *row_count = sc.row_count;
    int *row_off = sc.row_off;
    int *nb = n_blobs ? n_blobs : sc.n_fallback;
    const int gw = grid_for(ctx, total_words, 256, 8);
    const int gr = grid_for(ctx, total_rows * 32, 256, 8);
    BV_LAUNCH(ctx, ccl_init_kernel, gw, 256, 0, bits, parent, height, width, wpr, (uint32_t)total_words);
    if (outer) {
        const bool holes = root_px != nullptr;
        BV_LAUNCH(ctx, ccl_merge_kernel<false>, gw, 256, 0, bits, parent, height, width, wpr, (uint32_t)total_words);
        BV_LAUNCH(ctx, ccl_count_kernel, gr, 256, 0, bits, parent, row_count, height, width, wpr, total_rows);
        BV_CUDA(cudaMemsetAsync(outer, 0, (size_t)batch * (((size_t)height * width + 31) / 32) * 4, ctx->stream));
        const int ge = grid_for(ctx, (size_t)batch * (2 * width + 2 * height), 256, 8);
        if (!holes) {
            BV_LAUNCH(ctx, bg_outer_kernel<false>, ge, 256, 0, bits, parent, outer, height, width, wpr, batch, nullptr);
            return BV_OK;
        }
        BV_LAUNCH(ctx, bg_outer_kernel<true>, ge, 256, 0, bits, parent, outer, height, width, wpr, batch, row_count);
        BV_LAUNCH(ctx, ccl_scan_kernel, batch, 1024, 0, row_count, row_off, nb, height, nullptr, 0, width);
        BV_LAUNCH(ctx, ccl_rank_kernel<true>, gr, 256, 0, bits, parent, row_off, height, width, wpr, total_rows, root_px,
                  max_roots, outer);
        return BV_OK;
    }
    BV_LAUNCH(ctx, ccl_merge_kernel<true>, gw, 256, 0, bits, parent, height, width, wpr, (uint32_t)total_words);
    BV_LAUNCH(ctx, ccl_count_kernel, gr, 256, 0, bits, parent, row_count, height, width, wpr, total_rows);
    BV_LAUNCH(ctx, ccl_scan_kernel, batch, 1024, 0, row_count, row_off, nb, height, (max_blobs > 0 ? blobs : nullptr), max_blobs, width);
    BV_LAUNCH(ctx, ccl_rank_kernel<false>, gr, 256, 0, bits, parent, row_off, height, width, wpr, total_rows, root_px, max_roots,
              nullptr);
    if (labels || (blobs && max_blobs > 0))
        BV_LAUNCH(ctx, ccl_final_kernel, gw, 256, 0, bits, parent, labels, (max_blobs > 0 ? blobs : nullptr), max_blobs,
                  height, width, wpr, (uint32_t)total_words);
    return BV_OK;
}

// ----------------------------------------------------------------------------------------------
// Outer borders as cv2.findContours(RETR_EXTERNAL) follows them, with the Green's-theorem sums of
// cv2.moments(contour) -- the literal reference path outer_contours -> contour_centroid /
// contour_area (utils/feature.py:5-21,240-265), SURVEY.md 8f rank 1.
//
//  * the start pixel of a component's outer border is its first pixel in raster order, i.e. the
//    union-find root that the labelling already produces;
//  * RETR_EXTERNAL drops components that lie inside a hole of another one: a component is external
//    iff the background left of its start pixel belongs to a (4-connected) background region that
//    reaches the image frame; background regions are labelled with the same union-find machinery
//    on the inverted mask and the frame-touching ones are marked in a bitmap;
//  * one thread walks one border with Suzuki's 8-neighbour rule (clockwise search for the first
//    neighbour, then counter-clockwise from the direction it came from) and accumulates
//    a00 = sum(x' y - x y'), a10 = sum(dxy (x' + x)), a01 = sum(dxy (y' + y)) in int64: exact, and
//    independent of CHAIN_APPROX_SIMPLE (collinear points split a term into equal parts).
//
// Hole borders and the hierarchy (bv_find_contours, RETR_LIST / CCOMP / TREE): the background
// regions that do not reach the frame are the holes; the same count / scan / rank steps number
// them in raster order of their first pixel.  A hole border starts at the pixel left of the hole's
// first pixel and is followed by the same walk; the hole that encloses an outer border is the one
// left of its start pixel, and the component that encloses a hole border owns its start pixel.
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) invert_bits_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst,
                                                          int width, int wpr, uint32_t total_words) {
    const int tail = width - (wpr - 1) * 32;
    const uint32_t tail_mask = tail == 32 ? 0xFFFFFFFFu : ((1u << tail) - 1u);
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total_words; i += stride) {
        uint32_t w = ~src[i];
        if ((int)(i % (uint32_t)wpr) == wpr - 1) w &= tail_mask;
        dst[i] = w;
    }
}

// Copy of the bit mask laid out for the border walk.  Word (w, y + 1) holds the pixels 30w-1 .. 30w+30 of row y: 30 own
// pixels and one neighbour on either side, zero outside the frame, so the three pixels x-1, x, x+1 always sit in one
// word (no word-edge cases in the walk); rows -1 and `height` are stored as zero rows (no row checks either); and the
// words of one 30-pixel column are contiguous in y, so the rows y-1, y, y+1 are three adjacent words and a walk stays
// inside one 128-byte line for 32 rows.  A lone warp issues dependent instructions every ~5 cycles, so the walk is
// bound by the instruction count of one step, which this layout roughly halves.
constexpr unsigned kWalkPixelsPerWord = 30;

__global__ void __launch_bounds__(256) walk_bits_kernel(const uint32_t *__restrict__ bits, uint32_t *__restrict__ walk,
                                                        int height, int width, int wpr, int wcols, uint32_t total) {
    const uint32_t rows = (uint32_t)height + 2, per_frame = (uint32_t)wcols * rows;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const uint32_t f = i / per_frame, r = i - f * per_frame;
        const uint32_t w = r / rows;
        const int y = (int)(r - w * rows) - 1;
        uint32_t v = 0;
        if (y >= 0 && y < height) {
            const uint32_t *row = bits + ((size_t)f * height + y) * wpr;
            const int p = (int)(kWalkPixelsPerWord * w) - 1;  // first pixel of the word
            if (p < 0) {
                v = row[0] << 1;
            } else {
                const int i0 = p >> 5;
                v = __funnelshift_r(row[i0], i0 + 1 < wpr ? row[i0 + 1] : 0u, p & 31);
            }
            const int valid = width - p;  // >= 2
            if (valid < 32) v &= (1u << valid) - 1u;
        }
        walk[i] = v;
    }
}

// the 8 neighbours of (x, y) as a mask over the direction codes 0..7 = E, NE, N, NW, W, SW, S, SE
__device__ __forceinline__ uint32_t neighbours_at(const uint32_t *__restrict__ fw, unsigned rows, int x, int y) {
    const unsigned w = (unsigned)x / kWalkPixelsPerWord, sh = (unsigned)x - kWalkPixelsPerWord * w;
    const uint32_t *p = fw + (w * rows + (unsigned)y);  // rows are stored shifted down by one: p[0] is row y-1
    const uint32_t top = (p[0] >> sh) & 7u, mid = (p[1] >> sh) & 7u, bot = (p[2] >> sh) & 7u;
    return (mid >> 2) | ((__brev(top) >> 29) << 1) | ((mid & 1u) << 4) | (bot << 5);
}

constexpr int kContourLaneStride = 4;
constexpr int kChunkPoints = 31;                  // vertices per chunk
constexpr int kChunkInts = 2 * kChunkPoints + 2;  // + index of the next chunk + padding = 256 bytes
constexpr int kChunksOverflowed = -2;             // the pool ran dry under this border: it is walked again

// What the walk needs besides the RETR_EXTERNAL inputs when it serves bv_find_contours (TREE = true): records
// 0 .. n_outer-1 are the outer borders, as for RETR_EXTERNAL, and the hole borders follow them.
struct TreeArgs {
    const int *n_holes;       // [batch] holes per frame (ranked background labelling)
    const int *hole_px;       // [batch][max_contours] first pixel of every hole, raster order
    const uint32_t *fg_bits;  // the foreground mask, row-major words
    const int *fg_parent;     // the ranked foreground union-find: parent[root] = -label, other nodes point at their root
    int *enclosing;           // [batch][max_contours] out: outer border -> hole index or -1, hole border -> label - 1
    int none;                 // CHAIN_APPROX_NONE: every border pixel is a vertex
};

// hole index of the background pixel (x, y) once the holes are ranked (ccl_rank_kernel<true>); -1 for a frame-touching
// region, whose root keeps parent[root] == root
__device__ __forceinline__ int hole_of(const uint32_t *frame_inv, const int *frame_parent, int wpr, int width, int y, int x) {
    const int v = frame_parent[node_of(frame_inv, wpr, width, y, x)];
    if (v < 0) return -v - 1;
    const int r = frame_parent[v];
    return r < 0 ? -r - 1 : -1;
}

// records of frame f that the walk writes
template <bool TREE>
__device__ __forceinline__ int records_of(const int *n_blobs, const int *n_holes, int f, int max_contours) {
    if (!TREE) return min(n_blobs[f], max_contours);
    return (int)min((long long)n_blobs[f] + n_holes[f], (long long)max_contours);
}

// WRITE = false: first walk (sums, counts, externality).  WRITE = true: second walk of the borders that got a slot in
// the point list but whose vertices the pool could not hold.  TREE = false: the external borders' CHAIN_APPROX_SIMPLE
// vertices (bv_outer_contours); TREE = true: outer and hole borders, CHAIN_APPROX_SIMPLE or NONE (bv_find_contours).
template <bool WRITE, bool TREE>
__global__ void __launch_bounds__(128) contour_kernel(const uint32_t *__restrict__ bits, const uint32_t *__restrict__ inv,
                                                      const int *__restrict__ parent_bg, const uint32_t *__restrict__ outer,
                                                      const int *__restrict__ root_px, const int *__restrict__ n_blobs,
                                                      bv_contour *__restrict__ out, int max_contours, int height, int width,
                                                      int wpr, int wcols, int *__restrict__ points, int max_points, int lane_stride,
                                                      int *__restrict__ pool, int *__restrict__ pool_next, int pool_chunks,
                                                      TreeArgs ta) {
    const int f = blockIdx.y;
    const int n = records_of<TREE>(n_blobs, ta.n_holes, f, max_contours);
    // one border per thread, but only every fourth lane takes one: a warp-wide load of 32 walks touches 32 different
    // lines and every step waits for the slowest of them
    if (threadIdx.x % lane_stride) return;
    const int idx = (blockIdx.x * blockDim.x + threadIdx.x) / lane_stride;
    if (idx >= n) return;
    const unsigned rows = (unsigned)height + 2;
    const uint32_t *fw = bits + (size_t)f * wcols * rows;  // walk_bits_kernel's copy
    // a hole border starts at the pixel left of the hole's first pixel, and cv2 starts its clockwise search there from E
    // (from W for an outer border)
    const bool hole = TREE && idx >= n_blobs[f];
    const bool none = TREE && ta.none;
    bv_contour c;
    int *pts = nullptr;
    int x0, y0;
    if (WRITE) {
        c = out[(size_t)f * max_contours + idx];
        if ((!TREE && !c.external) || c.point_offset < 0 || c.reserved != kChunksOverflowed) return;  // the gather kernel served the rest
        pts = points + ((size_t)f * max_points + c.point_offset) * 2;
        x0 = c.start_x;
        y0 = c.start_y;
    } else if (hole) {
        const int start = ta.hole_px[(size_t)f * max_contours + idx - n_blobs[f]];
        y0 = start / width;
        x0 = start - y0 * width - 1;  // foreground: the hole does not reach the frame
        const int *fp = ta.fg_parent + (size_t)f * height * width;
        const int v = fp[node_of(ta.fg_bits + (size_t)f * height * wpr, wpr, width, y0, x0)];
        c.label = v < 0 ? -v : -fp[v];
        c.start_x = x0;
        c.start_y = y0;
        c.external = 0;
        ta.enclosing[(size_t)f * max_contours + idx] = c.label - 1;
    } else {
        const int start = root_px[(size_t)f * max_contours + idx];
        y0 = start / width;
        x0 = start - y0 * width;
        c.label = idx + 1;
        c.start_x = x0;
        c.start_y = y0;
        // external iff the background on the left reaches the frame (or the start pixel is on the frame)
        int external = 1;
        if (TREE) {
            const int h = x0 > 0 ? hole_of(inv + (size_t)f * height * wpr, parent_bg + (size_t)f * height * width, wpr,
                                           width, y0, x0 - 1)
                                 : -1;
            external = h < 0;
            ta.enclosing[(size_t)f * max_contours + idx] = h;
        } else if (x0 > 0) {
            const uint32_t *fi = inv + (size_t)f * height * wpr;
            const int node = node_of(fi, wpr, width, y0, x0 - 1);
            const int root = parent_bg[(size_t)f * height * width + node];
            const size_t words_per_frame = ((size_t)height * width + 31) / 32;
            external = (outer[(size_t)f * words_per_frame + (root >> 5)] >> (root & 31)) & 1u;
        }
        c.external = external;
    }
    // Suzuki border following, direction codes 0..7 = E, NE, N, NW, W, SW, S, SE (y grows downwards)
    // dx = {1,1,0,-1,-1,-1,0,1}, dy = {0,-1,-1,-1,0,1,1,1} as nibble tables (value + 1), so that the
    // dynamically indexed look-up stays in registers
#define dx(s) ((int)((0x21000122u >> (4 * (s))) & 0xFu) - 1)
#define dy(s) ((int)((0x22210001u >> (4 * (s))) & 0xFu) - 1)
    long long a00 = 0, a10 = 0, a01 = 0;
    int bx0 = x0, bx1 = x0, by0 = y0, by1 = y0, npts = 1, nsimple = 1;
    // first walk of a border whose vertices are wanted: they also go into a chain of 31-point chunks drawn from the
    // frame's pool, so that they need not be found again by a second walk once the offsets in the point list are known
    const bool store = !WRITE && pool != nullptr && (TREE || c.external);
    int *fpool = store ? pool + (size_t)f * pool_chunks * kChunkInts : nullptr;
    int first_chunk = -1, chunk = -1, slot = kChunkPoints;
    auto keep_vertex = [&](int vx, int vy) {
        if (!store || first_chunk == kChunksOverflowed) return;
        if (slot == kChunkPoints) {
            const int next = atomicAdd(pool_next + f, 1);
            if (next >= pool_chunks) {
                first_chunk = kChunksOverflowed;
                return;
            }
            if (chunk >= 0) fpool[(size_t)chunk * kChunkInts + 2 * kChunkPoints] = next; else first_chunk = next;
            chunk = next;
            slot = 0;
        }
        fpool[(size_t)chunk * kChunkInts + 2 * slot] = vx;
        fpool[(size_t)chunk * kChunkInts + 2 * slot + 1] = vy;
        ++slot;
    };
    int s = hole ? 0 : 4;
    bool found = false;
    const uint32_t nb0 = neighbours_at(fw, rows, x0, y0);
    for (int k = 0; k < 7; ++k) {  // clockwise from W: NW, N, NE, E, SE, S, SW (from E: SE, S, SW, W, NW, N, NE)
        s = (s - 1) & 7;
        if ((nb0 >> s) & 1u) {
            found = true;
            break;
        }
    }
    if (!found) {
        if (WRITE) {
            pts[0] = x0;
            pts[1] = y0;
        }
        keep_vertex(x0, y0);
    } else {
        const int x1 = x0 + dx(s), y1 = y0 + dy(s);  // i1: the first neighbour, where the walk will end
        int cx = x0, cy = y0;                        // i3
        // CHAIN_APPROX_SIMPLE: keep a point when the direction turns.  The walk ends with the step i1 -> i0, in direction
        // s ^ 4, so the start pixel is kept iff the chain turns there, as CHAIN_APPROX_SIMPLE treats it: always for an
        // outer border (its start is the component's first pixel), not always for a hole border.
        int prev_s = s ^ 4;
        npts = 0;
        nsimple = 0;
        for (;;) {
            // counter-clockwise, starting just after the direction we came from: the three rows around (cx, cy) are
            // fetched at once (independent loads), the first set neighbour is a rotate + find-first-set.  The pixel we
            // came from is always set, so the search cannot come up empty.
            const uint32_t nb = neighbours_at(fw, rows, cx, cy);
            const int first = (s + 1) & 7;
            s = (first + __ffs(((nb | (nb << 8)) >> first) & 0xFFu) - 1) & 7;
            const int ddx = dx(s), ddy = dy(s);
            const int nx = cx + ddx, ny = cy + ddy;
            const bool turn = s != prev_s;
            if (turn || none) {
                if (WRITE) {
                    const int k = none ? npts : nsimple;
                    pts[2 * k] = cx;
                    pts[2 * k + 1] = cy;
                }
                keep_vertex(cx, cy);
            }
            if (turn) {
                ++nsimple;
                prev_s = s;
            }
            if (!WRITE) {
                // polygon edge (cx,cy) -> (nx,ny)
                // cross = cx*ny - nx*cy = cx*dy - cy*dx fits 32 bits for a unit step; the products go to 64
                const int dxy = cx * ddy - cy * ddx;
                a00 += dxy;
                a10 += (long long)dxy * (cx + nx);
                a01 += (long long)dxy * (cy + ny);
                bx0 = min(bx0, cx); bx1 = max(bx1, cx); by0 = min(by0, cy); by1 = max(by1, cy);
            }
            ++npts;
            if (nx == x0 && ny == y0 && cx == x1 && cy == y1) break;
            cx = nx;
            cy = ny;
            s = (s + 4) & 7;
        }
    }
#undef dx
#undef dy
    if (WRITE) {
        out[(size_t)f * max_contours + idx].reserved = 0;
        return;
    }
    c.a00 = a00;
    c.a10 = a10;
    c.a01 = a01;
    c.x0 = bx0; c.y0 = by0; c.x1 = bx1; c.y1 = by1;
    c.n_points = npts;
    c.n_simple = nsimple;
    c.point_offset = -1;
    c.reserved = store ? first_chunk : 0;
    out[(size_t)f * max_contours + idx] = c;
}

// one block per frame: hand every border that lists its vertices (the external ones; TREE: all) its slice of the frame's
// point list (exclusive scan of the vertex counts in record order; sequential over chunks of blockDim contours)
template <bool TREE>
__global__ void __launch_bounds__(1024) contour_offsets_kernel(bv_contour *__restrict__ contours, const int *__restrict__ n_blobs,
                                                               int max_contours, int max_points, int *__restrict__ n_points,
                                                               const int *__restrict__ n_holes, int none) {
    __shared__ int warp_sums[32];
    __shared__ int carry;
    const int f = blockIdx.x;
    const int n = records_of<TREE>(n_blobs, n_holes, f, max_contours);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    bv_contour *fc = contours + (size_t)f * max_contours;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += blockDim.x) {
        const int i = base + threadIdx.x;
        const int v = (i < n && (TREE || fc[i].external)) ? (TREE && none ? fc[i].n_points : fc[i].n_simple) : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) warp_sums[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            int ws = warp_sums[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int o = __shfl_up_sync(0xFFFFFFFFu, ws, d);
                if (lane >= d) ws += o;
            }
            warp_sums[lane] = ws;
        }
        __syncthreads();
        const int before = carry + (wid ? warp_sums[wid - 1] : 0) + incl - v;
        if (i < n && v > 0 && before + v <= max_points) fc[i].point_offset = before;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0 && n_points) n_points[f] = carry;
}

// One warp per listed contour that got a slice of the point list: copies its chain of chunks into the slice.
template <bool TREE>
__global__ void __launch_bounds__(128) contour_gather_kernel(bv_contour *__restrict__ contours, const int *__restrict__ n_blobs,
                                                             int max_contours, const int *__restrict__ pool, int pool_chunks,
                                                             int *__restrict__ points, int max_points,
                                                             const int *__restrict__ n_holes, int none) {
    const int f = blockIdx.y;
    const int n = records_of<TREE>(n_blobs, n_holes, f, max_contours);
    const int lane = threadIdx.x & 31;
    const int idx = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (idx >= n) return;
    bv_contour *c = contours + (size_t)f * max_contours + idx;
    const int first = c->reserved, offset = c->point_offset, count = (TREE && none) ? c->n_points : c->n_simple;
    if (!TREE && !c->external) return;
    __syncwarp();
    if (first == kChunksOverflowed && offset >= 0) return;    // keeps the mark: the second walk writes its vertices
    if (lane == 0) c->reserved = 0;
    if (offset < 0 || first < 0) return;
    const int *fpool = pool + (size_t)f * pool_chunks * kChunkInts;
    int *dst = points + ((size_t)f * max_points + offset) * 2;
    int chunk = first;
    for (int done = 0; done < count; done += kChunkPoints) {
        const int *src = fpool + (size_t)chunk * kChunkInts;
        const int here = min(kChunkPoints, count - done);
        for (int k = lane; k < 2 * here; k += 32) dst[2 * done + k] = src[k];
        chunk = src[2 * kChunkPoints];
    }
}

// One block per frame: cv2's hierarchy rows (next, prev, first_child, parent) of the records the walk wrote, and the
// frame's two counts.  Parents follow from `enclosing` and the mode; siblings are the records with the same parent, linked
// in increasing record order.  `next` comes from one warp that runs over the records from the last to the first, 32 at a
// time, keeping head[parent + 1] = the smallest record seen so far with that parent; `prev` is its inverse and
// first_child[p] is head[p + 1] at the end.  No atomics: the result does not depend on scheduling.
__global__ void __launch_bounds__(1024) contour_tree_kernel(int *__restrict__ enclosing, const int *__restrict__ n_outer_of,
                                                            const int *__restrict__ n_holes_of, int max_contours, int mode,
                                                            int4 *__restrict__ hierarchy, int *__restrict__ n_contours,
                                                            int *head_global) {
    extern __shared__ int head_shared[];
    const int f = blockIdx.x;
    const int n_outer = n_outer_of[f];
    const int n = records_of<true>(n_outer_of, n_holes_of, f, max_contours);
    int *par = enclosing + (size_t)f * max_contours;
    int4 *hier = hierarchy + (size_t)f * max_contours;
    int *head = head_global ? head_global + (size_t)f * (max_contours + 1) : head_shared;  // head[0]: parent -1
    if (threadIdx.x == 0 && n_contours) {
        n_contours[2 * f] = n_outer;
        n_contours[2 * f + 1] = n_holes_of[f];
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int e = par[i];
        int p = -1;
        if (i >= n_outer)
            p = mode == BV_RETR_LIST ? -1 : e;                            // hole -> its component's outer border
        else if (mode == BV_RETR_TREE && e >= 0 && n_outer + e < n)
            p = n_outer + e;                                              // outer border -> the hole around it
        par[i] = p;
        hier[i] = make_int4(-1, -1, -1, p);
    }
    for (int k = threadIdx.x; k <= n; k += blockDim.x) head[k] = -1;
    __syncthreads();
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        for (int base = (n - 1) & ~31; base >= 0; base -= 32) {
            const int i = base + lane;
            const bool valid = i < n;
            const int key = valid ? par[i] + 1 : -1 - lane;               // invalid lanes match nobody
            const unsigned peers = __match_any_sync(0xFFFFFFFFu, key);
            const unsigned later = peers & ~((2u << lane) - 1u);
            const int next = !valid ? -1 : later ? base + __ffs(later) - 1 : head[key];
            __syncwarp();
            if (valid && !(peers & ((1u << lane) - 1u))) head[key] = i;   // the group's first record
            if (valid) {
                hier[i].x = next;
                if (next >= 0) hier[next].y = i;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) hier[i].z = head[i + 1];
}

// RETR_EXTERNAL (mode < 0, bv_outer_contours): the outer borders, the external ones with their CHAIN_APPROX_SIMPLE
// vertices, n_contours[batch].  RETR_LIST / CCOMP / TREE (bv_find_contours): the outer borders, then the hole borders,
// all with vertices, n_contours[batch][2], and the hierarchy.
static int contours_bits(bv_ctx *ctx, const uint32_t *bits, int batch, int height, int width, bv_contour *contours,
                         int max_contours, int32_t *n_contours, int32_t *points, int max_points, int32_t *n_points, int mode,
                         int none, int32_t *hierarchy) {
    const bool tree = mode >= 0;
    const int wpr = words_per_row(width);
    const size_t total_words = (size_t)batch * height * wpr;
    const size_t total_rows = (size_t)batch * height;
    const size_t px = (size_t)height * width;
    const size_t outer_words = (px + 31) / 32;
    BV_TRY(ensure_scratch(ctx, SCR_CCL_ROOTS, (size_t)batch * max_contours * sizeof(int)));
    BV_TRY(ensure_scratch(ctx, SCR_BITS_B, total_words * 8));
    BV_TRY(ensure_scratch(ctx, SCR_CCL_PARENT2, total_rows * width * sizeof(int)));
    BV_TRY(ensure_scratch(ctx, SCR_CCL_AUX2, (total_rows * 2 + batch + (size_t)batch * outer_words) * sizeof(int)));
    int *root_px = (int *)ctx->scratch[SCR_CCL_ROOTS];
    uint32_t *inv = (uint32_t *)ctx->scratch[SCR_BITS_B];
    LabelScratch bg;
    bg.parent = (int *)ctx->scratch[SCR_CCL_PARENT2];
    bg.row_count = (int *)ctx->scratch[SCR_CCL_AUX2];
    bg.row_off = bg.row_count + total_rows;
    bg.n_fallback = bg.row_off + total_rows;          // the hole count per frame
    uint32_t *outer = (uint32_t *)(bg.n_fallback + batch);
    // RETR_LIST / CCOMP / TREE: first pixel of every hole, the records' enclosing regions, the hierarchy's head table
    int *hole_px = nullptr, *enclosing = nullptr, *head_global = nullptr;
    const size_t head_bytes = ((size_t)max_contours + 1) * sizeof(int);
    const bool head_in_smem = head_bytes <= 48 * 1024;
    if (tree) {
        BV_TRY(ensure_scratch(ctx, SCR_CCL_TREE, (size_t)batch * (2 * (size_t)max_contours + (head_in_smem ? 0 : max_contours + 1)) *
                                                     sizeof(int)));
        hole_px = (int *)ctx->scratch[SCR_CCL_TREE];
        enclosing = hole_px + (size_t)batch * max_contours;
        if (!head_in_smem) head_global = enclosing + (size_t)batch * max_contours;
    }
    // foreground: labels are not needed, only the roots in raster order
    LabelScratch ls;
    BV_TRY(label_scratch(ctx, batch, height, width, &ls));
    // label_bits_ex writes the blob count to n_blobs (its own scratch when NULL)
    int *nb = tree ? ls.n_fallback : (n_contours ? n_contours : ls.n_fallback);
    BV_TRY(label_bits_ex(ctx, bits, nullptr, batch, height, width, nullptr, 0, nb, root_px, max_contours, ls));
    // background, 4-connected
    const int gw = grid_for(ctx, total_words, 256, 8);
    BV_LAUNCH(ctx, invert_bits_kernel, gw, 256, 0, bits, inv, width, wpr, (uint32_t)total_words);
    BV_TRY(label_bits_ex(ctx, inv, nullptr, batch, height, width, nullptr, 0, bg.n_fallback, hole_px, max_contours, bg, outer));
    const int wcols = (width + (int)kWalkPixelsPerWord - 1) / (int)kWalkPixelsPerWord;
    const size_t walk_words = (size_t)batch * wcols * (height + 2);
    BV_REQUIRE(walk_words < 0xFFFFFFFFull, "frames too large for the contour walk");
    BV_TRY(ensure_scratch(ctx, SCR_BITS_TILED, walk_words * 4));
    uint32_t *walk = (uint32_t *)ctx->scratch[SCR_BITS_TILED];
    BV_LAUNCH(ctx, walk_bits_kernel, grid_for(ctx, walk_words, 256, 8), 256, 0, bits, walk, height, width, wpr, wcols,
              (uint32_t)walk_words);
    const int lane_stride = kContourLaneStride;
    dim3 grid((unsigned)(((size_t)max_contours * lane_stride + 127) / 128), batch);
    const bool want_points = points && max_points > 0;
    int *pool = nullptr, *pool_next = nullptr;
    int pool_chunks = 0;
    if (want_points) {
        // every contour wastes less than one chunk, and the vertices that fit the list fill max_points / 31 of them
        pool_chunks = max_points / kChunkPoints + max_contours + 1;
        if (ctx->opt[BV_OPT_CONTOUR_POOL_CHUNKS] > 0) pool_chunks = ctx->opt[BV_OPT_CONTOUR_POOL_CHUNKS];
        BV_TRY(ensure_scratch(ctx, SCR_CONTOUR_POOL, ((size_t)batch * pool_chunks * kChunkInts + batch) * sizeof(int)));
        pool = (int *)ctx->scratch[SCR_CONTOUR_POOL];
        pool_next = pool + (size_t)batch * pool_chunks * kChunkInts;
        BV_CUDA(cudaMemsetAsync(pool_next, 0, batch * sizeof(int), ctx->stream));
    }
    const TreeArgs ta = tree ? TreeArgs{bg.n_fallback, hole_px, bits, ls.parent, enclosing, none} : TreeArgs{};
    const int *nh = ta.n_holes;
    if (tree) {
        BV_LAUNCH(ctx, (contour_kernel<false, true>), grid, 128, 0, walk, inv, bg.parent, outer, root_px, nb, contours,
                  max_contours, height, width, wpr, wcols, nullptr, 0, lane_stride, pool, pool_next, pool_chunks, ta);
    } else {
        BV_LAUNCH(ctx, (contour_kernel<false, false>), grid, 128, 0, walk, inv, bg.parent, outer, root_px, nb, contours,
                  max_contours, height, width, wpr, wcols, nullptr, 0, lane_stride, pool, pool_next, pool_chunks, ta);
    }
    if (want_points) {
        const dim3 gg((max_contours + 3) / 4, batch);
        if (tree) {
            BV_LAUNCH(ctx, contour_offsets_kernel<true>, batch, 1024, 0, contours, nb, max_contours, max_points, n_points, nh, none);
            BV_LAUNCH(ctx, contour_gather_kernel<true>, gg, 128, 0, contours, nb, max_contours, pool, pool_chunks, points,
                      max_points, nh, none);
            BV_LAUNCH(ctx, (contour_kernel<true, true>), grid, 128, 0, walk, inv, bg.parent, outer, root_px, nb, contours,
                      max_contours, height, width, wpr, wcols, points, max_points, lane_stride, nullptr, nullptr, 0, ta);
        } else {
            BV_LAUNCH(ctx, contour_offsets_kernel<false>, batch, 1024, 0, contours, nb, max_contours, max_points, n_points, nh, 0);
            BV_LAUNCH(ctx, contour_gather_kernel<false>, gg, 128, 0, contours, nb, max_contours, pool, pool_chunks, points,
                      max_points, nh, 0);
            // borders the pool could not hold (it is sized so that this needs more vertices than max_points): walked again
            BV_LAUNCH(ctx, (contour_kernel<true, false>), grid, 128, 0, walk, inv, bg.parent, outer, root_px, nb, contours,
                      max_contours, height, width, wpr, wcols, points, max_points, lane_stride, nullptr, nullptr, 0, ta);
        }
    }
    if (tree && (hierarchy || n_contours)) {
        if (!hierarchy) {
            BV_TRY(ensure_scratch(ctx, SCR_CCL_TREE_ROWS, (size_t)batch * max_contours * sizeof(int4)));
            hierarchy = (int32_t *)ctx->scratch[SCR_CCL_TREE_ROWS];
        }
        BV_LAUNCH(ctx, contour_tree_kernel, batch, 1024, head_in_smem ? head_bytes : 0, enclosing, nb, nh, max_contours, mode,
                  reinterpret_cast<int4 *>(hierarchy), n_contours, head_global);
    }
    return BV_OK;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_label(bv_ctx *ctx, const uint8_t *mask_dev, int32_t *labels_dev, int batch, int height, int width,
                        bv_blob *blobs_dev, int max_blobs, int32_t *n_blobs_dev) {
    BV_REQUIRE(ctx && mask_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(max_blobs >= 0, "max_blobs must be >= 0");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t words = (size_t)batch * bits_frame_words(height, width);
    BV_TRY(ensure_scratch(ctx, SCR_BITS_A, words * 4));
    uint32_t *bits = (uint32_t *)ctx->scratch[SCR_BITS_A];
    BV_TRY(mask_to_bits(ctx, mask_dev, bits, batch, height, width));
    return label_bits(ctx, bits, labels_dev, batch, height, width, blobs_dev, max_blobs, n_blobs_dev);
}

extern "C" int bv_outer_contours(bv_ctx *ctx, const uint8_t *mask_dev, int batch, int height, int width,
                                 bv_contour *contours_dev, int max_contours, int32_t *n_contours_dev, int32_t *points_dev,
                                 int max_points, int32_t *n_points_dev) {
    BV_REQUIRE(ctx && mask_dev && contours_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0 && max_contours > 0, "sizes must be positive");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t words = (size_t)batch * bits_frame_words(height, width);
    BV_TRY(ensure_scratch(ctx, SCR_BITS_A, words * 4));
    uint32_t *bits = (uint32_t *)ctx->scratch[SCR_BITS_A];
    BV_TRY(mask_to_bits(ctx, mask_dev, bits, batch, height, width));
    return contours_bits(ctx, bits, batch, height, width, contours_dev, max_contours, n_contours_dev, points_dev,
                         points_dev ? max_points : 0, n_points_dev, -1, 0, nullptr);
}

extern "C" int bv_find_contours(bv_ctx *ctx, const uint8_t *mask_dev, int batch, int height, int width, int mode, int method,
                                bv_contour *contours_dev, int32_t *hierarchy_dev, int max_contours, int32_t *n_contours_dev,
                                int32_t *points_dev, int max_points, int32_t *n_points_dev) {
    BV_REQUIRE(ctx && mask_dev && contours_dev, "null argument");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0 && max_contours > 0, "sizes must be positive");
    BV_REQUIRE(mode == BV_RETR_LIST || mode == BV_RETR_CCOMP || mode == BV_RETR_TREE,
               "mode must be BV_RETR_LIST, BV_RETR_CCOMP or BV_RETR_TREE (RETR_EXTERNAL: bv_outer_contours)");
    BV_REQUIRE(method == BV_CHAIN_APPROX_NONE || method == BV_CHAIN_APPROX_SIMPLE,
               "method must be BV_CHAIN_APPROX_NONE or BV_CHAIN_APPROX_SIMPLE");
    BV_REQUIRE(max_points >= 0, "max_points must be >= 0");
    BV_REQUIRE(((uintptr_t)hierarchy_dev & 15) == 0, "hierarchy_dev must be 16-byte aligned");
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t words = (size_t)batch * bits_frame_words(height, width);
    BV_TRY(ensure_scratch(ctx, SCR_BITS_A, words * 4));
    uint32_t *bits = (uint32_t *)ctx->scratch[SCR_BITS_A];
    BV_TRY(mask_to_bits(ctx, mask_dev, bits, batch, height, width));
    return contours_bits(ctx, bits, batch, height, width, contours_dev, max_contours, n_contours_dev, points_dev,
                         points_dev ? max_points : 0, n_points_dev, mode, method == BV_CHAIN_APPROX_NONE, hierarchy_dev);
}
