// rects.cu -- cv2.minAreaRect of every outer contour (modules/bins.py:60-69, utils/feature.py:301-312),
// on the device-side CHAIN_APPROX_SIMPLE vertex lists that bv_outer_contours leaves in HBM, so the
// module's rectangle filter needs no per-contour host round trip.
//
// One thread per contour (the point sets are tiny: tens to hundreds of vertices):
//   1. heap-sort a private copy of the vertices by (x, y); drop duplicates
//   2. Andrew's monotone chain with exact integer cross products -> convex hull, taken clockwise in
//      y-up axes (the orientation cv::minAreaRect feeds to its rotating calipers)
//   3. rotating calipers in float32 as OpenCV's rotatingCalipers(CALIPERS_MINAREARECT) does: the
//      base vector follows the hull edge with the smallest angle to one of the four caliper sides;
//      the rectangle of least area (ties: the last one met) is kept
//   4. centre / size / angle as cv::minAreaRect derives them, angle reported in [-90, 0) like
//      cv2 4.13.0 (quarter turns with the sides swapped until it is in range)
// Tolerance (stated, tests/test_gpu_morph_ccl.py): the area agrees with cv2 to 1e-4 relative; centre,
// size and angle to 1e-3 whenever the minimum is unique -- OpenCV's own float32 evaluation order is
// not reproduced bit for bit, so two hull edges whose rectangles tie to within rounding may swap.
#include <math.h>

#include "common.cuh"

namespace bv {

struct P2 {
    int x, y;
};

__device__ __forceinline__ bool p_less(const P2 &a, const P2 &b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }

__device__ void heap_sort(P2 *a, int n) {
    for (int start = n / 2 - 1; start >= 0; --start) {  // heapify
        int root = start;
        for (;;) {
            int child = 2 * root + 1;
            if (child >= n) break;
            if (child + 1 < n && p_less(a[child], a[child + 1])) ++child;
            if (!p_less(a[root], a[child])) break;
            const P2 t = a[root]; a[root] = a[child]; a[child] = t;
            root = child;
        }
    }
    for (int end = n - 1; end > 0; --end) {
        const P2 t = a[0]; a[0] = a[end]; a[end] = t;
        int root = 0;
        for (;;) {
            int child = 2 * root + 1;
            if (child >= end) break;
            if (child + 1 < end && p_less(a[child], a[child + 1])) ++child;
            if (!p_less(a[root], a[child])) break;
            const P2 u = a[root]; a[root] = a[child]; a[child] = u;
            root = child;
        }
    }
}

__device__ __forceinline__ long long cross3(const P2 &o, const P2 &a, const P2 &b) {
    return (long long)(a.x - o.x) * (b.y - o.y) - (long long)(a.y - o.y) * (b.x - o.x);
}

// hull vertex i of the clockwise (y-up) sequence = counter-clockwise sequence reversed
struct HullView {
    const P2 *h;
    int n;
    const float *ex, *ey, *el;  // edge vectors and inverse lengths computed once per edge (NULL: computed on demand)
    __device__ __forceinline__ float2 pt(int i) const {
        const P2 p = h[n - 1 - i];
        return make_float2((float)p.x, (float)p.y);
    }
    __device__ __forceinline__ void edge(int i, float &vx, float &vy, float &inv_len) const {
        if (ex) {
            vx = ex[i];
            vy = ey[i];
            inv_len = el[i];
            return;
        }
        compute_edge(i, vx, vy, inv_len);
    }
    __device__ __forceinline__ void compute_edge(int i, float &vx, float &vy, float &inv_len) const {
        const P2 a = h[n - 1 - i], b = h[n - 1 - (i + 1 == n ? 0 : i + 1)];
        const double dx = (double)b.x - (double)a.x, dy = (double)b.y - (double)a.y;
        vx = (float)dx;
        vy = (float)dy;
        inv_len = (float)(1. / sqrt(dx * dx + dy * dy));
    }
};

__device__ void rotating_calipers(const HullView &H, float out[6]) {
    const int n = H.n;
    int left = 0, bottom = 0, right = 0, top = 0;
    float2 p0 = H.pt(0);
    float left_x = p0.x, right_x = p0.x, top_y = p0.y, bottom_y = p0.y;
    for (int i = 0; i < n; ++i) {
        const float2 p = H.pt(i);
        if (p.x < left_x) { left_x = p.x; left = i; }
        if (p.x > right_x) { right_x = p.x; right = i; }
        if (p.y > top_y) { top_y = p.y; top = i; }
        if (p.y < bottom_y) { bottom_y = p.y; bottom = i; }
    }
    // orientation of the hull: sign of the first non-zero turn
    float orientation = 0.f;
    {
        float ax, ay, il;
        H.edge(n - 1, ax, ay, il);
        for (int i = 0; i < n; ++i) {
            float bx, by;
            H.edge(i, bx, by, il);
            const double convexity = (double)ax * by - (double)ay * bx;
            if (convexity != 0) {
                orientation = convexity > 0 ? 1.f : -1.f;
                break;
            }
            ax = bx;
            ay = by;
        }
    }
    float base_a = orientation, base_b = 0.f;
    int seq[4] = {bottom, right, top, left};
    float minarea = 3.402823466e+38f;
    int best_left = 0, best_bottom = 0;
    float best_a = 1.f, best_b = 0.f, best_w = 0.f, best_h = 0.f;
    for (int k = 0; k < n; ++k) {
        float vx[4], vy[4], il[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) H.edge(seq[q], vx[q], vy[q], il[q]);
        const float dp[4] = {+base_a * vx[0] + base_b * vy[0], -base_b * vx[1] + base_a * vy[1],
                             -base_a * vx[2] - base_b * vy[2], +base_b * vx[3] - base_a * vy[3]};
        float maxcos = dp[0] * il[0];
        int main_el = 0;
#pragma unroll
        for (int q = 1; q < 4; ++q) {
            const float c = dp[q] * il[q];
            if (c > maxcos) {
                main_el = q;
                maxcos = c;
            }
        }
        float lx = 0.f, ly = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q == main_el) {
                lx = vx[q] * il[q];
                ly = vy[q] * il[q];
            }
        if (main_el == 0) { base_a = lx; base_b = ly; }
        else if (main_el == 1) { base_a = ly; base_b = -lx; }
        else if (main_el == 2) { base_a = -lx; base_b = -ly; }
        else { base_a = -ly; base_b = lx; }
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q == main_el) seq[q] = seq[q] + 1 == n ? 0 : seq[q] + 1;
        const float2 pr = H.pt(seq[1]), pl = H.pt(seq[3]), pt_ = H.pt(seq[2]), pb = H.pt(seq[0]);
        float dx = pr.x - pl.x, dy = pr.y - pl.y;
        const float width = dx * base_a + dy * base_b;
        dx = pt_.x - pb.x;
        dy = pt_.y - pb.y;
        const float height = -dx * base_b + dy * base_a;
        const float area = width * height;
        if (area <= minarea) {
            minarea = area;
            best_left = seq[3];
            best_bottom = seq[0];
            best_a = base_a;
            best_b = base_b;
            best_w = width;
            best_h = height;
        }
    }
    const float A1 = best_a, B1 = best_b, A2 = -best_b, B2 = best_a;
    const float2 pl = H.pt(best_left), pb = H.pt(best_bottom);
    const float C1 = A1 * pl.x + pl.y * B1;
    const float C2 = A2 * pb.x + pb.y * B2;
    const float idet = 1.f / (A1 * B2 - A2 * B1);
    out[0] = (C1 * B2 - C2 * B1) * idet;
    out[1] = (A1 * C2 - A2 * C1) * idet;
    out[2] = A1 * best_w;
    out[3] = B1 * best_w;
    out[4] = A2 * best_h;
    out[5] = B2 * best_h;
}

// Akl-Toussaint prefilter + heap sort + monotone chain by ONE thread in global scratch: the fallback for contours whose
// kept vertices do not fit the warp's shared-memory buffer (or whose coordinates do not fit 16 bits).  Returns the hull size.
__device__ __noinline__ int hull_sequential(const P2 *__restrict__ src, int n_in, P2 *sorted, P2 *hull) {
    P2 ext[4] = {src[0], src[0], src[0], src[0]};
    for (int i = 1; i < n_in; ++i) {
        const P2 p = src[i];
        if (p.x < ext[0].x) ext[0] = p;
        if (p.y < ext[1].y) ext[1] = p;
        if (p.x > ext[2].x) ext[2] = p;
        if (p.y > ext[3].y) ext[3] = p;
    }
    long long area2 = 0;
    for (int k = 0; k < 4; ++k)
        area2 += (long long)ext[k].x * ext[(k + 1) & 3].y - (long long)ext[(k + 1) & 3].x * ext[k].y;
    int n_kept = 0;
    if (area2 == 0 || n_in <= 8) {
        for (int i = 0; i < n_in; ++i) sorted[n_kept++] = src[i];
    } else {
        for (int k = 0; k < 4; ++k) sorted[n_kept++] = ext[k];
        for (int i = 0; i < n_in; ++i) {
            const P2 p = src[i];
            bool outside = false;
            for (int k = 0; k < 4; ++k) {
                const long long c = cross3(ext[k], ext[(k + 1) & 3], p);
                outside |= area2 > 0 ? c < 0 : c > 0;
            }
            if (outside) sorted[n_kept++] = p;
        }
    }
    heap_sort(sorted, n_kept);
    int n = 0;
    for (int i = 0; i < n_kept; ++i)
        if (n == 0 || sorted[i].x != sorted[n - 1].x || sorted[i].y != sorted[n - 1].y) sorted[n++] = sorted[i];
    int m = 0;
    if (n <= 2) {
        for (int i = 0; i < n; ++i) hull[m++] = sorted[i];
    } else {
        for (int i = 0; i < n; ++i) {  // lower chain
            while (m >= 2 && cross3(hull[m - 2], hull[m - 1], sorted[i]) <= 0) --m;
            hull[m++] = sorted[i];
        }
        const int lower = m + 1;
        for (int i = n - 2; i >= 0; --i) {  // upper chain
            while (m >= lower && cross3(hull[m - 2], hull[m - 1], sorted[i]) <= 0) --m;
            hull[m++] = sorted[i];
        }
        --m;  // the first point again
    }
    return m;
}

// cv2.minAreaRect of a convex hull (counter-clockwise in hull[0..m), as the monotone chain leaves it)
__device__ void rect_from_hull(const HullView &H, bv_rrect &r) {
    const P2 *hull = H.h;
    const int m = H.n;
    float angle = 0.f;
    if (m > 2) {
        float o[6];
        rotating_calipers(H, o);
        r.cx = o[0] + (o[2] + o[4]) * 0.5f;
        r.cy = o[1] + (o[3] + o[5]) * 0.5f;
        r.width = (float)sqrt((double)o[2] * o[2] + (double)o[3] * o[3]);
        r.height = (float)sqrt((double)o[4] * o[4] + (double)o[5] * o[5]);
        angle = (float)atan2((double)o[3], (double)o[2]);
    } else if (m == 2) {
        const P2 a = hull[0], b = hull[1];  // (x, y)-sorted, the order cv::convexHull returns a segment in
        r.cx = ((float)a.x + (float)b.x) * 0.5f;
        r.cy = ((float)a.y + (float)b.y) * 0.5f;
        const double dx = (double)b.x - a.x, dy = (double)b.y - a.y;
        r.width = (float)sqrt(dx * dx + dy * dy);
        r.height = 0.f;
        angle = (float)atan2(dy, dx);
    } else {
        r.cx = (float)hull[0].x;
        r.cy = (float)hull[0].y;
    }
    angle = (float)((double)angle * 180. / 3.1415926535897932384626433832795);
    // cv2 4.13.0 reports the angle in [-90, 0): quarter turns, the sides swapping with each
    for (int q = 0; q < 4 && !(angle < 0.f); ++q) {
        angle -= 90.f;
        const float t = r.width; r.width = r.height; r.height = t;
    }
    for (int q = 0; q < 4 && angle < -90.f; ++q) {
        angle += 90.f;
        const float t = r.width; r.width = r.height; r.height = t;
    }
    r.angle = angle;
    r.valid = 1;
}

// One WARP per contour.  A thread per contour spends its time in a heap sort over global scratch (one dependent access
// after the other, the frame waits for its largest contour); here the 32 lanes find the extreme points, filter and
// compact the vertices into shared memory (ballot), sort them as packed 16+16-bit keys with a bitonic network, and
// compute the hull's edge vectors; only the monotone chain and the calipers, both O(hull), run on lane 0, out of
// shared memory.
constexpr int kRectCap = 512;      // vertices a warp keeps in shared memory; more (or coordinates > 65534) -> fallback
constexpr int kRectWarps = 2;      // warps per block

struct RectWarpSmem {
    uint32_t keys[kRectCap];
    P2 hull[kRectCap + 1];
    float ex[kRectCap], ey[kRectCap], el[kRectCap];
};

__device__ __forceinline__ P2 key_point(uint32_t k) { return P2{(int)(k >> 16), (int)(k & 0xFFFFu)}; }

// The convex hull of src[0 .. n_in) built by one warp: counter-clockwise in y-up axes (clockwise on the image), starting at
// the smallest (x, y), collinear points dropped.  Returns the vertex count on every lane; `hull` points at the warp's
// shared memory or, when the vertices do not fit it (`fallback`), at `scratch` + n_in + 4, the record's private global
// scratch of 2 n_in + 9 points.
__device__ __forceinline__ int warp_hull(const P2 *__restrict__ src, int n_in, int lane, RectWarpSmem &sm, P2 *scratch,
                                         const P2 *&hull, bool &fallback) {
    // extreme points: per lane, then across the warp (ties: any of the tied points will do)
    P2 ext[4] = {src[0], src[0], src[0], src[0]};
    for (int i = lane; i < n_in; i += 32) {
        const P2 p = src[i];
        if (p.x < ext[0].x) ext[0] = p;
        if (p.y < ext[1].y) ext[1] = p;
        if (p.x > ext[2].x) ext[2] = p;
        if (p.y > ext[3].y) ext[3] = p;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        P2 o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            o[k].x = __shfl_down_sync(0xFFFFFFFFu, ext[k].x, off);
            o[k].y = __shfl_down_sync(0xFFFFFFFFu, ext[k].y, off);
        }
        if (o[0].x < ext[0].x) ext[0] = o[0];
        if (o[1].y < ext[1].y) ext[1] = o[1];
        if (o[2].x > ext[2].x) ext[2] = o[2];
        if (o[3].y > ext[3].y) ext[3] = o[3];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        ext[k].x = __shfl_sync(0xFFFFFFFFu, ext[k].x, 0);
        ext[k].y = __shfl_sync(0xFFFFFFFFu, ext[k].y, 0);
    }
    long long area2 = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        area2 += (long long)ext[k].x * ext[(k + 1) & 3].y - (long long)ext[(k + 1) & 3].x * ext[k].y;
    // Akl-Toussaint: only the extremes and the vertices strictly outside their quadrilateral can be hull vertices
    const bool keep_all = area2 == 0 || n_in <= 8;
    int n_kept = 0;
    if (!keep_all) {
        if (lane < 4) sm.keys[lane] = ((uint32_t)ext[lane].x << 16) | (uint32_t)ext[lane].y;
        n_kept = 4;
    }
    bool wide = false;
    for (int base = 0; base < n_in; base += 32) {
        const int i = base + lane;
        bool keep = false;
        P2 p = P2{0, 0};
        if (i < n_in) {
            p = src[i];
            wide |= (unsigned)p.x > 65534u || (unsigned)p.y > 65534u;
            keep = keep_all;
            if (!keep_all) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const long long cr = cross3(ext[k], ext[(k + 1) & 3], p);
                    keep |= area2 > 0 ? cr < 0 : cr > 0;
                }
            }
        }
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, keep);
        const int pos = n_kept + __popc(mask & ((1u << lane) - 1u));
        if (keep && pos < kRectCap) sm.keys[pos] = ((uint32_t)p.x << 16) | (uint32_t)p.y;
        n_kept += __popc(mask);
    }
    wide = __any_sync(0xFFFFFFFFu, wide);
    int m = 0;
    fallback = wide || n_kept > kRectCap;  // warp-uniform
    hull = fallback ? scratch + n_in + 4 : sm.hull;
    if (fallback) {
        // private scratch: [sorted points (n_in + 4) | hull stack (one more: the chain closes on its first point)]
        if (lane == 0) m = hull_sequential(src, n_in, scratch, scratch + n_in + 4);
    } else {
        int np2 = 32;
        while (np2 < n_kept) np2 <<= 1;
        for (int i = n_kept + lane; i < np2; i += 32) sm.keys[i] = 0xFFFFFFFFu;  // above every real key
        __syncwarp();
        for (int k = 2; k <= np2; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < (np2 >> 1); t += 32) {
                    const int lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
                    const uint32_t a = sm.keys[lo], b = sm.keys[hi];
                    if ((a > b) == ((lo & k) == 0)) {
                        sm.keys[lo] = b;
                        sm.keys[hi] = a;
                    }
                }
                __syncwarp();
            }
        if (lane == 0) {
            int n = 0;
            for (int i = 0; i < n_kept; ++i)
                if (n == 0 || sm.keys[i] != sm.keys[n - 1]) sm.keys[n++] = sm.keys[i];
            if (n <= 2) {
                for (int i = 0; i < n; ++i) sm.hull[m++] = key_point(sm.keys[i]);
            } else {
                for (int i = 0; i < n; ++i) {  // lower chain
                    const P2 p = key_point(sm.keys[i]);
                    while (m >= 2 && cross3(sm.hull[m - 2], sm.hull[m - 1], p) <= 0) --m;
                    sm.hull[m++] = p;
                }
                const int lower = m + 1;
                for (int i = n - 2; i >= 0; --i) {  // upper chain
                    const P2 p = key_point(sm.keys[i]);
                    while (m >= lower && cross3(sm.hull[m - 2], sm.hull[m - 1], p) <= 0) --m;
                    sm.hull[m++] = p;
                }
                --m;  // the first point again
            }
        }
    }
    m = __shfl_sync(0xFFFFFFFFu, m, 0);
    __syncwarp();
    return m;
}

// cv2.minAreaRect of the hull warp_hull built; the result is valid on lane 0
__device__ __forceinline__ void warp_rect(const P2 *hull, int m, bool fallback, int lane, RectWarpSmem &sm, bv_rrect &r) {
    HullView H{hull, m, nullptr, nullptr, nullptr};
    if (!fallback && m > 2) {  // edge vectors and inverse lengths once per edge, 32 at a time
        for (int i = lane; i < m; i += 32) H.compute_edge(i, sm.ex[i], sm.ey[i], sm.el[i]);
        H.ex = sm.ex;
        H.ey = sm.ey;
        H.el = sm.el;
    }
    __syncwarp();
    if (lane == 0) rect_from_hull(H, r);
}

__global__ void __launch_bounds__(32 * kRectWarps) min_area_rect_kernel(const bv_contour *__restrict__ contours,
                                                                        const int32_t *__restrict__ n_contours,
                                                                        const int32_t *__restrict__ points, int max_contours,
                                                                        int max_points, P2 *__restrict__ scratch,
                                                                        bv_rrect *__restrict__ rects) {
    __shared__ RectWarpSmem smem[kRectWarps];
    const int frame = blockIdx.y;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ci = blockIdx.x * kRectWarps + wib;
    if (ci >= max_contours) return;  // warp-uniform
    RectWarpSmem &sm = smem[wib];
    bv_rrect r;
    r.cx = r.cy = r.width = r.height = r.angle = 0.f;
    r.valid = 0;
    const int total = min(n_contours[frame], max_contours);
    const bv_contour c = contours[(size_t)frame * max_contours + ci];
    if (ci < total && c.external && c.point_offset >= 0 && c.n_simple > 0 && c.point_offset + c.n_simple <= max_points) {
        const int n_in = c.n_simple;
        const P2 *src = reinterpret_cast<const P2 *>(points) + (size_t)frame * max_points + c.point_offset;
        P2 *rec_scratch = scratch + (size_t)frame * (2 * (size_t)max_points + 9 * (size_t)max_contours) + 2 * (size_t)c.point_offset +
                          9 * (size_t)ci;
        const P2 *hull;
        bool fallback;
        const int m = warp_hull(src, n_in, lane, sm, rec_scratch, hull, fallback);
        warp_rect(hull, m, fallback, lane, sm, r);
    }
    if (lane == 0) rects[(size_t)frame * max_contours + ci] = r;
}


// ---- shape descriptors of every record (bv_contour_shapes) ---------------------------------------------------------------

// Farthest candidate of one warp-wide scan: lane-strided partial maxima (strict >: the first in traversal order wins),
// then the larger distance, or on a tie the earlier traversal position, across the warp.  Returns the position.
__device__ __forceinline__ int warp_argmax_first(double d, int pos, double &best) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        const double od = __shfl_down_sync(0xFFFFFFFFu, d, off);
        const int op = __shfl_down_sync(0xFFFFFFFFu, pos, off);
        if (od > d || (od == d && op < pos)) {
            d = od;
            pos = op;
        }
    }
    best = __shfl_sync(0xFFFFFFFFu, d, 0);
    return __shfl_sync(0xFFFFFFFFu, pos, 0);
}

// cv::approxPolyDP(closed) on int points as OpenCV 4.13 computes it (approx.cpp approxPolyDP_): the farthest-point
// initialisation over 3 passes, the slice stack -- a slice is split at the point farthest from its chord segment (squared
// distance to the nearer end where the point projects outside the segment) unless that is <= eps^2 --, the final
// collinear clean-up.  All lanes hold the same state; the farthest-point scans are split
// over the warp, lane 0 writes.  dst holds the record's n slots: the output grows from the front, the stack of slices
// from the back (written points + stacked slices <= n, as the slices tile the n steps of the closed curve).  Returns the
// vertex count.  eps2 = eps * eps.
__device__ int warp_approx_poly(const P2 *__restrict__ src, int n, double eps2, int lane, int2 *dst) {
    int w = 0, top = 0;
    auto push = [&](int a, int b) {
        if (lane == 0) dst[n - 1 - top] = make_int2(a, b);
        ++top;
    };
    // 1. approximately the two farthest points
    int pos = 0, rs = 0;
    bool le_eps = false;
    P2 start = src[0];
    for (int it = 0; it < 3; ++it) {
        pos = (pos + rs) % n;
        start = src[pos];
        double best = 0., d = 0.;
        int j_best = 0x7FFFFFFF;
        for (int j = 1 + lane; j < n; j += 32) {
            const P2 p = src[(pos + j) % n];
            const double dx = (double)(p.x - start.x), dy = (double)(p.y - start.y);
            const double dist = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            if (dist > d) {
                d = dist;
                j_best = j;
            }
        }
        const int jb = warp_argmax_first(d, j_best, best);
        if (best > 0.) rs = jb;
        le_eps = best <= eps2;
    }
    if (!le_eps) {
        const int s0 = pos, e0 = (rs + pos) % n;
        push(e0, s0);  // right slice
        push(s0, e0);
    } else {
        if (lane == 0) dst[w] = make_int2(start.x, start.y);
        ++w;
    }
    __syncwarp();
    // 2. the slice stack
    while (top > 0) {
        --top;
        const int2 sl = dst[n - 1 - top];  // written by lane 0 before the last __syncwarp
        __syncwarp();
        const int s0 = sl.x, e0 = sl.y;
        const P2 sp = src[s0], ep = src[e0];
        const int len = (e0 - s0 + n) % n - 1;  // candidates s0+1 .. e0-1
        int split = -1;
        if (len > 0) {
            const double dx = (double)(ep.x - sp.x), dy = (double)(ep.y - sp.y);
            const double l2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
            double d = 0., best;
            int k_best = 0x7FFFFFFF;
            for (int k = lane; k < len; k += 32) {
                const P2 p = src[(s0 + 1 + k) % n];
                // squared distance to the chord segment: to the nearer end where p projects outside it
                const double px = (double)(p.x - sp.x), py = (double)(p.y - sp.y);
                const double dot = __dadd_rn(__dmul_rn(px, dx), __dmul_rn(py, dy));
                double dist;
                if (dot <= 0.) {
                    dist = __dadd_rn(__dmul_rn(px, px), __dmul_rn(py, py));
                } else if (dot >= l2) {
                    const double qx = (double)(p.x - ep.x), qy = (double)(p.y - ep.y);
                    dist = __dadd_rn(__dmul_rn(qx, qx), __dmul_rn(qy, qy));
                } else {
                    const double cr = __dsub_rn(__dmul_rn(py, dx), __dmul_rn(px, dy));
                    dist = __ddiv_rn(__dmul_rn(cr, cr), l2);
                }
                if (dist > d) {
                    d = dist;
                    k_best = k;
                }
            }
            const int kb = warp_argmax_first(d, k_best, best);
            if (!(best <= eps2)) split = (s0 + 1 + kb) % n;
        }
        if (split < 0) {
            if (lane == 0) dst[w] = make_int2(sp.x, sp.y);
            ++w;
        } else {
            push(split, e0);
            push(s0, split);
        }
        __syncwarp();
    }
    // 3. clean-up of the points on [almost] straight lines, sequential as in OpenCV
    int count = w;
    if (lane == 0) {
        int new_count = count, rp = count - 1, wpos;
        int2 st = dst[rp];
        if (++rp >= count) rp = 0;
        wpos = rp;
        int2 pt = dst[rp];
        if (++rp >= count) rp = 0;
        for (int i = 0; i < count && new_count > 2; ++i) {
            const int2 en = dst[rp];
            if (++rp >= count) rp = 0;
            const double dx = (double)(en.x - st.x), dy = (double)(en.y - st.y);
            const double dist = fabs(__dsub_rn(__dmul_rn((double)(pt.x - st.x), dy), __dmul_rn((double)(pt.y - st.y), dx)));
            const double sip = (double)((pt.x - st.x) * (en.x - pt.x) + (pt.y - st.y) * (en.y - pt.y));
            if (__dmul_rn(dist, dist) <= __dmul_rn(__dmul_rn(0.5, eps2), __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy))) &&
                dx != 0 && dy != 0 && sip >= 0) {
                --new_count;
                dst[wpos] = st = en;
                if (++wpos >= count) wpos = 0;
                pt = dst[rp];
                if (++rp >= count) rp = 0;
                ++i;
                continue;
            }
            dst[wpos] = st = pt;
            if (++wpos >= count) wpos = 0;
            pt = en;
        }
        count = new_count;
    }
    count = __shfl_sync(0xFFFFFFFFu, count, 0);
    __syncwarp();
    return count;
}

// cv::isContourConvex on int points, with its 32-bit products
__device__ int contour_convex(const int2 *p, int n) {
    if (n < 3) return 0;
    int2 prev = p[n - 2], cur = p[n - 1];
    int dx0 = cur.x - prev.x, dy0 = cur.y - prev.y, orientation = 0;
    for (int i = 0; i < n; ++i) {
        prev = cur;
        cur = p[i];
        const int dx = cur.x - prev.x, dy = cur.y - prev.y;
        const int dxdy0 = (int)((unsigned)dx * (unsigned)dy0), dydx0 = (int)((unsigned)dy * (unsigned)dx0);
        orientation |= dydx0 > dxdy0 ? 1 : (dydx0 < dxdy0 ? 2 : 3);
        if (orientation == 3) return 0;
        dx0 = dx;
        dy0 = dy;
    }
    return 1;
}

struct Circle {
    double x, y, r2;
};

__device__ __forceinline__ bool outside(const Circle &c, const P2 &p) {
    const double dx = p.x - c.x, dy = p.y - c.y;
    return dx * dx + dy * dy > c.r2 * (1. + 1e-12);
}

// First hull vertex (in the fixed visiting order q -> (q * stride) % m) among positions [lo, hi) outside c, or -1.
__device__ __forceinline__ int first_outside(const P2 *hull, int m, int stride, int lo, int hi, const Circle &c, int lane) {
    for (int base = lo; base < hi; base += 32) {
        const int q = base + lane;
        const bool out = q < hi && outside(c, hull[(int)(((long long)q * stride) % m)]);
        const uint32_t b = __ballot_sync(0xFFFFFFFFu, out);
        if (b) return base + __ffs(b) - 1;
    }
    return -1;
}

// The minimum enclosing circle of the hull in double: the incremental algorithm over a fixed permutation of the
// vertices, each "first vertex outside" search split over the warp.  Every lane computes the same circle.
__device__ Circle warp_enclosing_circle(const P2 *hull, int m, int lane) {
    int stride = 7919;  // any stride coprime with m visits every vertex once
    for (;;) {
        int a = stride, b = m;
        while (b) { const int t = a % b; a = b; b = t; }
        if (a == 1) break;
        stride += 2;
    }
    auto at = [&](int q) { return hull[(int)(((long long)q * stride) % m)]; };
    const P2 a0 = at(0);
    Circle c{(double)a0.x, (double)a0.y, 0.};
    for (int i = 1; i < m; ++i) {
        const P2 pi = at(i);
        if (!outside(c, pi)) continue;
        c = Circle{(double)pi.x, (double)pi.y, 0.};
        for (int j = first_outside(hull, m, stride, 0, i, c, lane); j >= 0;) {
            const P2 pj = at(j);
            c.x = 0.5 * ((double)pi.x + pj.x);
            c.y = 0.5 * ((double)pi.y + pj.y);
            c.r2 = 0.25 * (((double)pi.x - pj.x) * ((double)pi.x - pj.x) + ((double)pi.y - pj.y) * ((double)pi.y - pj.y));
            for (int k = first_outside(hull, m, stride, 0, j, c, lane); k >= 0;) {
                const P2 pk = at(k);
                // circumcircle of pi, pj, pk (three distinct hull vertices are never collinear)
                const double bx = (double)pj.x - pi.x, by = (double)pj.y - pi.y;
                const double cx = (double)pk.x - pi.x, cy = (double)pk.y - pi.y;
                const double d = 2. * (bx * cy - by * cx);
                const double b2 = bx * bx + by * by, c2 = cx * cx + cy * cy;
                const double ux = (cy * b2 - by * c2) / d, uy = (bx * c2 - cx * b2) / d;
                c = Circle{pi.x + ux, pi.y + uy, ux * ux + uy * uy};
                k = first_outside(hull, m, stride, k + 1, j, c, lane);
            }
            j = first_outside(hull, m, stride, j + 1, i, c, lane);
        }
    }
    return c;
}

__global__ void __launch_bounds__(32 * kRectWarps) contour_shapes_kernel(
    const bv_contour *__restrict__ contours, const int32_t *__restrict__ n_contours, int counts_per_frame,
    const int32_t *__restrict__ points, int max_contours, int max_points, int method, double approx_epsilon,
    double approx_relative, P2 *__restrict__ scratch, bv_shape *__restrict__ shapes, int32_t *__restrict__ hull_out,
    int32_t *__restrict__ approx_out) {
    __shared__ RectWarpSmem smem[kRectWarps];
    const int frame = blockIdx.y;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ci = blockIdx.x * kRectWarps + wib;
    if (ci >= max_contours) return;  // warp-uniform
    RectWarpSmem &sm = smem[wib];
    bv_shape out;
    memset(&out, 0, sizeof(out));
    int total = n_contours[(size_t)frame * counts_per_frame];
    if (counts_per_frame == 2) total += n_contours[(size_t)frame * 2 + 1];
    total = min(total, max_contours);
    const bv_contour c = contours[(size_t)frame * max_contours + ci];
    const int n_in = method == BV_CHAIN_APPROX_NONE ? c.n_points : c.n_simple;
    if (ci < total && c.point_offset >= 0 && n_in > 0 && c.point_offset <= max_points - n_in) {
        const size_t base = (size_t)frame * max_points + c.point_offset;
        const P2 *src = reinterpret_cast<const P2 *>(points) + base;
        // arcLength: float32 steps (exact integers in, correctly rounded sqrt), summed exactly in double
        double arc = 0.;
        for (int i = lane; i < n_in; i += 32) {
            const P2 p = src[i], q = src[i == 0 ? n_in - 1 : i - 1];
            const float dx = __fsub_rn((float)p.x, (float)q.x), dy = __fsub_rn((float)p.y, (float)q.y);
            arc += (double)__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) arc += __shfl_xor_sync(0xFFFFFFFFu, arc, off);
        out.arc_length = arc;

        P2 *rec_scratch = scratch + (size_t)frame * (2 * (size_t)max_points + 9 * (size_t)max_contours) + 2 * (size_t)c.point_offset +
                          9 * (size_t)ci;
        const P2 *hull;
        bool fallback;
        const int m = warp_hull(src, n_in, lane, sm, rec_scratch, hull, fallback);
        warp_rect(hull, m, fallback, lane, sm, out.rect);
        out.rect = {__shfl_sync(0xFFFFFFFFu, out.rect.cx, 0), __shfl_sync(0xFFFFFFFFu, out.rect.cy, 0),
                    __shfl_sync(0xFFFFFFFFu, out.rect.width, 0), __shfl_sync(0xFFFFFFFFu, out.rect.height, 0),
                    __shfl_sync(0xFFFFFFFFu, out.rect.angle, 0), 1};
        out.n_hull = m;

        const Circle cc = warp_enclosing_circle(hull, m, lane);
        out.circle_cx = (float)cc.x;
        out.circle_cy = (float)cc.y;
        out.circle_r = (float)(sqrt(cc.r2) + 1e-4);

        if (hull_out) {
            // cv2.convexHull's first vertex: where the vertices' first indices in the contour run cyclically up (or
            // down), the smallest (largest) of them; otherwise the largest (x, y)
            int *first = fallback ? reinterpret_cast<int *>(rec_scratch) : reinterpret_cast<int *>(sm.keys);
            int top = 0;
            for (int k = lane; k < m; k += 32) {
                first[k] = 0x7FFFFFFF;
                if (p_less(hull[top], hull[k])) top = k;
            }
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const int o = __shfl_xor_sync(0xFFFFFFFFu, top, off);
                if (o < m && p_less(hull[top], hull[o])) top = o;
            }
            __syncwarp();
            for (int i = lane; i < n_in; i += 32) {  // lower chain hull[0..top] ascends, upper hull[top..m) descends
                const P2 p = src[i];
                int lo = 0, hi = top, k = -1;
                while (lo <= hi) {
                    const int mid = (lo + hi) >> 1;
                    if (p_less(hull[mid], p)) lo = mid + 1;
                    else if (p_less(p, hull[mid])) hi = mid - 1;
                    else { k = mid; break; }
                }
                lo = top + 1, hi = m - 1;
                while (k < 0 && lo <= hi) {
                    const int mid = (lo + hi) >> 1;
                    if (p_less(p, hull[mid])) lo = mid + 1;
                    else if (p_less(hull[mid], p)) hi = mid - 1;
                    else { k = mid; break; }
                }
                if (k >= 0) atomicMin(first + k, i);
            }
            __syncwarp();
            int start = top;
            if (m >= 3) {
                int ups = 0, kmin = 0, kmax = 0;
                for (int k = lane; k < m; k += 32) {
                    ups += first[k + 1 == m ? 0 : k + 1] > first[k];
                    if (first[k] < first[kmin]) kmin = k;
                    if (first[k] > first[kmax]) kmax = k;
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    ups += __shfl_xor_sync(0xFFFFFFFFu, ups, off);
                    const int a = __shfl_xor_sync(0xFFFFFFFFu, kmin, off), b = __shfl_xor_sync(0xFFFFFFFFu, kmax, off);
                    if (first[a] < first[kmin]) kmin = a;
                    if (first[b] > first[kmax]) kmax = b;
                }
                if (ups == m - 1) start = kmin;
                else if (ups == 1) start = kmax;
            }
            int2 *dst = reinterpret_cast<int2 *>(hull_out) + base;
            for (int k = lane; k < m; k += 32) {
                const P2 p = hull[(start + k) % m];
                dst[k] = make_int2(p.x, p.y);
            }
        }

        if (approx_out) {
            const double eps = __dadd_rn(approx_epsilon, __dmul_rn(approx_relative, arc));
            int2 *dst = reinterpret_cast<int2 *>(approx_out) + base;
            out.n_approx = warp_approx_poly(src, n_in, __dmul_rn(eps, eps), lane, dst);
            if (lane == 0) out.approx_convex = contour_convex(dst, out.n_approx);
        }
        out.valid = 1;
    }
    if (lane == 0) shapes[(size_t)frame * max_contours + ci] = out;
}

}  // namespace bv

using namespace bv;

extern "C" int bv_min_area_rects(bv_ctx *ctx, const bv_contour *contours_dev, const int32_t *n_contours_dev,
                                 const int32_t *points_dev, int batch, int max_contours, int max_points, bv_rrect *rects_dev) {
    BV_REQUIRE(ctx && contours_dev && n_contours_dev && points_dev && rects_dev, "null argument");
    BV_REQUIRE(batch > 0 && batch <= 65535 && max_contours > 0 && max_points > 0, "sizes must be positive");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_scratch(ctx, SCR_HULL, sizeof(P2) * (size_t)batch * (2 * (size_t)max_points + 9 * (size_t)max_contours)));
    BV_LAUNCH(ctx, min_area_rect_kernel, dim3((max_contours + kRectWarps - 1) / kRectWarps, batch), 32 * kRectWarps, 0, contours_dev,
              n_contours_dev, points_dev, max_contours, max_points, (P2 *)ctx->scratch[SCR_HULL], rects_dev);
    return BV_OK;
}

extern "C" int bv_contour_shapes(bv_ctx *ctx, const bv_contour *contours_dev, const int32_t *n_contours_dev, int counts_per_frame,
                                 const int32_t *points_dev, int batch, int max_contours, int max_points, int method,
                                 double approx_epsilon, double approx_relative, bv_shape *shapes_dev, int32_t *hull_dev,
                                 int32_t *approx_dev) {
    BV_REQUIRE(ctx && contours_dev && n_contours_dev && points_dev && shapes_dev, "null argument");
    BV_REQUIRE(batch > 0 && batch <= 65535 && max_contours > 0 && max_points > 0, "sizes must be positive");
    BV_REQUIRE(counts_per_frame == 1 || counts_per_frame == 2, "counts_per_frame must be 1 or 2");
    BV_REQUIRE(method == BV_CHAIN_APPROX_NONE || method == BV_CHAIN_APPROX_SIMPLE, "unknown method");
    BV_REQUIRE(counts_per_frame == 2 || method == BV_CHAIN_APPROX_SIMPLE,
               "a bv_outer_contours table (counts_per_frame = 1) holds CHAIN_APPROX_SIMPLE vertices only");
    BV_REQUIRE(approx_epsilon >= 0 && approx_relative >= 0, "approximation accuracy must be non-negative");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_TRY(ensure_scratch(ctx, SCR_HULL, sizeof(P2) * (size_t)batch * (2 * (size_t)max_points + 9 * (size_t)max_contours)));
    BV_LAUNCH(ctx, contour_shapes_kernel, dim3((max_contours + kRectWarps - 1) / kRectWarps, batch), 32 * kRectWarps, 0, contours_dev,
              n_contours_dev, counts_per_frame, points_dev, max_contours, max_points, method, approx_epsilon, approx_relative,
              (P2 *)ctx->scratch[SCR_HULL], shapes_dev, hull_dev, approx_dev);
    return BV_OK;
}
