// common.cuh -- context, error plumbing and small device helpers shared by all translation units
// of libb200vision.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/b200vision.h"
#include "pixel_math.cuh"

namespace bv {

// ---- error plumbing ------------------------------------------------------------------------
void set_error(const char *fmt, ...);  // thread-local message, api.cu

#define BV_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            bv::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));   \
            return BV_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

#define BV_REQUIRE(cond, msg)                                                                      \
    do {                                                                                           \
        if (!(cond)) {                                                                             \
            bv::set_error("%s: %s", __func__, msg);                                                \
            return BV_ERR_INVALID;                                                                 \
        }                                                                                          \
    } while (0)

#define BV_TRY(expr)                                                                               \
    do {                                                                                           \
        int _s = (expr);                                                                           \
        if (_s != BV_OK) return _s;                                                                \
    } while (0)

// Launch + count + check.  Every kernel of the library goes through this macro so that
// bv_launch_count() is the true number of launches.
#define BV_LAUNCH(ctx, kernel, grid, block, smem, ...)                                             \
    do {                                                                                           \
        if ((ctx)->prof) bv::prof_begin((ctx), #kernel);                                           \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                           \
        (ctx)->launches++;                                                                         \
        if ((ctx)->prof) bv::prof_end((ctx));                                                      \
        BV_CUDA(cudaGetLastError());                                                               \
    } while (0)

// Programmatic dependent launch: the kernel may start (and run its prologue up to bv::grid_dependency_wait())
// while the previous kernel of the stream is still draining; everything it reads that the previous kernel wrote
// must come after that wait.  Same counting / profiling / checking as BV_LAUNCH.
#define BV_LAUNCH_PDL(ctx, kernel, grid, block, smem, ...)                                         \
    do {                                                                                           \
        if ((ctx)->prof) bv::prof_begin((ctx), #kernel);                                           \
        cudaLaunchConfig_t cfg_;                                                                   \
        memset(&cfg_, 0, sizeof(cfg_));                                                            \
        cfg_.gridDim = (grid);                                                                     \
        cfg_.blockDim = (block);                                                                   \
        cfg_.dynamicSmemBytes = (smem);                                                            \
        cfg_.stream = (ctx)->stream;                                                               \
        cudaLaunchAttribute attr_[1];                                                              \
        attr_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                          \
        attr_[0].val.programmaticStreamSerializationAllowed = 1;                                   \
        cfg_.attrs = attr_;                                                                        \
        cfg_.numAttrs = (ctx)->prof ? 0 : 1;                                                       \
        cudaError_t le_ = cudaLaunchKernelEx(&cfg_, kernel, __VA_ARGS__);                          \
        (ctx)->launches++;                                                                         \
        if ((ctx)->prof) bv::prof_end((ctx));                                                      \
        BV_CUDA(le_);                                                                              \
        BV_CUDA(cudaGetLastError());                                                               \
    } while (0)

// ---- scratch slots ---------------------------------------------------------------------------
enum ScratchSlot {
    SCR_BAL_STATE = 0,  // per-frame histograms, LUTs, stats of the colour balance
    SCR_BAL_TILES,      // per-tile histograms and tables (tiled equalisation)
    SCR_BAL_HSV,        // H,S,V image written by pass 2 and read by pass 3 (L2 resident per chunk)
    SCR_WARP,           // per-column / per-row fixed-point coordinate terms of warpAffine
    SCR_HSI,            // float32 H, S, I planes of one frame (HSI contrast branch)
    SCR_HSI_BGR,        // balanced BGR frames the HSI branch works on when the caller does not want them
    SCR_BITS_A,         // bit-packed masks (ping)
    SCR_BITS_B,         // bit-packed masks (pong)
    SCR_CONTOUR_POOL,   // chunked vertex storage of the contour walk (+ one allocation counter per frame)
    SCR_BITS_TILED,     // copy of the bit mask laid out for the contour walk (walk_bits_kernel)
    SCR_CCL_PARENT,     // union-find parents, int32 per pixel
    SCR_CCL_AUX,        // per-block root counts / offsets
    SCR_CCL_PARENT2,    // union-find parents of the background regions (outer contours)
    SCR_CCL_AUX2,       // background row counts / offsets, hole counts, frame-touching bitmap
    SCR_CCL_ROOTS,      // first pixel of every blob, raster order
    SCR_CCL_TREE,       // first pixel of every hole, enclosing region of every border, hierarchy head table (find_contours)
    SCR_CCL_TREE_ROWS,  // hierarchy rows when the caller passes none
    SCR_HULL,           // sorted vertices + hull stack per contour (minAreaRect)
    SCR_NOISE_RAW,      // raw MT19937 words replayed for the Gaussian-noise step
    SCR_NOISE_AUX,      // per-block accepted counts / offsets of the polar method
    SCR_MORPH_TMP,      // intermediate image of multi-step grey morphology
    SCR_MORPH_TMP2,
    SCR_MORPH_SE,       // structuring-element offsets
    SCR_STAGE_IMG,      // balanced frame when the caller does not want it
    SCR_LETTERBOX,      // per-image descriptors
    SCR_HOST_IN,        // device staging of bv_stage_host
    SCR_HOST_BAL,
    SCR_HOST_CVT,
    SCR_HOST_MASK,
    SCR_HOST_LABELS,
    SCR_HOST_BLOBS,
    SCR_HOST_NBLOBS,
    SCR_HOST1_IN,       // second staging set (slot 1 of bv_stage_host_submit), same order as the first
    SCR_HOST1_BAL,
    SCR_HOST1_CVT,
    SCR_HOST1_MASK,
    SCR_HOST1_LABELS,
    SCR_HOST1_BLOBS,
    SCR_HOST1_NBLOBS,
    SCR_IVL_FRAMES,     // hue-interval table composed with every frame's S / V stretch tables (balance.cu)
    SCR_INGEST,         // landing buffer of 4-channel frames ingested from a shared-memory ring (ingest.cu)
    SCR_HOUGH_TAB,      // trig table of the Hough transform, then per-frame edge and peak counts (hough.cu)
    SCR_HOUGH_ACC,      // int32 Hough accumulators of one group of frames
    SCR_HOUGH_KEYS,     // peak keys of one group of frames, two buffers for the radix sort
    SCR_HOUGH_EDGES,    // edge-pixel lists of one group of frames (+ their values with use_edgeval)
    SCR_THRESH_SMALL,   // per-frame histograms of the automatic thresholds, or the Gaussian taps of the adaptive one (thresh.cu)
    SCR_THRESH_PLANE,   // row prefix sums (MEAN_C) or float32 row-filtered frames (GAUSSIAN_C) of the adaptive threshold
    SCR_COUNT
};

}  // namespace bv

#define BV_MAX_CHUNKS 64
#define BV_MAX_SIDE 4
#define BV_HOST_SLOTS 2
#define BV_IVL_SLOTS 4

struct bv_ctx {
    int device;
    int sm_count;
    cudaStream_t own_stream;
    cudaStream_t stream;
    uint64_t launches;
    void *scratch[bv::SCR_COUNT];
    size_t scratch_bytes[bv::SCR_COUNT];
    uint16_t *d_lab_gamma;  // 256
    uint16_t *d_lab_cbrt;   // 3072, then the Lab->BGR tables: 512 x u16 (y, fy) and 4096 x u8 inverse gamma
    int16_t *d_luv_tab;     // 33^3 x 4 int16 nodes of BGR2LUV (cvt.cu), built on first use
    short *d_bilinear_tab;  // 32x32x4 int16 bilinear weights of cv::warpAffine / cv::remap (filter.cu), built on first use
    double *d_pow_quarter;  // 256: pow((255-x)/255, 0.25) from the host libm (adaptive cast correction)
    // host-memory pipeline (bv_stage_host): copy streams and per-chunk events
    cudaStream_t copy_in, copy_out;
    cudaEvent_t ev_in[BV_MAX_CHUNKS], ev_done[BV_MAX_CHUNKS];
    cudaEvent_t ev_slot[BV_HOST_SLOTS];  // end of the last download of the call in flight on each staging set
    int slot_busy[BV_HOST_SLOTS];
    int overlapped;  // the current call spreads its chunks over side streams (small grids per kernel)
    void *prof;  // per-kernel CUDA-event timing, only while bv_profile_enable(ctx, 1)
    // side streams: independent chunks of one call run concurrently so that the issue-bound final
    // pass of one chunk overlaps the atomics-bound histogram passes of the next
    cudaStream_t side[BV_MAX_SIDE];
    cudaEvent_t ev_fork, ev_join[BV_MAX_SIDE];
    // hue-interval tables of the HSV inRange fast path (balance.cu), one per distinct bounds set
    struct {
        uint8_t key[6];
        int state;         // 0 empty, 1 usable, 2 built but not representable (generic pass is used)
        uint16_t *table;   // 65536 entries, device
    } ivl[BV_IVL_SLOTS];
    int ivl_next;
    int ivl_attr_set;
    int lb_smem_set;     // same for letterbox_tma_kernel
    void *lb_cache;      // host copy of the letterbox descriptors whose tap table is on the device
    int lb_cache_n, lb_cache_ow, lb_cache_oh;
    int opt[BV_OPT_COUNT];  // tuning knobs, 0 = built-in default (bv_set_option)
    int *d_ivl_flag;
};

namespace bv {

int ensure_scratch(bv_ctx *ctx, int slot, size_t bytes);  // api.cu
void prof_begin(bv_ctx *ctx, const char *kernel);          // api.cu
void prof_end(bv_ctx *ctx);

// ---- device helpers --------------------------------------------------------------------------
#if defined(__CUDACC__)

// blocks until the previous kernel of the stream has completed and its writes are visible (no-op when the kernel
// was not launched with BV_LAUNCH_PDL)
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// streaming 128-bit load that does not pollute L1
__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
// plain 128-bit load (keeps the line in L1/L2: used when a later pass re-reads the frame)
__device__ __forceinline__ uint4 ld_keep(const uint4 *p) { return __ldg(p); }

__device__ __forceinline__ void st_stream(uint4 *p, const uint4 &v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
                 "r"(v.w));
}

// 16 interleaved 3-channel pixels = 48 bytes = 12 words
struct Px16 {
    uint32_t w[12];
};

template <bool KEEP>
__device__ __forceinline__ void load_px16(const uint8_t *base, size_t group, Px16 &p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(base) + group * 3;
    uint4 a, b, c;
    if (KEEP) {
        a = ld_keep(q);
        b = ld_keep(q + 1);
        c = ld_keep(q + 2);
    } else {
        a = ld_stream(q);
        b = ld_stream(q + 1);
        c = ld_stream(q + 2);
    }
    p.w[0] = a.x; p.w[1] = a.y; p.w[2] = a.z; p.w[3] = a.w;
    p.w[4] = b.x; p.w[5] = b.y; p.w[6] = b.z; p.w[7] = b.w;
    p.w[8] = c.x; p.w[9] = c.y; p.w[10] = c.z; p.w[11] = c.w;
}

__device__ __forceinline__ void store_px16(uint8_t *base, size_t group, const Px16 &p) {
    uint4 *q = reinterpret_cast<uint4 *>(base) + group * 3;
    st_stream(q, make_uint4(p.w[0], p.w[1], p.w[2], p.w[3]));
    st_stream(q + 1, make_uint4(p.w[4], p.w[5], p.w[6], p.w[7]));
    st_stream(q + 2, make_uint4(p.w[8], p.w[9], p.w[10], p.w[11]));
}

// byte k (compile-time constant after unrolling) of a packed word array
// (bytes 1 and 2 of a word through one byte-permute instead of shift + mask)
__device__ __forceinline__ uint32_t bv_word_byte(uint32_t w, int b) {
    return b == 0 ? (w & 0xFFu) : b == 3 ? (w >> 24) : __byte_perm(w, 0u, 0x4440u | (uint32_t)b);
}
#define BV_GETB(W, k) bv::bv_word_byte((W)[(k) >> 2], (k)&3)
#define BV_PUTB(W, k, v) ((W)[(k) >> 2] |= ((uint32_t)(v)) << (8 * ((k)&3)))

// ---- TMA bulk copy (cp.async.bulk, SASS: UBLKCP) completing on an mbarrier ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t phase) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"  // suspends up to the hint instead of spinning
        "@p bra LB_DONE_%=;\n"
        "bra LB_WAIT_%=;\n"
        "LB_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(phase), "r"(0x989680u)
        : "memory");
}

__device__ __forceinline__ bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

#endif  // __CUDACC__

inline bool host_aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Grid sizing for grid-stride kernels: a whole number of waves of 148-SM multiples.
inline int grid_for(const bv_ctx *ctx, size_t work_items, int block, int max_blocks_per_sm) {
    size_t need = (work_items + block - 1) / block;
    size_t cap = (size_t)ctx->sm_count * max_blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

}  // namespace bv
