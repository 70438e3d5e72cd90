// balance.cuh -- device-side state of the colour balance and the chunking policy of a batch, shared by balance.cu and
// stage.cu.
#pragma once
#include "common.cuh"

namespace bv {

// Chunking of a batch (bv_set_option / BV_* environment variables read at bv_create, see api.cu): independent chunks in
// flight on side streams, and the input bytes per chunk that keep a chunk and its H,S,V scratch in L2 across the passes.
inline int side_streams(const bv_ctx *ctx) {
    const int v = ctx->opt[BV_OPT_SIDE_STREAMS] > 0 ? ctx->opt[BV_OPT_SIDE_STREAMS] : 4;
    return v > BV_MAX_SIDE ? BV_MAX_SIDE : v;
}
inline size_t l2_chunk_bytes(const bv_ctx *ctx) { return (size_t)(ctx->opt[BV_OPT_L2_CHUNK_MB] > 0 ? ctx->opt[BV_OPT_L2_CHUNK_MB] : 33) << 20; }

// Runs fn(f0, nf) for consecutive chunks of the batch, alternating over the side streams (fork from / join into the
// context's stream).  ctx->overlapped tells the kernels' grid sizing whether chunks share the SMs.
template <class Fn>
int for_chunks_on_side_streams(bv_ctx *ctx, int batch, int chunk, Fn fn) {
    if (chunk < 1) chunk = 1;
    const int nchunks = (batch + chunk - 1) / chunk;
    int nside = side_streams(ctx);
    if (nside > nchunks) nside = nchunks;
    if (ctx->prof) nside = 1;  // per-kernel timing wants serialised launches
    cudaStream_t main_stream = ctx->stream;
    ctx->overlapped = nside > 1;
    if (nside > 1) {
        BV_CUDA(cudaEventRecord(ctx->ev_fork, main_stream));
        for (int i = 0; i < nside; ++i) BV_CUDA(cudaStreamWaitEvent(ctx->side[i], ctx->ev_fork, 0));
    }
    struct Restore {  // every exit path puts the context's stream back
        bv_ctx *c;
        cudaStream_t s;
        ~Restore() { c->stream = s; }
    } restore{ctx, main_stream};
    for (int k = 0; k < nchunks; ++k) {
        const int f0 = k * chunk, nf = (batch - f0 < chunk) ? batch - f0 : chunk;
        if (nside > 1) ctx->stream = ctx->side[k % nside];
        BV_TRY(fn(f0, nf));
    }
    ctx->stream = main_stream;
    if (nside > 1)
        for (int i = 0; i < nside; ++i) {
            BV_CUDA(cudaEventRecord(ctx->ev_join[i], ctx->side[i]));
            BV_CUDA(cudaStreamWaitEvent(main_stream, ctx->ev_join[i], 0));
        }
    return BV_OK;
}

// Per-frame working state in HBM (3.9 KB + 1.75 KB of tables per tile).
struct BalFrame {
    uint32_t hist_bgr[3][256];  // pass 1: histograms of B, G, R
    uint32_t hist_sv[2][256];   // pass 2: histograms of S, V after the BGR tables
    uint8_t lut_bgr[3][256];    // clip -> equalise -> rgb-contrast, composed per channel
    uint8_t lut_sv[2][256];     // clip -> stretch for S and V
    uint32_t ticket[2];         // blocks of pass 1 / pass 2 that have merged their histograms
    bv_balance_stats stats;
};

// Tiled equalisation (horizontal_blocks x vertical_blocks > 1, color_balance.cpp:441-544): every
// tile has its own local means, hence its own gains and composed tables.
struct BalTile {
    uint32_t hist[3][256];
    uint8_t lut[3][256];
};

struct TileGeom {
    int hb, vb;  // tiles across / down
    int bw, bh;  // tile size in pixels (the tiling must divide the frame)
    int width, height;
};

// What the final pass does with each balanced pixel.
struct BalOutputs {
    uint8_t *balanced;   // BGR after balance (may be null)
    uint8_t *converted;  // after the conversion CODE (may be null)
    uint8_t *mask;       // uint8 0/255 in-range mask (may be null)
    uint16_t *mask_bits; // bit-packed mask, one uint16 per 16-px group (needs width % 16 == 0)
    uint8_t lo[3], hi[3];
};

// Enqueues the complete colour balance of `batch` frames.  `out.balanced == src` is allowed.
// `after_chunk`, if given, is called for every chunk of frames [f0, f0 + nf) right after its last
// pass has been enqueued, with ctx->stream set to the stream that chunk runs on: work the caller
// enqueues there (morphology on the chunk's mask bits) overlaps the other chunks' passes.  It is
// not called for tiled equalisation.
struct ChunkHook {
    int (*fn)(void *self, bv_ctx *ctx, int f0, int nf);
    void *self;
};
int balance_run(bv_ctx *ctx, const uint8_t *src, int batch, int height, int width, const bv_balance_params &prm,
                int cvt_code, const BalOutputs &out, bv_balance_stats *stats_host, const ChunkHook *after_chunk = nullptr);

// Convert (+inRange) without balance, writing any of converted / mask / mask_bits.
int convert_run(bv_ctx *ctx, const uint8_t *src, int batch, int height, int width, int cvt_code,
                const BalOutputs &out);

}  // namespace bv
