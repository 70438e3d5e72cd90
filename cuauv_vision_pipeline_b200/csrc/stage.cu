// stage.cu -- the fused per-frame stage and the host-memory entry points.
//
// bv_stage strings the kernels of balance.cu / morph.cu / ccl.cu together without ever
// materialising intermediates the caller did not ask for:
//
//   frame (BGR, 3 B/px) --[balance passes 1-2: statistics only]--> pass 3 (balance -> convert ->
//   inRange) --> bit-packed mask (1/8 B/px, L2 resident) --> binary morphology on bits -->
//   {uint8 mask (1 B/px), labels (4 B/px), blob table}
//
// which is modules/bins.py:13-27 / modules/red_buoy.py:21-44 behind an optional balance()
// (modules/preprocessor.py:87-88) in one call.
//
// bv_stage_host and the legacy process_frame symbol take HOST buffers (the reference's calling
// convention, modules/color_balance.py:93-110): upload, run, download, return when done.
#include <stdlib.h>

#include <mutex>

#include "balance.cuh"
#include "morph.cuh"

namespace bv {
static int validate_desc(const bv_stage_desc *d) {
    BV_REQUIRE(d, "null stage description");
    BV_REQUIRE(d->n_morph >= 0 && d->n_morph <= 4, "n_morph must be 0..4");
    for (int i = 0; i < d->n_morph; ++i) {
        BV_REQUIRE(d->morph_op[i] >= BV_MORPH_ERODE && d->morph_op[i] <= BV_MORPH_GRADIENT, "unknown morphology op");
        BV_REQUIRE(d->morph_kw[i] >= 1 && d->morph_kh[i] >= 1 && d->morph_kw[i] <= 255 && d->morph_kh[i] <= 255,
                   "structuring element size must be 1..255");
        BV_REQUIRE(d->morph_iters[i] >= 0, "iterations must be >= 0");
    }
    BV_REQUIRE(d->cvt_code == -1 || d->cvt_code == BV_BGR2HSV || d->cvt_code == BV_BGR2LAB ||
                   d->cvt_code == BV_BGR2GRAY || d->cvt_code == BV_BGR2YCRCB || d->cvt_code == BV_BGR2HLS,
               "cvt_code must be -1, BGR2HSV, BGR2LAB, BGR2GRAY, BGR2YCRCB or BGR2HLS");
    return BV_OK;
}

// Everything behind the threshold for frames f0 .. f0 + nf - 1, on the context's CURRENT stream: uint8 mask -> bits (odd
// widths), the morphology steps, bits -> uint8 mask, labels + moments.  All buffers are whole-batch buffers; the chunk works
// on its own slices, so the chunks of one call run concurrently on the side streams: the latency-bound union-find kernels
// of one chunk fill the SMs together with the issue-bound pixel passes of the next.
struct StageTail {
    const bv_stage_desc *desc;
    int height, width;
    bool bits_direct, want_label;
    uint32_t *bits, *tmp, *tmp2, *tmp3;   // whole batch
    const uint8_t *thr_mask;       // thresholded uint8 mask when the bits do not come straight from the pixel pass
    uint8_t *mask;                 // caller's mask (may be null)
    int32_t *labels;
    bv_blob *blobs;
    int max_blobs;
    int32_t *n_blobs;
    LabelScratch ls;
    int calls;

    int run(bv_ctx *c, int f0, int nf) {
        ++calls;
        const size_t fw = bits_frame_words(height, width), fpx = (size_t)height * width;
        uint32_t *b = bits + f0 * fw, *t = tmp + f0 * fw, *t2 = tmp2 + f0 * fw, *t3 = tmp3 + f0 * fw;
        uint8_t *m = mask ? mask + f0 * fpx : nullptr;
        if (!bits_direct) BV_TRY(mask_to_bits(c, thr_mask + f0 * fpx, b, nf, height, width));
        const uint32_t *res = b;
        if (desc->n_morph > 0) {
            bool chained = false;   // one launch for the whole chain; it also expands the final bits into the uint8 mask
            BV_TRY(morph_bits_chain(c, b, want_label ? t : nullptr, m, nf, height, width, desc->n_morph, desc->morph_op,
                                    desc->morph_kw, desc->morph_kh, desc->morph_iters, &chained));
            if (chained) {
                if (want_label) res = t;
            } else {
                for (int i = 0; i < desc->n_morph; ++i)
                    BV_TRY(morph_bits_rect(c, b, t, t2, t3, nf, height, width, desc->morph_op[i], desc->morph_kw[i], desc->morph_kh[i],
                                           desc->morph_iters[i]));
                if (m) BV_TRY(bits_to_mask(c, b, m, nf, height, width));
            }
        }
        if (want_label)
            BV_TRY(label_bits_slice(c, res, labels ? labels + f0 * fpx : nullptr, f0, nf, height, width,
                                    blobs ? blobs + (size_t)f0 * max_blobs : nullptr, max_blobs, n_blobs ? n_blobs + f0 : nullptr, ls));
        return BV_OK;
    }
    static int hook(void *self, bv_ctx *c, int f0, int nf) { return ((StageTail *)self)->run(c, f0, nf); }
};

// Runs fn(f0, nf) for consecutive chunks of the batch, alternating over the side streams (fork from / join into the
// context's stream), like balance_run does for its own chunks.
template <class Fn>
static int for_chunks_on_side_streams(bv_ctx *ctx, int batch, int chunk, Fn fn) {
    if (chunk < 1) chunk = 1;
    const int nchunks = (batch + chunk - 1) / chunk;
    int nside = ctx->opt[BV_OPT_SIDE_STREAMS] > 0 ? ctx->opt[BV_OPT_SIDE_STREAMS] : 4;
    if (nside > BV_MAX_SIDE) nside = BV_MAX_SIDE;
    if (nside > nchunks) nside = nchunks;
    if (ctx->prof) nside = 1;  // per-kernel timing wants serialised launches
    cudaStream_t main_stream = ctx->stream;
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

int stage_run(bv_ctx *ctx, const bv_stage_desc *desc, const uint8_t *src, int batch, int height, int width,
              uint8_t *balanced, uint8_t *converted, uint8_t *mask, int32_t *labels, bv_blob *blobs, int max_blobs,
              int32_t *n_blobs) {
    const size_t npx = (size_t)height * width;
    const bool want_label = desc->do_label && (labels || blobs || n_blobs);
    const bool need_bits = desc->n_morph > 0 || want_label;
    BalOutputs out;
    memset(&out, 0, sizeof(out));
    out.balanced = balanced;
    out.converted = converted;
    for (int k = 0; k < 3; ++k) {
        out.lo[k] = desc->lo[k];
        out.hi[k] = desc->hi[k];
    }
    const bool tiled = desc->do_balance && (desc->balance.horizontal_blocks != 1 || desc->balance.vertical_blocks != 1);
    StageTail tail;
    memset(&tail, 0, sizeof(tail));
    tail.desc = desc;
    tail.height = height;
    tail.width = width;
    tail.want_label = want_label;
    tail.mask = mask;
    tail.labels = labels;
    tail.blobs = blobs;
    tail.max_blobs = max_blobs;
    tail.n_blobs = n_blobs;
    if (need_bits) {
        const size_t words = (size_t)batch * bits_frame_words(height, width);
        BV_TRY(ensure_scratch(ctx, SCR_BITS_A, words * 4));
        BV_TRY(ensure_scratch(ctx, SCR_BITS_B, words * 12));   // tmp, tmp2, tmp3
        tail.bits = (uint32_t *)ctx->scratch[SCR_BITS_A];
        tail.tmp = (uint32_t *)ctx->scratch[SCR_BITS_B];
        tail.tmp2 = tail.tmp + words;
        tail.tmp3 = tail.tmp2 + words;
        const bool aligned = host_aligned16(src) && (!balanced || host_aligned16(balanced)) &&
                             (!converted || host_aligned16(converted)) && (!mask || host_aligned16(mask));
        tail.bits_direct = aligned && (width % 16 == 0) && !tiled;
        if (tail.bits_direct) {
            if (width % 32 != 0) BV_CUDA(cudaMemsetAsync(tail.bits, 0, words * 4, ctx->stream));
            out.mask_bits = (uint16_t *)tail.bits;
            if (desc->n_morph == 0) out.mask = mask;  // the thresholded mask is already final
        } else {
            // odd widths: go through a uint8 mask (the caller's buffer doubles as the intermediate)
            if (mask) {
                out.mask = mask;
            } else {
                BV_TRY(ensure_scratch(ctx, SCR_STAGE_IMG, (size_t)batch * npx));
                out.mask = (uint8_t *)ctx->scratch[SCR_STAGE_IMG];
            }
            tail.thr_mask = out.mask;
        }
        if (want_label) BV_TRY(label_scratch(ctx, batch, height, width, &tail.ls));   // before any stream forks
    } else {
        out.mask = mask;
    }
    const bool pixel_pass = out.balanced || out.converted || out.mask || out.mask_bits;
    if (desc->do_balance) {
        // balance_run spreads its chunks over the side streams and calls the hook behind every chunk's last pass
        ChunkHook hook{&StageTail::hook, &tail};
        const bool use_hook = need_bits && !tiled;
        if (pixel_pass)
            BV_TRY(balance_run(ctx, src, batch, height, width, desc->balance, desc->cvt_code, out, nullptr, use_hook ? &hook : nullptr));
        if (need_bits && tail.calls == 0) BV_TRY(tail.run(ctx, 0, batch));   // tiled / HSI paths do not chunk
        return BV_OK;
    }
    // no balance: chunks of whole frames (input + outputs of a chunk stay in L2 between its kernels), on the side streams
    // when the work is worth splitting
    int chunk = batch;
    if (need_bits && batch > 1) {
        const size_t l2_chunk = (size_t)(ctx->opt[BV_OPT_L2_CHUNK_MB] > 0 ? ctx->opt[BV_OPT_L2_CHUNK_MB] : 33) << 20;
        chunk = (int)(l2_chunk / (npx * 3));
        const int quarter = (batch + 3) / 4;
        if (chunk > quarter) chunk = quarter;
        const size_t min_px = (size_t)1 << 20;   // below ~1 Mpx per chunk the launches cost more than the overlap returns
        if ((size_t)chunk * npx < min_px) chunk = (int)((min_px + npx - 1) / npx);
        if (chunk < 1) chunk = 1;
        if (chunk > batch) chunk = batch;
    }
    const size_t cvt_bpp = desc->cvt_code == BV_BGR2GRAY ? 1 : 3;
    return for_chunks_on_side_streams(ctx, batch, chunk, [&](int f0, int nf) -> int {
        if (pixel_pass) {
            BalOutputs co = out;
            const size_t po = (size_t)f0 * npx;
            if (co.balanced) co.balanced += po * 3;
            if (co.converted) co.converted += po * cvt_bpp;
            if (co.mask) co.mask += po;
            if (co.mask_bits) co.mask_bits += (size_t)f0 * height * (((width + 31) / 32) * 2);
            BV_TRY(convert_run(ctx, src + po * 3, nf, height, width, desc->cvt_code, co));
        }
        if (need_bits) BV_TRY(tail.run(ctx, f0, nf));
        return BV_OK;
    });
}

// process-wide context behind the legacy symbol
static std::mutex g_legacy_mutex;
static bv_ctx *g_legacy_ctx = nullptr;

}  // namespace bv

using namespace bv;

extern "C" int bv_stage(bv_ctx *ctx, const bv_stage_desc *desc, const uint8_t *src_dev, int batch, int height, int width,
                        uint8_t *balanced_dev, uint8_t *converted_dev, uint8_t *mask_dev, int32_t *labels_dev,
                        bv_blob *blobs_dev, int max_blobs, int32_t *n_blobs_dev) {
    BV_REQUIRE(ctx && src_dev, "null context or source");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(max_blobs >= 0, "max_blobs must be >= 0");
    BV_TRY(validate_desc(desc));
    BV_CUDA(cudaSetDevice(ctx->device));
    return stage_run(ctx, desc, src_dev, batch, height, width, balanced_dev, converted_dev, mask_dev, labels_dev,
                     blobs_dev, blobs_dev ? max_blobs : 0, n_blobs_dev);
}

// Enqueues one host-buffer call on staging set `slot`: uploads, kernels, downloads; no synchronisation.
static int stage_host_enqueue(bv_ctx *ctx, int slot, const bv_stage_desc *desc, const uint8_t *src_host, int batch, int height,
                              int width, uint8_t *balanced_host, uint8_t *converted_host, uint8_t *mask_host,
                              int32_t *labels_host, bv_blob *blobs_host, int max_blobs, int32_t *n_blobs_host) {
    BV_REQUIRE(ctx && src_host, "null context or source");
    BV_REQUIRE(slot >= 0 && slot < BV_HOST_SLOTS, "slot must be 0 or 1");
    BV_REQUIRE(batch > 0 && height > 0 && width > 0, "batch, height and width must be positive");
    BV_REQUIRE(max_blobs >= 0, "max_blobs must be >= 0");
    BV_TRY(validate_desc(desc));
    BV_CUDA(cudaSetDevice(ctx->device));
    const size_t npx = (size_t)height * width;
    const size_t cvt_bpp = desc->cvt_code == BV_BGR2GRAY ? 1 : 3;
    if (!blobs_host) max_blobs = 0;
    // device staging for the whole batch, one set per slot: no buffer is reused inside one call, so the three
    // streams below need no back-pressure
    const int base = SCR_HOST_IN + slot * (SCR_HOST_NBLOBS - SCR_HOST_IN + 1);
    const int s_in = base, s_bal = base + (SCR_HOST_BAL - SCR_HOST_IN), s_cvt = base + (SCR_HOST_CVT - SCR_HOST_IN),
              s_mask = base + (SCR_HOST_MASK - SCR_HOST_IN), s_lab = base + (SCR_HOST_LABELS - SCR_HOST_IN),
              s_blobs = base + (SCR_HOST_BLOBS - SCR_HOST_IN), s_nb = base + (SCR_HOST_NBLOBS - SCR_HOST_IN);
    BV_TRY(ensure_scratch(ctx, s_in, (size_t)batch * npx * 3));
    if (balanced_host) BV_TRY(ensure_scratch(ctx, s_bal, (size_t)batch * npx * 3));
    if (converted_host) BV_TRY(ensure_scratch(ctx, s_cvt, (size_t)batch * npx * cvt_bpp));
    if (mask_host) BV_TRY(ensure_scratch(ctx, s_mask, (size_t)batch * npx));
    if (labels_host) BV_TRY(ensure_scratch(ctx, s_lab, (size_t)batch * npx * 4));
    if (max_blobs) BV_TRY(ensure_scratch(ctx, s_blobs, (size_t)batch * max_blobs * sizeof(bv_blob)));
    BV_TRY(ensure_scratch(ctx, s_nb, (size_t)batch * sizeof(int32_t)));
    uint8_t *d_in = (uint8_t *)ctx->scratch[s_in];
    uint8_t *d_bal = balanced_host ? (uint8_t *)ctx->scratch[s_bal] : nullptr;
    uint8_t *d_cvt = converted_host ? (uint8_t *)ctx->scratch[s_cvt] : nullptr;
    uint8_t *d_mask = mask_host ? (uint8_t *)ctx->scratch[s_mask] : nullptr;
    int32_t *d_lab = labels_host ? (int32_t *)ctx->scratch[s_lab] : nullptr;
    bv_blob *d_blobs = max_blobs ? (bv_blob *)ctx->scratch[s_blobs] : nullptr;
    int32_t *d_nb = (int32_t *)ctx->scratch[s_nb];

    // chunked three-stage pipeline: H2D (copy-in stream) -> kernels (context stream) -> D2H
    // (copy-out stream); PCIe is full duplex, so uploads of chunk k+1 overlap downloads of k-1.
    // A lone call wants small pieces (16 MB: its first upload and last download overlap nothing); when the other slot
    // is in flight the overlap comes from that call, and whole batches keep the kernels efficient and the copies long
    // (tools/e2e_pipe_sweep.py: two batches in flight 5 056 frames/s with 16 MB pieces, 5 613 with one piece per batch).
    static const long env_chunk_mb = []() {
        const char *e = getenv("BV_HOST_CHUNK_MB");
        return e ? atol(e) : 0L;
    }();
    const bool pipelined = ctx->slot_busy[1 - slot] != 0;
    const size_t chunk_bytes = (size_t)(env_chunk_mb > 0 ? env_chunk_mb : (pipelined ? 256 : 16)) << 20;
    int chunk = (int)(chunk_bytes / (npx * 3));
    if (chunk < 1) chunk = 1;
    if (chunk > batch) chunk = batch;
    int nchunks = (batch + chunk - 1) / chunk;
    if (nchunks > BV_MAX_CHUNKS) {
        chunk = (batch + BV_MAX_CHUNKS - 1) / BV_MAX_CHUNKS;
        nchunks = (batch + chunk - 1) / chunk;
    }
    // BV_HOST_TIMELINE=1 (diagnostic): device time stamps of every chunk's upload, kernels and download, to stderr
    static const bool timeline = getenv("BV_HOST_TIMELINE") != nullptr;
    cudaEvent_t tl[3 * BV_MAX_CHUNKS + 1];
    if (timeline) {
        for (int i = 0; i < 3 * nchunks + 1; ++i) BV_CUDA(cudaEventCreate(&tl[i]));
        BV_CUDA(cudaEventRecord(tl[3 * nchunks], ctx->copy_in));
    }
    // every upload is enqueued before the first kernel: a download into PAGEABLE host memory (small result tables in plain
    // numpy arrays) blocks the calling thread until its chunk's kernels are done, and must not hold back the next uploads.
    // The per-chunk events are shared by both slots: a stream wait refers to the record that precedes it in program order.
    for (int k = 0; k < nchunks; ++k) {
        const int f0 = k * chunk, nf = (batch - f0 < chunk) ? batch - f0 : chunk;
        const size_t po = (size_t)f0 * npx;
        BV_CUDA(cudaMemcpyAsync(d_in + po * 3, src_host + po * 3, (size_t)nf * npx * 3, cudaMemcpyHostToDevice,
                                ctx->copy_in));
        if (timeline) BV_CUDA(cudaEventRecord(tl[3 * k], ctx->copy_in));
        BV_CUDA(cudaEventRecord(ctx->ev_in[k], ctx->copy_in));
    }
    for (int k = 0; k < nchunks; ++k) {
        const int f0 = k * chunk, nf = (batch - f0 < chunk) ? batch - f0 : chunk;
        const size_t po = (size_t)f0 * npx;
        BV_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[k], 0));
        BV_TRY(stage_run(ctx, desc, d_in + po * 3, nf, height, width, d_bal ? d_bal + po * 3 : nullptr,
                         d_cvt ? d_cvt + po * cvt_bpp : nullptr, d_mask ? d_mask + po : nullptr,
                         d_lab ? d_lab + po : nullptr, d_blobs ? d_blobs + (size_t)f0 * max_blobs : nullptr, max_blobs,
                         d_nb + f0));
        if (timeline) BV_CUDA(cudaEventRecord(tl[3 * k + 1], ctx->stream));
        BV_CUDA(cudaEventRecord(ctx->ev_done[k], ctx->stream));
        BV_CUDA(cudaStreamWaitEvent(ctx->copy_out, ctx->ev_done[k], 0));
        if (balanced_host)
            BV_CUDA(cudaMemcpyAsync(balanced_host + po * 3, d_bal + po * 3, (size_t)nf * npx * 3, cudaMemcpyDeviceToHost,
                                    ctx->copy_out));
        if (converted_host)
            BV_CUDA(cudaMemcpyAsync(converted_host + po * cvt_bpp, d_cvt + po * cvt_bpp, (size_t)nf * npx * cvt_bpp,
                                    cudaMemcpyDeviceToHost, ctx->copy_out));
        if (mask_host)
            BV_CUDA(cudaMemcpyAsync(mask_host + po, d_mask + po, (size_t)nf * npx, cudaMemcpyDeviceToHost, ctx->copy_out));
        if (labels_host)
            BV_CUDA(cudaMemcpyAsync(labels_host + po, d_lab + po, (size_t)nf * npx * 4, cudaMemcpyDeviceToHost,
                                    ctx->copy_out));
        if (max_blobs)
            BV_CUDA(cudaMemcpyAsync(blobs_host + (size_t)f0 * max_blobs, d_blobs + (size_t)f0 * max_blobs,
                                    (size_t)nf * max_blobs * sizeof(bv_blob), cudaMemcpyDeviceToHost, ctx->copy_out));
        if (n_blobs_host && desc->do_label)
            BV_CUDA(cudaMemcpyAsync(n_blobs_host + f0, d_nb + f0, (size_t)nf * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                    ctx->copy_out));
        if (timeline) BV_CUDA(cudaEventRecord(tl[3 * k + 2], ctx->copy_out));
    }
    BV_CUDA(cudaEventRecord(ctx->ev_slot[slot], ctx->copy_out));   // everything of this call precedes it on copy_out
    ctx->slot_busy[slot] = 1;
    if (timeline) {
        BV_CUDA(cudaEventSynchronize(ctx->ev_slot[slot]));
        for (int k = 0; k < nchunks; ++k) {
            float a = 0, b = 0, c = 0;
            cudaEventElapsedTime(&a, tl[3 * nchunks], tl[3 * k]);
            cudaEventElapsedTime(&b, tl[3 * nchunks], tl[3 * k + 1]);
            cudaEventElapsedTime(&c, tl[3 * nchunks], tl[3 * k + 2]);
            fprintf(stderr, "bv_stage_host chunk %2d: uploaded %8.1f us, kernels done %8.1f us, downloaded %8.1f us\n", k, a * 1e3,
                    b * 1e3, c * 1e3);
        }
        for (int i = 0; i < 3 * nchunks + 1; ++i) cudaEventDestroy(tl[i]);
    }
    return BV_OK;
}

// An enqueue that failed half-way (bad description, out of memory) may have copies and kernels of the call in flight with no
// completion event recorded: wait for them, so that the caller's buffers and the slot's staging are quiescent on return.
static void drain_after_failed_enqueue(bv_ctx *ctx) {
    cudaStreamSynchronize(ctx->copy_in);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copy_out);
    (void)cudaGetLastError();
}

extern "C" int bv_stage_host_wait(bv_ctx *ctx, int slot) {
    BV_REQUIRE(ctx, "null context");
    BV_REQUIRE(slot >= 0 && slot < BV_HOST_SLOTS, "slot must be 0 or 1");
    if (!ctx->slot_busy[slot]) return BV_OK;
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_CUDA(cudaEventSynchronize(ctx->ev_slot[slot]));
    ctx->slot_busy[slot] = 0;
    return BV_OK;
}

extern "C" int bv_stage_host_submit(bv_ctx *ctx, int slot, const bv_stage_desc *desc, const uint8_t *src_host, int batch,
                                    int height, int width, uint8_t *balanced_host, uint8_t *converted_host, uint8_t *mask_host,
                                    int32_t *labels_host, bv_blob *blobs_host, int max_blobs, int32_t *n_blobs_host) {
    BV_REQUIRE(ctx, "null context");
    BV_REQUIRE(slot >= 0 && slot < BV_HOST_SLOTS, "slot must be 0 or 1");
    BV_TRY(bv_stage_host_wait(ctx, slot));   // the slot's device staging is free again once its previous call has completed
    const int st = stage_host_enqueue(ctx, slot, desc, src_host, batch, height, width, balanced_host, converted_host, mask_host,
                                      labels_host, blobs_host, max_blobs, n_blobs_host);
    if (st != BV_OK) drain_after_failed_enqueue(ctx);
    return st;
}

extern "C" int bv_stage_host(bv_ctx *ctx, const bv_stage_desc *desc, const uint8_t *src_host, int batch, int height,
                             int width, uint8_t *balanced_host, uint8_t *converted_host, uint8_t *mask_host,
                             int32_t *labels_host, bv_blob *blobs_host, int max_blobs, int32_t *n_blobs_host) {
    BV_REQUIRE(ctx, "null context");
    BV_TRY(bv_stage_host_wait(ctx, 0));
    const int st = stage_host_enqueue(ctx, 0, desc, src_host, batch, height, width, balanced_host, converted_host, mask_host,
                                      labels_host, blobs_host, max_blobs, n_blobs_host);
    if (st != BV_OK) {
        drain_after_failed_enqueue(ctx);
        return st;
    }
    BV_TRY(bv_stage_host_wait(ctx, 0));
    BV_CUDA(cudaStreamSynchronize(ctx->stream));
    return BV_OK;
}

extern "C" int process_frame(unsigned char *arr, size_t height, size_t width, size_t depth, bool equalize_rgb,
                             bool rgb_contrast_correct, bool hsv_contrast_correct, bool hsi_contrast_correct,
                             bool rgb_extrema_clipping, bool adaptive_cast_correction, int horizontal_blocks,
                             int vertical_blocks) {
    if (!arr || height == 0 || width == 0 || depth != 3 || height > 65535 || width > 65535) {
        set_error("process_frame: need a non-empty height x width x 3 uint8 buffer");
        return BV_ERR_INVALID;
    }
    std::lock_guard<std::mutex> lock(g_legacy_mutex);
    if (!g_legacy_ctx) {
        const char *e = getenv("BV_DEVICE");
        BV_TRY(bv_create(e ? atoi(e) : 0, &g_legacy_ctx));
    }
    bv_stage_desc d;
    memset(&d, 0, sizeof(d));
    d.do_balance = 1;
    d.balance.equalize_rgb = equalize_rgb;
    d.balance.rgb_contrast_correct = rgb_contrast_correct;
    d.balance.hsv_contrast_correct = hsv_contrast_correct;
    d.balance.hsi_contrast_correct = hsi_contrast_correct;
    d.balance.rgb_extrema_clipping = rgb_extrema_clipping;
    d.balance.adaptive_cast_correction = adaptive_cast_correction;
    d.balance.horizontal_blocks = horizontal_blocks;
    d.balance.vertical_blocks = vertical_blocks;
    d.cvt_code = -1;
    for (int k = 0; k < 3; ++k) d.hi[k] = 255;
    return bv_stage_host(g_legacy_ctx, &d, arr, 1, (int)height, (int)width, arr, nullptr, nullptr, nullptr, nullptr, 0,
                         nullptr);
}

// ---- pinned host memory helpers (full PCIe speed for the *_host entry points) -----------------
extern "C" void *bv_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
        set_error("cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}

extern "C" void bv_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

extern "C" int bv_host_register(void *p, size_t bytes) {
    BV_REQUIRE(p && bytes, "null buffer");
    BV_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return BV_OK;
}

extern "C" int bv_host_unregister(void *p) {
    BV_REQUIRE(p, "null buffer");
    BV_CUDA(cudaHostUnregister(p));
    return BV_OK;
}
