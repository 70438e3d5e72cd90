// api.cu -- context management and error plumbing of libb200vision.so.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>

#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"
#include "lab_tables.inc"

namespace bv {

int rcp_tables_check(bv_ctx *ctx);  // balance.cu

static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int ensure_scratch(bv_ctx *ctx, int slot, size_t bytes) {
    if (ctx->scratch_bytes[slot] >= bytes) return BV_OK;
    // grow-only; steady state performs no allocation.  cudaFree synchronises the device, so any
    // kernel still using the old block has finished before it is released.
    if (ctx->scratch[slot]) {
        BV_CUDA(cudaFree(ctx->scratch[slot]));
        ctx->scratch[slot] = nullptr;
        ctx->scratch_bytes[slot] = 0;
    }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&ctx->scratch[slot], want);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu bytes) for scratch slot %d: %s", want, slot, cudaGetErrorString(e));
        (void)cudaGetLastError();
        return BV_ERR_NOMEM;
    }
    ctx->scratch_bytes[slot] = want;
    return BV_OK;
}

// ---- per-kernel timing with CUDA events on the launching stream (bench.py's roofline leg) ----
struct ProfRecord {
    const char *name;
    cudaEvent_t start, stop;
};
struct Profiler {
    std::vector<ProfRecord> records;
    std::vector<cudaEvent_t> pool;
    cudaEvent_t get() {
        if (!pool.empty()) {
            cudaEvent_t e = pool.back();
            pool.pop_back();
            return e;
        }
        cudaEvent_t e;
        cudaEventCreate(&e);
        return e;
    }
};

void prof_begin(bv_ctx *ctx, const char *kernel) {
    Profiler *p = (Profiler *)ctx->prof;
    ProfRecord r{kernel, p->get(), p->get()};
    cudaEventRecord(r.start, ctx->stream);
    p->records.push_back(r);
}

void prof_end(bv_ctx *ctx) {
    Profiler *p = (Profiler *)ctx->prof;
    cudaEventRecord(p->records.back().stop, ctx->stream);
}

}  // namespace bv

using namespace bv;

extern "C" int bv_profile_enable(bv_ctx *ctx, int on) {
    BV_REQUIRE(ctx, "null context");
    if (on && !ctx->prof) ctx->prof = new Profiler();
    if (!on && ctx->prof) {
        Profiler *p = (Profiler *)ctx->prof;
        cudaStreamSynchronize(ctx->stream);
        for (auto &r : p->records) {
            cudaEventDestroy(r.start);
            cudaEventDestroy(r.stop);
        }
        for (auto e : p->pool) cudaEventDestroy(e);
        delete p;
        ctx->prof = nullptr;
    }
    return BV_OK;
}

extern "C" int bv_profile_dump(bv_ctx *ctx, char *buf, size_t cap) {
    BV_REQUIRE(ctx && buf && cap > 2, "null argument");
    BV_REQUIRE(ctx->prof, "profiling is not enabled");
    Profiler *p = (Profiler *)ctx->prof;
    BV_CUDA(cudaStreamSynchronize(ctx->stream));
    std::map<std::string, std::pair<long, double>> agg;
    for (auto &r : p->records) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.start, r.stop) != cudaSuccess) (void)cudaGetLastError();
        std::string name(r.name);
        // "(final_kernel<MODE, CODE, true>)" -> "final_kernel"
        size_t b = name.find_first_not_of("( ");
        size_t e = name.find_first_of("<) ", b);
        name = name.substr(b, e == std::string::npos ? std::string::npos : e - b);
        auto &a = agg[name];
        a.first += 1;
        a.second += ms;
        p->pool.push_back(r.start);
        p->pool.push_back(r.stop);
    }
    p->records.clear();
    std::string out = "{";
    bool first = true;
    for (auto &kv : agg) {
        char tmp[256];
        snprintf(tmp, sizeof(tmp), "%s\"%s\": {\"launches\": %ld, \"ms\": %.6f}", first ? "" : ", ", kv.first.c_str(),
                 kv.second.first, kv.second.second);
        out += tmp;
        first = false;
    }
    out += "}";
    if (out.size() + 1 > cap) {
        set_error("bv_profile_dump: buffer too small (%zu needed)", out.size() + 1);
        return BV_ERR_CAPACITY;
    }
    memcpy(buf, out.c_str(), out.size() + 1);
    return BV_OK;
}

extern "C" int bv_version(void) { return BV_VERSION; }

extern "C" const char *bv_last_error(void) { return g_error; }

extern "C" int bv_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" void bv_balance_default(bv_balance_params *p) {
    if (!p) return;
    // defaults of balance(), modules/color_balance.py:93-96
    p->equalize_rgb = 1;
    p->rgb_contrast_correct = 0;
    p->hsv_contrast_correct = 1;
    p->hsi_contrast_correct = 0;
    p->rgb_extrema_clipping = 1;
    p->adaptive_cast_correction = 0;
    p->horizontal_blocks = 1;
    p->vertical_blocks = 1;
}

extern "C" int bv_create(int device, bv_ctx **out) {
    BV_REQUIRE(out, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("bv_create: no usable CUDA device (%s); this library has no CPU path",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        (void)cudaGetLastError();
        return BV_ERR_CUDA;
    }
    BV_REQUIRE(device >= 0 && device < n, "device index out of range");
    BV_CUDA(cudaSetDevice(device));
    bv_ctx *ctx = (bv_ctx *)calloc(1, sizeof(bv_ctx));
    if (!ctx) {
        set_error("bv_create: out of host memory");
        return BV_ERR_NOMEM;
    }
    ctx->device = device;
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        set_error("cudaGetDeviceProperties: %s", cudaGetErrorString(e));
        free(ctx);
        return BV_ERR_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
        set_error("cudaStreamCreate: %s", cudaGetErrorString(e));
        free(ctx);
        return BV_ERR_CUDA;
    }
    ctx->stream = ctx->own_stream;
    bool ok_aux = cudaStreamCreateWithFlags(&ctx->copy_in, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&ctx->copy_out, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok_aux && i < BV_MAX_CHUNKS; ++i)
        ok_aux = cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok_aux && i < BV_MAX_SIDE; ++i)
        ok_aux = cudaStreamCreateWithFlags(&ctx->side[i], cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&ctx->ev_join[i], cudaEventDisableTiming) == cudaSuccess;
    ok_aux = ok_aux && cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok_aux && i < BV_HOST_SLOTS; ++i)
        ok_aux = cudaEventCreateWithFlags(&ctx->ev_slot[i], cudaEventDisableTiming) == cudaSuccess;
    if (!ok_aux) {
        set_error("bv_create: stream/event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
        bv_destroy(ctx);
        return BV_ERR_CUDA;
    }
    double pow_tab[256];
    for (int x = 0; x < 256; ++x) pow_tab[x] = pow((255. - x) / 255., 0.25);  // color_balance.cpp:490
    bool ok = cudaMalloc(&ctx->d_lab_gamma, sizeof(kLabGammaTab)) == cudaSuccess &&
              cudaMalloc(&ctx->d_lab_cbrt, sizeof(kLabCbrtTab) + sizeof(kLabToYF) + sizeof(kLabInvGammaTab)) == cudaSuccess &&
              cudaMalloc(&ctx->d_pow_quarter, sizeof(pow_tab)) == cudaSuccess &&
              cudaMemcpy(ctx->d_lab_gamma, kLabGammaTab, sizeof(kLabGammaTab), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_lab_cbrt, kLabCbrtTab, sizeof(kLabCbrtTab), cudaMemcpyHostToDevice) == cudaSuccess &&
              // Lab -> BGR tables ride behind the cube-root table (convert.cuh: init_tabs<BV_LAB2BGR>)
              cudaMemcpy(ctx->d_lab_cbrt + kLabCbrtSize, kLabToYF, sizeof(kLabToYF), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_lab_cbrt + kLabCbrtSize + 512, kLabInvGammaTab, sizeof(kLabInvGammaTab), cudaMemcpyHostToDevice) == cudaSuccess &&
              cudaMemcpy(ctx->d_pow_quarter, pow_tab, sizeof(pow_tab), cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok) {
        set_error("bv_create: table upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        bv_destroy(ctx);
        return BV_ERR_CUDA;
    }
    if (bv::rcp_tables_check(ctx) != BV_OK) {
        bv_destroy(ctx);
        return BV_ERR_UNSUPPORTED;
    }
    static const char *const opt_env[BV_OPT_COUNT] = {"BV_HIST_BPS", "BV_FINAL_BPS", "BV_SIDE_STREAMS", "BV_L2_CHUNK_MB",
                                                      "BV_NO_HUE_TABLE", "BV_CONTOUR_POOL_CHUNKS", nullptr, "BV_MORPH_VARIANT",
                                                      nullptr, nullptr, "BV_MORPH_WARPS"};   // nullptr: retired option
    for (int i = 0; i < BV_OPT_COUNT; ++i) {
        const char *v = opt_env[i] ? getenv(opt_env[i]) : nullptr;
        ctx->opt[i] = v ? atoi(v) : 0;
    }
    *out = ctx;
    return BV_OK;
}

extern "C" int bv_set_option(bv_ctx *ctx, int option, int value) {
    BV_REQUIRE(ctx, "null context");
    BV_REQUIRE(option >= 0 && option < BV_OPT_COUNT, "unknown option");
    if (option == 6 || option == 8 || option == 9) {
        set_error("bv_set_option: option %d is retired (its alternative implementation was removed)", option);
        return BV_ERR_INVALID;
    }
    ctx->opt[option] = value > 0 ? value : 0;
    return BV_OK;
}

extern "C" void bv_destroy(bv_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    if (ctx->prof) {  // while the stream it synchronises on still exists
        ctx->stream = ctx->own_stream;
        bv_profile_enable(ctx, 0);
    }
    for (int i = 0; i < SCR_COUNT; ++i)
        if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
    if (ctx->d_lab_gamma) cudaFree(ctx->d_lab_gamma);
    if (ctx->d_lab_cbrt) cudaFree(ctx->d_lab_cbrt);
    if (ctx->d_pow_quarter) cudaFree(ctx->d_pow_quarter);
    if (ctx->lb_cache) free(ctx->lb_cache);
    if (ctx->d_luv_tab) cudaFree(ctx->d_luv_tab);
    if (ctx->d_bilinear_tab) cudaFree(ctx->d_bilinear_tab);
    if (ctx->d_ivl_flag) cudaFree(ctx->d_ivl_flag);
    for (int i = 0; i < BV_IVL_SLOTS; ++i)
        if (ctx->ivl[i].table) cudaFree(ctx->ivl[i].table);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_in) cudaStreamDestroy(ctx->copy_in);
    if (ctx->copy_out) cudaStreamDestroy(ctx->copy_out);
    for (int i = 0; i < BV_MAX_SIDE; ++i) {
        if (ctx->side[i]) cudaStreamDestroy(ctx->side[i]);
        if (ctx->ev_join[i]) cudaEventDestroy(ctx->ev_join[i]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    for (int i = 0; i < BV_HOST_SLOTS; ++i)
        if (ctx->ev_slot[i]) cudaEventDestroy(ctx->ev_slot[i]);
    for (int i = 0; i < BV_MAX_CHUNKS; ++i) {
        if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]);
        if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]);
    }
    (void)cudaGetLastError();
    free(ctx);
}

extern "C" int bv_sync(bv_ctx *ctx) {
    BV_REQUIRE(ctx, "null context");
    BV_CUDA(cudaSetDevice(ctx->device));
    BV_CUDA(cudaStreamSynchronize(ctx->stream));
    return BV_OK;
}

extern "C" void *bv_stream(bv_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

extern "C" int bv_set_stream(bv_ctx *ctx, void *cuda_stream) {
    BV_REQUIRE(ctx, "null context");
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return BV_OK;
}

extern "C" uint64_t bv_launch_count(const bv_ctx *ctx) { return ctx ? ctx->launches : 0; }
