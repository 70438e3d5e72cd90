// lsu_bench.cu -- what one shared-memory instruction costs on B200 (round 2 design micro-benchmark, not part of the library).
// Every kernel runs `iters` iterations of a body with U independent shared-memory operations per thread on pseudo-random
// addresses generated in registers (one IMAD + one shift per operation), 1 block of 256/512/1024 threads per SM x 148 SMs.
// Reported: SM clocks per WARP-instruction of the measured kind (clock64 per block, averaged), i.e. the reciprocal
// throughput the colour-balance passes run against.
//   lds8      LDS.U8  from a 256-byte table               (pass 2 / pass 3 byte tables, ~2 words per bank)
//   lds8rep   LDS.U8  from a per-lane replica             (a 128-byte row per index, lane l reads word l: bank = lane, conflict-free)
//   lds32     LDS.32  from a 256-entry int table          (sdiv / hdiv)
//   lds16c    LDS.U16 from a 3072-entry table             (Lab cube-root table)
//   atoms     ATOMS.POPC.INC on a per-warp 256-bin histogram, all lanes active
//   atomsK    the same with only lanes whose random value falls below K/32 active (K = 0, 1, 4, 16)
//   alu       the address arithmetic alone (baseline to subtract)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at line %d\n", cudaGetErrorString(e_), __LINE__); exit(1); } } while (0)

constexpr int U = 16;

template <int MODE>
__global__ void __launch_bounds__(1024) bench(uint32_t *out, long long *clocks, int iters, uint32_t frac) {
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t *sm32 = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < 24576; i += blockDim.x) sm32[i] = i * 2654435761u >> 8;   // 96 KB
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = (blockIdx.x * 1024 + threadIdx.x) * 747796405u + 2891336453u;
    uint32_t acc = 0;
    uint32_t *hist = sm32 + 8192 + warp * 256;   // per-warp histogram (32 warps x 1 KB above the first 32 KB)
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
            x = x * 1664525u + 1013904223u;
            const uint32_t r = x >> 24;             // 0..255
            if (MODE == 0) acc += r;                                                        // alu
            if (MODE == 1) acc += smem[r];                                                  // lds8
            if (MODE == 2) acc += smem[(r << 7) + (lane << 2)];                             // lds8rep (32 KB)
            if (MODE == 3) acc += sm32[r];                                                  // lds32
            if (MODE == 4) acc += reinterpret_cast<uint16_t *>(smem)[(x >> 20) % 3072u];    // lds16c
            if (MODE == 5) atomicAdd(&hist[r], 1u);                                         // atoms
            if (MODE == 6) { if (((x >> 8) & 0xFFFFu) < frac) atomicAdd(&hist[r], 1u); }    // atoms, a fraction of lanes
            if (MODE == 7) acc += sm32[(r << 5) + lane];                                    // lds32 conflict-free replica (32 KB)
            // image-like data: a warp's 32 values fall into a window of `frac` bins, so several lanes share an address
            // frac = window - 1 (a power of two minus one): no division in the loop
            if (MODE == 8) atomicAdd(&hist[100 + (r & frac)], 1u);                          // per-warp histogram
            if (MODE == 9) atomicAdd(&sm32[((100 + (r & frac)) << 5) + lane], 1u);          // per-lane striped (32 KB, bank = lane)
            if (MODE == 10) atomicAdd(&sm32[((100 + (r & frac)) << 3) + (lane & 7)], 1u);   // 8 copies (8 KB)
            if (MODE == 11) atomicAdd(&sm32[((100 + (r & frac)) << 1) + (lane & 1)], 1u);   // 2 copies
        }
    }
    const long long t1 = clock64();
    if (threadIdx.x == 0) clocks[blockIdx.x] = t1 - t0;
    if (acc == 0xFFFFFFFFu) out[0] = acc + hist[lane];
}

template <int MODE>
static void run(const char *name, int threads, int iters, uint32_t frac, uint32_t *d_out, long long *d_clk, double alu_base) {
    CK(cudaFuncSetAttribute(bench<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
    bench<MODE><<<148, threads, 98304>>>(d_out, d_clk, iters, frac);
    CK(cudaDeviceSynchronize());
    bench<MODE><<<148, threads, 98304>>>(d_out, d_clk, iters, frac);
    CK(cudaDeviceSynchronize());
    long long h[148];
    CK(cudaMemcpy(h, d_clk, sizeof(h), cudaMemcpyDeviceToHost));
    double avg = 0;
    for (int i = 0; i < 148; ++i) avg += (double)h[i];
    avg /= 148;
    const double warp_instr = (double)iters * U * (threads / 32);
    printf("%-14s thr=%4d  %7.3f clk / warp-instruction   (minus address arithmetic: %7.3f)\n", name, threads, avg / warp_instr,
           avg / warp_instr - alu_base);
}

int main() {
    uint32_t *d_out;
    long long *d_clk;
    CK(cudaMalloc(&d_out, 64));
    CK(cudaMalloc(&d_clk, 148 * sizeof(long long)));
    const int iters = 2000;
    for (int threads : {512, 1024}) {
        // baseline
        CK(cudaFuncSetAttribute(bench<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 98304));
        bench<0><<<148, threads, 98304>>>(d_out, d_clk, iters, 0);
        CK(cudaDeviceSynchronize());
        long long h[148];
        CK(cudaMemcpy(h, d_clk, sizeof(h), cudaMemcpyDeviceToHost));
        double avg = 0;
        for (int i = 0; i < 148; ++i) avg += (double)h[i];
        const double base = avg / 148 / ((double)iters * U * (threads / 32));
        printf("alu        thr=%4d  %7.3f clk / warp-iteration of the address arithmetic\n", threads, base);
        run<1>("lds8", threads, iters, 0, d_out, d_clk, base);
        run<2>("lds8rep", threads, iters, 0, d_out, d_clk, base);
        run<3>("lds32", threads, iters, 0, d_out, d_clk, base);
        run<7>("lds32rep", threads, iters, 0, d_out, d_clk, base);
        run<4>("lds16c", threads, iters, 0, d_out, d_clk, base);
        run<5>("atoms", threads, iters, 0, d_out, d_clk, base);
        run<6>("atoms0", threads, iters, 0, d_out, d_clk, base);
        run<6>("atoms1/32", threads, iters, 65536 / 32, d_out, d_clk, base);
        run<6>("atoms4/32", threads, iters, 65536 / 8, d_out, d_clk, base);
        run<6>("atoms16/32", threads, iters, 65536 / 2, d_out, d_clk, base);
        for (uint32_t win : {1u, 4u, 16u, 64u, 256u}) {
            char nm[32];
            snprintf(nm, sizeof nm, "atomsW%u", win); run<8>(nm, threads, iters, win - 1, d_out, d_clk, base);
            snprintf(nm, sizeof nm, "atomsW%u/s32", win); run<9>(nm, threads, iters, win - 1, d_out, d_clk, base);
            snprintf(nm, sizeof nm, "atomsW%u/s8", win); run<10>(nm, threads, iters, win - 1, d_out, d_clk, base);
            snprintf(nm, sizeof nm, "atomsW%u/s2", win); run<11>(nm, threads, iters, win - 1, d_out, d_clk, base);
        }
    }
    return 0;
}
