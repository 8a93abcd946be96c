// microbench.cu -- measured FP64 roofline denominators.
//
// MEASURED_PEAKS.json (driver-written) holds HBM GB/s and dense bf16 TFLOP/s only; the H(k) build runs
// on the FP64 pipes, so bench.py measures the two FP64 peaks on the same GPU in the same run:
//   kind 0: register-resident mma.sync.m8n8k4.f64 chains (SASS DMMA.8x8x4), 16 independent accumulators/warp
//   kind 1: register-resident DFMA chains, 16 independent accumulators/thread
// Both run one CTA of 256 threads x 4 per SM for `iters` iterations and are timed with CUDA events.
// measure_int8_peak: the INT8 tensor-core rate an exact digit-product GEMM could run at -- one CTA per SM issues
// tcgen05.mma.cta_group::1.kind::i8 (M 128, N 256, K 32, int32 accumulators in tensor memory) on shared-memory
// operands that never change, so nothing but the MMA pipe is timed.
#include "tbk_kernels.h"
#include "tcgen05.cuh"

namespace tbk {

namespace {

constexpr int ACC = 16;

__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double seed) {
    double c0[ACC], c1[ACC];
#pragma unroll
    for (int i = 0; i < ACC; ++i) {
        c0[i] = seed * i;
        c1[i] = -seed * i;
    }
    double a = seed + threadIdx.x * 1e-9, b = seed - threadIdx.x * 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < ACC; ++i)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c0[i]), "+d"(c1[i])
                         : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < ACC; ++i) s += c0[i] + c1[i];
    if (s == 123.456) out[0] = s;  // keep the chain alive
}

__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double seed) {
    double c[ACC];
#pragma unroll
    for (int i = 0; i < ACC; ++i) c[i] = seed * i;
    const double a = 1.0 + seed * 1e-9, b = seed * 1e-12 + threadIdx.x * 1e-15;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < ACC; ++i) c[i] = fma(c[i], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < ACC; ++i) s += c[i];
    if (s == 123.456) out[0] = s;
}

// both at once: do DMMA and DFMA share a datapath?  (reported sum of both flop counts)
__global__ void __launch_bounds__(256) mixed_peak_kernel(double* out, int iters, double seed) {
    double c0[ACC], c1[ACC], f[ACC];
#pragma unroll
    for (int i = 0; i < ACC; ++i) {
        c0[i] = seed * i;
        c1[i] = -seed * i;
        f[i] = seed * i;
    }
    double a = seed + threadIdx.x * 1e-9, b = seed - threadIdx.x * 1e-9;
    const double fa = 1.0 + seed * 1e-9, fb = seed * 1e-12;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < ACC; ++i) {
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c0[i]), "+d"(c1[i])
                         : "d"(a), "d"(b));
            f[i] = fma(f[i], fa, fb);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < ACC; ++i) s += c0[i] + c1[i] + f[i];
    if (s == 123.456) out[0] = s;
}

constexpr int I8_M = 128, I8_N = 256, I8_K = 32;

// 128 threads, one CTA per SM (it holds all 512 tensor-memory columns: two 128 x 256 int32 accumulators, alternated so
// back-to-back MMAs do not all chain on one accumulator).  Operands: pseudo-random int8, so the pipe toggles as in a
// real product.  Layout: K-major, no swizzle; core matrix (row group g, K half h) at g * 256 + h * 128 bytes.
__global__ void __launch_bounds__(128, 1) i8_peak_kernel(int* out, long iters, uint32_t seed) {
    __shared__ __align__(1024) uint32_t ab[(I8_M + I8_N) * I8_K / 4];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tbase;
    const int tid = threadIdx.x;
    for (int i = tid; i < (I8_M + I8_N) * I8_K / 4; i += 128) {
        uint32_t x = (uint32_t)i * 2654435761u ^ seed;
        x ^= x >> 15;
        x *= 2246822519u;
        ab[i] = x ^ (x >> 13);
    }
    if (tid == 0) tc5::mbar_init(tc5::smem_u32(&bar), 1);
    if (tid < 32) {
        tc5::tmem_alloc(tc5::smem_u32(&tbase), 512);
        tc5::tmem_relinquish();
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the MMA
    tc5::fence_before_sync();
    __syncthreads();
    tc5::fence_after_sync();
    const uint32_t d = tbase;
    if (tid == 0) {
        const uint32_t a_addr = tc5::smem_u32(ab), b_addr = a_addr + I8_M * I8_K;
        const uint64_t adesc = tc5::smem_desc(a_addr, 128, 256), bdesc = tc5::smem_desc(b_addr, 128, 256);
        constexpr uint32_t idesc = tc5::idesc_s8(I8_M, I8_N);
        for (long it = 0; it < iters; ++it) tc5::mma_i8(d + (uint32_t)(it & 1) * I8_N, adesc, bdesc, idesc, it >= 2);
        tc5::commit(tc5::smem_u32(&bar));
        tc5::mbar_wait_sleep(tc5::smem_u32(&bar), 0);
    }
    tc5::fence_before_sync();
    __syncthreads();
    tc5::fence_after_sync();
    if (tid < 32) {
        uint32_t v;  // one lane of the result keeps the chain observable
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n tcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(d) : "memory");
        if (v == 0x9E3779B9u) out[0] = (int)v;
        tc5::fence_before_sync();
        __syncwarp();
        tc5::tmem_dealloc(d, 512);
    }
}

}  // namespace

double measure_int8_peak(long iters) {
    int dev = 0, sms = 0;
    if (iters < 1 || cudaGetDevice(&dev) != cudaSuccess) return -1.0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int* out = nullptr;
    if (cudaMalloc(&out, 4) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double best = -1.0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0);
        i8_peak_kernel<<<sms, 128>>>(out, iters, 0x12345u + rep);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double ops = (double)sms * (double)iters * 2.0 * I8_M * I8_N * I8_K;
        const double tops = ops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tops > best) best = tops;  // first rep is warm-up
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return best;
}

double measure_fp64_peak(int kind, int iters) {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return -1.0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    double* out = nullptr;
    if (cudaMalloc(&out, 8) != cudaSuccess) return -1.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    const int blocks = sms * 4;
    double best = -1.0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0);
        if (kind == 0) dmma_peak_kernel<<<blocks, 256>>>(out, iters, 1.0);
        else if (kind == 1) dfma_peak_kernel<<<blocks, 256>>>(out, iters, 1.0);
        else mixed_peak_kernel<<<blocks, 256>>>(out, iters, 1.0);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -1.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double flops;
        if (kind == 0) flops = (double)blocks * 8 /*warps*/ * (double)iters * ACC * 512.0;   // 8x8x4 MACs x 2
        else if (kind == 1) flops = (double)blocks * 256 * (double)iters * ACC * 2.0;
        else flops = (double)blocks * 8 * (double)iters * ACC * 512.0 + (double)blocks * 256 * (double)iters * ACC * 2.0;
        const double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;  // first rep is warm-up
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    return best;
}

}  // namespace tbk
