// tcgen05.cuh -- the fifth-generation tensor core (tcgen05, sm_100a) as inline PTX: tensor-memory allocation, shared
// memory / instruction descriptors, MMA issue and commit.  Layout conventions are those of the PTX ISA
// ("Matrix descriptors", "Instruction descriptor"); only the forms the kernels here use are wrapped.
#pragma once
#include <stdint.h>

namespace tbk {
namespace tc5 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Warp-wide: allocate `cols` (power of two, 32 .. 512) tensor-memory columns; the base address lands in *dst (shared).
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor, no swizzle.  The operand is a grid of 8-row x 16-byte core matrices (128 contiguous
// bytes each); lbo = byte distance between core matrices adjacent along K, sbo = between 8-row groups along M / N.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46);  // bits 46-48 = 0b001: sm_100 descriptor
}

// Instruction descriptor of kind::i8: signed 8-bit A and B, both K-major, int32 accumulator, M x N.
__host__ __device__ constexpr uint32_t idesc_s8(int m, int n) {
    return (2u << 4)                      // D: s32
           | (1u << 7) | (1u << 10)       // A, B: signed
           | ((uint32_t)(n >> 3) << 17)   // N >> 3
           | ((uint32_t)(m >> 4) << 24);  // M >> 4
}

// D[tmem] (+)= A[smem] . B[smem]^T, issued by one thread; accumulate = 0 overwrites D.
__device__ __forceinline__ void mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

// Spin (try_wait suspends in hardware between polls) until the phase of the given parity completes; a completion that
// never comes becomes a trap, not a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    uint32_t spins = 0;
    do {
        if (++spins > (1u << 28)) __trap();
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
    } while (!ok);
}

// 1-D TMA bulk copy global -> shared, completion counted in bytes on the mbarrier.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

// Wait for the phase of the given parity to complete.  A completion that never comes (a lost arrive) traps after
// ~2^24 sleeps of >= 1 us instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    for (uint32_t spins = 0;; ++spins) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) return;
        if (spins > (1u << 24)) __trap();
        __nanosleep(1000);
    }
}

// Arrive once on the mbarrier when every MMA this thread issued before has completed.
__device__ __forceinline__ void commit(uint32_t bar_smem) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_smem) : "memory");
}

}  // namespace tc5
}  // namespace tbk
