// hk_gemm_i8.cu -- H(k) build from exact INT8 tensor-core digit products (tcgen05 kind::i8, sm_100a).
//
// The GEMM of hk_gemm.cu, Hp[k, j] = sum_r Q[k, r] W[r, j], with both operands split into balanced 7-bit digits
// (the Ozaki scheme; tests/hk_digits_reference.py restates it in Python and pins its error bound):
//     q    = sum_{a=0..7} q_a 2^(-6-7a),  q_a in [-64, 64], rounded at 2^-55        (|q| <= 1: cos / sin)
//     W/s_j = sum_{b=0..8} w_b 2^(-6-7b),  w_b in [-64, 64], rounded at 2^-62       (s_j: power of two > max_r |W_rj|)
// A digit product (a, b) belongs to class c = a + b, weight 2^(-12-7c).  The classes c <= 9 (51 products) are summed
// exactly in int32 (at most 8 pairs x 64^2 per row: < 2^31 for K < 2^16 rows), one tensor-memory accumulator each, and
// combined in FP64 from c = 9 down to 0 by Horner steps, then scaled by s_j 2^-12 (exact).  Integer sums do not depend
// on order, so a k-point's bits depend on nothing but its own digits: not on the batch, the chunk or the tiling.
//
// Three kernels:
//   hk_wdigits_kernel  once per handle: the digits of the tiled weights Wt (hk_gemm.cu layout) -> Wd, scales -> Wsc.
//                      It reads the device copy, so host-packed, device-packed (supercell) and block-sparse handles
//                      get their digits from one place.
//   hk_qdigits_kernel  per chunk, in place of hk_phase_kernel: the 8 digit planes of [cos | sin](2 pi k.R), with the
//                      phase computed exactly as hk_phase_kernel computes it.
//   hk_gemm_i8_kernel  one CTA per (128 packed columns, 48 k-points) tile.  A (M = 128) = the 9 digit planes of W,
//                      B (N) = the Q digit planes stacked along N, [Q_0 | Q_1 | ...] x 48 rows; for W digit b the
//                      planes 0 .. min(7, 9 - b) land on the contiguous accumulator range of classes b .. b + 7 (class
//                      c at tensor-memory columns 48 c .. 48 c + 47, 480 of 512 columns).  Every 32-row K step is one
//                      48 KB stage (36 KB of W digits + 12 KB of Q digits, both pre-laid out in the no-swizzle K-major
//                      core-matrix layout, so one bulk copy each) and 16 MMAs (kOps).  Warp 0 feeds a ring of stages
//                      with cp.async.bulk, warp 1 owns tensor memory and issues the MMAs, warps 2-5 (one TMEM lane
//                      quarter each) run the epilogue.  Two CTAs fit an SM: the second fills its ring while the first
//                      still holds tensor memory, and allocates it when the first releases it.
#include "tbk_kernels.h"
#include "tbk_math.cuh"
#include "tcgen05.cuh"

namespace tbk {

namespace {

constexpr int BM = kI8BM;      // packed columns per tile (M, tensor-memory lanes)
constexpr int BK = kI8BK;      // k-points per tile (N of one class)
constexpr int QD = 8;          // digits of q
constexpr int WD = 9;          // digits of W / s_j
constexpr int NCLS = 10;       // classes kept
constexpr int A_DIGIT = BM * 32;          // bytes of one W digit plane of a K step
constexpr int A_STAGE = WD * A_DIGIT;     // 36864
constexpr int B_PLANE = BK * 32;          // 1536
constexpr int B_STAGE = QD * B_PLANE;     // 12288
constexpr int STAGE = A_STAGE + B_STAGE;  // 49152
constexpr int STAGES = 2;  // 2 x 48 KB per CTA: two CTAs per SM (see the file header)
constexpr int THREADS = 192;
constexpr size_t SMEM = (size_t)STAGES * STAGE + 1024;  // + barriers, tensor-memory address, alignment slack

// Byte of (row, k byte) in an R x 32-byte operand block: 8-row x 16-byte core matrices, the two K halves of a row group
// adjacent (LBO = 128 bytes), row groups 256 bytes apart (SBO).
__host__ __device__ constexpr int core_off(int row, int kb) { return (row >> 3) * 256 + (kb >> 4) * 128 + (row & 7) * 16 + (kb & 15); }

// Balanced digits of x (|x| <= 1): D digits of weight 2^(-6-7a); every step is exact but the last rint.
template <int D>
__device__ __forceinline__ void split_digits(double x, int (&d)[D]) {
    double t = x * 64.0;
#pragma unroll
    for (int a = 0; a < D; ++a) {
        const double r = rint(t);
        d[a] = (int)r;
        t = (t - r) * 128.0;
    }
}

// One MMA of the K step: W digit b against Q planes [plane, plane + np) into classes b + plane ...  `init` marks the
// first write of its classes in K step 0 (accumulate off).  The order makes every MMA's class range either all fresh or
// all written, which two MMAs per digit cannot (N <= 256 = 5 planes of 48).
struct MmaOp {
    int b, plane, np, init;
};
__device__ constexpr MmaOp kOps[16] = {{0, 0, 5, 1}, {0, 5, 3, 1}, {1, 0, 5, 0}, {1, 5, 2, 0}, {1, 7, 1, 1}, {2, 0, 5, 0},
                                       {2, 5, 2, 0}, {2, 7, 1, 1}, {3, 0, 5, 0}, {3, 5, 2, 0}, {4, 0, 5, 0}, {4, 5, 1, 0},
                                       {5, 0, 5, 0}, {6, 0, 4, 0}, {7, 0, 3, 0}, {8, 0, 2, 0}};

__device__ __forceinline__ double wt_at(const double* Wt, int kchunks, int bn, int n_tiles, long q, long j) {
    const long nt = j / bn;
    if (nt >= n_tiles || q >= (long)kchunks * kGemmKC) return 0.0;
    const long c = q / kGemmKC, kk = q % kGemmKC;
    return Wt[((nt * kchunks + c) * kGemmKC + kk) * (bn + 4) + (j - nt * bn)];
}

// grid (m_tiles, ksteps), BM threads: thread = column j of the tile.  Wd[((mt * ksteps + s) * WD + b) * A_DIGIT + ...],
// Wsc[j] = s_j 2^-12 (0 for all-zero columns).
__global__ void __launch_bounds__(BM) hk_wdigits_kernel(const double* __restrict__ Wt, int kchunks, int bn, int n_tiles,
                                                        int ksteps, int8_t* __restrict__ Wd, double* __restrict__ Wsc) {
    const long j = (long)blockIdx.x * BM + threadIdx.x;
    const int s = blockIdx.y;
    double mx = 0.0;
    for (long q = 0; q < (long)kchunks * kGemmKC; ++q) mx = fmax(mx, fabs(wt_at(Wt, kchunks, bn, n_tiles, q, j)));
    int e = 0;
    frexp(mx, &e);  // 2^(e-1) <= mx < 2^e
    if (s == 0) Wsc[j] = mx > 0.0 ? ldexp(1.0, e - 12) : 0.0;
    uint32_t w[WD][8];
#pragma unroll
    for (int b = 0; b < WD; ++b)
#pragma unroll
        for (int i = 0; i < 8; ++i) w[b][i] = 0;
    if (mx > 0.0) {
        for (int kb = 0; kb < 32; ++kb) {
            int d[WD];
            split_digits<WD>(ldexp(wt_at(Wt, kchunks, bn, n_tiles, (long)s * 32 + kb, j), -e), d);
#pragma unroll
            for (int b = 0; b < WD; ++b) w[b][kb >> 2] |= (uint32_t)(d[b] & 0xFF) << (8 * (kb & 3));
        }
    }
    int8_t* base = Wd + ((size_t)blockIdx.x * ksteps + s) * A_STAGE + core_off(threadIdx.x, 0);
#pragma unroll
    for (int b = 0; b < WD; ++b) {
        *reinterpret_cast<uint4*>(base + b * A_DIGIT) = make_uint4(w[b][0], w[b][1], w[b][2], w[b][3]);
        *reinterpret_cast<uint4*>(base + b * A_DIGIT + 128) = make_uint4(w[b][4], w[b][5], w[b][6], w[b][7]);
    }
}

// grid (k_tiles, ysplit), 256 threads.  Qd[(kt * ksteps + s) * B_STAGE + a * B_PLANE + core_off(k, row)]: row 2 r' of
// K step s is cos, row 2 r' + 1 sin of R vector 16 s + r' (the row order of W).
__global__ void __launch_bounds__(256) hk_qdigits_kernel(const double* __restrict__ kpts, long nk, const double* __restrict__ Rd,
                                                         int dim, int kchunks, int ksteps, int8_t* __restrict__ Qd) {
    __shared__ double ks[BK * kMaxDim];
    __shared__ __align__(16) int8_t tile[B_STAGE];
    const int tid = threadIdx.x;
    const long kt = blockIdx.x;
    for (int i = tid; i < BK * dim; i += 256) {
        const long row = kt * BK + i / dim;
        ks[i] = (row < nk) ? kpts[row * dim + (i % dim)] : 0.0;  // rows past the batch: k = 0, never stored
    }
    __syncthreads();
    for (int s = blockIdx.y; s < ksteps; s += gridDim.y) {
        for (int p = tid; p < BK * 16; p += 256) {
            const int m = p % BK, rl = p / BK;
            const int r = s * 16 + rl;
            int dc[QD], dsn[QD];
            if (r < kchunks * 8) {
                double x = 0.0;  // as hk_phase_kernel: the same phase bits as the FP64 path
                for (int d = 0; d < dim; ++d) x = fma(ks[m * dim + d], __ldg(Rd + (size_t)r * dim + d), x);
                double sn, cs;
                sincospi_lean(2.0 * x, sn, cs);
                split_digits<QD>(cs, dc);
                split_digits<QD>(sn, dsn);
            } else {
#pragma unroll
                for (int a = 0; a < QD; ++a) dc[a] = dsn[a] = 0;
            }
#pragma unroll
            for (int a = 0; a < QD; ++a) {
                tile[a * B_PLANE + core_off(m, 2 * rl)] = (int8_t)dc[a];
                tile[a * B_PLANE + core_off(m, 2 * rl + 1)] = (int8_t)dsn[a];
            }
        }
        __syncthreads();
        uint4* dst = reinterpret_cast<uint4*>(Qd + ((size_t)kt * ksteps + s) * B_STAGE);
        for (int i = tid; i < B_STAGE / 16; i += 256) dst[i] = reinterpret_cast<const uint4*>(tile)[i];
        __syncthreads();
    }
}

__device__ __forceinline__ void named_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

// grid: k_tiles * m_tiles, column tile fastest (the m_tiles CTAs of a k tile share its Q digits in L2).
__global__ void __launch_bounds__(THREADS, STAGES <= 2 ? 2 : 1)
hk_gemm_i8_kernel(const int8_t* __restrict__ Wd, const double* __restrict__ Wsc, const int8_t* __restrict__ Qd, long nk,
                  int m_tiles, int ksteps, int NN, double* __restrict__ Hp) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* stages = smem_raw;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)STAGES * STAGE);
    uint64_t* empty = full + STAGES;
    uint64_t* accum = empty + STAGES;
    uint32_t* tbase = reinterpret_cast<uint32_t*>(accum + 1);

    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const long kt = blockIdx.x / m_tiles;
    const int mt = (int)(blockIdx.x - kt * m_tiles);

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc5::mbar_init(tc5::smem_u32(&full[s]), 1);
            tc5::mbar_init(tc5::smem_u32(&empty[s]), 1);
        }
        tc5::mbar_init(tc5::smem_u32(accum), 1);
    }
    __syncthreads();

    if (warp == 0) {
        if ((tid & 31) == 0) {
            const int8_t* asrc = Wd + (size_t)mt * ksteps * A_STAGE;
            const int8_t* bsrc = Qd + (size_t)kt * ksteps * B_STAGE;
            for (int c = 0; c < ksteps; ++c) {
                const int s = c % STAGES;
                if (c >= STAGES) tc5::mbar_wait(tc5::smem_u32(&empty[s]), (uint32_t)((c / STAGES - 1) & 1));
                const uint32_t bar = tc5::smem_u32(&full[s]);
                const uint32_t dst = tc5::smem_u32(stages + (size_t)s * STAGE);
                tc5::mbar_expect_tx(bar, STAGE);
                tc5::bulk_g2s(dst, asrc + (size_t)c * A_STAGE, A_STAGE, bar);
                tc5::bulk_g2s(dst + A_STAGE, bsrc + (size_t)c * B_STAGE, B_STAGE, bar);
            }
        }
        return;
    }

    if (warp == 1) {
        tc5::tmem_alloc(tc5::smem_u32(tbase), 512);  // waits while the other CTA on this SM holds tensor memory
        tc5::tmem_relinquish();
        tc5::fence_before_sync();
        named_sync(1, 160);  // tensor-memory address -> epilogue warps
        tc5::fence_after_sync();
        const uint32_t d0 = *tbase;
        if ((tid & 31) == 0) {
            for (int c = 0; c < ksteps; ++c) {
                const int s = c % STAGES;
                tc5::mbar_wait(tc5::smem_u32(&full[s]), (uint32_t)((c / STAGES) & 1));
                tc5::fence_after_sync();
                const uint32_t a0 = tc5::smem_u32(stages + (size_t)s * STAGE), b0 = a0 + A_STAGE;
#pragma unroll
                for (int o = 0; o < 16; ++o) {
                    const MmaOp op = kOps[o];
                    tc5::mma_i8(d0 + (uint32_t)((op.b + op.plane) * BK), tc5::smem_desc(a0 + op.b * A_DIGIT, 128, 256),
                                tc5::smem_desc(b0 + op.plane * B_PLANE, 128, 256), tc5::idesc_s8(BM, BK * op.np),
                                (c > 0 || !op.init) ? 1u : 0u);
                }
                tc5::commit(tc5::smem_u32(&empty[s]));  // stage s free once these MMAs have read it
            }
            tc5::commit(tc5::smem_u32(accum));
        }
        __syncwarp();
        named_sync(2, 160);  // the epilogue has read every accumulator
        tc5::fence_after_sync();
        tc5::tmem_dealloc(d0, 512);
        return;
    }

    // epilogue: warp w reads tensor-memory lanes 32 (w % 4) ..; thread = packed column j
    named_sync(1, 160);
    tc5::fence_after_sync();
    const uint32_t lane_q = (uint32_t)(warp & 3) * 32;
    const uint32_t taddr = *tbase + (lane_q << 16);
    const long j = (long)mt * BM + lane_q + (tid & 31);
    const double sc = Wsc[j];
    tc5::mbar_wait(tc5::smem_u32(accum), 0);
    tc5::fence_after_sync();
#pragma unroll 1
    for (int g = 0; g < BK / 8; ++g) {
        uint32_t v[NCLS][8];
#pragma unroll
        for (int c = 0; c < NCLS; ++c) tmem_ld8(taddr + (uint32_t)(c * BK + g * 8), v[c]);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            double t = (double)(int)v[NCLS - 1][i];
#pragma unroll
            for (int c = NCLS - 2; c >= 0; --c) t = fma(t, 0x1p-7, (double)(int)v[c][i]);
            const long k = kt * BK + g * 8 + i;
            if (k < nk && j < NN) Hp[k * NN + j] = t * sc;
        }
    }
    tc5::fence_before_sync();
    named_sync(2, 160);
}

}  // namespace

int hk_i8_ksteps(const ModelDev& md) { return (md.kchunks + 1) / 2; }

size_t hk_i8_q_bytes(const ModelDev& md, long nk) {
    return (size_t)((nk + BK - 1) / BK) * (size_t)hk_i8_ksteps(md) * B_STAGE;
}

size_t hk_i8_w_bytes(const ModelDev& md) {
    const long m_tiles = ((long)md.n * md.n + BM - 1) / BM;
    return (size_t)m_tiles * hk_i8_ksteps(md) * A_STAGE;
}

cudaError_t launch_hk_wdigits(const ModelDev& md, int8_t* Wd, double* Wsc, cudaStream_t st) {
    const long m_tiles = ((long)md.n * md.n + BM - 1) / BM;
    const int ks = hk_i8_ksteps(md);
    if (m_tiles <= 0 || ks <= 0) return cudaSuccess;
    if (m_tiles > 2147483647L || ks > 65535) return cudaErrorInvalidConfiguration;
    hk_wdigits_kernel<<<dim3((unsigned)m_tiles, (unsigned)ks), BM, 0, st>>>(md.Wt, md.kchunks, 16 * md.na, md.n_tiles, ks, Wd, Wsc);
    return cudaGetLastError();
}

cudaError_t launch_hk_qdigits(const ModelDev& md, const double* k, long nk, int8_t* Qd, cudaStream_t st) {
    const long k_tiles = (nk + BK - 1) / BK;
    const int ks = hk_i8_ksteps(md);
    if (k_tiles <= 0 || ks <= 0) return cudaSuccess;
    if (k_tiles > 2147483647L) return cudaErrorInvalidConfiguration;
    int ysplit = 1;
    while (k_tiles * ysplit < 592 && ysplit * 2 <= ks) ysplit *= 2;  // >= 4 CTAs per SM worth of work
    hk_qdigits_kernel<<<dim3((unsigned)k_tiles, (unsigned)ysplit), 256, 0, st>>>(k, nk, md.Rd, md.dim, md.kchunks, ks, Qd);
    return cudaGetLastError();
}

cudaError_t launch_hk_gemm_i8(const ModelDev& md, long nk, const int8_t* Qd, double* Hp, cudaStream_t st) {
    const long NN = (long)md.n * md.n;
    const long m_tiles = (NN + BM - 1) / BM;
    const long k_tiles = (nk + BK - 1) / BK;
    if (k_tiles <= 0 || m_tiles <= 0) return cudaSuccess;
    const long grid = k_tiles * m_tiles;
    if (grid > 2147483647L || NN > 2147483647L) return cudaErrorInvalidConfiguration;
    cudaError_t err = cudaFuncSetAttribute(hk_gemm_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    if (err != cudaSuccess) return err;
    hk_gemm_i8_kernel<<<(unsigned)grid, THREADS, SMEM, st>>>(md.Wd, md.Wsc, Qd, nk, (int)m_tiles, hk_i8_ksteps(md), (int)NN, Hp);
    return cudaGetLastError();
}

}  // namespace tbk
