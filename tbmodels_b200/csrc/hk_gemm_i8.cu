// hk_gemm_i8.cu -- H(k) build from exact INT8 tensor-core digit products (tcgen05 kind::i8, sm_100a).
//
// The GEMM of hk_gemm.cu, Hp[k, j] = sum_r Q[k, r] W[r, j], with both operands split into balanced 7-bit digits
// (the Ozaki scheme; tests/hk_digits_reference.py restates it bit for bit in Python and pins its error bound, and
// tests/test_gpu_hk_int8_exact.py requires this kernel's output to equal the restatement):
//     q    = sum_{a=0..7} q_a 2^(-6-7a),  q_a in [-64, 64], rounded at 2^-55        (|q| <= 1: cos / sin)
//     W/s_j = sum_{b=0..8} w_b 2^(-6-7b),  w_b in [-64, 64], rounded at 2^-62       (s_j: power of two > max_r |W_rj|)
// A digit product (a, b) belongs to class c = a + b, weight 2^(-12-7c).  The classes c <= 9 (51 products) are summed
// exactly in int32 (at most 8 pairs x 64^2 per row: < 2^31 for K < 2^16 rows), one tensor-memory accumulator each,
// combined exactly into two int64 parts and then in FP64 by one FMA (correctly rounded up to 31 K steps of 32 rows), and
// scaled by s_j 2^-12 (exact).  Integer sums do not depend
// on order, so a k-point's bits depend on nothing but its own digits: not on the batch, the chunk or the tiling.
//
// Three kernels:
//   hk_wdigits_kernel  once per handle: the digits of the tiled weights Wt (hk_gemm.cu layout) -> Wd, scales -> Wsc.
//                      It reads the device copy, so host-packed, device-packed (supercell) and block-sparse handles
//                      get their digits from one place.
//   hk_qdigits_kernel  per chunk, in place of hk_phase_kernel: the 8 digit planes of [cos | sin](2 pi k.R), with the
//                      phase computed exactly as hk_phase_kernel computes it.
//   hk_gemm_i8_kernel  tiles of 128 packed columns x 48 k-points.  A (M = 128) = the 9 digit planes of W,
//                      B (N) = the Q digit planes stacked along N, [Q_0 | Q_1 | ...] x 48 rows; for W digit b the
//                      planes 0 .. min(7, 9 - b) land on the contiguous accumulator range of classes b .. b + 7 (class
//                      c at tensor-memory columns 48 c .. 48 c + 47, 480 of 512 columns).  Every 32-row K step is one
//                      48 KB stage (36 KB of W digits + 12 KB of Q digits, both pre-laid out in the no-swizzle K-major
//                      core-matrix layout, so one bulk copy each) and 16 MMAs (kOps).  Persistent, one CTA per SM:
//                      warp 0 feeds a ring of stages with cp.async.bulk across tile boundaries, warp 1 owns tensor
//                      memory and issues the MMAs, warps 2-9 drain a tile's accumulators into registers, hand tensor
//                      memory back and convert and store while the MMAs of the CTA's next tile run.
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
constexpr int STAGES = 4;     // 4 x 48 KB: one CTA per SM
constexpr int EPI_WARPS = 8;  // two per tensor-memory lane quarter
constexpr int EPI_K = BK / 2;  // k-points per epilogue thread and tile
constexpr int THREADS = 64 + 32 * EPI_WARPS;
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

// split_digits<QD>(q) without conversions: rint(t) is (t + 1.5 2^52) - 1.5 2^52 (round half to even, |t| <= 65), and the
// low word of t + 1.5 2^52 is that integer in two's complement.  The same exact steps, so the same digits, byte for byte.
__device__ __forceinline__ void split_q_digits(double q, uint32_t (&d)[QD]) {
    constexpr double kMagic = 0x1.8p52;
    double t = q * 64.0;
#pragma unroll
    for (int a = 0; a < QD; ++a) {
        const double s = __dadd_rn(t, kMagic);
        d[a] = (uint32_t)__double2loint(s);
        t = (t - __dsub_rn(s, kMagic)) * 128.0;
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

// grid (k_tiles, ysplit), QTHREADS threads.  Qd[(kt * ksteps + s) * B_STAGE + a * B_PLANE + core_off(k, row)]: row
// 2 r' of K step s is cos, row 2 r' + 1 sin of R vector 16 s + r' (the row order of W).  A thread makes the digits of one
// k-point and two R vectors, which are one 32-bit word (cos, sin, cos, sin) of each digit plane; the lanes of a warp
// take 8 k-points x 4 R pairs, whose words fall in 32 different banks.
constexpr int QTHREADS = BK * 8;  // 384: one thread per (k-point, R pair) of a K step
__global__ void __launch_bounds__(QTHREADS) hk_qdigits_kernel(const double* __restrict__ kpts, long nk, const double* __restrict__ Rd,
                                                              int dim, int kchunks, int ksteps, int8_t* __restrict__ Qd) {
    __shared__ double ks[BK * kMaxDim];
    __shared__ __align__(16) uint32_t tile[B_STAGE / 4];
    const int tid = threadIdx.x;
    const long kt = blockIdx.x;
    for (int i = tid; i < BK * dim; i += QTHREADS) {
        const long row = kt * BK + i / dim;
        ks[i] = (row < nk) ? kpts[row * dim + (i % dim)] : 0.0;  // rows past the batch: k = 0, never stored
    }
    __syncthreads();
    const int m = (tid & 7) | ((tid >> 6) << 3);  // k-point of the tile
    const int rp = (tid >> 3) & 7;                // R pair: rows 4 rp .. 4 rp + 3 of the K step
    for (int s = blockIdx.y; s < ksteps; s += gridDim.y) {
        uint32_t w[QD];
#pragma unroll
        for (int a = 0; a < QD; ++a) w[a] = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = s * 16 + 2 * rp + h;
            if (r < kchunks * 8) {
                double x = 0.0;  // as hk_phase_kernel: the same phase bits as the FP64 path
                for (int d = 0; d < dim; ++d) x = fma(ks[m * dim + d], __ldg(Rd + (size_t)r * dim + d), x);
                double sn, cs;
                sincospi_lean(2.0 * x, sn, cs);
                uint32_t dc[QD], dsn[QD];
                split_q_digits(cs, dc);
                split_q_digits(sn, dsn);
#pragma unroll
                for (int a = 0; a < QD; ++a) w[a] |= ((dc[a] & 0xFF) | (dsn[a] & 0xFF) << 8) << (16 * h);
            }
        }
#pragma unroll
        for (int a = 0; a < QD; ++a) tile[(a * B_PLANE + core_off(m, 4 * rp)) >> 2] = w[a];
        __syncthreads();
        uint4* dst = reinterpret_cast<uint4*>(Qd + ((size_t)kt * ksteps + s) * B_STAGE);
        for (int i = tid; i < B_STAGE / 16; i += QTHREADS) dst[i] = reinterpret_cast<const uint4*>(tile)[i];
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

// Persistent: grid = min(tiles, SMs), one CTA per SM, tile t = blockIdx.x + i gridDim.x with the column tile fastest (the
// CTAs working on one k tile run together and share its Q digits in L2).  Barrier phases, with g the CTA's running K
// step count over all its tiles and i its tile count:
//   full[g % STAGES]    completes once per K step g (expect_tx of both copies)      MMA issuer waits parity (g / STAGES) & 1
//   empty[g % STAGES]   commit after K step g's MMAs                                producer waits parity (g / STAGES - 1) & 1
//   accum_full          commit after tile i's last K step                           epilogue waits parity i & 1
//   tmem_empty          one arrive per epilogue warp once tile i is drained          MMA issuer waits parity (i - 1) & 1, i >= 1
// Each barrier can be at most one phase ahead of its waiter, so parities are unambiguous.
__global__ void __launch_bounds__(THREADS, 1)
hk_gemm_i8_kernel(const int8_t* __restrict__ Wd, const double* __restrict__ Wsc, const int8_t* __restrict__ Qd, long nk,
                  int m_tiles, long tiles, int ksteps, int NN, double* __restrict__ Hp) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* stages = smem_raw;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)STAGES * STAGE);
    uint64_t* empty = full + STAGES;
    uint64_t* accum_full = empty + STAGES;
    uint64_t* tmem_empty = accum_full + 1;
    uint32_t* tbase = reinterpret_cast<uint32_t*>(tmem_empty + 1);

    const int tid = threadIdx.x;
    const int warp = tid >> 5;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            tc5::mbar_init(tc5::smem_u32(&full[s]), 1);
            tc5::mbar_init(tc5::smem_u32(&empty[s]), 1);
        }
        tc5::mbar_init(tc5::smem_u32(accum_full), 1);
        tc5::mbar_init(tc5::smem_u32(tmem_empty), EPI_WARPS);
    }
    __syncthreads();

    if (warp == 0) {  // producer: one stage ring across tile boundaries
        if ((tid & 31) == 0) {
            long g = 0;
            for (long t = blockIdx.x; t < tiles; t += gridDim.x) {
                const long kt = t / m_tiles;
                const int mt = (int)(t - kt * m_tiles);
                const int8_t* asrc = Wd + (size_t)mt * ksteps * A_STAGE;
                const int8_t* bsrc = Qd + (size_t)kt * ksteps * B_STAGE;
                for (int c = 0; c < ksteps; ++c, ++g) {
                    const int s = (int)(g % STAGES);
                    if (g >= STAGES) tc5::mbar_wait(tc5::smem_u32(&empty[s]), (uint32_t)((g / STAGES - 1) & 1));
                    const uint32_t bar = tc5::smem_u32(&full[s]);
                    const uint32_t dst = tc5::smem_u32(stages + (size_t)s * STAGE);
                    tc5::mbar_expect_tx(bar, STAGE);
                    tc5::bulk_g2s(dst, asrc + (size_t)c * A_STAGE, A_STAGE, bar);
                    tc5::bulk_g2s(dst + A_STAGE, bsrc + (size_t)c * B_STAGE, B_STAGE, bar);
                }
            }
        }
        return;
    }

    if (warp == 1) {  // tensor-memory owner for the kernel's lifetime, MMA issuer
        tc5::tmem_alloc(tc5::smem_u32(tbase), 512);
        tc5::tmem_relinquish();
        tc5::fence_before_sync();
        named_sync(1, 32 + 32 * EPI_WARPS);  // tensor-memory address -> epilogue warps
        tc5::fence_after_sync();
        const uint32_t d0 = *tbase;
        if ((tid & 31) == 0) {
            long g = 0, i = 0;
            for (long t = blockIdx.x; t < tiles; t += gridDim.x, ++i) {
                if (i > 0) {  // the epilogue has drained tile i - 1
                    tc5::mbar_wait(tc5::smem_u32(tmem_empty), (uint32_t)((i - 1) & 1));
                    tc5::fence_after_sync();
                }
                for (int c = 0; c < ksteps; ++c, ++g) {
                    const int s = (int)(g % STAGES);
                    tc5::mbar_wait(tc5::smem_u32(&full[s]), (uint32_t)((g / STAGES) & 1));
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
                tc5::commit(tc5::smem_u32(accum_full));
            }
        }
        __syncwarp();
        named_sync(2, 32 + 32 * EPI_WARPS);  // the epilogue has read every accumulator
        tc5::fence_after_sync();
        tc5::tmem_dealloc(d0, 512);
        return;
    }

    // epilogue: warps w and w + 4 read tensor-memory lanes 32 (w % 4) .., k-points 0 .. 23 and 24 .. 47 of the tile;
    // thread = packed column j.  The ten class sums of a k-point are combined exactly in two int64 parts,
    //   hi = sum_{c <= 4} s_c 2^(7 (4 - c)),   lo = sum_{c >= 5} s_c 2^(7 (9 - c)),   t = (hi + lo 2^-35) 2^-28,
    // (|s_c| < 2^20 K steps, so |hi|, |lo| < 2^49 K steps: no overflow for K steps <= kI8MaxKSteps), held in registers
    // while tensor memory goes back to the MMA issuer, and converted while the next tile's MMAs run.  Up to 31 K steps
    // hi and lo are exact doubles and t is the correctly rounded sum of the classes.
    named_sync(1, 32 + 32 * EPI_WARPS);
    tc5::fence_after_sync();
    const uint32_t lane_q = (uint32_t)(warp & 3) * 32;
    const int k0 = ((warp - 2) >> 2) * EPI_K;
    const uint32_t taddr = *tbase + (lane_q << 16) + (uint32_t)k0;
    long i = 0;
    for (long t = blockIdx.x; t < tiles; t += gridDim.x, ++i) {
        const long kt = t / m_tiles;
        const int mt = (int)(t - kt * m_tiles);
        const long j = (long)mt * BM + lane_q + (tid & 31);
        const double sc = Wsc[j];
        long long hi[EPI_K], lo[EPI_K];
        tc5::mbar_wait(tc5::smem_u32(accum_full), (uint32_t)(i & 1));
        tc5::fence_after_sync();
#pragma unroll
        for (int g = 0; g < EPI_K / 8; ++g) {
            uint32_t v[NCLS][8];
#pragma unroll
            for (int c = 0; c < NCLS; ++c) tmem_ld8(taddr + (uint32_t)(c * BK + g * 8), v[c]);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                long long h = 0, l = 0;
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                    h += (long long)(int)v[c][e] * (1LL << (7 * (4 - c)));
                    l += (long long)(int)v[c + 5][e] * (1LL << (7 * (4 - c)));
                }
                hi[g * 8 + e] = h;
                lo[g * 8 + e] = l;
            }
        }
        tc5::fence_before_sync();
        __syncwarp();
        if ((tid & 31) == 0) tc5::mbar_arrive(tc5::smem_u32(tmem_empty));
        if (j < NN) {
#pragma unroll
            for (int e = 0; e < EPI_K; ++e) {
                const long k = kt * BK + k0 + e;
                if (k < nk) Hp[k * NN + j] = fma((double)lo[e], 0x1p-35, (double)hi[e]) * 0x1p-28 * sc;
            }
        }
    }
    tc5::fence_before_sync();
    named_sync(2, 32 + 32 * EPI_WARPS);
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
    hk_qdigits_kernel<<<dim3((unsigned)k_tiles, (unsigned)ysplit), QTHREADS, 0, st>>>(k, nk, md.Rd, md.dim, md.kchunks, ks, Qd);
    return cudaGetLastError();
}

cudaError_t launch_hk_gemm_i8(const ModelDev& md, long nk, const int8_t* Qd, double* Hp, cudaStream_t st) {
    const long NN = (long)md.n * md.n;
    const long m_tiles = (NN + BM - 1) / BM;
    const long k_tiles = (nk + BK - 1) / BK;
    if (k_tiles <= 0 || m_tiles <= 0) return cudaSuccess;
    const long tiles = k_tiles * m_tiles;
    if (m_tiles > 2147483647L || NN > 2147483647L) return cudaErrorInvalidConfiguration;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const unsigned grid = (unsigned)std::min<long>(tiles, sms);
    cudaError_t err = cudaFuncSetAttribute(hk_gemm_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM);
    if (err != cudaSuccess) return err;
    hk_gemm_i8_kernel<<<grid, THREADS, SMEM, st>>>(md.Wd, md.Wsc, Qd, nk, (int)m_tiles, tiles, hk_i8_ksteps(md), (int)NN, Hp);
    return cudaGetLastError();
}

}  // namespace tbk
