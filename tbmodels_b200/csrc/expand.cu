// expand.cu -- packed Hermitian H(k) -> the dense complex128 [n_k][N][N] array Model.hamilton returns.
//
// Writes the upper triangle as the exact conjugate of the lower one with an exactly-zero imaginary
// diagonal, which is what the reference's  H += H.conjugate().transpose()  produces for convention 2
// (src/tbmodels/_tb_model.py:1123).  For convention == 1 it applies the orbital-position phases
//   H_ij <- conj(pe_i) * H_ij * pe_j,   pe_j = exp(2 pi i k.pos_j)         (:1124-1128)
// in the same association order as the reference expression.
#include "tbk_kernels.h"
#include "tbk_math.cuh"

namespace tbk {

namespace {

__device__ __forceinline__ double2 load_elem(const double* __restrict__ h, long nre, int i, int j) {
    const int lo = i < j ? i : j, hi = i < j ? j : i;
    const double re = __ldg(h + tri(hi) + lo);
    double im = 0.0;
    if (hi != lo) {
        im = __ldg(h + nre + trs(hi) + lo);
        if (j > i) im = -im;
    }
    return make_double2(re, im);
}

__device__ __forceinline__ double2 pos_phase(const double* __restrict__ kp, const double* __restrict__ pos, int dim,
                                             int orb) {
    double x = 0.0;
    for (int d = 0; d < dim; ++d) x = fma(kp[d], __ldg(pos + orb * dim + d), x);
    double sn, cs;
    sincospi_lean(2.0 * x, sn, cs);
    return make_double2(cs, sn);
}

__device__ __forceinline__ double2 apply_conv1(double2 h, double2 pi_, double2 pj) {
    // (conj(pe_i) * h) * pe_j
    const double tr = pi_.x * h.x + pi_.y * h.y;
    const double ti = pi_.x * h.y - pi_.y * h.x;
    return make_double2(tr * pj.x - ti * pj.y, tr * pj.y + ti * pj.x);
}

// Small N: one thread per output element across the whole batch.
__global__ void __launch_bounds__(256)
expand_flat_kernel(const double* __restrict__ Hp, const double* __restrict__ kpts, const double* __restrict__ pos, int n,
                   int dim, long nk, int convention, double2* __restrict__ out) {
    const long NN = (long)n * n;
    const long nre = tri(n);
    const long total = nk * NN;
    for (long gid = (long)blockIdx.x * blockDim.x + threadIdx.x; gid < total; gid += (long)gridDim.x * blockDim.x) {
        const long kk = gid / NN;
        const int idx = (int)(gid - kk * NN);
        const int i = idx / n, j = idx - i * n;
        double2 h = load_elem(Hp + kk * NN, nre, i, j);
        if (convention == 1) {
            const double* kp = kpts + kk * dim;
            h = apply_conv1(h, pos_phase(kp, pos, dim, i), pos_phase(kp, pos, dim, j));
        }
        out[gid] = h;
    }
}

// Larger N: one CTA per k-point, position phases computed once per k-point in shared memory.
__global__ void __launch_bounds__(256)
expand_block_kernel(const double* __restrict__ Hp, const double* __restrict__ kpts, const double* __restrict__ pos, int n,
                    int dim, long nk, int convention, double2* __restrict__ out) {
    extern __shared__ __align__(16) double2 pe[];
    const long NN = (long)n * n;
    const long nre = tri(n);
    for (long kk = blockIdx.x; kk < nk; kk += gridDim.x) {
        if (convention == 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) pe[i] = pos_phase(kpts + kk * dim, pos, dim, i);
            __syncthreads();
        }
        const double* h = Hp + kk * NN;
        double2* o = out + kk * NN;
        for (int idx = threadIdx.x; idx < NN; idx += blockDim.x) {
            const int i = idx / n, j = idx - i * n;
            double2 v = load_elem(h, nre, i, j);
            if (convention == 1) v = apply_conv1(v, pe[i], pe[j]);
            o[idx] = v;
        }
        if (convention == 1) __syncthreads();
    }
}

__global__ void __launch_bounds__(256) scale_pow2_kernel(double* __restrict__ p, long n, int s) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) p[i] = scalbn(p[i], s);
}

}  // namespace

// Multi-GPU exchange step fused behind the eigensolver (SURVEY.md section 8 e1): the rows one chunk just produced are
// stored straight into the result buffers of the peer GPUs (peer-mapped memory over NVLink / NVSwitch), while the next
// chunk computes.  One grid-stride pass, 16-byte stores, every peer gets the same rows at the same offset.
constexpr int kMaxPeers = 15;
struct PeerList {
    double* base[kMaxPeers];
    int n;
};

__global__ void __launch_bounds__(256)
push_rows_kernel(const double* __restrict__ src, long n_doubles, PeerList peers, long dst_offset) {
    const long stride = (long)gridDim.x * blockDim.x;
    const long i0 = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if ((((unsigned long long)src | (unsigned long long)(dst_offset * 8)) & 15ull) == 0) {
        const long n2 = n_doubles >> 1;
        const double2* s2 = reinterpret_cast<const double2*>(src);
        for (long i = i0; i < n2; i += stride) {
            const double2 v = s2[i];
            for (int p = 0; p < peers.n; ++p) reinterpret_cast<double2*>(peers.base[p] + dst_offset)[i] = v;
        }
        if ((n_doubles & 1) && i0 == 0)
            for (int p = 0; p < peers.n; ++p) peers.base[p][dst_offset + n_doubles - 1] = src[n_doubles - 1];
    } else {
        for (long i = i0; i < n_doubles; i += stride) {
            const double v = src[i];
            for (int p = 0; p < peers.n; ++p) peers.base[p][dst_offset + i] = v;
        }
    }
}

cudaError_t launch_scale_pow2(double* p, long n, int s, cudaStream_t st) {
    if (n <= 0 || s == 0) return cudaSuccess;
    long blocks = (n + 255) / 256;
    if (blocks > 4096) blocks = 4096;
    scale_pow2_kernel<<<(unsigned)blocks, 256, 0, st>>>(p, n, s);
    return cudaGetLastError();
}

cudaError_t launch_push_rows(const double* src, long n_doubles, double* const* peer_bases, int n_peers, long dst_offset,
                             cudaStream_t st) {
    if (n_doubles <= 0 || n_peers <= 0) return cudaSuccess;
    if (n_peers > kMaxPeers) return cudaErrorInvalidValue;
    PeerList pl;
    pl.n = n_peers;
    for (int p = 0; p < n_peers; ++p) pl.base[p] = peer_bases[p];
    // a SMALL grid on purpose: the copy only has to keep up with one chunk of compute (tens of MB per ~10 ms), and every
    // CTA it occupies is taken from the phase / GEMM kernels of the next chunk it overlaps (measured at 8 GPUs with a
    // 1184-CTA grid: the overlapped phase kernel slowed from 2.3 to 7.4 ms per 2^21 k-points)
    long blocks = (n_doubles / 2 + 255) / 256;
    if (blocks > 32) blocks = 32;
    if (blocks < 1) blocks = 1;
    push_rows_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, n_doubles, pl, dst_offset);
    return cudaGetLastError();
}

cudaError_t launch_expand(const ModelDev& md, const double* k, const double* Hp, long nk, int convention, double* out,
                          cudaStream_t st) {
    if (nk <= 0 || md.n <= 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (md.n <= 16) {
        const long total = nk * (long)md.n * md.n;
        long blocks = (total + 255) / 256;
        const long cap = (long)sms * 32;
        if (blocks > cap) blocks = cap;
        expand_flat_kernel<<<(unsigned)blocks, 256, 0, st>>>(Hp, k, md.pos, md.n, md.dim, nk, convention,
                                                             reinterpret_cast<double2*>(out));
    } else {
        long blocks = nk;
        const long cap = (long)sms * 16;
        if (blocks > cap) blocks = cap;
        // the per-orbital phase table is only used by convention 1; large N needs the opt-in limit (> 48 KB from N = 3073)
        const size_t smem = convention == 1 ? (size_t)md.n * sizeof(double2) : 0;
        if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
        if (smem > 48 * 1024) {
            cudaError_t err = cudaFuncSetAttribute(expand_block_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (err != cudaSuccess) return err;
        }
        expand_block_kernel<<<(unsigned)blocks, 256, smem, st>>>(Hp, k, md.pos, md.n, md.dim, nk, convention,
                                                                 reinterpret_cast<double2*>(out));
    }
    return cudaGetLastError();
}

}  // namespace tbk
