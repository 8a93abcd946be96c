// hk_small.cu -- fused thread-per-k-point path for few-band models (N <= 8).
//
// One thread owns one k-point end to end: k (D doubles) in, N eigenvalues (or the packed H(k)) out.
// Nothing else touches HBM: the Hermitian-split weights W [2 n_R][N^2] and the R vectors sit in shared
// memory, the N^2 accumulators in registers, phases come from sincospi(2 k.R) on chip.
// Replaces Model.hamilton's Fourier loop + H += H^dagger (reference src/tbmodels/_tb_model.py:1111-1123)
// and the per-k scipy eigvalsh loop of Model.eigenval (:1147-1150) for small N.
// Phases: for nearest-cell lattice vectors (all |R_d| <= 1, flagged on the host) e^{2 pi i k.R} is the product
// of per-dimension factors  f_d = 1, z_d or conj(z_d)  with z_d = e^{2 pi i k_d}  (one sincospi per dimension
// per k-point, then D - 1 complex multiplications per R, branch free); longer vectors call sincospi(2 k.R).
//   N = 1, 2 : closed-form eigenvalues.
//   N = 3..8 : per-thread Householder tridiagonalisation + implicit QL on a thread-strided shared-memory
//              scratch (tbk_math.cuh), i.e. every lane works on its own matrix -- no idle lanes, no shuffles.
#include <cstdlib>

#include "tbk_kernels.h"
#include "tbk_math.cuh"

namespace tbk {

namespace {

constexpr int TPB = 128;

// doubles occupied by the R tables in shared memory: [nR][dim] doubles + [nR] int flags, rounded to 16 bytes
__host__ __device__ inline size_t small_table_doubles(int nR, int dim) {
    const size_t d = (size_t)nR * dim + ((size_t)nR + 1) / 2;
    return (d + 1) & ~(size_t)1;
}

template <int N>
constexpr int scratch_doubles() {
    return (N > 2) ? (N * N + 6 * N) : 0;  // matrix + v/w work (4N) + d, e (2N)
}

template <int D>
__device__ __forceinline__ void load_kpoint(double (&kn)[D ? D : kMaxDim], const double* __restrict__ kpts, long idx,
                                            long nk, int dim) {
    if (idx >= nk) return;
    if (D == 2) {
        const double2 v = *reinterpret_cast<const double2*>(kpts + idx * 2);
        kn[0] = v.x;
        kn[D > 1 ? 1 : 0] = v.y;
    } else {
#pragma unroll
        for (int d = 0; d < (D ? D : kMaxDim); ++d) kn[d] = (d < dim) ? kpts[idx * dim + d] : 0.0;
    }
}

template <int N, int D>  // D = 0: run-time dimension (<= kMaxDim)
__global__ void __launch_bounds__(TPB)
hk_small_kernel(const double* __restrict__ kpts, long nk, const double* __restrict__ Rd, const int* __restrict__ Ri,
                const double* __restrict__ W, int dim_rt, int nR, int use_z, double* __restrict__ Hp,
                double* __restrict__ eig, int* __restrict__ fail_count) {
    constexpr int NN = N * N;
    const int dim = D ? D : dim_rt;
    extern __shared__ __align__(16) double sm[];
    double* Ws = sm;                             // [2 nR][NN]
    double* Rs = Ws + (size_t)2 * nR * NN;       // [nR][dim]
    int* Is = reinterpret_cast<int*>(Rs + (size_t)nR * dim);  // [nR] flag: phase = product of per-dimension factors
    double* scratch = Rs + small_table_doubles(nR, dim);

    const int tid = threadIdx.x;
    for (int i = tid; i < 2 * nR * NN; i += TPB) Ws[i] = W[i];
    for (int i = tid; i < nR * dim; i += TPB) Rs[i] = Rd[i];
    for (int i = tid; i < nR; i += TPB) Is[i] = Ri[i];
    __syncthreads();

    // KP k-points per thread and loop trip (2 for N <= 2): the R / W table reads and the loop bookkeeping are shared,
    // and two independent dependency chains are in flight.  The k-points of the next trip are prefetched.
    constexpr int KP = (N <= 2) ? 2 : 1;
    constexpr int DD = D ? D : kMaxDim;
    const long stride = (long)gridDim.x * TPB;
    long kk = (long)blockIdx.x * TPB + tid;
    double kn[KP][DD];
#pragma unroll
    for (int p = 0; p < KP; ++p) load_kpoint<D>(kn[p], kpts, kk + p * stride, nk, dim);
    for (; kk < nk; kk += KP * stride) {
        double kv[KP][DD];
#pragma unroll
        for (int p = 0; p < KP; ++p) {
#pragma unroll
            for (int d = 0; d < DD; ++d) kv[p][d] = kn[p][d];
            load_kpoint<D>(kn[p], kpts, kk + (KP + p) * stride, nk, dim);
        }

        double acc[KP][NN];
#pragma unroll
        for (int p = 0; p < KP; ++p)
#pragma unroll
            for (int e = 0; e < NN; ++e) acc[p][e] = 0.0;

        double zr[KP][DD], zi[KP][DD];
        if (use_z) {
#pragma unroll
            for (int p = 0; p < KP; ++p)
#pragma unroll
                for (int d = 0; d < DD; ++d)
                    if (d < dim) sincospi_lean(2.0 * kv[p][d], zi[p][d], zr[p][d]);
        }

        for (int r = 0; r < nR; ++r) {
            double sn[KP], cs[KP];
            double rd[DD];
#pragma unroll
            for (int d = 0; d < DD; ++d) rd[d] = (d < dim) ? Rs[r * dim + d] : 0.0;
            if (Is[r]) {  // CTA-uniform: all |R_d| <= 1, so R_d itself is the sign / presence of the factor
#pragma unroll
                for (int p = 0; p < KP; ++p) {
                    cs[p] = (rd[0] != 0.0) ? zr[p][0] : 1.0;
                    sn[p] = rd[0] * zi[p][0];
#pragma unroll
                    for (int d = 1; d < DD; ++d) {
                        if (d < dim) {
                            const double fr = (rd[d] != 0.0) ? zr[p][d] : 1.0;
                            const double fi = rd[d] * zi[p][d];
                            const double tr_ = cs[p] * fr - sn[p] * fi;
                            sn[p] = fma(cs[p], fi, sn[p] * fr);
                            cs[p] = tr_;
                        }
                    }
                }
            } else {
#pragma unroll
                for (int p = 0; p < KP; ++p) {
                    double x = 0.0;
#pragma unroll
                    for (int d = 0; d < DD; ++d)
                        if (d < dim) x = fma(kv[p][d], rd[d], x);
                    sincospi_lean(2.0 * x, sn[p], cs[p]);
                }
            }
            const double* w0 = Ws + (size_t)(2 * r) * NN;
            const double* w1 = w0 + NN;
            if (NN % 2 == 0) {
#pragma unroll
                for (int e = 0; e < NN; e += 2) {
                    const double2 a = *reinterpret_cast<const double2*>(w0 + e);
                    const double2 b = *reinterpret_cast<const double2*>(w1 + e);
#pragma unroll
                    for (int p = 0; p < KP; ++p) {
                        acc[p][e] = fma(cs[p], a.x, fma(sn[p], b.x, acc[p][e]));
                        acc[p][e + 1] = fma(cs[p], a.y, fma(sn[p], b.y, acc[p][e + 1]));
                    }
                }
            } else {
#pragma unroll
                for (int e = 0; e < NN; ++e) {
                    const double a = w0[e], b = w1[e];
#pragma unroll
                    for (int p = 0; p < KP; ++p) acc[p][e] = fma(cs[p], a, fma(sn[p], b, acc[p][e]));
                }
            }
        }

#pragma unroll
        for (int p = 0; p < KP; ++p) {
            const long idx = kk + p * stride;
            if (idx >= nk) continue;
            if (Hp != nullptr) {
                double* o = Hp + idx * NN;
                if (NN % 2 == 0) {
#pragma unroll
                    for (int e = 0; e < NN; e += 2)
                        *reinterpret_cast<double2*>(o + e) = make_double2(acc[p][e], acc[p][e + 1]);
                } else {
#pragma unroll
                    for (int e = 0; e < NN; ++e) o[e] = acc[p][e];
                }
            }
            if (eig != nullptr) {
                if (N == 1) {
                    eig[idx] = acc[p][0];
                } else if (N == 2) {
                    double lo, hi;
                    eig2_closed(acc[p][0], acc[p][2], acc[p][1], acc[p][3], lo, hi);
                    *reinterpret_cast<double2*>(eig + idx * 2) = make_double2(lo, hi);
                } else {
                    double* A = scratch + tid;  // element q at A[q * TPB]
#pragma unroll
                    for (int e = 0; e < NN; ++e) A[(long)e * TPB] = acc[p][e];
                    double* wv = A + (long)NN * TPB;
                    double* dd = wv + 4L * N * TPB;
                    double* ee = dd + (long)N * TPB;
                    hetrd_serial(N, A, TPB, dd, ee, TPB, wv);
                    const int fails = tridiag_ql(N, dd, ee, TPB);
                    if (fails && fail_count) atomicAdd(fail_count, fails);  // reported by tbk_model_check / the _host calls
                    double* o = eig + idx * N;
#pragma unroll
                    for (int i = 0; i < N; ++i) o[i] = dd[(long)i * TPB];
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Trigonometric-product form for nearest-cell models with N <= 2 (C2: the 2-band Haldane model).
// With every |R_d| <= 1,  e^{2 pi i k.R} = prod_d (c_d + i R_d s_d),  c_d = cos 2 pi k_d, s_d = sin 2 pi k_d, so
//   H(k) = sum_b phi_b(k) B_b ,   phi_b = prod_d {1, c_d, s_d}[t_d] ,   b = sum_d t_d 3^d   (3^D real functions),
// with the packed Hermitian coefficient matrices B_b accumulated once on the host (tbk_api.cu, tbk_model_create).
// Per k-point: D sincospi, 3^D - 2 D - 1 products, (3^D - 1) N^2 FMAs whose second operand is a uniform-register /
// constant-bank operand (the table is a kernel parameter): no shared memory, no loop over R, no selects.
// Same sum as the reference's Fourier loop (src/tbmodels/_tb_model.py:1111-1123), reassociated.
// KP k-points per thread and trip share the 64-bit immediates of the sincospi polynomials (two UMOVs each).
// ---------------------------------------------------------------------------------------------------------
template <int D>
struct Pow3 {
    static constexpr int value = 3 * Pow3<D - 1>::value;
};
template <>
struct Pow3<0> {
    static constexpr int value = 1;
};

template <int N, int D>
struct BasisTable {
    double w[Pow3<D>::value * N * N];
};

// sincospi_lean (tbk_math.cuh: same reduction, same polynomials) with a cheaper quadrant fix-up: one select per
// output and the signs applied as integer XORs on the high words.
__device__ __forceinline__ void sincospi_x(double t, double& s, double& c) {
    const double n = rint(t + t);
    const double r = fma(n, -0.5, t);
    const unsigned q = (unsigned)(long long)n;  // low bits of the (exact) integer n
    const double r2 = r * r;
    double ps = 0.00046221129498806536;
    ps = fma(ps, r2, -0.0073701436737117);
    ps = fma(ps, r2, 0.08214587730806341);
    ps = fma(ps, r2, -0.5992645291845754);
    ps = fma(ps, r2, 2.550164039876616);
    ps = fma(ps, r2, -5.167712780049969);
    double sv = fma(r * r2, ps, r * 1.2246467991473532e-16);  // pi = 3.141592653589793 + 1.2246467991473532e-16
    sv = fma(r, 3.141592653589793, sv);
    double pc = -0.00010370086335346046;
    pc = fma(pc, r2, 0.0019294938812021883);
    pc = fma(pc, r2, -0.025806887965145374);
    pc = fma(pc, r2, 0.2353306302840066);
    pc = fma(pc, r2, -1.3352627688538097);
    pc = fma(pc, r2, 4.058712126416765);
    pc = fma(pc, r2, -4.934802200544679);
    const double cv = fma(pc, r2, 1.0);
    // q mod 4:  0 -> (s, c),  1 -> (c, -s),  2 -> (-s, -c),  3 -> (-c, s)
    const bool odd = q & 1u;
    const double a = odd ? cv : sv, b = odd ? sv : cv;
    const unsigned qs = q << 30;  // bit 31 = bit 1 of q
    s = __hiloint2double(__double2hiint(a) ^ (int)(qs & 0x80000000u), __double2loint(a));
    c = __hiloint2double(__double2hiint(b) ^ (int)((qs + 0x40000000u) & 0x80000000u), __double2loint(b));
}

// sqrt(x) for finite x >= 0: hardware reciprocal-square-root seed (~2^-22), one coupled Newton step for g ~ sqrt(x) and
// h ~ 1 / (2 sqrt(x)) (~2^-44) and a residual correction g += (x - g^2) h (quadratic again: rounding-level error); x below
// DBL_MIN returns 0: zero (exact band degeneracy) or subnormal, which rsqrt.approx.ftz flushes.  A relative cut-off is not
// needed: the model's normalisation (tbk_api.cu, kScaleWindow) keeps every x that matters far above DBL_MIN.
__device__ __forceinline__ double sqrt_nonneg(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double g = x * y, h = 0.5 * y;
    const double r = fma(-g, h, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    const double d = fma(-g, g, x);
    g = fma(d, h, g);
    return (x >= DBL_MIN) ? g : 0.0;
}

// (Guarding the FMAs of exact-zero table entries -- 24 of 32 for the Haldane model -- with uniform predicates was measured
//  5 % slower than running them all: the kernel is issue bound as much as FP64-pipe bound.)
template <int N, int D, int KP>
__device__ __forceinline__ void basis_kpoints(const double (&kv)[KP][D], const BasisTable<N, D>& T,
                                              double (&acc)[KP][N * N]) {
    constexpr int NN = N * N;
    constexpr int NB3 = Pow3<D>::value;
    const double* __restrict__ w = T.w;
    double phi[KP][NB3];
    int n = 1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
        double sd[KP], cd[KP];
#pragma unroll
        for (int p = 0; p < KP; ++p) {
            sincospi_x(2.0 * kv[p][d], sd[p], cd[p]);
            phi[p][0] = 1.0;
            phi[p][n] = cd[p];
            phi[p][2 * n] = sd[p];
        }
#pragma unroll
        for (int b = 1; b < n; ++b) {
#pragma unroll
            for (int p = 0; p < KP; ++p) {
                phi[p][b + n] = phi[p][b] * cd[p];
                phi[p][b + 2 * n] = phi[p][b] * sd[p];
            }
        }
        n *= 3;
    }
#pragma unroll
    for (int p = 0; p < KP; ++p)
#pragma unroll
        for (int e = 0; e < NN; ++e) acc[p][e] = w[e];
#pragma unroll
    for (int b = 1; b < NB3; ++b)  // table entry outermost: one uniform operand feeds the KP k-points of the trip
#pragma unroll
        for (int e = 0; e < NN; ++e)
#pragma unroll
            for (int p = 0; p < KP; ++p) acc[p][e] = fma(phi[p][b], w[b * NN + e], acc[p][e]);
}

template <int N>
__device__ __forceinline__ void basis_store(const double (&acc)[N * N], long idx, double* __restrict__ Hp,
                                            double* __restrict__ eig) {
    // N = 2: the table was rotated on the host so that acc = (mean, Re h10, delta, Im h10) with mean = (h00 + h11) / 2,
    // delta = (h00 - h11) / 2 -- the closed form (tbk_math.cuh eig2_closed) needs exactly these
    constexpr int NN = N * N;
    if (Hp != nullptr) {
        if (N == 2) {
            Hp[idx * NN] = acc[0] + acc[2 % NN];
            Hp[idx * NN + 1] = acc[1 % NN];
            Hp[idx * NN + 2] = acc[0] - acc[2 % NN];
            Hp[idx * NN + 3] = acc[3 % NN];
        } else {
#pragma unroll
            for (int e = 0; e < NN; ++e) Hp[idx * NN + e] = acc[e];
        }
    }
    if (eig != nullptr) {
        if (N == 1) {
            eig[idx] = acc[0];
        } else {
            const double mean = acc[0], delta = acc[2 % NN];
            const double rad = sqrt_nonneg(fma(delta, delta, fma(acc[1 % NN], acc[1 % NN], acc[3 % NN] * acc[3 % NN])));
            *reinterpret_cast<double2*>(eig + idx * 2) = make_double2(mean - rad, mean + rad);
        }
    }
}

template <int D, int KP>
__device__ __forceinline__ void load_trip(double (&k)[KP][D], const double* __restrict__ kp) {
#pragma unroll
    for (int p = 0; p < KP; ++p) {
        if (D == 2) {
            const double2 v = *reinterpret_cast<const double2*>(kp + (long)p * TPB * D);
            k[p][0] = v.x;
            k[p][D - 1] = v.y;
        } else {
#pragma unroll
            for (int d = 0; d < D; ++d) k[p][d] = kp[(long)p * TPB * D + d];
        }
    }
}

// A CTA trip covers KP * TPB consecutive k-points; thread t owns t, t + TPB, ... (immediate offsets from one pointer).
template <int N, int D, int KP>
__global__ void __launch_bounds__(TPB)
hk_basis_kernel(const double* __restrict__ kpts, long nk, const __grid_constant__ BasisTable<N, D> T,
                double* __restrict__ Hp, double* __restrict__ eig) {
    constexpr int NN = N * N;
    constexpr long TRIP = (long)KP * TPB;
    const long step = (long)gridDim.x * TRIP;
    long base = (long)blockIdx.x * TRIP;
    double kn[KP][D];  // k-points of the next full trip (prefetched one trip ahead)
    if (base + TRIP <= nk) load_trip<D, KP>(kn, kpts + (base + threadIdx.x) * D);
    for (; base + TRIP <= nk; base += step) {  // full trips: no bounds checks
        double kv[KP][D];
#pragma unroll
        for (int p = 0; p < KP; ++p)
#pragma unroll
            for (int d = 0; d < D; ++d) kv[p][d] = kn[p][d];
        if (base + step + TRIP <= nk) load_trip<D, KP>(kn, kpts + (base + step + threadIdx.x) * D);
        double acc[KP][NN];
        basis_kpoints<N, D, KP>(kv, T, acc);
#pragma unroll
        for (int p = 0; p < KP; ++p) basis_store<N>(acc[p], base + threadIdx.x + (long)p * TPB, Hp, eig);
    }
    if (base < nk) {  // ragged last trip (at most one CTA gets here with work)
        for (long idx = base + threadIdx.x; idx < nk; idx += TPB) {
            double kv[1][D];
#pragma unroll
            for (int d = 0; d < D; ++d) kv[0][d] = kpts[idx * D + d];
            double acc[1][NN];
            basis_kpoints<N, D, 1>(kv, T, acc);
            basis_store<N>(acc[0], idx, Hp, eig);
        }
    }
}

template <int N, int D, int KP>
cudaError_t launch_basis_ndk(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, cudaStream_t st) {
    BasisTable<N, D> T;
    for (int i = 0; i < Pow3<D>::value * N * N; ++i) T.w[i] = md.basis[i];
    if (N == 2) {  // accumulate (mean, delta) of the diagonal instead of (h00, h11): see basis_store
        for (int b = 0; b < Pow3<D>::value; ++b) {
            const double h00 = md.basis[b * 4], h11 = md.basis[b * 4 + 2];
            T.w[b * (N * N)] = 0.5 * (h00 + h11);
            T.w[b * (N * N) + 2 % (N * N)] = 0.5 * (h00 - h11);
        }
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long blocks = (nk + KP * TPB - 1) / (KP * TPB);
    const long cap = (long)sms * 16;
    if (blocks > cap) blocks = cap;
    if (blocks <= 0) return cudaSuccess;
    hk_basis_kernel<N, D, KP><<<(unsigned)blocks, TPB, 0, st>>>(k, nk, T, Hp, eig);
    return cudaGetLastError();
}

template <int N, int D>
cudaError_t launch_basis_nd(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, cudaStream_t st) {
    if (D <= 2) {
        if (md.tune.basis_kp == 2) return launch_basis_ndk<N, D, 2>(md, k, nk, Hp, eig, st);  // tuning hook
        return launch_basis_ndk<N, D, 4>(md, k, nk, Hp, eig, st);
    }
    return launch_basis_ndk<N, D, 2>(md, k, nk, Hp, eig, st);
}

template <int N>
cudaError_t launch_basis_n(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, cudaStream_t st) {
    switch (md.dim) {
        case 1: return launch_basis_nd<N, 1>(md, k, nk, Hp, eig, st);
        case 2: return launch_basis_nd<N, 2>(md, k, nk, Hp, eig, st);
        case 3: return launch_basis_nd<N, 3>(md, k, nk, Hp, eig, st);
        default: return cudaErrorInvalidValue;
    }
}

template <int N, int D>
cudaError_t launch_nd(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, int* fail_count,
                      cudaStream_t st) {
    const size_t smem = hk_small_smem_bytes(N, md.dim, md.nR, TPB);
    cudaError_t err =
        cudaFuncSetAttribute(hk_small_kernel<N, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long blocks = (nk + TPB - 1) / TPB;
    if (N <= 2) blocks = (blocks + 1) / 2;  // two k-points per thread and trip
    // persistent-ish: the tables are loaded once per CTA, so cap the grid at a few waves
    const long cap = (long)sms * 16;
    if (blocks > cap) blocks = cap;
    if (blocks <= 0) return cudaSuccess;
    hk_small_kernel<N, D><<<(unsigned)blocks, TPB, smem, st>>>(k, nk, md.Rd, md.Ri, md.W, md.dim, md.nR, md.use_z, Hp,
                                                               eig, fail_count);
    return cudaGetLastError();
}

template <int N>
cudaError_t launch_n(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, int* fail_count,
                     cudaStream_t st) {
    switch (md.dim) {
        case 1: return launch_nd<N, 1>(md, k, nk, Hp, eig, fail_count, st);
        case 2: return launch_nd<N, 2>(md, k, nk, Hp, eig, fail_count, st);
        case 3: return launch_nd<N, 3>(md, k, nk, Hp, eig, fail_count, st);
        default: return launch_nd<N, 0>(md, k, nk, Hp, eig, fail_count, st);
    }
}

}  // namespace

size_t hk_small_smem_bytes(int n, int dim, int nR, int threads) {
    if (threads <= 0) threads = TPB;
    const size_t nn = (size_t)n * n;
    size_t doubles = 2 * (size_t)nR * nn + small_table_doubles(nR, dim);
    if (n > 2) doubles += (nn + 6 * (size_t)n) * threads;
    return doubles * 8;
}

cudaError_t launch_hk_small(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, int* fail_count,
                            cudaStream_t st) {
    if (md.basis_ok) {
        if (md.n == 1) return launch_basis_n<1>(md, k, nk, Hp, eig, st);
        if (md.n == 2) return launch_basis_n<2>(md, k, nk, Hp, eig, st);
    }
    switch (md.n) {
        case 1: return launch_n<1>(md, k, nk, Hp, eig, fail_count, st);
        case 2: return launch_n<2>(md, k, nk, Hp, eig, fail_count, st);
        case 3: return launch_n<3>(md, k, nk, Hp, eig, fail_count, st);
        case 4: return launch_n<4>(md, k, nk, Hp, eig, fail_count, st);
        case 5: return launch_n<5>(md, k, nk, Hp, eig, fail_count, st);
        case 6: return launch_n<6>(md, k, nk, Hp, eig, fail_count, st);
        case 7: return launch_n<7>(md, k, nk, Hp, eig, fail_count, st);
        case 8: return launch_n<8>(md, k, nk, Hp, eig, fail_count, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace tbk
