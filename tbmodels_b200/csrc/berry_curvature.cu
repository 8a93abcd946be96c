// berry_curvature.cu -- Berry curvature of every band from eigenvectors and dH/dk (tbk_berry_curvature, tbk_api.cu
// run_eigh).
//
// Inputs of k-point kk (all produced on the device by run_eigh):
//   eig [N]                ascending eigenvalues of the convention-2 H(k) (eigh_kernel)
//   V   [N][N] c128        eigenvectors, V[i][j] = component i of the eigenvector of eig[j] (eigh_kernel)
//   X   [terms][N][N] c128 the Taylor terms of kdotp_construct.cu: dH/dk_a for a < dim and, for convention 1, H(k) itself
//                          as term dim (the zero power tuple)
//
// 1. Product (launch_berry_product): M_a = V^H X'_a V for every direction a, with X'_a = dH/dk_a (convention 2) or
//    X'_a[i][j] = dH/dk_a[i][j] + 2 pi i (pos[j][a] - pos[i][a]) H[i][j] (convention 1, the k-derivative of
//    D H D^H, D = diag(e^{-2 pi i k.pos_i}), seen in the convention-2 eigenbasis), applied where X_a is loaded.  M_a
//    overwrites X_a.
//      N > kSmallMaxN: two batched complex GEMMs per direction on the FP64 tensor cores (mma.sync.m8n8k4.f64, SASS
//        DMMA.8x8x4), complex arithmetic as four real products: Y_a = X'_a V into the scratch Y, then M_a = V^H Y_a.
//        64 x 64 complex output tile per CTA, K in steps of 16 through shared memory, the next step prefetched into
//        registers; 8 warps of 32 x 16.  The K loop runs in order with no split, so every entry's sum has a fixed order.
//      N <= kSmallMaxN: one thread per (k-point, direction, column l) forms y = X'_a v_l in registers, then
//        M_a[:, l] = V^H y (plain DFMA); the CTA holds whole (k-point, direction) groups and writes after a barrier.
// 2. Curvature (launch_berry_curvature), one CTA per k-point.  Clusters as in band_velocity.cu: maximal runs of ascending
//    eigenvalues whose gaps are <= degen_tol * rho, rho = max_n |eig_n|.  For every pair a < b (pair index p in the order
//    (0,1), (0,2), ..., (1,2), ...):
//      a singleton n:  curv[n][p] = -2 sum_{l != n} Im(M_a[n][l] M_b[l][n]) / ((E_n - E_l)(E_n - E_l));
//      a cluster c:    the ascending eigenvalues (jacobi_eig.cuh) of the m x m Hermitian block
//                      F_nm = i sum_{l not in c} (M_a[n][l] M_b[l][m] - M_b[n][l] M_a[l][m]) / ((E_n - E_l)(E_m - E_l)),
//                      upper triangle computed, lower mirrored; the blocks live where band_velocity.cu keeps its blocks
//                      (shared memory, or eigh's global scratch for the sizes where eigh works there).
//    Sums over l run in ascending order.
// No atomics, nothing shared between k-points: the bits of a k-point do not depend on its chunk.  Every operation is
// exactly equivariant under a power-of-two scaling of H (M and E scale alike, quotients by products of computed
// differences, no approximate reciprocals), so the curvature of a model stored scaled equals the unscaled one's bit for
// bit.
#include "jacobi_eig.cuh"
#include "tbk_kernels.h"

namespace tbk {

namespace {

constexpr double kTwoPi = 6.28318530717958647692;

// ------------------------------------------------------------------------------------------ product, DMMA variant
constexpr int PT = 256;           // threads: 8 warps, 2 (rows) x 4 (columns), warp tile 32 x 16
constexpr int PBM = 64, PBN = 64; // complex output tile
constexpr int PBK = 16;           // K step
constexpr int PSA = PBK + 4;      // A row stride in doubles: fragment reads (row g, column t) hit (4 g + t) mod 16, distinct
constexpr int PSB = PBN + 4;      // B row stride in doubles: fragment reads (row t, column g) hit (4 t + g) mod 16, distinct
constexpr int P_LD = PBM * PBK / PT;  // complex elements of each operand tile loaded per thread (4)

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// One launch computes C[z][y] = op(A[z][y]) B[z][y] for the N x N complex matrices of k-point z = blockIdx.z and direction
// y = blockIdx.y, each at base + z * kstride + y * dstride (complex elements; dstride 0 = shared by the directions).
//   CONJ = false: op(A) = X'_y, A = X_y, with the convention-1 term added from H (H non-null; hstride per k-point).
//   CONJ = true:  op(A) = A^H (A = V).
template <bool CONJ>
__global__ void __launch_bounds__(PT)
berry_product_kernel(int N, int dim, const double2* __restrict__ A, long a_k, long a_d, const double2* __restrict__ B,
                     long b_k, long b_d, double2* __restrict__ C, long c_k, long c_d, const double2* __restrict__ H,
                     long h_k, const double* __restrict__ pos) {
    __shared__ __align__(16) double Ar[PBM * PSA], Ai[PBM * PSA], Br[PBK * PSB], Bi[PBK * PSB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp >> 2, wn = warp & 3, g = lane >> 2, t = lane & 3;
    const int tiles_n = (N + PBN - 1) / PBN;
    const int m0 = (blockIdx.x / tiles_n) * PBM, n0 = (blockIdx.x % tiles_n) * PBN;
    const int dir = blockIdx.y;
    const long kk = blockIdx.z;
    const double2* Ap = A + kk * a_k + dir * a_d;
    const double2* Bp = B + kk * b_k + dir * b_d;
    const double2* Hp = H ? H + kk * h_k : nullptr;
    double2* Cp = C + kk * c_k + dir * c_d;
    const double2 zero = make_double2(0.0, 0.0);

    // operand element e = tid + PT q of a tile: A (not CONJ) row e / PBK, column e % PBK (coalesced along the row of X);
    // A (CONJ) column e / PBM, row e % PBM (coalesced along the row of V); B row e / PBN, column e % PBN
    double2 ra[P_LD], rh[P_LD], rb[P_LD];
    auto fetch = [&](int k0) {
#pragma unroll
        for (int q = 0; q < P_LD; ++q) {
            const int e = tid + PT * q;
            if (CONJ) {
                const int r = m0 + e % PBM, c = k0 + e / PBM;
                ra[q] = (r < N && c < N) ? Ap[(size_t)c * N + r] : zero;
            } else {
                const int r = m0 + e / PBK, c = k0 + e % PBK;
                const bool in = r < N && c < N;
                ra[q] = in ? Ap[(size_t)r * N + c] : zero;
                if (Hp) rh[q] = in ? Hp[(size_t)r * N + c] : zero;
            }
            const int br = k0 + e / PBN, bc = n0 + e % PBN;
            rb[q] = (br < N && bc < N) ? Bp[(size_t)br * N + bc] : zero;
        }
    };
    auto stash = [&](int k0) {
#pragma unroll
        for (int q = 0; q < P_LD; ++q) {
            const int e = tid + PT * q;
            if (CONJ) {
                const int r = e % PBM, c = e / PBM;
                Ar[r * PSA + c] = ra[q].x;
                Ai[r * PSA + c] = -ra[q].y;
            } else {
                const int r = e / PBK, c = e % PBK;
                double2 x = ra[q];
                if (Hp && m0 + r < N && k0 + c < N) {
                    const double f = kTwoPi * (pos[(size_t)(k0 + c) * dim + dir] - pos[(size_t)(m0 + r) * dim + dir]);
                    x = make_double2(fma(-f, rh[q].y, x.x), fma(f, rh[q].x, x.y));
                }
                Ar[r * PSA + c] = x.x;
                Ai[r * PSA + c] = x.y;
            }
            const int br = e / PBN, bc = e % PBN;
            Br[br * PSB + bc] = rb[q].x;
            Bi[br * PSB + bc] = rb[q].y;
        }
    };

    double cr[4][2][2], ci[4][2][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) cr[i][j][0] = cr[i][j][1] = ci[i][j][0] = ci[i][j][1] = 0.0;

    fetch(0);
    for (int k0 = 0; k0 < N; k0 += PBK) {
        __syncthreads();  // every warp is done with the previous step's tiles
        stash(k0);
        __syncthreads();
        if (k0 + PBK < N) fetch(k0 + PBK);
#pragma unroll
        for (int k4 = 0; k4 < PBK / 4; ++k4) {
            double ar[4], ai[4], br[2], bi[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int o = (wm * 32 + i * 8 + g) * PSA + k4 * 4 + t;
                ar[i] = Ar[o];
                ai[i] = Ai[o];
            }
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int o = (k4 * 4 + t) * PSB + wn * 16 + j * 8 + g;
                br[j] = Br[o];
                bi[j] = Bi[o];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    dmma(cr[i][j][0], cr[i][j][1], ar[i], br[j]);
                    dmma(cr[i][j][0], cr[i][j][1], -ai[i], bi[j]);
                    dmma(ci[i][j][0], ci[i][j][1], ar[i], bi[j]);
                    dmma(ci[i][j][0], ci[i][j][1], ai[i], br[j]);
                }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = m0 + wm * 32 + i * 8 + g;
        if (r >= N) continue;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int c = n0 + wn * 16 + j * 8 + 2 * t;
            if (c < N) Cp[(size_t)r * N + c] = make_double2(cr[i][j][0], ci[i][j][0]);
            if (c + 1 < N) Cp[(size_t)r * N + c + 1] = make_double2(cr[i][j][1], ci[i][j][1]);
        }
    }
}

// ------------------------------------------------------------------------------------------ product, FMA variant
constexpr int PS_T = 128;

// Thread (group, l), group = (k-point, direction): y = X'_a v_l, then M_a[:, l] = V^H y, written over X_a once every
// thread of the CTA has read its operands (a CTA holds PS_T / NT whole groups).
template <int NT>
__global__ void __launch_bounds__(PS_T)
berry_product_small_kernel(int dim, long groups, const double2* __restrict__ V, double2* X, int terms, bool conv1,
                           const double* __restrict__ pos) {
    constexpr int NN = NT * NT;
    constexpr int GPC = PS_T / NT;
    const int l = threadIdx.x % NT;
    const long grp = (long)blockIdx.x * GPC + threadIdx.x / NT;
    const bool live = threadIdx.x < GPC * NT && grp < groups;
    double2 mv[NT];
    if (live) {
        const long kk = grp / dim;
        const int a = (int)(grp - kk * dim);
        const double2* Vk = V + kk * NN;
        const double2* Xa = X + (kk * terms + a) * NN;
        const double2* Hk = X + (kk * terms + dim) * NN;
        double2 y[NT];
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            double yr = 0.0, yi = 0.0;
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                double2 x = Xa[i * NT + j];
                if (conv1) {
                    const double f = kTwoPi * (pos[(size_t)j * dim + a] - pos[(size_t)i * dim + a]);
                    const double2 h = Hk[i * NT + j];
                    x = make_double2(fma(-f, h.y, x.x), fma(f, h.x, x.y));
                }
                const double2 v = Vk[j * NT + l];
                yr = fma(x.x, v.x, fma(-x.y, v.y, yr));
                yi = fma(x.x, v.y, fma(x.y, v.x, yi));
            }
            y[i] = make_double2(yr, yi);
        }
#pragma unroll
        for (int n = 0; n < NT; ++n) {
            double re = 0.0, im = 0.0;
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                const double2 u = Vk[i * NT + n];
                re = fma(u.x, y[i].x, fma(u.y, y[i].y, re));
                im = fma(u.x, y[i].y, fma(-u.y, y[i].x, im));
            }
            mv[n] = make_double2(re, im);
        }
    }
    __syncthreads();
    if (live) {
        const long kk = grp / dim;
        const int a = (int)(grp - kk * dim);
        double2* Ma = X + (kk * terms + a) * NN;
#pragma unroll
        for (int n = 0; n < NT; ++n) Ma[n * NT + l] = mv[n];
    }
}

template <int NT>
cudaError_t launch_small_t(int dim, long nk, const double* vec, double* X, int terms, bool conv1, const double* pos,
                           cudaStream_t st) {
    const long groups = nk * dim, gpc = PS_T / NT;
    const long blocks = (groups + gpc - 1) / gpc;
    if (blocks > 2147483647L) return cudaErrorInvalidConfiguration;
    berry_product_small_kernel<NT><<<(unsigned)blocks, PS_T, 0, st>>>(dim, groups, reinterpret_cast<const double2*>(vec),
                                                                      reinterpret_cast<double2*>(X), terms, conv1, pos);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------------ curvature
template <int T>
__global__ void __launch_bounds__(T)
berry_curvature_kernel(int N, int dim, long nk, const double* __restrict__ eig, const double2* __restrict__ M, int terms,
                       double degen_tol, double* __restrict__ curv, double2* __restrict__ gB) {
    extern __shared__ __align__(16) double2 smc[];
    const int tid = threadIdx.x;
    const long kk = blockIdx.x;
    if (kk >= nk) return;
    const size_t NN = (size_t)N * N;
    double2* B;  // block of the cluster starting at s: B[s * N + a * m + b]
    int* cst;    // [N] first index of the cluster of j
    if (gB) {
        B = gB + (size_t)kk * 2 * NN;
        cst = reinterpret_cast<int*>(smc);
    } else {
        B = smc;
        cst = reinterpret_cast<int*>(smc + NN);
    }
    int* csz = cst + N;  // [N] its size
    const double* e = eig + (size_t)kk * N;
    const int P = dim * (dim - 1) / 2;
    double* out = curv + (size_t)kk * N * P;

    // ---- clusters, exactly as band_velocity_kernel ----
    double rho = 0.0;
    for (int n = 0; n < N; ++n) rho = fmax(rho, fabs(e[n]));
    const double thr = degen_tol * rho;
    for (int j = tid; j < N; j += T) {
        int s = j;
        while (s > 0 && e[s] - e[s - 1] <= thr) --s;
        int t = j + 1;
        while (t < N && e[t] - e[t - 1] <= thr) ++t;
        cst[j] = s;
        csz[j] = t - s;
    }
    __syncthreads();

    int p = 0;
    for (int a = 0; a < dim; ++a)
        for (int b = a + 1; b < dim; ++b, ++p) {
            const double2* Ma = M + ((size_t)kk * terms + a) * NN;
            const double2* Mb = M + ((size_t)kk * terms + b) * NN;
            // ---- 1. singletons: their curvature; cluster columns j = s + q: entries (r, q), r <= q, of F ----
            for (int j = tid; j < N; j += T) {
                const int s = cst[j], m = csz[j];
                const double ej = e[j];
                if (m == 1) {
                    double acc = 0.0;
                    for (int l = 0; l < N; ++l) {
                        if (l == j) continue;
                        const double2 x = Ma[(size_t)j * N + l], y = Mb[(size_t)l * N + j];
                        const double d = ej - e[l];
                        acc += fma(x.x, y.y, x.y * y.x) / (d * d);  // Im(x y) / (E_j - E_l)^2
                    }
                    out[(size_t)j * P + p] = -2.0 * acc;
                    continue;
                }
                const int q = j - s;
                for (int r = 0; r <= q; ++r) {
                    const int nr = s + r;
                    const double er = e[nr];
                    double sr = 0.0, si = 0.0;
                    for (int l = 0; l < N; ++l) {
                        if (l == s) {
                            l = s + m - 1;
                            continue;
                        }
                        const double2 x1 = Ma[(size_t)nr * N + l], y1 = Mb[(size_t)l * N + j];
                        const double2 x2 = Mb[(size_t)nr * N + l], y2 = Ma[(size_t)l * N + j];
                        const double zr = fma(x1.x, y1.x, -x1.y * y1.y) - fma(x2.x, y2.x, -x2.y * y2.y);
                        const double zi = fma(x1.x, y1.y, x1.y * y1.x) - fma(x2.x, y2.y, x2.y * y2.x);
                        const double den = (er - e[l]) * (ej - e[l]);
                        sr += zr / den;
                        si += zi / den;
                    }
                    // F = i (sr + i si)
                    if (r == q) B[(size_t)s * N + (size_t)q * m + q] = make_double2(-si, 0.0);
                    else {
                        B[(size_t)s * N + (size_t)r * m + q] = make_double2(-si, sr);
                        B[(size_t)s * N + (size_t)q * m + r] = make_double2(-si, -sr);
                    }
                }
            }
            __syncthreads();
            // ---- 2. eigenvalues of every block: the thread of the cluster's first column ----
            for (int j = tid; j < N; j += T) {
                const int m = csz[j];
                if (m == 1 || cst[j] != j) continue;
                double2* blk = B + (size_t)j * N;
                jacobi_eigvals(blk, m);
                for (int c = 0; c < m; ++c) out[(size_t)(j + c) * P + p] = blk[c * m + c].x;
            }
            __syncthreads();  // B is reused by the next pair
        }
}

size_t curvature_smem(int n, bool global_b) { return (global_b ? 0 : (size_t)n * n * 16) + (size_t)2 * n * sizeof(int); }

template <int T>
cudaError_t launch_curv_t(int n, int dim, long nk, const double* eig, const double* M, int terms, double degen_tol,
                          double* curv, double2* gB, cudaStream_t st) {
    const size_t smem = curvature_smem(n, gB != nullptr);
    cudaError_t err = cudaFuncSetAttribute(berry_curvature_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    if (nk > 2147483647L) return cudaErrorInvalidConfiguration;
    berry_curvature_kernel<T><<<(unsigned)nk, T, smem, st>>>(n, dim, nk, eig, reinterpret_cast<const double2*>(M), terms,
                                                             degen_tol, curv, gB);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_berry_product(int n, int dim, long nk, const double* vec, double* X, int terms, bool conv1,
                                 const double* pos, double* Y, cudaStream_t st) {
    if (nk <= 0 || n <= 0) return cudaSuccess;
    switch (n) {
        case 1: return launch_small_t<1>(dim, nk, vec, X, terms, conv1, pos, st);
        case 2: return launch_small_t<2>(dim, nk, vec, X, terms, conv1, pos, st);
        case 3: return launch_small_t<3>(dim, nk, vec, X, terms, conv1, pos, st);
        case 4: return launch_small_t<4>(dim, nk, vec, X, terms, conv1, pos, st);
        case 5: return launch_small_t<5>(dim, nk, vec, X, terms, conv1, pos, st);
        case 6: return launch_small_t<6>(dim, nk, vec, X, terms, conv1, pos, st);
        case 7: return launch_small_t<7>(dim, nk, vec, X, terms, conv1, pos, st);
        case 8: return launch_small_t<8>(dim, nk, vec, X, terms, conv1, pos, st);
        default: break;
    }
    static_assert(kSmallMaxN == 8, "the FMA variant is instantiated for N = 1 .. kSmallMaxN");
    if (nk > 65535) return cudaErrorInvalidConfiguration;  // grid.z
    const long NN = (long)n * n;
    const int tiles = ((n + PBM - 1) / PBM) * ((n + PBN - 1) / PBN);
    const dim3 grid((unsigned)tiles, (unsigned)dim, (unsigned)nk);
    const double2* V = reinterpret_cast<const double2*>(vec);
    double2* Xc = reinterpret_cast<double2*>(X);
    double2* Yc = reinterpret_cast<double2*>(Y);
    // Y_a = X'_a V
    berry_product_kernel<false><<<grid, PT, 0, st>>>(n, dim, Xc, terms * NN, NN, V, NN, 0, Yc, dim * NN, NN,
                                                    conv1 ? Xc + dim * NN : nullptr, terms * NN, pos);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return err;
    // M_a = V^H Y_a, over X_a
    berry_product_kernel<true><<<grid, PT, 0, st>>>(n, dim, V, NN, 0, Yc, dim * NN, NN, Xc, terms * NN, NN, nullptr, 0, pos);
    return cudaGetLastError();
}

cudaError_t launch_berry_curvature(int n, int dim, long nk, const double* eig, const double* M, int terms,
                                   double degen_tol, double* curv, double* scratch, cudaStream_t st) {
    if (nk <= 0 || n <= 0 || dim < 2) return cudaSuccess;
    double2* gB = nullptr;
    if (!eigh_in_smem(n)) {
        if (!scratch) return cudaErrorInvalidValue;
        gB = reinterpret_cast<double2*>(scratch);
    }
    if (n <= 32) return launch_curv_t<32>(n, dim, nk, eig, M, terms, degen_tol, curv, gB, st);
    if (n <= 64) return launch_curv_t<64>(n, dim, nk, eig, M, terms, degen_tol, curv, gB, st);
    if (n <= 128) return launch_curv_t<128>(n, dim, nk, eig, M, terms, degen_tol, curv, gB, st);
    return launch_curv_t<256>(n, dim, nk, eig, M, terms, degen_tol, curv, gB, st);
}

}  // namespace tbk
