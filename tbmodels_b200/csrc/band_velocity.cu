// band_velocity.cu -- band velocities dE_n/dk_d from eigenvectors and dH/dk_d, one CTA per k-point.
//
// Inputs of k-point kk (all produced on the device by tbk_band_velocity, tbk_api.cu run_eigh):
//   eig [N]          ascending eigenvalues of H(k) (eigh_kernel)
//   V   [N][N] c128  eigenvectors, V[i][j] = component i of the eigenvector of eig[j] (numpy layout, eigh_kernel)
//   dH  [dim][N][N]  c128 dH/dk_d, full Hermitian matrices (the order-1 Taylor terms of kdotp_construct.cu)
// Output vel [N][dim].
//
// Clusters: maximal runs of ascending eigenvalues whose consecutive gaps are <= degen_tol * rho, rho = max_n |eig_n|.
//   m = 1 (a plain band): Hellmann-Feynman, vel[j][d] = Re(v_j^H dH_d v_j).
//   m > 1: degenerate perturbation theory, vel[s .. s+m)[d] = ascending eigenvalues of the m x m Hermitian block
//          B_ab = v_{s+a}^H dH_d v_{s+b}, by cyclic complex Jacobi (one thread per cluster, serial: speed matters only
//          for small m).
// Per direction: thread j forms y = dH_d v_j four rows at a time and accumulates Re(v_j^H y) (dim N^3 complex FMAs per
// k-point); the columns of clusters also store y in Y[.][j], the block entries are then v_a^H y_b, stored at B + s N
// (rows s .. s+m of an N x N array hold the m^2 entries, so the blocks of all clusters fit side by side).  Y and B live in
// shared memory or, for the sizes where eigh_kernel itself works on global scratch, on that same scratch (32 N^2 bytes
// per k-point, free once eigh is done).
// No atomics and nothing shared between CTAs: the bits of a k-point do not depend on its chunk or position.  Every
// operation is exactly equivariant under a power-of-two scaling of H (no approximate reciprocal square roots), so the
// results of a model stored scaled by 2^-s are exactly 2^-s times those of the unscaled model.
#include "jacobi_eig.cuh"
#include "tbk_kernels.h"

namespace tbk {

namespace {

constexpr int kRows = 4;          // rows of y per pass (register blocking of dH_d v_j)

template <int T>
__global__ void __launch_bounds__(T)
band_velocity_kernel(int N, int dim, long nk, const double* __restrict__ eig, const double* __restrict__ vec,
                     const double* __restrict__ dH, double degen_tol, double* __restrict__ vel, double2* __restrict__ gYB) {
    extern __shared__ __align__(16) double2 smv[];
    const int tid = threadIdx.x;
    const long kk = blockIdx.x;
    if (kk >= nk) return;
    const size_t NN = (size_t)N * N;
    double2* Y;  // Y[r * N + j] = (dH_d v_j)_r for the columns of clusters
    double2* B;  // block of the cluster starting at s: B[s * N + a * m + b]
    int* cst;    // [N] first index of the cluster of j
    int* csz;    // [N] its size
    if (gYB) {
        Y = gYB + (size_t)kk * 2 * NN;
        B = Y + NN;
        cst = reinterpret_cast<int*>(smv);
    } else {
        Y = smv;
        B = smv + NN;
        cst = reinterpret_cast<int*>(smv + 2 * NN);
    }
    csz = cst + N;
    const double* e = eig + (size_t)kk * N;
    const double2* V = reinterpret_cast<const double2*>(vec) + (size_t)kk * NN;
    double* out = vel + (size_t)kk * N * dim;

    // ---- clusters: a cut before n where the gap is not <= degen_tol * rho (a NaN gap cuts) ----
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

    for (int d = 0; d < dim; ++d) {
        const double2* A = reinterpret_cast<const double2*>(dH) + ((size_t)kk * dim + d) * NN;
        // ---- 1. every column: y = dH_d v_j, Re(v_j^H y); cluster columns keep y ----
        for (int j = tid; j < N; j += T) {
            const int s = cst[j], m = csz[j];
            double acc = 0.0;
            for (int r0 = 0; r0 < N; r0 += kRows) {
                double yr[kRows], yi[kRows];
#pragma unroll
                for (int q = 0; q < kRows; ++q) yr[q] = yi[q] = 0.0;
                const int nr = min(kRows, N - r0);
                if (nr == kRows) {
                    for (int i = 0; i < N; ++i) {
                        const double2 v = V[(size_t)i * N + j];
#pragma unroll
                        for (int q = 0; q < kRows; ++q) {
                            const double2 h = A[(size_t)(r0 + q) * N + i];
                            yr[q] = fma(h.x, v.x, fma(-h.y, v.y, yr[q]));
                            yi[q] = fma(h.x, v.y, fma(h.y, v.x, yi[q]));
                        }
                    }
                } else {
                    for (int i = 0; i < N; ++i) {
                        const double2 v = V[(size_t)i * N + j];
#pragma unroll
                        for (int q = 0; q < kRows; ++q) {
                            if (q >= nr) break;
                            const double2 h = A[(size_t)(r0 + q) * N + i];
                            yr[q] = fma(h.x, v.x, fma(-h.y, v.y, yr[q]));
                            yi[q] = fma(h.x, v.y, fma(h.y, v.x, yi[q]));
                        }
                    }
                }
#pragma unroll
                for (int q = 0; q < kRows; ++q) {
                    if (q >= nr) break;
                    const double2 u = V[(size_t)(r0 + q) * N + j];
                    acc = fma(u.x, yr[q], fma(u.y, yi[q], acc));  // Re(conj(u) y)
                    if (m > 1) Y[(size_t)(r0 + q) * N + j] = make_double2(yr[q], yi[q]);
                }
            }
            if (m == 1) out[(size_t)j * dim + d] = acc;
            else B[(size_t)s * N + (size_t)(j - s) * m + (j - s)] = make_double2(acc, 0.0);
        }
        __syncthreads();
        // ---- 2. off-diagonal block entries B_ab = v_a^H y_b, a < b: thread of column b ----
        for (int j = tid; j < N; j += T) {
            const int s = cst[j], m = csz[j];
            if (m == 1) continue;
            const int b = j - s;
            for (int a = 0; a < b; ++a) {
                double re = 0.0, im = 0.0;
                for (int r = 0; r < N; ++r) {
                    const double2 u = V[(size_t)r * N + s + a], y = Y[(size_t)r * N + j];
                    re = fma(u.x, y.x, fma(u.y, y.y, re));
                    im = fma(u.x, y.y, fma(-u.y, y.x, im));
                }
                B[(size_t)s * N + (size_t)a * m + b] = make_double2(re, im);
                B[(size_t)s * N + (size_t)b * m + a] = make_double2(re, -im);
            }
        }
        __syncthreads();
        // ---- 3. eigenvalues of every block: the thread of the cluster's first column ----
        for (int j = tid; j < N; j += T) {
            const int m = csz[j];
            if (m == 1 || cst[j] != j) continue;
            double2* blk = B + (size_t)j * N;
            jacobi_eigvals(blk, m);
            for (int a = 0; a < m; ++a) out[(size_t)(j + a) * dim + d] = blk[a * m + a].x;
        }
        __syncthreads();  // Y and B are reused by the next direction
    }
}

size_t velocity_smem(int n, bool global_yb) { return (global_yb ? 0 : (size_t)2 * n * n * 16) + (size_t)2 * n * sizeof(int); }

template <int T>
cudaError_t launch_t(int n, int dim, long nk, const double* eig, const double* vec, const double* dH, double degen_tol,
                     double* vel, double2* gYB, cudaStream_t st) {
    const size_t smem = velocity_smem(n, gYB != nullptr);
    cudaError_t err = cudaFuncSetAttribute(band_velocity_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    if (nk > 2147483647L) return cudaErrorInvalidConfiguration;
    band_velocity_kernel<T><<<(unsigned)nk, T, smem, st>>>(n, dim, nk, eig, vec, dH, degen_tol, vel, gYB);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_band_velocity(int n, int dim, long nk, const double* eig, const double* vec, const double* dH,
                                 double degen_tol, double* vel, double* scratch, cudaStream_t st) {
    if (nk <= 0 || n <= 0) return cudaSuccess;
    double2* gYB = nullptr;
    if (!eigh_in_smem(n)) {
        if (!scratch) return cudaErrorInvalidValue;
        gYB = reinterpret_cast<double2*>(scratch);
    }
    if (n <= 32) return launch_t<32>(n, dim, nk, eig, vec, dH, degen_tol, vel, gYB, st);
    if (n <= 64) return launch_t<64>(n, dim, nk, eig, vec, dH, degen_tol, vel, gYB, st);
    if (n <= 128) return launch_t<128>(n, dim, nk, eig, vec, dH, degen_tol, vel, gYB, st);
    return launch_t<256>(n, dim, nk, eig, vec, dH, degen_tol, vel, gYB, st);
}

}  // namespace tbk
