// eig_vectors.cu -- batched Hermitian eigen-decomposition WITH eigenvectors (`eigh`), one CTA per matrix.
//
// SURVEY.md section 8 row f4: the step right after Model.eigenval (reference src/tbmodels/_tb_model.py:1134-1150 calls
// scipy.linalg.eigvalsh, values only) for Berry-phase / Z2Pack-type consumers is scipy.linalg.eigh -- LAPACK zheev[rd]
// with JOBZ = 'V'.  Restated here in the classical three steps (EISPACK tred2 / tql2 organisation, LAPACK zhetd2
// reflector conventions as everywhere else in this library):
//   1. Householder reduction A = Q T Q^H with the unitary Q = H_0 H_1 ... H_{N-2} accumulated explicitly
//      (Q <- Q (I - tau v v^H) after every step);
//   2. implicit-shift QL on the real tridiagonal T (the same iteration as tbk_math.cuh tridiag_ql); one thread runs
//      the serial recurrence and records the plane rotations of a sweep, then ALL threads apply them to their rows
//      of Q (a row only ever mixes with itself under column rotations, so rows are independent);
//   3. eigenvalues sorted ascending, eigenvector columns permuted with them (v[:, j] belongs to w[j], like numpy).
// Layout: the matrix and Q^T are stored full (both triangles) with thread c owning COLUMN c: every inner loop reads
// element (j, c) for running j, which is bank-conflict free in shared memory and coalesced in global memory.  The
// Hermitian product uses A[c][j] = conj(A[j][c]), the rank-2 update touches both triangles.
// The same code runs with both arrays in shared memory (N <= 12) or on global scratch (L2 resident; faster above because
// shared memory would cap residency, see eigh_in_smem).  Not tuned further: the eigenvalue-only path is the benchmarked one.
// Eigenvectors are defined up to a phase (and up to a rotation inside degenerate subspaces); the parity tests check
// residual, orthonormality and the eigenvalues -- not the phase.
#include <cstdlib>

#include "tbk_kernels.h"
#include "tbk_math.cuh"

namespace tbk {

namespace {

__device__ __forceinline__ int itri(int i) { return (i * (i + 1)) >> 1; }
__device__ __forceinline__ int itrs(int i) { return (i * (i - 1)) >> 1; }

// Sum of a double2 over the CTA, result in every thread.  red: [T / 32] scratch.
template <int T>
__device__ __forceinline__ double2 block_sum2(double2 v, double2* red) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, off);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, off);
    }
    if constexpr (T == 32) {
        return v;
    } else {
        __syncthreads();  // red may still be read by the previous call
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
        __syncthreads();
        double2 s = make_double2(0.0, 0.0);
#pragma unroll
        for (int w = 0; w < T / 32; ++w) {
            s.x += red[w].x;
            s.y += red[w].y;
        }
        return s;
    }
}

template <int T>
__global__ void __launch_bounds__(T)
eigh_kernel(const double* __restrict__ Hp, int N, long nk, double* __restrict__ eig_out, double* __restrict__ vec_out,
            double2* __restrict__ gA, double2* __restrict__ gQ, int* __restrict__ fail_count) {
    extern __shared__ __align__(16) double2 sm[];
    const int tid = threadIdx.x;
    const long kk = blockIdx.x;
    if (kk >= nk) return;
    const int NN = N * N;
    double2* M;   // M[j * N + c]  = A[j][c]
    double2* QT;  // QT[j * N + r] = Q[r][j]
    double2* vecs;
    if (gA) {
        M = gA + (size_t)kk * NN;
        QT = gQ + (size_t)kk * NN;
        vecs = sm;
    } else {
        M = sm;
        QT = sm + NN;
        vecs = sm + 2 * NN;
    }
    double2* V = vecs;          // [N] reflector
    double2* W = V + N;         // [N] p, then w
    double2* CS = W + N;        // [N] (c, s) of the rotations of one QL sweep; later the sort permutation
    double2* red = CS + N;      // [T / 32]
    double* d = reinterpret_cast<double*>(red + T / 32);  // [N]
    double* e = d + N;                                     // [N]
    int* ctl = reinterpret_cast<int*>(e + N);              // [4]

    // ---- load: packed Hermitian (tbk_math.cuh layout) -> full matrix; Q = I ----
    {
        const double* src = Hp + (size_t)kk * NN;
        const int ntri = itri(N);
        for (int idx = tid; idx < NN; idx += T) {
            const int j = idx / N, c = idx - j * N;
            const int hi = j > c ? j : c, lo = j > c ? c : j;
            const double re = src[itri(hi) + lo];
            double im = (hi != lo) ? src[ntri + itrs(hi) + lo] : 0.0;
            if (c > j) im = -im;  // stored entry is (hi, lo); the upper triangle is its conjugate
            M[idx] = make_double2(re, im);
            QT[idx] = make_double2(j == c ? 1.0 : 0.0, 0.0);
        }
    }
    __syncthreads();

    // ---- 1. Householder reduction, Q accumulated ----
    for (int i = 0; i < N - 1; ++i) {
        // pivot column x_r = A[r][i] = conj(A[i][r]), r > i (row i is contiguous)
        double2 part = make_double2(0.0, 0.0);
        for (int c = i + 2 + tid; c < N; c += T) {
            const double2 z = M[i * N + c];
            part.x = fma(z.x, z.x, fma(z.y, z.y, part.x));
        }
        const double xn = block_sum2<T>(part, red).x;
        const double2 a0 = M[i * N + i + 1];
        double beta, tr, ti, sr, si;
        householder_gen(a0.x, -a0.y, xn, beta, tr, ti, sr, si);
        if (tid == 0) {
            d[i] = M[i * N + i].x;
            e[i] = beta;
        }
        if (tr == 0.0 && ti == 0.0) continue;  // uniform: every thread computed the same numbers
        for (int c = tid; c < N; c += T) {
            double2 v = make_double2(0.0, 0.0);
            if (c == i + 1) v.x = 1.0;
            else if (c > i + 1) {
                const double2 z = M[i * N + c];  // x_c = conj(z)
                v.x = z.x * sr + z.y * si;
                v.y = z.x * si - z.y * sr;
            }
            V[c] = v;
        }
        __syncthreads();
        // p = tau A v, p_c = tau sum_j conj(A[j][c]) v_j ;  dot = p^H v
        double2 dot = make_double2(0.0, 0.0);
        for (int c = i + 1 + tid; c < N; c += T) {
            double s0r = 0.0, s0i = 0.0, s1r = 0.0, s1i = 0.0;
            int j = i + 1;
            for (; j + 1 < N; j += 2) {
                const double2 a = M[j * N + c], v = V[j];
                const double2 b = M[(j + 1) * N + c], u = V[j + 1];
                s0r = fma(a.x, v.x, fma(a.y, v.y, s0r));
                s0i = fma(a.x, v.y, fma(-a.y, v.x, s0i));
                s1r = fma(b.x, u.x, fma(b.y, u.y, s1r));
                s1i = fma(b.x, u.y, fma(-b.y, u.x, s1i));
            }
            if (j < N) {
                const double2 a = M[j * N + c], v = V[j];
                s0r = fma(a.x, v.x, fma(a.y, v.y, s0r));
                s0i = fma(a.x, v.y, fma(-a.y, v.x, s0i));
            }
            const double sumr = s0r + s1r, sumi = s0i + s1i;
            const double pr = tr * sumr - ti * sumi, pi = tr * sumi + ti * sumr;
            W[c] = make_double2(pr, pi);
            const double2 v = V[c];
            dot.x += pr * v.x + pi * v.y;
            dot.y += pr * v.y - pi * v.x;
        }
        dot = block_sum2<T>(dot, red);
        const double alr = -0.5 * (tr * dot.x - ti * dot.y), ali = -0.5 * (tr * dot.y + ti * dot.x);
        for (int c = i + 1 + tid; c < N; c += T) {  // each thread finishes the entries it wrote itself
            const double2 v = V[c];
            double2 w = W[c];
            w.x += alr * v.x - ali * v.y;
            w.y += alr * v.y + ali * v.x;
            W[c] = w;
        }
        __syncthreads();
        // A -= v w^H + w v^H on the trailing block (both triangles), thread c owns column c
        for (int c = i + 1 + tid; c < N; c += T) {
            const double2 vc = V[c], wc = W[c];
            for (int j = i + 1; j < N; ++j) {
                const double2 vj = V[j], wj = W[j];
                double2 a = M[j * N + c];
                a.x -= vj.x * wc.x + vj.y * wc.y + wj.x * vc.x + wj.y * vc.y;
                a.y -= vj.y * wc.x - vj.x * wc.y + wj.y * vc.x - wj.x * vc.y;
                M[j * N + c] = a;
            }
        }
        // Q <- Q (I - tau v v^H): row r of Q (column r of QT): u = sum_j Q[r][j] v_j, Q[r][j] -= tau u conj(v_j)
        for (int r = tid; r < N; r += T) {
            double ur = 0.0, ui = 0.0;
            for (int j = i + 1; j < N; ++j) {
                const double2 q = QT[j * N + r], v = V[j];
                ur = fma(q.x, v.x, fma(-q.y, v.y, ur));
                ui = fma(q.x, v.y, fma(q.y, v.x, ui));
            }
            const double tur = tr * ur - ti * ui, tui = tr * ui + ti * ur;
            for (int j = i + 1; j < N; ++j) {
                const double2 v = V[j];
                double2 q = QT[j * N + r];
                q.x -= tur * v.x + tui * v.y;
                q.y -= tui * v.x - tur * v.y;
                QT[j * N + r] = q;
            }
        }
        __syncthreads();
    }
    if (tid == 0) {
        d[N - 1] = M[(N - 1) * N + N - 1].x;
        e[N - 1] = 0.0;
    }
    __syncthreads();

    // ---- 2. implicit QL on (d, e); rotations of a sweep recorded by thread 0, applied to the rows of Q by all ----
    for (int l = 0; l < N; ++l) {
        int iter = 0;
        while (true) {
            if (tid == 0) {
                int m;
                for (m = l; m < N - 1; ++m) {
                    const double dd = fabs(d[m]) + fabs(d[m + 1]);
                    if (fabs(e[m]) <= DBL_EPSILON * dd) break;
                }
                if (m == l) ctl[0] = 1;
                else if (iter == 64) ctl[0] = 2;
                else {
                    const double el = e[l];
                    double g = (d[l + 1] - d[l]) / (2.0 * el);
                    double r = sqrt(g * g + 1.0);
                    g = d[m] - d[l] + el / (g + (g >= 0.0 ? r : -r));
                    double s = 1.0, c = 1.0, p = 0.0;
                    int i;
                    bool underflow = false;
                    for (i = m - 1; i >= l; --i) {
                        const double ei = e[i];
                        const double f = s * ei;
                        const double b = c * ei;
                        const double h = f * f + g * g;
                        if (h == 0.0) {
                            e[i + 1] = 0.0;
                            d[i + 1] -= p;
                            e[m] = 0.0;
                            underflow = true;
                            break;
                        }
                        const double rinv = rsqrt(h);
                        r = h * rinv;
                        e[i + 1] = r;
                        s = f * rinv;
                        c = g * rinv;
                        g = d[i + 1] - p;
                        r = (d[i] - g) * s + 2.0 * c * b;
                        p = s * r;
                        d[i + 1] = g + p;
                        g = c * r - b;
                        CS[i] = make_double2(c, s);
                    }
                    if (!underflow) {
                        d[l] -= p;
                        e[l] = g;
                        e[m] = 0.0;
                    }
                    ctl[0] = 0;
                    ctl[1] = m;
                    ctl[2] = underflow ? i + 1 : l;
                }
            }
            __syncthreads();
            const int st = ctl[0], m = ctl[1], lo = ctl[2];
            if (st != 0) {
                if (st == 2 && tid == 0 && fail_count) atomicAdd(fail_count, 1);
                __syncthreads();  // everybody has read ctl before thread 0 overwrites it for the next l
                break;
            }
            for (int r = tid; r < N; r += T) {
                double2 hi = QT[m * N + r];
                for (int i = m - 1; i >= lo; --i) {
                    const double2 cs = CS[i];
                    const double2 g = QT[i * N + r];
                    // z[.][i+1] = s z[.][i] + c z[.][i+1];  z[.][i] = c z[.][i] - s z[.][i+1]
                    QT[(i + 1) * N + r] = make_double2(cs.y * g.x + cs.x * hi.x, cs.y * g.y + cs.x * hi.y);
                    hi = make_double2(cs.x * g.x - cs.y * hi.x, cs.x * g.y - cs.y * hi.y);
                }
                QT[lo * N + r] = hi;
            }
            __syncthreads();
            ++iter;
        }
    }

    // ---- 3. ascending order (stable rank), eigenvector columns permuted alongside ----
    // NaNs rank last: with plain comparisons a NaN (from a non-finite matrix) would share a rank, leave a slot of perm
    // unwritten and send the gather below outside QT
    int* perm = reinterpret_cast<int*>(CS);
    for (int t = tid; t < N; t += T) {
        const double x = d[t];
        const bool xnan = isnan(x);
        int rank = 0;
        for (int q = 0; q < N; ++q) {
            const double y = d[q];
            rank += (xnan ? (!isnan(y) || q < t) : (y < x || (y == x && q < t))) ? 1 : 0;
        }
        perm[rank] = t;
        eig_out[kk * N + rank] = x;
    }
    __syncthreads();
    double2* out = reinterpret_cast<double2*>(vec_out) + (size_t)kk * NN;
    for (int idx = tid; idx < NN; idx += T) {
        const int r = idx / N, j = idx - r * N;
        out[idx] = QT[perm[j] * N + r];  // v[r][j] = Q[r][perm[j]]
    }
}

size_t eigh_fixed_smem(int n, int t) { return (size_t)3 * n * 16 + (size_t)(t / 32) * 16 + (size_t)2 * n * 8 + 32; }

template <int T>
cudaError_t launch_eigh_t(int n, const double* Hp, long nk, double* eig, double* vec, double2* gA, double2* gQ,
                          int* fail_count, cudaStream_t st) {
    const size_t smem = eigh_fixed_smem(n, T) + (gA ? 0 : (size_t)2 * n * n * 16);
    cudaError_t err = cudaFuncSetAttribute(eigh_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return err;
    if (nk > 2147483647L) return cudaErrorInvalidConfiguration;
    eigh_kernel<T><<<(unsigned)nk, T, smem, st>>>(Hp, n, nk, eig, vec, gA, gQ, fail_count);
    return cudaGetLastError();
}

}  // namespace

// Where the matrix and the accumulated unitary live.  Shared memory (32 N^2 bytes per matrix) caps the CTAs an SM
// holds, and this kernel is latency bound (barriers, one thread's serial QL chain): measured on B200, ms per 1000
// matrices in shared memory / on L2-resident global scratch (as many CTAs resident as threads allow) -- N = 12: 0.035 /
// 0.035, 16: 0.063 / 0.058, 24: 0.197 / 0.139, 36: 0.864 / 0.584, 48: 3.23 / 1.25, 64: 10.9 / 3.34, 82: 17.8 / 9.07
// (gpurun_out/r03y_eigh.log, r03z_eigh.log).  So only the smallest matrices stay in shared memory.
// TBK_EIGH_SMEM_MAX overrides (tests, A/B runs).
bool eigh_in_smem(int n) {
    static const int limit = [] {
        const char* e = getenv("TBK_EIGH_SMEM_MAX");
        return e ? atoi(e) : 12;
    }();
    return n <= limit && eigh_fixed_smem(n, 128) + (size_t)2 * n * n * 16 <= 220 * 1024;
}

// Hp: packed Hermitian [nk][n*n] (not modified).  eig [nk][n] ascending, vec [nk][n][n] c128 (column j <-> eig[j]).
// scratch: 2 * nk * n * n double2 of global memory when !eigh_in_smem(n), else unused (may be null).
cudaError_t launch_eigh(int n, const double* Hp, long nk, double* eig, double* vec, double* scratch, int* fail_count,
                        cudaStream_t st) {
    if (nk <= 0 || n <= 0) return cudaSuccess;
    double2 *gA = nullptr, *gQ = nullptr;
    if (!eigh_in_smem(n)) {
        if (!scratch) return cudaErrorInvalidValue;
        gA = reinterpret_cast<double2*>(scratch);
        gQ = gA + (size_t)nk * n * n;
    }
    if (n <= 32) return launch_eigh_t<32>(n, Hp, nk, eig, vec, gA, gQ, fail_count, st);
    if (n <= 64) return launch_eigh_t<64>(n, Hp, nk, eig, vec, gA, gQ, fail_count, st);
    if (n <= 128) return launch_eigh_t<128>(n, Hp, nk, eig, vec, gA, gQ, fail_count, st);
    return launch_eigh_t<256>(n, Hp, nk, eig, vec, gA, gQ, fail_count, st);
}

}  // namespace tbk
