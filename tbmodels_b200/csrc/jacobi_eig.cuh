// jacobi_eig.cuh -- eigenvalues of small Hermitian blocks by cyclic complex Jacobi, one thread per block.  Used for the
// projected blocks of degenerate clusters (band_velocity.cu, berry_curvature.cu); serial, so speed matters only for small m.
#pragma once
#include <cfloat>

namespace tbk {

namespace {

constexpr int kJacobiSweeps = 60;

// Ascending eigenvalues of the Hermitian m x m matrix A (row-major, full, destroyed) into A's diagonal, sorted.
__device__ void jacobi_eigvals(double2* A, int m) {
    double fro2 = 0.0;
    for (int i = 0; i < m * m; ++i) fro2 = fma(A[i].x, A[i].x, fma(A[i].y, A[i].y, fro2));
    const double stop = DBL_EPSILON * DBL_EPSILON * fro2;
    for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
        double off = 0.0;
        for (int p = 0; p < m; ++p)
            for (int q = p + 1; q < m; ++q) off = fma(A[p * m + q].x, A[p * m + q].x, fma(A[p * m + q].y, A[p * m + q].y, off));
        if (!(off > stop)) break;  // also ends on NaN input
        for (int p = 0; p < m; ++p)
            for (int q = p + 1; q < m; ++q) {
                const double2 b = A[p * m + q];
                const double ab = sqrt(b.x * b.x + b.y * b.y);
                if (ab == 0.0) continue;
                // A <- U^H A U, U = diag(1, conj(e)) in the (p, q) plane (makes A_pq = |b| real) times a real rotation
                const double er = b.x / ab, ei = b.y / ab;  // e = b / |b|
                const double app = A[p * m + p].x, aqq = A[q * m + q].x;
                const double theta = (aqq - app) / (2.0 * ab);
                const double at = fabs(theta);
                double t = at > 1e150 ? 0.5 / at : 1.0 / (at + sqrt(fma(at, at, 1.0)));
                if (theta < 0.0) t = -t;
                const double c = 1.0 / sqrt(fma(t, t, 1.0)), s = t * c;
                for (int r = 0; r < m; ++r) {
                    if (r == p || r == q) continue;
                    const double2 xp = A[r * m + p];
                    const double2 x = A[r * m + q];
                    const double2 xq = make_double2(x.x * er + x.y * ei, x.y * er - x.x * ei);  // A_rq conj(e)
                    const double2 np_ = make_double2(c * xp.x - s * xq.x, c * xp.y - s * xq.y);
                    const double2 nq = make_double2(s * xp.x + c * xq.x, s * xp.y + c * xq.y);
                    A[r * m + p] = np_;
                    A[r * m + q] = nq;
                    A[p * m + r] = make_double2(np_.x, -np_.y);
                    A[q * m + r] = make_double2(nq.x, -nq.y);
                }
                A[p * m + p] = make_double2(app - t * ab, 0.0);
                A[q * m + q] = make_double2(aqq + t * ab, 0.0);
                A[p * m + q] = make_double2(0.0, 0.0);
                A[q * m + p] = make_double2(0.0, 0.0);
            }
    }
    // insertion sort of the diagonal (bounded indices whatever the values, NaN included)
    for (int i = 1; i < m; ++i) {
        const double x = A[i * m + i].x;
        int j = i - 1;
        while (j >= 0 && A[j * m + j].x > x) {
            A[(j + 1) * m + j + 1].x = A[j * m + j].x;
            --j;
        }
        A[(j + 1) * m + j + 1].x = x;
    }
}

}  // namespace

}  // namespace tbk
