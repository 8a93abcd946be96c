/* tbk.h -- C ABI of libtbk.so, the B200-native evaluator for the TBmodels k-space hot path.
 *
 * The reference (Z2PackDev/TBmodels v1.4.4) is pure Python and has no FFI seam; the boundary this
 * library sits behind is the pair of methods
 *     Model.hamilton(self, k, convention=2)      reference src/tbmodels/_tb_model.py:1076-1132
 *     Model.eigenval(self, k)                    reference src/tbmodels/_tb_model.py:1134-1150
 * plus the state they read: Model.hop (:206-218, half-set semantics from _reduce_hop :247-279),
 * Model.pos (:186-191), Model.size, Model.dim.  INTEGRATION.md shows the ctypes binding a maintainer
 * adds on the reference side.
 *
 * Conventions
 *   - every function returns an int status: 0 = OK, non-zero = error (TBK_E_*); the message for the last
 *     error on the calling thread is tbk_last_error().  No C++ exceptions cross the boundary.
 *   - plain pointers and sizes only; complex128 arrays are interleaved (re, im) doubles, row-major.
 *   - a handle is immutable after creation (re-create it when the model's hoppings change) and owns its
 *     device scratch; use one handle per GPU and one in-flight call per handle.
 *   - "_host" entry points take HOST pointers and run a chunked H2D -> kernels -> D2H pipeline on private
 *     streams (pinned buffers from tbk_host_alloc overlap fully; pageable memory works, slower); the plain
 *     entry points take DEVICE pointers, enqueue on the caller's stream and return without synchronising.
 *   - there is no CPU fallback: without a usable CUDA device every compute entry point fails.
 */
#ifndef TBK_H
#define TBK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TBK_OK 0
#define TBK_E_INVALID 1     /* bad argument (null pointer, size, convention, dimension) */
#define TBK_E_CUDA 2        /* CUDA runtime / launch failure */
#define TBK_E_UNSUPPORTED 3 /* model outside the supported envelope (dim > 8) */
#define TBK_E_NOCONV 4      /* QL iteration did not converge for some matrix */

typedef struct tbk_model tbk_model;

/* Library version (major * 100 + minor). */
int tbk_version(void);
/* Message describing the last error on this thread ("" if none). */
const char* tbk_last_error(void);

/* Pack a model onto GPU `device`.
 *   R    [n_R][dim]            int32   keys of Model.hop, in dict order            (_tb_model.py:1111)
 *   hop  [n_R][n_orb][n_orb]   c128    dense values of Model.hop; the R = 0 entry holds HALF the on-site
 *                                      block, exactly as the reference stores it     (:218, :268)
 *   pos  [n_orb][dim]          f64     Model.pos (reduced coordinates)              (:186-191)
 * All three are HOST pointers, copied during the call.  n_R may be 0 (H == 0).
 * Any finite magnitude is accepted: a model whose bound on |H(k)_ij|, max_ij sum_R (|T_R,ij| + |T_R,ji|) with
 * |z| = |Re z| + |Im z|, lies outside [2^-384, 2^384] is stored scaled by an even power of two and every result is scaled back (exact while results are normal); the
 * same holds for tbk_kdotp_create (the coefficients) and tbk_supercell_create (the base model). */
int tbk_model_create(int dim, int n_orb, int n_R, const int32_t* R, const double* hop, const double* pos,
                     int device, tbk_model** out);
/* Pack a k.p model (tbmodels.kdotp.KdotpModel, reference src/tbmodels/kdotp.py:19-49): H(k) = sum_q prod_d k_d^{p_qd} C_q.
 *   powers [n_terms][dim]            int32  keys of KdotpModel.taylor_coefficients
 *   coeff  [n_terms][n_orb][n_orb]   c128   the Hermitian coefficient matrices
 * The handle is used with tbk_hamilton[_host] (convention must be 2: a k.p model has none, kdotp.py:51-82) and
 * tbk_eigenval[_host] (kdotp.py:84-100). */
int tbk_kdotp_create(int dim, int n_orb, int n_terms, const int32_t* powers, const double* coeff, int device,
                     tbk_model** out);
/* Model.supercell (reference src/tbmodels/_tb_model.py:1645-1724) + packing, for a BASE model given like tbk_model_create
 * and size[dim] >= 1 cells per direction (SURVEY.md section 8 row f3).  The n_R' dense N' x N' matrices the reference
 * builds (N' = n_orb * prod(size)) are never materialised: the host enumerates the block list, a kernel gathers the
 * weights straight into the GEMM's tiles, and the all-zero (column tile, K-chunk) stages of the block-sparse result
 * are skipped by the H(k) GEMM.  The handle behaves like one from tbk_model_create on the supercell model (lattice
 * vectors folded onto the half set as Model(..., contains_cc=False) does, positions divided by size, :1670-1678).
 * tbk_model_info reports N' and n_R'; tbk_model_vectors copies the stored lattice vectors [n_R][dim] to the host. */
int tbk_supercell_create(int dim, int n_orb, int n_R, const int32_t* R, const double* hop, const double* pos,
                         const int32_t* size, int device, tbk_model** out);
int tbk_model_vectors(const tbk_model* m, int32_t* R_out);
int tbk_model_destroy(tbk_model* m);
/* path: 0 = fused thread-per-k kernel (N <= 8), 1 = DMMA GEMM + batched tridiagonal/QL eigensolver,
 *       2 = fused trigonometric-product kernel (N <= 2, dim <= 3, nearest-cell lattice vectors). */
int tbk_model_info(const tbk_model* m, int* n_orb, int* dim, int* n_R, int* path);

/* Model.hamilton for a batch (replaces _tb_model.py:1109-1128).
 *   k_dev   [n_k][dim]            f64   device
 *   out_dev [n_k][n_orb][n_orb]   c128  device
 *   convention  1 or 2 (anything else -> TBK_E_INVALID; the Python layer raises ValueError first, :1097-1102) */
int tbk_hamilton(tbk_model* m, const double* k_dev, int64_t n_k, int convention, double* out_dev, void* stream);
/* Model.eigenval for a batch (replaces _tb_model.py:1147-1149): convention-2 H(k), eigenvalues ascending.
 *   out_dev [n_k][n_orb] f64 device */
int tbk_eigenval(tbk_model* m, const double* k_dev, int64_t n_k, double* out_dev, void* stream);

/* Multi-GPU form of tbk_eigenval (SURVEY.md section 8 e1: the all-gather fused behind the eigensolver).  out_dev is this
 * rank's slice -- starting at row `row_offset` -- of a result buffer that exists on every GPU; peer_bases[p] are the
 * base addresses of the OTHER ranks' buffers, peer-mapped into this process (e.g. the buffer_ptrs of a
 * torch.distributed._symmetric_memory rendezvous, or cudaIpc / cuMem handles).  After every workspace chunk its rows are
 * stored into all peers at the same row offset by a copy kernel on a side stream (16-byte stores over NVLink /
 * NVSwitch), overlapping the next chunk's kernels; `stream` continues once the last store has completed.  The CALLER
 * synchronises the ranks afterwards (a device-side barrier of the symmetric-memory handle, or any collective) before
 * any rank reads rows it did not compute.  n_peers = 0 degenerates to tbk_eigenval. */
int tbk_eigenval_push(tbk_model* m, const double* k_dev, int64_t n_k, double* out_dev, void* const* peer_bases, int n_peers,
                      int64_t row_offset, void* stream);

/* Model.eigenval on a regular k-mesh without an explicit k array (SURVEY.md section 8 row f4): the mesh has dims[d]
 * points in dimension d, k_d = (i_d + shift_d) / dims[d] (shift may be NULL), ordered like
 * numpy.meshgrid(..., indexing="ij") flattened in C order -- the layout of the reference's k-grid workloads.  A LINE
 * is the run of dims[dim-1] consecutive mesh points along the last dimension; the call evaluates lines
 * [first_line, first_line + n_lines) (for sharding across GPUs) and writes
 *   out_dev [n_lines * dims[dim-1]][n_orb] f64 device, ascending per k-point.
 * Same results as tbk_eigenval on the explicit k-points within the parity bounds (the Fourier sum is factorised over
 * the last dimension where the model allows it, otherwise the k-points are generated on the device and the ordinary
 * path runs).  tbk_mesh_factorised reports which of the two will be used (1 / 0). */
int tbk_eigenval_mesh(tbk_model* m, const int64_t* dims, const double* shift, int64_t first_line, int64_t n_lines,
                      double* out_dev, void* stream);
int tbk_mesh_factorised(const tbk_model* m, const int64_t* dims);
/* Same with a HOST result buffer (pinned memory from tbk_host_alloc overlaps fully): groups of lines are evaluated into
 * two device buffers whose D2H copies overlap the next group's kernels; synchronous on return. */
int tbk_eigenval_mesh_host(tbk_model* m, const int64_t* dims, const double* shift, int64_t first_line, int64_t n_lines,
                           double* out_host);

/* Eigenvalues AND eigenvectors of the convention-2 H(k) (SURVEY.md section 8 row f4; what scipy.linalg.eigh returns where
 * Model.eigenval calls scipy.linalg.eigvalsh, _tb_model.py:1149): Householder reduction with the unitary accumulated,
 * implicit QL with the rotations applied to it, ascending order.
 *   eig_dev [n_k][n_orb]          f64   device, ascending
 *   vec_dev [n_k][n_orb][n_orb]   c128  device, vec[k][i][j] = component i of the eigenvector of eig[k][j] (numpy layout);
 *                                       unit norm, phase arbitrary */
int tbk_eigh(tbk_model* m, const double* k_dev, int64_t n_k, double* eig_dev, double* vec_dev, void* stream);
int tbk_eigh_host(tbk_model* m, const double* k_host, int64_t n_k, double* eig_host, double* vec_host);

/* Band velocities vel[k][n][d] = dE_n/dk_d of the ascending eigenvalues eig[k][n] of the convention-2 H(k) (eigenvalues
 * do not depend on the convention, so neither do their derivatives).  k is in reduced coordinates, as for tbk_hamilton;
 * the velocities are in energy units per unit of reduced k (Cartesian: v_cart = v @ uc / (2 pi), uc the lattice vectors
 * as rows).
 *   - a band whose eigenvalue is separated from its neighbours: the Hellmann-Feynman value Re(v_n^H dH/dk_d v_n);
 *   - a degenerate cluster, a maximal run of ascending eigenvalues whose consecutive gaps are <= degen_tol * rho with
 *     rho = max_n |eig_n|, is treated as one level: for every direction d separately the velocities of its m members are
 *     the eigenvalues, ascending, of the m x m Hermitian block V_c^H dH/dk_d V_c (degenerate perturbation theory, the
 *     only choice that does not depend on the basis eigh picks inside the subspace).  So inside a cluster the value at
 *     index n in direction 0 and the one at index n in direction 1 need not belong to the same state.  eig is returned
 *     as tbk_eigh computes it (bit for bit), not averaged over clusters.
 *   - degen_tol >= 0 (a negative or NaN value -> TBK_E_INVALID); 1e-8 is a good default: an eigenvector with gap g is
 *     accurate to about eps rho / g, so a pair left unmerged has a velocity error of at most about eps / degen_tol
 *     ||dH/dk_d||, 2e-8 ||dH/dk_d|| at 1e-8.
 * dH/dk_d are the order-1 terms of tbk_kdotp_coefficients.  Handles from tbk_model_create and tbk_supercell_create;
 * handles from tbk_kdotp_create -> TBK_E_INVALID.
 *   eig_dev [n_k][n_orb]        f64  device
 *   vel_dev [n_k][n_orb][dim]   f64  device */
int tbk_band_velocity(tbk_model* m, const double* k_dev, int64_t n_k, double degen_tol, double* eig_dev, double* vel_dev,
                      void* stream);
/* Same with HOST buffers (copies inside, synchronous on return). */
int tbk_band_velocity_host(tbk_model* m, const double* k_host, int64_t n_k, double degen_tol, double* eig_host,
                           double* vel_host);

/* Berry curvature curv[k][n][p] of every band at the reduced k-points k (units of (reduced k)^-2), for every pair a < b of
 * directions in the order p = (0,1), (0,2), ..., (0,dim-1), (1,2), ... (dim (dim - 1) / 2 pairs; dim = 3: 01, 02, 12).
 * With V the eigenvectors of tbk_eigh, E = eig and M_a = V^H X_a V, X_a the k_a-derivative of H(k) in the convention:
 *   - a band separated from its neighbours: Omega_n^ab = -2 Im sum_{l != n} M_a[n][l] M_b[l][n] / ((E_n - E_l)(E_n - E_l)),
 *     the curl of the Berry connection A = i <u|grad u>;
 *   - a degenerate cluster c (as for tbk_band_velocity: a maximal run of ascending eigenvalues whose gaps are
 *     <= degen_tol * rho, rho = max_n |eig_n|): its m members get, per pair separately, the ascending eigenvalues of the
 *     m x m Hermitian non-Abelian curvature F_nm = i sum_{l not in c} (M_a[n][l] M_b[l][m] - M_b[n][l] M_a[l][m]) /
 *     ((E_n - E_l)(E_m - E_l)), n, m in c.  Its trace is the sum of the members' Abelian curvatures, and its eigenvalues do
 *     not depend on the basis eigh picks inside the cluster.
 *   - convention: the local curvature depends on it (Chern numbers do not).  2: X_a = dH/dk_a, the order-1 terms of
 *     tbk_kdotp_coefficients, as for tbk_band_velocity.  1: X_a = dH/dk_a + 2 pi i [H, T_a], T_a = diag(pos[:, a]), i.e.
 *     X_a[i][j] = dH/dk_a[i][j] + 2 pi i (pos[j][a] - pos[i][a]) H[i][j] with the convention-2 H (H_1 = D H_2 D^H,
 *     D = diag(e^{-2 pi i k.pos_i})).
 *   - sum over a 2-d mesh of n_k points of curv[.][n][p] / n_k, divided by 2 pi, tends to the Chern number of band n in
 *     plane p.  Cartesian tensor: uc^T Omega_red uc / (4 pi^2), Omega_red the full antisymmetric dim x dim matrix and uc
 *     the lattice vectors as rows.
 *   - Omega does not change under H -> 2^e H: a model stored scaled (tbk_model_create) gives the unscaled model's curvature
 *     bit for bit; eig is returned as tbk_eigh computes it (bit for bit).  N = 1 and H = 0 give zeros.
 * TBK_E_INVALID: convention other than 1 or 2, degen_tol negative or NaN, dim < 2, a handle from tbk_kdotp_create, null
 * buffers with n_k > 0.
 *   eig_dev  [n_k][n_orb]                     f64  device
 *   curv_dev [n_k][n_orb][dim (dim - 1) / 2]  f64  device */
int tbk_berry_curvature(tbk_model* m, const double* k_dev, int64_t n_k, int convention, double degen_tol, double* eig_dev,
                        double* curv_dev, void* stream);
/* Same with HOST buffers (copies inside, synchronous on return). */
int tbk_berry_curvature_host(tbk_model* m, const double* k_host, int64_t n_k, int convention, double degen_tol,
                             double* eig_host, double* curv_host);

/* Model.construct_kdotp (reference src/tbmodels/_tb_model.py:942-982), batched over expansion points: the Taylor
 * coefficients C_p = (2 pi i)^|p| / p! * sum_R [R^p e^{2 pi i k.R} T_R + (-R)^p e^{-2 pi i k.R} T_R^H] of H around k
 * (convention 2), the same Fourier sum as tbk_hamilton with R^p weights (SURVEY.md section 8 row f2).
 *   k_dev   [n_k][dim]                       f64    device: expansion points
 *   powers  [n_terms][dim]                   int32  HOST: the power tuples p (keys of KdotpModel.taylor_coefficients),
 *                                                   each component in [0, 64]
 *   out_dev [n_k][n_terms][n_orb][n_orb]     c128   device: exactly Hermitian matrices
 * Not defined for handles made by tbk_kdotp_create (TBK_E_INVALID). */
int tbk_kdotp_coefficients(tbk_model* m, const double* k_dev, int64_t n_k, const int32_t* powers, int n_terms,
                           double* out_dev, void* stream);
/* Same with HOST buffers for k and out (synchronous on return). */
int tbk_kdotp_coefficients_host(tbk_model* m, const double* k_host, int64_t n_k, const int32_t* powers, int n_terms,
                                double* out_host);

/* Same two operations with HOST buffers (copies inside, synchronous on return). */
int tbk_hamilton_host(tbk_model* m, const double* k_host, int64_t n_k, int convention, double* out_host);
int tbk_eigenval_host(tbk_model* m, const double* k_host, int64_t n_k, double* out_host);

/* Synchronise the handle's device and report deferred errors (QL non-convergence) of the device-pointer calls. */
int tbk_model_check(tbk_model* m);
/* Number of kernels launched through this handle so far. */
int64_t tbk_launch_count(const tbk_model* m);
/* Per-kernel-class device timing with CUDA events recorded on the launching stream.
 * Classes: 0 H(k) DMMA GEMM, 1 fused small-N kernel, 2 expand (and the k.p coefficient kernel, which also builds the
 * dH/dk_d of tbk_band_velocity and tbk_berry_curvature), 3 tridiagonalisation, 4 tridiagonal QL, 5 phase tiles for the
 * GEMM (and the small mesh helper kernels), 6 line expansion of the regular-mesh path, 7 eigen-decomposition with
 * eigenvectors (and the band velocity kernel of tbk_band_velocity, the product and curvature kernels of
 * tbk_berry_curvature), 8 peer stores of tbk_eigenval_push, 9 rescaling of the results of a
 * model stored scaled by a power of two (see tbk_model_create).
 * tbk_profile(m, 1) starts recording; tbk_profile_read synchronises, returns the accumulated milliseconds
 * and launch counts per class since the last read (arrays of TBK_PROFILE_CLASSES) and resets them. */
#define TBK_PROFILE_CLASSES 10
int tbk_profile(tbk_model* m, int enable);
int tbk_profile_read(tbk_model* m, double* ms, int64_t* count);
/* Bytes of device scratch currently held by the handle. */
int64_t tbk_workspace_bytes(const tbk_model* m);

/* Page-locked host memory for the _host entry points. */
int tbk_host_alloc(void** p, size_t bytes);
int tbk_host_free(void* p);

/* Measured FP64 peaks of the current device, TFLOP/s (kind 0: DMMA mma.sync.m8n8k4.f64, 1: DFMA). < 0 on error. */
double tbk_measure_fp64_peak(int kind, int iters);
/* Measured INT8 tensor-core peak of the current device, TOP/s (tcgen05.mma kind::i8, M 128 N 256 K 32, int32
 * accumulators in tensor memory; `iters` MMAs per SM). < 0 on error. */
double tbk_measure_int8_peak(int64_t iters);

/* ---- host-side debug entry points: run the exact scalar code of the kernels on the CPU (tests only) ---- */
/* In-place eigenvalues of a real symmetric tridiagonal matrix; d[n], e[n] (e[n-1] scratch). Returns #failures. */
int tbk_host_tridiag_ql(int n, double* d, double* e);
/* sin(pi t), cos(pi t) as the fused small-N kernel computes them (tbk_math.cuh sincospi_lean). */
int tbk_host_sincospi(double t, double* s, double* c);
/* Same result by bisection with Sturm counts (the large-N device path); e is not modified. */
int tbk_host_tridiag_bisect(int n, double* d, const double* e);
/* Packed Hermitian (n*n doubles, destroyed) -> d[n], e[n]. */
int tbk_host_hetrd(int n, double* hp, double* d, double* e);
/* Hermitian-split weights W[2*n_R][n_orb*n_orb] the kernels consume, from hop[n_R][n_orb][n_orb] c128. */
int tbk_host_pack_weights(int n_orb, int n_R, const double* hop, double* W);

#ifdef __cplusplus
}
#endif
#endif /* TBK_H */
