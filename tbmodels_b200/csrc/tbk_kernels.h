// tbk_kernels.h -- internal launcher interface between the C-ABI layer (tbk_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tbk {

constexpr int kMaxDim = 8;        // largest lattice dimension supported on the device
constexpr int kSmallMaxN = 8;     // thread-per-k fused kernel handles N <= 8 (if its tables fit in smem)
constexpr int kGemmBM = 128;      // k-points per CTA tile of the H(k) GEMM
constexpr int kGemmKC = 16;       // K (= 2 * R-vectors) per pipeline stage
constexpr int kGemmStages = 5;
constexpr int kI8BM = 128;       // INT8 digit GEMM (hk_gemm_i8.cu): packed columns per tile
constexpr int kI8BK = 48;        //   k-points per tile
constexpr int kI8MaxKSteps = 2047;  //   32-row K steps whose int32 class sums cannot overflow
constexpr int kI8MinKSteps = 6;  //   default from this many K steps (>= 81 stored R): below, the per-tile epilogue costs more
                                 //   than the MMAs save (C4, 1 step: 19.9 vs 11.8 ms per 12 500 k; C3, 16 steps: 443 vs 673 ms)
constexpr int kTridiagRegMaxN = 48;  // register-resident warp-per-matrix tridiagonalisation (eig_tridiag_reg.cu)

// Tuning / test hooks, read from the environment ONCE per handle at tbk_model_create (never on the launch path).
// Defaults are the measured best; none of them depends on the batch.
struct Tuning {
    long workspace_mb = 2048;   // TBK_WORKSPACE_MB: scratch budget that sizes the k-point chunk of the GEMM path
    long host_chunk_mb = 64;    // TBK_HOST_CHUNK_MB: chunk of the H2D | kernels | D2H pipeline of the _host entry points
    int no_mesh_factor = 0;     // TBK_NO_MESH_FACTOR: tbk_eigenval_mesh generates explicit k-points instead
    int basis_kp = 0;           // TBK_BASIS_KP: k-points per thread of the trigonometric-product kernel (0 = default)
    int tridiag_g = 0;          // TBK_TRIDIAG_G: shared-memory kernel: threads per matrix (1 = tensor-core variant)
    int tridiag_cs = 1;         // TBK_TRIDIAG_CS: column slices
    int tridiag_g1 = 0;         // TBK_TRIDIAG_G1 / _CS1: threads / column slices of the staged kernel while N > 112 (0 = default)
    int tridiag_cs1 = 0;
    int tridiag_mpb = 0;        // TBK_TRIDIAG_MPB: matrices per CTA (0 = maximise residency)
    int tridiag_stages = -1;    // TBK_TRIDIAG_STAGES: staged reduction, size ratio between launches in percent (0 = off,
                                //   -1 = by size: stages end where one more matrix fits an SM for blocks > 88, else ratio 67
                                //   -- gpurun_out/r02s_sweep.log, r03f_sweep.log)
    int tridiag_panel_min = 0;  // TBK_TRIDIAG_PANEL_MIN: blocked kernel from this N on (0 = default 120)
    int tridiag_panel_stop = -1;   // TBK_TRIDIAG_PANEL_STOP: the blocked kernel hands its trailing block to the staged
                                   //   shared-memory / register kernels once at most this many rows are left (0 = never,
                                   //   -1 = by size: 112 for N <= 256, 160 above)
    int tridiag_nopanel = 0;    // TBK_TRIDIAG_NOPANEL
    int tridiag_oldbig = 0;     // TBK_TRIDIAG_OLDBIG
    int tridiag_reg_min = 21;   // TBK_TRIDIAG_REG_MIN / _MAX: sizes served by the register-resident kernel
    int tridiag_reg_max = 40;   //   (TBK_TRIDIAG_REG_MAX=0 disables it; 41 .. 48 measured equal through the staged path)
    int tridiag_reg_bw = 4;     // TBK_TRIDIAG_REG_BW: build of the register kernel: 4 = default per size, 8 = lookahead + 255
                                //   registers, 1 = plain loop, 2 = lookahead at the default register budget
    int tridiag_reg_stop = 16;  // TBK_TRIDIAG_REG_STOP: staged register reduction, the two-matrices-per-warp kernel takes
                                //   over at this block size (2 .. 16; 0 = single launch)
    int tridiag_reg_mid = 0;    // TBK_TRIDIAG_REG_MID: optional middle stage of the staged register reduction (a smaller
                                //   build from this block size down to _STOP; 0 = none, the measured best)
    int panel_t = 0;            // TBK_PANEL_T: blocked kernel: threads per matrix
    int panel_lpr = 0;          // TBK_PANEL_LPR: lanes per row
    int panel_pfd = 1;          // TBK_PANEL_PFD: L2 prefetch distance in warp trips
    int ql_bisect_min = 0;      // TBK_QL_BISECT_MIN: bisection instead of QL from this N on (0 = default)
    int ql_global_min = 0;      // TBK_QL_GLOBAL_MIN: thread-per-matrix QL in global memory from this N on (0 = never)
    int ql_overlap = 0;         // TBK_QL_OVERLAP=1: run chunk i's QL in the background of chunk i + 1.  Off by default: measured
                                //   on B200 the co-resident QL slows the GEMM / tridiagonalisation by what it saves (C3 explicit
                                //   191.7 vs 189.0 ms per 2^21, k-grid 154.7 vs 128.1 ms; gpurun_out/r02u_*)
    int tridiag_twostage = -1;  // TBK_TRIDIAG_TWOSTAGE: two-stage reduction (band + bulge chasing, eig_band.cu) from this N on
                                //   (0 = never, -1 = default)
    int band_t = 0;             // TBK_BAND_T: threads per matrix of the band reduction (0 = by size)
    int band_stage2 = 1;        // TBK_BAND_STAGE2=0: timing hook, skip the bulge chasing (results are then meaningless)
    int band_chase = 0;         // TBK_BAND_CHASE: 1 = first form of the bulge chasing (four matrices per warp, one sweep
                                //   each), 4 = pipelined form at 16 warps per SM (128 registers, spills)
    int band_wave = 0;          // TBK_BAND_WAVE: matrices per launch of the bulge chasing (0 = one resident wave)
    long band_group_mb = 2048;  // TBK_BAND_GROUP_MB: band arrays collected before one bulge-chasing launch
    int gemm_dense = 0;         // TBK_GEMM_DENSE: never skip all-zero weight stages (block-sparse models; A/B tests)
    int hk_fp64 = -1;           // TBK_HK_FP64: explicit-k H(k) builds on the FP64 DMMA GEMM (1) or the INT8 digit GEMM (0);
                                //   -1 = by K: INT8 from kI8MinKSteps K steps on
};
Tuning read_tuning();

// Device-resident packed model (see DESIGN.md "Data layout in HBM").
struct ModelDev {
    int n = 0;        // orbitals
    int dim = 0;      // lattice dimension
    int nR = 0;       // stored (half-set) R vectors that are non-zero matrices
    int nRpad = 0;    // nR rounded up to a multiple of 8 (padding rows: R = 0, zero weights)
    const double* Rd = nullptr;   // [nRpad][dim]   R vectors as doubles
    const int* Ri = nullptr;      // [nR]  fused path: 1 = all |R_d| <= 1, phase is a product of per-dimension factors
    int use_z = 0;                // fused path: any R uses the product form
    const double* W = nullptr;    // [2*nR][n*n]    Hermitian-split weights, row 2r = hp(T_r + T_r^H), row 2r+1 = hp(i(T_r - T_r^H))
    const double* Wt = nullptr;   // tiled copy of W for the GEMM: [n_tiles][kchunks][kGemmKC][bn + 4]
    const double* pos = nullptr;  // [n][dim]
    int na = 0;        // GEMM: n-atoms (8 columns) per warp -> bn = 16 * na
    int n_tiles = 0;   // GEMM: column tiles
    int kchunks = 0;   // GEMM: nRpad / 8
    // GEMM, block-sparse weights (supercells): per column tile the K-chunks whose stage block of Wt is not all zero;
    // null when every stage is populated (then the dense K loop runs)
    const int* kc_cnt = nullptr;  // [n_tiles]
    const int* kc_idx = nullptr;  // [n_tiles][kchunks], first kc_cnt[t] entries valid (ascending)
    int small_ok = 0;  // fused thread-per-k kernel usable
    // N <= 2, dim <= 3, all |R_d| <= 1: H(k) as a linear combination of the 3^dim products of {1, cos 2 pi k_d,
    // sin 2 pi k_d} (hk_small.cu, hk_basis_kernel); basis[b * n * n + e], b = sum_d t_d 3^d, t_d in {0: 1, 1: cos, 2: sin}
    int basis_ok = 0;
    double basis[27 * 4] = {0};
    // regular k-meshes (hk_mesh.cu): stored R vectors sorted into classes by their last component
    int nclass = 0;               // 0: mesh factorisation not available (fused path, k.p model, dim < 2)
    const int* Rc = nullptr;      // [nRpad] class of every R vector (-1 for the padding rows)
    const double* zc = nullptr;   // [nclass] last component of the class
    // k.p models (reference src/tbmodels/kdotp.py:51-82): kind = 1, the GEMM coefficients are the monomials
    // prod_d k_d^{p_d} instead of [cos | sin] phases; Pw holds the integer powers [kchunks * 16][dim]
    int kind = 0;
    const int* Pw = nullptr;
    // INT8 digit GEMM (hk_gemm_i8.cu), phase handles only: W digits [m_tiles][ksteps][9][128 x 32] and s_j 2^-12
    // [m_tiles * 128]; null when the handle builds H(k) on the DMMA GEMM only
    const int8_t* Wd = nullptr;
    const double* Wsc = nullptr;
    Tuning tune;  // environment hooks, captured when the handle was created
};

// H(k) build on the FP64 tensor cores: Hp[k][0..n*n) (packed Hermitian, see tbk_math.cuh).
// Two launches per chunk: launch_hk_phase fills Qt (hk_gemm_q_doubles(md, nk) doubles of scratch) with the
// [cos | sin] tiles, launch_hk_gemm contracts them with the tiled weights.
cudaError_t launch_hk_phase(const ModelDev& md, const double* k, long nk, double* Qt, cudaStream_t st);
cudaError_t launch_hk_gemm(const ModelDev& md, long nk, const double* Qt, double* Hp, cudaStream_t st);
size_t hk_gemm_q_doubles(const ModelDev& md, long nk);
size_t hk_gemm_smem_bytes(const ModelDev& md);  // dynamic shared memory of one GEMM CTA (one CTA per SM)
// The same H(k) from exact INT8 tensor-core digit products (hk_gemm_i8.cu).  launch_hk_wdigits fills md.Wd / md.Wsc
// (hk_i8_w_bytes(md) and m_tiles * 128 doubles) from md.Wt once per handle; per chunk launch_hk_qdigits writes the phase
// digits (hk_i8_q_bytes(md, nk) bytes of scratch) and launch_hk_gemm_i8 contracts them.
int hk_i8_ksteps(const ModelDev& md);
size_t hk_i8_w_bytes(const ModelDev& md);
size_t hk_i8_q_bytes(const ModelDev& md, long nk);
cudaError_t launch_hk_wdigits(const ModelDev& md, int8_t* Wd, double* Wsc, cudaStream_t st);
cudaError_t launch_hk_qdigits(const ModelDev& md, const double* k, long nk, int8_t* Qd, cudaStream_t st);
cudaError_t launch_hk_gemm_i8(const ModelDev& md, long nk, const int8_t* Qd, double* Hp, cudaStream_t st);
// Fused thread-per-k-point path for N <= 8: writes packed H (if Hp) and/or ascending eigenvalues (if eig).
// fail_count (may be null): incremented by the number of eigenvalues whose QL iteration did not converge.
cudaError_t launch_hk_small(const ModelDev& md, const double* k, long nk, double* Hp, double* eig, int* fail_count,
                            cudaStream_t st);
size_t hk_small_smem_bytes(int n, int dim, int nR, int threads);
// packed H -> full complex128 [nk][n][n]; convention 1 applies the orbital-position phases.
cudaError_t launch_expand(const ModelDev& md, const double* k, const double* Hp, long nk, int convention,
                          double* out, cudaStream_t st);
// p[0 .. n) *= 2^s in place (expand.cu): undoes the power-of-two normalisation of a model on its results.
cudaError_t launch_scale_pow2(double* p, long n, int s, cudaStream_t st);
// Peer push (expand.cu): src[0 .. n_doubles) -> peer_bases[p][dst_offset ..] for every peer (peer-mapped device memory).
cudaError_t launch_push_rows(const double* src, long n_doubles, double* const* peer_bases, int n_peers, long dst_offset,
                             cudaStream_t st);
// Taylor coefficients of Model.construct_kdotp (kdotp_construct.cu): out [nk][n_terms][n][n] c128; powers [n_terms][dim]
// and fac [n_terms] (the real prefactor of every term) are device arrays.
cudaError_t launch_kdotp_coeff(const ModelDev& md, const double* k, long nk, const int* powers, const double* fac,
                               int n_terms, double* out, cudaStream_t st);
// Regular k-mesh path (hk_mesh.cu): lines along the last mesh dimension; see the file header.
cudaError_t launch_mesh_phase(const ModelDev& m, const int64_t* dims, const double* shift, long line0, long n_lines,
                              double* Qt, cudaStream_t st);
cudaError_t launch_mesh_qz(const ModelDev& m, long nz, double shift, double* Qz, cudaStream_t st);
cudaError_t launch_mesh_lines(const ModelDev& m, const double* AB, const double* Qz, long nz, long n_lines, double* Hp,
                              cudaStream_t st);
cudaError_t launch_mesh_kpoints(int dim, const int64_t* dims, const double* shift, long first, long count, double* k,
                                cudaStream_t st);
size_t mesh_lines_smem_bytes(int K2);
// Batched Hermitian -> tridiagonal reduction (Hp is destroyed). D, E: [nk][n].
cudaError_t launch_tridiag(int n, double* Hp, long nk, double* D, double* E, cudaStream_t st, const Tuning& tune);
// Two-stage variant (eig_band.cu): Hermitian -> band (half bandwidth 8) on the tensor cores, band -> tridiagonal by bulge chasing.
bool tridiag_twostage_fits(int n);
bool tridiag_twostage_default(int n, const Tuning& tune);  // the size is served by the two-stage reduction
size_t tridiag_twostage_scratch_bytes(int n, long nk);
// The two stages are launched separately: the band arrays of several workspace chunks are collected (they are 16 / n of a
// matrix) and chased in one launch, which gives the latency-bound second stage enough matrices to fill the GPU.
cudaError_t launch_band_reduce(int n, double* Hp, long nk, double* band_ws, cudaStream_t st, const Tuning& tune);
long band_chase_wave_matrices(const Tuning& tune);  // matrices one resident wave of the second stage holds
cudaError_t launch_band_chase(int n, double* band_ws, long nk, double* D, double* E, cudaStream_t st, const Tuning& tune);
// Register-resident warp-per-matrix variant (eig_tridiag_reg.cu), n <= kTridiagRegMaxN.  The matrix of problem k is the
// packed n x n block at Hp + k * mstride; results go to D / E [k * ldo + off + i] (mstride = 0 -> n * n, ldo = 0 -> n).
bool tridiag_reg_fits(int n);
cudaError_t launch_tridiag_reg(int n, double* Hp, long nk, double* D, double* E, cudaStream_t st, long mstride,
                               int ldo, int off, int bw, int stop, int mid);
// Blocked (panel + tensor-core her2k) variant for matrices that live in L2 / HBM (eig_tridiag_panel.cu).
bool tridiag_panel_fits(int n);
// n_stop > 0: staged -- stop at the first panel boundary with at most n_stop rows left (tridiag_panel_handover(n, n_stop)
// of them), write d / e of the eliminated rows and leave the trailing block packed at the head of each matrix' slot.
cudaError_t launch_tridiag_panel(int n, double* Hp, long nk, double* D, double* E, cudaStream_t st, const Tuning& tune,
                                 int n_stop = 0);
int tridiag_panel_handover(int n, int n_stop);
// Supercell packing on the device (supercell_pack.cu).  One SupEntry per base hopping matrix that lands in a block of a
// folded supercell matrix: base matrix index, Hermitian-transposed or not, scale (1/2 for the R' = 0 symmetrisation).
// table[(q * vol + a) * vol + b] = (first entry, count) of block (a, b) of new lattice vector q.
struct SupEntry {
    int r;
    int herm;
    double scale;
};
cudaError_t launch_supercell_pack(int n_base, int vol, int nq, int bn, int kchunks, const double* base_hop,
                                  const int2* table, const SupEntry* entries, double* Wt, cudaStream_t st);
cudaError_t launch_stage_flags(const double* Wt, long n_stages, int stage_doubles, unsigned char* flags, cudaStream_t st);
// Eigenvalues AND eigenvectors (eig_vectors.cu): Hp packed Hermitian [nk][n*n] (kept), eig [nk][n] ascending, vec
// [nk][n][n] c128 with column j belonging to eig[j]; scratch = 2 nk n^2 complex numbers of global memory when
// !eigh_in_smem(n).
bool eigh_in_smem(int n);
cudaError_t launch_eigh(int n, const double* Hp, long nk, double* eig, double* vec, double* scratch, int* fail_count,
                        cudaStream_t st);
// Band velocities (band_velocity.cu): eig [nk][n] ascending and vec [nk][n][n] c128 as launch_eigh writes them, dH
// [nk][dim][n][n] c128 (dH/dk_d) -> vel [nk][n][dim]; degenerate clusters (gaps <= degen_tol * max|eig|) get the
// eigenvalues of their projected blocks.  scratch: the eigh scratch (2 nk n^2 complex numbers) when !eigh_in_smem(n).
cudaError_t launch_band_velocity(int n, int dim, long nk, const double* eig, const double* vec, const double* dH,
                                 double degen_tol, double* vel, double* scratch, cudaStream_t st);
// Berry curvature (berry_curvature.cu).  launch_berry_product: vec [nk][n][n] c128 as launch_eigh writes them and X
// [nk][terms][n][n] c128, the Taylor terms of launch_kdotp_coeff (dH/dk_a for a < dim, then H(k) when conv1) -> M_a =
// V^H X'_a V over X_a (X'_a = dH/dk_a, plus 2 pi i (pos_j,a - pos_i,a) H_ij when conv1); Y: [nk][dim][n][n] c128 scratch
// (n > kSmallMaxN; nk <= 65535).  launch_berry_curvature: curv [nk][n][dim (dim - 1) / 2] from eig and those M_a; scratch as
// for launch_band_velocity.
cudaError_t launch_berry_product(int n, int dim, long nk, const double* vec, double* X, int terms, bool conv1,
                                 const double* pos, double* Y, cudaStream_t st);
cudaError_t launch_berry_curvature(int n, int dim, long nk, const double* eig, const double* M, int terms,
                                   double degen_tol, double* curv, double* scratch, cudaStream_t st);
// Batched tridiagonal QL: D (in: diagonal, out: ascending eigenvalues), E sub-diagonal (destroyed). fail_count may be null.
cudaError_t launch_ql(int n, double* D, double* E, long nk, int* fail_count, cudaStream_t st, const Tuning& tune);
// Background variant for overlapping chunk i's QL with chunk i + 1's build (eig_ql.cu); cudaErrorNotSupported = not
// applicable at this size, use launch_ql.
cudaError_t launch_ql_background(int n, double* D, double* E, long nk, int* fail_count, unsigned long long* counter,
                                 size_t smem_budget, cudaStream_t st, const Tuning& tune);
// Matrices per full wave of the QL kernel on the current device (chunks are sized in whole waves); 0 if n/a.
long ql_wave_matrices(int n, const Tuning& tune);

// FP64 peak micro-benchmarks (bench.py roofline denominators). Return achieved TFLOP/s, or < 0 on error.
double measure_fp64_peak(int kind /*0 = DMMA, 1 = DFMA*/, int iters);
// INT8 tensor-core (tcgen05 kind::i8) peak, TOP/s; iters MMAs of 128 x 256 x 32 per SM.
double measure_int8_peak(long iters);

}  // namespace tbk
