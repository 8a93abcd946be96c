// tbk_api.cu -- the C ABI (include/tbk.h): model packing, chunked launch sequences, host pipelines.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>  // header-only; ranges cost a few ns unless a profiler is attached

#include "../../include/tbk.h"
#include "tbk_kernels.h"
#include "tbk_math.cuh"

using namespace tbk;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return fail(TBK_E_CUDA, "%s -> %s", #call, cudaGetErrorString(e_)); \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = (cudaSetDevice(dev) == cudaSuccess);
    }
    ~DeviceGuard() {
        int cur = -1;
        if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
    }
};

void pack_weights_host(int n, int nR, const double* hop, double* W) {
    const long NN = (long)n * n;
    const long nre = tri(n);
    for (int r = 0; r < nR; ++r) {
        const double* T = hop + (size_t)r * NN * 2;
        double* w0 = W + (size_t)(2 * r) * NN;
        double* w1 = w0 + NN;
        for (int i = 0; i < n; ++i) {
            for (int j = 0; j <= i; ++j) {
                const double tr_ij = T[((long)i * n + j) * 2], ti_ij = T[((long)i * n + j) * 2 + 1];
                const double tr_ji = T[((long)j * n + i) * 2], ti_ji = T[((long)j * n + i) * 2 + 1];
                // A = T + T^H ; B = i (T - T^H)
                w0[tri(i) + j] = tr_ij + tr_ji;
                w1[tri(i) + j] = -(ti_ij + ti_ji);
                if (j < i) {
                    w0[nre + trs(i) + j] = ti_ij - ti_ji;
                    w1[nre + trs(i) + j] = tr_ij - tr_ji;
                }
            }
        }
    }
}

// one row per Taylor term: the packed lower triangle of the (Hermitian) coefficient matrix itself
void pack_hermitian_rows_host(int n, int nterms, const double* mats, double* W) {
    const long NN = (long)n * n;
    const long nre = tri(n);
    for (int q = 0; q < nterms; ++q) {
        const double* C = mats + (size_t)q * NN * 2;
        double* w = W + (size_t)q * NN;
        for (int i = 0; i < n; ++i)
            for (int j = 0; j <= i; ++j) {
                w[tri(i) + j] = C[((long)i * n + j) * 2];
                if (j < i) w[nre + trs(i) + j] = C[((long)i * n + j) * 2 + 1];
            }
    }
}

// Power-of-two normalisation.  B = max_ij sum_R (|T_R,ij| + |T_R,ji|) bounds |H(k)_ij| at every k, so ||H(k)||_2 <= N B
// with N <= 8192 = 2^13.  The solvers square entries with no scaling (Householder norms, QL rotations, the Sturm
// sequence's e^2, the 2 x 2 closed form) and switch to their fast reciprocal (square root) paths inside 1e+-280 (about
// 2^+-930).  For 2^-W <= B < 2^W:
//   * the largest square, a sum of N squares of entries <= N B, stays below N^3 B^2 <= 2^(39 + 2W);
//   * the smallest square that moves a result at the eps rho level, (eps B)^2, stays above 2^(-104 - 2W);
// both inside (2^-930, 2^930) while W <= 412.  W = 384 keeps a margin of 2^50 on both sides (B is computed with
// |Re| + |Im| for the modulus, at most sqrt(2) above the sum of moduli: half a binade of that margin).  A model outside the window
// is scaled by 2^-s on upload, s even so that the hardware rsqrt seeds (exact under even exponent shifts) give the
// bits of the same model at its normalised scale; B 2^-s then lies in [1, 4).  Every result is scaled back by 2^s.  Models
// inside the window (every physical unit system) keep s = 0: the same kernels and launches as without normalisation.
constexpr int kScaleWindow = 384;

// B for n_mats complex [N][N] matrices (hoppings of the half set, or k.p coefficients), with |re| + |im| in place of the
// modulus: within a factor sqrt(2) of the bound, which is all the choice of s needs, and a contiguous walk as cheap as
// the packing's.
double coupling_bound(int n, int n_mats, const double* mats) {
    const size_t NN = (size_t)n * n;
    std::vector<double> acc(NN, 0.0);
    for (int r = 0; r < n_mats; ++r) {
        const double* T = mats + (size_t)r * NN * 2;
        for (size_t e = 0; e < NN; ++e) acc[e] += std::fabs(T[2 * e]) + std::fabs(T[2 * e + 1]);
    }
    double B = 0.0;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j <= i; ++j) B = std::max(B, acc[(size_t)i * n + j] + acc[(size_t)j * n + i]);
    return B;
}

int normalise_exponent(double B) {
    if (!(B > 0.0) || !std::isfinite(B)) return 0;  // empty model, or non-finite input: nothing to normalise
    const int x = std::ilogb(B);
    if (x >= -kScaleWindow && x < kScaleWindow) return 0;
    return x & ~1;
}

// mats * 2^-s into `keep`; returns the pointer to use in place of `mats`
const double* scaled_copy(const double* mats, size_t n_doubles, int s, std::vector<double>& keep) {
    if (s == 0) return mats;
    keep.resize(n_doubles);
    for (size_t i = 0; i < n_doubles; ++i) keep[i] = std::ldexp(mats[i], -s);
    return keep.data();
}

int env_int(const char* name, int dflt) {
    const char* s = getenv(name);
    return s ? atoi(s) : dflt;
}

}  // namespace

namespace tbk {
// Environment hooks (DESIGN.md section 5), read once per handle: tbk_model_create / tbk_kdotp_create.
Tuning read_tuning() {
    Tuning t;
    const long ws = env_int("TBK_WORKSPACE_MB", 0), hc = env_int("TBK_HOST_CHUNK_MB", 0);
    if (ws > 0) t.workspace_mb = ws;
    if (hc > 0) t.host_chunk_mb = hc;
    t.no_mesh_factor = getenv("TBK_NO_MESH_FACTOR") ? 1 : 0;
    t.basis_kp = env_int("TBK_BASIS_KP", 0);
    t.tridiag_g = env_int("TBK_TRIDIAG_G", 0);
    t.tridiag_cs = env_int("TBK_TRIDIAG_CS", 1);
    t.tridiag_mpb = env_int("TBK_TRIDIAG_MPB", 0);
    t.tridiag_g1 = env_int("TBK_TRIDIAG_G1", 0);
    t.tridiag_cs1 = env_int("TBK_TRIDIAG_CS1", 0);
    t.tridiag_stages = env_int("TBK_TRIDIAG_STAGES", t.tridiag_stages);
    t.tridiag_panel_min = env_int("TBK_TRIDIAG_PANEL_MIN", 0);
    t.tridiag_nopanel = getenv("TBK_TRIDIAG_NOPANEL") ? 1 : 0;
    t.tridiag_panel_stop = env_int("TBK_TRIDIAG_PANEL_STOP", t.tridiag_panel_stop);
    t.tridiag_oldbig = getenv("TBK_TRIDIAG_OLDBIG") ? 1 : 0;
    t.tridiag_reg_min = env_int("TBK_TRIDIAG_REG_MIN", t.tridiag_reg_min);
    t.tridiag_reg_max = env_int("TBK_TRIDIAG_REG_MAX", t.tridiag_reg_max);
    if (t.tridiag_reg_max > kTridiagRegMaxN) t.tridiag_reg_max = kTridiagRegMaxN;
    t.tridiag_reg_bw = env_int("TBK_TRIDIAG_REG_BW", t.tridiag_reg_bw);
    t.tridiag_reg_stop = env_int("TBK_TRIDIAG_REG_STOP", t.tridiag_reg_stop);
    t.tridiag_reg_mid = env_int("TBK_TRIDIAG_REG_MID", t.tridiag_reg_mid);
    t.panel_t = env_int("TBK_PANEL_T", 0);
    t.panel_lpr = env_int("TBK_PANEL_LPR", 0);
    t.panel_pfd = env_int("TBK_PANEL_PFD", 1);
    t.ql_bisect_min = env_int("TBK_QL_BISECT_MIN", 0);
    t.gemm_dense = getenv("TBK_GEMM_DENSE") ? 1 : 0;
    t.hk_fp64 = env_int("TBK_HK_FP64", t.hk_fp64);
    t.tridiag_twostage = env_int("TBK_TRIDIAG_TWOSTAGE", t.tridiag_twostage);
    t.band_t = env_int("TBK_BAND_T", t.band_t);
    t.band_stage2 = env_int("TBK_BAND_STAGE2", t.band_stage2);
    t.band_group_mb = env_int("TBK_BAND_GROUP_MB", (int)t.band_group_mb);
    t.band_wave = env_int("TBK_BAND_WAVE", t.band_wave);
    t.band_chase = env_int("TBK_BAND_CHASE", t.band_chase);
    t.ql_global_min = env_int("TBK_QL_GLOBAL_MIN", 0);
    t.ql_overlap = env_int("TBK_QL_OVERLAP", t.ql_overlap);
    return t;
}
}  // namespace tbk

struct tbk_model {
    int device = 0;
    ModelDev md;
    int scale_exp = 0;  // the device copy holds the model times 2^-scale_exp (normalise_exponent); results are scaled back
    double* dRd = nullptr;
    double* dW = nullptr;
    int* dRi = nullptr;
    int* dPw = nullptr;
    double* dWt = nullptr;
    double* dPos = nullptr;
    int* dFail = nullptr;
    int* dKcCnt = nullptr;  // block-sparse weights: non-zero K-chunks per column tile (hk_gemm.cu, SP = true)
    int* dKcIdx = nullptr;
    int8_t* dWd = nullptr;   // INT8 digit GEMM: weight digits and column scales (hk_gemm_i8.cu)
    double* dWsc = nullptr;
    // scratch for the device-pointer entry points
    double* wsH = nullptr;  // [chunk][n*n] packed H(k)
    double* wsE = nullptr;  // [chunk][n]   sub-diagonals
    // two-stage reduction (sizes it serves only): band arrays [band_cap][n][16] complex of up to band_cap matrices -- several
    // workspace chunks -- and their sub-diagonals; the bulge chasing and the tridiagonal solver run once per group
    double* wsB = nullptr;
    double* wsEg = nullptr;
    long band_cap = 0, band_fill = 0, band_first_row = 0;
    double* band_D0 = nullptr;
    double* wsQ = nullptr;  // phase tiles of the chunk (GEMM path only)
    // regular k-mesh entry point (tbk_eigenval_mesh)
    int* dRc = nullptr;       // [nRpad] class (last component) of every stored R
    double* dZc = nullptr;    // [nclass]
    double* wsAB = nullptr;   // [lines][2 nclass][n*n] line coefficients (stage A output)
    double* wsQz = nullptr;   // [n_z][2 nclass] cos / sin along the last mesh dimension
    double* wsK = nullptr;    // explicit k-points of a mesh range (ordinary-path fallback)
    double* wsV = nullptr;    // eigh, N > 82: full matrix + accumulated unitary of every matrix in flight
    size_t v_bytes = 0;
    double* wsKp = nullptr;   // construct_kdotp: [n_terms] prefactors followed by the int powers [n_terms][dim]
    double* dDerivKp = nullptr;  // run_eigh: the same arrays for the dim unit power tuples and the zero tuple (H(k))
    double* wsVel = nullptr;  // run_eigh, velocities and curvature: [chunk] eigenvectors [n][n] c128, then [chunk][terms]
                              // Taylor terms [n][n] c128 (curvature: then [chunk][dim] product scratch)
    size_t vel_bytes = 0;
    size_t ab_bytes = 0, qz_bytes = 0, k_bytes = 0, kp_bytes = 0;
    long chunk = 0;
    size_t ws_bytes = 0;
    size_t model_bytes = 0;
    // host pipeline
    cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    double* hk[2] = {nullptr, nullptr};
    double* ho[2] = {nullptr, nullptr};
    size_t hk_bytes = 0, ho_bytes = 0;
    int64_t launches = 0;
    // background QL (chunk i's tridiagonal eigenvalues behind chunk i + 1's build): side stream, second E buffer, events
    cudaStream_t s_ql = nullptr;
    cudaEvent_t ev_td[2] = {nullptr, nullptr}, ev_ql[2] = {nullptr, nullptr};
    double* wsE2 = nullptr;
    unsigned long long* dCounter = nullptr;
    bool ql_pending[2] = {false, false};
    bool ql_bg_ok = false;
    long eig_chunk_index = 0;
    // peer push of the multi-GPU entry point (tbk_eigenval_push): side stream + events ordering it against the chunks
    cudaStream_t s_push = nullptr;
    cudaEvent_t ev_chunk = nullptr, ev_push = nullptr;
    // The handle has ONE scratch set (wsH / wsE / wsQ / ...).  Every entry point records ev_busy on the stream it used
    // when its launches are queued and makes its stream wait on the previous record first, so calls on different
    // streams (a device-pointer call on a torch stream followed by a _host call on s_comp, two torch streams, ...)
    // are ordered on the device instead of racing on the scratch.
    cudaEvent_t ev_busy = nullptr;
    bool busy_recorded = false;
    // optional per-kernel-class CUDA-event timing (tbk_profile / tbk_profile_read)
    bool prof_on = false;
    struct ProfRec {
        cudaEvent_t a, b;
        int cls;
    };
    std::vector<ProfRec> prof;
    double prof_ms[TBK_PROFILE_CLASSES] = {0};
    int64_t prof_n[TBK_PROFILE_CLASSES] = {0};
};

// NVTX range names of the kernel classes (SURVEY.md section 5: tracing) -- visible in Nsight Systems / ncu --nvtx.
static const char* const kClassName[TBK_PROFILE_CLASSES] = {"tbk:hk_gemm", "tbk:hk_small", "tbk:expand", "tbk:tridiag",
                                                           "tbk:ql", "tbk:hk_phase", "tbk:mesh_lines", "tbk:eigh",
                                                           "tbk:peer_push", "tbk:rescale"};
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

// Launch wrapper: counts the launch and, when profiling is on, brackets it with events on the launch stream.
#define LAUNCH(cls, st, call)                                        \
    do {                                                             \
        NvtxRange nvtx_(kClassName[(cls)]);                          \
        tbk_model::ProfRec rec_{nullptr, nullptr, (cls)};            \
        if (m->prof_on) {                                            \
            CU(cudaEventCreate(&rec_.a));                            \
            CU(cudaEventCreate(&rec_.b));                            \
            CU(cudaEventRecord(rec_.a, (st)));                       \
        }                                                            \
        CU(call);                                                    \
        if (m->prof_on) {                                            \
            CU(cudaEventRecord(rec_.b, (st)));                       \
            m->prof.push_back(rec_);                                 \
        }                                                            \
        m->launches += 1;                                            \
    } while (0)

namespace {

// Column-tile width that wastes the fewest padded columns (ties -> wider), tile and K-chunk counts.
void choose_gemm_tiling(ModelDev& md, int n_rows) {
    const long NN = (long)md.n * md.n;
    const int cands[3] = {4, 8, 9};
    long best_cols = -1;
    for (int c : cands) {
        const long bn = 16L * c;
        const long cols = ((NN + bn - 1) / bn) * bn;
        if (best_cols < 0 || cols <= best_cols) {
            best_cols = cols;
            md.na = c;
        }
    }
    md.n_tiles = (int)((NN + 16 * md.na - 1) / (16 * md.na));
    md.kchunks = (n_rows + kGemmKC - 1) / kGemmKC;
}

// Block-sparse weights: nz[tile * kchunks + c] says whether stage (tile, c) of Wt holds anything non-zero.  If some
// stage is empty the GEMM gets the per-tile lists of populated K-chunks and skips the rest (hk_gemm.cu, SP = true).
int upload_stage_lists(tbk_model* m, const std::vector<unsigned char>& nz) {
    ModelDev& md = m->md;
    const size_t total = (size_t)md.n_tiles * md.kchunks;
    size_t populated = 0;
    for (size_t i = 0; i < total; ++i) populated += nz[i] ? 1 : 0;
    if (populated == total || md.tune.gemm_dense) return TBK_OK;
    std::vector<int> cnt((size_t)md.n_tiles, 0), idx(std::max<size_t>(total, 1), 0);
    for (int nt = 0; nt < md.n_tiles; ++nt)
        for (int c = 0; c < md.kchunks; ++c)
            if (nz[(size_t)nt * md.kchunks + c]) idx[(size_t)nt * md.kchunks + cnt[nt]++] = c;
    CU(cudaMalloc(&m->dKcCnt, cnt.size() * sizeof(int)));
    CU(cudaMemcpy(m->dKcCnt, cnt.data(), cnt.size() * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&m->dKcIdx, idx.size() * sizeof(int)));
    CU(cudaMemcpy(m->dKcIdx, idx.data(), idx.size() * sizeof(int), cudaMemcpyHostToDevice));
    md.kc_cnt = m->dKcCnt;
    md.kc_idx = m->dKcIdx;
    m->model_bytes += (cnt.size() + idx.size()) * sizeof(int);
    return TBK_OK;
}

// Tile the weight rows W[n_rows][n*n] for the GEMM (column tiles x 16-row K stages, padding baked in) and upload.
int upload_gemm_weights(tbk_model* m, const std::vector<double>& W, int n_rows) {
    ModelDev& md = m->md;
    const long NN = (long)md.n * md.n;
    choose_gemm_tiling(md, n_rows);
    const int bn = 16 * md.na, sb = bn + 4;
    const size_t stage = (size_t)kGemmKC * sb;
    std::vector<double> Wt((size_t)std::max(md.n_tiles * md.kchunks, 1) * stage, 0.0);
    std::vector<unsigned char> nz((size_t)std::max(md.n_tiles * md.kchunks, 1), 0);
    for (int nt = 0; nt < md.n_tiles; ++nt)
        for (int c = 0; c < md.kchunks; ++c) {
            double* blk = Wt.data() + ((size_t)nt * md.kchunks + c) * stage;
            unsigned char any = 0;
            for (int kk = 0; kk < kGemmKC; ++kk) {
                const long q = (long)c * kGemmKC + kk;
                if (q >= n_rows) continue;
                const double* src = W.data() + (size_t)q * NN;
                for (int col = 0; col < bn; ++col) {
                    const long e = (long)nt * bn + col;
                    if (e < NN) {
                        blk[(size_t)kk * sb + col] = src[e];
                        any |= src[e] != 0.0;
                    }
                }
            }
            nz[(size_t)nt * md.kchunks + c] = any;
        }
    CU(cudaMalloc(&m->dWt, Wt.size() * 8));
    CU(cudaMemcpy(m->dWt, Wt.data(), Wt.size() * 8, cudaMemcpyHostToDevice));
    md.Wt = m->dWt;
    m->model_bytes += Wt.size() * 8;
    return upload_stage_lists(m, nz);
}

// Digits of the tiled weights for the INT8 GEMM of the explicit-k H(k) builds: phase handles whose K fits the int32
// class sums and is long enough for the INT8 GEMM to win (kI8MinKSteps), unless TBK_HK_FP64 decides.  k.p handles stay on
// DMMA (their monomial rows are not bounded by 1, which the fixed-point phase digits need).
int prepare_hk_i8(tbk_model* m) {
    ModelDev& md = m->md;
    const int ks = hk_i8_ksteps(md);
    if (md.kind != 0 || md.small_ok || md.tune.hk_fp64 == 1 || ks < 1 || ks > kI8MaxKSteps) return TBK_OK;
    if (md.tune.hk_fp64 < 0 && ks < kI8MinKSteps) return TBK_OK;
    const size_t sc_bytes = (size_t)(((long)md.n * md.n + kI8BM - 1) / kI8BM) * kI8BM * 8;
    CU(cudaMalloc(&m->dWd, hk_i8_w_bytes(md)));
    CU(cudaMalloc(&m->dWsc, sc_bytes));
    CU(launch_hk_wdigits(md, m->dWd, m->dWsc, nullptr));
    CU(cudaDeviceSynchronize());
    m->launches += 1;
    md.Wd = m->dWd;
    md.Wsc = m->dWsc;
    m->model_bytes += hk_i8_w_bytes(md) + sc_bytes;
    return TBK_OK;
}

// Classes of the stored R vectors by their last component (regular k-mesh path, hk_mesh.cu).
int setup_mesh_classes(tbk_model* m, const int32_t* R, int n_R) {
    ModelDev& md = m->md;
    const int dim = md.dim;
    if (dim < 2 || n_R <= 0) return TBK_OK;
    std::vector<int> zs;
    for (int r = 0; r < n_R; ++r) zs.push_back(R[(size_t)r * dim + dim - 1]);
    std::vector<int> uniq(zs);
    std::sort(uniq.begin(), uniq.end());
    uniq.erase(std::unique(uniq.begin(), uniq.end()), uniq.end());
    std::vector<int> Rc((size_t)md.kchunks * 8, -1);
    for (int r = 0; r < n_R; ++r) Rc[r] = (int)(std::lower_bound(uniq.begin(), uniq.end(), zs[r]) - uniq.begin());
    std::vector<double> zc(uniq.begin(), uniq.end());
    CU(cudaMalloc(&m->dRc, Rc.size() * sizeof(int)));
    CU(cudaMemcpy(m->dRc, Rc.data(), Rc.size() * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&m->dZc, zc.size() * 8));
    CU(cudaMemcpy(m->dZc, zc.data(), zc.size() * 8, cudaMemcpyHostToDevice));
    md.Rc = m->dRc;
    md.zc = m->dZc;
    md.nclass = (int)uniq.size();
    return TBK_OK;
}

long pick_chunk(const tbk_model* m) {
    const size_t budget_mb = (size_t)m->md.tune.workspace_mb;
    const size_t per_k = ((size_t)m->md.n * m->md.n + m->md.n + (m->md.small_ok ? 0 : (size_t)m->md.kchunks * kGemmKC)) * 8;
    long chunk = (long)((budget_mb << 20) / per_k);
    if (chunk < 1) chunk = 1;
    if (chunk > (1L << 22)) chunk = 1L << 22;
    if (chunk >= 1024) chunk &= ~127L;  // whole GEMM row tiles
    if (!m->md.small_ok) {
        // whole waves of the thread-per-matrix QL kernel (its threads all run equally long: a partial wave idles SMs)
        const long wave = ql_wave_matrices(m->md.n, m->md.tune);
        if (wave > 0 && chunk > wave) chunk -= chunk % wave;
    }
    return chunk;
}

int ensure_workspace(tbk_model* m, long nk) {
    const long want = std::min(nk, pick_chunk(m));
    const bool two = !m->md.small_ok && tridiag_twostage_default(m->md.n, m->md.tune);
    long group = 0;  // matrices whose band arrays are collected before the second stage runs
    if (two) {
        const long per = (long)tridiag_twostage_scratch_bytes(m->md.n, 1);
        group = std::min(nk, std::max(want, (m->md.tune.band_group_mb << 20) / per));
    }
    if (want <= m->chunk && group <= m->band_cap) return TBK_OK;
    if (m->wsH) cudaFree(m->wsH);
    if (m->wsE) cudaFree(m->wsE);
    if (m->wsQ) cudaFree(m->wsQ);
    if (m->wsE2) cudaFree(m->wsE2);
    if (m->wsB) cudaFree(m->wsB);
    if (m->wsEg) cudaFree(m->wsEg);
    m->wsH = m->wsE = m->wsQ = m->wsE2 = m->wsB = m->wsEg = nullptr;
    m->band_cap = m->band_fill = 0;
    m->chunk = 0;
    m->ws_bytes = 0;
    const size_t hb = (size_t)want * m->md.n * m->md.n * 8;
    const size_t eb = (size_t)want * m->md.n * 8;
    CU(cudaMalloc(&m->wsH, hb));
    CU(cudaMalloc(&m->wsE, eb));
    size_t qb = 0;
    if (!m->md.small_ok) {
        qb = std::max<size_t>(hk_gemm_q_doubles(m->md, want) * 8, 16);
        if (m->md.Wd) qb = std::max(qb, hk_i8_q_bytes(m->md, want));
        CU(cudaMalloc(&m->wsQ, qb));
    }
    size_t eb2 = 0;
    if (!m->md.small_ok && m->md.tune.ql_overlap) {  // second sub-diagonal buffer: QL of chunk i overlaps chunk i + 1
        eb2 = eb;
        CU(cudaMalloc(&m->wsE2, eb2));
    }
    size_t bb = 0;
    if (two) {
        bb = tridiag_twostage_scratch_bytes(m->md.n, group) + (size_t)group * m->md.n * 8;
        CU(cudaMalloc(&m->wsB, tridiag_twostage_scratch_bytes(m->md.n, group)));
        CU(cudaMalloc(&m->wsEg, (size_t)group * m->md.n * 8));
        m->band_cap = group;
    }
    m->chunk = want;
    m->ws_bytes = hb + eb + qb + eb2 + bb;
    return TBK_OK;
}

// Peer destinations of tbk_eigenval_push: after every chunk its rows are stored into the peers' buffers on a side stream.
struct PushPlan {
    double* const* bases = nullptr;
    int n = 0;
    long row_offset = 0;  // row of out[0] inside the peers' buffers
};

int push_chunk(tbk_model* m, const PushPlan& plan, const double* rows, long first_row, long n_rows, cudaStream_t st) {
    if (plan.n <= 0 || n_rows <= 0) return TBK_OK;
    CU(cudaEventRecord(m->ev_chunk, st));
    CU(cudaStreamWaitEvent(m->s_push, m->ev_chunk, 0));
    LAUNCH(8, m->s_push, launch_push_rows(rows, n_rows * m->md.n, plan.bases, plan.n, (plan.row_offset + first_row) * m->md.n,
                                          m->s_push));
    return TBK_OK;
}

// Undo the model's power-of-two normalisation on n results (no launch for the models that needed none).
int unscale(tbk_model* m, double* p, long n, cudaStream_t st) {
    if (m->scale_exp == 0 || n <= 0) return TBK_OK;
    LAUNCH(9, st, launch_scale_pow2(p, n, m->scale_exp, st));
    return TBK_OK;
}

// Tridiagonalisation + tridiagonal eigenvalues of one chunk (packed H in wsH -> ascending eigenvalues in D).  With
// TBK_QL_OVERLAP=1 and more than one chunk in the call, the QL of every chunk but the last runs as a few
// persistent CTAs on a side stream (launch_ql_background) while the main stream already builds and tridiagonalises the
// next chunk; two sub-diagonal buffers alternate.  (Opt-in experiment: the step is throughput bound, not latency bound --
// the background QL slows its co-resident kernels by as much as it saves, see Tuning::ql_overlap.)  eig_begin / eig_drain bracket the chunks of one call.
int eig_begin(tbk_model* m, long n_chunks) {
    m->band_fill = 0;
    m->ql_pending[0] = m->ql_pending[1] = false;
    m->eig_chunk_index = 0;
    m->ql_bg_ok = m->md.tune.ql_overlap && n_chunks >= 2 && m->wsE2 != nullptr;
    if (m->ql_bg_ok && !m->s_ql) {
        CU(cudaStreamCreateWithFlags(&m->s_ql, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            CU(cudaEventCreateWithFlags(&m->ev_td[b], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&m->ev_ql[b], cudaEventDisableTiming));
        }
        CU(cudaMalloc(&m->dCounter, sizeof(unsigned long long)));
    }
    return TBK_OK;
}

// Two-stage sizes: second stage (bulge chasing), tridiagonal solver and peer push of the collected group.
int band_flush(tbk_model* m, cudaStream_t st, const PushPlan* plan) {
    const ModelDev& md = m->md;
    const long cnt = m->band_fill;
    if (cnt <= 0) return TBK_OK;
    m->band_fill = 0;
    if (md.tune.band_stage2) {
        // balanced launches of at most one resident wave of the bulge-chasing kernel (its warps all run equally long: a
        // launch of 1.3 waves takes as long as one of 2)
        const long wave = std::max<long>(1, band_chase_wave_matrices(md.tune));
        const long parts = (cnt + wave - 1) / wave;
        const long per = (cnt + parts - 1) / parts;
        for (long c0 = 0; c0 < cnt; c0 += per) {
            const long cn = std::min(per, cnt - c0);
            LAUNCH(3, st, launch_band_chase(md.n, m->wsB + (size_t)c0 * md.n * 32, cn, m->band_D0 + c0 * md.n,
                                            m->wsEg + c0 * md.n, st, md.tune));
        }
    }
    LAUNCH(4, st, launch_ql(md.n, m->band_D0, m->wsEg, cnt, m->dFail, st, md.tune));
    if (int rc = unscale(m, m->band_D0, cnt * md.n, st)) return rc;
    if (plan)
        if (int rc = push_chunk(m, *plan, m->band_D0, m->band_first_row, cnt, st)) return rc;
    return TBK_OK;
}

int eig_chunk(tbk_model* m, double* D, long cn, bool last, cudaStream_t st, const PushPlan* plan, long first_row) {
    const ModelDev& md = m->md;
    if (m->wsB != nullptr && tridiag_twostage_default(md.n, md.tune)) {
        // first stage now (the packed matrices live in the workspace chunk), band arrays collected over several chunks
        if (m->band_fill > 0 && (D != m->band_D0 + m->band_fill * md.n || m->band_fill + cn > m->band_cap))
            if (int rc = band_flush(m, st, plan)) return rc;
        if (m->band_fill == 0) {
            m->band_D0 = D;
            m->band_first_row = first_row;
        }
        LAUNCH(3, st, launch_band_reduce(md.n, m->wsH, cn, m->wsB + (size_t)m->band_fill * md.n * 32, st, md.tune));
        m->band_fill += cn;
        if (last || m->band_fill + m->chunk > m->band_cap) return band_flush(m, st, plan);
        return TBK_OK;
    }
    const int b = (int)(m->eig_chunk_index++ & 1);
    double* E = (m->ql_bg_ok && b) ? m->wsE2 : m->wsE;
    if (m->ql_pending[b]) {  // the QL two chunks back still owns this sub-diagonal buffer
        CU(cudaStreamWaitEvent(st, m->ev_ql[b], 0));
        m->ql_pending[b] = false;
    }
    LAUNCH(3, st, launch_tridiag(md.n, m->wsH, cn, D, E, st, md.tune));
    if (m->ql_bg_ok && !last) {
        CU(cudaEventRecord(m->ev_td[b], st));
        CU(cudaStreamWaitEvent(m->s_ql, m->ev_td[b], 0));
        const size_t gemm_smem = hk_gemm_smem_bytes(md);
        const size_t budget = gemm_smem + 4096 < 227 * 1024 ? 227 * 1024 - gemm_smem - 2048 : 0;
        tbk_model::ProfRec rec{nullptr, nullptr, 4};
        if (m->prof_on) {
            CU(cudaEventCreate(&rec.a));
            CU(cudaEventCreate(&rec.b));
            CU(cudaEventRecord(rec.a, m->s_ql));
        }
        const cudaError_t err = launch_ql_background(md.n, D, E, cn, m->dFail, m->dCounter, budget, m->s_ql, md.tune);
        if (err == cudaSuccess) {
            if (m->prof_on) {
                CU(cudaEventRecord(rec.b, m->s_ql));
                m->prof.push_back(rec);
            }
            m->launches += 1;
            if (int rc = unscale(m, D, cn * md.n, m->s_ql)) return rc;
            CU(cudaEventRecord(m->ev_ql[b], m->s_ql));
            m->ql_pending[b] = true;
            if (plan)
                if (int rc = push_chunk(m, *plan, D, first_row, cn, m->s_ql)) return rc;
            return TBK_OK;
        }
        if (m->prof_on) {
            cudaEventDestroy(rec.a);
            cudaEventDestroy(rec.b);
        }
        if (err != cudaErrorNotSupported) return fail(TBK_E_CUDA, "launch_ql_background -> %s", cudaGetErrorString(err));
        cudaGetLastError();
        m->ql_bg_ok = false;  // size served by bisection / no CTA shape fits: in stream order from here on
    }
    LAUNCH(4, st, launch_ql(md.n, D, E, cn, m->dFail, st, md.tune));
    if (int rc = unscale(m, D, cn * md.n, st)) return rc;
    if (plan)
        if (int rc = push_chunk(m, *plan, D, first_row, cn, st)) return rc;
    return TBK_OK;
}

int eig_drain(tbk_model* m, cudaStream_t st) {
    if (m->band_fill > 0)  // (the last chunk of a call flushes; kept for callers that stop early)
        if (int rc = band_flush(m, st, nullptr)) return rc;
    for (int b = 0; b < 2; ++b)
        if (m->ql_pending[b]) {
            CU(cudaStreamWaitEvent(st, m->ev_ql[b], 0));
            m->ql_pending[b] = false;
        }
    return TBK_OK;
}

// H(k) of cn explicit k-points through a GEMM, packed into wsH: the INT8 digit GEMM where the handle has digits, else
// the FP64 phase tiles and the DMMA GEMM.  (The mesh path's stage A calls the DMMA GEMM directly.)
int build_hk_gemm(tbk_model* m, const double* k, long cn, cudaStream_t st) {
    const ModelDev& md = m->md;
    if (md.Wd) {
        int8_t* Qd = reinterpret_cast<int8_t*>(m->wsQ);
        LAUNCH(5, st, launch_hk_qdigits(md, k, cn, Qd, st));
        LAUNCH(0, st, launch_hk_gemm_i8(md, cn, Qd, m->wsH, st));
    } else {
        LAUNCH(5, st, launch_hk_phase(md, k, cn, m->wsQ, st));
        LAUNCH(0, st, launch_hk_gemm(md, cn, m->wsQ, m->wsH, st));
    }
    return TBK_OK;
}

int run_eigenval(tbk_model* m, const double* k, long nk, double* out, cudaStream_t st, const PushPlan* plan = nullptr) {
    NvtxRange nvtx_call_("tbk:eigenval");
    const ModelDev& md = m->md;
    if (nk <= 0) return TBK_OK;
    if (md.small_ok) {
        // fused small-N kernel: cut the batch into a few launches so that the peer stores overlap the next launch
        const long step = plan ? std::max<long>(1L << 20, (nk + 7) / 8) : nk;
        for (long c0 = 0; c0 < nk; c0 += step) {
            const long cn = std::min(step, nk - c0);
            LAUNCH(1, st, launch_hk_small(md, k + c0 * md.dim, cn, nullptr, out + c0 * md.n, m->dFail, st));
            if (int rc = unscale(m, out + c0 * md.n, cn * md.n, st)) return rc;
            if (plan)
                if (int rc = push_chunk(m, *plan, out + c0 * md.n, c0, cn, st)) return rc;
        }
        return TBK_OK;
    }
    if (int rc = ensure_workspace(m, nk)) return rc;
    if (int rc = eig_begin(m, (nk + m->chunk - 1) / m->chunk)) return rc;
    for (long c0 = 0; c0 < nk; c0 += m->chunk) {
        const long cn = std::min(m->chunk, nk - c0);
        double* D = out + c0 * md.n;
        if (int rc = build_hk_gemm(m, k + c0 * md.dim, cn, st)) return rc;
        if (int rc = eig_chunk(m, D, cn, c0 + cn >= nk, st, plan, c0)) return rc;
    }
    return eig_drain(m, st);
}

int grow(double** p, size_t* have, size_t want) {
    if (want <= *have) return TBK_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *have = 0;
    CU(cudaMalloc(p, want));
    *have = want;
    return TBK_OK;
}

// Lines of a regular mesh can be factorised when the model runs on the GEMM path, has at least two dimensions, a line
// fits one workspace chunk and the 2 C pseudo k-points of a line are fewer than its mesh points.
bool mesh_factorised(const tbk_model* m, const int64_t* dims) {
    const ModelDev& md = m->md;
    if (md.small_ok || md.kind != 0 || md.nclass <= 0 || md.dim < 2) return false;
    if (md.tune.no_mesh_factor) return false;  // test hook: explicit k-points through the ordinary path
    const long nz = (long)dims[md.dim - 1];
    if (2L * md.nclass > nz || 2 * md.nclass > 256) return false;
    if (mesh_lines_smem_bytes(2 * md.nclass) > 200 * 1024) return false;
    return nz <= pick_chunk(m);
}

int run_eigenval_mesh(tbk_model* m, const int64_t* dims, const double* shift, long line0, long n_lines, double* out,
                      cudaStream_t st) {
    const ModelDev& md = m->md;
    const long nz = (long)dims[md.dim - 1];
    if (n_lines <= 0 || nz <= 0) return TBK_OK;
    if (!mesh_factorised(m, dims)) {
        // ordinary path on k-points generated on the device, one workspace chunk at a time
        const long total = n_lines * nz;
        const long kchunk = std::min<long>(total, 1L << 22);
        if (int rc = grow(&m->wsK, &m->k_bytes, (size_t)kchunk * md.dim * 8)) return rc;
        for (long c0 = 0; c0 < total; c0 += kchunk) {
            const long cn = std::min(kchunk, total - c0);
            LAUNCH(5, st, launch_mesh_kpoints(md.dim, dims, shift, line0 * nz + c0, cn, m->wsK, st));
            if (int rc = run_eigenval(m, m->wsK, cn, out + c0 * md.n, st)) return rc;
        }
        return TBK_OK;
    }
    const int K2 = 2 * md.nclass;
    const long NN = (long)md.n * md.n;
    if (int rc = ensure_workspace(m, n_lines * nz)) return rc;
    const long lchunk = std::max<long>(1, m->chunk / nz);  // whole lines per chunk (nz <= chunk was checked)
    const long lmax = std::min(lchunk, n_lines);
    if (int rc = grow(&m->wsAB, &m->ab_bytes, (size_t)lmax * K2 * NN * 8)) return rc;
    if (int rc = grow(&m->wsQz, &m->qz_bytes, (size_t)nz * K2 * 8)) return rc;
    LAUNCH(5, st, launch_mesh_qz(md, nz, shift ? shift[md.dim - 1] : 0.0, m->wsQz, st));
    if (int rc = eig_begin(m, (n_lines + lchunk - 1) / lchunk)) return rc;
    for (long l0 = 0; l0 < n_lines; l0 += lchunk) {
        const long ln = std::min(lchunk, n_lines - l0);
        const long cn = ln * nz;
        double* D = out + l0 * nz * md.n;
        // stage A: the 2 C line coefficients of every line as pseudo k-points through the DMMA GEMM
        LAUNCH(5, st, launch_mesh_phase(md, dims, shift, line0 + l0, ln, m->wsQ, st));
        LAUNCH(0, st, launch_hk_gemm(md, ln * K2, m->wsQ, m->wsAB, st));
        // stage B: expand every line along the last mesh dimension
        LAUNCH(6, st, launch_mesh_lines(md, m->wsAB, m->wsQz, nz, ln, m->wsH, st));
        if (int rc = eig_chunk(m, D, cn, l0 + ln >= n_lines, st, nullptr, 0)) return rc;
    }
    return eig_drain(m, st);
}

// H(k) of cn k-points, packed into wsH: the fused small-N kernel, or a GEMM (build_hk_gemm).
int build_hk(tbk_model* m, const double* k, long cn, cudaStream_t st) {
    const ModelDev& md = m->md;
    if (md.small_ok) {
        LAUNCH(1, st, launch_hk_small(md, k, cn, m->wsH, nullptr, nullptr, st));
        return TBK_OK;
    }
    return build_hk_gemm(m, k, cn, st);
}

int run_hamilton(tbk_model* m, const double* k, long nk, int convention, double* out, cudaStream_t st) {
    NvtxRange nvtx_call_("tbk:hamilton");
    const ModelDev& md = m->md;
    if (nk <= 0) return TBK_OK;
    if (int rc = ensure_workspace(m, nk)) return rc;
    const long NN = (long)md.n * md.n;
    for (long c0 = 0; c0 < nk; c0 += m->chunk) {
        const long cn = std::min(m->chunk, nk - c0);
        const double* kc = k + c0 * md.dim;
        if (int rc = build_hk(m, kc, cn, st)) return rc;
        LAUNCH(2, st, launch_expand(md, kc, m->wsH, cn, convention, out + c0 * NN * 2, st));
        if (int rc = unscale(m, out + c0 * NN * 2, cn * NN * 2, st)) return rc;
    }
    return TBK_OK;
}

// The kernel arguments of launch_kdotp_coeff: [n_terms] real prefactors followed by the int powers [n_terms][dim].
std::vector<double> kdotp_stage(const int32_t* powers, int n_terms, int dim) {
    const size_t fb = (size_t)n_terms * 8, pb = (size_t)n_terms * dim * sizeof(int);
    std::vector<double> stage((fb + pb + 7) / 8, 0.0);
    for (int t = 0; t < n_terms; ++t) {
        int order = 0;
        double f = 1.0;
        for (int d = 0; d < dim; ++d) {
            const int p = powers[(size_t)t * dim + d];
            order += p;
            for (int q = 2; q <= p; ++q) f /= (double)q;  // 1 / p_d!
        }
        for (int q = 0; q < order; ++q) f *= 2.0 * 3.14159265358979323846;
        const int flips = (order & 1) ? (order + 1) / 2 : order / 2;  // i^|p| (even) or i^(|p|+1) (odd) = (-1)^flips
        stage[t] = (flips & 1) ? -f : f;
    }
    memcpy(reinterpret_cast<char*>(stage.data()) + fb, powers, pb);
    return stage;
}

constexpr long kKdotpLaunchK = 32768;  // k-points per launch of run_kdotp_coeff

// Model.construct_kdotp (reference _tb_model.py:942-982): prefactors on the host, everything else in one kernel.
int run_kdotp_coeff(tbk_model* m, const double* k, long nk, const int32_t* powers, int n_terms, double* out, cudaStream_t st) {
    const ModelDev& md = m->md;
    if (nk <= 0 || n_terms <= 0) return TBK_OK;
    const size_t fb = (size_t)n_terms * 8, pb = (size_t)n_terms * md.dim * sizeof(int);
    if (int rc = grow(&m->wsKp, &m->kp_bytes, fb + pb)) return rc;
    const std::vector<double> stage = kdotp_stage(powers, n_terms, md.dim);
    // pageable source: the copy is staged by the driver before the call returns, so `stage` may go out of scope
    CU(cudaMemcpyAsync(m->wsKp, stage.data(), fb + pb, cudaMemcpyHostToDevice, st));
    const int* dpw = reinterpret_cast<const int*>(reinterpret_cast<const char*>(m->wsKp) + fb);
    for (long c0 = 0; c0 < nk; c0 += kKdotpLaunchK) {
        const long cn = std::min<long>(kKdotpLaunchK, nk - c0);
        LAUNCH(2, st, launch_kdotp_coeff(md, k + c0 * md.dim, cn, dpw, m->wsKp, n_terms,
                                         out + (size_t)c0 * n_terms * md.n * md.n * 2, st));
        if (int rc = unscale(m, out + (size_t)c0 * n_terms * md.n * md.n * 2, cn * n_terms * md.n * md.n * 2, st)) return rc;
    }
    return TBK_OK;
}

// What run_eigh computes after eigh: nothing (the eigenvectors are the result), band velocities, or Berry curvature.
struct EighOp {
    enum Kind { kEigh, kVelocity, kCurvature } kind = kEigh;
    int convention = 0;      // Berry curvature: 1 or 2
    double degen_tol = 0.0;  // band velocities, Berry curvature
};

// Taylor terms of launch_kdotp_coeff per k-point: dH/dk_d for every d and, for convention-1 curvature, H(k) itself.
int taylor_terms(const tbk_model* m, const EighOp& op) {
    if (op.kind == EighOp::kEigh) return 0;
    return m->md.dim + (op.kind == EighOp::kCurvature && op.convention == 1 ? 1 : 0);
}

// N x N c128 matrices per k-point in wsVel: eigenvectors, Taylor terms and (curvature) the dim product scratch matrices.
long vel_slots(const tbk_model* m, const EighOp& op) {
    return 1 + taylor_terms(m, op) + (op.kind == EighOp::kCurvature ? m->md.dim : 0);
}

// Doubles of run_eigh's second result per k-point: eigenvectors [N][N] c128, velocities [N][dim] or curvature [N][P].
size_t eigh_out_doubles(const tbk_model* m, const EighOp& op) {
    const size_t n = (size_t)m->md.n, dim = (size_t)m->md.dim;
    if (op.kind == EighOp::kEigh) return 2 * n * n;
    return op.kind == EighOp::kVelocity ? n * dim : n * (dim * (dim - 1) / 2);
}

// k-points per chunk of run_eigh, from the workspace chunk `base`.  Velocities and curvature keep vel_slots matrices per
// k-point in wsVel and, where eigh works on global scratch, its 32 N^2 bytes (which their kernels reuse for their blocks).
long eigh_chunk(const tbk_model* m, const EighOp& op, long base) {
    const ModelDev& md = m->md;
    const long NN = (long)md.n * md.n;
    const bool gscratch = !eigh_in_smem(md.n);
    long chunk = base;
    if (op.kind != EighOp::kEigh) {
        const size_t per_k = (size_t)NN * 16 * vel_slots(m, op) + (gscratch ? (size_t)NN * 32 : 0);
        chunk = std::min<long>(chunk, std::max<long>(1, (long)(((size_t)md.tune.workspace_mb << 20) / per_k)));
        chunk = std::min<long>(chunk, 65535);  // k-points per launch of launch_kdotp_coeff and of the product kernel
    }
    if (gscratch) chunk = std::max<long>(1, std::min<long>(chunk, (1L << 30) / (32L * NN)));  // eigh scratch: at most 1 GiB
    return chunk;
}

// kdotp_stage of the dim unit power tuples followed by the zero tuple, uploaded on first use: dH/dk_d and H(k) as
// Taylor terms.  Velocities use the first dim terms, curvature dim or dim + 1.  Returns the powers; the prefactors are
// at m->dDerivKp.
int derivative_terms(tbk_model* m, const int** powers) {
    const int dim = m->md.dim;
    if (!m->dDerivKp) {
        std::vector<int32_t> tuples((size_t)(dim + 1) * dim, 0);
        for (int d = 0; d < dim; ++d) tuples[(size_t)d * dim + d] = 1;
        const std::vector<double> stage = kdotp_stage(tuples.data(), dim + 1, dim);
        double* p = nullptr;
        CU(cudaMalloc(&p, stage.size() * 8));
        const cudaError_t e = cudaMemcpy(p, stage.data(), stage.size() * 8, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(p);
            return fail(TBK_E_CUDA, "derivative_terms: %s", cudaGetErrorString(e));
        }
        m->dDerivKp = p;
    }
    *powers = reinterpret_cast<const int*>(reinterpret_cast<const char*>(m->dDerivKp) + (size_t)(dim + 1) * 8);
    return TBK_OK;
}

// eigh and what follows it, chunk by chunk: H(k) build (packed, in wsH), eigh, then for velocities and curvature the
// Taylor terms of run_kdotp_coeff and their kernels.  eig [nk][N]; out [nk][eigh_out_doubles].  Eigenvectors go to out
// (eigh) or to wsVel, followed by the Taylor terms X and (curvature) the product scratch Y.  The curvature is invariant
// under H -> 2^e H and is not un-scaled.
int run_eigh(tbk_model* m, const double* k, long nk, const EighOp& op, double* eig, double* out, cudaStream_t st) {
    NvtxRange nvtx_call_(op.kind == EighOp::kEigh ? "tbk:eigh_call"
                         : op.kind == EighOp::kVelocity ? "tbk:band_velocity_call" : "tbk:berry_curvature_call");
    const ModelDev& md = m->md;
    if (nk <= 0) return TBK_OK;
    if (int rc = ensure_workspace(m, nk)) return rc;
    const long NN = (long)md.n * md.n;
    const int dim = md.dim, terms = taylor_terms(m, op);
    const size_t width = eigh_out_doubles(m, op);
    const long chunk = eigh_chunk(m, op, m->chunk);
    const long cc = std::min(chunk, nk);
    if (!eigh_in_smem(md.n))
        if (int rc = grow(&m->wsV, &m->v_bytes, (size_t)cc * NN * 32)) return rc;
    double *X = nullptr, *Y = nullptr;
    const int* dpw = nullptr;
    if (op.kind != EighOp::kEigh) {
        if (int rc = grow(&m->wsVel, &m->vel_bytes, (size_t)cc * NN * 16 * vel_slots(m, op))) return rc;
        if (int rc = derivative_terms(m, &dpw)) return rc;
        X = m->wsVel + (size_t)cc * NN * 2;
        Y = X + (size_t)cc * terms * NN * 2;
    }
    for (long c0 = 0; c0 < nk; c0 += chunk) {
        const long cn = std::min(chunk, nk - c0);
        const double* kc = k + c0 * dim;
        double* E = eig + c0 * md.n;
        double* O = out + (size_t)c0 * width;
        double* V = op.kind == EighOp::kEigh ? O : m->wsVel;
        if (int rc = build_hk(m, kc, cn, st)) return rc;
        LAUNCH(7, st, launch_eigh(md.n, m->wsH, cn, E, V, m->wsV, m->dFail, st));
        if (op.kind != EighOp::kEigh) LAUNCH(2, st, launch_kdotp_coeff(md, kc, cn, dpw, m->dDerivKp, terms, X, st));
        if (op.kind == EighOp::kVelocity)
            LAUNCH(7, st, launch_band_velocity(md.n, dim, cn, E, V, X, op.degen_tol, O, m->wsV, st));
        if (op.kind == EighOp::kCurvature) {
            LAUNCH(7, st, launch_berry_product(md.n, dim, cn, V, X, terms, op.convention == 1, md.pos, Y, st));
            LAUNCH(7, st, launch_berry_curvature(md.n, dim, cn, E, X, terms, op.degen_tol, O, m->wsV, st));
        }
        if (int rc = unscale(m, E, cn * md.n, st)) return rc;
        if (op.kind == EighOp::kVelocity)
            if (int rc = unscale(m, O, cn * (long)width, st)) return rc;
    }
    return TBK_OK;
}

// Order this call's use of the handle's scratch behind the previous call's (possibly on another stream).
int scratch_acquire(tbk_model* m, cudaStream_t st) {
    if (!m->ev_busy) CU(cudaEventCreateWithFlags(&m->ev_busy, cudaEventDisableTiming));
    if (m->busy_recorded) CU(cudaStreamWaitEvent(st, m->ev_busy, 0));
    return TBK_OK;
}

int scratch_release(tbk_model* m, cudaStream_t st) {
    CU(cudaEventRecord(m->ev_busy, st));
    m->busy_recorded = true;
    return TBK_OK;
}

int ensure_pipeline(tbk_model* m, size_t kbytes, size_t obytes) {
    if (!m->s_in) {
        CU(cudaStreamCreateWithFlags(&m->s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&m->s_comp, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&m->s_out, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            CU(cudaEventCreateWithFlags(&m->ev_in[b], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&m->ev_comp[b], cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&m->ev_out[b], cudaEventDisableTiming));
        }
    }
    if (kbytes > m->hk_bytes) {
        for (int b = 0; b < 2; ++b) {
            if (m->hk[b]) cudaFree(m->hk[b]);
            m->hk[b] = nullptr;
        }
        m->hk_bytes = 0;
        for (int b = 0; b < 2; ++b) CU(cudaMalloc(&m->hk[b], kbytes));
        m->hk_bytes = kbytes;
    }
    if (obytes > m->ho_bytes) {
        for (int b = 0; b < 2; ++b) {
            if (m->ho[b]) cudaFree(m->ho[b]);
            m->ho[b] = nullptr;
        }
        m->ho_bytes = 0;
        for (int b = 0; b < 2; ++b) CU(cudaMalloc(&m->ho[b], obytes));
        m->ho_bytes = obytes;
    }
    return TBK_OK;
}

// Chunked, double-buffered host pipeline shared by the two _host entry points.
// out_per_k: doubles written per k-point (n for eigenval, 2 n^2 for hamilton).
int run_host(tbk_model* m, const double* k_host, long nk, double* out_host, int convention /*0 = eigenval*/) {
    NvtxRange nvtx_call_("tbk:host_pipeline (H2D | kernels | D2H)");
    const ModelDev& md = m->md;
    if (nk <= 0) return TBK_OK;
    const size_t out_per_k = convention ? (size_t)2 * md.n * md.n : (size_t)md.n;
    const size_t bytes_per_k = ((size_t)md.dim + out_per_k) * 8;
    const size_t target_mb = (size_t)md.tune.host_chunk_mb;
    long hchunk = (long)((target_mb << 20) / bytes_per_k);
    if (hchunk < 1) hchunk = 1;
    if (hchunk >= 1024) hchunk &= ~127L;
    if (!md.small_ok) {  // whole workspace chunks per host chunk: no ragged (partial-wave) last launch in every group
        const long wchunk = pick_chunk(m);
        if (hchunk > wchunk) hchunk -= hchunk % wchunk;
    }
    if (hchunk > nk) hchunk = nk;
    if (int rc = ensure_pipeline(m, (size_t)hchunk * md.dim * 8, (size_t)hchunk * out_per_k * 8)) return rc;
    if (int rc = scratch_acquire(m, m->s_comp)) return rc;

    int it = 0;
    for (long c0 = 0; c0 < nk; c0 += hchunk, ++it) {
        const long cn = std::min(hchunk, nk - c0);
        const int b = it & 1;
        if (it >= 2) {
            CU(cudaStreamWaitEvent(m->s_in, m->ev_comp[b], 0));   // kernels of chunk it-2 consumed hk[b]
            CU(cudaStreamWaitEvent(m->s_comp, m->ev_out[b], 0));  // D2H of chunk it-2 drained ho[b]
        }
        CU(cudaMemcpyAsync(m->hk[b], k_host + c0 * md.dim, (size_t)cn * md.dim * 8, cudaMemcpyHostToDevice, m->s_in));
        CU(cudaEventRecord(m->ev_in[b], m->s_in));
        CU(cudaStreamWaitEvent(m->s_comp, m->ev_in[b], 0));
        int rc = convention ? run_hamilton(m, m->hk[b], cn, convention, m->ho[b], m->s_comp)
                            : run_eigenval(m, m->hk[b], cn, m->ho[b], m->s_comp);
        if (rc) return rc;
        CU(cudaEventRecord(m->ev_comp[b], m->s_comp));
        CU(cudaStreamWaitEvent(m->s_out, m->ev_comp[b], 0));
        CU(cudaMemcpyAsync(out_host + (size_t)c0 * out_per_k, m->ho[b], (size_t)cn * out_per_k * 8,
                           cudaMemcpyDeviceToHost, m->s_out));
        CU(cudaEventRecord(m->ev_out[b], m->s_out));
    }
    if (int rc = scratch_release(m, m->s_comp)) return rc;
    CU(cudaStreamSynchronize(m->s_in));
    CU(cudaStreamSynchronize(m->s_comp));
    CU(cudaStreamSynchronize(m->s_out));
    return TBK_OK;
}

// Regular mesh with a HOST result buffer: lines are evaluated in host-chunk sized groups into two device buffers whose
// D2H copies overlap the next group's kernels (the pipeline of run_host without the H2D leg: a mesh has no k array).
int run_mesh_host(tbk_model* m, const int64_t* dims, const double* shift, long line0, long n_lines, double* out_host) {
    NvtxRange nvtx_call_("tbk:mesh_host_pipeline (kernels | D2H)");
    const ModelDev& md = m->md;
    const long nz = (long)dims[md.dim - 1];
    if (n_lines <= 0 || nz <= 0) return TBK_OK;
    const size_t line_bytes = (size_t)nz * md.n * 8;
    long hl = (long)(((size_t)md.tune.host_chunk_mb << 20) / line_bytes);
    if (hl < 1) hl = 1;
    const long lchunk = std::max<long>(1, pick_chunk(m) / nz);  // whole workspace chunks per group: no ragged last launch
    if (hl > lchunk) hl -= hl % lchunk;
    if (hl > n_lines) hl = n_lines;
    if (int rc = ensure_pipeline(m, 0, (size_t)hl * line_bytes)) return rc;
    if (int rc = scratch_acquire(m, m->s_comp)) return rc;
    int it = 0;
    for (long l0 = 0; l0 < n_lines; l0 += hl, ++it) {
        const long ln = std::min(hl, n_lines - l0);
        const int b = it & 1;
        if (it >= 2) CU(cudaStreamWaitEvent(m->s_comp, m->ev_out[b], 0));  // D2H of group it-2 drained ho[b]
        if (int rc = run_eigenval_mesh(m, dims, shift, line0 + l0, ln, m->ho[b], m->s_comp)) return rc;
        CU(cudaEventRecord(m->ev_comp[b], m->s_comp));
        CU(cudaStreamWaitEvent(m->s_out, m->ev_comp[b], 0));
        CU(cudaMemcpyAsync(out_host + (size_t)l0 * nz * md.n, m->ho[b], (size_t)ln * line_bytes, cudaMemcpyDeviceToHost, m->s_out));
        CU(cudaEventRecord(m->ev_out[b], m->s_out));
    }
    if (int rc = scratch_release(m, m->s_comp)) return rc;
    CU(cudaStreamSynchronize(m->s_comp));
    CU(cudaStreamSynchronize(m->s_out));
    return TBK_OK;
}

int check_fail_flag(tbk_model* m) {
    int h = 0;
    CU(cudaMemcpy(&h, m->dFail, sizeof(int), cudaMemcpyDeviceToHost));
    if (h != 0) {
        cudaMemset(m->dFail, 0, sizeof(int));
        return fail(TBK_E_NOCONV, "tridiagonal QL did not converge for %d eigenvalue(s)", h);
    }
    return TBK_OK;
}

// The vector _host entry points (eigh, band velocities, Berry curvature, k.p coefficients): k [nk][dim] from the host
// through device staging buffers of one host chunk, run(dk, cn, d0, d1) on s_comp, then w0 (w1) doubles per k-point
// back into out0 (out1), one host chunk at a time.  A host chunk that holds several of the op's device chunks (dchunk)
// holds a whole number of them, so the batch is split where the device entry point splits it.  check_ql: report a QL
// failure of this call (eigh-based ops only; the flag is not set by the k.p kernel).
template <class Run>
int run_staged(tbk_model* m, const double* k_host, long nk, long dchunk, size_t w0, double* out0, size_t w1, double* out1,
               bool check_ql, Run run) {
    if (nk <= 0) return TBK_OK;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = ensure_pipeline(m, 0, 0)) return rc;
    const ModelDev& md = m->md;
    long hchunk = std::max<long>(1, (long)(((size_t)md.tune.host_chunk_mb << 20) / ((md.dim + w0 + w1) * 8)));
    if (hchunk > dchunk) hchunk -= hchunk % dchunk;
    hchunk = std::min(hchunk, nk);
    const size_t kb = (size_t)hchunk * md.dim * 8, b0 = (size_t)hchunk * w0 * 8, b1 = (size_t)hchunk * w1 * 8;
    double *dk = nullptr, *d0 = nullptr, *d1 = nullptr;
    cudaError_t e = cudaMalloc(&dk, kb);
    if (e == cudaSuccess) e = cudaMalloc(&d0, b0);
    if (e == cudaSuccess && b1) e = cudaMalloc(&d1, b1);
    int rc = e == cudaSuccess ? scratch_acquire(m, m->s_comp)
                              : fail(TBK_E_CUDA, "host staging: cannot allocate %zu bytes of device buffers", kb + b0 + b1);
    for (long c0 = 0; !rc && c0 < nk; c0 += hchunk) {
        const long cn = std::min(hchunk, nk - c0);
        e = cudaMemcpyAsync(dk, k_host + c0 * md.dim, (size_t)cn * md.dim * 8, cudaMemcpyHostToDevice, m->s_comp);
        if (e == cudaSuccess) rc = run(dk, cn, d0, d1);
        if (!rc && e == cudaSuccess)
            e = cudaMemcpyAsync(out0 + c0 * w0, d0, (size_t)cn * w0 * 8, cudaMemcpyDeviceToHost, m->s_comp);
        if (!rc && e == cudaSuccess && b1)
            e = cudaMemcpyAsync(out1 + c0 * w1, d1, (size_t)cn * w1 * 8, cudaMemcpyDeviceToHost, m->s_comp);
        if (!rc && e == cudaSuccess) e = cudaStreamSynchronize(m->s_comp);
        if (!rc && e != cudaSuccess) rc = fail(TBK_E_CUDA, "host staging: %s", cudaGetErrorString(e));
    }
    if (!rc) rc = scratch_release(m, m->s_comp);
    cudaStreamSynchronize(m->s_comp);
    cudaFree(dk);
    cudaFree(d0);
    cudaFree(d1);
    if (rc || !check_ql) return rc;
    return check_fail_flag(m);
}

// run_eigh through run_staged: eigenvalues into eig_host, the op's second result into out_host.
int run_eigh_host(tbk_model* m, const double* k_host, long nk, const EighOp& op, double* eig_host, double* out_host) {
    return run_staged(m, k_host, nk, eigh_chunk(m, op, pick_chunk(m)), m->md.n, eig_host, eigh_out_doubles(m, op),
                      out_host, true, [&](const double* dk, long cn, double* de, double* dout) {
                          return run_eigh(m, dk, cn, op, de, dout, m->s_comp);
                      });
}

}  // namespace

extern "C" {

int tbk_version(void) { return 103; }

const char* tbk_last_error(void) { return g_err.c_str(); }

int tbk_model_create(int dim, int n_orb, int n_R, const int32_t* R, const double* hop, const double* pos, int device,
                     tbk_model** out) {
    if (!out) return fail(TBK_E_INVALID, "tbk_model_create: out is null");
    *out = nullptr;
    if (n_orb < 1) return fail(TBK_E_INVALID, "tbk_model_create: n_orb = %d must be >= 1", n_orb);
    if (dim < 1) return fail(TBK_E_INVALID, "tbk_model_create: dim = %d must be >= 1", dim);
    if (dim > kMaxDim) return fail(TBK_E_UNSUPPORTED, "tbk_model_create: dim = %d > %d is not supported", dim, kMaxDim);
    if (n_R < 0 || (n_R > 0 && (!R || !hop))) return fail(TBK_E_INVALID, "tbk_model_create: bad hopping arrays");
    if (!pos) return fail(TBK_E_INVALID, "tbk_model_create: pos is null");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(TBK_E_CUDA, "tbk_model_create: no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(TBK_E_INVALID, "tbk_model_create: device %d out of range", device);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(TBK_E_CUDA, "tbk_model_create: cudaSetDevice(%d) failed", device);

    NvtxRange nvtx_call_("tbk:model_create (pack + upload)");
    tbk_model* m = new (std::nothrow) tbk_model();
    if (!m) return fail(TBK_E_INVALID, "out of host memory");
    m->device = device;
    m->scale_exp = normalise_exponent(coupling_bound(n_orb, n_R, hop));
    std::vector<double> hop_scaled;
    hop = scaled_copy(hop, (size_t)n_R * n_orb * n_orb * 2, m->scale_exp, hop_scaled);
    ModelDev& md = m->md;
    md.tune = read_tuning();
    md.n = n_orb;
    md.dim = dim;
    md.nR = n_R;
    md.nRpad = (n_R + 7) & ~7;
    const long NN = (long)n_orb * n_orb;

    auto bail = [&](int rc) {
        tbk_model_destroy(m);
        return rc;
    };
#define CUB(call)                                                                                             \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return bail(fail(TBK_E_CUDA, "%s -> %s", #call, cudaGetErrorString(e_)));      \
    } while (0)

    // R as doubles, padded with zero vectors
    std::vector<double> Rd((size_t)std::max(md.nRpad, 1) * dim, 0.0);
    for (int r = 0; r < n_R; ++r)
        for (int d = 0; d < dim; ++d) Rd[(size_t)r * dim + d] = (double)R[(size_t)r * dim + d];
    CUB(cudaMalloc(&m->dRd, Rd.size() * 8));
    CUB(cudaMemcpy(m->dRd, Rd.data(), Rd.size() * 8, cudaMemcpyHostToDevice));
    md.Rd = m->dRd;
    m->model_bytes += Rd.size() * 8;

    CUB(cudaMalloc(&m->dPos, (size_t)n_orb * dim * 8));
    CUB(cudaMemcpy(m->dPos, pos, (size_t)n_orb * dim * 8, cudaMemcpyHostToDevice));
    md.pos = m->dPos;
    m->model_bytes += (size_t)n_orb * dim * 8;

    CUB(cudaMalloc(&m->dFail, sizeof(int)));
    CUB(cudaMemset(m->dFail, 0, sizeof(int)));

    std::vector<double> W((size_t)std::max(2 * n_R, 1) * NN, 0.0);
    pack_weights_host(n_orb, n_R, hop, W.data());

    md.small_ok = (n_orb <= kSmallMaxN && hk_small_smem_bytes(n_orb, dim, n_R, 0) <= 220 * 1024) ? 1 : 0;
    if (getenv("TBK_FORCE_GEMM")) md.small_ok = 0;  // test hook: exercise the general path on small models
    if (md.small_ok) {
        CUB(cudaMalloc(&m->dW, W.size() * 8));
        CUB(cudaMemcpy(m->dW, W.data(), W.size() * 8, cudaMemcpyHostToDevice));
        md.W = m->dW;
        m->model_bytes += W.size() * 8;
        std::vector<int> Ri((size_t)std::max(n_R, 1), 0);
        for (int r = 0; r < n_R; ++r) {
            bool unit = true;
            for (int d = 0; d < dim; ++d) {
                const int v = R[(size_t)r * dim + d];
                if (v < -1 || v > 1) unit = false;
            }
            Ri[r] = unit ? 1 : 0;
            if (unit) md.use_z = 1;
        }
        // trigonometric-product table (hk_small.cu, hk_basis_kernel): N <= 2, dim <= 3, every R in {-1, 0, 1}^dim
        bool all_unit = true;
        for (int r = 0; r < n_R; ++r) all_unit = all_unit && Ri[r] == 1;
        if (n_orb <= 2 && dim <= 3 && all_unit && !getenv("TBK_NO_BASIS")) {
            int nb3 = 1;
            for (int d = 0; d < dim; ++d) nb3 *= 3;
            std::vector<double> cre((size_t)nb3), cim((size_t)nb3), tre((size_t)nb3), tim((size_t)nb3);
            for (int r = 0; r < n_R; ++r) {
                // expand prod_d (c_d + i R_d s_d) into the 3^dim products: complex coefficient per basis function
                std::fill(cre.begin(), cre.end(), 0.0);
                std::fill(cim.begin(), cim.end(), 0.0);
                cre[0] = 1.0;
                int stride3 = 1;
                for (int d = 0; d < dim; ++d, stride3 *= 3) {
                    const int v = R[(size_t)r * dim + d];
                    if (v == 0) continue;
                    std::fill(tre.begin(), tre.end(), 0.0);
                    std::fill(tim.begin(), tim.end(), 0.0);
                    for (int b = 0; b < stride3; ++b) {  // only dimensions < d have been expanded so far
                        tre[b + stride3] += cre[b];            // * c_d
                        tim[b + stride3] += cim[b];
                        tre[b + 2 * stride3] += -v * cim[b];   // * i v s_d
                        tim[b + 2 * stride3] += v * cre[b];
                    }
                    cre.swap(tre);
                    cim.swap(tim);
                }
                for (int b = 0; b < nb3; ++b)
                    for (long e = 0; e < NN; ++e)
                        md.basis[(size_t)b * NN + e] +=
                            cre[b] * W[(size_t)(2 * r) * NN + e] + cim[b] * W[(size_t)(2 * r + 1) * NN + e];
            }
            md.basis_ok = 1;
        }
        CUB(cudaMalloc(&m->dRi, Ri.size() * sizeof(int)));
        CUB(cudaMemcpy(m->dRi, Ri.data(), Ri.size() * sizeof(int), cudaMemcpyHostToDevice));
        md.Ri = m->dRi;
    } else {
        if (int rc = upload_gemm_weights(m, W, 2 * n_R)) return bail(rc);
        if (int rc = prepare_hk_i8(m)) return bail(rc);
        if (int rc = setup_mesh_classes(m, R, n_R)) return bail(rc);
    }
#undef CUB
    *out = m;
    return TBK_OK;
}

int tbk_supercell_create(int dim, int n_orb, int n_R, const int32_t* R, const double* hop, const double* pos,
                         const int32_t* size, int device, tbk_model** out) {
    if (!out) return fail(TBK_E_INVALID, "tbk_supercell_create: out is null");
    *out = nullptr;
    if (n_orb < 1 || dim < 1) return fail(TBK_E_INVALID, "tbk_supercell_create: bad sizes");
    if (dim > kMaxDim) return fail(TBK_E_UNSUPPORTED, "tbk_supercell_create: dim = %d > %d is not supported", dim, kMaxDim);
    if (n_R < 0 || (n_R > 0 && (!R || !hop)) || !pos || !size) return fail(TBK_E_INVALID, "tbk_supercell_create: bad arrays");
    long vol = 1;
    for (int d = 0; d < dim; ++d) {
        if (size[d] < 1) return fail(TBK_E_INVALID, "tbk_supercell_create: size[%d] = %d must be >= 1", d, size[d]);
        vol *= size[d];
        if (vol > 4096) return fail(TBK_E_UNSUPPORTED, "tbk_supercell_create: more than 4096 cells");
    }
    const long N = (long)n_orb * vol;
    if (N > 8192) return fail(TBK_E_UNSUPPORTED, "tbk_supercell_create: %ld orbitals (limit 8192)", N);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(TBK_E_CUDA, "tbk_supercell_create: no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(TBK_E_INVALID, "tbk_supercell_create: device %d out of range", device);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(TBK_E_CUDA, "tbk_supercell_create: cudaSetDevice(%d) failed", device);

    // ---- host: enumerate the blocks (reference :1687-1710) and fold onto the half set (:281-298) ----
    struct Raw {
        int q, a, b, r, herm;
        double scale;
    };
    std::vector<std::vector<int>> keys;  // folded lattice vectors in order of first appearance
    auto key_index = [&](const std::vector<int>& key) {
        for (size_t i = 0; i < keys.size(); ++i)
            if (keys[i] == key) return (int)i;
        keys.push_back(key);
        return (int)keys.size() - 1;
    };
    std::vector<long> mult((size_t)dim, 1);  // cell index = sum_d offset_d * prod_{e > d} size_e (itertools.product order)
    for (int d = dim - 2; d >= 0; --d) mult[d] = mult[d + 1] * size[d + 1];
    std::vector<Raw> raws;
    std::vector<int> off((size_t)dim), newR((size_t)dim);
    // pass 1 in the reference's loop order (cells outermost) so that the folded keys appear in the same order as in
    // Model(hop=new_hop, contains_cc=False): first the order of raw keys, then their folded images
    std::vector<std::vector<int>> raw_keys;
    for (long a = 0; a < vol; ++a) {
        long rem = a;
        for (int d = 0; d < dim; ++d) {
            off[d] = (int)(rem / mult[d]);
            rem %= mult[d];
        }
        for (int r = 0; r < n_R; ++r) {
            for (int d = 0; d < dim; ++d) {
                const int full = off[d] + R[(size_t)r * dim + d];
                int q = full / size[d];
                if (full % size[d] < 0) --q;  // floor division
                newR[d] = q;
            }
            bool seen = false;
            for (const auto& k : raw_keys) seen = seen || k == newR;
            if (!seen) raw_keys.push_back(newR);
        }
    }
    for (const auto& k : raw_keys) {
        int first = 0;
        for (int d = 0; d < dim && first == 0; ++d) first = k[d];
        std::vector<int> key(k);
        if (first < 0)
            for (int& x : key) x = -x;
        key_index(key);
    }
    for (long a = 0; a < vol; ++a) {
        long rem = a;
        for (int d = 0; d < dim; ++d) {
            off[d] = (int)(rem / mult[d]);
            rem %= mult[d];
        }
        for (int r = 0; r < n_R; ++r) {
            long b = 0;
            int first = 0;
            for (int d = 0; d < dim; ++d) {
                const int full = off[d] + R[(size_t)r * dim + d];
                int q = full / size[d], md_ = full % size[d];
                if (md_ < 0) {
                    --q;
                    md_ += size[d];
                }
                newR[d] = q;
                b += md_ * mult[d];
                if (first == 0) first = q;
            }
            std::vector<int> key(newR);
            if (first < 0)
                for (int& x : key) x = -x;
            const int q = key_index(key);
            if (first == 0) {  // R' = 0: 0.5 X + 0.5 X^H
                raws.push_back({q, (int)a, (int)b, r, 0, 0.5});
                raws.push_back({q, (int)b, (int)a, r, 1, 0.5});
            } else if (first > 0) raws.push_back({q, (int)a, (int)b, r, 0, 1.0});
            else raws.push_back({q, (int)b, (int)a, r, 1, 1.0});
        }
    }
    const int nq = (int)keys.size();
    if ((size_t)nq * vol * vol > (size_t)1 << 26) return fail(TBK_E_UNSUPPORTED, "tbk_supercell_create: block table too large");
    std::stable_sort(raws.begin(), raws.end(), [&](const Raw& x, const Raw& y) {
        if (x.q != y.q) return x.q < y.q;
        if (x.a != y.a) return x.a < y.a;
        return x.b < y.b;
    });
    std::vector<int2> table((size_t)std::max(nq, 1) * vol * vol, make_int2(0, 0));
    std::vector<SupEntry> entries(std::max<size_t>(raws.size(), 1));
    for (size_t i = 0; i < raws.size(); ++i) {
        entries[i] = {raws[i].r, raws[i].herm, raws[i].scale};
        int2& t = table[((size_t)raws[i].q * vol + raws[i].a) * vol + raws[i].b];
        if (t.y == 0) t.x = (int)i;
        t.y += 1;
    }

    tbk_model* m = new (std::nothrow) tbk_model();
    if (!m) return fail(TBK_E_INVALID, "out of host memory");
    m->device = device;
    // the supercell's bound is at most the base model's: every supercell element sums a subset of the base terms
    m->scale_exp = normalise_exponent(coupling_bound(n_orb, n_R, hop));
    std::vector<double> hop_scaled;
    hop = scaled_copy(hop, (size_t)n_R * n_orb * n_orb * 2, m->scale_exp, hop_scaled);
    ModelDev& md = m->md;
    md.tune = read_tuning();
    md.n = (int)N;
    md.dim = dim;
    md.nR = nq;
    md.nRpad = (nq + 7) & ~7;
    md.small_ok = 0;
    auto bail = [&](int rc) {
        tbk_model_destroy(m);
        return rc;
    };
#define CUB(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return bail(fail(TBK_E_CUDA, "%s -> %s", #call, cudaGetErrorString(e_))); \
    } while (0)
    std::vector<double> Rd((size_t)std::max(md.nRpad, 1) * dim, 0.0);
    std::vector<int32_t> Rn((size_t)std::max(nq, 1) * dim, 0);
    for (int q = 0; q < nq; ++q)
        for (int d = 0; d < dim; ++d) {
            Rd[(size_t)q * dim + d] = (double)keys[q][d];
            Rn[(size_t)q * dim + d] = keys[q][d];
        }
    CUB(cudaMalloc(&m->dRd, Rd.size() * 8));
    CUB(cudaMemcpy(m->dRd, Rd.data(), Rd.size() * 8, cudaMemcpyHostToDevice));
    md.Rd = m->dRd;
    // positions normalised to the supercell (reference :1670-1678): cell offsets outermost
    std::vector<double> npos((size_t)N * dim);
    for (long a = 0; a < vol; ++a) {
        long rem = a;
        for (int d = 0; d < dim; ++d) {
            off[d] = (int)(rem / mult[d]);
            rem %= mult[d];
        }
        for (int i = 0; i < n_orb; ++i)
            for (int d = 0; d < dim; ++d)
                npos[((size_t)a * n_orb + i) * dim + d] = pos[(size_t)i * dim + d] / (double)size[d] + (double)off[d] / (double)size[d];
    }
    CUB(cudaMalloc(&m->dPos, npos.size() * 8));
    CUB(cudaMemcpy(m->dPos, npos.data(), npos.size() * 8, cudaMemcpyHostToDevice));
    md.pos = m->dPos;
    CUB(cudaMalloc(&m->dFail, sizeof(int)));
    CUB(cudaMemset(m->dFail, 0, sizeof(int)));

    // ---- device: gather the Hermitian-split weights straight into the GEMM stage tiles ----
    choose_gemm_tiling(md, 2 * nq);
    const int bn = 16 * md.na;
    const size_t stage = (size_t)kGemmKC * (bn + 4);
    const size_t n_stages = (size_t)std::max(md.n_tiles * md.kchunks, 1);
    CUB(cudaMalloc(&m->dWt, n_stages * stage * 8));
    CUB(cudaMemset(m->dWt, 0, n_stages * stage * 8));
    md.Wt = m->dWt;
    m->model_bytes += n_stages * stage * 8;
    double* d_hop = nullptr;
    int2* d_table = nullptr;
    SupEntry* d_entries = nullptr;
    unsigned char* d_flags = nullptr;
    auto drop_tmp = [&]() {
        cudaFree(d_hop);
        cudaFree(d_table);
        cudaFree(d_entries);
        cudaFree(d_flags);
    };
    std::vector<unsigned char> nz(n_stages, 0);
    cudaError_t e = cudaMalloc(&d_hop, std::max<size_t>((size_t)n_R * n_orb * n_orb * 16, 16));
    if (e == cudaSuccess) e = cudaMalloc(&d_table, table.size() * sizeof(int2));
    if (e == cudaSuccess) e = cudaMalloc(&d_entries, entries.size() * sizeof(SupEntry));
    if (e == cudaSuccess) e = cudaMalloc(&d_flags, n_stages);
    if (e == cudaSuccess && n_R > 0) e = cudaMemcpy(d_hop, hop, (size_t)n_R * n_orb * n_orb * 16, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_table, table.data(), table.size() * sizeof(int2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d_entries, entries.data(), entries.size() * sizeof(SupEntry), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_supercell_pack(n_orb, (int)vol, nq, bn, md.kchunks, d_hop, d_table, d_entries, m->dWt, nullptr);
    if (e == cudaSuccess) e = launch_stage_flags(m->dWt, (long)n_stages, (int)stage, d_flags, nullptr);
    if (e == cudaSuccess) e = cudaMemcpy(nz.data(), d_flags, n_stages, cudaMemcpyDeviceToHost);
    drop_tmp();
    if (e != cudaSuccess) return bail(fail(TBK_E_CUDA, "tbk_supercell_create: %s", cudaGetErrorString(e)));
    m->launches += 2;
    if (int rc = upload_stage_lists(m, nz)) return bail(rc);
    if (int rc = prepare_hk_i8(m)) return bail(rc);
    if (int rc = setup_mesh_classes(m, Rn.data(), nq)) return bail(rc);
#undef CUB
    *out = m;
    return TBK_OK;
}

int tbk_model_vectors(const tbk_model* m, int32_t* R_out) {
    if (!m || !R_out) return fail(TBK_E_INVALID, "tbk_model_vectors: null argument");
    if (m->md.kind != 0) return fail(TBK_E_INVALID, "tbk_model_vectors: the handle is a k.p model");
    DeviceGuard guard(m->device);
    std::vector<double> Rd((size_t)std::max(m->md.nR, 1) * m->md.dim);
    if (m->md.nR > 0) CU(cudaMemcpy(Rd.data(), m->md.Rd, (size_t)m->md.nR * m->md.dim * 8, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < (size_t)m->md.nR * m->md.dim; ++i) R_out[i] = (int32_t)Rd[i];
    return TBK_OK;
}

int tbk_kdotp_create(int dim, int n_orb, int n_terms, const int32_t* powers, const double* coeff, int device,
                     tbk_model** out) {
    if (!out) return fail(TBK_E_INVALID, "tbk_kdotp_create: out is null");
    *out = nullptr;
    if (n_orb < 1 || dim < 1) return fail(TBK_E_INVALID, "tbk_kdotp_create: bad sizes");
    if (dim > kMaxDim) return fail(TBK_E_UNSUPPORTED, "tbk_kdotp_create: dim = %d > %d is not supported", dim, kMaxDim);
    if (n_terms < 0 || (n_terms > 0 && (!powers || !coeff))) return fail(TBK_E_INVALID, "tbk_kdotp_create: bad arrays");
    for (long i = 0; i < (long)n_terms * dim; ++i)
        if (powers[i] < 0 || powers[i] > 64) return fail(TBK_E_INVALID, "tbk_kdotp_create: powers must be in [0, 64]");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(TBK_E_CUDA, "tbk_kdotp_create: no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(TBK_E_INVALID, "tbk_kdotp_create: device %d out of range", device);
    DeviceGuard guard(device);
    if (!guard.ok) return fail(TBK_E_CUDA, "tbk_kdotp_create: cudaSetDevice(%d) failed", device);
    tbk_model* m = new (std::nothrow) tbk_model();
    if (!m) return fail(TBK_E_INVALID, "out of host memory");
    m->device = device;
    m->scale_exp = normalise_exponent(coupling_bound(n_orb, n_terms, coeff));
    std::vector<double> coeff_scaled;
    coeff = scaled_copy(coeff, (size_t)n_terms * n_orb * n_orb * 2, m->scale_exp, coeff_scaled);
    ModelDev& md = m->md;
    md.tune = read_tuning();
    md.n = n_orb;
    md.dim = dim;
    md.nR = n_terms;
    md.kind = 1;
    md.small_ok = 0;
    auto bail = [&](int rc) {
        tbk_model_destroy(m);
        return rc;
    };
#define CUB(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) return bail(fail(TBK_E_CUDA, "%s -> %s", #call, cudaGetErrorString(e_))); \
    } while (0)
    const long NN = (long)n_orb * n_orb;
    std::vector<double> W((size_t)std::max(n_terms, 1) * NN, 0.0);
    pack_hermitian_rows_host(n_orb, n_terms, coeff, W.data());
    if (int rc = upload_gemm_weights(m, W, n_terms)) return bail(rc);
    std::vector<int> Pw((size_t)std::max(md.kchunks, 1) * kGemmKC * dim, 0);
    for (long i = 0; i < (long)n_terms * dim; ++i) Pw[i] = powers[i];
    CUB(cudaMalloc(&m->dPw, Pw.size() * sizeof(int)));
    CUB(cudaMemcpy(m->dPw, Pw.data(), Pw.size() * sizeof(int), cudaMemcpyHostToDevice));
    md.Pw = m->dPw;
    std::vector<double> zeros((size_t)n_orb * dim, 0.0);
    CUB(cudaMalloc(&m->dPos, zeros.size() * 8));
    CUB(cudaMemcpy(m->dPos, zeros.data(), zeros.size() * 8, cudaMemcpyHostToDevice));
    md.pos = m->dPos;
    CUB(cudaMalloc(&m->dFail, sizeof(int)));
    CUB(cudaMemset(m->dFail, 0, sizeof(int)));
#undef CUB
    *out = m;
    return TBK_OK;
}

int tbk_model_destroy(tbk_model* m) {
    if (!m) return TBK_OK;
    DeviceGuard guard(m->device);
    cudaDeviceSynchronize();
    cudaFree(m->dRd);
    cudaFree(m->dW);
    cudaFree(m->dRi);
    cudaFree(m->dPw);
    cudaFree(m->dWt);
    cudaFree(m->dPos);
    cudaFree(m->dFail);
    cudaFree(m->dKcCnt);
    cudaFree(m->dKcIdx);
    cudaFree(m->dWd);
    cudaFree(m->dWsc);
    cudaFree(m->wsH);
    cudaFree(m->wsE);
    cudaFree(m->wsQ);
    cudaFree(m->dRc);
    cudaFree(m->dZc);
    cudaFree(m->wsAB);
    cudaFree(m->wsQz);
    cudaFree(m->wsK);
    cudaFree(m->wsKp);
    cudaFree(m->dDerivKp);
    cudaFree(m->wsVel);
    cudaFree(m->wsV);
    for (int b = 0; b < 2; ++b) {
        cudaFree(m->hk[b]);
        cudaFree(m->ho[b]);
        if (m->ev_in[b]) cudaEventDestroy(m->ev_in[b]);
        if (m->ev_comp[b]) cudaEventDestroy(m->ev_comp[b]);
        if (m->ev_out[b]) cudaEventDestroy(m->ev_out[b]);
    }
    if (m->ev_busy) cudaEventDestroy(m->ev_busy);
    for (int b = 0; b < 2; ++b) {
        if (m->ev_td[b]) cudaEventDestroy(m->ev_td[b]);
        if (m->ev_ql[b]) cudaEventDestroy(m->ev_ql[b]);
    }
    if (m->s_ql) cudaStreamDestroy(m->s_ql);
    cudaFree(m->wsE2);
    cudaFree(m->wsB);
    cudaFree(m->wsEg);
    cudaFree(m->dCounter);
    if (m->ev_chunk) cudaEventDestroy(m->ev_chunk);
    if (m->ev_push) cudaEventDestroy(m->ev_push);
    if (m->s_push) cudaStreamDestroy(m->s_push);
    if (m->s_in) cudaStreamDestroy(m->s_in);
    if (m->s_comp) cudaStreamDestroy(m->s_comp);
    if (m->s_out) cudaStreamDestroy(m->s_out);
    delete m;
    return TBK_OK;
}

int tbk_model_info(const tbk_model* m, int* n_orb, int* dim, int* n_R, int* path) {
    if (!m) return fail(TBK_E_INVALID, "tbk_model_info: null handle");
    if (n_orb) *n_orb = m->md.n;
    if (dim) *dim = m->md.dim;
    if (n_R) *n_R = m->md.nR;
    if (path) *path = m->md.small_ok ? (m->md.basis_ok ? 2 : 0) : 1;
    return TBK_OK;
}

int tbk_hamilton(tbk_model* m, const double* k_dev, int64_t n_k, int convention, double* out_dev, void* stream) {
    if (!m) return fail(TBK_E_INVALID, "tbk_hamilton: null handle");
    if (convention != 1 && convention != 2)
        return fail(TBK_E_INVALID, "Invalid value '%d' for 'convention': must be either '1' or '2'", convention);
    if (n_k < 0 || (n_k > 0 && (!k_dev || !out_dev))) return fail(TBK_E_INVALID, "tbk_hamilton: bad buffers");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_hamilton(m, k_dev, (long)n_k, convention, out_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_eigenval(tbk_model* m, const double* k_dev, int64_t n_k, double* out_dev, void* stream) {
    if (!m) return fail(TBK_E_INVALID, "tbk_eigenval: null handle");
    if (n_k < 0 || (n_k > 0 && (!k_dev || !out_dev))) return fail(TBK_E_INVALID, "tbk_eigenval: bad buffers");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_eigenval(m, k_dev, (long)n_k, out_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_eigenval_push(tbk_model* m, const double* k_dev, int64_t n_k, double* out_dev, void* const* peer_bases, int n_peers,
                      int64_t row_offset, void* stream) {
    if (!m) return fail(TBK_E_INVALID, "tbk_eigenval_push: null handle");
    if (n_k < 0 || (n_k > 0 && (!k_dev || !out_dev))) return fail(TBK_E_INVALID, "tbk_eigenval_push: bad buffers");
    if (n_peers < 0 || n_peers > 15 || (n_peers > 0 && !peer_bases) || row_offset < 0)
        return fail(TBK_E_INVALID, "tbk_eigenval_push: bad peer list (0 .. 15 peers)");
    for (int p = 0; p < n_peers; ++p)
        if (!peer_bases[p]) return fail(TBK_E_INVALID, "tbk_eigenval_push: peer %d has a null base pointer", p);
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!m->s_push) CU(cudaStreamCreateWithFlags(&m->s_push, cudaStreamNonBlocking));
    if (!m->ev_chunk) CU(cudaEventCreateWithFlags(&m->ev_chunk, cudaEventDisableTiming));
    if (!m->ev_push) CU(cudaEventCreateWithFlags(&m->ev_push, cudaEventDisableTiming));
    if (int rc = scratch_acquire(m, st)) return rc;
    PushPlan plan;
    plan.bases = reinterpret_cast<double* const*>(peer_bases);
    plan.n = n_peers;
    plan.row_offset = (long)row_offset;
    if (int rc = run_eigenval(m, k_dev, (long)n_k, out_dev, st, n_peers > 0 ? &plan : nullptr)) return rc;
    if (n_peers > 0 && n_k > 0) {  // the caller's stream continues only after the last peer store was issued and done
        CU(cudaEventRecord(m->ev_push, m->s_push));
        CU(cudaStreamWaitEvent(st, m->ev_push, 0));
    }
    return scratch_release(m, st);
}

static int mesh_args_ok(const tbk_model* m, const int64_t* dims, int64_t first_line, int64_t n_lines, const void* out,
                        const char* who) {
    if (!m) return fail(TBK_E_INVALID, "%s: null handle", who);
    if (!dims) return fail(TBK_E_INVALID, "%s: dims is null", who);
    int64_t lines = 1;
    for (int d = 0; d < m->md.dim; ++d) {
        if (dims[d] < 1) return fail(TBK_E_INVALID, "%s: dims[%d] = %lld must be >= 1", who, d, (long long)dims[d]);
        if (d < m->md.dim - 1) lines *= dims[d];
    }
    if (first_line < 0 || n_lines < 0 || first_line + n_lines > lines)
        return fail(TBK_E_INVALID, "%s: lines [%lld, %lld) outside the mesh (%lld lines)", who, (long long)first_line,
                    (long long)(first_line + n_lines), (long long)lines);
    if (n_lines > 0 && !out) return fail(TBK_E_INVALID, "%s: bad buffers", who);
    return TBK_OK;
}

int tbk_eigenval_mesh(tbk_model* m, const int64_t* dims, const double* shift, int64_t first_line, int64_t n_lines,
                      double* out_dev, void* stream) {
    if (int rc = mesh_args_ok(m, dims, first_line, n_lines, out_dev, "tbk_eigenval_mesh")) return rc;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_eigenval_mesh(m, dims, shift, (long)first_line, (long)n_lines, out_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_eigenval_mesh_host(tbk_model* m, const int64_t* dims, const double* shift, int64_t first_line, int64_t n_lines,
                           double* out_host) {
    if (int rc = mesh_args_ok(m, dims, first_line, n_lines, out_host, "tbk_eigenval_mesh_host")) return rc;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = run_mesh_host(m, dims, shift, (long)first_line, (long)n_lines, out_host)) return rc;
    return check_fail_flag(m);
}

int tbk_mesh_factorised(const tbk_model* m, const int64_t* dims) {
    if (!m || !dims) return 0;
    return mesh_factorised(m, dims) ? 1 : 0;
}

int tbk_eigh(tbk_model* m, const double* k_dev, int64_t n_k, double* eig_dev, double* vec_dev, void* stream) {
    if (!m) return fail(TBK_E_INVALID, "tbk_eigh: null handle");
    if (n_k < 0 || (n_k > 0 && (!k_dev || !eig_dev || !vec_dev))) return fail(TBK_E_INVALID, "tbk_eigh: bad buffers");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_eigh(m, k_dev, (long)n_k, EighOp{}, eig_dev, vec_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_eigh_host(tbk_model* m, const double* k_host, int64_t n_k, double* eig_host, double* vec_host) {
    if (!m) return fail(TBK_E_INVALID, "tbk_eigh_host: null handle");
    if (n_k < 0 || (n_k > 0 && (!k_host || !eig_host || !vec_host))) return fail(TBK_E_INVALID, "tbk_eigh_host: bad buffers");
    return run_eigh_host(m, k_host, (long)n_k, EighOp{}, eig_host, vec_host);
}

// Arguments of the band velocity (op.kind == kVelocity) and Berry curvature entry points.
static int band_args_ok(tbk_model* m, const void* k, int64_t n_k, const EighOp& op, const void* eig, const void* out,
                        const char* who) {
    const bool curv = op.kind == EighOp::kCurvature;
    if (!m) return fail(TBK_E_INVALID, "%s: null handle", who);
    if (m->md.kind != 0)
        return fail(TBK_E_INVALID, "%s: the handle is a k.p model (%s defined for Model handles)", who,
                    curv ? "Berry curvature is" : "band velocities are");
    if (curv && op.convention != 1 && op.convention != 2)
        return fail(TBK_E_INVALID, "%s: convention must be 1 or 2 (got %d)", who, op.convention);
    if (!(op.degen_tol >= 0.0)) return fail(TBK_E_INVALID, "%s: degen_tol must be >= 0 (got %g)", who, op.degen_tol);
    if (curv && m->md.dim < 2) return fail(TBK_E_INVALID, "%s: a %d-dimensional model has no Berry curvature", who, m->md.dim);
    if (n_k < 0 || (n_k > 0 && (!k || !eig || !out))) return fail(TBK_E_INVALID, "%s: bad buffers", who);
    if ((size_t)2 * m->md.nR * 8 > 200 * 1024) return fail(TBK_E_UNSUPPORTED, "%s: %d stored R vectors (limit 12800)", who, m->md.nR);
    return TBK_OK;
}

int tbk_band_velocity(tbk_model* m, const double* k_dev, int64_t n_k, double degen_tol, double* eig_dev, double* vel_dev,
                      void* stream) {
    const EighOp op{EighOp::kVelocity, 0, degen_tol};
    if (int rc = band_args_ok(m, k_dev, n_k, op, eig_dev, vel_dev, "tbk_band_velocity")) return rc;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_eigh(m, k_dev, (long)n_k, op, eig_dev, vel_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_band_velocity_host(tbk_model* m, const double* k_host, int64_t n_k, double degen_tol, double* eig_host,
                           double* vel_host) {
    const EighOp op{EighOp::kVelocity, 0, degen_tol};
    if (int rc = band_args_ok(m, k_host, n_k, op, eig_host, vel_host, "tbk_band_velocity_host")) return rc;
    return run_eigh_host(m, k_host, (long)n_k, op, eig_host, vel_host);
}

int tbk_berry_curvature(tbk_model* m, const double* k_dev, int64_t n_k, int convention, double degen_tol, double* eig_dev,
                        double* curv_dev, void* stream) {
    const EighOp op{EighOp::kCurvature, convention, degen_tol};
    if (int rc = band_args_ok(m, k_dev, n_k, op, eig_dev, curv_dev, "tbk_berry_curvature")) return rc;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_eigh(m, k_dev, (long)n_k, op, eig_dev, curv_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_berry_curvature_host(tbk_model* m, const double* k_host, int64_t n_k, int convention, double degen_tol,
                             double* eig_host, double* curv_host) {
    const EighOp op{EighOp::kCurvature, convention, degen_tol};
    if (int rc = band_args_ok(m, k_host, n_k, op, eig_host, curv_host, "tbk_berry_curvature_host")) return rc;
    return run_eigh_host(m, k_host, (long)n_k, op, eig_host, curv_host);
}

static int kdotp_args_ok(tbk_model* m, const void* k, int64_t n_k, const int32_t* powers, int n_terms, const void* out,
                         const char* who) {
    if (!m) return fail(TBK_E_INVALID, "%s: null handle", who);
    if (m->md.kind != 0) return fail(TBK_E_INVALID, "%s: the handle is a k.p model (construct_kdotp is a Model method)", who);
    if (n_k < 0 || n_terms < 0 || (n_k > 0 && n_terms > 0 && (!k || !out || !powers)))
        return fail(TBK_E_INVALID, "%s: bad buffers", who);
    if (n_terms > 65535) return fail(TBK_E_UNSUPPORTED, "%s: %d Taylor terms (limit 65535)", who, n_terms);
    if ((size_t)2 * m->md.nR * 8 > 200 * 1024) return fail(TBK_E_UNSUPPORTED, "%s: %d stored R vectors (limit 12800)", who, m->md.nR);
    for (long i = 0; i < (long)n_terms * m->md.dim; ++i)
        if (powers[i] < 0 || powers[i] > 64) return fail(TBK_E_INVALID, "%s: powers must be in [0, 64]", who);
    return TBK_OK;
}

int tbk_kdotp_coefficients(tbk_model* m, const double* k_dev, int64_t n_k, const int32_t* powers, int n_terms,
                           double* out_dev, void* stream) {
    if (int rc = kdotp_args_ok(m, k_dev, n_k, powers, n_terms, out_dev, "tbk_kdotp_coefficients")) return rc;
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = scratch_acquire(m, (cudaStream_t)stream)) return rc;
    if (int rc = run_kdotp_coeff(m, k_dev, (long)n_k, powers, n_terms, out_dev, (cudaStream_t)stream)) return rc;
    return scratch_release(m, (cudaStream_t)stream);
}

int tbk_kdotp_coefficients_host(tbk_model* m, const double* k_host, int64_t n_k, const int32_t* powers, int n_terms,
                                double* out_host) {
    if (int rc = kdotp_args_ok(m, k_host, n_k, powers, n_terms, out_host, "tbk_kdotp_coefficients_host")) return rc;
    if (n_terms == 0) return TBK_OK;
    return run_staged(m, k_host, (long)n_k, kKdotpLaunchK, (size_t)n_terms * m->md.n * m->md.n * 2, out_host, 0, nullptr,
                      false, [&](const double* dk, long cn, double* dout, double*) {
                          return run_kdotp_coeff(m, dk, cn, powers, n_terms, dout, m->s_comp);
                      });
}

int tbk_hamilton_host(tbk_model* m, const double* k_host, int64_t n_k, int convention, double* out_host) {
    if (!m) return fail(TBK_E_INVALID, "tbk_hamilton_host: null handle");
    if (convention != 1 && convention != 2)
        return fail(TBK_E_INVALID, "Invalid value '%d' for 'convention': must be either '1' or '2'", convention);
    if (n_k < 0 || (n_k > 0 && (!k_host || !out_host))) return fail(TBK_E_INVALID, "tbk_hamilton_host: bad buffers");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    return run_host(m, k_host, (long)n_k, out_host, convention);
}

int tbk_eigenval_host(tbk_model* m, const double* k_host, int64_t n_k, double* out_host) {
    if (!m) return fail(TBK_E_INVALID, "tbk_eigenval_host: null handle");
    if (n_k < 0 || (n_k > 0 && (!k_host || !out_host))) return fail(TBK_E_INVALID, "tbk_eigenval_host: bad buffers");
    DeviceGuard guard(m->device);
    if (!guard.ok) return fail(TBK_E_CUDA, "cudaSetDevice(%d) failed", m->device);
    if (int rc = run_host(m, k_host, (long)n_k, out_host, 0)) return rc;
    return check_fail_flag(m);
}

int tbk_model_check(tbk_model* m) {
    if (!m) return fail(TBK_E_INVALID, "tbk_model_check: null handle");
    DeviceGuard guard(m->device);
    CU(cudaDeviceSynchronize());
    return check_fail_flag(m);
}

int64_t tbk_launch_count(const tbk_model* m) { return m ? m->launches : 0; }

int tbk_profile(tbk_model* m, int enable) {
    if (!m) return fail(TBK_E_INVALID, "tbk_profile: null handle");
    m->prof_on = enable != 0;
    return TBK_OK;
}

int tbk_profile_read(tbk_model* m, double* ms, int64_t* count) {
    if (!m) return fail(TBK_E_INVALID, "tbk_profile_read: null handle");
    DeviceGuard guard(m->device);
    CU(cudaDeviceSynchronize());
    for (auto& r : m->prof) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) {
            m->prof_ms[r.cls] += t;
            m->prof_n[r.cls] += 1;
        }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    m->prof.clear();
    for (int i = 0; i < TBK_PROFILE_CLASSES; ++i) {
        if (ms) ms[i] = m->prof_ms[i];
        if (count) count[i] = m->prof_n[i];
        m->prof_ms[i] = 0.0;
        m->prof_n[i] = 0;
    }
    return TBK_OK;
}

int64_t tbk_workspace_bytes(const tbk_model* m) {
    return m ? (int64_t)(m->ws_bytes + 2 * m->hk_bytes + 2 * m->ho_bytes + m->model_bytes) : 0;
}

int tbk_host_alloc(void** p, size_t bytes) {
    if (!p) return fail(TBK_E_INVALID, "tbk_host_alloc: null");
    CU(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
    return TBK_OK;
}

int tbk_host_free(void* p) {
    if (p) CU(cudaFreeHost(p));
    return TBK_OK;
}

double tbk_measure_fp64_peak(int kind, int iters) { return measure_fp64_peak(kind, iters); }
double tbk_measure_int8_peak(int64_t iters) { return measure_int8_peak((long)iters); }

int tbk_host_tridiag_ql(int n, double* d, double* e) { return tridiag_ql(n, d, e, 1); }

int tbk_host_sincospi(double t, double* s, double* c) {
    sincospi_lean(t, *s, *c);
    return TBK_OK;
}

int tbk_host_tridiag_bisect(int n, double* d, const double* e) {
    if (n < 1) return fail(TBK_E_INVALID, "n < 1");
    std::vector<double> dd(d, d + n), e2((size_t)n, 0.0);
    double lo = 1e300, hi = -1e300, emax = 0.0;
    for (int i = 0; i < n; ++i) {
        const double el = i > 0 ? fabs(e[i - 1]) : 0.0, er = i + 1 < n ? fabs(e[i]) : 0.0;
        e2[i] = er * er;
        lo = std::min(lo, dd[i] - el - er);
        hi = std::max(hi, dd[i] + el + er);
        emax = std::max(emax, er * er);
    }
    const double pivmin = DBL_MIN * std::max(1.0, emax);
    const double span = std::max(fabs(lo), fabs(hi));
    const double gl = lo - 2.0 * DBL_EPSILON * span * n - 2.0 * pivmin, gu = hi + 2.0 * DBL_EPSILON * span * n + 2.0 * pivmin;
    for (int i = 0; i < n; ++i) d[i] = bisect_eig(n, dd.data(), e2.data(), i, gl, gu, pivmin);
    return TBK_OK;
}

int tbk_host_hetrd(int n, double* hp, double* d, double* e) {
    if (n < 1) return fail(TBK_E_INVALID, "n < 1");
    std::vector<double> wv((size_t)4 * n);
    hetrd_serial(n, hp, 1, d, e, 1, wv.data());
    e[n - 1] = 0.0;
    return TBK_OK;
}

int tbk_host_pack_weights(int n_orb, int n_R, const double* hop, double* W) {
    if (n_orb < 1 || n_R < 0) return fail(TBK_E_INVALID, "bad sizes");
    pack_weights_host(n_orb, n_R, hop, W);
    return TBK_OK;
}

}  // extern "C"
