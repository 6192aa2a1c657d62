// Internal declarations shared by the translation units of libpigp.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <string>
#include <vector>

#include "../../include/pigp.h"

namespace pigp {

constexpr int TILE = PIGP_TILE;        // 128: padding unit and GEMM tile
constexpr int ASM_TR = 64;             // assembly tile rows (a multiple of 16; 128 must be a multiple of it)
constexpr int ASM_TC = 128;            // assembly tile cols
constexpr int MAX_THETA = PIGP_MAX_GROUPS * 4 + 1;  // 16 kernel hyper-parameters + noise

void set_error(const std::string& msg);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define PIGP_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            pigp::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                \
            return PIGP_ECUDA;                                                                  \
        }                                                                                       \
    } while (0)

#define PIGP_TRY(expr)                 \
    do {                               \
        int _rc = (expr);              \
        if (_rc != PIGP_OK) return _rc; \
    } while (0)

// ---- optional per-class event timing (pigp_profile_start / _stop)
enum { PROF_ASSEMBLE = 0, PROF_GEMM = 1, PROF_POTF2 = 2, PROF_GRAD = 3, PROF_MISC = 4 };
extern bool g_prof_on;
void prof_push(int cls, cudaStream_t st, bool begin, double flops);
void prof_note(int m, int n, int k, int mode);  // shape of the next record (written to $PIGP_PROF_DUMP by pigp_profile_stop)
struct ProfScope {
    int cls; cudaStream_t st; bool on;
    ProfScope(int c, cudaStream_t s, double flops = 0.0) : cls(c), st(s), on(g_prof_on) { if (on) prof_push(cls, st, true, flops); }
    ~ProfScope() { if (on) prof_push(cls, st, false, 0.0); }
};

// Force-load a kernel (CUDA loads kernels lazily on first launch, and that load can block behind a spinning flag wait
// of another rank that shares the process): every kernel is touched once when a multi-rank solver is created.
#define PIGP_PRELOAD(f)                                        \
    do {                                                       \
        cudaFuncAttributes _a;                                 \
        PIGP_CUDA(cudaFuncGetAttributes(&_a, f));              \
    } while (0)
int preload_dense();
int set_potf2_debug(long long* dev_buf);  // 17 clock64 stamps of the next k_potf2 launches (nullptr: off)
int preload_assemble();

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// One rectangle of the output matrix, evaluated by one CTA of the assembly / gradient kernels.
struct AsmTile {
    int32_t row0, col0;    // output coordinates of the tile origin
    int32_t nrows, ncols;  // extent (<= ASM_TR x ASM_TC)
    int32_t desc;          // block descriptor index, -1 = zero fill (Kzero or padding)
    int32_t flags;         // ASM_* bits
};
enum {
    ASM_SWAP = 1,   // first kernel argument is the COLUMN point (lower half of an upper-table block)
    ASM_LOWER = 2,  // write / weigh only entries with row >= col
    ASM_PAD = 4,    // padding region: zero, 1.0 on the diagonal
    ASM_MIRROR = 8, // also store the strictly-lower entries transposed (full layout of a symmetric matrix)
    ASM_DIAG = 16,  // store only the diagonal entries (R == C), to K[R]: the diagonal of a symmetric matrix as a vector
};

}  // namespace pigp

struct pigp_plan {
    int dim = 0, product_form = 1, n_groups = 0, symmetric = 0;
    int kernel_type = 0;  // 0 squared exponential; 52 / 72 / 92 Matern
    int n_row_blocks = 0, n_col_blocks = 0;
    std::vector<int64_t> sec_row, sec_col;
    int64_t rows = 0, cols = 0;
    double lbox[3] = {0, 0, 0};
    int noise_lo_block = -1, noise_hi_block = -1;
    int64_t noise_lo = 0, noise_hi = 0;  // row range carrying exp(noise)
    int theta_len = 0;                   // incl. noise
    int device = 0;
    std::vector<pigp_block_desc> table;  // host copy, n_row_blocks x n_col_blocks
    // device state
    double* d_pts_row = nullptr;  // [dim][rows] (structure of arrays)
    double* d_pts_col = nullptr;  // [dim][cols]; == d_pts_row when symmetric
    pigp_block_desc* d_table = nullptr;
    pigp::AsmTile* d_tiles_full = nullptr;
    int64_t n_tiles_full = 0;
    pigp::AsmTile* d_tiles_lower = nullptr;  // symmetric plans only
    int64_t n_tiles_lower = 0;
    pigp::AsmTile* d_tiles_diag = nullptr;   // symmetric plans only: the diagonal as a vector
    int64_t n_tiles_diag = 0;
    double* d_khost = nullptr;               // staging of pigp_assemble_host (grow-only)
    size_t d_khost_bytes = 0;
    double* d_theta_stage = nullptr;  // MAX_THETA doubles, for the _host entry points
    double* h_pin = nullptr;          // pinned staging
    int64_t h_pin_bytes = 0;
};

namespace pigp {

// ---- arguments shared by the block evaluators (pigp_assemble.cu: squared exponential; pigp_matern.cu: Matern)
struct AsmArgs {
    const AsmTile* tiles;
    const pigp_block_desc* table;
    const double* pts_row;  // [DIM][n_row_pts]
    const double* pts_col;  // [DIM][n_col_pts]
    int64_t n_row_pts, n_col_pts;
    const double* theta;
    int n_groups;
    int has_noise;      // theta[n_groups*(1+DIM)] is the noise parameter
    int64_t noise_lo, noise_hi;
    double eps;
    int add_diag;
    double lbox[3];
    double* K;          // assembly output
    int64_t ld;
    // gradient-only
    const double* X;    // K^-1, lower triangle
    const double* alpha;
    double* partials;   // [n_tiles][MAX_THETA]
    // batch: nb slots share the points and the tile list; slot b = blockIdx.y reads and writes its pointers offset by b times
    // these strides (0: shared by every slot)
    int nb;
    int64_t s_theta, s_K, s_X, s_alpha, s_partials;
};

AsmArgs make_args(const pigp_plan* p, const AsmTile* tiles, const double* theta, double eps, int add_diag);
int launch_blocks_matern(const pigp_plan* p, const AsmArgs& a, int64_t n_tiles, bool grad, cudaStream_t st);
int preload_matern();

#ifdef __CUDACC__
__device__ __forceinline__ double diag_addon(const AsmArgs& a, int64_t R, double noise_exp) {
    // GP/gp.py:23-42 (_add_jiggle) and :44-70 (_add_jiggle_noise)
    if (!a.has_noise) return a.eps;
    if (R < a.noise_lo) return 1.0;
    if (R < a.noise_hi) return noise_exp;
    return a.eps;
}

// the slot's pointers (once, at kernel entry).  The evaluators are instantiated twice, with and without this: the single-slot
// kernels stay exactly as register-tight as they were (several run at their register cap)
__device__ __forceinline__ void slot_args(AsmArgs& a) {
    const int64_t b = blockIdx.y;
    a.theta += b * a.s_theta;
    a.K += b * a.s_K;
    a.X += b * a.s_X;
    a.alpha += b * a.s_alpha;
    a.partials += b * a.s_partials;
}

#endif

// ---- assembly / gradient (pigp_assemble.cu).  The trailing nb and strides batch a launch over nb slots (one more grid
// dimension): slot b reads theta_dev + b * s_theta and writes K + b * s_K, and so on.
int launch_assemble(const pigp_plan* p, const AsmTile* tiles, int64_t n_tiles, const double* theta_dev, double eps,
                    int add_diag, double* K, int64_t ld, cudaStream_t st, int nb = 1, int64_t s_theta = 0, int64_t s_K = 0);
// zero-fill + unit diagonal for rows/cols outside the plan's extent, up to rows_pad x cols_pad
int launch_pad(double* K, int64_t ld, int64_t rows, int64_t cols, int64_t rows_pad, int64_t cols_pad, int unit_diag,
               int lower_only, cudaStream_t st, int nb = 1, int64_t s_K = 0);
// partials[n_tiles_lower][MAX_THETA] <- per-tile sums of (X - alpha alpha^T) * dK/dtheta ; then reduce into grad
// (slot b: grad_out + b * s_grad)
int launch_grad(const pigp_plan* p, const AsmTile* tiles, int64_t n_tiles, const double* theta_dev, const double* X, int64_t ld,
                const double* alpha, double* partials, double* grad_out, cudaStream_t st, int nb = 1, int64_t s_theta = 0,
                int64_t s_X = 0, int64_t s_alpha = 0, int64_t s_partials = 0, int64_t s_grad = 0);
// lower-triangle tiles of a symmetric plan whose 128-row tile belongs to `rank` (tile t -> rank t mod world); tiles never
// straddle a 128-row boundary
void build_lower_tiles_owned(const pigp_plan* p, int rank, int world, std::vector<AsmTile>& out);

// ---- the matrix the tile Cholesky of pigp_dist.cu factors in place, and what the posterior driver reads of a (world = 1)
// solver's factor after an NLL evaluation
struct FactorView {
    double* L;       // K -> lower Cholesky factor, row-major, leading dimension ld
    int64_t ld;
    int T;           // row tiles of the matrix proper (npad / 128)
    int end;         // one past the last row tile that rides through the panel TRSMs and trailing updates (>= T)
    double* invd;    // T inverse diagonal tiles
    int32_t* info;   // first failing pivot (may be null)
    int rank, world; // 128-row tile t belongs to rank t mod world
    double* v;       // L^-1 y (npad entries; zeros beyond n): solver only
    // batch (world = 1): nb matrices factored by the same launches; slot b's L (and v) at + b * sL, its invd at + b * sI,
    // its info at + b
    int nb;
    int64_t sL, sI;
    // first own tile >= a
    int first_own(int a) const { return a + ((rank - a) % world + world) % world; }
    int count_own(int a, int b) const { const int f = first_own(a); return f < b ? (b - f + world - 1) / world : 0; }
};
FactorView factor_view(pigp_dsolver* s);
// pigp_nll_grad_batch on the solver's world = 1 block-cyclic solver (pigp_dist.cu): nb slots, one pass of the schedule
int dsolver_nll_grad_batch(pigp_dsolver* s, int nb, const double* thetas_dev, const double* y_dev, double eps, double* nll_dev,
                           double* grad_dev, int32_t* info_dev, void* stream);

// ---- dense linear algebra (pigp_dense.cu)
struct GemmDesc {
    int M, N, K;
    double alpha, beta;
    const double* A; int64_t lda; int a_kcontig;
    const double* B; int64_t ldb; int b_kcontig;
    double* C; int64_t ldc;
    int lower_only;  // skip tiles with tn > tm
    int kmode;       // 0: all k; 1: k_tile >= m_tile; 2: k_tile <= m_tile
    // ---- generalised addressing (block-cyclic row tiles; zero-initialised = plain GEMM)
    int gen;         // 1: rectangular tile raster with the predicates below evaluated on GLOBAL tile indices
    int m_ts;        // row tile tm lives at rows tm * m_ts * 128 of A and C (0 is read as 1)
    int m_gt0;       // global tile index of row tile 0:  gm = m_gt0 + tm * m_ts
    int n_gt0;       // global tile index (128 units) of column 0 of C
    int k_gt0;       // global tile index of k = 0 (kmode 1: k_tile >= gm, kmode 2: k_tile <= gm, in global tiles)
    int force_bn128; // one CTA per 128 x 128 tile (required when C aliases A: the CTA reads its rows before it writes them)
    // ---- triangular solve by the inverse diagonal tile with one step of iterative refinement (N = K = 128, in place):
    //      X0 = A W^T;  X = X0 + (A - X0 Lkk^T) W^T   with B = W = inv(Lkk).  |W Lkk - I| grows like n u cond(Lkk)
    //      (1e-8 for the eps = 1e-6 Stokes matrices); the refinement step brings the panel back to substitution quality.
    const double* Lkk; int64_t ldl;
    // ---- stores mirrored into peer memory (NVLink P2P) for row tiles with gm < push_gm_end
    int npeers;
    int push_gm_end;
    double* Cpeer[7];  // the address of C[0][0] in each peer's buffer (same ldc)
    // ---- flag wait fused into the prologue: every CTA waits until flags[wait_idx0 + t * wait_stride] >= wait_val for
    // t in [0, wait_count), t != wait_skip (bounded spin; *wait_err is set on time-out)
    const unsigned long long* wait_flags;
    int wait_idx0, wait_stride, wait_count, wait_skip;
    unsigned long long wait_val;
    unsigned long long wait_timeout_ns;
    int* wait_err;
    // ---- flag signal fused into the epilogue: the last of sig_total CTAs stores sig_val to the sig_n peer flags
    // (small-tile kernel only; sig_total must equal the number of CTAs that reach the epilogue)
    unsigned int* sig_counter;
    int sig_total, sig_n;
    unsigned long long sig_val;
    unsigned long long* sig_flag[7];
    // ---- batch: nb (0 is read as 1) independent products of this shape in one launch (grid dimension y = slot); slot b
    //      works on A + b * sa, B + b * sb, C + b * sc and Lkk + b * sl.  Every choice of kernel variant is made from the
    //      shape of one slot, so a slot's result does not depend on nb.
    int nb;
    int64_t sa, sb, sc, sl;
};
int launch_gemm(const GemmDesc& g, cudaStream_t st);
// factor one 128 x 128 diagonal tile in place; invd receives the four diagonal 32 x 32 blocks of inv(L) only
// (nb slots: A + b * sA, invd + b * sI, info + b)
int launch_potf2(double* A, int64_t ld, double* invd, int32_t* info, int base, cudaStream_t st, int nb = 1, int64_t sA = 0,
                 int64_t sI = 0);
// complete the inverse tiles c = first + i * stride (i < count) from L_cc and their diagonal blocks; Y != nullptr: also
// write inv(L_cc)^T into the diagonal tile c of Y (row stride ldy).  nb slots: L + b * sL, invd + b * sI, Y + b * sY
int launch_tile_inv(const double* L, int64_t ld, double* invd, int first, int stride, int count, double* Y, int64_t ldy, cudaStream_t st,
                    int zero_upper = 0, int nb = 1, int64_t sL = 0, int64_t sI = 0, int64_t sY = 0);
// pigp_potrf_lower (pigp_dist.cu: the solver's factorisation over the caller's buffer)
int potrf_lower(double* A, int64_t ld, int64_t n, int64_t m_extra, double* invd, int32_t* info, cudaStream_t st);
int potri_lower(const double* L, int64_t ld, int64_t n, const double* invd, double* W, double* X, cudaStream_t st);
// out[0] = sum_{i<n} log A[i*ld+i]; out[1] = sum_{j<n} v[j]^2  (nb slots: A + b * sA, v + b * sv, out2 + 2 b)
int launch_logdet_quad(const double* A, int64_t ld, int64_t n, const double* v, double* out2, cudaStream_t st, int nb = 1,
                       int64_t sA = 0, int64_t sv = 0);
// y[i] = sum_j A[i*ld+j] x[j], A (m x n) row-major
int launch_gemv(const double* A, int64_t ld, int64_t m, int64_t n, const double* x, double* y, cudaStream_t st);

}  // namespace pigp
