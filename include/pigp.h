/*
 * pigp.h -- C ABI of the B200-native PIGP hot path (libpigp.so).
 *
 * Drop-in boundary for the covariance-assembly -> Cholesky -> NLL / dK/dtheta
 * trace gradient -> posterior path of ogaken1104/stopro.  Every entry point
 * names the reference interface it replaces (paths relative to the reference
 * tree).  Plain pointers and sizes only; no torch / JAX types.  All functions
 * return 0 on success and a negative PIGP_E* code on failure; the message is
 * available from pigp_last_error() (thread local).  Nothing throws or aborts
 * across the ABI.  Work is enqueued on the caller's stream (a cudaStream_t
 * passed as void*, NULL = default stream); "_dev" pointers are device memory,
 * "_host" pointers are host memory.  Functions whose name ends in _host copy
 * their inputs to the device and their results back, and synchronise the
 * stream before returning; the others never synchronise.
 *
 * Threads: the device-pointer entry points (pigp_assemble, pigp_assemble_diag, and the test building blocks
 * pigp_assemble_owned and pigp_trace_grad, whose tile lists and partial sums are stream-ordered allocations on the
 * caller's stream) only read a plan, so one plan may serve
 * several threads / streams at once.  pigp_plan_set_points_host and every _host entry point use staging buffers owned by
 * the plan or the solver and are NOT thread-safe per handle.  A solver (pigp_solver / pigp_dsolver) owns its workspace and
 * must be used by one thread at a time -- use one solver per thread / stream.  Every entry point switches the calling
 * thread to the device its plan was created on (cudaSetDevice).  pigp_last_error() is thread local.  The measurement aids (pigp_profile_*, pigp_set_side_stream,
 * pigp_debug_*) are process-global switches for single-threaded benchmarks.
 *
 * Environment knobs read once at first use (tuning / debugging only; defaults are the measured-best settings):
 *   PIGP_GEMM_BN=128      one 128 x 128 CTA per SM instead of two 128 x 64 CTAs
 *   PIGP_GEMM_SMALL=0     disable the small-tile GEMM for latency-bound launches
 *   PIGP_SIDE_CHUNK=<t>   issue the side stream's products in k-chunks of t tiles
 *   PIGP_FUSE_WAITS=1     spin on the DIAG flag inside the consuming TRSM instead of a one-CTA wait kernel
 *   PIGP_PROF_DUMP=<csv>  per-launch timeline written by pigp_profile_stop
 *   PIGP_LOOKAHEAD=<W>    panel schedule with look-ahead, W tile columns per panel (see pigp_set_lookahead)
 *   PIGP_EARLY_KINV=0     compute K^-1 = Y Y^T in one product at the end instead of accumulating it from finished column ranges
 *                         of Y underneath the factorisation (single GPU, 8..32 tiles; costs one more N^2 buffer)
 *   PIGP_WAIT_TIMEOUT_S / PIGP_BARRIER_TIMEOUT_S   flag-wait limits of the multi-GPU path (see pigp_dsolver_reset)
 */
#ifndef PIGP_H
#define PIGP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIGP_ABI_VERSION 3
#define PIGP_MAX_TERMS 8   /* monomials per block (3-D Kfzfz needs 7) */
#define PIGP_MAX_GROUPS 4  /* hyper-parameter groups per model (ux, uy, uz, pp); a block may use all of them */
#define PIGP_TILE 128      /* row/column padding unit of every factorisation buffer */
#define PIGP_MAX_BATCH 65535 /* hyper-parameter vectors of one batched evaluation / starts of one multi-start Adam run */

enum {
    PIGP_OK = 0,
    PIGP_EINVAL = -1,   /* bad argument */
    PIGP_ECUDA = -2,    /* CUDA runtime error (message in pigp_last_error) */
    PIGP_ENOMEM = -3,
    PIGP_ENOTPD = -4    /* informational: a non-positive pivot was met; results are NaN like the reference's */
};

/* One monomial of a block:  coef * gamma_g * prod_d G_{order[d]}(r_d - r'_d ; l_{g,d}),
 * G_n = (d/ds)^n exp(-s^2 / (2 l^2)), sum_d order[d] <= 4.  Additive kernel form (k = gamma sum_d E_d,
 * GP/kernels.py:57-61): exactly one order[d] >= 0 per term (the dimension the term lives on), -1 elsewhere.  Replaces the nested jax.grad / jax.hessian
 * operators of GP/gp_2D.py:16-86, GP/gp_3D.py:12-35, GP/gp_1D_laplacian.py:35-46. */
typedef struct {
    int32_t group;     /* theta offset of the group = group * (1 + dim): [log gamma, log l_0 ..] (sub_modules/init_modules.py:5-54) */
    int32_t order[3];
    double coef;
} pigp_term;

/* One block function K_AB(r, r') of GP/gp_2D_stokes_independent.py:22-246 /
 * GP/gp_3D_stokes_independent.py:25-239.  Terms must be sorted by group.
 * shift_first / shift_second are the periodic-difference wrappers of GP/gp.py:374-410
 * (setup_kernel_include_difference: first argument; ..._prime: second argument; difdif: both). */
typedef struct {
    int32_t n_terms;       /* 0 = the reference's Kzero block */
    int32_t shift_first;
    int32_t shift_second;
    int32_t reserved;
    pigp_term terms[PIGP_MAX_TERMS];
} pigp_block_desc;

/* A block-structured covariance matrix: what GPmodel.set_constants (GP/gp.py:263-285) fixes
 * (sec_tr / sec_te, the jitter rule) together with the class's trainingKs / mixedKs / testKs
 * table (e.g. GP/gp_poiseuille_independent.py:21-42). */
typedef struct {
    int32_t dim;            /* 1, 2 or 3 */
    int32_t product_form;   /* 1: k = gamma prod_d E_d (kernels.py:64-77); 0: additive, gamma sum_d E_d (kernels.py:57-61) */
    int32_t n_groups;
    int32_t symmetric;      /* 1: rows == cols (training / test matrix, GP/gp.py:122-189); 0: rectangular (GP/gp.py:191-211) */
    int32_t n_row_blocks;
    int32_t n_col_blocks;   /* ignored when symmetric */
    const int64_t* sec_row; /* n_row_blocks + 1 offsets (GP/gp.py:258-261 calc_sec) */
    const int64_t* sec_col; /* ignored when symmetric */
    const double* pts_row_host; /* [sec_row[last]][dim] row-major; first kernel argument */
    const double* pts_col_host; /* second kernel argument; ignored when symmetric */
    const pigp_block_desc* table; /* n_row_blocks x n_col_blocks row-major; symmetric plans read entries (i, j >= i) only,
                                     first argument = block i points, second = block j points, as Ks[i][j-i] in GP/gp.py:140 */
    double lbox[3];         /* periodic shift vector (self.lbox) */
    int32_t noise_lo_block; /* index_optimize_noise[0], or -1: plain jitter (GP/gp.py:23-42) */
    int32_t noise_hi_block; /* index_optimize_noise[-1]: diagonal add-on is 1 before the range, exp(noise) inside, eps after (GP/gp.py:44-70) */
    int32_t kernel_type;    /* params_model["kernel_type"] (GP/kernels.py:331-427): PIGP_KERNEL_SE, or PIGP_KERNEL_MT52 / _MT72 /
                               _MT92 = the Matern kernels of GP/kernels.py:127-205, G_n then being the n-th derivative of
                               q(rho) exp(-rho), rho = kappa |s| / l, with the reference's autodiff value 0 at s = 0 for n >= 1 */
    int32_t reserved;
} pigp_plan_desc;
enum { PIGP_KERNEL_SE = 0, PIGP_KERNEL_MT52 = 52, PIGP_KERNEL_MT72 = 72, PIGP_KERNEL_MT92 = 92 };

typedef struct pigp_plan pigp_plan;
typedef struct pigp_solver pigp_solver;

enum { PIGP_LAYOUT_FULL = 0, PIGP_LAYOUT_LOWER = 1 };

int pigp_abi_version(void);
const char* pigp_last_error(void);

/* Device selection for everything created afterwards by this thread (cudaSetDevice). */
int pigp_set_device(int device);

/* --- plans ------------------------------------------------------------------------------- */
int pigp_plan_create(const pigp_plan_desc* desc, pigp_plan** out);
void pigp_plan_destroy(pigp_plan* plan);
int64_t pigp_plan_rows(const pigp_plan* plan);
int64_t pigp_plan_cols(const pigp_plan* plan);
int32_t pigp_plan_theta_len(const pigp_plan* plan); /* n_groups*(1+dim) (+1 when noise is optimised) */
/* Replace the coordinates (same block sizes); side 0 = rows / first argument, 1 = columns.  The points are transposed
 * into the plan's pinned staging buffer, copied on `stream`, and the stream is synchronised before returning (the staging
 * buffer is reused by the next call). */
int pigp_plan_set_points_host(pigp_plan* plan, int side, const double* pts_host, void* stream);

/* trainingK_all / mixedK_all / testK_all (GP/gp.py:287-306): K_dev[row * ld + col], row-major.
 * add_diag != 0 also applies add_eps_to_sigma (GP/gp.py:23-70) -- symmetric plans only. */
int pigp_assemble(const pigp_plan* plan, const double* theta_dev, double eps, int add_diag,
                  double* K_dev, int64_t ld, int layout, void* stream);
int pigp_assemble_host(pigp_plan* plan, const double* theta_host, double eps, int add_diag,
                       double* K_host, int layout);
/* Only the diagonal of a symmetric plan's matrix, diag_dev[rows]: what the callers of predictingFunction_all consume
 * (std = sqrt(diag(Sigma_post)), test/test_1_sinusoidal_direct_main.py:144) -- M kernel values instead of M x M. */
int pigp_assemble_diag(const pigp_plan* plan, const double* theta_dev, double eps, int add_diag, double* diag_dev, void* stream);

/* --- solver: factorisation workspace bound to a training plan ----------------------------- */
int pigp_solver_create(pigp_plan* training_plan, pigp_solver** out);
void pigp_solver_destroy(pigp_solver* s);
/* The same handle over a K dealt block-cyclically over `world` GPUs (see the multi-GPU section below): every rank creates
 * one, wires the peers through the borrowed pigp_dsolver handle (pigp_dsolver_ipc_handle / _connect) and then all ranks
 * issue the same sequence of pigp_nll / pigp_nll_grad / pigp_predict calls.  After a factorisation every rank holds the
 * whole factor, so pigp_predict may be given a different (disjoint) set of test points on every rank. */
typedef struct pigp_dsolver pigp_dsolver;
int pigp_solver_create_dist(pigp_plan* training_plan, int rank, int world, pigp_solver** out);
pigp_dsolver* pigp_solver_dsolver(pigp_solver* s);

/* trainingFunction_all (GP/gp.py:213-224, logpGP :72-89): NLL = 0.5 |L^-1 y|^2 + sum log L_ii + 0.5 n log 2pi.
 * out_dev[0] = NLL.  info_dev (may be NULL): 0, the 1-based index of the first non-positive pivot, or -1 when a peer's flag
 * never arrived (multi-GPU only). */
int pigp_nll(pigp_solver* s, const double* theta_dev, const double* y_dev, double eps,
             double* out_dev, int32_t* info_dev, void* stream);
/* NLL and d_trainingFunction_all (GP/gp.py:412-488) from one factorisation:
 * grad[p] = 0.5 * sum_jk (K^-1 - alpha alpha^T)_jk dK_jk/dtheta_p.  The +sum(theta) prior of
 * sub_modules/loss_modules.py:5-13 and the +1.0 of d_logposterior (GP/gp.py:491-493) stay with the caller. */
int pigp_nll_grad(pigp_solver* s, const double* theta_dev, const double* y_dev, double eps,
                  double* nll_dev, double* grad_dev, int32_t* info_dev, void* stream);
/* Host-buffer variant: the call a user of the reference makes every optimiser step
 * (func(theta, r_train, delta_y, eps), solver/optimizers.py:173-176).  pts_host may be NULL to keep the
 * plan's coordinates; otherwise they are re-uploaded.  want_grad = 0 skips the gradient. */
int pigp_nll_grad_host(pigp_solver* s, const double* theta_host, const double* pts_host, const double* y_host,
                       double eps, int want_grad, double* nll_host, double* grad_host, int32_t* info_host);
/* pigp_nll_grad for n_theta hyper-parameter vectors that share the training points, y and eps, in one pass: every launch
 * of the schedule is issued once, with one grid dimension more for the slot, so the launch count does not depend on
 * n_theta.  Slot b reads thetas_dev[b][theta_len] and writes nll_dev[b], grad_dev[b][theta_len] (grad_dev NULL: NLL
 * only) and info_dev[b] (may be NULL).  Each slot's results equal pigp_nll_grad / pigp_nll of its theta bit for bit; a
 * non-positive pivot in one slot gives NaN and info for that slot only.  pigp_nll and pigp_nll_grad are the
 * n_theta = 1 case.  Runs on the caller's stream and never synchronises, like pigp_nll_grad.
 * PIGP_EINVAL before any launch for n_theta outside [1, PIGP_MAX_BATCH], a null pointer, or a sharded solver
 * (world > 1).
 * Memory: for n_theta > 1 the solver keeps a batch workspace, grown to the largest batch seen and freed by
 * pigp_solver_destroy.  Per slot, with npad = N rounded up to 128: (npad + 128) * npad + npad * 128 doubles for L, its y
 * row tile and the inverse diagonal tiles, plus npad^2 for L^-T when the gradient is asked for, plus npad^2 for K^-1 when
 * 8 <= npad / 128 <= 32.  PIGP_ENOMEM when it cannot grow: nothing was launched, and the solver remains usable for single
 * calls and smaller batches. */
int pigp_nll_grad_batch(pigp_solver* s, int n_theta, const double* thetas_dev, const double* y_dev, double eps,
                        double* nll_dev, double* grad_dev, int32_t* info_dev, void* stream);
/* Host-buffer variant: thetas_host[n_theta][theta_len] -> nll_host[n_theta], grad_host[n_theta][theta_len] (want_grad),
 * info_host[n_theta] (may be NULL). */
int pigp_nll_grad_batch_host(pigp_solver* s, int n_theta, const double* thetas_host, const double* y_host, double eps,
                             int want_grad, double* nll_host, double* grad_host, int32_t* info_host);

/* predictingFunction_all (GP/gp.py:226-256, postGP :91-120).  mixed: rows = test points, cols = training points;
 * test: symmetric plan over the test points.  mu_dev[M] = K_ab K_bb^-1 y (mu_test is added by the caller);
 * cov_dev: full M x M posterior covariance K_aa - V^T V (ld = M) when want_full_cov, else its diagonal (M).
 * PIGP_EINVAL before any launch when mixed is not (M x N training points), test is not symmetric over the M test points,
 * or either plan's dim, kernel_type, product_form or n_groups differs from the training plan's (both read theta as the
 * training plan lays it out, noise entry excepted). */
int pigp_predict(pigp_solver* s, const pigp_plan* mixed, const pigp_plan* test, const double* theta_dev,
                 const double* y_dev, double eps, double* mu_dev, double* cov_dev, int want_full_cov,
                 int32_t* info_dev, void* stream);
int pigp_predict_host(pigp_solver* s, pigp_plan* mixed, pigp_plan* test, const double* theta_host,
                      const double* y_host, double eps, double* mu_host, double* cov_host, int want_full_cov,
                      int32_t* info_host);
/* The interval_check loop of the reference's scripts (predictor(theta[i], ...) for a list of recorded hyper-parameter
 * vectors, test/test_1_sinusoidal_direct_main.py:111-131) as ONE call: thetas_host[n_theta][theta_len] ->
 * mu_host[n_theta][M], cov_host[n_theta][M] (or [n_theta][M][M] when want_full_cov); info_host[n_theta] (or one entry
 * when n_theta == 1).  Results are staged on the device and copied back once. */
int pigp_predict_batch_host(pigp_solver* s, pigp_plan* mixed, pigp_plan* test, int n_theta, const double* thetas_host,
                            const double* y_host, double eps, double* mu_host, double* cov_host, int want_full_cov,
                            int32_t* info_host);

/* optimize_by_adam (solver/optimizers.py:94-263) with the hyper-parameters, the Adam moments and the histories resident
 * on the device: per iteration one NLL + gradient evaluation and one update kernel, enqueued back to back; the host reads
 * the state every check_every iterations.  Semantics kept: loss = (NLL + sum(theta) [+ ridge_alpha sum exp(theta)^2]) /
 * ntraining, gradient = (dNLL + 1 [+ ridge term when ridge_in_grad: the autodiff scripts; the explicit-derivative scripts
 * drop it, GP/gp.py:491-493]) / ntraining, optax.adam defaults, entries with fixed_host[i] != 0 held fixed
 * (index_fixed), stop when |loss_t - loss_{t-1}| < stop_eps twice in a row.
 * Outputs: theta_hist_host[(n_done + 1) x P] (row 0 = theta0), loss_hist_host[n_done + 1] (entry 0 = "loss before
 * optimize" = entry 1), norm_hist_host[n_done]; *status_host: 0 max_iter reached, 1 converged, 2 gradient NaN,
 * 3 theta NaN, 4 initial loss NaN (the reference raises in cases 2-4). */
int pigp_adam_host(pigp_solver* s, const double* theta0_host, const double* y_host, double eps, int max_iter, double lr,
                   double stop_eps, double ntraining, double ridge_alpha, int ridge_in_grad, const int32_t* fixed_host,
                   int check_every, double* theta_hist_host, double* loss_hist_host, double* norm_hist_host,
                   int32_t* n_done_host, int32_t* status_host);
/* pigp_adam_host from n_start starting points theta0s_host[n_start][P] at once: one batched NLL + gradient evaluation
 * (pigp_nll_grad_batch) and one update kernel (one warp per start) per iteration.  A start that has stopped (status != 0)
 * is frozen: its later updates are no-ops.  The loop ends when every start has stopped or max_iter is reached.  Start b's
 * outputs are theta_hist_host[b][max_iter + 1][P], loss_hist_host[b][max_iter + 1], norm_hist_host[b][max_iter] (the
 * first n_done_host[b] + 1, n_done_host[b] + 1 and n_done_host[b] entries are written), n_done_host[b] and
 * status_host[b], each equal bit for bit to pigp_adam_host from theta0s_host[b] alone.  pigp_adam_host is the
 * n_start = 1 case, and like it runs on a sharded solver (every rank makes the same call); several starts need a
 * world = 1 solver.  The loop runs on a stream of its own per solver.  PIGP_EINVAL for n_start outside
 * [1, PIGP_MAX_BATCH], a null pointer, or n_start > 1 on a sharded solver. */
int pigp_adam_batch_host(pigp_solver* s, int n_start, const double* theta0s_host, const double* y_host, double eps,
                         int max_iter, double lr, double stop_eps, double ntraining, double ridge_alpha, int ridge_in_grad,
                         const int32_t* fixed_host, int check_every, double* theta_hist_host, double* loss_hist_host,
                         double* norm_hist_host, int32_t* n_done_host, int32_t* status_host);

/* --- building blocks exposed for tests and benchmarks (device pointers, n multiple of PIGP_TILE) --- */
/* In-place lower Cholesky of the leading n x n of A (row-major, ld), applying L^-T to the m_extra rows below it
 * (jnp.linalg.cholesky + jnp.linalg.solve of GP/gp.py:83-84, :106-118).  invd_dev: n/128 inverse diagonal tiles
 * (128*128 doubles each), workspace output.  Only the lower triangle of A is defined on output (the part above the
 * diagonal is not referenced by any consumer and is left partly overwritten).  Runs the solver's factorisation with the
 * panel width of an NLL-only evaluation (pigp_set_lookahead); the panel schedule's bulk stream is one per device,
 * shared by the calling threads. */
int pigp_potrf_lower(double* A_dev, int64_t ld, int64_t n, int64_t m_extra, double* invd_dev,
                     int32_t* info_dev, void* stream);
/* K^-1 (lower triangle, into X_dev) from the factor L (lower of L_dev) -- replaces solve(L.T, solve(L, I)),
 * GP/gp.py:431-432.  W_dev receives L^-1 (lower); its upper triangle is scratch. X_dev may alias L_dev. */
int pigp_potri_lower(const double* L_dev, int64_t ld, int64_t n, const double* invd_dev, double* W_dev,
                     double* X_dev, void* stream);
/* C[MxN] = alpha * A * B^T + beta * C with A(m,k), B(n,k); *_kcontig selects which index is contiguous.
 * M, N and K multiples of 128.  lower_only skips tiles above the diagonal. */
int pigp_dgemm(int M, int N, int K, double alpha, const double* A_dev, int64_t lda, int a_kcontig,
               const double* B_dev, int64_t ldb, int b_kcontig, double beta, double* C_dev, int64_t ldc,
               int lower_only, void* stream);
/* The lower-triangle entries of the 128-row tiles of a symmetric plan's matrix that `rank` owns (tile t belongs to rank
 * t mod world), over exactly the tile list the block-cyclic solver assembles into (64-row tiles, or 16-row tiles when
 * that leaves fewer than two per SM).  Nothing else of K_dev (ld >= cols) is written. */
int pigp_assemble_owned(const pigp_plan* plan, int rank, int world, const double* theta_dev, double eps, int add_diag,
                        double* K_dev, int64_t ld, void* stream);
/* The solver's fused trace gradient over the same owned tiles:  grad[p] = 1/2 sum_jk w_jk (X_jk - alpha_j alpha_k)
 * dK_jk/dtheta_p  over the owned lower entries, w = 1 on the diagonal and 2 below it (X is read below the diagonal only;
 * any 8-byte-aligned X_dev).  Summing grad over the ranks of a world gives the world = 1 result. */
int pigp_trace_grad(const pigp_plan* plan, int rank, int world, const double* theta_dev, const double* X_dev, int64_t ld,
                    const double* alpha_dev, double* grad_dev, void* stream);

/* --- multi-GPU evaluation (new; the reference is single device).  One pigp_dsolver per rank; 128-row tile t of K
 * belongs to rank t mod world.  Ranks exchange data by stores into each other's slab over NVLink (P2P) and epoch flags;
 * the slabs are made mutually visible either with CUDA IPC (one process per GPU: _ipc_handle on every rank, exchange
 * the 64-byte handles with any host-side transport, pigp_ipc_open, _connect) or by passing raw pointers (several ranks
 * in one process).  Every rank must issue the same sequence of pigp_dsolver_nll_grad calls.  All ranks receive the
 * same NLL and (bitwise) the same gradient. */
#define PIGP_IPC_HANDLE_BYTES 64
int pigp_dsolver_create(pigp_plan* training_plan, int rank, int world, pigp_dsolver** out);
void pigp_dsolver_destroy(pigp_dsolver* s);
int pigp_dsolver_slab(const pigp_dsolver* s, void** ptr, int64_t* bytes);
int pigp_dsolver_ipc_handle(const pigp_dsolver* s, void* handle64);
int pigp_ipc_open(const void* handle64, void** ptr);
int pigp_ipc_close(void* ptr);
int pigp_dsolver_connect(pigp_dsolver* s, void* const* slabs /* world pointers; entry [rank] is ignored */);
/* Whether another rank computes on the same physical GPU (tests).  _connect detects it for peers of the same process;
 * with CUDA IPC the caller compares pigp_device_uuid() across ranks and says so.  Ranks that share a GPU wait for flags
 * in separate one-CTA kernels instead of inside the consuming GEMMs (spinning grids could starve their producer). */
int pigp_dsolver_set_shared_device(pigp_dsolver* s, int shared);
int pigp_device_uuid(void* out16);
/* trainingFunction_all + d_trainingFunction_all (GP/gp.py:213-224, :412-488) over the sharded K.  grad_dev may be NULL
 * (NLL only).  Asynchronous on `stream`. */
int pigp_dsolver_nll_grad(pigp_dsolver* s, const double* theta_dev, const double* y_dev, double eps, double* nll_dev,
                          double* grad_dev, int32_t* info_dev, void* stream);
int pigp_dsolver_nll_grad_host(pigp_dsolver* s, const double* theta_host, const double* y_host, double eps, int want_grad,
                               double* nll_host, double* grad_host, int32_t* info_host);
/* Failure handling.  Every flag wait is bounded (PIGP_WAIT_TIMEOUT_S, default 10 s, inside a factorisation;
 * PIGP_BARRIER_TIMEOUT_S, default 300 s, for the barrier that opens a call and absorbs host-side skew between ranks):
 * a lost peer gives NaN results and info = -1 on every surviving rank (and PIGP_ECUDA from the _host call), never a
 * hung GPU.  The condition is sticky; pigp_dsolver_reset -- called on EVERY rank, with a host-side barrier before the
 * next evaluation -- drains the solver's streams and re-arms it.  Ranks must also pass a host-side barrier between
 * pigp_dsolver_connect and their first evaluation. */
int pigp_dsolver_reset(pigp_dsolver* s);

/* Kernel launches issued by this library since load (all threads); for bench.py's gpu_launches. */
int64_t pigp_launch_count(void);

/* Per-kernel-class device timing for bench.py's roofline object (not part of the reference interface).
 * Between start and stop every launch is bracketed by a CUDA event pair on its stream; stop synchronises and
 * returns, per class, the summed kernel time [ms], the number of launches and (GEMM class) the flops executed
 * at tile granularity.  Classes: 0 assemble, 1 gemm (DMMA), 2 potf2, 3 gradient, 4 everything else. */
#define PIGP_PROF_CLASSES 5
/* on = 1 (default): the Y = L^-T products run on a side stream concurrently with the Cholesky chain.  on = 0 puts every
 * kernel on one stream, so that per-launch event times do not overlap (used by the per-class timing pass of bench.py). */
int pigp_set_side_stream(int on);
/* Panel schedule of the factorisation (solver evaluations and pigp_potrf_lower): tiles = 0 is the plain recursion;
 * tiles = W > 0 factors coarse panels of W tile columns on the chain stream and applies each panel to the rest of the
 * matrix on a bulk stream, one panel ahead (the big trailing updates leave the N/128-step dependency chain); tiles < 0 =
 * automatic, which is the default when PIGP_LOOKAHEAD is unset.  The automatic width depends on the tile count T = N/128
 * and applies to single-GPU evaluations only (sharded ones keep the plain recursion): NLL-only evaluations (and
 * pigp_predict and pigp_potrf_lower) have no L^-T work to fill the chain's bubbles and take W = 2 for 12 <= T < 64, 4 for
 * T < 128 and 16 above; NLL + gradient evaluations take W = 2 for 16 <= T < 32 and W = 4 for 32 <= T < 96, where the
 * L^-T products leave bubbles that panels still fill.  Otherwise the plain recursion.  Process-global. */
int pigp_set_lookahead(int tiles);
int pigp_profile_start(void);
int pigp_profile_stop(double* ms_out, int64_t* launches_out, double* flops_out);

/* Debug aid of tools/potf2_bench.py: when dev_buf != NULL the following k_potf2 launches write 17 clock64 phase
 * stamps (thread 0) to it. */
int pigp_debug_potf2_stamps(long long* dev_buf);

#ifdef __cplusplus
}
#endif
#endif /* PIGP_H */
