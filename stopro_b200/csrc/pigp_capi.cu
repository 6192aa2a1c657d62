// extern "C" surface of libpigp.so: plans, solver workspace, NLL / gradient / posterior drivers.
// See include/pigp.h for the contract and the reference interfaces each entry point replaces.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "pigp_internal.cuh"

namespace pigp {

static thread_local std::string t_error;
void set_error(const std::string& msg) { t_error = msg; }
std::atomic<long long> g_launches{0};

bool g_prof_on = false;
struct ProfRec { int cls; cudaEvent_t e0, e1; double flops; int m, n, k, mode; cudaStream_t st; };
static int g_note[4] = {0, 0, 0, 0};
void prof_note(int m, int n, int k, int mode) { g_note[0] = m; g_note[1] = n; g_note[2] = k; g_note[3] = mode; }
static std::vector<ProfRec> g_prof;
static std::mutex g_prof_mu;
void prof_push(int cls, cudaStream_t st, bool begin, double flops) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (begin) {
        ProfRec r{cls, nullptr, nullptr, flops, g_note[0], g_note[1], g_note[2], g_note[3], st};
        g_note[0] = g_note[1] = g_note[2] = g_note[3] = 0;
        cudaEventCreate(&r.e0);
        cudaEventCreate(&r.e1);
        cudaEventRecord(r.e0, st);
        g_prof.push_back(r);
    } else {
        for (size_t i = g_prof.size(); i-- > 0;)
            if (g_prof[i].cls == cls && g_prof[i].st == st && g_prof[i].e1 != nullptr) { cudaEventRecord(g_prof[i].e1, st); break; }
    }
}

static void add_tiles(std::vector<AsmTile>& out, int64_t r0, int64_t r1, int64_t c0, int64_t c1, int desc, int flags) {
    for (int64_t r = r0; r < r1; r += ASM_TR) {
        const int nr = (int)std::min<int64_t>(ASM_TR, r1 - r);
        for (int64_t c = c0; c < c1; c += ASM_TC) {
            if ((flags & ASM_LOWER) && r + nr - 1 < c) continue;  // entirely above the diagonal
            const int nc = (int)std::min<int64_t>(ASM_TC, c1 - c);
            out.push_back(AsmTile{(int32_t)r, (int32_t)c, nr, nc, desc, flags});
        }
    }
}

// (row cap of a tile: ASM_TR = 64 rows, or 16 when that leaves fewer tiles than two per SM -- the kernels of a small problem
// are latency bound, and a CTA's time is proportional to its rows)
static void build_lower_tiles_capped(const pigp_plan* p, int rank, int world, int row_cap, std::vector<AsmTile>& out);

void build_lower_tiles_owned(const pigp_plan* p, int rank, int world, std::vector<AsmTile>& out) {
    build_lower_tiles_capped(p, rank, world, ASM_TR, out);
    if ((int64_t)out.size() < 2 * 148) {
        out.clear();
        build_lower_tiles_capped(p, rank, world, 16, out);
    }
}

static void build_lower_tiles_capped(const pigp_plan* p, int rank, int world, int row_cap, std::vector<AsmTile>& out) {
    const int nb = p->n_row_blocks;
    for (int i = 0; i < nb; ++i)
        for (int j = 0; j <= i; ++j) {
            const pigp_block_desc& b = p->table[(size_t)j * nb + i];  // lower block (i, j) = transpose of table[j][i]
            const int desc = b.n_terms > 0 ? j * nb + i : -1;
            const int flags = (i == j) ? ASM_LOWER : ASM_SWAP;
            const int64_t r1 = p->sec_row[i + 1], c0 = p->sec_row[j], c1 = p->sec_row[j + 1];
            for (int64_t r = p->sec_row[i]; r < r1;) {
                const int nr = (int)std::min<int64_t>(std::min<int64_t>(row_cap, r1 - r), TILE - r % TILE);
                if ((int)((r / TILE) % world) == rank)
                    for (int64_t c = c0; c < c1; c += ASM_TC) {
                        if ((flags & ASM_LOWER) && r + nr - 1 < c) continue;
                        out.push_back(AsmTile{(int32_t)r, (int32_t)c, nr, (int)std::min<int64_t>(ASM_TC, c1 - c), desc, flags});
                    }
                r += nr;
            }
        }
}

static int upload_tiles(const std::vector<AsmTile>& v, AsmTile** dev, int64_t* n) {
    *n = (int64_t)v.size();
    *dev = nullptr;
    if (v.empty()) return PIGP_OK;
    PIGP_CUDA(cudaMalloc(dev, v.size() * sizeof(AsmTile)));
    PIGP_CUDA(cudaMemcpy(*dev, v.data(), v.size() * sizeof(AsmTile), cudaMemcpyHostToDevice));
    return PIGP_OK;
}

// host [n][dim] (array of points) -> pinned [dim][n] -> device
static int upload_points(pigp_plan* p, const double* host, int64_t n, double* dev, cudaStream_t st) {
    const int64_t bytes = n * p->dim * (int64_t)sizeof(double);
    if (bytes > p->h_pin_bytes) {
        if (p->h_pin) cudaFreeHost(p->h_pin);
        p->h_pin = nullptr;
        PIGP_CUDA(cudaMallocHost(&p->h_pin, bytes));
        p->h_pin_bytes = bytes;
    }
    for (int64_t i = 0; i < n; ++i)
        for (int d = 0; d < p->dim; ++d) p->h_pin[d * n + i] = host[i * p->dim + d];
    PIGP_CUDA(cudaMemcpyAsync(dev, p->h_pin, bytes, cudaMemcpyHostToDevice, st));
    PIGP_CUDA(cudaStreamSynchronize(st));  // the pinned buffer is reused by the next call
    return PIGP_OK;
}

__global__ void k_rowsumsq_sub(const double* Vt, int64_t ld, int64_t m, int64_t n, const double* kdiag, double* var) {
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= m) return;
    const int lane = threadIdx.x & 31;
    double s = 0.0;
    for (int64_t j = lane; j < n; j += 32) {
        const double x = Vt[row * ld + j];
        s = fma(x, x, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) var[row] = kdiag[row] - s;
}

// ---- device-resident optimiser step (solver/optimizers.py:173-235): one warp per start, thread i owns hyper-parameter i
// (start b's arrays at + b times the size of one start's)
struct AdamArgs {
    int P, max_iter;
    double lr, stop_eps, ntraining, ridge_alpha;
    int ridge_in_grad;
    const int32_t* fixed;   // P entries (1 = held fixed: params_optimization["index_fixed"]) or nullptr
    double* theta;          // current hyper-parameters (read by the evaluation, advanced here)
    const double* nll;      // likelihood value and gradient of the evaluation just finished
    const double* grad;
    double *m, *v;          // Adam moments
    double* prev_loss;
    int32_t* istate;        // [0] t, [1] converged once, [2] status (0 running), [3] iterations done
    double *theta_hist, *loss_hist, *norm_hist;
};
__global__ void k_adam_step(AdamArgs a) {
    const int64_t b = blockIdx.x;
    a.theta += b * a.P; a.m += b * a.P; a.v += b * a.P;
    a.nll += b; a.grad += b * a.P; a.prev_loss += b;
    a.istate += 4 * b;
    a.theta_hist += b * (int64_t)(a.max_iter + 1) * a.P;
    a.loss_hist += b * (int64_t)(a.max_iter + 1);
    a.norm_hist += b * (int64_t)a.max_iter;
    const int i = threadIdx.x;
    const int t = a.istate[0];
    if (a.istate[2] != 0 || t >= a.max_iter) return;
    const bool on = i < a.P;
    const double th = on ? a.theta[i] : 0.0;
    if (on && t == 0) a.theta_hist[i] = th;  // row 0 of the history: the starting point
    const double e2 = on ? exp(2.0 * th) : 0.0;
    double s_th = th, s_e2 = e2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s_th += __shfl_xor_sync(0xffffffffu, s_th, o);
        s_e2 += __shfl_xor_sync(0xffffffffu, s_e2, o);
    }
    // logposterior = NLL + sum(theta) [+ ridge_alpha sum exp(theta)^2] (sub_modules/loss_modules.py:5-13), divided by the
    // number of training points (optimizers.py:136-139); gradient: +1 per component (GP/gp.py:491-493)
    const double value = (*a.nll + s_th + a.ridge_alpha * s_e2) / a.ntraining;
    double g = 0.0;
    if (on && !(a.fixed && a.fixed[i])) g = (a.grad[i] + 1.0 + (a.ridge_in_grad ? 2.0 * a.ridge_alpha * e2 : 0.0)) / a.ntraining;
    const unsigned nan_g = __ballot_sync(0xffffffffu, g != g);
    if (t == 0 && value != value) {  // "loss is nan at the initial hyper-parameters" (optimizers.py:245-246)
        if (i == 0) { a.istate[2] = 4; a.loss_hist[0] = value; }
        return;
    }
    if (nan_g) {                     // "gradient of loss became nan" (optimizers.py:182-183)
        if (i == 0) a.istate[2] = 2;
        return;
    }
    double g2 = g * g;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) g2 += __shfl_xor_sync(0xffffffffu, g2, o);
    double th_new = th;
    if (on) {
        // optax.adam defaults: b1 = 0.9, b2 = 0.999, eps = 1e-8, eps_root = 0
        const double b1 = 0.9, b2 = 0.999;
        const double m = b1 * a.m[i] + (1.0 - b1) * g;
        const double v = b2 * a.v[i] + (1.0 - b2) * g * g;
        a.m[i] = m;
        a.v[i] = v;
        const double mhat = m / (1.0 - pow(b1, (double)(t + 1))), vhat = v / (1.0 - pow(b2, (double)(t + 1)));
        th_new = th - a.lr * mhat / (sqrt(vhat) + 1e-8);
        a.theta[i] = th_new;
        a.theta_hist[(int64_t)(t + 1) * a.P + i] = th_new;
    }
    const unsigned nan_th = __ballot_sync(0xffffffffu, th_new != th_new);
    if (i == 0) {
        if (t == 0) a.loss_hist[0] = value;  // "loss before optimize": the same evaluation (optimizers.py:239-244)
        a.loss_hist[t + 1] = value;
        a.norm_hist[t] = sqrt(g2);
        int status = 0, once = a.istate[1];
        if (t >= 1) {                         // two-in-a-row plateau rule and divergence guard (optimizers.py:218-233)
            if (fabs(value - *a.prev_loss) < a.stop_eps) {
                if (once) status = 1; else once = 1;
            } else if (nan_th) {
                status = 3;
            } else {
                once = 0;
            }
        }
        *a.prev_loss = value;
        a.istate[0] = t + 1;
        a.istate[1] = once;
        a.istate[2] = status;
        a.istate[3] = t + 1;
    }
}

}  // namespace pigp

using namespace pigp;

template <class T>
static int grow(T** buf, int64_t* have, int64_t need) {
    if (need <= *have) return PIGP_OK;
    cudaFree(*buf);
    *buf = nullptr;
    *have = 0;
    PIGP_CUDA(cudaMalloc(buf, sizeof(T) * (size_t)need));
    *have = need;
    return PIGP_OK;
}


struct pigp_solver {
    pigp_plan* plan = nullptr;
    pigp_dsolver* ds = nullptr;  // the block-cyclic solver (world = 1 unless created with _create_dist): NLL, gradient, factor
    int world = 1;
    int64_t n = 0, npad = 0;
    int32_t* info = nullptr;
    // posterior workspace (allocated on first use, grow-only)
    double* V = nullptr;     // mpad x npad: K_ab -> K_ab L^-T
    int64_t v_elems = 0;
    double* T = nullptr;     // mpad x mpad test covariance (full posterior covariance only)
    int64_t t_elems = 0;
    double* kdiag = nullptr; // diag(K_aa)
    int64_t kdiag_elems = 0;
    double* d_mu = nullptr;  // staging of the _host entry points: mu, then cov / var
    double* d_cov = nullptr;
    int64_t mu_elems = 0, cov_elems = 0;
    // staging for the _host entry points
    double* d_theta = nullptr;
    double* d_y = nullptr;
    double* d_res = nullptr;  // nll + grad
    double* h_res = nullptr;  // pinned
    double* d_batch = nullptr;  // pigp_nll_grad_batch_host: thetas, nll, grad (grow-only)
    int64_t batch_elems = 0;
    int32_t* d_binfo = nullptr;
    int64_t binfo_elems = 0;
    // the device Adam loop runs on its own stream: ranks of a sharded solver that share a process must not share one
    cudaStream_t adam_stream = nullptr;
};

static cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// every entry point works on the device its plan was created on, whatever the calling thread's current device is
static int use_device(const pigp_plan* p) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != p->device) PIGP_CUDA(cudaSetDevice(p->device));
    return PIGP_OK;
}

extern "C" {

int pigp_abi_version(void) { return PIGP_ABI_VERSION; }
const char* pigp_last_error(void) { return t_error.c_str(); }
int64_t pigp_launch_count(void) { return (int64_t)g_launches.load(); }

int pigp_profile_start(void) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.clear();
    g_prof_on = true;
    return PIGP_OK;
}

int pigp_profile_stop(double* ms_out, int64_t* launches_out, double* flops_out) {
    g_prof_on = false;
    PIGP_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int c = 0; c < PIGP_PROF_CLASSES; ++c) {
        if (ms_out) ms_out[c] = 0.0;
        if (launches_out) launches_out[c] = 0;
        if (flops_out) flops_out[c] = 0.0;
    }
    FILE* dump = nullptr;
    if (const char* path = getenv("PIGP_PROF_DUMP")) dump = fopen(path, "w");
    if (dump) fprintf(dump, "class,ms,flops,m,n,k,mode,start_ms,stream\n");
    for (auto& r : g_prof) {
        float ms = 0.f, t0 = 0.f;
        cudaEventElapsedTime(&ms, r.e0, r.e1);
        if (dump) {
            cudaEventElapsedTime(&t0, g_prof.front().e0, r.e0);
            fprintf(dump, "%d,%.6f,%.0f,%d,%d,%d,%d,%.6f,%p\n", r.cls, ms, r.flops, r.m, r.n, r.k, r.mode, t0, (void*)r.st);
        }
        if (ms_out) ms_out[r.cls] += ms;
        if (launches_out) launches_out[r.cls] += 1;
        if (flops_out) flops_out[r.cls] += r.flops;
    }
    for (auto& r : g_prof) {
        cudaEventDestroy(r.e0);
        cudaEventDestroy(r.e1);
    }
    if (dump) fclose(dump);
    g_prof.clear();
    return PIGP_OK;
}

int pigp_set_device(int device) {
    PIGP_CUDA(cudaSetDevice(device));
    return PIGP_OK;
}

void pigp_plan_destroy(pigp_plan* p) {
    if (!p) return;
    if (p->d_pts_col && p->d_pts_col != p->d_pts_row) cudaFree(p->d_pts_col);
    cudaFree(p->d_pts_row);
    cudaFree(p->d_table);
    cudaFree(p->d_tiles_full);
    cudaFree(p->d_tiles_lower);
    cudaFree(p->d_tiles_diag);
    cudaFree(p->d_khost);
    cudaFree(p->d_theta_stage);
    if (p->h_pin) cudaFreeHost(p->h_pin);
    delete p;
}

int pigp_plan_create(const pigp_plan_desc* d, pigp_plan** out) {
    if (!d || !out) { set_error("pigp_plan_create: null argument"); return PIGP_EINVAL; }
    *out = nullptr;
    if (d->dim < 1 || d->dim > 3 || d->n_groups < 1 || d->n_groups > PIGP_MAX_GROUPS || d->n_row_blocks < 1 ||
        (!d->symmetric && d->n_col_blocks < 1) || !d->sec_row || !d->pts_row_host || !d->table) {
        set_error("pigp_plan_create: bad dimensions or null arrays");
        return PIGP_EINVAL;
    }
    pigp_plan* p = new pigp_plan();
    p->dim = d->dim;
    p->product_form = d->product_form ? 1 : 0;
    p->n_groups = d->n_groups;
    p->symmetric = d->symmetric ? 1 : 0;
    p->n_row_blocks = d->n_row_blocks;
    p->n_col_blocks = p->symmetric ? d->n_row_blocks : d->n_col_blocks;
    p->sec_row.assign(d->sec_row, d->sec_row + d->n_row_blocks + 1);
    if (p->symmetric) p->sec_col = p->sec_row;
    else p->sec_col.assign(d->sec_col, d->sec_col + d->n_col_blocks + 1);
    p->rows = p->sec_row.back();
    p->cols = p->sec_col.back();
    for (int k = 0; k < 3; ++k) p->lbox[k] = d->lbox[k];
    p->noise_lo_block = d->noise_lo_block;
    p->noise_hi_block = d->noise_hi_block;
    p->kernel_type = d->kernel_type;
    p->theta_len = d->n_groups * (1 + d->dim);
    auto fail = [&](const char* msg) {
        set_error(msg);
        pigp_plan_destroy(p);
        return PIGP_EINVAL;
    };
    for (size_t i = 0; i + 1 < p->sec_row.size(); ++i)
        if (p->sec_row[i + 1] < p->sec_row[i]) return fail("pigp_plan_create: sec_row must be non-decreasing");
    for (size_t i = 0; i + 1 < p->sec_col.size(); ++i)
        if (p->sec_col[i + 1] < p->sec_col[i]) return fail("pigp_plan_create: sec_col must be non-decreasing");
    if (p->kernel_type != PIGP_KERNEL_SE && p->kernel_type != PIGP_KERNEL_MT52 && p->kernel_type != PIGP_KERNEL_MT72 &&
        p->kernel_type != PIGP_KERNEL_MT92)
        return fail("pigp_plan_create: unknown kernel_type");
    if (p->rows <= 0 || p->cols <= 0 || p->rows > (1 << 30) || p->cols > (1 << 30))
        return fail("pigp_plan_create: empty or oversized matrix");
    if (p->noise_lo_block >= 0) {
        if (!p->symmetric || p->noise_hi_block < p->noise_lo_block || p->noise_hi_block >= p->n_row_blocks)
            return fail("pigp_plan_create: bad noise block range");
        p->noise_lo = p->sec_row[p->noise_lo_block];
        p->noise_hi = p->sec_row[p->noise_hi_block + 1];
        p->theta_len += 1;
    }
    const int nrb = p->n_row_blocks, ncb = p->n_col_blocks;
    p->table.assign(d->table, d->table + (size_t)nrb * ncb);
    for (int i = 0; i < nrb; ++i)
        for (int j = (p->symmetric ? i : 0); j < ncb; ++j) {
            const pigp_block_desc& b = p->table[(size_t)i * ncb + j];
            if (b.n_terms < 0 || b.n_terms > PIGP_MAX_TERMS) return fail("pigp_plan_create: n_terms out of range");
            for (int t = 0; t < b.n_terms; ++t) {
                if (b.terms[t].group < 0 || b.terms[t].group >= p->n_groups) return fail("pigp_plan_create: term group out of range");
                if (t && b.terms[t].group < b.terms[t - 1].group) return fail("pigp_plan_create: terms must be sorted by group");
                int active = 0, total = 0;
                for (int k = 0; k < p->dim; ++k) {
                    if (b.terms[t].order[k] < -1 || b.terms[t].order[k] > 4) return fail("pigp_plan_create: derivative order out of range");
                    if (b.terms[t].order[k] >= 0) { ++active; total += b.terms[t].order[k]; }
                }
                if (total > 4) return fail("pigp_plan_create: total derivative order of a term exceeds 4");
                if (!p->product_form && p->dim > 1 && active != 1)
                    return fail("pigp_plan_create: additive kernel form: every term must act on exactly one dimension (order -1 elsewhere)");
            }
        }
    if (p->product_form) {
        // the evaluator groups the terms of a block into runs of equal (group, parity pattern of the derivative orders)
        auto key = [&](const pigp_term& t) {
            int pm = 0;
            for (int k = 0; k < p->dim; ++k) pm |= (std::max(t.order[k], 0) & 1) << k;
            return t.group * 8 + pm;
        };
        for (pigp_block_desc& b : p->table)
            std::stable_sort(b.terms, b.terms + std::max(0, std::min(b.n_terms, PIGP_MAX_TERMS)),
                             [&](const pigp_term& x, const pigp_term& y) { return key(x) < key(y); });
    }
    if (cudaGetDevice(&p->device) != cudaSuccess) return fail("pigp_plan_create: no CUDA device");

    int rc = PIGP_OK;
    auto cuda_ok = [&](cudaError_t e, const char* what) {
        if (e != cudaSuccess && rc == PIGP_OK) {
            set_error(std::string(what) + ": " + cudaGetErrorString(e));
            rc = PIGP_ECUDA;
        }
    };
    cuda_ok(cudaMalloc(&p->d_pts_row, sizeof(double) * p->dim * p->rows), "cudaMalloc pts_row");
    if (p->symmetric) p->d_pts_col = p->d_pts_row;
    else cuda_ok(cudaMalloc(&p->d_pts_col, sizeof(double) * p->dim * p->cols), "cudaMalloc pts_col");
    cuda_ok(cudaMalloc(&p->d_table, sizeof(pigp_block_desc) * p->table.size()), "cudaMalloc table");
    cuda_ok(cudaMalloc(&p->d_theta_stage, sizeof(double) * MAX_THETA), "cudaMalloc theta");
    if (rc == PIGP_OK)
        cuda_ok(cudaMemcpy(p->d_table, p->table.data(), sizeof(pigp_block_desc) * p->table.size(), cudaMemcpyHostToDevice), "copy table");
    if (rc == PIGP_OK) rc = upload_points(p, d->pts_row_host, p->rows, p->d_pts_row, 0);
    if (rc == PIGP_OK && !p->symmetric) {
        if (!d->pts_col_host || !d->sec_col) { pigp_plan_destroy(p); set_error("pigp_plan_create: rectangular plan needs column points"); return PIGP_EINVAL; }
        rc = upload_points(p, d->pts_col_host, p->cols, p->d_pts_col, 0);
    }
    if (rc == PIGP_OK) {
        std::vector<AsmTile> full, lower;
        auto desc_of = [&](int i, int j) { return p->table[(size_t)i * ncb + j].n_terms > 0 ? i * ncb + j : -1; };
        for (int i = 0; i < nrb; ++i)
            for (int j = 0; j < ncb; ++j) {
                const int64_t r0 = p->sec_row[i], r1 = p->sec_row[i + 1], c0 = p->sec_col[j], c1 = p->sec_col[j + 1];
                if (!p->symmetric) add_tiles(full, r0, r1, c0, c1, desc_of(i, j), 0);
                if (p->symmetric && i == j) add_tiles(lower, r0, r1, c0, c1, desc_of(i, i), ASM_LOWER);
                if (p->symmetric && i > j) add_tiles(lower, r0, r1, c0, c1, desc_of(j, i), ASM_SWAP);  // lower block = transpose of table[j][i]
            }
        if (p->symmetric) {
            // full layout = the lower tiles, each also stored transposed: half the evaluations, exact symmetry
            full = lower;
            for (AsmTile& t : full) t.flags |= ASM_MIRROR;
            // the diagonal alone (posterior variance: callers only ever take sqrt(diag), test_1:144): 16 x 16 tiles
            // astride the diagonal of every diagonal block
            std::vector<AsmTile> diag;
            for (int i = 0; i < nrb; ++i)
                for (int64_t r = p->sec_row[i]; r < p->sec_row[i + 1]; r += ASM_TR)
                    diag.push_back(AsmTile{(int32_t)r, (int32_t)r, (int32_t)std::min<int64_t>(ASM_TR, p->sec_row[i + 1] - r),
                                           (int32_t)std::min<int64_t>(ASM_TR, p->sec_row[i + 1] - r), desc_of(i, i), ASM_DIAG});
            rc = upload_tiles(diag, &p->d_tiles_diag, &p->n_tiles_diag);
        }
        if (rc == PIGP_OK) rc = upload_tiles(full, &p->d_tiles_full, &p->n_tiles_full);
        if (rc == PIGP_OK) rc = upload_tiles(lower, &p->d_tiles_lower, &p->n_tiles_lower);
    }
    if (rc != PIGP_OK) { pigp_plan_destroy(p); return rc; }
    *out = p;
    return PIGP_OK;
}

int64_t pigp_plan_rows(const pigp_plan* p) { return p ? p->rows : 0; }
int64_t pigp_plan_cols(const pigp_plan* p) { return p ? p->cols : 0; }
int32_t pigp_plan_theta_len(const pigp_plan* p) { return p ? p->theta_len : 0; }

int pigp_plan_set_points_host(pigp_plan* p, int side, const double* pts_host, void* stream) {
    if (!p || !pts_host) { set_error("pigp_plan_set_points_host: null argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(p));
    if (side == 0 || p->symmetric) return upload_points(p, pts_host, p->rows, p->d_pts_row, as_stream(stream));
    return upload_points(p, pts_host, p->cols, p->d_pts_col, as_stream(stream));
}

int pigp_assemble(const pigp_plan* p, const double* theta_dev, double eps, int add_diag, double* K_dev, int64_t ld,
                  int layout, void* stream) {
    if (!p || !theta_dev || !K_dev || ld < p->cols) { set_error("pigp_assemble: bad argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(p));
    if (add_diag && !p->symmetric) { set_error("pigp_assemble: add_diag needs a symmetric plan"); return PIGP_EINVAL; }
    if (layout == PIGP_LAYOUT_LOWER) {
        if (!p->symmetric) { set_error("pigp_assemble: LOWER layout needs a symmetric plan"); return PIGP_EINVAL; }
        return launch_assemble(p, p->d_tiles_lower, p->n_tiles_lower, theta_dev, eps, add_diag, K_dev, ld, as_stream(stream));
    }
    return launch_assemble(p, p->d_tiles_full, p->n_tiles_full, theta_dev, eps, add_diag, K_dev, ld, as_stream(stream));
}

int pigp_assemble_host(pigp_plan* p, const double* theta_host, double eps, int add_diag, double* K_host, int layout) {
    if (!p || !theta_host || !K_host) { set_error("pigp_assemble_host: null argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(p));
    const size_t bytes = sizeof(double) * (size_t)p->rows * p->cols;
    if (bytes > p->d_khost_bytes) {  // grow-only staging buffer owned by the plan (not thread-safe per plan: see pigp.h)
        cudaFree(p->d_khost);
        p->d_khost = nullptr;
        p->d_khost_bytes = 0;
        PIGP_CUDA(cudaMalloc(&p->d_khost, bytes));
        p->d_khost_bytes = bytes;
    }
    double* K = p->d_khost;
    PIGP_CUDA(cudaMemcpy(p->d_theta_stage, theta_host, sizeof(double) * p->theta_len, cudaMemcpyHostToDevice));
    if (layout == PIGP_LAYOUT_LOWER) PIGP_CUDA(cudaMemset(K, 0, bytes));
    PIGP_TRY(pigp_assemble(p, p->d_theta_stage, eps, add_diag, K, p->cols, layout, nullptr));
    PIGP_CUDA(cudaMemcpy(K_host, K, bytes, cudaMemcpyDeviceToHost));
    return PIGP_OK;
}

int pigp_assemble_diag(const pigp_plan* p, const double* theta_dev, double eps, int add_diag, double* diag_dev, void* stream) {
    if (!p || !theta_dev || !diag_dev || !p->symmetric) { set_error("pigp_assemble_diag: needs a symmetric plan and device buffers"); return PIGP_EINVAL; }
    return launch_assemble(p, p->d_tiles_diag, p->n_tiles_diag, theta_dev, eps, add_diag, diag_dev, 0, as_stream(stream));
}

// ------------------------------------------------------------------------------------------------ solver
void pigp_solver_destroy(pigp_solver* s) {
    if (!s) return;
    pigp_dsolver_destroy(s->ds);
    cudaFree(s->info); cudaFree(s->V); cudaFree(s->T); cudaFree(s->kdiag); cudaFree(s->d_mu); cudaFree(s->d_cov);
    cudaFree(s->d_theta); cudaFree(s->d_y); cudaFree(s->d_res); cudaFree(s->d_batch); cudaFree(s->d_binfo);
    if (s->adam_stream) cudaStreamDestroy(s->adam_stream);
    if (s->h_res) cudaFreeHost(s->h_res);
    delete s;
}

int pigp_solver_create(pigp_plan* plan, pigp_solver** out) { return pigp_solver_create_dist(plan, 0, 1, out); }

pigp_dsolver* pigp_solver_dsolver(pigp_solver* s) { return s ? s->ds : nullptr; }

int pigp_solver_create_dist(pigp_plan* plan, int rank, int world, pigp_solver** out) {
    if (!plan || !out || !plan->symmetric) { set_error("pigp_solver_create: needs a symmetric training plan"); return PIGP_EINVAL; }
    *out = nullptr;
    PIGP_TRY(use_device(plan));
    pigp_solver* s = new pigp_solver();
    s->plan = plan;
    s->world = world;
    s->n = plan->rows;
    s->npad = round_up(s->n, TILE);
    int rc = pigp_dsolver_create(plan, rank, world, &s->ds);
    auto cuda_ok = [&](cudaError_t e, const char* what) {
        if (e != cudaSuccess && rc == PIGP_OK) { set_error(std::string(what) + ": " + cudaGetErrorString(e)); rc = PIGP_ECUDA; }
    };
    cuda_ok(cudaMalloc(&s->info, sizeof(int32_t)), "cudaMalloc info");
    cuda_ok(cudaMalloc(&s->d_theta, sizeof(double) * MAX_THETA), "cudaMalloc theta");
    cuda_ok(cudaMalloc(&s->d_y, sizeof(double) * s->n), "cudaMalloc y");
    cuda_ok(cudaMalloc(&s->d_res, sizeof(double) * (1 + MAX_THETA)), "cudaMalloc res");
    cuda_ok(cudaMallocHost(&s->h_res, sizeof(double) * (2 + 2 * MAX_THETA) + sizeof(double) * s->n), "cudaMallocHost res");
    cuda_ok(cudaStreamCreateWithFlags(&s->adam_stream, cudaStreamNonBlocking), "cudaStreamCreate adam");
    if (rc != PIGP_OK) { pigp_solver_destroy(s); return rc; }
    *out = s;
    return PIGP_OK;
}

// V[:, tiles c0 .. c0 + nt) <- V L^-T restricted to those columns: recursive (the flops are GEMMs with large K), the
// leaf multiplies by the inverse diagonal tile in place
static int trsm_rec(double* V, int64_t ldv, int64_t m, const FactorView& f, int c0, int nt, cudaStream_t st) {
    if (nt == 1) {
        GemmDesc g{};
        g.M = (int)m; g.N = TILE; g.K = TILE;
        g.alpha = 1.0; g.beta = 0.0;
        g.A = V + (int64_t)c0 * TILE; g.lda = ldv; g.a_kcontig = 1;
        g.B = f.invd + (int64_t)c0 * TILE * TILE; g.ldb = TILE; g.b_kcontig = 1;
        g.C = V + (int64_t)c0 * TILE; g.ldc = ldv;
        g.force_bn128 = 1;  // in place: a CTA reads its 128 columns of its rows before it writes them
        g.Lkk = f.L + (int64_t)c0 * TILE * f.ld + (int64_t)c0 * TILE; g.ldl = f.ld;  // block substitution with refinement (k_trsm_blk)
        return launch_gemm(g, st);
    }
    const int n1 = nt / 2, n2 = nt - n1;
    PIGP_TRY(trsm_rec(V, ldv, m, f, c0, n1, st));
    GemmDesc g{};
    g.M = (int)m; g.N = n2 * TILE; g.K = n1 * TILE;
    g.alpha = -1.0; g.beta = 1.0;
    g.A = V + (int64_t)c0 * TILE; g.lda = ldv; g.a_kcontig = 1;
    g.B = f.L + (int64_t)(c0 + n1) * TILE * f.ld + (int64_t)c0 * TILE; g.ldb = f.ld; g.b_kcontig = 1;
    g.C = V + (int64_t)(c0 + n1) * TILE; g.ldc = ldv;
    PIGP_TRY(launch_gemm(g, st));
    return trsm_rec(V, ldv, m, f, c0 + n1, n2, st);
}

int pigp_nll(pigp_solver* s, const double* theta_dev, const double* y_dev, double eps, double* out_dev, int32_t* info_dev,
             void* stream) {
    if (!s || !theta_dev || !y_dev || !out_dev) { set_error("pigp_nll: null argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(s->plan));
    return pigp_dsolver_nll_grad(s->ds, theta_dev, y_dev, eps, out_dev, nullptr, info_dev ? info_dev : s->info, stream);
}

int pigp_nll_grad(pigp_solver* s, const double* theta_dev, const double* y_dev, double eps, double* nll_dev, double* grad_dev,
                  int32_t* info_dev, void* stream) {
    if (!s || !theta_dev || !y_dev || !nll_dev || !grad_dev) { set_error("pigp_nll_grad: null argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(s->plan));
    return pigp_dsolver_nll_grad(s->ds, theta_dev, y_dev, eps, nll_dev, grad_dev, info_dev ? info_dev : s->info, stream);
}

int pigp_nll_grad_host(pigp_solver* s, const double* theta_host, const double* pts_host, const double* y_host, double eps,
                       int want_grad, double* nll_host, double* grad_host, int32_t* info_host) {
    if (!s || !theta_host || !y_host || !nll_host || (want_grad && !grad_host)) { set_error("pigp_nll_grad_host: null argument"); return PIGP_EINVAL; }
    pigp_plan* p = s->plan;
    PIGP_TRY(use_device(p));
    const int P = p->theta_len;
    cudaStream_t st = 0;
    if (pts_host) PIGP_TRY(upload_points(p, pts_host, p->rows, p->d_pts_row, st));
    if (s->world > 1)  // sharded: the block-cyclic solver's own host entry point (own stream, time-out reporting)
        return pigp_dsolver_nll_grad_host(s->ds, theta_host, y_host, eps, want_grad, nll_host, grad_host, info_host);
    double* h_theta = s->h_res + 2 + MAX_THETA;
    double* h_y = h_theta + MAX_THETA;
    std::memcpy(h_theta, theta_host, sizeof(double) * P);
    std::memcpy(h_y, y_host, sizeof(double) * s->n);
    PIGP_CUDA(cudaMemcpyAsync(s->d_theta, h_theta, sizeof(double) * P, cudaMemcpyHostToDevice, st));
    PIGP_CUDA(cudaMemcpyAsync(s->d_y, h_y, sizeof(double) * s->n, cudaMemcpyHostToDevice, st));
    if (want_grad) PIGP_TRY(pigp_nll_grad(s, s->d_theta, s->d_y, eps, s->d_res, s->d_res + 1, s->info, st));
    else PIGP_TRY(pigp_nll(s, s->d_theta, s->d_y, eps, s->d_res, s->info, st));
    PIGP_CUDA(cudaMemcpyAsync(s->h_res, s->d_res, sizeof(double) * (1 + (want_grad ? P : 0)), cudaMemcpyDeviceToHost, st));
    int32_t* h_info = reinterpret_cast<int32_t*>(s->h_res + 1 + MAX_THETA);
    PIGP_CUDA(cudaMemcpyAsync(h_info, s->info, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PIGP_CUDA(cudaStreamSynchronize(st));
    *nll_host = s->h_res[0];
    if (want_grad) std::memcpy(grad_host, s->h_res + 1, sizeof(double) * P);
    if (info_host) *info_host = *h_info;
    return PIGP_OK;
}

int pigp_nll_grad_batch(pigp_solver* s, int n_theta, const double* thetas_dev, const double* y_dev, double eps, double* nll_dev,
                        double* grad_dev, int32_t* info_dev, void* stream) {
    if (!s || !thetas_dev || !y_dev || !nll_dev) { set_error("pigp_nll_grad_batch: null argument"); return PIGP_EINVAL; }
    if (n_theta < 1 || n_theta > PIGP_MAX_BATCH) { set_error("pigp_nll_grad_batch: n_theta must be in [1, 65535]"); return PIGP_EINVAL; }
    if (s->world != 1) { set_error("pigp_nll_grad_batch: sharded solvers (world > 1) evaluate one theta at a time"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(s->plan));
    return dsolver_nll_grad_batch(s->ds, n_theta, thetas_dev, y_dev, eps, nll_dev, grad_dev, info_dev, stream);
}

int pigp_nll_grad_batch_host(pigp_solver* s, int n_theta, const double* thetas_host, const double* y_host, double eps,
                             int want_grad, double* nll_host, double* grad_host, int32_t* info_host) {
    if (!s || !thetas_host || !y_host || !nll_host || (want_grad && !grad_host)) { set_error("pigp_nll_grad_batch_host: null argument"); return PIGP_EINVAL; }
    if (n_theta < 1 || n_theta > PIGP_MAX_BATCH) { set_error("pigp_nll_grad_batch_host: n_theta must be in [1, 65535]"); return PIGP_EINVAL; }
    if (s->world != 1) { set_error("pigp_nll_grad_batch_host: sharded solvers (world > 1) evaluate one theta at a time"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(s->plan));
    const int64_t P = s->plan->theta_len, nb = n_theta;
    PIGP_TRY(grow(&s->d_batch, &s->batch_elems, nb * (2 * P + 1)));
    PIGP_TRY(grow(&s->d_binfo, &s->binfo_elems, nb));
    double* th = s->d_batch;
    double* nll = th + nb * P;
    double* grad = nll + nb;
    PIGP_CUDA(cudaMemcpy(th, thetas_host, sizeof(double) * nb * P, cudaMemcpyHostToDevice));
    PIGP_CUDA(cudaMemcpy(s->d_y, y_host, sizeof(double) * s->n, cudaMemcpyHostToDevice));
    PIGP_TRY(pigp_nll_grad_batch(s, n_theta, th, s->d_y, eps, nll, want_grad ? grad : nullptr, s->d_binfo, nullptr));
    PIGP_CUDA(cudaMemcpy(nll_host, nll, sizeof(double) * nb, cudaMemcpyDeviceToHost));
    if (want_grad) PIGP_CUDA(cudaMemcpy(grad_host, grad, sizeof(double) * nb * P, cudaMemcpyDeviceToHost));
    if (info_host) PIGP_CUDA(cudaMemcpy(info_host, s->d_binfo, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost));
    return PIGP_OK;
}

int pigp_predict(pigp_solver* s, const pigp_plan* mixed, const pigp_plan* test, const double* theta_dev, const double* y_dev,
                 double eps, double* mu_dev, double* cov_dev, int want_full_cov, int32_t* info_dev, void* stream) {
    if (!s || !mixed || !test || !theta_dev || !y_dev || !mu_dev || !cov_dev) { set_error("pigp_predict: null argument"); return PIGP_EINVAL; }
    if (mixed->symmetric || mixed->cols != s->n || !test->symmetric || test->rows != mixed->rows) {
        set_error("pigp_predict: mixed must be (test x train) and test symmetric over the same test points");
        return PIGP_EINVAL;
    }
    for (const pigp_plan* p : {mixed, test})
        if (p->dim != s->plan->dim || p->kernel_type != s->plan->kernel_type || p->product_form != s->plan->product_form ||
            p->n_groups != s->plan->n_groups) {
            set_error("pigp_predict: mixed and test plans must have the training plan's dim, kernel_type, product_form and n_groups");
            return PIGP_EINVAL;
        }
    PIGP_TRY(use_device(s->plan));
    cudaStream_t st = as_stream(stream);
    int32_t* info = info_dev ? info_dev : s->info;
    const int64_t m = mixed->rows, mpad = round_up(m, TILE), ld = s->npad;
    PIGP_TRY(grow(&s->V, &s->v_elems, mpad * ld));
    // L and L^-1 y from the solver's own factorisation (the NLL value is a by-product, parked in d_res)
    PIGP_TRY(pigp_dsolver_nll_grad(s->ds, theta_dev, y_dev, eps, s->d_res, nullptr, info, stream));
    const FactorView f = factor_view(s->ds);
    // V = K_ab L^-T: rows = test points (first kernel argument), columns = training points
    PIGP_TRY(launch_assemble(mixed, mixed->d_tiles_full, mixed->n_tiles_full, theta_dev, 0.0, 0, s->V, ld, st));
    PIGP_TRY(launch_pad(s->V, ld, m, s->n, mpad, s->npad, 0, 0, st));
    PIGP_TRY(trsm_rec(s->V, ld, mpad, f, 0, f.T, st));
    // mu = K_ab K_bb^-1 y = (K_ab L^-T)(L^-1 y)
    PIGP_TRY(launch_gemv(s->V, ld, m, s->n, f.v, mu_dev, st));
    if (want_full_cov) {
        // K_aa - V V^T
        PIGP_TRY(grow(&s->T, &s->t_elems, mpad * mpad));
        PIGP_TRY(launch_assemble(test, test->d_tiles_full, test->n_tiles_full, theta_dev, 0.0, 0, s->T, mpad, st));
        PIGP_TRY(launch_pad(s->T, mpad, m, m, mpad, mpad, 0, 0, st));
        GemmDesc g{};
        g.M = (int)mpad; g.N = (int)mpad; g.K = (int)s->npad;
        g.alpha = -1.0; g.beta = 1.0;
        g.A = s->V; g.lda = ld; g.a_kcontig = 1;
        g.B = s->V; g.ldb = ld; g.b_kcontig = 1;
        g.C = s->T; g.ldc = mpad;
        PIGP_TRY(launch_gemm(g, st));
        PIGP_CUDA(cudaMemcpy2DAsync(cov_dev, sizeof(double) * m, s->T, sizeof(double) * mpad, sizeof(double) * m, m,
                                    cudaMemcpyDeviceToDevice, st));
    } else {
        // only diag(K_aa) is evaluated (M values, not M x M) and only the row norms of V are formed
        PIGP_TRY(grow(&s->kdiag, &s->kdiag_elems, mpad));
        PIGP_TRY(launch_assemble(test, test->d_tiles_diag, test->n_tiles_diag, theta_dev, 0.0, 0, s->kdiag, 0, st));
        k_rowsumsq_sub<<<(unsigned)((m + 7) / 8), 256, 0, st>>>(s->V, ld, m, s->n, s->kdiag, cov_dev);
        count_launch();
        PIGP_CUDA(cudaGetLastError());
    }
    return PIGP_OK;
}

int pigp_predict_host(pigp_solver* s, pigp_plan* mixed, pigp_plan* test, const double* theta_host, const double* y_host,
                      double eps, double* mu_host, double* cov_host, int want_full_cov, int32_t* info_host) {
    return pigp_predict_batch_host(s, mixed, test, 1, theta_host, y_host, eps, mu_host, cov_host, want_full_cov, info_host);
}

int pigp_predict_batch_host(pigp_solver* s, pigp_plan* mixed, pigp_plan* test, int n_theta, const double* thetas_host,
                            const double* y_host, double eps, double* mu_host, double* cov_host, int want_full_cov,
                            int32_t* info_host) {
    if (!s || !mixed || !test || !thetas_host || !y_host || !mu_host || !cov_host || n_theta < 1) { set_error("pigp_predict_batch_host: bad argument"); return PIGP_EINVAL; }
    PIGP_TRY(use_device(s->plan));
    const int P = s->plan->theta_len;
    const int64_t m = mixed->rows;
    const int64_t cov_each = want_full_cov ? m * m : m;
    // results of all n_theta evaluations are staged on the device and copied back once
    PIGP_TRY(grow(&s->d_mu, &s->mu_elems, m * n_theta));
    PIGP_TRY(grow(&s->d_cov, &s->cov_elems, cov_each * n_theta));
    PIGP_CUDA(cudaMemcpy(s->d_y, y_host, sizeof(double) * s->n, cudaMemcpyHostToDevice));
    int32_t worst = 0;
    for (int b = 0; b < n_theta; ++b) {
        PIGP_CUDA(cudaMemcpy(s->d_theta, thetas_host + (int64_t)b * P, sizeof(double) * P, cudaMemcpyHostToDevice));
        PIGP_TRY(pigp_predict(s, mixed, test, s->d_theta, s->d_y, eps, s->d_mu + (int64_t)b * m, s->d_cov + (int64_t)b * cov_each,
                              want_full_cov, s->info, nullptr));
        int32_t inf = 0;
        PIGP_CUDA(cudaMemcpy(&inf, s->info, sizeof(int32_t), cudaMemcpyDeviceToHost));  // also orders theta's reuse
        if (inf != 0 && worst == 0) worst = inf;
        if (info_host && n_theta > 1) info_host[b] = inf;
    }
    PIGP_CUDA(cudaMemcpy(mu_host, s->d_mu, sizeof(double) * m * n_theta, cudaMemcpyDeviceToHost));
    PIGP_CUDA(cudaMemcpy(cov_host, s->d_cov, sizeof(double) * cov_each * n_theta, cudaMemcpyDeviceToHost));
    if (info_host && n_theta == 1) *info_host = worst;
    return PIGP_OK;
}

int pigp_adam_host(pigp_solver* s, const double* theta0_host, const double* y_host, double eps, int max_iter, double lr,
                   double stop_eps, double ntraining, double ridge_alpha, int ridge_in_grad, const int32_t* fixed_host,
                   int check_every, double* theta_hist_host, double* loss_hist_host, double* norm_hist_host,
                   int32_t* n_done_host, int32_t* status_host) {
    return pigp_adam_batch_host(s, 1, theta0_host, y_host, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha, ridge_in_grad,
                                fixed_host, check_every, theta_hist_host, loss_hist_host, norm_hist_host, n_done_host, status_host);
}

int pigp_adam_batch_host(pigp_solver* s, int n_start, const double* theta0s_host, const double* y_host, double eps, int max_iter,
                         double lr, double stop_eps, double ntraining, double ridge_alpha, int ridge_in_grad,
                         const int32_t* fixed_host, int check_every, double* theta_hist_host, double* loss_hist_host,
                         double* norm_hist_host, int32_t* n_done_host, int32_t* status_host) {
    if (!s || !theta0s_host || !y_host || !theta_hist_host || !loss_hist_host || !norm_hist_host || !n_done_host || !status_host ||
        max_iter < 1 || !(ntraining > 0.0) || n_start < 1 || n_start > PIGP_MAX_BATCH || (n_start > 1 && s->world != 1)) {
        set_error("pigp_adam_host: bad argument (null pointer, max_iter < 1, ntraining <= 0, n_start outside [1, 65535], or "
                  "several starts on a sharded solver)");
        return PIGP_EINVAL;
    }
    PIGP_TRY(use_device(s->plan));
    const int P = s->plan->theta_len;
    const int64_t nb = n_start, H = (int64_t)(max_iter + 1) * P;
    if (check_every < 1) check_every = 16;
    // workspace, one array of n_start entries each: theta, m, v, grad [P], nll, prev_loss, theta / loss / norm histories;
    // integer state [4] per start, then the mask
    const size_t n_d = (size_t)nb * (4 * P + 2 + H + (max_iter + 1) + max_iter);
    double* ws = nullptr;
    int32_t* iws = nullptr;
    if (cudaMalloc(&ws, sizeof(double) * n_d) != cudaSuccess) { cudaGetLastError(); set_error("pigp_adam_host: out of memory"); return PIGP_ENOMEM; }
    if (cudaMalloc(&iws, sizeof(int32_t) * (4 * nb + MAX_THETA)) != cudaSuccess) { cudaGetLastError(); cudaFree(ws); set_error("pigp_adam_host: out of memory"); return PIGP_ENOMEM; }
    int rc = PIGP_OK;
    auto ck = [&](cudaError_t e) { if (e != cudaSuccess && rc == PIGP_OK) { set_error(std::string("pigp_adam_host: ") + cudaGetErrorString(e)); rc = PIGP_ECUDA; } };
    cudaStream_t st = s->adam_stream;
    ck(cudaMemsetAsync(ws, 0, sizeof(double) * n_d, st));
    ck(cudaMemsetAsync(iws, 0, sizeof(int32_t) * (4 * nb + MAX_THETA), st));
    AdamArgs a{};
    a.P = P; a.max_iter = max_iter; a.lr = lr; a.stop_eps = stop_eps; a.ntraining = ntraining;
    a.ridge_alpha = ridge_alpha; a.ridge_in_grad = ridge_in_grad;
    a.theta = ws; a.m = ws + nb * P; a.v = ws + 2 * nb * P;
    double* d_grad = ws + 3 * nb * P;
    double* d_nll = ws + 4 * nb * P;
    a.nll = d_nll; a.grad = d_grad;
    a.prev_loss = d_nll + nb;
    a.theta_hist = a.prev_loss + nb;
    a.loss_hist = a.theta_hist + nb * H;
    a.norm_hist = a.loss_hist + nb * (max_iter + 1);
    a.istate = iws;
    a.fixed = fixed_host ? iws + 4 * nb : nullptr;
    ck(cudaMemcpyAsync(a.theta, theta0s_host, sizeof(double) * nb * P, cudaMemcpyHostToDevice, st));
    ck(cudaMemcpyAsync(s->d_y, y_host, sizeof(double) * s->n, cudaMemcpyHostToDevice, st));
    if (fixed_host) ck(cudaMemcpyAsync(iws + 4 * nb, fixed_host, sizeof(int32_t) * P, cudaMemcpyHostToDevice, st));
    std::vector<int32_t> ist((size_t)4 * nb, 0);
    auto running = [&]() {
        for (int64_t b = 0; b < nb; ++b)
            if (ist[4 * b + 2] == 0) return true;
        return false;
    };
    // theta never leaves the device: evaluation and update are enqueued back to back, the host looks at the state only
    // every check_every iterations (a start that stopped in between leaves its remaining queued updates as no-ops)
    for (int it = 0; it < max_iter && rc == PIGP_OK && running(); it += check_every) {
        const int nk = std::min(check_every, max_iter - it);
        for (int k = 0; k < nk && rc == PIGP_OK; ++k) {
            // one start: the single-theta evaluation, which sharded solvers run too
            rc = nb == 1 ? pigp_dsolver_nll_grad(s->ds, a.theta, s->d_y, eps, d_nll, d_grad, s->info, st)
                         : pigp_nll_grad_batch(s, n_start, a.theta, s->d_y, eps, d_nll, d_grad, nullptr, st);
            if (rc == PIGP_OK) {
                k_adam_step<<<(unsigned)nb, 32, 0, st>>>(a);
                count_launch();
                ck(cudaGetLastError());
            }
        }
        ck(cudaMemcpyAsync(ist.data(), iws, sizeof(int32_t) * 4 * nb, cudaMemcpyDeviceToHost, st));
        ck(cudaStreamSynchronize(st));
    }
    for (int64_t b = 0; b < nb && rc == PIGP_OK; ++b) {
        const int done = ist[4 * b + 3];
        ck(cudaMemcpyAsync(theta_hist_host + b * H, a.theta_hist + b * H, sizeof(double) * (size_t)(done + 1) * P,
                           cudaMemcpyDeviceToHost, st));
        ck(cudaMemcpyAsync(loss_hist_host + b * (max_iter + 1), a.loss_hist + b * (max_iter + 1), sizeof(double) * (size_t)(done + 1),
                           cudaMemcpyDeviceToHost, st));
        if (done > 0)
            ck(cudaMemcpyAsync(norm_hist_host + b * max_iter, a.norm_hist + b * max_iter, sizeof(double) * (size_t)done,
                               cudaMemcpyDeviceToHost, st));
        n_done_host[b] = done;
        status_host[b] = ist[4 * b + 2];
    }
    ck(cudaStreamSynchronize(st));
    cudaFree(ws);
    cudaFree(iws);
    return rc;
}

// ------------------------------------------------------------------------------------------------ building blocks
int pigp_potrf_lower(double* A_dev, int64_t ld, int64_t n, int64_t m_extra, double* invd_dev, int32_t* info_dev, void* stream) {
    if (!A_dev || !invd_dev) { set_error("pigp_potrf_lower: null argument"); return PIGP_EINVAL; }
    if (info_dev) PIGP_CUDA(cudaMemsetAsync(info_dev, 0, sizeof(int32_t), as_stream(stream)));
    return potrf_lower(A_dev, ld, n, m_extra, invd_dev, info_dev, as_stream(stream));
}

int pigp_debug_potf2_stamps(long long* dev_buf) { return set_potf2_debug(dev_buf); }

int pigp_potri_lower(const double* L_dev, int64_t ld, int64_t n, const double* invd_dev, double* W_dev, double* X_dev, void* stream) {
    if (!L_dev || !invd_dev || !W_dev || !X_dev) { set_error("pigp_potri_lower: null argument"); return PIGP_EINVAL; }
    return potri_lower(L_dev, ld, n, invd_dev, W_dev, X_dev, as_stream(stream));
}

int pigp_dgemm(int M, int N, int K, double alpha, const double* A_dev, int64_t lda, int a_kcontig, const double* B_dev, int64_t ldb,
               int b_kcontig, double beta, double* C_dev, int64_t ldc, int lower_only, void* stream) {
    GemmDesc g{};
    g.M = M; g.N = N; g.K = K; g.alpha = alpha; g.beta = beta;
    g.A = A_dev; g.lda = lda; g.a_kcontig = a_kcontig;
    g.B = B_dev; g.ldb = ldb; g.b_kcontig = b_kcontig;
    g.C = C_dev; g.ldc = ldc; g.lower_only = lower_only;
    return launch_gemm(g, as_stream(stream));
}

// The owned lower tiles of build_lower_tiles_owned in a stream-ordered device buffer (freed by the caller with
// cudaFreeAsync on the same stream), so that neither entry point below synchronises.
static int owned_tiles(const pigp_plan* p, int rank, int world, cudaStream_t st, AsmTile** dev, int64_t* n) {
    std::vector<AsmTile> v;
    build_lower_tiles_owned(p, rank, world, v);
    *n = (int64_t)v.size();
    *dev = nullptr;
    if (v.empty()) return PIGP_OK;
    PIGP_CUDA(cudaMallocAsync(reinterpret_cast<void**>(dev), v.size() * sizeof(AsmTile), st));
    const cudaError_t e = cudaMemcpyAsync(*dev, v.data(), v.size() * sizeof(AsmTile), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) {
        cudaFreeAsync(*dev, st);
        *dev = nullptr;
        PIGP_CUDA(e);
    }
    return PIGP_OK;
}

int pigp_assemble_owned(const pigp_plan* p, int rank, int world, const double* theta_dev, double eps, int add_diag,
                        double* K_dev, int64_t ld, void* stream) {
    if (!p || !p->symmetric || !theta_dev || !K_dev || world < 1 || rank < 0 || rank >= world || ld < p->cols) {
        set_error("pigp_assemble_owned: needs a symmetric plan, 0 <= rank < world, ld >= cols and device buffers");
        return PIGP_EINVAL;
    }
    PIGP_TRY(use_device(p));
    const cudaStream_t st = as_stream(stream);
    AsmTile* tiles = nullptr;
    int64_t n = 0;
    PIGP_TRY(owned_tiles(p, rank, world, st, &tiles, &n));
    const int rc = launch_assemble(p, tiles, n, theta_dev, eps, add_diag, K_dev, ld, st);
    if (tiles) PIGP_CUDA(cudaFreeAsync(tiles, st));
    return rc;
}

int pigp_trace_grad(const pigp_plan* p, int rank, int world, const double* theta_dev, const double* X_dev, int64_t ld,
                    const double* alpha_dev, double* grad_dev, void* stream) {
    if (!p || !p->symmetric || !theta_dev || !X_dev || !alpha_dev || !grad_dev || world < 1 || rank < 0 || rank >= world ||
        ld < p->cols) {
        set_error("pigp_trace_grad: needs a symmetric plan, 0 <= rank < world, ld >= cols and device buffers");
        return PIGP_EINVAL;
    }
    PIGP_TRY(use_device(p));
    const cudaStream_t st = as_stream(stream);
    AsmTile* tiles = nullptr;
    int64_t n = 0;
    PIGP_TRY(owned_tiles(p, rank, world, st, &tiles, &n));
    double* partials = nullptr;
    int rc = PIGP_OK;
    const cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&partials), sizeof(double) * MAX_THETA * std::max<int64_t>(n, 1), st);
    if (e != cudaSuccess) {
        set_error(std::string("pigp_trace_grad: cudaMallocAsync: ") + cudaGetErrorString(e));
        rc = PIGP_ECUDA;
    }
    if (rc == PIGP_OK) rc = launch_grad(p, tiles, n, theta_dev, X_dev, ld, alpha_dev, partials, grad_dev, st);
    if (partials) cudaFreeAsync(partials, st);
    if (tiles) cudaFreeAsync(tiles, st);
    return rc;
}

}  // extern "C"
