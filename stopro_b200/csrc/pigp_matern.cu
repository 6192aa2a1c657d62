// Block evaluator for the Matern-5/2, 7/2 and 9/2 kernels of the reference (GP/kernels.py:127-205), under the same
// differential operators, block tables, layouts and gradient reduction as the squared-exponential path
// (pigp_assemble.cu) -- SURVEY.md 8(f) row n4.
//
// One-dimensional factor:  M(s) = q(rho) exp(-rho),  rho = c |s|,  c = kappa / l
//     mt52: kappa = sqrt 5, q = 1 + rho + rho^2/3            mt72: kappa = sqrt 7, q = 1 + rho + 2 rho^2/5 + rho^3/15
//     mt92: kappa = 3,      q = 1 + rho + 3 rho^2/7 + 2 rho^3/21 + rho^4/105
//     (d/ds)^n M = c^n sgn(s)^n q_n(rho) exp(-rho),  q_{n+1} = q_n' - q_n
//     d/dlog l [c^n q_n(rho) e^-rho] = c^n e^-rho u_n(rho),  u_n = -n q_n + rho (q_n - q_n')
// Autodiff quirk kept for parity: the reference differentiates through jnp.abs (derivative sgn(0) = 0 at the origin), so
// for s = 0 every derivative of order >= 1 is 0 -- sgn(s)^n with sgn(0) = 0 -- also the even ones.
// This path is written for coverage, not speed: one thread per entry, terms evaluated one by one.
#include <mutex>

#include "pigp_internal.cuh"

namespace pigp {

// [kind 0..2 = 52, 72, 92][n 0..4][0: q_n, 1: u_n][ascending coefficients, degree <= 5]
__constant__ double c_mat[3][5][2][6];
__constant__ double c_kappa[3];

static void poly_tables(double out[3][5][2][6], double kappa[3]) {
    // q scaled by a common denominator, so that the recurrences run on exact integers: a coefficient that is 0 (the
    // constant term of q_3 for mt52 and mt72, which makes the third derivative vanish at s = 0) stays exactly 0, and every
    // other one is rounded once, by the final division
    const double base[3][5] = {{3, 3, 1, 0, 0}, {15, 15, 6, 1, 0}, {105, 105, 45, 10, 1}};
    const double denom[3] = {3, 15, 105};
    kappa[0] = sqrt(5.0); kappa[1] = sqrt(7.0); kappa[2] = 3.0;
    for (int k = 0; k < 3; ++k) {
        double q[6] = {base[k][0], base[k][1], base[k][2], base[k][3], base[k][4], 0.0};
        for (int n = 0; n < 5; ++n) {
            double dq[6] = {0, 0, 0, 0, 0, 0};
            for (int i = 0; i < 5; ++i) dq[i] = (i + 1) * q[i + 1];
            for (int i = 0; i < 6; ++i) out[k][n][0][i] = q[i] / denom[k];
            // u = -n q + rho (q - q')
            for (int i = 0; i < 6; ++i) out[k][n][1][i] = (-n * q[i] + (i > 0 ? q[i - 1] - dq[i - 1] : 0.0)) / denom[k];
            for (int i = 0; i < 6; ++i) q[i] = dq[i] - q[i];  // q_{n+1}
        }
    }
}

static int upload_tables() {
    static std::once_flag once[64];
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    cudaError_t err = cudaSuccess;
    std::call_once(once[dev & 63], [&] {
        double t[3][5][2][6], kappa[3];
        poly_tables(t, kappa);
        err = cudaMemcpyToSymbol(c_mat, t, sizeof(t));
        if (err == cudaSuccess) err = cudaMemcpyToSymbol(c_kappa, kappa, sizeof(kappa));
    });
    if (err != cudaSuccess) { set_error(std::string("matern tables: ") + cudaGetErrorString(err)); return PIGP_ECUDA; }
    return PIGP_OK;
}

__device__ __forceinline__ double horner6(const double* c, double x) {
    double acc = c[5];
#pragma unroll
    for (int i = 4; i >= 0; --i) acc = fma(acc, x, c[i]);
    return acc;
}

// factor of order n in one dimension, without exp(-rho): (value, d/dlog l)
__device__ __forceinline__ void mat_factor(int kind, int n, double s, double c, double rho, double& f, double& df) {
    const double q = horner6(c_mat[kind][n][0], rho), u = horner6(c_mat[kind][n][1], rho);
    double pref = 1.0;
    if (n > 0) {
        const double sg = (s > 0.0) ? 1.0 : ((s < 0.0) ? -1.0 : 0.0);
        pref = (n & 1) ? sg : sg * sg;
        double cn = c;
        for (int i = 1; i < n; ++i) cn *= c;
        pref *= cn;
    }
    f = pref * q;
    df = pref * u;
}

struct MatShared {
    pigp_block_desc sd;
    double gamma[PIGP_MAX_GROUPS], c[PIGP_MAX_GROUPS][3];
    double noise;
    double red[8][1 + 3];
};

// value of the block at first - second = s (already with the shifts applied), restricted to the terms of group g (g < 0:
// all groups); GRAD: also d/d[log gamma, log l_0 ..] of that group into dv[0 .. DIM]
template <int DIM, bool PRODUCT, bool GRAD>
__device__ __forceinline__ double mat_eval(const MatShared& sh, int kind, const double* s, int g_only, double* dv) {
    double val = 0.0;
    const int nt = sh.sd.n_terms;
    for (int t = 0; t < nt; ++t) {
        const int g = sh.sd.terms[t].group;
        if (g_only >= 0 && g != g_only) continue;
        double f[DIM], df[DIM], esum = 0.0;
        bool on[DIM];
#pragma unroll
        for (int d = 0; d < DIM; ++d) {
            const int n = sh.sd.terms[t].order[d];
            on[d] = PRODUCT || n >= 0;
            f[d] = 1.0;
            df[d] = 0.0;
            if (on[d]) {
                const double rho = sh.c[g][d] * fabs(s[d]);
                mat_factor(kind, max(n, 0), s[d], sh.c[g][d], rho, f[d], df[d]);
                esum += rho;
            }
        }
        const double w = sh.sd.terms[t].coef * sh.gamma[g] * exp(-esum);
        double all = w;
#pragma unroll
        for (int d = 0; d < DIM; ++d) all *= f[d];
        val += all;
        if (GRAD) {
            dv[0] += all;
#pragma unroll
            for (int e = 0; e < DIM; ++e) {
                if (!on[e]) continue;
                double pe = w * df[e];
#pragma unroll
                for (int d = 0; d < DIM; ++d)
                    if (d != e) pe *= f[d];
                dv[1 + e] += pe;
            }
        }
    }
    return val;
}

template <int DIM, bool PRODUCT, bool GRAD, bool BATCH>
__global__ void __launch_bounds__(256) k_blocks_matern(AsmArgs a, int kind) {
    __shared__ MatShared sh;
    if (BATCH) slot_args(a);
    const AsmTile tl = a.tiles[blockIdx.x];
    const int tid = threadIdx.x;
    const bool live = tl.desc >= 0;
    if (live) {
        const int* src = reinterpret_cast<const int*>(&a.table[tl.desc]);
        int* dst = reinterpret_cast<int*>(&sh.sd);
        for (int i = tid; i < (int)(sizeof(pigp_block_desc) / sizeof(int)); i += 256) dst[i] = src[i];
    }
    if (tid < a.n_groups) {
        const double* th = a.theta + tid * (1 + DIM);
        sh.gamma[tid] = exp(th[0]);
#pragma unroll
        for (int d = 0; d < DIM; ++d) sh.c[tid][d] = c_kappa[kind] * exp(-th[1 + d]);
    }
    if (tid == 32) sh.noise = a.has_noise ? exp(a.theta[a.n_groups * (1 + DIM)]) : 0.0;
    __syncthreads();
    const bool swap = tl.flags & ASM_SWAP, lower = tl.flags & ASM_LOWER;
    const int sfm = live ? sh.sd.shift_first : 0, ssm = live ? sh.sd.shift_second : 0;
    const int n_entries = tl.nrows * tl.ncols;

    auto entry = [&](int e, int g_only, double* dv) {
        const int lr = e / tl.ncols, lc = e % tl.ncols;
        const int64_t R = tl.row0 + lr, C = tl.col0 + lc;
        double first0[DIM], second0[DIM];
#pragma unroll
        for (int d = 0; d < DIM; ++d) {
            const double xr = a.pts_row[d * a.n_row_pts + R], xc = a.pts_col[d * a.n_col_pts + C];
            first0[d] = swap ? xc : xr;
            second0[d] = swap ? xr : xc;
        }
        double val = 0.0;
        for (int sf = 0; sf <= sfm; ++sf)
            for (int ss = 0; ss <= ssm; ++ss) {
                const double sign = ((sfm - sf + ssm - ss) & 1) ? -1.0 : 1.0;
                double s[DIM], part[1 + DIM];
#pragma unroll
                for (int d = 0; d < DIM; ++d) {
                    // the shifted point is formed first (r + lbox), then the difference, as in GP/gp.py:381, 392
                    const double f = sf ? first0[d] + a.lbox[d] : first0[d];
                    const double g = ss ? second0[d] + a.lbox[d] : second0[d];
                    s[d] = f - g;
                }
#pragma unroll
                for (int d = 0; d <= DIM; ++d) part[d] = 0.0;
                val += sign * mat_eval<DIM, PRODUCT, GRAD>(sh, kind, s, g_only, part);
                if (GRAD)
#pragma unroll
                    for (int d = 0; d <= DIM; ++d) dv[d] += sign * part[d];
            }
        return val;
    };

    if (!GRAD) {
        for (int e = tid; e < n_entries; e += 256) {
            const int lr = e / tl.ncols, lc = e % tl.ncols;
            const int64_t R = tl.row0 + lr, C = tl.col0 + lc;
            if (lower && C > R) continue;
            if ((tl.flags & ASM_DIAG) && R != C) continue;
            double v = live ? entry(e, -1, nullptr) : 0.0;
            if (R == C && a.add_diag) v += diag_addon(a, R, sh.noise);
            if (tl.flags & ASM_DIAG) { a.K[R] = v; continue; }
            a.K[R * a.ld + C] = v;
            if ((tl.flags & ASM_MIRROR) && C < R) a.K[C * a.ld + R] = v;
        }
    } else {
        double* out = a.partials + (int64_t)blockIdx.x * MAX_THETA;
        const int noise_idx = a.n_groups * (1 + DIM);
        for (int g = 0; g <= a.n_groups; ++g) {  // g == n_groups: the noise parameter
            double acc[1 + DIM];
#pragma unroll
            for (int d = 0; d <= DIM; ++d) acc[d] = 0.0;
            for (int e = tid; e < n_entries; e += 256) {
                const int lr = e / tl.ncols, lc = e % tl.ncols;
                const int64_t R = tl.row0 + lr, C = tl.col0 + lc;
                if (lower && C > R) continue;
                const double w = ((lower && C == R) ? 1.0 : 2.0) * (a.X[R * a.ld + C] - a.alpha[R] * a.alpha[C]);
                if (g == a.n_groups) {
                    if (a.has_noise && R == C && R >= a.noise_lo && R < a.noise_hi) acc[0] += w * sh.noise;
                } else if (live) {
                    double dv[1 + DIM];
#pragma unroll
                    for (int d = 0; d <= DIM; ++d) dv[d] = 0.0;
                    entry(e, g, dv);
#pragma unroll
                    for (int d = 0; d <= DIM; ++d) acc[d] = fma(w, dv[d], acc[d]);
                }
            }
            // deterministic CTA reduction: warp shuffles, then the 8 warp sums in order
#pragma unroll
            for (int d = 0; d <= DIM; ++d) {
                double v = acc[d];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if ((tid & 31) == 0) sh.red[tid >> 5][d] = v;
            }
            __syncthreads();
            if (tid <= DIM) {
                double v = 0.0;
                for (int k = 0; k < 8; ++k) v += sh.red[k][tid];
                if (g < a.n_groups) out[g * (1 + DIM) + tid] = v;
                else if (tid == 0 && a.has_noise) out[noise_idx] = v;
            }
            __syncthreads();
        }
    }
}

template <int DIM, bool PRODUCT, bool GRAD>
static void launch_k(const AsmArgs& a, int64_t n_tiles, int kind, cudaStream_t st) {
    const dim3 grid((unsigned)n_tiles, (unsigned)a.nb), block(256);
    if (a.nb > 1) k_blocks_matern<DIM, PRODUCT, GRAD, true><<<grid, block, 0, st>>>(a, kind);
    else k_blocks_matern<DIM, PRODUCT, GRAD, false><<<grid, block, 0, st>>>(a, kind);
}

template <bool GRAD>
static int launch_t(const pigp_plan* p, const AsmArgs& a, int64_t n_tiles, int kind, cudaStream_t st) {
    ProfScope prof(GRAD ? PROF_GRAD : PROF_ASSEMBLE, st);
    if (p->dim == 1) launch_k<1, true, GRAD>(a, n_tiles, kind, st);
    else if (p->dim == 2) {
        if (p->product_form) launch_k<2, true, GRAD>(a, n_tiles, kind, st);
        else launch_k<2, false, GRAD>(a, n_tiles, kind, st);
    } else {
        if (p->product_form) launch_k<3, true, GRAD>(a, n_tiles, kind, st);
        else launch_k<3, false, GRAD>(a, n_tiles, kind, st);
    }
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

int launch_blocks_matern(const pigp_plan* p, const AsmArgs& a, int64_t n_tiles, bool grad, cudaStream_t st) {
    const int kind = p->kernel_type == 52 ? 0 : (p->kernel_type == 72 ? 1 : 2);
    PIGP_TRY(upload_tables());
    return grad ? launch_t<true>(p, a, n_tiles, kind, st) : launch_t<false>(p, a, n_tiles, kind, st);
}

int preload_matern() {
    PIGP_TRY(upload_tables());
    PIGP_PRELOAD((k_blocks_matern<1, true, false, false>)); PIGP_PRELOAD((k_blocks_matern<1, true, true, false>));
    PIGP_PRELOAD((k_blocks_matern<2, true, false, false>)); PIGP_PRELOAD((k_blocks_matern<2, true, true, false>));
    PIGP_PRELOAD((k_blocks_matern<2, false, false, false>)); PIGP_PRELOAD((k_blocks_matern<2, false, true, false>));
    PIGP_PRELOAD((k_blocks_matern<3, true, false, false>)); PIGP_PRELOAD((k_blocks_matern<3, true, true, false>));
    PIGP_PRELOAD((k_blocks_matern<3, false, false, false>)); PIGP_PRELOAD((k_blocks_matern<3, false, true, false>));
    return PIGP_OK;
}

}  // namespace pigp
