// FP64 dense linear algebra for the PIGP path on sm_100a (K3/K4/K5/K7).
//
// Replaces the library calls of the reference: jnp.linalg.cholesky (GP/gp.py:83, :106, :430), the general
// jnp.linalg.solve calls on the triangular factor (:84, :109, :118, :432-433) and the per-parameter
// Sigma_inv @ dK matmuls (:481-485).
//
// * k_gemm: C = alpha * A * B^T + beta * C on 128 x 128 tiles, operands staged through shared memory by a
//   3-stage cp.async pipeline, the products issued as FP64 tensor-core MMAs (mma.sync.m8n8k4.f64, SASS DMMA.8x8x4;
//   tcgen05 has no f64 kind).  Either index of A / B may be the contiguous one, k-ranges can follow a triangular
//   operand tile by tile and tiles above the diagonal can be skipped, so that the same kernel is the SYRK/GEMM
//   trailing update of the Cholesky, the TRSM-by-inverse, both TRTRI products and the LAUUM.
// * k_potf2: one CTA factors a 128 x 128 diagonal tile in shared memory (32 x 32 blocks: one warp eliminates column pairs,
//   a second warp inverts the block behind it); k_tile_inv completes inverse tiles off the critical path.
// * k_trsm_blk: the panel solve X = A inv(L_kk)^T by block forward substitution with refined 32 x 32 diagonal solves.
// * Host drivers: TRTRI + LAUUM for K^-1.  The Cholesky that drives k_potf2, k_trsm_blk and k_gemm is in pigp_dist.cu.
#include <algorithm>
#include <cstdlib>

#include "pigp_internal.cuh"

namespace pigp {

// ----------------------------------------------------------------------------------------------- GEMM
constexpr int BM = 128;
#ifndef PIGP_GEMM_BK
#define PIGP_GEMM_BK 16
#endif
constexpr int BK = PIGP_GEMM_BK;
// Shared-memory operand tiles.  Fragments are fetched with 16-byte loads (two k values, or two rows, per load):
//   k-contiguous operand  [128][BK + 8]  row stride = 8 mod 16 doubles  -> the 8 lanes of a quarter warp hit 8 distinct 16-byte slots
//   m-contiguous operand  [BK][130]      row stride = 2 mod 8 doubles   -> same property for the (k, row-pair) pattern
constexpr int LDS_K = BK + 8;
__host__ __device__ constexpr int lds_m(int rows) { return rows + 2; }
__host__ __device__ constexpr int opd(int rows) { return (rows * LDS_K > BK * lds_m(rows)) ? rows * LDS_K : BK * lds_m(rows); }  // doubles per operand tile
__host__ __device__ constexpr int gemm_smem(int bn, int stages) { return stages * (opd(BM) + opd(bn)) * (int)sizeof(double); }
constexpr int SUPER = 12;  // tiles are issued in 12 x 12 super-tiles so that the ~148 resident CTAs share operand panels in L2

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}
// Shared-memory mbarriers (producer / consumer hand-off between warps of a CTA)
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("{\n .reg .b64 t;\n mbarrier.arrive.shared::cta.b64 t, [%0];\n}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, int parity) {
    const unsigned addr = (unsigned)__cvta_generic_to_shared(bar);
    unsigned ok;
    do {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <bool KC, int ROWS, int THREADS>
__device__ __forceinline__ void load_operand(double* sm, const double* G, int64_t ld, int64_t row0, int64_t k0, int tid) {
    constexpr int PER_THREAD = ROWS * BK / 2 / THREADS;
    if (KC) {  // X(row, k) = G[row*ld + k]: ROWS rows x BK doubles, BK/2 16-byte chunks per row
#pragma unroll
        for (int i = 0; i < PER_THREAD; ++i) {
            const int c = tid + i * THREADS;
            const int r = c / (BK / 2), ch = c % (BK / 2);
            cp_async16(sm + r * LDS_K + ch * 2, G + (row0 + r) * ld + k0 + ch * 2);
        }
    } else {   // X(row, k) = G[k*ld + row]: BK k-rows x ROWS doubles, ROWS/2 chunks per k-row
#pragma unroll
        for (int i = 0; i < PER_THREAD; ++i) {
            const int c = tid + i * THREADS;
            const int kr = c / (ROWS / 2), ch = c % (ROWS / 2);
            cp_async16(sm + kr * lds_m(ROWS) + ch * 2, G + (k0 + kr) * ld + row0 + ch * 2);
        }
    }
}

// Fragments of one 8-wide k group for NT 8-row sub-tiles starting at row `base` of the operand tile.
// frag[i].x feeds the MMA over k = {0,2,4,6} + k8 (lane tig supplies k8 + 2 tig), frag[i].y the one over {1,3,5,7} + k8.
// k-contiguous: sub-tile i = rows base + 8 i + gid.  m-contiguous: sub-tiles (2p, 2p+1) = rows base + 16 p + 2 gid + {0, 1}.
template <bool KC, int NT, int ROWS>
__device__ __forceinline__ void load_frags(double2* frag, const double* sm, int base, int k8, int gid, int tig) {
    if (KC) {
#pragma unroll
        for (int i = 0; i < NT; ++i)
            frag[i] = *reinterpret_cast<const double2*>(sm + (base + 8 * i + gid) * LDS_K + k8 + 2 * tig);
    } else {
#pragma unroll
        for (int p = 0; p < NT / 2; ++p) {
            const double2 e = *reinterpret_cast<const double2*>(sm + (k8 + 2 * tig) * lds_m(ROWS) + base + 16 * p + 2 * gid);
            const double2 o = *reinterpret_cast<const double2*>(sm + (k8 + 2 * tig + 1) * lds_m(ROWS) + base + 16 * p + 2 * gid);
            frag[2 * p] = make_double2(e.x, o.x);
            frag[2 * p + 1] = make_double2(e.y, o.y);
        }
    }
}

// the slot's operands (batched launches: once, at kernel entry)
__device__ __forceinline__ void slot_ptrs(GemmDesc& g) {
    const int64_t b = blockIdx.y;
    g.A += b * g.sa;
    g.B += b * g.sb;
    g.C += b * g.sc;
    if (g.Lkk) g.Lkk += b * g.sl;
}

// Bounded spin on epoch flags written by peers (st.release.sys); see pigp_dist.cu.
__device__ __forceinline__ void wait_flags(const GemmDesc& g, int tid) {
    if (g.wait_count <= 0) return;
    if (tid < g.wait_count && tid != g.wait_skip && *reinterpret_cast<volatile int*>(g.wait_err) == 0) {
        const unsigned long long* p = g.wait_flags + g.wait_idx0 + (int64_t)tid * g.wait_stride;
        unsigned long long t0, now, v;
        asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t0));
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
            if (v >= g.wait_val) break;
            asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
            if (now - t0 > g.wait_timeout_ns) { atomicExch(g.wait_err, 1); break; }
            __nanosleep(64);
        }
    }
    __syncthreads();
}

// BN_ = 128: 8 warps, one CTA per SM.  BN_ = 64: 4 warps, two CTAs per SM (independent barriers: while one CTA waits at its
// barrier or on shared-memory loads, the other keeps the FP64 tensor pipe busy).
// BATCH: the launch covers g.nb slots (grid dimension y).  The kernels that can be batched are instantiated twice: the
// single-slot instantiation is the kernel as it was before batching existed, instruction for instruction.
template <bool AKC, bool BKC, int BN_, int STAGES_, bool BATCH>
__global__ void __launch_bounds__(BN_ * 2, 128 / BN_) k_gemm(GemmDesc g) {
    constexpr int THREADS = BN_ * 2;
    constexpr int OPA = opd(BM), OPB = opd(BN_), STG = OPA + OPB;
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gid = lane >> 2, tig = lane & 3;
    const int wm = warp & 1, wn = warp >> 1;  // 2 x (BN_/32) warps, warp tile 64 x 32

    const int nt = g.N / BN_;
    const int mt = (g.lower_only && !g.gen) ? g.N / BM : g.M / BM;  // a plain lower_only launch covers the square part only
    int tm, tn;
    {
        constexpr int SN = SUPER * (BM / BN_);  // column tiles per super-tile (super-tiles are square in elements)
        const int sidx = blockIdx.x / (SUPER * SN), local = blockIdx.x % (SUPER * SN);
        int sm_, sn_;
        if (g.lower_only && !g.gen) {  // super-tiles in lower-triangular order
            sm_ = (int)((sqrt(8.0 * sidx + 1.0) - 1.0) * 0.5);
            while ((sm_ + 1) * (sm_ + 2) / 2 <= sidx) ++sm_;
            while (sm_ * (sm_ + 1) / 2 > sidx) --sm_;
            sn_ = sidx - sm_ * (sm_ + 1) / 2;
        } else {
            const int smt = (mt + SUPER - 1) / SUPER;
            sm_ = sidx % smt;
            sn_ = sidx / smt;
        }
        tm = sm_ * SUPER + local % SUPER;
        tn = sn_ * SN + local / SUPER;
        if (tm >= mt || tn >= nt) return;
    }
    const int gm = g.m_gt0 + tm * g.m_ts;  // global row tile (== tm for a plain GEMM)
    if (g.lower_only && (int64_t)g.n_gt0 * BM + (int64_t)tn * BN_ > (int64_t)gm * BM + (BM - BN_)) return;
    const int64_t m0 = (int64_t)tm * g.m_ts * BM, n0 = (int64_t)tn * BN_;
    int kt_begin = 0, kt_end = g.K / BK;
    if (g.kmode == 1) kt_begin = max(0, gm - g.k_gt0) * (BM / BK);
    else if (g.kmode == 2) kt_end = min(kt_end, (gm - g.k_gt0 + 1) * (BM / BK));
    if (kt_end <= kt_begin && g.beta == 1.0) return;  // nothing to add
    wait_flags(g, tid);
    if (BATCH) slot_ptrs(g);

    double acc[8][4][2];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int nk = kt_end - kt_begin;
#pragma unroll
    for (int s = 0; s < STAGES_ - 1; ++s) {
        if (s < nk) {
            load_operand<AKC, BM, THREADS>(smem + s * STG, g.A, g.lda, m0, (int64_t)(kt_begin + s) * BK, tid);
            load_operand<BKC, BN_, THREADS>(smem + s * STG + OPA, g.B, g.ldb, n0, (int64_t)(kt_begin + s) * BK, tid);
        }
        cp_async_commit();
    }
    for (int it = 0; it < nk; ++it) {
        cp_async_wait<STAGES_ - 2>();
        __syncthreads();
        {
            const int nx = it + STAGES_ - 1;
            if (nx < nk) {
                const int s = nx % STAGES_;
                load_operand<AKC, BM, THREADS>(smem + s * STG, g.A, g.lda, m0, (int64_t)(kt_begin + nx) * BK, tid);
                load_operand<BKC, BN_, THREADS>(smem + s * STG + OPA, g.B, g.ldb, n0, (int64_t)(kt_begin + nx) * BK, tid);
            }
            cp_async_commit();
        }
        const double* sA = smem + (it % STAGES_) * STG;
        const double* sB = sA + OPA;
#pragma unroll
        for (int k8 = 0; k8 < BK; k8 += 8) {
            double2 af[8], bf[4];
            load_frags<AKC, 8, BM>(af, sA, wm * 64, k8, gid, tig);
            load_frags<BKC, 4, BN_>(bf, sB, wn * 32, k8, gid, tig);
#pragma unroll
            for (int mi = 0; mi < 8; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], af[mi].x, bf[ni].x);
#pragma unroll
            for (int mi = 0; mi < 8; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], af[mi].y, bf[ni].y);
        }
    }
    cp_async_wait<0>();

    // epilogue.  Row of (sub-tile mi, lane group gid): 8 mi + gid (k-contiguous A) or 16 (mi/2) + 2 gid + (mi & 1).
    // Columns: k-contiguous B: sub-tile ni holds columns 8 ni + 2 tig + {0,1}; m-contiguous B: the pair (2q, 2q+1) holds
    // the four columns 16 q + 4 tig + {0,1,2,3} = {acc[2q][0], acc[2q+1][0], acc[2q][1], acc[2q+1][1]}.
#pragma unroll
    for (int mi = 0; mi < 8; ++mi) {
        const int lr = AKC ? (8 * mi + gid) : (16 * (mi >> 1) + 2 * gid + (mi & 1));
        double* crow = g.C + (m0 + wm * 64 + lr) * g.ldc + n0 + wn * 32;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            double v[4];
            int c0, c1;
            if (BKC) {
                v[0] = acc[mi][2 * q][0]; v[1] = acc[mi][2 * q][1]; v[2] = acc[mi][2 * q + 1][0]; v[3] = acc[mi][2 * q + 1][1];
                c0 = 16 * q + 2 * tig;
                c1 = c0 + 8;
            } else {
                v[0] = acc[mi][2 * q][0]; v[1] = acc[mi][2 * q + 1][0]; v[2] = acc[mi][2 * q][1]; v[3] = acc[mi][2 * q + 1][1];
                c0 = 16 * q + 4 * tig;
                c1 = c0 + 2;
            }
            double2* p0 = reinterpret_cast<double2*>(crow + c0);
            double2* p1 = reinterpret_cast<double2*>(crow + c1);
            double2 o0 = make_double2(g.alpha * v[0], g.alpha * v[1]);
            double2 o1 = make_double2(g.alpha * v[2], g.alpha * v[3]);
            if (g.beta != 0.0) {
                const double2 a0 = *p0, a1 = *p1;
                o0.x = fma(g.beta, a0.x, o0.x); o0.y = fma(g.beta, a0.y, o0.y);
                o1.x = fma(g.beta, a1.x, o1.x); o1.y = fma(g.beta, a1.y, o1.y);
            }
            *p0 = o0;
            *p1 = o1;
            if (g.npeers > 0 && gm < g.push_gm_end) {
                const int64_t off = (crow - g.C) + c0, d1 = c1 - c0;
                for (int p = 0; p < g.npeers; ++p) {
                    double* q = g.Cpeer[p] + off;
                    *reinterpret_cast<double2*>(q) = o0;
                    *reinterpret_cast<double2*>(q + d1) = o1;
                }
            }
        }
    }
}

template <int BN_, int STAGES_, bool BATCH>
static int gemm_attrs_b() {
    constexpr int SMEM = gemm_smem(BN_, STAGES_);
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm<true, true, BN_, STAGES_, BATCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm<true, false, BN_, STAGES_, BATCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm<false, true, BN_, STAGES_, BATCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm<false, false, BN_, STAGES_, BATCH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    PIGP_PRELOAD((k_gemm<true, true, BN_, STAGES_, BATCH>));
    PIGP_PRELOAD((k_gemm<true, false, BN_, STAGES_, BATCH>));
    PIGP_PRELOAD((k_gemm<false, true, BN_, STAGES_, BATCH>));
    PIGP_PRELOAD((k_gemm<false, false, BN_, STAGES_, BATCH>));
    return PIGP_OK;
}
template <int BN_, int STAGES_>
static int gemm_attrs() {
    PIGP_TRY((gemm_attrs_b<BN_, STAGES_, false>()));
    return gemm_attrs_b<BN_, STAGES_, true>();
}

// ----------------------------------------------------------------------------------------------- small-tile GEMM
// Same contract as k_gemm for k-contiguous A and B in `gen` addressing, with BM_ x BN_ CTA tiles (BM_ = 32 or 64) for
// the latency-bound launches of the factorisation (the K = 128 TRSM by the inverse diagonal tile, the low levels of
// the trailing updates): 4-8 x more CTAs than 128 x 64 tiles, so that a 26-row-tile panel still covers the GPU.
// BN_ = 128 with N = 128 is safe in place (C aliasing A): a CTA reads all 128 columns of its rows before it writes.
template <int BM_, int BN_, int STAGES_, bool BATCH>
__global__ void __launch_bounds__(BN_ * 2) k_gemm_s(GemmDesc g) {
    constexpr int THREADS = BN_ * 2;
    constexpr int MI = BM_ / 16;  // 8-row MMA tiles per warp (2 warps along M)
    constexpr int OPA = BM_ * LDS_K, OPB = BN_ * LDS_K, STG = OPA + OPB;
    extern __shared__ __align__(16) double smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gid = lane >> 2, tig = lane & 3;
    const int wm = warp & 1, wn = warp >> 1;

    const int nt = g.N / BN_, mt = g.M / BM_;
    const int tn = blockIdx.x % nt, tm = blockIdx.x / nt;
    if (tm >= mt) return;
    constexpr int SUB = BM / BM_;                      // CTA row tiles per 128-row tile
    const int gm = g.m_gt0 + (tm / SUB) * g.m_ts;      // global 128-row tile
    const int64_t rg = (int64_t)gm * BM + (tm % SUB) * BM_, cg = (int64_t)g.n_gt0 * BM + (int64_t)tn * BN_;
    if (g.lower_only && cg >= rg + BM_) return;
    const int64_t m0 = (int64_t)(tm / SUB) * g.m_ts * BM + (tm % SUB) * BM_, n0 = (int64_t)tn * BN_;
    int kt_begin = 0, kt_end = g.K / BK;
    if (g.kmode == 1) kt_begin = max(0, gm - g.k_gt0) * (BM / BK);
    if (kt_end <= kt_begin && g.beta == 1.0) return;
    wait_flags(g, tid);
    if (BATCH) slot_ptrs(g);

    // C -= A B^T (the trailing updates on the latency-bound chain): the accumulators start from -C, fetched while the first
    // operand tiles are still in flight, instead of a read-modify-write of C after the last MMA
    const bool fold = (g.alpha == -1.0 && g.beta == 1.0);
    double acc[MI][4][2];
#pragma unroll
    for (int i = 0; i < MI; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int nk = kt_end - kt_begin;
#pragma unroll
    for (int s = 0; s < STAGES_ - 1; ++s) {
        if (s < nk) {
            load_operand<true, BM_, THREADS>(smem + s * STG, g.A, g.lda, m0, (int64_t)(kt_begin + s) * BK, tid);
            load_operand<true, BN_, THREADS>(smem + s * STG + OPA, g.B, g.ldb, n0, (int64_t)(kt_begin + s) * BK, tid);
        }
        cp_async_commit();
    }
    if (fold) {
#pragma unroll
        for (int mi = 0; mi < MI; ++mi) {
            const double* crow = g.C + (m0 + wm * (BM_ / 2) + 8 * mi + gid) * g.ldc + n0 + wn * 32;
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const double2 a0 = *reinterpret_cast<const double2*>(crow + 16 * q + 2 * tig);
                const double2 a1 = *reinterpret_cast<const double2*>(crow + 16 * q + 2 * tig + 8);
                acc[mi][2 * q][0] = -a0.x; acc[mi][2 * q][1] = -a0.y;
                acc[mi][2 * q + 1][0] = -a1.x; acc[mi][2 * q + 1][1] = -a1.y;
            }
        }
    }
    for (int it = 0; it < nk; ++it) {
        cp_async_wait<STAGES_ - 2>();
        __syncthreads();
        {
            const int nx = it + STAGES_ - 1;
            if (nx < nk) {
                const int s = nx % STAGES_;
                load_operand<true, BM_, THREADS>(smem + s * STG, g.A, g.lda, m0, (int64_t)(kt_begin + nx) * BK, tid);
                load_operand<true, BN_, THREADS>(smem + s * STG + OPA, g.B, g.ldb, n0, (int64_t)(kt_begin + nx) * BK, tid);
            }
            cp_async_commit();
        }
        const double* sA = smem + (it % STAGES_) * STG;
        const double* sB = sA + OPA;
#pragma unroll
        for (int k8 = 0; k8 < BK; k8 += 8) {
            double2 af[MI], bf[4];
            load_frags<true, MI, BM_>(af, sA, wm * (BM_ / 2), k8, gid, tig);
            load_frags<true, 4, BN_>(bf, sB, wn * 32, k8, gid, tig);
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], af[mi].x, bf[ni].x);
#pragma unroll
            for (int mi = 0; mi < MI; ++mi)
#pragma unroll
                for (int ni = 0; ni < 4; ++ni) dmma(acc[mi][ni][0], acc[mi][ni][1], af[mi].y, bf[ni].y);
        }
    }
    cp_async_wait<0>();
    if (BN_ == 128 && g.C == g.A) __syncthreads();  // in place: every warp has consumed the CTA's rows

    const bool push = g.npeers > 0 && gm < g.push_gm_end;
#pragma unroll
    for (int mi = 0; mi < MI; ++mi) {
        const int lr = 8 * mi + gid;
        double* crow = g.C + (m0 + wm * (BM_ / 2) + lr) * g.ldc + n0 + wn * 32;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int c0 = 16 * q + 2 * tig, c1 = c0 + 8;
            double2* p0 = reinterpret_cast<double2*>(crow + c0);
            double2* p1 = reinterpret_cast<double2*>(crow + c1);
            double2 o0 = make_double2(g.alpha * acc[mi][2 * q][0], g.alpha * acc[mi][2 * q][1]);
            double2 o1 = make_double2(g.alpha * acc[mi][2 * q + 1][0], g.alpha * acc[mi][2 * q + 1][1]);
            if (g.beta != 0.0 && !fold) {
                const double2 a0 = *p0, a1 = *p1;
                o0.x = fma(g.beta, a0.x, o0.x); o0.y = fma(g.beta, a0.y, o0.y);
                o1.x = fma(g.beta, a1.x, o1.x); o1.y = fma(g.beta, a1.y, o1.y);
            }
            *p0 = o0;
            *p1 = o1;
            if (push) {
                const int64_t off = (crow - g.C) + c0;
                for (int p = 0; p < g.npeers; ++p) {
                    double* qd = g.Cpeer[p] + off;
                    *reinterpret_cast<double2*>(qd) = o0;
                    *reinterpret_cast<double2*>(qd + 8) = o1;
                }
            }
        }
    }
    if (g.sig_total > 0) {
        // the last CTA to finish publishes the epoch to the peers (release: all stores above are fenced first)
        __threadfence_system();
        __syncthreads();
        if (tid == 0) {
            const unsigned int done = atomicAdd(g.sig_counter, 1u);
            if (done == (unsigned int)g.sig_total - 1u) {
                *g.sig_counter = 0u;
                __threadfence_system();
                for (int p = 0; p < g.sig_n; ++p)
                    asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(g.sig_flag[p]), "l"(g.sig_val) : "memory");
            }
        }
    }
}

template <int BM_, int BN_, int STAGES_>
static int launch_gemm_small(const GemmDesc& d, cudaStream_t st) {
    constexpr int SMEM = STAGES_ * (BM_ + BN_) * LDS_K * (int)sizeof(double);
    static bool attr_done[64] = {};
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        PIGP_CUDA(cudaFuncSetAttribute(k_gemm_s<BM_, BN_, STAGES_, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        PIGP_CUDA(cudaFuncSetAttribute(k_gemm_s<BM_, BN_, STAGES_, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        attr_done[dev & 63] = true;
    }
    const int64_t ctas = (int64_t)(d.M / BM_) * (d.N / BN_);
    double flops = 0.0;
    if (g_prof_on) {
        const int kt = d.K / BK, per = BM / BK;
        for (int t = 0; t < d.M / BM; ++t) {
            const int gm = d.m_gt0 + t * d.m_ts;
            const int ncols = d.lower_only ? std::max(0, std::min(d.N / BM, gm - d.n_gt0 + 1)) : d.N / BM;
            const int kb = d.kmode == 1 ? std::max(0, gm - d.k_gt0) * per : 0;
            flops += 2.0 * BM * BM * BK * (double)std::max(0, kt - kb) * ncols;
        }
        prof_note(d.M, d.N, d.K, 100 + d.kmode * 10 + d.lower_only);
    }
    ProfScope prof(PROF_GEMM, st, flops * d.nb);
    const dim3 grid((unsigned)ctas, (unsigned)d.nb);
    if (d.nb > 1) k_gemm_s<BM_, BN_, STAGES_, true><<<grid, BN_ * 2, SMEM, st>>>(d);
    else k_gemm_s<BM_, BN_, STAGES_, false><<<grid, BN_ * 2, SMEM, st>>>(d);
    count_launch();
    return PIGP_OK;
}

// ----------------------------------------------------------------------------------------------- block TRSM
// X = A inv(Lkk)^T for TR_BM-row slabs of a 128-column panel, in place, by forward substitution over the four 32-column
// blocks of Lkk, each diagonal solve done with the block's explicit inverse plus one refinement step:
//   T_j = A_j - sum_{i<j} X_i L_ji^T;   X0 = T_j W_j^T,  R = T_j - X0 L_jj^T,  X_j = X0 + R W_j^T      (W_j = inv(L_jj))
// Only the diagonal 32 x 32 blocks of the inverse tile are read (k_potf2 produces exactly those on the critical path; the
// rest of the tile is completed off it by k_tile_inv).  Against three full 128-deep products this is 2.7 x fewer flops, and
// the refinement acts on blocks whose condition number is far below the tile's: row-wise backward stable like LAPACK's
// substitution.  One CTA per slab, everything in shared memory after one wave of asynchronous copies; each of the 15
// barrier-separated phases is a K = 32..96 product of 8 x 8 DMMA tiles spread over the warps (all four tensor pipes).
constexpr int TB_SLD = 132, TB_LD = 36;  // row strides = 4 mod 16 doubles: conflict-free 8-byte fragment loads
__host__ __device__ constexpr int tb_smem(int bm) { return (bm * TB_SLD + 5 * bm * TB_LD + 14 * 32 * TB_LD) * (int)sizeof(double); }

// (d, e) += A[row gid][k..k+K) * B[col gid][k..k+K)^T as four independent DMMA chains (two per accumulator pair)
template <int K>
__device__ __forceinline__ void tile_mma(double (&d)[2], double (&e)[2], const double* Arow, const double* Brow, int tig) {
    double a[K / 4], b[K / 4];
#pragma unroll
    for (int q = 0; q < K / 4; ++q) {
        a[q] = Arow[4 * q + tig];
        b[q] = Brow[4 * q + tig];
    }
    double f[2] = {0.0, 0.0}, h[2] = {0.0, 0.0};
#pragma unroll
    for (int q = 0; q < K / 4; q += 4) {
        dmma(d[0], d[1], a[q], b[q]);
        dmma(e[0], e[1], a[q + 1], b[q + 1]);
        dmma(f[0], f[1], a[q + 2], b[q + 2]);
        dmma(h[0], h[1], a[q + 3], b[q + 3]);
    }
    d[0] += f[0]; d[1] += f[1];
    e[0] += h[0]; e[1] += h[1];
}

template <int TR_BM, bool BATCH>
__global__ void __launch_bounds__(256) k_trsm_blk(GemmDesc g) {
    constexpr int N_TILES = TR_BM / 8 * 4;                 // 8 x 8 tiles of one TR_BM x 32 block
    constexpr int TPW = N_TILES >= 8 ? N_TILES / 8 : 1;    // tiles per warp
    extern __shared__ __align__(16) double smem[];
    double* S = smem;                         // TR_BM x 128: A, then per block T / R
    double* Xb = S + TR_BM * TB_SLD;          // 4 solved blocks, TR_BM x 32 each
    double* X0 = Xb + 4 * TR_BM * TB_LD;      // TR_BM x 32
    double* Ls = X0 + TR_BM * TB_LD;          // blocks (jb, ib <= jb) of Lkk at index jb (jb + 1) / 2 + ib, 32 x 32 each
    double* Ws = Ls + 10 * 32 * TB_LD;        // the four diagonal blocks of inv(Lkk)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gid = lane >> 2, tig = lane & 3;
    constexpr int SUB = BM / TR_BM;
    const int tm = blockIdx.x;
    const int64_t m0 = (int64_t)(tm / SUB) * g.m_ts * BM + (tm % SUB) * TR_BM;
    wait_flags(g, tid);
    if (BATCH) slot_ptrs(g);
    // one group of asynchronous copies per column block: what step jb needs (its 32 columns of the slab, row jb of the
    // blocks of Lkk, W_jb) arrives while steps 0 .. jb - 1 compute.  Thread (lr, lch) copies 16 bytes of rows lr and
    // lr + 16 of every 32 x 32 block: all offsets are compile-time multiples of the row strides (the issue of these ~30
    // copies per thread was 45 % of the kernel with per-copy index arithmetic).
    {
        const int lr = tid >> 4, lch = (tid & 15) * 2;
        const double* srcA = g.A + (m0 + lr) * g.lda + lch;
        const double* srcL = g.Lkk + (int64_t)lr * g.ldl + lch;
        const double* srcW = g.B + (int64_t)lr * g.ldb + lch;
        double* dstS = S + lr * TB_SLD + lch;
        double* dstL = Ls + lr * TB_LD + lch;
        double* dstW = Ws + lr * TB_LD + lch;
        const int64_t l16 = 16 * (int64_t)g.ldl, w16 = 16 * (int64_t)g.ldb;
#pragma unroll
        for (int jb = 0; jb < 4; ++jb) {
            if (lr < TR_BM) cp_async16(dstS + 32 * jb, srcA + 32 * jb);
            if (TR_BM > 16) cp_async16(dstS + 16 * TB_SLD + 32 * jb, srcA + 16 * g.lda + 32 * jb);
            const double* rowL = srcL + 2 * jb * l16;
#pragma unroll
            for (int ib = 0; ib <= jb; ++ib) {
                double* d = dstL + (jb * (jb + 1) / 2 + ib) * 32 * TB_LD;
                cp_async16(d, rowL + 32 * ib);
                cp_async16(d + 16 * TB_LD, rowL + l16 + 32 * ib);
            }
            const double* rowW = srcW + 2 * jb * w16 + 32 * jb;
            cp_async16(dstW + jb * 32 * TB_LD, rowW);
            cp_async16(dstW + jb * 32 * TB_LD + 16 * TB_LD, rowW + w16);
            cp_async_commit();
        }
    }
    const bool active = warp * TPW < N_TILES;
    const int rt = (warp * TPW) >> 2, ct0 = (warp * TPW) & 3;  // this warp's tiles: row tile rt, column tiles ct0 .. ct0 + TPW
    const int row = 8 * rt + gid;
#pragma unroll
    for (int jb = 0; jb < 4; ++jb) {
        double* Sj = S + 32 * jb;  // block jb of the slab
        if (jb == 0) cp_async_wait<3>();
        else if (jb == 1) cp_async_wait<2>();
        else if (jb == 2) cp_async_wait<1>();
        else cp_async_wait<0>();
        __syncthreads();
        if (jb > 0) {
            // T_j = A_j - sum_{i<j} X_i L_ji^T
            if (active) {
#pragma unroll
                for (int t = 0; t < TPW; ++t) {
                    const int ct = ct0 + t;
                    double d[2] = {0.0, 0.0}, e[2] = {0.0, 0.0};
#pragma unroll
                    for (int i = 0; i < jb; ++i)
                        tile_mma<32>(d, e, Xb + (i * TR_BM + row) * TB_LD, Ls + ((jb * (jb + 1) / 2 + i) * 32 + 8 * ct + gid) * TB_LD, tig);
                    double2* p = reinterpret_cast<double2*>(Sj + row * TB_SLD + 8 * ct + 2 * tig);
                    double2 v = *p;
                    v.x -= d[0] + e[0];
                    v.y -= d[1] + e[1];
                    *p = v;
                }
            }
            __syncthreads();
        }
        const double* Wj = Ws + jb * 32 * TB_LD;
        const double* Ljj = Ls + (jb * (jb + 1) / 2 + jb) * 32 * TB_LD;
        // X0 = T_j W_j^T
        if (active) {
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const int ct = ct0 + t;
                double d[2] = {0.0, 0.0}, e[2] = {0.0, 0.0};
                tile_mma<32>(d, e, Sj + row * TB_SLD, Wj + (8 * ct + gid) * TB_LD, tig);
                *reinterpret_cast<double2*>(X0 + row * TB_LD + 8 * ct + 2 * tig) = make_double2(d[0] + e[0], d[1] + e[1]);
            }
        }
        __syncthreads();
        // R = T_j - X0 L_jj^T (in place of T_j: a warp only reads its own tiles of T_j here)
        if (active) {
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const int ct = ct0 + t;
                double d[2] = {0.0, 0.0}, e[2] = {0.0, 0.0};
                tile_mma<32>(d, e, X0 + row * TB_LD, Ljj + (8 * ct + gid) * TB_LD, tig);
                double2* p = reinterpret_cast<double2*>(Sj + row * TB_SLD + 8 * ct + 2 * tig);
                double2 v = *p;
                v.x -= d[0] + e[0];
                v.y -= d[1] + e[1];
                *p = v;
            }
        }
        __syncthreads();
        // X_j = X0 + R W_j^T
        if (active) {
#pragma unroll
            for (int t = 0; t < TPW; ++t) {
                const int ct = ct0 + t;
                double d[2] = {0.0, 0.0}, e[2] = {0.0, 0.0};
                tile_mma<32>(d, e, Sj + row * TB_SLD, Wj + (8 * ct + gid) * TB_LD, tig);
                const double2 x0 = *reinterpret_cast<const double2*>(X0 + row * TB_LD + 8 * ct + 2 * tig);
                *reinterpret_cast<double2*>(Xb + (jb * TR_BM + row) * TB_LD + 8 * ct + 2 * tig) =
                    make_double2(x0.x + d[0] + e[0], x0.y + d[1] + e[1]);
            }
        }
        if (jb == 3) __syncthreads();  // (the other steps are followed by the barrier that opens the next one)
    }
    for (int c = tid; c < TR_BM * 64; c += 256) {
        const int r = c >> 6, j2 = (c & 63) * 2;
        *reinterpret_cast<double2*>(g.C + (m0 + r) * g.ldc + j2) =
            *reinterpret_cast<const double2*>(Xb + ((j2 >> 5) * TR_BM + r) * TB_LD + (j2 & 31));
    }
}

template <int TR_BM>
static int launch_trsm_blk_t(const GemmDesc& d, cudaStream_t st) {
    static bool attr_done[64] = {};
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        PIGP_CUDA(cudaFuncSetAttribute(k_trsm_blk<TR_BM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tb_smem(TR_BM)));
        PIGP_CUDA(cudaFuncSetAttribute(k_trsm_blk<TR_BM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tb_smem(TR_BM)));
        attr_done[dev & 63] = true;
    }
    double flops = 0.0;
    if (g_prof_on) {
        flops = 18.0 * 2.0 * d.M * 32.0 * 32.0;
        prof_note(d.M, d.N, d.K, 200);
    }
    ProfScope prof(PROF_GEMM, st, flops * d.nb);
    const dim3 grid((unsigned)(d.M / TR_BM), (unsigned)d.nb);
    if (d.nb > 1) k_trsm_blk<TR_BM, true><<<grid, 256, tb_smem(TR_BM), st>>>(d);
    else k_trsm_blk<TR_BM, false><<<grid, 256, tb_smem(TR_BM), st>>>(d);
    count_launch();
    return PIGP_OK;
}

// Short panels are latency bound (the phases of a slab run back to back on one SM), so the slab height shrinks with the
// panel until the CTAs no longer cover the 148 SMs.
static int launch_trsm_blk(const GemmDesc& d, cudaStream_t st) {
    if (d.M > 148 * 16) return launch_trsm_blk_t<32>(d, st);
    if (d.M > 148 * 8) return launch_trsm_blk_t<16>(d, st);
    return launch_trsm_blk_t<8>(d, st);
}

static int g_gemm_bn = 0;  // 0: read PIGP_GEMM_BN once (kernel tuning); 128 or 64

template <int BN_, int STAGES_>
static int launch_gemm_cfg(const GemmDesc& d, cudaStream_t st) {
    constexpr int SMEM = gemm_smem(BN_, STAGES_);
    static bool attr_done[64] = {};
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    bool& attr_set = attr_done[dev & 63];
    if (!attr_set) {
        PIGP_TRY((gemm_attrs<BN_, STAGES_>()));
        attr_set = true;
    }
    const bool tri = d.lower_only && !d.gen;
    const int dmt = tri ? d.N / BM : d.M / BM, dnt_e = d.N / BM;  // in 128-element units
    const int smt = (dmt + SUPER - 1) / SUPER, snt = (dnt_e + SUPER - 1) / SUPER;
    const int64_t supers = tri ? (int64_t)smt * (smt + 1) / 2 : (int64_t)smt * snt;
    const dim3 grid((unsigned)(supers * SUPER * SUPER * (BM / BN_)), (unsigned)d.nb), block(BN_ * 2);
    double flops = 0.0;
    if (g_prof_on) {  // flops executed at 128-tile granularity
        const int kt = d.K / BK, per = BM / BK;
        for (int tm = 0; tm < dmt; ++tm) {
            const int gm = d.m_gt0 + tm * d.m_ts;
            const int ncols = d.lower_only ? std::max(0, std::min(dnt_e, gm - d.n_gt0 + 1)) : dnt_e;
            int kb = 0, ke = kt;
            if (d.kmode == 1) kb = std::max(0, gm - d.k_gt0) * per;
            else if (d.kmode == 2) ke = std::min(kt, (gm - d.k_gt0 + 1) * per);
            flops += 2.0 * BM * BM * BK * (double)std::max(0, ke - kb) * ncols;
        }
        prof_note(tri ? d.N : d.M, d.N, d.K, d.kmode * 10 + d.lower_only);
    }
    ProfScope prof(PROF_GEMM, st, flops * d.nb);
    if (d.nb > 1) {
        if (d.a_kcontig && d.b_kcontig) k_gemm<true, true, BN_, STAGES_, true><<<grid, block, SMEM, st>>>(d);
        else if (d.a_kcontig) k_gemm<true, false, BN_, STAGES_, true><<<grid, block, SMEM, st>>>(d);
        else if (d.b_kcontig) k_gemm<false, true, BN_, STAGES_, true><<<grid, block, SMEM, st>>>(d);
        else k_gemm<false, false, BN_, STAGES_, true><<<grid, block, SMEM, st>>>(d);
    } else {
        if (d.a_kcontig && d.b_kcontig) k_gemm<true, true, BN_, STAGES_, false><<<grid, block, SMEM, st>>>(d);
        else if (d.a_kcontig) k_gemm<true, false, BN_, STAGES_, false><<<grid, block, SMEM, st>>>(d);
        else if (d.b_kcontig) k_gemm<false, true, BN_, STAGES_, false><<<grid, block, SMEM, st>>>(d);
        else k_gemm<false, false, BN_, STAGES_, false><<<grid, block, SMEM, st>>>(d);
    }
    count_launch();
    return PIGP_OK;
}

int launch_gemm(const GemmDesc& g_in, cudaStream_t st) {
    GemmDesc g = g_in;
    if (g.M <= 0 || g.N <= 0) return PIGP_OK;
    if (g.M % BM || g.N % BM || g.K % 128 || g.K <= 0) {
        set_error("pigp gemm: M, N and K must be multiples of 128");
        return PIGP_EINVAL;
    }
    // the operand loads are 16-byte cp.async copies of element pairs: every row must start 16-byte aligned
    if (g.lda % 2 || g.ldb % 2 || g.ldc % 2 || (g.Lkk && g.ldl % 2)) {
        set_error("pigp gemm: lda, ldb and ldc must be even");
        return PIGP_EINVAL;
    }
    if (g.m_ts == 0) g.m_ts = 1;
    if (g.nb <= 0) g.nb = 1;
    if (g.Lkk) {
        if (g.N != BM || g.K != BM || !g.a_kcontig || !g.b_kcontig || g.C != g.A || g.sc != g.sa || g.alpha != 1.0 || g.beta != 0.0) {
            set_error("pigp gemm: the block TRSM is in place with N = K = 128 and k-contiguous operands");
            return PIGP_EINVAL;
        }
        PIGP_TRY(launch_trsm_blk(g, st));
        PIGP_CUDA(cudaGetLastError());
        return PIGP_OK;
    }
    if (g.lower_only && !g.gen && g.M < g.N) { set_error("pigp gemm: lower_only needs M >= N"); return PIGP_EINVAL; }
    if (g_gemm_bn == 0) {
        const char* e = getenv("PIGP_GEMM_BN");
        g_gemm_bn = (e && atoi(e) == 128) ? 128 : 64;
    }
    static int small_on = -1;
    if (small_on < 0) { const char* e = getenv("PIGP_GEMM_SMALL"); small_on = (e && atoi(e) == 0) ? 0 : 1; }
    if (small_on && g.gen && g.a_kcontig && g.b_kcontig && g.kmode != 2) {
        // latency-bound launches: fewer than one wave of 128 x 64 tiles
        if (g.force_bn128 && g.N == BM) {
            PIGP_TRY((launch_gemm_small<32, 128, 3>(g, st)));
            PIGP_CUDA(cudaGetLastError());
            return PIGP_OK;
        }
        const int64_t tiles = (int64_t)(g.M / BM) * (g.N / 64) / (g.lower_only ? 2 : 1);
        if (!g.force_bn128 && tiles < 74) {  // under half a wave of 64 x 64 tiles: halve the per-CTA DMMA chain instead
            PIGP_TRY((launch_gemm_small<32, 64, 3>(g, st)));
            PIGP_CUDA(cudaGetLastError());
            return PIGP_OK;
        }
        if (!g.force_bn128 && tiles < 2 * 148) {
            PIGP_TRY((launch_gemm_small<64, 64, 3>(g, st)));
            PIGP_CUDA(cudaGetLastError());
            return PIGP_OK;
        }
    }
    if (g.sig_total > 0) { set_error("pigp gemm: fused signal needs the small-tile kernel"); return PIGP_EINVAL; }
    auto run = [&](const GemmDesc& d) {
        return (g_gemm_bn == 128 || d.force_bn128) ? launch_gemm_cfg<128, 4>(d, st) : launch_gemm_cfg<64, 3>(d, st);
    };
    PIGP_TRY(run(g));
    if (g.lower_only && !g.gen && g.M > g.N) {
        // rectangular remainder below the square part: rows [N, M)
        GemmDesc r = g;
        r.lower_only = 0;
        r.M = g.M - g.N;
        r.A = g.a_kcontig ? g.A + (int64_t)g.N * g.lda : g.A + g.N;
        r.C = g.C + (int64_t)g.N * g.ldc;
        if (g.kmode != 0) { set_error("pigp gemm: kmode with rectangular lower_only is unsupported"); return PIGP_EINVAL; }
        PIGP_TRY(run(r));
    }
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

// ----------------------------------------------------------------------------------------------- POTF2 (128 x 128)
// k_potf2: one CTA (8 warps) factors a 128 x 128 diagonal tile held in shared memory and leaves the four diagonal
// 32 x 32 blocks of its inverse; k_tile_inv (same shared-memory layout) completes inverse tiles off the critical path.
// Blocked with 32 x 32 blocks so that only 4 x 16 column-pair steps are sequential:
//   per block column kb: warp 0 factors the 32 x 32 diagonal block in registers (lane = row, column pairs, the pivot
//   chain by shuffles), warp 1 inverts it behind warp 0; the panel  L_ik = A_ik inv(L_kk)^T  and the trailing update
//   A_ij -= L_ik L_jk^T  are 8 x 32 strips of FP64 MMAs (DMMA) out of shared memory -- the part the next diagonal block
//   needs by warps 0-3 alone on the tensor pipe, the rest by background warps underneath the next factorisation.
//   k_tile_inv: the two 64 x 64 diagonal halves from their 32-blocks, then W21 = -W22 (L21 W11); the (unused) upper-right
//   64 x 64 quadrant of the tile is the scratch for L21 W11.
constexpr int PT = 128;
constexpr int PLD = PT + 4;   // 132 = 4 mod 16: conflict-free DMMA fragment loads in both orientations
constexpr int SLD = 36;       // 32 x 32 scratch blocks, same residue
constexpr int N_SCRATCH = 6;  // inv(L_kk) x 4, two temporaries (k_tile_inv)
constexpr int POTF2_SMEM = (PT * PLD + N_SCRATCH * 32 * SLD + 2 * 32 * 4 + 32 + 16) * (int)sizeof(double);

// C(8 x 32 strip) = (accumulate ? C : 0) + alpha * sum_k A(row, k) * Bop(col, k);  Bop(col,k) = B_KN ? B[k][col] : B[col][k].
// Pointers are pre-offset to the strip / operand origin.  n_tiles (1..4) of the four 8 x 8 column tiles are stored.
// K is processed in chunks of 32 whose operands are fetched up front (40 shared loads in flight), and each 8 x 8 tile
// accumulates in two independent chains, so a strip costs ~4 dependent DMMAs per 32 of K instead of 8 load-use steps.
template <bool B_KN, int K>
__device__ __forceinline__ void strip_mma(double* C, int ldc, const double* A, int lda, const double* B, int ldb,
                                          double alpha, bool accumulate, int n_tiles, int lane) {
    const int gid = lane >> 2, tig = lane & 3;
    double acc[4][2], acc2[4][2];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (accumulate && t < n_tiles) {
            const double2 c = *reinterpret_cast<const double2*>(C + gid * ldc + t * 8 + tig * 2);
            acc[t][0] = c.x;
            acc[t][1] = c.y;
        } else {
            acc[t][0] = acc[t][1] = 0.0;
        }
        acc2[t][0] = acc2[t][1] = 0.0;
    }
#pragma unroll
    for (int kc = 0; kc < K; kc += 32) {
        double a[8], b[8][4];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            a[q] = alpha * A[gid * lda + kc + 4 * q + tig];
#pragma unroll
            for (int t = 0; t < 4; ++t)
                b[q][t] = B_KN ? B[(kc + 4 * q + tig) * ldb + t * 8 + gid] : B[(t * 8 + gid) * ldb + kc + 4 * q + tig];
        }
#pragma unroll
        for (int q = 0; q < 8; q += 2)
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                dmma(acc[t][0], acc[t][1], a[q], b[q][t]);
                dmma(acc2[t][0], acc2[t][1], a[q + 1], b[q + 1][t]);
            }
    }
#pragma unroll
    for (int t = 0; t < 4; ++t)
        if (t < n_tiles)
            *reinterpret_cast<double2*>(C + gid * ldc + t * 8 + tig * 2) = make_double2(acc[t][0] + acc2[t][0], acc[t][1] + acc2[t][1]);
}

__device__ long long* g_potf2_dbg = nullptr;  // optional phase stamps (tools/potf2_bench.py)
#define POTF2_STAMP(i) do { if (g_potf2_dbg && threadIdx.x == 0) g_potf2_dbg[i] = clock64(); } while (0)

// 1 / sqrt(d) for the pivots: MUFU seed (~20 bits, from the high word) and one third-order correction,
// y (1 + e/2 + 3 e^2/8) with e = 1 - d y^2 -- ~1 ulp, 5 dependent FP64 operations, branch-free (two of them interleave).
// d < 0 or NaN -> NaN, d = 0 -> NaN as well (inf * 0): a failed factorisation is NaN from that column on.
__device__ __forceinline__ double rsqrt_pivot(double d) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    const double e = fma(-(d * y), y, 1.0);
    const double p = fma(0.375, e, 0.5);
    return fma(y * e, p, y);
}

// Warp-level Cholesky of the 32 x 32 block at D (shared memory, row stride ld), and its inverse by a second warp.
// Factor (warp_factor32): lane i owns row i of the block in registers.  The 32 columns are eliminated in 16 pairs: for
// the 2 x 2 pivot block [d0 b; b d1] the two reciprocal roots rsqrt(d0) and rsqrt(d0 d1 - b^2) are independent, so the
// pivot -> rsqrt -> scale -> pivot dependency chain has 16 links instead of 32.  Every lane rebuilds the next pivot block
// redundantly from seven shuffled numbers (L[i][j], L[i][j+1], the future pivots S[i][i] of rows j+2, j+3 and
// S[j+3][j+2]) ahead of the rank-2 update of the rows, so that the chain (~10 dependent FP64 operations of ~25 cycles plus
// the MUFU seed) runs underneath the update.  L overwrites the lower triangle of D (zeros above).
// Inverse (warp_inverse32): lane c solves column c of W = inv(L) right-looking (w_j = r_j / L_jj; r_m -= L[m][j] w_j),
// two columns of L at a time as soon as the factoring warp has released them (one mbarrier per column pair), with
// the factor's entries coming from broadcast loads.  W goes to Winv (row stride SLD, zeros above the diagonal).

// (The finished column pairs go from the factoring warp to the inverting warp through mbarriers: arrive (release) does
// not block the producer, try_wait (acquire) orders the consumer's loads behind the producer's stores.)

// Scalars of the 2 x 2 pivot block [d0 b; b d1]: r0 = 1 / l00, l10, l00 and rdet = 1 / sqrt(d0 d1 - b^2), from which
// 1 / l11 = rdet l00.  Branch-free (a non-positive pivot is recorded in `fail`, 1-based column inside the block, first
// one wins; NaNs propagate).  d0 d1 is formed (with its rounding error) while b is still on its way, so the determinant
// costs two dependent operations after b.
struct PairScal { double r0, l10, l00, rdet; };

__device__ __forceinline__ PairScal pivot_block(double d0, double d1, double b, int col, int& fail) {
    const double dd = d0 * d1, dde = fma(d0, d1, -dd);
    const double det = fma(-b, b, dd) + dde;
    fail = (fail == 0 && !(d0 > 0.0)) ? col + 1 : fail;
    fail = (fail == 0 && !(det > 0.0)) ? col + 2 : fail;
    const double r0 = rsqrt_pivot(d0), rdet = rsqrt_pivot(det);
    PairScal sc;
    sc.r0 = r0;
    sc.l10 = b * r0;
    sc.l00 = d0 * r0;
    sc.rdet = rdet;
    return sc;
}

// (template recursion instead of #pragma unroll: the rows must stay in registers, and the unroller gives up on the long
// inner loops of the first pairs, which would put the array into local memory)
template <int K>
__device__ __forceinline__ void pair_update(double (&a)[32], const double2* nxt, double l0, double l1) {
    if constexpr (K < 32) {
        const double2 c = nxt[K];  // (L[K][j], L[K][j+1]): broadcast load
        a[K] = fma(-l1, c.y, fma(-l0, c.x, a[K]));
        pair_update<K + 1>(a, nxt, l0, l1);
    }
}

// One pair of columns.  Every lane applies the same formulas: for the block's own rows they reproduce l00, l10 and l11
// (lane J holds d0 in a[J]; lane J + 1 holds b and d1), rows above the block compute garbage that nobody reads and that
// is masked when the columns are stored -- straight-line code.  The new columns go to shared memory for the rank-2 update
// (broadcast loads) and for the inverting warp; the seven numbers the next pivot block depends on travel by shuffles,
// so that the dependency chain per pair is shuffle -> 4 operations -> rsqrt (MUFU + 4) -> 2 operations.
template <int J>
__device__ __forceinline__ void pair_step(double (&a)[32], double& piv, const PairScal sc, int& fail, double2* xch, double* D,
                                          int ld, double* rdiag, unsigned long long* bars, int lane) {
    if constexpr (J < 32) {
        const double l0 = a[J] * sc.r0;
        const double l1 = (fma(-l0, sc.l10, a[J + 1]) * sc.l00) * sc.rdet;
        piv = fma(-l1, l1, fma(-l0, l0, piv));
        PairScal nsc{};
        if constexpr (J + 3 < 32) {
            constexpr unsigned FULL = 0xffffffffu;
            const double p2l0 = __shfl_sync(FULL, l0, J + 2), p3l0 = __shfl_sync(FULL, l0, J + 3);
            const double p3sub = __shfl_sync(FULL, a[J + 2], J + 3);
            const double p2l1 = __shfl_sync(FULL, l1, J + 2), p3l1 = __shfl_sync(FULL, l1, J + 3);
            const double d0 = __shfl_sync(FULL, piv, J + 2), d1 = __shfl_sync(FULL, piv, J + 3);
            nsc = pivot_block(d0, d1, fma(-p3l1, p2l1, fma(-p3l0, p2l0, p3sub)), J + 2, fail);
        }
        double2* nxt = xch + (((J >> 1) + 1) & 1) * 32;
        nxt[lane] = make_double2(l0, l1);
        // columns J, J + 1 of L are final: back to shared memory at once (frees their registers, feeds the inverting warp)
        *reinterpret_cast<double2*>(D + lane * ld + J) = make_double2(lane >= J ? l0 : 0.0, lane > J ? l1 : 0.0);
        if (lane == 0) *reinterpret_cast<double2*>(rdiag + J) = make_double2(sc.r0, sc.rdet * sc.l00);
        mbar_arrive(bars + (J >> 1));  // all 32 lanes: each releases its own row's stores
        __syncwarp();
        pair_update<J + 2>(a, nxt, l0, l1);
        pair_step<J + 2>(a, piv, nsc, fail, xch, D, ld, rdiag, bars, lane);
    }
}

__device__ __noinline__ void warp_factor32(double* D, int ld, double* xch_sm, double* rdiag, unsigned long long* bars,
                                              int32_t* info, int base, int lane) {
    double2* xch = reinterpret_cast<double2*>(xch_sm);  // 2 x 32 entries, double-buffered
    double a[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = (c <= lane) ? D[lane * ld + c] : 0.0;
    double piv = D[lane * ld + lane];
    int fail = 0;
    constexpr unsigned FULL = 0xffffffffu;
    const PairScal sc = pivot_block(__shfl_sync(FULL, piv, 0), __shfl_sync(FULL, piv, 1), __shfl_sync(FULL, a[0], 1), 0, fail);
    pair_step<0>(a, piv, sc, fail, xch, D, ld, rdiag, bars, lane);
    if (lane == 0 && info && fail) atomicCAS(info, 0, base + fail);
    POTF2_STAMP(13);
}

template <int K>
__device__ __forceinline__ void inv_update(double (&r)[32], const double* Dj, int ld, double w0, double w1) {
    if constexpr (K < 32) {
        const double2 c = *reinterpret_cast<const double2*>(Dj + K * ld);  // (L[K][j], L[K][j+1]): broadcast load
        r[K] = fma(-c.y, w1, fma(-c.x, w0, r[K]));
        inv_update<K + 1>(r, Dj, ld, w0, w1);
    }
}

template <int J>
__device__ __forceinline__ void inv_step(double (&r)[32], const double* D, int ld, double* Winv, const double* rdiag,
                                         unsigned long long* bars, int parity, int lane) {
    if constexpr (J < 32) {
        mbar_wait(bars + (J >> 1), parity);
        const double2 rd = *reinterpret_cast<const double2*>(rdiag + J);  // (1 / L[J][J], 1 / L[J+1][J+1])
        const double l10 = D[(J + 1) * ld + J];
        const double w0 = r[J] * rd.x;
        const double w1 = fma(-l10, w0, r[J + 1]) * rd.y;
        Winv[J * SLD + lane] = w0;
        Winv[(J + 1) * SLD + lane] = w1;
        inv_update<J + 2>(r, D + J, ld, w0, w1);
        inv_step<J + 2>(r, D, ld, Winv, rdiag, bars, parity, lane);
    }
}

__device__ __noinline__ void warp_inverse32(const double* D, int ld, double* Winv, const double* rdiag, unsigned long long* bars,
                                               int parity, int lane) {
    double r[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) r[c] = (c == lane) ? 1.0 : 0.0;
    inv_step<0>(r, D, ld, Winv, rdiag, bars, parity, lane);
    POTF2_STAMP(14);
}

// Factor the lower triangle of the 128 x 128 tile at A in place (the upper part of the tile is set to zero) and write
// inv(L) (lower, zeros above) to invd[128*128].  Non-positive pivot -> *info = base + column + 1 (first one wins)
// and NaNs propagate, which is what jnp.linalg.cholesky gives the reference.
// Peers (multi-GPU) receive inv(L) and the diagonal of L -- what their TRSMs and their log-det read -- then the flag.
template <bool BATCH>
__global__ void __launch_bounds__(256, 1) k_potf2(double* A, int64_t ld, double* invd, int32_t* info, int base, int64_t sA, int64_t sI) {
    extern __shared__ __align__(16) double sm[];
    if (BATCH) {
        A += blockIdx.y * sA;
        invd += blockIdx.y * sI;
        if (info) info += blockIdx.y;
    }
    double* scratch = sm + PT * PLD;
    double* xch = scratch + N_SCRATCH * 32 * SLD;    // exchange area of warp_factor32: 2 x 32 x 4 doubles
    double* rdiag = xch + 2 * 32 * 4;                 // 1 / L_ii of the block being factored
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(rdiag + 32);  // one mbarrier per column pair of a block
    if (threadIdx.x < 16) mbar_init(bars + threadIdx.x, 32);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    POTF2_STAMP(0);
    // lower 32 x 32 blocks of the tile -> shared memory (16-byte asynchronous copies, all in flight at once).  The strictly
    // upper blocks are never read; the upper triangles of the diagonal blocks are zeroed by the factoring warp when it
    // writes the columns back.  (Bulk copies of the 256-byte block rows through the TMA engine were measured slower here
    // and in k_trsm_blk: 4.6k vs 3.0k cycles for this tile.)
#pragma unroll 8
    for (int c = tid; c < PT * PT / 2; c += 256) {
        const int i = c >> 6, j2 = (c & 63) * 2;
        if ((j2 >> 5) <= (i >> 5)) cp_async16(sm + i * PLD + j2, A + (int64_t)i * ld + j2);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    POTF2_STAMP(1);
    // kb = -1: factor block 0.  kb >= 0: warps 0-3 solve the first four 8-row strips of panel kb (L_ik = A_ik inv(L_kk)^T, in
    // place) and update the next diagonal block with them -- two strip products, alone on the SM's FP64 tensor pipe -- after
    // which warp 0 factors that block and warp 1 inverts it behind warp 0.  Underneath, warps 2, 3, 5, 6, 7 solve the rest of
    // the panel, apply the trailing update to everything but the diagonal block and store what has become final (warp 4
    // shares warp 0's scheduler and FP64 pipe and stays idle: the factoring warp's DFMA chain is the critical path).
    // (One call site of the factor / inverse: their straight-line code is ~50 KB, a second copy would thrash the
    // instruction cache -- the loop start is opaque so that the first iteration is not peeled.)
    const int kb_first = (ld < 0) ? 0 : -1;
    const int bg = warp < 4 ? warp - 2 : warp - 3;  // background warps 2, 3, 5, 6, 7 -> 0 .. 4
#pragma unroll 1
    for (int kb = kb_first; kb < 3; ++kb) {
        const int o = 32 * kb;
        const int r_lo = o + 32;
        const int n_strips = (PT - r_lo) / 8;
        double* Dblk = sm + r_lo * PLD + r_lo;
        const double* invk = scratch + kb * 32 * SLD;
        if (kb >= 0) {
            if (warp < 4) {
                double* X = sm + (r_lo + warp * 8) * PLD + o;
                strip_mma<false, 32>(X, PLD, X, PLD, invk, SLD, 1.0, false, 4, lane);
                asm volatile("bar.sync 1, 128;\n" ::: "memory");
                strip_mma<false, 32>(sm + (r_lo + warp * 8) * PLD + r_lo, PLD, X, PLD, sm + r_lo * PLD + o, PLD, -1.0, true, warp + 1, lane);
            }
            __syncthreads();
        }
        POTF2_STAMP(3 + 2 * kb);
        if (warp == 0) {
            warp_factor32(Dblk, PLD, xch, rdiag, bars, info, base + r_lo, lane);
        } else if (warp == 1) {
            warp_inverse32(Dblk, PLD, scratch + (kb + 1) * 32 * SLD, rdiag, bars, (kb + 1) & 1, lane);
        } else if (kb >= 0 && warp != 4) {
            for (int st = 4 + bg; st < n_strips; st += 5) {
                double* X = sm + (r_lo + st * 8) * PLD + o;
                strip_mma<false, 32>(X, PLD, X, PLD, invk, SLD, 1.0, false, 4, lane);
            }
            asm volatile("bar.sync 2, 160;\n" ::: "memory");  // every strip of panel kb is final
            // trailing update (lower): tasks = (8-row strip below the diagonal block, 32-column group at or left of it)
            int task = 0;
            for (int st = 4; st < n_strips; ++st) {
                const int n_groups = st / 4 + 1;
                for (int cg = 0; cg < n_groups; ++cg, ++task) {
                    if (task % 5 != bg) continue;
                    const int r0 = r_lo + st * 8, c0 = r_lo + cg * 32;
                    const int n_tiles = min(4, (r0 - c0) / 8 + 1);  // tiles at or left of the diagonal tile
                    strip_mma<false, 32>(sm + r0 * PLD + c0, PLD, sm + r0 * PLD + o, PLD, sm + c0 * PLD + o, PLD, -1.0, true,
                                         n_tiles, lane);
                }
            }
            // block column kb of L (diagonal block and panel) and block kb of the inverse are final: to global memory now,
            // underneath the factorisation of the next block (a single SM stores ~32 B/clk, 80 KB at the end would be 2.7k cycles)
            const int t5 = bg * 32 + lane;
            for (int q = t5; q < (PT - o) * 16; q += 160) {
                const int i = o + (q >> 4), ch = (q & 15) * 2;
                *reinterpret_cast<double2*>(A + (int64_t)i * ld + o + ch) = *reinterpret_cast<const double2*>(sm + i * PLD + o + ch);
            }
            for (int q = t5; q < 32 * 16; q += 160) {
                const int i = q >> 4, ch = (q & 15) * 2;
                *reinterpret_cast<double2*>(invd + (o + i) * PT + o + ch) = *reinterpret_cast<const double2*>(scratch + (kb * 32 + i) * SLD + ch);
            }
        }
        __syncthreads();
        POTF2_STAMP(4 + 2 * kb);
    }
    POTF2_STAMP(9);
    // the last diagonal block of L and of the inverse (everything else was stored underneath the factorisation)
    for (int q = tid; q < 32 * 16; q += 256) {
        const int i = q >> 4, ch = (q & 15) * 2;
        *reinterpret_cast<double2*>(A + (int64_t)(96 + i) * ld + 96 + ch) = *reinterpret_cast<const double2*>(sm + (96 + i) * PLD + 96 + ch);
        *reinterpret_cast<double2*>(invd + (96 + i) * PT + 96 + ch) = *reinterpret_cast<const double2*>(scratch + (3 * 32 + i) * SLD + ch);
    }
    POTF2_STAMP(10);
    POTF2_STAMP(11);
    POTF2_STAMP(12);
}

// Complete inverse diagonal tiles: W = inv(L_cc) from L_cc and the four diagonal 32 x 32 blocks of W that k_potf2 left in
// invd[c] (one CTA per tile c = first + blockIdx.x * stride):
//   the two 64 x 64 diagonal halves from their 32-blocks, W_ba = -inv(L_b) (L_ba inv(L_a)); then W21 = -W22 (L21 W11), with
//   the (unused) upper-right 64 x 64 quadrant of the tile as scratch for L21 W11.
// Optionally also writes the tile transposed into Yt (the diagonal tile of Y = L^-T, zeros below its diagonal).
template <bool BATCH>
__global__ void __launch_bounds__(256, 1) k_tile_inv(const double* L, int64_t ld, double* invd, int first, int stride, double* Y, int64_t ldy,
                                                      int zero_upper, int64_t sL, int64_t sI, int64_t sY) {
    extern __shared__ __align__(16) double sm[];
    if (BATCH) {
        L += blockIdx.y * sL;
        invd += blockIdx.y * sI;
        if (Y) Y += blockIdx.y * sY;
    }
    double* scratch = sm + PT * PLD;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = first + blockIdx.x * stride;
    const double* Lcc = L + (int64_t)c * PT * ld + (int64_t)c * PT;
    double* W = invd + (int64_t)c * PT * PT;
    // sub-diagonal 32-blocks of L_cc -> tile; diagonal blocks of W -> scratch 0-3; blocks (0,1) and (2,3) of the tile are
    // read by the products below and must be zero
#pragma unroll 8
    for (int q = tid; q < PT * PT / 2; q += 256) {
        const int i = q >> 6, j2 = (q & 63) * 2;
        if ((j2 >> 5) < (i >> 5)) cp_async16(sm + i * PLD + j2, Lcc + (int64_t)i * ld + j2);
    }
    for (int e = tid; e < 4 * 32 * 16; e += 256) {
        const int kb = e >> 9, i = (e >> 4) & 31, j2 = (e & 15) * 2;
        cp_async16(scratch + (kb * 32 + i) * SLD + j2, W + (32 * kb + i) * PT + 32 * kb + j2);
    }
    cp_async_commit();
    for (int e = tid; e < 2 * 32 * 32; e += 256) {
        const int half = e >> 10, i = (e >> 5) & 31, j = e & 31;
        sm[(64 * half + i) * PLD + 64 * half + 32 + j] = 0.0;
    }
    cp_async_wait<0>();
    __syncthreads();
    // Step 1: off-diagonal 32-blocks of the two 64 x 64 halves, W_ba = -inv(L_b) (L_ba inv(L_a)).
    {
        const int half = warp >> 2, w4 = warp & 3;         // warps 0-3: blocks (1,0); warps 4-7: blocks (3,2)
        const int ra = 64 * half, rb = ra + 32;
        const double* inva = scratch + (2 * half) * 32 * SLD;
        const double* invb = scratch + (2 * half + 1) * 32 * SLD;
        double* tmp = scratch + (4 + half) * 32 * SLD;
        double* Lba = sm + rb * PLD + ra;
        strip_mma<true, 32>(tmp + w4 * 8 * SLD, SLD, Lba + w4 * 8 * PLD, PLD, inva, SLD, 1.0, false, 4, lane);
        __syncthreads();
        strip_mma<true, 32>(Lba + w4 * 8 * PLD, PLD, invb + w4 * 8 * SLD, SLD, tmp, SLD, -1.0, false, 4, lane);
    }
    __syncthreads();
    // Step 2: diagonal 32-blocks <- inv(L_kk) (full blocks, zeros above the diagonal)
    for (int e = tid; e < 4 * 32 * 32; e += 256) {
        const int kb = e >> 10, i = (e >> 5) & 31, j = e & 31;
        sm[(32 * kb + i) * PLD + 32 * kb + j] = scratch[kb * 32 * SLD + i * SLD + j];
    }
    __syncthreads();
    // Step 3: T = L21 W11 into the upper-right quadrant; 16 tasks (8 strips x 2 column groups).  W11 is lower triangular:
    // its second column group only has rows k >= 32.  Every warp takes one task of each kind.
    {
        const int st = warp;
        strip_mma<true, 64>(sm + (st * 8) * PLD + 64, PLD, sm + (64 + st * 8) * PLD, PLD, sm, PLD, 1.0, false, 4, lane);
        strip_mma<true, 32>(sm + (st * 8) * PLD + 96, PLD, sm + (64 + st * 8) * PLD + 32, PLD, sm + 32 * PLD + 32, PLD, 1.0, false, 4, lane);
    }
    __syncthreads();
    // Step 4: W21 = -W22 T.  W22 is lower triangular: its first four row strips only have columns k < 32.  Warp w takes
    // strip w for the first column group and strip 7 - w for the second (one short and one long product each).
#pragma unroll
    for (int cg = 0; cg < 2; ++cg) {
        const int st = cg == 0 ? warp : 7 - warp;
        double* C = sm + (64 + st * 8) * PLD + cg * 32;
        const double* Aw = sm + (64 + st * 8) * PLD + 64;
        const double* Bt = sm + 64 + cg * 32;
        if (st < 4) strip_mma<true, 32>(C, PLD, Aw, PLD, Bt, PLD, -1.0, false, 4, lane);
        else strip_mma<true, 64>(C, PLD, Aw, PLD, Bt, PLD, -1.0, false, 4, lane);
    }
    __syncthreads();
#pragma unroll 8
    for (int q = tid; q < PT * PT / 2; q += 256) {
        const int i = q >> 6, j2 = (q & 63) * 2;
        // the strictly lower 32-blocks: the diagonal blocks are in place (and may be being read by the panel's TRSM); the
        // blocks above are zero in the solver's workspace and are cleared here for caller-provided buffers (zero_upper)
        if ((j2 >> 5) < (i >> 5)) *reinterpret_cast<double2*>(W + i * PT + j2) = *reinterpret_cast<const double2*>(sm + i * PLD + j2);
        else if (zero_upper && (j2 >> 5) > (i >> 5)) *reinterpret_cast<double2*>(W + i * PT + j2) = make_double2(0.0, 0.0);
    }
    if (Y) {
        double* Yt = Y + (int64_t)c * PT * ldy + (int64_t)c * PT;
        for (int e = tid; e < PT * PT; e += 256) {
            const int j = e >> 7, i = e & 127;  // Y[j][i] = W[i][j]
            Yt[(int64_t)j * ldy + i] = (i >= j) ? sm[i * PLD + j] : 0.0;
        }
    }
}

int launch_tile_inv(const double* L, int64_t ld, double* invd, int first, int stride, int count, double* Y, int64_t ldy, cudaStream_t st, int zero_upper,
                    int nb, int64_t sL, int64_t sI, int64_t sY) {
    if (count <= 0) return PIGP_OK;
    static bool attr_done[64] = {};
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    if (!attr_done[dev & 63]) {
        PIGP_CUDA(cudaFuncSetAttribute(k_tile_inv<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
        PIGP_CUDA(cudaFuncSetAttribute(k_tile_inv<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
        attr_done[dev & 63] = true;
    }
    ProfScope prof(PROF_POTF2, st);
    const dim3 grid((unsigned)count, (unsigned)nb);
    if (nb > 1) k_tile_inv<true><<<grid, 256, POTF2_SMEM, st>>>(L, ld, invd, first, stride, Y, ldy, zero_upper, sL, sI, sY);
    else k_tile_inv<false><<<grid, 256, POTF2_SMEM, st>>>(L, ld, invd, first, stride, Y, ldy, zero_upper, sL, sI, sY);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

int set_potf2_debug(long long* dev_buf) {
    PIGP_CUDA(cudaMemcpyToSymbol(g_potf2_dbg, &dev_buf, sizeof(dev_buf)));
    return PIGP_OK;
}

int launch_potf2(double* A, int64_t ld, double* invd, int32_t* info, int base, cudaStream_t st, int nb, int64_t sA, int64_t sI) {
    static bool attr_done[64] = {};
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    bool& attr_set = attr_done[dev & 63];
    if (!attr_set) {
        PIGP_CUDA(cudaFuncSetAttribute(k_potf2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
        PIGP_CUDA(cudaFuncSetAttribute(k_potf2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
        attr_set = true;
    }
    ProfScope prof(PROF_POTF2, st);
    if (nb > 1) k_potf2<true><<<dim3(1, (unsigned)nb), 256, POTF2_SMEM, st>>>(A, ld, invd, info, base, sA, sI);
    else k_potf2<false><<<1, 256, POTF2_SMEM, st>>>(A, ld, invd, info, base, sA, sI);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

// ----------------------------------------------------------------------------------------------- TRTRI + LAUUM
__global__ void k_place_diag(double* W, int64_t ld, const double* invd) {
    // diagonal tile b of W <- invd[b] (full tile, zeros above the diagonal)
    const int b = blockIdx.x;
    double* dst = W + (int64_t)b * TILE * ld + (int64_t)b * TILE;
    const double* src = invd + (int64_t)b * TILE * TILE;
    for (int e = threadIdx.x; e < TILE * TILE; e += blockDim.x) dst[(int64_t)(e >> 7) * ld + (e & 127)] = src[e];
}

static int trtri_rec(const double* L, double* W, int64_t ld, int64_t n, cudaStream_t st) {
    if (n == TILE) return PIGP_OK;  // diagonal tiles were placed up front
    const int64_t n1 = (n / TILE / 2) * TILE, n2 = n - n1;
    PIGP_TRY(trtri_rec(L, W, ld, n1, st));
    PIGP_TRY(trtri_rec(L + n1 * ld + n1, W + n1 * ld + n1, ld, n2, st));
    double* Tt = W + n1;  // scratch in the strictly upper part of W: Tt (n1 x n2) = W11^T * L21^T
    {
        GemmDesc g{};
        g.M = (int)n1; g.N = (int)n2; g.K = (int)n1;
        g.alpha = 1.0; g.beta = 0.0;
        g.A = W; g.lda = ld; g.a_kcontig = 0;  // A(m,k) = W11[k][m], non-zero for k >= m
        g.B = L + n1 * ld; g.ldb = ld; g.b_kcontig = 1;  // B(n,k) = L21[n][k]
        g.C = Tt; g.ldc = ld;
        g.kmode = 1;
        PIGP_TRY(launch_gemm(g, st));
    }
    {
        // W21 = -W22 * T,  T[k][n] = Tt[n][k]
        GemmDesc g{};
        g.M = (int)n2; g.N = (int)n1; g.K = (int)n2;
        g.alpha = -1.0; g.beta = 0.0;
        g.A = W + n1 * ld + n1; g.lda = ld; g.a_kcontig = 1;  // A(m,k) = W22[m][k], non-zero for k <= m
        g.B = Tt; g.ldb = ld; g.b_kcontig = 1;
        g.C = W + n1 * ld; g.ldc = ld;
        g.kmode = 2;
        PIGP_TRY(launch_gemm(g, st));
    }
    return PIGP_OK;
}

int potri_lower(const double* L, int64_t ld, int64_t n, const double* invd, double* W, double* X, cudaStream_t st) {
    if (n <= 0 || n % TILE || ld % 2) {
        set_error("pigp potri: n must be a multiple of 128 and ld even");
        return PIGP_EINVAL;
    }
    {
        ProfScope prof(PROF_MISC, st);
        k_place_diag<<<(unsigned)(n / TILE), 256, 0, st>>>(W, ld, invd);
        count_launch();
    }
    PIGP_CUDA(cudaGetLastError());
    PIGP_TRY(trtri_rec(L, W, ld, n, st));
    // X (lower) = W^T W :  X_ij = sum_{k >= i} W[k][i] W[k][j]
    GemmDesc g{};
    g.M = (int)n; g.N = (int)n; g.K = (int)n;
    g.alpha = 1.0; g.beta = 0.0;
    g.A = W; g.lda = ld; g.a_kcontig = 0;
    g.B = W; g.ldb = ld; g.b_kcontig = 0;
    g.C = X; g.ldc = ld;
    g.lower_only = 1;
    g.kmode = 1;
    return launch_gemm(g, st);
}

// ----------------------------------------------------------------------------------------------- reductions / BLAS-2
// out2[0] = sum_{i<n} log A[i][i],  out2[1] = sum_{j<n} v[j]^2   (single CTA, fixed order: deterministic)
__global__ void __launch_bounds__(1024) k_logdet_quad(const double* A, int64_t ld, int64_t n, const double* v, double* out2, int64_t sA,
                                                      int64_t sv) {
    __shared__ double sh[2][32];
    A += blockIdx.y * sA;
    v += blockIdx.y * sv;
    out2 += 2 * blockIdx.y;
    double s0 = 0.0, s1 = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
        s0 += log(A[i * ld + i]);
        const double x = v[i];
        s1 = fma(x, x, s1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s0; sh[1][threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x < 32) {
        s0 = sh[0][threadIdx.x];
        s1 = sh[1][threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s0 += __shfl_xor_sync(0xffffffffu, s0, o);
            s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        }
        if (threadIdx.x == 0) { out2[0] = s0; out2[1] = s1; }
    }
}

int launch_logdet_quad(const double* A, int64_t ld, int64_t n, const double* v, double* out2, cudaStream_t st, int nb, int64_t sA,
                       int64_t sv) {
    ProfScope prof(PROF_MISC, st);
    k_logdet_quad<<<dim3(1, (unsigned)nb), 1024, 0, st>>>(A, ld, n, v, out2, sA, sv);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

// y[i] = sum_j A[i][j] x[j]: one warp per row
__global__ void __launch_bounds__(256) k_gemv(const double* A, int64_t ld, int64_t m, int64_t n, const double* x, double* y) {
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= m) return;
    const int lane = threadIdx.x & 31;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const double* a = A + row * ld;
    int64_t j = lane;
    for (; j + 96 < n; j += 128) {
        s0 = fma(a[j], x[j], s0);
        s1 = fma(a[j + 32], x[j + 32], s1);
        s2 = fma(a[j + 64], x[j + 64], s2);
        s3 = fma(a[j + 96], x[j + 96], s3);
    }
    for (; j < n; j += 32) s0 = fma(a[j], x[j], s0);
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) y[row] = s;
}

int launch_gemv(const double* A, int64_t ld, int64_t m, int64_t n, const double* x, double* y, cudaStream_t st) {
    if (m <= 0) return PIGP_OK;
    ProfScope prof(PROF_MISC, st);
    k_gemv<<<(unsigned)((m + 7) / 8), 256, 0, st>>>(A, ld, m, n, x, y);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

int preload_dense() {
    // (the batched instantiations of k_gemm_s / k_trsm_blk / k_potf2 / k_tile_inv are left to their launchers: a batch never
    // runs on a multi-rank solver, whose creation is what this is for)
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm_s<32, 128, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (32 + 128) * LDS_K * (int)sizeof(double)));
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm_s<64, 64, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (64 + 64) * LDS_K * (int)sizeof(double)));
    PIGP_CUDA(cudaFuncSetAttribute(k_gemm_s<32, 64, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * (32 + 64) * LDS_K * (int)sizeof(double)));
    PIGP_PRELOAD((k_gemm_s<32, 128, 3, false>));
    PIGP_PRELOAD((k_gemm_s<64, 64, 3, false>));
    PIGP_PRELOAD((k_gemm_s<32, 64, 3, false>));
    PIGP_CUDA(cudaFuncSetAttribute(k_trsm_blk<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tb_smem(8)));
    PIGP_CUDA(cudaFuncSetAttribute(k_trsm_blk<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tb_smem(16)));
    PIGP_CUDA(cudaFuncSetAttribute(k_trsm_blk<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tb_smem(32)));
    PIGP_PRELOAD((k_trsm_blk<8, false>));
    PIGP_PRELOAD((k_trsm_blk<16, false>));
    PIGP_PRELOAD((k_trsm_blk<32, false>));
    PIGP_TRY((gemm_attrs<128, 4>()));
    PIGP_TRY((gemm_attrs<64, 3>()));
    PIGP_CUDA(cudaFuncSetAttribute(k_potf2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
    PIGP_PRELOAD(k_potf2<false>);
    PIGP_CUDA(cudaFuncSetAttribute(k_tile_inv<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, POTF2_SMEM));
    PIGP_PRELOAD(k_tile_inv<false>);
    PIGP_PRELOAD(k_place_diag);
    PIGP_PRELOAD(k_logdet_quad);
    PIGP_PRELOAD(k_gemv);
    return PIGP_OK;
}

}  // namespace pigp
