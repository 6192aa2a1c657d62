// Multi-GPU evaluation of the PIGP path (K8): NLL + dK/dtheta trace gradient with K dealt block-cyclically over ranks.
//
// The reference has no distributed code at all (SURVEY.md 2.1); this is the sharded form of GP/gp.py:213-224 and
// :412-488 that BASELINE.json's north star asks for.  One pigp_dsolver per rank (one process per GPU, or several
// ranks in one process for tests).  Ownership: 128-row tile t of K belongs to rank t mod P.
//
// Data path = stores into peer memory over NVLink from inside the producing kernels + epoch flags; no library
// collective:
//   * every rank assembles its own row tiles of K (lower part) into a GLOBAL-layout buffer L (npad columns);
//   * recursive right-looking Cholesky restricted to own row tiles.  k_potf2 of the tile owner stores L_kk and
//     inv(L_kk) into every peer; the TRSM GEMM (own rows x inv(L_kk)^T) stores its result tiles into every peer from
//     its epilogue, so L ends up replicated and every trailing update reads local memory only;
//   * Y = L^-T (row tile j of Y = column tile j of L^-1) needs only L: own row tiles, no communication, then one bulk
//     push of the finished rows to all peers;
//   * K^-1 = Y Y^T on own row tiles, fused trace-gradient reduction on own tiles, P partial gradients exchanged by
//     peer stores and summed in rank order (deterministic, identical on every rank);
//   * log-det, |L^-1 y|^2 and alpha = K^-1 y are computed redundantly from the replicated L / Y; each rank carries its
//     own y row tile (placed at the first tile index >= npad/128 that it owns) through the TRSMs.
// The factorisation (leaf, rec, chol_lookahead over a FactorView) is also pigp_potrf_lower's, on one rank.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "pigp_internal.cuh"

namespace pigp {

typedef unsigned long long u64;

struct PeerFlags { int n; u64* f[7]; };

__global__ void k_signal(PeerFlags pf, int idx, u64 val) {
    if ((int)threadIdx.x < pf.n) {
        __threadfence_system();
        u64* p = pf.f[threadIdx.x] + idx;
        asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(p), "l"(val) : "memory");
    }
}

// thread t waits until flags[idx0 + t * stride] >= val (t == skip is not waited for).  Bounded: after timeout_ns the
// error flag is raised and the kernel returns, so a lost peer can never hang the device.
__global__ void k_wait(const u64* flags, int idx0, int stride, int count, int skip, u64 val, int* err, u64 timeout_ns) {
    const int t = threadIdx.x;
    if (t >= count || t == skip) return;
    const u64* p = flags + idx0 + (int64_t)t * stride;
    if (*reinterpret_cast<volatile int*>(err) != 0) return;  // a wait already timed out in this solver: fail fast
    u64 t0 = 0, now = 0;
    asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(t0));
    for (;;) {
        u64 v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];\n" : "=l"(v) : "l"(p) : "memory");
        if (v >= val) break;
        asm volatile("mov.u64 %0, %%globaltimer;\n" : "=l"(now));
        if (now - t0 > timeout_ns) { atomicExch(err, 1); break; }
        __nanosleep(100);
    }
}

// rows [tile * 128, +128), columns [tile * 128, npad) of the own Y row tiles -> the same place in every peer
struct PeerBufs { int n; double* p[7]; };
__global__ void __launch_bounds__(256) k_push_rows(const double* Y, int64_t ld, int64_t npad, int first, int stride, PeerBufs pb) {
    const int tile = first + (blockIdx.x >> 7) * stride;
    const int64_t row = (int64_t)tile * 128 + (blockIdx.x & 127);
    const int64_t c0 = (int64_t)tile * 128;
    const double2* src = reinterpret_cast<const double2*>(Y + row * ld + c0);
    const int64_t n2 = (npad - c0) >> 1;
    for (int64_t i = threadIdx.x; i < n2; i += 256) {
        const double2 v = src[i];
        for (int p = 0; p < pb.n; ++p) reinterpret_cast<double2*>(pb.p[p] + row * ld + c0)[i] = v;
    }
}

// Publication to the peers by dedicated multi-CTA kernels on their own stream, off the Cholesky chain: coalesced 16-byte
// stores over NVLink; the last CTA to finish (system-scope fence, arrival counter) releases the epoch flag on every peer.
struct PushSig { unsigned int* counter; int idx; u64 val; int n; u64* flag[8]; };  // peers' flag arrays and this rank's own
__device__ __forceinline__ void push_done(const PushSig& sg) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int done = atomicAdd(sg.counter, 1u);
        if (done == gridDim.x - 1) {
            *sg.counter = 0u;
            __threadfence_system();
            for (int p = 0; p < sg.n; ++p)
                asm volatile("st.release.sys.global.u64 [%0], %1;\n" ::"l"(sg.flag[p] + sg.idx), "l"(sg.val) : "memory");
        }
    }
}
// rows of the own tiles first, first + stride, ... (count tiles) x columns [col0, col0 + 128) of L; 4 CTAs per tile
__global__ void __launch_bounds__(256) k_push_panel(const double* L, int64_t ld, int64_t col0, int first, int stride, PeerBufs pb, PushSig sg) {
    const int tile = first + (blockIdx.x >> 2) * stride;
    const int64_t row0 = (int64_t)tile * 128 + (blockIdx.x & 3) * 32;
    for (int e = threadIdx.x; e < 32 * 64; e += 256) {
        const int64_t off = (row0 + (e >> 6)) * ld + col0 + (e & 63) * 2;
        const double2 v = *reinterpret_cast<const double2*>(L + off);
        for (int p = 0; p < pb.n; ++p) *reinterpret_cast<double2*>(pb.p[p] + off) = v;
    }
    push_done(sg);
}
// inverse diagonal tile (lower triangle) and L_kk itself (full tile, zeros above the diagonal: the peers' refined TRSMs
// multiply by it, and their log-det reads its diagonal); 8 CTAs
struct PeerDiag { int n; double* invd[7]; double* lkk[7]; };
__global__ void __launch_bounds__(256) k_push_diag(const double* invk, const double* Lkk, int64_t ld, PeerDiag pd, PushSig sg) {
    const int r0 = blockIdx.x * 16;
    for (int e = threadIdx.x; e < 16 * 64; e += 256) {
        const int i = r0 + (e >> 6), j2 = (e & 63) * 2;
        if (j2 <= i && (j2 >> 5) == (i >> 5)) {  // the diagonal 32-blocks of the inverse: all that a peer's TRSM reads
            const double2 v = *reinterpret_cast<const double2*>(invk + i * 128 + j2);
            for (int p = 0; p < pd.n; ++p) *reinterpret_cast<double2*>(pd.invd[p] + i * 128 + j2) = v;
        }
        if ((j2 >> 5) <= (i >> 5)) {  // the lower 32-blocks of L_kk (k_potf2 does not define the others)
            const double2 l = *reinterpret_cast<const double2*>(Lkk + (int64_t)i * ld + j2);
            for (int p = 0; p < pd.n; ++p) *reinterpret_cast<double2*>(pd.lkk[p] + (int64_t)i * ld + j2) = l;
        }
    }
    push_done(sg);
}

// The small kernels below take one grid dimension (y) more per batch slot b: b's vectors of npad entries follow each other,
// its matrices are at + b * sL (L and its y tile) or + b * sY (Y).
// alpha[j] = sum_{k >= tile(j) * 128} Y[j][k] v[k]   (one warp per row; Y upper triangular by tiles)
__global__ void __launch_bounds__(256) k_gemv_upper(const double* Y, int64_t ld, int64_t npad, const double* v, double* alpha, int64_t sY) {
    Y += blockIdx.y * sY;
    v += blockIdx.y * npad;
    alpha += blockIdx.y * npad;
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= npad) return;
    const int lane = threadIdx.x & 31;
    const double* a = Y + row * ld;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int64_t j = (row >> 7 << 7) + lane;
    for (; j + 96 < npad; j += 128) {
        s0 = fma(a[j], v[j], s0);
        s1 = fma(a[j + 32], v[j + 32], s1);
        s2 = fma(a[j + 64], v[j + 64], s2);
        s3 = fma(a[j + 96], v[j + 96], s3);
    }
    for (; j < npad; j += 32) s0 = fma(a[j], v[j], s0);
    double s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) alpha[row] = s;
}

// own y tile: first row = [y, 0 ...], other rows zero
__global__ void __launch_bounds__(256) k_set_ytile(double* tile, int64_t ld, int64_t n, int64_t npad, const double* y, int64_t sL) {
    tile += blockIdx.y * sL;
    const int64_t total = 128 * npad;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / npad, c = e % npad;
        tile[r * ld + c] = (r == 0 && c < n) ? y[c] : 0.0;
    }
}

__global__ void k_push_vec(const double* src, int len, int slot, double* local_slots, PeerBufs pb, int64_t s_slots) {
    const int i = threadIdx.x;
    if (i >= len) return;
    src += blockIdx.y * MAX_THETA;
    local_slots += blockIdx.y * s_slots;
    const double v = src[i];
    local_slots[slot * MAX_THETA + i] = v;
    for (int p = 0; p < pb.n; ++p) pb.p[p][slot * MAX_THETA + i] = v;
}

__global__ void k_sum_slots(const double* slots, int world, int len, double* out, const int32_t* info, const int* err, int64_t s_slots) {
    const int i = threadIdx.x;
    if (i >= len) return;
    slots += blockIdx.y * s_slots;
    out += blockIdx.y * len;
    if (info) info += blockIdx.y;
    double s = 0.0;
    for (int r = 0; r < world; ++r) s += slots[r * MAX_THETA + i];  // rank order: same result on every rank
    if ((info && *info != 0) || (err && *err != 0)) s = nan("");
    out[i] = s;
}

__global__ void k_finish_nll_d(const double* out2, int64_t n, int32_t* info, const int* err, double* nll) {
    out2 += 2 * blockIdx.y;
    info += blockIdx.y;
    nll += blockIdx.y;
    double v = 0.5 * out2[1] + out2[0] + 0.5 * (double)n * log(2.0 * 3.14159265358979323846);  // GP/gp.py:85-89
    if (err && *err != 0) *info = -1;  // a peer's flag never arrived: reported through info (device-pointer API) as well
    if (*info != 0) v = nan("");
    *nll = v;
}

// info <- 1-based index of the first diagonal entry of the replicated factor that is not a positive number (0: none).
// Every rank derives the same value from its copy of L (the owner's k_potf2 saw the pivot itself).
__global__ void __launch_bounds__(1024) k_diag_info(const double* L, int64_t ld, int64_t n, int32_t* info, int64_t sL) {
    __shared__ int best;
    L += blockIdx.y * sL;
    info += blockIdx.y;
    if (threadIdx.x == 0) best = 0x7fffffff;
    __syncthreads();
    int mine = 0x7fffffff;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x)
        if (!(L[i * ld + i] > 0.0)) { mine = (int)i + 1; break; }
    if (mine != 0x7fffffff) atomicMin(&best, mine);
    __syncthreads();
    if (threadIdx.x == 0) *info = (best == 0x7fffffff) ? 0 : best;
}

__global__ void k_copy_v(const double* row, int64_t npad, double* v, int64_t sL) {
    row += blockIdx.y * sL;
    v += blockIdx.y * npad;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < npad) v[i] = row[i];
}

// Streams and events of the panel schedule (chol_lookahead): the bulk stream of the trailing updates, per coarse panel
// "chain done" and "next panel's columns updated", and the event that joins the bulk stream back.  Grows on demand.
struct PanelSched {
    bool low_priority = false;  // the solver's bulk stream yields to its chains; pigp_potrf_lower's has the default priority
    cudaStream_t bulk = nullptr;
    std::vector<cudaEvent_t> pan, next;
    cudaEvent_t done = nullptr;

    int ensure(int panels) {
        if (!bulk) {
            int lo = 0, hi = 0;
            if (low_priority) PIGP_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
            PIGP_CUDA(cudaStreamCreateWithPriority(&bulk, cudaStreamNonBlocking, lo));
            PIGP_CUDA(cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
        }
        while ((int)pan.size() < panels) {
            cudaEvent_t a = nullptr, b = nullptr;
            PIGP_CUDA(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
            PIGP_CUDA(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
            pan.push_back(a);
            next.push_back(b);
        }
        return PIGP_OK;
    }
    void destroy() {
        if (bulk) cudaStreamDestroy(bulk);
        if (done) cudaEventDestroy(done);
        for (cudaEvent_t e : pan) cudaEventDestroy(e);
        for (cudaEvent_t e : next) cudaEventDestroy(e);
    }
};

}  // namespace pigp

using namespace pigp;

static bool g_side_stream = true;
// Flag waits inside the prologue of the consuming GEMM save one tiny kernel per wait, but a grid of spinning CTAs can
// keep this rank's own publication kernels (which a peer's progress depends on) off the SMs: off unless PIGP_FUSE_WAITS=1.
static int g_fuse_waits = -1;
// k-extent (in 128-tiles) of one launch of the side stream's products: PIGP_SIDE_CHUNK (default 0 = unchunked)
static int g_side_chunk = -1;
static int side_chunk_tiles() {
    if (g_side_chunk < 0) {
        const char* e = getenv("PIGP_SIDE_CHUNK");
        g_side_chunk = e ? atoi(e) : 0;
        if (g_side_chunk <= 0) g_side_chunk = 1 << 20;
    }
    return g_side_chunk;
}
// Time-outs of the flag waits.  Inside a factorisation every rank is running, so a flag that stays down for seconds
// means a lost peer (PIGP_WAIT_TIMEOUT_S, default 10 s).  The barrier that opens a call also absorbs host-side skew
// between the ranks -- first-call module loading, a slow set_points on one rank, a garbage-collection pause -- and gets
// its own, much longer limit (PIGP_BARRIER_TIMEOUT_S, default 300 s).
static u64 env_seconds_ns(const char* name, double dflt) {
    const char* e = getenv(name);
    double v = e ? atof(e) : dflt;
    if (!(v > 0.0)) v = dflt;
    return (u64)(v * 1e9);
}
static u64 wait_timeout_ns() { static u64 v = env_seconds_ns("PIGP_WAIT_TIMEOUT_S", 10.0); return v; }
static u64 barrier_timeout_ns() { static u64 v = env_seconds_ns("PIGP_BARRIER_TIMEOUT_S", 300.0); return v; }

static bool fuse_waits() {
    if (g_fuse_waits < 0) { const char* e = getenv("PIGP_FUSE_WAITS"); g_fuse_waits = (e && atoi(e) == 1) ? 1 : 0; }
    return g_fuse_waits == 1;
}

struct pigp_dsolver {
    pigp_plan* plan = nullptr;
    int rank = 0, world = 1;
    int64_t n = 0, npad = 0, ld = 0;
    int T = 0;    // row tiles of the padded matrix
    int gy = 0;   // tile index of this rank's y tile (>= T, == rank mod world)
    char* slab = nullptr;
    size_t slab_bytes = 0;
    double* L = nullptr;       // (T + world) * 128 rows x ld: K -> L (replicated) -> own rows of K^-1
    double* Y = nullptr;       // npad x ld: L^-T, upper
    double* invd = nullptr;    // T inverse diagonal tiles
    double* gslots = nullptr;  // world x MAX_THETA partial gradients
    u64* flags = nullptr;
    int n_flags = 0;
    char* peer_slab[8] = {};
    bool connected = false;
    bool shared_device = false;  // a peer rank lives on this device (tests): flag waits stay in their own 1-CTA kernels,
                                 // because a grid of spinning CTAs could starve the producer it is waiting for
    u64 epoch = 0;
    bool y_lazy = false;  // Y is a separate allocation made on the first gradient request (world == 1)
    bool broken = false;  // an enqueue failed part-way through a call: the solver must be reset (or destroyed)
    // private (not shared)
    AsmTile* d_tiles = nullptr;
    int64_t n_tiles = 0;
    double *partials = nullptr, *gpart = nullptr, *out2 = nullptr, *v = nullptr, *alpha = nullptr;
    int32_t* info = nullptr;
    int* err = nullptr;
    unsigned int* sig_counter = nullptr;  // arrival counter of the fused panel signal
    double *d_theta = nullptr, *d_y = nullptr, *d_res = nullptr, *h_res = nullptr;
    cudaStream_t own_stream = nullptr;  // the _host entry point runs here (ranks sharing a process must not share a stream)
    // internal streams: `sa` (high priority) carries the latency-bound Cholesky chain, `sb` the Y = L^-T products that
    // depend only on finished panels, so that they fill the bubbles of the chain
    cudaStream_t sa = nullptr, sb = nullptr, sc = nullptr;  // sc: publication kernels (peer stores), off the chain
    cudaEvent_t ev_in = nullptr, ev_bar = nullptr, ev_b = nullptr, ev_c = nullptr, ev_out = nullptr, ev_y0 = nullptr;
    std::vector<cudaEvent_t> ev_diag, ev_upd, ev_inv;
    // single-rank, mid-size problems: K^-1 = Y Y^T accumulates in its own buffer from column ranges of Y as they become final,
    // on a low-priority stream underneath the latency-bound chains, instead of one product at the end
    double* Kinv = nullptr;
    cudaStream_t sk = nullptr;
    cudaEvent_t ev_k = nullptr, ev_kd = nullptr;
    int k_done = 0;
    cudaStream_t se = nullptr;  // completes the inverse diagonal tiles (k_tile_inv) as soon as L_kk exists, off both chains
    PanelSched panels{true};
    // batch workspace (world = 1; Work below): per-slot copies of L with its y tile, invd and the small vectors, grown to the
    // largest batch seen; Y and K^-1 separately, to the largest batch that needed them
    int b_cap = 0, b_cap_y = 0, b_cap_k = 0;
    double *bL = nullptr, *binvd = nullptr, *bvec = nullptr, *bY = nullptr, *bK = nullptr;
    int32_t* binfo = nullptr;

    int f_diag(int k) const { return k; }
    int f_panel(int k, int src) const { return T + k * world + src; }
    int f_ydone(int src) const { return T + T * world + src; }
    int f_grad(int src) const { return T + T * world + world + src; }
    int f_bar(int src) const { return T + T * world + 2 * world + src; }
    template <class P> P* peer(int p, P* local) const { return reinterpret_cast<P*>(peer_slab[p] + (reinterpret_cast<char*>(local) - slab)); }
};

namespace pigp {
FactorView factor_view(pigp_dsolver* s) {
    FactorView f{};
    f.L = s->L; f.ld = s->ld; f.T = s->T; f.invd = s->invd; f.info = s->info;
    f.end = s->gy + 1;  // this rank's y tile rides through the TRSMs: L^-1 y comes out of the same launches
    f.rank = s->rank; f.world = s->world;
    f.v = s->L + (int64_t)s->gy * TILE * s->ld;  // first row of the y tile: L^-1 y after the factorisation
    f.nb = 1; f.sL = (int64_t)(s->T + s->world) * TILE * s->ld; f.sI = (int64_t)s->T * TILE * TILE;
    return f;
}
}  // namespace pigp

namespace {

// The buffers one evaluation works in.  A single-theta call uses the solver's own (nb = 1); a batch of nb slots uses the
// batch workspace, where slot b's copy of a buffer is at + b * its stride: sL for L, sI for invd, sY for Y and K^-1,
// npad for v and alpha, 2 for out2, one per slot for info, max(n_tiles, 1) * MAX_THETA for partials, MAX_THETA for gpart
// and world * MAX_THETA for gslots.
struct Work {
    int nb;
    double* L; int64_t sL;      // (T + world) * 128 rows x ld: K -> L, the y tile below it
    double* invd; int64_t sI;
    double *Y, *Kinv; int64_t sY;  // npad x ld each; only with the gradient (K^-1 only with the early products)
    double *partials, *gpart, *gslots, *out2, *v, *alpha;
    int32_t* info;
};

struct Ctx {
    FactorView f;      // the matrix being factored
    pigp_dsolver* s;   // everything else of the solver: only with grad or peers (null under pigp_potrf_lower)
    double *Y, *Kinv;  // L^-T and the early K^-1 (grad only); slot b at + b * sY
    int64_t sY;
    cudaStream_t st;   // chain stream
    cudaStream_t sb;   // side stream (Y = L^-T), used when grad is set
    cudaStream_t sc;   // publication stream
    cudaStream_t se;   // inverse-tile stream
    cudaStream_t sk;   // early K^-1 products
    bool early_kinv;
    int kinv_gran;
    bool grad;
    PeerFlags pf;
    int npeers;
    int others[7];
};

Ctx make_ctx(pigp_dsolver* s, cudaStream_t st, const Work& w) {
    Ctx c{};
    c.f = factor_view(s); c.s = s; c.st = st;
    c.f.L = w.L; c.f.invd = w.invd; c.f.info = w.info; c.f.v = w.L + (int64_t)s->gy * TILE * s->ld;
    c.f.nb = w.nb; c.f.sL = w.sL; c.f.sI = w.sI;
    c.Y = w.Y; c.Kinv = w.Kinv; c.sY = w.sY;
    int k = 0;
    for (int p = 0; p < s->world; ++p)
        if (p != s->rank) { c.others[k] = p; c.pf.f[k] = s->peer(p, s->flags); ++k; }
    c.pf.n = c.npeers = k;
    return c;
}

int signal(const Ctx& c, int idx) {
    if (c.npeers == 0) return PIGP_OK;
    ProfScope prof(PROF_MISC, c.st);
    k_signal<<<1, 32, 0, c.st>>>(c.pf, idx, c.s->epoch);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

int wait_one(const Ctx& c, int idx, cudaStream_t st) {
    if (c.npeers == 0) return PIGP_OK;
    ProfScope prof(PROF_MISC, st);
    k_wait<<<1, 32, 0, st>>>(c.s->flags, idx, 0, 1, -1, c.s->epoch, c.s->err, wait_timeout_ns());
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

// flags[idx0 + src] for every src != rank
int wait_all(const Ctx& c, int idx0, cudaStream_t st, u64 timeout_ns = 0) {
    if (c.npeers == 0) return PIGP_OK;
    ProfScope prof(PROF_MISC, st);
    k_wait<<<1, 32, 0, st>>>(c.s->flags, idx0, 1, c.s->world, c.s->rank, c.s->epoch, c.s->err,
                             timeout_ns ? timeout_ns : wait_timeout_ns());
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    return PIGP_OK;
}

// wait for flag idx before GEMM g on stream st: fused into the GEMM prologue, or (ranks sharing a device) its own kernel
int set_wait_one(const Ctx& c, GemmDesc& g, int idx, cudaStream_t st) {
    if (c.npeers == 0) return PIGP_OK;
    if (c.s->shared_device || !fuse_waits()) return wait_one(c, idx, st);
    g.wait_flags = c.s->flags; g.wait_idx0 = idx; g.wait_stride = 0; g.wait_count = 1; g.wait_skip = -1;
    g.wait_val = c.s->epoch; g.wait_err = c.s->err; g.wait_timeout_ns = wait_timeout_ns();
    return PIGP_OK;
}
// wait for every peer's flag idx0 + src before GEMM g: always its own kernel -- the consumers are full-GPU grids, and a
// grid of spinning CTAs keeps this rank's publication kernels off the SMs (dead-lock observed at 8 GPUs)
int set_wait_all(const Ctx& c, GemmDesc& /*g*/, int idx0, cudaStream_t st) {
    return wait_all(c, idx0, st);
}

// ---- merged recursion over column tiles [c0, c0 + nt): Cholesky on the chain stream; when the gradient is wanted,
// the products of Y = L^-T that depend only on finished panels are issued on the side stream, publication to the
// peers on the publication stream; events order those streams behind this rank's own producers, flags behind the peers'.
PushSig make_sig(const Ctx& c, int idx) {
    PushSig sg{};
    sg.counter = c.s->sig_counter + 1; sg.idx = idx; sg.val = c.s->epoch;
    for (int q = 0; q < c.npeers; ++q) sg.flag[q] = c.pf.f[q];
    sg.flag[c.npeers] = c.s->flags;
    sg.n = c.npeers + 1;
    return sg;
}

// every slot of a batch runs the same product: A, B, C (and Lkk) in buffers of these per-slot strides
void set_slots(GemmDesc& g, const Ctx& c, int64_t sa, int64_t sb, int64_t sc, int64_t sl = 0) {
    g.nb = c.f.nb; g.sa = sa; g.sb = sb; g.sc = sc; g.sl = sl;
}

int leaf(const Ctx& c, int k) {
    const FactorView& f = c.f;
    pigp_dsolver* s = c.s;
    const int64_t ld = f.ld;
    double* invk = f.invd + (int64_t)k * TILE * TILE;
    double* Akk = f.L + (int64_t)k * TILE * ld + (int64_t)k * TILE;
    const bool mine = (k % f.world == f.rank), multi = c.npeers > 0;
    if (mine) PIGP_TRY(launch_potf2(Akk, ld, invk, f.info, k * TILE, c.st, f.nb, f.sL, f.sI));
    if (c.grad || multi) PIGP_CUDA(cudaEventRecord(s->ev_diag[k], c.st));  // mine: inv(L_kk) is ready; else: the chain has reached leaf k
    if (mine && multi) {
        // publish inv(L_kk) and diag(L_kk) from the publication stream while the chain goes on with this rank's own TRSM
        PIGP_CUDA(cudaStreamWaitEvent(c.sc, s->ev_diag[k], 0));
        PeerDiag pd{};
        pd.n = c.npeers;
        for (int q = 0; q < c.npeers; ++q) { pd.invd[q] = s->peer(c.others[q], invk); pd.lkk[q] = s->peer(c.others[q], Akk); }
        ProfScope prof(PROF_MISC, c.sc);
        k_push_diag<<<8, 256, 0, c.sc>>>(invk, Akk, ld, pd, make_sig(c, s->f_diag(k)));
        count_launch();
        PIGP_CUDA(cudaGetLastError());
    }
    {
        // L_ik = A_ik inv(L_kk)^T for the own row tiles below (and the rows below the matrix)
        const int first = f.first_own(k + 1), cnt = f.count_own(k + 1, f.end);
        if (cnt > 0) {
            GemmDesc g{};
            g.M = cnt * TILE; g.N = TILE; g.K = TILE;
            g.alpha = 1.0; g.beta = 0.0;
            double* Cb = f.L + (int64_t)first * TILE * ld + (int64_t)k * TILE;
            g.A = Cb; g.lda = ld; g.a_kcontig = 1;
            g.B = invk; g.ldb = TILE; g.b_kcontig = 1;
            g.C = Cb; g.ldc = ld;
            g.gen = 1; g.m_ts = f.world; g.m_gt0 = first; g.n_gt0 = k; g.k_gt0 = k;
            g.force_bn128 = 1;  // in place
            g.Lkk = Akk; g.ldl = ld;  // refined: needs L_kk itself next to its inverse (peers receive both)
            set_slots(g, c, f.sL, f.sI, f.sL, f.sL);
            if (!mine) PIGP_TRY(set_wait_one(c, g, s->f_diag(k), c.st));
            PIGP_TRY(launch_gemm(g, c.st));
        }
        if (c.grad || multi) PIGP_CUDA(cudaEventRecord(s->ev_upd[k], c.st));  // this rank's rows of panel k are final
        if (multi) {
            // publish them (rows of the matrix proper; the y tile is private) and raise PANEL[k][rank] on every peer
            PIGP_CUDA(cudaStreamWaitEvent(c.sc, s->ev_upd[k], 0));
            const int pcnt = f.count_own(k + 1, f.T);
            ProfScope prof(PROF_MISC, c.sc);
            if (pcnt > 0) {
                PeerBufs pb{};
                pb.n = c.npeers;
                for (int q = 0; q < c.npeers; ++q) pb.p[q] = s->peer(c.others[q], s->L);
                k_push_panel<<<pcnt * 4, 256, 0, c.sc>>>(s->L, ld, (int64_t)k * TILE, first, s->world, pb, make_sig(c, s->f_panel(k, s->rank)));
            } else {
                k_signal<<<1, 32, 0, c.sc>>>(c.pf, s->f_panel(k, s->rank), s->epoch);
            }
            count_launch();
            PIGP_CUDA(cudaGetLastError());
        }
    }
    if (c.grad) {
        // Y[j, k] = R[j, k] inv(L_kk)^T for own row tiles j < k; Y[k, k] = inv(L_kk)^T.  The factorisation only produced
        // the diagonal 32-blocks of inv(L_kk); every rank completes the tile itself from its copy of L_kk, here, off the chain
        // (on its own stream: it depends on L_kk only, so it runs ahead of the L^-T chain instead of inside it)
        PIGP_CUDA(cudaStreamWaitEvent(c.se, s->ev_diag[k], 0));
        if (!mine) PIGP_TRY(wait_one(c, s->f_diag(k), c.se));
        PIGP_TRY(launch_tile_inv(f.L, ld, f.invd, k, 1, 1, mine ? c.Y : nullptr, ld, c.se, 0, f.nb, f.sL, f.sI, c.sY));
        PIGP_CUDA(cudaEventRecord(s->ev_inv[k], c.se));
        PIGP_CUDA(cudaStreamWaitEvent(c.sb, s->ev_inv[k], 0));
        const int first = f.first_own(0), cnt = f.count_own(0, k);
        if (cnt > 0) {
            GemmDesc g{};
            g.M = cnt * TILE; g.N = TILE; g.K = TILE;
            g.alpha = 1.0; g.beta = 0.0;
            double* Cb = c.Y + (int64_t)first * TILE * ld + (int64_t)k * TILE;
            g.A = Cb; g.lda = ld; g.a_kcontig = 1;
            g.B = invk; g.ldb = TILE; g.b_kcontig = 1;
            g.C = Cb; g.ldc = ld;
            g.gen = 1; g.m_ts = s->world; g.m_gt0 = first; g.n_gt0 = k; g.k_gt0 = k;
            g.force_bn128 = 1;
            set_slots(g, c, c.sY, f.sI, c.sY);
            PIGP_TRY(launch_gemm(g, c.sb));
        }
        // columns [k_done, k + 1) of Y are final once the side stream gets here: their share of K^-1 = Y Y^T,
        //   Kinv[i, j] += sum_{k in range, k >= i} Y[i, k] Y[j, k]   (rows / columns 0 .. k, lower part),
        // goes to the low-priority product stream now, while the chains are still running
        if (c.early_kinv && (k + 1 - s->k_done >= c.kinv_gran || k + 1 == s->T)) {
            const int a = s->k_done, b = k + 1;
            PIGP_CUDA(cudaEventRecord(s->ev_k, c.sb));
            PIGP_CUDA(cudaStreamWaitEvent(c.sk, s->ev_k, 0));
            GemmDesc g{};
            g.M = b * TILE; g.N = b * TILE; g.K = (b - a) * TILE;
            g.alpha = 1.0; g.beta = 1.0;
            g.A = c.Y + (int64_t)a * TILE; g.lda = ld; g.a_kcontig = 1;
            g.B = c.Y + (int64_t)a * TILE; g.ldb = ld; g.b_kcontig = 1;
            g.C = c.Kinv; g.ldc = ld;
            g.lower_only = 1; g.kmode = 1;
            g.gen = 1; g.m_ts = 1; g.m_gt0 = 0; g.n_gt0 = 0; g.k_gt0 = a;
            set_slots(g, c, c.sY, c.sY, c.sY);
            PIGP_TRY(launch_gemm(g, c.sk));
            s->k_done = b;
        }
    }
    return PIGP_OK;
}

int rec(const Ctx& c, int c0, int nt) {
    if (nt == 1) return leaf(c, c0);
    const FactorView& f = c.f;
    pigp_dsolver* s = c.s;
    const int64_t ld = f.ld;
    const int n1 = nt / 2, n2 = nt - n1;
    PIGP_TRY(rec(c, c0, n1));
    const int k1 = c0 + n1 - 1;  // once every peer's PANEL[k1] flag is up, all rows of the panels [c0, c0 + n1) have arrived
    {
        // trailing update of the own row tiles: C[i, J2] -= L[i, K1] L[J2, K1]^T (lower part)
        const int first = f.first_own(c0 + n1), cnt = f.count_own(c0 + n1, f.end);
        if (cnt > 0) {
            GemmDesc g{};
            g.M = cnt * TILE; g.N = n2 * TILE; g.K = n1 * TILE;
            g.alpha = -1.0; g.beta = 1.0;
            g.A = f.L + (int64_t)first * TILE * ld + (int64_t)c0 * TILE; g.lda = ld; g.a_kcontig = 1;
            g.B = f.L + (int64_t)(c0 + n1) * TILE * ld + (int64_t)c0 * TILE; g.ldb = ld; g.b_kcontig = 1;
            g.C = f.L + (int64_t)first * TILE * ld + (int64_t)(c0 + n1) * TILE; g.ldc = ld;
            g.lower_only = 1;
            g.gen = 1; g.m_ts = f.world; g.m_gt0 = first; g.n_gt0 = c0 + n1; g.k_gt0 = c0;
            set_slots(g, c, f.sL, f.sL, f.sL);
            if (c.npeers > 0) PIGP_TRY(set_wait_all(c, g, s->f_panel(k1, 0), c.st));
            PIGP_TRY(launch_gemm(g, c.st));
        }
    }
    if (c.grad) {
        // Y[j, J2] -= sum_{k in K1, k >= j} Y[j, k] L[J2, k]^T for the own row tiles j < c0 + n1
        PIGP_CUDA(cudaStreamWaitEvent(c.sb, s->ev_upd[k1], 0));
        const int first = f.first_own(0), cnt = f.count_own(0, c0 + n1);
        if (cnt > 0) {
            GemmDesc g{};
            g.M = cnt * TILE; g.N = n2 * TILE; g.K = n1 * TILE;
            g.alpha = -1.0; g.beta = 1.0;
            g.A = c.Y + (int64_t)first * TILE * ld + (int64_t)c0 * TILE; g.lda = ld; g.a_kcontig = 1;
            g.B = f.L + (int64_t)(c0 + n1) * TILE * ld + (int64_t)c0 * TILE; g.ldb = ld; g.b_kcontig = 1;
            g.C = c.Y + (int64_t)first * TILE * ld + (int64_t)(c0 + n1) * TILE; g.ldc = ld;
            g.kmode = 1;
            g.gen = 1; g.m_ts = s->world; g.m_gt0 = first; g.n_gt0 = c0 + n1; g.k_gt0 = c0;
            set_slots(g, c, c.sY, f.sL, c.sY);
            PIGP_TRY(set_wait_all(c, g, s->f_panel(k1, 0), c.sb));
            // Optionally issued in k-chunks (PIGP_SIDE_CHUNK = tiles per launch): a CTA of a K = 10k product holds its SM
            // slot for ~1 ms, and the chain's (and the publication stream's) small high-priority kernels can only start
            // when slots drain -- stream priority does not preempt.  Measured at N = 20k: chunks of 2048 cost more GEMM
            // efficiency than the chain gains (1 GPU 254.3 -> 256.4 ms, 2 GPUs 138.1 -> 140.0 ms), so the default is
            // one launch.
            const int chunk = side_chunk_tiles();
            for (int kc = 0; kc < n1; kc += chunk) {
                GemmDesc h = g;
                h.A = g.A + (int64_t)kc * TILE;
                h.B = g.B + (int64_t)kc * TILE;
                h.K = std::min(chunk, n1 - kc) * TILE;
                h.k_gt0 = c0 + kc;
                if (kc > 0) h.wait_count = 0;
                PIGP_TRY(launch_gemm(h, c.sb));
            }
        }
    }
    return rec(c, c0 + n1, n2);
}

// ---- Panel schedule with look-ahead (PIGP_LOOKAHEAD=<W tiles>; 0 = the plain recursion).
// Coarse right-looking panels of W tile columns with the recursive factorisation inside a panel and a depth-1
// look-ahead: the chain stream factors panel p (rec over its W columns, all own rows below), the bulk stream applies
// panel p to the columns of panel p + 1 first (the chain waits only for that) and to the rest afterwards, concurrently
// with the chain's work on panel p + 1.  The big trailing updates thereby leave the N/128-step dependency chain; the
// L^-T products get the matching right-looking update V_p on the side stream.  Uses the existing kernels only.
// Width: PIGP_LOOKAHEAD / pigp_set_lookahead(W >= 0) fix it (0 = plain recursion); unset (or a negative W) = automatic:
// a single-rank NLL-only evaluation (and pigp_potrf_lower) has no L^-T work on the side stream to fill the bubbles of the
// potf2 -> TRSM chain, and the panel schedule measured 18 % / 13 % / 5 % faster there at N = 5018 / 10570 / 20000
// (profiles/r02_lookahead.txt); with the gradient requested the L^-T products fill most of those bubbles (a few per cent
// gain at mid sizes only), and sharded runs keep the plain recursion.
static int g_lookahead = -2;  // -2: read PIGP_LOOKAHEAD once; -1: automatic; >= 0: fixed
static int lookahead_width(int T, int world, bool grad) {
    if (g_lookahead == -2) { const char* e = getenv("PIGP_LOOKAHEAD"); g_lookahead = e ? std::max(0, atoi(e)) : -1; }
    if (g_lookahead >= 0) return g_lookahead;
    if (world != 1 || T < 12) return 0;
    if (grad) return (T >= 16 && T < 32) ? 2 : (T >= 32 && T < 96) ? 4 : 0;  // -6 % at N = 2640, -4 % at 5018
    return T < 64 ? 2 : T < 128 ? 4 : 16;
}

// C[i, J] -= L[i, Kp] L[J, Kp]^T for the own row tiles i >= jc0 (lower part), J = [jc0, jc1), Kp = [k0, k1)
static int panel_update(const Ctx& c, int k0, int k1, int jc0, int jc1, cudaStream_t st) {
    const FactorView& f = c.f;
    if (jc1 <= jc0) return PIGP_OK;
    const int64_t ld = f.ld;
    const int first = f.first_own(jc0), cnt = f.count_own(jc0, f.end);
    if (cnt <= 0) return PIGP_OK;
    GemmDesc g{};
    g.M = cnt * TILE; g.N = (jc1 - jc0) * TILE; g.K = (k1 - k0) * TILE;
    g.alpha = -1.0; g.beta = 1.0;
    g.A = f.L + (int64_t)first * TILE * ld + (int64_t)k0 * TILE; g.lda = ld; g.a_kcontig = 1;
    g.B = f.L + (int64_t)jc0 * TILE * ld + (int64_t)k0 * TILE; g.ldb = ld; g.b_kcontig = 1;
    g.C = f.L + (int64_t)first * TILE * ld + (int64_t)jc0 * TILE; g.ldc = ld;
    g.lower_only = 1;
    g.gen = 1; g.m_ts = f.world; g.m_gt0 = first; g.n_gt0 = jc0; g.k_gt0 = k0;
    set_slots(g, c, f.sL, f.sL, f.sL);
    return launch_gemm(g, st);
}

static int chol_lookahead(const Ctx& c, int W, PanelSched& ps) {
    const FactorView& f = c.f;
    pigp_dsolver* s = c.s;
    const int64_t ld = f.ld;
    const int T = f.T;
    PIGP_TRY(ps.ensure((T + W - 1) / W));
    for (int j0 = 0, p = 0; j0 < T; j0 += W, ++p) {
        const int j1 = std::min(j0 + W, T);
        PIGP_TRY(rec(c, j0, j1 - j0));  // chain: panel p, all own rows below (and the intra-panel L^-T products on sb)
        if (j1 >= T) break;
        PIGP_CUDA(cudaEventRecord(ps.pan[p], c.st));
        // bulk stream: panel p -> columns of panel p + 1 (the chain waits for this), then -> everything right of it
        PIGP_CUDA(cudaStreamWaitEvent(ps.bulk, ps.pan[p], 0));
        if (c.npeers > 0) PIGP_TRY(wait_all(c, s->f_panel(j1 - 1, 0), ps.bulk));  // every peer's rows of the panel have arrived
        const int jn = std::min(j1 + W, T);
        PIGP_TRY(panel_update(c, j0, j1, j1, jn, ps.bulk));
        PIGP_CUDA(cudaEventRecord(ps.next[p], ps.bulk));
        PIGP_TRY(panel_update(c, j0, j1, jn, T, ps.bulk));
        PIGP_CUDA(cudaStreamWaitEvent(c.st, ps.next[p], 0));
        if (c.grad) {
            // V_p: Y[j, [j1, T)] -= sum_{k in panel p, k >= j} Y[j, k] L[[j1, T), k]^T for the own row tiles j < j1
            PIGP_CUDA(cudaStreamWaitEvent(c.sb, ps.pan[p], 0));
            PIGP_TRY(wait_all(c, s->f_panel(j1 - 1, 0), c.sb));
            const int first = f.first_own(0), cnt = f.count_own(0, j1);
            if (cnt > 0) {
                GemmDesc g{};
                g.M = cnt * TILE; g.N = (T - j1) * TILE; g.K = (j1 - j0) * TILE;
                g.alpha = -1.0; g.beta = 1.0;
                g.A = c.Y + (int64_t)first * TILE * ld + (int64_t)j0 * TILE; g.lda = ld; g.a_kcontig = 1;
                g.B = f.L + (int64_t)j1 * TILE * ld + (int64_t)j0 * TILE; g.ldb = ld; g.b_kcontig = 1;
                g.C = c.Y + (int64_t)first * TILE * ld + (int64_t)j1 * TILE; g.ldc = ld;
                g.kmode = 1;
                g.gen = 1; g.m_ts = s->world; g.m_gt0 = first; g.n_gt0 = j1; g.k_gt0 = j0;
                set_slots(g, c, c.sY, f.sL, c.sY);
                PIGP_TRY(launch_gemm(g, c.sb));
            }
        }
    }
    PIGP_CUDA(cudaEventRecord(ps.done, ps.bulk));
    PIGP_CUDA(cudaStreamWaitEvent(c.st, ps.done, 0));
    return PIGP_OK;
}

int preload_dist() {
    PIGP_TRY(preload_dense());
    PIGP_TRY(preload_assemble());
    PIGP_TRY(preload_matern());
    PIGP_PRELOAD(k_signal); PIGP_PRELOAD(k_wait); PIGP_PRELOAD(k_push_rows);
    PIGP_PRELOAD(k_gemv_upper); PIGP_PRELOAD(k_set_ytile); PIGP_PRELOAD(k_push_vec); PIGP_PRELOAD(k_sum_slots);
    PIGP_PRELOAD(k_finish_nll_d); PIGP_PRELOAD(k_diag_info); PIGP_PRELOAD(k_copy_v); PIGP_PRELOAD(k_push_panel); PIGP_PRELOAD(k_push_diag);
    return PIGP_OK;
}

// pigp_potrf_lower's panel streams: one set per device, shared by the host threads that factor on it
PanelSched g_panels[64];
std::mutex g_panels_mutex;

}  // namespace

// pigp_potrf_lower: the solver's factorisation, on one rank, of the caller's buffer; its m_extra rows below the matrix
// ride through the TRSMs and trailing updates as the solver's y tile does.
int pigp::potrf_lower(double* A, int64_t ld, int64_t n, int64_t m_extra, double* invd, int32_t* info, cudaStream_t st) {
    if (n <= 0 || n % TILE || m_extra % TILE || m_extra < 0 || ld % 2) {
        set_error("pigp potrf: n and m_extra must be multiples of 128 and ld even");
        return PIGP_EINVAL;
    }
    Ctx c{};
    c.st = st;
    c.f.L = A; c.f.ld = ld; c.f.invd = invd; c.f.info = info;
    c.f.T = (int)(n / TILE); c.f.end = (int)((n + m_extra) / TILE);
    c.f.rank = 0; c.f.world = 1;
    c.f.nb = 1;
    const int W = lookahead_width(c.f.T, 1, false);
    if (W > 0 && c.f.T > W) {
        int dev = 0;
        PIGP_CUDA(cudaGetDevice(&dev));
        std::lock_guard<std::mutex> lock(g_panels_mutex);
        PIGP_TRY(chol_lookahead(c, W, g_panels[dev & 63]));
    } else {
        PIGP_TRY(rec(c, 0, c.f.T));
    }
    // the factorisation leaves the diagonal 32-blocks of the inverse tiles; callers of this entry point get complete tiles
    return launch_tile_inv(A, ld, invd, 0, 1, c.f.T, nullptr, 0, st, 1);
}

extern "C" {

void pigp_dsolver_destroy(pigp_dsolver* s) {
    if (!s) return;
    if (s->y_lazy) cudaFree(s->Y);
    cudaFree(s->slab); cudaFree(s->d_tiles); cudaFree(s->partials); cudaFree(s->gpart); cudaFree(s->out2); cudaFree(s->v);
    cudaFree(s->alpha); cudaFree(s->info); cudaFree(s->err); cudaFree(s->sig_counter); cudaFree(s->d_theta); cudaFree(s->d_y); cudaFree(s->d_res);
    if (s->h_res) cudaFreeHost(s->h_res);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    if (s->sa) cudaStreamDestroy(s->sa);
    if (s->sb) cudaStreamDestroy(s->sb);
    if (s->sc) cudaStreamDestroy(s->sc);
    s->panels.destroy();
    for (cudaEvent_t e : {s->ev_in, s->ev_bar, s->ev_b, s->ev_c, s->ev_out, s->ev_y0}) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s->ev_diag) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s->ev_upd) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s->ev_inv) if (e) cudaEventDestroy(e);
    if (s->se) cudaStreamDestroy(s->se);
    if (s->sk) cudaStreamDestroy(s->sk);
    if (s->ev_k) cudaEventDestroy(s->ev_k);
    if (s->ev_kd) cudaEventDestroy(s->ev_kd);
    cudaFree(s->Kinv);
    cudaFree(s->bL); cudaFree(s->binvd); cudaFree(s->bvec); cudaFree(s->bY); cudaFree(s->bK); cudaFree(s->binfo);
    delete s;
}

int pigp_dsolver_create(pigp_plan* plan, int rank, int world, pigp_dsolver** out) {
    if (!plan || !out || !plan->symmetric || world < 1 || world > 8 || rank < 0 || rank >= world) {
        set_error("pigp_dsolver_create: needs a symmetric training plan and 0 <= rank < world <= 8");
        return PIGP_EINVAL;
    }
    *out = nullptr;
    PIGP_TRY(preload_dist());
    pigp_dsolver* s = new pigp_dsolver();
    s->plan = plan; s->rank = rank; s->world = world;
    s->n = plan->rows;
    s->npad = round_up(s->n, TILE);
    s->ld = s->npad;
    s->T = (int)(s->npad / TILE);
    s->gy = factor_view(s).first_own(s->T);  // the y tile: the first own tile past the matrix
    s->n_flags = s->T + s->T * world + 3 * world;
    const size_t l_bytes = sizeof(double) * (size_t)(s->T + world) * TILE * s->ld;
    // Y = L^-T is needed by the gradient only.  A single-rank solver (the handle behind pigp_solver: NLL-only and
    // posterior users) allocates it on the first gradient request; sharded solvers keep it inside the peer-visible slab.
    s->y_lazy = (world == 1);
    const size_t y_bytes = s->y_lazy ? 0 : sizeof(double) * (size_t)s->npad * s->ld;
    const size_t i_bytes = sizeof(double) * (size_t)s->T * TILE * TILE;
    const size_t g_bytes = sizeof(double) * (size_t)world * MAX_THETA;
    const size_t f_bytes = (sizeof(u64) * (size_t)s->n_flags + 255) / 256 * 256;
    s->slab_bytes = l_bytes + y_bytes + i_bytes + ((g_bytes + 255) / 256 * 256) + f_bytes;
    int rc = PIGP_OK;
    auto cuda_ok = [&](cudaError_t e, const char* what) {
        if (e != cudaSuccess && rc == PIGP_OK) { set_error(std::string(what) + ": " + cudaGetErrorString(e)); rc = PIGP_ECUDA; }
    };
    cuda_ok(cudaMalloc(&s->slab, s->slab_bytes), "cudaMalloc slab");
    if (rc == PIGP_OK) {
        char* p = s->slab;
        s->L = reinterpret_cast<double*>(p); p += l_bytes;
        s->Y = s->y_lazy ? nullptr : reinterpret_cast<double*>(p); p += y_bytes;
        s->invd = reinterpret_cast<double*>(p); p += i_bytes;
        s->gslots = reinterpret_cast<double*>(p); p += (g_bytes + 255) / 256 * 256;
        s->flags = reinterpret_cast<u64*>(p);
        // zero everything once: flags and slots start at epoch 0, and the upper triangles of the inverse diagonal tiles
        // (never written on peers) must read as zero
        cuda_ok(cudaMemset(s->slab, 0, s->slab_bytes), "memset slab");
        s->peer_slab[rank] = s->slab;
    }
    std::vector<AsmTile> tiles;
    build_lower_tiles_owned(plan, rank, world, tiles);
    s->n_tiles = (int64_t)tiles.size();
    if (rc == PIGP_OK && !tiles.empty()) {
        cuda_ok(cudaMalloc(&s->d_tiles, tiles.size() * sizeof(AsmTile)), "cudaMalloc tiles");
        if (rc == PIGP_OK) cuda_ok(cudaMemcpy(s->d_tiles, tiles.data(), tiles.size() * sizeof(AsmTile), cudaMemcpyHostToDevice), "copy tiles");
    }
    cuda_ok(cudaMalloc(&s->partials, sizeof(double) * std::max<int64_t>(s->n_tiles, 1) * MAX_THETA), "cudaMalloc partials");
    cuda_ok(cudaMalloc(&s->gpart, sizeof(double) * MAX_THETA), "cudaMalloc gpart");
    cuda_ok(cudaMalloc(&s->out2, sizeof(double) * 2), "cudaMalloc out2");
    cuda_ok(cudaMalloc(&s->v, sizeof(double) * s->npad), "cudaMalloc v");
    cuda_ok(cudaMalloc(&s->alpha, sizeof(double) * s->npad), "cudaMalloc alpha");
    cuda_ok(cudaMalloc(&s->info, sizeof(int32_t)), "cudaMalloc info");
    cuda_ok(cudaMalloc(&s->err, sizeof(int)), "cudaMalloc err");
    if (rc == PIGP_OK) cuda_ok(cudaMemset(s->err, 0, sizeof(int)), "memset err");
    cuda_ok(cudaMalloc(&s->sig_counter, 2 * sizeof(unsigned int)), "cudaMalloc sig_counter");
    if (rc == PIGP_OK) cuda_ok(cudaMemset(s->sig_counter, 0, 2 * sizeof(unsigned int)), "memset sig_counter");
    cuda_ok(cudaMalloc(&s->d_theta, sizeof(double) * MAX_THETA), "cudaMalloc theta");
    cuda_ok(cudaMalloc(&s->d_y, sizeof(double) * s->n), "cudaMalloc y");
    cuda_ok(cudaMalloc(&s->d_res, sizeof(double) * (1 + MAX_THETA)), "cudaMalloc res");
    cuda_ok(cudaMallocHost(&s->h_res, sizeof(double) * (4 + 2 * MAX_THETA) + sizeof(double) * s->n), "cudaMallocHost res");
    cuda_ok(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking), "cudaStreamCreate");
    {
        int lo = 0, hi = 0;
        cuda_ok(cudaDeviceGetStreamPriorityRange(&lo, &hi), "cudaDeviceGetStreamPriorityRange");
        cuda_ok(cudaStreamCreateWithPriority(&s->sa, cudaStreamNonBlocking, hi), "cudaStreamCreate sa");
        cuda_ok(cudaStreamCreateWithPriority(&s->sb, cudaStreamNonBlocking, lo), "cudaStreamCreate sb");
        cuda_ok(cudaStreamCreateWithPriority(&s->sc, cudaStreamNonBlocking, hi), "cudaStreamCreate sc");
        for (cudaEvent_t* e : {&s->ev_in, &s->ev_bar, &s->ev_b, &s->ev_c, &s->ev_out, &s->ev_y0}) cuda_ok(cudaEventCreateWithFlags(e, cudaEventDisableTiming), "cudaEventCreate");
        s->ev_diag.assign(s->T, nullptr);
        s->ev_upd.assign(s->T, nullptr);
        s->ev_inv.assign(s->T, nullptr);
        cuda_ok(cudaStreamCreateWithPriority(&s->se, cudaStreamNonBlocking, lo), "cudaStreamCreate se");
        cuda_ok(cudaStreamCreateWithPriority(&s->sk, cudaStreamNonBlocking, lo), "cudaStreamCreate sk");
        cuda_ok(cudaEventCreateWithFlags(&s->ev_k, cudaEventDisableTiming), "cudaEventCreate");
        cuda_ok(cudaEventCreateWithFlags(&s->ev_kd, cudaEventDisableTiming), "cudaEventCreate");
        for (int k = 0; k < s->T; ++k) {
            cuda_ok(cudaEventCreateWithFlags(&s->ev_diag[k], cudaEventDisableTiming), "cudaEventCreate");
            cuda_ok(cudaEventCreateWithFlags(&s->ev_upd[k], cudaEventDisableTiming), "cudaEventCreate");
            cuda_ok(cudaEventCreateWithFlags(&s->ev_inv[k], cudaEventDisableTiming), "cudaEventCreate");
        }
    }
    // The zeroed flags, error flag and arrival counters must be in place before a peer signals into them, and cudaMemset
    // is asynchronous to the host on the legacy stream, which does not order with any solver's non-blocking streams.
    if (rc == PIGP_OK) cuda_ok(cudaStreamSynchronize(0), "cudaStreamSynchronize");
    if (rc != PIGP_OK) { pigp_dsolver_destroy(s); return rc; }
    s->connected = (world == 1);
    *out = s;
    return PIGP_OK;
}

int pigp_set_lookahead(int tiles) {
    g_lookahead = tiles < 0 ? -1 : tiles;
    return PIGP_OK;
}

int pigp_set_side_stream(int on) {
    g_side_stream = on != 0;
    return PIGP_OK;
}

int pigp_dsolver_slab(const pigp_dsolver* s, void** ptr, int64_t* bytes) {
    if (!s) { set_error("pigp_dsolver_slab: null solver"); return PIGP_EINVAL; }
    if (ptr) *ptr = s->slab;
    if (bytes) *bytes = (int64_t)s->slab_bytes;
    return PIGP_OK;
}

int pigp_dsolver_ipc_handle(const pigp_dsolver* s, void* handle64) {
    if (!s || !handle64) { set_error("pigp_dsolver_ipc_handle: null argument"); return PIGP_EINVAL; }
    static_assert(sizeof(cudaIpcMemHandle_t) == PIGP_IPC_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    PIGP_CUDA(cudaIpcGetMemHandle(&h, s->slab));
    std::memcpy(handle64, &h, sizeof(h));
    return PIGP_OK;
}

int pigp_ipc_open(const void* handle64, void** ptr) {
    if (!handle64 || !ptr) { set_error("pigp_ipc_open: null argument"); return PIGP_EINVAL; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, sizeof(h));
    PIGP_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return PIGP_OK;
}

int pigp_ipc_close(void* ptr) {
    if (ptr) PIGP_CUDA(cudaIpcCloseMemHandle(ptr));
    return PIGP_OK;
}

int pigp_dsolver_connect(pigp_dsolver* s, void* const* slabs) {
    if (!s || !slabs) { set_error("pigp_dsolver_connect: null argument"); return PIGP_EINVAL; }
    int me = 0;
    PIGP_CUDA(cudaGetDevice(&me));
    for (int p = 0; p < s->world; ++p) {
        if (p == s->rank) continue;
        if (!slabs[p]) { set_error("pigp_dsolver_connect: missing peer slab"); return PIGP_EINVAL; }
        s->peer_slab[p] = static_cast<char*>(slabs[p]);
        cudaPointerAttributes at{};
        const bool known = cudaPointerGetAttributes(&at, slabs[p]) == cudaSuccess && at.type == cudaMemoryTypeDevice;
        if (known && at.device == me) s->shared_device = true;
        if (known && at.device != me) {
            const cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);  // same-process peers on another device
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                set_error(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
                return PIGP_ECUDA;
            }
        }
        cudaGetLastError();
    }
    s->connected = true;
    return PIGP_OK;
}

int pigp_dsolver_set_shared_device(pigp_dsolver* s, int shared) {
    if (!s) { set_error("pigp_dsolver_set_shared_device: null solver"); return PIGP_EINVAL; }
    s->shared_device = shared != 0;
    return PIGP_OK;
}

int pigp_device_uuid(void* out16) {
    if (!out16) { set_error("pigp_device_uuid: null argument"); return PIGP_EINVAL; }
    int dev = 0;
    PIGP_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    PIGP_CUDA(cudaGetDeviceProperties(&prop, dev));
    std::memcpy(out16, &prop.uuid, 16);
    return PIGP_OK;
}

// PIGP_EARLY_KINV=0 switches the early K^-1 products off.  Worth it while the evaluation is latency bound and its GEMMs
// are short: -9 % at N = 1180, -7.5 % at 2640.  From N ~ 5000 on nothing is gained (measured 5018 ... 12700): the
// product's CTAs then hold every SM for tens of microseconds, and each of the chains' launches waits that long for a slot
// -- priorities do not pre-empt
static bool early_kinv_on(const pigp_dsolver* s, bool grad) {
    static int early = -1;
    if (early < 0) { const char* e = getenv("PIGP_EARLY_KINV"); early = (e && atoi(e) == 0) ? 0 : 1; }
    return early && grad && s->world == 1 && s->T >= 8 && s->T <= 32;
}

// the solver's own buffers (one slot); Y (world = 1) and K^-1 are allocated on the first call that needs them
static int own_work(pigp_dsolver* s, bool grad, Work& w) {
    if (grad && !s->Y) PIGP_CUDA(cudaMalloc(&s->Y, sizeof(double) * (size_t)s->npad * s->ld));
    if (early_kinv_on(s, grad) && !s->Kinv) PIGP_CUDA(cudaMalloc(&s->Kinv, sizeof(double) * (size_t)s->npad * s->ld));
    const FactorView f = factor_view(s);
    w = Work{};
    w.nb = 1;
    w.L = s->L; w.sL = f.sL; w.invd = s->invd; w.sI = f.sI;
    w.Y = s->Y; w.Kinv = s->Kinv; w.sY = s->npad * s->ld;
    w.partials = s->partials; w.gpart = s->gpart; w.gslots = s->gslots; w.out2 = s->out2; w.v = s->v; w.alpha = s->alpha;
    w.info = s->info;
    return PIGP_OK;
}

// per-slot vectors of the batch workspace, one array each: partials, gpart, gslots, out2, v, alpha
static int64_t vec_len(const pigp_dsolver* s) { return std::max<int64_t>(s->n_tiles, 1) * MAX_THETA + 2 * MAX_THETA + 2 + 2 * s->npad; }

// Grow the batch workspace to nb slots.  Runs before anything is enqueued: on PIGP_ENOMEM nothing was launched, and the
// solver stays usable for single calls and for the batches that still fit.  New buffers are zeroed on the caller's stream
// `user`, which the schedule then waits for (the solver's own streams do not order with the legacy stream).
static int batch_work(pigp_dsolver* s, int nb, bool grad, cudaStream_t user, Work& w) {
    const FactorView f = factor_view(s);
    const size_t mat = sizeof(double) * (size_t)s->npad * s->ld;
    auto alloc = [&](void** p, size_t bytes) {
        if (cudaMalloc(p, bytes) == cudaSuccess && cudaMemsetAsync(*p, 0, bytes, user) == cudaSuccess) return true;
        cudaFree(*p);
        *p = nullptr;
        cudaGetLastError();  // not sticky: clear it, so that it is not reported by the next launch check
        set_error("pigp_nll_grad_batch: out of device memory for the batch workspace");
        return false;
    };
    if (nb > s->b_cap) {
        cudaFree(s->bL); cudaFree(s->binvd); cudaFree(s->bvec); cudaFree(s->binfo);
        s->bL = s->binvd = s->bvec = nullptr; s->binfo = nullptr;
        s->b_cap = 0;
        // zeroed once like the solver's slab: the parts of the inverse tiles above their diagonal blocks are read as zero
        if (!alloc((void**)&s->bL, sizeof(double) * (size_t)f.sL * nb) || !alloc((void**)&s->binvd, sizeof(double) * (size_t)f.sI * nb) ||
            !alloc((void**)&s->bvec, sizeof(double) * (size_t)vec_len(s) * nb) || !alloc((void**)&s->binfo, sizeof(int32_t) * (size_t)nb)) {
            cudaFree(s->bL); cudaFree(s->binvd); cudaFree(s->bvec); cudaFree(s->binfo);
            s->bL = s->binvd = s->bvec = nullptr; s->binfo = nullptr;
            return PIGP_ENOMEM;
        }
        s->b_cap = nb;
    }
    if (grad && nb > s->b_cap_y) {
        cudaFree(s->bY);
        s->bY = nullptr;
        s->b_cap_y = 0;
        if (!alloc((void**)&s->bY, mat * nb)) return PIGP_ENOMEM;
        s->b_cap_y = nb;
    }
    if (early_kinv_on(s, grad) && nb > s->b_cap_k) {
        cudaFree(s->bK);
        s->bK = nullptr;
        s->b_cap_k = 0;
        if (!alloc((void**)&s->bK, mat * nb)) return PIGP_ENOMEM;
        s->b_cap_k = nb;
    }
    const int64_t cap = s->b_cap, pt = std::max<int64_t>(s->n_tiles, 1) * MAX_THETA;
    w = Work{};
    w.nb = nb;
    w.L = s->bL; w.sL = f.sL; w.invd = s->binvd; w.sI = f.sI;
    w.Y = s->bY; w.Kinv = s->bK; w.sY = s->npad * s->ld;
    w.partials = s->bvec;
    w.gpart = w.partials + cap * pt;
    w.gslots = w.gpart + cap * MAX_THETA;
    w.out2 = w.gslots + cap * MAX_THETA;
    w.v = w.out2 + cap * 2;
    w.alpha = w.v + cap * s->npad;
    w.info = s->binfo;
    return PIGP_OK;
}

static int dsolver_enqueue(pigp_dsolver* s, const Work& w, const double* theta_dev, const double* y_dev, double eps,
                           double* nll_dev, double* grad_dev, int32_t* info_dev, cudaStream_t st);

// One evaluation of w.nb slots: slot b reads theta_dev + b * theta_len and writes nll_dev + b, grad_dev + b * theta_len and
// info_dev + b.  Every launch is issued once, for all slots.
static int dsolver_call(pigp_dsolver* s, int nb, const double* theta_dev, const double* y_dev, double eps, double* nll_dev,
                        double* grad_dev, int32_t* info_dev, void* stream) {
    if (!s->connected) { set_error("pigp_dsolver_nll_grad: peers are not connected"); return PIGP_EINVAL; }
    if (s->broken) { set_error("pigp_dsolver_nll_grad: an earlier call failed part-way; call pigp_dsolver_reset on every rank"); return PIGP_ECUDA; }
    cudaStream_t user = reinterpret_cast<cudaStream_t>(stream);
    cudaStream_t st = s->sa;
    {
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && cur != s->plan->device) PIGP_CUDA(cudaSetDevice(s->plan->device));
    }
    Work w;
    if (nb == 1) PIGP_TRY(own_work(s, grad_dev != nullptr, w));
    else PIGP_TRY(batch_work(s, nb, grad_dev != nullptr, user, w));
    PIGP_CUDA(cudaEventRecord(s->ev_in, user));
    PIGP_CUDA(cudaStreamWaitEvent(st, s->ev_in, 0));
    s->epoch += 1;
    // From here on the peers expect this rank's publications of epoch `epoch`: if an enqueue fails below, the call still
    // joins the user's stream to whatever was enqueued (so nothing runs unordered) and the solver is marked broken; the
    // peers' waits for the missing flags end at their time-out with info = -1 / NaN results.
    const int rc = dsolver_enqueue(s, w, theta_dev, y_dev, eps, nll_dev, grad_dev, info_dev, st);
    if (rc != PIGP_OK) s->broken = true;
    const cudaError_t e1 = cudaEventRecord(s->ev_out, st);
    const cudaError_t e2 = (e1 == cudaSuccess) ? cudaStreamWaitEvent(user, s->ev_out, 0) : e1;
    if (rc != PIGP_OK) return rc;
    if (e2 != cudaSuccess) { s->broken = true; set_error(std::string("pigp_dsolver_nll_grad: ") + cudaGetErrorString(e2)); return PIGP_ECUDA; }
    return PIGP_OK;
}

int pigp_dsolver_nll_grad(pigp_dsolver* s, const double* theta_dev, const double* y_dev, double eps, double* nll_dev,
                          double* grad_dev, int32_t* info_dev, void* stream) {
    if (!s || !theta_dev || !y_dev || !nll_dev) { set_error("pigp_dsolver_nll_grad: null argument"); return PIGP_EINVAL; }
    return dsolver_call(s, 1, theta_dev, y_dev, eps, nll_dev, grad_dev, info_dev, stream);
}

}  // extern "C"

int pigp::dsolver_nll_grad_batch(pigp_dsolver* s, int nb, const double* thetas_dev, const double* y_dev, double eps,
                                 double* nll_dev, double* grad_dev, int32_t* info_dev, void* stream) {
    if (!s || !thetas_dev || !y_dev || !nll_dev) { set_error("pigp_nll_grad_batch: null argument"); return PIGP_EINVAL; }
    if (nb < 1 || nb > PIGP_MAX_BATCH) { set_error("pigp_nll_grad_batch: n_theta must be in [1, 65535]"); return PIGP_EINVAL; }
    if (s->world != 1) { set_error("pigp_nll_grad_batch: sharded solvers (world > 1) evaluate one theta at a time"); return PIGP_EINVAL; }
    return dsolver_call(s, nb, thetas_dev, y_dev, eps, nll_dev, grad_dev, info_dev, stream);
}

extern "C" {

static int dsolver_enqueue(pigp_dsolver* s, const Work& w, const double* theta_dev, const double* y_dev, double eps,
                           double* nll_dev, double* grad_dev, int32_t* info_dev, cudaStream_t st) {
    const pigp_plan* p = s->plan;
    const int64_t ld = s->ld;
    const int nb = w.nb, P = p->theta_len;
    Ctx c = make_ctx(s, st, w);
    // serial mode: everything on the chain stream -- for the per-kernel timing pass, and for three or more ranks that share
    // one device (tests): the emulation would otherwise keep more streams with spinning waits alive than the device has
    // independent hardware queues, and a producer queued behind another rank's wait would dead-lock until the time-out
    const bool serial = !g_side_stream || (s->shared_device && s->world >= 3);
    c.sb = serial ? st : s->sb;
    c.sc = serial ? st : s->sc;
    // ranks sharing one device (tests) keep the inverse tiles on the side stream: a fifth stream per rank with its own spinning
    // flag waits would exceed the device's 8 hardware queues, and a producer queued behind a wait dead-locks until the time-out
    c.se = serial ? st : (s->shared_device ? c.sb : s->se);
    c.grad = grad_dev != nullptr;
    c.sk = serial ? st : s->sk;
    c.early_kinv = early_kinv_on(s, c.grad);
    c.kinv_gran = std::max(2, s->T / 8);
    int32_t* info = w.info;
    PIGP_CUDA(cudaMemsetAsync(info, 0, sizeof(int32_t) * nb, st));
    // every peer has finished reading what the previous call left in this rank's buffers
    PIGP_TRY(signal(c, s->f_bar(s->rank)));
    PIGP_TRY(wait_all(c, s->f_bar(0), st, barrier_timeout_ns()));
    const int first = c.f.first_own(0), cnt = c.f.count_own(0, s->T);
    if (c.grad) {
        PIGP_CUDA(cudaEventRecord(s->ev_bar, st));
        PIGP_CUDA(cudaStreamWaitEvent(c.sb, s->ev_bar, 0));
        // (a batch has world = 1: its slots' Y follow each other, so their row tiles are one run of cnt * nb tiles)
        if (cnt > 0)
            PIGP_CUDA(cudaMemset2DAsync(c.Y + (int64_t)first * TILE * ld, sizeof(double) * TILE * ld * s->world, 0,
                                        sizeof(double) * TILE * ld, (size_t)cnt * nb, c.sb));
        // the inverse-tile stream writes the diagonal tiles of Y: behind the clearing of Y
        PIGP_CUDA(cudaEventRecord(s->ev_y0, c.sb));
        PIGP_CUDA(cudaStreamWaitEvent(c.se, s->ev_y0, 0));
        if (c.early_kinv) {
            PIGP_CUDA(cudaStreamWaitEvent(c.sk, s->ev_bar, 0));  // the previous evaluation's gradient kernel has read Kinv
            PIGP_CUDA(cudaMemsetAsync(c.Kinv, 0, sizeof(double) * (size_t)s->npad * s->ld * nb, c.sk));
            s->k_done = 0;
        }
    }
    // own rows of K (lower, jitter added), identity padding (owner of the last tile), own y tile
    PIGP_TRY(launch_assemble(p, s->d_tiles, s->n_tiles, theta_dev, eps, 1, w.L, ld, st, nb, P, w.sL));
    if (s->n < s->npad && (s->T - 1) % s->world == s->rank)
        PIGP_TRY(launch_pad(w.L, ld, s->n, s->n, s->npad, s->npad, 1, 1, st, nb, w.sL));
    double* ytile = w.L + (int64_t)s->gy * TILE * ld;
    {
        ProfScope prof(PROF_MISC, st);
        k_set_ytile<<<dim3(148, nb), 256, 0, st>>>(ytile, ld, s->n, s->npad, y_dev, w.sL);
        count_launch();
    }
    PIGP_CUDA(cudaGetLastError());
    const int law = lookahead_width(s->T, s->world, c.grad);
    if (law > 0 && c.sb != st && s->T > law) PIGP_TRY(chol_lookahead(c, law, s->panels));
    else PIGP_TRY(rec(c, 0, s->T));
    if (c.npeers > 0) {
        // the diagonal of every L_kk (log-det) travels with the DIAG flags; a GEMM only waits for the flags it consumes
        ProfScope prof(PROF_MISC, st);
        for (int k0 = 0; k0 < s->T; k0 += 32) {
            k_wait<<<1, 32, 0, st>>>(s->flags, s->f_diag(k0), 1, std::min(32, s->T - k0), -1, s->epoch, s->err, wait_timeout_ns());
            count_launch();
        }
        PIGP_CUDA(cudaGetLastError());
        PIGP_CUDA(cudaEventRecord(s->ev_c, c.sc));
        PIGP_CUDA(cudaStreamWaitEvent(st, s->ev_c, 0));
    }
    // every rank holds all of L now (the panel flags of every peer were awaited inside rec for all but the final leaf,
    // whose diagonal tile arrives with its DIAG flag)
    PIGP_TRY(launch_logdet_quad(w.L, ld, s->n, ytile, w.out2, st, nb, w.sL, w.sL));
    k_diag_info<<<dim3(1, nb), 1024, 0, st>>>(w.L, ld, s->n, info, w.sL);
    count_launch();
    k_finish_nll_d<<<dim3(1, nb), 1, 0, st>>>(w.out2, s->n, info, s->err, nll_dev);
    count_launch();
    PIGP_CUDA(cudaGetLastError());
    if (c.grad) {
        PIGP_CUDA(cudaEventRecord(s->ev_b, c.sb));
        PIGP_CUDA(cudaStreamWaitEvent(st, s->ev_b, 0));  // own rows of Y are complete
        if (c.npeers > 0) {
            if (cnt > 0) {
                PeerBufs pb{};
                pb.n = c.npeers;
                for (int q = 0; q < c.npeers; ++q) pb.p[q] = s->peer(c.others[q], s->Y);
                ProfScope prof(PROF_MISC, st);
                k_push_rows<<<cnt * TILE, 256, 0, st>>>(s->Y, ld, s->npad, first, s->world, pb);
                count_launch();
                PIGP_CUDA(cudaGetLastError());
            }
            PIGP_TRY(signal(c, s->f_ydone(s->rank)));
            PIGP_TRY(wait_all(c, s->f_ydone(0), st));
        }
        // alpha = K^-1 y = Y (L^-1 y), redundantly on every rank
        {
            ProfScope prof(PROF_MISC, st);
            k_copy_v<<<dim3((unsigned)((s->npad + 255) / 256), nb), 256, 0, st>>>(ytile, s->npad, w.v, w.sL);
            k_gemv_upper<<<dim3((unsigned)((s->npad + 7) / 8), nb), 256, 0, st>>>(c.Y, ld, s->npad, w.v, w.alpha, c.sY);
            count_launch(2);
        }
        PIGP_CUDA(cudaGetLastError());
        // own row tiles of K^-1 = Y Y^T (lower) over the own rows of L -- unless it was accumulated along the way
        if (c.early_kinv) {
            PIGP_CUDA(cudaEventRecord(s->ev_kd, c.sk));
            PIGP_CUDA(cudaStreamWaitEvent(st, s->ev_kd, 0));
        } else if (cnt > 0) {
            GemmDesc g{};
            g.M = cnt * TILE; g.N = (int)s->npad; g.K = (int)s->npad;
            g.alpha = 1.0; g.beta = 0.0;
            g.A = c.Y + (int64_t)first * TILE * ld; g.lda = ld; g.a_kcontig = 1;
            g.B = c.Y; g.ldb = ld; g.b_kcontig = 1;
            g.C = w.L + (int64_t)first * TILE * ld; g.ldc = ld;
            g.lower_only = 1; g.kmode = 1;
            g.gen = 1; g.m_ts = s->world; g.m_gt0 = first; g.n_gt0 = 0; g.k_gt0 = 0;
            set_slots(g, c, c.sY, c.sY, w.sL);
            PIGP_TRY(launch_gemm(g, st));
        }
        PIGP_TRY(launch_grad(p, s->d_tiles, s->n_tiles, theta_dev, c.early_kinv ? c.Kinv : w.L, ld, w.alpha, w.partials, w.gpart, st,
                             nb, P, c.early_kinv ? c.sY : w.sL, s->npad, std::max<int64_t>(s->n_tiles, 1) * MAX_THETA, MAX_THETA));
        {
            PeerBufs pb{};
            pb.n = c.npeers;
            for (int q = 0; q < c.npeers; ++q) pb.p[q] = s->peer(c.others[q], s->gslots);
            ProfScope prof(PROF_GRAD, st);
            k_push_vec<<<dim3(1, nb), 32, 0, st>>>(w.gpart, p->theta_len, s->rank, w.gslots, pb, (int64_t)s->world * MAX_THETA);
            count_launch();
        }
        PIGP_CUDA(cudaGetLastError());
        PIGP_TRY(signal(c, s->f_grad(s->rank)));
        PIGP_TRY(wait_all(c, s->f_grad(0), st));
        k_sum_slots<<<dim3(1, nb), 32, 0, st>>>(w.gslots, s->world, p->theta_len, grad_dev, info, s->err, (int64_t)s->world * MAX_THETA);
        count_launch();
        PIGP_CUDA(cudaGetLastError());
    }
    if (info_dev) PIGP_CUDA(cudaMemcpyAsync(info_dev, info, sizeof(int32_t) * nb, cudaMemcpyDeviceToDevice, st));
    return PIGP_OK;
}

int pigp_dsolver_reset(pigp_dsolver* s) {
    if (!s) { set_error("pigp_dsolver_reset: null solver"); return PIGP_EINVAL; }
    // Drain this rank's streams and clear the sticky time-out flag.  Call it on EVERY rank after a failed evaluation
    // (info = -1, NaN results or PIGP_ECUDA from a _host call), with a host-side barrier between the resets and the
    // next evaluation; epochs keep counting, so stale flags of the failed call are never mistaken for new ones.
    PIGP_CUDA(cudaStreamSynchronize(s->sa));
    PIGP_CUDA(cudaStreamSynchronize(s->sb));
    PIGP_CUDA(cudaStreamSynchronize(s->sc));
    PIGP_CUDA(cudaStreamSynchronize(s->se));
    PIGP_CUDA(cudaStreamSynchronize(s->sk));
    if (s->panels.bulk) PIGP_CUDA(cudaStreamSynchronize(s->panels.bulk));
    PIGP_CUDA(cudaMemset(s->err, 0, sizeof(int)));
    PIGP_CUDA(cudaMemset(s->sig_counter, 0, 2 * sizeof(unsigned int)));
    // the ranks' call counters may have drifted apart (a rank that never made the failed call): everybody restarts at
    // epoch 0 with clean flags.  The host-side barrier AFTER the resets keeps a fast rank's new flags from being erased.
    PIGP_CUDA(cudaMemset(s->flags, 0, sizeof(u64) * (size_t)s->n_flags));
    PIGP_CUDA(cudaMemset(s->gslots, 0, sizeof(double) * (size_t)s->world * MAX_THETA));
    PIGP_CUDA(cudaStreamSynchronize(0));  // the memsets are complete when the host-side barrier is passed
    s->epoch = 0;
    s->broken = false;
    return PIGP_OK;
}

int pigp_dsolver_nll_grad_host(pigp_dsolver* s, const double* theta_host, const double* y_host, double eps, int want_grad,
                               double* nll_host, double* grad_host, int32_t* info_host) {
    if (!s || !theta_host || !y_host || !nll_host || (want_grad && !grad_host)) { set_error("pigp_dsolver_nll_grad_host: null argument"); return PIGP_EINVAL; }
    const int P = s->plan->theta_len;
    cudaStream_t st = s->own_stream;
    double* h_theta = s->h_res + 4 + MAX_THETA;
    double* h_y = h_theta + MAX_THETA;
    std::memcpy(h_theta, theta_host, sizeof(double) * P);
    std::memcpy(h_y, y_host, sizeof(double) * s->n);
    PIGP_CUDA(cudaMemcpyAsync(s->d_theta, h_theta, sizeof(double) * P, cudaMemcpyHostToDevice, st));
    PIGP_CUDA(cudaMemcpyAsync(s->d_y, h_y, sizeof(double) * s->n, cudaMemcpyHostToDevice, st));
    PIGP_TRY(pigp_dsolver_nll_grad(s, s->d_theta, s->d_y, eps, s->d_res, want_grad ? s->d_res + 1 : nullptr, nullptr, st));
    PIGP_CUDA(cudaMemcpyAsync(s->h_res, s->d_res, sizeof(double) * (1 + (want_grad ? P : 0)), cudaMemcpyDeviceToHost, st));
    int32_t* h_info = reinterpret_cast<int32_t*>(s->h_res + 1 + MAX_THETA);
    PIGP_CUDA(cudaMemcpyAsync(h_info, s->info, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    PIGP_CUDA(cudaMemcpyAsync(h_info + 1, s->err, sizeof(int), cudaMemcpyDeviceToHost, st));
    PIGP_CUDA(cudaStreamSynchronize(st));
    *nll_host = s->h_res[0];
    if (want_grad) std::memcpy(grad_host, s->h_res + 1, sizeof(double) * P);
    if (info_host) *info_host = h_info[0];
    if (h_info[1] != 0) { set_error("pigp_dsolver: a peer flag wait timed out (a rank is missing or failed)"); return PIGP_ECUDA; }
    return PIGP_OK;
}

}  // extern "C"
