"""Entry-wise GPU tests of the dense path in every size regime it dispatches on, with stale workspaces and after a failed
factorisation.

Which code runs depends on the tile count T = round_up(N, 128) / 128 (or n / 128 for the building blocks):

  regime                                          threshold (file:line)                       covered by
  ----------------------------------------------  ------------------------------------------  ---------------------------------
  pigp_potrf_lower: recursion / panels W=2/4/16   pigp_dist.cu:579-581 (12, 64, 128)           test_potrf_potri_exact, T in
                                                  (the solver's NLL-only rule)                 POTRF_T (both sides of each break,
                                                                                               odd T, short last panel), T 17/65
                                                                                               with pigp_set_lookahead(0)
  block-TRSM slab height 8 / 16 / 32 rows         pigp_dense.cu:614-618 (1184 / 2368 rows)     same (panel heights up to 16.8k)
  k_gemm BN 64 / 128, lower_only, remainder       pigp_dense.cu:689-722, PIGP_GEMM_BN           test_dgemm_*, test_knobs
  small-tile GEMMs (solver launches)              pigp_dense.cu:689-707, PIGP_GEMM_SMALL        test_solver_regime, test_knobs
  solver NLL + gradient: rec / W=2 / W=4 / rec    pigp_dist.cu:580 (16, 32, 96)                test_solver_regime, SOLVER_T
  solver NLL only: rec / W=2 / 4 / 16             pigp_dist.cu:579-581 (12, 64, 128)           test_solver_regime (also width 0)
  early K^-1 accumulation (one rank, 8..32)       pigp_dist.cu:929; late product :1016-1026    test_solver_regime (T 7/8, 32/33),
                                                                                               test_knobs (PIGP_EARLY_KINV=0)
  pigp_predict (factors through NLL only)         pigp_capi.cu:606                             test_solver_regime (M = 300)
  block-cyclic ranks                              pigp_dist.cu                                 test_ranks_at_33_tiles
  reuse of one solver after a failed evaluation   pigp_dist.cu:933-958                         test_reuse_after_failure (T 4/16/40),
                                                                                               test_adam_after_failure

References: the exact-factor SPD family L0 = c I + R (R strictly lower in {-1, 0, 1}, c a power of two >= 4 sqrt(n)) has the
exact Cholesky factor L0 of A = L0 L0^T (exact in float64; every pivot is c^2); integer GEMM operands make every product and
partial sum exact, so pigp_dgemm must equal torch bit for bit.  The solver is compared with a float64 evaluation of its own
matrix (Plan.assemble, itself checked against oracle.closed_form) through torch / cuSOLVER, with dK/dtheta from the
oracle's closed-form derivatives evaluated on the GPU (closed_form_grad; checked against the numpy oracle's gradient in
tests/test_grad_reference_cpu.py).  Finite differences of the assembly are not accurate enough for that reference: the
gradient sum_jk M_jk dK_jk cancels ~1e4-fold, so the smooth O(h^4) truncation error of a Richardson-extrapolated central
difference (2e-11 of max |dK| entry-wise) reaches 6e-10 of max |grad| at N = 890, above the 1e-10 bar.
Every case prints T, the regime, the largest error and the bar.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from stopro_b200 import synthetic

pytestmark = pytest.mark.gpu

U = 2.0 ** -52
COND_FRAC = 0.05            # of cond(K) * u, the rule of tests/test_gpu_parity.py
GRAD_SPREAD = 10.0          # gradient bar: times the spread of two float64 references (Problem.reference)
TILE = 128
SENTINEL = 7.25             # guard value: exactly representable, never produced by the integer-valued cases
POTRF_T = [1, 2, 3, 5, 11, 12, 13, 17, 33, 63, 64, 65, 127, 128, 131]
SOLVER_T = [7, 8, 15, 16, 32, 33, 63, 64, 95, 96, 127, 128]


def closed_form_grad(cfg, theta, M):
    """0.5 sum_jk M_jk dK_jk/dtheta_p for M = K^-1 - alpha alpha^T (torch, float64, on M's device), dK/dtheta from the
    closed-form derivatives of oracle.closed_form evaluated block by block on M's device: independent of the fused
    analytic evaluator of the CUDA path (squared-exponential kernels, no noise parameter)."""
    import torch

    from conftest import oracle_for
    from oracle import blocks_ref, closed_form

    ref = oracle_for(cfg)
    assert ref.kernel_type == "se" and not ref.index_optimize_noise
    pts = [torch.as_tensor(np.asarray(p, dtype=np.float64).reshape(len(p), -1), device=M.device) for p in cfg["r_train"]]
    sec = np.concatenate([[0], np.cumsum([len(p) for p in pts])])
    lbox = None if ref.lbox is None else torch.as_tensor(ref.lbox, device=M.device)
    th = np.asarray(theta, dtype=np.float64)
    rows, blocks, groups = ref.table["training"], ref.table["blocks"], ref.table["groups"]
    g = np.zeros(len(th))
    for i in range(len(pts)):
        for j in range(i, len(pts)):
            terms, shift = blocks_ref.parse_spec(blocks[rows[i][j - i]], blocks)
            Mij = M[sec[i]:sec[i + 1], sec[j]:sec[j + 1]]
            w = 1.0 if i == j else 2.0  # M and K are symmetric: block (j, i) is the transpose of (i, j)
            for sign, op, group in terms:
                sl = groups[group]

                def base(a, b):
                    return closed_form.eval_operator(op, a, b, th[sl], ref.form, ref.dim, with_grad=True)[1]

                a, b = pts[i], pts[j]
                if shift is None:
                    dG = base(a, b)
                elif shift == "Xp":
                    dG = base(a, b + lbox) - base(a, b)
                elif shift == "X":
                    dG = base(a + lbox, b) - base(a, b)
                else:
                    dG = base(a + lbox, b + lbox) - base(a + lbox, b) - base(a, b + lbox) + base(a, b)
                for q, p in enumerate(list(range(len(th)))[sl]):
                    g[p] += w * sign * float((Mij * dG[q]).sum())
    return 0.5 * g


def _lib():
    from stopro_b200 import _lib as L

    return L


def _nan_like(t):
    import torch

    return torch.full_like(t, float("nan"))


def relerr(a, b):
    d = (a - b).abs().max().item()
    return d / max(b.abs().max().item(), 1e-300)


def exact_factor(n, dev, seed):
    """L0 = c I + R with R strictly lower in {-1, 0, 1} and c the power of two >= 4 sqrt(n); A = L0 L0^T exactly."""
    import torch

    g = torch.Generator(device=dev).manual_seed(seed)
    c = 2.0 ** int(np.ceil(np.log2(4.0 * np.sqrt(n))))
    R = torch.randint(-1, 2, (n, n), generator=g, device=dev).to(torch.float64).tril(-1)
    L0 = R + c * torch.eye(n, dtype=torch.float64, device=dev)
    return L0, L0 @ L0.t()


def tri_inv(L):
    import torch

    return torch.linalg.solve_triangular(L, torch.eye(L.shape[0], dtype=L.dtype, device=L.device), upper=False)


def _potrf_case(n, m_extra, ld, seed, dev, extra_rows=2):
    """Buffer with rows [0, n) = A (strictly upper part NaN), [n, n + m_extra) = E, `extra_rows` guard rows below, guard
    columns [n, ld) holding SENTINEL."""
    import torch

    L0, A = exact_factor(n, dev, seed)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    E = torch.randint(-2, 3, (m_extra, n), generator=g, device=dev).to(torch.float64)
    buf = torch.full((n + m_extra + extra_rows, ld), SENTINEL, dtype=torch.float64, device=dev)
    buf[:n, :n] = A.tril() + torch.full_like(A, float("nan")).triu(1)
    buf[n:n + m_extra, :n] = E
    return L0, E, buf


def _check_guards(buf, n, rows):
    """Guard columns [n, ld) of every row and the guard rows below the matrix still hold SENTINEL."""
    assert bool((buf[:, n:] == SENTINEL).all()), "guard columns were written"
    assert bool((buf[rows:] == SENTINEL).all()), "guard rows were written"


def _potrf_width(T):
    return 0 if T < 12 else 2 if T < 64 else 4 if T < 128 else 16


@pytest.mark.parametrize("T,lookahead", [pytest.param(T, -1, id=str(T)) for T in POTRF_T] +
                         [pytest.param(T, 0, id=f"{T}-lookahead0") for T in (17, 65)])
def test_potrf_potri_exact(cuda_device, T, lookahead):
    """pigp_potrf_lower / pigp_potri_lower against the exact factor, with poisoned inputs and workspaces, padded ld and
    extra rows; every inverse diagonal tile checked.  lookahead = 0: pigp_set_lookahead(0), which steers pigp_potrf_lower
    as it steers the solver, makes it take the plain recursion where the automatic width would take panels."""
    import torch

    L = _lib()
    lib = L.lib()
    dev = cuda_device
    n = T * TILE
    # each T takes one (m_extra, ld) pair; over POTRF_T every value of each meets small and large T
    m_extra = [0, 128, n + 256][T % 3]
    ld = [n, n + 2, n + 256][(T // 3) % 3]
    L0, E, buf = _potrf_case(n, m_extra, ld, T, dev)
    invd = torch.full((T, TILE, TILE), float("nan"), dtype=torch.float64, device=dev)
    info = torch.full((1,), -7, dtype=torch.int32, device=dev)
    L.check(lib.pigp_set_lookahead(lookahead))
    try:
        L.check(lib.pigp_potrf_lower(buf.data_ptr(), ld, n, m_extra, invd.data_ptr(), info.data_ptr(), None))
        torch.cuda.synchronize()
    finally:
        L.check(lib.pigp_set_lookahead(-1))
    assert int(info.item()) == 0
    _check_guards(buf, n, n + m_extra)
    e_L = relerr(buf[:n, :n].tril(), L0)
    W0 = tri_inv(L0)
    e_E = relerr(buf[n:n + m_extra, :n], E @ W0.t()) if m_extra else 0.0
    e_inv = 0.0
    for k in range(T):
        Wk = invd[k]
        assert float(Wk.triu(1).abs().max()) == 0.0, f"inverse tile {k} is not zero above its diagonal"
        e_inv = max(e_inv, relerr(Wk, tri_inv(L0[k * TILE:(k + 1) * TILE, k * TILE:(k + 1) * TILE])))
    W = _potrf_width(T) if lookahead < 0 else lookahead
    print(f"\n[potrf T={T} W={W} m_extra={m_extra} ld={ld}] L {e_L:.1e} extra {e_E:.1e} "
          f"invd {e_inv:.1e} (bars 1e-13 / 1e-12 / 1e-12)")
    assert e_L <= 1e-13 and e_E <= 1e-12 and e_inv <= 1e-12

    # potri into NaN-filled W and X (X separate), then with X aliasing L
    Ainv = W0.t() @ W0
    Lbuf = buf[:n + m_extra]  # same ld
    Wb = torch.full((n + 2, ld), float("nan"), dtype=torch.float64, device=dev)
    Wb[n:] = SENTINEL
    Wb[:n, n:] = SENTINEL
    Xb = Wb.clone()
    L.check(lib.pigp_potri_lower(Lbuf.data_ptr(), ld, n, invd.data_ptr(), Wb.data_ptr(), Xb.data_ptr(), None))
    torch.cuda.synchronize()
    _check_guards(Wb, n, n)
    _check_guards(Xb, n, n)
    e_W = relerr(Wb[:n, :n].tril(), W0)
    e_X = relerr(Xb[:n, :n].tril(), Ainv.tril())
    L.check(lib.pigp_potri_lower(Lbuf.data_ptr(), ld, n, invd.data_ptr(), Wb.data_ptr(), Lbuf.data_ptr(), None))
    torch.cuda.synchronize()
    _check_guards(buf, n, n + m_extra)
    e_alias = relerr(buf[:n, :n].tril(), Ainv.tril())
    print(f"[potri T={T}] L^-1 {e_W:.1e} A^-1 {e_X:.1e} aliased {e_alias:.1e} (bar 1e-12)")
    assert e_W <= 1e-12 and e_X <= 1e-12 and e_alias <= 1e-12


@pytest.mark.parametrize("n,how", [(640, "extended"), (2176, "cusolver"), (8320, "cusolver")])
def test_potrf_potri_random_spd(cuda_device, n, how):
    """X X^T / n + I: against the long-double oracle (n <= 1024) or cuSOLVER float64, whose own error at this
    conditioning (cond ~ 5) is a few u."""
    import torch

    L = _lib()
    lib = L.lib()
    dev = cuda_device
    g = torch.Generator(device=dev).manual_seed(n)
    X = torch.randn(n, n, dtype=torch.float64, device=dev, generator=g)
    S = X @ X.t() / n + torch.eye(n, dtype=torch.float64, device=dev)
    if how == "extended":
        from oracle import extended

        Ld = extended.cholesky_lower(S.cpu().numpy())
        Wd = extended.tri_inv_lower(Ld)
        Lref = torch.as_tensor(Ld.astype(np.float64), device=dev)
        Wref = torch.as_tensor(Wd.astype(np.float64), device=dev)
        Xref = torch.as_tensor((Wd.T @ Wd).astype(np.float64), device=dev)
    else:
        Lref = torch.linalg.cholesky(S)
        Wref = tri_inv(Lref)
        Xref = torch.cholesky_inverse(Lref)
    buf = S.tril() + torch.full_like(S, float("nan")).triu(1)
    invd = torch.full((n // TILE, TILE, TILE), float("nan"), dtype=torch.float64, device=dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    L.check(lib.pigp_potrf_lower(buf.data_ptr(), n, n, 0, invd.data_ptr(), info.data_ptr(), None))
    Wb, Xb = _nan_like(S), _nan_like(S)
    L.check(lib.pigp_potri_lower(buf.data_ptr(), n, n, invd.data_ptr(), Wb.data_ptr(), Xb.data_ptr(), None))
    torch.cuda.synchronize()
    assert int(info.item()) == 0
    e = (relerr(buf.tril(), Lref), relerr(Wb.tril(), Wref), relerr(Xb.tril(), Xref.tril()))
    print(f"\n[random SPD n={n} T={n // TILE} vs {how}] L {e[0]:.1e} L^-1 {e[1]:.1e} A^-1 {e[2]:.1e} (bars 1e-12 / 1e-11)")
    assert e[0] <= 1e-12 and e[1] <= 1e-11 and e[2] <= 1e-11


@pytest.mark.parametrize("T,cols", [(16, [12 * 128 + 37]), (16, [13 * 128, 15 * 128 + 127]),
                                    (65, [40 * 128 + 77]), (65, [64 * 128 + 5]), (65, [12 * 128 + 1, 50 * 128 + 64])])
def test_failing_pivot_under_the_panel_schedule(cuda_device, T, cols):
    """A non-positive pivot inside a panel of the look-ahead schedule: info = the first bad column (1-based), columns
    before it exact, NaN from it on."""
    import torch

    L = _lib()
    lib = L.lib()
    dev = cuda_device
    n = T * TILE
    L0, A = exact_factor(n, dev, 100 + T)
    c2 = float(L0[0, 0]) ** 2
    for j in cols:
        A[j, j] -= 1.5 * c2  # pivot c^2 - 1.5 c^2 < 0, exactly
    j = cols[0]
    buf = A.tril() + torch.full_like(A, float("nan")).triu(1)
    invd = torch.full((T, TILE, TILE), float("nan"), dtype=torch.float64, device=dev)
    info = torch.zeros(1, dtype=torch.int32, device=dev)
    L.check(lib.pigp_potrf_lower(buf.data_ptr(), n, n, 0, invd.data_ptr(), info.data_ptr(), None))
    torch.cuda.synchronize()
    # as LAPACK's potrf: the leading j x j factor is valid.  Rows below it are valid left of the failing 128-column
    # tile (earlier panels); inside that tile their TRSM uses the tile's inverse, which the failed pivot has poisoned.
    t0 = TILE * (j // TILE)
    e = max(relerr(buf[:j, :j].tril(), L0[:j, :j]), relerr(buf[j:, :t0], L0[j:, :t0]) if t0 else 0.0)
    trail = buf[j:, j:].tril()
    mask = torch.ones_like(trail, dtype=torch.bool).tril()
    nan_left = int(torch.isnan(buf[j:, t0:j]).sum())
    print(f"\n[failing pivot T={T} W={_potrf_width(T)} cols={cols}] info {int(info.item())} error before the column "
          f"{e:.1e} (bar 1e-13); NaN below row j in the failing tile's earlier columns: {nan_left}")
    assert int(info.item()) == j + 1
    assert e <= 1e-13
    assert bool(torch.isnan(trail[mask]).all())


# ------------------------------------------------------------------------------------------------------------ GEMM
GEMM_SHAPES = [(2048, 2048, 2048), (4096, 1024, 512), (128, 4096, 256), (1024, 1024, 384), (1536, 1024, 2560)]
ALPHA_BETA = [(1.0, 1.0), (-1.0, 0.5), (0.5, -2.0), (-2.0, 0.0)]


def _gemm_operands(M, N, K, akc, bkc, dev, g, integer):
    """A(m,k), B(n,k) stored k-contiguous ([m][k]) or m-contiguous ([k][m]) with a padded, even leading dimension."""
    import torch

    def make(rows, cols):
        if integer:
            return torch.randint(-2, 3, (rows, cols), generator=g, device=dev).to(torch.float64)
        return torch.randn(rows, cols, generator=g, device=dev, dtype=torch.float64)

    A, B = make(M, K), make(N, K)

    def store(X, kc):
        Xs = X if kc else X.t()
        s = torch.full((Xs.shape[0], Xs.shape[1] + 6), SENTINEL, dtype=torch.float64, device=dev)
        s[:, :Xs.shape[1]] = Xs
        return s

    return A, B, store(A, akc), store(B, bkc)


def _run_gemm(M, N, K, alpha, beta, As, akc, Bs, bkc, C, lower):
    L = _lib()
    return L.lib().pigp_dgemm(M, N, K, alpha, As.data_ptr(), As.stride(0), akc, Bs.data_ptr(), Bs.stride(0), bkc, beta,
                              C.data_ptr(), C.stride(0), lower, None)


@pytest.mark.parametrize("lower", [0, 1])
@pytest.mark.parametrize("shape", GEMM_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_dgemm_exact(cuda_device, shape, lower):
    """Integer operands: every partial sum is exact in any order, so C must equal alpha A B^T + beta C0 bit for bit.
    lower_only writes whole 128-row diagonal tiles and every tile left of them (and, for M > N, every row below N): the
    tiles strictly above the diagonal tile row keep their sentinel.  beta = 0 ignores a NaN-filled C.  Guard columns
    (ldc = N + 4) and a guard row stay untouched.  One float-valued case per orientation at 1e-13."""
    import torch

    L = _lib()
    dev = cuda_device
    M, N, K = shape
    g = torch.Generator(device=dev).manual_seed(M + 3 * N + 7 * K + lower)
    if lower and M < N:
        A, B, As, Bs = _gemm_operands(M, N, K, 1, 1, dev, g, True)
        C = torch.zeros(M + 1, N + 4, dtype=torch.float64, device=dev)
        before = L.launch_count()
        assert _run_gemm(M, N, K, 1.0, 0.0, As, 1, Bs, 1, C, 1) == -1  # PIGP_EINVAL
        assert L.launch_count() == before
        return
    rows = torch.arange(M, device=dev).view(-1, 1) // TILE
    cols = torch.arange(N, device=dev).view(1, -1) // TILE
    written = (cols <= rows) if lower else torch.ones(M, N, dtype=torch.bool, device=dev)
    worst = 0.0
    for i, (akc, bkc) in enumerate([(1, 1), (1, 0), (0, 1), (0, 0)]):
        for integer in (True, False):
            alpha, beta = ALPHA_BETA[i] if integer else (-0.5, 2.0)
            A, B, As, Bs = _gemm_operands(M, N, K, akc, bkc, dev, g, integer)
            C0 = (torch.randint(-3, 4, (M, N), generator=g, device=dev).to(torch.float64) if integer
                  else torch.randn(M, N, generator=g, device=dev, dtype=torch.float64))
            C = torch.full((M + 1, N + 4), SENTINEL, dtype=torch.float64, device=dev)
            C[:M, :N] = torch.where(written, C0 if beta != 0.0 else torch.full_like(C0, float("nan")),
                                    torch.full_like(C0, SENTINEL))
            L.check(_run_gemm(M, N, K, alpha, beta, As, akc, Bs, bkc, C, lower))
            torch.cuda.synchronize()
            want = alpha * (A @ B.t()) + (beta * C0 if beta != 0.0 else 0.0)
            got = C[:M, :N]
            assert bool((C[M:] == SENTINEL).all()) and bool((C[:, N:] == SENTINEL).all()), "guards written"
            assert bool((got[~written] == SENTINEL).all()), "a tile above the diagonal tile row was written"
            if integer:
                assert torch.equal(got[written], want[written]), f"akc={akc} bkc={bkc}: not exact"
            else:
                e = relerr(torch.where(written, got, 0.0), torch.where(written, want, 0.0))
                worst = max(worst, e)
                assert e < 1e-13, (akc, bkc, e)
    print(f"\n[dgemm {M}x{N}x{K} lower_only={lower}] integer cases exact; float worst {worst:.1e} (bar 1e-13)")


@pytest.mark.parametrize("which", ["lda", "ldb", "ldc"])
def test_dgemm_rejects_odd_leading_dimension(cuda_device, which):
    """The operand copies are 16-byte cp.async of element pairs: an odd leading dimension is refused before any launch."""
    import torch

    L = _lib()
    buf = torch.zeros(128 * 130, dtype=torch.float64, device=cuda_device)
    ld = {"lda": 128, "ldb": 128, "ldc": 128}
    ld[which] = 129
    before = L.launch_count()
    rc = L.lib().pigp_dgemm(128, 128, 128, 1.0, buf.data_ptr(), ld["lda"], 1, buf.data_ptr(), ld["ldb"], 1, 0.0,
                            buf.data_ptr(), ld["ldc"], 0, None)
    assert rc == -1 and b"even" in L.lib().pigp_last_error()
    assert L.launch_count() == before


# ---------------------------------------------------------------------------------------------------------- solver
def _n_for(T):
    """N = 128 T - r with r in 1..127 (padding), and the exact multiple for T = 64."""
    return 128 * T - (0 if T == 64 else 1 + (37 * T) % 127)


def _nll_width(T):
    return 0 if T < 12 else 2 if T < 64 else 4 if T < 128 else 16


def _grad_width(T):
    return 2 if 16 <= T < 32 else 4 if 32 <= T < 96 else 0


def _theta(cfg):
    return cfg["theta0"] + 0.05 * np.random.default_rng(11).standard_normal(len(cfg["theta0"]))


class Problem:
    """stokes2d_scaling(N) with eps = 1 and its float64 reference on the GPU: K from the solver's own plan (checked
    against oracle.closed_form on sampled entries), L and K^-1 from cuSOLVER, dK/dtheta from closed_form_grad."""

    def __init__(self, N, dev, n_test=100):
        import torch

        self.cfg = dict(synthetic.stokes2d_scaling(N, n_test=n_test), eps=1.0)
        self.N, self.dev = N, dev
        self.gp = synthetic.make_model(self.cfg)
        c = self.cfg
        self.gp.set_constants(c["r_test"], c["mu_test"], c["r_train"], c["delta_y"], c["eps"])
        self.plan = self.gp._training_plan(c["r_train"])
        self.th = _theta(c)
        self.y = torch.as_tensor(c["delta_y"], device=dev)

    def solver(self):
        return self.gp._solver_for(self.cfg["r_train"])

    def assemble(self, plan, th, eps, add_diag):
        import torch

        K = torch.empty(plan.rows, plan.cols, dtype=torch.float64, device=self.dev)
        t = torch.as_tensor(np.asarray(th, dtype=np.float64), device=self.dev)
        plan.assemble(t.data_ptr(), eps, add_diag, K.data_ptr(), plan.cols)
        torch.cuda.synchronize()
        return K

    def K(self, th):
        return self.assemble(self.plan, th, self.cfg["eps"], 1)

    def check_assembly(self, K):
        """20 000 sampled entries of the plan's K against oracle.closed_form (the reference must not just echo the CUDA
        assembly)."""
        from conftest import oracle_for

        ref = oracle_for(self.cfg)
        pts = ref._pts(self.cfg["r_train"])
        sec = np.concatenate([[0], np.cumsum([len(p) for p in pts])])
        rng = np.random.default_rng(self.N)
        R, Cc = np.sort(rng.choice(self.N, 150, replace=False)), np.sort(rng.choice(self.N, 134, replace=False))
        want = np.zeros((len(R), len(Cc)))
        table = ref.table["training"]
        for bi in range(len(pts)):
            ri = np.nonzero((R >= sec[bi]) & (R < sec[bi + 1]))[0]
            for bj in range(len(pts)):
                cj = np.nonzero((Cc >= sec[bj]) & (Cc < sec[bj + 1]))[0]
                if len(ri) == 0 or len(cj) == 0:
                    continue
                a, b = pts[bi][R[ri] - sec[bi]], pts[bj][Cc[cj] - sec[bj]]
                blk = (ref.block(table[bi][bj - bi], a, b, self.th) if bi <= bj
                       else ref.block(table[bj][bi - bj], b, a, self.th).T)
                want[np.ix_(ri, cj)] = blk
        want[R[:, None] == Cc[None, :]] += self.cfg["eps"]
        import torch

        got = K[torch.as_tensor(R, device=K.device)][:, torch.as_tensor(Cc, device=K.device)].cpu().numpy()
        e = np.max(np.abs(got - want)) / K.abs().max().item()
        assert e <= 1e-12, f"Plan.assemble differs from oracle.closed_form by {e:.2e}"
        return e

    def reference(self):
        """-> dict(nll, grad, L, cond) in float64 (torch / cuSOLVER)."""
        import torch

        K = self.K(self.th)
        e_asm = self.check_assembly(K)
        L = torch.linalg.cholesky(K)
        v = torch.linalg.solve_triangular(L, self.y.view(-1, 1), upper=False).view(-1)
        nll = 0.5 * float(v @ v) + float(torch.log(torch.diagonal(L)).sum()) + 0.5 * self.N * np.log(2.0 * np.pi)
        Kinv = torch.cholesky_inverse(L)
        alpha = Kinv @ self.y
        M = Kinv - torch.outer(alpha, alpha)
        # cond_2(K) from power iterations on K and K^-1 (symmetric positive definite)
        lam = []
        for Mat in (K, Kinv):
            x = torch.ones(self.N, dtype=torch.float64, device=self.dev)
            for _ in range(60):
                x = Mat @ x
                x /= x.norm()
            lam.append(float(x @ (Mat @ x)))
        cond = lam[0] * lam[1]
        del Kinv
        grad = closed_form_grad(self.cfg, self.th, M)
        # The gradient sum_jk M_jk dK_jk cancels: at N = 16k its terms exceed the result ~1e4-fold, so two correct float64
        # evaluations differ by more than cond(K) u.  The spread between this reference and a second one through an
        # LU-based inverse (another algorithm, same data) measures that; the gradient bar is the larger of the NLL bar
        # and GRAD_SPREAD times the spread.
        del M
        Kinv2 = torch.linalg.inv(K)
        alpha2 = torch.linalg.solve(K, self.y)
        M2 = 0.5 * (Kinv2 + Kinv2.t()) - torch.outer(alpha2, alpha2)
        del Kinv2, K
        spread = np.max(np.abs(closed_form_grad(self.cfg, self.th, M2) - grad)) / np.max(np.abs(grad))
        tol = max(1e-10, COND_FRAC * cond * U)
        return dict(nll=nll, grad=grad, L=L, cond=cond, e_asm=e_asm, tol=tol, spread=spread,
                    tol_g=max(tol, GRAD_SPREAD * spread))

    def close(self):
        self.gp.close()


def _nll_dev(solver, th, y, eps, want_grad):
    """One device-pointer evaluation -> (nll, grad or None, info)."""
    import torch

    dev = y.device
    t = torch.as_tensor(np.asarray(th, dtype=np.float64), device=dev)
    out = torch.full((1 + len(th),), float("nan"), dtype=torch.float64, device=dev)
    info = torch.full((1,), -7, dtype=torch.int32, device=dev)
    if want_grad:
        solver.nll_grad(t.data_ptr(), y.data_ptr(), eps, out.data_ptr(), out.data_ptr() + 8, info.data_ptr(), None)
    else:
        solver.nll(t.data_ptr(), y.data_ptr(), eps, out.data_ptr(), info.data_ptr(), None)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    return o[0], (o[1:] if want_grad else None), int(info.item())


@pytest.mark.parametrize("T", SOLVER_T)
def test_solver_regime(cuda_device, T):
    """NLL + gradient, NLL only (automatic width, and width 0 where the automatic one is 4 or 16) and pigp_predict (mean,
    full covariance, variances; M = 300 test points) against the float64 reference of the solver's own matrix."""
    import torch

    L = _lib()
    pb = Problem(_n_for(T), cuda_device)
    try:
        ref = pb.reference()
        tol, tol_g = ref["tol"], ref["tol_g"]
        solver, eps = pb.solver(), pb.cfg["eps"]
        early = T >= 8 and T <= 32
        nll, grad, info = _nll_dev(solver, pb.th, pb.y, eps, True)
        assert info == 0
        e_n = abs(nll - ref["nll"]) / abs(ref["nll"])
        e_g = np.max(np.abs(grad - ref["grad"])) / np.max(np.abs(ref["grad"]))
        print(f"\n[solver T={T} N={pb.N}] cond(K) {ref['cond']:.2e} tol {tol:.1e}; assembly vs oracle {ref['e_asm']:.1e}; "
              f"gradient tol {tol_g:.1e} (reference spread {ref['spread']:.1e})\n"
              f"  NLL+grad (W={_grad_width(T)}, {'early' if early else 'late'} K^-1): nll {e_n:.1e} grad {e_g:.1e}")
        assert e_n <= tol and e_g <= tol_g
        widths = [-1] + ([0] if _nll_width(T) >= 4 else [])
        try:
            for w in widths:
                L.check(L.lib().pigp_set_lookahead(w))
                v, _, info = _nll_dev(solver, pb.th, pb.y, eps, False)
                e = abs(v - ref["nll"]) / abs(ref["nll"])
                print(f"  NLL only (W={_nll_width(T) if w < 0 else w}{' auto' if w < 0 else ''}): nll {e:.1e}")
                assert info == 0 and e <= tol
        finally:
            L.check(L.lib().pigp_set_lookahead(-1))
        c = pb.cfg
        mixed, test = pb.gp._mixed_plan(c["r_test"], c["r_train"]), pb.gp._test_plan(c["r_test"])
        Kab = pb.assemble(mixed, pb.th, 0.0, 0)
        Kaa = pb.assemble(test, pb.th, 0.0, 0)
        Lr = ref["L"]
        alpha = torch.cholesky_solve(pb.y.view(-1, 1), Lr).view(-1)
        V = torch.linalg.solve_triangular(Lr, Kab.t(), upper=False)
        mu_ref = (Kab @ alpha).cpu().numpy()
        cov_ref = (Kaa - V.t() @ V).cpu().numpy()
        mu, cov, info = solver.predict_host(mixed, test, pb.th, c["delta_y"], eps, full_cov=True)
        mu_d, var, info_d = solver.predict_host(mixed, test, pb.th, c["delta_y"], eps, full_cov=False)
        assert info == 0 and info_d == 0
        scale_cov = max(np.max(np.abs(Kaa.cpu().numpy())), np.max(np.abs(cov_ref)))
        e_mu = np.max(np.abs(mu - mu_ref)) / np.max(np.abs(mu_ref))
        e_cov = np.max(np.abs(cov - cov_ref)) / scale_cov
        e_var = np.max(np.abs(var - np.diag(cov))) / scale_cov
        print(f"  predict (M=300, NLL-only factor W={_nll_width(T)}): mu {e_mu:.1e} cov {e_cov:.1e} var-vs-diag {e_var:.1e}")
        assert mu.shape == (300,) and cov.shape == (300, 300)
        assert e_mu <= tol and e_cov <= tol and e_var <= tol
        assert np.array_equal(mu_d, mu)
    finally:
        pb.close()


@pytest.mark.parametrize("world", [2, 3])
def test_ranks_at_33_tiles(cuda_device, world):
    """Two and three in-process ranks at T = 33 against the same float64 reference (bitwise equal across ranks)."""
    from test_gpu_dist import run_ranks

    pb = Problem(_n_for(33), cuda_device)
    try:
        ref = pb.reference()
        tol, tol_g = ref["tol"], ref["tol_g"]
        out = run_ranks(pb.gp, pb.cfg, pb.th, world)
        for nll, grad, info in out:
            assert info == 0
            e_n = abs(nll - ref["nll"]) / abs(ref["nll"])
            e_g = np.max(np.abs(grad - ref["grad"])) / np.max(np.abs(ref["grad"]))
            assert e_n <= tol and e_g <= tol_g
        print(f"\n[ranks T=33 world={world}] nll {e_n:.1e} grad {e_g:.1e} tol {tol:.1e} gradient tol {tol_g:.1e}")
        for nll, grad, _ in out[1:]:
            assert nll == out[0][0] and np.array_equal(grad, out[0][1])
    finally:
        pb.close()


# -------------------------------------------------------------------------------------------- reuse after a failure
def _two_models(T, dev):
    """(used, fresh): two models (one solver each) over the same T-tile problem."""
    N = _n_for(T)
    return Problem(N, dev), Problem(N, dev)


@pytest.mark.parametrize("T", [4, 16, 40])
def test_reuse_after_failure(cuda_device, T):
    """After a non-positive-definite evaluation (eps = -10: info != 0, NaN results) the same solver's next NLL-only,
    NLL + gradient and predict calls equal a fresh solver's, bitwise; so do alternating NLL-only / NLL + gradient calls
    (at T = 40 their panel widths differ: 2 and 4)."""
    used, fresh = _two_models(T, cuda_device)
    try:
        s, f = used.solver(), fresh.solver()
        c = used.cfg
        for grad in (True, False):
            nll, g, info = _nll_dev(s, used.th, used.y, -10.0, grad)
            assert info != 0 and np.isnan(nll) and (g is None or np.all(np.isnan(g)))
        mixed, test = used.gp._mixed_plan(c["r_test"], c["r_train"]), used.gp._test_plan(c["r_test"])
        fm, ft = fresh.gp._mixed_plan(c["r_test"], c["r_train"]), fresh.gp._test_plan(c["r_test"])
        for grad in (False, True, False, True):
            a = _nll_dev(s, used.th, used.y, c["eps"], grad)
            b = _nll_dev(f, fresh.th, fresh.y, c["eps"], grad)
            assert a[2] == 0 and b[2] == 0
            assert a[0] == b[0] and (not grad or np.array_equal(a[1], b[1])), f"grad={grad}: {a[0]!r} vs {b[0]!r}"
            # fail again before the next good call
            _nll_dev(s, used.th, used.y, -10.0, not grad)
        for full in (True, False):
            _nll_dev(s, used.th, used.y, -10.0, True)
            mu, cov, info = s.predict_host(mixed, test, used.th, c["delta_y"], c["eps"], full_cov=full)
            mu0, cov0, info0 = f.predict_host(fm, ft, fresh.th, c["delta_y"], c["eps"], full_cov=full)
            assert info == 0 and info0 == 0
            assert np.array_equal(mu, mu0) and np.array_equal(cov, cov0), f"predict full_cov={full}"
        print(f"\n[reuse T={T} NLL W={_nll_width(T)} grad W={_grad_width(T)}] bitwise equal to a fresh solver")
    finally:
        used.close()
        fresh.close()


def test_adam_after_failure(cuda_device):
    """pigp_adam_host from a good theta0 after a run that ended with a NaN status equals the same run on a fresh solver."""
    used, fresh = _two_models(16, cuda_device)
    try:
        s, f = used.solver(), fresh.solver()
        c = used.cfg
        args = dict(max_iter=6, lr=1e-2, stop_eps=0.0, ntraining=float(used.N), check_every=2)
        _, _, _, status = s.adam_host(used.th, c["delta_y"], -10.0, **args)
        assert status == 4  # initial loss NaN
        a = s.adam_host(used.th, c["delta_y"], c["eps"], **args)
        b = f.adam_host(fresh.th, c["delta_y"], c["eps"], **args)
        assert a[3] == b[3] == 0
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(x, y)
        print(f"\n[adam after failure T=16] {len(a[1]) - 1} iterations bitwise equal to a fresh solver")
    finally:
        used.close()
        fresh.close()


# ----------------------------------------------------------------------------------------- knobs read once per process
def knob_child_checks():
    """What a child process started with one of the knobs set runs: a GEMM, a potrf / potri case and an NLL + gradient at
    T = 16, each against the references above."""
    import torch

    dev = torch.device("cuda:0")
    test_dgemm_exact(dev, (2048, 2048, 2048), 1)
    test_dgemm_exact(dev, (4096, 1024, 512), 1)
    test_potrf_potri_exact(dev, 17, -1)
    pb = Problem(_n_for(16), dev)
    try:
        ref = pb.reference()
        tol, tol_g = ref["tol"], ref["tol_g"]
        nll, grad, info = _nll_dev(pb.solver(), pb.th, pb.y, pb.cfg["eps"], True)
        e_n = abs(nll - ref["nll"]) / abs(ref["nll"])
        e_g = np.max(np.abs(grad - ref["grad"])) / np.max(np.abs(ref["grad"]))
        print(f"[T=16 NLL+grad] nll {e_n:.1e} grad {e_g:.1e} tol {tol:.1e} gradient tol {tol_g:.1e}")
        assert info == 0 and e_n <= tol and e_g <= tol_g
    finally:
        pb.close()


@pytest.mark.parametrize("knob", ["PIGP_GEMM_BN=128", "PIGP_GEMM_SMALL=0", "PIGP_EARLY_KINV=0"])
def test_knobs(cuda_device, knob):
    """The tuning knobs are read into statics at first use, so each runs in a child process of its own."""
    key, val = knob.split("=")
    env = dict(os.environ, **{key: val})
    here = os.path.dirname(os.path.abspath(__file__))
    code = f"import sys; sys.path.insert(0, {here!r}); import test_gpu_regimes as t; t.knob_child_checks()"
    r = subprocess.run([sys.executable, "-c", code], cwd=os.path.dirname(here), env=env, capture_output=True, text=True,
                       timeout=900)
    print(f"\n[{knob}]\n{r.stdout[-3000:]}")
    assert r.returncode == 0, r.stderr[-4000:]
