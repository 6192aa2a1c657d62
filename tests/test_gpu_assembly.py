"""Entry-wise GPU tests of covariance assembly (k_blocks<.., false>, k_blocks_matern) and of the fused trace gradient
(k_blocks<.., true>, k_blocks_matern<.., true>, k_reduce_partials) against oracle.desc_ref, an extended-precision
(numpy.longdouble) evaluator of the same descriptor tables.

Error bars (u = 2^-53).  The reference takes the float64 differences s the kernels form (r + lbox first, then the
difference), so only the kernels' own roundings count:

  K entry:   |K_gpu - K_ref| <= C_K u A (1 + U)
     A = sum of |monomial| * exponential over every term and shift combination (desc_ref), U = largest exponent argument.
     Derivation of C_K = 64: gamma, a (or c) = exp of theta: <= 2u each; powers a^k and coefficient products (total
     derivative order <= 4, <= 3 dimensions): <= 12u; Horner over <= 10 coefficients: <= 20u; the sum over <= 8 runs x 4
     shift combinations (or <= 8 terms x 4 combinations for Matern): <= 31u -- all relative to A.  The exponent argument
     is formed from a rounded a and s^2 with <= 3 fma: relative error <= 6u, which exp turns into <= 6u U; exp itself
     <= 2u.  Total < 64u A + 6u A U <= C_K u A (1 + U).
     Where the argument is formed exactly (dyadic points with theta = 0: a = gamma = 1, s^2 and the fma chain exact),
     the U term is absent: |K_gpu - K_ref| <= C_K u A.
     Entries whose argument exceeds 700 are clamped by exp_neg: they must be finite, within exp(-699) A / E of the
     reference (E = the entry's exponential).
  Gradient:  |g_p - g_ref,p| <= C_K u sum_jk w (|X| + |alpha alpha^T|)_jk Dabs_p,jk (1 + U_jk)
                                + (D + n_tiles / 256) u sum_jk |w (X - alpha alpha^T)_jk dK_jk/dtheta_p|
     Dabs = desc_ref's absolute-monomial sum of dK/dtheta_p; the first term also covers the rounding of the weights
     w (X - alpha alpha^T).  D bounds the depth of the kernels' summation: per thread <= 8 row slots x 4 shift
     combinations x 3 dimensions (additive form) x 4 entries = 384 accumulations, then 5 warp-shuffle levels, the 8 warp
     sums, <= 8 runs, and in k_reduce_partials n_tiles / 256 strided adds plus an 8-level tree: D = 420.

The layouts are checked bit for bit against one another (every layout runs the same per-entry arithmetic), and every
entry a call must not write keeps its NaN: above the diagonal (LOWER, owned), rows of other ranks (owned), the ld
padding and a guard row above and below the matrix.  Every case prints its largest err / bar for K and the gradient.
"""
import ctypes as C

import numpy as np
import pytest

from oracle import desc_ref
from stopro_b200 import _lib, operators

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
C_K = 64.0
D_SUM = 420.0
LD = np.longdouble
TINY = np.longdouble("1e-4000")  # bar floor: an entry whose bar is 0 must be exact
SWITCH_TILES = 2 * 148  # build_lower_tiles_owned: 16-row tiles when 64-row tiles would leave fewer than two per SM


# ------------------------------------------------------------------------------------------------ plans and references
def owned_tiles(sec, rank, world):
    """Python restatement of build_lower_tiles_owned: [(row0, col0, nrows, ncols)]."""
    nb = len(sec) - 1

    def capped(cap):
        out = []
        for i in range(nb):
            for j in range(i + 1):
                r, r1, c0, c1 = int(sec[i]), int(sec[i + 1]), int(sec[j]), int(sec[j + 1])
                while r < r1:
                    nr = min(cap, r1 - r, 128 - r % 128)
                    if (r // 128) % world == rank:
                        for c in range(c0, c1, 128):
                            if not (i == j and r + nr - 1 < c):
                                out.append((r, c, nr, min(128, c1 - c)))
                    r += nr
        return out

    t = capped(64)
    return t if len(t) >= SWITCH_TILES else capped(16)


class Case:
    def __init__(self, name, dim, product, kernel, n_groups, sizes, pts, table, theta, lbox=None, noise_blocks=None,
                 eps=1e-4, exact_arg=False, col_sizes=None, col_pts=None):
        self.name, self.dim, self.product, self.kernel, self.n_groups = name, dim, product, kernel, n_groups
        self.sec = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self.pts = np.ascontiguousarray(pts, dtype=np.float64).reshape(-1, dim)
        self.symmetric = col_sizes is None
        self.sec_col = self.sec if self.symmetric else np.concatenate([[0], np.cumsum(col_sizes)]).astype(np.int64)
        self.pts_col = self.pts if self.symmetric else np.ascontiguousarray(col_pts, dtype=np.float64).reshape(-1, dim)
        self.table, self.lbox, self.noise_blocks = table, lbox, noise_blocks
        self.theta, self.eps, self.exact_arg = np.asarray(theta, dtype=np.float64), eps, exact_arg
        self.rows, self.cols = int(self.sec[-1]), int(self.sec_col[-1])
        self.ref = desc_ref.PlanRef(dim, product, kernel, n_groups, self.sec, self.pts, table,
                                    None if self.symmetric else self.sec_col, None if self.symmetric else self.pts_col,
                                    lbox, noise_blocks)
        d = _lib.PlanDesc()
        d.dim, d.product_form, d.n_groups, d.symmetric = dim, int(product), n_groups, int(self.symmetric)
        d.n_row_blocks, d.n_col_blocks = len(self.sec) - 1, len(self.sec_col) - 1
        d.kernel_type = _lib.KERNEL_TYPES[kernel]
        d.sec_row = self.sec.ctypes.data_as(C.POINTER(C.c_int64))
        d.sec_col = self.sec_col.ctypes.data_as(C.POINTER(C.c_int64))
        d.pts_row_host = self.pts.ctypes.data_as(C.POINTER(C.c_double))
        d.pts_col_host = self.pts_col.ctypes.data_as(C.POINTER(C.c_double))
        d.table = table
        lb = np.zeros(3) if lbox is None else np.concatenate([np.asarray(lbox, dtype=np.float64), np.zeros(3)])[:3]
        for k in range(3):
            d.lbox[k] = float(lb[k])
        d.noise_lo_block, d.noise_hi_block = noise_blocks if noise_blocks else (-1, -1)
        h = C.c_void_p()
        _lib.check(_lib.lib().pigp_plan_create(C.byref(d), C.byref(h)))
        self.handle = h
        assert _lib.lib().pigp_plan_theta_len(h) == len(self.theta) == self.ref.theta_len

    def close(self):
        _lib.lib().pigp_plan_destroy(self.handle)


def obs_table(dim, product, names, obs, fields, zero=()):
    """Symmetric block table of operators.make_desc over the observables `names` ((i, j) in zero: Kzero)."""
    nb = len(names)
    table = (_lib.BlockDesc * (nb * nb))()
    for i in range(nb):
        for j in range(i, nb):
            if (i, j) not in zero:
                table[i * nb + j] = operators.make_desc(obs[names[i]], obs[names[j]], fields, dim, product)
    return table


def random_desc(rng, dim, product, n_groups, shift=(0, 0), eight_runs=False):
    """Seeded random descriptor: 1-8 signed terms sorted by group, total order <= 4, one nearly cancelling pair."""
    d = _lib.BlockDesc()
    terms = []
    if eight_runs:  # dim 3 product: 8 distinct (group, parity pattern) runs
        pats = [(1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (2, 1, 1), (0, 2, 0), (1, 1, 1), (0, 0, 2)]
        for k in range(8):
            terms.append([k // 2, list(pats[k]), rng.uniform(-2, 2)])
    else:
        for _ in range(int(rng.integers(1, 8))):
            g = int(rng.integers(0, n_groups))
            if product:
                order = [0] * dim
                for _ in range(int(rng.integers(0, 5))):
                    order[int(rng.integers(0, dim))] += 1
            else:
                order = [-1] * dim
                order[int(rng.integers(0, dim))] = int(rng.integers(0, 5))
            terms.append([g, order, rng.uniform(-2, 2)])
        g, order, c = terms[0]
        terms.append([g, list(order), -c * (1.0 - 1e-7)])  # nearly cancels terms[0]
    terms.sort(key=lambda t: t[0])
    d.n_terms = len(terms)
    d.shift_first, d.shift_second = shift
    for k, (g, order, c) in enumerate(terms):
        d.terms[k].group, d.terms[k].coef = g, c
        for i in range(3):
            d.terms[k].order[i] = order[i] if i < dim else -1
    return d


def random_table(rng, dim, product, n_groups, nb, zero=(), eight_runs_at=None):
    table = (_lib.BlockDesc * (nb * nb))()
    for i in range(nb):
        for j in range(i, nb):
            if (i, j) in zero:
                continue
            shift = (int(rng.integers(0, 2)), int(rng.integers(0, 2)))
            table[i * nb + j] = random_desc(rng, dim, product, n_groups, shift, eight_runs=(i, j) == eight_runs_at)
    return table


def random_theta(rng, n_groups, dim, noise):
    th = []
    for _ in range(n_groups):
        th += [rng.uniform(-1, 1)] + list(rng.uniform(-3, 3, dim))  # length scales e^-3 .. e^3
    if noise:
        th.append(rng.uniform(-6, -2))
    return np.array(th)


def points(rng, sizes, dim, scale=1.0):
    """Random points with coincident pairs inside a block and across blocks."""
    pts = scale * rng.random((int(sum(sizes)), dim))
    sec = np.concatenate([[0], np.cumsum(sizes)])
    for b in range(len(sizes)):
        n = sizes[b]
        if n >= 4:
            pts[sec[b] + n - 1] = pts[sec[b]]                 # inside the block
        if b > 0 and n >= 2:
            pts[sec[b] + 1] = pts[sec[b - 1]]                 # across blocks
    return pts


def _stokes(dim, product, kernel, names, sizes, seed, noise=True, lbox=None, zero=()):
    rng = np.random.default_rng(seed)
    obs, fields = operators.stokes_observables(dim) if dim > 1 else operators.scalar_observables(1)
    table = obs_table(dim, product, names, obs, fields, zero)
    nb = (1, 2) if noise else None
    return dict(dim=dim, product=product, kernel=kernel, n_groups=len(fields), sizes=sizes,
                pts=points(rng, sizes, dim), table=table, theta=random_theta(rng, len(fields), dim, noise),
                lbox=lbox, noise_blocks=nb)


def _random(dim, product, kernel, sizes, seed, zero=((0, 2),), eight_runs_at=None):
    rng = np.random.default_rng(seed)
    nb = len(sizes)
    table = random_table(rng, dim, product, 4, nb, zero, eight_runs_at)
    return dict(dim=dim, product=product, kernel=kernel, n_groups=4, sizes=sizes, pts=points(rng, sizes, dim),
                table=table, theta=random_theta(rng, 4, dim, True), lbox=np.array([0.75, -1.25, 0.5])[:dim],
                noise_blocks=(1, nb - 2))


def _far():
    """theta = 0 (a = gamma = 1) and dyadic points: every exponent argument is formed exactly; pairs with arguments
    in [690, 700] and beyond 700 (the exp_neg clamp)."""
    rng = np.random.default_rng(11)
    sizes = [65, 64, 1]
    n = sum(sizes)
    x = np.where(rng.random(n) < 0.5, rng.integers(0, 64, n) / 64.0, 37.0 + rng.integers(0, 96, n) / 64.0)
    y = rng.integers(0, 16, n) / 64.0
    pts = np.stack([x, y], 1)
    obs, fields = operators.stokes_observables(2)
    table = obs_table(2, True, ["ux", "fx", "p"], obs, fields)
    return dict(dim=2, product=True, kernel="se", n_groups=3, sizes=sizes, pts=pts, table=table, theta=np.zeros(9),
                noise_blocks=None, exact_arg=True)


def _large(n_target, seed):
    names = ["ux", "p", "fx", "div"]
    base = np.array([0.3, 0.2, 0.3, 0.2])
    sizes = [int(v) for v in np.round(base * n_target)]
    sizes[0] += 1  # odd block offsets
    return _stokes(2, True, "se", names, sizes, seed, noise=True)


def _large_sizes():
    """Totals just below and just above the 16 / 64-row switch of build_lower_tiles_owned at world = 1."""
    names_frac = np.array([0.3, 0.2, 0.3, 0.2])

    def n64(n):  # number of 64-row tiles
        sizes = [int(v) for v in np.round(names_frac * n)]
        sizes[0] += 1
        sec = np.concatenate([[0], np.cumsum(sizes)])
        tiles = 0
        for i in range(len(sizes)):
            for j in range(i + 1):
                r, r1, c0, c1 = sec[i], sec[i + 1], sec[j], sec[j + 1]
                while r < r1:
                    nr = min(64, r1 - r, 128 - r % 128)
                    tiles += sum(1 for c in range(c0, c1, 128) if not (i == j and r + nr - 1 < c))
                    r += nr
        return tiles

    n = 1000
    while n64(n) < SWITCH_TILES:
        n += 16
    assert n64(n - 48) < SWITCH_TILES <= n64(n)
    return n - 48, n


STOKES2 = ["ux", "uy", "p", "fx", "fy", "div", "difux", "difp"]
SIZES2 = [65, 1, 129, 63, 127, 64, 1, 128]
CASES = {
    "stokes2d_se_product": lambda: _stokes(2, True, "se", STOKES2, SIZES2, 1, lbox=np.array([2.5, 0.75]), zero=((0, 1),)),
    "stokes2d_se_additive": lambda: _stokes(2, False, "se", STOKES2, SIZES2, 2, lbox=np.array([2.5, 0.75])),
    "stokes3d_se": lambda: _stokes(3, True, "se", ["ux", "uy", "uz", "p", "fx", "fy", "fz", "div"],
                                   [64, 1, 63, 65, 64, 1, 63, 65], 3),
    "laplacian1d_se": lambda: dict(_stokes(1, True, "se", ["y", "ly"], [129, 63], 4, noise=False)),
    "random_1d_se": lambda: _random(1, True, "se", [63, 1, 64, 65], 5),
    "random_2d_se_product": lambda: _random(2, True, "se", [65, 1, 127, 64, 63], 6),
    "random_3d_se_product_8runs": lambda: _random(3, True, "se", [64, 129, 1, 63], 7, eight_runs_at=(1, 1)),
    "random_3d_se_additive": lambda: _random(3, False, "se", [127, 1, 65, 64], 8),
    "random_2d_se_additive": lambda: _random(2, False, "se", [1, 64, 129, 63], 9),
    "stokes2d_mt52_product": lambda: _stokes(2, True, "mt52", STOKES2, [33, 1, 65, 31, 63, 64, 1, 64], 10,
                                             lbox=np.array([2.5, 0.75])),
    "stokes2d_mt72_additive": lambda: _stokes(2, False, "mt72", STOKES2, [33, 1, 65, 31, 63, 64, 1, 64], 12,
                                              lbox=np.array([2.5, 0.75])),
    "random_3d_mt92_product": lambda: _random(3, True, "mt92", [63, 1, 64, 65], 13),
    "random_2d_mt52_additive": lambda: _random(2, False, "mt52", [65, 1, 63, 64], 14),
    "far_dyadic_se": _far,
    "large_below_switch": lambda: _large(_large_sizes()[0], 15),
    "large_above_switch": lambda: _large(_large_sizes()[1], 16),
}


def lower_entries(n):
    R, Cc = np.tril_indices(n)
    return R.astype(np.int64), Cc.astype(np.int64)


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    """The plan, its reference over every lower entry (value, A, U) and the reference trace sums for the X kinds."""
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = Case(request.param, **CASES[request.param]())
    rng = np.random.default_rng(100)
    n = c.rows
    Xs = {"random": (rng.standard_normal((n, n)), rng.standard_normal(n))}
    Xs["random"] = ((Xs["random"][0] + Xs["random"][0].T) / 2, Xs["random"][1])
    Xs["zero_alpha"] = (np.zeros((n, n)), rng.standard_normal(n))
    P = c.ref.theta_len
    R, Cc = lower_entries(n)
    val, A = np.zeros(len(R), LD), np.zeros(len(R), LD)  # A in longdouble: entries beyond exp(-708) stay normal
    Uarg = np.zeros(len(R))
    sums = {k: dict(g=np.zeros(P, LD), m1=np.zeros(P), m2=np.zeros(P)) for k in Xs}
    step = 1 << 18
    for s0 in range(0, len(R), step):
        sl = slice(s0, s0 + step)
        v, g, a, u, dabs = c.ref.entries(R[sl], Cc[sl], c.theta)
        val[sl], A[sl], Uarg[sl] = v, a, u.astype(np.float64)
        w = np.where(R[sl] == Cc[sl], 1.0, 2.0)
        for k, (X, al) in Xs.items():
            x = X[R[sl], Cc[sl]]
            aa = al[R[sl]] * al[Cc[sl]]
            W = w * (x.astype(LD) - al[R[sl]].astype(LD) * al[Cc[sl]].astype(LD))
            sums[k]["g"] += (W * g).sum(axis=1) / 2
            sums[k]["m1"] += ((w * (np.abs(x) + np.abs(aa)) * (1 + u.astype(np.float64))) * dabs.astype(np.float64)).sum(axis=1)
            sums[k]["m2"] += np.abs((W * g).astype(np.float64)).sum(axis=1)
    c.lower = (R, Cc)
    c.val, c.A, c.U, c.Xs, c.sums = val, A, Uarg, Xs, sums
    c.n_tiles = len(owned_tiles(c.sec, 0, 1))
    c.dev = torch.device("cuda:0")
    c.theta_dev = torch.as_tensor(c.theta, device=c.dev)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ device buffers
def guarded(rows, ld, off, dev):
    """NaN buffer with one guard row above and below the rows x ld matrix, which starts `off` doubles into it."""
    import torch

    buf = torch.full((off + (rows + 2) * ld + 2,), float("nan"), dtype=torch.float64, device=dev)
    return buf, buf.data_ptr() + 8 * (off + ld)


def unpack(buf, rows, ld, off):
    """-> (matrix rows x ld as numpy, guard rows all NaN?)."""
    b = buf.cpu().numpy()
    body = b[off + ld:off + ld + rows * ld].reshape(rows, ld)
    guards = np.concatenate([b[:off + ld], b[off + ld + rows * ld:]])
    return body, bool(np.isnan(guards).all())


def assemble(c, how, ld, off, add_diag=False, rank=0, world=1):
    import torch

    buf, ptr = guarded(c.rows, ld, off, c.dev)
    L = _lib.lib()
    if how == "full":
        _lib.check(L.pigp_assemble(c.handle, c.theta_dev.data_ptr(), c.eps, int(add_diag), ptr, ld, _lib.LAYOUT_FULL, None))
    elif how == "lower":
        _lib.check(L.pigp_assemble(c.handle, c.theta_dev.data_ptr(), c.eps, int(add_diag), ptr, ld, _lib.LAYOUT_LOWER, None))
    else:
        _lib.check(L.pigp_assemble_owned(c.handle, rank, world, c.theta_dev.data_ptr(), c.eps, int(add_diag), ptr, ld, None))
    torch.cuda.synchronize()
    body, guards_ok = unpack(buf, c.rows, ld, off)
    assert guards_ok, f"{how}: a guard row was written"
    assert np.isnan(body[:, c.cols:]).all(), f"{how}: the ld padding was written"
    return body[:, :c.cols]


def diag_addon(c):
    add = np.full(c.rows, c.eps, dtype=LD)
    if c.ref.noise is not None:
        lo, hi = c.ref.noise
        add[:lo] = 1
        add[lo:hi] = np.exp(LD(c.theta[-1]))
    return add


def bitwise_equal(a, b):
    return np.array_equal(a.view(np.int64), b.view(np.int64))


# ------------------------------------------------------------------------------------------------ tests
def check_entries(c, got, val, A, Uarg, what):
    """Entry bar; returns the largest err / bar."""
    assert np.isfinite(got).all(), f"{what}: non-finite entries"
    err = np.abs(got.astype(LD) - val)
    bar = C_K * U * A * (1 if c.exact_arg else 1.0 + Uarg.astype(LD))
    far = Uarg > 700.0  # clamped by exp_neg: within exp(-699) A / E, E = exp(-Uarg)
    bar = np.where(far, A * np.exp(Uarg.astype(LD) - 699) + bar, bar)
    ratio = (err / np.maximum(bar, TINY)).astype(np.float64)
    worst = int(np.argmax(ratio))
    assert ratio[worst] <= 1.0, (f"{what}: entry {worst} err {float(err[worst]):.3e} bar {float(bar[worst]):.3e} "
                                 f"val {float(val[worst]):.6e} A {float(A[worst]):.3e} U {Uarg[worst]:.1f}")
    return float(ratio[worst])


def test_assembly_entrywise_and_layouts(case):
    c = case
    n = c.rows
    R, Cc = c.lower
    full = assemble(c, "full", c.cols, 0)
    worst = check_entries(c, full[R, Cc], c.val, c.A, c.U, "FULL")
    assert bitwise_equal(full, np.ascontiguousarray(full.T)), "FULL is not exactly symmetric"
    for ld, off in ((c.cols + 1, 0), (c.cols + 64, 1), (c.cols, 1)):
        assert bitwise_equal(assemble(c, "full", ld, off), full), f"FULL ld={ld} off={off}"
    upper = np.triu(np.ones((n, n), bool), 1)
    for ld, off in ((c.cols, 0), (c.cols + 1, 1), (c.cols + 64, 0)):
        low = assemble(c, "lower", ld, off)
        assert np.isnan(low[upper]).all(), "LOWER wrote above the diagonal"
        assert bitwise_equal(low[R, Cc], full[R, Cc]), f"LOWER ld={ld} off={off}"
    for world in (1, 2, 3):
        union = np.full((n, n), np.nan)
        for rank in range(world):
            ld, off = ((c.cols + 64, 0), (c.cols, 1), (c.cols + 1, 0))[rank]
            part = assemble(c, "owned", ld, off, rank=rank, world=world)
            mine = ((np.arange(n) // 128) % world == rank)[:, None] & ~upper
            assert np.isnan(part[~mine]).all(), f"owned rank {rank}/{world} wrote outside its lower rows"
            assert not np.isnan(part[mine]).any(), f"owned rank {rank}/{world} left an owned entry unwritten"
            union[mine] = part[mine]
        assert bitwise_equal(union[R, Cc], full[R, Cc]), f"owned union world={world}"
    # add_diag: off-diagonal entries unchanged bit for bit, the diagonal gains the jitter / noise add-on
    fd = assemble(c, "full", c.cols + 1, 1, add_diag=True)
    off_diag = ~np.eye(n, dtype=bool)
    assert bitwise_equal(fd[off_diag], full[off_diag])
    di = np.arange(n)
    dmask = R == Cc
    add = diag_addon(c)
    worst = max(worst, check_entries(c, fd[di, di], c.val[dmask] + add, c.A[dmask] + np.abs(add), c.U[dmask],
                                     "FULL + add_diag"))
    od = assemble(c, "owned", c.cols, 0, add_diag=True, rank=1, world=2)
    mine = (di // 128) % 2 == 1
    assert bitwise_equal(od[di[mine], di[mine]], fd[di[mine], di[mine]])
    # pigp_assemble_diag == diag(FULL) bit for bit
    import torch

    for add_d in (0, 1):
        buf = torch.full((n + 2,), float("nan"), dtype=torch.float64, device=c.dev)
        _lib.check(_lib.lib().pigp_assemble_diag(c.handle, c.theta_dev.data_ptr(), c.eps, add_d, buf.data_ptr() + 8, None))
        b = buf.cpu().numpy()
        assert np.isnan(b[0]) and np.isnan(b[-1]), "DIAG wrote outside its vector"
        assert bitwise_equal(b[1:-1], (fd if add_d else full)[di, di]), "DIAG differs from diag(FULL)"
    print(f"\n[{c.name}] N={n} tiles={c.n_tiles} K max err/bar {worst:.3e}")


def trace_grad(c, X, alpha, rank=0, world=1, ld=None, off=0):
    import torch

    n = c.rows
    ld = c.cols if ld is None else ld
    buf = torch.full((off + n * ld,), float("nan"), dtype=torch.float64, device=c.dev)
    Xt = torch.as_tensor(X, device=c.dev)
    buf[off:].view(n, ld)[:, :n] = Xt
    al = torch.as_tensor(alpha, device=c.dev)
    g = torch.full((c.ref.theta_len,), float("nan"), dtype=torch.float64, device=c.dev)
    _lib.check(_lib.lib().pigp_trace_grad(c.handle, rank, world, c.theta_dev.data_ptr(), buf.data_ptr() + 8 * off, ld,
                                          al.data_ptr(), g.data_ptr(), None))
    torch.cuda.synchronize()
    return g.cpu().numpy()


def test_trace_gradient(case):
    c = case
    if not c.symmetric:
        pytest.skip("gradient of a symmetric plan only")
    worst = 0.0
    for kind, (X, alpha) in c.Xs.items():
        s = c.sums[kind]
        bar = C_K * U * s["m1"] + (D_SUM + c.n_tiles / 256.0) * U * s["m2"]
        g1 = trace_grad(c, X, alpha)
        err = np.abs(g1.astype(LD) - s["g"]).astype(np.float64)
        ratio = err / np.maximum(bar, 1e-300)
        assert (ratio <= 1.0).all(), (kind, err, bar)
        worst = max(worst, float(ratio.max()))
        # odd ld and an X one double off 16-byte alignment: the scalar weight loads give the same sums bit for bit
        assert bitwise_equal(trace_grad(c, X, alpha, ld=c.cols + 1, off=1), g1), kind
        assert bitwise_equal(trace_grad(c, X, alpha, ld=c.cols + 64, off=0), g1), kind
        for world in (2, 3):
            tot = sum(trace_grad(c, X, alpha, rank=r, world=world) for r in range(world))
            assert (np.abs(tot - g1) <= 2 * bar).all(), (kind, world, tot - g1, bar)
    # one-hot probes X = e_j e_k^T + e_k e_j^T, alpha = 0: grad = dK_jk/dtheta (j != k) or dK_jj/dtheta (j == k)
    n = c.rows
    picks = {0, n - 1, 63, 64, 127, 128, 129}
    picks |= {int(v) for v in c.sec[1:-1]} | {int(v) - 1 for v in c.sec[1:-1]}
    picks = sorted(p for p in picks if 0 <= p < n)
    probes = [(j, j) for j in picks[:6]] + [(j, k) for j in picks for k in picks if k < j][:14]
    zero = np.zeros(n)
    for j, k in probes:
        X = np.zeros((n, n))
        X[j, k] += 1.0
        X[k, j] += 1.0
        g = trace_grad(c, X, zero)
        _, gr, _, u, dabs = c.ref.entries(np.array([j]), np.array([k]), c.theta)
        want = gr[:, 0]
        bar = (C_K * U * (1 + u[0]) + (D_SUM + c.n_tiles / 256.0) * U) * dabs[:, 0]
        if u[0] > 700:  # clamped by exp_neg
            bar += dabs[:, 0] * np.exp(u[0] - 699)
        err = np.abs(g.astype(LD) - want)
        assert (err <= bar).all(), ((j, k), g, want.astype(np.float64), bar.astype(np.float64))
        worst = max(worst, float((err / np.maximum(bar, TINY)).max()))
    print(f"\n[{c.name}] N={n} tiles={c.n_tiles} gradient max err/bar {worst:.3e}")


def test_mixed_plan_entrywise(cuda_device):
    """Rectangular (test x training) plan: FULL layout, odd ld, K one double off alignment."""
    import torch

    rng = np.random.default_rng(21)
    obs, fields = operators.stokes_observables(2)
    rows, cols = ["ux", "fx", "difp"], ["uy", "p", "fy", "div", "difux"]
    rs, cs = [65, 1, 63], [64, 127, 1, 65, 33]
    table = (_lib.BlockDesc * (len(rows) * len(cols)))()
    for i in range(len(rows)):
        for j in range(len(cols)):
            table[i * len(cols) + j] = operators.make_desc(obs[rows[i]], obs[cols[j]], fields, 2, True)
    pr, pc = points(rng, rs, 2), points(rng, cs, 2)
    pr[:3] = pc[:3]
    c = Case("mixed", 2, True, "se", 3, rs, pr, table, random_theta(rng, 3, 2, False), lbox=np.array([1.5, 0.5]),
             col_sizes=cs, col_pts=pc)
    c.dev = torch.device("cuda:0")
    c.theta_dev = torch.as_tensor(c.theta, device=c.dev)
    R, Cc = [a.ravel() for a in np.meshgrid(np.arange(c.rows), np.arange(c.cols), indexing="ij")]
    val, _, A, Uarg, _ = c.ref.entries(R, Cc, c.theta)
    full = assemble(c, "full", c.cols, 0)
    worst = check_entries(c, full[R, Cc], val, A, Uarg.astype(np.float64), "mixed")
    for ld, off in ((c.cols + 1, 1), (c.cols + 64, 0)):
        assert bitwise_equal(assemble(c, "full", ld, off), full)
    c.close()
    print(f"\n[mixed] {c.rows} x {c.cols} K max err/bar {worst:.3e}")


def test_owned_entry_points_reject_bad_arguments(cuda_device):
    import torch

    c = Case("args", **_stokes(1, True, "se", ["y", "ly"], [3, 2], 0, noise=False))
    th = torch.as_tensor(c.theta, device="cuda:0")
    K = torch.zeros(64, dtype=torch.float64, device="cuda:0")
    L = _lib.lib()
    for rank, world, ld in ((1, 1, 5), (-1, 2, 5), (0, 0, 5), (0, 1, 4)):
        assert L.pigp_assemble_owned(c.handle, rank, world, th.data_ptr(), 0.0, 0, K.data_ptr(), ld, None) == -1
        assert L.pigp_trace_grad(c.handle, rank, world, th.data_ptr(), K.data_ptr(), ld, K.data_ptr(), K.data_ptr(),
                                 None) == -1
    assert L.pigp_trace_grad(c.handle, 0, 1, th.data_ptr(), None, 5, K.data_ptr(), K.data_ptr(), None) == -1
    assert L.pigp_assemble_owned(c.handle, 0, 1, th.data_ptr(), 0.0, 0, None, 5, None) == -1
    torch.cuda.synchronize()
    c.close()
