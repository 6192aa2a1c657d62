"""Extended-precision evaluator of `pigp_block_desc` tables (TEST INFRASTRUCTURE, see oracle/__init__.py).

Evaluates a descriptor exactly as include/pigp.h defines it, independently of the fused CUDA evaluators
(csrc/pigp_assemble.cu, csrc/pigp_matern.cu): every monomial is formed on its own, in the requested dtype
(numpy.longdouble for the entry-wise GPU tests; float64 for the CPU checks of the descriptor compiler).

A term  coef * gamma_g * prod_d G_{n_d}(s_d)  with
    SE:      G_n = (d/ds)^n exp(-a s^2 / 2) = g_n(s, a) exp(-a s^2 / 2),  g_n = sum_i kappa_{n,i} a^((n+i)/2) s^i,
             a = exp(-2 log l)
    Matern:  G_n = (d/ds)^n q(rho) e^-rho = c^n sgn(s)^n q_n(rho) e^-rho,  rho = c |s|,  c = kappa / l,
             with sgn(0) = 0 for n >= 1 (the reference's autodiff value at coincident points, also for even n)
runs over every dimension in the product form (an absent order counts as 0) and over the one dimension it lives on in
the additive form.  The periodic wrappers evaluate the block at the shifted points, r + lbox formed first, then the
difference, both in float64 as the kernels do, with the sign (-1)^(shifts not taken).  Lower blocks of a symmetric
plan are the transposes of the table's upper blocks (first argument = the column point).

For every entry, entries() also returns
    A  = sum over terms and shift combinations of |coef| gamma prod_d (sum_i |monomial_i|) * exponential:
         the condition of the entry's sum, which bounds the rounding of any evaluation that forms these monomials;
    U  = the largest exponent argument  1/2 sum_d a_d s_d^2  (SE) or  sum_d rho_d  (Matern)  over terms and shifts;
    Dabs[p] = the same absolute-monomial sum for dK/dtheta_p.
"""
from fractions import Fraction

import numpy as np

LD = np.longdouble

# g_n(s, a) = sum_i HERM[n][i] a^((n + i) / 2) s^i
HERM = {0: {0: 1}, 1: {1: -1}, 2: {2: 1, 0: -1}, 3: {3: -1, 1: 3}, 4: {4: 1, 2: -6, 0: 3}}
MATERN = {"mt52": (5, [1, 1, Fraction(1, 3)]),
          "mt72": (7, [1, 1, Fraction(2, 5), Fraction(1, 15)]),
          "mt92": (9, [1, 1, Fraction(3, 7), Fraction(2, 21), Fraction(1, 105)])}
KERNEL_NAMES = {0: "se", 52: "mt52", 72: "mt72", 92: "mt92"}


def _matern_polys(kind, n):
    """(q_n, u_n) as exact rational coefficient lists (ascending powers of rho)."""
    q = list(MATERN[kind][1]) + [0] * 6
    for _ in range(n):
        dq = [(i + 1) * q[i + 1] for i in range(len(q) - 1)] + [0]
        q = [dq[i] - q[i] for i in range(len(q))]
    dq = [(i + 1) * q[i + 1] for i in range(len(q) - 1)] + [0]
    u = [-n * q[i] + ((q[i - 1] - dq[i - 1]) if i > 0 else 0) for i in range(len(q))]
    return q, u


def _poly_abs(coefs, x, dtype):
    """(sum_i c_i x^i, sum_i |c_i x^i|) for x >= 0."""
    val = np.zeros_like(x)
    mag = np.zeros_like(x)
    for i, c in enumerate(coefs):
        if c == 0:
            continue
        m = dtype(c.numerator) / dtype(c.denominator) if isinstance(c, Fraction) else dtype(c)
        t = m * x ** i
        val = val + t
        mag = mag + np.abs(t)
    return val, mag


def _se_dim(n, s, a):
    """g_n, sum |monomials|, h = (d/dlog l of g_n E) / E = -2 sum kappa k a^k s^i + a s^2 g_n, and its magnitude."""
    g = np.zeros_like(s)
    gm = np.zeros_like(s)
    h = np.zeros_like(s)
    hm = np.zeros_like(s)
    for i, kap in HERM[n].items():
        k = (n + i) // 2
        mono = kap * a ** k * s ** i
        g = g + mono
        gm = gm + np.abs(mono)
        h = h - 2 * k * mono
        hm = hm + 2 * k * np.abs(mono)
    x = a * s * s
    return g, gm, h + x * g, hm + x * gm


def _mt_dim(kind, n, s, c, dtype):
    """Matern factor without e^-rho: f, |f| monomial sum, d/dlog l, its magnitude; and rho."""
    rho = c * np.abs(s)
    q, u = _matern_polys(kind, n)
    fq, fm = _poly_abs(q, rho, dtype)
    fu, um = _poly_abs(u, rho, dtype)
    if n > 0:
        sg = np.sign(s) ** n  # sgn(0) = 0 for every order >= 1
        pref = c ** n * sg
        fq, fu = pref * fq, pref * fu
        fm, um = np.abs(pref) * fm, np.abs(pref) * um
    return fq, fm, fu, um, rho


def eval_terms(desc, dim, s, theta, product, kernel="se", dtype=LD):
    """One descriptor at differences s (list of dim arrays, already shifted), without the shift wrappers.

    Returns (val, grad[n_groups * (1 + dim)], A, U, Dabs[n_groups * (1 + dim)]) as arrays shaped like s[0]."""
    theta = np.asarray(theta, dtype=dtype)
    n_hyp = (len(theta) // (1 + dim)) * (1 + dim)
    shape = np.shape(s[0])
    val, A, U = np.zeros(shape, dtype), np.zeros(shape, dtype), np.zeros(shape, dtype)
    grad = np.zeros((n_hyp,) + shape, dtype)
    dabs = np.zeros((n_hyp,) + shape, dtype)
    for t in range(desc.n_terms):
        term = desc.terms[t]
        g = term.group
        th = theta[g * (1 + dim):(g + 1) * (1 + dim)]
        gamma = np.exp(th[0])
        dims = list(range(dim)) if product else [d for d in range(dim) if term.order[d] >= 0]
        f, fm, df, dfm = {}, {}, {}, {}
        arg = np.zeros(shape, dtype)
        for d in dims:
            n = max(int(term.order[d]), 0)
            if kernel == "se":
                a = np.exp(dtype(-2) * th[1 + d])
                f[d], fm[d], df[d], dfm[d] = _se_dim(n, s[d], a)
                arg = arg + a * s[d] * s[d] / 2
            else:
                c = np.sqrt(dtype(MATERN[kernel][0])) * np.exp(-th[1 + d])
                f[d], fm[d], df[d], dfm[d], rho = _mt_dim(kernel, n, s[d], c, dtype)
                arg = arg + rho
        E = np.exp(-arg)
        w = dtype(term.coef) * gamma * E
        wm = np.abs(w)
        v, m = w, wm
        for d in dims:
            v, m = v * f[d], m * fm[d]
        val += v
        A += m
        U = np.maximum(U, arg)
        base = g * (1 + dim)
        grad[base] += v
        dabs[base] += m
        for e in dims:
            pe, pm = w * df[e], wm * dfm[e]
            for d in dims:
                if d != e:
                    pe, pm = pe * f[d], pm * fm[d]
            grad[base + 1 + e] += pe
            dabs[base + 1 + e] += pm
    return val, grad, A, U, dabs


def shifted_differences(first, second, lbox, sf, ss, dim):
    """s_d = (first_d [+ lbox_d]) - (second_d [+ lbox_d]), formed in float64 as the kernels form it."""
    out = []
    for d in range(dim):
        f = np.asarray(first[:, d], dtype=np.float64)
        g = np.asarray(second[:, d], dtype=np.float64)
        if sf:
            f = f + np.float64(lbox[d])
        if ss:
            g = g + np.float64(lbox[d])
        out.append(f - g)
    return out


def eval_desc_all(desc, dim, first, second, theta, lbox, product, kernel="se", dtype=LD):
    """A descriptor with its shift wrappers at point pairs (first[j], second[j]) (float64 arrays (n, dim))."""
    lb = np.zeros(3) if lbox is None else np.concatenate([np.asarray(lbox, dtype=np.float64).ravel(), np.zeros(3)])[:3]
    n = len(first)
    n_hyp = (len(theta) // (1 + dim)) * (1 + dim)
    val, A, U = np.zeros(n, dtype), np.zeros(n, dtype), np.zeros(n, dtype)
    grad, dabs = np.zeros((n_hyp, n), dtype), np.zeros((n_hyp, n), dtype)
    sfm, ssm = int(desc.shift_first), int(desc.shift_second)
    for sf in range(sfm + 1):
        for ss in range(ssm + 1):
            sign = -1 if (sfm - sf + ssm - ss) % 2 else 1
            s = [x.astype(dtype) for x in shifted_differences(first, second, lb, sf, ss, dim)]
            v, g, a, u, dm = eval_terms(desc, dim, s, theta, product, kernel, dtype)
            val += sign * v
            grad += sign * g
            A += a
            dabs += dm
            U = np.maximum(U, u)
    return val, grad, A, U, dabs


def eval_desc(desc, dim, r, rp, theta, lbox=None, product=True, kernel="se", dtype=np.float64):
    """Dense block of one descriptor on points r (n, dim) x rp (m, dim): the value only."""
    r = np.asarray(r, dtype=np.float64).reshape(len(r), dim)
    rp = np.asarray(rp, dtype=np.float64).reshape(len(rp), dim)
    n, m = len(r), len(rp)
    first = np.repeat(r, m, axis=0)
    second = np.tile(rp, (n, 1))
    val = eval_desc_all(desc, dim, first, second, np.asarray(theta), lbox, product, kernel, dtype)[0]
    return val.reshape(n, m)


class PlanRef:
    """Entry-wise reference of a plan (pigp_plan_desc): block table, points, shifts, jitter and noise range."""

    def __init__(self, dim, product, kernel, n_groups, sec_row, pts_row, table, sec_col=None, pts_col=None, lbox=None,
                 noise_blocks=None):
        self.dim, self.product, self.kernel, self.n_groups = dim, bool(product), kernel, n_groups
        self.symmetric = sec_col is None
        self.sec_row = np.asarray(sec_row, dtype=np.int64)
        self.sec_col = self.sec_row if self.symmetric else np.asarray(sec_col, dtype=np.int64)
        self.pts_row = np.asarray(pts_row, dtype=np.float64).reshape(-1, dim)
        self.pts_col = self.pts_row if self.symmetric else np.asarray(pts_col, dtype=np.float64).reshape(-1, dim)
        self.table = table  # flat, n_row_blocks x n_col_blocks
        self.ncb = len(self.sec_col) - 1
        self.lbox = lbox
        self.noise = None
        if noise_blocks is not None:
            self.noise = (int(self.sec_row[noise_blocks[0]]), int(self.sec_row[noise_blocks[1] + 1]))
        self.theta_len = n_groups * (1 + dim) + (self.noise is not None)

    def entries(self, R, C, theta, eps=0.0, add_diag=False, dtype=LD):
        """(val, grad[theta_len], A, U, Dabs[theta_len]) at global entries (R[j], C[j])."""
        R, C = np.asarray(R, dtype=np.int64), np.asarray(C, dtype=np.int64)
        theta = np.asarray(theta, dtype=np.float64)
        n, P = len(R), self.theta_len
        val, A, U = np.zeros(n, dtype), np.zeros(n, dtype), np.zeros(n, dtype)
        grad, dabs = np.zeros((P, n), dtype), np.zeros((P, n), dtype)
        bi = np.searchsorted(self.sec_row, R, side="right") - 1
        bj = np.searchsorted(self.sec_col, C, side="right") - 1
        th = theta[:self.n_groups * (1 + self.dim)].astype(dtype)
        nh = len(th)
        key = bi * self.ncb + bj
        for k in np.unique(key):
            sel = np.nonzero(key == k)[0]
            i, j = divmod(int(k), self.ncb)
            if self.symmetric and i > j:  # lower block = transpose of table[j][i]: first argument = the column point
                desc, first, second = self.table[j * self.ncb + i], self.pts_col[C[sel]], self.pts_row[R[sel]]
            else:
                desc, first, second = self.table[i * self.ncb + j], self.pts_row[R[sel]], self.pts_col[C[sel]]
            if desc.n_terms == 0:
                continue
            v, g, a, u, dm = eval_desc_all(desc, self.dim, first, second, th, self.lbox, self.product, self.kernel, dtype)
            val[sel], A[sel], U[sel] = v, a, u
            grad[:nh, sel], dabs[:nh, sel] = g, dm
        if self.symmetric:
            diag = R == C
            if add_diag:
                add = np.full(n, dtype(eps), dtype=dtype)
                if self.noise is not None:
                    lo, hi = self.noise
                    add[R < lo] = 1
                    add[(R >= lo) & (R < hi)] = np.exp(dtype(theta[-1]))
                val[diag] += add[diag]
                A[diag] += np.abs(add[diag])
            if self.noise is not None:  # dK/dnoise = exp(noise) on the diagonal of the noise range
                lo, hi = self.noise
                on = diag & (R >= lo) & (R < hi)
                grad[P - 1, on] = np.exp(dtype(theta[-1]))
                dabs[P - 1, on] = np.exp(dtype(theta[-1]))
        return val, grad, A, U, dabs
