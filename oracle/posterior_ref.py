"""Extended-precision posterior of a block-structured GP (TEST INFRASTRUCTURE, see oracle/__init__.py).

The reference behind tests/test_gpu_posterior.py.  It builds the same descriptor tables the plans of
stopro_b200.plan.Plan build (operators.make_desc per block, Kzero test blocks, shift wrappers, jitter and noise range),
evaluates every entry with oracle.desc_ref in numpy.longdouble and factors K_bb with oracle.extended:

    mu  = K_ab alpha,          alpha = K_bb^-1 y
    cov = K_aa - V V^T,        V = K_ab L^-T,   L L^T = K_bb
    var = diag(K_aa) - rowsum(V * V)

Posterior rows are independent, so one Posterior holds the truth for a pool of test points per block; a test set that
takes the first m_b points of every pool block is an index into it (Posterior.rows).  Covariance entries are formed on
request for any (i, j), so a large test set is checked on sampled pairs plus the whole diagonal instead of M^2 N
longdouble products.

Besides the values it keeps what the error bars of the GPU test need, in float64 (they are bounds, not truth):
|L| |L|^T, A_bb / A_ab / A_aa (desc_ref's absolute-monomial sums times (1 + U)), alpha, z = L^-1 y, V and
W = K_ab K_bb^-1.  The longdouble work is O(N^3 + M_pool N^2) in numpy loops (no LAPACK for longdouble): keep
N <= ~1024.
"""
import numpy as np

from stopro_b200 import _lib, operators

from . import desc_ref, extended

LD = np.longdouble


def block_table(obs, fields, dim, product, row_names, col_names=None, zero=()):
    """The descriptor table of Plan(...): symmetric (upper blocks only, Kzero at `zero`) when col_names is None."""
    sym = col_names is None
    cols = row_names if sym else col_names
    nr, nc = len(row_names), len(cols)
    table = (_lib.BlockDesc * (nr * nc))()
    for i in range(nr):
        for j in range(nc):
            if (sym and j < i) or (i, j) in zero:
                continue
            table[i * nc + j] = operators.make_desc(obs[row_names[i]], obs[cols[j]], fields, dim, product)
    return table


def _flat(pts, dim):
    arrs = [np.asarray(p, dtype=np.float64).reshape(-1, dim) for p in pts]
    sec = np.concatenate([[0], np.cumsum([len(a) for a in arrs])]).astype(np.int64)
    return np.concatenate(arrs, axis=0), sec


class Posterior:
    """Truth of the posterior of (training set, theta, y, eps) at a pool of test points per test block.

    obs / fields: operators.stokes_observables(dim) or scalar_observables(dim); train_names / test_names: observable
    names per block; theta: the training plan's hyper-parameters (with the noise entry last when noise_blocks is set:
    the mixed and test plans read only the kernel entries before it)."""

    def __init__(self, dim, product, kernel, obs, fields, train_names, r_train, test_names, r_test, theta, y, eps,
                 lbox=None, noise_blocks=None, test_zero=()):
        self.dim, self.theta, self.eps = dim, np.asarray(theta, dtype=np.float64), float(eps)
        ng = len(fields)
        self.pts_tr, self.sec_tr = _flat(r_train, dim)
        self.pts_te, self.sec_te = _flat(r_test, dim)
        nb = (noise_blocks[0], noise_blocks[-1]) if noise_blocks else None
        self.train = desc_ref.PlanRef(dim, product, kernel, ng, self.sec_tr, self.pts_tr,
                                      block_table(obs, fields, dim, product, train_names), lbox=lbox, noise_blocks=nb)
        self.mixed = desc_ref.PlanRef(dim, product, kernel, ng, self.sec_te, self.pts_te,
                                      block_table(obs, fields, dim, product, test_names, train_names),
                                      sec_col=self.sec_tr, pts_col=self.pts_tr, lbox=lbox)
        self.test = desc_ref.PlanRef(dim, product, kernel, ng, self.sec_te, self.pts_te,
                                     block_table(obs, fields, dim, product, test_names, zero=test_zero), lbox=lbox)
        assert self.train.theta_len == len(self.theta)
        N, M = len(self.pts_tr), len(self.pts_te)
        self.N, self.M = N, M
        # K_bb with jitter / noise, lower entries mirrored
        R, C = np.tril_indices(N)
        v, _, a, u, _ = self.train.entries(R, C, self.theta, eps, add_diag=True)
        K = np.zeros((N, N), dtype=LD)
        K[R, C] = v
        K[C, R] = v
        Abb = np.zeros((N, N))
        Abb[R, C] = (a * (1 + u)).astype(np.float64)
        Abb[C, R] = Abb[R, C]
        self.K, self.A_bb = K, Abb
        L = extended.cholesky_lower(K)
        Li = extended.tri_inv_lower(L)
        yl = np.asarray(y, dtype=LD)
        self.z = Li @ yl                       # L^-1 y
        self.alpha = Li.T @ self.z             # K^-1 y
        self.L = L
        L64 = np.abs(L.astype(np.float64))
        self.LLt = L64 @ L64.T                 # |L| |L|^T: the Cholesky backward-error pattern
        # K_ab and its magnitudes
        R, C = [x.ravel() for x in np.meshgrid(np.arange(M), np.arange(N), indexing="ij")]
        v, _, a, u, _ = self.mixed.entries(R, C, self.theta)
        self.Kab = v.reshape(M, N)
        self.A_ab = (a * (1 + u)).astype(np.float64).reshape(M, N)
        self.V = self.Kab @ Li.T               # K_ab L^-T (longdouble)
        self.W = self.V.astype(np.float64) @ Li.astype(np.float64)  # K_ab K^-1 (float64: bars only)
        self.mu = self.Kab @ self.alpha
        d = np.arange(M)
        kd, _, a, u, _ = self.test.entries(d, d, self.theta)
        self.kdiag, self.A_aa_diag = kd, (a * (1 + u)).astype(np.float64)
        self.var = kd - np.sum(self.V * self.V, axis=1)

    @classmethod
    def for_model(cls, gp, r_train, r_test, theta, y, eps):
        """The posterior of a stopro_b200 GPmodel's plans (its observables, lbox, noise range and Kzero test blocks)."""
        return cls(gp.dim, gp.product_form, gp.kernel_type, gp._obs, gp._fields, gp.train_observables[:len(r_train)],
                   r_train, gp.test_observables[:len(r_test)], r_test, theta, y, eps, lbox=gp.lbox,
                   noise_blocks=gp.index_optimize_noise or None, test_zero=gp.test_zero_blocks)

    def rows(self, counts):
        """Pool rows of the test set made of the first counts[b] points of every test block."""
        return np.concatenate([np.arange(self.sec_te[b], self.sec_te[b] + c) for b, c in enumerate(counts)]).astype(np.int64)

    def cov(self, I, J):
        """Covariance entries (I[k], J[k]) (pool indices) -> (value, A_aa of the entry)."""
        I, J = np.asarray(I, dtype=np.int64), np.asarray(J, dtype=np.int64)
        k, _, a, u, _ = self.test.entries(I, J, self.theta)
        out = np.empty(len(I), dtype=LD)
        step = 4096
        for s in range(0, len(I), step):
            sl = slice(s, s + step)
            out[sl] = k[sl] - np.einsum("ij,ij->i", self.V[I[sl]], self.V[J[sl]])
        return out, (a * (1 + u)).astype(np.float64)

    def cov_full(self, rows):
        """Dense covariance over pool rows `rows` -> (value, A_aa) as (m, m) arrays."""
        rows = np.asarray(rows, dtype=np.int64)
        m = len(rows)
        I, J = [x.ravel() for x in np.meshgrid(rows, rows, indexing="ij")]
        k, _, a, u, _ = self.test.entries(I, J, self.theta)
        Vr = self.V[rows]
        return k.reshape(m, m) - Vr @ Vr.T, (a * (1 + u)).astype(np.float64).reshape(m, m)
