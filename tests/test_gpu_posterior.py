"""Entry-wise GPU tests of the posterior (pigp_predict, pigp_predict_host, pigp_predict_batch_host) against
oracle.posterior_ref, an extended-precision (numpy.longdouble) posterior of the same descriptor tables.

What runs, in csrc/pigp_capi.cu and csrc/pigp_dense.cu: the NLL-only factorisation (L and z = L^-1 y), the mixed
assembly, launch_pad, V = K_ab L^-T by trsm_rec (leaf: k_trsm_blk over mpad rows in 8-, 16- or 32-row slabs, chosen
by mpad <= 1184 / <= 2368 / above; the split n1 = nt / 2 is uneven for odd tile counts), mu = V z by k_gemv, and
either var = diag(K_aa) - rowsum(V * V) by k_rowsumsq_sub or cov = K_aa - V V^T by an mpad x mpad GEMM with beta = 1.

Error bars (u = 2^-53), first order, evaluated from the truth.  Notation: k_i = row i of K_ab, w_i = row i of
W = K_ab K^-1, v_i = row i of V, z = L^-1 y, alpha = K^-1 y; A = desc_ref's absolute-monomial sum of an entry times
(1 + U) (the assembly bar of tests/test_gpu_assembly.py is C1 u A); npad = N rounded up to 128.

  mean:  |mu_i - mu*_i| <= u ( C1 sum_j A^ab_ij |alpha_j| + |w_i|^T (c2 |L||L|^T + C1 A^bb) |alpha|
                               + c3 sum_j |v_ij| |z_j| )
  cov:   |cov_ij - cov*_ij| <= u ( C1 A^aa_ij + C1 sum_k (A^ab_ik |w_jk| + |w_ik| A^ab_jk)
                                   + |w_i|^T (c2 |L||L|^T + C1 A^bb) |w_j| + c4 sum_k |v_ik| |v_jk| )
  var:   the covariance bar with i = j.

Derivation.  Entry errors of K_ab: mu_i = k_i^T alpha and cov_ij = K^aa_ij - k_i^T w_j - w_i^T k_j + ..., so an error
of at most C1 u A in every entry (C1 = 64) gives the A^ab terms, and C1 u A^aa_ij is that of K_aa.  Entry errors dK of
K_bb change alpha by -K^-1 dK alpha and K^-1 by -K^-1 dK K^-1: -w_i^T dK alpha and +w_i^T dK w_j, hence C1 A^bb.  The
factorisation: the Cholesky factor of the bordered matrix [K y] (the solver factors y as one more row, so z comes from
the same blocked recursion) has a backward error |dK| <= gamma_npad |L||L|^T; each triangular solve with L (z, V) has
|dL| <= gamma_npad |L|, which moves mu_i by v_i^T dL^T alpha or w_i^T dL L^T alpha and cov_ij by v_i^T dL^T w_j
(+ transpose); since |v_i| <= |L|^T |w_i| every one of these three is bounded by gamma_npad |w_i|^T |L||L|^T |.| :
c2 = 3 (npad + 1).  The final sums: k_gemv and k_rowsumsq_sub add <= n / 32 terms per lane and 5 shuffle levels, the
GEMM <= npad products per entry: c3 = c4 = npad + 8.  The bars do not grow with cond(K) but only through |w_i| and
|alpha|, so they stay meaningful at eps = 1e-6.  Every case prints its worst err / bar for mu, var and cov.

The full covariance of a large test set is checked on its whole diagonal and on a dense sample of rows (block edges
and random rows) against the same bar.  K_aa is assembled mirrored (exactly symmetric), so cov - cov^T comes from the
GEMM alone: it is held to u c4 (|V||V|^T)_ij over all pairs.  var and diag(cov) are each held to the bar; they sum in
different orders and are not required to be equal.

Bitwise: a solver reused across test-set sizes, test plans, output kinds and NLL + gradient evaluations equals a fresh
solver; every slot of pigp_predict_batch_host equals the single-theta call, also next to a theta whose factorisation
fails; the device entry point on a non-default stream equals the host entry point.  Sharded solvers (world 2 and 3,
in-process ranks, device entry points on one non-blocking stream per rank) must meet the bar on the full test set and on
the shards of GPmodel.shard_points, with ranks that own an empty slice of a block or no test points at all.
"""
import ctypes as C
import threading

import numpy as np
import pytest

from oracle import posterior_ref
from stopro_b200 import _lib, operators, synthetic
from stopro_b200.GP.gp import GPmodel
from stopro_b200.plan import Plan, Solver

pytestmark = pytest.mark.gpu

U = 2.0 ** -53
C1 = 64.0
LD = np.longdouble
M_SWEEP = [1, 2, 127, 128, 129, 300, 1152, 1153, 2304, 2305]


def slab_height(m):
    mpad = -(-m // 128) * 128
    return 32 if mpad > 148 * 16 else 16 if mpad > 148 * 8 else 8


def split(m, sizes):
    """m test points over blocks of pool sizes `sizes` (per-block prefixes, roughly proportional)."""
    tot = sum(sizes)
    c = [m * s // tot for s in sizes]
    for b in range(len(sizes)):
        while sum(c) < m and c[b] < sizes[b]:
            c[b] += 1
    assert sum(c) == m
    return c


# ------------------------------------------------------------------------------------------------------- cases
class Case:
    """A training set and theta of a model class, a pool of test points per test block, and the truth."""

    def __init__(self, name, cfg, test_names=None, pool=None, theta=None, eps=None, kernel_type=None, form=None):
        if form is not None:
            cfg["kernel"] = dict(cfg["kernel"], kernel_form=form)
        if kernel_type is not None:
            cfg["kernel"] = dict(cfg["kernel"], kernel_type=kernel_type)
        self.name, self.cfg = name, cfg
        self.gp = synthetic.make_model(cfg)
        self.r_train, self.y = cfg["r_train"], np.asarray(cfg["delta_y"], dtype=np.float64)
        self.eps = cfg["eps"] if eps is None else eps
        self.theta = np.asarray(cfg["theta0"] if theta is None else theta, dtype=np.float64)
        self.test_names = list(test_names or self.gp.test_observables)
        self.pool = pool if pool is not None else cfg["r_test"][:len(self.test_names)]
        gp = self.gp
        self.post = posterior_ref.Posterior(gp.dim, gp.product_form, gp.kernel_type, gp._obs, gp._fields,
                                            gp.train_observables[:len(self.r_train)], self.r_train, self.test_names,
                                            self.pool, self.theta, self.y, self.eps, lbox=gp.lbox,
                                            noise_blocks=gp.index_optimize_noise or None)
        self.N = self.post.N
        self.npad = -(-self.N // 128) * 128
        self.T = self.npad // 128
        p = self.post
        B = 3.0 * (self.npad + 1) * p.LLt + C1 * p.A_bb
        self.absW = np.abs(p.W)
        self.G = self.absW @ B                      # |w_i|^T (c2 |L||L|^T + C1 A_bb)
        self.absV = np.abs(p.V.astype(np.float64))
        self.c34 = self.npad + 8.0
        al, z = np.abs(p.alpha.astype(np.float64)), np.abs(p.z.astype(np.float64))
        self.bar_mu = U * (C1 * (p.A_ab @ al) + self.G @ al + self.c34 * (self.absV @ z))
        self.bar_var = U * (C1 * p.A_aa_diag + 2 * C1 * np.sum(p.A_ab * self.absW, axis=1)
                            + np.sum(self.G * self.absW, axis=1) + self.c34 * np.sum(self.absV ** 2, axis=1))
        self._plans = {}

    # -- plans
    def training_plan(self):
        gp = self.gp
        if "train" not in self._plans:
            self._plans["train"] = Plan(gp.dim, gp.product_form, gp._fields, gp._observables(gp.train_observables[:len(self.r_train)]),
                                        self.r_train, lbox=gp.lbox, noise_blocks=gp.index_optimize_noise or None,
                                        kernel_type=gp.kernel_type)
        return self._plans["train"]

    def test_plans(self, counts):
        """(mixed, test, pool rows) of the test set made of the first counts[b] pool points of every block."""
        key = tuple(counts)
        if key not in self._plans:
            gp = self.gp
            pts = [np.asarray(self.pool[b])[:c] for b, c in enumerate(counts)]
            te = gp._observables(self.test_names)
            mixed = Plan(gp.dim, gp.product_form, gp._fields, te, pts, gp._observables(gp.train_observables[:len(self.r_train)]),
                         self.r_train, lbox=gp.lbox, kernel_type=gp.kernel_type)
            test = Plan(gp.dim, gp.product_form, gp._fields, te, pts, lbox=gp.lbox, kernel_type=gp.kernel_type)
            self._plans[key] = (mixed, test, self.post.rows(counts))
        return self._plans[key]

    def counts(self, m):
        return split(m, [len(p) for p in self.pool])

    def close(self):
        for v in self._plans.values():
            for p in (v if isinstance(v, tuple) else (v,)):
                if isinstance(p, Plan):
                    p.close()
        self._plans = {}
        self.gp.close()

    # -- bars
    def check(self, rows, mu, var=None, cov=None, sample=200, what=""):
        """Entry-wise check of a prediction over pool rows `rows` -> dict of worst err / bar."""
        p = self.post
        out = {}
        assert np.isfinite(mu).all(), f"{what}: non-finite mean"
        r = (np.abs(mu.astype(LD) - p.mu[rows]).astype(np.float64)) / np.maximum(self.bar_mu[rows], 1e-300)
        out["mu"] = float(r.max()) if len(r) else 0.0
        assert out["mu"] <= 1.0, f"{what}: mean row {int(np.argmax(r))} err/bar {out['mu']:.3e}"
        diag = var if var is not None else np.diag(cov)
        r = (np.abs(diag.astype(LD) - p.var[rows]).astype(np.float64)) / np.maximum(self.bar_var[rows], 1e-300)
        key = "var" if var is not None else "diag(cov)"
        out[key] = float(r.max())
        assert out[key] <= 1.0, f"{what}: {key} row {int(np.argmax(r))} err/bar {out[key]:.3e}"
        if cov is not None:
            m = len(rows)
            # asymmetry: the GEMM's rounding only (K_aa is mirrored)
            asym = np.abs(cov - cov.T)
            gemm = U * self.c34 * (self.absV[rows] @ self.absV[rows].T)
            out["asym"] = float(asym.max())
            assert (asym <= gemm).all(), f"{what}: |cov - cov^T| {asym.max():.3e} exceeds the GEMM bound"
            # dense sample: block edges and random rows
            sec = np.searchsorted(rows, p.sec_te)
            pick = {0, m - 1} | {int(s) for s in sec if s < m} | {int(s) - 1 for s in sec if 0 < s <= m}
            rng = np.random.default_rng(m)
            pick |= {int(v) for v in rng.choice(m, min(m, sample), replace=False)}
            S = np.array(sorted(pick))
            R = rows[S]
            truth, Aaa = p.cov_full(R)
            bar = U * (C1 * Aaa + C1 * (p.A_ab[R] @ self.absW[R].T + self.absW[R] @ p.A_ab[R].T)
                       + self.G[R] @ self.absW[R].T + self.c34 * (self.absV[R] @ self.absV[R].T))
            err = np.abs(cov[np.ix_(S, S)].astype(LD) - truth).astype(np.float64)
            ratio = err / np.maximum(bar, 1e-300)
            out["cov"] = float(ratio.max())
            i, j = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
            assert out["cov"] <= 1.0, f"{what}: cov ({S[i]}, {S[j]}) err {err[i, j]:.3e} bar {bar[i, j]:.3e}"
        return out


def _se2d(n, form="product", kernel_type=None, eps=1e-3, n_test=100, seed=0):
    cfg = dict(synthetic.stokes2d_scaling(n, seed=seed, n_test=n_test), eps=eps)
    th = cfg["theta0"] + 0.05 * np.random.default_rng(n).standard_normal(9)
    return dict(cfg=cfg, theta=th, form=form, kernel_type=kernel_type)


def _pool_2d(sizes, seed):
    rng = np.random.default_rng(seed)
    return [rng.random((s, 2)) for s in sizes]


POOL_SIZES = [461, 0, 1152, 692]  # 2305 points; p, an empty ux block, fy, uy


def _sweep_case():
    """N = 300 (T = 3, odd split), test blocks in another order than the training blocks, uneven, one empty; the pool
    holds 2305 points so the M sweep crosses both slab-height switches."""
    d = _se2d(300)
    return dict(d, test_names=["p", "ux", "fy", "uy"], pool=_pool_2d(POOL_SIZES, 1))


def _drag3d():
    cfg = dict(synthetic.drag3d(n_u=5, n_f=4, n_test=14), eps=1e-3)
    th = cfg["theta0"] + 0.05 * np.random.default_rng(3).standard_normal(len(cfg["theta0"]))
    return dict(cfg=cfg, theta=th)


def _sinusoidal():
    cfg = dict(synthetic.sinusoidal(u_num=20, f_nx=16, f_ny=8, dif_num=10, n_test=12), eps=1e-3)
    th = cfg["theta0"] + 0.05 * np.random.default_rng(4).standard_normal(len(cfg["theta0"]))
    # mixed blocks with shift wrappers: the test points against the difux / difuy / difp training blocks
    return dict(cfg=cfg, theta=th, test_names=["uy", "ux"], pool=[cfg["r_test"][0][:101], cfg["r_test"][1][:60]])


def _matern():
    """Matern-5/2, product form, on the value blocks ux, uy, p only (the kernel is twice differentiable)."""
    cfg = dict(synthetic.stokes2d_scaling(400, seed=5, n_test=100), eps=1e-3)
    rng = np.random.default_rng(6)
    cfg["r_train"] = [rng.random((n, 2)) for n in (150, 121, 129)]
    cfg["delta_y"] = rng.standard_normal(400)
    th = np.tile([0.0, np.log(0.3), np.log(0.4)], 3) + 0.05 * rng.standard_normal(9)
    return dict(cfg=cfg, theta=th, kernel_type="mt52")


def _sin1d():
    cfg = synthetic.sin_1d_naive(n=32, n_test=300)
    th = cfg["theta0"] + np.array([0.1, -0.2, 0.0])
    return dict(cfg=cfg, theta=th)


CASES = {
    "se2d_N300_sweep": _sweep_case,
    "se2d_N32": lambda: _se2d(32, n_test=43),
    "se2d_N97": lambda: _se2d(97, n_test=43),
    "se2d_N128": lambda: _se2d(128, n_test=43),
    "se2d_N129": lambda: _se2d(129, n_test=43),
    "se2d_N600_T5": lambda: _se2d(600),
    "se2d_N900_T8": lambda: _se2d(900),
    "se2d_additive_N600": lambda: _se2d(560, form="additive"),
    "mt52_N400": _matern,
    "drag3d": _drag3d,
    "sinusoidal_shifts": _sinusoidal,
    "sin1d_naive_noise": _sin1d,
    "stokes_eps1e-6": lambda: _se2d(400, eps=1e-6),
}
_CACHE = {}


def get_case(name):
    if name not in _CACHE:
        _CACHE[name] = Case(name, **CASES[name]())
    return _CACHE[name]


@pytest.fixture(scope="module", autouse=True)
def _close_cases():
    yield
    for c in _CACHE.values():
        c.close()
    _CACHE.clear()


def predict(solver, mixed, test, theta, y, eps, full):
    mu, cov, info = solver.predict_host(mixed, test, theta, y, eps, full_cov=full)
    assert info == 0
    return mu, cov


def _report(c, m, res, tag=""):
    print(f"\n[{c.name}{tag}] M={m} N={c.N} T={c.T} slab={slab_height(m)} " + " ".join(f"{k} {v:.2e}" for k, v in res.items()))


# ------------------------------------------------------------------------------------------------------- tests
def test_m_sweep(cuda_device):
    """Test-point counts on both sides of the 128-row tile and of the 8 -> 16 and 16 -> 32 slab switches."""
    c = get_case("se2d_N300_sweep")
    solver = Solver(c.training_plan())
    try:
        for m in M_SWEEP:
            mixed, test, rows = c.test_plans(c.counts(m))
            mu, cov = predict(solver, mixed, test, c.theta, c.y, c.eps, True)
            mu_d, var = predict(solver, mixed, test, c.theta, c.y, c.eps, False)
            assert np.array_equal(mu_d, mu)
            res = c.check(rows, mu, cov=cov, what=f"M={m} full")
            res.update(c.check(rows, mu_d, var=var, what=f"M={m} diag"))
            _report(c, m, res)
    finally:
        solver.close()


@pytest.mark.parametrize("name", [n for n in CASES if n != "se2d_N300_sweep"])
def test_case(cuda_device, name):
    """Training sizes around the k_gemv / k_rowsumsq_sub chunks and the tile edge, T = 1 ... 8, SE product and
    additive, 3-D, Matern, shift wrappers, a noise parameter, eps = 1e-6."""
    c = get_case(name)
    solver = Solver(c.training_plan())
    try:
        for m in sorted({1, min(129, c.post.M), c.post.M}):
            mixed, test, rows = c.test_plans(c.counts(m))
            mu, cov = predict(solver, mixed, test, c.theta, c.y, c.eps, True)
            mu_d, var = predict(solver, mixed, test, c.theta, c.y, c.eps, False)
            assert np.array_equal(mu_d, mu)
            res = c.check(rows, mu, cov=cov, what=f"{name} M={m}")
            res.update(c.check(rows, mu_d, var=var, what=f"{name} M={m} diag"))
            _report(c, m, res)
    finally:
        solver.close()


def test_workspace_reuse_bitwise(cuda_device):
    """One solver: large M, small M, another test plan, full / diagonal alternating, NLL + gradient in between (which
    leaves K^-1 where L was) -- each result equals a fresh solver's bit for bit."""
    c = get_case("se2d_N300_sweep")
    other = Case("other_plan", **dict(_se2d(300), test_names=["fx", "div", "uy"], pool=_pool_2d([40, 1, 88], 9)))
    used = Solver(c.training_plan())
    try:
        seq = [(c, 2305, True), (c, 129, False), (other, 129, True), (c, 1153, False), (c, 1153, True),
               ("grad", None, None), (c, 300, False), ("grad", None, None), (c, 300, True), (other, 129, False)]
        for k, (cc, m, full) in enumerate(seq):
            if cc == "grad":
                nll, grad, info = used.nll_grad_host(c.theta, c.y, c.eps, want_grad=True)
                assert info == 0 and np.isfinite(grad).all()
                continue
            mixed, test, _ = cc.test_plans(cc.counts(m))
            got = predict(used, mixed, test, cc.theta, cc.y, cc.eps, full)
            fresh = Solver(cc.training_plan())
            try:
                want = predict(fresh, mixed, test, cc.theta, cc.y, cc.eps, full)
            finally:
                fresh.close()
            for a, b in zip(got, want):
                assert a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64)), f"step {k}: M={m} full={full}"
    finally:
        used.close()
        other.close()


def test_batch_slots_bitwise(cuda_device):
    c = get_case("se2d_N600_T5")
    mixed, test, _ = c.test_plans(c.counts(129))
    rng = np.random.default_rng(8)
    thetas = [c.theta + 0.05 * rng.standard_normal(len(c.theta)) for _ in range(5)]
    solver = Solver(c.training_plan())
    try:
        for full in (False, True):
            single = [solver.predict_host(mixed, test, t, c.y, c.eps, full_cov=full) for t in thetas]
            for nb in (1, 2, 5):
                mu, cov, info = solver.predict_batch_host(mixed, test, thetas[:nb], c.y, c.eps, full_cov=full)
                assert (info == 0).all()
                for b in range(nb):
                    assert np.array_equal(mu[b], single[b][0]) and np.array_equal(cov[b], single[b][1]), (nb, b, full)
    finally:
        solver.close()


def test_batch_failed_slot(cuda_device):
    """One theta whose factorisation fails (K ~ eps I with eps < 0) among positive definite ones (a large signal
    variance with a tiny length scale keeps K ~ gamma I): that slot gives NaN and info != 0, its neighbours are the
    single-theta results bit for bit."""
    obs, fields = operators.scalar_observables(1)
    y_obs = [obs["y"]]
    x = np.linspace(0.0, 6.0, 40)
    xt = np.linspace(0.05, 5.95, 23)
    y = np.sin(x)
    eps = -1e-3
    ok = [np.array([2.0, -6.0]), np.array([1.5, -5.0]), np.array([2.5, -7.0]), np.array([1.0, -6.5])]
    bad = np.array([-30.0, -6.0])
    thetas = [ok[0], ok[1], bad, ok[2], ok[3]]
    plan = Plan(1, True, fields, y_obs, [x])
    mixed = Plan(1, True, fields, y_obs, [xt], y_obs, [x])
    test = Plan(1, True, fields, y_obs, [xt])
    solver = Solver(plan)
    try:
        for full in (False, True):
            mu, cov, info = solver.predict_batch_host(mixed, test, thetas, y, eps, full_cov=full)
            assert info[2] != 0 and np.isnan(mu[2]).all() and np.isnan(cov[2]).all(), (info, full)
            for b in (0, 1, 3, 4):
                m1, c1, i1 = solver.predict_host(mixed, test, thetas[b], y, eps, full_cov=full)
                assert info[b] == 0 and i1 == 0
                assert np.array_equal(mu[b], m1) and np.array_equal(cov[b], c1), (b, full)
                assert np.isfinite(mu[b]).all()
    finally:
        solver.close()
        for p in (plan, mixed, test):
            p.close()


def _device_predict(solver, mixed, test, theta_t, y_t, eps, full, stream, mu_t, cov_t, info_t):
    _lib.check(_lib.lib().pigp_predict(solver.handle, mixed.handle, test.handle, theta_t.data_ptr(), y_t.data_ptr(),
                                       float(eps), mu_t.data_ptr(), cov_t.data_ptr(), int(full), info_t.data_ptr(),
                                       C.c_void_p(stream.cuda_stream)))


def test_device_entry_on_a_stream(cuda_device):
    """pigp_predict on a non-default stream, theta and y written on that stream just before the call and the outputs
    read on it just after: equal to the host entry point bit for bit."""
    import torch

    c = get_case("se2d_N300_sweep")
    solver = Solver(c.training_plan())
    try:
        for m in (129, 1153):
            mixed, test, _ = c.test_plans(c.counts(m))
            st = torch.cuda.Stream()
            for full in (True, False):
                want = solver.predict_host(mixed, test, c.theta, c.y, c.eps, full_cov=full)
                with torch.cuda.stream(st):
                    th = torch.empty(len(c.theta), dtype=torch.float64, device=cuda_device)
                    y = torch.empty(c.N, dtype=torch.float64, device=cuda_device)
                    mu = torch.full((m,), float("nan"), dtype=torch.float64, device=cuda_device)
                    cov = torch.full((m * m if full else m,), float("nan"), dtype=torch.float64, device=cuda_device)
                    info = torch.full((1,), -7, dtype=torch.int32, device=cuda_device)
                    th.copy_(torch.as_tensor(c.theta).pin_memory(), non_blocking=True)
                    y.copy_(torch.as_tensor(c.y).pin_memory(), non_blocking=True)
                    _device_predict(solver, mixed, test, th, y, c.eps, full, st, mu, cov, info)
                    out = (mu.to("cpu", non_blocking=False), cov.to("cpu"), info.to("cpu"))
                st.synchronize()
                assert int(out[2][0]) == 0
                assert np.array_equal(out[0].numpy(), want[0])
                assert np.array_equal(out[1].numpy(), want[1].reshape(-1)), (m, full)
    finally:
        solver.close()


# ------------------------------------------------------------------------------------------------------- sharded
def _wired_solvers(plan, world):
    """In-process ranks wired like DistSolver.connect_pointers, on one shared device."""
    solvers = [Solver(plan, r, world) for r in range(world)]
    L = _lib.lib()
    slabs = []
    for s in solvers:
        ptr, nbytes = C.c_void_p(), C.c_int64()
        _lib.check(L.pigp_dsolver_slab(s._ds, C.byref(ptr), C.byref(nbytes)))
        slabs.append(ptr.value)
    arr = (C.c_void_p * world)(*[C.c_void_p(p) for p in slabs])
    for s in solvers:
        _lib.check(L.pigp_dsolver_connect(s._ds, arr))
        _lib.check(L.pigp_dsolver_set_shared_device(s._ds, 1))
    return solvers


def _run_ranks(c, solvers, jobs, full):
    """jobs[r] = (mixed, test, m) or None (NLL only); one thread and one non-blocking stream per rank, device entry
    points -> [(mu, cov) or nll]."""
    import torch

    dev = torch.device("cuda:0")
    world = len(solvers)
    th = torch.as_tensor(c.theta, device=dev)
    y = torch.as_tensor(c.y, device=dev)
    bufs = []
    for r in range(world):
        m = jobs[r][2] if jobs[r] else 0
        bufs.append((torch.full((max(m, 1),), float("nan"), dtype=torch.float64, device=dev),
                     torch.full((max(m * m if full else m, 1),), float("nan"), dtype=torch.float64, device=dev),
                     torch.full((1,), -7, dtype=torch.int32, device=dev)))
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    torch.cuda.synchronize()
    errs = [None] * world

    def work(r):
        try:
            mu, cov, info = bufs[r]
            if jobs[r] is None:
                _lib.check(_lib.lib().pigp_nll(solvers[r].handle, th.data_ptr(), y.data_ptr(), float(c.eps), mu.data_ptr(),
                                               info.data_ptr(), C.c_void_p(streams[r].cuda_stream)))
            else:
                mixed, test, _ = jobs[r]
                _device_predict(solvers[r], mixed, test, th, y, c.eps, full, streams[r], mu, cov, info)
            streams[r].synchronize()
        except Exception as exc:  # noqa: BLE001
            errs[r] = exc

    ts = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for e in errs:
        if e is not None:
            raise e
    out = []
    for r in range(world):
        mu, cov, info = (b.cpu().numpy() for b in bufs[r])
        assert int(info[0]) == 0, f"rank {r}: info {int(info[0])}"
        m = jobs[r][2] if jobs[r] else 0
        out.append((mu[:m], cov[:m * m].reshape(m, m) if full else cov[:m]) if jobs[r] else float(mu[0]))
    return out


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_ranks(cuda_device, world):
    c = get_case("se2d_N600_T5")
    plan = c.training_plan()
    solvers = _wired_solvers(plan, world)
    extra = []
    try:
        single = Solver(plan)
        mixed, test, rows = c.test_plans(c.counts(300))
        want = [predict(single, mixed, test, c.theta, c.y, c.eps, f) for f in (True, False)]
        single.close()
        # every rank predicts the full test set
        agree = True
        for full in (True, False):
            out = _run_ranks(c, solvers, [(mixed, test, len(rows))] * world, full)
            for r, (mu, cv) in enumerate(out):
                res = c.check(rows, mu, **({"cov": cv} if full else {"var": cv}), what=f"world {world} rank {r}")
                _report(c, len(rows), res, tag=f" rank {r}/{world}")
            agree &= all(np.array_equal(o[0], out[0][0]) and np.array_equal(o[1], out[0][1]) for o in out)
            agree &= np.array_equal(out[0][0], want[0][0]) and np.array_equal(out[0][1], want[0 if full else 1][1])
        print(f"\n[{c.name}] world={world}: ranks and the single solver agree bitwise: {agree}")
        # shards of GPmodel.shard_points; block 1 has fewer points than ranks, so rank 0's slice of it is empty
        counts = [5, 1, 7]
        pts = [np.asarray(c.pool[b])[:n] for b, n in enumerate(counts)]
        jobs, rowsets = [], []
        gp = c.gp
        for r in range(world):
            shard, slices = GPmodel.shard_points(pts, r, world)
            assert r > 0 or len(shard[1]) == 0
            k = [len(s) for s in shard]
            if sum(k) == 0:
                jobs.append(None)
                rowsets.append(None)
                continue
            te = gp._observables(c.test_names)
            mx = Plan(gp.dim, gp.product_form, gp._fields, te, shard, gp._observables(gp.train_observables), c.r_train,
                      lbox=gp.lbox, kernel_type=gp.kernel_type)
            ts = Plan(gp.dim, gp.product_form, gp._fields, te, shard, lbox=gp.lbox, kernel_type=gp.kernel_type)
            extra += [mx, ts]
            jobs.append((mx, ts, sum(k)))
            rowsets.append(np.concatenate([c.post.sec_te[b] + np.arange(a, z) for b, (a, z) in enumerate(slices)]).astype(np.int64))
        for full in (False, True):
            out = _run_ranks(c, solvers, jobs, full)
            for r in range(world):
                if jobs[r] is None:
                    continue
                mu, cv = out[r]
                res = c.check(rowsets[r], mu, **({"cov": cv} if full else {"var": cv}), what=f"shard {r}/{world}")
                print(f"  shard rank {r}/{world} M={len(rowsets[r])}: " + " ".join(f"{k} {v:.2e}" for k, v in res.items()))
        # a rank with no test points takes part through an NLL-only evaluation
        jobs = [None] + [(mixed, test, len(rows))] * (world - 1)
        out = _run_ranks(c, solvers, jobs, False)
        for r in range(1, world):
            c.check(rows, out[r][0], var=out[r][1], what=f"world {world} rank {r} next to an NLL-only rank")
        assert np.isfinite(out[0])
    finally:
        for s in solvers:
            s.close()
        for p in extra:
            p.close()


# ------------------------------------------------------------------------------------------------------- arguments
def test_predict_rejects_bad_arguments(cuda_device):
    """Null arguments, a symmetric mixed plan, wrong column / row counts, a rectangular test plan, and (new) mixed or
    test plans whose dim, kernel type, form or number of hyper-parameter groups differ from the training plan's: every
    one is PIGP_EINVAL before any launch."""
    import torch

    so, sf = operators.stokes_observables(2)
    co, cf = operators.scalar_observables(2)
    rng = np.random.default_rng(2)
    tr_pts = [rng.random((20, 2)), rng.random((9, 2))]
    te_pts = [rng.random((7, 2))]
    tr_names = [so["ux"], so["p"]]
    plan = Plan(2, True, sf, tr_names, tr_pts)
    good_mixed = Plan(2, True, sf, [so["uy"]], te_pts, tr_names, tr_pts)
    good_test = Plan(2, True, sf, [so["uy"]], te_pts)
    plans = [plan, good_mixed, good_test]

    def mk(*a, **k):
        p = Plan(*a, **k)
        plans.append(p)
        return p

    tr1 = [np.concatenate(tr_pts)[:, :1]]
    te1 = [te_pts[0][:, :1]]
    o1, f1 = operators.scalar_observables(1)
    bad = {
        "mixed symmetric": (mk(2, True, sf, [so["uy"]], [rng.random((29, 2))]), good_test),
        "mixed cols": (mk(2, True, sf, [so["uy"]], te_pts, [so["ux"]], [tr_pts[0]]), good_test),
        "test rectangular": (good_mixed, mk(2, True, sf, [so["uy"]], te_pts, [so["uy"]], te_pts)),
        "test rows": (good_mixed, mk(2, True, sf, [so["uy"]], [te_pts[0][:6]])),
        "mixed dim": (mk(1, True, f1, [o1["y"]], te1, [o1["y"]], tr1), good_test),
        "test dim": (good_mixed, mk(1, True, f1, [o1["y"]], te1)),
        "mixed kernel": (mk(2, True, sf, [so["uy"]], te_pts, tr_names, tr_pts, kernel_type="mt52"), good_test),
        "test kernel": (good_mixed, mk(2, True, sf, [so["uy"]], te_pts, kernel_type="mt72")),
        "mixed form": (mk(2, False, sf, [so["uy"]], te_pts, tr_names, tr_pts), good_test),
        "test form": (good_mixed, mk(2, False, sf, [so["uy"]], te_pts)),
        "mixed groups": (mk(2, True, cf, [co["y"]], te_pts, [co["y"], co["y"]], tr_pts), good_test),
        "test groups": (good_mixed, mk(2, True, cf, [co["y"]], te_pts)),
    }
    solver = Solver(plan)
    dev = torch.device("cuda:0")
    th = torch.zeros(plan.theta_len, dtype=torch.float64, device=dev)
    y = torch.zeros(plan.rows, dtype=torch.float64, device=dev)
    mu = torch.zeros(64, dtype=torch.float64, device=dev)
    cov = torch.zeros(64, dtype=torch.float64, device=dev)
    L = _lib.lib()
    try:
        torch.cuda.synchronize()
        before = _lib.launch_count()
        for what, (mx, te) in bad.items():
            rc = L.pigp_predict(solver.handle, mx.handle, te.handle, th.data_ptr(), y.data_ptr(), 1e-2, mu.data_ptr(),
                                cov.data_ptr(), 1, None, None)
            assert rc == -1, what
        args = [solver.handle, good_mixed.handle, good_test.handle, th.data_ptr(), y.data_ptr(), 1e-2, mu.data_ptr(),
                cov.data_ptr(), 1, None, None]
        for k in (0, 1, 2, 3, 4, 6, 7):
            a = list(args)
            a[k] = None
            assert L.pigp_predict(*a) == -1, f"null argument {k}"
        assert _lib.launch_count() == before, "a rejected call launched a kernel"
        # the same plans through the batched host entry
        for what, (mx, te) in bad.items():
            with pytest.raises(_lib.PigpError):
                solver.predict_host(mx, te, np.zeros(plan.theta_len), np.zeros(plan.rows), 1e-2)
        mu_h, cov_h, info = solver.predict_host(good_mixed, good_test, np.zeros(plan.theta_len), np.zeros(plan.rows), 1e-2)
        assert info == 0 and np.isfinite(cov_h).all()
    finally:
        solver.close()
        for p in plans:
            p.close()
