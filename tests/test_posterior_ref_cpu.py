"""CPU tests of oracle.posterior_ref, the extended-precision posterior behind tests/test_gpu_posterior.py.

It is pinned to the two references the repository already trusts, on small configurations: one with a noise parameter
(sin1d_naive: the training theta has one entry more than the mixed and test plans read) and one with shift wrappers on
the mixed blocks (the sinusoidal channel, lbox = [2.5, 0]):
  * oracle.extended.truth (oracle.closed_form blocks in longdouble, the same factorisation): mu, var and alpha agree
    within cond(K) u.  The two differ only in their data: desc_ref forms the point differences in float64, as the
    kernels do, closed_form in longdouble, a relative perturbation of at most u per difference;
  * oracle.gp_ref in float64 (LAPACK): mu and the full covariance agree within that evaluation's own conditioning,
    cond(K) u relative to the largest entry.
"""
import numpy as np
import pytest

from oracle import extended, posterior_ref
from oracle.gp_ref import GPRef
from stopro_b200 import synthetic

LD = np.longdouble


def _sinusoidal():
    return dict(synthetic.sinusoidal(u_num=8, f_nx=5, f_ny=3, dif_num=4, n_test=4), eps=1e-4)


def _sin1d():
    return synthetic.sin_1d_naive(n=24, n_test=17)


CASES = {"sin1d_naive_noise": _sin1d, "sinusoidal_shifts": _sinusoidal}


@pytest.fixture(scope="module", params=list(CASES))
def case(request):
    cfg = CASES[request.param]()
    rng = np.random.default_rng(5)
    th = cfg["theta0"].copy()
    noise = bool(cfg["model_kwargs"].get("index_optimize_noise"))
    nk = len(th) - noise
    th[:nk] += 0.2 * rng.standard_normal(nk)
    gp = synthetic.make_model(cfg)
    post = posterior_ref.Posterior.for_model(gp, cfg["r_train"], cfg["r_test"], th, cfg["delta_y"], cfg["eps"])
    kw = cfg["model_kwargs"]

    def gpref(dtype):
        g = GPRef(cfg["model"], kernel_form=cfg["kernel"]["kernel_form"], dim=cfg["kernel"]["input_dim"],
                  lbox=kw.get("lbox"), index_optimize_noise=kw.get("index_optimize_noise"), backend="closed",
                  dtype=dtype)
        g.set_constants(cfg["r_test"], cfg["mu_test"], cfg["r_train"], cfg["delta_y"], cfg["eps"])
        return g

    return dict(cfg=cfg, th=th, post=post, gpref=gpref, name=request.param)


def test_matches_extended_truth(case):
    cfg, post = case["cfg"], case["post"]
    ref = case["gpref"](LD)
    t = extended.truth(ref, case["th"], ref._pts(cfg["r_train"]), cfg["delta_y"], cfg["eps"], r_test=cfg["r_test"],
                       want_grad=False)
    # mixed blocks with shift wrappers are differences of nearly equal terms: compare against the magnitudes
    scale_mu = np.max(np.abs(post.A_ab) @ np.abs(post.alpha.astype(np.float64)))
    scale_var = max(np.max(post.A_aa_diag), np.max(np.sum(np.abs(post.V.astype(np.float64)) ** 2, axis=1)))
    e_mu = np.max(np.abs(post.mu.astype(np.float64) - t["mu"]))
    e_var = np.max(np.abs(post.var.astype(np.float64) - t["var"]))
    e_alpha = np.max(np.abs(post.alpha.astype(np.float64) - t["alpha"])) / np.max(np.abs(t["alpha"]))
    print(f"\n[{case['name']}] N={post.N} M={post.M} vs extended.truth: mu {e_mu / scale_mu:.1e} var {e_var / scale_var:.1e} "
          f"alpha {e_alpha:.1e}")
    # longdouble evaluations of data that differ by the rounding of the point differences (float64 here)
    cond = np.linalg.cond(post.K.astype(np.float64))
    tol = cond * 2.0 ** -53
    assert e_mu <= tol * scale_mu and e_var <= tol * scale_var and e_alpha <= tol


def test_matches_float64_gp_ref(case):
    cfg, post = case["cfg"], case["post"]
    ref = case["gpref"](np.float64)
    mus, covs = ref.predictingFunction_all(case["th"], cfg["r_test"], cfg["mu_test"], cfg["r_train"], cfg["delta_y"],
                                           cfg["eps"])
    mu = np.concatenate(mus)
    rows = np.arange(post.M)
    cov, _ = post.cov_full(rows)
    cov = cov.astype(np.float64)
    sec = post.sec_te
    cond = np.linalg.cond(post.K.astype(np.float64))
    tol = max(1e-12, 0.05 * cond * 2.0 ** -53)
    e_mu = np.max(np.abs(post.mu.astype(np.float64) - mu)) / np.max(np.abs(mu))
    e_cov = max(np.max(np.abs(cov[sec[b]:sec[b + 1], sec[b]:sec[b + 1]] - covs[b])) for b in range(len(covs)))
    e_cov /= max(np.max(np.abs(c)) for c in covs)
    # the diagonal of the full covariance is the variance the reference keeps separately
    assert np.max(np.abs(np.diag(cov) - post.var.astype(np.float64))) <= 1e-15 * np.max(np.abs(cov))
    print(f"\n[{case['name']}] cond(K) {cond:.1e} vs gp_ref float64: mu {e_mu:.1e} cov {e_cov:.1e} (tol {tol:.1e})")
    assert e_mu <= tol and e_cov <= tol


def test_pool_prefixes_and_sampled_entries(case):
    """A prefix test set indexes the pool's truth; cov(I, J) equals the dense covariance entry for entry."""
    post = case["post"]
    counts = [max(0, (post.sec_te[b + 1] - post.sec_te[b]) // 2) for b in range(len(post.sec_te) - 1)]
    rows = post.rows(counts)
    assert len(rows) == sum(counts)
    dense, A = post.cov_full(rows)
    I, J = [x.ravel() for x in np.meshgrid(rows, rows, indexing="ij")]
    got, A2 = post.cov(I, J)
    assert np.max(np.abs(got.reshape(dense.shape) - dense)) <= 1e-17 * np.max(np.abs(dense))
    assert np.array_equal(A2.reshape(A.shape), A)
    assert np.max(np.abs(np.diag(dense) - post.var[rows])) <= 1e-17 * np.max(np.abs(dense))
