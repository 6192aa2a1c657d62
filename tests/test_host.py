"""CPU tests (no GPU): the C-ABI library loads and exports what include/pigp.h declares; the descriptor compiler
reproduces every block of the reference's library (checked against the oracle's hand-written tables); the host-side
mirror of the reference interface (logposterior, optimiser driver, theta handling) behaves like the reference's."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import blocks_ref, closed_form
from oracle.desc_ref import eval_desc
from stopro_b200 import _lib, operators

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="session")
def built_lib():
    if not os.path.exists(_lib.LIB_PATH):
        subprocess.run(["make", "-C", os.path.join(ROOT, "stopro_b200", "csrc"), "-j4"], check=True)
    return ctypes.CDLL(_lib.LIB_PATH)


def test_library_exports_every_declared_symbol(built_lib):
    header = open(os.path.join(ROOT, "include", "pigp.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(pigp_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 20
    for name in sorted(declared):
        assert hasattr(built_lib, name), f"{name} is declared in include/pigp.h but not exported"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    built_lib.pigp_abi_version.restype = ctypes.c_int
    assert built_lib.pigp_abi_version() == _lib.ABI_VERSION
    # a freshly loaded library has launched nothing (no compute without a GPU); checked in a process of its own because
    # GPU tests earlier in the session share this process's copy of the library and its launch counter
    code = ("import ctypes, sys; lib = ctypes.CDLL(sys.argv[1]); lib.pigp_launch_count.restype = ctypes.c_int64; "
            "print(lib.pigp_launch_count())")
    res = subprocess.run([sys.executable, "-c", code, _lib.LIB_PATH], capture_output=True, text=True, check=True)
    assert int(res.stdout) == 0


def test_struct_layout_matches_header():
    # pigp_term: int32 + 3*int32 + double = 24 bytes; pigp_block_desc: 4*int32 + 8 terms
    assert ctypes.sizeof(_lib.Term) == 24
    assert ctypes.sizeof(_lib.BlockDesc) == 16 + 8 * 24
    assert _lib.PlanDesc.lbox.offset % 8 == 0


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.PigpError, match="no CPU fallback"):
        _lib.lib()


@pytest.mark.parametrize("dim,form", [(2, "product"), (2, "additive"), (3, "product")])
def test_descriptor_compiler_reproduces_the_block_library(dim, form):
    """Every K<a><b> of gp_2D_stokes_independent.py / gp_3D_stokes_independent.py: derived descriptor == the
    oracle's hand-written spec, evaluated on random points."""
    rng = np.random.default_rng(dim)
    obs, fields = operators.stokes_observables(dim)
    table = blocks_ref.TABLES["poiseuille" if dim == 2 else "stokes3d"]
    theta = 0.3 * rng.standard_normal(len(fields) * (1 + dim))
    r, rp = rng.random((5, dim)), rng.random((4, dim))
    lbox = np.array([2.5, 0.0, 0.0])[:dim]

    def op_eval(op, a, b, th):
        return closed_form.eval_operator(op, a, b, th, form, dim)

    checked = 0
    for name in table["blocks"]:
        try:
            oa, ob = operators.parse_block_name(name, obs)
        except KeyError:
            continue
        want = blocks_ref.eval_block(name, table, op_eval, r, rp, theta, lbox, lambda n, m: np.zeros((n, m)))
        if name in ("Kuydifux",):  # reference quirk: built from Kuxuy == 0 (gp_2D_stokes_independent.py:164-165)
            assert not want.any()
        desc = operators.make_desc(oa, ob, fields, dim, form == "product")
        got = eval_desc(desc, dim, r, rp, theta, lbox, product=form == "product")
        scale = max(np.max(np.abs(want)), 1.0)
        assert np.max(np.abs(got - want)) <= 1e-12 * scale, name
        checked += 1
    assert checked >= (60 if dim == 2 else 70)


def test_scalar_models_descriptors():
    rng = np.random.default_rng(0)
    obs, fields = operators.scalar_observables(1)
    r, rp, theta = rng.random(6), rng.random(5), np.array([0.2, -0.3])
    for a, b, op in [("y", "y", "K"), ("y", "ly", "L1K"), ("ly", "ly", "LLK")]:
        desc = operators.make_desc(obs[a], obs[b], fields, 1, True)
        got = eval_desc(desc, 1, r, rp, theta)
        want = closed_form.eval_operator(op, r, rp, theta, "product", 1)
        assert np.max(np.abs(got - want)) <= 1e-13 * np.max(np.abs(want))


def test_define_kernel_semantics():
    from stopro_b200.GP.kernels import define_kernel

    k = define_kernel(dict(kernel_type="se", kernel_form="additive", input_dim=2, distance_func=False))
    assert not k.product_form and k.input_dim == 2
    r1, r2, th = np.array([0.1, 0.2]), np.array([0.4, 0.9]), np.array([0.3, -0.2, 0.1])
    want = np.exp(0.3) * (np.exp(-0.5 * (0.3 * np.exp(0.2)) ** 2) + np.exp(-0.5 * (0.7 * np.exp(-0.1)) ** 2))
    assert abs(k(r1, r2, th) - want) < 1e-15
    # the reference ignores kernel_form for 3-D inputs (kernels.py:419-426)
    assert define_kernel(dict(kernel_type="se", kernel_form="additive", input_dim=3, distance_func=False)).product_form
    # Matern kernels of GP/kernels.py:127-205
    m = define_kernel(dict(kernel_type="mt52", kernel_form="product", input_dim=2, distance_func=False))
    rho = np.sqrt(5.0) * np.abs(r1 - r2) * np.exp(-th[1:])
    want = np.exp(0.3) * np.prod((1.0 + rho + rho ** 2 / 3.0) * np.exp(-rho))
    assert m.kernel_type == "mt52" and abs(m(r1, r2, th) - want) < 1e-15
    assert define_kernel(dict(kernel_type="mt92", kernel_form="additive", input_dim=3, distance_func=False)).product_form
    with pytest.raises(NotImplementedError):
        define_kernel(dict(kernel_type="rq", kernel_form="product", input_dim=2, distance_func=False))
    with pytest.raises(NotImplementedError):
        define_kernel(dict(kernel_type="mt52", kernel_form="product", input_dim=3, distance_func=False))


class _FakeModel:
    """Quadratic 'likelihood' with a known gradient, standing in for a GP model on the CPU."""

    def __init__(self):
        self.calls = 0

    def value_and_grad(self, theta, r, y, eps, want_grad=True):
        self.calls += 1
        theta = np.asarray(theta)
        return float(np.sum((theta - 1.0) ** 2)), 2.0 * (theta - 1.0)

    def trainingFunction_all(self, theta, *args):
        return self.value_and_grad(theta, *args)[0]


def test_logposterior_and_prior_terms():
    from stopro_b200.sub_modules.loss_modules import hessian, logposterior

    m = _FakeModel()
    th = np.array([0.5, -0.25, 2.0])
    f = logposterior(m.trainingFunction_all, {"loss_ridge_regression": False})
    assert abs(f(th, None, None, 0.0) - (np.sum((th - 1) ** 2) + np.sum(th))) < 1e-15
    v, g = f.value_and_grad(th, None, None, 0.0)
    assert np.allclose(g, 2 * (th - 1) + 1.0)  # +1.0: gradient of the sum(theta) prior (gp.py:491-493)
    fr = logposterior(m.trainingFunction_all, {"loss_ridge_regression": True, "ridge_alpha": 0.1})
    assert abs(fr(th, None, None, 0.0) - (f(th, None, None, 0.0) + 0.1 * np.sum(np.exp(th) ** 2))) < 1e-14
    assert np.allclose(fr.grad(th, None, None, 0.0), g + 0.2 * np.exp(th) ** 2)
    hessian(f)  # construction must not fail (the reference never evaluates it)


def test_optimize_by_adam_matches_reference_semantics():
    from stopro_b200.solver.optimizers import optimize_by_adam
    from stopro_b200.sub_modules.loss_modules import logposterior

    m = _FakeModel()
    f = logposterior(m.trainingFunction_all, {"loss_ridge_regression": False})
    r_train = [np.zeros((3, 2)), np.zeros((2, 2))]  # ntraining = 5 (optimizers.py:131-139)
    po = dict(maxiter_GD=200, lr=0.05, eps=1e-12, maxiter_scipy=[0], method_GD="adam", method_scipy=["Nelder-Mead"],
              print_process=False, index_fixed=None)
    init = np.array([0.0, 2.0])
    opt, loss, theta, norms = optimize_by_adam(f, f.grad, None, init, po, r_train, None, 0.0)
    assert len(theta) == len(loss) == 201 and len(norms) == 200
    assert abs(loss[0] - f(init, r_train, None, 0.0) / 5) < 1e-15      # loss before optimize, normalised
    assert np.allclose(opt, 0.5, atol=1e-3)                            # argmin of (t-1)^2 + t
    # first Adam step moves every coordinate by lr against the gradient sign
    assert np.allclose(theta[1], init - 0.05 * np.sign(2 * (init - 1) + 1), atol=1e-6)
    # plateau stop: |dloss| < eps twice in a row (optimizers.py:224-229)
    po2 = dict(po, eps=1e-3, maxiter_GD=2000)
    _, loss2, _, _ = optimize_by_adam(f, f.grad, None, init, po2, r_train, None, 0.0)
    assert len(loss2) < 2001
    # NaN loss at the start raises, like the reference (optimizers.py:245-246)
    bad = logposterior(lambda th, *a: float("nan"), {"loss_ridge_regression": False})
    with pytest.raises(Exception):
        optimize_by_adam(bad, lambda th, *a: np.zeros_like(th), None, init, po, r_train, None, 0.0)
