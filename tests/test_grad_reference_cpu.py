"""The gradient reference of the GPU regime tests (tests/test_gpu_regimes.py::closed_form_grad) evaluates the oracle's
closed-form dK/dtheta block by block with torch.  Here it runs on the CPU against the numpy oracle's own gradient
(oracle.gp_ref.GPRef.d_trainingFunction_all) on the same matrix."""
import numpy as np
import torch

from conftest import oracle_for
from stopro_b200 import synthetic
from test_gpu_regimes import closed_form_grad


def test_closed_form_grad_matches_the_oracle():
    cfg = dict(synthetic.stokes2d_scaling(300, n_test=8), eps=1.0)
    ref = oracle_for(cfg)
    th = cfg["theta0"] + 0.05 * np.random.default_rng(11).standard_normal(len(cfg["theta0"]))
    r, y = cfg["r_train"], cfg["delta_y"]
    S = torch.as_tensor(ref.training_sigma(th, r, cfg["eps"]))
    L = torch.linalg.cholesky(S)
    Kinv = torch.cholesky_inverse(L)
    alpha = Kinv @ torch.as_tensor(y)
    got = closed_form_grad(cfg, th, Kinv - torch.outer(alpha, alpha))
    want = ref.d_trainingFunction_all(th, r, y, cfg["eps"])
    e = np.max(np.abs(got - want)) / np.max(np.abs(want))
    print(f"\n[closed-form gradient reference, N = 300] {e:.1e} (bar 1e-12)")
    assert e <= 1e-12
