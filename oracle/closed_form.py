"""Closed-form numpy restatement of the reference's autodiff operators.

The reference (GP/gp_2D.py:16-86, GP/gp_3D.py:12-35, GP/gp_1D_laplacian.py:35-46)
obtains every operator by automatic differentiation of the squared-exponential
kernels of GP/kernels.py:36-77.  For those kernels the derivatives are known in
closed form.  With s = r_d - r'_d, a = exp(-2 logl_d), E = exp(-a s^2 / 2):

    (d/ds)^n E = g_n(s, a) E,   g0 = 1, g1 = -a s, g2 = a^2 s^2 - a,
                                g3 = -a^3 s^3 + 3 a^2 s, g4 = a^4 s^4 - 6 a^3 s^2 + 3 a^2

d/dr_d = d/ds and d/dr'_d = -d/ds.  An operator is a polynomial in
(d/dr, d/dr'); a monomial with orders (alpha, beta) applied to
  product  k = gamma prod_d E_d  gives  (-1)^|beta| gamma prod_d G_{alpha_d+beta_d}^d
  additive k = gamma sum_d E_d   gives  (-1)^|beta| gamma G_n^e if all derivatives
           fall on one dimension e, gamma sum_d E_d if there are none, else 0.

``oracle.autodiff_ops`` (the literal restatement) is the check for this file:
tests/test_oracle.py compares every operator, both forms, 1-/2-/3-D.
This is test infrastructure (see oracle/__init__.py).  eval_operator also takes torch tensors for the points (same
formulas, float64 on their device), so that large float64 references can be evaluated on a GPU.
"""
import itertools

import numpy as np


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _exp_for(x):
    if _is_torch(x):
        import torch

        return torch.exp
    return np.exp


def _prod(factors):
    out = factors[0]
    for f in factors[1:]:
        out = out * f
    return out


def _stack(arrs):
    if _is_torch(arrs[0]):
        import torch

        return torch.stack(arrs)
    return np.stack(arrs)


def _e(i, dim):
    v = [0] * dim
    v[i] = 1
    return tuple(v)


def _add(*vs):
    return tuple(sum(c) for c in zip(*vs))


def operator_polynomial(name, dim):
    """name -> list of (coef, alpha, beta); alpha/beta are per-dimension derivative orders."""
    z = (0,) * dim
    two = [tuple(2 * c for c in _e(d, dim)) for d in range(dim)]
    if name == "K":
        return [(1.0, z, z)]
    if name in ("L0", "L0K"):
        return [(1.0, two[d], z) for d in range(dim)]
    if name in ("L1", "L1K"):
        return [(1.0, z, two[d]) for d in range(dim)]
    if name in ("LL", "LLK"):
        return [(1.0, two[d], two[f]) for d in range(dim) for f in range(dim)]
    if len(name) == 3 and name[0] == "d" and name[1] in "01" and name[2].isdigit():
        i = int(name[2])  # d0i = d/dr_i, d1i = d/dr'_i
        return [(1.0, _e(i, dim), z)] if name[1] == "0" else [(1.0, z, _e(i, dim))]
    if len(name) == 4 and name[0] == "d" and name[2] == "d":
        return [(1.0, _e(int(name[1]), dim), _e(int(name[3]), dim))]  # didj = d/dr_i d/dr'_j
    if len(name) == 3 and name[0] == "d" and name[2] == "L":
        return [(1.0, _e(int(name[1]), dim), two[d]) for d in range(dim)]  # diL = d/dr_i Lap_r'
    if len(name) == 3 and name[:2] == "Ld":
        return [(1.0, two[d], _e(int(name[2]), dim)) for d in range(dim)]  # Ldi = Lap_r d/dr'_i
    raise KeyError(name)


def _g(n, s, a):
    t = a * s * s
    if n == 0:
        return s * 0.0 + 1.0
    if n == 1:
        return -a * s
    if n == 2:
        return a * (t - 1.0)
    if n == 3:
        return a * a * s * (3.0 - t)
    if n == 4:
        return a * a * (t * t - 6.0 * t + 3.0)
    raise ValueError(n)


def _dg_da(n, s, a):
    """d g_n / d a."""
    s2 = s * s
    if n == 0:
        return s * 0.0
    if n == 1:
        return -s
    if n == 2:
        return 2.0 * a * s2 - 1.0
    if n == 3:
        return -3.0 * a * a * s2 * s + 6.0 * a * s
    if n == 4:
        return 4.0 * a ** 3 * s2 * s2 - 18.0 * a * a * s2 + 6.0 * a
    raise ValueError(n)


def _prep(r, rp, dim, dtype=np.float64):
    if not _is_torch(r):
        r = np.asarray(r, dtype=dtype)
        rp = np.asarray(rp, dtype=dtype)
    if dim == 1:
        r = r.reshape(-1, 1)
        rp = rp.reshape(-1, 1)
    return [r[:, None, d] - rp[None, :, d] for d in range(dim)]


def eval_operator(name, r, rp, theta, form, dim, with_grad=False, dtype=np.float64):
    """Dense block of operator ``name`` on points r (n,dim), rp (m,dim).

    theta = [log gamma, logl_0 .. logl_{dim-1}].  With ``with_grad`` also returns
    d block / d theta as an array (1+dim, n, m).  ``dtype=np.longdouble`` evaluates the same formulas in extended
    precision (the higher-precision truth of oracle/extended.py).
    """
    theta = np.asarray(theta, dtype=dtype)
    gamma = np.exp(theta[0])
    a = np.exp(-2.0 * theta[1:1 + dim])
    if _is_torch(r):  # plain floats: a numpy scalar on the left of a tensor product would convert the tensor
        gamma, a = float(gamma), [float(x) for x in a]
    s = _prep(r, rp, dim, dtype)
    exp = _exp_for(s[0])
    E = [exp(-0.5 * a[d] * s[d] * s[d]) for d in range(dim)]

    def G(n, d):
        return _g(n, s[d], a[d]) * E[d]

    def dG_dlogl(n, d):
        # d/dlogl = -2a d/da ; d(g E)/da = (dg/da - s^2/2 g) E
        return -2.0 * a[d] * (_dg_da(n, s[d], a[d]) - 0.5 * s[d] * s[d] * _g(n, s[d], a[d])) * E[d]

    val = s[0] * 0.0
    grad = [s[0] * 0.0 for _ in range(1 + dim)] if with_grad else None
    for coef, alpha, beta in operator_polynomial(name, dim):
        sign = coef * (-1.0) ** sum(beta)
        order = _add(alpha, beta)
        if form == "product":
            factors = [G(order[d], d) for d in range(dim)]
            term = sign * gamma * _prod(factors)
            val += term
            if with_grad:
                grad[0] += term
                for e in range(dim):
                    others = [factors[d] for d in range(dim) if d != e]
                    rest = _prod(others) if others else 1.0
                    grad[1 + e] += sign * gamma * dG_dlogl(order[e], e) * rest
        elif form == "additive":
            active = [d for d in range(dim) if order[d] > 0]
            if len(active) == 0:
                for d in range(dim):
                    term = sign * gamma * G(0, d)
                    val += term
                    if with_grad:
                        grad[0] += term
                        grad[1 + d] += sign * gamma * dG_dlogl(0, d)
            elif len(active) == 1:
                e = active[0]
                term = sign * gamma * G(order[e], e)
                val += term
                if with_grad:
                    grad[0] += term
                    grad[1 + e] += sign * gamma * dG_dlogl(order[e], e)
        else:
            raise ValueError(form)
    if with_grad:
        grad = _stack(grad)
    return (val, grad) if with_grad else val
