"""optimize_by_adam_many through its host fallback (no GP model behind the loss): one optimize_by_adam per start, every
start's results equal to optimize_by_adam from it alone, and the failures optimize_by_adam raises for reported as a
status instead."""
import numpy as np

from stopro_b200.solver.optimizers import optimize_by_adam, optimize_by_adam_many

CENTRE = np.array([0.5, -1.0, 2.0])


def loss(p, r, y, eps):
    """A non-convex loss with several minima (cosine ripple on a quadratic bowl)."""
    return float(np.sum(np.cos(3.0 * p) + (p - CENTRE) ** 2))


def grad(p, r, y, eps):
    return -3.0 * np.sin(3.0 * p) + 2.0 * (p - CENTRE)


def _args():
    return ([np.zeros((40, 2)), np.zeros((24, 2))], np.zeros(64), 1e-6)


def test_optimize_by_adam_many_host_fallback():
    po = dict(maxiter_GD=300, lr=5e-2, eps=1e-7, index_fixed=None)
    inits = [np.array([0.0, 0.0, 0.0]), np.array([2.0, -3.0, 1.0]), np.array([np.nan, 0.0, 0.0]), np.array([-1.0, 1.0, 3.0])]
    many = optimize_by_adam_many(loss, grad, None, inits, po, *_args())
    assert len(many) == len(inits)
    assert many[2] == (None, None, None, None, "initial_nan")
    statuses = set()
    for b, x in enumerate(inits):
        if b == 2:
            continue
        ref = optimize_by_adam(loss, grad, None, x, po, *_args())
        theta_final, losses, theta, norms, status = many[b]
        assert np.array_equal(theta_final, ref[0]) and losses == ref[1] and norms == ref[3]
        assert len(theta) == len(ref[2]) and all(np.array_equal(a, r) for a, r in zip(theta, ref[2]))
        assert status == ("converged" if len(norms) < po["maxiter_GD"] else "max_iter")
        statuses.add(status)
    assert statuses == {"converged"}


def test_optimize_by_adam_many_reports_max_iter_and_keeps_index_fixed():
    po = dict(maxiter_GD=20, lr=1e-2, eps=1e-12, index_fixed=[1])
    inits = [np.array([0.1, 0.2, 0.3]), np.array([1.0, 1.5, -0.5])]
    many = optimize_by_adam_many(loss, grad, None, inits, po, *_args())
    for b, x in enumerate(inits):
        ref = optimize_by_adam(loss, grad, None, x, po, *_args())
        assert many[b][4] == "max_iter" and len(many[b][3]) == 20
        assert np.array_equal(many[b][0], ref[0]) and many[b][0][1] == x[1]
