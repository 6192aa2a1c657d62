"""optimize_by_adam with the reference's signature and stopping rules (solver/optimizers.py:94-263).

What is kept: normalisation of loss and gradient by the number of training points (:131-139), "loss before optimize"
as first loss entry and NaN guard (:239-246), the Adam update (optax.adam defaults: b1 = 0.9, b2 = 0.999,
eps = 1e-8), history lists of theta / loss / gradient norm, the two-in-a-row plateau stop on |delta loss| < eps
(:224-229) and the NaN guards on gradient and theta (:182-183, :230-232).  What differs: value and gradient come from
ONE factorisation (``f.value_and_grad`` of stopro_b200's logposterior) instead of func + dfunc assembling and
factorising K twice per step (:148-150); and when the loss is stopro_b200's logposterior over a GP model the whole loop
runs on the device (``_device_loop`` -> pigp_adam_host), the host loop below being the fallback.  The optional scipy pre-stage is delegated to scipy.optimize.minimize.
``optimize_by_adam_many`` runs optimize_by_adam from several starting points (multi-start fitting: the marginal
likelihood is not convex in theta); on the device all starts share one batched evaluation per iteration.
"""
import numpy as np


def _value_and_grad(f, df):
    if hasattr(f, "value_and_grad"):
        return f.value_and_grad
    if df is None:
        raise ValueError("a gradient function is required")
    return lambda p, *args: (f(p, *args), df(p, *args))


def _device_kwargs(f, df, params_optimization, ntraining, index_fixed, method):
    """Arguments of GPmodel.adam_device / adam_device_many, or None when the device loop does not apply: the loss is not
    stopro_b200's logposterior over a GP model, or there is a scipy pre-stage, print_process (per-step run.out lines) or
    params_optimization["device_loop"] = False."""
    model = getattr(f, "model", None)
    if (model is None or not hasattr(model, method) or not params_optimization.get("device_loop", True)
            or params_optimization.get("print_process", False) or not params_optimization.get("maxiter_GD")
            or (params_optimization.get("maxiter_scipy") or [0])[0]):
        return None
    # jit(grad(func)) differentiates the ridge term; the explicit-derivative scripts (df = gp.d_logposterior) drop it
    explicit = getattr(df, "__func__", None) is getattr(type(model), "d_logposterior", None) and df is not None
    return dict(max_iter=params_optimization["maxiter_GD"], lr=params_optimization["lr"], stop_eps=params_optimization["eps"],
                ntraining=ntraining, ridge_alpha=getattr(f, "ridge_alpha", 0.0), ridge_in_grad=not explicit,
                fixed=index_fixed or None)


def _device_loop(f, df, init, params_optimization, ntraining, index_fixed, args):
    """The whole Adam loop on the device (pigp_adam_host) when the loss is stopro_b200's logposterior over a GP model:
    theta, the moments and the histories stay in HBM, evaluation and update are enqueued back to back and the host only
    looks at the stop flag every few iterations.  Same lists and exceptions as the host loop below."""
    kw = _device_kwargs(f, df, params_optimization, ntraining, index_fixed, "adam_device")
    if kw is None:
        return None
    out = f.model.adam_device(init, *args, **kw)
    if out is None:
        return None
    theta_hist, loss_hist, norms, status = out
    print(f"loss before optimize: {loss_hist[0]}")
    if status == 4:
        raise Exception("loss is nan at the initial hyper-parameters")
    if status == 2:
        raise Exception("gradient of loss became nan")
    if status == 3:
        print("diverged")
        raise Exception("theta became nan")
    if status == 1:
        print("converged")
    theta = [t.copy() for t in theta_hist]
    return theta[-1], [float(v) for v in loss_hist], theta, [float(v) for v in norms]


def optimize_by_adam(f, df, hf, init, params_optimization, *args):
    maxiter_GD = params_optimization["maxiter_GD"]
    lr = params_optimization["lr"]
    eps = params_optimization["eps"]
    maxiter_scipy = params_optimization.get("maxiter_scipy", [0])
    method_scipy = params_optimization.get("method_scipy", [])
    print_process = params_optimization.get("print_process", False)
    index_fixed = params_optimization.get("index_fixed")
    if params_optimization.get("method_GD", "adam") != "adam":
        raise NotImplementedError("only method_GD == 'adam' is supported")

    r_train = args[0]
    ntraining = sum(np.shape(r)[0] for r in r_train)
    init = np.asarray(init, dtype=np.float64).copy()
    device = _device_loop(f, df, init, params_optimization, ntraining, index_fixed, args)
    if device is not None:
        return device
    vg = _value_and_grad(f, df)
    free = np.ones(len(init), dtype=bool)
    if index_fixed:
        free[np.asarray(index_fixed, dtype=int)] = False

    def value_and_grad(theta):
        v, g = vg(theta, *args)
        return v / ntraining, np.where(free, g, 0.0) / ntraining

    loss, theta, norms = [], [init.copy()], []
    loss_before = f(init, *args) / ntraining
    print(f"loss before optimize: {loss_before}")
    loss.append(loss_before)
    if np.isnan(loss_before):
        raise Exception("loss is nan at the initial hyper-parameters")

    if maxiter_scipy and maxiter_scipy[0]:
        from scipy.optimize import minimize

        x = theta[-1]
        for method, maxiter in zip(method_scipy, maxiter_scipy):
            res = minimize(lambda p: value_and_grad(p)[0], x, jac=(lambda p: value_and_grad(p)[1]) if method != "Nelder-Mead" else None,
                           method=method, options={"maxiter": maxiter})
            x = np.where(free, res.x, init)
            theta.append(x.copy())
            loss.append(float(res.fun))

    m, v = np.zeros_like(init), np.zeros_like(init)
    b1, b2, adam_eps = 0.9, 0.999, 1e-8
    converged_once = False
    for t in range(maxiter_GD):
        cur = theta[-1]
        value, grads = value_and_grad(cur)
        if np.any(np.isnan(grads)):
            raise Exception("gradient of loss became nan")
        m = b1 * m + (1.0 - b1) * grads
        v = b2 * v + (1.0 - b2) * grads * grads
        mhat, vhat = m / (1.0 - b1 ** (t + 1)), v / (1.0 - b2 ** (t + 1))
        new = cur - lr * mhat / (np.sqrt(vhat) + adam_eps)
        norms.append(float(np.linalg.norm(grads)))
        theta.append(new)
        loss.append(value)
        if print_process:
            with open("run.out", "a") as fh:
                fh.write(f"step{t:4} loss: {value:.4f} max_grad: {np.max(np.abs(grads)):.5f}, arg={np.argmax(np.abs(grads))}\n")
                fh.write(f"norm_of_grads: {norms[-1]:.5f}\n")
        if t < 1:
            continue
        if abs(loss[-1] - loss[-2]) < eps:
            if converged_once:
                print("converged")
                break
            converged_once = True
        elif np.any(np.isnan(theta[-1])):
            print("diverged")
            raise Exception("theta became nan")
        else:
            converged_once = False
    return theta[-1], loss, theta, norms


# device status of pigp_adam_host -> status of optimize_by_adam_many; the exception messages of optimize_by_adam
_STATUS = {0: "max_iter", 1: "converged", 2: "grad_nan", 3: "theta_nan", 4: "initial_nan"}
_RAISED = {"loss is nan at the initial hyper-parameters": "initial_nan", "gradient of loss became nan": "grad_nan",
           "theta became nan": "theta_nan"}


def optimize_by_adam_many(f, df, hf, inits, params_optimization, *args):
    """optimize_by_adam from every starting point in ``inits`` -> one (theta_final, loss, theta_hist, norms, status) per
    start, status one of "max_iter", "converged", "grad_nan", "theta_nan" and "initial_nan".  A start that
    optimize_by_adam would raise for reports that status with None in place of its results; no start raises.  On the
    device (GPmodel.adam_device_many) every start gets exactly the results optimize_by_adam gives it alone, from one
    batched evaluation per iteration; elsewhere optimize_by_adam runs once per start."""
    r_train = args[0]
    ntraining = sum(np.shape(r)[0] for r in r_train)
    inits = [np.asarray(x, dtype=np.float64).copy() for x in inits]
    index_fixed = params_optimization.get("index_fixed")
    kw = _device_kwargs(f, df, params_optimization, ntraining, index_fixed, "adam_device_many")
    outs = f.model.adam_device_many(inits, *args, **kw) if kw is not None else None
    if outs is not None:
        res = []
        for theta_hist, loss_hist, norms, status in outs:
            st = _STATUS[status]
            if st in _RAISED.values():
                res.append((None, None, None, None, st))
                continue
            theta = [t.copy() for t in theta_hist]
            res.append((theta[-1], [float(v) for v in loss_hist], theta, [float(v) for v in norms], st))
        return res
    res = []
    eps = params_optimization["eps"]
    for x in inits:
        try:
            theta_final, loss, theta, norms = optimize_by_adam(f, df, hf, x, params_optimization, *args)
        except Exception as e:
            if str(e) not in _RAISED:
                raise
            res.append((None, None, None, None, _RAISED[str(e)]))
            continue
        # the loop stops early only on the two-in-a-row plateau rule, checked from the third step on
        conv = len(norms) >= 3 and abs(loss[-1] - loss[-2]) < eps and abs(loss[-2] - loss[-3]) < eps
        res.append((theta_final, loss, theta, norms, "converged" if conv else "max_iter"))
    return res
