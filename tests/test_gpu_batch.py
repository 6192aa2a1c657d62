"""GPU tests of the batched evaluation (pigp_nll_grad_batch / _host, Solver.nll_grad_batch_host, GPmodel.value_and_grad_many)
and of multi-start Adam (pigp_adam_batch_host, optimize_by_adam_many).

A batch runs every launch of the world-1 schedule once, with one grid dimension more for the slot, and makes every kernel
and schedule choice from the shape of one slot.  So each slot must equal the single-theta call of its theta bit for bit,
whatever the batch size.  The reference is always a second, fresh model whose solver evaluates the slots' thetas one
after another through pigp_nll_grad / pigp_nll.  The tile counts T cross the early-K^-1 window (8 <= T <= 32) and every
look-ahead width of both the NLL-only rule (0 / 2 / 4 below T = 12 / 64 / 128) and the gradient rule (2 for 16 <= T < 32,
4 for 32 <= T < 96)."""
import ctypes as C

import numpy as np
import pytest

from stopro_b200 import _lib, synthetic
from stopro_b200.plan import Solver
from stopro_b200.solver.optimizers import optimize_by_adam, optimize_by_adam_many
from stopro_b200.sub_modules.loss_modules import logposterior
from test_gpu_regimes import _n_for, _nll_dev

pytestmark = pytest.mark.gpu

EINVAL = -1  # PIGP_EINVAL
BATCH_T = [1, 4, 8, 10, 12, 16, 21, 32, 33, 64]


def _model(cfg):
    gp = synthetic.make_model(cfg)
    gp.set_constants(cfg["r_train"], cfg["delta_y"], cfg["eps"], only_training=True)
    return gp


def _thetas(theta0, nb, seed, scale=0.05):
    rng = np.random.default_rng(seed)
    return [np.asarray(theta0, dtype=np.float64) + scale * rng.standard_normal(len(theta0)) for _ in range(nb)]


def _stokes(T):
    return dict(synthetic.stokes2d_scaling(_n_for(T), n_test=8), eps=1.0)


def _kinds():
    """SE product and additive, 3-D, Matern 5/2, a noise parameter, shift wrappers."""
    se = dict(synthetic.stokes2d_scaling(600, seed=2, n_test=8), eps=1e-3)
    add = dict(se, kernel=dict(se["kernel"], kernel_form="additive"))
    mat = dict(synthetic.stokes2d_scaling(400, seed=5, n_test=8), eps=1e-3)
    rng = np.random.default_rng(6)
    mat["r_train"] = [rng.random((n, 2)) for n in (150, 121, 129)]
    mat["delta_y"] = rng.standard_normal(400)
    mat["kernel"] = dict(mat["kernel"], kernel_type="mt52")
    mat["theta0"] = np.tile([0.0, np.log(0.3), np.log(0.4)], 3)
    return {
        "se_product": se,
        "se_additive": add,
        "drag3d": dict(synthetic.drag3d(n_u=5, n_f=4, n_test=14), eps=1e-3),
        "matern52": mat,
        "sin1d_noise": synthetic.sin_1d_naive(n=150, n_test=8),
        "sinusoidal_shift": dict(synthetic.sinusoidal(u_num=20, f_nx=16, f_ny=8, dif_num=10, n_test=12), eps=1e-3),
    }


def _singles(gp, cfg, thetas, want_grad):
    """Each theta through pigp_nll_grad / pigp_nll of gp's solver, one after another -> (nll (B,), grad (B, P), info (B,))."""
    import torch

    solver = gp._solver_for(cfg["r_train"])
    y = torch.as_tensor(np.asarray(cfg["delta_y"], dtype=np.float64), device="cuda")
    out = [_nll_dev(solver, th, y, cfg["eps"], want_grad) for th in thetas]
    return (np.array([o[0] for o in out]), np.stack([o[1] for o in out]) if want_grad else None,
            np.array([o[2] for o in out], dtype=np.int32))


def _same(a, b):
    """Bitwise equality of float arrays (NaN payloads included)."""
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def _check_batches(cfg, sizes, seed, label):
    gp, fresh = _model(cfg), _model(cfg)
    try:
        solver = gp._solver_for(cfg["r_train"])
        thetas = _thetas(cfg["theta0"], max(sizes), seed)
        for want_grad in (False, True):
            ref = _singles(fresh, cfg, thetas, want_grad)
            for nb in sizes:
                nll, grad, info = solver.nll_grad_batch_host(thetas[:nb], cfg["delta_y"], cfg["eps"], want_grad=want_grad)
                assert np.all(info == 0) and np.array_equal(info, ref[2][:nb])
                assert _same(nll, ref[0][:nb]), f"{label} B={nb} grad={want_grad}: NLL differs from the single calls"
                assert want_grad == (grad is not None)
                if want_grad:
                    assert _same(grad, ref[1][:nb]), f"{label} B={nb}: gradient differs from the single calls"
        print(f"\n[{label}] B = {sizes}, NLL only and NLL + gradient: every slot bitwise equal to its single call")
    finally:
        gp.close()
        fresh.close()


@pytest.mark.parametrize("T", BATCH_T)
def test_batch_equals_single_calls(cuda_device, T):
    _check_batches(_stokes(T), [1, 2, 3, 7] + ([33] if T <= 16 else []), T, f"T={T}")


@pytest.mark.parametrize("kind", list(_kinds()))
def test_batch_equals_single_calls_per_model_class(cuda_device, kind):
    _check_batches(_kinds()[kind], [1, 3], 7, kind)


def test_failed_slots_leave_their_neighbours_alone(cuda_device):
    """Two failing slots among good ones, with eps = 1e-6.  Slot 2 is not positive definite in floating point: its pressure
    group has variance e^30 and length scale e^2 (far beyond the unit square), so the pressure block is numerically of
    low rank and its Schur complements are rounding noise of order e^30 u >> eps; the first non-positive pivot lies in the
    pressure rows, past tile 0.  Slot 4 has a NaN length scale.  Each reports the info and the NaN results of its single
    call, every other slot is unchanged bit for bit.  Afterwards the same solver's single call, a smaller batch and a larger
    batch all equal a fresh solver."""
    cfg = dict(_stokes(16), eps=1e-6)
    gp, fresh = _model(cfg), _model(cfg)
    try:
        solver = gp._solver_for(cfg["r_train"])
        thetas = _thetas(cfg["theta0"], 9, 3)
        bad = [t.copy() for t in thetas[:6]]
        bad[2][6:9] = [30.0, 2.0, 2.0]
        bad[4][1] = np.nan
        for want_grad in (True, False):
            nll, grad, info = solver.nll_grad_batch_host(bad, cfg["delta_y"], cfg["eps"], want_grad=want_grad)
            ref = _singles(fresh, cfg, bad, want_grad)
            print(f"\n[failed slots T=16 grad={want_grad}] info {info.tolist()} (single calls {ref[2].tolist()})")
            assert np.array_equal(info, ref[2]) and np.nonzero(info)[0].tolist() == [2, 4]
            assert info[2] > 128 and info[4] > 0  # slot 2 fails in a later tile than the first
            assert np.isnan(nll[2]) and np.isnan(nll[4])
            assert _same(nll, ref[0]) and (not want_grad or _same(grad, ref[1]))
            if want_grad:
                assert np.all(np.isnan(grad[[2, 4]]))
        ref = _singles(fresh, cfg, thetas, True)
        one = _singles(gp, cfg, thetas[:1], True)
        assert _same(one[0], ref[0][:1]) and _same(one[1], ref[1][:1])
        for nb in (3, 9):
            nll, grad, info = solver.nll_grad_batch_host(thetas[:nb], cfg["delta_y"], cfg["eps"])
            assert np.all(info == 0) and _same(nll, ref[0][:nb]) and _same(grad, ref[1][:nb])
    finally:
        gp.close()
        fresh.close()


def test_device_entry_on_a_side_stream_equals_host_entry(cuda_device):
    """The first batched call of a fresh solver goes through the device entry point on a non-default stream, so the batch
    workspace is allocated and zeroed by that call; it equals the host entry point and the single calls."""
    import torch

    cfg = _stokes(12)
    gp, fresh = _model(cfg), _model(cfg)
    try:
        solver = gp._solver_for(cfg["r_train"])
        thetas = _thetas(cfg["theta0"], 5, 4)
        P = len(thetas[0])
        th = torch.as_tensor(np.stack(thetas), device=cuda_device)
        y = torch.as_tensor(np.asarray(cfg["delta_y"], dtype=np.float64), device=cuda_device)
        nll = torch.full((5,), float("nan"), dtype=torch.float64, device=cuda_device)
        grad = torch.full((5, P), float("nan"), dtype=torch.float64, device=cuda_device)
        info = torch.full((5,), -7, dtype=torch.int32, device=cuda_device)
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            solver.nll_grad_batch(5, th.data_ptr(), y.data_ptr(), cfg["eps"], nll.data_ptr(), grad.data_ptr(), info.data_ptr(),
                                  C.c_void_p(stream.cuda_stream))
        stream.synchronize()
        nll_h, grad_h, info_h = solver.nll_grad_batch_host(thetas, cfg["delta_y"], cfg["eps"])
        ref = _singles(fresh, cfg, thetas, True)
        assert _same(nll.cpu().numpy(), nll_h) and _same(grad.cpu().numpy(), grad_h)
        assert np.array_equal(info.cpu().numpy(), info_h) and np.all(info_h == 0)
        assert _same(nll_h, ref[0]) and _same(grad_h, ref[1])
    finally:
        gp.close()
        fresh.close()


@pytest.mark.parametrize("want_grad", [False, True])
def test_batch_is_one_pass(cuda_device, want_grad):
    """pigp_launch_count grows by as much for a 6-slot call as for one single-theta call at the same N."""
    cfg = _stokes(21)
    gp = _model(cfg)
    try:
        solver = gp._solver_for(cfg["r_train"])
        thetas = _thetas(cfg["theta0"], 6, 5)
        solver.nll_grad_batch_host(thetas, cfg["delta_y"], cfg["eps"], want_grad=want_grad)  # workspace grown
        n0 = _lib.launch_count()
        solver.nll_grad_host(thetas[0], cfg["delta_y"], cfg["eps"], want_grad=want_grad)
        n1 = _lib.launch_count()
        solver.nll_grad_batch_host(thetas, cfg["delta_y"], cfg["eps"], want_grad=want_grad)
        n2 = _lib.launch_count()
        print(f"\n[one pass T=21 grad={want_grad}] single call {n1 - n0} launches, 6 slots {n2 - n1}")
        assert n1 - n0 == n2 - n1 > 0
    finally:
        gp.close()


def test_rejections_before_any_launch(cuda_device):
    import torch

    cfg = _stokes(4)
    gp = _model(cfg)
    plan = gp._training_plan(cfg["r_train"])
    sharded = Solver(plan, 0, 2)  # in-process world-2 rank: a batch is refused before anything else is looked at
    try:
        solver = gp._solver_for(cfg["r_train"])
        L = _lib.lib()
        P = plan.theta_len
        th = torch.zeros((2, P), dtype=torch.float64, device=cuda_device)
        y = torch.as_tensor(np.asarray(cfg["delta_y"], dtype=np.float64), device=cuda_device)
        out = torch.zeros(2 * (P + 1), dtype=torch.float64, device=cuda_device)
        h_th = np.zeros((2, P))
        h_y = np.asarray(cfg["delta_y"], dtype=np.float64)
        h_out = np.zeros(2 * (P + 1))
        h_n, h_s = np.zeros(2, dtype=np.int32), np.zeros(2, dtype=np.int32)
        t, yp, o = th.data_ptr(), y.data_ptr(), out.data_ptr()
        ht, hy, ho = h_th.ctypes.data, h_y.ctypes.data, h_out.ctypes.data
        adam = lambda s, n, t0: L.pigp_adam_batch_host(s, n, t0, hy, 1.0, 4, 1e-2, 0.0, 100.0, 0.0, 1, None, 2, ho, ho, ho,
                                                       h_n.ctypes.data, h_s.ctypes.data)
        calls = {
            "n_theta = 0": lambda: L.pigp_nll_grad_batch(solver.handle, 0, t, yp, 1.0, o, o, None, None),
            "n_theta = 65536": lambda: L.pigp_nll_grad_batch(solver.handle, 65536, t, yp, 1.0, o, o, None, None),
            "null solver": lambda: L.pigp_nll_grad_batch(None, 2, t, yp, 1.0, o, o, None, None),
            "null thetas": lambda: L.pigp_nll_grad_batch(solver.handle, 2, None, yp, 1.0, o, o, None, None),
            "null y": lambda: L.pigp_nll_grad_batch(solver.handle, 2, t, None, 1.0, o, o, None, None),
            "null nll": lambda: L.pigp_nll_grad_batch(solver.handle, 2, t, yp, 1.0, None, o, None, None),
            "world 2": lambda: L.pigp_nll_grad_batch(sharded.handle, 2, t, yp, 1.0, o, o, None, None),
            "host n_theta = 0": lambda: L.pigp_nll_grad_batch_host(solver.handle, 0, ht, hy, 1.0, 1, ho, ho, None),
            "host n_theta = 65536": lambda: L.pigp_nll_grad_batch_host(solver.handle, 65536, ht, hy, 1.0, 1, ho, ho, None),
            "host null thetas": lambda: L.pigp_nll_grad_batch_host(solver.handle, 2, None, hy, 1.0, 1, ho, ho, None),
            "host null grad": lambda: L.pigp_nll_grad_batch_host(solver.handle, 2, ht, hy, 1.0, 1, ho, None, None),
            "host world 2": lambda: L.pigp_nll_grad_batch_host(sharded.handle, 2, ht, hy, 1.0, 1, ho, ho, None),
            "adam n_start = 0": lambda: adam(solver.handle, 0, ht),
            "adam n_start = 65536": lambda: adam(solver.handle, 65536, ht),
            "adam null theta0s": lambda: adam(solver.handle, 2, None),
            "adam world 2": lambda: adam(sharded.handle, 2, ht),
        }
        torch.cuda.synchronize()
        for what, call in calls.items():
            n0 = _lib.launch_count()
            rc = call()
            assert rc == EINVAL and _lib.launch_count() == n0, f"{what}: rc {rc}"
    finally:
        sharded.close()
        gp.close()


ADAM_ARGS = dict(max_iter=24, lr=2e-2, check_every=4)


def _adam_case(cfg, gp, fresh, thetas, stop_eps, fixed):
    kw = dict(ADAM_ARGS, stop_eps=stop_eps, ntraining=float(len(cfg["delta_y"])), fixed=fixed)
    many = gp._solver_for(cfg["r_train"]).adam_batch_host(thetas, cfg["delta_y"], cfg["eps"], **kw)
    one = fresh._solver_for(cfg["r_train"])
    for b, th in enumerate(thetas):
        ref = one.adam_host(th, cfg["delta_y"], cfg["eps"], **kw)
        assert many[b][3] == ref[3], f"start {b}: status {many[b][3]} vs {ref[3]}"
        for x, r in zip(many[b][:3], ref[:3]):
            assert _same(x, r), f"start {b}: histories differ ({len(x)} vs {len(r)} entries)"
    return [m[3] for m in many], [len(m[2]) for m in many]


def test_multi_start_adam_equals_single_runs(cuda_device):
    """Each start's theta, loss and gradient-norm histories, iteration count and status equal pigp_adam_host from that
    start alone: with a plateau threshold at which the first start converges early while others keep going, with
    index_fixed, and with a start whose initial loss is NaN."""
    cfg = _stokes(10)
    thetas = _thetas(cfg["theta0"], 4, 8, scale=0.2)
    thetas.insert(2, np.full_like(thetas[0], np.nan))  # NaN initial loss
    gp, fresh = _model(cfg), _model(cfg)
    try:
        # a threshold that start 0 crosses two steps in a row by step 10: it converges there
        probe = fresh._solver_for(cfg["r_train"]).adam_host(thetas[0], cfg["delta_y"], cfg["eps"],
                                                            **dict(ADAM_ARGS, stop_eps=0.0, ntraining=float(len(cfg["delta_y"]))))
        d = np.abs(np.diff(probe[1][1:]))
        stop_eps = float(np.max(d[8:10])) * (1.0 + 1e-9)
        status, n_done = _adam_case(cfg, gp, fresh, thetas, stop_eps, None)
        print(f"\n[multi-start adam, plateau {stop_eps:.2e}] status {status} iterations {n_done}")
        # start 0 stops early and stays frozen while the others go on to their own stopping steps
        assert status[0] == 1 and n_done[0] <= 11 and status[2] == 4 and len(set(n_done[:2] + n_done[3:])) > 1
        status, n_done = _adam_case(cfg, gp, fresh, thetas, 0.0, [0, 4])
        print(f"[multi-start adam, index_fixed] status {status} iterations {n_done}")
        assert status == [0, 0, 4, 0, 0] and n_done == [24, 24, 0, 24, 24]
    finally:
        gp.close()
        fresh.close()


def test_single_start_adam_on_a_sharded_solver(cuda_device):
    """pigp_adam_host (the one-start case of pigp_adam_batch_host) runs on sharded solvers as before: two in-process ranks of
    a world-2 solver, one host thread each, give the same histories bit for bit, and agree with the single-GPU run."""
    import threading

    cfg = _stokes(10)
    gp = _model(cfg)
    plan = gp._training_plan(cfg["r_train"])
    ranks = [Solver(plan, k, 2) for k in range(2)]
    try:
        L = _lib.lib()
        slabs = []
        for r in ranks:
            ptr, nbytes = C.c_void_p(), C.c_int64()
            _lib.check(L.pigp_dsolver_slab(r._ds, C.byref(ptr), C.byref(nbytes)))
            slabs.append(ptr.value)
        for r in ranks:
            _lib.check(L.pigp_dsolver_connect(r._ds, (C.c_void_p * 2)(*[C.c_void_p(p) for p in slabs])))
        theta0 = _thetas(cfg["theta0"], 1, 12, scale=0.2)[0]
        kw = dict(ADAM_ARGS, stop_eps=0.0, ntraining=float(len(cfg["delta_y"])), fixed=[1])
        out = [None, None]

        def work(k):
            try:
                out[k] = ranks[k].adam_host(theta0, cfg["delta_y"], cfg["eps"], **kw)
            except Exception as exc:  # noqa: BLE001
                out[k] = exc

        threads = [threading.Thread(target=work, args=(k,)) for k in range(2)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for o in out:
            if isinstance(o, Exception):
                raise o
        ref = gp._solver_for(cfg["r_train"]).adam_host(theta0, cfg["delta_y"], cfg["eps"], **kw)
        assert out[0][3] == out[1][3] == ref[3] == 0
        for x, y in zip(out[0][:3], out[1][:3]):
            assert _same(x, y)
        assert len(out[0][2]) == ADAM_ARGS["max_iter"] and np.all(out[0][0][:, 1] == theta0[1])
        e_loss = np.max(np.abs(out[0][1] - ref[1]) / np.abs(ref[1]))
        e_theta = np.max(np.abs(out[0][0] - ref[0]))
        print(f"\n[adam world 2] {len(out[0][2])} iterations; vs one GPU: loss {e_loss:.1e}, theta {e_theta:.1e}")
        assert e_loss < 1e-7 and e_theta < 1e-7
    finally:
        for r in ranks:
            r.close()
        gp.close()


def test_optimize_by_adam_many_on_a_logposterior(cuda_device):
    cfg = dict(synthetic.poiseuille(u_num=7, p_num=7, f_num=8, n_test=4, kernel_form="product"), eps=1e-4)
    po = dict(maxiter_GD=30, lr=1e-2, eps=1e-6, loss_ridge_regression=False, index_fixed=None)
    gp = _model(cfg)
    try:
        args = (cfg["r_train"], cfg["delta_y"], cfg["eps"])
        f = logposterior(gp.trainingFunction_all, po)
        inits = _thetas(cfg["theta0"], 3, 9, scale=0.1)
        bad = cfg["theta0"].copy()
        bad[1] = np.nan  # the initial loss is NaN
        inits.insert(1, bad)
        many = optimize_by_adam_many(f, f.grad, None, inits, dict(po, device_loop=True), *args)
        assert many[1][:4] == (None, None, None, None) and many[1][4] == "initial_nan"
        for b, x in enumerate(inits):
            if b == 1:
                with pytest.raises(Exception, match="initial"):
                    optimize_by_adam(f, f.grad, None, x, dict(po, device_loop=True), *args)
                continue
            ref = optimize_by_adam(f, f.grad, None, x, dict(po, device_loop=True), *args)
            theta_final, loss, theta, norms, status = many[b]
            assert _same(theta_final, ref[0]) and loss == ref[1] and norms == ref[3]
            assert all(_same(a, r) for a, r in zip(theta, ref[2])) and len(theta) == len(ref[2])
            assert status == ("max_iter" if len(norms) == po["maxiter_GD"] else "converged")
    finally:
        gp.close()


def test_value_and_grad_many(cuda_device):
    """GPmodel.value_and_grad_many: rows equal value_and_grad bit for bit, including the zero gradient of the dropped
    cross-covariance entries of a longer caller theta; the value_and_grad cache stays valid."""
    cfg = _stokes(4)
    gp = _model(cfg)
    try:
        args = (cfg["r_train"], cfg["delta_y"], cfg["eps"])
        thetas = _thetas(cfg["theta0"], 3, 10)
        longer = [np.append(t, [0.3, -0.2, 0.1]) for t in thetas]
        first = gp.value_and_grad(thetas[0], *args)
        calls = gp._solver_for(cfg["r_train"])
        for ths in (thetas, longer):
            nll, grad = gp.value_and_grad_many(ths, *args)
            for b, t in enumerate(ths):
                v, g = gp.value_and_grad(t, *args)
                assert nll[b] == v and _same(grad[b], g)
            assert grad.shape == (3, len(ths[0]))
        nll, grad = gp.value_and_grad_many(thetas, *args, want_grad=False)
        assert grad is None and nll.shape == (3,)
        # the cache: value_and_grad(thetas[0]) is served without an evaluation after a batch
        gp.value_and_grad(thetas[0], *args)
        gp.value_and_grad_many(thetas[1:], *args)
        n0 = _lib.launch_count()
        again = gp.value_and_grad(thetas[0], *args)
        assert _lib.launch_count() == n0 and again[0] == first[0] and _same(again[1], first[1])
        assert calls is gp._solver_for(cfg["r_train"])
    finally:
        gp.close()
