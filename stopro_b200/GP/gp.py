"""GPmodel: the reference's base-class interface (GP/gp.py) over the CUDA path.

Same public methods, argument meaning and failure behaviour as /root/reference/GP/gp.py:
  set_constants :263-285, trainingK_all / mixedK_all / testK_all :287-306, trainingFunction_all :213-224,
  predictingFunction_all :226-256, d_trainingFunction_all :412-488, d_logposterior :491-493,
  setup_Ks_dKdtheta :322-330 (kept as a no-op: dK/dtheta is evaluated in closed form inside the gradient kernel).
Inputs are lists of per-variable point arrays, flat delta_y and a log-space theta; outputs are numpy float64.
A non-positive-definite K gives NaN (as jnp.linalg.cholesky does), never an exception.

A model is a list of *observables* per training / test block (see stopro_b200.operators); the block functions of
the reference's library (Kuxux, Kfxdiv, Kuxdifux, ...) are available by name through ``model.K<a><b>(r, rp, theta)``.
"""
import os

import numpy as np

from .. import _lib, operators
from ..plan import Plan, Solver


class GPmodel:
    #: names of the observables per training / test block, in block order; set by subclasses
    train_observables = ()
    test_observables = ()
    system = "stokes"  # "stokes" | "scalar"
    #: (i, j), i <= j, blocks of the test table that the reference fills with a zero block although the observables
    #: are correlated (kept quirks, e.g. gp_sinusoidal_infer_difp.py:97)
    test_zero_blocks = frozenset()

    def __init__(self, Kernel=None, index_optimize_noise=None, lbox=None, distributed=None, process_group=None):
        """``distributed`` (not part of the reference's signature; default: the STOPRO_B200_DISTRIBUTED environment
        variable): when true and a torch.distributed process group with more than one rank is up (one process per GPU,
        e.g. under torchrun), K is dealt block-cyclically over the ranks and every rank must make the same sequence of
        calls; all ranks receive identical results.  The YAML schema is untouched (SURVEY.md 5.6)."""
        if Kernel is None:
            raise ValueError("Kernel is required (use stopro_b200.GP.kernels.define_kernel)")
        self.Kernel = Kernel
        self.dim = Kernel.input_dim
        self.product_form = Kernel.product_form
        self.kernel_type = getattr(Kernel, "kernel_type", "se")
        self.index_optimize_noise = index_optimize_noise if index_optimize_noise else False
        self.lbox = None if lbox is None else np.asarray(lbox, dtype=np.float64)
        if self.system == "stokes":
            self._obs, self._fields = operators.stokes_observables(self.dim)
        else:
            self._obs, self._fields = operators.scalar_observables(self.dim)
        self.n_kernel_theta = len(self._fields) * (1 + self.dim)
        if distributed is None:
            distributed = os.environ.get("STOPRO_B200_DISTRIBUTED", "0") not in ("", "0", "false", "False")
        self._distributed, self._group = bool(distributed), process_group
        self._plans = {}
        self._solver = None
        self._cache = None  # (theta bytes, y id, eps) -> (nll, grad)
        self._grad_seen = False  # a caller has asked for gradients: func(theta) then evaluates value AND gradient at once

    # ------------------------------------------------------------------ bookkeeping (gp.py:258-285)
    @staticmethod
    def calc_sec(pts):
        return np.concatenate([np.zeros(1, dtype=int), np.cumsum([len(x) for x in pts])])

    def set_constants(self, *args, only_training=False):
        if only_training:
            r_train, delta_y_train, eps = args
        else:
            r_test, mu_test, r_train, delta_y_train, eps = args
            self.num_te = len(r_test)
            self.sec_te = self.calc_sec(r_test)
        self.num_tr = len(r_train)
        self.sec_tr = self.calc_sec(r_train)
        self._training_plan(r_train)
        if not only_training:
            self._mixed_plan(r_test, r_train)
            self._test_plan(r_test)

    def split_hyp_and_noise(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        if self.index_optimize_noise:
            return theta[:-1], theta[-1]
        return theta, None

    def setup_Ks_dKdtheta(self):
        """Kept for call compatibility (gp.py:322-330); nothing to build."""
        return None

    # ------------------------------------------------------------------ plans
    def _observables(self, names):
        return [self._obs[n] for n in names]

    def _plan(self, key, build, row_pts, col_pts=None):
        plan = self._plans.get(key)
        sizes = tuple(len(p) for p in row_pts) + ((-1,) + tuple(len(p) for p in col_pts) if col_pts is not None else ())
        if plan is not None and plan._sizes == sizes:
            if not plan.same_points(row_pts, col_pts):
                plan.set_points(0, row_pts)
                if col_pts is not None:
                    plan.set_points(1, col_pts)
                self._cache = None
            return plan
        if plan is not None:
            if key == "train" and self._solver is not None:
                self._solver.close()
                self._solver = None
            plan.close()
        plan = build()
        plan._sizes = sizes
        self._plans[key] = plan
        self._cache = None
        return plan

    def _training_plan(self, r_train):
        names = self.train_observables[:len(r_train)]
        if len(names) != len(r_train):
            raise ValueError(f"{type(self).__name__} has {len(self.train_observables)} training blocks, got {len(r_train)} point sets")
        return self._plan("train", lambda: Plan(self.dim, self.product_form, self._fields, self._observables(names), r_train,
                                                lbox=self.lbox, noise_blocks=self.index_optimize_noise or None,
                                                kernel_type=self.kernel_type), r_train)

    def _mixed_plan(self, r_test, r_train):
        tr = self.train_observables[:len(r_train)]
        te = self.test_observables[:len(r_test)]
        return self._plan("mixed", lambda: Plan(self.dim, self.product_form, self._fields, self._observables(te), r_test,
                                                self._observables(tr), r_train, lbox=self.lbox, kernel_type=self.kernel_type),
                          r_test, r_train)

    def _test_plan(self, r_test):
        te = self.test_observables[:len(r_test)]
        return self._plan("test", lambda: Plan(self.dim, self.product_form, self._fields, self._observables(te), r_test,
                                               lbox=self.lbox, zero_blocks=self.test_zero_blocks, kernel_type=self.kernel_type),
                          r_test)

    def enable_distributed(self, process_group=None, on=True):
        """Select the sharded solver after construction (the subclasses keep the reference's constructor signatures, so
        the switch is this method or the STOPRO_B200_DISTRIBUTED environment variable -- never the YAML)."""
        if self._solver is not None:
            self._solver.close()
            self._solver = None
        self._distributed, self._group, self._cache = bool(on), process_group, None
        return self

    def _rank_world(self):
        """(rank, world) of the sharded evaluation; (0, 1) unless ``distributed`` was asked for and a group is up."""
        if not self._distributed:
            return 0, 1
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()):
            return 0, 1
        return dist.get_rank(self._group), dist.get_world_size(self._group)

    def _solver_for(self, r_train):
        plan = self._training_plan(r_train)
        if self._solver is None or self._solver.plan is not plan:
            if self._solver is not None:
                self._solver.close()
            rank, world = self._rank_world()
            self._solver = Solver(plan, rank, world)
            self._solver.connect_ipc(self._group)
        return self._solver

    @staticmethod
    def shard_points(pts, rank, world):
        """The rank's share of every test block (contiguous slices): the factor is replicated after a sharded
        factorisation, so posterior rows are independent work."""
        out, slices = [], []
        for p in pts:
            n = len(p)
            lo, hi = (n * rank) // world, (n * (rank + 1)) // world
            out.append(np.asarray(p)[lo:hi])
            slices.append((lo, hi))
        return out, slices

    def _reduce_theta(self, theta):
        """theta as the caller holds it -> (theta the plan consumes, positions of those entries in the caller's theta or
        None when they coincide).  params_main.yaml may carry the cross-covariance groups uxuy / uxp / uyp after the
        ones the independent models use (default_params/sinusoidal/params_main.yaml; get_init appends them,
        sub_modules/init_modules.py:37-48): the reference's theta slices ind_uxux / ind_uyuy / ind_pp simply never touch
        them, so they are dropped here and their gradient is zero.  The noise parameter, if any, is the last entry."""
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64).ravel())
        n_noise = 1 if self.index_optimize_noise else 0
        expected = self.n_kernel_theta + n_noise
        if th.size == expected:
            return th, None
        if th.size < expected:
            raise ValueError(f"theta has {th.size} entries, {type(self).__name__} needs {expected}")
        idx = np.arange(self.n_kernel_theta)
        if n_noise:
            idx = np.append(idx, th.size - 1)
        return np.ascontiguousarray(th[idx]), idx

    def _kernel_theta(self, theta, plan):
        th = np.asarray(theta, dtype=np.float64).ravel()
        if th.size > self.n_kernel_theta and th.size != plan.theta_len:
            th = th[:self.n_kernel_theta]  # unused cross-covariance groups (see _reduce_theta)
        if th.size == plan.theta_len - 1 and self.index_optimize_noise:
            th = np.append(th, 0.0)  # builders take theta without the noise entry (gp.py:221-222)
        return th

    # ------------------------------------------------------------------ covariance builders (gp.py:287-306)
    def trainingK_all(self, theta, train_pts):
        plan = self._training_plan(train_pts)
        return plan.assemble_host(self._kernel_theta(theta, plan), 0.0, False)

    def mixedK_all(self, theta, test_pts, train_pts):
        plan = self._mixed_plan(test_pts, train_pts)
        return plan.assemble_host(np.asarray(theta, dtype=np.float64)[:self.n_kernel_theta], 0.0, False)

    def testK_all(self, theta, test_pts):
        plan = self._test_plan(test_pts)
        return plan.assemble_host(np.asarray(theta, dtype=np.float64)[:self.n_kernel_theta], 0.0, False)

    def add_eps_to_sigma(self, Sigma, eps, noise_parameter=None):
        """gp.py:23-70 on a host matrix (the fused device path adds the diagonal inside the assembly kernel)."""
        n = len(Sigma)
        d = np.ones(n)
        if self.index_optimize_noise:
            lo = self.sec_tr[self.index_optimize_noise[0]]
            hi = self.sec_tr[self.index_optimize_noise[-1] + 1]
            d[lo:hi] *= np.exp(noise_parameter)
            d[hi:] *= eps
        else:
            d *= eps
        return Sigma + np.diag(d)

    def training_sigma(self, theta, train_pts, eps):
        """trainingK_all + add_eps_to_sigma in one kernel (gp.py:221-223)."""
        plan = self._training_plan(train_pts)
        return plan.assemble_host(self._reduce_theta(theta)[0], eps, True)

    # ------------------------------------------------------------------ likelihood and gradient
    def value_and_grad(self, theta, r, delta_y, eps, want_grad=True):
        """(NLL, dNLL/dtheta) from ONE factorisation; cached so that func(theta) followed by dfunc(theta)
        (solver/optimizers.py:148-150) costs one evaluation."""
        th, idx = self._reduce_theta(theta)
        y = np.ascontiguousarray(np.asarray(delta_y, dtype=np.float64).ravel())
        solver = self._solver_for(r)
        key = (th.tobytes(), y.tobytes(), float(eps))
        if self._cache is not None and self._cache[0] == key and (self._cache[2] is not None or not want_grad):
            nll, grad = self._cache[1], self._cache[2]
        else:
            nll, grad, _info = solver.nll_grad_host(th, y, eps, want_grad=want_grad)
            self._cache = (key, nll, grad)
        if idx is not None and grad is not None:
            full = np.zeros(np.asarray(theta).size, dtype=np.float64)
            full[idx] = grad
            grad = full
        return nll, grad

    def value_and_grad_many(self, thetas, r, delta_y, eps, want_grad=True):
        """value_and_grad for every row of ``thetas`` -> (nll (B,), grad (B, P_caller) or None).  One pass of the
        factorisation schedule evaluates all of them (Solver.nll_grad_batch_host); row b equals value_and_grad(thetas[b])
        bit for bit.  A sharded model evaluates them one after another, so that every rank issues the same calls.  The
        value_and_grad cache is left as it was."""
        thetas = [np.asarray(t, dtype=np.float64).ravel() for t in thetas]
        y = np.ascontiguousarray(np.asarray(delta_y, dtype=np.float64).ravel())
        solver = self._solver_for(r)
        if solver.world > 1:
            cache = self._cache
            out = [self.value_and_grad(t, r, y, eps, want_grad=want_grad) for t in thetas]
            self._cache = cache
            nll = np.array([o[0] for o in out])
            return nll, (np.stack([o[1] for o in out]) if want_grad else None)
        reduced = [self._reduce_theta(t) for t in thetas]
        nll, grad, _info = solver.nll_grad_batch_host([th for th, _ in reduced], y, eps, want_grad=want_grad)
        if grad is not None and any(idx is not None for _, idx in reduced):
            full = np.zeros((len(thetas), thetas[0].size), dtype=np.float64)
            for b, (_, idx) in enumerate(reduced):
                full[b, slice(None) if idx is None else idx] = grad[b]
            grad = full
        return nll, grad

    def trainingFunction_all(self, theta, *args):
        """NLL (gp.py:213-224).  Once a gradient has been requested from this model (the explicit-derivative scripts call
        func(theta) and then dfunc(theta) every step, solver/optimizers.py:148-150), the gradient is evaluated along with
        the value so that the pair costs ONE factorisation instead of the reference's two."""
        r, delta_y, eps = args
        return self.value_and_grad(theta, r, delta_y, eps, want_grad=self._grad_seen)[0]

    def d_trainingFunction_all(self, theta, *args):
        r, delta_y, eps = args
        self._grad_seen = True
        return self.value_and_grad(theta, r, delta_y, eps, want_grad=True)[1].copy()

    def adam_device(self, theta0, r, delta_y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=0.0, ridge_in_grad=True,
                    fixed=None, check_every=16):
        """optimize_by_adam's loop (solver/optimizers.py:173-235) resident on the device.  Returns (theta history
        (n+1, P_caller), loss history, gradient-norm history, status) or None when theta carries extra entries that are
        held by the caller only (cross-covariance groups of the YAML schema)."""
        th, idx = self._reduce_theta(theta0)
        if idx is not None:
            return None
        solver = self._solver_for(r)
        self._cache = None
        return solver.adam_host(th, delta_y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=ridge_alpha,
                                ridge_in_grad=ridge_in_grad, fixed=fixed, check_every=check_every)

    def adam_device_many(self, theta0s, r, delta_y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=0.0,
                         ridge_in_grad=True, fixed=None, check_every=16):
        """adam_device from several starting points in one device loop (one batched evaluation per iteration) -> list of
        adam_device's tuples, or None when a start carries entries held by the caller only, or the model is sharded."""
        reduced = [self._reduce_theta(t) for t in theta0s]
        if any(idx is not None for _, idx in reduced):
            return None
        solver = self._solver_for(r)
        if solver.world > 1:
            return None
        self._cache = None
        return solver.adam_batch_host([th for th, _ in reduced], delta_y, eps, max_iter, lr, stop_eps, ntraining,
                                      ridge_alpha=ridge_alpha, ridge_in_grad=ridge_in_grad, fixed=fixed,
                                      check_every=check_every)

    def d_logposterior(self, theta, *args):
        return self.d_trainingFunction_all(theta, *args) + 1.0  # gradient of the sum(theta) prior (gp.py:491-493)

    # ------------------------------------------------------------------ posterior (gp.py:226-256)
    def predictingFunction_all(self, theta, *args, full_cov=True):
        mus, covs = self.predict_many([theta], *args, full_cov=full_cov)
        return mus[0], covs[0]

    def predict_many(self, thetas, *args, full_cov=False):
        """predictingFunction_all for a list of hyper-parameter vectors in one library call: the ``interval_check`` loop of
        the reference's scripts (test/test_1_sinusoidal_direct_main.py:111-131).  Returns (list over thetas of [mu per test
        block], list over thetas of [variance (or covariance) per test block]).  In a sharded run with diagonal-only
        output every rank evaluates its own slice of the test points and the slices are gathered."""
        r_test, mu_test, r_train, delta_y_train, eps = args
        solver = self._solver_for(r_train)
        rank, world = solver.rank, solver.world
        shard = world > 1 and not full_cov
        pts, slices = self.shard_points(r_test, rank, world) if shard else (r_test, [(0, len(p)) for p in r_test])
        ths = [self._reduce_theta(t)[0] for t in thetas]
        if sum(len(p) for p in pts) > 0:
            mixed = self._mixed_plan(pts, r_train)
            test = self._test_plan(pts)
            mu, cov, _info = solver.predict_batch_host(mixed, test, ths, delta_y_train, eps, full_cov=full_cov)
        else:  # more ranks than test points: this rank only takes part in the factorisations
            for t in ths:
                solver.nll_grad_host(t, delta_y_train, eps, want_grad=False)
            mu = np.zeros((len(ths), 0))
            cov = np.zeros((len(ths), 0))
        self._cache = None
        if shard:
            import torch.distributed as dist

            parts = [None] * world
            dist.all_gather_object(parts, (mu, cov, slices), group=self._group)
        else:
            parts = [(mu, cov, slices)]
        out_mu, out_cov = [], []
        for b in range(len(ths)):
            mus = [np.empty(len(p)) for p in r_test]
            covs = [np.empty((len(p), len(p)) if full_cov else len(p)) for p in r_test]
            for pmu, pcov, psl in parts:
                lo = 0
                for i, (a, z) in enumerate(psl):
                    hi = lo + (z - a)
                    mus[i][a:z] = pmu[b, lo:hi]
                    if full_cov:
                        covs[i][:] = pcov[b, lo:hi, lo:hi]
                    else:
                        covs[i][a:z] = pcov[b, lo:hi]
                    lo = hi
            for i in range(len(r_test)):
                mus[i] = mus[i] + np.asarray(mu_test[i], dtype=np.float64)
            out_mu.append(mus)
            out_cov.append(covs)
        return out_mu, out_cov

    # ------------------------------------------------------------------ named blocks of the reference's library
    def __getattr__(self, name):
        # K<a><b>(r, rp, theta): cov(a(r), b(rp)), e.g. Kuxfx, Kfxdiv, Kdifuxdifux, Kpdifp (gp_2D_stokes_independent.py:22-246)
        if name.startswith("K") and not name.startswith("Kernel") and "_obs" in self.__dict__:
            try:
                oa, ob = operators.parse_block_name(name, self._obs)
            except KeyError:
                raise AttributeError(name) from None

            def block(r, rp, theta):
                plan = Plan(self.dim, self.product_form, self._fields, [oa], [r], [ob], [rp], lbox=self.lbox,
                            kernel_type=self.kernel_type)
                try:
                    return plan.assemble_host(np.asarray(theta, dtype=np.float64)[:self.n_kernel_theta])
                finally:
                    plan.close()

            return block
        raise AttributeError(name)

    def close(self):
        if self._solver is not None:
            self._solver.close()
            self._solver = None
        for p in self._plans.values():
            p.close()
        self._plans = {}
