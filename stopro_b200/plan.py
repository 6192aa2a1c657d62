"""Python handles over the C ABI: Plan (block-structured covariance) and Solver (factorisation workspace)."""
import ctypes as C

import numpy as np

from . import _lib, operators


def stack_points(pts, dim):
    """list of (n_i, dim) arrays ((n_i,) when dim == 1) -> (N, dim) float64 C-contiguous, plus section offsets
    (GP/gp.py:258-261 calc_sec)."""
    arrs = []
    for p in pts:
        a = np.asarray(p, dtype=np.float64)
        if dim == 1:
            a = a.reshape(-1, 1)
        if a.ndim != 2 or a.shape[1] != dim:
            raise ValueError(f"expected points of shape (n, {dim}), got {a.shape}")
        arrs.append(a)
    sec = np.concatenate([[0], np.cumsum([len(a) for a in arrs])]).astype(np.int64)
    flat = np.ascontiguousarray(np.concatenate(arrs, axis=0)) if arrs else np.zeros((0, dim))
    return flat, sec


def _ptr(a, typ=C.c_double):
    return a.ctypes.data_as(C.POINTER(typ))


class Plan:
    """A block matrix  [cov(A_i(r_i), B_j(r'_j))]_{ij}  bound to its point sets."""

    def __init__(self, dim, product_form, fields, row_obs, row_pts, col_obs=None, col_pts=None, lbox=None,
                 noise_blocks=None, zero_blocks=(), kernel_type="se"):
        self.dim, self.product_form, self.fields = dim, bool(product_form), list(fields)
        self.kernel_type = kernel_type
        self.symmetric = col_obs is None
        self.row_obs, self.col_obs = list(row_obs), (list(row_obs) if col_obs is None else list(col_obs))
        self._rows, self.sec_row = stack_points(row_pts, dim)
        if self.symmetric:
            self._cols, self.sec_col = self._rows, self.sec_row
        else:
            self._cols, self.sec_col = stack_points(col_pts, dim)
        if len(self.row_obs) != len(self.sec_row) - 1 or len(self.col_obs) != len(self.sec_col) - 1:
            raise ValueError("one observable per point block is required")
        nr, nc = len(self.row_obs), len(self.col_obs)
        table = (_lib.BlockDesc * (nr * nc))()
        for i in range(nr):
            for j in range(nc):
                if self.symmetric and j < i:
                    continue
                if (i, j) in zero_blocks:
                    continue  # zero-initialised descriptor: n_terms = 0, the reference's Kzero
                table[i * nc + j] = operators.make_desc(self.row_obs[i], self.col_obs[j], self.fields, dim,
                                                        self.product_form)
        self._table = table
        d = _lib.PlanDesc()
        d.dim, d.product_form, d.n_groups, d.symmetric = dim, int(self.product_form), len(self.fields), int(self.symmetric)
        d.n_row_blocks, d.n_col_blocks = nr, nc
        d.kernel_type = _lib.KERNEL_TYPES[kernel_type]
        d.sec_row, d.sec_col = _ptr(self.sec_row, C.c_int64), _ptr(self.sec_col, C.c_int64)
        d.pts_row_host, d.pts_col_host = _ptr(self._rows), _ptr(self._cols)
        d.table = table
        lb = np.zeros(3) if lbox is None else np.concatenate([np.asarray(lbox, dtype=np.float64).ravel(), np.zeros(3)])[:3]
        for k in range(3):
            d.lbox[k] = float(lb[k])
        if noise_blocks:
            d.noise_lo_block, d.noise_hi_block = int(noise_blocks[0]), int(noise_blocks[-1])
        else:
            d.noise_lo_block = d.noise_hi_block = -1
        h = C.c_void_p()
        _lib.check(_lib.lib().pigp_plan_create(C.byref(d), C.byref(h)))
        self.handle = h
        self.rows, self.cols = int(self.sec_row[-1]), int(self.sec_col[-1])
        self.theta_len = int(_lib.lib().pigp_plan_theta_len(h))

    def close(self):
        if getattr(self, "handle", None):
            _lib.lib().pigp_plan_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def same_points(self, row_pts, col_pts=None):
        def eq(flat, pts):
            try:
                a, _ = stack_points(pts, self.dim)
            except ValueError:
                return False
            return a.shape == flat.shape and np.array_equal(a, flat)

        return eq(self._rows, row_pts) and (self.symmetric or eq(self._cols, col_pts))

    def set_points(self, side, pts):
        flat, sec = stack_points(pts, self.dim)
        ref_sec = self.sec_row if (side == 0 or self.symmetric) else self.sec_col
        if not np.array_equal(sec, ref_sec):
            raise ValueError("block sizes differ from the plan's")
        _lib.check(_lib.lib().pigp_plan_set_points_host(self.handle, side, flat.ctypes.data, None))
        if side == 0 or self.symmetric:
            self._rows = flat
            if self.symmetric:
                self._cols = flat
        else:
            self._cols = flat

    def _theta(self, theta):
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64).ravel())
        if th.size != self.theta_len:
            raise ValueError(f"theta has {th.size} entries, the model needs {self.theta_len}")
        return th

    def assemble_host(self, theta, eps=0.0, add_diag=False, layout=_lib.LAYOUT_FULL):
        th = self._theta(theta)
        K = np.empty((self.rows, self.cols), dtype=np.float64)
        _lib.check(_lib.lib().pigp_assemble_host(self.handle, th.ctypes.data, float(eps), int(add_diag), K.ctypes.data,
                                                 int(layout)))
        return K

    def assemble_diag(self, theta_ptr, eps, add_diag, out_ptr, stream=None):
        """Only the diagonal of a symmetric plan's matrix (device pointers)."""
        _lib.check(_lib.lib().pigp_assemble_diag(self.handle, theta_ptr, float(eps), int(add_diag), out_ptr, stream))

    def assemble(self, theta_ptr, eps, add_diag, out_ptr, ld, layout=_lib.LAYOUT_FULL, stream=None):
        """Device-pointer form (theta_ptr / out_ptr are integers, e.g. torch.Tensor.data_ptr())."""
        _lib.check(_lib.lib().pigp_assemble(self.handle, theta_ptr, float(eps), int(add_diag), out_ptr, int(ld), int(layout),
                                            stream))


class Solver:
    """Factorisation workspace bound to a training plan (pigp_solver).  With world > 1 the covariance matrix is dealt
    block-cyclically over the ranks of one NVLink box (one process per GPU): every rank creates Solver(plan, rank, world),
    calls connect_ipc() once, and then all ranks issue the same sequence of evaluations."""

    def __init__(self, plan, rank=0, world=1):
        if not plan.symmetric:
            raise ValueError("Solver needs the symmetric training plan")
        self.plan, self.rank, self.world = plan, int(rank), int(world)
        h = C.c_void_p()
        _lib.check(_lib.lib().pigp_solver_create_dist(plan.handle, self.rank, self.world, C.byref(h)))
        self.handle = h
        self._opened = []

    # -- multi-GPU wiring (no-ops for world == 1)
    @property
    def _ds(self):
        return C.c_void_p(_lib.lib().pigp_solver_dsolver(self.handle))

    def connect_ipc(self, group=None):
        """Exchange the CUDA-IPC handles of the solver slabs over torch.distributed (any backend) and map the peers."""
        if self.world == 1:
            return
        import torch.distributed as dist

        from .dist import exchange_handles

        lib = _lib.lib()
        buf = (C.c_char * _lib.IPC_HANDLE_BYTES)()
        _lib.check(lib.pigp_dsolver_ipc_handle(self._ds, buf))
        uuid = (C.c_char * 16)()
        _lib.check(lib.pigp_device_uuid(uuid))
        both = exchange_handles(bytes(buf) + bytes(uuid), group)
        slab, nbytes = C.c_void_p(), C.c_int64()
        _lib.check(lib.pigp_dsolver_slab(self._ds, C.byref(slab), C.byref(nbytes)))
        slabs, shared = [], False
        for r, b in enumerate(both):
            if r == self.rank:
                slabs.append(slab.value)
                continue
            shared |= b[_lib.IPC_HANDLE_BYTES:] == bytes(uuid)
            ptr = C.c_void_p()
            _lib.check(lib.pigp_ipc_open(b[:_lib.IPC_HANDLE_BYTES], C.byref(ptr)))
            self._opened.append(ptr.value)
            slabs.append(ptr.value)
        arr = (C.c_void_p * self.world)(*[C.c_void_p(p) for p in slabs])
        _lib.check(lib.pigp_dsolver_connect(self._ds, arr))
        _lib.check(lib.pigp_dsolver_set_shared_device(self._ds, int(shared)))
        dist.barrier(group=group)  # every rank is wired before anyone's first flag wait

    def reset(self):
        """Re-arm after a failed sharded evaluation (call on every rank, then barrier)."""
        if self.world > 1:
            _lib.check(_lib.lib().pigp_dsolver_reset(self._ds))

    def close(self):
        if getattr(self, "handle", None):
            _lib.lib().pigp_solver_destroy(self.handle)
            self.handle = None
            for ptr in self._opened:
                _lib.lib().pigp_ipc_close(ptr)
            self._opened = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def nll_grad_host(self, theta, y, eps, want_grad=True, pts=None):
        """One NLL (+ gradient) evaluation with host buffers in and out -> (nll, grad or None, info)."""
        p = self.plan
        th = p._theta(theta)
        yy = np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        if yy.size != p.rows:
            raise ValueError(f"delta_y has {yy.size} entries, the training set has {p.rows}")
        pts_ptr = None
        if pts is not None:
            flat, sec = stack_points(pts, p.dim)
            if not np.array_equal(sec, p.sec_row):
                raise ValueError("block sizes differ from the plan's")
            pts_ptr = flat.ctypes.data
        nll = C.c_double()
        grad = np.empty(p.theta_len, dtype=np.float64)
        info = C.c_int32()
        _lib.check(_lib.lib().pigp_nll_grad_host(self.handle, th.ctypes.data, pts_ptr, yy.ctypes.data, float(eps),
                                                 int(want_grad), C.addressof(nll), grad.ctypes.data, C.addressof(info)))
        return nll.value, (grad if want_grad else None), info.value

    def nll_grad_batch_host(self, thetas, y, eps, want_grad=True):
        """NLL (+ gradient) of B hyper-parameter vectors (rows of ``thetas``) in one pass of the factorisation schedule
        (pigp_nll_grad_batch_host) -> (nll (B,), grad (B, P) or None, info (B,)).  Slot b equals nll_grad_host(thetas[b])
        bit for bit."""
        p = self.plan
        th = np.ascontiguousarray(np.stack([p._theta(t) for t in thetas]))
        yy = np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        if yy.size != p.rows:
            raise ValueError(f"delta_y has {yy.size} entries, the training set has {p.rows}")
        nb = len(th)
        nll = np.empty(nb, dtype=np.float64)
        grad = np.empty((nb, p.theta_len), dtype=np.float64)
        info = np.zeros(nb, dtype=np.int32)
        _lib.check(_lib.lib().pigp_nll_grad_batch_host(self.handle, nb, th.ctypes.data, yy.ctypes.data, float(eps),
                                                       int(want_grad), nll.ctypes.data, grad.ctypes.data, info.ctypes.data))
        return nll, (grad if want_grad else None), info

    def nll_grad_batch(self, n_theta, thetas_ptr, y_ptr, eps, nll_ptr, grad_ptr=None, info_ptr=None, stream=None):
        _lib.check(_lib.lib().pigp_nll_grad_batch(self.handle, int(n_theta), thetas_ptr, y_ptr, float(eps), nll_ptr, grad_ptr,
                                                  info_ptr, stream))

    def nll_grad(self, theta_ptr, y_ptr, eps, nll_ptr, grad_ptr, info_ptr=None, stream=None):
        _lib.check(_lib.lib().pigp_nll_grad(self.handle, theta_ptr, y_ptr, float(eps), nll_ptr, grad_ptr, info_ptr, stream))

    def nll(self, theta_ptr, y_ptr, eps, nll_ptr, info_ptr=None, stream=None):
        _lib.check(_lib.lib().pigp_nll(self.handle, theta_ptr, y_ptr, float(eps), nll_ptr, info_ptr, stream))

    def adam_host(self, theta0, y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=0.0, ridge_in_grad=True, fixed=None,
                  check_every=16):
        """Device-resident optimize_by_adam loop (pigp_adam_host) -> (theta_hist (n+1, P), loss_hist (n+1,),
        gradnorm_hist (n,), status)."""
        return self.adam_batch_host([theta0], y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=ridge_alpha,
                                    ridge_in_grad=ridge_in_grad, fixed=fixed, check_every=check_every)[0]

    def adam_batch_host(self, theta0s, y, eps, max_iter, lr, stop_eps, ntraining, ridge_alpha=0.0, ridge_in_grad=True,
                        fixed=None, check_every=16):
        """adam_host from every row of ``theta0s`` at once (pigp_adam_batch_host: one batched evaluation per iteration)
        -> list over starts of (theta_hist, loss_hist, gradnorm_hist, status), each equal to adam_host from that start."""
        p = self.plan
        th = np.ascontiguousarray(np.stack([p._theta(t) for t in theta0s]))
        yy = np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        nb, P = len(th), p.theta_len
        theta_hist = np.empty((nb, max_iter + 1, P), dtype=np.float64)
        loss_hist = np.empty((nb, max_iter + 1), dtype=np.float64)
        norm_hist = np.empty((nb, max_iter), dtype=np.float64)
        mask = None
        if fixed is not None and len(fixed):
            mask = np.zeros(P, dtype=np.int32)
            mask[np.asarray(fixed, dtype=int)] = 1
        n_done = np.zeros(nb, dtype=np.int32)
        status = np.zeros(nb, dtype=np.int32)
        _lib.check(_lib.lib().pigp_adam_batch_host(self.handle, nb, th.ctypes.data, yy.ctypes.data, float(eps), int(max_iter),
                                                   float(lr), float(stop_eps), float(ntraining), float(ridge_alpha),
                                                   int(ridge_in_grad), mask.ctypes.data if mask is not None else None,
                                                   int(check_every), theta_hist.ctypes.data, loss_hist.ctypes.data,
                                                   norm_hist.ctypes.data, n_done.ctypes.data, status.ctypes.data))
        return [(theta_hist[b, :n + 1].copy(), loss_hist[b, :n + 1].copy(), norm_hist[b, :n].copy(), int(status[b]))
                for b, n in enumerate(n_done)]

    def predict_host(self, mixed, test, theta, y, eps, full_cov=True):
        mu, cov, info = self.predict_batch_host(mixed, test, [theta], y, eps, full_cov=full_cov)
        return mu[0], cov[0], int(info[0])

    def predict_batch_host(self, mixed, test, thetas, y, eps, full_cov=False):
        """Posterior for a list of hyper-parameter vectors in ONE library call (the interval_check loop of the reference's
        scripts) -> mu (n_theta, M), cov (n_theta, M[, M]), info (n_theta,)."""
        p = self.plan
        th = np.ascontiguousarray(np.stack([p._theta(t) for t in thetas]))
        yy = np.ascontiguousarray(np.asarray(y, dtype=np.float64).ravel())
        nb, m = len(th), mixed.rows
        mu = np.empty((nb, m), dtype=np.float64)
        cov = np.empty((nb, m, m) if full_cov else (nb, m), dtype=np.float64)
        info = np.zeros(nb, dtype=np.int32)
        _lib.check(_lib.lib().pigp_predict_batch_host(self.handle, mixed.handle, test.handle, nb, th.ctypes.data,
                                                      yy.ctypes.data, float(eps), mu.ctypes.data, cov.ctypes.data,
                                                      int(full_cov), info.ctypes.data))
        return mu, cov, info
