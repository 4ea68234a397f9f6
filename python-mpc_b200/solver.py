"""Batched MPC-QP solver object: the host-side mirror of ``osqp.OSQP()`` for a batch of MPC QPs.

Reference surface mirrored (names and meaning follow the reference's use of OSQP):
    prob = osqp.OSQP(); prob.setup(P, q, A, l, u, warm_start=True)   mpc_kinematics.py:205-206
    prob.update(q=q_new, l=l_new, u=u_new)                            vehicle_lateral_mpc_slack_increment.py:237
    res = prob.solve(); res.x; res.info.status                        ...:248-253

Here the QP is given by its stage data (A_k, B_k, g_k, x_init, Xr, weights, bounds) instead of
assembled sparse matrices — the CUDA kernels apply the structured operators directly.
torch is used for device memory and streams only; every computation is a kernel of
libmpc_b200.so called through the C ABI (include/mpc_b200.h).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import MPCB_F32, MPCB_F64, MpcError, Problem, Settings, ptr

OSQP_DEFAULTS = dict(rho=0.1, sigma=1e-6, alpha=1.6, eps_abs=1e-3, eps_rel=1e-3, eps_prim_inf=1e-4,
                     eps_dual_inf=1e-4, max_iter=4000, scaling=10, check_termination=25, warm_start=True)


def _diag(v, n, name):
    if v is None:
        return np.zeros(n)
    if hasattr(v, "diagonal") and getattr(v, "ndim", 1) == 2:      # scipy.sparse.diags / dense matrix
        d = np.asarray(v.diagonal(), dtype=np.float64).ravel()
        dense = v.toarray() if hasattr(v, "toarray") else np.asarray(v)
        if np.any(dense - np.diag(d) != 0):
            raise ValueError("%s must be diagonal (the reference only uses sparse.diags / eye weights)" % name)
    else:
        d = np.asarray(v, dtype=np.float64).ravel()
    if d.size == 1 and n > 1:
        d = np.full(n, float(d[0]))
    if d.size != n:
        raise ValueError("%s has %d entries, expected %d" % (name, d.size, n))
    return d


class SolveInfo:
    """Per-batch solve information (``res.info`` of OSQP, vectorised)."""

    def __init__(self, iters, status_val, pri_res, dua_res):
        self.iter = iters
        self.status_val = status_val
        self.pri_res = pri_res
        self.dua_res = dua_res

    @property
    def status(self):
        return [_lib.STATUS_STRING.get(int(s), "unknown") for s in self.status_val.tolist()]


class BatchSolver:
    """One ``mpcb_solver``: B independent MPC QPs of identical shape, solved by OSQP-equivalent ADMM."""

    def __init__(self, N, nx, nu, Q, QN, R, xmin, xmax, umin, umax, slack=False, W=None, S=None,
                 dtype=torch.float32, time_varying=False, shared_model=False, stage_reference=False,
                 capacity=1, _backend=None, **settings):
        self.be = _backend if _backend is not None else _lib.cuda_backend()
        self.N, self.nx, self.nu, self.slack = int(N), int(nx), int(nu), bool(slack)
        if dtype not in (torch.float32, torch.float64):
            raise ValueError("dtype must be torch.float32 or torch.float64")
        self.dtype = dtype
        self.time_varying, self.shared_model, self.stage_reference = bool(time_varying), bool(shared_model), bool(stage_reference)
        p = Problem()
        p.horizon, p.nx, p.nu, p.slack = self.N, self.nx, self.nu, int(self.slack)
        p.dtype = MPCB_F32 if dtype == torch.float32 else MPCB_F64
        p.time_varying, p.shared_model, p.stage_reference = int(time_varying), int(shared_model), int(stage_reference)
        if self.nx > _lib.MPCB_MAX_NX or self.nu > _lib.MPCB_MAX_NU:
            raise ValueError("nx <= %d and nu <= %d" % (_lib.MPCB_MAX_NX, _lib.MPCB_MAX_NU))
        for name, val, n in (("Q", Q, nx), ("QN", QN, nx), ("R", R, nu), ("W", W, nx), ("S", S, nx),
                             ("xmin", xmin, nx), ("xmax", xmax, nx), ("umin", umin, nu), ("umax", umax, nu)):
            d = _diag(val, n, name)
            arr = getattr(p, name)
            for i in range(n):
                arr[i] = d[i]
        if np.any(_diag(Q, nx, "Q") < 0) or np.any(_diag(QN, nx, "QN") < 0) or np.any(_diag(R, nu, "R") < 0) \
                or np.any(_diag(W, nx, "W") < 0):
            raise ValueError("weights must be non-negative (P must be positive semidefinite)")
        self._problem = p
        self.settings = dict(OSQP_DEFAULTS)
        self._apply_settings_dict(settings)
        s = self._settings_struct()
        self.capacity = int(capacity)
        h = C.c_void_p()
        self.be.check(self.be.lib.mpcb_create(C.byref(p), C.byref(s), self.capacity, C.byref(h)))
        self._h = h
        self.ld = (self.capacity + 31) // 32 * 32
        self.nvar = self.be.lib.mpcb_num_variables(h)
        self.ncon = self.be.lib.mpcb_num_constraints(h)
        self.batch = 0
        self._keep = {}
        self._buffers = {}

    # ------------------------------------------------------------------ settings
    def _apply_settings_dict(self, settings):
        for k, v in settings.items():
            if k in ("verbose", "linsys_solver", "time_limit"):
                continue
            if k in ("adaptive_rho", "polish"):
                if v:
                    raise ValueError("%s is not part of this path (north_star: adaptive_rho and polish off)" % k)
                continue
            if k not in self.settings:
                raise TypeError("unknown setting %r" % k)
            self.settings[k] = v

    def _settings_struct(self):
        o = self.settings
        return Settings(o["rho"], o["sigma"], o["alpha"], o["eps_abs"], o["eps_rel"], o["eps_prim_inf"],
                        o["eps_dual_inf"], int(o["max_iter"]), int(o["scaling"]), int(o["check_termination"]),
                        int(bool(o["warm_start"])))

    def update_settings(self, **settings):
        self._apply_settings_dict(settings)
        s = self._settings_struct()
        self.be.check(self.be.lib.mpcb_set_settings(self._h, C.byref(s)))

    def set_stage_bounds(self, lo, hi):
        """Per-stage state boxes (lb_x/ub_x... of mpc_ in mpc_kinematics.py:215): lo, hi of shape (N+1, nx)."""
        box = np.stack([np.asarray(lo, dtype=np.float64), np.asarray(hi, dtype=np.float64)], axis=1)
        if box.shape != (self.N + 1, 2, self.nx):
            raise ValueError("stage bounds must have shape (N+1, nx)")
        box = np.ascontiguousarray(box)
        self.be.check(self.be.lib.mpcb_set_stage_bounds(self._h, box.ctypes.data_as(C.POINTER(C.c_double))))

    # ------------------------------------------------------------------ layout
    def _dev(self, a):
        if a is None:
            return None
        t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.asarray(a))
        return t.to(device=self.be.device, dtype=self.dtype).contiguous()

    def buffer(self, name, shape, dtype=None):
        """Persistent device buffer owned by the solver (reused across calls: no allocator traffic in the hot path)."""
        dtype = dtype or self.dtype
        t = self._buffers.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = self._buffers[name] = torch.zeros(shape, device=self.be.device, dtype=dtype)
        return t

    def to_element_major(self, a_bm, rows, elems, ld, out=None):
        """(rows, elems) batch-major tensor -> (elems, ld) element-major tensor (a kernel, not torch.t())."""
        src = self._dev(a_bm).reshape(rows, elems)
        dst = out if out is not None else torch.empty((elems, ld), device=self.be.device, dtype=self.dtype)
        if ld > rows and out is None:
            dst[:, rows:] = 0
        self.be.check(self.be.lib.mpcb_to_element_major(self._problem.dtype, rows, elems, ld, ptr(src), ptr(dst),
                                                        self.be.stream()))
        return dst

    def _bm(self, em, rows, elems):
        """(elems, ld) element-major -> (rows, elems) batch-major (kernel)."""
        dst = torch.empty((rows, elems), device=self.be.device, dtype=self.dtype)
        self.be.check(self.be.lib.mpcb_to_batch_major(self._problem.dtype, rows, elems, em.shape[1], ptr(em), ptr(dst),
                                                      self.be.stream()))
        return dst

    def _model_em(self, M, per_stage_shape, batch):
        """Natural-shape model array -> element-major.  Accepts (B, [N,] r, c), or for a shared model ([N,] r, c)."""
        if M is None:
            return None
        t = self._dev(M)
        stages = self.N if self.time_varying else 1
        elems = stages * int(np.prod(per_stage_shape))
        if self.shared_model:
            if t.numel() != elems:
                raise ValueError("shared model array has %d entries, expected %d" % (t.numel(), elems))
            return t.reshape(elems, 1).contiguous()
        if t.numel() != batch * elems:
            raise ValueError("model array has %d entries, expected %d x %d" % (t.numel(), batch, elems))
        return self.to_element_major(t, batch, elems, self.ld)

    # ------------------------------------------------------------------ OSQP-like surface
    def setup(self, Ad, Bd, gd, x_init, Xr, element_major=False):
        """prob.setup(...): Ruiz scaling + cached KKT factorisation for a batch.

        Batch-major inputs (default): Ad (B,[N,]nx,nx) | shared ([N,]nx,nx); Bd likewise; gd (B,[N,]nx) | None;
        x_init (B,nx); Xr (B,nx) or, with stage_reference, (B,nx,N+1) like the reference's Xr.
        element_major=True: tensors already in the device layout [elems, ld]."""
        if element_major:
            batch = int(x_init.shape[1]) if self.batch == 0 else self.batch
            ems = [Ad, Bd, gd, x_init, Xr]
        else:
            x0 = self._dev(x_init).reshape(-1, self.nx)
            batch = x0.shape[0]
            if batch > self.capacity:
                raise ValueError("batch %d exceeds solver capacity %d" % (batch, self.capacity))
            xr = self._dev(Xr)
            if self.stage_reference:
                xr = xr.reshape(batch, self.nx, self.N + 1).transpose(1, 2).contiguous()   # -> stage-major
                xr_elems = (self.N + 1) * self.nx
            else:
                xr = xr.reshape(batch, self.nx)
                xr_elems = self.nx
            ems = [self._model_em(Ad, (self.nx, self.nx), batch), self._model_em(Bd, (self.nx, self.nu), batch),
                   self._model_em(gd, (self.nx,), batch), self.to_element_major(x0, batch, self.nx, self.ld),
                   self.to_element_major(xr, batch, xr_elems, self.ld)]
        self.batch = batch
        self._keep = dict(zip(("Ad", "Bd", "gd", "x_init", "Xr"), ems))      # borrowed by the library
        self.be.check(self.be.lib.mpcb_setup(self._h, batch, self.ld, ptr(ems[0]), ptr(ems[1]), ptr(ems[2]),
                                             ptr(ems[3]), ptr(ems[4]), self.be.stream()))
        return self

    def set_batch(self, batch):
        self.batch = int(batch)

    def update(self, x_init=None, Xr=None, element_major=False):
        """prob.update(q=..., l=..., u=...): new initial state and/or reference, same scaling and factor."""
        if x_init is not None:
            self._keep["x_init"] = x_init if element_major else self.to_element_major(
                self._dev(x_init).reshape(self.batch, self.nx), self.batch, self.nx, self.ld)
        if Xr is not None:
            if element_major:
                self._keep["Xr"] = Xr
            else:
                xr = self._dev(Xr)
                if self.stage_reference:
                    xr = xr.reshape(self.batch, self.nx, self.N + 1).transpose(1, 2).contiguous()
                    self._keep["Xr"] = self.to_element_major(xr, self.batch, (self.N + 1) * self.nx, self.ld)
                else:
                    self._keep["Xr"] = self.to_element_major(xr.reshape(self.batch, self.nx), self.batch, self.nx, self.ld)
        self.be.check(self.be.lib.mpcb_update(self._h, ptr(self._keep["x_init"]), ptr(self._keep["Xr"])))
        return self

    def update_bounds(self, xmin=None, xmax=None, umin=None, umax=None, stage_lo=None, stage_hi=None):
        """The inequality part of prob.update(l=l_new, u=u_new): new state / input bounds after setup
        (vehicle_lateral_mpc_slack_increment.py:158-172, applied at :237).  OSQP's update_bounds semantics: the
        existing scaling is kept, the per-row rho type is re-evaluated and the KKT factor is rebuilt only for QPs in
        which a row changed type; the iterates stay (warm start).  None = unchanged; stage_lo / stage_hi (N+1, nx)
        replace the per-stage state boxes."""
        dp = C.POINTER(C.c_double)
        keep = []

        def arr(v, n, name):
            if v is None:
                return dp()
            a = np.ascontiguousarray(_diag(v, n, name), dtype=np.float64)
            keep.append(a)
            return a.ctypes.data_as(dp)

        box = dp()
        if (stage_lo is None) != (stage_hi is None):
            raise ValueError("stage_lo and stage_hi go together")
        if stage_lo is not None:
            b = np.ascontiguousarray(np.stack([np.asarray(stage_lo, dtype=np.float64), np.asarray(stage_hi, dtype=np.float64)],
                                              axis=1))
            if b.shape != (self.N + 1, 2, self.nx):
                raise ValueError("stage bounds must have shape (N+1, nx)")
            keep.append(b)
            box = b.ctypes.data_as(dp)
        self.be.check(self.be.lib.mpcb_update_bounds(self._h, arr(xmin, self.nx, "xmin"), arr(xmax, self.nx, "xmax"),
                                                     arr(umin, self.nu, "umin"), arr(umax, self.nu, "umax"), box,
                                                     self.be.stream()))
        return self

    def solve(self):
        """res = prob.solve() for the whole batch (asynchronous on the current stream)."""
        self.be.check(self.be.lib.mpcb_solve(self._h, self.be.stream()))
        return self

    def iterate(self, iters):
        self.be.check(self.be.lib.mpcb_iterate(self._h, int(iters), self.be.stream()))
        return self

    def cold_start(self):
        self.be.check(self.be.lib.mpcb_cold_start(self._h, self.be.stream()))
        return self

    def solution(self, want_x=True, want_y=False, want_u=True, reuse=False):
        """(x, y, u): res.x (B,nvar) / res.y (B,ncon) in the reference's ordering, and the input sequence (B,N,nu).
        reuse=True returns views of persistent buffers (overwritten by the next call)."""
        B = self.batch
        mk = (lambda n, nm: self.buffer("out_" + nm, (B, n))) if reuse else \
             (lambda n, nm: torch.empty((B, n), device=self.be.device, dtype=self.dtype))
        x = mk(self.nvar, "x") if want_x else None
        y = mk(self.ncon, "y") if want_y else None
        u = mk(self.N * self.nu, "u") if want_u else None
        self.be.check(self.be.lib.mpcb_get_solution(self._h, ptr(x), ptr(y), ptr(u), self.be.stream()))
        return x, y, (u.reshape(B, self.N, self.nu) if u is not None else None)

    def info(self, reuse=False):
        B = self.batch
        if reuse:
            it, st = self.buffer("info_it", (B,), torch.int32), self.buffer("info_st", (B,), torch.int32)
            pr, du = self.buffer("info_pr", (B,)), self.buffer("info_du", (B,))
        else:
            it = torch.empty(B, device=self.be.device, dtype=torch.int32)
            st = torch.empty(B, device=self.be.device, dtype=torch.int32)
            pr = torch.empty(B, device=self.be.device, dtype=self.dtype)
            du = torch.empty(B, device=self.be.device, dtype=self.dtype)
        self.be.check(self.be.lib.mpcb_get_info(self._h, ptr(it), ptr(st), ptr(pr), ptr(du), self.be.stream()))
        return SolveInfo(it, st, pr, du)

    def build_qp(self):
        """The explicit (Pdiag, q, A values, l, u) of every QP, batch-major, plus A's shared CSC pattern."""
        B, ld = self.batch, self.ld
        nnz = self.be.lib.mpcb_qp_pattern(self._h, None, None)
        Ap = np.zeros(self.nvar + 1, dtype=np.int32); Ai = np.zeros(nnz, dtype=np.int32)
        self.be.lib.mpcb_qp_pattern(self._h, Ap.ctypes.data_as(C.POINTER(C.c_int)), Ai.ctypes.data_as(C.POINTER(C.c_int)))
        mk = lambda n: torch.zeros((n, ld), device=self.be.device, dtype=self.dtype)
        Pd, q, Av, l, u = mk(self.nvar), mk(self.nvar), mk(nnz), mk(self.ncon), mk(self.ncon)
        self.be.check(self.be.lib.mpcb_build_qp(self._h, ptr(Pd), ptr(q), ptr(Av), ptr(l), ptr(u), self.be.stream()))
        out = [t[:, :B].t().contiguous() for t in (Pd, q, Av, l, u)]
        return out[0], out[1], out[2], out[3], out[4], Ap, Ai

    def scaling(self):
        """The Ruiz scaling of the last setup, OSQP's (D, E, c): D (B,nvar), E (B,ncon) in the reference's ordering, c (B,)."""
        B = self.batch
        mk = lambda *shape: torch.empty(shape, device=self.be.device, dtype=self.dtype)
        D, E, c = mk(B, self.nvar), mk(B, self.ncon), mk(B)
        self.be.check(self.be.lib.mpcb_get_scaling(self._h, ptr(D), ptr(E), ptr(c), self.be.stream()))
        return D, E, c

    def solve_host(self, Ad, Bd, gd, x_init, Xr, want_x=True, want_u=True):
        """The host front door: numpy-layout HOST arrays in and out, copies inside (mpcb_solve_host)."""
        npdt = np.float32 if self.dtype == torch.float32 else np.float64
        c = lambda a: None if a is None else np.ascontiguousarray(np.asarray(a, dtype=npdt))
        x0 = c(x_init).reshape(-1, self.nx)
        B = x0.shape[0]
        xr = c(Xr)
        if self.stage_reference:
            xr = np.ascontiguousarray(xr.reshape(B, self.nx, self.N + 1).transpose(0, 2, 1))
        Ad, Bd, gd = c(Ad), c(Bd), c(gd)
        xo = np.empty((B, self.nvar), dtype=npdt) if want_x else None
        uo = np.empty((B, self.N * self.nu), dtype=npdt) if want_u else None
        it = np.empty(B, dtype=np.int32); st = np.empty(B, dtype=np.int32)
        vp = lambda a: C.c_void_p(0) if a is None else C.c_void_p(a.ctypes.data)
        self.be.check(self.be.lib.mpcb_solve_host(self._h, B, vp(Ad), vp(Bd), vp(gd), vp(x0), vp(xr), vp(xo), vp(uo),
                                                  vp(it), vp(st)))
        self.batch = B
        return xo, (uo.reshape(B, self.N, self.nu) if uo is not None else None), it, st

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.be.lib.mpcb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
