"""ORACLE — test infrastructure only.  ctypes front-end of oracle/osqp_admm.c."""
import ctypes as C

import numpy as np
import scipy.sparse as sp

from .library import build


class Settings(C.Structure):
    _fields_ = [("rho", C.c_double), ("sigma", C.c_double), ("alpha", C.c_double), ("eps_abs", C.c_double),
                ("eps_rel", C.c_double), ("eps_prim_inf", C.c_double), ("eps_dual_inf", C.c_double),
                ("max_iter", C.c_int), ("scaling", C.c_int), ("check_termination", C.c_int),
                ("warm_start", C.c_int)]


class Info(C.Structure):
    _fields_ = [("iter", C.c_int), ("status", C.c_int), ("pri_res", C.c_double), ("dua_res", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.oracle_osqp_solve.restype = C.c_int
        _lib.oracle_solve_batch.restype = C.c_int
        _lib.oracle_closed_loop_batch.restype = C.c_int
    return _lib


def make_settings(rho=0.1, sigma=1e-6, alpha=1.6, eps_abs=1e-3, eps_rel=1e-3, eps_prim_inf=1e-4,
                  eps_dual_inf=1e-4, max_iter=4000, scaling=10, check_termination=25, warm_start=1, **_):
    return Settings(rho, sigma, alpha, eps_abs, eps_rel, eps_prim_inf, eps_dual_inf, max_iter, scaling,
                    check_termination, int(warm_start))


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _csc(P, A):
    Pu = sp.triu(sp.csc_matrix(P, dtype=np.float64), format="csc"); Pu.sort_indices()
    A = sp.csc_matrix(A, dtype=np.float64); A.sort_indices()
    return Pu, A


def solve(P, q, A, l, u, perm=None, x0=None, y0=None, **settings):
    Pu, A = _csc(P, A)
    n, m = Pu.shape[0], A.shape[0]
    s = make_settings(**settings)
    info = Info()
    x = np.zeros(n); y = np.zeros(m)
    q = np.ascontiguousarray(q, dtype=np.float64); l = np.ascontiguousarray(l, dtype=np.float64)
    u = np.ascontiguousarray(u, dtype=np.float64)
    Pp = Pu.indptr.astype(np.int32); Pi = Pu.indices.astype(np.int32)
    Ap = A.indptr.astype(np.int32); Ai = A.indices.astype(np.int32)
    permp = None if perm is None else _p(np.ascontiguousarray(perm, dtype=np.int32), C.c_int)
    keep = [np.ascontiguousarray(v, dtype=np.float64) if v is not None else None for v in (x0, y0)]
    rc = lib().oracle_osqp_solve(C.c_int(n), C.c_int(m), _p(Pp, C.c_int), _p(Pi, C.c_int), _p(Pu.data, C.c_double),
                                 _p(q, C.c_double), _p(Ap, C.c_int), _p(Ai, C.c_int), _p(A.data, C.c_double),
                                 _p(l, C.c_double), _p(u, C.c_double), permp, C.byref(s),
                                 None if keep[0] is None else _p(keep[0], C.c_double),
                                 None if keep[1] is None else _p(keep[1], C.c_double),
                                 _p(x, C.c_double), _p(y, C.c_double), C.byref(info))
    if rc != 0:
        raise RuntimeError("oracle: reduced KKT matrix not positive definite")
    return x, y, info.iter, info.status, info.pri_res, info.dua_res


def solve_batch(P, A, Pvals, q, Avals, l, u, perm=None, nthreads=0, **settings):
    """P, A give the shared CSC pattern (P upper triangle); Pvals[B,pnz], Avals[B,anz] in that pattern's order."""
    Pu, A = _csc(P, A)
    n, m = Pu.shape[0], A.shape[0]
    B = q.shape[0]
    s = make_settings(**settings)
    x = np.zeros((B, n)); y = np.zeros((B, m)); it = np.zeros(B, dtype=np.int32); st = np.zeros(B, dtype=np.int32)
    arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (Pvals, q, Avals, l, u)]
    Pp = Pu.indptr.astype(np.int32); Pi = Pu.indices.astype(np.int32)
    Ap = A.indptr.astype(np.int32); Ai = A.indices.astype(np.int32)
    permp = None if perm is None else _p(np.ascontiguousarray(perm, dtype=np.int32), C.c_int)
    used = lib().oracle_solve_batch(C.c_int(B), C.c_int(n), C.c_int(m), _p(Pp, C.c_int), _p(Pi, C.c_int),
                                    _p(arrs[0], C.c_double), _p(arrs[1], C.c_double), _p(Ap, C.c_int), _p(Ai, C.c_int),
                                    _p(arrs[2], C.c_double), _p(arrs[3], C.c_double), _p(arrs[4], C.c_double), permp,
                                    C.byref(s), _p(x, C.c_double), _p(y, C.c_double), _p(it, C.c_int), _p(st, C.c_int),
                                    C.c_int(nthreads))
    return x, y, it, st, used


def closed_loop_batch(P, A, Pvals, q, Avals, l, u, Apl, Bpl, x0, steps, u_index, perm=None, nthreads=0, schedule=None,
                      **settings):
    """oracle_closed_loop_batch: setup once per scenario, then `steps` x (update(l, u) with the initial-state rows,
    warm-started solve, plant step).  schedule: {step: (l_row [m], u_row [m])} inequality bounds switched in at a step.
    Returns (iters [B, steps], status [B, steps], u_applied [B, steps, nu], traj [B, steps+1, nx], threads used)."""
    Pu, A = _csc(P, A)
    n, m = Pu.shape[0], A.shape[0]
    B, nx = x0.shape
    nu = Bpl.shape[-1]
    settings = dict(settings); settings.setdefault("warm_start", 1)
    s = make_settings(**settings)
    arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (Pvals, q, Avals, l, u, Apl, Bpl, x0)]
    Pp = Pu.indptr.astype(np.int32); Pi = Pu.indices.astype(np.int32)
    Ap = A.indptr.astype(np.int32); Ai = A.indices.astype(np.int32)
    permp = None if perm is None else _p(np.ascontiguousarray(perm, dtype=np.int32), C.c_int)
    sched = sorted((schedule or {}).items())
    ss = np.array([k for k, _ in sched], dtype=np.int32)
    ls = np.ascontiguousarray(np.stack([v[0] for _, v in sched]) if sched else np.zeros((1, m)), dtype=np.float64)
    us = np.ascontiguousarray(np.stack([v[1] for _, v in sched]) if sched else np.zeros((1, m)), dtype=np.float64)
    it = np.zeros((B, steps), dtype=np.int32); st = np.zeros((B, steps), dtype=np.int32)
    ua = np.zeros((B, steps, nu)); traj = np.zeros((B, steps + 1, nx))
    used = lib().oracle_closed_loop_batch(C.c_int(B), C.c_int(n), C.c_int(m), _p(Pp, C.c_int), _p(Pi, C.c_int),
                                          _p(arrs[0], C.c_double), _p(arrs[1], C.c_double), _p(Ap, C.c_int), _p(Ai, C.c_int),
                                          _p(arrs[2], C.c_double), _p(arrs[3], C.c_double), _p(arrs[4], C.c_double), permp,
                                          C.byref(s), C.c_int(steps), C.c_int(nx), C.c_int(nu), C.c_int(u_index),
                                          _p(arrs[5], C.c_double), _p(arrs[6], C.c_double), _p(arrs[7], C.c_double),
                                          C.c_int(len(sched)), _p(ss if len(sched) else np.zeros(1, dtype=np.int32), C.c_int),
                                          _p(ls, C.c_double), _p(us, C.c_double), _p(it, C.c_int), _p(st, C.c_int),
                                          _p(ua, C.c_double), _p(traj, C.c_double), C.c_int(nthreads))
    return it, st, ua, traj, used
