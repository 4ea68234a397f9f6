"""prob.update(l=, u=) after a setup (mpcb_update_bounds): the per-QP refactor of RefactorFn / bounds_change_row_types, the
per-stage box buffers (xbox / xbox_alt), the batch-wide infinite-bound flag (inf_bounds) and the reset of the dense path's
inverse, through bound changes that change a row's rho type (equality / inequality / unbounded) in some QPs or in all:

  T1  a state row narrowed to a gap g that is an equality after scaling (E g < RHO_TOL) in some QPs only
  T2  T1 reversed (equality -> inequality)
  T3  a state row made unbounded on both sides in a problem without an infinite bound (inf_bounds 0 -> 1); T4 reversed
  T5  umin = umax on an input (the bu rows become equalities), and back
  T6  a type change at one stage only, through a per-stage box (from no box to a box)
  T7  bounds that move without a type change (nothing is refactored, the warm start is kept)

(a) Ruiz scaling never reads l or u, and the factor depends on the bounds only through the row types: a solver set up
    with L0 and updated to L1 equals, bit for bit, a solver set up with L1 — scaling, the first iterates from a cold
    start, and a solve of exactly 30 iterations (which reaches every ADMM path).
(b) A warm-started sequence of solves in which T1..T7 alternate with new initial states, against the oracle's
    update(l=, u=) on one oracle object per QP kept for the whole sequence; the iterates after each update; which QPs
    the oracle refactors; closed loops with a bound switch that changes a row's type against oracle_closed_loop_batch.
(c) On the GPU, (a) and (b) on every ADMM path: warp-per-tile and lane-per-QP (also against each other), the CTA kernel
    (5- and 3-buffer, time-varying), the dense kernel and the chunked main loop with compaction and a CTA straggler tail.
(d) A rejected update leaves the solver unchanged; an update before setup is plain problem data."""
import copy

import numpy as np
import pytest
import torch

import parity_cases as pc
import python_mpc_b200 as pm
from python_mpc_b200 import workloads
from oracle import c_oracle, osqp_admm, ref_qp, workload_qp
from test_setup_scaling import B, RES_ATOL, RES_RTOL, SHAPES, Problem, _bitwise, _with

RHO_TOL, INF = osqp_admm.RHO_TOL, osqp_admm.OSQP_INFTY
# every path runs exactly 30 iterations: a termination test at 25 that nothing passes, then the iteration limit
SOLVE30 = dict(eps_abs=1e-12, eps_rel=1e-12, max_iter=30, check_termination=25, warm_start=False)
ITERS = (1, 2, 7)
# warm-started sequences against the oracle
SEQ = dict(rho=1.0, eps_abs=1e-4, eps_rel=1e-4, max_iter=1000, warm_start=True)
ITER_TOL = 1e-10
HORIZONS = (1, 2, 7, 31, 32, 33)


class Bounds:
    """The bounds of a problem: state bounds per stage lo, hi (N+1, nx), input bounds, and whether the state bounds are a
    per-stage box (else lo / hi hold xmin / xmax at every stage)."""

    def __init__(self, lo, hi, umin, umax, box):
        self.lo, self.hi, self.umin, self.umax, self.box = lo, hi, umin, umax, box

    @classmethod
    def of(cls, prob):
        if prob.box is not None:
            return cls(prob.box[0].copy(), prob.box[1].copy(), prob.umin.copy(), prob.umax.copy(), True)
        t = lambda v: np.tile(v, (prob.N + 1, 1))
        return cls(t(prob.xmin), t(prob.xmax), prob.umin.copy(), prob.umax.copy(), False)

    def copy(self):
        return Bounds(self.lo.copy(), self.hi.copy(), self.umin.copy(), self.umax.copy(), self.box)

    def kwargs(self):
        """update_bounds(...) arguments (a box replaces the state bounds of every stage)."""
        if self.box:
            return dict(stage_lo=self.lo, stage_hi=self.hi, umin=self.umin, umax=self.umax)
        return dict(xmin=self.lo[0], xmax=self.hi[0], umin=self.umin, umax=self.umax)

    def apply(self, prob):
        """The problem with these bounds (the constructor's xmin / xmax stay when the state bounds are a box)."""
        p = copy.copy(prob)
        p.umin, p.umax = self.umin, self.umax
        if self.box:
            p.box = (self.lo, self.hi)
        else:
            p.box, p.xmin, p.xmax = None, self.lo[0], self.hi[0]
        return p


def finite_problem(nx, nu, slack, N, seed, f32=False, box=None, batch=B):
    """A seeded Problem whose bounds are all finite (T3 brings in the first infinite bound)."""
    p = Problem(nx, nu, slack, N, seed, f32=f32, box=box, batch=batch)
    fin = lambda v, s: np.where(np.isfinite(v), v, s * 4.0)
    p.xmin, p.xmax = fin(p.xmin, -1), fin(p.xmax, 1)
    if p.box is not None:
        p.box = (fin(p.box[0], -1), fin(p.box[1], 1))
    return p


def _rnd(dtype):
    return (lambda v: np.asarray(v, dtype=np.float32).astype(np.float64)) if dtype == torch.float32 else \
           (lambda v: np.asarray(v, dtype=np.float64))


def row_types(prob, bd, E):
    """OSQP's constr_type (auxil.c: set_rho_vec) of the bx and bu rows of every QP, from the scalings E (B, ncon) of the
    device: -1 unbounded, 1 equality, 0 inequality.  Asserts that no finite scaled gap lies within 1 % of RHO_TOL, so
    that f32 and f64 decide every row alike."""
    N, nx, nu = prob.N, prob.nx, prob.nu
    bx0, bu0 = (N + 1) * nx, 2 * (N + 1) * nx
    out = []
    for El, lo, hi in ((E[:, bx0:bu0].reshape(-1, N + 1, nx), bd.lo, bd.hi),
                       (E[:, bu0:].reshape(-1, N, nu), np.tile(bd.umin, (N, 1)), np.tile(bd.umax, (N, 1)))):
        l, u = El * np.maximum(lo, -INF), El * np.minimum(hi, INF)
        unc = (l < -INF * osqp_admm.MIN_SCALING) & (u > INF * osqp_admm.MIN_SCALING)
        gap = u - l
        fin = np.isfinite(lo) & np.isfinite(hi) & np.ones_like(El, dtype=bool)
        assert (np.abs(gap[fin] / RHO_TOL - 1) > 0.01).all(), "a scaled gap within 1 % of RHO_TOL"
        out.append(np.where(unc, -1, np.where(gap < RHO_TOL, 1, 0)).reshape(El.shape[0], -1))
    return np.concatenate(out, axis=1)


def split_gap(e):
    """A gap g for which the row of scalings e (B, stages) is an equality after scaling (e g < RHO_TOL at some stage) in
    some QPs and an inequality in the others, no scaled gap within 2 % of RHO_TOL.  Returns (the smaller of the two sets,
    g); (0, g) with every QP on the equality side when the QPs scale the row alike."""
    m, v = e.min(axis=1), np.unique(e)
    best = (0, v[-1] * 1.5)
    for a, b in zip(v[:-1], v[1:]):
        if b > 1.05 * a:
            t = np.sqrt(a * b)
            n = int((m < t).sum())
            if min(n, len(m) - n) > best[0]:
                best = (min(n, len(m) - n), t)
    return best[0], RHO_TOL / best[1]


def transitions(prob, E, x, dtype):
    """T1..T7 from the bounds of `prob` (L0) as [(name, bounds, which QPs refactor: 'some' | 'any' | 'all' | 'none')].
    T1 and T6 narrow the state row that splits the batch best (split_gap) around the current solution x (B, nvar)."""
    r = _rnd(dtype)
    N, nx, nu = prob.N, prob.nx, prob.nu
    L0 = Bounds.of(prob)
    bx = lambda k, j: (N + 1) * nx + k * nx + j

    def narrow(bd, ks, skip=()):
        """(bounds, 'some' when the row splits the batch, else 'any')"""
        n, g, j = max(split_gap(E[:, [bx(k, j) for k in ks]]) + (-j,) for j in range(nx) if j not in skip)
        j = -j
        v = x[:, [k * nx + j for k in ks]]
        c = float(np.median(v[np.isfinite(v)])) if np.isfinite(v).any() else 0.0   # (no solution: infeasible QPs)
        bd.lo[ks, j], bd.hi[ks, j] = r(c - g / 2), r(c + g / 2)
        return bd, "some" if n else "any"
    L1, some = narrow(L0.copy(), list(range(N + 1)), skip=(nx - 1,))
    L3 = L0.copy(); L3.lo[:, nx - 1], L3.hi[:, nx - 1] = -np.inf, np.inf
    L5 = L0.copy(); L5.umin[nu - 1] = L5.umax[nu - 1] = r(0.5 * (L0.umin[nu - 1] + L0.umax[nu - 1]))
    L6 = L0.copy(); L6.box = True
    L6, some6 = narrow(L6, [min(1, N)])
    L7 = L6.copy()                                   # the box and the input bounds move by a representable step
    L7.lo, L7.hi = r(L6.lo + 0.125), r(L6.hi + 0.125)
    L7.umin, L7.umax = r(L6.umin - 0.0625), r(L6.umax - 0.0625)
    return [("T1", L1, some), ("T2", L0, some), ("T3", L3, "all"), ("T4", L0, "all"), ("T5", L5, "all"),
            ("T5 back", L0, "all"), ("T6", L6, some6), ("T7", L7, "none")]


def _changed(prob, old, new, E, expect, tag):
    """The QPs whose row types change, asserted against the expectation of the transition."""
    ch = (row_types(prob, old, E) != row_types(prob, new, E)).any(axis=1)
    n = int(ch.sum())
    assert {"some": 0 < n < len(ch), "any": n > 0, "all": n == len(ch), "none": n == 0}[expect], (tag, expect, n)
    return ch


def _close(a, b, tol):
    """a and b (device tensors) have NaN (no solution: an infeasibility certificate) in the same places and agree
    elsewhere to tol relative to max(1, |b|)."""
    na, nb = a.isnan(), b.isnan()
    assert torch.equal(na, nb)
    if bool(na.all()):
        return True
    return float((a - b)[~na].abs().max()) <= tol * max(1.0, float(b[~nb].abs().max()))


def _scal(s):
    return [t.cpu().numpy().astype(np.float64) for t in s.scaling()]


def _out(s):
    x, y, _ = s.solution(want_y=True)
    inf = s.info()
    return x, y, inf.iter, inf.status_val, inf.pri_res, inf.dua_res


# ---------------------------------------------------------------------------------------------------------------------
# (a) a refactor equals a fresh setup, bit for bit
def check_refactor_equals_fresh(be, prob, dtype):
    """solver 1: set up with L0, then T1..T7 in sequence through update_bounds, a 30-iteration solve after each; solver 2,
    after each update: a fresh setup with the new bounds.  Scaling, x and y after cold_start(); iterate(k), and the
    30-iteration solve agree to the bit.  (Solver 1 solves before every update, so that whatever a solve leaves behind —
    the factor form of the records, the dense path's inverse, the per-stage box buffers — is there to go stale.)"""
    s = prob.setup(prob.solver(be, dtype, **SOLVE30))
    s.solve()
    E = _scal(s)[1]
    x = s.solution()[0].cpu().double().numpy()
    prev = Bounds.of(prob)
    split = {}
    for name, bd, expect in transitions(prob, E, x, dtype):
        tag = (prob.nx, prob.nu, prob.slack, prob.N, prob.tv, prob.shared, dtype, name)
        split[name] = expect == "some"
        _changed(prob, prev, bd, E, expect, tag)
        s.update_bounds(**bd.kwargs())
        pf = bd.apply(prob)
        f = pf.setup(pf.solver(be, dtype, **SOLVE30))
        for a, b in zip(s.scaling(), f.scaling()):
            assert _bitwise(a, b), tag
        # the solve first: it reads the factor in the form the update left it (on the CTA path Linv' Linv; a solve or an
        # iterate on another path re-factors every QP into its own form, which would hide a refactor in the wrong form)
        s.solve(); f.solve()
        for a, b in zip(_out(s), _out(f)):
            assert _bitwise(a, b), (tag, "solve")
        for k in ITERS:
            s.cold_start().iterate(k); f.cold_start().iterate(k)
            for a, b in zip(s.solution(want_y=True)[:2], f.solution(want_y=True)[:2]):
                assert _bitwise(a, b), (tag, k)
        s.solve(); f.solve()            # (and the solve path's factor form again before the next update)
        for a, b in zip(_out(s), _out(f)):
            assert _bitwise(a, b), (tag, "solve")
        assert int(_out(s)[2].max()) == 30, tag
        f.close()
        prev = bd
    s.close()
    return split


def refactor_problems(dtype, shapes=SHAPES, per_shape=2, box=None, modes=None):
    """Problems for (a): every shape, the horizons of HORIZONS spread over the shapes (different ones in f32), the model
    modes cycled through by seed (or restricted to `modes`: a predicate of Problem)."""
    f32 = dtype == torch.float32
    out = []
    for si, (nx, nu, slack) in enumerate(SHAPES):
        if (nx, nu, slack) not in shapes:
            continue
        for j in range(per_shape):
            N = HORIZONS[(per_shape * si + j + (3 if f32 else 0)) % len(HORIZONS)]
            seed = 40 * si + 7 * j + (1 if f32 else 0)
            while modes is not None and not modes(Problem(nx, nu, slack, 1, seed)):
                seed += 1
            out.append(finite_problem(nx, nu, slack, N, seed, f32=f32, box=box))
    return out


def run_refactor_equals_fresh(be, dtype, **kw):
    """Returns the modes seen; asserts that T1 and T6 each split the batch (some QPs refactor, others not) in a third of the problems at least
    (a row narrowed at every stage splits only where the smallest scaling of the row over the stages differs by QP)."""
    seen, splits = set(), []
    for prob in refactor_problems(dtype, **kw):
        split = check_refactor_equals_fresh(be, prob, dtype)
        seen.add((prob.tv, prob.shared, prob.box is not None, prob.N))
        splits.append((split["T1"], split["T6"]))
    assert min(sum(a for a, _ in splits), sum(b for _, b in splits)) >= len(splits) // 3, splits
    return seen


# ---------------------------------------------------------------------------------------------------------------------
# (b) against OSQP's update semantics: one oracle object per sampled QP for the whole warm-started sequence
def _oracle_lu(prob, bd, b, x0):
    _, _, _, l, u = ref_qp.assemble(bd.apply(prob).qp(b, x0=x0))
    return dict(l=l, u=u)


def _compare_solve(got, r, tag):
    x, y, it, st, pri, dua = got
    assert (it, st) == (r.info.iter, r.info.status_val), (tag, it, st, r.info.iter, r.info.status)
    if r.info.status_val in (1, 2, -2):
        assert pc.rel(x, r.x) < 1e-6 and pc.rel(y, r.y) < 1e-6, tag
        atol = RES_ATOL * max(1.0, float(np.abs(r.x).max()), float(np.abs(r.y).max()))
    else:
        assert np.isnan(x).all() and np.isnan(y).all(), tag
        atol = RES_ATOL
    for g, ref in ((pri, r.info.pri_res), (dua, r.info.dua_res)):
        assert abs(g - ref) <= atol + RES_RTOL * abs(ref), (tag, g, ref)


def check_oracle_sequence(be, prob, iters=5, nsamples=6):
    """A warm-started sequence: T1..T7 alternating with new initial states (f64).  Per sampled QP (some that T1 turns into
    equalities, some that it does not): status and iteration count equal to the oracle's, x and y within 1e-6, the
    residuals within RES_RTOL / RES_ATOL; the QPs whose constr_type changed in the oracle are those predicted from the
    device's E; after each update, `cold_start(); iterate(k)` of a second solver against the oracle's iterate() x k.
    Returns the device's results of every step (for the bitwise comparison of two kernels)."""
    dt = torch.float64
    s = prob.setup(prob.solver(be, dt, **SEQ))
    s2 = prob.setup(prob.solver(be, dt, **SEQ))
    s.solve()
    E = _scal(s)[1]
    x = s.solution()[0].cpu().numpy()
    steps = transitions(prob, E, x, dt)
    assert steps[0][2] == "some", "T1 does not split the batch"
    rng = np.random.default_rng(prob.N)
    x0s = [prob.x0 * f + 0.05 * rng.standard_normal(prob.x0.shape) for f in (0.5, -0.8, 1.2)]
    new_x0 = [("x0", v, "none") for v in x0s]
    seq = [steps[0], new_x0[0], steps[1], steps[2], new_x0[1], steps[3], steps[4], steps[5], steps[6], new_x0[2], steps[7]]
    # the sampled QPs: both sides of T1's split
    ch1 = _changed(prob, Bounds.of(prob), steps[0][1], E, steps[0][2], "T1")
    eq, ne = np.flatnonzero(ch1), np.flatnonzero(~ch1)
    samples = sorted(set(eq[:nsamples // 2].tolist() + ne[:nsamples // 2].tolist() + [0, prob.B - 1]))
    bd, x0 = Bounds.of(prob), prob.x0
    oracles = {b: osqp_admm.OSQP().setup(*ref_qp.assemble(prob.qp(b)), **SEQ) for b in samples}
    results = []

    def compare(tag):
        got = [t.cpu().numpy() for t in _out(s)]
        results.append(_out(s))
        for b in samples:
            _compare_solve([g[b] for g in got], oracles[b].solve(), tag + (b,))
    compare(("setup",))
    for name, what, expect in seq:
        tag = (prob.nx, prob.nu, prob.slack, prob.N, prob.tv, prob.shared, name)
        if name == "x0":
            x0 = what
            s.update(x_init=x0); s2.update(x_init=x0)
            ch = np.zeros(prob.B, dtype=bool)
        else:
            ch = _changed(prob, bd, what, E, expect, tag)
            bd = what
            s.update_bounds(**bd.kwargs()); s2.update_bounds(**bd.kwargs())
        types = row_types(prob, bd, E)
        for b in samples:
            o = oracles[b]
            old = o.constr_type.copy()
            o.update(**_oracle_lu(prob, bd, b, x0[b]))
            assert bool((old != o.constr_type).any()) == bool(ch[b]), (tag, b)
            assert np.array_equal(o.constr_type[(prob.N + 1) * prob.nx:], types[b]), (tag, b)
        # the iterates after the update, from a cold start
        s2.cold_start().iterate(iters)
        xi, yi, _ = s2.solution(want_y=True)
        xi, yi = xi.cpu().numpy(), yi.cpu().numpy()
        for b in samples:
            o = oracles[b]
            keep = o.x, o.z, o.y
            o.x, o.z, o.y = np.zeros(o.n), np.zeros(o.m), np.zeros(o.m)
            for _ in range(iters):
                o.iterate()
            assert pc.rel(xi[b], o.D * o.x) < ITER_TOL and pc.rel(yi[b], o.cinv * o.E * o.y) < ITER_TOL, (tag, b)
            o.x, o.z, o.y = keep
        s.solve()
        compare(tag)
    s.close(); s2.close()
    return results


def oracle_problems(be, shapes=SHAPES, tv=None):
    """Problems for (b): every shape, per-QP models, no box (T6 brings the first one), the first seed whose T1 splits
    the batch."""
    out = []
    for si, (nx, nu, slack) in enumerate(SHAPES):
        if (nx, nu, slack) not in shapes:
            continue
        seed = 11 * si
        while True:
            prob = finite_problem(nx, nu, slack, 3 + 2 * si, seed, box=False)
            if not prob.shared and (tv is None or prob.tv == tv):
                s = prob.setup(prob.solver(be, torch.float64))
                E = _scal(s)[1]
                s.close()
                if transitions(prob, E, np.zeros((prob.B, (prob.N + 1) * prob.nx)), torch.float64)[0][2] == "some":
                    break
            seed += 1
        out.append(prob)
    return out


def run_oracle_sequences(be, **kw):
    return [check_oracle_sequence(be, prob) for prob in oracle_problems(be, **kw)]


def check_closed_loop_type_switch(be, B_=6, steps=14, rho=5.0, N=20, seed=43, switch=(4, 9)):
    """LateralMPC.closed_loop_batch(bounds_at=) with a switch that makes the yaw-error row an equality after scaling
    (xmin[2] = xmax[2] - 1e-6) and back, against oracle_closed_loop_batch(schedule=), which refactors on a type change:
    iteration counts of every step equal, applied inputs and trajectories to 1e-9."""
    wl = workloads.LateralWorkload(B_, N, True, True, seed, torch.float64)
    eq = wl.xmin.copy(); eq[2] = wl.xmax[2] - 1e-6
    sched = {switch[0]: dict(xmin=eq), switch[1]: dict(xmin=wl.xmin)}
    ctl = wl.make_controller(_backend=be, rho=rho, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
    traj, us, its = ctl.closed_loop_batch(wl.x0, wl.xr, wl.speed, steps=steps, bounds_at=lambda k: sched.get(k))
    Pu, A0, Pv, q, Av, l, u, perm = workload_qp.lateral_batch_csc(wl)
    Ad, Bd = workload_qp.lateral_models(wl.speed)
    At, Bt, _ = ref_qp.augment_increment(Ad, Bd, None)
    nx = 5
    bx = slice((N + 1) * nx, 2 * (N + 1) * nx)
    rows = {}
    for k, bd in sched.items():
        lk = l[0].copy(); lk[bx] = np.tile(bd["xmin"], N + 1)
        rows[k] = (lk, u[0].copy())
    it, st, ua, tr, _ = c_oracle.closed_loop_batch(Pu, A0, Pv, q, Av, l, u, At, Bt, wl.x0, steps, (N + 1) * nx, perm=perm,
                                                   schedule=rows, rho=rho, eps_abs=1e-4, eps_rel=1e-4)
    assert (st == 1).all()
    assert np.array_equal(it, its.cpu().numpy().T)
    assert np.abs(ua - us.cpu().numpy().transpose(1, 0, 2)).max() < 1e-9
    assert np.abs(tr - traj.cpu().numpy().transpose(1, 0, 2)).max() < 1e-9
    # (the switch changes the iteration counts: the new type is in force)
    assert not np.array_equal(it[:, switch[0]:switch[1]], it[:, switch[0] - 1:switch[1] - 1])


def check_single_vehicle(be, N=20, seed=3):
    """LateralMPC.solve (a batch of one; on the GPU the dense kernel): warm-started solves through T1- and T5-type updates
    (a yaw-error row made an equality, the delta-u bound closed) against the continued oracle."""
    wl = workloads.LateralWorkload(1, N, True, True, seed, torch.float64, shared_speed=11.0)
    ctl = wl.make_controller(_backend=be, rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
    o = osqp_admm.OSQP().setup(*ref_qp.assemble(workload_qp.lateral_qp(wl, 0)), rho=5.0, eps_abs=1e-4, eps_rel=1e-4,
                               warm_start=True)
    eq = wl.xmin.copy(); eq[2] = wl.xmax[2] - 1e-6
    seq = [None, dict(xmin=eq), None, dict(umin=np.zeros(1), umax=np.zeros(1)), dict(xmin=wl.xmin, umin=wl.umin,
                                                                                      umax=wl.umax), None]
    x0, cur = wl.x0[0].copy(), dict(xmin=wl.xmin, xmax=wl.xmax, umin=wl.umin, umax=wl.umax)
    for i, upd in enumerate(seq):
        if upd is not None:
            ctl.update_bounds(**upd)
            cur.update(upd)
        if i:
            x0 = 0.7 * x0
        ctl.solve(x0, wl.xr[0])
        qp = ref_qp.canonical(N, *_lateral_model(wl), None, np.r_[wl.Q, 0.0], np.r_[wl.Q, 0.0], wl.R,
                              np.r_[wl.xr[0], 0.0], cur["xmin"], cur["xmax"], cur["umin"], cur["umax"], x0,
                              slack=True, W=wl.W, S=wl.S)
        _, _, _, l, u = ref_qp.assemble(qp)
        if i:
            old = o.constr_type.copy()
            o.update(l=l, u=u)
            assert bool((old != o.constr_type).any()) == (upd is not None and i in (1, 3, 4)), i
        r = o.solve()
        assert int(ctl.last.info.iter[0]) == r.info.iter and r.info.status_val == 1, (i, int(ctl.last.info.iter[0]), r.info.iter)
        assert pc.rel(ctl.last.x[0].cpu().numpy(), r.x) < 1e-6, i


def _lateral_model(wl):
    Ad, Bd = workload_qp.lateral_model(float(wl.speed[0]))
    At, Bt, _ = ref_qp.augment_increment(Ad, Bd, None)
    return At, Bt


# ---------------------------------------------------------------------------------------------------------------------
# (d) a rejected update; an update before setup
def check_rejected_update(be, dtype=torch.float64):
    """Inverted bounds, global or per-stage, are rejected and leave the solver as it was: the next solve equals, bit for
    bit, a solve without the rejected call — also when the rejected call carries a type change in another row."""
    for si, (nx, nu, slack) in enumerate(SHAPES):
        prob = finite_problem(nx, nu, slack, 5 + si, seed=600 + si, box=si % 2 == 0)
        E = None
        outs = []
        for reject in (False, True):
            s = prob.setup(prob.solver(be, dtype, **dict(SEQ, max_iter=200)))
            s.solve()
            if E is None:
                E = _scal(s)[1]
                T1 = transitions(prob, E, s.solution()[0].cpu().double().numpy(), dtype)[0][1]
            if reject:
                bad = T1.copy(); bad.lo[:, nx - 1] = bad.hi[:, nx - 1] + 1.0
                with pytest.raises(pm.MpcError, match="lower bound must be lower than or equal to upper bound"):
                    s.update_bounds(**bad.kwargs())
                bad = T1.copy(); bad.box = True; bad.lo[-1, nx - 1] = bad.hi[-1, nx - 1] + 1.0
                with pytest.raises(pm.MpcError, match="lower bound must be lower than or equal to upper bound"):
                    s.update_bounds(**bad.kwargs())
                bad = T1.copy(); bad.umin[0] = bad.umax[0] + 1.0
                with pytest.raises(pm.MpcError, match="lower bound must be lower than or equal to upper bound"):
                    s.update_bounds(**bad.kwargs())
            s.update(x_init=0.5 * prob.x0).solve()
            outs.append(_out(s) + tuple(s.scaling()))
            s.close()
        for a, b in zip(*outs):
            assert _bitwise(a, b), (nx, nu, slack)


def check_update_before_setup(be, dtype):
    """update_bounds before the first setup is problem data: the solve equals a solver constructed with those bounds —
    a narrowed row, an unbounded one (inf_bounds) and a per-stage box."""
    r = _rnd(dtype)
    for si, (nx, nu, slack) in enumerate(SHAPES):
        prob = finite_problem(nx, nu, slack, 4 + si, seed=700 + si, f32=dtype == torch.float32, box=False)
        bd = Bounds.of(prob)
        bd.lo[:, 0], bd.hi[:, 0] = r(bd.lo[:, 0] * 0.5), r(bd.lo[:, 0] * 0.5 + 1e-6)
        bd.lo[:, nx - 1], bd.hi[:, nx - 1] = -np.inf, np.inf
        bd.umin[0] = bd.umax[0] = r(0.5 * (bd.umin[0] + bd.umax[0]))
        for box in (False, True):
            bd.box = box
            a = prob.solver(be, dtype, **SOLVE30)
            a.update_bounds(**bd.kwargs())
            prob.setup(a).solve()
            pf = bd.apply(prob)
            f = pf.setup(pf.solver(be, dtype, **SOLVE30)).solve()
            for x, y in zip(_out(a) + tuple(a.scaling()), _out(f) + tuple(f.scaling())):
                assert _bitwise(x, y), (nx, nu, slack, box)
            a.close(); f.close()


# ---------------------------------------------------------------------------------------------------------------------
# (c) GPU paths that neither mpcb_iterate nor the emu build reach
def check_dense_path(be, N=12, seed=1):
    """The dense kernel (shared model, xr = 0, f64, N + 1 <= 32: every QP has the same scaling and changes type alike):
    (a) against a fresh setup with the dense path, then a warm-started sequence through T1 and T5 with dense = 1 against
    dense = 0 (equal iteration counts, x to 1e-9) and the oracle."""
    for si, (nx, nu, slack) in enumerate(SHAPES):
        seed_ = 20 * si + seed
        while not Problem(nx, nu, slack, 1, seed_).shared:
            seed_ += 1
        prob = finite_problem(nx, nu, slack, N, seed_, box=False)
        prob.Xr[:] = 0.0
        _with(be, dict(dense=1), lambda: check_refactor_equals_fresh(be, prob, torch.float64))
        runs = []
        for dense in (1, 0):
            def run():
                s = prob.setup(prob.solver(be, torch.float64, **SEQ))
                s.solve()
                T = dict((n, bd) for n, bd, _ in transitions(prob, _scal(s)[1], s.solution()[0].cpu().numpy(), torch.float64))
                bds = [Bounds.of(prob), T["T1"], T["T2"], T["T5"], T["T5 back"]]
                out = [[t.clone() for t in _out(s)]]
                for bd in bds[1:]:
                    s.update_bounds(**bd.kwargs())
                    s.update(x_init=prob.x0 * 0.9).solve()
                    out.append([t.clone() for t in _out(s)])
                s.close()
                return out, bds
            runs.append(_with(be, dict(dense=dense), run))
        (d, bds), (a, _) = runs
        for k, (od, oa) in enumerate(zip(d, a)):
            assert torch.equal(od[2], oa[2]) and torch.equal(od[3], oa[3]), (nx, nu, slack, k)
            assert _close(od[0], oa[0], 1e-9), (nx, nu, slack, k)
        # the oracle, continued through the same updates
        for b in (0, prob.B - 1):
            o = osqp_admm.OSQP().setup(*ref_qp.assemble(prob.qp(b)), **SEQ)
            for k, bd in enumerate(bds):
                x0 = prob.x0[b] if k == 0 else prob.x0[b] * 0.9
                if k:
                    o.update(**_oracle_lu(prob, bd, b, x0))
                _compare_solve([t.cpu().numpy()[b] for t in d[k]], o.solve(), (nx, nu, slack, k, b))


def check_chunked_main_loop(be, B_=10240, N=10, seed=0):
    """About 10240 QPs under the default options: the warp-per-tile kernel on the home workspace, compaction, the CTA kernel
    for the stragglers.  T1 on part of the batch, then a warm-started solve: the chunked schedule without the CTA kernel
    ("cta" 0) equals the unchunked one ("retile" 0) bit for bit, the default schedule agrees with both to 1e-10; against
    the oracle on the stragglers and on a spread of QPs."""
    prob = finite_problem(4, 1, True, N, seed, box=False, batch=B_)
    assert not prob.shared and not prob.tv
    runs = []
    for opts in (dict(), dict(cta=0), dict(cta=0, retile=0)):
        def run():
            s = prob.setup(prob.solver(be, torch.float64, capacity=B_, **SEQ))
            s.solve()
            E = _scal(s)[1]
            T1 = transitions(prob, E, s.solution()[0].cpu().numpy(), torch.float64)[0][1]
            ch = _changed(prob, Bounds.of(prob), T1, E, "some", "T1")
            s.update_bounds(**T1.kwargs())
            s.update(x_init=prob.x0 * 0.8).solve()
            out = [t.clone() for t in _out(s)]
            s.close()
            return out, ch, T1
        runs.append(_with(be, opts, run))
    (d, ch, T1), (c0, _, _), (r0, _, _) = runs
    for a, b in zip(c0, r0):
        assert _bitwise(a, b)
    it = d[2].cpu().numpy()
    assert np.array_equal(it, c0[2].cpu().numpy()) and torch.equal(d[3], c0[3]) and len(np.unique(it)) >= 3
    for a, b in zip(d[:2], c0[:2]):
        assert _close(a, b, 1e-10)
    slow = np.argsort(it, kind="stable")[-3:]
    samples = sorted(set(slow.tolist() + list(range(0, B_, B_ // 6)) + np.flatnonzero(ch)[:2].tolist()
                         + np.flatnonzero(~ch)[:2].tolist()))
    got = [t.cpu().numpy() for t in d]
    for b in samples:
        o = osqp_admm.OSQP().setup(*ref_qp.assemble(prob.qp(b)), **SEQ)
        o.solve()
        o.update(**_oracle_lu(prob, T1, b, prob.x0[b] * 0.8))
        _compare_solve([g[b] for g in got], o.solve(), ("chunked", b, bool(ch[b])))


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_refactor_equals_fresh_setup_cpu(emu_backend, dtype):
    seen = run_refactor_equals_fresh(emu_backend, dtype)
    assert {tv for tv, _, _, _ in seen} == {False, True} and {sh for _, sh, _, _ in seen} == {False, True}


def test_update_sequence_against_oracle_cpu(emu_backend):
    run_oracle_sequences(emu_backend)


def test_closed_loop_type_switch_cpu(emu_backend):
    check_closed_loop_type_switch(emu_backend)


def test_single_vehicle_type_changes_cpu(emu_backend):
    check_single_vehicle(emu_backend)


def test_rejected_update_leaves_solver_unchanged_cpu(emu_backend):
    check_rejected_update(emu_backend)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_update_before_setup_is_problem_data_cpu(emu_backend, dtype):
    check_update_before_setup(emu_backend, dtype)


PATHS = {"tma": dict(cta=0), "lane": dict(cta=0, tma=0), "cta": dict()}


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_refactor_equals_fresh_setup_gpu(cuda_backend, dtype, path):
    _with(cuda_backend, PATHS[path], lambda: run_refactor_equals_fresh(cuda_backend, dtype))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_refactor_equals_fresh_setup_cta_three_buffer_gpu(cuda_backend, dtype, monkeypatch):
    monkeypatch.setenv("MPCB_NO_CTA_DEEP", "1")
    run_refactor_equals_fresh(cuda_backend, dtype)


@pytest.mark.gpu
def test_update_sequence_against_oracle_gpu(cuda_backend, monkeypatch):
    """every path; the warp-per-tile and the lane-per-QP kernels agree bit for bit through the whole sequence"""
    tma = _with(cuda_backend, PATHS["tma"], lambda: run_oracle_sequences(cuda_backend))
    lane = _with(cuda_backend, PATHS["lane"], lambda: run_oracle_sequences(cuda_backend))
    for a, b in zip(tma, lane):
        for sa, sb in zip(a, b):
            for x, y in zip(sa, sb):
                assert _bitwise(x, y)
    run_oracle_sequences(cuda_backend)                      # the CTA kernel (5-buffer; time-varying problems included)
    monkeypatch.setenv("MPCB_NO_CTA_DEEP", "1")
    run_oracle_sequences(cuda_backend, tv=True)             # 3-buffer, stage models staged by TMA


@pytest.mark.gpu
def test_closed_loop_and_single_vehicle_gpu(cuda_backend):
    check_closed_loop_type_switch(cuda_backend)
    check_single_vehicle(cuda_backend)


@pytest.mark.gpu
def test_dense_path_after_type_changes_gpu(cuda_backend):
    check_dense_path(cuda_backend)


@pytest.mark.gpu
def test_chunked_main_loop_after_type_change_gpu(cuda_backend):
    check_chunked_main_loop(cuda_backend)


@pytest.mark.gpu
def test_rejected_update_and_update_before_setup_gpu(cuda_backend):
    check_rejected_update(cuda_backend)
    for dt in (torch.float64, torch.float32):
        check_update_before_setup(cuda_backend, dt)
