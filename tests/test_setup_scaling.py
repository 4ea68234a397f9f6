"""prob.setup() on its own: the Ruiz equilibration (D, E, c; mpcb_get_scaling) against the oracle's scale_data at every
compiled shape, the edge horizons and pass counts, in both precisions; the two Ruiz kernels (scale_warp_kernel for
N + 1 <= 32, scale_one otherwise) against each other; the cached factor in both forms (Linv and Linv' Linv) through the
first iterates; sigma, alpha and scaling set to other values than OSQP's defaults; settings changed after a setup; the
scaling kept by update, update_bounds, compaction and closed-loop steps, as OSQP's update keeps it; and the premise of the
shared-KKT dense path, that a batch with one model and xr = 0 has one scaling.  CPU (tests/emu: scale_one and the
lane-per-QP loop, the same source as host loops) and GPU (-m gpu).

The random batches have B = 37 QPs in a solver of capacity 64: the last tile is ragged, the leading dimension exceeds the
batch, and the batch is not a multiple of the 8 QPs per CTA of scale_warp_kernel."""
import itertools

import numpy as np
import pytest
import torch

import parity_cases as pc
import python_mpc_b200 as pm
from python_mpc_b200 import vehicle_models, workloads
from oracle import osqp_admm, ref_qp, workload_qp

B, CAP = 37, 64
SAMPLES = (0, 31, 32, B - 1)
SHAPES = ((4, 1, False), (4, 1, True), (5, 1, False), (5, 1, True), (4, 2, False), (6, 2, False), (8, 2, False))
HORIZONS = (1, 2, 7, 30, 31, 32, 33, 64)
# (time_varying, shared_model, affine term g): cycled through by seed
MODES = ((False, False, False), (False, True, True), (True, False, True), (False, False, True), (True, False, False),
         (False, True, False))
# D, E, c against the oracle, elementwise relative: f64 (the same operations, rsqrt to the last bit or two, another order
# of the sum in c) and f32 (against the f64 oracle on the same f32-representable data)
SCALE_TOL = {torch.float64: 1e-13, torch.float32: 1e-5}
ITER_TOL = 1e-11                    # x, y after the first iterations, f64
RES_RTOL, RES_ATOL = 1e-6, 1e-10    # residuals against the oracle (as test_fused_termination.py)
DEFAULT_OPTS = dict(warp_setup=1, cta=1, dense=1, retile=1, retile_min_batch=4096, certificates=1)


def _with(be, opts, fn):
    for k, v in opts.items():
        be.set_option(k, v)
    try:
        return fn()
    finally:
        for k, v in DEFAULT_OPTS.items():
            be.set_option(k, v)


def _bitwise(a, b):
    """Equal to the bit, NaN (the solution of an infeasible QP) included."""
    return a.shape == b.shape and a.dtype == b.dtype and bool(((a == b) | (a.isnan() & b.isnan())).all())


def _rel(a, b):
    """Elementwise relative deviation (the oracle's scalings are positive)."""
    a = np.asarray(a, dtype=np.float64)
    return float(np.max(np.abs(a - b) / np.abs(b)))


class _ScaleOnly(osqp_admm.OSQP):
    """The oracle's setup without the KKT factorisation (only D, E, c are read)."""

    def _factor(self):
        pass


class Problem:
    """A seeded random batch of MPC QPs of one shape (modelled on parity_cases.check_random_problems): models per QP or
    shared, time-invariant or per stage, with or without affine term; weights with zeros; bounds with infinities,
    optionally per-stage boxes.  `f32`: every number is f32-representable, nonzero weights in [0.05, 50] (no norm near
    the MIN/MAX_SCALING clamps).  `wide`: weights from 1e-8 to 1e8, a slack column with W = S = 0 and a model column of
    zeros."""

    def __init__(self, nx, nu, slack, N, seed, f32=False, wide=False, box=None, batch=B):
        rng = np.random.default_rng(seed)
        self.nx, self.nu, self.slack, self.N, self.B = nx, nu, slack, N, batch
        self.tv, self.shared, has_g = MODES[seed % len(MODES)]
        r = (lambda a: np.asarray(a, dtype=np.float32).astype(np.float64)) if f32 else (lambda a: np.asarray(a, dtype=np.float64))
        stages, nm = (N if self.tv else 1), (1 if self.shared else batch)
        A = np.eye(nx) + 0.15 * rng.standard_normal((nm, stages, nx, nx))
        Bm = 0.3 * rng.standard_normal((nm, stages, nx, nu))
        if wide:
            A[..., :, nx - 1] = 0.0          # a state that nothing depends on
            Bm[..., :, nu - 1] = 0.0         # an input that moves nothing
        self.A, self.Bm = r(A), r(Bm)
        self.g = r(0.05 * rng.standard_normal((nm, stages, nx))) if has_g else None

        def w(n, zero=0.25, wide=wide):
            v = np.exp(rng.uniform(np.log(1e-8), np.log(1e8), n)) if wide else rng.uniform(0.05, 50.0, n)
            return r(v * (rng.random(n) > zero))
        self.Q, self.QN, self.R = w(nx), w(nx), w(nu, 0.2)
        # (the slack weights stay in [0.05, 50] with `wide`: a slack column whose norm is its P entry alone is equilibrated
        # to W D^2 = 1 by the first pass, and once the cost scaling c clamps at 1 / MAX_SCALING the next pass sees the norm
        # c W D^2 = MIN_SCALING up to the last bit of 1/sqrt — a tie that the rounding of each implementation decides)
        self.W = w(nx, wide=False) if slack else None
        self.S = r(np.where(rng.random(nx) > 0.3, rng.uniform(0.05, 50.0, nx) if wide or f32 else 1.0, 0.0)) if slack else None
        if slack and wide:
            self.W[0] = self.S[0] = 0.0      # a slack column of zeros: zero norm, scaling 1
            self.W[self.S == 0] = 0.0        # (no column with a P entry alone, see above)
        xmax = r(rng.uniform(0.5, 4.0, nx)); xmin = r(-rng.uniform(0.5, 4.0, nx))
        inf = rng.random(nx) < 0.3
        xmax[inf], xmin[inf] = np.inf, -np.inf
        self.xmin, self.xmax = xmin, xmax
        self.umax, self.umin = r(rng.uniform(0.2, 2.0, nu)), r(-rng.uniform(0.2, 2.0, nu))
        self.box = None
        if box if box is not None else seed % 3 == 2:     # per-stage boxes: a corridor that moves along the horizon
            lo = np.tile(xmin, (N + 1, 1)); hi = np.tile(xmax, (N + 1, 1))
            shift = r(np.linspace(-0.3, 0.3, N + 1))
            lo[:, 0] = np.where(inf[0], lo[:, 0], lo[:, 0] + shift); hi[:, 0] = np.where(inf[0], hi[:, 0], hi[:, 0] + shift)
            self.box = (lo, hi)
        self.x0 = r(rng.uniform(-0.4, 0.4, (batch, nx)))
        self.Xr = r(rng.uniform(-0.3, 0.3, (batch, nx, N + 1)))

    def solver(self, be, dtype, capacity=CAP, **settings):
        s = pm.BatchSolver(self.N, self.nx, self.nu, self.Q, self.QN, self.R, self.xmin, self.xmax, self.umin, self.umax,
                           slack=self.slack, W=self.W, S=self.S, dtype=dtype, time_varying=self.tv,
                           shared_model=self.shared, stage_reference=True, capacity=capacity, _backend=be,
                           **dict(dict(rho=1.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False, max_iter=1000), **settings))
        if self.box is not None:
            s.set_stage_bounds(*self.box)
        return s

    def setup(self, s, x0=None, Xr=None):
        sq = lambda M: None if M is None else (M if self.tv else M[:, 0])
        A, Bm, g = sq(self.A), sq(self.Bm), sq(self.g)
        if self.shared:
            A, Bm, g = A[0], Bm[0], None if g is None else g[0]
        s.setup(A, Bm, g, self.x0 if x0 is None else x0, self.Xr if Xr is None else Xr)
        return s

    def qp(self, b, x0=None):
        mb = 0 if self.shared else b
        pick = lambda M: None if M is None else (M[mb] if self.tv else M[mb, 0][None] if M.ndim == 3 else M[mb, 0])
        lo, hi = self.box if self.box is not None else (self.xmin, self.xmax)
        return ref_qp.canonical(self.N, pick(self.A), pick(self.Bm), pick(self.g), self.Q, self.QN, self.R, self.Xr[b],
                                lo, hi, self.umin, self.umax, self.x0[b] if x0 is None else x0,
                                slack=self.slack, W=self.W, S=self.S)

    def oracle_scaling(self, b, scaling):
        o = _ScaleOnly().setup(*ref_qp.assemble(self.qp(b)), scaling=scaling)
        return o.D, o.E, o.c


def _scaling(s):
    return [t.cpu().numpy().astype(np.float64) for t in s.scaling()]


def _check_scaling_vs_oracle(prob, got, scaling, tol, samples=SAMPLES):
    """(D, E, c) of the device against the oracle on the sampled QPs; returns the worst relative deviation."""
    D, E, c = got
    if scaling == 0:
        assert (D == 1).all() and (E == 1).all() and (c == 1).all()
        return 0.0
    worst = 0.0
    for b in samples:
        Do, Eo, co = prob.oracle_scaling(b, scaling)
        dev = max(_rel(D[b], Do), _rel(E[b], Eo), _rel(c[b], co))
        assert dev <= tol, (prob.nx, prob.nu, prob.slack, prob.N, scaling, b, dev)
        worst = max(worst, dev)
    return worst


# ---------------------------------------------------------------------------------------------------------------------
# (a) D, E, c against the oracle: every shape, the edge horizons (the warp kernel's N = 31 / 32 switch), pass counts 0,
#     1, 3 (odd: scale_one copies its result home from the scratch buffer) and 10, both precisions
def check_scaling_against_oracle(be, dtype, horizons=HORIZONS, scalings=(0, 1, 3, 10)):
    worst = 0.0
    f32 = dtype == torch.float32
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for hi, N in enumerate(horizons):
            prob = Problem(nx, nu, slack, N, seed=100 * si + hi, f32=f32)
            for sc in scalings:
                s = prob.setup(prob.solver(be, dtype, scaling=sc))
                worst = max(worst, _check_scaling_vs_oracle(prob, _scaling(s), sc, SCALE_TOL[dtype]))
                s.close()
    return worst


# (b) clamps and zero columns, f64
def check_clamps_and_zero_columns(be, horizons=(3, 31, 33)):
    worst = 0.0
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for hi, N in enumerate(horizons):
            prob = Problem(nx, nu, slack, N, seed=7000 + 10 * si + hi, wide=True)
            s = prob.setup(prob.solver(be, torch.float64))
            D, E, c = got = _scaling(s)
            worst = max(worst, _check_scaling_vs_oracle(prob, got, 10, SCALE_TOL[torch.float64]))
            if slack:         # the zero slack column s_k[0] of every stage: scaling 1 in every pass
                s0 = (N + 1) * nx + N * nu
                assert (D[:, s0::nx] == 1).all()
            assert np.isfinite(D).all() and np.isfinite(E).all() and (D > 0).all() and (E > 0).all()
            s.close()
    return worst


# (d) the cached factor, through the first iterates from a cold start: iterate(1), then iterate(2) (a second launch)
def _iterates_vs_oracle(prob, x, y, iters, settings, samples):
    worst = 0.0
    for b in samples:
        o = osqp_admm.OSQP().setup(*ref_qp.assemble(prob.qp(b)), **settings)
        for _ in range(iters):
            o.iterate()
        worst = max(worst, pc.rel(x[b], o.D * o.x), pc.rel(y[b], o.cinv * o.E * o.y))
    assert worst <= ITER_TOL, (prob.nx, prob.nu, prob.slack, prob.N, iters, worst)
    return worst


FACTOR_SETTINGS = dict(rho=1.0, sigma=1e-3)


def check_factor_iterates(be, horizons=(1, 7), samples=(0, B - 1)):
    """The Linv form (the sweeps of the lane-per-QP / warp-per-tile drivers, mpcb_iterate)."""
    worst = 0.0
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for hi, N in enumerate(horizons):
            prob = Problem(nx, nu, slack, N, seed=300 + 10 * si + hi)
            s = prob.setup(prob.solver(be, torch.float64, **FACTOR_SETTINGS))
            s.cold_start().iterate(1)
            x, y, _ = s.solution(want_y=True)
            worst = max(worst, _iterates_vs_oracle(prob, x.cpu().numpy(), y.cpu().numpy(), 1, FACTOR_SETTINGS, samples))
            s.iterate(2)
            x, y, _ = s.solution(want_y=True)
            worst = max(worst, _iterates_vs_oracle(prob, x.cpu().numpy(), y.cpu().numpy(), 3, FACTOR_SETTINGS, samples))
            s.close()
    return worst


# (e) full solves with sigma, alpha and scaling other than OSQP's defaults: a covering set of combinations per shape
SETTINGS = list(itertools.product((1e-6, 1e-3, 0.1), (1.0, 1.6, 1.9), (0, 1, 10)))      # (sigma, alpha, scaling)


def _solve_vs_oracle(prob, s, samples, settings):
    s.solve()
    x, y, _ = s.solution(want_y=True)
    inf = s.info()
    x, y = x.cpu().numpy(), y.cpu().numpy()
    it, st = inf.iter.cpu().numpy(), inf.status_val.cpu().numpy()
    pri, dua = inf.pri_res.cpu().numpy(), inf.dua_res.cpu().numpy()
    for b in samples:
        r = pc.oracle_solve(prob.qp(b), **settings)
        tag = (prob.nx, prob.nu, prob.slack, prob.N, settings, b)
        assert (it[b], st[b]) == (r.info.iter, r.info.status_val), (tag, it[b], st[b], r.info.iter, r.info.status)
        if r.info.status_val in (1, 2, -2):
            assert pc.rel(x[b], r.x) < 1e-6 and pc.rel(y[b], r.y) < 1e-6, tag
        # (a converged residual is a difference of terms of the size of x and y: its absolute rounding scales with them)
        atol = RES_ATOL * max(1.0, float(np.abs(r.x).max()), float(np.abs(r.y).max())) \
            if r.info.status_val in (1, 2, -2) else RES_ATOL
        for got, ref in ((pri[b], r.info.pri_res), (dua[b], r.info.dua_res)):
            assert abs(got - ref) <= atol + RES_RTOL * abs(ref), (tag, got, ref)
    return it


def check_settings(be, per_shape=6, samples=(0, B - 1)):
    seen = set()
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for j in range(per_shape):
            sigma, alpha, sc = SETTINGS[(per_shape * si + j) % len(SETTINGS)]
            seen.add((sigma, alpha, sc))
            prob = Problem(nx, nu, slack, 3 + (5 * si + 3 * j) % 12, seed=500 + 10 * si + j)
            settings = dict(rho=1.0, sigma=sigma, alpha=alpha, scaling=sc, eps_abs=1e-4, eps_rel=1e-4, max_iter=1000)
            s = prob.setup(prob.solver(be, torch.float64, **settings))
            _solve_vs_oracle(prob, s, samples, settings)
            s.close()
    assert len(seen) == len(SETTINGS)


def check_dense_settings(be, B_=64):
    """The shared-KKT dense path (configs[1]-style batch, f64) with sigma 1e-3 and alpha 1.0, against the oracle and
    against the per-QP kernels."""
    wl = workloads.LateralWorkload(B_, 20, False, False, 321, torch.float64, shared_speed=8.3128334)
    settings = dict(rho=5.0, sigma=1e-3, alpha=1.0, eps_abs=1e-4, eps_rel=1e-4)
    out = []
    for dense in (1, 0):
        def run():
            ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, warm_start=False,
                                     **settings)
            r = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
            return [t.clone() for t in (r.x, r.info.iter, r.info.status_val, r.info.pri_res, r.info.dua_res)]
        out.append(_with(be, dict(dense=dense), run))
    (x, it, st, pri, dua), (x0, it0, st0, _, _) = out
    assert torch.equal(it, it0) and torch.equal(st, st0)
    assert pc.rel(x.cpu().numpy(), x0.cpu().numpy()) < 1e-9
    for b in (0, B_ // 2, B_ - 1):
        r = pc.oracle_solve(workload_qp.lateral_qp(wl, b), **settings)
        assert (int(it[b]), int(st[b])) == (r.info.iter, r.info.status_val), (b, int(it[b]), r.info.iter)
        assert pc.rel(x[b].cpu().numpy(), r.x) < 1e-6
        for got, ref in ((float(pri[b]), r.info.pri_res), (float(dua[b]), r.info.dua_res)):
            assert abs(got - ref) <= RES_ATOL + RES_RTOL * abs(ref), (b, got, ref)


# (f) settings that invalidate the setup (rho, sigma, scaling), changed after a setup and a solve: the next setup equals a
#     fresh solver's with those settings, bit for bit
def check_settings_changed_after_setup(be, dtype=torch.float64):
    changes = (dict(rho=5.0, sigma=1e-3, scaling=3), dict(rho=0.1, sigma=0.1, scaling=0), dict(scaling=1))
    for si, (nx, nu, slack) in enumerate(SHAPES):
        prob = Problem(nx, nu, slack, 12 + si, seed=900 + si)
        ch = changes[si % len(changes)]
        s = prob.setup(prob.solver(be, dtype))
        s.solve()
        s.update_settings(**ch)
        with pytest.raises(pm.MpcError, match="before setup"):
            s.scaling()
        with pytest.raises(pm.MpcError, match="before setup"):
            s.solve()
        prob.setup(s).solve()
        fresh = prob.setup(prob.solver(be, dtype, **ch)).solve()
        for a, b in zip(_state(s), _state(fresh)):
            assert _bitwise(a, b), (nx, nu, slack, ch)
        s.close(); fresh.close()


def _state(s):
    x, y, _ = s.solution(want_y=True)
    inf = s.info()
    return (x, y, inf.iter, inf.status_val) + tuple(s.scaling())


# (g) the scaling of a setup is kept by update (x0 and the reference: q changes, D, E, c do not — osqp_update_lin_cost),
#     update_bounds (including a row that becomes an equality: the refactor path), a chunked solve whose unsolved QPs are
#     compacted into the scratch workspace, and closed-loop steps
def check_scaling_kept(be):
    wl = workloads.lateral_slack_increment(B, seed=77, dtype=torch.float64)

    def run():
        ctl = wl.make_controller(capacity=CAP, vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=5.0,
                                 eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
        r = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
        assert len(np.unique(r.info.iter.cpu().numpy())) > 2          # the chunked solves compact
        ref = [t.clone() for t in ctl.solver.scaling()]

        def same(what):
            for a, b in zip(ctl.solver.scaling(), ref):
                assert torch.equal(a, b), what
        same("solve")
        xr = np.random.default_rng(1).uniform(-0.5, 0.5, (B, 4))
        ctl.update_batch(wl.x0 * 0.9, references=xr)
        same("update")
        eq = wl.xmin.copy(); eq[2] = wl.xmax[2] - 1e-6
        ctl.update_bounds(xmin=eq)
        same("update_bounds")
        ctl.update_batch(wl.x0 * 0.5)
        same("solve after update_bounds")
        ctl.update_bounds(xmin=wl.xmin)
        _, _, its = ctl.closed_loop_batch(wl.x0, wl.xr, wl.speed, steps=4)
        same("closed loop")
        return its
    _with(be, dict(cta=0, retile_min_batch=2), run)


# (h) the premise of the dense path: one model, xr = 0 -> one scaling for the whole batch; diverging references -> c differs
def check_shared_kkt_premise(be, kernels=(1,)):
    for warp in kernels:
        def run():
            wl = workloads.lateral_vanilla_shared(B, seed=5)
            ctl = wl.make_controller(capacity=CAP, _backend=be, rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
            ctl.solve_batch(wl.x0, wl.xr, wl.speed)
            D, E, c = ctl.solver.scaling()
            for t in (D, E, c):
                assert torch.equal(t, t[:1].expand_as(t)), "QPs of one shared model scale differently"
            o = _ScaleOnly().setup(*ref_qp.assemble(workload_qp.lateral_qp(wl, 0)))
            D, E, c = D.cpu().numpy(), E.cpu().numpy(), c.cpu().numpy()
            assert max(_rel(D[0], o.D), _rel(E[0], o.E), _rel(c[0], o.c)) <= SCALE_TOL[torch.float64]
            wl.xr = np.random.default_rng(5).uniform(-3.0, 3.0, (B, 4))
            ctl.solve_batch(wl.x0, wl.xr, wl.speed)
            c = ctl.solver.scaling()[2].cpu().numpy()
            assert len(np.unique(c)) > B // 2, "the references do not reach the cost scaling"
            for b in (0, B - 1):
                o = _ScaleOnly().setup(*ref_qp.assemble(workload_qp.lateral_qp(wl, b)))
                assert _rel(c[b], o.c) <= SCALE_TOL[torch.float64]
            return c
        _with(be, dict(warp_setup=warp), run)


# (c) the two Ruiz kernels against each other (GPU): scale_warp_kernel ("warp_setup" 1) and scale_one ("warp_setup" 0)
ULP = {torch.float64: float(np.finfo(np.float64).eps), torch.float32: float(np.finfo(np.float32).eps)}


def check_ruiz_kernels_agree(be, dtype, horizons=tuple(range(1, 33))):
    worst = 0.0
    f32 = dtype == torch.float32
    settings = dict(rho=0.1, eps_abs=1e-3, eps_rel=1e-3, max_iter=400) if f32 else dict(rho=1.0, max_iter=400)
    xtol = 1e-4 if f32 else 1e-10
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for N in horizons:
            prob = Problem(nx, nu, slack, N, seed=2000 + 100 * si + N, f32=f32)
            out = []
            for warp in (1, 0):
                def run():
                    s = prob.setup(prob.solver(be, dtype, **settings))
                    sc = [t.clone() for t in s.scaling()]
                    s.solve()
                    x, _, _ = s.solution()
                    inf = s.info()
                    s.close()
                    return sc, (x.clone(), inf.iter.clone(), inf.status_val.clone())
                out.append(_with(be, dict(warp_setup=warp), run))
            (sw, rw), (s1, r1) = out
            tag = (nx, nu, slack, N, dtype)
            if N == 32:       # N + 1 > 32: both settings take scale_one
                for a, b in zip(sw + list(rw), s1 + list(r1)):
                    assert _bitwise(a, b), tag
                continue
            for a, b in zip(sw, s1):
                a, b = a.cpu().double().numpy(), b.cpu().double().numpy()
                dev = float(np.max(np.abs(a - b) / np.abs(b))) / ULP[dtype]
                assert dev <= 4, (tag, dev)
                worst = max(worst, dev)
            assert torch.equal(rw[1], r1[1]) and torch.equal(rw[2], r1[2]), tag
            nan = rw[0].isnan().all(dim=1)                  # infeasible QPs: NaN like OSQP's results
            assert torch.equal(nan, r1[0].isnan().all(dim=1)), tag
            if not bool(nan.all()):
                assert pc.rel(rw[0][~nan].cpu().numpy(), r1[0][~nan].cpu().numpy()) <= xtol, tag
    return worst


# (d) on the GPU, the block-inverse form Linv' Linv of admm_cta_kernel ("cta" 2 forces it): a solve capped at 1 and at 3
#     iterations from a cold start
def check_factor_block_inverse(be, horizons=(1, 7), samples=(0, B - 1)):
    worst = 0.0
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for hi, N in enumerate(horizons):
            prob = Problem(nx, nu, slack, N, seed=300 + 10 * si + hi)
            for iters in (1, 3):
                def run():
                    s = prob.setup(prob.solver(be, torch.float64, max_iter=iters, **FACTOR_SETTINGS))
                    s.solve()
                    x, y, _ = s.solution(want_y=True)
                    s.close()
                    return x.cpu().numpy(), y.cpu().numpy()
                x, y = _with(be, dict(cta=2, certificates=0), run)
                worst = max(worst, _iterates_vs_oracle(prob, x, y, iters, FACTOR_SETTINGS, samples))
    return worst


# ---------------------------------------------------------------------------------------------------------------------
def test_scaling_against_oracle_f64_cpu(emu_backend):
    print("worst rel. deviation of D, E, c from the oracle (emu, f64): %.2e" % check_scaling_against_oracle(emu_backend, torch.float64))


def test_scaling_against_oracle_f32_cpu(emu_backend):
    print("worst rel. deviation of D, E, c from the oracle (emu, f32): %.2e" % check_scaling_against_oracle(emu_backend, torch.float32))


def test_scaling_clamps_and_zero_columns_cpu(emu_backend):
    check_clamps_and_zero_columns(emu_backend)


def test_factor_first_iterates_cpu(emu_backend):
    print("worst rel. deviation of x, y after 1 and 3 iterations (emu, Linv): %.2e" % check_factor_iterates(emu_backend))


def test_non_default_settings_cpu(emu_backend):
    check_settings(emu_backend)


def test_settings_changed_after_setup_cpu(emu_backend):
    check_settings_changed_after_setup(emu_backend)


def test_scaling_kept_after_setup_cpu(emu_backend):
    check_scaling_kept(emu_backend)


def test_shared_kkt_premise_cpu(emu_backend):
    check_shared_kkt_premise(emu_backend)


@pytest.mark.gpu
def test_scaling_against_oracle_f64_gpu(cuda_backend):
    print("worst rel. deviation of D, E, c from the oracle (GPU, f64): %.2e" % check_scaling_against_oracle(cuda_backend, torch.float64))


@pytest.mark.gpu
def test_scaling_against_oracle_f32_gpu(cuda_backend):
    print("worst rel. deviation of D, E, c from the oracle (GPU, f32): %.2e" % check_scaling_against_oracle(cuda_backend, torch.float32))


@pytest.mark.gpu
def test_scaling_clamps_and_zero_columns_gpu(cuda_backend):
    check_clamps_and_zero_columns(cuda_backend)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_ruiz_kernels_agree_gpu(cuda_backend, dtype):
    print("worst deviation between the two Ruiz kernels (%s): %.2f ulp" % (dtype, check_ruiz_kernels_agree(cuda_backend, dtype)))


@pytest.mark.gpu
def test_factor_first_iterates_gpu(cuda_backend):
    w1 = _with(cuda_backend, dict(cta=0), lambda: check_factor_iterates(cuda_backend))
    w2 = check_factor_block_inverse(cuda_backend)
    print("worst rel. deviation of x, y after 1 and 3 iterations (GPU): Linv %.2e, Linv'Linv %.2e" % (w1, w2))


@pytest.mark.gpu
def test_non_default_settings_gpu(cuda_backend):
    check_settings(cuda_backend)
    check_dense_settings(cuda_backend)


@pytest.mark.gpu
def test_settings_changed_after_setup_gpu(cuda_backend):
    check_settings_changed_after_setup(cuda_backend)


@pytest.mark.gpu
def test_scaling_kept_after_setup_gpu(cuda_backend):
    check_scaling_kept(cuda_backend)


@pytest.mark.gpu
def test_shared_kkt_premise_gpu(cuda_backend):
    check_shared_kkt_premise(cuda_backend, kernels=(1, 0))
