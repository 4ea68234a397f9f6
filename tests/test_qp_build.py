"""The QP build path ("cast the MPC problem to a QP") against the oracle, at every compiled shape and in both precisions:
mpcb_build_qp (build_one) and mpcb_qp_pattern against ref_qp.assemble; the vehicle-model kernels (lateral_discretize,
dynamics_linearize, dynamics_step, kinematics_linearize, kinematics_step) against oracle/workload_qp.py and
oracle/vehicle_ref.py; augment_increment and plant_step; the layout helpers; and the host front door mpcb_solve_host
against setup + solve on the device path.  CPU (tests/emu) and GPU (-m gpu).

The solve path never materialises P or A, so no solve test can see an error of build_one.  Every kernel is called
through its C entry point, into outputs that hold NaN in the columns [0, batch) and a sentinel past them: each check
asserts that every slot of the batch was written and that nothing past the batch was touched.  Random batches have
B = 37 QPs in a capacity of 64 (ld = 64 > B, a ragged last tile).

Most of the build is copies and products of f32-representable inputs, so most comparisons are exact.  Model kernels
are compared with the f64 oracle on the same (f32-representable) inputs, relative to each output's max-norm per QP."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import python_mpc_b200 as pm
from python_mpc_b200 import workloads
from python_mpc_b200._lib import MPCB_F32, MPCB_F64, ptr
from oracle import ref_qp, vehicle_ref, workload_qp
from test_setup_scaling import B, CAP, MODES, SHAPES, Problem, _bitwise

E_ARG, E_STATE = -1, -3
SENT = 777.0                         # fills the columns past the batch (and every output of a call that must fail)
GUARD = 64                           # rows of SENT after each output: a write past its end fails a check, corrupts nothing
INFTY = 1e30                         # OSQP_INFTY: OSQP's Python interface clips infinite bounds to it
BUILD_HORIZONS = (1, 2, 7, 31, 32, 33, 64)
FULL_CHECK_MAX_N = 33                # every QP of the batch up to this horizon, SAMPLES beyond
SAMPLES = (0, 31, 32, B - 1)
MODEL_BATCHES = ((1, 1), (1, 64), (B, B), (B, 64))          # (batch, ld)
# relative to each output's max-norm per QP: f64 (libm, FMA contraction) and f32 against the f64 oracle on the same
# f32-representable inputs
TOL = {"lateral": {torch.float64: 1e-12, torch.float32: 2e-5},
       "dynamics": {torch.float64: 1e-13, torch.float32: 2e-6},
       "kinematics": {torch.float64: 1e-13, torch.float32: 2e-6}}
LATERAL_PARAMS = (1300., 1.25, 1.40, 2555.88174, 11979.9261, 11140.9949, 0.02)         # m, l_f, l_r, Iz, Cf, Cr, dt
DYN = dict(m=1300., l_f=1.25, l_r=1.40, width=1.78, length=4.25, C_d=0.34, A_f=2.0, C_roll=0.015)
WHEELBASE = 1.25 + 1.40


def _dt(dtype):
    return MPCB_F32 if dtype == torch.float32 else MPCB_F64


def _npdt(dtype):
    return np.float32 if dtype == torch.float32 else np.float64


def _f32(a):
    """Round to the nearest f32 (inputs that both precisions hold exactly)."""
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def _out(be, dtype, elems, batch, ld):
    """An element-major output [elems, ld] followed by GUARD rows: NaN in the batch's columns, SENT everywhere else."""
    t = torch.full((elems + GUARD, ld), SENT, dtype=dtype, device=be.device)
    t[:elems, :batch] = float("nan")
    return t


def _em(be, dtype, a, ld):
    """(batch, elems) host array -> element-major device input [elems, ld], NaN past the batch (a kernel must not read it)."""
    a = np.asarray(a, dtype=np.float64).reshape(len(a), -1)
    t = torch.full((a.shape[1], ld), float("nan"), dtype=dtype, device=be.device)
    t[:, :a.shape[0]] = torch.as_tensor(a.T.copy()).to(device=be.device, dtype=dtype)
    return t


def _written(t, batch, cols=None):
    """Asserts that every slot of the batch was written and the columns past it are untouched; returns the batch's
    columns (or `cols`) batch-major as float64 numpy."""
    assert bool((t[-GUARD:] == SENT).all()), "a write past the end of the output"
    t = t[:-GUARD]
    assert not bool(t[:, :batch].isnan().any()), "a slot of the batch was not written"
    assert bool((t[:, batch:] == SENT).all()), "a column past the batch was written"
    sel = t[:, :batch] if cols is None else t[:, cols]
    return sel.t().cpu().numpy()


def _untouched(*ts):
    for t in ts:
        assert bool((t == SENT).all()), "an output of a rejected call was written"


def _rel_dev(got, ref):
    """Worst deviation over the QPs of a batch, relative to the max-norm of each QP's reference output."""
    got = np.asarray(got, dtype=np.float64).reshape(len(got), -1)
    ref = np.asarray(ref, dtype=np.float64).reshape(len(ref), -1)
    nrm = np.abs(ref).max(axis=1)
    nrm[nrm == 0] = 1.0
    return float((np.abs(got - ref).max(axis=1) / nrm).max())


# ---------------------------------------------------------------------------------------------------------------------
# 1. mpcb_build_qp against ref_qp.assemble
NAMES = ("Pdiag", "q", "Avals", "l", "u")


def _oracle_qp(prob, b, f32):
    """(Pdiag, q, A values on the CSC pattern, l, u) of QP b in the device's precision.  The inputs are representable in
    it, so every entry is a copy or ONE rounded product (q = -(Q xr)): the f64 oracle rounded to f32 is exact."""
    P, q, A, l, u = ref_qp.assemble(prob.qp(b))
    A = sp.csc_matrix(A); A.sort_indices()
    out = [P.diagonal(), q, A.data, np.clip(l, -INFTY, INFTY), np.clip(u, -INFTY, INFTY)]
    return [v.astype(np.float32) if f32 else v for v in out]


def _build(s, be, nnz, skip=None):
    """mpcb_build_qp into NaN / sentinel-filled outputs; output `skip` passed as NULL (returned as None)."""
    outs = [None if i == skip else _out(be, s.dtype, n, s.batch, s.ld)
            for i, n in enumerate((s.nvar, s.nvar, nnz, s.ncon, s.ncon))]
    be.check(be.lib.mpcb_build_qp(s._h, *[ptr(t) for t in outs], be.stream()))
    return [None if t is None else _written(t, s.batch).astype(_npdt(s.dtype)) for t in outs]


def _check_build(prob, got, f32, samples, tag):
    for b in samples:
        for name, g, r in zip(NAMES, got, _oracle_qp(prob, b, f32)):
            if g is not None:
                assert np.array_equal(g[b], r), (tag, name, b, float(np.abs(g[b].astype(np.float64) - r).max()))


def _solver(prob, be, dtype, stage_reference=True, capacity=CAP):
    """Problem.solver with the choice of one reference per QP (the oracle's Xr then repeats it over the stages)."""
    if not stage_reference:
        prob.Xr = np.repeat(prob.Xr[:, :, :1], prob.N + 1, axis=2)
    s = pm.BatchSolver(prob.N, prob.nx, prob.nu, prob.Q, prob.QN, prob.R, prob.xmin, prob.xmax, prob.umin, prob.umax,
                       slack=prob.slack, W=prob.W, S=prob.S, dtype=dtype, time_varying=prob.tv, shared_model=prob.shared,
                       stage_reference=stage_reference, capacity=capacity, _backend=be, rho=1.0, max_iter=1)
    if prob.box is not None:
        s.set_stage_bounds(*prob.box)
    return s


def _setup(prob, s):
    return prob.setup(s, Xr=None if s.stage_reference else prob.Xr[:, :, 0])


def check_build_qp(be, dtype, horizons=BUILD_HORIZONS):
    """Every shape x horizon; the (time-varying, shared, g) mode cycles with the seed, per-stage boxes on alternate shapes,
    one reference per QP at every third horizon; infinite bounds where Problem draws them (30 % of the state bounds)."""
    f32 = dtype == torch.float32
    seen = set()
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for hi, N in enumerate(horizons):
            prob = Problem(nx, nu, slack, N, seed=6000 + 7 * si + hi, f32=f32, box=si % 2 == 0)
            stage_ref = hi % 3 != 1
            s = _setup(prob, _solver(prob, be, dtype, stage_ref))
            nnz = be.lib.mpcb_qp_pattern(s._h, None, None)
            samples = range(B) if N <= FULL_CHECK_MAX_N else SAMPLES
            _check_build(prob, _build(s, be, nnz), f32, samples, (nx, nu, slack, N, dtype))
            seen.add((prob.tv, prob.shared, prob.g is not None, prob.box is not None, stage_ref,
                      bool(np.isinf(prob.xmin).any())))
            s.close()
    assert {m[:3] for m in seen} == set(MODES)
    assert any(m[3] for m in seen) and any(not m[4] for m in seen) and any(m[5] for m in seen)


def check_build_after_updates(be, dtype, N=7):
    """update (x_init, Xr) and update_bounds (xmin / umax, then per-stage boxes) reach the build; a rejected update
    leaves it unchanged; each output set to NULL on its own leaves the other four as they were."""
    f32 = dtype == torch.float32
    r = _f32 if f32 else (lambda a: np.asarray(a, dtype=np.float64))
    for si, (nx, nu, slack) in enumerate(SHAPES):
        prob = Problem(nx, nu, slack, N, seed=6500 + si, f32=f32, box=si % 2 == 1)
        tag = (nx, nu, slack, prob.tv, prob.shared, dtype)
        s = _setup(prob, _solver(prob, be, dtype, stage_reference=si % 3 != 1))
        nnz = be.lib.mpcb_qp_pattern(s._h, None, None)
        rng = np.random.default_rng(si)
        # new initial states and references: rows dyn_0 and q follow
        x0 = r(rng.uniform(-0.4, 0.4, (B, nx))); Xr = r(rng.uniform(-0.3, 0.3, (B, nx, N + 1)))
        if not s.stage_reference:
            Xr = np.repeat(Xr[:, :, :1], N + 1, axis=2)
        s.update(x0, Xr if s.stage_reference else Xr[:, :, 0])
        prob.x0, prob.Xr = x0, Xr
        _check_build(prob, _build(s, be, nnz), f32, range(B), tag + ("update",))
        # new xmin / umax (no effect on the state rows while per-stage boxes are set), then new per-stage boxes
        xmin = prob.xmin.copy(); xmin[0] = -0.75
        umax = r(prob.umax + 0.5)
        s.update_bounds(xmin=xmin, umax=umax)
        prob.xmin, prob.umax = xmin, umax
        _check_build(prob, _build(s, be, nnz), f32, range(B), tag + ("update_bounds",))
        lo = np.tile(prob.xmin, (N + 1, 1)) - r(np.linspace(0.0, 0.5, N + 1))[:, None]
        hi = np.tile(prob.xmax, (N + 1, 1)) + 0.25
        s.update_bounds(stage_lo=lo, stage_hi=hi)
        prob.box = (lo, hi)
        full = _build(s, be, nnz)
        _check_build(prob, full, f32, range(B), tag + ("stage boxes",))
        # rejected updates (inverted bounds) change nothing
        with pytest.raises(pm.MpcError):
            s.update_bounds(umin=prob.umax + 1.0)
        with pytest.raises(pm.MpcError):
            s.update_bounds(stage_lo=hi + 1.0, stage_hi=hi)
        for a, b in zip(_build(s, be, nnz), full):
            assert np.array_equal(a, b), tag + ("rejected update",)
        # each output NULL on its own
        for skip in range(5):
            part = _build(s, be, nnz, skip=skip)
            for i, (a, b) in enumerate(zip(part, full)):
                assert (a is None) == (i == skip) and (a is None or np.array_equal(a, b)), tag + ("NULL", NAMES[skip])
        s.close()


def check_build_before_setup(be):
    prob = Problem(4, 1, False, 3, seed=1)
    s = prob.solver(be, torch.float64)
    outs = [torch.full((n, s.ld), SENT, dtype=torch.float64, device=be.device) for n in (s.nvar, s.nvar, 200, s.ncon, s.ncon)]
    assert be.lib.mpcb_build_qp(s._h, *[ptr(t) for t in outs], be.stream()) == E_STATE
    _untouched(*outs)
    s.close()


def check_build_qp_at_scale(be, batch=65536, N=20, stride=1024):
    """The qp_build workload of bench.py: 65536 QPs of the slack + delta-u lateral MPC.  Every slot written; a strided
    sample and the last QP equal the oracle's assembly of the model the solver holds, bit for bit."""
    wl = workloads.lateral_slack_increment(batch, N=N, seed=11, dtype=torch.float64)
    ctl = wl.make_controller(capacity=batch, _backend=be, rho=5.0, warm_start=False, max_iter=1)
    ctl.solve_batch(wl.x0, wl.xr, wl.speed, want_x=False)
    s = ctl.solver
    nnz = be.lib.mpcb_qp_pattern(s._h, None, None)
    cols = list(range(0, batch, stride)) + [batch - 1]
    outs = [_out(be, s.dtype, n, s.batch, s.ld) for n in (s.nvar, s.nvar, nnz, s.ncon, s.ncon)]
    be.check(be.lib.mpcb_build_qp(s._h, *[ptr(t) for t in outs], be.stream()))
    got = [_written(t, s.batch, cols) for t in outs]
    Ad = s._keep["Ad"][:, cols].t().cpu().numpy(); Bd = s._keep["Bd"][:, cols].t().cpu().numpy()
    for j, b in enumerate(cols):
        p = workload_qp.lateral_qp(wl, b)
        p.A[:] = Ad[j].reshape(p.nx, p.nx); p.B[:] = Bd[j].reshape(p.nx, p.nu)
        P, q, A, l, u = ref_qp.assemble(p)
        A = sp.csc_matrix(A); A.sort_indices()
        for name, g, ref in zip(NAMES, got, (P.diagonal(), q, A.data, l, u)):
            assert np.array_equal(g[j], ref), (name, b)
    s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. mpcb_qp_pattern: the CSC pattern of the oracle's A
def check_pattern(be, horizons=BUILD_HORIZONS):
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for N in horizons:
            prob = Problem(nx, nu, slack, N, seed=si, batch=1)
            s = prob.solver(be, torch.float64, capacity=1)
            nnz = be.lib.mpcb_qp_pattern(s._h, None, None)
            Ap = np.full(s.nvar + 1, -1, dtype=np.int32); Ai = np.full(nnz, -1, dtype=np.int32)
            assert be.lib.mpcb_qp_pattern(s._h, Ap.ctypes.data_as(C.POINTER(C.c_int)),
                                          Ai.ctypes.data_as(C.POINTER(C.c_int))) == nnz
            A = sp.csc_matrix(ref_qp.assemble(prob.qp(0))[2]); A.sort_indices()
            assert np.array_equal(Ap, A.indptr) and np.array_equal(Ai, A.indices), (nx, nu, slack, N)
            s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. model kernels
def _model_kernel(be, dtype, name, ins, params, out_elems, ld, null=()):
    """One call of a model kernel on batch-major host inputs; returns its outputs batch-major (None where passed NULL)."""
    batch = len(ins[0])
    tin = [_em(be, dtype, a, ld) for a in ins]
    touts = [None if i in null else _out(be, dtype, n, batch, ld) for i, n in enumerate(out_elems)]
    par = (C.c_double * len(params))(*params)
    be.check(getattr(be.lib, name)(_dt(dtype), batch, ld, *[ptr(t) for t in tin], par, *[ptr(t) for t in touts],
                                   be.stream()))
    return [None if t is None else _written(t, batch) for t in touts]


def _chunks(n, batch):
    """Index sets of `batch` inputs covering range(n) (the last one overlaps); every fifth input alone for batch 1."""
    if batch == 1:
        return [[i] for i in range(0, n, 5)]
    return [list(range(i, i + batch)) if i + batch <= n else list(range(n - batch, n)) for i in range(0, n, batch)]


def _lateral_speeds():
    edge = [0.0, 0.05, -0.05, 0.0999, -0.0999, 0.1, -0.1, 0.5, 8.3128334, 35.0, 60.0]
    return _f32(np.concatenate([edge, np.linspace(-40.0, 60.0, 26)]))


def _dynamics_inputs(golden):
    """The golden points, random states and vx on and one f32 ulp either side of each guard boundary (0, +-0.3, +-0.5)
    with nonzero vy, wz and steer that the guards must zero; all f32-representable."""
    g = golden["vehicle_models"]
    rng = np.random.default_rng(3)
    n = 40
    xr = np.stack([rng.uniform(-50, 50, n), rng.uniform(-50, 50, n), rng.uniform(-np.pi, np.pi, n),
                   rng.uniform(-30, 30, n), rng.uniform(-2, 2, n), rng.uniform(-1, 1, n)], axis=1)
    ur = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-3, 3, n)], axis=1)
    vx = []
    for v in (0.0, 0.3, -0.3, 0.5, -0.5):
        f = np.float32(v)
        vx += [f, np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(-np.inf))]
    xg = np.array([[1.0, -2.0, 0.3, float(v), 0.7, -0.4] for v in vx])
    ug = np.tile([0.2, 1.0], (len(vx), 1))
    return _f32(np.concatenate([g["dyn_x"], xr, xg])), _f32(np.concatenate([g["dyn_u"], ur, ug])), float(g["dyn_dt"])


def _kinematics_inputs(golden):
    g = golden["vehicle_models"]
    rng = np.random.default_rng(4)
    n = 40
    xr = np.stack([rng.uniform(-50, 50, n), rng.uniform(-50, 50, n), rng.uniform(-5, 30, n),
                   rng.uniform(-np.pi, np.pi, n)], axis=1)
    ur = np.stack([rng.uniform(-0.5, 0.5, n), rng.uniform(-3, 3, n)], axis=1)
    return _f32(np.concatenate([g["kin_x"], xr])), _f32(np.concatenate([g["kin_u"], ur])), float(g["kin_dt"])


def check_lateral(be, dtype):
    v = _lateral_speeds()
    Ao, Bo = workload_qp.lateral_models(v)
    worst = 0.0
    for batch, ld in MODEL_BATCHES:
        for idx in _chunks(len(v), batch):
            A, Bm = _model_kernel(be, dtype, "mpcb_lateral_discretize", [v[idx, None]], LATERAL_PARAMS, (16, 4), ld)
            dev = max(_rel_dev(A, Ao[idx]), _rel_dev(Bm, Bo[idx]))
            assert dev <= TOL["lateral"][dtype], (dtype, batch, ld, v[idx], dev)
            worst = max(worst, dev)
    return worst


def check_dynamics(be, dtype, golden):
    x, u, dt = _dynamics_inputs(golden)
    params = (DYN["m"], DYN["l_f"], DYN["l_r"], 1 / 12 * DYN["m"] * (DYN["width"] ** 2 + DYN["length"] ** 2), DYN["C_d"],
              DYN["A_f"], DYN["C_roll"], dt)
    ref_lin = [vehicle_ref.dynamics_model(x[i], u[i], dt=dt, **DYN) for i in range(len(x))]
    ref_step = [vehicle_ref.dynamics_step(x[i], u[i], dt=dt, **DYN) for i in range(len(x))]
    tol = TOL["dynamics"][dtype]
    worst = {"linearize": 0.0, "step": 0.0}
    for batch, ld in MODEL_BATCHES:
        for idx in _chunks(len(x), batch):
            got = _model_kernel(be, dtype, "mpcb_dynamics_linearize", [x[idx], u[idx]], params, (36, 12, 6), ld)
            dev = max(_rel_dev(got[k], np.stack([ref_lin[i][k] for i in idx])) for k in range(3))
            assert dev <= tol, (dtype, "linearize", batch, ld, x[idx], dev)
            worst["linearize"] = max(worst["linearize"], dev)
            xn, al = _model_kernel(be, dtype, "mpcb_dynamics_step", [x[idx], u[idx]], params, (6, 2), ld)
            dev = max(_rel_dev(xn, np.stack([ref_step[i][0] for i in idx])),
                      _rel_dev(al, np.array([ref_step[i][1:] for i in idx])))
            assert dev <= tol, (dtype, "step", batch, ld, x[idx], dev)
            worst["step"] = max(worst["step"], dev)
            xn2, none = _model_kernel(be, dtype, "mpcb_dynamics_step", [x[idx], u[idx]], params, (6, 2), ld, null=(1,))
            assert none is None and np.array_equal(xn2, xn)          # alpha = NULL: the same step
    return worst


def check_kinematics(be, dtype, golden):
    x, u, dt = _kinematics_inputs(golden)
    ref_lin = [vehicle_ref.kinematics_model(x[i], u[i], WHEELBASE, dt) for i in range(len(x))]
    ref_step = np.stack([vehicle_ref.kinematics_step(x[i], u[i], WHEELBASE, dt) for i in range(len(x))])
    tol = TOL["kinematics"][dtype]
    worst = {"linearize": 0.0, "step": 0.0}
    for batch, ld in MODEL_BATCHES:
        for idx in _chunks(len(x), batch):
            got = _model_kernel(be, dtype, "mpcb_kinematics_linearize", [x[idx], u[idx]], (WHEELBASE, dt), (16, 8, 4), ld)
            dev = max(_rel_dev(got[k], np.stack([ref_lin[i][k] for i in idx])) for k in range(3))
            assert dev <= tol, (dtype, "linearize", batch, ld, dev)
            worst["linearize"] = max(worst["linearize"], dev)
            xn, = _model_kernel(be, dtype, "mpcb_kinematics_step", [x[idx], u[idx]], (WHEELBASE, dt), (4,), ld)
            dev = _rel_dev(xn, ref_step[idx])
            assert dev <= tol, (dtype, "step", batch, ld, dev)
            worst["step"] = max(worst["step"], dev)
    return worst


def check_augment(be, dtype):
    """Bit-exact copies: A~ = [[Ad, Bd], [0, I]], B~ = [[Bd], [I]], g~ = [gd; 0] (zeros when gd is NULL)."""
    rng = np.random.default_rng(5)
    npdt = _npdt(dtype)
    for nx, nu in ((4, 1), (4, 2), (6, 2)):
        na = nx + nu
        for stages in (1, 7):
            for batch, ld in MODEL_BATCHES:
                Ad = _f32(rng.standard_normal((batch, stages, nx, nx)))
                Bd = _f32(rng.standard_normal((batch, stages, nx, nu)))
                gd = _f32(rng.standard_normal((batch, stages, nx)))
                At_o, Bt_o, gt_o = ref_qp.augment_increment(Ad, Bd, gd)
                for with_gd, with_gt in ((True, True), (False, True), (True, False), (False, False)):
                    tin = [_em(be, dtype, a, ld) for a in (Ad, Bd, gd)]
                    At, Bt, gt = (_out(be, dtype, stages * n, batch, ld) for n in (na * na, na * nu, na))
                    be.check(be.lib.mpcb_augment_increment(_dt(dtype), batch, ld, nx, nu, stages, ptr(tin[0]), ptr(tin[1]),
                                                           ptr(tin[2] if with_gd else None), ptr(At), ptr(Bt),
                                                           ptr(gt if with_gt else None), be.stream()))
                    tag = (nx, nu, stages, batch, ld, with_gd, with_gt, dtype)
                    assert np.array_equal(_written(At, batch), At_o.reshape(batch, -1).astype(npdt)), tag
                    assert np.array_equal(_written(Bt, batch), Bt_o.reshape(batch, -1).astype(npdt)), tag
                    if with_gt:
                        ref = gt_o if with_gd else np.zeros_like(gt_o)
                        assert np.array_equal(_written(gt, batch), ref.reshape(batch, -1).astype(npdt)), tag
                    else:
                        assert bool(gt[:-GUARD, :batch].isnan().all()) and bool((gt[:, batch:] == SENT).all()), tag


def check_plant(be, dtype, N=7):
    """x_next = A x + B u + g against a long-double reference, within the bound of a sum of n = nx + nu + 1 terms:
    n eps (|A||x| + |B||u| + |g|) per component; shared models, no g, the closed loop's u stride N nu, x_next aliasing x."""
    rng = np.random.default_rng(6)
    eps = float(np.finfo(_npdt(dtype)).eps)
    worst = 0.0
    for nx, nu in ((4, 1), (5, 1), (6, 2), (8, 2), (10, 2)):
        for shared in (0, 1):
            for has_g in (False, True):
                for u_stride in (nu, N * nu):
                    for alias in (False, True):
                        for batch, ld in ((1, 1), (B, CAP)):
                            nm, mld = (1, 1) if shared else (batch, ld)
                            A = _f32(rng.standard_normal((nm, nx, nx))); Bm = _f32(rng.standard_normal((nm, nx, nu)))
                            g = _f32(rng.standard_normal((nm, nx))) if has_g else None
                            x = _f32(rng.standard_normal((batch, nx))); u = _f32(rng.standard_normal((batch, u_stride)))
                            tA, tB = _em(be, dtype, A, mld), _em(be, dtype, Bm, mld)
                            tg = _em(be, dtype, g, mld) if has_g else None
                            tx = _em(be, dtype, x, ld)
                            tu = torch.as_tensor(u).to(device=be.device, dtype=dtype)
                            xn = _out(be, dtype, nx, batch, ld)
                            if alias:
                                xn[:nx, :batch] = tx[:, :batch]
                                tx = xn
                            be.check(be.lib.mpcb_plant_step(_dt(dtype), batch, ld, nx, nu, shared, ptr(tA), ptr(tB), ptr(tg),
                                                            ptr(tx), ptr(tu), u_stride, ptr(xn), be.stream()))
                            got = _written(xn, batch)
                            Al, Bl = A.astype(np.longdouble), Bm.astype(np.longdouble)
                            ul = u[:, :nu].astype(np.longdouble)
                            ref = np.einsum("bij,bj->bi", Al, x.astype(np.longdouble)) + np.einsum("bij,bj->bi", Bl, ul)
                            mag = np.einsum("bij,bj->bi", np.abs(A), np.abs(x)) + np.einsum("bij,bj->bi", np.abs(Bm), np.abs(u[:, :nu]))
                            if has_g:
                                ref = ref + g; mag = mag + np.abs(g)
                            err = np.abs(got - ref.astype(np.float64)) / ((nx + nu + 1) * eps * mag)
                            tag = (nx, nu, shared, has_g, u_stride, alias, batch, dtype)
                            assert float(err.max()) <= 1.0, tag
                            worst = max(worst, float(err.max()))
    return worst


def check_model_argument_errors(be, dtype):
    """Rejected calls return MPCB_E_ARG and write nothing: ld < batch, batch = 0, a NULL input; for plant_step also
    u_stride < nu, nx > 10 and nu > 2."""
    dt, st, L = _dt(dtype), be.stream(), be.lib
    buf = lambda n: torch.full((n, CAP), SENT, dtype=dtype, device=be.device)
    p7, p8, p2 = (C.c_double * 7)(*LATERAL_PARAMS), (C.c_double * 8)(*([1.0] * 8)), (C.c_double * 2)(WHEELBASE, 0.02)
    ins = {n: torch.zeros((n, CAP), dtype=dtype, device=be.device) for n in (1, 2, 4, 6, 16)}
    for batch, ld, null in ((B, B - 1, False), (0, CAP, False), (B, CAP, True)):
        i = lambda n: None if null else ins[n]          # the first input of each call
        calls = (("mpcb_lateral_discretize", lambda o: (ptr(i(1)), p7, ptr(o[0]), ptr(o[1])), (16, 4)),
                 ("mpcb_dynamics_linearize", lambda o: (ptr(i(6)), ptr(ins[2]), p8, ptr(o[0]), ptr(o[1]), ptr(o[2])), (36, 12, 6)),
                 ("mpcb_dynamics_step", lambda o: (ptr(i(6)), ptr(ins[2]), p8, ptr(o[0]), ptr(o[1])), (6, 2)),
                 ("mpcb_kinematics_linearize", lambda o: (ptr(i(4)), ptr(ins[2]), p2, ptr(o[0]), ptr(o[1]), ptr(o[2])), (16, 8, 4)),
                 ("mpcb_kinematics_step", lambda o: (ptr(i(4)), ptr(ins[2]), p2, ptr(o[0])), (4,)))
        for name, args, sizes in calls:
            o = [buf(n) for n in sizes]
            assert getattr(L, name)(dt, batch, ld, *args(o), st) == E_ARG, (name, batch, ld, null)
            _untouched(*o)
        o = [buf(n) for n in (25, 5, 5)]
        assert L.mpcb_augment_increment(dt, batch, ld, 4, 1, 1, ptr(i(16)), ptr(ins[4]), ptr(None), ptr(o[0]), ptr(o[1]),
                                        ptr(o[2]), st) == E_ARG, ("augment", batch, ld, null)
        _untouched(*o)
        o = buf(4)
        assert L.mpcb_plant_step(dt, batch, ld, 4, 1, 0, ptr(i(16)), ptr(ins[4]), ptr(None), ptr(ins[4]), ptr(ins[1]), 1,
                                 ptr(o), st) == E_ARG, ("plant", batch, ld, null)
        _untouched(o)
    for nx, nu, u_stride in ((4, 2, 1), (11, 1, 1), (4, 3, 3)):
        o = buf(16)
        assert L.mpcb_plant_step(dt, B, CAP, nx, nu, 0, ptr(ins[16]), ptr(ins[16]), ptr(None), ptr(ins[16]), ptr(ins[16]),
                                 u_stride, ptr(o), st) == E_ARG, ("plant", nx, nu, u_stride)
        _untouched(o)


# ---------------------------------------------------------------------------------------------------------------------
# 4. layout helpers
def check_layout(be, dtype):
    gen = torch.Generator().manual_seed(9)
    dt, st = _dt(dtype), be.stream()
    for batch in (1, 31, 32, 33, 37):
        for elems in (1, 5, 105):
            for ld in sorted({batch, (batch + 31) // 32 * 32, batch + 7}):
                src = torch.randn((batch, elems), generator=gen, dtype=torch.float64).to(device=be.device, dtype=dtype)
                em = _out(be, dtype, elems, batch, ld)
                be.check(be.lib.mpcb_to_element_major(dt, batch, elems, ld, ptr(src), ptr(em), st))
                assert np.array_equal(_written(em, batch), src.cpu().numpy()), (batch, elems, ld)
                bm = torch.full((batch * elems + 64,), SENT, dtype=dtype, device=be.device)
                bm[:batch * elems] = float("nan")
                be.check(be.lib.mpcb_to_batch_major(dt, batch, elems, ld, ptr(em), ptr(bm), st))
                assert torch.equal(bm[:batch * elems].reshape(batch, elems), src), (batch, elems, ld)
                assert bool((bm[batch * elems:] == SENT).all()), (batch, elems, ld)
    src = torch.zeros((B, 5), dtype=dtype, device=be.device)
    for batch, elems, ld, s_ok, d_ok in ((B, 5, B - 1, 1, 1), (0, 5, CAP, 1, 1), (B, 0, CAP, 1, 1), (B, 5, CAP, 0, 1),
                                         (B, 5, CAP, 1, 0)):
        dst = torch.full((5, CAP), SENT, dtype=dtype, device=be.device)
        for fn in (be.lib.mpcb_to_element_major, be.lib.mpcb_to_batch_major):
            assert fn(dt, batch, elems, ld, ptr(src if s_ok else None), ptr(dst if d_ok else None), st) == E_ARG
        _untouched(dst)


# ---------------------------------------------------------------------------------------------------------------------
# 5. mpcb_solve_host against setup + solve on the device path
def _inputs(prob, n):
    """Natural-shape inputs of the first n QPs: models ([n,] [N,] r, c) — one row for a shared model — x0, Xr (n, nx, N+1)."""
    out = []
    for M in (prob.A, prob.Bm, prob.g):
        if M is not None:
            M = M[0] if prob.shared else M[:n]
            if not prob.tv:
                M = M[0] if prob.shared else M[:, 0]
        out.append(M)
    return out + [prob.x0[:n], prob.Xr[:n]]


def _device_path(s, prob, n):
    s.setup(*_inputs(prob, n)).solve()
    x, _, u = s.solution()
    inf = s.info()
    return x.cpu(), u.reshape(n, -1).cpu(), inf.iter.cpu(), inf.status_val.cpu()


def _host_path(s, prob, n, want_x=True, want_u=True):
    """mpcb_solve_host with numpy-layout host buffers; outputs pre-filled with SENT / -999 (slots it must write)."""
    npdt = _npdt(s.dtype)
    A, Bm, g, x0, Xr = _inputs(prob, n)
    c = lambda a: None if a is None else np.ascontiguousarray(np.asarray(a, dtype=npdt))
    A, Bm, g, x0 = c(A), c(Bm), c(g), c(x0)
    xr = c(np.transpose(Xr, (0, 2, 1)))                  # (n, N+1, nx): stage-major rows
    xo = np.full((n, s.nvar), SENT, dtype=npdt) if want_x else None
    uo = np.full((n, s.N * s.nu), SENT, dtype=npdt) if want_u else None
    it = np.full(n, -999, dtype=np.int32); st = np.full(n, -999, dtype=np.int32)
    vp = lambda a: C.c_void_p(0) if a is None else C.c_void_p(a.ctypes.data)
    s.be.check(s.be.lib.mpcb_solve_host(s._h, n, vp(A), vp(Bm), vp(g), vp(x0), vp(xr), vp(xo), vp(uo), vp(it), vp(st)))
    t = lambda a: None if a is None else torch.from_numpy(a)
    return t(xo), t(uo), t(it), t(st)


def check_solve_host(be, dtype):
    """Every shape x every mode (a shared model takes the single-row shortcut), per-stage boxes on alternate cases; on one
    mode per shape also a smaller batch first (the staging buffers grow on the second call) and x_out / u_out NULL."""
    f32 = dtype == torch.float32
    settings = dict(rho=0.1 if f32 else 1.0, eps_abs=1e-3, eps_rel=1e-3, max_iter=300)
    for si, (nx, nu, slack) in enumerate(SHAPES):
        for mi in range(len(MODES)):
            N = 2 + (si + mi) % 6
            prob = Problem(nx, nu, slack, N, seed=7200 + 6 * si + mi, f32=f32, box=(si + mi) % 2 == 0)
            assert MODES[mi] == (prob.tv, prob.shared, prob.g is not None)
            dev = prob.solver(be, dtype, **settings)
            host = prob.solver(be, dtype, **settings)
            tag = (nx, nu, slack, N, MODES[mi], dtype)
            extra = mi == si % len(MODES)
            if extra:
                small = 9
                for a, b in zip(_host_path(host, prob, small), _device_path(dev, prob, small)):
                    assert _bitwise(a, b), tag + ("batch 9",)
            ref = _device_path(dev, prob, B)
            for a, b in zip(_host_path(host, prob, B), ref):
                assert _bitwise(a, b), tag
            if extra:
                xo, uo, it, st = _host_path(host, prob, B, want_x=False)
                assert xo is None and _bitwise(uo, ref[1]) and _bitwise(it, ref[2]) and _bitwise(st, ref[3]), tag + ("x_out NULL",)
                xo, uo, it, st = _host_path(host, prob, B, want_u=False)
                assert uo is None and _bitwise(xo, ref[0]) and _bitwise(it, ref[2]) and _bitwise(st, ref[3]), tag + ("u_out NULL",)
            dev.close(); host.close()


# ---------------------------------------------------------------------------------------------------------------------
DTYPES = pytest.mark.parametrize("dtype", [torch.float64, torch.float32], ids=["f64", "f32"])


@DTYPES
def test_build_qp_cpu(emu_backend, dtype):
    check_build_qp(emu_backend, dtype)


@DTYPES
def test_build_qp_after_updates_cpu(emu_backend, dtype):
    check_build_after_updates(emu_backend, dtype)


def test_build_qp_before_setup_cpu(emu_backend):
    check_build_before_setup(emu_backend)


def test_qp_pattern_cpu(emu_backend):
    check_pattern(emu_backend)


@DTYPES
def test_model_kernels_cpu(emu_backend, golden, dtype):
    lat = check_lateral(emu_backend, dtype)
    dyn = check_dynamics(emu_backend, dtype, golden)
    kin = check_kinematics(emu_backend, dtype, golden)
    print("worst rel. deviation (emu, %s): lateral %.2e, dynamics %.2e / step %.2e, kinematics %.2e / step %.2e"
          % (dtype, lat, dyn["linearize"], dyn["step"], kin["linearize"], kin["step"]))


@DTYPES
def test_augment_and_plant_cpu(emu_backend, dtype):
    check_augment(emu_backend, dtype)
    print("plant step (emu, %s): worst error %.2f of its bound" % (dtype, check_plant(emu_backend, dtype)))


@DTYPES
def test_model_argument_errors_cpu(emu_backend, dtype):
    check_model_argument_errors(emu_backend, dtype)


@DTYPES
def test_layout_round_trip_cpu(emu_backend, dtype):
    check_layout(emu_backend, dtype)


@DTYPES
def test_solve_host_cpu(emu_backend, dtype):
    check_solve_host(emu_backend, dtype)


@pytest.mark.gpu
@DTYPES
def test_build_qp_gpu(cuda_backend, dtype):
    check_build_qp(cuda_backend, dtype)
    check_build_after_updates(cuda_backend, dtype)


@pytest.mark.gpu
def test_build_qp_before_setup_and_pattern_gpu(cuda_backend):
    check_build_before_setup(cuda_backend)
    check_pattern(cuda_backend)


@pytest.mark.gpu
def test_build_qp_at_scale_gpu(cuda_backend):
    check_build_qp_at_scale(cuda_backend)


@pytest.mark.gpu
@DTYPES
def test_model_kernels_gpu(cuda_backend, golden, dtype):
    lat = check_lateral(cuda_backend, dtype)
    dyn = check_dynamics(cuda_backend, dtype, golden)
    kin = check_kinematics(cuda_backend, dtype, golden)
    print("worst rel. deviation (GPU, %s): lateral %.2e, dynamics %.2e / step %.2e, kinematics %.2e / step %.2e"
          % (dtype, lat, dyn["linearize"], dyn["step"], kin["linearize"], kin["step"]))


@pytest.mark.gpu
@DTYPES
def test_augment_plant_layout_and_errors_gpu(cuda_backend, dtype):
    check_augment(cuda_backend, dtype)
    print("plant step (GPU, %s): worst error %.2f of its bound" % (dtype, check_plant(cuda_backend, dtype)))
    check_model_argument_errors(cuda_backend, dtype)
    check_layout(cuda_backend, dtype)


@pytest.mark.gpu
@DTYPES
def test_solve_host_gpu(cuda_backend, dtype):
    check_solve_host(cuda_backend, dtype)
