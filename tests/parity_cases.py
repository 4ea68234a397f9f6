"""Parity cases shared by the CPU suite (kernel code run through tests/emu) and the GPU suite (-m gpu,
the real libmpc_b200.so).  Every case compares the product path with the oracle (oracle/) on the same
seeded inputs or with the committed golden fixtures captured from the reference's own code."""
import numpy as np
import scipy.sparse as sp
import torch

import python_mpc_b200 as pm
from python_mpc_b200 import mpc as pmpc
from python_mpc_b200 import vehicle_models, workloads
from oracle import osqp_admm, ref_qp, workload_qp

DEG = np.pi / 180
# north_star tolerances: primal solutions agree within 1e-6 relative in FP64, 1e-4 in FP32
TOL = {torch.float64: 1e-6, torch.float32: 1e-4}


def rel(a, b):
    return float(np.abs(np.asarray(a, dtype=np.float64) - b).max() / np.abs(b).max())


def oracle_solve(qp, **settings):
    return osqp_admm.OSQP().setup(*ref_qp.assemble(qp), **settings).solve()


def check_lateral_batch(be, slack, increment, dtype, B=6, rho=5.0, shared=False, seed=11, eps=1e-4, max_iter=4000,
                        samples=None):
    """LateralMPC.solve_batch vs the oracle: same status, same iteration count, primal within tolerance."""
    if shared:
        wl = workloads.LateralWorkload(B, 20, slack, increment, seed, dtype, shared_speed=8.3128334)
    else:
        wl = workloads.LateralWorkload(B, 20, slack, increment, seed, dtype)
    veh = vehicle_models.Vehicle_Lateral(dtype=dtype, _backend=be)
    ctl = wl.make_controller(vehicle=veh, _backend=be, rho=rho, eps_abs=eps, eps_rel=eps, warm_start=False,
                             max_iter=max_iter)
    res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    x = res.x.cpu().numpy(); it = res.info.iter.cpu().numpy(); st = res.info.status_val.cpu().numpy()
    worst = 0.0
    for b in (range(B) if samples is None else samples):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=rho, eps_abs=eps, eps_rel=eps, max_iter=max_iter)
        assert st[b] == r.info.status_val, (b, st[b], r.info.status)
        if dtype == torch.float64:
            assert it[b] == r.info.iter, (b, it[b], r.info.iter)
        worst = max(worst, rel(x[b], r.x))
        N, nx = wl.N, wl.nx
        np.testing.assert_allclose(res.u[b].cpu().numpy().ravel(), x[b][(N + 1) * nx:(N + 1) * nx + N], rtol=0, atol=0)
    assert worst < TOL[dtype], worst
    return worst


def check_iterates(be, dtype, iters, rho, B=4, seed=5):
    """Exactly `iters` ADMM iterations from a cold start, no termination test: iterate-for-iterate parity."""
    wl = workloads.lateral_slack_increment(B, seed=seed, dtype=dtype)
    ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(dtype=dtype, _backend=be), _backend=be, rho=rho,
                             warm_start=False, max_iter=1)
    ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    s = ctl.solver
    s.cold_start(); s.iterate(iters)
    x, y, _ = s.solution(want_y=True)
    worst = 0.0
    for b in range(B):
        o = osqp_admm.OSQP().setup(*ref_qp.assemble(workload_qp.lateral_qp(wl, b)), rho=rho)
        for _ in range(iters):
            o.iterate()
        xo = o.D * o.x; yo = o.cinv * o.E * o.y
        worst = max(worst, rel(x[b].cpu().numpy(), xo), rel(y[b].cpu().numpy(), yo))
    assert worst < TOL[dtype], worst
    return worst


def check_build_qp_against_reference_capture(be, golden):
    """mpcb_build_qp (explicit P, q, A, l, u) vs the matrices the reference's own code assembled."""
    g = golden["lateral_slack_increment_closed_loop"]
    N = int(g["N"])
    xmin = np.array([-np.pi, -0.5 * np.pi, -15 * DEG, -10., -30 * DEG])
    ctl = pmpc.LateralMPC(N, [5., 5., 10., 10.], [10.], xmin, -xmin, [-0.5 * DEG], [0.5 * DEG], slack=True, increment=True,
                          W=[10., 10., 10., 10., 0.], S=[1., 1., 1., 1., 0.], Ad=g["Ad"], Bd=g["Bd"], _backend=be, max_iter=1)
    ctl.solve_batch(np.array([[0., 0., 5 * DEG, 3., 0.]]), np.zeros((1, 4)))
    Pd, q, Av, l, u, Ap, Ai = ctl.solver.build_qp()
    A = sp.csc_matrix((Av[0].cpu().numpy(), Ai, Ap), shape=(ctl.solver.ncon, ctl.solver.nvar)).toarray()
    assert np.array_equal(A, g["A"])
    assert np.array_equal(np.diag(Pd[0].cpu().numpy()), g["P"])
    assert np.array_equal(q[0].cpu().numpy(), g["q"])
    assert np.array_equal(l[0].cpu().numpy(), g["l"]) and np.array_equal(u[0].cpu().numpy(), g["u"])


def check_models_against_reference(be, golden):
    g = golden["vehicle_models"]
    vd = vehicle_models.Vehicle_Dynamics(dt=float(g["dyn_dt"]), _backend=be)
    A, B, gd = vd.get_dynamics_model(g["dyn_x"], g["dyn_u"])
    np.testing.assert_allclose(A.cpu().numpy(), g["dyn_Ad"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(B.cpu().numpy(), g["dyn_Bd"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(gd.cpu().numpy(), g["dyn_gd"], rtol=0, atol=1e-11)
    a1, b1, g1 = vd.get_dynamics_model(g["dyn_x"][7], g["dyn_u"][7])       # single-vehicle, reference shapes
    assert a1.shape == (6, 6) and b1.shape == (6, 2) and g1.shape == (6, 1)
    np.testing.assert_allclose(a1, g["dyn_Ad"][7], atol=1e-12)
    vk = vehicle_models.Vehicle_Kinematics(dt=float(g["kin_dt"]), _backend=be)
    A, B, C = vk.get_kinematics_model(g["kin_x"], g["kin_u"])
    np.testing.assert_allclose(A.cpu().numpy(), g["kin_A"], rtol=0, atol=1e-14)
    np.testing.assert_allclose(B.cpu().numpy(), g["kin_B"], rtol=0, atol=1e-14)
    np.testing.assert_allclose(C.cpu().numpy(), g["kin_C"], rtol=0, atol=1e-14)
    # the nonlinear plant steps (update_dynamics_model incl. its low-speed guards, update_kinematics_model)
    xn, _ = vd.update_dynamics_model(g["dyn_x"], g["dyn_u"])
    np.testing.assert_allclose(xn.cpu().numpy(), g["dyn_xnext"], rtol=0, atol=1e-11)
    x1, af, ar = vd.update_dynamics_model(g["dyn_x"][7], g["dyn_u"][7])
    assert x1.shape == (6, 1) and np.abs(x1[:, 0] - g["dyn_xnext"][7]).max() < 1e-11 and np.isfinite(af) and np.isfinite(ar)
    xn = vk.update_kinematics_model(g["kin_x"], g["kin_u"])
    np.testing.assert_allclose(xn.cpu().numpy(), g["kin_xnext"], rtol=0, atol=1e-13)
    assert np.abs(vk.update_kinematics_model(g["kin_x"][3], g["kin_u"][3]) - g["kin_xnext"][3]).max() < 1e-13
    vl = vehicle_models.Vehicle_Lateral(_backend=be)
    v = np.array([0.05, 1.0, 8.3128334, 20.0, 35.0, -6.0])
    A, B = vl.get_lateral_model(v)
    for i, vi in enumerate(v):
        Ao, Bo = workload_qp.lateral_model(float(vi))
        np.testing.assert_allclose(A[i].cpu().numpy(), Ao, rtol=0, atol=1e-12)
        np.testing.assert_allclose(B[i].cpu().numpy(), Bo, rtol=0, atol=1e-12)
    gl = golden["lateral_slack_increment_closed_loop"]                      # the reference's hard-coded literals
    assert np.abs(A[2].cpu().numpy() - gl["Ad"]).max() < 2.5e-3 and np.abs(B[2].cpu().numpy() - gl["Bd"]).max() < 1e-4


def check_reference_functions(be, golden):
    """mpc / mpc_lists / mpc_increment with the reference's signatures vs fixtures made by the reference's
    own functions (assembly) + the oracle (solve)."""
    s = dict(eps_abs=1e-4, eps_rel=1e-4, _backend=be)
    g = golden["qp_vanilla_kinematic"]
    res = pmpc.mpc(g["Ad"], g["Bd"], g["gd"].reshape(-1, 1), g["x_init"], g["Xr"], sp.diags(g["Q"]), sp.diags(g["QN"]),
                   sp.diags(g["R"]), int(g["N"]), g["xmin"], g["xmax"], g["umin"], g["umax"], **s)
    assert res.info.status_val == int(g["sol_status"]) and res.info.iter == int(g["sol_iter"])
    assert rel(res.x, g["sol_x"]) < 1e-6
    g = golden["qp_vanilla_dynamic"]
    N = int(g["N"])
    px, pu = np.zeros((6, N + 1)), np.zeros((2, N + 1))
    px, pu = pmpc.mpc_lists(list(g["Ad"]), list(g["Bd"]), [v.reshape(-1, 1) for v in g["gd"]], g["x_init"], g["Xr"], px, pu,
                            sp.diags(g["Q"]), sp.diags(g["QN"]), sp.diags(g["R"]), N, g["xmin"], g["xmax"], g["umin"],
                            g["umax"], **s)
    assert rel(px, g["pred_x"]) < 1e-6 and rel(pu, g["pred_u"]) < 1e-6
    g = golden["qp_increment_dynamic"]
    px, pdu = np.zeros((8, N + 1)), np.zeros((2, N + 1))
    px, pdu = pmpc.mpc_increment(list(g["Ad"]), list(g["Bd"]), [v.reshape(-1, 1) for v in g["gd"]], g["x_init"], g["Xr"],
                                 px, pdu, sp.diags(g["Q"]), sp.diags(g["QN"]), sp.diags(g["R"]), N, g["xmin"], g["xmax"],
                                 g["umin"], g["umax"], **s)
    assert rel(px, g["pred_x"]) < 1e-6 and rel(pdu, g["pred_du"]) < 1e-6


def check_kinematic_corridor_and_predmatrix(be, golden):
    """mpc_ (per-stage position corridor, mpc_kinematics.py:202), mpc__ (per-stage linearisations,
    mpc_kinematics_pred_matrix.py:268) and the kinematic mpc_increment (mpc_increment_kinematics_pred_matrix.py:150)
    with the reference's signatures vs a fixture made by the reference's own functions (assembly) + the oracle."""
    g = golden["qp_kinematic_corridor_predmatrix"]
    N = int(g["N"])
    s = dict(eps_abs=1e-4, eps_rel=1e-4, _backend=be)
    Q, QN, R = sp.diags(g["Q"]), sp.diags(g["QN"]), sp.diags(g["R"])
    res = pmpc.mpc_(g["Ad"], g["Bd"], g["gd"].reshape(-1, 1), g["x_init"], g["Xr"], Q, QN, R, N, g["lb_x"], g["ub_x"],
                    g["lb_y"], g["ub_y"], g["umin"], g["umax"], **s)
    assert res.info.status_val == int(g["corr_status"]) and res.info.iter == int(g["corr_iter"])
    assert rel(res.x, g["corr_x"]) < 1e-6
    X = res.x[:(N + 1) * 4].reshape(N + 1, 4)                       # the corridor is what binds this solution
    assert (X[:, 0] >= g["lb_x"] - 1e-3).all() and (X[:, 0] <= g["ub_x"] + 1e-3).all()
    res = pmpc.mpc__(list(g["Ad_list"]), list(g["Bd_list"]), [v.reshape(-1, 1) for v in g["gd_list"]], g["x_init"], g["Xr"],
                     Q, QN, R, N, g["xmin"], g["xmax"], g["umin"], g["umax"], **s)
    assert res.info.status_val == int(g["list_status"]) and res.info.iter == int(g["list_iter"])
    assert rel(res.x, g["list_x"]) < 1e-6
    px, pdu = np.zeros((6, N + 1)), np.zeros((2, N + 1))
    px, pdu = pmpc.mpc_increment(list(g["Ad_list"]), list(g["Bd_list"]), [v.reshape(-1, 1) for v in g["gd_list"]],
                                 np.concatenate([g["x_init"], g["u_init"]]), g["Xr"], px, pdu, Q, QN, R, N, g["xmin_t"],
                                 g["xmax_t"], g["del_umin"], g["del_umax"], **s)
    assert rel(px, g["inc_pred_x"]) < 1e-6 and rel(pdu, g["inc_pred_du"]) < 1e-6


def check_closed_loop(be, golden, steps=None):
    """The reference script's closed loop (setup once, update(q,l,u) + warm-started solve every step) through
    LateralMPC.solve: lateral-error trajectory within 1e-3 m of the fixture (north_star bound)."""
    g = golden["lateral_slack_increment_closed_loop"]
    N = int(g["N"]); nsim = int(g["nsim"]) if steps is None else steps
    xmin = np.array([-np.pi, -0.5 * np.pi, -15 * DEG, -10., -30 * DEG])
    ctl = pmpc.LateralMPC(N, [5., 5., 10., 10.], [10.], xmin, -xmin, [-0.5 * DEG], [0.5 * DEG], slack=True, increment=True,
                          W=[10., 10., 10., 10., 0.], S=[1., 1., 1., 1., 0.], Ad=g["Ad"], Bd=g["Bd"], _backend=be,
                          eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
    At, Bt, _ = ref_qp.augment_increment(g["Ad"], g["Bd"], None)
    x0 = np.array([0., 0., 5 * DEG, 3., 0.])
    ey, du, its = [], [], []
    for i in range(nsim):
        ey.append(x0[3])
        useq = ctl.solve(x0, np.zeros(4))
        its.append(int(ctl.last.info.iter[0]))
        du.append(useq[0, 0])
        x0 = At @ x0 + Bt @ useq[0]
    assert np.abs(np.array(ey) - g["x4"][:nsim]).max() < 1e-3
    assert np.abs(np.array(du) - g["del_u"][:nsim]).max() < 1e-5
    assert its == g["iters"][:nsim].tolist()


def check_closed_loop_full(be, golden, steps=None):
    """The UNMODIFIED reference script (N = 100, 1500 closed-loop steps) through LateralMPC: setup once, then per step
    prob.update(q, l, u) — with the tightened lateral-error bound xmin_tilda[3] = 2 for steps 401..900
    (vehicle_lateral_mpc_slack_increment.py:158-172, :237) — and a warm-started prob.solve().  Against the fixture made by
    the script itself + the oracle: e_y within 1e-3 m (north_star), delta-u within 1e-5, the slack the script plots
    (res.x[-(N+1)*nx:][3], :259) and the iteration count of every step."""
    g = golden["lateral_slack_increment_closed_loop_full"]
    N = int(g["N"]); nsim = int(g["nsim"]) if steps is None else steps
    xmin = np.array([-np.pi, -0.5 * np.pi, -15 * DEG, -10., -30 * DEG])
    tight = xmin.copy(); tight[3] = 2.0
    ctl = pmpc.LateralMPC(N, [5., 5., 10., 10.], [10.], xmin, -xmin, [-0.5 * DEG], [0.5 * DEG], slack=True, increment=True,
                          W=[10., 10., 10., 10., 0.], S=[1., 1., 1., 1., 0.], Ad=g["Ad"], Bd=g["Bd"], _backend=be,
                          rho=float(g["rho"]), eps_abs=float(g["eps"]), eps_rel=float(g["eps"]), warm_start=True)
    At, Bt, _ = ref_qp.augment_increment(g["Ad"], g["Bd"], None)
    x0 = np.array([0., 0., 5 * DEG, 3., 0.])
    nx = 5
    ey, du, its, slack = [], [], [], []
    for i in range(nsim):
        if i == 401:
            ctl.update_bounds(xmin=tight)
        elif i == 901:
            ctl.update_bounds(xmin=xmin)
        ey.append(x0[3])
        useq = ctl.solve(x0, np.zeros(4))
        its.append(int(ctl.last.info.iter[0]))
        du.append(useq[0, 0])
        slack.append(float(ctl.last.x[0, -(N + 1) * nx:][3]))
        x0 = At @ x0 + Bt @ useq[0]
    assert np.abs(np.array(ey) - g["x4"][:nsim]).max() < 1e-3
    assert np.abs(np.array(du) - g["del_u"][:nsim]).max() < 1e-5
    assert np.abs(np.array(slack) - g["slack"][:nsim]).max() < 1e-5
    assert its == g["iters"][:nsim].tolist()
    if nsim > 450:
        assert np.abs(np.array(slack)[401:nsim]).max() > 1.0      # the regime where the soft constraint works
    return np.array(slack)


def check_bound_updates(be, B=6, steps=36, rho=5.0, N=20, seed=41, switch=(6, 24)):
    """prob.update(l=l_new, u=u_new) with CHANGED inequality bounds (vehicle_lateral_mpc_slack_increment.py:158-172, :237)
    in a batched closed loop: at step switch[0] the lateral-error lower bound is tightened to +2 (slack becomes active for
    every scenario below it), at switch[1] it is relaxed again.  Every step is compared with the oracle's update()
    (osqp_update_bounds: same scaling, rho types re-evaluated, refactor if a type changed) + warm-started solve:
    iteration counts, applied input, slack of the lateral-error row, trajectory."""
    dt = torch.float64
    wl = workloads.LateralWorkload(B, N, True, True, seed, dt)
    wl.x0[:, 3] = np.linspace(-1.0, 3.5, B)          # some scenarios start below the tightened bound, some above
    ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=rho, eps_abs=1e-4,
                             eps_rel=1e-4, warm_start=True)
    tight = wl.xmin.copy(); tight[3] = 2.0
    sched = {switch[0]: dict(xmin=tight), switch[1]: dict(xmin=wl.xmin)}
    xs_gpu = []

    class Rec:                       # record res.x of every step through the public API
        pass
    s = ctl.solver
    traj, us, its = ctl.closed_loop_batch(wl.x0, wl.xr, wl.speed, steps=steps, bounds_at=lambda k: sched.get(k))
    traj = traj.cpu().numpy(); us = us.cpu().numpy(); its = its.cpu().numpy()
    x_last, _, _ = s.solution()
    x_last = x_last.cpu().numpy()
    nx = 5
    slack_seen = 0.0
    for b in range(B):
        Ad, Bd = workload_qp.lateral_model(float(wl.speed[b]))
        At, Bt, _ = ref_qp.augment_increment(Ad, Bd, None)
        P, q, A, l, u = ref_qp.assemble(workload_qp.lateral_qp(wl, b))
        o = osqp_admm.OSQP().setup(P, q, A, l, u, rho=rho, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
        x = wl.x0[b].copy()
        bx0 = (N + 1) * nx                      # first bx row
        for k in range(steps):
            if k in sched:
                lo = sched[k]["xmin"]
                l[bx0:bx0 + (N + 1) * nx] = np.tile(lo, N + 1)
            if k > 0:
                l[:nx] = -x; u[:nx] = -x
            if k > 0 or k in sched:
                o.update(l=l, u=u)
            r = o.solve()
            assert r.info.status_val == 1
            assert r.info.iter == its[k, b], (b, k, r.info.iter, its[k, b])
            du = r.x[(N + 1) * nx:(N + 1) * nx + 1]
            assert abs(du[0] - us[k, b, 0]) < 1e-6 * max(1.0, abs(du[0])), (b, k, du[0], us[k, b, 0])
            slack_seen = max(slack_seen, float(np.abs(r.x[-(N + 1) * nx:]).max()))
            x = At @ x + Bt @ du
            assert np.abs(x - traj[k + 1, b]).max() < 1e-3 and abs(x[3] - traj[k + 1, b, 3]) < 1e-6
        assert rel(x_last[b], r.x) < 1e-6
    assert slack_seen > 0.1, "the tightened bound never activated the slack (%g)" % slack_seen
    # a bound that turns a row into an equality (u - l < RHO_TOL after scaling) changes its rho type: refactor path
    eq = wl.xmin.copy(); eq[2] = wl.xmax[2] - 1e-6
    ctl.update_bounds(xmin=eq)
    res = ctl.update_batch(traj[-1])
    for b in (0, B - 1):
        Ad, Bd = workload_qp.lateral_model(float(wl.speed[b]))
        P, q, A, l, u = ref_qp.assemble(workload_qp.lateral_qp(wl, b))
        o = osqp_admm.OSQP().setup(P, q, A, l, u, rho=rho, eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
        types0 = o.constr_type.copy()
        l[bx0:bx0 + (N + 1) * nx] = np.tile(eq, N + 1)
        l[:nx] = -traj[-1, b]; u[:nx] = -traj[-1, b]
        o.update(l=l, u=u)
        assert (types0 != o.constr_type).any()
        r = o.solve()
        # (cold-started comparison of the optimum only: the warm-start history of the GPU side differs)
        assert int(res.info.status_val[b]) == r.info.status_val
        if r.info.status_val == 1:
            assert rel(res.x[b].cpu().numpy(), r.x) < 5e-3
    # inverted bounds are rejected like OSQP's update
    try:
        ctl.update_bounds(xmin=wl.xmax + 1.0)
        raise AssertionError("expected an error")
    except pm.MpcError as e:
        assert "lower bound must be lower than or equal to upper bound" in str(e)
    return slack_seen


def check_setup_resets_iterates(be, B=8):
    """prob.setup() leaves x = z = y = 0: a second solve_batch on the same controller equals a fresh controller's
    (no warm start across setups, ADVICE r1), while update + solve keeps the warm start."""
    dt = torch.float64
    wa = workloads.lateral_slack_increment(B, seed=51, dtype=dt)
    wb = workloads.lateral_slack_increment(B, seed=52, dtype=dt)
    mk = lambda w: w.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=5.0,
                                     eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
    c1 = mk(wa)
    c1.solve_batch(wa.x0, wa.xr, wa.speed)
    r1 = c1.solve_batch(wb.x0, wb.xr, wb.speed)
    r2 = mk(wb).solve_batch(wb.x0, wb.xr, wb.speed)
    assert torch.equal(r1.info.iter, r2.info.iter) and torch.equal(r1.x, r2.x)
    # warm start across update() is kept: re-solving the same data converges at the first termination test
    r3 = c1.update_batch(wb.x0)
    assert int(r3.info.iter.max()) == 25


def check_host_front_door(be, dtype=torch.float64):
    """mpcb_solve_host (numpy-layout host buffers, copies inside) equals the device path."""
    wl = workloads.lateral_slack_increment(5, seed=21, dtype=dtype)
    Ad, Bd = zip(*[workload_qp.lateral_model(float(v)) for v in wl.speed])
    At, Bt, _ = ref_qp.augment_increment(np.stack(Ad), np.stack(Bd), None)
    s = pm.BatchSolver(20, 5, 1, np.concatenate([wl.Q, [0]]), np.concatenate([wl.Q, [0]]), wl.R, wl.xmin, wl.xmax, wl.umin,
                       wl.umax, slack=True, W=wl.W, S=wl.S, dtype=dtype, capacity=8, _backend=be, rho=5.0, eps_abs=1e-4,
                       eps_rel=1e-4, warm_start=False)
    xr = np.zeros((5, 5))
    xo, uo, it, st = s.solve_host(At, Bt, None, wl.x0, xr)
    for b in range(5):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert st[b] == 1 and it[b] == r.info.iter
        assert rel(xo[b], r.x) < TOL[dtype]
        np.testing.assert_array_equal(uo[b].ravel(), xo[b][105:125])


def check_edge_cases(be):
    dt = torch.float64
    xmin = np.array([-np.pi, -0.5 * np.pi, -15 * DEG, -10.])
    mk = lambda **kw: pmpc.LateralMPC(20, [5., 5., 10., 10.], [10.], xmin, -xmin, [-30 * DEG], [30 * DEG], dtype=dt,
                                      _backend=be, **kw)
    # ragged batch sizes (not a multiple of the warp / leading dimension) and batch < capacity
    for B, cap in ((1, 1), (3, 64), (33, 40)):
        wl = workloads.LateralWorkload(B, 20, False, False, 3, dt)
        ctl = mk(capacity=cap, rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
        r = oracle_solve(workload_qp.lateral_qp(wl, B - 1), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert rel(res.x[B - 1].cpu().numpy(), r.x) < 1e-6 and int(res.info.iter[B - 1]) == r.info.iter
    # iteration cap: same status as OSQP ("maximum iterations reached" = -2), same iterate
    wl = workloads.LateralWorkload(2, 20, False, False, 4, dt)
    ctl = mk(capacity=2, rho=0.1, eps_abs=1e-7, eps_rel=1e-7, max_iter=40)
    res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    r = oracle_solve(workload_qp.lateral_qp(wl, 0), rho=0.1, eps_abs=1e-7, eps_rel=1e-7, max_iter=40)
    assert int(res.info.status_val[0]) == r.info.status_val == -2 and int(res.info.iter[0]) == 40
    assert rel(res.x[0].cpu().numpy(), r.x) < 1e-6
    # single-vehicle drop-in raises like the reference when OSQP does not return 'solved'
    try:
        ctl.solve(wl.x0[0], wl.xr[0], speed=float(wl.speed[0]))
        raise AssertionError("expected ValueError")
    except ValueError as e:
        assert "OSQP did not solve the problem!" in str(e)
    # batch larger than capacity, inverted bounds, unsupported shapes, calls out of order, an unknown option
    for bad in (lambda: mk(capacity=2).solve_batch(np.zeros((3, 4)), np.zeros((3, 4)), np.ones(3)),
                lambda: pmpc.LateralMPC(20, [5.] * 4, [10.], -xmin, xmin, [-1.], [1.], _backend=be),
                lambda: pm.BatchSolver(20, 7, 2, np.ones(7), np.ones(7), np.ones(2), -np.ones(7), np.ones(7), [-1, -1], [1, 1],
                                       _backend=be),
                lambda: pm.BatchSolver(0, 4, 1, np.ones(4), np.ones(4), [1.], -np.ones(4), np.ones(4), [-1], [1], _backend=be),
                lambda: mk(capacity=2).solver.solve(),
                lambda: mk(capacity=2, rho=-1.0),
                lambda: mk(capacity=2, adaptive_rho=True),
                lambda: be.set_option("wide", 1)):
        try:
            bad()
        except (pm.MpcError, ValueError, TypeError):
            continue
        raise AssertionError("expected an error")


def check_primal_infeasibility(be, B=5, retile=False):
    """Vanilla (hard-constraint) lateral MPC whose initial state violates the state box: dyn_0 pins x_0 = x_init, bx_0
    excludes it.  OSQP's certificate (auxil.c: is_primal_infeasible) must fire at the same termination test as in the
    oracle, per QP, next to feasible QPs of the same batch; infeasible QPs return NaN like OSQP's results."""
    dt = torch.float64
    wl = workloads.LateralWorkload(B, 20, False, False, 9, dt)
    wl.x0[1, 3] = 14.0          # lateral error beyond xmax[3] = 10
    wl.x0[3, 2] = -0.5          # heading error beyond xmin[2] = -15 deg
    if retile:
        be.set_option("retile_min_batch", 2)
    try:
        ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(dtype=dt, _backend=be), _backend=be, rho=5.0,
                                 eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
        res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    finally:
        be.set_option("retile_min_batch", 4096)
    x = res.x.cpu().numpy(); it = res.info.iter.cpu().numpy(); st = res.info.status_val.cpu().numpy()
    for b in range(B):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert st[b] == r.info.status_val and it[b] == r.info.iter, (b, st[b], it[b], r.info.status, r.info.iter)
        if b in (1, 3):
            assert st[b] == -3 and res.info.status[b] == "primal infeasible"
            assert np.isnan(x[b]).all() and np.isnan(res.u[b].cpu().numpy()).all()
        else:
            assert st[b] == 1 and rel(x[b], r.x) < 1e-6
    # the single-vehicle drop-in raises like the reference script (status != 'solved')
    try:
        ctl.solve(wl.x0[1], wl.xr[1], speed=float(wl.speed[1]))
        raise AssertionError("expected ValueError")
    except ValueError as e:
        assert "OSQP did not solve the problem!" in str(e)
    # approximate certificate at the iteration cap (tolerances x10): OSQP's "primal infeasible inaccurate"
    ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(dtype=dt, _backend=be), _backend=be, rho=5.0,
                             eps_abs=1e-4, eps_rel=1e-4, eps_prim_inf=1e-9, warm_start=False, max_iter=60)
    res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    st = res.info.status_val.cpu().numpy()
    for b in (1, 3):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4, eps_prim_inf=1e-9, max_iter=60)
        assert st[b] == r.info.status_val, (b, st[b], r.info.status)
    # the same certificate with unbounded rows in the problem (delta-y is projected on the recession cone of each row's
    # bound type first): kinematic model, x/y position unbounded, initial speed above its upper bound
    N, nx, nu = 12, 4, 2
    kin = vehicle_models.Vehicle_Kinematics(dt=0.02, _backend=be)
    x = np.array([0.0, 0.0, 5.0, 30 * DEG]); u = np.array([0.02, 0.01])
    A, Bm, C = kin.get_kinematics_model(x, u)
    Q = np.array([1., 1., 5., 10.]); QN = np.array([10., 10., 50., 50.]); R = np.array([0.1, 0.1])
    umin = np.array([-15 * DEG, -3.]); umax = np.array([15 * DEG, 1.])
    lo = np.array([-np.inf, -np.inf, -10., -np.pi]); hi = np.array([np.inf, np.inf, 4.0, np.pi])
    Xr = np.zeros((nx, N + 1)); Xr[2] = 5.0
    s = pm.BatchSolver(N, nx, nu, Q, QN, R, lo, hi, umin, umax, dtype=torch.float64, stage_reference=True, capacity=1,
                       _backend=be, eps_abs=1e-5, eps_rel=1e-5, warm_start=False)
    s.setup(A[None], Bm[None], C.reshape(1, nx), x[None], Xr[None]); s.solve()
    r = oracle_solve(ref_qp.canonical(N, A, Bm, C.reshape(1, nx), Q, QN, R, Xr, lo, hi, umin, umax, x), eps_abs=1e-5,
                     eps_rel=1e-5)
    inf = s.info()
    assert r.info.status_val == -3 and int(inf.status_val[0]) == -3 and int(inf.iter[0]) == r.info.iter, \
        (r.info.status, r.info.iter, int(inf.status_val[0]), int(inf.iter[0]))
    # feasible problems never trip a certificate: the dual one cannot hold for this family (the cost is a sum of
    # squares, q = -Q xr), and the oracle agrees on every status of the feasible batches in this module
    return st


def check_infinite_bounds_and_stage_boxes(be):
    """-inf/+inf bounds (RHO_MIN rows) and per-stage state boxes (mpc_ of mpc_kinematics.py:215)."""
    rng = np.random.default_rng(2)
    N, nx, nu = 12, 4, 2
    kin = vehicle_models.Vehicle_Kinematics(dt=0.02, _backend=be)
    x = np.array([0.0, 0.0, 5.0, 30 * DEG]); u = np.array([0.02, 0.01])
    A, B, C = kin.get_kinematics_model(x, u)
    Q = np.array([1., 1., 5., 10.]); QN = np.array([10., 10., 50., 50.]); R = np.array([0.1, 0.1])
    umin = np.array([-15 * DEG, -3.]); umax = np.array([15 * DEG, 1.])
    lo = np.tile(np.array([-np.inf, -np.inf, -10., -np.pi]), (N + 1, 1)); hi = -lo
    lo[:, 0] = np.linspace(-1, 0.5, N + 1); hi[:, 0] = lo[:, 0] + 2.0
    lo[:, 1] = -3.0; hi[:, 1] = 3.0
    Xr = np.zeros((nx, N + 1)); Xr[0] = np.linspace(0, 1, N + 1); Xr[2] = 5.0
    s = pm.BatchSolver(N, nx, nu, Q, QN, R, lo[0], hi[0], umin, umax, dtype=torch.float64, stage_reference=True, capacity=1,
                       _backend=be, eps_abs=1e-5, eps_rel=1e-5, warm_start=False)
    s.set_stage_bounds(lo, hi)
    s.setup(A[None], B[None], C.reshape(1, nx), x[None], Xr[None]); s.solve()
    xg, _, _ = s.solution()
    qp = ref_qp.canonical(N, A, B, C.reshape(1, nx), Q, QN, R, Xr, lo, hi, umin, umax, x)
    r = oracle_solve(qp, eps_abs=1e-5, eps_rel=1e-5)
    assert int(s.info().iter[0]) == r.info.iter and rel(xg[0].cpu().numpy(), r.x) < 1e-6
    # prob.update(l=, u=) with a MOVED corridor (per-stage boxes through mpcb_update_bounds): scaling kept, warm start kept
    lo_b = lo.copy(); hi_b = hi.copy()
    lo_b[:, 0] += 0.3; hi_b[:, 0] += 0.3; hi_b[:, 1] = 2.5
    s.update_bounds(stage_lo=lo_b, stage_hi=hi_b)
    s.update_settings(warm_start=True)
    s.solve()
    Pm, qv, Am, lv, uv = ref_qp.assemble(qp)
    o = osqp_admm.OSQP().setup(Pm, qv, Am, lv, uv, eps_abs=1e-5, eps_rel=1e-5, warm_start=True)
    o.solve()
    _, _, _, l2, u2 = ref_qp.assemble(ref_qp.canonical(N, A, B, C.reshape(1, nx), Q, QN, R, Xr, lo_b, hi_b, umin, umax, x))
    o.update(l=l2, u=u2)
    r_b = o.solve()
    assert int(s.info().iter[0]) == r_b.info.iter and rel(s.solution()[0][0].cpu().numpy(), r_b.x) < 1e-6
    # same problem with the unbounded rows of the reference (xmin = -inf ...): constraint type "unconstrained"
    lo2 = np.array([-np.inf, -np.inf, -100., -np.pi]); hi2 = -lo2
    s2 = pm.BatchSolver(N, nx, nu, Q, QN, R, lo2, hi2, umin, umax, dtype=torch.float64, stage_reference=True, capacity=1,
                        _backend=be, eps_abs=1e-5, eps_rel=1e-5, warm_start=False)
    s2.setup(A[None], B[None], C.reshape(1, nx), x[None], Xr[None]); s2.solve()
    r2 = oracle_solve(ref_qp.canonical(N, A, B, C.reshape(1, nx), Q, QN, R, Xr, lo2, hi2, umin, umax, x), eps_abs=1e-5,
                      eps_rel=1e-5)
    assert int(s2.info().iter[0]) == r2.info.iter and rel(s2.solution()[0][0].cpu().numpy(), r2.x) < 1e-6


SHAPES = ((4, 1, False), (4, 1, True), (5, 1, False), (5, 1, True), (4, 2, False), (6, 2, False), (8, 2, False))


def check_random_problems(be, seeds=(0, 1), B=3, shapes=SHAPES, horizons=None):
    """Seeded random MPC QPs over every compiled (nx, nu, slack) shape: random horizon, models (per QP or shared,
    time-invariant or per stage, with / without affine term), weights (some zero), bounds (some infinite, some tight,
    sometimes excluding the initial state -> primal infeasible), rho.  Status, iteration count and primal solution
    of every QP against the oracle."""
    worst = 0.0
    seen = set()
    for nx, nu, slack in shapes:
        for seed in seeds:
            rng = np.random.default_rng(1000 * nx + 100 * nu + 10 * int(slack) + seed)
            N = int(rng.integers(3, 25))
            if horizons is not None:
                N = int(horizons[seed % len(horizons)])     # (edge horizons: the stage-buffer rotations of the TMA kernels)
            tv = bool(rng.integers(0, 2)); shared = (not tv) and bool(rng.integers(0, 2)); has_g = bool(rng.integers(0, 2))
            rho = float(rng.choice([0.1, 1.0, 5.0]))
            stages = N if tv else 1
            nm = 1 if shared else B
            A = np.eye(nx) + 0.15 * rng.standard_normal((nm, stages, nx, nx))
            Bm = 0.3 * rng.standard_normal((nm, stages, nx, nu))
            g = 0.05 * rng.standard_normal((nm, stages, nx)) if has_g else None
            Q = rng.uniform(0.5, 20, nx) * (rng.random(nx) > 0.2); QN = Q * rng.uniform(1, 10)
            R = rng.uniform(0.05, 10, nu)
            W = rng.uniform(1, 50, nx) * (rng.random(nx) > 0.2) if slack else None
            S = (rng.random(nx) > 0.3).astype(float) if slack else None
            xmax = rng.uniform(0.5, 4.0, nx); xmin = -rng.uniform(0.5, 4.0, nx)
            inf_mask = rng.random(nx) < 0.3
            xmax[inf_mask] = np.inf; xmin[inf_mask] = -np.inf
            umax = rng.uniform(0.2, 2.0, nu); umin = -rng.uniform(0.2, 2.0, nu)
            x0 = rng.uniform(-0.4, 0.4, (B, nx))
            if seed % 2 == 1 and not slack and not inf_mask[0]:
                x0[0, 0] = xmax[0] + 1.0          # outside a hard state bound: primal infeasible
            Xr = rng.uniform(-0.3, 0.3, (B, nx, N + 1))
            solver = pm.BatchSolver(N, nx, nu, Q, QN, R, xmin, xmax, umin, umax, slack=slack, W=W, S=S, dtype=torch.float64,
                                    time_varying=tv, shared_model=shared, stage_reference=True, capacity=B, _backend=be,
                                    rho=rho, eps_abs=1e-4, eps_rel=1e-4, warm_start=False, max_iter=400)
            sq = lambda M: M if tv else M[:, 0]
            Ain, Bin = sq(A), sq(Bm)
            gin = None if g is None else sq(g)
            if shared:
                Ain, Bin = Ain[0], Bin[0]
                gin = None if gin is None else gin[0]
            solver.setup(Ain, Bin, gin, x0, Xr)
            solver.solve()
            x, _, _ = solver.solution()
            inf = solver.info()
            for b in range(B):
                mb = 0 if shared else b
                qp = ref_qp.canonical(N, A[mb] if tv else A[mb, 0], Bm[mb] if tv else Bm[mb, 0],
                                      None if g is None else (g[mb] if tv else g[mb, 0][None]), Q, QN, R, Xr[b], xmin, xmax,
                                      umin, umax, x0[b], slack=slack, W=W, S=S)
                r = oracle_solve(qp, rho=rho, eps_abs=1e-4, eps_rel=1e-4, max_iter=400)
                tag = (nx, nu, slack, seed, b)
                assert int(inf.status_val[b]) == r.info.status_val, (tag, int(inf.status_val[b]), r.info.status)
                assert int(inf.iter[b]) == r.info.iter, (tag, int(inf.iter[b]), r.info.iter)
                seen.add(r.info.status_val)
                if r.info.status_val in (1, 2, -2):
                    worst = max(worst, rel(x[b].cpu().numpy(), r.x))
                    assert worst < 1e-6, (tag, worst)
                else:
                    assert np.isnan(x[b].cpu().numpy()).all()
            solver.close()
    return worst, seen


def check_closed_loop_sweep(be, B=6, steps=6, rho=5.0, sample=None, wl=None):
    """configs[4] in small: B scenarios x `steps` warm-started MPC steps on the device vs the oracle run scenario by
    scenario with OSQP's update()/warm-start semantics.  Lateral-error trajectories within 1e-3 m (north_star).
    `sample`: number of scenarios checked against the oracle (default all) — the ones with the most iterations in any
    step (the stragglers: compacted, finished in another kernel) plus evenly spaced ones.  Returns (its, us)."""
    dt = torch.float64
    if wl is None:
        wl = workloads.lateral_slack_increment(B, seed=31, dtype=dt)
    ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=rho, eps_abs=1e-4,
                             eps_rel=1e-4, warm_start=True)
    traj, us, its = ctl.closed_loop_batch(wl.x0, wl.xr, wl.speed, steps=steps)
    traj = traj.cpu().numpy(); us = us.cpu().numpy(); its = its.cpu().numpy()
    which = range(B)
    if sample is not None and sample < B:
        slow = np.unique(its.argmax(axis=1))[: sample // 2]
        which = sorted(set(int(b) for b in slow) | set(int(b) for b in np.linspace(0, B - 1, sample - len(slow)).astype(int)))
    for b in which:
        Ad, Bd = workload_qp.lateral_model(float(wl.speed[b]))
        At, Bt, _ = ref_qp.augment_increment(Ad, Bd, None)
        qp = workload_qp.lateral_qp(wl, b)
        P, q, A, l, u = ref_qp.assemble(qp)
        o = osqp_admm.OSQP().setup(P, q, A, l, u, rho=rho, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
        x = wl.x0[b].copy()
        for k in range(steps):
            if k > 0:
                l[:5] = -x; u[:5] = -x
                o.update(l=l, u=u)
            r = o.solve()
            assert r.info.iter == its[k, b], (b, k, r.info.iter, its[k, b])
            du = r.x[105:106]
            assert abs(du[0] - us[k, b, 0]) < 1e-6 * max(1.0, abs(du[0]))
            x = At @ x + Bt @ du
            assert np.abs(x - traj[k + 1, b]).max() < 1e-3 and abs(x[3] - traj[k + 1, b, 3]) < 1e-6
    return its, us


def check_dynamic_long_horizon(be, B=2, N=30, rho=0.1, samples=(0,), eps=1e-4):
    """configs[3]: time-varying (per-stage) linearisation of the combined longitudinal-lateral dynamics model,
    long horizon, f64.  GPU/emu rollout + solve vs the oracle on the same per-stage matrices."""
    wl = workloads.DynamicWorkload(B, N=N, seed=1)
    veh = vehicle_models.Vehicle_Dynamics(dt=wl.dt, _backend=be)
    A, Bm, g, _, ld = workloads.rollout_linearisation(veh, wl.x0, wl.u0, N)
    Xr = wl.references()
    s = pm.BatchSolver(N, 6, 2, wl.Q, wl.QN, wl.R, wl.xmin, wl.xmax, wl.umin, wl.umax, dtype=torch.float64,
                       time_varying=True, stage_reference=True, capacity=B, _backend=be, rho=rho, eps_abs=eps, eps_rel=eps,
                       warm_start=False)
    assert s.ld == ld
    xr = torch.as_tensor(Xr).transpose(1, 2).contiguous()
    s.batch = B
    s.setup(A, Bm, g, s.to_element_major(wl.x0, B, 6, ld), s.to_element_major(xr, B, (N + 1) * 6, ld), element_major=True)
    s.solve()
    inf = s.info()
    st = inf.status_val.cpu().numpy(); it = inf.iter.cpu().numpy()
    assert (st == 1).all(), np.unique(st, return_counts=True)
    x, _, _ = s.solution()
    Ab = s._bm(A, B, N * 36).reshape(B, N, 6, 6).cpu().numpy()
    Bb = s._bm(Bm, B, N * 12).reshape(B, N, 6, 2).cpu().numpy()
    gb = s._bm(g, B, N * 6).reshape(B, N, 6).cpu().numpy()
    for b in samples:
        # the per-stage matrices themselves equal the reference's get_dynamics_model along the same rollout
        xk = wl.x0[b].copy()
        import oracle.vehicle_ref as vr
        for k in (0, 1, N - 1):
            if k <= 1:
                a_ref, b_ref, g_ref = vr.dynamics_model(xk, wl.u0[b], dt=wl.dt)
                assert np.abs(a_ref - Ab[b, k]).max() < 1e-11 and np.abs(g_ref - gb[b, k]).max() < 1e-10
                xk = a_ref @ xk + b_ref @ wl.u0[b] + g_ref
        qp = ref_qp.canonical(N, Ab[b], Bb[b], gb[b], wl.Q, wl.QN, wl.R, Xr[b], wl.xmin, wl.xmax, wl.umin, wl.umax, wl.x0[b])
        r = oracle_solve(qp, rho=rho, eps_abs=eps, eps_rel=eps)
        assert r.info.iter == it[b] and r.info.status_val == 1
        assert rel(x[b].cpu().numpy(), r.x) < 1e-6
    return it


def check_retiling_is_bitwise_neutral(be, B=96):
    """The chunked ADMM loop with re-tiling of unconverged QPs must give bit-identical results to the single launch
    (rows stay in p-form across chunk boundaries; a QP's arithmetic does not depend on the tile it sits in); the
    stragglers, which finish in the scratch workspace, agree with the oracle."""
    wl = workloads.lateral_slack_increment(B, seed=77, dtype=torch.float64)
    out = []
    for retile in (0, 1):
        be.set_option("retile", retile); be.set_option("retile_min_batch", 2)
        be.set_option("cta", 0)         # (a batch this small would go to the CTA-per-tile kernel: this test is about the main loop)
        try:
            ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=5.0, eps_abs=1e-4,
                                     eps_rel=1e-4, warm_start=True)
            n0 = be.launch_count()
            r1 = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
            n1 = be.launch_count() - n0
            x1, y1, _ = ctl.solver.solution(want_y=True)
            r2 = ctl.update_batch(wl.x0 * 0.9)                 # warm-started second solve reads the (z, y) left behind
            out.append((x1.clone(), y1.clone(), r1.info.iter.clone(), r2.x.clone(), r2.info.iter.clone(), n1))
        finally:
            be.set_option("retile", 1); be.set_option("retile_min_batch", 4096); be.set_option("cta", 1)
    a, b_ = out
    it = a[2].cpu().numpy()
    assert len(np.unique(it)) > 1 and (it == it.max()).mean() <= 0.5, "workload does not exercise re-tiling: %s" % np.unique(it, return_counts=True)
    # the chunked run launched at least: one more ADMM chunk, the re-tiling copy, the un-tiling copy
    assert b_[5] >= a[5] + 3, "the chunked loop did not re-tile (%d vs %d launches)" % (b_[5], a[5])
    for u, v in zip(a[:5], b_[:5]):
        assert torch.equal(u, v)
    for b in np.flatnonzero(it == it.max())[:3]:
        r = oracle_solve(workload_qp.lateral_qp(wl, int(b)), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert r.info.iter == it[b] and rel(b_[0][b].cpu().numpy(), r.x) < 1e-6


def check_dense_shared_kkt(be, B=1024):
    """The shared-KKT dense path (admm_dense.cuh: explicit inverse of the reduced KKT matrix, DMMA GEMM over all right-hand
    sides) against the per-QP kernels and the oracle: one shared linearisation, (a) vanilla = BASELINE configs[1],
    (b) slack + delta-u; warm-started second solve after update(); a batch whose references differ (scalings differ per
    QP -> the dense path must decline and the per-QP kernels run)."""
    out = []
    for slack, inc in ((False, False), (True, True)):
        wl = workloads.LateralWorkload(B, 20, slack, inc, 321, torch.float64, shared_speed=8.3128334)
        res = []
        for dense in (0, 1):
            be.set_option("dense", dense)
            try:
                ctl = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
                n0 = be.launch_count()
                r1 = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
                x1, y1, _ = ctl.solver.solution(want_y=True)
                r2 = ctl.update_batch(wl.x0 * 0.9)
                res.append((r1.x.clone(), y1.clone(), r1.info.iter.clone(), r1.info.status_val.clone(), r2.x.clone(),
                            r2.info.iter.clone(), be.launch_count() - n0))
            finally:
                be.set_option("dense", 1)
        a, d = res
        assert torch.equal(a[2], d[2]) and torch.equal(a[3], d[3]) and torch.equal(a[5], d[5])
        sx, sy = float(a[0].abs().max()), float(a[1].abs().max())
        assert float((a[0] - d[0]).abs().max()) < 1e-9 * sx and float((a[4] - d[4]).abs().max()) < 1e-9 * sx
        assert float((a[1] - d[1]).abs().max()) < 1e-8 * sy
        it = d[2].cpu().numpy()
        for b in list(range(0, B, max(1, B // 6)))[:6]:
            r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
            assert r.info.iter == it[b] and r.info.status_val == 1
            assert rel(d[0][b].cpu().numpy(), r.x) < 1e-6
        out.append((np.unique(it, return_counts=True), a[6], d[6]))
    # references that differ per QP change the cost scaling c (and with it D, E): no shared KKT matrix
    wl = workloads.LateralWorkload(64, 20, False, False, 77, torch.float64, shared_speed=8.3128334)
    wl.xr = np.random.default_rng(5).uniform(-3.0, 3.0, (64, 4))
    ctl = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
    r1 = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    for b in (0, 31, 63):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert r.info.iter == int(r1.info.iter[b]) and rel(r1.x[b].cpu().numpy(), r.x) < 1e-6
    return out


def check_cta_kernel_agrees(be, B=2048):
    """The CTA-per-tile kernel (admm_cta.cuh: a warp per component, records staged by TMA, the whole loop in one launch)
    against the warp-per-tile kernel on time-invariant problems (option "cta" = 2 forces it): statuses and iteration counts
    equal, solutions to the last bits, warm-started second solve, primal infeasibility; and against the oracle."""
    out = []
    for slack, inc in ((True, True), (False, False)):
        wl = workloads.LateralWorkload(B, 20, slack, inc, 99, torch.float64)
        wl.x0[5, 3] = 14.0 if not slack else wl.x0[5, 3]        # hard-constraint formulation: one infeasible QP in the batch
        res = []
        for cta in (0, 2):
            be.set_option("cta", cta)
            try:
                ctl = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
                r1 = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
                x1, y1, _ = ctl.solver.solution(want_y=True)
                r2 = ctl.update_batch(wl.x0 * 0.9)
                res.append((r1.x.clone(), y1.clone(), r1.info.iter.clone(), r1.info.status_val.clone(), r2.x.clone(),
                            r2.info.iter.clone(), r2.info.status_val.clone()))
            finally:
                be.set_option("cta", 1)
        a, d = res
        assert torch.equal(a[2], d[2]) and torch.equal(a[3], d[3]), (a[2] != d[2]).sum()
        assert torch.equal(a[5], d[5]) and torch.equal(a[6], d[6])
        ok = a[3] == 1
        sx, sy = float(a[0][ok].abs().max()), float(a[1][ok].abs().max())
        assert float((a[0][ok] - d[0][ok]).abs().max()) < 1e-10 * sx and float((a[1][ok] - d[1][ok]).abs().max()) < 1e-9 * sy
        ok2 = a[6] == 1
        assert float((a[4][ok2] - d[4][ok2]).abs().max()) < 1e-10 * sx
        if not slack:
            assert int(d[3][5]) == -3 and bool(torch.isnan(d[0][5]).all())
        it = d[2].cpu().numpy()
        for b in (0, 5, B - 1):
            r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
            assert r.info.iter == it[b] and r.info.status_val == int(d[3][b])
            if r.info.status_val == 1:
                assert rel(d[0][b].cpu().numpy(), r.x) < 1e-6
        out.append(np.unique(it, return_counts=True))
    return out


def check_cta_retiling_is_bitwise_neutral(be, B=4608, N=40):
    """Time-varying batch through the CTA-per-tile kernel: one launch (retile off) vs the chunked loop that compacts the
    unsolved QPs — records, headers AND staged stage models — every time half of the set has terminated.  A QP's arithmetic
    does not depend on the tile it sits in: bit-identical results, iteration counts and duals."""
    wl = workloads.DynamicWorkload(B, N=N, seed=4)
    veh = vehicle_models.Vehicle_Dynamics(dt=wl.dt, _backend=be)
    A, Bm, g, _, ld = workloads.rollout_linearisation(veh, wl.x0, wl.u0, N)
    Xr = wl.references()
    xr = torch.as_tensor(Xr).transpose(1, 2).contiguous()
    out = []
    for retile in (0, 1):
        be.set_option("retile", retile)
        try:
            s = pm.BatchSolver(N, 6, 2, wl.Q, wl.QN, wl.R, wl.xmin, wl.xmax, wl.umin, wl.umax, dtype=torch.float64,
                               time_varying=True, stage_reference=True, capacity=B, _backend=be, rho=0.1, eps_abs=1e-4,
                               eps_rel=1e-4, warm_start=False)
            s.batch = B
            n0 = be.launch_count()
            s.setup(A, Bm, g, s.to_element_major(wl.x0, B, 6, ld), s.to_element_major(xr, B, (N + 1) * 6, ld), element_major=True)
            s.solve()
            x, y, _ = s.solution(want_y=True)
            inf = s.info()
            out.append((x.clone(), y.clone(), inf.iter.clone(), inf.status_val.clone(), be.launch_count() - n0))
        finally:
            be.set_option("retile", 1)
    a, b_ = out
    it = a[2].cpu().numpy()
    assert len(np.unique(it)) > 2 and b_[4] > a[4] + 2, (np.unique(it, return_counts=True), a[4], b_[4])
    for u, v in zip(a[:4], b_[:4]):
        assert torch.equal(u, v)
    return np.unique(it, return_counts=True)


def check_fp32_batch(be, B=4096, rho=0.1, eps=1e-3):
    """FP32 mode at batch scale (north_star: primal within 1e-4 in FP32).  Same QPs in f32 and f64 at rho = 0.1 — the
    largest rho at which f32 round-off (multiplied by rho_eq = 1e3 rho into the duals) stays below OSQP's termination
    tolerance, DESIGN.md section 6:
      * every QP reports 'solved' in both precisions, and the f64 run matches the oracle (status, iterations, primal);
      * after the SAME number of iterations (no termination test) the f32 iterate is within 1e-4 of the f64 one for EVERY QP;
      * with the termination test on, a QP that stops at the same iteration in both precisions (> 98 % of them) is within
        1e-4; the rest stop one check later or earlier (a residual within f32 round-off of the tolerance) and stay within
        the termination tolerance itself."""
    res = {}
    for dt in (torch.float32, torch.float64):
        wl = workloads.lateral_slack_increment(B, seed=31, dtype=dt)
        ctl = wl.make_controller(capacity=B, rho=rho, eps_abs=eps, eps_rel=eps, warm_start=False)
        r = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
        s = ctl.solver
        s.cold_start(); s.iterate(200)
        xi, _, _ = s.solution()
        res[dt] = (r.x.double().clone(), r.info.iter.clone(), r.info.status_val.clone(), xi.double().clone(), wl)
    x32, it32, st32, xi32, _ = res[torch.float32]
    x64, it64, st64, xi64, wl = res[torch.float64]
    assert bool((st32 == 1).all()) and bool((st64 == 1).all())
    scale = xi64.abs().amax(dim=1)
    dev_fixed = ((xi32 - xi64).abs().amax(dim=1) / scale).max().item()
    assert dev_fixed < 1e-4, dev_fixed
    same = it32 == it64
    frac_same = same.double().mean().item()
    assert frac_same > 0.98, frac_same
    dev = (x32 - x64).abs().amax(dim=1) / x64.abs().amax(dim=1)
    assert dev[same].max().item() < 1e-4, dev[same].max().item()
    assert dev.max().item() < 10 * eps, dev.max().item()
    for b in (0, B // 2, B - 1):
        r = oracle_solve(workload_qp.lateral_qp(wl, b), rho=rho, eps_abs=eps, eps_rel=eps)
        assert r.info.iter == int(it64[b]) and rel(x64[b].cpu().numpy(), r.x) < 1e-6
    return dev_fixed, frac_same, dev.max().item()
