"""The oracle pinned against everything available for this path (the reference has no tests of its own):
the reference's own QP assembly executed from /root/reference (tests/golden), OSQP's documented demo QP,
KKT optimality checked independently of ADMM, and the C port against the numpy restatement."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import c_oracle, osqp_admm, ref_qp, workload_qp

DEG = np.pi / 180


def kkt_violation(P, q, A, l, u, x, y):
    """Independent optimality check: stationarity, primal feasibility, sign/complementarity of the multipliers."""
    P = sp.csc_matrix(P); A = sp.csc_matrix(A)
    Ax = A @ x
    stat = np.abs(P @ x + q + A.T @ y).max()
    feas = max(np.maximum(l - Ax, 0).max(), np.maximum(Ax - u, 0).max())
    comp = max(np.abs(np.minimum(y, 0) * (Ax - l)).max(), np.abs(np.maximum(y, 0) * (u - Ax)).max())
    return stat, feas, comp


def test_osqp_documented_demo_qp():
    # "Setup and solve" example of the OSQP documentation: optimal x = [0.3, 0.7], objective 1.88
    P = sp.csc_matrix([[4, 1], [1, 2]]); q = np.array([1., 1.]); A = sp.csc_matrix([[1, 1], [1, 0], [0, 1]])
    l = np.array([1., 0., 0.]); u = np.array([1., 0.7, 0.7])
    r = osqp_admm.OSQP().setup(P, q, A, l, u, eps_abs=1e-9, eps_rel=1e-9).solve()
    assert r.info.status == "solved"
    np.testing.assert_allclose(r.x, [0.3, 0.7], atol=1e-7)
    assert abs(r.info.obj_val - 1.88) < 1e-7
    x, y, it, st, _, _ = c_oracle.solve(P, q, A, l, u, eps_abs=1e-9, eps_rel=1e-9)
    assert st == 1 and it == r.info.iter
    np.testing.assert_allclose(x, r.x, atol=1e-12)


@pytest.mark.parametrize("shared_dir", ["absent", "world_writable", "foreign_owner"])
def test_stale_oracle_in_a_read_only_tree_is_rebuilt_outside_it(tmp_path, monkeypatch, shared_dir):
    """bench.py may run from a tree it cannot write: a missing or stale library is then built in a per-user temporary
    directory, reused while current — and never loaded from that directory when another user could have written it."""
    import ctypes
    import os
    import tempfile
    from oracle import library
    monkeypatch.setattr(library, "SO", str(tmp_path / "tree" / "liboracle_osqp.so"))
    monkeypatch.setattr(library, "_writable", lambda d: False)
    (tmp_path / "tmp").mkdir()
    monkeypatch.setattr(tempfile, "tempdir", str(tmp_path / "tmp"))
    uid = os.getuid()
    if shared_dir == "foreign_owner":
        monkeypatch.setattr(os, "getuid", lambda: uid + 1)              # the directory below belongs to "another" user
    planted = tmp_path / "tmp" / ("mpcb_oracle_%d_%s" % (os.getuid(), library._stamp()[:16]))
    if shared_dir != "absent":
        planted.mkdir(mode=0o700)
        (planted / "liboracle_osqp.so").write_bytes(b"planted")
        (planted / "liboracle_osqp.sha256").write_text(library._stamp())
        if shared_dir == "world_writable":
            planted.chmod(0o777)
    so = library.build()
    assert so.startswith(str(tmp_path / "tmp")) and not (tmp_path / "tree").exists()
    assert hasattr(ctypes.CDLL(so), "oracle_osqp_solve")
    if shared_dir == "absent":
        assert os.path.dirname(so) == str(planted) and planted.stat().st_mode & 0o777 == 0o700
        mtime = os.path.getmtime(so)
        assert library.build() == so and os.path.getmtime(so) == mtime      # up to date: found again, not rebuilt
    else:
        assert os.path.dirname(so) != str(planted) and (planted / "liboracle_osqp.so").read_bytes() == b"planted"


def test_restated_assembly_equals_reference_slack_increment(golden):
    g = golden["lateral_slack_increment_closed_loop"]
    p = ref_qp.qp_slack_increment(g["Ad"], g["Bd"], np.array([0., 0., 5 * DEG, 3., 0.]), np.zeros(4),
                                  [5., 5., 10., 10.], [10.], [10., 10., 10., 10., 0.], [1., 1., 1., 1., 0.], int(g["N"]),
                                  np.array([-np.pi, -0.5 * np.pi, -15 * DEG, -10., -30 * DEG]),
                                  np.array([np.pi, 0.5 * np.pi, 15 * DEG, 10., 30 * DEG]), [-0.5 * DEG], [0.5 * DEG])
    P, q, A, l, u = ref_qp.assemble(p)
    assert np.array_equal(P.toarray(), g["P"]) and np.array_equal(A.toarray(), g["A"])
    assert np.array_equal(q, g["q"]) and np.array_equal(l, g["l"]) and np.array_equal(u, g["u"])


@pytest.mark.parametrize("name", ["qp_vanilla_kinematic", "qp_vanilla_dynamic", "qp_increment_dynamic"])
def test_restated_assembly_equals_reference(golden, name):
    g = golden[name]
    N = int(g["N"])
    if name == "qp_vanilla_kinematic":
        p = ref_qp.qp_vanilla(g["Ad"], g["Bd"], g["gd"], g["x_init"], g["Xr"], g["Q"], g["QN"], g["R"], N,
                              g["xmin"], g["xmax"], g["umin"], g["umax"])
    elif name == "qp_vanilla_dynamic":
        p = ref_qp.qp_vanilla(list(g["Ad"]), list(g["Bd"]), list(g["gd"]), g["x_init"], g["Xr"], g["Q"], g["QN"], g["R"],
                              N, g["xmin"], g["xmax"], g["umin"], g["umax"])
    else:
        p = ref_qp.qp_increment(list(g["Ad"]), list(g["Bd"]), list(g["gd"]), g["x_init"], g["Xr"], g["Q"], g["QN"],
                                g["R"], N, g["xmin"], g["xmax"], g["umin"], g["umax"])
    P, q, A, l, u = ref_qp.assemble(p)
    assert np.array_equal(P.toarray(), g["P"]) and np.array_equal(A.toarray(), g["A"])
    np.testing.assert_array_equal(q, g["q"])
    np.testing.assert_array_equal(l, g["l"]); np.testing.assert_array_equal(u, g["u"])


def test_numpy_and_c_oracle_agree_and_reproduce_golden_solution(golden):
    g = golden["qp_increment_dynamic"]
    s = dict(eps_abs=1e-4, eps_rel=1e-4)
    r = osqp_admm.OSQP().setup(g["P"], g["q"], g["A"], g["l"], g["u"], **s).solve()
    assert r.info.iter == int(g["sol_iter"]) and r.info.status_val == int(g["sol_status"])
    np.testing.assert_allclose(r.x, g["sol_x"], rtol=0, atol=1e-10)
    x, y, it, st, _, _ = c_oracle.solve(g["P"], g["q"], g["A"], g["l"], g["u"], **s)
    assert it == r.info.iter and st == r.info.status_val
    np.testing.assert_allclose(x, r.x, rtol=0, atol=1e-9 * np.abs(r.x).max())


def test_converged_point_satisfies_kkt(golden):
    g = golden["lateral_slack_increment_closed_loop"]
    P, q, A, l, u = [g[k] for k in "PqAlu"]
    r = osqp_admm.OSQP().setup(P, q, A, l, u, rho=5.0, eps_abs=1e-10, eps_rel=1e-10, max_iter=20000).solve()
    assert r.info.status == "solved"
    stat, feas, comp = kkt_violation(P, q, A, l, u, r.x, r.y)
    assert stat < 1e-7 and feas < 1e-8 and comp < 1e-7
    # a different rho converges to the same optimum (the QP solution does not depend on ADMM parameters)
    r2 = osqp_admm.OSQP().setup(P, q, A, l, u, rho=0.7, eps_abs=1e-10, eps_rel=1e-10, max_iter=100000).solve()
    np.testing.assert_allclose(r2.x, r.x, atol=2e-6)


def test_update_and_warm_start_follow_osqp_semantics(golden):
    g = golden["lateral_slack_increment_closed_loop"]
    P, q, A, l, u = [g[k] for k in "PqAlu"]
    o = osqp_admm.OSQP().setup(P, q, A, l, u, rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
    cold = o.solve().info.iter
    o.update(l=g["l_updates"][1], u=g["l_updates"][1] * 0 + np.where(np.arange(u.size) < 5, g["l_updates"][1], u))
    warm = o.solve().info.iter
    assert warm <= cold
    with pytest.raises(ValueError):
        o.update(l=u + 1.0, u=u)


def test_closed_loop_fixture_is_consistent(golden):
    """The reference script's closed loop (run through the oracle when the fixture was made) regulates the
    lateral error and respects the rate bound — sanity of the captured trajectory itself."""
    g = golden["lateral_slack_increment_closed_loop"]
    assert np.abs(g["x4"]).max() < 10.0 and g["x4"].min() < 0 < g["x4"].max()      # crosses the reference, stays in the box
    assert np.all(np.abs(g["del_u"]) <= 0.5 * DEG + 1.2e-3)                        # rate bound up to eps_prim
    assert g["iters"].min() >= 25 and g["iters"].max() <= 4000


def test_lateral_model_matches_reference_literals(golden):
    """oracle lateral bicycle (ZOH) at the nominal speed reproduces Ad_sys/Bd_sys hard-coded in
    vehicle_lateral_mpc_slack_increment.py:32-43 to their printed precision."""
    g = golden["lateral_slack_increment_closed_loop"]
    Ad, Bd = workload_qp.lateral_model(8.3128334)
    assert np.abs(Ad - g["Ad"]).max() < 2.5e-3
    assert np.abs(Bd - g["Bd"]).max() < 1e-4


def test_dynamics_model_restatement_equals_reference(golden):
    """oracle/vehicle_ref.py vs the outputs of the reference's own get_dynamics_model (run when the fixture was
    made), including the low-speed guard branches."""
    from oracle import vehicle_ref
    g = golden["vehicle_models"]
    for i in range(g["dyn_x"].shape[0]):
        A, B, gd = vehicle_ref.dynamics_model(g["dyn_x"][i], g["dyn_u"][i], dt=float(g["dyn_dt"]))
        np.testing.assert_allclose(A, g["dyn_Ad"][i], rtol=0, atol=1e-12)
        np.testing.assert_allclose(B, g["dyn_Bd"][i], rtol=0, atol=1e-12)
        np.testing.assert_allclose(gd, g["dyn_gd"][i], rtol=0, atol=1e-11)


def test_plant_step_and_kinematics_restatements_equal_reference(golden):
    """oracle/vehicle_ref.py's dynamics_step, kinematics_model and kinematics_step vs the outputs of the reference's own
    update_dynamics_model (low-speed guards included), get_kinematics_model and update_kinematics_model."""
    from oracle import vehicle_ref
    g = golden["vehicle_models"]
    for i in range(g["dyn_x"].shape[0]):
        xn, af, ar = vehicle_ref.dynamics_step(g["dyn_x"][i], g["dyn_u"][i], dt=float(g["dyn_dt"]))
        np.testing.assert_allclose(xn, g["dyn_xnext"][i], rtol=0, atol=1e-12)
        assert np.isfinite(af) and np.isfinite(ar)
    for i in range(g["kin_x"].shape[0]):
        A, B, C = vehicle_ref.kinematics_model(g["kin_x"][i], g["kin_u"][i], dt=float(g["kin_dt"]))
        np.testing.assert_allclose(A, g["kin_A"][i], rtol=0, atol=1e-15)
        np.testing.assert_allclose(B, g["kin_B"][i], rtol=0, atol=1e-15)
        np.testing.assert_allclose(C, g["kin_C"][i], rtol=0, atol=1e-15)
        xn = vehicle_ref.kinematics_step(g["kin_x"][i], g["kin_u"][i], dt=float(g["kin_dt"]))
        np.testing.assert_allclose(xn, g["kin_xnext"][i], rtol=0, atol=1e-14)
    # the yaw update sees the new speed: with the old one the fixture is missed wherever steer and acceleration are nonzero
    x, u = g["kin_x"], g["kin_u"]
    old = x[:, 3] + x[:, 2] / (1.25 + 1.40) * np.tan(u[:, 0]) * float(g["kin_dt"])
    assert np.abs(old - g["kin_xnext"][:, 3]).max() > 1e-6


def test_c_closed_loop_driver_reproduces_reference_script_fixture(golden):
    """oracle_closed_loop_batch (the CPU arm of bench.py's configs[4] record): setup once, update(l, u) + warm-started
    solve + plant step per scenario — against the closed-loop fixture of the reference script (H = 20 head) and, with a
    bound schedule, against the numpy oracle's update()."""
    g = golden["lateral_slack_increment_closed_loop"]
    N = int(g["N"]); steps = 40
    At, Bt, _ = ref_qp.augment_increment(g["Ad"], g["Bd"], None)
    P = sp.csc_matrix(g["P"]); A = sp.csc_matrix(g["A"])
    Pu = sp.triu(P, format="csc"); Pu.sort_indices(); Ac = A.copy(); Ac.sort_indices()
    x0 = np.array([[0., 0., 5 * DEG, 3., 0.]])
    it, st, ua, traj, _ = c_oracle.closed_loop_batch(P, A, Pu.data[None], g["q"][None], Ac.data[None], g["l"][None], g["u"][None],
                                                     At[None], Bt[None], x0, steps, (N + 1) * 5, eps_abs=1e-4, eps_rel=1e-4)
    assert (st == 1).all() and it[0].tolist() == g["iters"][:steps].tolist()
    assert np.abs(traj[0, :steps, 3] - g["x4"][:steps]).max() < 1e-9 and np.abs(ua[0, :, 0] - g["del_u"][:steps]).max() < 1e-10
    # bound switch at step 5 / back at step 12 (rho = 5): the numpy oracle step by step
    l2 = g["l"].copy(); l2[(N + 1) * 5 + 3:(N + 1) * 10:5] = 2.0
    sched = {5: (l2, g["u"]), 12: (g["l"], g["u"])}
    it, st, ua, traj, _ = c_oracle.closed_loop_batch(P, A, Pu.data[None], g["q"][None], Ac.data[None], g["l"][None], g["u"][None],
                                                     At[None], Bt[None], x0, 20, (N + 1) * 5, schedule=sched, rho=5.0,
                                                     eps_abs=1e-4, eps_rel=1e-4)
    o = osqp_admm.OSQP().setup(P, g["q"], A, g["l"], g["u"], rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=True)
    x = x0[0].copy(); l = g["l"].copy(); u = g["u"].copy()
    for k in range(20):
        if k in sched:
            l[5:] = sched[k][0][5:]
        l[:5] = -x; u[:5] = -x
        if k > 0 or k in sched:
            o.update(l=l, u=u)
        r = o.solve()
        assert r.info.iter == it[0, k] and r.info.status_val == st[0, k]
        x = At @ x + Bt @ r.x[(N + 1) * 5:(N + 1) * 5 + 1]
        assert np.abs(x - traj[0, k + 1]).max() < 1e-9
    assert np.abs(ua[0, 5:12]).max() > 0


def test_batch_csc_builders_equal_the_per_qp_assembly():
    """The vectorised CSC batches the CPU arm of bench.py feeds to oracle_solve_batch hold exactly the per-QP assembly."""
    import torch
    from python_mpc_b200 import workloads
    wl = workloads.lateral_slack_increment(5, seed=3, dtype=torch.float64)
    Pu, A0, Pv, q, Av, l, u, perm = workload_qp.lateral_batch_csc(wl)
    for b in range(5):
        P, qq, A, ll, uu = ref_qp.assemble(workload_qp.lateral_qp(wl, b))
        A = sp.csc_matrix(A); A.sort_indices()
        assert np.array_equal(A.indices, A0.indices) and np.array_equal(Av[b], A.data)
        assert np.array_equal(q[b], qq) and np.array_equal(l[b], ll) and np.array_equal(u[b], uu)
    rng = np.random.default_rng(0)
    dw = workloads.DynamicWorkload(4, N=7, seed=2)
    A = np.eye(6) + 0.1 * rng.standard_normal((4, 7, 6, 6)); Bm = rng.standard_normal((4, 7, 6, 2)); g = rng.standard_normal((4, 7, 6))
    Xr = dw.references()
    Pu, A0, Pv, q, Av, l, u, perm = workload_qp.dynamic_batch_csc(dw, A, Bm, g, Xr, np.array([3, 1]))
    for r, b in enumerate((3, 1)):
        P, qq, Aq, ll, uu = ref_qp.assemble(ref_qp.canonical(7, A[b], Bm[b], g[b], dw.Q, dw.QN, dw.R, Xr[b], dw.xmin, dw.xmax,
                                                             dw.umin, dw.umax, dw.x0[b]))
        Aq = sp.csc_matrix(Aq); Aq.sort_indices()
        assert np.array_equal(Aq.indices, A0.indices) and np.array_equal(Av[r], Aq.data)
        assert np.array_equal(q[r], qq) and np.array_equal(l[r], np.maximum(ll, -np.inf)) and np.array_equal(u[r], uu)
