"""GPU suite (-m gpu): the parity tests proper — libmpc_b200.so through the C ABI on a B200, against the oracle on
the same seeded inputs, the golden fixtures, and size-independent properties at BASELINE.json's full sizes."""
import numpy as np
import pytest
import torch

import parity_cases as pc

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("slack,increment", [(True, True), (False, False), (True, False), (False, True)])
def test_lateral_formulations_fp64(cuda_backend, slack, increment):
    pc.check_lateral_batch(cuda_backend, slack, increment, torch.float64, B=48)


def test_lateral_shared_linearisation_fp64(cuda_backend):
    pc.check_lateral_batch(cuda_backend, False, False, torch.float64, B=40, shared=True)


def test_lateral_fp32_within_1e4(cuda_backend):
    pc.check_lateral_batch(cuda_backend, True, True, torch.float32, B=8, rho=0.1, max_iter=400, eps=1e-3)


def test_fp32_batch_4096_within_1e4(cuda_backend):
    pc.check_fp32_batch(cuda_backend, B=4096)


def test_iterates_match_oracle(cuda_backend):
    pc.check_iterates(cuda_backend, torch.float64, iters=60, rho=5.0, B=8)
    pc.check_iterates(cuda_backend, torch.float32, iters=60, rho=0.1, B=8)


def test_build_qp_equals_reference_assembly(cuda_backend, golden):
    pc.check_build_qp_against_reference_capture(cuda_backend, golden)


def test_vehicle_models_equal_reference(cuda_backend, golden):
    pc.check_models_against_reference(cuda_backend, golden)


def test_reference_signature_functions(cuda_backend, golden):
    pc.check_reference_functions(cuda_backend, golden)


def test_kinematic_corridor_and_predmatrix_functions(cuda_backend, golden):
    pc.check_kinematic_corridor_and_predmatrix(cuda_backend, golden)


def test_closed_loop_trajectory(cuda_backend, golden):
    pc.check_closed_loop(cuda_backend, golden)


def test_closed_loop_full_reference_script_with_bound_switches(cuda_backend, golden):
    """the unmodified reference script: N = 100, all 1500 steps, bound switches at 401 and 901, slack active in between"""
    slack = pc.check_closed_loop_full(cuda_backend, golden)
    assert np.abs(slack[401:901]).max() > 1.9 and np.abs(slack[1000:]).max() < 1e-3


def test_closed_loop_sweep_warm_started(cuda_backend):
    pc.check_closed_loop_sweep(cuda_backend, B=40, steps=8)


def test_closed_loop_large_batch_schedules_agree(cuda_backend):
    """20000 scenarios x 5 warm-started steps — beyond one wave of CTAs: the warp-per-tile kernel with repeated compaction, the
    stragglers finished by the CTA-per-tile kernel, learnt / probed compaction points from step to step.  Stragglers and a
    spread of scenarios against the oracle; every scenario against the schedule without the CTA kernel ("cta", 0)."""
    from python_mpc_b200 import workloads
    its, us = pc.check_closed_loop_sweep(cuda_backend, B=20000, steps=5, sample=8)
    cuda_backend.set_option("cta", 0)
    try:
        its0, us0 = pc.check_closed_loop_sweep(cuda_backend, B=20000, steps=5, sample=2)
    finally:
        cuda_backend.set_option("cta", 1)
    assert np.array_equal(its, its0) and len(np.unique(its)) >= 3
    assert np.abs(us - us0).max() < 1e-9 * max(1.0, np.abs(us0).max())
    # the configs[4] sweep workload (a third to a half of the scenarios terminate at the first test -> compaction at 25) with
    # every 40th scenario started far from its reference (stragglers beyond the second test -> a second compaction, from the
    # scratch workspace, into the CTA-per-tile kernel)
    def mixed():
        wl = workloads.lateral_closed_loop_sweep(20000, seed=77)
        wl.x0[::40] *= 12.0
        return wl
    its, us = pc.check_closed_loop_sweep(cuda_backend, B=20000, steps=6, sample=8, wl=mixed())
    cuda_backend.set_option("cta", 0)
    try:
        its0, us0 = pc.check_closed_loop_sweep(cuda_backend, B=20000, steps=6, sample=2, wl=mixed())
    finally:
        cuda_backend.set_option("cta", 1)
    assert np.array_equal(its, its0) and len(np.unique(its)) >= 3
    assert np.abs(us - us0).max() < 1e-9 * max(1.0, np.abs(us0).max())


def test_config3_long_horizon_dynamic_8192_f64(cuda_backend):
    """BASELINE configs[3] at full size: batch 8192, H = 100, combined longitudinal-lateral dynamics model, FP64."""
    it = pc.check_dynamic_long_horizon(cuda_backend, B=8192, N=100, samples=(0, 4097))
    assert it.max() <= 4000 and (it % 25 == 0).all()


def test_config1_vanilla_shared_1024_f64(cuda_backend):
    """BASELINE configs[1] at full size: batch 1024 vanilla lateral MPC, one shared linearisation, FP64."""
    pc.check_lateral_batch(cuda_backend, False, False, torch.float64, B=1024, shared=True, samples=range(0, 1024, 128))


def test_retiling_is_bitwise_neutral(cuda_backend):
    pc.check_retiling_is_bitwise_neutral(cuda_backend, B=4096)


def test_wide_straggler_kernel_agrees(cuda_backend):
    pc.check_wide_kernel_agrees(cuda_backend, B=4096)


def test_dense_shared_kkt_path(cuda_backend):
    """configs[1] (batch 1024 vanilla, one linearisation): DMMA GEMM with the explicit reduced-KKT inverse vs the per-QP kernels"""
    pc.check_dense_shared_kkt(cuda_backend, B=1024)


def test_cta_per_tile_kernel_agrees(cuda_backend):
    pc.check_cta_kernel_agrees(cuda_backend, B=2048)


def test_cta_three_buffer_instantiation_on_small_batches(cuda_backend, monkeypatch):
    """Launches of at most one tile per SM use the 5-buffer / one-CTA-per-SM instantiation of the CTA kernel; the 3-buffer one
    (full batches) on the same small problems, incl. the edge horizons"""
    monkeypatch.setenv("MPCB_NO_CTA_DEEP", "1")
    pc.check_cta_kernel_agrees(cuda_backend)
    worst, seen = pc.check_random_problems(cuda_backend, seeds=(2, 3, 4, 5, 6, 7), B=37, horizons=(1, 2, 3, 4, 5, 33))
    assert worst < 1e-9


def test_cta_retiling_is_bitwise_neutral(cuda_backend):
    pc.check_cta_retiling_is_bitwise_neutral(cuda_backend)


def test_tma_and_plain_kernels_agree_bitwise(cuda_backend):
    """The TMA-staged warp-per-tile kernel and the lane-per-QP kernel run the same stage functions."""
    from python_mpc_b200 import workloads, vehicle_models
    wl = workloads.lateral_slack_increment(300, seed=8, dtype=torch.float64)
    res = []
    for tma in (1, 0):
        cuda_backend.set_option("tma", tma); cuda_backend.set_option("cta", 0)
        try:
            r = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False).solve_batch(wl.x0, wl.xr, wl.speed)
            res.append((r.x.clone(), r.info.iter.clone()))
        finally:
            cuda_backend.set_option("tma", 1); cuda_backend.set_option("cta", 1)
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])


def test_bound_updates_keep_osqp_update_semantics(cuda_backend):
    """batched closed loop with the bound switch of vehicle_lateral_mpc_slack_increment.py:158-172: slack columns active"""
    assert pc.check_bound_updates(cuda_backend, B=40, steps=36) > 0.1


def test_setup_resets_iterates(cuda_backend):
    pc.check_setup_resets_iterates(cuda_backend, B=64)


def test_host_front_door(cuda_backend):
    pc.check_host_front_door(cuda_backend)


def test_edge_cases_and_errors(cuda_backend):
    pc.check_edge_cases(cuda_backend)


def test_primal_infeasibility_certificate(cuda_backend):
    pc.check_primal_infeasibility(cuda_backend, B=70)
    pc.check_primal_infeasibility(cuda_backend, B=70, retile=True)


def test_random_problems_every_shape(cuda_backend):
    worst, seen = pc.check_random_problems(cuda_backend, seeds=(0, 1, 2, 3), B=35)
    assert {1, -3} <= seen and worst < 1e-9


def test_random_problems_edge_horizons(cuda_backend):
    """horizons 1..7, 33, 64 (the 3- and 5-deep stage-buffer rotations of the TMA kernels at their edges), a partial tile"""
    worst, seen = pc.check_random_problems(cuda_backend, seeds=tuple(range(2, 11)), B=37, horizons=(1, 2, 3, 4, 5, 6, 7, 33, 64))
    assert {1, -3} <= seen and worst < 1e-9
    cuda_backend.set_option("cta", 0)           # ... and the warp-per-tile / 8-lanes kernels on the same problems
    try:
        worst, seen = pc.check_random_problems(cuda_backend, seeds=(2, 3, 4, 5, 6), B=37, horizons=(1, 2, 3, 4, 5, 6, 7, 33, 64))
    finally:
        cuda_backend.set_option("cta", 1)
    assert worst < 1e-9


def test_infinite_bounds_and_stage_boxes(cuda_backend):
    pc.check_infinite_bounds_and_stage_boxes(cuda_backend)


def test_full_size_batch_properties(cuda_backend):
    """BASELINE configs[2] at full size (65536 QPs): properties that need no oracle run.
    (1) every QP reports 'solved'; (2) the reported unscaled residuals satisfy OSQP's termination inequalities
    against an independent torch evaluation of the dynamics rows; (3) batch invariance: a QP's answer does not
    depend on its position in the batch; (4) the oracle agrees on a strided sample."""
    from python_mpc_b200 import workloads
    from oracle import workload_qp
    B = 65536
    wl = workloads.lateral_slack_increment(B, seed=99, dtype=torch.float64)
    ctl = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
    res = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    st = res.info.status_val.cpu().numpy(); it = res.info.iter.cpu().numpy()
    assert (st == 1).all()
    assert it.min() >= 25 and (it % 25 == 0).all()
    x = res.x
    _, y, _ = ctl.solver.solution(want_x=False, want_y=True, want_u=False)      # res.y of the whole batch
    N, nx = 20, 5
    X = x[:, :(N + 1) * nx].reshape(B, N + 1, nx); U = x[:, (N + 1) * nx:(N + 1) * nx + N]
    # dynamics rows re-evaluated with torch from independently discretised models of a sample
    idx = np.arange(0, B, 4099)
    for b in idx:
        Ad, Bd = workload_qp.lateral_model(float(wl.speed[b]))
        Xb = X[b].cpu().numpy(); Ub = U[b].cpu().numpy()
        At = np.zeros((5, 5)); At[:4, :4] = Ad; At[:4, 4:] = Bd; At[4, 4] = 1; Bt = np.vstack([Bd, [[1.0]]])
        resid = Xb[1:] - Xb[:-1] @ At.T - Ub[:, None] * Bt.T
        assert np.abs(resid).max() < 2e-3 and np.abs(Xb[0] - wl.x0[b]).max() < 2e-3
        r = pc.oracle_solve(workload_qp.lateral_qp(wl, b), rho=5.0, eps_abs=1e-4, eps_rel=1e-4)
        assert r.info.iter == it[b] and pc.rel(x[b].cpu().numpy(), r.x) < 1e-6
        assert pc.rel(y[b].cpu().numpy(), r.y) < 1e-6                       # the duals too (res.y)
    # batch invariance: re-solve a permuted sub-batch
    perm = torch.randperm(4096, generator=torch.Generator().manual_seed(1)).numpy()
    pidx = torch.as_tensor(perm, device=x.device)
    cuda_backend.set_option("cta", 0)       # one set of kernels for both sizes: bit-identical whatever the position or batch
    try:
        big = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False).solve_batch(wl.x0, wl.xr, wl.speed)
        sub = wl.make_controller(capacity=4096, rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
        r2 = sub.solve_batch(wl.x0[perm], wl.xr[perm], wl.speed[perm])
    finally:
        cuda_backend.set_option("cta", 1)
    assert torch.equal(r2.x, big.x[pidx])
    # ... and the default schedule of the big batch (stragglers finish in the CTA-per-tile kernel) agrees with it to the last bits
    assert torch.equal(big.info.iter, res.info.iter) and torch.equal(big.info.status_val, res.info.status_val)
    assert float((big.x - x).abs().max()) < 1e-10 * float(x.abs().max())
    # default schedule of a 4096-QP batch (the CTA-per-tile kernel): same iteration counts, solutions to the last bits
    sub = wl.make_controller(capacity=4096, rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False)
    r3 = sub.solve_batch(wl.x0[perm], wl.xr[perm], wl.speed[perm])
    assert torch.equal(r3.info.iter, res.info.iter[pidx])
    assert float((r3.x - x[pidx]).abs().max()) < 1e-10 * float(x.abs().max())
    # duals of the whole batch: finite, and complementary with the bound rows (y > 0 only at an upper bound, y < 0 only
    # at a lower bound, up to the primal tolerance) — checked on the input-rate rows bu_k of every QP
    assert bool(torch.isfinite(y).all())
    ybu = y[:, 2 * (N + 1) * nx:]
    du = U
    dmax = 0.5 * np.pi / 180
    ytol = 1e-6 * float(ybu.abs().max())
    assert float((dmax - du)[ybu > ytol].max()) < 2e-3 and float((du + dmax)[ybu < -ytol].max()) < 2e-3


def test_bench_dump_outputs_are_the_last_timed_step(cuda_backend, tmp_path):
    """`bench.py --dump-outputs`, twice with the same arguments: identical files, holding what LateralMPC.solve_batch returns
    for the inputs of the last timed step (--warmup 1 --steps 1: the headline's batch of seed 1)."""
    import os, subprocess, sys
    from python_mpc_b200 import workloads
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = ("u", "iter", "status_val", "pri_res", "dua_res")
    out = []
    for d in ("a", "b"):
        p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--batch", "256", "--steps", "1", "--warmup", "1",
                            "--records", "none", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / d)],
                           capture_output=True, text=True, timeout=600, cwd=root)
        assert p.returncode == 0, p.stderr[-2000:]
        assert sorted(os.listdir(tmp_path / d)) == sorted(n + ".npy" for n in names)
        out.append({n: np.load(tmp_path / d / (n + ".npy")) for n in names})
    for n in names:
        assert out[0][n].dtype == np.float64 and np.array_equal(out[0][n], out[1][n]), n
    wl = workloads.lateral_slack_increment(256, seed=1, dtype=torch.float64)
    r = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False).solve_batch(wl.x0, wl.xr, wl.speed, want_x=False)
    u = r.u.cpu().numpy()
    assert out[0]["u"].shape == u.shape == (256, 20, 1)
    assert np.array_equal(out[0]["iter"], r.info.iter.cpu().numpy()) and (out[0]["status_val"] == 1).all()
    assert np.abs(out[0]["u"] - u).max() <= 1e-10 * np.abs(u).max()


def test_rate_bounds_hold_at_full_size(cuda_backend):
    from python_mpc_b200 import workloads
    wl = workloads.lateral_slack_increment(65536, seed=5, dtype=torch.float64)
    res = wl.make_controller(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False).solve_batch(wl.x0, wl.xr, wl.speed, want_x=False)
    assert float(res.u.abs().max()) <= 0.5 * np.pi / 180 + 2e-3        # delta-u bound up to eps_prim
