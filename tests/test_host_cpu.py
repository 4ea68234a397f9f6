"""CPU suite (-m "not gpu"): the host logic and the kernel arithmetic, run through tests/emu's host compilation of
the CUDA source, against the oracle and the golden fixtures.  No GPU compute happens here."""
import numpy as np
import pytest
import torch

import parity_cases as pc


@pytest.mark.parametrize("slack,increment", [(True, True), (False, False), (True, False), (False, True)])
def test_lateral_formulations_fp64(emu_backend, slack, increment):
    pc.check_lateral_batch(emu_backend, slack, increment, torch.float64, B=4)


def test_lateral_shared_linearisation_fp64(emu_backend):
    pc.check_lateral_batch(emu_backend, False, False, torch.float64, B=5, shared=True)


def test_lateral_fp32_within_1e4(emu_backend):
    # FP32 reaches OSQP's own termination test only for small rho_eq = 1e3*rho (DESIGN.md, "precision")
    pc.check_lateral_batch(emu_backend, True, True, torch.float32, B=3, rho=0.1, max_iter=400, eps=1e-3)


def test_iterates_match_oracle(emu_backend):
    pc.check_iterates(emu_backend, torch.float64, iters=60, rho=5.0)
    pc.check_iterates(emu_backend, torch.float32, iters=60, rho=0.1)


def test_build_qp_equals_reference_assembly(emu_backend, golden):
    pc.check_build_qp_against_reference_capture(emu_backend, golden)


def test_vehicle_models_equal_reference(emu_backend, golden):
    pc.check_models_against_reference(emu_backend, golden)


def test_reference_signature_functions(emu_backend, golden):
    pc.check_reference_functions(emu_backend, golden)


def test_kinematic_corridor_and_predmatrix_functions(emu_backend, golden):
    pc.check_kinematic_corridor_and_predmatrix(emu_backend, golden)


def test_closed_loop_trajectory(emu_backend, golden):
    pc.check_closed_loop(emu_backend, golden, steps=40)


def test_closed_loop_full_reference_script_with_bound_switches(emu_backend, golden):
    slack = pc.check_closed_loop_full(emu_backend, golden)
    assert np.abs(slack[401:901]).max() > 1.9 and np.abs(slack[1000:]).max() < 1e-3


def test_closed_loop_sweep_warm_started(emu_backend):
    pc.check_closed_loop_sweep(emu_backend, B=4, steps=5)


def test_long_horizon_time_varying_dynamics(emu_backend):
    pc.check_dynamic_long_horizon(emu_backend, B=2, N=30)


def test_retiling_is_bitwise_neutral_and_stragglers_match_oracle(emu_backend):
    pc.check_retiling_is_bitwise_neutral(emu_backend, B=40)


def test_bound_updates_keep_osqp_update_semantics(emu_backend):
    assert pc.check_bound_updates(emu_backend, B=4, steps=30) > 0.1


def test_setup_resets_iterates(emu_backend):
    pc.check_setup_resets_iterates(emu_backend)


def test_host_front_door(emu_backend):
    pc.check_host_front_door(emu_backend)


def test_edge_cases_and_errors(emu_backend):
    pc.check_edge_cases(emu_backend)


def test_primal_infeasibility_certificate(emu_backend):
    pc.check_primal_infeasibility(emu_backend)
    pc.check_primal_infeasibility(emu_backend, retile=True)


def test_random_problems_every_shape(emu_backend):
    worst, seen = pc.check_random_problems(emu_backend, seeds=(0, 1, 2, 3, 4, 5))
    assert {1, -3} <= seen and worst < 1e-9


def test_infinite_bounds_and_stage_boxes(emu_backend):
    pc.check_infinite_bounds_and_stage_boxes(emu_backend)


def test_bench_reference_arm_emits_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to the GPU arm): one JSON line with the contract's keys,
    the same `config` keys as the GPU arm, no GPU involved."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--batch", "512", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    import bench
    ns = type("A", (), dict(batch=512, horizon=20, rho=5.0, eps=1e-4))()
    assert set(line["config"]) == set(bench.workload_config(ns, 1))
    # a rank other than 0 of a torchrun launch exits without work and without output
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "2", "--batch", "512",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=root, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_dump_outputs_are_float_bounded_and_repeatable(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float32 / float64 .npy files; beyond the size bound one sample of QPs, the same in every array
    (u of two ranks: the same QPs of each rank's block) and in every run."""
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 100000)
    arrays = {"u": np.arange(2000 * 20, dtype=np.float64).reshape(2000, 20, 1), "iter": np.arange(1000, dtype=np.int32),
              "pri_res": np.arange(1000, dtype=np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    out = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in arrays}
    assert out["u"].dtype == np.float64 and out["iter"].dtype == np.float64 and out["pri_res"].dtype == np.float32
    assert sum(v.nbytes for v in out.values()) <= 100000 and 0 < out["iter"].size < 1000
    qps = out["iter"].astype(int)
    assert (np.diff(qps) > 0).all() and np.array_equal(out["pri_res"], qps)
    assert np.array_equal(out["u"], arrays["u"][np.concatenate([qps, 1000 + qps])])   # rank 0's QPs, then the same of rank 1
    for k in arrays:
        assert np.array_equal(out[k], np.load(tmp_path / "b" / (k + ".npy")))
    bench.dump_outputs(str(tmp_path / "c"), {"iter": arrays["iter"]})             # within the bound: everything
    assert np.array_equal(np.load(tmp_path / "c" / "iter.npy"), arrays["iter"])
