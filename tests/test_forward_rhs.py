"""The forward sweep that starts from the local right-hand side r^ left in the t slots by the previous backward sweep
(mpcb_set_option("fwd_rhs", 1), the default) against the forward sweep that forms the whole right-hand side ("fwd_rhs", 0):
the same iteration count and status for every QP and the same iterates up to rounding, on the schedules whose launches
continue from the t slots of an earlier launch — a chunked batch whose unsolved QPs are compacted into the scratch
workspace (and copied home and compacted again), warm-started closed-loop steps with bound updates, partial tiles and edge
horizons.  CPU (tests/emu: the same kernel code as host loops) and GPU (admm_tma_kernel)."""
import numpy as np
import pytest
import torch

import parity_cases as pc
from python_mpc_b200 import vehicle_models, workloads

RTOL = 1e-10


def _with(be, opts, fn):
    for k, v in opts.items():
        be.set_option(k, v)
    try:
        return fn()
    finally:
        be.set_option("fwd_rhs", 1); be.set_option("retile", 1); be.set_option("retile_min_batch", 4096)
        be.set_option("cta", 1)


def _both(be, fn, **opts):
    """fn() with r^ on and off; the results (tensors) compared: integers exactly, floats within RTOL relative."""
    on = _with(be, dict(opts, fwd_rhs=1), fn)
    off = _with(be, dict(opts, fwd_rhs=0), fn)
    for a, b in zip(on, off):
        a, b = a.cpu(), b.cpu()
        if a.dtype.is_floating_point:
            assert pc.rel(a.numpy(), b.numpy()) <= RTOL
        else:
            assert torch.equal(a, b)
    return on, off


def _cold_then_warm(be, B, N, seed=77):
    wl = workloads.lateral_slack_increment(B, N=N, seed=seed, dtype=torch.float64)

    def fn():
        ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=5.0, eps_abs=1e-4,
                                 eps_rel=1e-4, warm_start=True)
        r1 = ctl.solve_batch(wl.x0, wl.xr, wl.speed)
        out = [r1.x.clone(), r1.info.iter.clone(), r1.info.status_val.clone()]
        r2 = ctl.update_batch(wl.x0 * 0.9)              # warm-started: starts from the (z, y) the first solve left behind
        return out + [r2.x.clone(), r2.info.iter.clone(), r2.info.status_val.clone()]
    return fn


def check_chunked_compacted(be, B):
    """Chunks of check_termination iterations, the unsolved QPs compacted every time a fifth of the set has terminated."""
    on, off = _both(be, _cold_then_warm(be, B, 20), retile=1, retile_min_batch=2, cta=0)
    assert not torch.equal(on[0], off[0]), "the option selects the same arithmetic"      # (two forms of r, other rounding)
    it = on[1].cpu().numpy()
    assert len(np.unique(it)) > 2, "workload does not exercise the compaction: %s" % np.unique(it)
    # with r^ the chunked loop is still bit-identical to one launch
    one = _with(be, dict(fwd_rhs=1, retile=0, cta=0), _cold_then_warm(be, B, 20))
    for a, b in zip(on, one):
        assert torch.equal(a.cpu(), b.cpu())


def check_closed_loop_bound_updates(be, B=6, steps=14, N=20):
    """Warm-started closed-loop steps; the lateral-error lower bound is tightened at step 4 and relaxed at step 9."""
    wl = workloads.LateralWorkload(B, N, True, True, 41, torch.float64)
    wl.x0[:, 3] = np.linspace(-1.0, 3.5, B)
    tight = wl.xmin.copy(); tight[3] = 2.0
    sched = {4: dict(xmin=tight), 9: dict(xmin=wl.xmin)}

    def fn():
        ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(_backend=be), _backend=be, rho=5.0, eps_abs=1e-4,
                                 eps_rel=1e-4, warm_start=True)
        traj, us, its = ctl.closed_loop_batch(wl.x0, wl.xr, wl.speed, steps=steps, bounds_at=lambda k: sched.get(k))
        return [traj.clone(), us.clone(), its.clone()]
    _both(be, fn, retile=1, retile_min_batch=2, cta=0)


def check_edge_horizons(be, B=37):
    """Horizons 1, 2 and 33 (stage 0 next to stage N, the turn-around stages), a ragged last tile."""
    for N in (1, 2, 33):
        _both(be, _cold_then_warm(be, B, N, seed=5), retile=1, retile_min_batch=2, cta=0)


def test_fwd_rhs_chunked_compacted_cpu(emu_backend):
    check_chunked_compacted(emu_backend, 96)


def test_fwd_rhs_closed_loop_bound_updates_cpu(emu_backend):
    check_closed_loop_bound_updates(emu_backend)


def test_fwd_rhs_edge_horizons_cpu(emu_backend):
    check_edge_horizons(emu_backend)


@pytest.mark.gpu
def test_fwd_rhs_chunked_compacted_gpu(cuda_backend):
    check_chunked_compacted(cuda_backend, 4096)


@pytest.mark.gpu
def test_fwd_rhs_closed_loop_bound_updates_gpu(cuda_backend):
    check_closed_loop_bound_updates(cuda_backend, B=64)


@pytest.mark.gpu
def test_fwd_rhs_edge_horizons_gpu(cuda_backend):
    check_edge_horizons(cuda_backend, B=100)
