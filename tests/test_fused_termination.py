"""The termination test evaluated by the backward sweep of the tested iteration (admm_bwd_stage in mode kBwdTest): residuals
and infeasibility certificates against the oracle — iteration count, status, primal and dual residual — on the schedules
that reach the test from unusual places: a test at every iteration (the first iteration of a solve is tested), a cap that
is not a multiple of check_termination, primal-infeasible QPs with and without certificates, the edge horizons on a
ragged last tile, and a chunked, compacted batch followed by a warm-started solve.  CPU (tests/emu: the lane-per-QP driver,
the same stage code as host loops) and GPU (admm_tma_kernel, compared with the lane-per-QP and CTA kernels as well)."""
import numpy as np
import pytest
import torch

import parity_cases as pc
from python_mpc_b200 import vehicle_models, workloads
from oracle import workload_qp

# residuals against the oracle (another implementation: near convergence a residual is a sum that cancels, so its rounding
# differs in absolute terms, a millionth of the 1e-4 tolerances it is compared with)
RES_RTOL, RES_ATOL = 1e-6, 1e-10


def _opts(be, opts):
    for k, v in opts.items():
        be.set_option(k, v)


def _reset(be):
    _opts(be, dict(retile=1, retile_min_batch=4096, cta=1, tma=1, certificates=1))


def _solve(be, wl, opts=None, **settings):
    _opts(be, opts or {})
    try:
        ctl = wl.make_controller(vehicle=vehicle_models.Vehicle_Lateral(dtype=wl.dtype, _backend=be), _backend=be,
                                 **dict(dict(rho=5.0, eps_abs=1e-4, eps_rel=1e-4, warm_start=False), **settings))
        return ctl, ctl.solve_batch(wl.x0, wl.xr, wl.speed)
    finally:
        _reset(be)


def _against_oracle(wl, res, samples, **settings):
    it = res.info.iter.cpu().numpy(); st = res.info.status_val.cpu().numpy()
    pri = res.info.pri_res.cpu().numpy(); dua = res.info.dua_res.cpu().numpy()
    s = dict(dict(rho=5.0, eps_abs=1e-4, eps_rel=1e-4), **settings)
    for b in samples:
        r = pc.oracle_solve(workload_qp.lateral_qp(wl, int(b)), **s)
        assert (it[b], st[b]) == (r.info.iter, r.info.status_val), (b, it[b], st[b], r.info.iter, r.info.status)
        for got, ref in ((pri[b], r.info.pri_res), (dua[b], r.info.dua_res)):
            assert abs(got - ref) <= RES_ATOL + RES_RTOL * abs(ref), (b, got, ref)
    return it, st


def check_every(be, B=37):
    """check_termination 1, 2 and 25; a cap (37) that is not a multiple of check_termination ends in the approximate test."""
    wl = workloads.lateral_slack_increment(B, seed=3, dtype=torch.float64)
    for ce, mi in ((1, 4000), (2, 4000), (25, 4000), (25, 37), (2, 37)):
        _, res = _solve(be, wl, dict(cta=0), check_termination=ce, max_iter=mi)
        it, _ = _against_oracle(wl, res, (0, 17, B - 1), check_termination=ce, max_iter=mi)
        if mi == 37:
            assert (it == 37).any()
    # max_iter = 1: the only iteration is the first one of the solve, and it is tested
    _, res = _solve(be, wl, dict(cta=0), max_iter=1)
    assert (res.info.iter.cpu().numpy() == 1).all()
    _against_oracle(wl, res, (0, B - 1), max_iter=1)


def check_primal_infeasible(be, B=37):
    """Hard-constraint QPs whose initial state violates the state box, next to feasible ones; certificates on and off."""
    wl = workloads.LateralWorkload(B, 20, False, False, 9, torch.float64)
    wl.x0[1, 3] = 14.0
    wl.x0[B - 1, 2] = -0.5
    _, res = _solve(be, wl, dict(cta=0))
    _, st = _against_oracle(wl, res, (0, 1, 5, B - 1))
    assert st[1] == -3 and st[B - 1] == -3
    # without certificates an infeasible QP runs to the cap, where OSQP's final test consults them
    _, res = _solve(be, wl, dict(cta=0, certificates=0), max_iter=60)
    it = res.info.iter.cpu().numpy()
    assert it[1] == 60 and it[B - 1] == 60
    _against_oracle(wl, res, (0, 5), max_iter=60)


def check_edge_horizons(be, B=37):
    for N in (1, 2, 33):
        wl = workloads.LateralWorkload(B, N, True, True, 5, torch.float64)
        _, res = _solve(be, wl, dict(cta=0))
        _against_oracle(wl, res, (0, 31, B - 1))


def check_chunked_then_warm(be, B):
    """Chunks of check_termination iterations with compaction, then a warm-started solve: the oracle for the cold solve,
    the single launch bit for bit for both."""
    wl = workloads.lateral_slack_increment(B, seed=77, dtype=torch.float64)
    out = []
    for retile in (1, 0):
        ctl, r1 = _solve(be, wl, dict(cta=0, retile=retile, retile_min_batch=2), warm_start=True)
        if retile:
            it, _ = _against_oracle(wl, r1, np.flatnonzero(r1.info.iter.cpu().numpy() == int(r1.info.iter.max()))[:2])
            assert len(np.unique(it)) > 2, np.unique(it)
        _opts(be, dict(cta=0, retile=retile, retile_min_batch=2))
        try:
            r2 = ctl.update_batch(wl.x0 * 0.9)
        finally:
            _reset(be)
        out.append([t.clone() for r in (r1, r2) for t in (r.x, r.info.iter, r.info.status_val, r.info.pri_res,
                                                             r.info.dua_res)])
    for a, b in zip(*out):
        assert torch.equal(a, b)


def check_tested_sweep_keeps_iterates(be, B=37):
    """The tested backward sweep computes the iterates of the plain one bit for bit: at a cap of 30 iterations, the QPs
    that a test at iteration 25 does not stop end where they end without that test."""
    wl = workloads.lateral_slack_increment(B, seed=3, dtype=torch.float64)
    for opts in (dict(cta=0), dict(cta=0, tma=0)):
        _, r0 = _solve(be, wl, opts, check_termination=0, max_iter=30)
        x0, it0 = r0.x.clone(), r0.info.iter.clone()
        _, r1 = _solve(be, wl, opts, check_termination=25, max_iter=30)
        assert (it0 == 30).all()
        cont = r1.info.iter == 30
        assert int(cont.sum()) > 0
        assert torch.equal(x0[cont], r1.x[cont])


def test_tested_sweep_keeps_iterates_cpu(emu_backend):
    check_tested_sweep_keeps_iterates(emu_backend)


def test_check_every_cpu(emu_backend):
    check_every(emu_backend)


def test_primal_infeasible_cpu(emu_backend):
    check_primal_infeasible(emu_backend)


def test_edge_horizons_cpu(emu_backend):
    check_edge_horizons(emu_backend)


def test_chunked_then_warm_cpu(emu_backend):
    check_chunked_then_warm(emu_backend, 96)


@pytest.mark.gpu
def test_tested_sweep_keeps_iterates_gpu(cuda_backend):
    check_tested_sweep_keeps_iterates(cuda_backend, B=100)


@pytest.mark.gpu
def test_check_every_gpu(cuda_backend):
    check_every(cuda_backend, B=100)


@pytest.mark.gpu
def test_primal_infeasible_gpu(cuda_backend):
    check_primal_infeasible(cuda_backend, B=100)


@pytest.mark.gpu
def test_edge_horizons_gpu(cuda_backend):
    check_edge_horizons(cuda_backend, B=100)


@pytest.mark.gpu
def test_chunked_then_warm_gpu(cuda_backend):
    check_chunked_then_warm(cuda_backend, 4096)


@pytest.mark.gpu
def test_tma_kernel_agrees_with_lane_and_cta_kernels(cuda_backend):
    """admm_tma_kernel against the lane-per-QP kernel (the same stage functions: bit for bit, residuals included) and the
    CTA-per-tile kernel (its own sweeps and termination sweep: same iterations and statuses, iterates and residuals to
    rounding), at check_termination 25 and 1."""
    wl = workloads.lateral_slack_increment(300, seed=8, dtype=torch.float64)
    for ce in (25, 1):
        res = {}
        for name, opts in (("tma", dict(cta=0, tma=1)), ("lane", dict(cta=0, tma=0)), ("cta", dict(cta=2))):
            _, r = _solve(cuda_backend, wl, opts, check_termination=ce)
            res[name] = [t.clone() for t in (r.x, r.info.iter, r.info.status_val, r.info.pri_res, r.info.dua_res)]
        for a, b in zip(res["tma"], res["lane"]):
            assert torch.equal(a, b)
        a, c = res["tma"], res["cta"]
        assert torch.equal(a[1], c[1]) and torch.equal(a[2], c[2])
        assert pc.rel(a[0].cpu().numpy(), c[0].cpu().numpy()) < 1e-10
        for k in (3, 4):
            assert float(((a[k] - c[k]).abs() - RES_RTOL * c[k].abs()).max()) <= RES_ATOL
