#!/usr/bin/env python
"""Headline benchmark: lateral-MPC QP solves/sec (BASELINE.json metric) + one record per other BASELINE config.

Headline workload (config.workload): configs[2] of BASELINE.json — a batch of 65536 soft-constraint + incremental
(slack + delta-u) lateral MPC QPs per GPU, H = 20, every QP linearised at its own vehicle speed, OSQP-equivalent ADMM with
fixed rho/sigma/alpha, adaptive_rho and polish off, eps_abs = eps_rel = 1e-4.  One "step" = one pass of the hot path over
one synthetic batch:
    QP build (discretise A,B per speed, delta-u augmentation, layout) -> Ruiz scaling + cached KKT factorisation
    -> ADMM to convergence -> gather of the control sequences (+ NCCL all_gather of them at N > 1).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--records all|none|a,b,..] [--dump-outputs DIR]

value   : whole-job QP solves/sec with the inputs already resident in HBM (weak scaling: 65536 QPs per GPU)
e2e     : the same through the public API (LateralMPC.solve_batch) from pinned HOST buffers, H2D of the inputs, the
          all_gather and D2H of the control sequences inside the timed region
records : the other configurations, each with its own roofline and cpu_baseline —
          strong    global batch 65536 split over the N GPUs (sharding.solve_sharded)
          qp_build  "cast MPC problem to a QP" alone: per-speed discretisation, delta-u augmentation and the explicit
                    P/q/A/l/u assembly of the 65536 configs[2] QPs (north_star (1))           (N = 1 only)
          configs1  batch 1024 vanilla lateral MPC, one shared linearisation, f64     (N = 1 only)
          configs3  batch 8192, H = 100, time-varying combined dynamics model, f64     (N = 1 only)
          configs4  closed-loop sweep, 131072 scenarios per GPU x 200 warm-started steps (1M scenarios at N = 8)
          fp32      configs[2] solved in f32 at rho = 0.1 next to f64 at the same rho  (N = 1 only)
--impl reference : the reference's per-QP OSQP loop restated in C (oracle/osqp_admm.c), all host threads, the full
          65536-QP batch per step (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "lateral-MPC QP solves/sec (batch 65536, H=20)"
UNIT = "QP solves/s"
ALL_RECORDS = ("strong", "qp_build", "configs1", "configs3", "configs4", "fp32")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline and of its e2e figure (the records keep their own step counts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="QPs per GPU (weak scaling)")
    ap.add_argument("--horizon", type=int, default=20)
    ap.add_argument("--rho", type=float, default=5.0)
    ap.add_argument("--eps", type=float, default=1e-4)
    ap.add_argument("--dtype", default="f64", choices=["f32", "f64"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="QPs in the cpu_baseline sample of the headline (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--records", default="all", help="all | none | comma-separated subset of " + ",".join(ALL_RECORDS))
    ap.add_argument("--sweep-scenarios", type=int, default=131072, help="configs4: closed-loop scenarios per GPU")
    ap.add_argument("--sweep-steps", type=int, default=200, help="configs4: closed-loop steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline returned to its caller as DIR/<name>.npy: u (the control "
                         "sequences; at N > 1 every rank's, rank by rank), iter, status_val, pri_res, dua_res (rank 0's QPs); "
                         "float32 or float64, at most 64 MB in all (beyond that one fixed, seeded sample of QPs in every array)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


def host_cores():
    return len(os.sched_getaffinity(0))


DUMP_BYTES = 63 * 10 ** 6          # --dump-outputs: at most 64 MB in all, .npy headers included


def dump_outputs(d, arrays, seed=0):
    """np.save of each array as d/<name>.npy, float32 kept, anything else as float64.  Every array holds n rows (one per QP)
    or k blocks of n rows (at N > 1, u: one block per rank, in rank order).  Arrays that together exceed DUMP_BYTES keep the
    same QPs: one sorted sample r of the n rows, drawn with a fixed seed (the same from run to run), from every block."""
    os.makedirs(d, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_BYTES:
        n = min(v.shape[0] for v in arrays.values())
        r = np.sort(np.random.default_rng(seed).choice(n, max(1, n * DUMP_BYTES // total), replace=False))
        arrays = {k: v.reshape(-1, n, *v.shape[1:])[:, r].reshape(-1, *v.shape[1:]) for k, v in arrays.items()}
    for k, v in arrays.items():
        np.save(os.path.join(d, k + ".npy"), v)


def workload_config(a, n_gpus):
    """The workload description — identical in the GPU arm and the reference arm."""
    return {"workload": "BASELINE configs[2]: batch %d slack+delta-u lateral MPC QPs per GPU, H=%d, per-QP speed linearisation"
                        % (a.batch, a.horizon),
            "batch_per_gpu": a.batch, "global_batch": a.batch * n_gpus, "horizon": a.horizon,
            "nvar": (a.horizon + 1) * 5 * 2 + a.horizon, "ncon": 2 * (a.horizon + 1) * 5 + a.horizon,
            "rho": a.rho, "sigma": 1e-6, "alpha": 1.6, "eps_abs": a.eps, "eps_rel": a.eps, "max_iter": 4000,
            "check_termination": 25, "scaling": 10, "adaptive_rho": False, "polish": False, "warm_start": False,
            "l2": "per-step working set (~1.6 GB per GPU) exceeds the 126 MB L2; 4 distinct seeded batches cycle through the steps",
            "host_cores": host_cores(),
            "parallelism": "independent QPs sharded across %d GPU(s); NCCL all_gather of control sequences only" % n_gpus}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port, timed on the host cores (cpu_baseline legs and --impl reference)
# ------------------------------------------------------------------------------------------------
def cpu_lateral_inputs(wl):
    from oracle import workload_qp
    return workload_qp.lateral_batch_csc(wl)


def cpu_solve(inputs, rho, eps, repeats=1, max_iter=4000):
    """oracle_solve_batch on every host core.  Returns (QPs/s, cores, mean iterations, fraction solved, seconds)."""
    from oracle import c_oracle
    Pu, A0, Pv, q, Av, l, u, perm = inputs
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        x, y, it, st, used = c_oracle.solve_batch(Pu, A0, Pv, q, Av, l, u, perm=perm, nthreads=host_cores(), rho=rho,
                                                  eps_abs=eps, eps_rel=eps, max_iter=max_iter)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return q.shape[0] / best, used, float(it.mean()), float((st == 1).mean()), best


def cpu_solves_per_sec(a, sample, seed, repeats=1):
    import torch
    from python_mpc_b200 import workloads
    wl = workloads.lateral_slack_increment(sample, N=a.horizon, seed=seed, dtype=torch.float64)
    return cpu_solve(cpu_lateral_inputs(wl), a.rho, a.eps, repeats)


def run_reference(a):
    """The reference arm: torchrun starts one process per GPU; rank 0 alone runs the CPU loop."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from python_mpc_b200 import workloads
    B = a.batch                                                   # the full batch of the named config per step
    sets = [cpu_lateral_inputs(workloads.lateral_slack_increment(B, N=a.horizon, seed=1000 + i, dtype=torch.float64))
            for i in range(min(a.warmup + a.steps, 2))]
    times, info = [], None
    for i in range(a.warmup + a.steps):
        v, cores, iters, solved, dt = cpu_solve(sets[i % len(sets)], a.rho, a.eps)
        if i >= a.warmup:
            times.append(dt)
        info = (cores, iters, solved)
    tot = sum(times)
    value = B * a.steps / tot
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(a, a.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": info[0], "kind": "port",
                             "sample": "the full batch of %d QPs per step (oracle/osqp_admm.c, -O3 -march=native, OpenMP over "
                                       "QPs); mean %.1f ADMM iterations, %.3f solved" % (B, info[1], info[2])},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled in-process every ~20 ms (the
    timed region is a few steps of ~25 ms, too short for `nvidia-smi -lms`); nvidia-smi is the fallback."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t, self.h, self.nv = index, [], False, None, None, None
        self.sm_max, self.source = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ent = vis.split(",")[index].strip()
                phys = int(ent) if ent.isdigit() else None
                if phys is None:
                    self.h = pynvml.nvmlDeviceGetHandleByUUID(ent.encode() if hasattr(ent, "encode") else ent)
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv, self.source = pynvml, "nvml"
        except Exception:
            self.h = None

    def _poll_nvml(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), float(mhz), int(mask)))
            except Exception:
                pass
            time.sleep(0.02)       # NVML queries take the driver lock: polled sparingly so that they do not perturb the steps

    def _poll_smi(self):
        names = [0x8, 0x40, 0x20, 0x4]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                r = [c.strip() for c in out.strip().splitlines()[0].split(",")]
                mask = 0
                for bit, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        mask |= bit
                self.sm_max = float(r[1])
                self.rows.append((time.perf_counter(), float(r[0]), mask))
            except Exception:
                time.sleep(0.05)

    def start(self):
        if self.h is None:
            self.source = "nvidia-smi"
        self.t = threading.Thread(target=self._poll_nvml if self.h is not None else self._poll_smi, daemon=True)
        self.t.start()

    def window(self, t0, t1):
        """Summary of the samples taken inside [t0, t1] (perf_counter times bracketing the timed region)."""
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        sm = [r[1] for r in rows]
        mask = 0
        for r in rows:
            mask |= r[2]
        reasons = sorted(n for b, n in self.REASONS.items() if mask & b)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.sm_max, "reasons": reasons,
                "samples": len(sm), "source": self.source}

    def stop(self):
        self.stop_flag = True
        if self.t is not None:
            self.t.join(timeout=6)


def load_peak():
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        v = json.load(open(pk)).get("hbm_gbs")
        if v:
            return float(v), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of that kernel
    (profiles/traffic.json), reported only while the kernel sources are the ones that were profiled (content hash)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, None
    try:
        import __graft_entry__ as g
        ent = json.load(open(path)).get(kernel_key)
        if not ent or ent.get("csrc_sha256") != g.csrc_digest(ent.get("csrc_files")):
            return None, None
        return ent["dram_bytes"], ent["source"]
    except Exception:
        return None, None


def run_ours(a):
    import torch
    import torch.distributed as dist
    import python_mpc_b200 as pm
    from python_mpc_b200 import roofline, sharding, vehicle_models, workloads

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    want = set(ALL_RECORDS) if a.records == "all" else set() if a.records == "none" else set(a.records.split(","))
    dtype = torch.float32 if a.dtype == "f32" else torch.float64
    esz = 4 if a.dtype == "f32" else 8
    B, N = a.batch, a.horizon
    be = pm.cuda_backend()
    peak, peak_src = load_peak()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    def timed(step_fn, steps):
        """`steps` calls bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step_fn(i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))[0]

    # ------------------------------------------------------------------------------------------ headline: configs[2]
    nsets = a.warmup + a.steps
    sets = [workloads.lateral_slack_increment(B, N=N, seed=100 * rank + i, dtype=dtype) for i in range(min(nsets, 4))]
    dev_in = [(torch.as_tensor(w.x0).to(dev, dtype), torch.as_tensor(w.xr).to(dev, dtype),
               torch.as_tensor(w.speed).to(dev, dtype)) for w in sets]
    host_in = [(torch.as_tensor(w.x0).to(dtype).pin_memory(), torch.as_tensor(w.xr).to(dtype).pin_memory(),
                torch.as_tensor(w.speed).to(dtype).pin_memory()) for w in sets]
    ctl = sets[0].make_controller(capacity=B, rho=a.rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=False)

    # The path's only collective, the all_gather of the control sequences, is issued asynchronously from a staging copy of the
    # step's controls (two buffers): the solve of step i + 1 does not depend on it, so a rank only waits for the gather of
    # step i - 1 — without that slack every step costs the slowest rank's time (the batches differ in their straggler tails)
    # and the N = 8 line measured 0.95 of 8 x one GPU.  All gathers complete inside the timed region (drain() before the
    # closing barrier).
    stage_u = [torch.empty((B, N, 1), device=dev, dtype=dtype) for _ in range(2)] if world > 1 else None
    gathered = [torch.empty((B * world, N, 1), device=dev, dtype=dtype) for _ in range(2)] if world > 1 else None
    pending = [None, None]

    def drain():
        for j in range(2):
            if pending[j] is not None:
                pending[j].wait()
                pending[j] = None

    def step(i):
        x0, xr, sp = dev_in[i % len(dev_in)]
        res = ctl.solve_batch(x0, xr, sp, want_x=False, reuse=True)
        u_all = res.u
        if world > 1:
            j = i & 1
            if pending[j] is not None:
                pending[j].wait()                    # (the gather of two steps ago: long finished)
            stage_u[j].copy_(res.u)
            pending[j] = dist.all_gather_into_tensor(gathered[j], stage_u[j], async_op=True)
            u_all = gathered[j]
        return res, u_all

    # the clock sampler starts BEFORE the warm-up (NVML's first queries take milliseconds); only the samples that fall
    # inside the timed region are reported
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for i in range(max(a.warmup, 1)):        # (at least one untimed step: allocations, the learnt re-tile point)
        res, _ = step(i)
    drain()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
    # per-step solver info goes into buffers allocated BEFORE the timed region: a fresh allocation inside it can make the
    # caching allocator call cudaMalloc, which synchronises the device (seen as one 5-15 ms slower step)
    it_buf = torch.empty((a.steps, B), device=dev, dtype=res.info.iter.dtype)
    st_buf = torch.empty((a.steps, B), device=dev, dtype=res.info.status_val.dtype)
    step(0)                                  # one more untimed step after the allocations above
    drain()
    barrier()
    launches0 = be.launch_count()
    wall0 = time.perf_counter()
    ev[0].record()
    for i in range(a.steps):
        res, u_all = step(a.warmup + i)
        it_buf[i].copy_(res.info.iter); st_buf[i].copy_(res.info.status_val)
        ev[i + 1].record()
    drain()
    end_ev = torch.cuda.Event(enable_timing=True)
    end_ev.record()
    barrier()
    wall1 = time.perf_counter()
    if a.dump_outputs and rank == 0:
        # the last step's results are views of the solver's reused buffers: copied out before any later solve
        inf = res.info
        dump_outputs(a.dump_outputs, {"u": u_all.cpu().numpy(), "iter": inf.iter.cpu().numpy(), "status_val": inf.status_val.cpu().numpy(),
                                      "pri_res": inf.pri_res.cpu().numpy(), "dua_res": inf.dua_res.cpu().numpy()})
    launches = be.launch_count() - launches0
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)]
    total_ms = ev[0].elapsed_time(end_ev)
    clocks = sampler.window(wall0, wall1) if rank == 0 else None
    solved = (st_buf == 1).double().mean().item()
    mean_iter = it_buf.reshape(-1).double().mean().item()

    # ---- dominant kernel alone (the ADMM loop): CUDA events on the launching stream
    s = ctl.solver
    admm_ms = []
    for i in range(max(2, min(a.steps, 5))):
        x0, xr, sp = dev_in[i % len(dev_in)]
        ctl.solve_batch(x0, xr, sp, want_x=False)          # sets the batch up
        s.cold_start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(); s.solve(); e1.record()
        torch.cuda.synchronize()
        admm_ms.append(e0.elapsed_time(e1))
    admm_avg_ms = float(np.mean(admm_ms))
    warp_iters = s.info().iter.double().reshape(-1, 32).max(dim=1).values.sum().item() * 32   # iterations the warps executed

    # ---- e2e: public API from pinned host buffers; copies and the all_gather inside the timed region
    # the step's result on the host: rank 0 reads the whole gathered array (the job's result), every other rank its own shard
    # (eight ranks each pulling the same 84 MB through the host's PCIe root measured 15 M instead of 19 M solves/s at N = 8)
    out_rows = B * world if rank == 0 else B
    out_host = torch.empty((out_rows, N, 1), dtype=dtype).pin_memory()

    def e2e_step(i):
        hx0, hxr, hsp = host_in[i % len(host_in)]
        r = ctl.solve_batch(hx0.to(dev, non_blocking=True), hxr.to(dev, non_blocking=True),
                            hsp.to(dev, non_blocking=True), want_x=False, reuse=True)
        u_all = sharding.gather_controls(r.u, B * world) if world > 1 else r.u
        out_host.copy_(u_all if rank == 0 else r.u, non_blocking=True)
        torch.cuda.synchronize()

    for i in range(2):
        e2e_step(i)
    e2e_ms = timed(e2e_step, a.steps)
    if rank == 0:
        sampler.stop()
    total_ms = max_over_ranks(total_ms)[0]

    line = None
    if rank == 0:
        bytes_qp_iter = roofline.admm_bytes_per_qp_iteration(N, 5, 1, True, esz)
        achieved = bytes_qp_iter * B * mean_iter / (admm_avg_ms * 1e-3) / 1e9
        default_cfg = (B == 65536 and N == 20 and a.dtype == "f64" and a.rho == 5.0 and a.eps == 1e-4)
        traffic, traffic_src = ncu_traffic("admm_tma_kernel/configs2") if default_cfg else (None, None)
        cfg = workload_config(a, world)
        line = {"metric": METRIC, "value": B * world * a.steps / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": total_ms / a.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic", "config": cfg,
                "solve_stats": {"mean_admm_iterations": mean_iter, "fraction_solved": solved,
                                "workspace_mb": s.be.lib.mpcb_workspace_bytes(s._h) / 1e6},
                "p50_batch_latency_ms": float(np.median(step_ms)), "step_ms": [round(v, 2) for v in step_ms],
                "clocks": clocks,
                "e2e": {"value": B * world * a.steps / (e2e_ms * 1e-3), "unit": UNIT,
                        "h2d_bytes_per_step": B * (5 + 4 + 1) * esz, "d2h_bytes_per_step": B * world * N * esz,
                        "note": "bytes of rank 0 (it reads the whole gathered result; the other ranks read their own shard)"},
                "gpu_launches": launches,
                "roofline": {"kernel": "admm_tma_kernel (ADMM loop: phase-1 launch; + admm_wide_kernel and the tested iteration of the stragglers)",
                             "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_unit": "bytes per solve (the admm_tma_kernel launches: phase 1 + the stragglers' tested iteration)",
                             "traffic_source": traffic_src, "peak_source": peak_src,
                             "algorithmic_bytes_per_qp_iteration": bytes_qp_iter,
                             "algorithmic_bytes_per_solve": bytes_qp_iter * B * mean_iter,
                             "avg_launch_ms": admm_avg_ms,
                             "note": "algorithmic bytes = 164 record elements per stage and iteration x the iterations each "
                                     "QP needs (termination sweeps, certificate sweeps and the old-state copies are not "
                                     "counted); a warp streams its tile's records until its slowest lane converges "
                                     "(%.2fx the needed lane-iterations without re-tiling), which is why unconverged QPs "
                                     "are re-tiled" % (warp_iters / (B * mean_iter))}}
        if not a.no_cpu_baseline:
            sample = a.cpu_sample or 65536                      # the full batch of the named config, once
            v, cores, cit, csolved, dt = cpu_solves_per_sec(a, sample, seed=4242, repeats=1)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d QPs of the same workload (oracle/osqp_admm.c, -O3 -march=native, OpenMP over QPs, "
                                              "%.1f s); mean %.1f ADMM iterations, %.3f solved" % (sample, dt, cit, csolved)}
    del ctl, s, dev_in, host_in, out_host
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------------------------------ records
    records = {}
    ctx = dict(a=a, torch=torch, dist=dist, pm=pm, workloads=workloads, sharding=sharding, roofline=roofline,
               vehicle_models=vehicle_models, dev=dev, world=world, rank=rank, barrier=barrier, timed=timed,
               max_over_ranks=max_over_ranks, peak=peak, peak_src=peak_src, be=be)
    single_gpu_only = {"configs1": record_configs1, "configs3": record_configs3, "fp32": record_fp32, "qp_build": record_qp_build}
    for name in ALL_RECORDS:
        if name not in want:
            continue
        try:
            if name == "strong":
                rec = record_strong(ctx)
            elif name == "configs4":
                rec = record_configs4(ctx)
            elif world == 1:
                rec = single_gpu_only[name](ctx)
            else:
                rec = None                      # single-GPU configurations: measured by the N = 1 run
            if rec is not None and rank == 0:
                records[name] = rec
        except Exception as e:                  # a failing record must not cost the headline line
            if rank == 0:
                records[name] = {"error": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()
    if rank == 0:
        line["records"] = records
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def record_strong(c):
    """Strong scaling of the named batch: ONE global batch of 65536 QPs split over the N GPUs (north_star (3))."""
    a, torch, sharding, workloads = c["a"], c["torch"], c["sharding"], c["workloads"]
    world, rank, dev = c["world"], c["rank"], c["dev"]
    total, N = 65536, a.horizon
    lo, hi = sharding.shard_range(total, rank, world)
    sets = [workloads.lateral_slack_increment(total, N=N, seed=7000 + i, dtype=torch.float64) for i in range(2)]
    dev_in = [tuple(torch.as_tensor(v[lo:hi]).to(dev, torch.float64) for v in (w.x0, w.xr, w.speed)) for w in sets]
    ctl = sets[0].make_controller(capacity=hi - lo, rho=a.rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=False)

    def step(i):
        x0, xr, sp = dev_in[i % 2]
        r = ctl.solve_batch(x0, xr, sp, want_x=False, reuse=True)
        return sharding.gather_controls(r.u, total) if world > 1 else r.u

    for i in range(3):
        step(i)
    steps = max(a.steps, 5)
    ms = c["timed"](step, steps)
    return {"what": "strong scaling: global batch %d (configs[2]) split over %d GPU(s), all_gather of the control sequences "
                    "inside the step" % (total, world),
            "global_batch": total, "batch_per_gpu": hi - lo, "n_gpus": world, "steps": steps, "ms_per_step": ms / steps,
            "value": total * steps / (ms * 1e-3), "unit": UNIT, "scaling": "strong"}


def record_qp_build(c):
    """north_star (1): the QP build as batched kernels — discretisation of A, B per vehicle speed (ZOH), delta-u augmentation
    and the explicit P/q/A/l/u assembly in the reference's ordering (what the reference hands to prob.setup(); the solve path
    itself never materialises it) for the 65536 configs[2] QPs."""
    a, torch, workloads = c["a"], c["torch"], c["workloads"]
    dev = c["dev"]
    B, N = a.batch, a.horizon
    wl = workloads.lateral_slack_increment(B, N=N, seed=11, dtype=torch.float64)
    x0, xr, sp = (torch.as_tensor(v).to(dev, torch.float64) for v in (wl.x0, wl.xr, wl.speed))
    ctl = wl.make_controller(capacity=B, rho=a.rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=False, max_iter=1)
    ctl.solve_batch(x0, xr, sp, want_x=False)          # borrows the inputs, allocates the workspace
    s = ctl.solver
    be = s.be
    import ctypes as C
    from python_mpc_b200._lib import ptr
    nnz = be.lib.mpcb_qp_pattern(s._h, None, None)
    ld = s.ld
    mk = lambda n: torch.empty((n, ld), device=dev, dtype=torch.float64)
    Pd, q, Av, l, u = mk(s.nvar), mk(s.nvar), mk(nnz), mk(s.ncon), mk(s.ncon)
    st = lambda: be.stream()

    def models(i):
        ctl._model(sp, B)

    def assemble(i):
        be.check(be.lib.mpcb_build_qp(s._h, ptr(Pd), ptr(q), ptr(Av), ptr(l), ptr(u), st()))

    models(0); assemble(0)
    steps = 10
    ms_model = c["timed"](models, steps) / steps
    ms_asm = c["timed"](assemble, steps) / steps
    out_bytes = (2 * s.nvar + nnz + 2 * s.ncon) * 8 * B
    in_bytes = (25 + 5 + 5 + 5) * 8 * B                  # A~, B~, x_init, xr of every QP
    ach = (out_bytes + in_bytes) / (ms_asm * 1e-3) / 1e9
    model_bytes = (1 + 16 + 4 + 16 + 4 + 25 + 5) * 8 * B   # speed -> Ad, Bd (written, read back) -> A~, B~
    return {"what": "north_star (1), the QP build of the %d configs[2] QPs as batched kernels: (a) per-speed ZOH discretisation of "
                    "the lateral bicycle model + delta-u augmentation (mpcb_lateral_discretize, mpcb_augment_increment, layout), "
                    "(b) explicit P (diagonal), q, A (CSC values, %d nonzeros), l, u in the reference's ordering (mpcb_build_qp)"
                    % (B, nnz),
            "batch": B, "model_ms": ms_model, "assemble_ms": ms_asm,
            "value": B / ((ms_model + ms_asm) * 1e-3), "unit": "QP builds/s",
            "roofline": {"kernel": "lambda_kernel<BuildFn> (build_one: one lane per QP, element-major outputs, coalesced over the batch)",
                         "bound": "hbm", "achieved": ach, "peak": c["peak"], "unit": "GB/s", "frac": ach / c["peak"],
                         "traffic": None,
                         "peak_source": c["peak_src"], "algorithmic_bytes_per_qp": (out_bytes + in_bytes) / B},
            "model_kernels_gbs": model_bytes / (ms_model * 1e-3) / 1e9}


def record_configs1(c):
    """BASELINE configs[1]: batch 1024 vanilla lateral MPC QPs, H = 20, ONE shared linearisation, f64, one GPU."""
    a, torch, workloads, roofline, be = c["a"], c["torch"], c["workloads"], c["roofline"], c["be"]
    dev = c["dev"]
    Bq, N = 1024, 20
    sets = [workloads.lateral_vanilla_shared(Bq, N=N, seed=300 + i) for i in range(4)]
    dev_in = [(torch.as_tensor(w.x0).to(dev), torch.as_tensor(w.xr).to(dev)) for w in sets]
    host_in = [(torch.as_tensor(w.x0).pin_memory(), torch.as_tensor(w.xr).pin_memory()) for w in sets]
    ctl = sets[0].make_controller(rho=a.rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=False)
    s = ctl.solver
    its = []

    def step(i):
        x0, xr = dev_in[i % 4]
        return ctl.solve_batch(x0, xr, None, want_x=False, reuse=True)

    for i in range(4):
        its.append(step(i).info.iter.double().clone())
    steps = 20
    n0 = be.launch_count()
    ms = c["timed"](step, steps)
    launches = (be.launch_count() - n0) / steps
    out_host = torch.empty((Bq, N, 1), dtype=torch.float64).pin_memory()

    def e2e_step(i):
        hx0, hxr = host_in[i % 4]
        r = ctl.solve_batch(hx0.to(dev, non_blocking=True), hxr.to(dev, non_blocking=True), None, want_x=False, reuse=True)
        out_host.copy_(r.u, non_blocking=True)
        torch.cuda.synchronize()

    e2e_step(0)
    e2e_ms = c["timed"](e2e_step, steps)
    # the ADMM loop alone (one launch of admm_dense_kernel when the batch shares its KKT matrix)
    loop_ms = []
    for i in range(4):
        step(i); s.cold_start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(); s.solve(); e1.record(); torch.cuda.synchronize()
        loop_ms.append(e0.elapsed_time(e1))
    it_all = torch.stack(its)
    mean_it, max_it = it_all.mean().item(), it_all.max(dim=1).values.mean().item()
    flops = roofline.dense_flops_per_qp_iteration(N, 4, 1) * Bq * mean_it
    ach = flops / (float(np.mean(loop_ms)) * 1e-3) / 1e12
    rec = {"what": "BASELINE configs[1]: batch 1024 vanilla lateral MPC QPs, H=20, one shared linearisation (one speed), f64, 1 GPU; "
                   "step = QP build + Ruiz + factor + shared-KKT inverse + ADMM (admm_dense_kernel, one launch) + gather",
           "batch": Bq, "steps": steps, "ms_per_step": ms / steps, "value": Bq * steps / (ms * 1e-3), "unit": UNIT,
           "e2e": {"value": Bq * steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": Bq * 8 * 8,
                   "d2h_bytes_per_step": Bq * N * 8},
           "mean_admm_iterations": mean_it, "max_admm_iterations": max_it, "gpu_launches_per_step": launches,
           "admm_loop_ms": float(np.mean(loop_ms)),
           "us_per_iteration_of_the_slowest_qp": 1e3 * float(np.mean(loop_ms)) / max_it,
           "roofline": {"kernel": "admm_dense_kernel (explicit reduced-KKT inverse, DMMA m8n8k4 GEMM over the right-hand sides)",
                        "bound": "tensor", "achieved": ach, "peak": roofline.FP64_TENSOR_PEAK_TFLOPS, "unit": "TFLOP/s",
                        "frac": ach / roofline.FP64_TENSOR_PEAK_TFLOPS, "traffic": None,
                        "peak_source": "NVIDIA B200 FP64 tensor specification (MEASURED_PEAKS.json has no FP64 figure)",
                        "note": "latency-bound by construction: 1024 QPs are 128 CTAs of 8 QPs, and the launch lasts as long as "
                                "the slowest QP needs (max vs mean iterations above); the figure of merit is the time per "
                                "iteration of one QP"}}
    if not a.no_cpu_baseline:
        big = workloads.lateral_vanilla_shared(16 * Bq, N=N, seed=300)      # 16 batches of the same workload: a sample long enough to time
        v, cores, cit, csolved, dt = cpu_solve(cpu_lateral_inputs(big), a.rho, a.eps, repeats=2)
        rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "16 batches of 1024 QPs of the same workload (oracle/osqp_admm.c, OpenMP over QPs, %.3f s); "
                                         "mean %.1f ADMM iterations, %.3f solved" % (dt, cit, csolved)}
    return rec


def record_configs3(c):
    """BASELINE configs[3]: batch 8192, H = 100, combined longitudinal-lateral dynamics model linearised per stage, f64."""
    a, torch, pm, workloads, roofline, vehicle_models = c["a"], c["torch"], c["pm"], c["workloads"], c["roofline"], c["vehicle_models"]
    Bq, N, rho = 8192, 100, 0.1
    wl = workloads.DynamicWorkload(Bq, N=N, seed=1)
    veh = vehicle_models.Vehicle_Dynamics(dt=wl.dt)
    A, Bm, g, _, ld = workloads.rollout_linearisation(veh, wl.x0, wl.u0, N)
    Xr = wl.references()
    s = pm.BatchSolver(N, 6, 2, wl.Q, wl.QN, wl.R, wl.xmin, wl.xmax, wl.umin, wl.umax, dtype=torch.float64, time_varying=True,
                       stage_reference=True, capacity=Bq, rho=rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=False)
    xr = torch.as_tensor(Xr).transpose(1, 2).contiguous()
    s.batch = Bq
    x_em = s.to_element_major(wl.x0, Bq, 6, ld); xr_em = s.to_element_major(xr, Bq, (N + 1) * 6, ld)

    def step(i):
        s.setup(A, Bm, g, x_em, xr_em, element_major=True)
        s.solve()
        return s.solution(want_x=False, want_u=True, reuse=True)

    step(0)
    steps = 3
    ms = c["timed"](step, steps)
    inf = s.info()
    mean_it = inf.iter.double().mean().item()
    ms_build = c["timed"](lambda i: workloads.rollout_linearisation(veh, wl.x0, wl.u0, N), 2) / 2
    s.setup(A, Bm, g, x_em, xr_em, element_major=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record(); s.solve(); e1.record(); torch.cuda.synchronize()
    loop_ms = e0.elapsed_time(e1)
    bqi = roofline.admm_bytes_per_qp_iteration(N, 6, 2, False, 8, time_varying=True)
    ach = bqi * Bq * mean_it / (loop_ms * 1e-3) / 1e9
    rec = {"what": "BASELINE configs[3]: batch 8192, H=100, combined longitudinal-lateral dynamics model linearised per stage "
                   "along each vehicle's prediction (time-varying), f64, rho=0.1 (OSQP default), 1 GPU; step = Ruiz + factor + ADMM "
                   "+ gather (the rollout + linearisation of the 8192 x 100 stage models is timed apart: qp_build_ms)",
           "batch": Bq, "horizon": N, "steps": steps, "ms_per_step": ms / steps, "value": Bq * steps / (ms * 1e-3), "unit": UNIT,
           "qp_build_ms": ms_build, "mean_admm_iterations": mean_it,
           "fraction_solved": (inf.status_val == 1).double().mean().item(), "admm_loop_ms": loop_ms,
           "roofline": {"kernel": "admm_cta_kernel (CTA per tile, record + stage model staged by TMA; one launch per check interval, unsolved QPs compacted between launches)", "bound": "hbm",
                        "achieved": ach, "peak": c["peak"], "unit": "GB/s", "frac": ach / c["peak"],
                        "traffic": ncu_traffic("admm_cta_kernel/configs3")[0], "traffic_unit": "bytes per solve (all admm_cta launches of the chunked loop)",
                        "traffic_source": ncu_traffic("admm_cta_kernel/configs3")[1],
                        "peak_source": c["peak_src"], "algorithmic_bytes_per_qp_iteration": bqi}}
    if not a.no_cpu_baseline:
        from oracle import workload_qp
        idx = np.arange(0, Bq, Bq // 512)[:512]
        Ab = s._bm(A, Bq, N * 36).reshape(Bq, N, 6, 6)[idx].cpu().numpy()
        Bb = s._bm(Bm, Bq, N * 12).reshape(Bq, N, 6, 2)[idx].cpu().numpy()
        gb = s._bm(g, Bq, N * 6).reshape(Bq, N, 6)[idx].cpu().numpy()
        sub = workloads.DynamicWorkload(Bq, N=N, seed=1)
        sub.x0 = wl.x0[idx]
        v, cores, cit, csolved, dt = cpu_solve(workload_qp.dynamic_batch_csc(sub, Ab, Bb, gb, Xr[idx], np.arange(idx.size)), rho, a.eps)
        rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                               "sample": "%d of the same QPs (every %dth; oracle/osqp_admm.c, OpenMP over QPs, %.2f s); mean %.1f "
                                         "ADMM iterations, %.3f solved" % (idx.size, Bq // 512, dt, cit, csolved)}
    return rec


def record_configs4(c):
    """BASELINE configs[4]: closed-loop sweep — random initial states / speeds, warm-started ADMM, sharded over the GPUs."""
    a, torch, dist, workloads, roofline, sharding = c["a"], c["torch"], c["dist"], c["workloads"], c["roofline"], c["sharding"]
    world, rank, dev = c["world"], c["rank"], c["dev"]
    Bs, steps, N = a.sweep_scenarios, a.sweep_steps, a.horizon
    wl = workloads.lateral_closed_loop_sweep(Bs, N=N, seed=9000 + rank)
    x0, xr, sp = (torch.as_tensor(v).to(dev, torch.float64) for v in (wl.x0, wl.xr, wl.speed))
    ctl = wl.make_controller(capacity=Bs, rho=a.rho, eps_abs=a.eps, eps_rel=a.eps, warm_start=True)
    ctl.closed_loop_batch(x0, xr, sp, steps=3, record=False)            # warm-up: allocations, the learnt re-tile point
    c["barrier"]()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, us, its = ctl.closed_loop_batch(x0, xr, sp, steps=steps, record=False)
    u_last = sharding.gather_controls(us[-1], Bs * world) if world > 1 else us[-1]      # the final gather
    e1.record()
    c["barrier"]()
    ms = c["max_over_ranks"](e0.elapsed_time(e1))[0]
    tot_it = its.double().sum().item()
    mean_it = tot_it / (Bs * steps)
    bqi = roofline.admm_bytes_per_qp_iteration(N, 5, 1, True, 8)
    ach = bqi * tot_it / (ms * 1e-3) / 1e9
    rec = {"what": "BASELINE configs[4]: closed-loop sweep, %d scenarios per GPU x %d GPU(s) = %d scenarios, %d MPC steps each "
                   "(step 0: setup + cold solve; then prob.update(l,u) + warm-started solve + plant step), random initial states, "
                   "references and speeds (workloads.lateral_closed_loop_sweep), f64; no collective inside the sweep, one all_gather of the last controls"
                   % (Bs, world, Bs * world, steps),
           "scenarios_per_gpu": Bs, "scenarios": Bs * world, "closed_loop_steps": steps, "n_gpus": world,
           "wall_ms": ms, "ms_per_closed_loop_step": ms / steps, "value": Bs * world * steps / (ms * 1e-3), "unit": UNIT,
           "mean_admm_iterations": mean_it, "u_last_shape": list(u_last.shape), "scaling": "weak",
           "roofline": {"kernel": "the whole closed-loop step (ADMM kernels + update / gather / plant kernels)", "bound": "hbm",
                        "achieved": ach, "peak": c["peak"], "unit": "GB/s", "frac": ach / c["peak"],
                        "traffic": None,
                        "peak_source": c["peak_src"], "algorithmic_bytes_per_qp_iteration": bqi,
                        "note": "ADMM record traffic only, over the wall time of the whole sweep (a lower bound on the kernels' own rate)"}}
    if rank == 0 and not a.no_cpu_baseline:
        from oracle import c_oracle, ref_qp, workload_qp
        nb, nsteps = 1024, 50
        sub = workloads.lateral_closed_loop_sweep(nb, N=N, seed=9000)
        Pu, A0, Pv, q, Av, l, u, perm = workload_qp.lateral_batch_csc(sub)
        Ad, Bd = workload_qp.lateral_models(sub.speed)
        At, Bt, _ = ref_qp.augment_increment(Ad, Bd, None)
        t0 = time.perf_counter()
        it, st, ua, traj, used = c_oracle.closed_loop_batch(Pu, A0, Pv, q, Av, l, u, At, Bt, sub.x0, nsteps, (N + 1) * 5, perm=perm,
                                                            nthreads=host_cores(), rho=a.rho, eps_abs=a.eps, eps_rel=a.eps)
        dt = time.perf_counter() - t0
        rec["cpu_baseline"] = {"value": nb * nsteps / dt, "unit": UNIT, "cores": used, "kind": "port",
                               "sample": "%d scenarios x %d closed-loop steps of the same workload (oracle_closed_loop_batch: setup "
                                         "once, update + warm-started solve + plant step; OpenMP over scenarios, %.2f s); mean %.1f "
                                         "ADMM iterations, %.3f solved" % (nb, nsteps, dt, float(it.mean()), float((st == 1).mean()))}
    return rec


def record_fp32(c):
    """configs[2] is named FP32: the same QPs in f32 and in f64 at rho = 0.1 (the largest rho at which f32 reaches OSQP's own
    termination test, DESIGN.md §6) — iteration counts, throughput and the deviation of the f32 optimum."""
    a, torch, workloads = c["a"], c["torch"], c["workloads"]
    dev = c["dev"]
    Bq, N, rho, eps = 16384, a.horizon, 0.1, 1e-3
    out = {}
    for name, dt in (("f32", torch.float32), ("f64", torch.float64)):
        wl = workloads.lateral_slack_increment(Bq, N=N, seed=31, dtype=dt)
        x0, xr, sp = (torch.as_tensor(v).to(dev, dt) for v in (wl.x0, wl.xr, wl.speed))
        ctl = wl.make_controller(capacity=Bq, rho=rho, eps_abs=eps, eps_rel=eps, warm_start=False)
        step = lambda i: ctl.solve_batch(x0, xr, sp, want_x=True, reuse=True)
        step(0)
        ms = c["timed"](step, 2) / 2
        r = step(0)
        out[name] = dict(ms=ms, x=r.x.double().clone(), it=r.info.iter.double().mean().item(),
                         solved=(r.info.status_val == 1).double().mean().item())
        del ctl
    ok = (out["f32"]["x"] - out["f64"]["x"]).abs().amax(dim=1) / out["f64"]["x"].abs().amax(dim=1)
    return {"what": "configs[2] workload (16384 QPs) solved in f32 and in f64 at rho=0.1, eps=1e-3 (OSQP defaults): f32 is a "
                    "supported mode only where its round-off (multiplied by rho_eq = 1e3 rho into the duals) stays below the "
                    "termination tolerance; the headline runs f64 at rho=%g" % a.rho,
            "batch": Bq, "rho": rho, "eps": eps,
            "f32": {"ms_per_step": out["f32"]["ms"], "value": Bq / (out["f32"]["ms"] * 1e-3), "unit": UNIT,
                    "mean_admm_iterations": out["f32"]["it"], "fraction_solved": out["f32"]["solved"]},
            "f64": {"ms_per_step": out["f64"]["ms"], "value": Bq / (out["f64"]["ms"] * 1e-3), "unit": UNIT,
                    "mean_admm_iterations": out["f64"]["it"], "fraction_solved": out["f64"]["solved"]},
            "f32_vs_f64_primal_rel_deviation": {"max": ok.max().item(), "median": ok.median().item(),
                                                "fraction_within_1e-4": (ok < 1e-4).double().mean().item()}}


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
