"""Algorithmic work of the kernels (DESIGN.md §5) — used by bench.py for the roofline figures."""


def admm_elements_per_stage(nx, nu, slack, time_varying=False):
    """Elements one QP moves per stage and per ADMM iteration in the streaming ADMM kernels (stage records, csrc/mpc_common.h).

    warp-per-tile kernel (admm_tma_kernel), steady state:
      forward sweep : D_x, D_u, E_dyn(k+1), the factor block Linv_k, the local right-hand side r^_k, row state p of
                      dyn_{k+1};                                                             writes t_k
      backward sweep: the whole record (scalings, Linv_k, t_k, old p, old x/s/u);            writes new x/s/u, p, r^_k
    time_varying (admm_cta_kernel, which forms the whole right-hand side in its forward sweep):
      forward sweep : scalings of the stage (D_x, D_s, D_u, E_bx, E_bu, E_dyn(k+1)), iterates x_k/s_k/u_k,
                      row state p of bx_k, bu_k, dyn_{k+1}, the factor block;              writes t_k
      backward sweep: scalings (E_dyn(k) instead of E_dyn(k+1)), t_k, the factor block, old x/s/u, old p;  writes new x/s/u, p
      + the stage's own linearisation (A_k, B_k, g_k), read by both sweeps
    """
    ns = nx if slack else 0
    nw, vs, cs = nx + nu, nx + ns + nu, 2 * nx + nu
    fac = nw * (nw + 1) // 2
    coef = 3 * nx + ns + 2 * nu
    if not time_varying:
        reads = (2 * nx + nu + fac + nw + nx) + (coef + vs + cs + fac + nw)
        return reads, nw + vs + cs + nw
    reads = 2 * coef + 2 * vs + 2 * cs + 2 * fac + nw
    reads += 2 * (nx * nx + nx * nu + nx)
    writes = nw + vs + cs
    return reads, writes


def admm_bytes_per_qp_iteration(N, nx, nu, slack, elem_size, time_varying=False):
    r, w = admm_elements_per_stage(nx, nu, slack, time_varying)
    return (N + 1) * (r + w) * elem_size


def dense_flops_per_qp_iteration(N, nx, nu):
    """Shared-KKT dense path (csrc/admm_dense.cuh): one right-hand side through the explicit n_w x n_w inverse of the
    reduced KKT matrix per QP and iteration (multiply-add = 2 flop); the O(n_w) row updates are not counted."""
    nw = (N + 1) * (nx + nu)
    return 2 * nw * nw


# FP64 tensor-core (DMMA) peak of a B200: NVIDIA's specification (40 TFLOP/s); MEASURED_PEAKS.json has no FP64 figure
FP64_TENSOR_PEAK_TFLOPS = 40.0
