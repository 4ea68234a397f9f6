/* mpc_b200 — C ABI of the B200-native batched linear-MPC QP path.
 *
 * This is the drop-in boundary for the hot path of hynkis/Python-MPC: "cast the MPC problem
 * to a QP and solve it with OSQP".  The reference is pure Python; the natural binding is
 * ctypes (see INTEGRATION.md).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns 0 on success or a negative
 *     MPCB_E_* code, with a message available from mpcb_last_error();
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls are
 *     asynchronous on that stream unless stated otherwise;
 *   - DEVICE arrays are element-major ("SoA"):  a[e * ld + b], b = QP index, ld >= batch;
 *     matrices inside an element range are row-major; dtype is the solver's (float/double);
 *   - HOST arrays (the *_host entry points) are batch-major row-major, i.e. exactly the
 *     numpy arrays the reference builds: a[b * elems + e].
 */
#ifndef MPC_B200_H
#define MPC_B200_H
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPCB_MAX_NX 10
#define MPCB_MAX_NU 2

enum { MPCB_F32 = 0, MPCB_F64 = 1 };

enum {
    MPCB_OK = 0,
    MPCB_E_ARG = -1,        /* invalid argument / unsupported shape */
    MPCB_E_CUDA = -2,       /* CUDA runtime error */
    MPCB_E_STATE = -3,      /* call order violated (e.g. solve before setup) */
    MPCB_E_ALLOC = -4
};

/* status values written per QP — identical to OSQP's status_val (osqp/include/constants.h) */
enum {
    MPCB_SOLVED = 1,
    MPCB_SOLVED_INACCURATE = 2,
    MPCB_PRIMAL_INFEASIBLE_INACCURATE = 3,
    MPCB_DUAL_INFEASIBLE_INACCURATE = 4,
    MPCB_MAX_ITER_REACHED = -2,
    MPCB_PRIMAL_INFEASIBLE = -3,   /* certificate of auxil.c: is_primal_infeasible found at a termination test */
    MPCB_DUAL_INFEASIBLE = -4,     /* certificate of auxil.c: is_dual_infeasible */
    MPCB_NON_CVX = -7,
    MPCB_UNSOLVED = -10
};

/* The stage-structured MPC problem family (all formulations of the reference):
 *   min  sum_k 1/2 x_k'Q_k x_k - (Q_k xr_k)'x_k + 1/2 u_k'R u_k + 1/2 s_k'W s_k
 *   s.t. -x_0 = -x_init ;  A_k x_k + B_k u_k - x_{k+1} = -g_k
 *        xmin <= x_k + S s_k <= xmax ;  umin <= u_k <= umax
 * with diagonal Q, QN, R, W, S — Control/MPC/mpc_kinematics.py:150-213 (vanilla),
 * Control/MPC/mpc_dynamics.py:156-252 (time-varying), :284-402 (delta-u, after augmentation),
 * vehicle_lateral_mpc_slack_increment.py:32-121 (slack + delta-u). */
typedef struct mpcb_problem {
    int horizon;            /* N */
    int nx;                 /* stage state dimension (after delta-u augmentation) */
    int nu;                 /* stage input dimension */
    int slack;              /* 1: slack variables s_k on the state bounds */
    int dtype;              /* MPCB_F32 | MPCB_F64 */
    int time_varying;       /* 1: model arrays hold one (A_k,B_k,g_k) per stage (Ad_list/Bd_list/gd_list) */
    int shared_model;       /* 1: ONE linearisation shared by the whole batch (model arrays have ld = 1) */
    int stage_reference;    /* 1: Xr holds N+1 stage references (Xr[:,k]); 0: one xr per QP */
    double Q[MPCB_MAX_NX], QN[MPCB_MAX_NX], R[MPCB_MAX_NU];
    double W[MPCB_MAX_NX];  /* slack cost   (W_tilda == WN) */
    double S[MPCB_MAX_NX];  /* slack coupling (weight_slack_tilda) */
    double xmin[MPCB_MAX_NX], xmax[MPCB_MAX_NX], umin[MPCB_MAX_NU], umax[MPCB_MAX_NU];
} mpcb_problem;

/* OSQP settings honoured by this path (adaptive_rho and polish are always off). */
typedef struct mpcb_settings {
    double rho, sigma, alpha, eps_abs, eps_rel, eps_prim_inf, eps_dual_inf;
    int max_iter, scaling, check_termination, warm_start;
} mpcb_settings;

typedef struct mpcb_solver mpcb_solver;

const char* mpcb_last_error(void);
int mpcb_version(void);
void mpcb_default_settings(mpcb_settings* s);        /* OSQP 0.6 defaults, adaptive_rho/polish off */

/* ---- solver object: replaces `prob = osqp.OSQP()` for a batch of `capacity` QPs ---------- */
int mpcb_create(const mpcb_problem* prob, const mpcb_settings* settings, int capacity, mpcb_solver** out);
void mpcb_destroy(mpcb_solver* s);
int mpcb_set_settings(mpcb_solver* s, const mpcb_settings* settings);
int mpcb_set_stage_bounds(mpcb_solver* s, const double* xbox_host /* [(N+1)][2][nx] lo,hi */);
size_t mpcb_workspace_bytes(const mpcb_solver* s);
int mpcb_num_variables(const mpcb_solver* s);         /* (N+1)nx + N nu + (N+1)ns */
int mpcb_num_constraints(const mpcb_solver* s);       /* 2(N+1)nx + N nu */

/* replaces `prob.setup(P, q, A, l, u, ...)` (mpc_kinematics.py:206, mpc_dynamics.py:249/399,
 * vehicle_lateral_mpc_slack_increment.py:121): Ruiz scaling + cached KKT factorisation.
 * Device pointers are BORROWED until the next setup/update call.
 *   Ad [(N*)nx*nx], Bd [(N*)nx*nu], gd [(N*)nx] or NULL, x_init [nx], Xr [(N+1)*nx or nx] */
int mpcb_setup(mpcb_solver* s, int batch, size_t ld, const void* Ad, const void* Bd, const void* gd,
               const void* x_init, const void* Xr, void* stream);
/* replaces the q / equality part of `prob.update(q=q_new, l=l_new, u=u_new)`
 * (vehicle_lateral_mpc_slack_increment.py:237, and :267-269 for the initial-state rows):
 * new initial state / reference under the existing scaling and factorisation. */
int mpcb_update(mpcb_solver* s, const void* x_init, const void* Xr);
/* replaces the INEQUALITY part of `prob.update(l=l_new, u=u_new)`: new state / input bounds after setup
 * (vehicle_lateral_mpc_slack_increment.py:158-172 tightens xmin_tilda[3] for steps 401..900, applied at :237).
 * osqp_update_bounds semantics (osqp.c): the new bounds are scaled with the EXISTING E, the per-row rho type
 * (equality / inequality / unbounded, auxil.c: update_rho_vec) is re-evaluated per QP and the KKT matrix is
 * refactored only for QPs in which a row changed type; iterates (x, z, y) are kept for the warm start.
 * HOST arrays; NULL = unchanged.  xmin/xmax [nx], umin/umax [nu]; xbox [(N+1)][2][nx] per-stage state boxes
 * (replaces the boxes of mpcb_set_stage_bounds).  Returns MPCB_E_ARG if a lower bound exceeds its upper bound. */
int mpcb_update_bounds(mpcb_solver* s, const double* xmin, const double* xmax, const double* umin,
                       const double* umax, const double* xbox, void* stream);
/* replaces `res = prob.solve()`: the ADMM loop. */
int mpcb_solve(mpcb_solver* s, void* stream);
/* one iterate-exact building block for tests: run exactly `iters` ADMM iterations, no termination test */
int mpcb_iterate(mpcb_solver* s, int iters, void* stream);
int mpcb_cold_start(mpcb_solver* s, void* stream);

/* replaces `res.x` / `res.y` / `res.info.*`: outputs are batch-major row-major DEVICE arrays in
 * the reference's ordering x = (x_0..x_N, u_0..u_{N-1}, s_0..s_N); any pointer may be NULL.
 *   x_out [batch][nvar], y_out [batch][ncon], u_out [batch][N*nu], iter/status [batch] */
int mpcb_get_solution(mpcb_solver* s, void* x_out, void* y_out, void* u_out, void* stream);
int mpcb_get_info(mpcb_solver* s, int* iter_out, int* status_out, void* pri_res_out, void* dua_res_out,
                  void* stream);

/* HOST front door (what a reference user calls): numpy-layout host buffers in, host buffers out;
 * host<->device copies, layout change, setup, solve and gather all inside, synchronous.
 *   Ad [batch|1][(N*)nx*nx] ... x_out [batch][nvar], u_out [batch][N*nu] */
int mpcb_solve_host(mpcb_solver* s, int batch, const void* Ad, const void* Bd, const void* gd,
                    const void* x_init, const void* Xr, void* x_out, void* u_out, int* iter_out,
                    int* status_out);

/* ---- QP build kernels ("cast MPC problem to a QP") ---------------------------------------- */
/* Lateral bicycle model, discretised per vehicle speed (ZOH, matrix exponential):
 * state [side-slip, yaw-rate, yaw-error, lateral-error], input steer.  Produces the per-QP
 * Ad_sys/Bd_sys that vehicle_lateral_mpc_slack_increment.py:32-43 hard-codes for one speed.
 *   speed [batch] -> Ad [16][ld], Bd [4][ld]   params: m, l_f, l_r, Iz, Cf, Cr, dt */
int mpcb_lateral_discretize(int dtype, int batch, size_t ld, const void* speed, const double* params7,
                            void* Ad, void* Bd, void* stream);
/* Vehicle_Dynamics.get_dynamics_model (Vehicle_Dynamics/vehicle_models.py:52-340), batched:
 *   x [6][ld], u [2][ld] -> Ad [36][ld], Bd [12][ld], gd [6][ld]; params: m,l_f,l_r,Iz,C_d,A_f,C_roll,dt */
int mpcb_dynamics_linearize(int dtype, int batch, size_t ld, const void* x, const void* u,
                            const double* params8, void* Ad, void* Bd, void* gd, void* stream);
/* Vehicle_Kinematics.get_kinematics_model (vehicle_models.py:835-863), batched:
 *   x [4][ld], u [2][ld] -> A [16][ld], B [8][ld], C [4][ld]; params: wheelbase, dt */
int mpcb_kinematics_linearize(int dtype, int batch, size_t ld, const void* x, const void* u,
                              const double* params2, void* Ad, void* Bd, void* gd, void* stream);
/* Vehicle_Dynamics.update_dynamics_model (vehicle_models.py:343-482), batched: one explicit Euler step of the nonlinear
 * single-track model with Pacejka tyres (the simulated vehicle of the scripts; also extends the prediction by one stage,
 * mpc_dynamics.py:607):  x [6][ld], u [2][ld] -> x_next [6][ld], alpha [2][ld] (front / rear side slip; may be NULL).
 * params as for mpcb_dynamics_linearize */
int mpcb_dynamics_step(int dtype, int batch, size_t ld, const void* x, const void* u, const double* params8,
                       void* x_next, void* alpha, void* stream);
/* Vehicle_Kinematics.update_kinematics_model (vehicle_models.py:866-882), batched (the yaw update uses the NEW speed,
 * like the reference's in-place update):  x [4][ld], u [2][ld] -> x_next [4][ld]; params: wheelbase, dt */
int mpcb_kinematics_step(int dtype, int batch, size_t ld, const void* x, const void* u, const double* params2,
                         void* x_next, void* stream);
/* delta-u augmentation (mpc_dynamics.py:337-341; vehicle_lateral_mpc_slack_increment.py:48-52):
 *   (Ad [nx*nx], Bd [nx*nu], gd [nx]|NULL) x stages -> A~ [(nx+nu)^2], B~ [(nx+nu)*nu], g~ [nx+nu] */
int mpcb_augment_increment(int dtype, int batch, size_t ld, int nx, int nu, int stages, const void* Ad,
                           const void* Bd, const void* gd, void* At, void* Bt, void* gt, void* stream);
/* Plant update of the closed loop (vehicle_lateral_mpc_slack_increment.py:256-257, mpc_kinematics.py:472,
 * mpc_dynamics.py:590-592): x_next = A x + B u0 + g with the QP's own stage-0 model, batched.
 *   A [nx*nx][ld|1], B [nx*nu][ld|1], g [nx][ld|1] or NULL (element-major; shared_model: ld = 1),
 *   x [nx][ld] element-major in, x_next [nx][ld] out (may alias x), u batch-major [batch][u_stride] whose
 *   first nu entries are the applied input (the head of the control sequence). */
int mpcb_plant_step(int dtype, int batch, size_t ld, int nx, int nu, int shared_model, const void* A, const void* B,
                    const void* g, const void* x, const void* u, int u_stride, void* x_next, void* stream);

/* Explicit P/q/A/l/u assembly in the reference's ordering — the arrays the reference hands to
 * prob.setup()/prob.update() (mpc_kinematics.py:158-203, mpc_dynamics.py:163-245/300-396,
 * vehicle_lateral_mpc_slack_increment.py:79-115).  The solve path never materialises them; this
 * is for inspection, parity tests and users who want the QP itself.  Uses the stage data of the
 * last mpcb_setup/mpcb_update.  Infinite bounds come out as +-OSQP_INFTY (1e30), the values OSQP's
 * Python interface passes on for them.  Element-major outputs (any may be NULL):
 *   Pdiag [nvar][ld], q [nvar][ld], Avals [nnz][ld] (CSC values, pattern below), l/u [ncon][ld] */
int mpcb_build_qp(mpcb_solver* s, void* Pdiag, void* q, void* Avals, void* l, void* u, void* stream);
/* The Ruiz scaling of the last mpcb_setup — OSQP's D, E and cost scaling c (scaling.c: scale_data) — for inspection and
 * parity tests.  mpcb_update, mpcb_update_bounds and the solves keep it, like OSQP's update.  Batch-major DEVICE arrays
 * in the reference's ordering, any pointer may be NULL:
 *   D_out [batch][nvar] (x_0..x_N, u_0..u_{N-1}, s_0..s_N), E_out [batch][ncon] (dyn_0..dyn_N, bx_0..bx_N,
 *   bu_0..bu_{N-1}), c_out [batch].  Returns MPCB_E_STATE before setup (or after settings that invalidate it). */
int mpcb_get_scaling(mpcb_solver* s, void* D_out, void* E_out, void* c_out, void* stream);
/* CSC pattern of A shared by the whole batch: Ap [nvar+1], Ai [nnz] (host arrays); returns nnz.
 * Pass NULLs to query nnz. */
int mpcb_qp_pattern(const mpcb_solver* s, int* Ap, int* Ai);

/* layout helpers: batch-major row-major <-> element-major */
int mpcb_to_element_major(int dtype, int batch, int elems, size_t ld, const void* src_rowmajor, void* dst, void* stream);
int mpcb_to_batch_major(int dtype, int batch, int elems, size_t ld, const void* src, void* dst_rowmajor, void* stream);

/* Process-wide tunables (also read once from the environment: MPCB_NO_TMA, MPCB_NO_RETILE, MPCB_RETILE_MIN_BATCH,
 * MPCB_NO_CERT, MPCB_NO_DENSE, MPCB_NO_CTA, MPCB_NO_WARP_SETUP, MPCB_NO_FWD_RHS):
 *   "tma"              1 (default) warp-per-tile ADMM kernel with TMA-staged stage records; 0: one lane per QP from global memory
 *   "retile"           1 (default) run the ADMM loop in chunks and re-tile unconverged QPs; 0: one asynchronous launch
 *   "retile_min_batch" smallest batch that is run in chunks (default 4096)
 *   "fwd_rhs"          1 (default) the forward sweeps of the warp-per-tile and lane-per-QP kernels after the first iteration
 *                      of a solve start from the local right-hand side each backward sweep leaves in the stage record and
 *                      read 43 instead of 65 elements of a configs[2] record; 0: they form the whole right-hand side from
 *                      the record (the same arithmetic in another order: results agree to rounding)
 *   "dense"            1 (default) a batch that shares ONE KKT matrix (shared_model, identical Ruiz scaling of every QP, f64,
 *                      (N+1)(nx+nu) <= 128) runs its steady-state iterations as a dense FP64 tensor-core GEMM with the
 *                      explicit inverse of the reduced KKT matrix (admm_dense.cuh); 0: the per-QP kernels
 *   "cta"              1 (default) time-varying problems (one linearisation per stage) and every batch that fits the GPU in
 *                      one wave of CTAs (two per SM: up to 9472 QPs on 148 SMs; shapes with nx + nu <= 8) run their whole
 *                      ADMM loop in the CTA-per-tile kernel (admm_cta.cuh: a warp per component of the stage vector, record
 *                      AND stage model staged by TMA, symmetric block inverse in the records); 2: every problem does; 0: never
 *                      (MPCB_NO_CTA_DEEP=1 in the environment keeps its 5-buffer / one-CTA-per-SM instantiation out)
 *   "warp_setup"       1 (default) Ruiz equilibration with a warp per QP, one lane per stage, scalings in registers over all
 *                      passes (setup_warp.cuh; horizons up to 31); 0: the lane-per-QP kernel that ping-pongs them through HBM
 *   "certificates"     1 (default, OSQP's behaviour) evaluate the primal / dual infeasibility certificates whenever a
 *                      residual test fails; 0: a diagnostic switch that skips them (statuses solved / solved inaccurate /
 *                      maximum iterations reached only), used to measure what the certificates cost
 * MPCB_TRACE=1 in the environment prints the launch sequence of every ADMM loop to stderr (iterations, set size, kernel,
 * a timestamp per launch — tracing drains the stream after every launch, it is a diagnostic, not a product path).
 * MPCB_CHUNK_FINE=<n> sets the work-item length (iterations) the warp-per-tile kernel uses for launches of one to four
 * waves (default 5; 0: always a whole check interval).
 * Returns 0, or MPCB_E_ARG for an unknown name. */
int mpcb_set_option(const char* name, int value);

/* number of kernels this library launched since load (bench.py's gpu_launches) */
long long mpcb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MPC_B200_H */
