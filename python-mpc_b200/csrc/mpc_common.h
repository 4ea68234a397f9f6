// Shared declarations for the mpc_b200 kernels (device + host).
//
// Vocabulary (follows the reference, Control/MPC/*.py): a *QP* is one MPC problem over a
// horizon of N *stages*; its variables are the stage states x_k, inputs u_k and (soft
// constraint formulation) slacks s_k; its rows are the dynamics rows dyn_k and the bound
// rows bx_k / bu_k.  A *batch* is B independent QPs.
//
// Data layout in HBM.
//   INPUTS (borrowed from the caller) are element-major: a[e * ld + b], b = QP index.
//   The solver WORKSPACE is tiled: a tile is 32 consecutive QPs (one warp, lane = b % 32).  Per tile
//   and per stage k there is one contiguous *stage record* of REC elements x 32 lanes
//       rec[((tile*(N+1) + k)*REC + e)*32 + lane]
//       e:  [ D (VS) | E (CS) | Linv (LT) | t (NW) | p (CS) | x (VS) ]
//   holding everything one ADMM sweep needs at that stage: the Ruiz scalings of the stage's
//   variables [s_k | x_k | u_k] (D) and of the rows the stage OWNS [dyn_{k+1} | bx_k | bu_k] (E), the
//   inverse Cholesky block Linv_k, the t slots, the row state p (= z between solves) and the iterates
//   x.  The t slots hold the forward-substitution intermediate t between the forward and the backward
//   sweep, and the stage's local forward right-hand side r^ (written by the backward sweep) between the
//   backward sweep and the next forward sweep.  Because a record is contiguous (REC*256 bytes in FP64)
//   a warp stages it into shared memory with ONE cp.async.bulk, and every access inside the record
//   has a compile-time offset.  The order puts what a forward sweep reads from r^ on in two runs
//   (FA: D_x | D_u | E_dyn, FB: Linv | r^ | p_dyn), so that it streams 2 NX + NU + LT + NW + NX
//   elements of the record instead of all but t.  A small per-QP header holds the dyn_0 rows (E, p, y) and the cost
//   scaling c; the duals y (touched only on entry/exit of a solve) live in a separate tiled array.
//   (The u / bu slots of stage N and its dyn_{N+1} slot are unused padding.)  The reference's
//   ordering (x_0..x_N, u_0..u_{N-1}, s_0..s_N) is produced by the gather kernels in mpc_b200.cu.
#pragma once
#include <math.h>
#include <stddef.h>

#ifdef __CUDACC__
#define MPCB_HD __host__ __device__ __forceinline__
#else
#define MPCB_HD inline
#endif

namespace mpcb {

constexpr int MAXNX = 10;
constexpr int MAXNU = 2;

// osqp/include/constants.h (0.6.x) — the same constants as oracle/osqp_admm.{py,c}
constexpr double kOsqpInfty = 1e30;
constexpr double kRhoMin = 1e-6;
constexpr double kRhoMax = 1e6;
constexpr double kRhoEqOverRhoIneq = 1e3;
constexpr double kRhoTol = 1e-4;
constexpr double kMinScaling = 1e-4;
constexpr double kMaxScaling = 1e4;

enum Status : int {
    kSolved = 1,
    kSolvedInaccurate = 2,
    kPrimalInfeasibleInaccurate = 3,
    kDualInfeasibleInaccurate = 4,
    kMaxIterReached = -2,
    kPrimalInfeasible = -3,
    kDualInfeasible = -4,
    kUnsolved = -10,
};

// Everything a per-QP kernel needs, passed by value as the kernel argument.
template <typename T>
struct KParams {
    int N;            // horizon
    int B;            // QPs in this launch
    size_t ld;        // leading dimension of every SoA array
    // ---- model (inputs): A_k (NX*NX), B_k (NX*NU), g_k (NX), row-major inside a stage
    const T* Ad;
    const T* Bd;
    const T* gd;      // may be null (zero)
    int tv;           // 1: one (A,B,g) per stage, stage stride = element count; 0: one per QP
    int model_bs;     // batch stride of the model arrays: 1 per-QP linearisation, 0 one shared linearisation
    const T* x_init;  // (NX)
    const T* Xr;      // (NX) or (N+1)*(NX)
    int xr_tv;
    int xr_smem;      // TMA kernel: keep the per-QP reference in the warp's shared-memory slice (set by the launcher when it fits)
    // ---- weights and bounds, shared by the whole batch (constructor arguments of the controller)
    T Q[MAXNX], QN[MAXNX], R[MAXNU], W[MAXNX], S[MAXNX];
    T xmin[MAXNX], xmax[MAXNX], umin[MAXNU], umax[MAXNU];
    int inf_bounds;   // 1 if any state/input bound of the problem is infinite (batch-uniform)
    const T* xbox;    // optional per-stage state bounds, shared: [(N+1)][2][NX] (mpc_ of mpc_kinematics.py:215); null -> xmin/xmax
    // ---- OSQP settings
    T rho, sigma, alpha, eps_abs, eps_rel, eps_pinf, eps_dinf;
    T rho_c, rho_eq_c; // rho clamped to OSQP's [RHO_MIN, RHO_MAX] and RHO_EQ_OVER_RHO_INEQ times it, evaluated on the host: kernel
                      //   parameters cost a sweep no registers (admm_cta_kernel)
    int max_iter, scaling, check_every;
    int certs;        // 1 (default): evaluate OSQP's infeasibility certificates when a residual test fails; 0: statuses
                      //   solved / solved inaccurate / max-iter only (mpcb_set_option("certificates", 0), a diagnostic switch)
    int warm;         // 0: cold start (x = z = y = 0); 1: keep the iterates already in the workspace
    int fwd_rhs;      // 1 (default): the forward sweeps after the first iteration of a solve start from the local right-hand
                      //   side r^ the previous backward sweep left in the t slots; 0: every forward sweep forms the whole
                      //   right-hand side from the record (mpcb_set_option("fwd_rhs", 0))
    // ---- one CHUNK of the ADMM loop (the host runs the loop in chunks so that unconverged QPs can be re-tiled):
    int it0;          // iterations already done; this launch runs it0+1 .. it_stop.  Rows are explicit (z, y) on
    int it_stop;      //   entry when it0 == 0 and stay in p-form across chunk boundaries (bitwise continuation)
    int chunk_len;    // the TMA kernel hands the launch out as (tile, chunk of chunk_len iterations) work items
    int* tile_prog;   //   [tiles] number of chunks completed per tile (dependency between a tile's consecutive chunks)
    int list_survivors;  // 1: lanes left unsolved at it_stop put themselves on the survivor list
    const int* qp_map;   // workspace slot -> QP index for inputs/outputs (null: identity); set after a re-tiling
    int* survivors;      // QP indices left unsolved by this chunk ...
    int* n_survivors;    // ... and their count
    // ---- workspace (tiled, see the layout note at the top of this file)
    T* rec;           // [tiles][(N+1)][REC][32]   stage records
    T* hdr;           // [tiles][HDR][32]          E, p, y of the dyn_0 rows; cost scaling c
    T* yrows;         // [tiles][(N+1)][CS][32]    duals y between solves
    T* scr;           // [tiles][(N+1)][VS+CS][32] second D/E buffer of the Ruiz ping-pong
    T* scr_hdr;       // [tiles][NX][32]           second buffer for E of dyn_0
    int minv;         // form of the factor block R_F of the records: 0 = Linv_k (lower triangle), 1 = Linv_k' Linv_k (lower triangle of
                      //   the symmetric block inverse — what admm_cta_kernel multiplies with: one product instead of two per stage)
    const T* mdl;     // [tiles][N][A|B|g][32]     time-varying problems: the stage linearisations tiled like the records, so
                      //                           that admm_cta_kernel stages them by TMA next to the record (null otherwise)
    int* iter;        // [B]
    int* status;      // [B]
    T* pri_res;       // [B]
    T* dua_res;       // [B]
};

constexpr int TILE = 32;     // QPs per workspace tile = lanes of a warp

template <int NX_, int NU_, bool SLACK_>
struct Lay {
    static constexpr int NX = NX_, NU = NU_;
    static constexpr bool SLACK = SLACK_;
    static constexpr int NS = SLACK_ ? NX_ : 0;
    static constexpr int NW = NX_ + NU_;
    static constexpr int VS = NX_ + NS + NU_;
    static constexpr int CS = 2 * NX_ + NU_;
    static constexpr int LT = NW * (NW + 1) / 2;
    static constexpr int FS = NX_ * NW;
    static constexpr int OS = 0, OX = NS, OU = NS + NX_;       // variables inside a D / x block
    static constexpr int ODN = 0, OBX = NX_, OBU = 2 * NX_;    // rows inside an E / p block: dyn_{k+1}, bx_k, bu_k
    static constexpr int R_D = 0, R_E = VS, R_F = VS + CS, R_T = R_F + LT, R_P = R_T + NW, R_X = R_P + CS,
                         REC = R_X + VS;
    // the two runs a forward sweep that starts from r^ reads: FA = D_x | D_u | E_dyn, FB = Linv | r^ | p_dyn
    static constexpr int FA = R_D + OX, FA_N = R_E + ODN + NX_ - FA;
    static constexpr int FB = R_F, FB_N = R_P + ODN + NX_ - FB;
    static constexpr int H_E0 = 0, H_P0 = NX_, H_Y0 = 2 * NX_, H_C = 3 * NX_, HDR = 3 * NX_ + 1;
    static MPCB_HD int nvar(int N) { return (N + 1) * NX + N * NU + (N + 1) * NS; }
    static MPCB_HD int ncon(int N) { return 2 * (N + 1) * NX + N * NU; }
};

}  // namespace mpcb
