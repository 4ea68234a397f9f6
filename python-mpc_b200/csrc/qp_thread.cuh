// Per-QP device functions of the batched MPC-QP solver: one GPU thread (lane) owns one QP, one
// warp owns one workspace tile of 32 QPs (layout: mpc_common.h).
//
//   scale_one   Ruiz equilibration + cost scaling of the stage-structured KKT matrix
//               (OSQP scaling.c: scale_data; paper Algorithm 2)                      -> D, E, c
//   factor_one  cached factorisation of the reduced KKT matrix
//               M = P^ + sigma I + A^' diag(rho) A^   (block tridiagonal over stages after the
//               slack variables are eliminated in closed form) as a block-bidiagonal Cholesky;
//               stores the inverse diagonal blocks Linv_k only: the coupling blocks
//               F_k = C_k Linv_k' are re-applied from the model and the scalings    -> Linv
//   admm_fwd_stage / admm_bwd_stage / admm_test_stage / admm_exit_stage
//               one stage of the OSQP ADMM loop (osqp.c: update_xz_tilde / update_x / update_z /
//               update_y; auxil.c: check_termination) with fixed rho / sigma / alpha.  The loop that
//               drives them (and stages the records through shared memory with TMA bulk copies on
//               the GPU) is admm_loop in admm_kernel.cuh.
//
// Replaces, for a batch, the per-QP `osqp.OSQP().setup(P, q, A, l, u); prob.solve()` of
//   /root/reference/Control/MPC/mpc_kinematics.py:205-211
//   /root/reference/Control/MPC/mpc_dynamics.py:248-252, 398-402
//   /root/reference/vehicle_lateral_mpc_slack_increment.py:118-121, 237-248
// The QP itself (P, q, A, l, u of those files) is never materialised on this path: the
// kernels read the stage data (A_k, B_k, g_k, x_init, Xr, weights, bounds) and apply the
// structured operators directly.  build_one (mpc_b200.cu) materialises it for inspection/parity.
//
// All functions are __host__ __device__ so that tests/emu can run the identical code on the
// CPU of the (GPU-less) build container; the product only ever launches them as kernels.
#pragma once
#include "mpc_common.h"

namespace mpcb {

MPCB_HD float msqrt(float v) { return sqrtf(v); }
MPCB_HD double msqrt(double v) { return sqrt(v); }
template <typename T> MPCB_HD T tmax(T a, T b) { return a > b ? a : b; }
template <typename T> MPCB_HD T tmin(T a, T b) { return a < b ? a : b; }
template <typename T> MPCB_HD T tabs(T a) { return a < (T)0 ? -a : a; }
template <typename T> MPCB_HD T limit_scaling(T v) {
    v = v < (T)kMinScaling ? (T)1 : v;
    return v > (T)kMaxScaling ? (T)kMaxScaling : v;
}
template <typename T> MPCB_HD T clip_infty(T v) {
    return tmin(tmax(v, (T)-kOsqpInfty), (T)kOsqpInfty);
}
// auxil.c: set_rho_vec, evaluated on the scaled bounds of one row
template <typename T> MPCB_HD T row_rho(T l, T u, T rho, T rho_eq) {
    if (l < (T)(-kOsqpInfty * kMinScaling) && u > (T)(kOsqpInfty * kMinScaling)) return (T)kRhoMin;
    if (u - l < (T)kRhoTol) return rho_eq;
    return rho;
}
// same, when the host has established that no bound of the problem is infinite (batch-uniform flag)
template <typename T> MPCB_HD T row_rho(bool inf_possible, T l, T u, T rho, T rho_eq) {
    if (inf_possible) return row_rho(l, u, rho, rho_eq);
    return (u - l < (T)kRhoTol) ? rho_eq : rho;
}
template <typename T> MPCB_HD T clamp_rho(T rho) {
    return tmin(tmax(rho, (T)kRhoMin), (T)kRhoMax);
}
// 1/v for a positive, well-scaled v.  FP64 division costs ~25 instructions on the GPU; a single
// hardware seed with two Newton steps is exact to the last bit or two and costs 5.
MPCB_HD float fast_rcp(float v) { return 1.0f / v; }
MPCB_HD double fast_rcp(double v) {
#ifdef __CUDA_ARCH__
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));      // MUFU.RCP64H seed, ~20 bits
    r = r * (2.0 - v * r);
    r = r * (2.0 - v * r);
    return r;
#else
    return 1.0 / v;
#endif
}

// 1/sqrt(v) for a positive, well-scaled v (the Ruiz norms are clamped to [1e-4, 1e4]).  FP64 sqrt followed by a
// division is ~70 instructions on the GPU; the hardware seed (MUFU.RSQ64H, ~22 bits) with two Newton steps in
// residual form is 10 and exact to the last bit or two.
MPCB_HD float fast_rsqrt(float v) { return 1.0f / sqrtf(v); }
MPCB_HD double fast_rsqrt(double v) {
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(v));
    double e = fma(-(v * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-(v * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    return y;
#else
    return 1.0 / sqrt(v);
#endif
}

template <typename T, typename L>
struct Model {
    T A[L::NX][L::NX];
    T B[L::NX][L::NU];
};
// affine term g_k[i] of the stage model: read where it is used (rows dyn_{k+1}) instead of living in registers next
// to A and B — the lateral models have none, and the ADMM sweeps sit at the register limit
template <typename T, typename L>
MPCB_HD T model_g(const KParams<T>& p, int b, int k, int i) {
    if (!p.gd) return (T)0;
    const size_t og = p.tv ? (size_t)k * L::NX : 0;
    return p.model_bs ? p.gd[(og + i) * p.ld + b] : p.gd[og + i];
}

template <typename T, typename L>
MPCB_HD void load_model(const KParams<T>& p, int b, int k, Model<T, L>& m) {
    constexpr int NX = L::NX, NU = L::NU;
    const size_t bo = p.model_bs ? (size_t)b : 0;
    const size_t ld = p.model_bs ? p.ld : 1;
    const size_t oa = p.tv ? (size_t)k * NX * NX : 0, ob = p.tv ? (size_t)k * NX * NU : 0;
#pragma unroll
    for (int i = 0; i < NX; ++i) {
#pragma unroll
        for (int j = 0; j < NX; ++j) m.A[i][j] = p.Ad[(oa + i * NX + j) * ld + bo];
#pragma unroll
        for (int j = 0; j < NU; ++j) m.B[i][j] = p.Bd[(ob + i * NU + j) * ld + bo];
    }
}

template <typename T, typename L>
MPCB_HD void stage_box(const KParams<T>& p, int k, T* lo, T* hi) {
#pragma unroll
    for (int i = 0; i < L::NX; ++i) {
        T a = p.xbox ? p.xbox[(k * 2 + 0) * L::NX + i] : p.xmin[i];
        T c = p.xbox ? p.xbox[(k * 2 + 1) * L::NX + i] : p.xmax[i];
        lo[i] = a;        // already clipped to +-OSQP_INFTY on the host (make_params / mpcb_set_stage_bounds)
        hi[i] = c;
    }
}

// ---- addressing of the tiled workspace (one lane) ------------------------------------------
template <typename T, typename L>
struct Ws {
    T* rec;      // record of stage 0 of this lane; stage k at rec + k*REC*32, element e at [e*32]
    T* hdr;
    T* y;        // y rows of stage 0; stage k at y + k*CS*32
    T* scr;
    T* scr_hdr;
    MPCB_HD Ws(const KParams<T>& p, int b) {
        const size_t tile = (size_t)(b >> 5), lane = (size_t)(b & 31);
        const size_t S1 = (size_t)(p.N + 1);
        rec = p.rec + tile * S1 * L::REC * TILE + lane;
        hdr = p.hdr + tile * L::HDR * TILE + lane;
        y = p.yrows + tile * S1 * L::CS * TILE + lane;
        scr = p.scr + tile * S1 * (L::VS + L::CS) * TILE + lane;
        scr_hdr = p.scr_hdr + tile * L::NX * TILE + lane;
    }
    MPCB_HD T* R(int k) const { return rec + (size_t)k * L::REC * TILE; }
    MPCB_HD T* Y(int k) const { return y + (size_t)k * L::CS * TILE; }
    MPCB_HD T* S(int k) const { return scr + (size_t)k * (L::VS + L::CS) * TILE; }
};
#define MPCB_AT(ptr, e) (ptr)[(e) * TILE]

// ------------------------------------------------------------------------------------------
// Ruiz equilibration (scaling.c: scale_data).  The scaled matrices are never stored: entry
// (i,j) of the scaled A is E_i * A_ij * D_j with the running D, E.  Stage k handles the columns
// x_k, s_k, u_k and the rows it owns (dyn_{k+1}, bx_k, bu_k; dyn_0 at k = 0).
// ------------------------------------------------------------------------------------------
// The scalings of one stage: D of its variables [x | s | u], E of the rows it owns [dyn_{k+1} | bx | bu].
template <typename T, typename L>
struct ScaleStage {
    T Dx[L::NX], Dsl[L::NX], Du[L::NU], Ebx[L::NX], Ebu[L::NU], Edn[L::NX];
};
// One Ruiz pass for ONE stage (scaling.c: scale_data, one iteration of the loop restricted to the columns x_k, s_k, u_k
// and the rows dyn_{k+1}, bx_k, bu_k — plus dyn_0 at k = 0): new scalings `n` from the old scalings `o` of this stage, the old
// E of rows dyn_k (Ed_cur: the previous stage's, or the header's) and the old D_x of stage k+1 (Dx_next).  A pass is a
// Jacobi step — every new value depends on OLD values only — so the stages of a pass are independent: scale_pass walks
// them one after the other in one thread, scale_warp_kernel gives each to a lane.  Adds this stage's terms to the
// statistics of the cost normalisation (sumP, maxq), which are the only coupling between the stages of a pass.
template <typename T, typename L>
MPCB_HD void scale_stage_update(const KParams<T>& p, const Model<T, L>& m, T c, int b, int k, const ScaleStage<T, L>& o,
                                const T* Ed_cur, const T* Dx_next, ScaleStage<T, L>& n, T* E0new, T& sumP, T& maxq) {
    constexpr int NX = L::NX, NU = L::NU, NS = L::NS;
    const bool last = (k == p.N);
    const T* Qk = last ? p.QN : p.Q;
    // ---- column norms of the KKT matrix -> new D
    // every |entry| of [A B] scaled by its row's E and its column's D enters one column norm and one row norm:
    // formed once (the maxima are exact, so the order in which they are taken does not matter)
    T colx[NX], colu[NU], rowd[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        T v = c * tabs(Qk[j]) * o.Dx[j] * o.Dx[j];
        v = tmax(v, Ed_cur[j] * o.Dx[j]);
        colx[j] = tmax(v, o.Ebx[j] * o.Dx[j]);
        rowd[j] = o.Edn[j] * Dx_next[j];
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) colu[j] = tmax(c * tabs(p.R[j]) * o.Du[j] * o.Du[j], o.Ebu[j] * o.Du[j]);
    if (!last) {
#pragma unroll
        for (int i = 0; i < NX; ++i) {
#pragma unroll
            for (int j = 0; j < NX; ++j) {
                const T gij = tabs(m.A[i][j]) * o.Edn[i] * o.Dx[j];
                colx[j] = tmax(colx[j], gij); rowd[i] = tmax(rowd[i], gij);
            }
#pragma unroll
            for (int j = 0; j < NU; ++j) {
                const T gij = tabs(m.B[i][j]) * o.Edn[i] * o.Du[j];
                colu[j] = tmax(colu[j], gij); rowd[i] = tmax(rowd[i], gij);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        n.Dx[j] = o.Dx[j] * fast_rsqrt(limit_scaling(colx[j]));
        if (NS) {
            T w = tmax(c * tabs(p.W[j]) * o.Dsl[j] * o.Dsl[j], tabs(p.S[j]) * o.Ebx[j] * o.Dsl[j]);
            n.Dsl[j] = o.Dsl[j] * fast_rsqrt(limit_scaling(w));
        } else {
            n.Dsl[j] = (T)1;
        }
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) n.Du[j] = last ? (T)1 : o.Du[j] * fast_rsqrt(limit_scaling(colu[j]));
    // ---- row norms of A -> new E
    if (k == 0) {
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            T v = Ed_cur[i] * o.Dx[i];
            E0new[i] = Ed_cur[i] * fast_rsqrt(limit_scaling(v));
        }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        T en = (T)1;
        if (!last) en = o.Edn[i] * fast_rsqrt(limit_scaling(rowd[i]));
        n.Edn[i] = en;
        T w = o.Ebx[i] * o.Dx[i];
        if (NS) w = tmax(w, tabs(p.S[i]) * o.Ebx[i] * o.Dsl[i]);
        n.Ebx[i] = o.Ebx[i] * fast_rsqrt(limit_scaling(w));
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) {
        T w = o.Ebu[j] * o.Du[j];
        n.Ebu[j] = last ? (T)1 : o.Ebu[j] * fast_rsqrt(limit_scaling(w));
    }
    // ---- the cost-normalisation statistics with the new D
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        sumP += c * tabs(Qk[j]) * n.Dx[j] * n.Dx[j];
        const T xr = p.Xr[((p.xr_tv ? (size_t)k * NX : 0) + j) * p.ld + b];
        maxq = tmax(maxq, tabs(c * n.Dx[j] * (-(Qk[j] * xr))));
        if (NS) sumP += c * tabs(p.W[j]) * n.Dsl[j] * n.Dsl[j];
    }
#pragma unroll
    for (int j = 0; j < NU; ++j)
        if (!last) sumP += c * tabs(p.R[j]) * n.Du[j] * n.Du[j];
}
// the new cost scaling from the statistics of a pass
template <typename T, typename L>
MPCB_HD T scale_cost_update(T c, T sumP, T maxq, int N) {
    T c_temp = sumP / (T)L::nvar(N);
    const T nq = limit_scaling(maxq);
    c_temp = tmax(c_temp, nq);
    c_temp = (T)1 / limit_scaling(c_temp);
    return c * c_temp;
}

// one Ruiz pass over the stages; ODD is a compile-time constant so that every D/E access has a fixed offset
// (even passes read the records and write the scratch, odd ones the reverse)
template <typename T, typename L, bool ODD>
MPCB_HD void scale_pass(const KParams<T>& p, int b, const Ws<T, L>& ws, Model<T, L>& m, T& c) {
    constexpr int NX = L::NX, NU = L::NU, NS = L::NS;
    constexpr bool odd = ODD;
    const int N = p.N;
    const T* E0s = odd ? ws.scr_hdr : ws.hdr + L::H_E0 * TILE;
    T* E0d = odd ? ws.hdr + L::H_E0 * TILE : ws.scr_hdr;
    T sumP = 0, maxq = 0;
    T Ed_cur[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) Ed_cur[i] = MPCB_AT(E0s, i);
    for (int k = 0; k <= N; ++k) {
        const bool last = (k == N);
        const T* Ds = odd ? ws.S(k) : ws.R(k) + L::R_D * TILE;
        const T* Es = odd ? ws.S(k) + L::VS * TILE : ws.R(k) + L::R_E * TILE;
        T* Dd = odd ? ws.R(k) + L::R_D * TILE : ws.S(k);
        T* Ed = odd ? ws.R(k) + L::R_E * TILE : ws.S(k) + L::VS * TILE;
        const T* Dsn_ = last ? Ds : (odd ? ws.S(k + 1) : ws.R(k + 1) + L::R_D * TILE);
        if (p.tv && !last) load_model<T, L>(p, b, k, m);
        ScaleStage<T, L> o, n;
        T Dx_next[NX], E0new[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            o.Dx[i] = MPCB_AT(Ds, L::OX + i);
            o.Dsl[i] = NS ? MPCB_AT(Ds, L::OS + (NS ? i : 0)) : (T)1;
            o.Ebx[i] = MPCB_AT(Es, L::OBX + i);
            o.Edn[i] = last ? (T)1 : MPCB_AT(Es, L::ODN + i);
            Dx_next[i] = last ? (T)1 : MPCB_AT(Dsn_, L::OX + i);
        }
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            o.Du[j] = MPCB_AT(Ds, L::OU + j);
            o.Ebu[j] = MPCB_AT(Es, L::OBU + j);
        }
        scale_stage_update<T, L>(p, m, c, b, k, o, Ed_cur, Dx_next, n, E0new, sumP, maxq);
        if (k == 0) {
#pragma unroll
            for (int i = 0; i < NX; ++i) MPCB_AT(E0d, i) = E0new[i];
        }
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            MPCB_AT(Ed, L::ODN + i) = n.Edn[i];
            MPCB_AT(Ed, L::OBX + i) = n.Ebx[i];
            MPCB_AT(Dd, L::OX + i) = n.Dx[i];
            if (NS) MPCB_AT(Dd, L::OS + (NS ? i : 0)) = n.Dsl[i];
        }
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            MPCB_AT(Ed, L::OBU + j) = n.Ebu[j];
            MPCB_AT(Dd, L::OU + j) = n.Du[j];
        }
#pragma unroll
        for (int i = 0; i < NX; ++i) Ed_cur[i] = o.Edn[i];
    }
    c = scale_cost_update<T, L>(c, sumP, maxq, N);
}

template <typename T, typename L>
MPCB_HD void scale_one(const KParams<T>& p, int b) {
    constexpr int NX = L::NX;
    const int N = p.N;
    Ws<T, L> ws(p, b);
    for (int k = 0; k <= N; ++k) {
        T* R = ws.R(k);
        for (int e = 0; e < L::VS + L::CS; ++e) MPCB_AT(R, L::R_D + e) = (T)1;
    }
    for (int i = 0; i < NX; ++i) MPCB_AT(ws.hdr, L::H_E0 + i) = (T)1;
    T c = (T)1;
    Model<T, L> m;
    if (!p.tv) load_model<T, L>(p, b, 0, m);
    for (int it = 0; it < p.scaling; ++it) {
        if (it & 1) scale_pass<T, L, true>(p, b, ws, m, c);
        else scale_pass<T, L, false>(p, b, ws, m, c);
    }
    if (p.scaling & 1) {          // result of the last iteration is in the scratch: bring it home
        for (int k = 0; k <= N; ++k)
            for (int e = 0; e < L::VS + L::CS; ++e) MPCB_AT(ws.R(k), L::R_D + e) = MPCB_AT(ws.S(k), e);
        for (int i = 0; i < NX; ++i) MPCB_AT(ws.hdr, L::H_E0 + i) = MPCB_AT(ws.scr_hdr, i);
    }
    MPCB_AT(ws.hdr, L::H_C) = c;
}

// ------------------------------------------------------------------------------------------
// Cached factorisation of the reduced KKT matrix (the "cached KKT Cholesky").
//   ex_k = E_dyn(k) D_x(k)   |-I| entry of row dyn_k          bx, bs, bu  entries of the bound rows
//   A^_k = E_dyn(k+1) A_k D_x(k),  B^_k likewise               rho per row from its scaled bounds
// ------------------------------------------------------------------------------------------
template <typename T, typename L>
MPCB_HD void factor_one(const KParams<T>& p, int b) {
    constexpr int NX = L::NX, NU = L::NU, NW = L::NW, NS = L::NS;
    const int N = p.N;
    Ws<T, L> ws(p, b);
    const T c = MPCB_AT(ws.hdr, L::H_C);
    const T rho = clamp_rho(p.rho), rho_eq = (T)kRhoEqOverRhoIneq * rho, sigma = p.sigma;
    Model<T, L> m;
    if (!p.tv) load_model<T, L>(p, b, 0, m);
    T Fprev[NX][NW];
    T Ed_cur[NX];
#pragma unroll
    for (int i = 0; i < NX; ++i) Ed_cur[i] = MPCB_AT(ws.hdr, L::H_E0 + i);
    int bad = 0;
    for (int k = 0; k <= N; ++k) {
        const bool last = (k == N);
        T* R = ws.R(k);
        if (p.tv && !last) load_model<T, L>(p, b, k, m);
        const T* Qk = last ? p.QN : p.Q;
        T lo[NX], hi[NX];
        stage_box<T, L>(p, k, lo, hi);
        T Dx[NX], Du[NU], Ed_next[NX];
        T Sm[NW][NW];
#pragma unroll
        for (int a = 0; a < NW; ++a)
#pragma unroll
            for (int d = 0; d < NW; ++d) Sm[a][d] = 0;
#pragma unroll
        for (int j = 0; j < NX; ++j) {
            Dx[j] = MPCB_AT(R, L::R_D + L::OX + j);
            Ed_next[j] = last ? (T)1 : MPCB_AT(R, L::R_E + L::ODN + j);
            const T Ebx = MPCB_AT(R, L::R_E + L::OBX + j);
            const T ex = Ed_cur[j] * Dx[j], bx = Ebx * Dx[j];
            const T rb = row_rho(Ebx * lo[j], Ebx * hi[j], rho, rho_eq);
            T d = c * Qk[j] * Dx[j] * Dx[j] + sigma + rho_eq * ex * ex + rb * bx * bx;
            if (NS) {
                const T Dsl = MPCB_AT(R, L::R_D + L::OS + (NS ? j : 0));
                const T bs = p.S[j] * Ebx * Dsl;
                const T mss = c * p.W[j] * Dsl * Dsl + sigma + rb * bs * bs;
                const T mxs = rb * bx * bs;
                d -= mxs * mxs / mss;
            }
            Sm[j][j] = d;
        }
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            Du[j] = last ? (T)1 : MPCB_AT(R, L::R_D + L::OU + j);
            const T Ebu = MPCB_AT(R, L::R_E + L::OBU + j);
            const T bu = Ebu * Du[j];
            const T rb = row_rho(Ebu * p.umin[j], Ebu * p.umax[j], rho, rho_eq);
            Sm[NX + j][NX + j] = last ? (T)1 : c * p.R[j] * Du[j] * Du[j] + sigma + rb * bu * bu;
        }
        T G[NX][NW];      // [A^ B^] of rows dyn_{k+1}
#pragma unroll
        for (int i = 0; i < NX; ++i) {
#pragma unroll
            for (int j = 0; j < NX; ++j) G[i][j] = last ? (T)0 : Ed_next[i] * m.A[i][j] * Dx[j];
#pragma unroll
            for (int j = 0; j < NU; ++j) G[i][NX + j] = last ? (T)0 : Ed_next[i] * m.B[i][j] * Du[j];
        }
        if (!last) {
#pragma unroll
            for (int a = 0; a < NW; ++a)
#pragma unroll
                for (int d = 0; d <= a; ++d) {
                    T acc = 0;
#pragma unroll
                    for (int i = 0; i < NX; ++i) acc += G[i][a] * G[i][d];
                    Sm[a][d] += rho_eq * acc;
                }
        }
        if (k > 0) {
#pragma unroll
            for (int a = 0; a < NX; ++a)
#pragma unroll
                for (int d = 0; d <= a; ++d) {
                    T acc = 0;
#pragma unroll
                    for (int e = 0; e < NW; ++e) acc += Fprev[a][e] * Fprev[d][e];
                    Sm[a][d] -= acc;
                }
        }
        // Cholesky, lower, in place
#pragma unroll
        for (int j = 0; j < NW; ++j) {
            T d = Sm[j][j];
#pragma unroll
            for (int e = 0; e < j; ++e) d -= Sm[j][e] * Sm[j][e];
            if (!(d > (T)0)) { bad = 1; d = (T)1e-30; }
            d = msqrt(d);
            Sm[j][j] = d;
            const T inv = (T)1 / d;
#pragma unroll
            for (int i = j + 1; i < NW; ++i) {
                T v = Sm[i][j];
#pragma unroll
                for (int e = 0; e < j; ++e) v -= Sm[i][e] * Sm[j][e];
                Sm[i][j] = v * inv;
            }
        }
        // inverse of the lower-triangular factor
        T Li[NW][NW];
#pragma unroll
        for (int j = 0; j < NW; ++j) {
            Li[j][j] = (T)1 / Sm[j][j];
#pragma unroll
            for (int i = j + 1; i < NW; ++i) {
                T v = 0;
#pragma unroll
                for (int e = j; e < i; ++e) v += Sm[i][e] * Li[e][j];
                Li[i][j] = -v / Sm[i][i];
            }
        }
        if (p.minv) {                            // the symmetric block inverse Linv' Linv (KParams::minv)
#pragma unroll
            for (int a = 0; a < NW; ++a)
#pragma unroll
                for (int d = 0; d <= a; ++d) {
                    T acc = 0;
#pragma unroll
                    for (int e = a; e < NW; ++e) acc += Li[e][a] * Li[e][d];
                    MPCB_AT(R, L::R_F + a * (a + 1) / 2 + d) = acc;
                }
        } else {
#pragma unroll
            for (int a = 0; a < NW; ++a)
#pragma unroll
                for (int d = 0; d <= a; ++d) MPCB_AT(R, L::R_F + a * (a + 1) / 2 + d) = Li[a][d];
        }
        if (!last) {
            // coupling block C_k = M[x_{k+1}, w_k] = -rho_eq ex_{k+1} (.) [A^ B^];  F_k = C_k Linv_k'
            const T* Rn = ws.R(k + 1);
#pragma unroll
            for (int i = 0; i < NX; ++i) {
                const T exn = Ed_next[i] * MPCB_AT(Rn, L::R_D + L::OX + i);
#pragma unroll
                for (int a = 0; a < NW; ++a) {
                    T acc = 0;
#pragma unroll
                    for (int d = 0; d <= a; ++d) acc += G[i][d] * Li[a][d];
                    Fprev[i][a] = -rho_eq * exn * acc;      // only needed for the next Schur complement
                }
            }
        }
#pragma unroll
        for (int i = 0; i < NX; ++i) Ed_cur[i] = Ed_next[i];
    }
    if (bad) p.status[b] = -7;   // OSQP_NON_CVX: reduced KKT matrix lost positive definiteness
}

// ------------------------------------------------------------------------------------------
// The ADMM iteration, one stage at a time.
//
// Row state.  Between solves a row holds (z, y) like OSQP.  Inside the loop, after the first
// iteration, a row holds the single number p = z_relaxed + y/rho from which
//     z = clip(p, l, u),   y/rho = p - z                       (osqp.c: update_z / update_y)
// are recovered on the fly; this halves the row traffic and removes every division.  The first
// iteration of a launch reads the explicit (z, y) (cold-start zeros, a warm start, or the previous
// solve's values — those were projected onto the PREVIOUS bounds, so they cannot be recovered from
// p); the exit pass of a launch writes explicit (z, y) back.
//
// Linear solve.  M = L L' with L block lower bidiagonal: diagonal blocks L_kk (stored inverted,
// Linv_k) and sub-diagonal blocks F_k = C_k Linv_k', C_k = -rho_eq ex_{k+1} (.) [A^_k B^_k] the
// coupling of x_{k+1} with (x_k, u_k).  F_k is never stored:
//     forward   t_k = Linv_k ( r_k - [F_{k-1} t_{k-1}] ),   F_{k-1} t_{k-1} = C_{k-1} (Linv_{k-1}' t_{k-1})
//     backward  w_k = Linv_k' ( t_k - Linv_k (C_k' w^x_{k+1}) )
//
// `S` is the lane's view of the stage record the sweep READS (global memory, or the copy a TMA bulk
// transfer staged in shared memory — same [element][32 lanes] shape); `R` is the record in global
// memory that receives the WRITES.
// ------------------------------------------------------------------------------------------
template <typename T>
struct Row {      // z and y/rho of one row
    T z, yr;
};
template <typename T>
MPCB_HD Row<T> row_state(bool first, T zp, T yv, T l, T u, T rinv) {
    Row<T> r;
    if (first) { r.z = zp; r.yr = yv * rinv; }
    else { r.z = tmin(tmax(zp, l), u); r.yr = zp - r.z; }
    return r;
}
// bound rows: 1/rho is only needed by the first iteration of a launch, pick it lazily
template <typename T, typename Q>
MPCB_HD Row<T> row_state_b(bool first, T zp, const T* yptr, T l, T u, T rb, const Q& q) {
    Row<T> r;
    if (first) { r.z = zp; r.yr = *yptr * q.rinv_of(rb); }
    else { r.z = tmin(tmax(zp, l), u); r.yr = zp - r.z; }
    return r;
}
// new p from z~ (relaxation and dual step folded): p+ = alpha z~ + (1-alpha) z + y/rho
template <typename T>
MPCB_HD T row_next(T zt, const Row<T>& r, T alpha) {
    return alpha * zt + ((T)1 - alpha) * r.z + r.yr;
}

template <typename T, typename L>
struct AdmmConst {
    T c, cinv, rho, rho_eq, sigma, alpha;
    // reference of the QP when it is not stage-wise: element j at xr[j * xr_stride].  The TMA kernel keeps it in the
    // warp's slice of shared memory (5 loop-invariant doubles the register allocator would otherwise spill), the
    // lane-per-QP kernel reads it from the input array
    const T* xr;
    size_t xr_stride;
    bool inf_bounds;      // some bound of the problem is infinite (rows of type "unconstrained" may exist)
    // 1/rho of a row: only the first iteration of a solve (explicit y on entry) needs it — computed there, not kept
    MPCB_HD T rinv_of(T rb) const { return (T)1 / rb; }
    MPCB_HD T rinv_eq() const { return (T)1 / rho_eq; }
};

// state carried from stage to stage by the forward sweep
template <typename T, typename L>
struct FwdCarry {
    T Ed_cur[L::NX];     // E of rows dyn_k
    T vd_cur[L::NX];     // rho z - y of rows dyn_k
    T cprev[L::NX];      // [A_{k-1} B_{k-1}] (D (.) Linv_{k-1}' t_{k-1})
};

// RHS: the right-hand side is r^ (read from the t slots, written by the previous backward sweep) plus the two terms that come
// from stage k-1; the stage reads only the runs FA and FB of its record (mpc_common.h).  Otherwise it is formed from the
// whole record (the first iteration of a solve, or with KParams::fwd_rhs = 0).
template <typename T, typename L, bool FIRST, bool RHS = false>
MPCB_HD void admm_fwd_stage(const KParams<T>& p, const AdmmConst<T, L>& q, const Model<T, L>& m, int b, int k,
                            const T* S, const T* Yk, T* R, FwdCarry<T, L>& cy) {
    constexpr bool first = FIRST;     // compile-time: the steady-state sweeps carry no trace of the (z, y) entry form
    static_assert(!(FIRST && RHS), "r^ is formed from p-form rows: there is none before the first backward sweep");
    constexpr int NX = L::NX, NU = L::NU, NW = L::NW, NS = L::NS;
    const bool last = (k == p.N);
    const T* Qk = last ? p.QN : p.Q;
    T lo[NX], hi[NX];
    stage_box<T, L>(p, k, lo, hi);
    T Dx[NX], Du[NU], Ed_next[NX], wv[NX], vd_next[NX], r[NW];
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        Dx[i] = MPCB_AT(S, L::R_D + L::OX + i);
        if (!last) {
            Ed_next[i] = MPCB_AT(S, L::R_E + L::ODN + i);
            const T beq = -Ed_next[i] * model_g<T, L>(p, b, k, i);
            const Row<T> rw = row_state(first, MPCB_AT(S, L::R_P + L::ODN + i), first ? MPCB_AT(Yk, L::ODN + i) : (T)0,
                                        beq, beq, q.rinv_eq());
            vd_next[i] = q.rho_eq * (rw.z - rw.yr);
        } else {
            Ed_next[i] = 1; vd_next[i] = 0;
        }
        wv[i] = Ed_next[i] * vd_next[i];
    }
    if (RHS) {
#pragma unroll
        for (int j = 0; j < NX; ++j) {
            const T ex = cy.Ed_cur[j] * Dx[j];
            T v = MPCB_AT(S, L::R_T + j) - ex * cy.vd_cur[j];
            if (k > 0) v += q.rho_eq * ex * cy.Ed_cur[j] * cy.cprev[j];
            r[j] = v;
        }
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            Du[j] = last ? (T)1 : MPCB_AT(S, L::R_D + L::OU + j);
            r[NX + j] = MPCB_AT(S, L::R_T + NX + j);
        }
    } else {
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        const T Ebx = MPCB_AT(S, L::R_E + L::OBX + j);
        const T bx = Ebx * Dx[j], lb = Ebx * lo[j], ub = Ebx * hi[j];
        const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
        const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + L::OBX + j), Yk + (L::OBX + j) * TILE, lb, ub, rb, q);
        const T vbx = rb * (rw.z - rw.yr);
        const T xr = p.xr_tv ? p.Xr[((size_t)k * NX + j) * p.ld + b] : q.xr[(size_t)j * q.xr_stride];
        const T qh = q.c * Dx[j] * (-(Qk[j] * xr));
        T acc = 0;
        if (!last) {
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += m.A[i][j] * wv[i];
        }
        const T ex = cy.Ed_cur[j] * Dx[j];
        T v = q.sigma * MPCB_AT(S, L::R_X + L::OX + j) - qh - ex * cy.vd_cur[j] + bx * vbx + Dx[j] * acc;
        if (NS) {
            const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? j : 0));
            const T bs = p.S[j] * Ebx * Dsl;
            const T mss = q.c * p.W[j] * Dsl * Dsl + q.sigma + rb * bs * bs;
            const T mxs = rb * bx * bs;
            const T rs = q.sigma * MPCB_AT(S, L::R_X + L::OS + (NS ? j : 0)) + bs * vbx;
            v -= mxs * fast_rcp(mss) * rs;
        }
        if (k > 0) v += q.rho_eq * ex * cy.Ed_cur[j] * cy.cprev[j];
        r[j] = v;
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) {
        T v = 0;
        Du[j] = 1;
        if (!last) {
            Du[j] = MPCB_AT(S, L::R_D + L::OU + j);
            const T Ebu = MPCB_AT(S, L::R_E + L::OBU + j);
            const T bu = Ebu * Du[j], lb = Ebu * p.umin[j], ub = Ebu * p.umax[j];
            const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
            const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + L::OBU + j), Yk + (L::OBU + j) * TILE, lb, ub, rb, q);
            T acc = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += m.B[i][j] * wv[i];
            v = q.sigma * MPCB_AT(S, L::R_X + L::OU + j) + bu * (rb * (rw.z - rw.yr)) + Du[j] * acc;
        }
        r[NX + j] = v;
    }
    }
    (void)wv;
    // t = Linv r ;  g = Linv' t ;  h = D (.) g ;  cprev = [A B] h
    T Li[L::LT], t[NW], h[NW];
#pragma unroll
    for (int e = 0; e < L::LT; ++e) Li[e] = MPCB_AT(S, L::R_F + e);
#pragma unroll
    for (int a = 0; a < NW; ++a) {
        T acc = 0;
#pragma unroll
        for (int d = 0; d <= a; ++d) acc += Li[a * (a + 1) / 2 + d] * r[d];
        t[a] = acc;
        MPCB_AT(R, L::R_T + a) = acc;
    }
    if (!last) {
#pragma unroll
        for (int d = 0; d < NW; ++d) {
            T acc = 0;
#pragma unroll
            for (int a = d; a < NW; ++a) acc += Li[a * (a + 1) / 2 + d] * t[a];
            h[d] = (d < NX ? Dx[d < NX ? d : 0] : Du[d >= NX ? d - NX : 0]) * acc;
        }
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            T acc = 0;
#pragma unroll
            for (int j = 0; j < NX; ++j) acc += m.A[i][j] * h[j];
#pragma unroll
            for (int j = 0; j < NU; ++j) acc += m.B[i][j] * h[NX + j];
            cy.cprev[i] = acc;
        }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) { cy.Ed_cur[i] = Ed_next[i]; cy.vd_cur[i] = vd_next[i]; }
}

// state carried from stage to stage by the backward sweep
template <typename T, typename L>
struct BwdCarry {
    T xt_next[L::NX];    // x~_{k+1}
    T Dx_next[L::NX];    // D_x(k+1)
};

// ---- termination test on the unscaled residuals (auxil.c: check_termination), one stage
template <typename T>
struct Resid {
    T pri, dua, nz, nAx, nq, nAty, nPx;
};
// The accumulators of one evaluation of the termination test.  ONE set of terms serves both evaluations OSQP makes at a
// termination test:
//   the residuals of (x, y)                                        (auxil.c: compute_pri_res / compute_dua_res, tolerances)
//   the infeasibility certificates of (dx, dy) = (x - x_old, y - y_old)   (is_primal/dual_infeasible)
// Both need the same linear forms — E^-1 A v by rows, D^-1 A'w and D^-1 P v by columns — applied to v = x, w = y or to
// v = dx, w = dy.
template <typename T>
struct TestAcc {
    T pri, dua, nz, nAx, nq, nAty, nPx;      // residual norms; nAty = ||D^-1 A'w||, nPx = ||D^-1 P v|| serve both evaluations
    T nEw, lhs, nDv, qv, aup, alo;           // certificate terms: ||E w||, u'w+ + l'w-, ||D v||, q'v, max / min of E^-1 A v
};
template <typename T>
MPCB_HD void test_reset(TestAcc<T>& a) {
    a.pri = a.dua = a.nz = a.nAx = a.nq = a.nAty = a.nPx = 0;
    a.nEw = a.lhs = a.nDv = a.qv = 0;
    a.aup = (T)-kOsqpInfty; a.alo = (T)kOsqpInfty;
}
// is_primal_infeasible projects dy on the recession cone of the row's bound type first
template <typename T>
MPCB_HD T cert_project(bool inf_possible, T dy, T lb, T ub) {
    if (inf_possible) {
        const bool up_inf = ub > (T)(kOsqpInfty * kMinScaling), lo_inf = lb < (T)(-kOsqpInfty * kMinScaling);
        if (up_inf && lo_inf) dy = 0;
        else if (up_inf) dy = tmin(dy, (T)0);
        else if (lo_inf) dy = tmax(dy, (T)0);
    }
    return dy;
}

// The termination test of a tested iteration, evaluated by its backward sweep (admm_bwd_stage in mode kBwdTest).  At stage k
// the sweep holds the new x_k and p in registers and the old ones — x^{k-1}, y^{k-1} of the certificates — in the record it
// reads.  Every norm is a max-norm except lhs and qv, so the order of the stages does not matter.  A stage's row dyn_{k+1}
// needs the new x_{k+1}, and the dual residual of column x_k needs the new row dyn_k, which stage k-1 forms: both are
// carried here.  `r` gets the residual terms of (x, y), `c` the certificate terms of (dx, dy); admm_test_stage evaluates the
// same expressions.
template <typename T, typename L>
struct BwdTest {
    TestAcc<T> r, c;
    T x_next[L::NX], dx_next[L::NX];              // new x_{k+1}, x_{k+1} - x_{k+1}^old
    T own_r[L::NX], qpx_r[L::NX], own_c[L::NX];   // column x_{k+1} without its row dyn_{k+1}: A'y part, q + P x; A'dy part
};
enum { kBwdPlain, kBwdTest };
// A copy of v that the compiler cannot trace back to v's expression.  The test terms form their products from such copies
// so that they share none with the iterate arithmetic: the compiler fuses a product into an FMA only when every use of it
// is an addition, so one more use by the test would change how the tested iteration's iterates round.
MPCB_HD float opaque(float v) {
#ifdef __CUDA_ARCH__
    asm("" : "+f"(v));
#endif
    return v;
}
MPCB_HD double opaque(double v) {
#ifdef __CUDA_ARCH__
    asm("" : "+d"(v));
#endif
    return v;
}
template <typename T, typename L>
MPCB_HD void test_reset(BwdTest<T, L>& ts) { test_reset(ts.r); test_reset(ts.c); }
// the dual residual of column x_{k+1} (carried) once its row dyn_{k+1} is known: E y of that row is wr times the row's E,
// ex = E_dyn(k+1) D_x(k+1)
template <typename T, typename L>
MPCB_HD void test_close_column(BwdTest<T, L>& ts, int i, T ex, T wr, T wc, T Dinv) {
    T atyr = ts.own_r[i], atyc = ts.own_c[i];
    atyr -= ex * wr;
    atyc -= ex * wc;
    ts.r.dua = tmax(ts.r.dua, tabs(Dinv * (ts.qpx_r[i] + atyr)));
    ts.r.nAty = tmax(ts.r.nAty, tabs(Dinv * atyr));
    ts.c.nAty = tmax(ts.c.nAty, tabs(Dinv * atyc));
}

// MODE kBwdTest: the iteration ends with a termination test, accumulated into ts (BwdTest); the iterate arithmetic and the
// stores are those of kBwdPlain.
// Every instantiation leaves r^_k in the t slots of R: the part of the next forward sweep's right-hand side r_k that depends
// on stage k alone (sigma x, the cost term, the bound rows and the slack elimination, A'w / B'w of rows dyn_{k+1}), formed
// from the new x_k and the new p-form rows — all in registers here, while the next forward sweep would have to read them.
// S may alias R (the lane-per-QP kernel): every old value is read before the stage writes it.
template <typename T, typename L, bool FIRST, int MODE>
MPCB_HD void admm_bwd_stage(const KParams<T>& p, const AdmmConst<T, L>& q, const Model<T, L>& m, int b, int k,
                            const T* S, const T* Yk, T* R, BwdCarry<T, L>& cy, BwdTest<T, L>& ts) {
    constexpr bool first = FIRST;
    constexpr bool TEST = MODE == kBwdTest;
    constexpr int NX = L::NX, NU = L::NU, NW = L::NW, NS = L::NS;
    const bool last = (k == p.N);
    T lo[NX], hi[NX];
    stage_box<T, L>(p, k, lo, hi);
    T Dx[NX], Du[NU], Ed_next[NX], exn[NX], rhs[NW], w[NW], Li[L::LT];
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        Dx[i] = MPCB_AT(S, L::R_D + L::OX + i);
        Ed_next[i] = last ? (T)1 : MPCB_AT(S, L::R_E + L::ODN + i);
        exn[i] = Ed_next[i] * cy.Dx_next[i];              // ex_{k+1} = E_dyn(k+1) D_x(k+1)
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) Du[j] = last ? (T)1 : MPCB_AT(S, L::R_D + L::OU + j);
#pragma unroll
    for (int e = 0; e < L::LT; ++e) Li[e] = MPCB_AT(S, L::R_F + e);
#pragma unroll
    for (int a = 0; a < NW; ++a) rhs[a] = MPCB_AT(S, L::R_T + a);
    if (!last) {
        T cv[NW], om[NX];
#pragma unroll
        for (int i = 0; i < NX; ++i) om[i] = Ed_next[i] * exn[i] * cy.xt_next[i];
#pragma unroll
        for (int a = 0; a < NW; ++a) {
            T acc = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += (a < NX ? m.A[i][a < NX ? a : 0] : m.B[i][a >= NX ? a - NX : 0]) * om[i];
            cv[a] = -q.rho_eq * (a < NX ? Dx[a < NX ? a : 0] : Du[a >= NX ? a - NX : 0]) * acc;
        }
#pragma unroll
        for (int a = 0; a < NW; ++a) {
            T acc = 0;
#pragma unroll
            for (int d = 0; d <= a; ++d) acc += Li[a * (a + 1) / 2 + d] * cv[d];
            rhs[a] -= acc;
        }
    }
#pragma unroll
    for (int d = 0; d < NW; ++d) {
        T acc = 0;
#pragma unroll
        for (int a = d; a < NW; ++a) acc += Li[a * (a + 1) / 2 + d] * rhs[a];
        w[d] = acc;
    }
    // rows bx_k (+ slack recovery), x_k / s_k
    T rh[NW];         // r^_k
    // kBwdTest: the new x_k, u_k and their deltas; the columns x_k / u_k until the new rows dyn_{k+1} are known
    T xn_a[NX], dx_a[NX], ownr_x[NX], ownc_x[NX], qpx_x[NX], un_a[NU], du_a[NU], ownr_u[NU], ownc_u[NU], pxr_u[NU];
    (void)xn_a; (void)dx_a; (void)ownr_x; (void)ownc_x; (void)qpx_x; (void)un_a; (void)du_a; (void)ownr_u; (void)ownc_u;
    (void)pxr_u;
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        const T Ebx = MPCB_AT(S, L::R_E + L::OBX + j);
        const T bx = Ebx * Dx[j], lb = Ebx * lo[j], ub = Ebx * hi[j];
        const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
        const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + L::OBX + j), Yk + (L::OBX + j) * TILE, lb, ub, rb, q);
        const T xo = TEST ? MPCB_AT(S, L::R_X + L::OX + j) : (T)0;     // (old x_k; S may alias R)
        T ztil = bx * w[j];
        T sn = 0, bs = 0, mxs = 0, mss = 1, so = 0;
        if (NS) {
            const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? j : 0));
            bs = p.S[j] * Ebx * Dsl;
            mss = q.c * p.W[j] * Dsl * Dsl + q.sigma + rb * bs * bs;
            mxs = rb * bx * bs;
            const T sold = MPCB_AT(S, L::R_X + L::OS + (NS ? j : 0));
            if (TEST) so = sold;
            const T rs = q.sigma * sold + bs * (rb * (rw.z - rw.yr));
            const T st = (rs - mxs * w[j]) * fast_rcp(mss);
            ztil += bs * st;
            sn = q.alpha * st + ((T)1 - q.alpha) * sold;
            MPCB_AT(R, L::R_X + L::OS + (NS ? j : 0)) = sn;
        }
        const T pn = row_next(ztil, rw, q.alpha);
        const T xn = q.alpha * w[j] + ((T)1 - q.alpha) * MPCB_AT(S, L::R_X + L::OX + j);
        MPCB_AT(R, L::R_P + L::OBX + j) = pn;
        MPCB_AT(R, L::R_X + L::OX + j) = xn;
        // r^: sigma x - q + bx' (rho (z - y/rho)) of the new state, minus the slack elimination (A'w of rows dyn_{k+1} below)
        const Row<T> rn = row_state(false, pn, (T)0, lb, ub, (T)0);
        const T vbx = rb * (rn.z - rn.yr);
        const T xr = p.xr_tv ? p.Xr[((size_t)k * NX + j) * p.ld + b] : q.xr[(size_t)j * q.xr_stride];
        const T qh = q.c * Dx[j] * (-((last ? p.QN : p.Q)[j] * xr));
        T v = q.sigma * xn - qh + bx * vbx;
        if (NS) v -= mxs * fast_rcp(mss) * (q.sigma * sn + bs * vbx);
        rh[j] = v;
        if (TEST) {       // row bx_k and columns s_k; column x_k without the rows dyn_k, dyn_{k+1}
            const T Einv = fast_rcp(Ebx), Dinv = fast_rcp(Dx[j]);
            const T vx = xn - xo, vs = sn - so;
            T wr = rb * (pn - rn.z);
            T wc = wr;
            wc -= rb * rw.yr;
            wc = cert_project(q.inf_bounds, wc, lb, ub);
            const T axr = bx * xn + bs * sn, axc = bx * vx + bs * vs;
            ts.r.pri = tmax(ts.r.pri, tabs(Einv * (axr - rn.z)));
            ts.r.nz = tmax(ts.r.nz, tabs(Einv * rn.z));
            ts.r.nAx = tmax(ts.r.nAx, tabs(Einv * axr));
            if (!q.inf_bounds || ub < (T)(kOsqpInfty * kMinScaling)) ts.c.aup = tmax(ts.c.aup, Einv * axc);
            if (!q.inf_bounds || lb > (T)(-kOsqpInfty * kMinScaling)) ts.c.alo = tmin(ts.c.alo, Einv * axc);
            ts.c.nEw = tmax(ts.c.nEw, tabs(Ebx * wc));
            ts.c.lhs += ub * tmax(wc, (T)0) + lb * tmin(wc, (T)0);
            const T Qkj = (last ? p.QN : p.Q)[j];
            const T qt = q.c * Dx[j] * (-(Qkj * opaque(xr)));      // = qh
            const T pxr = q.c * Qkj * Dx[j] * Dx[j] * xn, pxc = q.c * Qkj * Dx[j] * Dx[j] * vx;
            ts.r.nq = tmax(ts.r.nq, tabs(Dinv * qt));
            ts.r.nPx = tmax(ts.r.nPx, tabs(Dinv * pxr));
            ts.c.nPx = tmax(ts.c.nPx, tabs(Dinv * pxc));
            ts.c.nDv = tmax(ts.c.nDv, tabs(Dx[j] * vx));
            ts.c.qv += qt * vx;
            xn_a[j] = xn; dx_a[j] = vx; ownr_x[j] = bx * wr; ownc_x[j] = bx * wc; qpx_x[j] = qt + pxr;
            if (NS) {
                const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? j : 0)), Dsinv = fast_rcp(Dsl);
                const T pd = q.c * p.W[j] * opaque(Dsl) * Dsl;
                const T atys = bs * wr, pxs = pd * sn, atyc = bs * wc, pxsc = pd * vs;
                ts.r.dua = tmax(ts.r.dua, tabs(Dsinv * (atys + pxs)));
                ts.r.nAty = tmax(ts.r.nAty, tabs(Dsinv * atys));
                ts.r.nPx = tmax(ts.r.nPx, tabs(Dsinv * pxs));
                ts.c.nAty = tmax(ts.c.nAty, tabs(Dsinv * atyc));
                ts.c.nPx = tmax(ts.c.nPx, tabs(Dsinv * pxsc));
                ts.c.nDv = tmax(ts.c.nDv, tabs(Dsl * vs));
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NU; ++j) rh[NX + j] = 0;
    T wyr[NX], wyc[NX];      // kBwdTest: E y and E dy of the new rows dyn_{k+1}
    (void)wyr; (void)wyc;
    if (!last) {
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            const T Ebu = MPCB_AT(S, L::R_E + L::OBU + j);
            const T bu = Ebu * Du[j], lb = Ebu * p.umin[j], ub = Ebu * p.umax[j];
            const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
            const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + L::OBU + j), Yk + (L::OBU + j) * TILE, lb, ub, rb, q);
            const T uo = TEST ? MPCB_AT(S, L::R_X + L::OU + j) : (T)0;     // (old u_k)
            const T pn = row_next(bu * w[NX + j], rw, q.alpha);
            const T un = q.alpha * w[NX + j] + ((T)1 - q.alpha) * MPCB_AT(S, L::R_X + L::OU + j);
            MPCB_AT(R, L::R_P + L::OBU + j) = pn;
            MPCB_AT(R, L::R_X + L::OU + j) = un;
            const Row<T> rn = row_state(false, pn, (T)0, lb, ub, (T)0);
            rh[NX + j] = q.sigma * un + bu * (rb * (rn.z - rn.yr));
            if (TEST) {   // row bu_k; column u_k without the rows dyn_{k+1}
                const T Einv = fast_rcp(Ebu), Dinv = fast_rcp(Du[j]);
                const T vu = un - uo;
                T wr = rb * (pn - rn.z);
                T wc = wr;
                wc -= rb * rw.yr;
                wc = cert_project(q.inf_bounds, wc, lb, ub);
                const T axr = bu * un, axc = bu * vu;
                ts.r.pri = tmax(ts.r.pri, tabs(Einv * (axr - rn.z)));
                ts.r.nz = tmax(ts.r.nz, tabs(Einv * rn.z));
                ts.r.nAx = tmax(ts.r.nAx, tabs(Einv * axr));
                if (!q.inf_bounds || ub < (T)(kOsqpInfty * kMinScaling)) ts.c.aup = tmax(ts.c.aup, Einv * axc);
                if (!q.inf_bounds || lb > (T)(-kOsqpInfty * kMinScaling)) ts.c.alo = tmin(ts.c.alo, Einv * axc);
                ts.c.nEw = tmax(ts.c.nEw, tabs(Ebu * wc));
                ts.c.lhs += ub * tmax(wc, (T)0) + lb * tmin(wc, (T)0);
                const T pxr = q.c * p.R[j] * Du[j] * Du[j] * un, pxc = q.c * p.R[j] * Du[j] * Du[j] * vu;
                ts.r.nPx = tmax(ts.r.nPx, tabs(Dinv * pxr));
                ts.c.nPx = tmax(ts.c.nPx, tabs(Dinv * pxc));
                ts.c.nDv = tmax(ts.c.nDv, tabs(Du[j] * vu));
                un_a[j] = un; du_a[j] = vu; ownr_u[j] = bu * wr; ownc_u[j] = bu * wc; pxr_u[j] = pxr;
            }
        }
        // rows dyn_{k+1}:  E (A D x~_k + B D u~_k) - ex_{k+1} x~_{k+1} = -E g_k
        T wv[NX];     // E (rho z - y) of the new rows dyn_{k+1}
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            T acc = 0;
#pragma unroll
            for (int j = 0; j < NX; ++j) acc += m.A[i][j] * (Dx[j] * w[j]);
#pragma unroll
            for (int j = 0; j < NU; ++j) acc += m.B[i][j] * (Du[j] * w[NX + j]);
            const T ztil = Ed_next[i] * acc - exn[i] * cy.xt_next[i];
            const T beq = -Ed_next[i] * model_g<T, L>(p, b, k, i);
            const Row<T> rw = row_state(first, MPCB_AT(S, L::R_P + L::ODN + i), first ? MPCB_AT(Yk, L::ODN + i) : (T)0,
                                        beq, beq, q.rinv_eq());
            const T pn = row_next(ztil, rw, q.alpha);
            MPCB_AT(R, L::R_P + L::ODN + i) = pn;
            const Row<T> rn = row_state(false, pn, (T)0, beq, beq, (T)0);
            wv[i] = Ed_next[i] * (q.rho_eq * (rn.z - rn.yr));
            if (TEST) {   // row dyn_{k+1}; column x_{k+1} gets its row dyn_{k+1}
                T ar = 0, ac = 0;
#pragma unroll
                for (int j = 0; j < NX; ++j) { ar += m.A[i][j] * (Dx[j] * xn_a[j]); ac += m.A[i][j] * (Dx[j] * dx_a[j]); }
#pragma unroll
                for (int j = 0; j < NU; ++j) { ar += m.B[i][j] * (Du[j] * un_a[j]); ac += m.B[i][j] * (Du[j] * du_a[j]); }
                const T axr = Ed_next[i] * ar - exn[i] * ts.x_next[i], axc = Ed_next[i] * ac - exn[i] * ts.dx_next[i];
                const T Einv = fast_rcp(Ed_next[i]);
                ts.r.pri = tmax(ts.r.pri, tabs(Einv * (axr - beq)));
                ts.r.nz = tmax(ts.r.nz, tabs(Einv * beq));
                ts.r.nAx = tmax(ts.r.nAx, tabs(Einv * axr));
                ts.c.aup = tmax(ts.c.aup, Einv * axc);
                ts.c.alo = tmin(ts.c.alo, Einv * axc);
                T wr = q.rho_eq * (pn - beq);
                T wc = wr;
                wc -= q.rho_eq * rw.yr;
                ts.c.nEw = tmax(ts.c.nEw, tabs(Ed_next[i] * wc));
                ts.c.lhs += beq * wc;
                wyr[i] = Ed_next[i] * wr; wyc[i] = Ed_next[i] * wc;
                test_close_column(ts, i, exn[i], wr, wc, fast_rcp(cy.Dx_next[i]));
            }
        }
        if (TEST) {       // columns x_k and u_k get their rows dyn_{k+1}
#pragma unroll
            for (int j = 0; j < NX; ++j) {
                T ar = 0, ac = 0;
#pragma unroll
                for (int i = 0; i < NX; ++i) { ar += m.A[i][j] * wyr[i]; ac += m.A[i][j] * wyc[i]; }
                ownr_x[j] += Dx[j] * ar;
                ownc_x[j] += Dx[j] * ac;
            }
#pragma unroll
            for (int j = 0; j < NU; ++j) {
                T ar = 0, ac = 0;
#pragma unroll
                for (int i = 0; i < NX; ++i) { ar += m.B[i][j] * wyr[i]; ac += m.B[i][j] * wyc[i]; }
                T atyr = ownr_u[j], atyc = ownc_u[j];
                atyr += Du[j] * ar;
                atyc += Du[j] * ac;
                const T Dinv = fast_rcp(Du[j]);
                ts.r.dua = tmax(ts.r.dua, tabs(Dinv * (atyr + pxr_u[j])));
                ts.r.nAty = tmax(ts.r.nAty, tabs(Dinv * atyr));
                ts.c.nAty = tmax(ts.c.nAty, tabs(Dinv * atyc));
            }
        }
#pragma unroll
        for (int j = 0; j < NX; ++j) {
            T acc = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += m.A[i][j] * wv[i];
            rh[j] += Dx[j] * acc;
        }
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            T acc = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += m.B[i][j] * wv[i];
            rh[NX + j] += Du[j] * acc;
        }
    }
#pragma unroll
    for (int a = 0; a < NW; ++a) MPCB_AT(R, L::R_T + a) = rh[a];
#pragma unroll
    for (int i = 0; i < NX; ++i) { cy.xt_next[i] = w[i]; cy.Dx_next[i] = Dx[i]; }
    if (TEST) {
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            ts.x_next[i] = xn_a[i]; ts.dx_next[i] = dx_a[i];
            ts.own_r[i] = ownr_x[i]; ts.qpx_r[i] = qpx_x[i]; ts.own_c[i] = ownc_x[i];
        }
    }
}

// rows dyn_0 (header): updated after the backward sweep reached stage 0 (cy holds x~_0 and D_x(0))
template <typename T, typename L, bool FIRST, int MODE>
MPCB_HD void admm_bwd_header(const KParams<T>& p, const AdmmConst<T, L>& q, int b, T* H, const BwdCarry<T, L>& cy,
                             BwdTest<T, L>& ts) {
    constexpr bool first = FIRST;
#pragma unroll
    for (int i = 0; i < L::NX; ++i) {
        const T E0 = MPCB_AT(H, L::H_E0 + i);
        const T beq = -E0 * p.x_init[(size_t)i * p.ld + b];
        const Row<T> rw = row_state(first, MPCB_AT(H, L::H_P0 + i), first ? MPCB_AT(H, L::H_Y0 + i) : (T)0, beq, beq,
                                    q.rinv_eq());
        const T pn = row_next(-(E0 * cy.Dx_next[i]) * cy.xt_next[i], rw, q.alpha);
        MPCB_AT(H, L::H_P0 + i) = pn;
        if (MODE == kBwdTest) {     // rows dyn_0; column x_0 gets its row dyn_0
            const T ex = E0 * cy.Dx_next[i], Einv = fast_rcp(E0);
            const T axr = -ex * ts.x_next[i], axc = -ex * ts.dx_next[i];
            ts.r.pri = tmax(ts.r.pri, tabs(Einv * (axr - beq)));
            ts.r.nz = tmax(ts.r.nz, tabs(Einv * beq));
            ts.r.nAx = tmax(ts.r.nAx, tabs(Einv * axr));
            ts.c.aup = tmax(ts.c.aup, Einv * axc);
            ts.c.alo = tmin(ts.c.alo, Einv * axc);
            T wr = q.rho_eq * (pn - beq);
            T wc = wr;
            wc -= q.rho_eq * rw.yr;
            ts.c.nEw = tmax(ts.c.nEw, tabs(E0 * wc));
            ts.c.lhs += beq * wc;
            test_close_column(ts, i, ex, wr, wc, fast_rcp(cy.Dx_next[i]));
        }
    }
}

// Accumulators of the infeasibility certificates (auxil.c: is_primal_infeasible / is_dual_infeasible, paper
// eq. (22), (24)) over delta_y = y^k - y^{k-1} and delta_x = x^k - x^{k-1} of the iteration being tested.  The
// backward sweep of a tested iteration (kBwdTest) forms them from the old state in the records it reads; the CTA and
// dense kernels copy the pre-update state of that iteration into the old-state buffer O (the Ruiz scratch, free after
// setup): [x (VS) | p (CS)] per stage, rows in the form they had then (p-form; explicit z with y in the y rows on the
// first iteration of a solve).
template <typename T>
struct Cert {
    T ndy, lhs, nAtdy;            // ||E dy||_inf, u'max(dy,0) + l'min(dy,0), ||Dinv A'dy||_inf
    T ndx, qdx, nPdx, aup, alo;   // ||D dx||_inf, q'dx, ||Dinv P dx||_inf, max/min of Einv A dx over rows with finite u / l
};
template <typename T>
MPCB_HD bool cert_primal_infeasible(const Cert<T>& c, T eps) {
    return c.ndy > eps && c.lhs < -eps * c.ndy && c.nAtdy < eps * c.ndy;
}
template <typename T>
MPCB_HD bool cert_dual_infeasible(const Cert<T>& c, T cost_scaling, T eps) {
    return c.ndx > eps && c.qdx < -cost_scaling * eps * c.ndx && c.nPdx < cost_scaling * eps * c.ndx &&
           c.aup <= eps * c.ndx && c.alo >= -eps * c.ndx;
}

// y^{k-1}/rho of a row from its saved state
template <typename T>
MPCB_HD T old_yr(bool first, T p_old, T y_old, T lb, T ub, T rho_row) {
    if (first) return y_old * ((T)1 / rho_row);      // explicit y on entry of a solve (cold path: one FP64 division)
    return p_old - tmin(tmax(p_old, lb), ub);
}

// ---- the termination sweep of the CTA and dense kernels, one stage: the terms of BwdTest as a sweep of its own over the new
// state, once for each evaluation:
//   cert = false: the residuals of (x, y)
//   cert = true : the infeasibility certificates of (dx, dy), the old state read from the old-state buffer O
// The second evaluation re-runs the same instructions instead of adding as many again (the kernel's code footprint, not
// its flop count, is what the instruction cache of an SM with six warps at different places of a long unrolled loop
// feels).  The column sums are associated like the backward sweep's (test_close_column).
template <typename T, typename L>
struct TestCarry {
    T Ed_cur[L::NX], wd_cur[L::NX];          // E and w of rows dyn_k
};

template <typename T, typename L>
MPCB_HD void admm_test_stage(const KParams<T>& p, const AdmmConst<T, L>& q, const Model<T, L>& m, int b, int k,
                             const T* S, const T* Sn, TestCarry<T, L>& cy, TestAcc<T>& t, bool cert, bool first,
                             const T* Yk, const T* O, const T* On) {
    constexpr int NX = L::NX, NU = L::NU, NS = L::NS;
    const bool last = (k == p.N);
    const T* Qk = last ? p.QN : p.Q;
    T lo[NX], hi[NX];
    stage_box<T, L>(p, k, lo, hi);
    // the old state of the tested iteration comes from global memory (L2): a stage's loads are issued together
    T ox[L::VS], op[L::CS], onx[NX];
#pragma unroll
    for (int e = 0; e < L::VS; ++e) ox[e] = 0;
#pragma unroll
    for (int e = 0; e < L::CS; ++e) op[e] = 0;
#pragma unroll
    for (int i = 0; i < NX; ++i) onx[i] = 0;
    if (cert) {
#pragma unroll
        for (int e = 0; e < L::VS; ++e) ox[e] = MPCB_AT(O, e);
#pragma unroll
        for (int e = 0; e < L::CS; ++e) op[e] = MPCB_AT(O, L::VS + e);
        if (!last) {
#pragma unroll
            for (int i = 0; i < NX; ++i) onx[i] = MPCB_AT(On, L::OX + i);
        }
    }
    T vx[NX], Dx[NX], vu[NU], Du[NU], w_next[NX], Ed_next[NX], wy[NX];
#pragma unroll
    for (int j = 0; j < NX; ++j) { vx[j] = MPCB_AT(S, L::R_X + L::OX + j) - ox[L::OX + j]; Dx[j] = MPCB_AT(S, L::R_D + L::OX + j); }
#pragma unroll
    for (int j = 0; j < NU; ++j) {
        vu[j] = last ? (T)0 : MPCB_AT(S, L::R_X + L::OU + j) - ox[L::OU + j];
        Du[j] = last ? (T)1 : MPCB_AT(S, L::R_D + L::OU + j);
    }
    if (k == 0) {
#pragma unroll
        for (int i = 0; i < NX; ++i) {
            const T Einv = fast_rcp(cy.Ed_cur[i]);
            const T ax = -(cy.Ed_cur[i] * Dx[i]) * vx[i], zz = -cy.Ed_cur[i] * p.x_init[(size_t)i * p.ld + b];
            const T zr = cert ? (T)0 : Einv * zz;
            t.pri = tmax(t.pri, tabs(Einv * (cert ? ax : ax - zz)));
            t.nz = tmax(t.nz, tabs(zr));
            t.nAx = tmax(t.nAx, tabs(Einv * ax));
            t.aup = tmax(t.aup, Einv * ax);
            t.alo = tmin(t.alo, Einv * ax);
        }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) {
        if (!last) {
            Ed_next[i] = MPCB_AT(S, L::R_E + L::ODN + i);
            const T beq = -Ed_next[i] * model_g<T, L>(p, b, k, i);
            const T pd = MPCB_AT(S, L::R_P + L::ODN + i);
            T w = q.rho_eq * (pd - beq);
            if (cert) w -= q.rho_eq * old_yr(first, op[L::ODN + i], first ? MPCB_AT(Yk, L::ODN + i) : (T)0, beq, beq, q.rho_eq);
            w_next[i] = w;
            T acc = 0;
#pragma unroll
            for (int j = 0; j < NX; ++j) acc += m.A[i][j] * (Dx[j] * vx[j]);
#pragma unroll
            for (int j = 0; j < NU; ++j) acc += m.B[i][j] * (Du[j] * vu[j]);
            const T exn = Ed_next[i] * MPCB_AT(Sn, L::R_D + L::OX + i);
            const T ax = Ed_next[i] * acc - exn * (MPCB_AT(Sn, L::R_X + L::OX + i) - onx[i]);
            const T Einv = fast_rcp(Ed_next[i]);
            const T zb = cert ? (T)0 : beq;
            t.pri = tmax(t.pri, tabs(Einv * (ax - zb)));
            t.nz = tmax(t.nz, tabs(Einv * zb));
            t.nAx = tmax(t.nAx, tabs(Einv * ax));
            t.aup = tmax(t.aup, Einv * ax);
            t.alo = tmin(t.alo, Einv * ax);
            t.nEw = tmax(t.nEw, tabs(Ed_next[i] * w));
            t.lhs += beq * w;
        } else {
            Ed_next[i] = 1; w_next[i] = 0;
        }
        wy[i] = Ed_next[i] * w_next[i];
    }
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        const T Dinv = fast_rcp(Dx[j]);
        const T Ebx = MPCB_AT(S, L::R_E + L::OBX + j), Einv = fast_rcp(Ebx);
        const T bx = Ebx * Dx[j], lb = Ebx * lo[j], ub = Ebx * hi[j];
        const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
        const T pp = MPCB_AT(S, L::R_P + L::OBX + j);
        const T zbx = tmin(tmax(pp, lb), ub);
        T wbx = rb * (pp - zbx);
        if (cert) {
            wbx -= rb * old_yr(first, op[L::OBX + j], first ? MPCB_AT(Yk, L::OBX + j) : (T)0, lb, ub, rb);
            wbx = cert_project(q.inf_bounds, wbx, lb, ub);
        }
        T vs = 0, bs = 0;
        if (NS) {
            vs = MPCB_AT(S, L::R_X + L::OS + (NS ? j : 0)) - ox[L::OS + (NS ? j : 0)];
            bs = p.S[j] * Ebx * MPCB_AT(S, L::R_D + L::OS + (NS ? j : 0));
        }
        const T ax = bx * vx[j] + bs * vs;
        const T zb = cert ? (T)0 : zbx;
        t.pri = tmax(t.pri, tabs(Einv * (ax - zb)));
        t.nz = tmax(t.nz, tabs(Einv * zb));
        t.nAx = tmax(t.nAx, tabs(Einv * ax));
        if (!q.inf_bounds || ub < (T)(kOsqpInfty * kMinScaling)) t.aup = tmax(t.aup, Einv * ax);
        if (!q.inf_bounds || lb > (T)(-kOsqpInfty * kMinScaling)) t.alo = tmin(t.alo, Einv * ax);
        t.nEw = tmax(t.nEw, tabs(Ebx * wbx));
        t.lhs += ub * tmax(wbx, (T)0) + lb * tmin(wbx, (T)0);
        const T xr = p.xr_tv ? p.Xr[((size_t)k * NX + j) * p.ld + b] : q.xr[(size_t)j * q.xr_stride];
        const T qh = q.c * Dx[j] * (-(Qk[j] * xr));
        T acc = 0;
#pragma unroll
        for (int i = 0; i < NX; ++i) acc += m.A[i][j] * wy[i];
        T aty = bx * wbx;
        if (!last) aty += Dx[j] * acc;
        aty -= (cy.Ed_cur[j] * Dx[j]) * cy.wd_cur[j];
        const T px = q.c * Qk[j] * Dx[j] * Dx[j] * vx[j];
        t.dua = tmax(t.dua, tabs(Dinv * ((qh + px) + aty)));
        t.nq = tmax(t.nq, tabs(Dinv * qh));
        t.nAty = tmax(t.nAty, tabs(Dinv * aty));
        t.nPx = tmax(t.nPx, tabs(Dinv * px));
        t.nDv = tmax(t.nDv, tabs(Dx[j] * vx[j]));
        t.qv += qh * vx[j];
        if (NS) {
            const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? j : 0)), Dsinv = fast_rcp(Dsl);
            const T atys = bs * wbx, pxs = q.c * p.W[j] * Dsl * Dsl * vs;
            t.dua = tmax(t.dua, tabs(Dsinv * (atys + pxs)));
            t.nAty = tmax(t.nAty, tabs(Dsinv * atys));
            t.nPx = tmax(t.nPx, tabs(Dsinv * pxs));
            t.nDv = tmax(t.nDv, tabs(Dsl * vs));
        }
    }
    if (!last) {
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            const T Dinv = fast_rcp(Du[j]);
            const T Ebu = MPCB_AT(S, L::R_E + L::OBU + j), Einv = fast_rcp(Ebu);
            const T bu = Ebu * Du[j], lb = Ebu * p.umin[j], ub = Ebu * p.umax[j];
            const T rb = row_rho(q.inf_bounds, lb, ub, q.rho, q.rho_eq);
            const T pp = MPCB_AT(S, L::R_P + L::OBU + j);
            const T zbu = tmin(tmax(pp, lb), ub);
            T wbu = rb * (pp - zbu);
            if (cert) {
                wbu -= rb * old_yr(first, op[L::OBU + j], first ? MPCB_AT(Yk, L::OBU + j) : (T)0, lb, ub, rb);
                wbu = cert_project(q.inf_bounds, wbu, lb, ub);
            }
            const T ax = bu * vu[j];
            const T zb = cert ? (T)0 : zbu;
            t.pri = tmax(t.pri, tabs(Einv * (ax - zb)));
            t.nz = tmax(t.nz, tabs(Einv * zb));
            t.nAx = tmax(t.nAx, tabs(Einv * ax));
            if (!q.inf_bounds || ub < (T)(kOsqpInfty * kMinScaling)) t.aup = tmax(t.aup, Einv * ax);
            if (!q.inf_bounds || lb > (T)(-kOsqpInfty * kMinScaling)) t.alo = tmin(t.alo, Einv * ax);
            t.nEw = tmax(t.nEw, tabs(Ebu * wbu));
            t.lhs += ub * tmax(wbu, (T)0) + lb * tmin(wbu, (T)0);
            T acc = 0;
#pragma unroll
            for (int i = 0; i < NX; ++i) acc += m.B[i][j] * wy[i];
            T aty = bu * wbu;
            aty += Du[j] * acc;
            const T px = q.c * p.R[j] * Du[j] * Du[j] * vu[j];
            t.dua = tmax(t.dua, tabs(Dinv * (aty + px)));
            t.nAty = tmax(t.nAty, tabs(Dinv * aty));
            t.nPx = tmax(t.nPx, tabs(Dinv * px));
            t.nDv = tmax(t.nDv, tabs(Du[j] * vu[j]));
        }
    }
#pragma unroll
    for (int i = 0; i < NX; ++i) { cy.Ed_cur[i] = Ed_next[i]; cy.wd_cur[i] = w_next[i]; }
}

// ---- exit pass: leave explicit (z, y) behind for the next solve and the gather, one stage
template <typename T, typename L>
MPCB_HD void admm_exit_stage(const KParams<T>& p, const AdmmConst<T, L>& q, int b, int k, T* R, T* Yk) {
    constexpr int NX = L::NX, NU = L::NU;
    const bool last = (k == p.N);
    T lo[NX], hi[NX];
    stage_box<T, L>(p, k, lo, hi);
#pragma unroll
    for (int j = 0; j < NX; ++j) {
        const T Ebx = MPCB_AT(R, L::R_E + L::OBX + j);
        const T lb = Ebx * lo[j], ub = Ebx * hi[j];
        const T rb = row_rho(lb, ub, q.rho, q.rho_eq);
        const T pp = MPCB_AT(R, L::R_P + L::OBX + j);
        const T z = tmin(tmax(pp, lb), ub);
        MPCB_AT(R, L::R_P + L::OBX + j) = z;
        MPCB_AT(Yk, L::OBX + j) = rb * (pp - z);
        if (!last) {
            const T beq = -MPCB_AT(R, L::R_E + L::ODN + j) * model_g<T, L>(p, b, k, j);
            const T pd = MPCB_AT(R, L::R_P + L::ODN + j);
            MPCB_AT(R, L::R_P + L::ODN + j) = beq;
            MPCB_AT(Yk, L::ODN + j) = q.rho_eq * (pd - beq);
        }
    }
    if (!last) {
#pragma unroll
        for (int j = 0; j < NU; ++j) {
            const T Ebu = MPCB_AT(R, L::R_E + L::OBU + j);
            const T lb = Ebu * p.umin[j], ub = Ebu * p.umax[j];
            const T rb = row_rho(lb, ub, q.rho, q.rho_eq);
            const T pp = MPCB_AT(R, L::R_P + L::OBU + j);
            const T z = tmin(tmax(pp, lb), ub);
            MPCB_AT(R, L::R_P + L::OBU + j) = z;
            MPCB_AT(Yk, L::OBU + j) = rb * (pp - z);
        }
    }
}

}  // namespace mpcb
