// Everything of the library that is instantiated per compiled (nx, nu, slack) shape and dtype: the per-QP kernels, the
// ADMM launchers and the host-side ADMM loop.  A translation unit (shape_tu.cu) instantiates ONE (shape, dtype) and
// exports its entry points as a ShapeOps table; the ABI layer (mpc_b200.cu) looks the table up.  Splitting the
// library this way lets the build compile the shapes in parallel (the ADMM kernels are tens of KB of straight-line
// SASS per instantiation).
#pragma once
#include <chrono>
#include "runtime.cuh"
#include "admm_kernel.cuh"
#include "admm_dense.cuh"
#include "admm_cta.cuh"
#include "setup_warp.cuh"

// Explicit QP data in the reference's ordering (see mpcb_build_qp in the header).
struct BuildOut {
    void *Pdiag, *q, *Avals, *l, *u;
};

// The Ruiz scalings in the reference's ordering (see mpcb_get_scaling in the header).
struct ScalingOut {
    void *D, *E, *c;
};

// entry points of one compiled (shape, dtype)
struct ShapeOps {
    int nx, nu, slack, dtype;
    int (*setup)(mpcb_solver* s, rt_stream st);                                             // Ruiz scaling + factorisation
    int (*refactor)(mpcb_solver* s, const mpcb_problem* np, void* new_box, rt_stream st);   // after a bound update
    int (*run_admm)(mpcb_solver* s, int max_iter, int check_every, int warm, rt_stream st);
    int (*cold_start)(mpcb_solver* s, rt_stream st);
    int (*build_qp)(mpcb_solver* s, const BuildOut* o, rt_stream st);
    int (*get_scaling)(mpcb_solver* s, const ScalingOut* o, rt_stream st);
};

// =============================================================================================
// per-QP kernel bodies
// =============================================================================================
struct ScaleOp { static const char* name() { return "scale"; } template <typename T, typename L> static MPCB_HD void run(const KParams<T>& p, int b) { scale_one<T, L>(p, b); } };
struct FactorOp { static const char* name() { return "factor"; } template <typename T, typename L> static MPCB_HD void run(const KParams<T>& p, int b) { factor_one<T, L>(p, b); } };
struct AdmmOp { static const char* name() { return "admm"; } template <typename T, typename L> static MPCB_HD void run(const KParams<T>& p, int b) { admm_one<T, L>(p, b); } };
struct ColdOp { static const char* name() { return "cold_start"; } template <typename T, typename L> static MPCB_HD void run(const KParams<T>& p, int b) { Ws<T, L> ws(p, b); admm_cold_start<T, L>(p, ws); } };

template <typename T, typename L>
MPCB_HD void build_one(const KParams<T>& p, const BuildOut& o, int b) {
    constexpr int NX = L::NX, NU = L::NU, NS = L::NS;
    const int N = p.N;
    const size_t ld = p.ld;
    T* Pd = (T*)o.Pdiag; T* q = (T*)o.q; T* Av = (T*)o.Avals; T* lo = (T*)o.l; T* up = (T*)o.u;
    const size_t ux0 = (size_t)(N + 1) * NX, sx0 = ux0 + (size_t)N * NU;      // variable offsets
    const size_t bx0 = (size_t)(N + 1) * NX, bu0 = 2 * (size_t)(N + 1) * NX;  // row offsets
    // CSC value offsets: x columns of stage k<N hold (2+NX) values, of stage N hold 2; u columns NX+1; s columns 1
    const size_t nnz_x = (size_t)N * NX * (2 + NX) + (size_t)NX * 2;
    const size_t nnz_u = (size_t)N * NU * (NX + 1);
    Model<T, L> m;
    if (!p.tv) load_model<T, L>(p, b, 0, m);
    for (int k = 0; k <= N; ++k) {
        const bool last = (k == N);
        if (p.tv && !last) load_model<T, L>(p, b, k, m);
        const T* Qk = last ? p.QN : p.Q;
        T blo[NX], bhi[NX];
        for (int i = 0; i < NX; ++i) {
            blo[i] = p.xbox ? p.xbox[(k * 2 + 0) * NX + i] : p.xmin[i];
            bhi[i] = p.xbox ? p.xbox[(k * 2 + 1) * NX + i] : p.xmax[i];
        }
        for (int j = 0; j < NX; ++j) {
            const size_t v = (size_t)k * NX + j;
            const T xr = p.Xr[((p.xr_tv ? (size_t)k * NX : 0) + j) * ld + b];
            if (Pd) Pd[v * ld + b] = Qk[j];
            if (q) q[v * ld + b] = -(Qk[j] * xr);
            if (Av) {
                size_t a = (size_t)k * NX * (2 + NX) + (size_t)j * (last ? 2 : 2 + NX);
                Av[a++ * ld + b] = (T)-1;
                if (!last)
                    for (int i = 0; i < NX; ++i) Av[a++ * ld + b] = m.A[i][j];
                Av[a * ld + b] = (T)1;
            }
            // rows dyn_k, bx_k
            const T beq = k == 0 ? -p.x_init[(size_t)j * ld + b] : (T)0;   // dyn_k for k>0 written below via g_{k-1}
            if (k == 0) { if (lo) lo[v * ld + b] = beq; if (up) up[v * ld + b] = beq; }
            if (!last) {
                const size_t r = (size_t)(k + 1) * NX + j;
                if (lo) lo[r * ld + b] = -model_g<T, L>(p, b, k, j);
                if (up) up[r * ld + b] = -model_g<T, L>(p, b, k, j);
            }
            if (lo) lo[(bx0 + v) * ld + b] = blo[j];
            if (up) up[(bx0 + v) * ld + b] = bhi[j];
            if (NS) {
                const size_t sv = sx0 + v;
                if (Pd) Pd[sv * ld + b] = p.W[j];
                if (q) q[sv * ld + b] = (T)0;
                if (Av) Av[(nnz_x + nnz_u + v) * ld + b] = p.S[j];
            }
        }
        if (!last) {
            for (int j = 0; j < NU; ++j) {
                const size_t v = ux0 + (size_t)k * NU + j;
                if (Pd) Pd[v * ld + b] = p.R[j];
                if (q) q[v * ld + b] = (T)0;
                if (Av) {
                    size_t a = nnz_x + ((size_t)k * NU + j) * (NX + 1);
                    for (int i = 0; i < NX; ++i) Av[a++ * ld + b] = m.B[i][j];
                    Av[a * ld + b] = (T)1;
                }
                if (lo) lo[(bu0 + (size_t)k * NU + j) * ld + b] = p.umin[j];
                if (up) up[(bu0 + (size_t)k * NU + j) * ld + b] = p.umax[j];
            }
        }
    }
}

template <typename T, typename L>
struct BuildFn {
    KParams<T> p;
    BuildOut o;
    MPCB_HD void operator()(int b) const { build_one<T, L>(p, o, b); }
};

// D, E, c of one QP from its home records and header, batch-major in the reference's ordering.  The slots without a
// variable or row in the reference (u_N, dyn_{N+1} and bu_N of stage N) are skipped.
template <typename T, typename L>
MPCB_HD void scaling_one(const KParams<T>& p, const ScalingOut& o, int b) {
    constexpr int NX = L::NX, NU = L::NU, NS = L::NS;
    const int N = p.N;
    const size_t nvar = (size_t)L::nvar(N), ncon = (size_t)L::ncon(N);
    const size_t ux0 = (size_t)(N + 1) * NX, sx0 = ux0 + (size_t)N * NU;      // variable offsets
    const size_t bx0 = (size_t)(N + 1) * NX, bu0 = 2 * (size_t)(N + 1) * NX;  // row offsets
    T* D = o.D ? (T*)o.D + (size_t)b * nvar : nullptr;
    T* E = o.E ? (T*)o.E + (size_t)b * ncon : nullptr;
    const Ws<T, L> ws(p, b);
    for (int k = 0; k <= N; ++k) {
        const T* R = ws.R(k);
        for (int j = 0; j < NX; ++j) {
            if (D) D[(size_t)k * NX + j] = MPCB_AT(R, L::R_D + L::OX + j);
            if (D && NS) D[sx0 + (size_t)k * NX + j] = MPCB_AT(R, L::R_D + L::OS + (NS ? j : 0));
            if (E && k < N) E[(size_t)(k + 1) * NX + j] = MPCB_AT(R, L::R_E + L::ODN + j);
            if (E) E[bx0 + (size_t)k * NX + j] = MPCB_AT(R, L::R_E + L::OBX + j);
        }
        if (k < N)
            for (int j = 0; j < NU; ++j) {
                if (D) D[ux0 + (size_t)k * NU + j] = MPCB_AT(R, L::R_D + L::OU + j);
                if (E) E[bu0 + (size_t)k * NU + j] = MPCB_AT(R, L::R_E + L::OBU + j);
            }
    }
    if (E)
        for (int i = 0; i < NX; ++i) E[i] = MPCB_AT(ws.hdr, L::H_E0 + i);        // rows dyn_0 live in the header
    if (o.c) ((T*)o.c)[b] = MPCB_AT(ws.hdr, L::H_C);
}

template <typename T, typename L>
struct ScalingFn {
    KParams<T> p;
    ScalingOut o;
    MPCB_HD void operator()(int b) const { scaling_one<T, L>(p, o, b); }
};

// osqp_update_bounds (osqp.c) + update_rho_vec (auxil.c) for one QP: did a bound row change its type between the old and
// the new bounds?  The rows' rho is a function of the scaled bounds (row_rho), evaluated on the fly by every kernel, so
// the cached factor must be rebuilt exactly when OSQP rebuilds its KKT matrix.
template <typename T, typename L>
MPCB_HD bool bounds_change_row_types(const KParams<T>& po, const KParams<T>& pn, int b) {
    constexpr int NX = L::NX, NU = L::NU;
    Ws<T, L> ws(pn, b);
    const T rho = clamp_rho(pn.rho), rho_eq = (T)kRhoEqOverRhoIneq * rho;
    bool changed = false;
    for (int k = 0; k <= pn.N; ++k) {
        const T* R = ws.R(k);
        T lo0[NX], hi0[NX], lo1[NX], hi1[NX];
        stage_box<T, L>(po, k, lo0, hi0);
        stage_box<T, L>(pn, k, lo1, hi1);
        for (int j = 0; j < NX; ++j) {
            const T E = MPCB_AT(R, L::R_E + L::OBX + j);
            changed |= row_rho(E * lo0[j], E * hi0[j], rho, rho_eq) != row_rho(E * lo1[j], E * hi1[j], rho, rho_eq);
        }
        if (k < pn.N)
            for (int j = 0; j < NU; ++j) {
                const T E = MPCB_AT(R, L::R_E + L::OBU + j);
                changed |= row_rho(E * po.umin[j], E * po.umax[j], rho, rho_eq) !=
                           row_rho(E * pn.umin[j], E * pn.umax[j], rho, rho_eq);
            }
    }
    return changed;
}
template <typename T, typename L>
struct RefactorFn {
    KParams<T> po, pn;
    MPCB_HD void operator()(int b) const {
        if (bounds_change_row_types<T, L>(po, pn, b)) factor_one<T, L>(pn, b);
    }
};

// The ADMM launch: warp-per-tile with TMA-staged stage records when two record buffers per warp fit in
// shared memory (every shape of the reference does), else one lane per QP straight from global memory.
// MPCB_NO_TMA=1 forces the latter (used to cross-check the two kernels in tests).
template <typename T, typename L>
static int launch_admm(const KParams<T>& p, mpcb_solver* s, rt_stream st) {
#ifndef MPCB_EMU
    const bool no_tma = g_opt_tma.load() == 0;
    const int max_smem = s->dev_max_smem, sms = s->dev_sms;      // of the solver's own device (queried at mpcb_create)
    const size_t per_warp = 2 * (size_t)L::REC * TILE * sizeof(T) + 16;      // two record buffers + two mbarriers
    int warps = (int)(((size_t)max_smem - 128 - 16) / per_warp);
    if (warps > 8) warps = 8;
    if (!no_tma && warps >= 2) {
        const int warps_max = warps;
        RT_CHECK(cudaFuncSetAttribute(admm_tma_kernel<T, L>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)((size_t)max_smem - 128)));
        const int ntiles = (p.B + TILE - 1) / TILE;
        // few tiles (small batches, the straggler launch after a re-tiling): spread them over the SMs with fewer
        // warps per CTA instead of packing them on a handful of SMs — such launches are latency-bound
        int wpc = (ntiles + sms - 1) / sms;
        if (wpc > warps) wpc = warps;
        warps = wpc < 1 ? 1 : wpc;
        int grid = (ntiles + warps - 1) / warps;
        if (grid > sms) grid = sms;              // persistent CTAs, one per SM; work items are handed out dynamically
        // behind the buffers: a slice per warp for the per-QP reference (used when it does not cost a warp of shared
        // memory at full occupancy; the slot is laid out either way) and 16 bytes for the CTA's round counter
        KParams<T> pk = p;
        // Work items are (tile, chunk_len iterations).  A launch ends when its last items do, and a warp needs ~0.1 ms per
        // iteration of a tile however empty the GPU is: with items of a whole check interval the last wave of e.g. 2011 tiles
        // on 888 warps (the second launch of a warm-started closed-loop step) runs a quarter full for 2.6 ms.  Launches of
        // one to four waves get items of 5 iterations (measured: that launch 8.45 -> 7.6 ms); longer launches keep 25 — an
        // item costs ~3 % of five iterations in set-up (the headline's phase 1: 21.3 vs 21.6 ms).
        {
            const int span = p.it_stop - p.it0, cl = p.chunk_len > 0 && p.chunk_len < span ? p.chunk_len : span;
            const long long items = (long long)((span + cl - 1) / cl) * ntiles, total_warps = (long long)grid * warps;
            static const int fine = std::getenv("MPCB_CHUNK_FINE") ? std::atoi(std::getenv("MPCB_CHUNK_FINE")) : 5;
            // (only where every warp has a tile: below that the launch is latency-bound and finer items cost 1-1.5 %)
            if (fine > 0 && fine < cl && ntiles >= total_warps && items < 4 * total_warps) pk.chunk_len = fine;
        }
        const size_t xr_bytes = (size_t)L::NX * TILE * sizeof(T);
        pk.xr_smem = (!p.xr_tv && (size_t)warps_max * (per_warp + xr_bytes) + 16 + 128 <= (size_t)max_smem) ? 1 : 0;
        const size_t smem = (size_t)warps * per_warp + (pk.xr_smem ? (size_t)warps * xr_bytes : 0) + 16;
        if (int r = rt_memset(s->tile_counter, 0, sizeof(int), st)) return r;
        if (int r = rt_memset(s->tile_prog, 0, (size_t)ntiles * sizeof(int), st)) return r;
        admm_tma_kernel<T, L><<<grid, warps * 32, smem, st>>>(pk, s->tile_counter);
        ++g_launches;
        return rt_launch_check("admm_tma");
    }
#endif
    (void)s;
    return launch_qp<AdmmOp, T, L>(p, st);
}

// ---- CTA-per-tile kernel (admm_cta.cuh) ------------------------------------------------------------------------------
#ifndef MPCB_EMU
template <typename T, typename L>
static bool cta_fits(const mpcb_solver* s, bool tv) {
    const size_t need = tv ? CtaSmem<T, L, true>::BYTES : CtaSmem<T, L, false>::BYTES;
    return need + 1024 <= (size_t)s->dev_max_smem;
}
#endif
// tile a time-varying model (and the stage references) like the records: mdl[((tile*(N+1) + k)*COUNT + e)*32 + lane]
template <typename T, typename L>
static int tile_model(mpcb_solver* s, const KParams<T>& p, rt_stream st) {
#ifndef MPCB_EMU
    typedef CtaModel<L> CM;
    const int N = p.N, S1 = N + 1, ntiles = (p.B + TILE - 1) / TILE;
    const size_t need = (size_t)ntiles * S1 * CM::COUNT * TILE * sizeof(T);
    if (s->mdl_bytes < need) {
        rt_free(s->mdl); s->mdl = nullptr; s->mdl_bytes = 0;
        const size_t cap_tiles = (s->ld + TILE - 1) / TILE;
        const size_t want = cap_tiles * S1 * CM::COUNT * TILE * sizeof(T);
        if (int r = rt_malloc(&s->mdl, want)) return r;
        s->mdl_bytes = want;
        s->ws_bytes += want;
    }
    T* mdl = (T*)s->mdl;
    const T* Ad = p.Ad; const T* Bd = p.Bd; const T* gd = p.gd; const T* Xr = p.Xr;
    const size_t ld = p.model_bs ? p.ld : 1, ldx = p.ld;
    const int bs = p.model_bs, B = p.B, xr_tv = p.xr_tv;
    const size_t total = (size_t)ntiles * S1 * CM::COUNT * TILE;
    if (total > 0x7fffffffull) return fail(MPCB_E_ARG, "time-varying model too large to tile");
    return launch_1d((int)total, st, MPCB_LAMBDA(int idx) {
        const int lane = idx & 31;
        int r = idx >> 5;
        const int e = r % CM::COUNT; r /= CM::COUNT;
        const int k = r % S1, tile = r / S1;
        int b = tile * TILE + lane;
        if (b >= B) b = B - 1;
        const size_t bo = bs ? (size_t)b : 0;
        T v = 0;
        if (e >= CM::M_XR) v = Xr[((xr_tv ? (size_t)k * L::NX : 0) + (e - CM::M_XR)) * ldx + b];
        else if (k < N) {
            if (e < CM::M_G) {
                const int i = e / L::NW, j = e % L::NW;
                v = j < L::NX ? Ad[((size_t)k * L::NX * L::NX + i * L::NX + j) * ld + bo]
                              : Bd[((size_t)k * L::NX * L::NU + i * L::NU + (j - L::NX)) * ld + bo];
            } else v = gd ? gd[((size_t)k * L::NX + (e - CM::M_G)) * ld + bo] : (T)0;
        }
        mdl[idx] = v;
    });
#else
    (void)s; (void)p; (void)st;
    return 0;
#endif
}
template <typename T, typename L>
static bool cta_applicable(const mpcb_solver* s, const KParams<T>& p) {
#ifndef MPCB_EMU
    return g_opt_cta.load() != 0 && cta_fits<T, L>(s, p.tv != 0) && !(p.tv && !p.mdl);
#else
    (void)s; (void)p;
    return false;
#endif
}
// Which solves go to admm_cta_kernel: time-varying problems; time-invariant batches that fit the GPU in one wave of CTAs
// (two per SM: 9472 QPs on 148 SMs) — below that the warp-per-tile kernel runs at one or two warps per SM, 104 us per
// iteration; the CTA kernel needs 45 us per iteration up to one tile per SM and ~65 us at two (scripts/strong_probe.py:
// 4.7 vs 5.3 ms per step at 256..2048 QPs, 4.7 vs 8.1 ms at 4096, 7.0 vs 8.7 ms at 8192; a second wave loses: 11.6 vs
// ~9 ms at 10240); everything with "cta" = 2.
template <typename T, typename L>
static bool cta_planned(const mpcb_solver* s, int B, bool tv, int check_every) {
    const int opt = g_opt_cta.load();
    const bool window = !tv && opt == 1 && B <= 2 * s->dev_sms * TILE && L::NW <= 8;
    return (tv || opt == 2 || window) && opt != 0 && check_every > 0;
}
// The factor block of the records comes in two forms (KParams::minv): Linv_k for the sweeps that solve with the two
// triangles one after the other, Linv_k' Linv_k for admm_cta_kernel.  A solve that takes the other path than the previous
// one re-runs the factorisation (same inputs, same Linv to the bit).
template <typename T, typename L>
static int ensure_factor_form(mpcb_solver* s, KParams<T>& p, bool minv, rt_stream st) {
    if (s->rec_minv == minv) return 0;
    s->rec_minv = minv;
    p.minv = minv ? 1 : 0;
    KParams<T> pf = make_params<T>(s);
    return launch_qp<FactorOp, T, L>(pf, st);
}
// Factor blocks of a (re-tiled) workspace from Linv to Linv' Linv in place: one thread per (QP, stage).  The stragglers of a
// large batch finish in admm_cta_kernel; their home records keep Linv (un-tiling copies iterates only).
template <typename T, typename L>
struct MinvFromLinvFn {
    T* rec; int S1, n;
    MPCB_HD void operator()(int idx) const {
        constexpr int NW = L::NW;
        const int j = idx % n, k = idx / n;                     // slot fastest: coalesced over the lanes of a tile
        T* R = rec + (((size_t)(j >> 5) * S1 + k) * L::REC) * TILE + (j & 31);
        T Li[L::LT];
#pragma unroll
        for (int e = 0; e < L::LT; ++e) Li[e] = MPCB_AT(R, L::R_F + e);
#pragma unroll
        for (int a = 0; a < NW; ++a)
#pragma unroll
            for (int d = 0; d <= a; ++d) {
                T acc = 0;
#pragma unroll
                for (int e = a; e < NW; ++e) acc += Li[e * (e + 1) / 2 + a] * Li[e * (e + 1) / 2 + d];
                MPCB_AT(R, L::R_F + a * (a + 1) / 2 + d) = acc;
            }
    }
};
// Iterations it0+1 .. it_stop with the CTA-per-tile kernel.  Returns 1 when not applicable, -1 on error.
template <typename T, typename L>
static int launch_cta(const KParams<T>& p, mpcb_solver* s, rt_stream st) {
#ifndef MPCB_EMU
    const bool tv = p.tv != 0;
    if (!cta_applicable<T, L>(s, p) || !p.minv) return 1;
    const int ntiles = (p.B + TILE - 1) / TILE;
    cudaError_t e;
    // at most one tile per SM: the deep-prefetch instantiation (latency-bound launches; admm_cta.cuh)
    const bool deep = ntiles <= s->dev_sms && std::getenv("MPCB_NO_CTA_DEEP") == nullptr &&
                      (tv ? CtaSmem<T, L, true, CTA_NBUF_DEEP>::BYTES : CtaSmem<T, L, false, CTA_NBUF_DEEP>::BYTES) + 1024 <= (size_t)s->dev_max_smem;
    auto go = [&](auto kernel, size_t bytes) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e == cudaSuccess) kernel<<<ntiles, L::NW * 32, bytes, st>>>(p);
    };
    if (tv) {
        if (deep) go(admm_cta_kernel<T, L, true, CTA_NBUF_DEEP>, CtaSmem<T, L, true, CTA_NBUF_DEEP>::BYTES);
        else go(admm_cta_kernel<T, L, true, CTA_NBUF>, CtaSmem<T, L, true, CTA_NBUF>::BYTES);
    } else {
        if (deep) go(admm_cta_kernel<T, L, false, CTA_NBUF_DEEP>, CtaSmem<T, L, false, CTA_NBUF_DEEP>::BYTES);
        else go(admm_cta_kernel<T, L, false, CTA_NBUF>, CtaSmem<T, L, false, CTA_NBUF>::BYTES);
    }
    if (e != cudaSuccess) { fail(MPCB_E_CUDA, std::string("admm_cta: ") + cudaGetErrorString(e)); return -1; }
    ++g_launches;
    return rt_launch_check("admm_cta") ? -1 : 0;
#else
    (void)p; (void)s; (void)st;
    return 1;
#endif
}

// ---- shared-KKT dense path (admm_dense.cuh) ------------------------------------------------------------------------
template <typename T, typename L>
struct SameScalingFn {
    KParams<T> p;
    int* flag;
    MPCB_HD void operator()(int b) const { if (!dense_same_scaling<T, L>(p, b)) *flag = 1; }
};
template <typename T, typename L>
struct InverseColumnFn {
    KParams<T> p;
    T* Minv; T* tbuf;
    int nwp, nw;
    MPCB_HD void operator()(int col) const { dense_inverse_column<T, L>(p, col, Minv, nwp, tbuf + (size_t)col * nw); }
};
// the static part of that decision (what the setup can know before the scalings exist)
template <typename T, typename L>
static bool dense_candidate(const mpcb_solver* s) {
#ifndef MPCB_EMU
    if constexpr (std::is_same<T, double>::value) {
        const int N = s->prob.horizon, nwp = dense_nwp(N, L::NW);
        return (s->prob.shared_model || s->batch == 1) && N + 1 <= 32 && nwp <= DENSE_MAX_NW && g_opt_dense.load() != 0 &&
               s->batch <= 16384 && dense_smem_bytes(nwp, DenseC<L>::COUNT) + 1024 <= (size_t)s->dev_max_smem;
    }
#endif
    (void)s;
    return false;
}
// Decide (once per setup / bound update) whether the batch shares one KKT matrix, and if so form its inverse.
// One read-back of a flag; the inverse is (N+1)(nx+nu) independent structured solves with the cached factor.
template <typename T, typename L>
static int dense_prepare(mpcb_solver* s, rt_stream st) {
    if (s->dense_state != 0) return 0;
    s->dense_state = -1;
#ifndef MPCB_EMU
    if constexpr (std::is_same<T, double>::value) {
        const int N = s->prob.horizon, nw = (N + 1) * L::NW, nwp = dense_nwp(N, L::NW);
        // one linearisation for the whole batch — or a batch of one (the single-vehicle calls of the reference's mpc functions)
        if (!dense_candidate<T, L>(s)) return 0;
        KParams<T> p = make_params<T>(s);
        if (!s->dense_flag) if (int r = rt_malloc((void**)&s->dense_flag, 64)) return r;
        if (int r = rt_memset(s->dense_flag, 0, sizeof(int), st)) return r;
        if (int r = launch_1d(p.B, st, SameScalingFn<T, L>{p, s->dense_flag})) return r;
        int differs = 0;
        if (int r = rt_d2h(&differs, s->dense_flag, sizeof(int), st)) return r;
        if (int r = rt_sync(st)) return r;
        if (differs) return 0;
        const size_t bytes = (size_t)nwp * nwp * sizeof(T);
        if (s->dense_bytes < 2 * bytes) {
            rt_free(s->dense_minv); s->dense_minv = nullptr; s->dense_bytes = 0;
            if (int r = rt_malloc(&s->dense_minv, 2 * bytes)) return r;
            s->dense_bytes = 2 * bytes;
        }
        if (int r = rt_memset(s->dense_minv, 0, 2 * bytes, st)) return r;
        T* Minv = (T*)s->dense_minv;
        if (int r = launch_1d(nw, st, InverseColumnFn<T, L>{p, Minv, Minv + (size_t)nwp * nwp, nwp, nw})) return r;
        s->dense_state = 1;
    }
#endif
    return 0;
}
// The ADMM loop of a batch that shares one KKT matrix (admm_dense_kernel).  Returns 1 when not applicable.
template <typename T, typename L>
static int launch_dense(const KParams<T>& p, mpcb_solver* s, rt_stream st) {
#ifndef MPCB_EMU
    if constexpr (std::is_same<T, double>::value) {
        if (s->dense_state != 1) return 1;
        const int nwp = dense_nwp(p.N, L::NW);
        const size_t smem = dense_smem_bytes(nwp, DenseC<L>::COUNT);
        if (cudaFuncSetAttribute(admm_dense_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            fail(MPCB_E_CUDA, "cudaFuncSetAttribute(admm_dense_kernel)");
            return -1;
        }
        admm_dense_kernel<L><<<(p.B + DENSE_QPB - 1) / DENSE_QPB, DENSE_QPB * 32, smem, st>>>(p, (const double*)s->dense_minv, nwp);
        ++g_launches;
        return rt_launch_check("admm_dense") ? -1 : 0;
    }
#endif
    (void)p; (void)s; (void)st;
    return 1;
}

// copy the workspace columns of the surviving QPs from the home workspace into dense tiles of the scratch one
// (records and headers; the duals y are not needed: unsolved rows are in p-form)
template <typename T>
static int retile_impl(mpcb_solver* s, int n, const int* list, rt_stream st) {
    const size_t S1 = (size_t)(s->prob.horizon + 1), REC = (size_t)s->REC, HDR = (size_t)s->HDR;
    const T* rec = (const T*)s->rec; const T* hdr = (const T*)s->hdr;
    T* rec2 = (T*)s->rec2; T* hdr2 = (T*)s->hdr2;
    const int per = (int)(S1 * REC + HDR);
    // thread = (element, destination slot) with the slot fastest: destination writes are coalesced
    return launch_1d(n * per, st, MPCB_LAMBDA(int idx) {
        const int e = idx / n, j = idx - e * n;
        const int b = list[j];
        const size_t ts = (size_t)(b >> 5), ls = (size_t)(b & 31), td = (size_t)(j >> 5), ldn = (size_t)(j & 31);
        if ((size_t)e < S1 * REC) rec2[(td * S1 * REC + e) * TILE + ldn] = rec[(ts * S1 * REC + e) * TILE + ls];
        else { const size_t h = (size_t)e - S1 * REC; hdr2[(td * HDR + h) * TILE + ldn] = hdr[(ts * HDR + h) * TILE + ls]; }
    });
}
// bring x, z, y of the re-tiled QPs back to their home columns, and the t slots with them: they hold r^ of an unsolved
// QP (mpc_common.h), which a later compaction copies from the home workspace
template <typename T>
static int untile_impl(mpcb_solver* s, int n, const int* list, rt_stream st) {
    const size_t S1 = (size_t)(s->prob.horizon + 1), REC = (size_t)s->REC, HDR = (size_t)s->HDR, CS = (size_t)s->CS,
                 VS = (size_t)s->VS;
    const size_t R_T = VS + CS + (size_t)s->LT, nxp = (size_t)s->NW + CS + VS, NX = (size_t)s->prob.nx;     // t | p | x
    T* rec = (T*)s->rec; T* hdr = (T*)s->hdr; T* yr = (T*)s->yrows;
    const T* rec2 = (const T*)s->rec2; const T* hdr2 = (const T*)s->hdr2; const T* yr2 = (const T*)s->yrows2;
    const int per = (int)(S1 * (nxp + CS) + 2 * NX);
    return launch_1d(n * per, st, MPCB_LAMBDA(int idx) {
        const int e = idx / n, j = idx - e * n;
        const int b = list[j];
        const size_t td = (size_t)(b >> 5), ldn = (size_t)(b & 31), ts = (size_t)(j >> 5), ls = (size_t)(j & 31);
        size_t r = (size_t)e;
        if (r < S1 * nxp) {                      // t, p (= z) and x blocks of every record
            const size_t k = r / nxp, o = R_T + (r - k * nxp);
            rec[((td * S1 + k) * REC + o) * TILE + ldn] = rec2[((ts * S1 + k) * REC + o) * TILE + ls];
            return;
        }
        r -= S1 * nxp;
        if (r < S1 * CS) { yr[(td * S1 * CS + r) * TILE + ldn] = yr2[(ts * S1 * CS + r) * TILE + ls]; return; }
        r -= S1 * CS;                             // header: p (= z) and y of the dyn_0 rows
        hdr[(td * HDR + NX + r) * TILE + ldn] = hdr2[(ts * HDR + NX + r) * TILE + ls];
    });
}


// the staged stage models of the surviving QPs -> dense tiles of the scratch copy (see retile_impl)
template <typename T, typename L>
static int retile_model(mpcb_solver* s, int n, const int* list, rt_stream st) {
#ifndef MPCB_EMU
    const size_t per = (size_t)(s->prob.horizon + 1) * CtaModel<L>::COUNT;
    const T* mdl = (const T*)s->mdl; T* mdl2 = (T*)s->mdl2;
    if ((size_t)n * per > 0x7fffffffull) return fail(MPCB_E_ARG, "time-varying model too large to re-tile");
    return launch_1d((int)(n * per), st, MPCB_LAMBDA(int idx) {
        const int e = idx / n, j = idx - e * n;
        const int b = list[j];
        mdl2[(((size_t)(j >> 5)) * per + e) * TILE + (j & 31)] = mdl[(((size_t)(b >> 5)) * per + e) * TILE + (b & 31)];
    });
#else
    (void)s; (void)n; (void)list; (void)st;
    return 0;
#endif
}
static int ensure_scratch(mpcb_solver* s, int n_unc, size_t mdl_per_qp_bytes) {
    const size_t ld2 = ((size_t)n_unc + 31) / 32 * 32, S1 = (size_t)(s->prob.horizon + 1), e = s->esz;
    if (ld2 > s->ld2) {
        rt_free(s->rec2); rt_free(s->hdr2); rt_free(s->yrows2); rt_free(s->mdl2);
        s->rec2 = s->hdr2 = s->yrows2 = s->mdl2 = nullptr; s->ld2 = 0;
        // half the capacity covers the classic "re-tile when half is left"; the eager compaction of warm-started steps asks
        // for up to four fifths, a different count every step: grow once, to the full capacity (a cudaFree / cudaMalloc
        // pair inside a closed loop is a device synchronisation and milliseconds each time)
        const size_t half = ((size_t)s->ld / 2 + 31) / 32 * 32, full = ((size_t)s->ld + 31) / 32 * 32;
        const size_t want = ld2 <= half ? half : (ld2 <= full ? full : ld2);
        if (int r = rt_malloc(&s->rec2, S1 * s->REC * want * e)) return r;
        if (int r = rt_malloc(&s->hdr2, (size_t)s->HDR * want * e)) return r;
        if (int r = rt_malloc(&s->yrows2, S1 * s->CS * want * e)) return r;
        s->ld2 = want;
        s->ws_bytes += (S1 * s->REC + s->HDR + S1 * s->CS) * want * e;
    }
    if (mdl_per_qp_bytes && !s->mdl2) {
        if (int r = rt_malloc(&s->mdl2, mdl_per_qp_bytes * s->ld2)) return r;
        s->ws_bytes += mdl_per_qp_bytes * s->ld2;
    }
    return 0;
}
// The set of QPs a chunked host loop iterates on: the whole batch in the home workspace until the first compaction, then
// the survivors in dense tiles of the scratch workspace (map[j] = home slot of scratch slot j).
template <typename T, typename L>
struct LoopSet {
    int n;                        // QPs in the set
    int which = 0;                // the next launch lists the set's survivors in s->surv[which]
    const int* map = nullptr;     // null while the set is the home workspace
    // Compact the n_unc survivors listed by the last launch into the scratch workspace — records, headers and, when
    // mdl_per (bytes per QP) is not 0, the staged stage models — and point p at them.  Compaction always reads the home
    // workspace: a set that already sits in the scratch workspace is copied home first.
    int compact(mpcb_solver* s, KParams<T>& p, int n_unc, size_t mdl_per, rt_stream st) {
        if (int r = copy_home(s, st)) return r;
        if (int r = ensure_scratch(s, n_unc, mdl_per)) return r;
        if (int r = retile_impl<T>(s, n_unc, s->surv[which], st)) return r;
        if (mdl_per) if (int r = retile_model<T, L>(s, n_unc, s->surv[which], st)) return r;
        map = s->surv[which];
        which ^= 1;               // the next launches list their survivors in the other buffer
        n = n_unc;
        p.rec = (T*)s->rec2; p.hdr = (T*)s->hdr2; p.yrows = (T*)s->yrows2;
        if (mdl_per) p.mdl = (const T*)s->mdl2;
        return 0;
    }
    // x, z, y of a compacted set back to their home columns
    int copy_home(mpcb_solver* s, rt_stream st) const { return map ? untile_impl<T>(s, n, map, st) : 0; }
};

// The host loop of the CTA-per-tile kernel.  Small sets: ONE launch, termination tests included, nothing to read back.
// Large sets: one launch per check interval; after each the number of unsolved QPs is read back, and every time at
// most four fifths of the current set are left the survivors are compacted into dense tiles of the scratch workspace (their
// records, headers and staged stage models) — a tile streams 32 QPs' records until its slowest QP terminates, and the
// iteration counts of a batch spread widely (configs[3]: 150 .. 450).
template <typename T, typename L>
static int run_cta_loop(mpcb_solver* s, KParams<T> p, int max_iter, int check_every, bool chunked, rt_stream st) {
#ifndef MPCB_EMU
    if (!chunked) {
        p.it0 = 0; p.it_stop = max_iter; p.list_survivors = 0;
        return launch_cta<T, L>(p, s, st);
    }
    const int retile_floor = 1024;          // (fewer QPs than this leave most SMs idle either way: compaction buys nothing)
    const size_t mdl_per = p.tv ? (size_t)(p.N + 1) * CtaModel<L>::COUNT * sizeof(T) : 0;
    int it0 = 0;
    LoopSet<T, L> set{p.B};
    const bool trace = std::getenv("MPCB_TRACE") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    while (it0 < max_iter) {
        p.B = set.n; p.survivors = s->surv[set.which]; p.qp_map = set.map;
        p.it0 = it0; p.it_stop = it0 + check_every < max_iter ? it0 + check_every : max_iter; p.list_survivors = 1;
        const int rc = launch_cta<T, L>(p, s, st);
        if (rc != 0) return rc;
        it0 = p.it_stop;
        int n_unc = 0;
        if (int r = rt_d2h(&n_unc, s->n_surv, sizeof(int), st)) return -1;
        if (int r = rt_sync(st)) return -1;
        if (int r = rt_memset(s->n_surv, 0, sizeof(int), st)) return -1;
        if (trace) std::fprintf(stderr, "[mpcb] cta ..%d n=%d -> %d unsolved (scratch=%d)  t=%.3f ms\n", it0, set.n, n_unc, (int)(set.map != nullptr),
                                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
        if (n_unc == 0 || it0 >= max_iter) break;
        if (5 * n_unc <= 4 * set.n && set.n >= retile_floor)      // a fifth of the tiles to gain: worth the two copies
            if (set.compact(s, p, n_unc, mdl_per, st)) return -1;
    }
    if (set.copy_home(s, st)) return -1;
    return 0;
#else
    (void)s; (void)p; (void)max_iter; (void)check_every; (void)chunked; (void)st;
    return 1;
#endif
}

// The ADMM loop on the host side.  The device runs it in chunks of `check_termination` iterations (a chunk ends right
// after a termination test; unsolved rows stay in p-form, so chunking does not change a single bit).  A batch that shares
// one KKT matrix runs in admm_dense_kernel, one that the CTA-per-tile kernel serves in run_cta_loop; every other batch below
// retile_min_batch (and every batch with MPCB_NO_RETILE=1) runs the whole loop as ONE asynchronous launch of
// admm_tma_kernel.  A larger batch runs phase 1 on the home workspace, then reads the number of unsolved QPs back after
// each tested launch (a stream synchronisation) and compacts them — their workspace columns are copied into dense tiles
// of a scratch workspace — every time a fifth of the set has terminated, so that warps stop streaming the records of 32
// QPs for the sake of one straggler; the tail finishes in the CTA-per-tile kernel.  At the end the compacted QPs are
// copied back to their home columns.
template <typename T, typename L>
static int run_admm_impl(mpcb_solver* s, int max_iter, int check_every, int warm, rt_stream st) {
    const bool no_retile = g_opt_retile.load() == 0;
    const int retile_min = g_opt_retile_min.load();
    const int B = s->batch;
    if (s->cold_pending) { warm = 0; s->cold_pending = false; }      // first launch after prob.setup(): x = z = y = 0
    const bool chunked = !no_retile && check_every > 0 && check_every < max_iter && B >= retile_min;
    int* status = s->status;
    if (int r = launch_1d(B, st, MPCB_LAMBDA(int b) { status[b] = status[b] == -7 ? -7 : (int)kUnsolved; })) return r;
    if (int r = rt_memset(s->n_surv, 0, sizeof(int), st)) return r;
    KParams<T> p = make_params<T>(s);
    p.max_iter = max_iter; p.check_every = check_every; p.warm = warm;
    p.chunk_len = check_every;
    // Time-varying problems (one linearisation per stage: BASELINE configs[3]): the CTA-per-tile kernel runs the whole loop
    // in one launch — first iteration, termination tests, certificates, exit pass — with the stage models staged by TMA
    // A batch that shares ONE KKT matrix (one linearisation and identical scalings, or a batch of one): the whole loop as a
    // dense GEMM on the FP64 tensor cores in one launch, termination tests included — nothing to read back (admm_dense.cuh)
    // (also offered to time-varying batches of up to 16384 QPs with nx + nu <= 8: moved to another kernel, their results
    // would change in the last bits)
    const bool dense_window = B < retile_min || (p.tv && B <= 16384 && L::NW <= 8);
    if (dense_window && !no_retile && check_every > 1 && check_every < max_iter) {
        if (s->dense_state == 0 && dense_candidate<T, L>(s))
            if (int r = ensure_factor_form<T, L>(s, p, false, st)) return r;      // (reads Linv)
        if (int r = dense_prepare<T, L>(s, st)) return r;
        if (s->dense_state == 1) {
            p.it0 = 0; p.it_stop = max_iter; p.list_survivors = 0;
            const int rd = launch_dense<T, L>(p, s, st);
            if (rd <= 0) return rd < 0 ? (int)MPCB_E_CUDA : 0;
        }
    }
    if (p.tv && s->mdl && s->mdl_dirty) {
        if (int r = tile_model<T, L>(s, p, st)) return r;
    }
    s->mdl_dirty = false;
    const bool use_cta = cta_planned<T, L>(s, B, p.tv != 0, check_every) && cta_applicable<T, L>(s, p);
    if (int r = ensure_factor_form<T, L>(s, p, use_cta, st)) return r;
    if (use_cta) {
        const bool cta_chunked = !no_retile && check_every < max_iter && B >= retile_min;
        const int rc = run_cta_loop<T, L>(s, p, max_iter, check_every, cta_chunked, st);
        if (rc <= 0) return rc < 0 ? (int)MPCB_E_CUDA : 0;
    }
    if (!chunked) {
        p.it0 = 0; p.it_stop = max_iter; p.list_survivors = 0;
        return launch_admm<T, L>(p, s, st);
    }
    // Large batches: phase 1 on the home workspace up to the iteration count at which the previous solve of this
    // solver compacted (one launch; unknown on the first solve: explore check by check), then compaction (below).
    // (cold and warm-started solves of one solver converge very differently — the closed loop's step 0 against every later
    // step — so each keeps its own learnt point)
    const int rt_slot = warm ? 1 : 0;
    int it0 = 0;
    LoopSet<T, L> set{B};
    const bool trace = std::getenv("MPCB_TRACE") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto trace_ms = [&]() {            // (MPCB_TRACE only) drains the stream: a timestamp per launch, not a product path
        rt_sync(st);
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    };
    bool learnt_now = false;
    while (it0 < max_iter) {
        int stop = it0 + check_every;
        if (it0 == 0 && s->retile_at[rt_slot] > 0) stop = s->retile_at[rt_slot];
        p.B = set.n; p.survivors = s->surv[set.which]; p.qp_map = set.map;
        p.it0 = it0; p.it_stop = stop < max_iter ? stop : max_iter; p.list_survivors = 1;
        if (int r = launch_admm<T, L>(p, s, st)) return r;
        if (trace) std::fprintf(stderr, "[mpcb] admm %d..%d n=%d scratch=%d  t=%.3f ms\n", p.it0 + 1, p.it_stop, set.n, (int)(set.map != nullptr), trace_ms());
        it0 = p.it_stop;
        int n_unc = 0;
        if (int r = rt_d2h(&n_unc, s->n_surv, sizeof(int), st)) return r;
        if (int r = rt_sync(st)) return r;
        if (int r = rt_memset(s->n_surv, 0, sizeof(int), st)) return r;
        if (n_unc == 0 || it0 >= max_iter) {
            // Everything terminated where nothing had been compacted: the next solve of this kind runs up to here in one launch
            // — and, once in a while, stops one test earlier to see whether a compaction there pays (a warm-started closed
            // loop drifts from "all at 50" to "half at 25, half at 50" as the scenarios settle).
            if (!set.map && !learnt_now && n_unc == 0) {
                int& at = s->retile_at[rt_slot];
                int& backoff = s->retile_backoff[rt_slot];
                if (at == it0 && it0 > check_every && backoff == 0) at = it0 - check_every;
                else if (at == 0) at = it0;
                if (backoff > 0) --backoff;
            }
            break;
        }
        // Compaction.  Copying a QP's records into a dense tile (and its iterates back later) costs about the traffic of 1.5
        // iterations of that QP; a tile streams the records of all 32 slots as long as one of them is unsolved.  So a large
        // batch is compacted every time a fifth of the set has terminated (the warm-started closed loop loses 30-50 % of its
        // QPs at the first test, a cold batch 96 % at the third), and as soon as the unsolved set fits one wave of CTAs it
        // finishes in the CTA-per-tile kernel (below).
        // (Measured against it: compacting the cold headline batch already at iteration 50, where 13 % have terminated —
        //  27.5 instead of 25.0 ms per step: a launch boundary costs the warp-per-tile kernel a partly filled last wave,
        //  ~2 ms at this size, more than the 1 ms of traffic the compaction saves.)
#ifndef MPCB_EMU
        const bool tail_cta = !p.tv && cta_planned<T, L>(s, n_unc, false, check_every) && cta_applicable<T, L>(s, p);
#else
        const bool tail_cta = false;
#endif
        if (tail_cta || (5 * n_unc <= 4 * set.n && set.n >= (retile_min < 1024 ? retile_min : 1024))) {
            if (!learnt_now) { s->retile_at[rt_slot] = it0; learnt_now = true; }
            if (int r = set.compact(s, p, n_unc, 0, st)) return r;
#ifndef MPCB_EMU
            // The stragglers of a large batch are a small batch: when they fit one wave of CTAs they finish in the CTA-per-tile
            // kernel, all remaining iterations, tests and exits in ONE launch (41 us per iteration, nothing read back per
            // test).  It multiplies with the block inverse: the factor blocks of the compacted copies are converted in place.
            if (tail_cta) {
                if (int r = launch_1d(set.n * (p.N + 1), st, MinvFromLinvFn<T, L>{p.rec, p.N + 1, set.n})) return r;
                KParams<T> pc = p;
                pc.minv = 1; pc.B = set.n; pc.qp_map = set.map; pc.survivors = s->surv[set.which];
                pc.it0 = it0; pc.it_stop = max_iter; pc.list_survivors = 0;
                const int rc = launch_cta<T, L>(pc, s, st);
                if (rc < 0) return (int)MPCB_E_CUDA;
                if (trace) std::fprintf(stderr, "[mpcb] cta %d..%d n=%d scratch=1 (stragglers)  t=%.3f ms\n", it0 + 1, max_iter, set.n, trace_ms());
                if (rc == 0) break;
            }
#endif
        } else if (!set.map && !learnt_now && it0 == s->retile_at[rt_slot]) {
            s->retile_at[rt_slot] = 0;                 // the learnt point no longer fits this workload: explore again next time
            s->retile_backoff[rt_slot] = 16;           // (and leave earlier probes alone for a while)
        }
    }
    return set.copy_home(s, st);
}

// =============================================================================================
// the ops table of this (shape, dtype)
// =============================================================================================
template <typename T, typename L>
static int setup_impl(mpcb_solver* s, rt_stream st) {
    KParams<T> p = make_params<T>(s);
    if (int r = rt_memset(s->status, 0, s->ld * sizeof(int), st)) return r;
#ifndef MPCB_EMU
    if (p.N + 1 <= 32 && g_opt_warp_setup.load() != 0) {      // Ruiz with a warp per QP, scalings in registers (setup_warp.cuh)
        scale_warp_kernel<T, L><<<(p.B + SCALE_WARPS - 1) / SCALE_WARPS, SCALE_WARPS * 32, 0, st>>>(p);
        ++g_launches;
        if (int r = rt_launch_check("scale_warp")) return r;
    } else
#endif
    if (int r = launch_qp<ScaleOp, T, L>(p, st)) return r;
    // solves that will go to admm_cta_kernel: factor blocks in its form from the start (ensure_factor_form)
#ifndef MPCB_EMU
    s->rec_minv = cta_planned<T, L>(s, p.B, p.tv != 0, s->set.check_termination) && cta_fits<T, L>(s, p.tv != 0) &&
                  !dense_candidate<T, L>(s);           // (the dense path reads Linv)
#else
    s->rec_minv = false;
#endif
    p.minv = s->rec_minv ? 1 : 0;
    if (int r = launch_qp<FactorOp, T, L>(p, st)) return r;
    s->mdl_dirty = false;
    if (p.tv && g_opt_cta.load() != 0) return tile_model<T, L>(s, p, st);      // staged by admm_cta_kernel next to the records
    return 0;
}
template <typename T, typename L>
static int refactor_impl(mpcb_solver* s, const mpcb_problem* np, void* new_box, rt_stream st) {
    RefactorFn<T, L> fn;
    fn.po = make_params<T>(s);
    const mpcb_problem keep = s->prob;
    void* keep_box = s->xbox;
    s->prob = *np; s->xbox = new_box;
    fn.pn = make_params<T>(s);
    s->prob = keep; s->xbox = keep_box;
    // either set of bounds may hold an infinity: both evaluations take the general row_rho
    return launch_1d(fn.pn.B, st, fn);
}
template <typename T, typename L>
static int cold_impl(mpcb_solver* s, rt_stream st) {
    KParams<T> p = make_params<T>(s);
    return launch_qp<ColdOp, T, L>(p, st);
}
template <typename T, typename L>
static int build_impl(mpcb_solver* s, const BuildOut* o, rt_stream st) {
    KParams<T> p = make_params<T>(s);
    return launch_1d(p.B, st, BuildFn<T, L>{p, *o});
}
template <typename T, typename L>
static int scaling_impl(mpcb_solver* s, const ScalingOut* o, rt_stream st) {
    KParams<T> p = make_params<T>(s);
    return launch_1d(p.B, st, ScalingFn<T, L>{p, *o});
}
template <typename T, typename L>
static ShapeOps make_shape_ops() {
    ShapeOps o;
    o.nx = L::NX; o.nu = L::NU; o.slack = L::SLACK ? 1 : 0;
    o.dtype = std::is_same<T, float>::value ? MPCB_F32 : MPCB_F64;
    o.setup = &setup_impl<T, L>; o.refactor = &refactor_impl<T, L>; o.run_admm = &run_admm_impl<T, L>;
    o.cold_start = &cold_impl<T, L>; o.build_qp = &build_impl<T, L>; o.get_scaling = &scaling_impl<T, L>;
    return o;
}
