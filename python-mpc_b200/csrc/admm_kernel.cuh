// The ADMM loop drivers.
//
//   admm_one          one lane runs its QP straight out of global memory (every record access has a compile-time
//                     offset).  Used for shapes whose stage record is too large to double-buffer in shared memory,
//                     with MPCB_NO_TMA=1, and by tests/emu.
//   admm_tma_kernel   (GPU only) a warp runs a tile of 32 QPs with the stage records staged through shared memory:
//                     while stage k is being computed, ONE elected lane has already issued a cp.async.bulk (TMA) for
//                     the whole record of the next stage, completion tracked by an mbarrier per buffer; all writes go
//                     straight to global memory.  Persistent CTAs; the warps of a CTA take (chunk, tile) work items
//                     together and meet at a CTA barrier once per iteration (instruction-cache sharing).
//   Both drive the same stage functions (qp_thread.cuh): forward / backward sweep, with first-iteration and tested-iteration
//   variants as template instantiations.  The backward sweep of a tested iteration (kBwdTest) also evaluates the
//   termination test — the residuals of (x, y) and the infeasibility certificates of (dx, dy) — from what it holds anyway:
//   the new state in registers, the old one in the record it reads.  A tested iteration therefore costs no memory traffic
//   beyond its two sweeps, and needs no copy of the old state.
#pragma once
#include "qp_thread.cuh"
#include <type_traits>

namespace mpcb {

template <typename T, typename L>
MPCB_HD void admm_setup_const(const KParams<T>& p, int b, const Ws<T, L>& ws, AdmmConst<T, L>& q) {
    q.c = MPCB_AT(ws.hdr, L::H_C);
    q.cinv = (T)1 / q.c;
    q.rho = clamp_rho(p.rho);
    q.rho_eq = (T)kRhoEqOverRhoIneq * q.rho;
    q.sigma = p.sigma;
    q.alpha = p.alpha;
    q.inf_bounds = p.inf_bounds != 0;
    q.xr = p.Xr + b; q.xr_stride = p.ld;      // (unused when the reference is stage-wise)
}

template <typename T, typename L>
MPCB_HD void admm_cold_start(const KParams<T>& p, const Ws<T, L>& ws) {
    for (int k = 0; k <= p.N; ++k) {
        T* R = ws.R(k);
        T* Y = ws.Y(k);
        for (int e = 0; e < L::VS; ++e) MPCB_AT(R, L::R_X + e) = 0;
        for (int e = 0; e < L::CS; ++e) { MPCB_AT(R, L::R_P + e) = 0; MPCB_AT(Y, e) = 0; }
    }
    for (int i = 0; i < L::NX; ++i) { MPCB_AT(ws.hdr, L::H_P0 + i) = 0; MPCB_AT(ws.hdr, L::H_Y0 + i) = 0; }
}

template <typename T>
MPCB_HD bool admm_is_tested(const KParams<T>& p, int it) {
    return (p.check_every > 0 && (it % p.check_every == 0)) || it == p.max_iter;
}

template <typename T, typename L, bool FIRST>
MPCB_HD void admm_fwd_begin(const KParams<T>& p, const AdmmConst<T, L>& q, int b, const T* H, FwdCarry<T, L>& cy) {
#pragma unroll
    for (int i = 0; i < L::NX; ++i) {
        cy.Ed_cur[i] = MPCB_AT(H, L::H_E0 + i);
        const T beq = -cy.Ed_cur[i] * p.x_init[(size_t)i * p.ld + b];
        const Row<T> rw = row_state(FIRST, MPCB_AT(H, L::H_P0 + i), FIRST ? MPCB_AT(H, L::H_Y0 + i) : (T)0, beq, beq,
                                    q.rinv_eq());
        cy.vd_cur[i] = q.rho_eq * (rw.z - rw.yr);
        cy.cprev[i] = 0;
    }
}

// start of a termination sweep of the CTA and dense kernels: rows dyn_0 (header)
template <typename T, typename L>
MPCB_HD void admm_test_begin(const KParams<T>& p, const AdmmConst<T, L>& q, int b, const T* H, TestCarry<T, L>& cy,
                             TestAcc<T>& t, bool cert, bool first, const T* O0) {
    test_reset(t);
#pragma unroll
    for (int i = 0; i < L::NX; ++i) {
        cy.Ed_cur[i] = MPCB_AT(H, L::H_E0 + i);
        const T beq = -cy.Ed_cur[i] * p.x_init[(size_t)i * p.ld + b];
        T w = q.rho_eq * (MPCB_AT(H, L::H_P0 + i) - beq);
        if (cert) w -= q.rho_eq * old_yr(first, MPCB_AT(O0, i), first ? MPCB_AT(H, L::H_Y0 + i) : (T)0, beq, beq, q.rho_eq);
        cy.wd_cur[i] = w;
        t.nEw = tmax(t.nEw, tabs(cy.Ed_cur[i] * w));
        t.lhs += beq * w;
    }
}
template <typename T>
MPCB_HD void test_to_resid(const TestAcc<T>& t, Resid<T>& rs) {
    rs.pri = t.pri; rs.dua = t.dua; rs.nz = t.nz; rs.nAx = t.nAx; rs.nq = t.nq; rs.nAty = t.nAty; rs.nPx = t.nPx;
}
template <typename T>
MPCB_HD void test_to_cert(const TestAcc<T>& t, Cert<T>& c) {
    c.ndy = t.nEw; c.lhs = t.lhs; c.nAtdy = t.nAty; c.ndx = t.nDv; c.qdx = t.qv; c.nPdx = t.nPx; c.aup = t.aup; c.alo = t.alo;
}

// osqp.c / auxil.c: the decision taken after a residual evaluation, in two steps.
//   admm_residual_test: true when the exact residual test passes (status solved — OSQP evaluates no certificate
//   then); otherwise the certificates are consulted and admm_decide concludes.
template <typename T, typename L>
MPCB_HD bool admm_residual_test(const KParams<T>& p, const AdmmConst<T, L>& q, Resid<T>& rs) {
    rs.dua *= q.cinv;
    return rs.pri < p.eps_abs + p.eps_rel * tmax(rs.nz, rs.nAx) &&
           rs.dua < p.eps_abs + p.eps_rel * q.cinv * tmax(rs.nq, tmax(rs.nAty, rs.nPx));
}
// auxil.c: check_termination with every tolerance multiplied by `mult` (1: exact, 10: approximate).  Returns 0 when
// nothing can be concluded, else the status (the *_inaccurate variants for the approximate test).
template <typename T, typename L>
MPCB_HD int admm_test(const KParams<T>& p, const AdmmConst<T, L>& q, const Resid<T>& rs, const Cert<T>& ct, T mult) {
    const bool approx = mult != (T)1;
    const T ea = mult * p.eps_abs, er = mult * p.eps_rel;
    const bool prim_ok = rs.pri < ea + er * tmax(rs.nz, rs.nAx);
    if (!prim_ok && cert_primal_infeasible(ct, mult * p.eps_pinf))
        return approx ? kPrimalInfeasibleInaccurate : kPrimalInfeasible;
    const bool dual_ok = rs.dua < ea + er * q.cinv * tmax(rs.nq, tmax(rs.nAty, rs.nPx));
    if (!dual_ok && cert_dual_infeasible(ct, q.c, mult * p.eps_dinf))
        return approx ? kDualInfeasibleInaccurate : kDualInfeasible;
    if (prim_ok && dual_ok) return approx ? kSolvedInaccurate : kSolved;
    return 0;
}
// after the certificates of a QP that failed the residual test (rs.dua already unscaled by admm_residual_test).
// Returns true when the loop ends.
template <typename T, typename L>
MPCB_HD bool admm_decide(const KParams<T>& p, const AdmmConst<T, L>& q, const Resid<T>& rs, const Cert<T>& ct, bool at_cap,
                         int& status) {
    // exact test: at a check iteration, or at the cap if it was not done this iteration (end of osqp_solve)
    if (const int st = admm_test<T, L>(p, q, rs, ct, (T)1)) { status = st; return true; }
    if (at_cap) {
        // the approximate test (tolerances x10) before declaring max-iter
        const int st = admm_test<T, L>(p, q, rs, ct, (T)10);
        status = st ? st : (int)kMaxIterReached;
        return true;
    }
    return false;
}

template <typename T, typename L>
MPCB_HD void admm_exit_header(const KParams<T>& p, const AdmmConst<T, L>& q, int b, T* H) {
#pragma unroll
    for (int i = 0; i < L::NX; ++i) {
        const T beq = -MPCB_AT(H, L::H_E0 + i) * p.x_init[(size_t)i * p.ld + b];
        const T pp = MPCB_AT(H, L::H_P0 + i);
        MPCB_AT(H, L::H_P0 + i) = beq;
        MPCB_AT(H, L::H_Y0 + i) = q.rho_eq * (pp - beq);
    }
}

// what a lane does when its chunk ends: converged / capped lanes leave explicit (z, y) behind, unsolved lanes of a
// non-final chunk keep their rows in p-form and put themselves on the survivor list
template <typename T, typename L>
MPCB_HD void admm_finish(const KParams<T>& p, const AdmmConst<T, L>& q, Model<T, L>& m, const Ws<T, L>& ws, int bi,
                         int status, int it_done, const Resid<T>& rs) {
    if (status == kUnsolved) {
        if (!p.list_survivors) return;
#ifdef __CUDA_ARCH__
        const int slot = atomicAdd(p.n_survivors, 1);
#else
        const int slot = (*p.n_survivors)++;
#endif
        p.survivors[slot] = bi;
        return;
    }
    admm_exit_header<T, L>(p, q, bi, ws.hdr);
    for (int k = 0; k <= p.N; ++k) admm_exit_stage<T, L>(p, q, bi, k, ws.R(k), ws.Y(k));
    (void)m;
    p.iter[bi] = it_done;
    p.status[bi] = status;
    p.pri_res[bi] = rs.pri;
    p.dua_res[bi] = rs.dua;
}

// Forward and backward sweep of one iteration straight out of global memory.  FIRST (iteration 1 of a solve: rows
// enter as explicit (z, y)), RHS (the forward sweep starts from r^) and MODE (kBwdTest: the iteration is tested) are
// template parameters: the steady-state instantiation carries none of that code or state.
template <typename T, typename L, bool FIRST, bool RHS = false>
MPCB_HD void admm_one_fwd(const KParams<T>& p, const AdmmConst<T, L>& q, Model<T, L>& m, int bi, const Ws<T, L>& ws) {
    FwdCarry<T, L> cy;
    admm_fwd_begin<T, L, FIRST>(p, q, bi, ws.hdr, cy);
    for (int k = 0; k <= p.N; ++k) {
        if (p.tv && k < p.N) load_model<T, L>(p, bi, k, m);
        admm_fwd_stage<T, L, FIRST, RHS>(p, q, m, bi, k, ws.R(k), ws.Y(k), ws.R(k), cy);
    }
}
template <typename T, typename L, bool FIRST, int MODE>
MPCB_HD void admm_one_bwd(const KParams<T>& p, const AdmmConst<T, L>& q, Model<T, L>& m, int bi, const Ws<T, L>& ws,
                          BwdTest<T, L>& ts) {
    BwdCarry<T, L> cy;
#pragma unroll
    for (int i = 0; i < L::NX; ++i) { cy.xt_next[i] = 0; cy.Dx_next[i] = 1; }
    if (MODE == kBwdTest) test_reset(ts);
    for (int k = p.N; k >= 0; --k) {
        if (p.tv && k < p.N) load_model<T, L>(p, bi, k, m);
        admm_bwd_stage<T, L, FIRST, MODE>(p, q, m, bi, k, ws.R(k), ws.Y(k), ws.R(k), cy, ts);
    }
    admm_bwd_header<T, L, FIRST, MODE>(p, q, bi, ws.hdr, cy, ts);
}
// The termination test of a tested iteration, after its backward sweep (kBwdTest) accumulated ts.  Returns true when the
// QP's loop ends (status set).  The certificates are consulted only when the residual test fails, as in OSQP.
template <typename T, typename L>
MPCB_HD bool admm_conclude(const KParams<T>& p, const AdmmConst<T, L>& q, const BwdTest<T, L>& ts, int it, Resid<T>& rs,
                           int& status) {
    test_to_resid(ts.r, rs);
    if (admm_residual_test<T, L>(p, q, rs)) { status = kSolved; return true; }
    if (!p.certs && it != p.max_iter) return false;
    Cert<T> ct;
    test_to_cert(ts.c, ct);
    return admm_decide<T, L>(p, q, rs, ct, it == p.max_iter, status);
}
// The CTA and dense kernels evaluate the certificates of a tested iteration `it` in a sweep of their own, from a copy of
// the old state: made by the backward sweep of iteration it-1 when that was a steady-state iteration, else (it <= 2: the
// state a solve starts from, or the one its first iteration left) before the iteration.
template <typename T>
MPCB_HD bool admm_saves(const KParams<T>& p, int it) { return it >= 2 && admm_is_tested(p, it + 1); }
template <typename T>
MPCB_HD bool admm_needs_copy(const KParams<T>& p, int it) { return it <= 2 && admm_is_tested(p, it); }

template <typename T, typename L>
MPCB_HD void admm_one(const KParams<T>& p, int b) {
    const int bi = p.qp_map ? p.qp_map[b] : b;          // QP index for inputs and outputs; b is the workspace slot
    if (p.status[bi] != kUnsolved) return;               // solved in an earlier chunk, or not factorable (-7)
    Ws<T, L> ws(p, b);
    AdmmConst<T, L> q;
    admm_setup_const<T, L>(p, bi, ws, q);
    Model<T, L> m;
    if (!p.tv) load_model<T, L>(p, bi, 0, m);
    if (p.it0 == 0 && !p.warm) admm_cold_start<T, L>(p, ws);
    int status = kUnsolved, it = 0;
    Resid<T> rs;
    rs.pri = rs.dua = 0;
    BwdTest<T, L> ts;
    for (it = p.it0 + 1; it <= p.it_stop; ++it) {
        const bool tested = admm_is_tested(p, it);
        if (it == 1) {
            admm_one_fwd<T, L, true>(p, q, m, bi, ws);
            if (tested) admm_one_bwd<T, L, true, kBwdTest>(p, q, m, bi, ws, ts);
            else admm_one_bwd<T, L, true, kBwdPlain>(p, q, m, bi, ws, ts);
        } else {
            if (p.fwd_rhs) admm_one_fwd<T, L, false, true>(p, q, m, bi, ws);
            else admm_one_fwd<T, L, false>(p, q, m, bi, ws);
            if (tested) admm_one_bwd<T, L, false, kBwdTest>(p, q, m, bi, ws, ts);
            else admm_one_bwd<T, L, false, kBwdPlain>(p, q, m, bi, ws, ts);
        }
        if (tested && admm_conclude<T, L>(p, q, ts, it, rs, status)) break;
    }
    admm_finish<T, L>(p, q, m, ws, bi, status, it > p.it_stop ? p.it_stop : it, rs);
}

#if defined(__CUDACC__) && !defined(MPCB_EMU)
// ==============================================================================================
// Warp-per-tile ADMM with the stage records staged through shared memory by TMA bulk copies.
// ==============================================================================================
__device__ __forceinline__ unsigned smem_u32(const void* ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// one TMA bulk copy global -> shared (1-D, no tensor map needed for a contiguous record)
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// order this thread's generic-proxy writes before later async-proxy (TMA) reads of the same memory
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }

// What a TMA load of a stage record brings into a record buffer (one mbarrier transaction, one or two bulk copies):
//   kLoadAll  the whole record: the backward sweep, and stage 0 / stage N of a forward sweep (the backward turn-around)
//   kLoadFwd  all but t: a forward sweep that forms the whole right-hand side
//   kLoadRhs  the runs FA and FB: a forward sweep that starts from r^ (mpc_common.h)
enum { kLoadAll, kLoadFwd, kLoadRhs };
template <typename T, typename L, int WHAT>
__device__ __forceinline__ void tma_load_stage(T* dst, const T* src, unsigned long long* bar) {
    constexpr unsigned E = TILE * sizeof(T);
    if (WHAT == kLoadRhs) {
        mbar_expect_tx(bar, (L::FA_N + L::FB_N) * E);
        tma_load_1d(dst + L::FA * TILE, src + L::FA * TILE, L::FA_N * E, bar);
        tma_load_1d(dst + L::FB * TILE, src + L::FB * TILE, L::FB_N * E, bar);
    } else if (WHAT == kLoadFwd) {
        mbar_expect_tx(bar, (L::REC - L::NW) * E);
        tma_load_1d(dst, src, L::R_T * E, bar);
        tma_load_1d(dst + L::R_P * TILE, src + L::R_P * TILE, (L::REC - L::R_P) * E, bar);
    } else {
        mbar_expect_tx(bar, L::REC * E);
        tma_load_1d(dst, src, L::REC * E, bar);
    }
}

// Forward and backward sweep of one iteration of a tile: record k is resident in one of the warp's two buffers while
// the elected lane has the TMA bulk load of the next record in flight into the other.  FIRST = iteration 1 of a solve
// (rows enter as explicit (z, y)), RHS = the forward sweep starts from r^ and loads only the runs FA and FB of the
// records in between, MODE = kBwdTest: the iteration is tested (the backward sweep accumulates the test into ts); the
// steady-state instantiation carries none of that code or state.  Record 0 of a forward sweep is resident whole (the
// backward turn-around patches it, or a kLoadAll), so is record N (loaded whole for the backward turn-around).
template <typename T, typename L, bool FIRST, bool RHS>
__device__ __forceinline__ void admm_tma_fwd(const KParams<T>& p, const AdmmConst<T, L>& q, Model<T, L>& m,
                                             const Ws<T, L>& ws, int bb, int lane, bool active, T* buf0,
                                             unsigned long long* bar, unsigned& ph, int& cur, const T* rec_tile) {
    const int N = p.N;
#define MPCB_BUF(c) (buf0 + (c) * (L::REC * TILE))
    // ---------------- forward sweep: record k is resident in MPCB_BUF(cur); prefetch k+1
    {
        FwdCarry<T, L> cy;
        admm_fwd_begin<T, L, FIRST>(p, q, bb, ws.hdr, cy);
        for (int k = 0; k <= N; ++k) {
            if (k < N && lane == 0) {
                const T* src = rec_tile + (size_t)(k + 1) * L::REC * TILE;
                if (k + 1 == N) tma_load_stage<T, L, kLoadAll>(MPCB_BUF(cur ^ 1), src, &bar[cur ^ 1]);
                else tma_load_stage<T, L, RHS ? kLoadRhs : kLoadFwd>(MPCB_BUF(cur ^ 1), src, &bar[cur ^ 1]);
            }
            if (k > 0) { mbar_wait(&bar[cur], (ph >> cur) & 1u); ph ^= 1u << cur; }
            if (active) {
                if (p.tv && k < N) load_model<T, L>(p, bb, k, m);
                admm_fwd_stage<T, L, FIRST, RHS>(p, q, m, bb, k, MPCB_BUF(cur) + lane, ws.Y(k), ws.R(k), cy);
                if (k == N) {                     // turn-around: backward stage N reuses this buffer, give it t_N
#pragma unroll
                    for (int a = 0; a < L::NW; ++a)
                        MPCB_AT(MPCB_BUF(cur) + lane, L::R_T + a) = MPCB_AT(ws.R(k), L::R_T + a);
                }
            }
            if (k == N) fence_proxy_async();      // t_0..t_N (generic stores) before the backward sweep's TMA reads
            __syncwarp();
            if (k < N) cur ^= 1;
        }
    }
#undef MPCB_BUF
}
template <typename T, typename L, bool FIRST, int MODE>
__device__ __forceinline__ void admm_tma_bwd(const KParams<T>& p, const AdmmConst<T, L>& q, Model<T, L>& m,
                                             const Ws<T, L>& ws, int bb, int lane, bool active, T* buf0,
                                             unsigned long long* bar, unsigned& ph, int& cur, const T* rec_tile,
                                             BwdTest<T, L>& ts) {
    const int N = p.N;
#define MPCB_BUF(c) (buf0 + (c) * (L::REC * TILE))
    // ---------------- backward sweep: record N is resident in MPCB_BUF(cur); prefetch k-1 (with t)
    {
        BwdCarry<T, L> cy;
#pragma unroll
        for (int i = 0; i < L::NX; ++i) { cy.xt_next[i] = 0; cy.Dx_next[i] = 1; }
        if (MODE == kBwdTest) test_reset(ts);
        for (int k = N; k >= 0; --k) {
            if (k > 0 && lane == 0)
                tma_load_stage<T, L, kLoadAll>(MPCB_BUF(cur ^ 1), rec_tile + (size_t)(k - 1) * L::REC * TILE, &bar[cur ^ 1]);
            if (k < N) { mbar_wait(&bar[cur], (ph >> cur) & 1u); ph ^= 1u << cur; }
            if (active) {
                if (p.tv && k < N) load_model<T, L>(p, bb, k, m);
                admm_bwd_stage<T, L, FIRST, MODE>(p, q, m, bb, k, MPCB_BUF(cur) + lane, ws.Y(k), ws.R(k), cy, ts);
                if (k == 0) {                     // turn-around: the next forward stage 0 reuses this buffer: new r^, p, x
#pragma unroll
                    for (int e = 0; e < L::NW + L::CS + L::VS; ++e)
                        MPCB_AT(MPCB_BUF(cur) + lane, L::R_T + e) = MPCB_AT(ws.R(0), L::R_T + e);
                }
            }
            if (k == 0) fence_proxy_async();      // new r^, x, p (generic stores) before the next sweep's TMA reads
            __syncwarp();
            if (k > 0) cur ^= 1;
        }
        if (active) admm_bwd_header<T, L, FIRST, MODE>(p, q, bb, ws.hdr, cy, ts);
    }
#undef MPCB_BUF
}

template <typename T, typename L>
__global__ void __launch_bounds__(256, 1) admm_tma_kernel(const __grid_constant__ KParams<T> p, int* tile_counter) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr unsigned REC_BYTES = L::REC * TILE * sizeof(T);
    const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ntiles = (p.B + TILE - 1) / TILE;
    T* const buf0 = reinterpret_cast<T*>(smem_raw + (size_t)warp * 2 * REC_BYTES);     // two record buffers of this warp
#define MPCB_BUF(c) (buf0 + (c) * (L::REC * TILE))
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem_raw + (size_t)warps * 2 * REC_BYTES) + warp * 2;
    if (lane == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_proxy_async();
    __syncwarp();
    unsigned ph = 0u;                                  // bit c: phase parity of the mbarrier of buffer c

    // The launch covers iterations it0+1 .. it_stop of every tile.  It is handed out as (chunk, tile) work items of
    // chunk_len iterations, chunk-major, through one atomic counter: with ~2 tiles per warp a tile-granular split
    // leaves the last wave of the persistent grid one third full, a chunk-granular one does not.  A tile's state
    // lives in global memory between its chunks (rows in p-form), so any warp can continue any tile; the only
    // dependency — chunk c of a tile after its chunk c-1 — is tracked in tile_prog[] (release/acquire).
    //
    // The warps of a CTA take their items TOGETHER (one round = `warps` consecutive items) and meet at a CTA barrier
    // once per iteration.  The sweeps are long straight-line code, and the tested backward sweep is a variant that a warp
    // walks once per check_termination iterations: with the warps in step each fetched instruction line serves all of
    // them, out of step the rarely run code is an instruction-cache miss from end to end (measured, round 1:
    // `no_instruction` was 70 % of the then separate termination sweep's stall samples and a third of the sweeps').
    // Every barrier below is reached by
    // every thread of the CTA the same number of times: base, total_items and chunk_len are CTA-uniform, and a warp
    // without work (no item, nothing left in its tile, all its QPs done) keeps walking the round's barriers.
    const int span = p.it_stop - p.it0;
    const int chunk_len = p.chunk_len > 0 && p.chunk_len < span ? p.chunk_len : span;
    const int nchunks = (span + chunk_len - 1) / chunk_len;
    const int total_items = nchunks * ntiles;
    int* const s_base = reinterpret_cast<int*>(smem_raw + (size_t)warps * (2 * REC_BYTES + 16 + (p.xr_smem ? L::NX * TILE * sizeof(T) : 0)));
    for (int round = 0;; ++round) {
        if (threadIdx.x == 0) s_base[round & 1] = atomicAdd(tile_counter, warps);
        __syncthreads();
        const int base = s_base[round & 1];
        if (base >= total_items) break;                  // CTA-uniform
        const int item = base + warp;
        const bool has_item = item < total_items;
        const int chunk = has_item ? item / ntiles : 0, tile = has_item ? item - chunk * ntiles : 0;
        const int it_begin = p.it0 + chunk * chunk_len;
        const int it_end = it_begin + chunk_len < p.it_stop ? it_begin + chunk_len : p.it_stop;
        const bool last_chunk = (chunk == nchunks - 1);
        if (has_item && chunk > 0) {
            if (lane == 0) {
                int done;
                const long long t0 = clock64();
                do {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(done) : "l"(p.tile_prog + tile) : "memory");
                    if (done < chunk && clock64() - t0 > 20000000000LL) __trap();     // ~10 s: a lost dependency must not hang the GPU
                } while (done < chunk);
            }
            __syncwarp();
            fence_proxy_async();
        }
        // lanes of a ragged last tile (b >= B) own padding columns: they load like everyone, never write
        const int b = tile * TILE + lane;                 // workspace slot
        const int bb = has_item && b < p.B ? (p.qp_map ? p.qp_map[b] : b) : 0;      // QP index for inputs and outputs
        const bool valid = has_item && b < p.B && p.status[bb] == kUnsolved;      // not solved in an earlier chunk, factorable
        bool alive = __any_sync(0xffffffffu, valid);      // this warp has sweeps to run in this round
        if (has_item && !alive && !last_chunk && lane == 0)       // nothing left to do in this tile: still publish the chunk
            asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p.tile_prog + tile), "r"(chunk + 1) : "memory");
        Ws<T, L> ws(p, b);
        const T* rec_tile = ws.rec - lane;               // base of the warp's tile (what TMA copies from)
        AdmmConst<T, L> q;
        Model<T, L> m;
        bool active = valid;
        int status = kUnsolved, it_done = 0;
        Resid<T> rs;
        rs.pri = rs.dua = 0;
        int cur = 0;
        if (alive) {
            admm_setup_const<T, L>(p, bb, ws, q);
            if (p.xr_smem) {                              // the QP's reference: loop-invariant, parked in shared memory
                T* xs = reinterpret_cast<T*>(smem_raw + (size_t)warps * (2 * REC_BYTES + 16)) + (size_t)warp * L::NX * TILE + lane;
#pragma unroll
                for (int i = 0; i < L::NX; ++i) xs[i * TILE] = p.Xr[(size_t)i * p.ld + bb];
                q.xr = xs; q.xr_stride = TILE;
            }
            if (!p.tv) load_model<T, L>(p, bb, 0, m);
            if (valid && it_begin == 0 && !p.warm) admm_cold_start<T, L>(p, ws);
            fence_proxy_async();
            __syncwarp();
            // record 0 for the first forward sweep
            if (lane == 0) tma_load_stage<T, L, kLoadAll>(MPCB_BUF(cur), rec_tile, &bar[cur]);
            mbar_wait(&bar[cur], (ph >> cur) & 1u); ph ^= 1u << cur;
        }

        BwdTest<T, L> ts;
        for (int r = 0; r < chunk_len; ++r) {
            const int it = it_begin + 1 + r;
            const bool run = alive && it <= it_end;
            if (!__syncthreads_or(run)) break;           // CTA-uniform: nobody has an iteration left in this round
            if (run) {
                // ---------------- forward and backward sweep (the steady-state instantiation has no first-iteration code).
                // A tested iteration's backward sweep evaluates the termination test; record 0 stays resident, patched by
                // the backward turn-around, for the next forward sweep.
                const bool tested = admm_is_tested(p, it);
                if (it == 1) {
                    admm_tma_fwd<T, L, true, false>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile);
                    if (tested) admm_tma_bwd<T, L, true, kBwdTest>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile, ts);
                    else admm_tma_bwd<T, L, true, kBwdPlain>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile, ts);
                } else {
                    if (p.fwd_rhs) admm_tma_fwd<T, L, false, true>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile);
                    else admm_tma_fwd<T, L, false, false>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile);
                    if (tested) admm_tma_bwd<T, L, false, kBwdTest>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile, ts);
                    else admm_tma_bwd<T, L, false, kBwdPlain>(p, q, m, ws, bb, lane, active, buf0, bar, ph, cur, rec_tile, ts);
                }
                if (tested) {
                    if (active && admm_conclude<T, L>(p, q, ts, it, rs, status)) { active = false; it_done = it; }
                    if (!__any_sync(0xffffffffu, active)) alive = false;     // every QP of the tile is done: no more sweeps
                }
            }
        }
        if (has_item && __any_sync(0xffffffffu, valid)) {
            if (valid && (status != kUnsolved || last_chunk)) admm_finish<T, L>(p, q, m, ws, bb, status, active ? it_end : it_done, rs);
            if (!last_chunk) {                               // publish: this tile's next chunk may start
                __syncwarp();
                __threadfence();
                if (lane == 0) asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p.tile_prog + tile), "r"(chunk + 1) : "memory");
            }
            fence_proxy_async();
            __syncwarp();
        }
    }
}
#undef MPCB_BUF
#endif   // __CUDACC__ && !MPCB_EMU

}  // namespace mpcb
