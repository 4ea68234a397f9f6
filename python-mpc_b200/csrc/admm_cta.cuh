// CTA-per-tile ADMM: one thread block owns a workspace tile of 32 QPs; warp a owns component a of the stage vector
// w = [x | u] (a < NX: state row / column a and its slack, NX <= a < NW: input a - NX), lane = QP.
//
// Why.  admm_tma_kernel (a WARP per tile, lane = QP, the whole 6x6 / 8x8 stage algebra in one thread's registers) needs
// a few thousand tiles to fill the GPU and ~2.5-5 us of dependent FP64 issue per stage: fine for 65536 QPs of the
// lateral shapes, but a batch of 8192 long-horizon QPs of the dynamic model (BASELINE configs[3]: 256 tiles, 142
// elements per stage with the per-stage linearisation) leaves three quarters of the schedulers idle — and so does every
// batch below ~10 k QPs.  Here the stage algebra is spread over NW warps — every product of the stage becomes one
// multiply-add per thread and operand, the operands exchanged through shared memory (2 exchanges per stage and sweep, one
// CTA barrier each) — so a tile keeps NW warps busy and a stage sweep takes 1.0-1.3 us; the stage record AND the stage's
// own linearisation ([A_k | B_k], g_k, tiled like the records at setup: KParams::mdl) arrive by TMA bulk copies, three or
// five buffers deep, on one mbarrier per buffer.  Shared-memory reads are conflict-free by construction (element-major
// records, lane = QP).
//
// The linear solve differs from the other kernels in form, not in content: the records hold the symmetric block inverse
// Linv_k' Linv_k (KParams::minv), so the forward sweep computes g_k = M_k^-1 (r_k - C_{k-1} g_{k-1}) and the backward sweep
// w_k = g_k - M_k^-1 C_k' w_{k+1} with ONE product per stage each instead of the two triangular ones.
//
// What sets its speed (ncu, profiles/r2y_cta_*): with the GPU full (two CTAs per SM) HBM — 5.8 TB/s; with at most one tile
// per SM the number of instructions a warp issues per stage (~290; one every ~8 cycles: fixed-latency dependencies,
// shared-memory and barrier waits).  Hence: one instruction stream for state and input warps, loop-invariant per-thread
// data in small shared-memory tables instead of registers that end up as spill slots, a 255-register instantiation for
// launches that have an SM to themselves.
//
// Functionally a drop-in for admm_tma_kernel: iterations it0+1 .. it_stop of every unsolved QP of the launch's
// tiles, first iteration from explicit (z, y), termination tests every check_termination iterations (the stage
// functions of qp_thread.cuh, the stages split over the warps, norms combined in shared memory), infeasibility
// certificates, exit pass, survivor list.  The kernels agree to the last bits, not bitwise.
#pragma once
#include "admm_kernel.cuh"

#if defined(__CUDACC__) && !defined(MPCB_EMU)
namespace mpcb {

// stage buffers per CTA: 3 with two CTAs per SM (full batches: the kernel is then bound by HBM), 5 when the launch has at most
// one tile per SM — stragglers after a compaction, small batches: those are bound by latency, a deeper prefetch keeps the
// HBM latency of 100+ concurrent streams off the stage chain and a lone CTA may use 255 registers (no spill slots)
constexpr int CTA_NBUF = 3, CTA_NBUF_DEEP = 5;

template <typename L>
struct CtaModel {      // what a time-varying stage stages behind its record: [A | B] (NX x NW, row-major: column a and row i at
                       // fixed strides for every warp) | g | xr (the stage's reference); N + 1 blocks per QP (stage N: xr only,
                       // the rest zero)
    static constexpr int M_AB = 0, M_G = L::NX * L::NW, M_XR = M_G + L::NX, COUNT = M_XR + L::NX;
};

// 1/rho of a row — needed only by the first iteration of a solve (explicit y on entry).  Inline Newton reciprocal: a true
// FP64 division is an out-of-line call, and a call inside the sweeps costs them registers on every iteration.
template <typename T>
struct CtaRinv {
    T rho_eq;
    __device__ __forceinline__ T rinv_of(T rb) const { return fast_rcp(rb); }
    __device__ __forceinline__ T rinv_eq() const { return fast_rcp(rho_eq); }
};

template <typename T, typename L, bool TV, int NBUF = CTA_NBUF>
struct CtaSmem {
    // elements per staged stage: the record and, behind it, A | B | g of the stage; the stage's reference xr rides in the
    // record's t slot during the forward sweep (which does not read t) — the budget is two CTAs per SM
    static constexpr int RS = L::REC + (TV ? CtaModel<L>::M_XR : 0);
    static_assert(!TV || L::NX <= L::NW, "xr fits the t slot");
    static constexpr size_t BUF_BYTES = (size_t)RS * TILE * sizeof(T);
    // exchange areas: [NW] for the single products, [NW | NX] for the merged one; consecutive exchanges alternate between
    // the two, which is what makes one barrier per exchange enough
    static constexpr size_t XCH_BYTES = (size_t)(2 * L::NW + L::NX) * TILE * sizeof(T);
    static constexpr size_t CQ_BYTES = (size_t)TILE * sizeof(T);            // cost scaling c per lane (read once per stage)
    static constexpr size_t MT_BYTES = (size_t)L::NW * ((L::NW + 7) / 8) * 8 * sizeof(int);      // record offsets of row a of the block inverse
    static constexpr size_t CT_BYTES = (size_t)L::NW * 4 * sizeof(T);       // Q, QN, lower, upper bound of component a
    static constexpr size_t BYTES = NBUF * BUF_BYTES + 64 + XCH_BYTES + CQ_BYTES + CT_BYTES + MT_BYTES;
    // (the termination test works in the record buffers — free at that point: per-warp partial norms, the residuals of the
    //  last test per lane, the open / active flags)
    static constexpr size_t RED_ELEMS = (size_t)(L::NW * 13 + 5) * TILE;
    static_assert((RED_ELEMS + 2 * TILE) * sizeof(T) + 64 * sizeof(int) <= NBUF * BUF_BYTES, "test scratch fits the buffers");
};

// Termination sweep of the stages [k0, k1) of one QP (lane) — out of line: it runs once every check_termination
// iterations and must not set the register allocation of the sweeps (two CTAs of NW warps per SM: 128 registers).
template <typename T, typename L>
__device__ __noinline__ void cta_test_range(const KParams<T>& p, const AdmmConst<T, L>& q, const Ws<T, L>& ws, int bb, int k0, int k1,
                                            bool cert, bool first, TestAcc<T>& t) {
    constexpr int NX = L::NX;
    const int N = p.N;
    TestCarry<T, L> cy;
    Model<T, L> m;
    if (!p.tv) load_model<T, L>(p, bb, 0, m);
    if (k0 == 0) {
        admm_test_begin<T, L>(p, q, bb, ws.hdr, cy, t, cert, first, ws.scr_hdr);
    } else {
        test_reset(t);
        const T* Rp = ws.R(k0 - 1);
#pragma unroll
        for (int i = 0; i < NX; ++i) {           // what stage k0 - 1 hands over: E and w (= y, or dy) of rows dyn_{k0}
            const T Ed = MPCB_AT(Rp, L::R_E + L::ODN + i);
            const T beq = -Ed * model_g<T, L>(p, bb, k0 - 1, i);
            T w = q.rho_eq * (MPCB_AT(Rp, L::R_P + L::ODN + i) - beq);
            if (cert) w -= q.rho_eq * old_yr(first, MPCB_AT(ws.S(k0 - 1), L::VS + L::ODN + i),
                                             first ? MPCB_AT(ws.Y(k0 - 1), L::ODN + i) : (T)0, beq, beq, q.rho_eq);
            cy.Ed_cur[i] = Ed; cy.wd_cur[i] = w;
        }
    }
    for (int k = k0; k < k1; ++k) {
        if (p.tv && k < N) load_model<T, L>(p, bb, k, m);
        admm_test_stage<T, L>(p, q, m, bb, k, ws.R(k), ws.R(k < N ? k + 1 : k), cy, t, cert, first, ws.Y(k), ws.S(k),
                              ws.S(k < N ? k + 1 : k));
    }
}
template <typename T, typename L>
__device__ __noinline__ void cta_exit_range(const KParams<T>& p, const AdmmConst<T, L>& q, const Ws<T, L>& ws, int bb, int kfirst,
                                            int kstep) {
    for (int k = kfirst; k <= p.N; k += kstep) admm_exit_stage<T, L>(p, q, bb, k, ws.R(k), ws.Y(k));
}

__device__ __forceinline__ void cta_sync() { asm volatile("bar.sync 0;" ::: "memory"); }
__device__ __forceinline__ int cta_opaque(int v) { asm volatile("" : "+r"(v)); return v; }

// (A variant with the warp's component index as a template parameter — every record offset an immediate, the triangular
// products without their structural zeros — was measured: 7 % faster for a lone tile, 60 % SLOWER for a full batch: eight
// specialised bodies, two CTAs per SM, thrash the instruction cache.  One body, run-time component index.)
template <typename T, typename L, bool TV, int NBUF = CTA_NBUF>
__global__ void __launch_bounds__(L::NW * 32, NBUF == CTA_NBUF ? 2 : 1) admm_cta_kernel(const __grid_constant__ KParams<T> p) {
    constexpr int NX = L::NX, NU = L::NU, NW = L::NW, NS = L::NS;
    typedef CtaSmem<T, L, TV, NBUF> SM;
    typedef CtaModel<L> CM;
    constexpr int RS = SM::RS;
    // the forward sweep forms its whole right-hand side: it loads all of a record but the t slots (two runs)
    constexpr unsigned REC_BYTES = L::REC * TILE * sizeof(T), FWD_BYTES = (L::REC - L::NW) * TILE * sizeof(T),
                       MDL_BYTES = CM::M_XR * TILE * sizeof(T), XR_BYTES = L::NX * TILE * sizeof(T);
    extern __shared__ __align__(128) unsigned char smem_raw[];
    T* const bufs = reinterpret_cast<T*>(smem_raw);
    unsigned long long* const bar = reinterpret_cast<unsigned long long*>(smem_raw + NBUF * SM::BUF_BYTES);
    T* const xch = reinterpret_cast<T*>(smem_raw + NBUF * SM::BUF_BYTES + 64);
    T* const csm = reinterpret_cast<T*>(smem_raw + NBUF * SM::BUF_BYTES + 64 + SM::XCH_BYTES);      // [32]
    constexpr int MTW = ((NW + 7) / 8) * 8;                 // offsets per row of the table, padded to whole int4 loads
    T* const ctab = csm + TILE;                             // [NW][4]
    int* const mtab = reinterpret_cast<int*>(ctab + NW * 4);      // [NW][MTW]
    T* const red = bufs;                                    // the termination test reads global memory: the buffers are free then
    T* const res = red + SM::RED_ELEMS;                     // [2][32]
    int* const flags = reinterpret_cast<int*>(res + 2 * TILE);      // [32] per-lane, [32..] CTA-wide

    // (opaque: the compiler would otherwise re-read the thread index — an S2R, ~20 cycles — wherever it needs a or lane again)
    //  — measured: pays with 255 registers (deep instantiation), costs spill slots with 128)
    const int a = NBUF == CTA_NBUF ? (int)(threadIdx.x >> 5) : cta_opaque((int)(threadIdx.x >> 5));
    const int lane = NBUF == CTA_NBUF ? (int)(threadIdx.x & 31) : cta_opaque((int)(threadIdx.x & 31));
    const int N = p.N, tile = blockIdx.x;
    const int b = tile * TILE + lane;
    const int bb = b < p.B ? (p.qp_map ? p.qp_map[b] : b) : 0;
    const bool valid = b < p.B && p.status[bb] == kUnsolved;
    if (!__any_sync(0xffffffffu, valid)) return;            // nothing left to do in this tile (every warp sees the same 32 QPs)
    const bool isx = a < NX, isu = !isx;
    const int jx = isx ? a : 0, ju = isu ? a - NX : 0;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NBUF; ++i) mbar_init(&bar[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    Ws<T, L> ws(p, b);
    const T* const rec_tile = ws.rec - lane;                // base of the tile's records (what TMA copies from)
    const T* const mdl_tile = TV ? p.mdl + (size_t)tile * (N + 1) * CM::COUNT * TILE : nullptr;
    AdmmConst<T, L> q;
    admm_setup_const<T, L>(p, bb, ws, q);
    if (a == 0) csm[lane] = q.c;
    // row r of the symmetric block inverse (lower triangle stored): (r, d <= r) at tri(r) + d, (r, d > r) = (d, r) at tri(d) + r.
    // The offsets live in shared memory and are re-read every stage (two vector loads): eight registers per thread held
    // across the sweeps end up as spill slots, and re-deriving them from the thread index costs ~90 instructions per stage.
    if (threadIdx.x < NW) {                                 // weights and bounds of component r (inputs: no linear cost term)
        const int r = threadIdx.x, rx = r < NX ? r : 0, ru = r >= NX ? r - NX : 0;
        ctab[r * 4 + 0] = r < NX ? p.Q[rx] : (T)0;
        ctab[r * 4 + 1] = r < NX ? p.QN[rx] : (T)0;
        ctab[r * 4 + 2] = r < NX ? p.xmin[rx] : p.umin[ru];
        ctab[r * 4 + 3] = r < NX ? p.xmax[rx] : p.umax[ru];
    }
    for (int i = threadIdx.x; i < NW * MTW; i += NW * 32) {
        const int r = i / MTW, d = i % MTW;
        mtab[i] = d < NW ? (L::R_F + (d <= r ? r * (r + 1) / 2 + d : d * (d + 1) / 2 + r)) * TILE : 0;
    }
    const T rho = p.rho_c, rho_eq = p.rho_eq_c, sigma = p.sigma, alpha = p.alpha;      // (== q.rho, q.rho_eq)
    const bool inf_bounds = q.inf_bounds;
    const CtaRinv<T> qr{rho_eq};
    if (valid && p.it0 == 0 && !p.warm) {                   // cold start: x = z = y = 0 (stages split over the warps)
        for (int k = a; k <= N; k += NW) {
            T* R = ws.R(k); T* Y = ws.Y(k);
            for (int e = 0; e < L::VS; ++e) MPCB_AT(R, L::R_X + e) = 0;
            for (int e = 0; e < L::CS; ++e) { MPCB_AT(R, L::R_P + e) = 0; MPCB_AT(Y, e) = 0; }
        }
        if (a == 0)
            for (int i = 0; i < NX; ++i) { MPCB_AT(ws.hdr, L::H_P0 + i) = 0; MPCB_AT(ws.hdr, L::H_Y0 + i) = 0; }
    }
    // column a and row a of [A | B]: loop-invariant for a time-invariant model (registers), part of the staged record otherwise
    const size_t bo = p.model_bs ? (size_t)bb : 0, ldm = p.model_bs ? p.ld : 1;
    T col0[NX], row0[NW], g0 = 0;
#pragma unroll
    for (int i = 0; i < NX; ++i)
        col0[i] = TV ? (T)0 : (isx ? p.Ad[(size_t)(i * NX + jx) * ldm + bo] : p.Bd[(size_t)(i * NU + ju) * ldm + bo]);
#pragma unroll
    for (int j = 0; j < NW; ++j)
        row0[j] = (TV || !isx) ? (T)0 : (j < NX ? p.Ad[(size_t)(jx * NX + (j < NX ? j : 0)) * ldm + bo]
                                                : p.Bd[(size_t)(jx * NU + (j >= NX ? j - NX : 0)) * ldm + bo]);
    if (!TV && isx) g0 = model_g<T, L>(p, bb, 0, jx);
    // (a time-invariant problem with per-stage references keeps reading them from the input array)
    const T xr0 = (!TV && isx && !p.xr_tv) ? p.Xr[(size_t)jx * p.ld + bb] : (T)0;
    const T xr_first = (TV && isx) ? mdl_tile[(size_t)(CM::M_XR + jx) * TILE + lane] : (T)0;
    const T Sj = (NS && isx) ? p.S[jx] : (T)0, Wj = (NS && isx) ? p.W[jx] : (T)0;
    // this component's weights and (stage-independent) bounds: indexed by the run-time component, read once
    // (weights and bounds of the component are re-read from a small shared-memory table every stage: a register each, held
    //  across the sweeps at 128 registers per thread, is a spill slot in local memory — and the L1 left beside 2 x 114 KB of
    //  shared memory does not hold the spill slots of 512 threads)
    const T E0 = isx ? MPCB_AT(ws.hdr, L::H_E0 + jx) : (T)0;
    const T beq0 = isx ? -E0 * p.x_init[(size_t)jx * p.ld + bb] : (T)0;
    fence_proxy_async();
    cta_sync();

    unsigned ph = 0u;                                       // bit i: phase parity of the mbarrier of buffer i
    bool active = valid;
    int status = kUnsolved, it_done = 0;

    // Loop-invariant record offsets of this warp's component.  Variables of a stage are laid out slack | x | u and the bound
    // rows bx | bu are contiguous, so component a — a state or an input — finds its scaling, iterate and bound row at one
    // run-time offset each: the x warps and the u warps run the SAME instructions (an input is a state without dynamics
    // rows, cost-reference and slack: its E_dyn, Q and W factors are zero), which is what keeps the stage at ~200
    // instructions per warp — the chain of a stage is bound by issue latency, not by the FP64 pipe.
    static_assert(L::OBU == L::OBX + NX && L::OU == L::OX + NX, "component a: variable OX + a, bound row OBX + a");
    const int cv = isx ? L::OX + jx : L::OU + ju;           // my variable inside D / x
    constexpr int RB = L::OBX;                              // my bound row: RB + a
    const int4* const mrow = reinterpret_cast<const int4*>(mtab + a * MTW);
    const bool has_xbox = p.xbox != nullptr;                // per-stage state boxes (mpc_): states only
    // (the last warp — an input: the least work per stage — drives the TMA)
    const int biN = N % NBUF;                           // buffer of stage N

    // the elected thread starts the bulk copies of stage k into buffer bi (record, and the stage's model behind it)
    auto issue = [&](int k, int bi, bool fwd) {
        if (a == NW - 1 && lane == 0) {
            unsigned long long* br = &bar[bi];
            T* dst = bufs + (size_t)bi * (RS * TILE);
            const unsigned rb = fwd ? FWD_BYTES : REC_BYTES;
            mbar_expect_tx(br, rb + (TV ? MDL_BYTES : 0u) + ((TV && fwd) ? XR_BYTES : 0u));
            const T* src = rec_tile + (size_t)k * L::REC * TILE;
            if (fwd) {
                tma_load_1d(dst, src, L::R_T * TILE * sizeof(T), br);
                tma_load_1d(dst + L::R_P * TILE, src + L::R_P * TILE, (L::REC - L::R_P) * TILE * sizeof(T), br);
            } else {
                tma_load_1d(dst, src, rb, br);
            }
            if (TV) tma_load_1d(dst + L::REC * TILE, mdl_tile + (size_t)k * CM::COUNT * TILE, MDL_BYTES, br);
            if (TV && fwd) tma_load_1d(dst + L::R_T * TILE, mdl_tile + ((size_t)k * CM::COUNT + CM::M_XR) * TILE, XR_BYTES, br);
        }
    };
    auto wait = [&](int bi) {
        mbar_wait(&bar[bi], (ph >> bi) & 1u);
        ph ^= 1u << bi;
    };
    // Exchanges.  Every warp contributes its component, a CTA barrier, every warp reads what it needs:  sum_d coef[d] * v_d
    // (three partial sums: the chain of a stage is bound by the FP64 dependent-issue latency).  The coefficients are fetched
    // from the staged record BEFORE the exchange (arrays in registers): their shared-memory latency hides behind the barrier.
    // xdot uses area X0, xdotA / xdotB / xdot2 the areas XA | XB; the sweeps alternate between the two families, so a warp
    // that runs ahead to the next exchange never overwrites what a slower warp is still reading.
    T* const X0 = xch + lane;
    T* const XA = xch + (size_t)NW * TILE + lane;
    T* const XB = xch + (size_t)2 * NW * TILE + lane;
    auto dot3 = [&](const T* coef, int nt, const T* slot) -> T {
        T s0 = 0, s1 = 0, s2 = 0;
#pragma unroll
        for (int d = 0; d < NW; d += 3) {
            if (d < nt) s0 += coef[d] * slot[d * TILE];
            if (d + 1 < nt) s1 += coef[d + 1] * slot[(d + 1) * TILE];
            if (d + 2 < nt) s2 += coef[d + 2] * slot[(d + 2) * TILE];
        }
        return (s0 + s1) + s2;
    };
    auto xdot = [&](const T* coef, T v) -> T {              // all NW components
        X0[a * TILE] = v;
        cta_sync();
        return dot3(coef, NW, X0);
    };
    auto xdotA = [&](const T* coef, T v) -> T {
        XA[a * TILE] = v;
        cta_sync();
        return dot3(coef, NW, XA);
    };
    auto xdotB = [&](const T* coef, T v) -> T {             // the NX state components (only state warps contribute)
        if (isx) XB[a * TILE] = v;
        cta_sync();
        return dot3(coef, NX, XB);
    };

    // stage 0 for the first forward sweep
    issue(0, 0, true);
    wait(0);

    for (int it = p.it0 + 1; it <= p.it_stop; ++it) {
        const bool wr = active;
        const bool save = wr && admm_saves(p, it);          // the next iteration is tested: duplicate the new state
        if (admm_needs_copy(p, it)) {                       // (tested at it <= 2: the certificates' old state is the entry state)
            if (wr) {
                for (int k = a; k <= N; k += NW) {
                    const T* R = ws.R(k); T* O = ws.S(k);
                    for (int e = 0; e < L::VS; ++e) MPCB_AT(O, e) = MPCB_AT(R, L::R_X + e);
                    for (int e = 0; e < L::CS; ++e) MPCB_AT(O, L::VS + e) = MPCB_AT(R, L::R_P + e);
                }
                if (a == 0)
                    for (int i = 0; i < NX; ++i) MPCB_AT(ws.scr_hdr, i) = MPCB_AT(ws.hdr, L::H_P0 + i);
            }
        }
        // the two sweeps of one iteration; FIRST (iteration 1 of a solve: rows enter as explicit (z, y)) is a compile-time
        // flag: the steady-state instantiation carries none of that code
        auto sweeps = [&](auto first_tag) {
        constexpr bool first = decltype(first_tag)::value;
        T P0 = isx ? MPCB_AT(ws.hdr, L::H_P0 + jx) : (T)0;
        T z0 = 0, y0 = 0;
        if (isx) {
            const Row<T> r0 = row_state(first, P0, first ? MPCB_AT(ws.hdr, L::H_Y0 + jx) : (T)0, beq0, beq0, qr.rinv_eq());
            z0 = r0.z; y0 = r0.yr;
        }
        // ================================================================== forward sweep:  g_k = M_k^-1 (r_k - C_{k-1} g_{k-1})
        // Two exchanges per stage: the product with the block inverse, then ONE exchange for both the coupling into stage
        // k + 1 ([A_k B_k] D g_k) and the dynamics rows of stage k + 1 (column a of [A_{k+1} B_{k+1}] times their duals).
        {
            T Ed_cur = E0, vd_cur = rho_eq * (z0 - y0), cprev = 0;      // (input warps: E0 = 0, their dynamics terms vanish)
            int bi = 0;
            T* Rg = ws.R(0);
#pragma unroll
            for (int j = 1; j < NBUF; ++j)
                if (j <= N) issue(j, j, true);
            T* S = bufs + lane;                             // stage 0 is in buffer 0
            // my row of dyn_{k+1} (state warps, k < N): E and rho (z - y/rho)
            auto dyn_row = [&](const T* Sk, const T* Mk, const T* Yk_, T& Edn, T& vdn) {
                Edn = MPCB_AT(Sk, L::R_E + L::ODN + jx);
                const T gk = TV ? MPCB_AT(Mk, CM::M_G + jx) : g0;
                const T beq = -Edn * gk;
                const Row<T> rd = row_state(first, MPCB_AT(Sk, L::R_P + L::ODN + jx), first ? MPCB_AT(Yk_, L::ODN + jx) : (T)0,
                                            beq, beq, qr.rinv_eq());
                vdn = rho_eq * (rd.z - rd.yr);
            };
            T Ed_next = 0, vd_next = 0, acc;
            {
                if (isx && N >= 1) dyn_row(S, S + L::REC * TILE, ws.Y(0), Ed_next, vd_next);
                T colv[NX];
#pragma unroll
                for (int i = 0; i < NX; ++i) colv[i] = TV ? MPCB_AT(S + L::REC * TILE, CM::M_AB + i * NW + a) : col0[i];
                acc = xdotB(colv, Ed_next * vd_next);
            }
            for (int k = 0; k <= N; ++k) {
                const bool last = (k == N);
                const T* M = S + L::REC * TILE;
                const T* Yk = ws.Y(k);
                const bool idle = last && isu;              // there is no input at stage N
                const T Da = idle ? (T)1 : MPCB_AT(S, L::R_D + cv);
                T Mrow[NW];
                {
                    int mo[MTW];
#pragma unroll
                    for (int v = 0; v < MTW / 4; ++v) {
                        const int4 o4 = mrow[v];
                        mo[4 * v] = o4.x; mo[4 * v + 1] = o4.y; mo[4 * v + 2] = o4.z; mo[4 * v + 3] = o4.w;
                    }
#pragma unroll
                    for (int d = 0; d < NW; ++d) Mrow[d] = S[mo[d]];
                }
                // my bound row, my cost gradient, my part of the couplings with stage k - 1 / k + 1
                const T Eb = MPCB_AT(S, L::R_E + RB + a);
                const T blo = (has_xbox && isx) ? p.xbox[(k * 2 + 0) * NX + jx] : ctab[a * 4 + 2];
                const T bhi = (has_xbox && isx) ? p.xbox[(k * 2 + 1) * NX + jx] : ctab[a * 4 + 3];
                const T bx = Eb * Da, lb = Eb * blo, ub = Eb * bhi;
                const T rb = row_rho(inf_bounds, lb, ub, rho, rho_eq);
                const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + RB + a), Yk + (size_t)(RB + a) * TILE, lb, ub, rb, qr);
                const T vbx = rb * (rw.z - rw.yr);
                const T Qj = ctab[a * 4 + (last ? 1 : 0)];   // (inputs: 0 — R sits in the matrix, there is no linear term)
                const T xr = TV ? MPCB_AT(S, L::R_T + jx) : (p.xr_tv ? p.Xr[((size_t)k * NX + jx) * p.ld + bb] : xr0);
                const T c = csm[lane];
                const T qh = c * Da * (-(Qj * xr));
                const T ex = Ed_cur * Da;
                T v = sigma * MPCB_AT(S, L::R_X + cv) - qh - ex * vd_cur + bx * vbx + Da * acc;
                if (NS && isx) {
                    const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? jx : 0));
                    const T bs = Sj * Eb * Dsl;
                    const T mss = c * Wj * Dsl * Dsl + sigma + rb * bs * bs;
                    const T mxs = rb * bx * bs;
                    const T rsl = sigma * MPCB_AT(S, L::R_X + L::OS + (NS ? jx : 0)) + bs * vbx;
                    v -= mxs * fast_rcp(mss) * rsl;
                }
                if (k > 0) v += rho_eq * ex * Ed_cur * cprev;
                const T g = xdot(Mrow, idle ? (T)0 : v);    // g = M_k^-1 r
                if (wr) MPCB_AT(Rg, L::R_T + a) = g;
                if (last) { MPCB_AT(S, L::R_T + a) = g; break; }      // turn-around: backward stage N reuses this buffer
                // row a of [A_k | B_k]  (input warps read row 0: their product is never used)
                T rowv[NW];
#pragma unroll
                for (int j = 0; j < NW; ++j) rowv[j] = TV ? MPCB_AT(M, CM::M_AB + jx * NW + j) : row0[j];
                // stage k + 1: its dynamics rows ride in the same exchange
                const int bn = bi == NBUF - 1 ? 0 : bi + 1;
                wait(bn);
                T* Sn = bufs + (size_t)bn * (RS * TILE) + lane;
                Ed_cur = Ed_next; vd_cur = vd_next;
                Ed_next = 0; vd_next = 0;
                if (isx && k + 1 < N) dyn_row(Sn, Sn + L::REC * TILE, ws.Y(k + 1), Ed_next, vd_next);
                XA[a * TILE] = Da * g;
                if (isx) XB[a * TILE] = Ed_next * vd_next;
                cta_sync();
                // the buffer of stage k is free once every warp is past this exchange
                if (k + NBUF <= N) issue(k + NBUF, bi, true);
                T colv[NX];
#pragma unroll
                for (int i = 0; i < NX; ++i) colv[i] = TV ? MPCB_AT(Sn + L::REC * TILE, CM::M_AB + i * NW + a) : col0[i];
                cprev = dot3(rowv, NW, XA);                 // [A B] (D (.) g)
                acc = dot3(colv, NX, XB);
                S = Sn; bi = bn;
                Rg += (size_t)L::REC * TILE;
            }
        }
        fence_proxy_async();                                // g_0 .. g_N (generic stores) before the backward sweep's TMA reads
        cta_sync();
        // ================================================================== backward sweep:  w_k = g_k - M_k^-1 C_k' w_{k+1}
        // Two exchanges per stage here too: D w_k (for the rows dyn_{k+1}) shares its exchange with the coupling of stage
        // k - 1 (column a of [A_{k-1} B_{k-1}] times E ex w_k).
        {
            T xt_next = 0, Dx_next = 1;
            int bi = biN;
            T* Rw = ws.R(N);
            T* Ow = ws.S(N);
            {
                int bj = bi;
#pragma unroll
                for (int j = 1; j < NBUF; ++j) {
                    bj = bj == 0 ? NBUF - 1 : bj - 1;
                    if (N - j >= 0) issue(N - j, bj, false);
                }
            }
            T* S = bufs + (size_t)bi * (RS * TILE) + lane;
            T acc = 0;                                      // stage N has no successor
            T Ed_next = 1, exn = 1;
            for (int k = N; k >= 0; --k) {
                const bool last = (k == N);
                const T* M = S + L::REC * TILE;
                const T* Yk = ws.Y(k);
                const bool idle = last && isu;
                const T Da = idle ? (T)1 : MPCB_AT(S, L::R_D + cv);
                const T gfw = MPCB_AT(S, L::R_T + a);
                T Mrow[NW];
                {
                    int mo[MTW];
#pragma unroll
                    for (int v = 0; v < MTW / 4; ++v) {
                        const int4 o4 = mrow[v];
                        mo[4 * v] = o4.x; mo[4 * v + 1] = o4.y; mo[4 * v + 2] = o4.z; mo[4 * v + 3] = o4.w;
                    }
#pragma unroll
                    for (int d = 0; d < NW; ++d) Mrow[d] = S[mo[d]];
                }
                const T w = gfw - xdot(Mrow, -rho_eq * Da * acc);
                // every warp is past the first exchange of stage k: the buffer of stage k + 1 is free
                if (k <= N - 1 && k + 1 - NBUF >= 0) issue(k + 1 - NBUF, bi == NBUF - 1 ? 0 : bi + 1, false);
                T rowv[NW];
#pragma unroll
                for (int j = 0; j < NW; ++j) rowv[j] = TV ? MPCB_AT(M, CM::M_AB + jx * NW + j) : row0[j];
                // stage k - 1: ex_k = E_dyn(k) D_x(k), its coupling product rides in the same exchange
                const int bp = bi == 0 ? NBUF - 1 : bi - 1;
                T* Sp = S;
                T Ed_prev = 1, exp_ = 1;
                if (k > 0) {
                    wait(bp);
                    Sp = bufs + (size_t)bp * (RS * TILE) + lane;
                    if (isx) { Ed_prev = MPCB_AT(Sp, L::R_E + L::ODN + jx); exp_ = Ed_prev * Da; }
                }
                XA[a * TILE] = Da * w;
                if (isx) XB[a * TILE] = Ed_prev * exp_ * w;
                cta_sync();
                T colv[NX];
#pragma unroll
                for (int i = 0; i < NX; ++i) colv[i] = TV ? MPCB_AT(Sp + L::REC * TILE, CM::M_AB + i * NW + a) : col0[i];
                const T accd = dot3(rowv, NW, XA);          // rows dyn_{k+1} need D (.) w of every component
                acc = dot3(colv, NX, XB);
                // my bound row and my variable
                const T Eb = MPCB_AT(S, L::R_E + RB + a);
                const T blo = (has_xbox && isx) ? p.xbox[(k * 2 + 0) * NX + jx] : ctab[a * 4 + 2];
                const T bhi = (has_xbox && isx) ? p.xbox[(k * 2 + 1) * NX + jx] : ctab[a * 4 + 3];
                const T bx = Eb * Da, lb = Eb * blo, ub = Eb * bhi;
                const T rb = row_rho(inf_bounds, lb, ub, rho, rho_eq);
                const Row<T> rw = row_state_b(first, MPCB_AT(S, L::R_P + RB + a), Yk + (size_t)(RB + a) * TILE, lb, ub, rb, qr);
                T ztil = bx * w;
                if (NS && isx) {
                    const T c = csm[lane];
                    const T Dsl = MPCB_AT(S, L::R_D + L::OS + (NS ? jx : 0));
                    const T bs = Sj * Eb * Dsl;
                    const T mss = c * Wj * Dsl * Dsl + sigma + rb * bs * bs;
                    const T mxs = rb * bx * bs;
                    const T sold = MPCB_AT(S, L::R_X + L::OS + (NS ? jx : 0));
                    const T rsl = sigma * sold + bs * (rb * (rw.z - rw.yr));
                    const T st = (rsl - mxs * w) * fast_rcp(mss);
                    ztil += bs * st;
                    const T sn = alpha * st + ((T)1 - alpha) * sold;
                    if (wr) MPCB_AT(Rw, L::R_X + L::OS + (NS ? jx : 0)) = sn;
                    if (save) MPCB_AT(Ow, L::OS + (NS ? jx : 0)) = sn;
                    if (k == 0) MPCB_AT(S, L::R_X + L::OS + (NS ? jx : 0)) = sn;
                }
                if (!idle) {
                    const T pn = row_next(ztil, rw, alpha);
                    const T xnw = alpha * w + ((T)1 - alpha) * MPCB_AT(S, L::R_X + cv);
                    if (wr) { MPCB_AT(Rw, L::R_P + RB + a) = pn; MPCB_AT(Rw, L::R_X + cv) = xnw; }
                    if (save) { MPCB_AT(Ow, L::VS + RB + a) = pn; MPCB_AT(Ow, cv) = xnw; }
                    if (k == 0) { MPCB_AT(S, L::R_P + RB + a) = pn; MPCB_AT(S, L::R_X + cv) = xnw; }     // turn-around
                }
                if (isx) {
                    if (!last) {
                        // row dyn_{k+1}:  E (A D x~_k + B D u~_k) - ex_{k+1} x~_{k+1} = -E g_k
                        const T zt = Ed_next * accd - exn * xt_next;
                        const T gk = TV ? MPCB_AT(M, CM::M_G + jx) : g0;
                        const T beq = -Ed_next * gk;
                        const Row<T> rd = row_state(first, MPCB_AT(S, L::R_P + L::ODN + jx), first ? MPCB_AT(Yk, L::ODN + jx) : (T)0,
                                                    beq, beq, qr.rinv_eq());
                        const T pdn = row_next(zt, rd, alpha);
                        if (wr) MPCB_AT(Rw, L::R_P + L::ODN + jx) = pdn;
                        if (save) MPCB_AT(Ow, L::VS + L::ODN + jx) = pdn;
                        if (k == 0) MPCB_AT(S, L::R_P + L::ODN + jx) = pdn;
                    }
                    // (stage 0 enters the next forward sweep in this buffer: its reference goes where the forward loads put it)
                    if (TV && k == 0) MPCB_AT(S, L::R_T + jx) = xr_first;
                    xt_next = w; Dx_next = Da;
                }
                Ed_next = Ed_prev; exn = exp_;
                S = Sp; bi = bp;
                Rw -= (size_t)L::REC * TILE;
                Ow -= (size_t)(L::VS + L::CS) * TILE;
            }
            // rows dyn_0 (header)
            if (isx) {
                Row<T> rw; rw.z = z0; rw.yr = y0;
                P0 = row_next(-(E0 * Dx_next) * xt_next, rw, alpha);
                if (wr) MPCB_AT(ws.hdr, L::H_P0 + jx) = P0;
                if (save) MPCB_AT(ws.scr_hdr, jx) = P0;
            }
        }
        };
        const bool first = (it == 1);
        if (first) sweeps(std::true_type{}); else sweeps(std::false_type{});
        fence_proxy_async();                                // new x, p (generic stores) before the next sweep's TMA reads
        cta_sync();
        // ================================================================== termination test (auxil.c: check_termination)
        if (admm_is_tested(p, it)) {                        // CTA-uniform
            const bool was_active = active;                 // (consistent over the warps: synchronised at the end of every test)
            const int per = (N + 1 + NW - 1) / NW;
            const int k0 = a * per < N + 1 ? a * per : N + 1, k1 = k0 + per < N + 1 ? k0 + per : N + 1;
            if (a == 0) { flags[lane] = active ? 1 : 0; }   // 1: still open in the current pass
            cta_sync();
            for (int pass = 0; pass < 2; ++pass) {          // residuals of (x, y), then certificates of (dx, dy)
                const bool cert = pass == 1;
                TestAcc<T> t;
                test_reset(t);
                if (flags[lane] && k0 < k1) cta_test_range<T, L>(p, q, ws, bb, k0, k1, cert, first, t);
                T* mine = red + ((size_t)a * 13) * TILE + lane;
                mine[0 * TILE] = t.pri; mine[1 * TILE] = t.dua; mine[2 * TILE] = t.nz; mine[3 * TILE] = t.nAx; mine[4 * TILE] = t.nq;
                mine[5 * TILE] = t.nAty; mine[6 * TILE] = t.nPx; mine[7 * TILE] = t.nEw; mine[8 * TILE] = t.nDv; mine[9 * TILE] = t.aup;
                mine[10 * TILE] = t.alo; mine[11 * TILE] = t.lhs; mine[12 * TILE] = t.qv;
                cta_sync();
                if (a == 0) {
                    int open_after = 0;
                    if (flags[lane]) {
                        for (int w2 = 1; w2 < NW; ++w2) {
                            const T* o = red + ((size_t)w2 * 13) * TILE + lane;
                            t.pri = tmax(t.pri, o[0 * TILE]); t.dua = tmax(t.dua, o[1 * TILE]); t.nz = tmax(t.nz, o[2 * TILE]);
                            t.nAx = tmax(t.nAx, o[3 * TILE]); t.nq = tmax(t.nq, o[4 * TILE]); t.nAty = tmax(t.nAty, o[5 * TILE]);
                            t.nPx = tmax(t.nPx, o[6 * TILE]); t.nEw = tmax(t.nEw, o[7 * TILE]); t.nDv = tmax(t.nDv, o[8 * TILE]);
                            t.aup = tmax(t.aup, o[9 * TILE]); t.alo = tmin(t.alo, o[10 * TILE]); t.lhs += o[11 * TILE]; t.qv += o[12 * TILE];
                        }
                        if (!cert) {
                            Resid<T> rs;
                            test_to_resid(t, rs);
                            if (admm_residual_test<T, L>(p, q, rs)) { status = kSolved; active = false; it_done = it; }
                            else if (p.certs || it == p.max_iter) open_after = 1;
                            res[lane] = rs.pri; res[TILE + lane] = rs.dua;
                            // (the certificate pass needs the norms of this one: parked in the reduction area of warp 0)
                            T* keep = red + (size_t)NW * 13 * TILE + lane;
                            keep[0 * TILE] = rs.nz; keep[1 * TILE] = rs.nAx; keep[2 * TILE] = rs.nq; keep[3 * TILE] = rs.nAty; keep[4 * TILE] = rs.nPx;
                        } else {
                            Resid<T> rs;
                            const T* keep = red + (size_t)NW * 13 * TILE + lane;
                            rs.pri = res[lane]; rs.dua = res[TILE + lane];
                            rs.nz = keep[0 * TILE]; rs.nAx = keep[1 * TILE]; rs.nq = keep[2 * TILE]; rs.nAty = keep[3 * TILE]; rs.nPx = keep[4 * TILE];
                            Cert<T> ct;
                            test_to_cert(t, ct);
                            if (admm_decide<T, L>(p, q, rs, ct, it == p.max_iter, status)) { active = false; it_done = it; }
                        }
                    }
                    flags[lane] = cert ? 0 : open_after;
                    flags[32 + lane] = active ? 1 : 0;
                }
                cta_sync();
                int any_open = 0;
                if (!cert) any_open = __any_sync(0xffffffffu, flags[lane] != 0);
                if (cert || !any_open) break;
            }
            // a QP that terminated leaves explicit (z, y) behind (stages split over the warps); warp 0 owns the header
            const bool now_active = flags[32 + lane] != 0;
            const bool finished = was_active && !now_active;
            if (finished) cta_exit_range<T, L>(p, q, ws, bb, a, NW);
            if (a == 0 && finished) {
                admm_exit_header<T, L>(p, q, bb, ws.hdr);
                p.iter[bb] = it_done; p.pri_res[bb] = res[lane]; p.dua_res[bb] = res[TILE + lane];
            }
            active = now_active;
            cta_sync();
            if (a == 0 && finished) p.status[bb] = status;      // (after the exit pass: the status gates every later launch)
            if (!__any_sync(0xffffffffu, active)) return;     // every QP of the tile is done (the same answer in every warp)
            // the buffers served the reduction: stage 0 again for the next forward sweep
            fence_proxy_async();
            cta_sync();
            if (it < p.it_stop) { issue(0, 0, true); wait(0); }
        }
    }
    // unsolved QPs of a non-final launch keep their rows in p-form and put themselves on the survivor list
    if (a == 0 && active && p.list_survivors) {
        const int slot = atomicAdd(p.n_survivors, 1);
        p.survivors[slot] = bb;
    }
}

}  // namespace mpcb
#endif
