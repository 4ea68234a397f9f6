// Runtime layer shared by the translation units of libmpc_b200.so: CUDA runtime wrappers (or, for tests/emu, their host
// stand-ins), kernel launchers, the solver object and the kernel-parameter block built from it.
#pragma once
#include "../../include/mpc_b200.h"
#include "mpc_common.h"
#include "qp_thread.cuh"

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>

using namespace mpcb;

// =============================================================================================
// runtime layer
// =============================================================================================
// process-wide state, defined once in mpc_b200.cu (the library is built from several translation units: one per
// compiled (shape, dtype) plus the ABI layer — see __graft_entry__.build_cuda)
namespace mpcb_rt {
extern std::atomic<long long> g_launches;
extern std::atomic<int> g_opt_tma, g_opt_retile, g_opt_cert, g_opt_dense, g_opt_cta, g_opt_warp_setup, g_opt_retile_min, g_opt_fwd_rhs;
int fail(int code, const std::string& msg);      // records the message for mpcb_last_error(), returns `code`
}
struct ShapeOps;
namespace mpcb_rt { void register_shape_ops(const ShapeOps* ops); }
using namespace mpcb_rt;

#ifndef MPCB_EMU
#include <cuda_runtime.h>
typedef cudaStream_t rt_stream;
#define RT_CHECK(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(MPCB_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));      \
    } while (0)
static int rt_malloc(void** p, size_t n) { RT_CHECK(cudaMalloc(p, n ? n : 1)); return 0; }
static void rt_free(void* p) { if (p) cudaFree(p); }
static int rt_memset(void* p, int v, size_t n, rt_stream s) { RT_CHECK(cudaMemsetAsync(p, v, n, s)); return 0; }
static int rt_h2d(void* d, const void* h, size_t n, rt_stream s) { RT_CHECK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s)); return 0; }
static int rt_d2h(void* h, const void* d, size_t n, rt_stream s) { RT_CHECK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s)); return 0; }
static int rt_sync(rt_stream s) { RT_CHECK(cudaStreamSynchronize(s)); return 0; }
// MPCB_DEBUG_SYNC=1: synchronise after every launch so that a faulting kernel is named in the error
static bool debug_sync() {
    static const bool on = std::getenv("MPCB_DEBUG_SYNC") != nullptr;
    return on;
}
static int rt_launch_check(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && debug_sync()) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return fail(MPCB_E_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    return 0;
}

#ifndef MPCB_QP_THREADS
#define MPCB_QP_THREADS 128     // threads per CTA of the per-QP kernels
#endif
#ifndef MPCB_QP_MINBLOCKS
#define MPCB_QP_MINBLOCKS 2     // resident CTAs per SM the register allocation must allow
#endif
template <typename Op, typename T, typename L>
__global__ void __launch_bounds__(MPCB_QP_THREADS, MPCB_QP_MINBLOCKS) qp_kernel(const KParams<T> p) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < p.B) Op::template run<T, L>(p, b);
}
template <typename Op, typename T, typename L>
static int launch_qp(const KParams<T>& p, rt_stream st) {
    const int threads = MPCB_QP_THREADS;
    qp_kernel<Op, T, L><<<(p.B + threads - 1) / threads, threads, 0, st>>>(p);
    ++g_launches;
    return rt_launch_check(Op::name());
}
template <typename F>
__global__ void __launch_bounds__(128) lambda_kernel(int n, F f) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n) f(b);
}
#define MPCB_LAMBDA [=] __device__
template <typename F>
static int launch_1d(int n, rt_stream st, F f) {
    if (n <= 0) return 0;
    lambda_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, f);
    ++g_launches;
    return rt_launch_check("lambda_kernel");
}
#else   // ---------------------------------------------------------------- MPCB_EMU (tests only)
typedef void* rt_stream;
static int rt_malloc(void** p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? 0 : fail(MPCB_E_ALLOC, "malloc"); }
static void rt_free(void* p) { std::free(p); }
static int rt_memset(void* p, int v, size_t n, rt_stream) { std::memset(p, v, n); return 0; }
static int rt_h2d(void* d, const void* h, size_t n, rt_stream) { std::memcpy(d, h, n); return 0; }
static int rt_d2h(void* h, const void* d, size_t n, rt_stream) { std::memcpy(h, d, n); return 0; }
static int rt_sync(rt_stream) { return 0; }
template <typename Op, typename T, typename L>
static int launch_qp(const KParams<T>& p, rt_stream) {
    for (int b = 0; b < p.B; ++b) Op::template run<T, L>(p, b);
    ++g_launches;
    return 0;
}
#define MPCB_LAMBDA [=]
template <typename F>
static int launch_1d(int n, rt_stream, F f) {
    for (int b = 0; b < n; ++b) f(b);
    ++g_launches;
    return 0;
}
#endif

// =============================================================================================
// solver object
// =============================================================================================
struct mpcb_solver {
    mpcb_problem prob;
    mpcb_settings set;
    int cap = 0, batch = 0;
    size_t ld = 0;
    bool is_setup = false;
    size_t esz = 4;
    // workspace
    void *rec = nullptr, *hdr = nullptr, *yrows = nullptr, *scr = nullptr, *scr_hdr = nullptr;
    void *pri = nullptr, *dua = nullptr, *xbox = nullptr, *xbox_alt = nullptr;   // xbox_alt: the other buffer of an update
    int inf_prob = 0, inf_box = 0;      // an infinite bound among the constructor bounds / the per-stage boxes
    int *iter = nullptr, *status = nullptr, *tile_counter = nullptr;
    // re-tiling of unconverged QPs (see run_admm): survivor lists and a half-size scratch workspace
    int *surv[2] = {nullptr, nullptr}, *n_surv = nullptr, *tile_prog = nullptr;
    int retile_at[2] = {0, 0};  // iteration count at which the previous cold [0] / warm-started [1] solve re-tiled (0: not known yet)
    int retile_backoff[2] = {0, 0};                 // solves to wait before probing an earlier compaction point again
    void *rec2 = nullptr, *hdr2 = nullptr, *yrows2 = nullptr;
    void* mdl2 = nullptr;                           // ... of the re-tiled survivors (scratch workspace)
    void* mdl = nullptr; size_t mdl_bytes = 0;      // tiled copy of a time-varying model (KParams::mdl), filled by setup
    bool rec_minv = false;                          // the records hold Linv' Linv instead of Linv (KParams::minv; CTA-kernel solves)
    bool mdl_dirty = false;                         // the stage references changed (mpcb_update): re-tile before the next solve
    size_t ld2 = 0;
    // borrowed inputs
    const void *Ad = nullptr, *Bd = nullptr, *gd = nullptr, *x_init = nullptr, *Xr = nullptr;
    // staging for the host front door
    void* stage_in = nullptr; size_t stage_in_bytes = 0;
    void* stage_out = nullptr; size_t stage_out_bytes = 0;
    void* soa_in = nullptr; size_t soa_in_bytes = 0;
    size_t ws_bytes = 0;
    int VS = 0, CS = 0, NW = 0, LT = 0, REC = 0, HDR = 0, nvar = 0, ncon = 0;
    int inf_bounds = 0;
    // prob.setup() leaves x = z = y = 0 (osqp.c: osqp_setup -> cold_start): the first ADMM launch after a setup starts
    // cold whatever warm_start says; readers of the iterates before that launch get the zeros written on demand
    // shared-KKT dense path (admm_dense.cuh): 0 = not decided since the last setup / bound update, 1 = the batch shares one
    // KKT matrix and dense_minv holds its inverse, -1 = not applicable
    int dense_state = 0;
    void* dense_minv = nullptr; size_t dense_bytes = 0;
    int* dense_flag = nullptr;
    bool cold_pending = false;
    int dev = 0, dev_max_smem = 0, dev_sms = 0;      // device the workspace lives on and its launch-sizing attributes
};

template <typename T>
static KParams<T> make_params(const mpcb_solver* s) {
    KParams<T> p;
    std::memset(&p, 0, sizeof(p));
    const mpcb_problem& q = s->prob;
    p.N = q.horizon; p.B = s->batch; p.ld = s->ld;
    p.Ad = (const T*)s->Ad; p.Bd = (const T*)s->Bd; p.gd = (const T*)s->gd;
    p.tv = q.time_varying; p.model_bs = q.shared_model ? 0 : 1;
    p.x_init = (const T*)s->x_init; p.Xr = (const T*)s->Xr; p.xr_tv = q.stage_reference;
    for (int i = 0; i < MAXNX; ++i) {
        p.Q[i] = (T)q.Q[i]; p.QN[i] = (T)q.QN[i]; p.W[i] = (T)q.W[i]; p.S[i] = (T)q.S[i];
        p.xmin[i] = (T)clip_infty(q.xmin[i]); p.xmax[i] = (T)clip_infty(q.xmax[i]);     // python interface of OSQP: +-inf -> +-OSQP_INFTY
    }
    for (int i = 0; i < MAXNU; ++i) {
        p.R[i] = (T)q.R[i]; p.umin[i] = (T)clip_infty(q.umin[i]); p.umax[i] = (T)clip_infty(q.umax[i]);
    }
    p.xbox = (const T*)s->xbox;
    p.inf_bounds = s->inf_bounds;
    p.certs = g_opt_cert.load();
    p.fwd_rhs = g_opt_fwd_rhs.load();
    const mpcb_settings& o = s->set;
    p.rho_c = (T)o.rho < (T)kRhoMin ? (T)kRhoMin : ((T)o.rho > (T)kRhoMax ? (T)kRhoMax : (T)o.rho);
    p.rho_eq_c = (T)kRhoEqOverRhoIneq * p.rho_c;
    p.rho = (T)o.rho; p.sigma = (T)o.sigma; p.alpha = (T)o.alpha; p.eps_abs = (T)o.eps_abs; p.eps_rel = (T)o.eps_rel;
    p.eps_pinf = (T)o.eps_prim_inf; p.eps_dinf = (T)o.eps_dual_inf;
    p.max_iter = o.max_iter; p.scaling = o.scaling; p.check_every = o.check_termination; p.warm = o.warm_start;
    p.rec = (T*)s->rec; p.hdr = (T*)s->hdr; p.yrows = (T*)s->yrows; p.scr = (T*)s->scr; p.scr_hdr = (T*)s->scr_hdr;
    p.mdl = (const T*)s->mdl;
    p.minv = s->rec_minv ? 1 : 0;
    p.iter = s->iter; p.status = s->status; p.pri_res = (T*)s->pri; p.dua_res = (T*)s->dua;
    p.it0 = 0; p.it_stop = o.max_iter; p.qp_map = nullptr; p.survivors = s->surv[0]; p.n_survivors = s->n_surv;
    p.chunk_len = o.check_termination; p.tile_prog = s->tile_prog; p.list_survivors = 0;
    return p;
}

// ---- shape dispatch: the (nx, nu, slack) combinations of the reference's formulations
//   lateral (4,1): vanilla / slack;  lateral delta-u (5,1): plain / slack  (vehicle_lateral_mpc_slack_increment.py)
//   kinematic (4,2) and its delta-u form (6,2)   (mpc_kinematics*.py, mpc_incre_kine_func.py)

