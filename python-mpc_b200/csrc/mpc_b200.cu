// mpc_b200 — the C ABI (include/mpc_b200.h) and every kernel that does not depend on the compiled QP shape.
//
// libmpc_b200.so (the product, nvcc, sm_100a) is linked from this file plus one object per compiled (shape, dtype) —
// shape_tu.cu, which instantiates the per-QP kernels, the ADMM kernels and the host-side ADMM loop of shape_ops.cuh
// and exports them as a ShapeOps table.  tests/emu compiles the same sources with g++ and -DMPCB_EMU: kernel launches
// become host loops and the CUDA runtime calls become malloc/memcpy, so that the whole C ABI can be exercised in the
// GPU-less build container.  That build is test infrastructure only; the product loader (python-mpc_b200/_lib.py)
// never looks for it.
#include "shape_ops.cuh"
#include "models.cuh"

// =============================================================================================
// process-wide state
// =============================================================================================
static thread_local std::string g_err;
static int env_int(const char* name, int dflt) { const char* v = std::getenv(name); return v ? std::atoi(v) : dflt; }
namespace mpcb_rt {
std::atomic<long long> g_launches{0};
std::atomic<int> g_opt_tma{std::getenv("MPCB_NO_TMA") ? 0 : 1};
std::atomic<int> g_opt_retile{std::getenv("MPCB_NO_RETILE") ? 0 : 1};
std::atomic<int> g_opt_cert{std::getenv("MPCB_NO_CERT") ? 0 : 1};
std::atomic<int> g_opt_dense{std::getenv("MPCB_NO_DENSE") ? 0 : 1};
std::atomic<int> g_opt_cta{std::getenv("MPCB_NO_CTA") ? 0 : 1};
std::atomic<int> g_opt_warp_setup{std::getenv("MPCB_NO_WARP_SETUP") ? 0 : 1};
std::atomic<int> g_opt_retile_min{env_int("MPCB_RETILE_MIN_BATCH", 4096)};
std::atomic<int> g_opt_fwd_rhs{std::getenv("MPCB_NO_FWD_RHS") ? 0 : 1};
int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
}  // namespace mpcb_rt

// ---- the compiled (nx, nu, slack) shapes of the reference's formulations, each in f32 and f64
//   lateral (4,1): vanilla / slack;  lateral delta-u (5,1): plain / slack  (vehicle_lateral_mpc_slack_increment.py)
//   kinematic (4,2) and its delta-u form (6,2)   (mpc_kinematics*.py, mpc_incre_kine_func.py)
//   dynamic (6,2) and its delta-u form (8,2)     (mpc_dynamics.py)
// The list lives in the build (__graft_entry__.SHAPES): every shape_tu.cu object registers its table when the library
// is loaded.
static const ShapeOps** registry(int* count_out, const ShapeOps* add) {
    static const ShapeOps* table[64];
    static int count = 0;
    if (add && count < 64) table[count++] = add;
    if (count_out) *count_out = count;
    return table;
}
namespace mpcb_rt {
void register_shape_ops(const ShapeOps* ops) { registry(nullptr, ops); }
}
static const ShapeOps* find_ops(int nx, int nu, int slack, int dtype) {
    int n = 0;
    const ShapeOps** t = registry(&n, nullptr);
    for (int i = 0; i < n; ++i)
        if (t[i]->nx == nx && t[i]->nu == nu && (t[i]->slack != 0) == (slack != 0) && t[i]->dtype == dtype) return t[i];
    return nullptr;
}
static const ShapeOps* ops_of(const mpcb_solver* s) {
    return find_ops(s->prob.nx, s->prob.nu, s->prob.slack, s->prob.dtype);
}

// anything this large can scale past the OSQP_INFTY test of set_rho_vec (E is at least MIN_SCALING)
static bool is_big(double v) { return !(std::fabs(v) < kOsqpInfty * kMinScaling * 1e-6); }
static int problem_has_inf_bounds(const mpcb_problem& q) {
    for (int i = 0; i < q.nx; ++i) if (is_big(q.xmin[i]) || is_big(q.xmax[i])) return 1;
    for (int i = 0; i < q.nu; ++i) if (is_big(q.umin[i]) || is_big(q.umax[i])) return 1;
    return 0;
}

static bool shape_supported(int nx, int nu, int slack) { return find_ops(nx, nu, slack, MPCB_F64) != nullptr; }

// All mpcb_* functions below are declared extern "C" by include/mpc_b200.h.

const char* mpcb_last_error(void) { return g_err.c_str(); }
int mpcb_version(void) { return 100; }
long long mpcb_launch_count(void) { return g_launches.load(); }

int mpcb_set_option(const char* name, int value) {
    if (!name) return fail(MPCB_E_ARG, "null option name");
    const std::string n(name);
    if (n == "tma") g_opt_tma = value != 0;
    else if (n == "retile") g_opt_retile = value != 0;
    else if (n == "certificates") g_opt_cert = value != 0;
    else if (n == "dense") g_opt_dense = value != 0;
    else if (n == "warp_setup") g_opt_warp_setup = value != 0;
    else if (n == "cta") g_opt_cta = value < 0 ? 0 : (value > 2 ? 2 : value);
    else if (n == "retile_min_batch") g_opt_retile_min = value;
    else if (n == "fwd_rhs") g_opt_fwd_rhs = value != 0;
    else return fail(MPCB_E_ARG, "unknown option: " + n);
    return 0;
}

void mpcb_default_settings(mpcb_settings* s) {
    s->rho = 0.1; s->sigma = 1e-6; s->alpha = 1.6; s->eps_abs = 1e-3; s->eps_rel = 1e-3;
    s->eps_prim_inf = 1e-4; s->eps_dual_inf = 1e-4; s->max_iter = 4000; s->scaling = 10;
    s->check_termination = 25; s->warm_start = 1;
}

static int check_settings(const mpcb_settings* o) {
    if (!(o->rho > 0) || !(o->sigma > 0) || !(o->alpha > 0 && o->alpha < 2) || o->max_iter <= 0 ||
        o->scaling < 0 || o->check_termination < 0 || o->eps_abs < 0 || o->eps_rel < 0 ||
        (o->eps_abs == 0 && o->eps_rel == 0))
        return fail(MPCB_E_ARG, "invalid settings (rho, sigma > 0; 0 < alpha < 2; max_iter > 0; eps >= 0, not both 0)");
    return 0;
}

int mpcb_create(const mpcb_problem* prob, const mpcb_settings* settings, int capacity, mpcb_solver** out) {
    if (!prob || !out || capacity <= 0) return fail(MPCB_E_ARG, "null problem / non-positive capacity");
    if (prob->horizon < 1) return fail(MPCB_E_ARG, "horizon must be >= 1");
    if (prob->dtype != MPCB_F32 && prob->dtype != MPCB_F64) return fail(MPCB_E_ARG, "dtype must be MPCB_F32 or MPCB_F64");
    if (!shape_supported(prob->nx, prob->nu, prob->slack))
        return fail(MPCB_E_ARG, "unsupported (nx, nu, slack) combination");
    for (int i = 0; i < prob->nx; ++i)
        if (prob->xmin[i] > prob->xmax[i]) return fail(MPCB_E_ARG, "lower bound must be lower than or equal to upper bound");
    for (int i = 0; i < prob->nu; ++i)
        if (prob->umin[i] > prob->umax[i]) return fail(MPCB_E_ARG, "lower bound must be lower than or equal to upper bound");
    mpcb_settings def;
    mpcb_default_settings(&def);
    if (!settings) settings = &def;
    if (int rc = check_settings(settings)) return rc;
    mpcb_solver* s = new (std::nothrow) mpcb_solver();
    if (!s) return fail(MPCB_E_ALLOC, "out of host memory");
    s->prob = *prob; s->set = *settings; s->cap = capacity;
#ifndef MPCB_EMU
    if (cudaGetDevice(&s->dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&s->dev_max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, s->dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&s->dev_sms, cudaDevAttrMultiProcessorCount, s->dev) != cudaSuccess) {
        const std::string msg = std::string("cuda device query: ") + cudaGetErrorString(cudaGetLastError());
        delete s;
        return fail(MPCB_E_CUDA, msg);
    }
#endif
    s->inf_prob = problem_has_inf_bounds(*prob);
    s->inf_bounds = s->inf_prob;
    s->esz = prob->dtype == MPCB_F32 ? 4 : 8;
    const int N = prob->horizon, nx = prob->nx, nu = prob->nu, ns = prob->slack ? nx : 0;
    s->VS = nx + ns + nu; s->CS = 2 * nx + nu; s->NW = nx + nu; s->LT = s->NW * (s->NW + 1) / 2;
    s->REC = 2 * s->VS + 2 * s->CS + s->LT + s->NW; s->HDR = 3 * nx + 1;
    s->nvar = (N + 1) * nx + N * nu + (N + 1) * ns; s->ncon = 2 * (N + 1) * nx + N * nu;
    s->ld = ((size_t)capacity + 31) / 32 * 32;
    const size_t ld = s->ld, e = s->esz, S1 = (size_t)(N + 1);
    struct { void** p; size_t n; } allocs[] = {
        {&s->rec, S1 * s->REC * ld * e}, {&s->hdr, (size_t)s->HDR * ld * e}, {&s->yrows, S1 * s->CS * ld * e},
        {&s->scr, S1 * (s->VS + s->CS) * ld * e}, {&s->scr_hdr, (size_t)nx * ld * e}, {&s->pri, ld * e},
        {&s->dua, ld * e}, {(void**)&s->iter, ld * sizeof(int)}, {(void**)&s->status, ld * sizeof(int)},
        {(void**)&s->tile_counter, 64}, {(void**)&s->surv[0], ld * sizeof(int)}, {(void**)&s->surv[1], ld * sizeof(int)},
        {(void**)&s->n_surv, 64}, {(void**)&s->tile_prog, (ld / 32 + 1) * sizeof(int)}};
    for (auto& a : allocs) {
        if (int rc = rt_malloc(a.p, a.n)) { mpcb_destroy(s); return rc; }
        s->ws_bytes += a.n;
    }
    rt_memset(s->rec, 0, S1 * s->REC * ld * e, 0);
    rt_memset(s->hdr, 0, (size_t)s->HDR * ld * e, 0);
    rt_memset(s->yrows, 0, S1 * s->CS * ld * e, 0);
    rt_memset(s->status, 0, ld * sizeof(int), 0);
    rt_sync(0);
    *out = s;
    return 0;
}

void mpcb_destroy(mpcb_solver* s) {
    if (!s) return;
    void* ptrs[] = {s->rec, s->hdr, s->yrows, s->scr, s->scr_hdr, s->pri, s->dua, s->iter, s->status, s->tile_counter,
                    s->surv[0], s->surv[1], s->n_surv, s->tile_prog, s->rec2, s->hdr2, s->yrows2,
                    s->xbox, s->xbox_alt, s->stage_in, s->stage_out, s->soa_in, s->dense_minv, s->dense_flag, s->mdl, s->mdl2};
    for (void* p : ptrs) rt_free(p);
    delete s;
}

int mpcb_set_settings(mpcb_solver* s, const mpcb_settings* o) {
    if (!s || !o) return fail(MPCB_E_ARG, "null argument");
    if (int rc = check_settings(o)) return rc;
    const bool refactor = o->rho != s->set.rho || o->sigma != s->set.sigma || o->scaling != s->set.scaling;
    if (o->check_termination != s->set.check_termination || o->max_iter != s->set.max_iter || refactor)
        s->retile_at[0] = s->retile_at[1] = 0;      // the learnt re-tiling points are multiples of the old check interval
    s->set = *o;
    if (refactor) s->is_setup = false;    // like osqp_update_rho: the cached factorisation is stale
    return 0;
}

// validate per-stage state boxes [(N+1)][2][nx] and upload them (clipped to +-OSQP_INFTY) into *dst
static int upload_stage_boxes(mpcb_solver* s, const double* xbox_host, void** dst, int* has_inf, rt_stream st) {
    const size_t n = (size_t)(s->prob.horizon + 1) * 2 * s->prob.nx;
    for (int k = 0; k <= s->prob.horizon; ++k)
        for (int i = 0; i < s->prob.nx; ++i)
            if (xbox_host[(k * 2) * s->prob.nx + i] > xbox_host[(k * 2 + 1) * s->prob.nx + i])
                return fail(MPCB_E_ARG, "lower bound must be lower than or equal to upper bound");
    *has_inf = 0;
    for (size_t i = 0; i < n; ++i) if (is_big(xbox_host[i])) *has_inf = 1;
    if (!*dst) if (int r = rt_malloc(dst, n * s->esz)) return r;
    void* tmp = std::malloc(n * s->esz);
    if (!tmp) return fail(MPCB_E_ALLOC, "out of host memory");
    for (size_t i = 0; i < n; ++i) {
        if (s->esz == 4) ((float*)tmp)[i] = (float)clip_infty(xbox_host[i]);
        else ((double*)tmp)[i] = clip_infty(xbox_host[i]);
    }
    int r = rt_h2d(*dst, tmp, n * s->esz, st);
    if (!r) r = rt_sync(st);
    std::free(tmp);
    return r;
}

int mpcb_set_stage_bounds(mpcb_solver* s, const double* xbox_host) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!xbox_host) {
        rt_sync(0);
        rt_free(s->xbox); s->xbox = nullptr; s->inf_box = 0;
    } else {
        int has_inf = 0;
        if (int r = upload_stage_boxes(s, xbox_host, &s->xbox, &has_inf, 0)) return r;
        s->inf_box = has_inf;
    }
    s->inf_bounds = s->inf_prob | s->inf_box;
    s->is_setup = false;      // problem data of the next prob.setup(); after a setup use mpcb_update_bounds
    return 0;
}

size_t mpcb_workspace_bytes(const mpcb_solver* s) { return s ? s->ws_bytes : 0; }
int mpcb_num_variables(const mpcb_solver* s) { return s ? s->nvar : 0; }
int mpcb_num_constraints(const mpcb_solver* s) { return s ? s->ncon : 0; }

int mpcb_setup(mpcb_solver* s, int batch, size_t ld, const void* Ad, const void* Bd, const void* gd,
               const void* x_init, const void* Xr, void* stream) {
    if (!s || !Ad || !Bd || !x_init || !Xr) return fail(MPCB_E_ARG, "null argument");
    if (batch <= 0 || batch > s->cap) return fail(MPCB_E_ARG, "batch must be in [1, capacity]");
    if (ld != s->ld) return fail(MPCB_E_ARG, "ld must equal the solver's leading dimension (capacity rounded up to 32)");
    s->batch = batch; s->Ad = Ad; s->Bd = Bd; s->gd = gd; s->x_init = x_init; s->Xr = Xr;
    int rc = ops_of(s)->setup(s, (rt_stream)stream);
    if (rc) return rc;
    s->is_setup = true;
    s->dense_state = 0;
    s->cold_pending = true;      // osqp_setup leaves x = z = y = 0: nothing of an earlier problem may warm-start this one
    return 0;
}

int mpcb_update(mpcb_solver* s, const void* x_init, const void* Xr) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->is_setup) return fail(MPCB_E_STATE, "update before setup");
    if (x_init) s->x_init = x_init;
    if (Xr) { s->Xr = Xr; s->mdl_dirty = true; }
    return 0;
}

int mpcb_update_bounds(mpcb_solver* s, const double* xmin, const double* xmax, const double* umin, const double* umax,
                       const double* xbox_host, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    rt_stream st = (rt_stream)stream;
    mpcb_problem np = s->prob;
    for (int i = 0; i < np.nx; ++i) { if (xmin) np.xmin[i] = xmin[i]; if (xmax) np.xmax[i] = xmax[i]; }
    for (int i = 0; i < np.nu; ++i) { if (umin) np.umin[i] = umin[i]; if (umax) np.umax[i] = umax[i]; }
    for (int i = 0; i < np.nx; ++i)
        if (np.xmin[i] > np.xmax[i]) return fail(MPCB_E_ARG, "lower bound must be lower than or equal to upper bound");
    for (int i = 0; i < np.nu; ++i)
        if (np.umin[i] > np.umax[i]) return fail(MPCB_E_ARG, "lower bound must be lower than or equal to upper bound");
    if (!s->is_setup) {           // before prob.setup(): plain problem data
        if (xbox_host) if (int r = mpcb_set_stage_bounds(s, xbox_host)) return r;
        s->prob = np;
        s->inf_prob = problem_has_inf_bounds(np);
        s->inf_bounds = s->inf_prob | s->inf_box;
        return 0;
    }
    void* new_box = s->xbox;
    int new_inf_box = s->inf_box;
    if (xbox_host) {
        if (int r = upload_stage_boxes(s, xbox_host, &s->xbox_alt, &new_inf_box, st)) return r;
        new_box = s->xbox_alt;
    }
    int rc = ops_of(s)->refactor(s, &np, new_box, st);
    if (rc) return rc;
    s->dense_state = 0;           // the factor may have changed: the shared inverse is rebuilt on demand
    s->prob = np;
    if (xbox_host) { s->xbox_alt = s->xbox; s->xbox = new_box; s->inf_box = new_inf_box; }
    s->inf_prob = problem_has_inf_bounds(np);
    s->inf_bounds = s->inf_prob | s->inf_box;
    return 0;
}

static int run_admm(mpcb_solver* s, int max_iter, int check_every, int warm, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->is_setup) return fail(MPCB_E_STATE, "solve before setup (or settings changed since setup)");
    return ops_of(s)->run_admm(s, max_iter, check_every, warm, (rt_stream)stream);
}

int mpcb_solve(mpcb_solver* s, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    return run_admm(s, s->set.max_iter, s->set.check_termination, s->set.warm_start, stream);
}

int mpcb_iterate(mpcb_solver* s, int iters, void* stream) {
    if (iters <= 0) return fail(MPCB_E_ARG, "iters must be positive");
    return run_admm(s, iters, 0, 1, stream);
}

int mpcb_cold_start(mpcb_solver* s, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->is_setup) return fail(MPCB_E_STATE, "cold_start before setup");
    s->cold_pending = false;
    return ops_of(s)->cold_start(s, (rt_stream)stream);
}

// ---- gather: scaled iterates of the tiled workspace -> unscaled batch-major outputs in reference order
template <typename T>
static int gather_impl(mpcb_solver* s, void* x_out, void* y_out, void* u_out, rt_stream st) {
    const int N = s->prob.horizon, nx = s->prob.nx, nu = s->prob.nu, ns = s->prob.slack ? nx : 0;
    const int VS = s->VS, CS = s->CS, REC = s->REC, nvar = s->nvar, ncon = s->ncon, B = s->batch;
    // record layout (Lay, mpc_common.h): [ D | E | Linv | t | p | x ], variables s | x | u inside D and x
    const int R_D = 0, R_E = VS, R_X = VS + CS + s->LT + s->NW + CS, H_E0 = 0, H_Y0 = 2 * nx, H_C = 3 * nx, HDR = s->HDR;
    const size_t S1 = (size_t)(N + 1);
    const T* rec = (const T*)s->rec; const T* hdr = (const T*)s->hdr; const T* yr = (const T*)s->yrows;
    // a QP that ended with an infeasibility certificate has no solution: NaN like OSQP's results (osqp.c: store_solution)
    const int* stt = s->status;
    const T nanv = (T)NAN;
#define MPCB_NO_SOLUTION(b) (stt[b] == kPrimalInfeasible || stt[b] == kDualInfeasible || \
                             stt[b] == kPrimalInfeasibleInaccurate || stt[b] == kDualInfeasibleInaccurate)
    if (x_out || u_out) {
        T* xo = (T*)x_out; T* uo = (T*)u_out;
        const int per = (N + 1) * VS;
        // one thread per (QP, internal element); consecutive threads walk the elements of one QP so
        // the batch-major writes are contiguous
        int rc = launch_1d(B * per, st, MPCB_LAMBDA(int idx) {
            const int b = idx / per, e = idx - b * per;
            const int k = e / VS, o = e - k * VS;
            const T* R = rec + (((size_t)(b >> 5) * S1 + k) * REC) * TILE + (b & 31);
            const T v = MPCB_NO_SOLUTION(b) ? nanv : R[(size_t)(R_D + o) * TILE] * R[(size_t)(R_X + o) * TILE];
            if (o < ns) { if (xo) xo[(size_t)b * nvar + (N + 1) * nx + N * nu + k * nx + o] = v; }
            else if (o < ns + nx) { if (xo) xo[(size_t)b * nvar + k * nx + (o - ns)] = v; }
            else if (k < N) {
                const int j = o - nx - ns;
                if (xo) xo[(size_t)b * nvar + (N + 1) * nx + k * nu + j] = v;
                if (uo) uo[(size_t)b * N * nu + k * nu + j] = v;
            }
        });
        if (rc) return rc;
    }
    if (y_out) {
        T* yo = (T*)y_out;
        const int per = nx + (N + 1) * CS;
        int rc = launch_1d(B * per, st, MPCB_LAMBDA(int idx) {
            const int b = idx / per, e = idx - b * per;
            const size_t tile = (size_t)(b >> 5), lane = (size_t)(b & 31);
            const T* H = hdr + tile * HDR * TILE + lane;
            const T cinv = MPCB_NO_SOLUTION(b) ? nanv : (T)1 / H[(size_t)H_C * TILE];
            if (e < nx) {                                  // rows dyn_0 live in the header
                yo[(size_t)b * ncon + e] = H[(size_t)(H_E0 + e) * TILE] * H[(size_t)(H_Y0 + e) * TILE] * cinv;
                return;
            }
            const int k = (e - nx) / CS, o = (e - nx) - k * CS;
            const T v = rec[((tile * S1 + k) * REC + R_E + o) * TILE + lane] * yr[((tile * S1 + k) * CS + o) * TILE + lane] * cinv;
            if (o < nx) { if (k < N) yo[(size_t)b * ncon + (k + 1) * nx + o] = v; }            // dyn_{k+1}
            else if (o < 2 * nx) yo[(size_t)b * ncon + (N + 1) * nx + k * nx + (o - nx)] = v;     // bx_k
            else if (k < N) yo[(size_t)b * ncon + 2 * (N + 1) * nx + k * nu + (o - 2 * nx)] = v; // bu_k
        });
        if (rc) return rc;
    }
#undef MPCB_NO_SOLUTION
    return 0;
}

int mpcb_get_solution(mpcb_solver* s, void* x_out, void* y_out, void* u_out, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->is_setup) return fail(MPCB_E_STATE, "get_solution before setup");
    rt_stream st = (rt_stream)stream;
    if (s->cold_pending) if (int r = mpcb_cold_start(s, stream)) return r;      // set up, not solved yet: the zeros of osqp_setup
    return s->esz == 4 ? gather_impl<float>(s, x_out, y_out, u_out, st) : gather_impl<double>(s, x_out, y_out, u_out, st);
}

int mpcb_get_info(mpcb_solver* s, int* iter_out, int* status_out, void* pri_out, void* dua_out, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    rt_stream st = (rt_stream)stream;
    const int B = s->batch;
    const int* it = s->iter; const int* stt = s->status;
    if (iter_out || status_out) {
        int rc = launch_1d(B, st, MPCB_LAMBDA(int b) {
            if (iter_out) iter_out[b] = it[b];
            if (status_out) status_out[b] = stt[b];
        });
        if (rc) return rc;
    }
    if (pri_out || dua_out) {
        const size_t e = s->esz;
        const char* pr = (const char*)s->pri; const char* du = (const char*)s->dua;
        char* po = (char*)pri_out; char* dq = (char*)dua_out;
        int rc = launch_1d(B, st, MPCB_LAMBDA(int b) {
            for (size_t i = 0; i < e; ++i) {
                if (po) po[b * e + i] = pr[b * e + i];
                if (dq) dq[b * e + i] = du[b * e + i];
            }
        });
        if (rc) return rc;
    }
    return 0;
}

// ---- layout helpers ---------------------------------------------------------------------------
template <typename T>
static int to_em(int B, int elems, size_t ld, const T* src, T* dst, rt_stream st) {
    // thread per (element, QP) with the QP index fastest: coalesced element-major writes
    return launch_1d(B * elems, st, MPCB_LAMBDA(int idx) {
        const int e = idx / B, b = idx - e * B;
        dst[(size_t)e * ld + b] = src[(size_t)b * elems + e];
    });
}
template <typename T>
static int to_bm(int B, int elems, size_t ld, const T* src, T* dst, rt_stream st) {
    return launch_1d(B * elems, st, MPCB_LAMBDA(int idx) {
        const int b = idx / elems, e = idx - b * elems;
        dst[(size_t)b * elems + e] = src[(size_t)e * ld + b];
    });
}

int mpcb_to_element_major(int dtype, int batch, int elems, size_t ld, const void* src, void* dst, void* stream) {
    if (!src || !dst || batch <= 0 || elems <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad layout arguments");
    rt_stream st = (rt_stream)stream;
    return dtype == MPCB_F32 ? to_em<float>(batch, elems, ld, (const float*)src, (float*)dst, st)
                             : to_em<double>(batch, elems, ld, (const double*)src, (double*)dst, st);
}
int mpcb_to_batch_major(int dtype, int batch, int elems, size_t ld, const void* src, void* dst, void* stream) {
    if (!src || !dst || batch <= 0 || elems <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad layout arguments");
    rt_stream st = (rt_stream)stream;
    return dtype == MPCB_F32 ? to_bm<float>(batch, elems, ld, (const float*)src, (float*)dst, st)
                             : to_bm<double>(batch, elems, ld, (const double*)src, (double*)dst, st);
}

// ---- model kernels ----------------------------------------------------------------------------
int mpcb_lateral_discretize(int dtype, int batch, size_t ld, const void* speed, const double* q, void* Ad, void* Bd,
                            void* stream) {
    if (!speed || !q || !Ad || !Bd || batch <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        LateralParams<float> lp{(float)q[0], (float)q[1], (float)q[2], (float)q[3], (float)q[4], (float)q[5], (float)q[6]};
        const float* sp = (const float*)speed; float* A = (float*)Ad; float* Bm = (float*)Bd;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { lateral_one<float>(lp, sp, A, Bm, ld, b); });
    }
    LateralParams<double> lp{q[0], q[1], q[2], q[3], q[4], q[5], q[6]};
    const double* sp = (const double*)speed; double* A = (double*)Ad; double* Bm = (double*)Bd;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { lateral_one<double>(lp, sp, A, Bm, ld, b); });
}

int mpcb_dynamics_linearize(int dtype, int batch, size_t ld, const void* x, const void* u, const double* q, void* Ad,
                            void* Bd, void* gd, void* stream) {
    if (!x || !u || !q || !Ad || !Bd || !gd || batch <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        DynParams<float> dp{(float)q[0], (float)q[1], (float)q[2], (float)q[3], (float)q[4], (float)q[5], (float)q[6], (float)q[7]};
        const float* xx = (const float*)x; const float* uu = (const float*)u;
        float* A = (float*)Ad; float* Bm = (float*)Bd; float* g = (float*)gd;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { dynamics_one<float>(dp, xx, uu, A, Bm, g, ld, b); });
    }
    DynParams<double> dp{q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7]};
    const double* xx = (const double*)x; const double* uu = (const double*)u;
    double* A = (double*)Ad; double* Bm = (double*)Bd; double* g = (double*)gd;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { dynamics_one<double>(dp, xx, uu, A, Bm, g, ld, b); });
}

int mpcb_kinematics_linearize(int dtype, int batch, size_t ld, const void* x, const void* u, const double* q, void* Ad,
                              void* Bd, void* gd, void* stream) {
    if (!x || !u || !q || !Ad || !Bd || !gd || batch <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        const float wb = (float)q[0], dt = (float)q[1];
        const float* xx = (const float*)x; const float* uu = (const float*)u;
        float* A = (float*)Ad; float* Bm = (float*)Bd; float* g = (float*)gd;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { kinematics_one<float>(wb, dt, xx, uu, A, Bm, g, ld, b); });
    }
    const double wb = q[0], dt = q[1];
    const double* xx = (const double*)x; const double* uu = (const double*)u;
    double* A = (double*)Ad; double* Bm = (double*)Bd; double* g = (double*)gd;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { kinematics_one<double>(wb, dt, xx, uu, A, Bm, g, ld, b); });
}

int mpcb_dynamics_step(int dtype, int batch, size_t ld, const void* x, const void* u, const double* q, void* x_next,
                       void* alpha, void* stream) {
    if (!x || !u || !q || !x_next || batch <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        DynParams<float> dp{(float)q[0], (float)q[1], (float)q[2], (float)q[3], (float)q[4], (float)q[5], (float)q[6], (float)q[7]};
        const float* xx = (const float*)x; const float* uu = (const float*)u;
        float* xn = (float*)x_next; float* al = (float*)alpha;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { dynamics_step_one<float>(dp, xx, uu, xn, al, ld, b); });
    }
    DynParams<double> dp{q[0], q[1], q[2], q[3], q[4], q[5], q[6], q[7]};
    const double* xx = (const double*)x; const double* uu = (const double*)u;
    double* xn = (double*)x_next; double* al = (double*)alpha;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { dynamics_step_one<double>(dp, xx, uu, xn, al, ld, b); });
}

int mpcb_kinematics_step(int dtype, int batch, size_t ld, const void* x, const void* u, const double* q, void* x_next,
                         void* stream) {
    if (!x || !u || !q || !x_next || batch <= 0 || ld < (size_t)batch) return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        const float wb = (float)q[0], dt = (float)q[1];
        const float* xx = (const float*)x; const float* uu = (const float*)u; float* xn = (float*)x_next;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { kinematics_step_one<float>(wb, dt, xx, uu, xn, ld, b); });
    }
    const double wb = q[0], dt = q[1];
    const double* xx = (const double*)x; const double* uu = (const double*)u; double* xn = (double*)x_next;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { kinematics_step_one<double>(wb, dt, xx, uu, xn, ld, b); });
}

int mpcb_augment_increment(int dtype, int batch, size_t ld, int nx, int nu, int stages, const void* Ad, const void* Bd,
                           const void* gd, void* At, void* Bt, void* gt, void* stream) {
    if (!Ad || !Bd || !At || !Bt || batch <= 0 || nx <= 0 || nu <= 0 || stages <= 0 || ld < (size_t)batch)
        return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32) {
        const float* A = (const float*)Ad; const float* Bm = (const float*)Bd; const float* g = (const float*)gd;
        float* A2 = (float*)At; float* B2 = (float*)Bt; float* g2 = (float*)gt;
        return launch_1d(batch, st, MPCB_LAMBDA(int b) { augment_one<float>(nx, nu, stages, A, Bm, g, A2, B2, g2, ld, b); });
    }
    const double* A = (const double*)Ad; const double* Bm = (const double*)Bd; const double* g = (const double*)gd;
    double* A2 = (double*)At; double* B2 = (double*)Bt; double* g2 = (double*)gt;
    return launch_1d(batch, st, MPCB_LAMBDA(int b) { augment_one<double>(nx, nu, stages, A, Bm, g, A2, B2, g2, ld, b); });
}

template <typename T>
static int plant_impl(int B, size_t ld, int nx, int nu, int shared, const T* A, const T* Bm, const T* g, const T* x,
                      const T* u, int us, T* xn, rt_stream st) {
    return launch_1d(B, st, MPCB_LAMBDA(int b) {
        const size_t mld = shared ? 1 : ld, bo = shared ? 0 : (size_t)b;
        T xo[MAXNX], acc[MAXNX];
        for (int j = 0; j < nx; ++j) xo[j] = x[(size_t)j * ld + b];
        for (int i = 0; i < nx; ++i) {
            T v = g ? g[(size_t)i * mld + bo] : (T)0;
            for (int j = 0; j < nx; ++j) v += A[(size_t)(i * nx + j) * mld + bo] * xo[j];
            for (int j = 0; j < nu; ++j) v += Bm[(size_t)(i * nu + j) * mld + bo] * u[(size_t)b * us + j];
            acc[i] = v;
        }
        for (int i = 0; i < nx; ++i) xn[(size_t)i * ld + b] = acc[i];
    });
}

int mpcb_plant_step(int dtype, int batch, size_t ld, int nx, int nu, int shared_model, const void* A, const void* Bm,
                    const void* g, const void* x, const void* u, int u_stride, void* x_next, void* stream) {
    if (!A || !Bm || !x || !u || !x_next || batch <= 0 || nx <= 0 || nx > MAXNX || nu <= 0 || nu > MAXNU ||
        ld < (size_t)batch || u_stride < nu)
        return fail(MPCB_E_ARG, "bad arguments");
    rt_stream st = (rt_stream)stream;
    if (dtype == MPCB_F32)
        return plant_impl<float>(batch, ld, nx, nu, shared_model, (const float*)A, (const float*)Bm, (const float*)g,
                                 (const float*)x, (const float*)u, u_stride, (float*)x_next, st);
    return plant_impl<double>(batch, ld, nx, nu, shared_model, (const double*)A, (const double*)Bm, (const double*)g,
                              (const double*)x, (const double*)u, u_stride, (double*)x_next, st);
}

// ---- explicit QP --------------------------------------------------------------------------------
int mpcb_qp_pattern(const mpcb_solver* s, int* Ap, int* Ai) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    const int N = s->prob.horizon, nx = s->prob.nx, nu = s->prob.nu, ns = s->prob.slack ? nx : 0;
    const int bx0 = (N + 1) * nx, bu0 = 2 * (N + 1) * nx;
    int nnz = 0, col = 0;
    for (int k = 0; k <= N; ++k)
        for (int j = 0; j < nx; ++j) {
            if (Ap) Ap[col] = nnz;
            if (Ai) Ai[nnz] = k * nx + j;
            ++nnz;
            if (k < N)
                for (int i = 0; i < nx; ++i) { if (Ai) Ai[nnz] = (k + 1) * nx + i; ++nnz; }
            if (Ai) Ai[nnz] = bx0 + k * nx + j;
            ++nnz; ++col;
        }
    for (int k = 0; k < N; ++k)
        for (int j = 0; j < nu; ++j) {
            if (Ap) Ap[col] = nnz;
            for (int i = 0; i < nx; ++i) { if (Ai) Ai[nnz] = (k + 1) * nx + i; ++nnz; }
            if (Ai) Ai[nnz] = bu0 + k * nu + j;
            ++nnz; ++col;
        }
    for (int k = 0; k <= N && ns; ++k)
        for (int j = 0; j < nx; ++j) {
            if (Ap) Ap[col] = nnz;
            if (Ai) Ai[nnz] = bx0 + k * nx + j;
            ++nnz; ++col;
        }
    if (Ap) Ap[col] = nnz;
    return nnz;
}

int mpcb_build_qp(mpcb_solver* s, void* Pdiag, void* q, void* Avals, void* l, void* u, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->Ad || !s->x_init) return fail(MPCB_E_STATE, "build_qp before setup");
    rt_stream st = (rt_stream)stream;
    BuildOut o{Pdiag, q, Avals, l, u};
    return ops_of(s)->build_qp(s, &o, st);
}

int mpcb_get_scaling(mpcb_solver* s, void* D_out, void* E_out, void* c_out, void* stream) {
    if (!s) return fail(MPCB_E_ARG, "null solver");
    if (!s->is_setup) return fail(MPCB_E_STATE, "get_scaling before setup (or settings changed since setup)");
    ScalingOut o{D_out, E_out, c_out};
    return ops_of(s)->get_scaling(s, &o, (rt_stream)stream);
}

// ---- host front door ----------------------------------------------------------------------------
static int ensure(void** p, size_t* have, size_t need) {
    if (*have >= need) return 0;
    rt_free(*p); *p = nullptr; *have = 0;
    if (rt_malloc(p, need)) return MPCB_E_ALLOC;
    *have = need;
    return 0;
}

int mpcb_solve_host(mpcb_solver* s, int batch, const void* Ad, const void* Bd, const void* gd, const void* x_init,
                    const void* Xr, void* x_out, void* u_out, int* iter_out, int* status_out) {
    if (!s || !Ad || !Bd || !x_init || !Xr) return fail(MPCB_E_ARG, "null argument");
    if (batch <= 0 || batch > s->cap) return fail(MPCB_E_ARG, "batch must be in [1, capacity]");
    const mpcb_problem& q = s->prob;
    const int N = q.horizon, nx = q.nx, nu = q.nu;
    const size_t e = s->esz, ld = s->ld;
    const int stages = q.time_varying ? N : 1;
    const int nA = stages * nx * nx, nB = stages * nx * nu, nG = gd ? stages * nx : 0, nX0 = nx,
              nXr = (q.stage_reference ? N + 1 : 1) * nx;
    const int mb = q.shared_model ? 1 : batch;                // model rows on the host side
    const size_t model_elems = (size_t)nA + nB + nG;
    const size_t in_bytes = (model_elems * mb + (size_t)(nX0 + nXr) * batch) * e;
    const size_t mld = q.shared_model ? 1 : ld;
    const size_t soa_bytes = (model_elems * mld + (size_t)(nX0 + nXr) * ld) * e;
    const size_t out_elems = (size_t)(x_out ? s->nvar : 0) + (u_out ? N * nu : 0);
    const size_t out_bytes = out_elems * batch * e + 2 * (size_t)batch * sizeof(int);
    if (ensure(&s->stage_in, &s->stage_in_bytes, in_bytes) || ensure(&s->soa_in, &s->soa_in_bytes, soa_bytes) ||
        ensure(&s->stage_out, &s->stage_out_bytes, out_bytes))
        return MPCB_E_ALLOC;
    rt_stream st = 0;
    char* din = (char*)s->stage_in;
    char* soa = (char*)s->soa_in;
    struct Part { const void* h; int elems; int rows; size_t pld; const void** dev; };
    const void *dA = nullptr, *dB = nullptr, *dG = nullptr, *dX0 = nullptr, *dXr = nullptr;
    Part parts[] = {{Ad, nA, mb, mld, &dA}, {Bd, nB, mb, mld, &dB}, {gd, nG, mb, mld, &dG},
                    {x_init, nX0, batch, ld, &dX0}, {Xr, nXr, batch, ld, &dXr}};
    for (auto& pt : parts) {
        if (!pt.h || pt.elems == 0) continue;
        const size_t nbytes = (size_t)pt.elems * pt.rows * e;
        if (int r = rt_h2d(din, pt.h, nbytes, st)) return r;
        if (pt.rows == 1 && pt.pld == 1) {
            *pt.dev = din;                                  // a single row is already element-major
        } else {
            if (int r = mpcb_to_element_major(q.dtype, pt.rows, pt.elems, pt.pld, din, soa, st)) return r;
            *pt.dev = soa;
            soa += (size_t)pt.elems * pt.pld * e;
        }
        din += nbytes;
    }
    if (int r = mpcb_setup(s, batch, ld, dA, dB, dG, dX0, dXr, st)) return r;
    if (int r = run_admm(s, s->set.max_iter, s->set.check_termination, 0, st)) return r;
    char* dout = (char*)s->stage_out;
    void* dx = nullptr; void* du = nullptr;
    if (x_out) { dx = dout; dout += (size_t)s->nvar * batch * e; }
    if (u_out) { du = dout; dout += (size_t)N * nu * batch * e; }
    int* dit = (int*)dout; int* dst = dit + batch;
    if (int r = mpcb_get_solution(s, dx, nullptr, du, st)) return r;
    if (int r = mpcb_get_info(s, dit, dst, nullptr, nullptr, st)) return r;
    if (x_out) if (int r = rt_d2h(x_out, dx, (size_t)s->nvar * batch * e, st)) return r;
    if (u_out) if (int r = rt_d2h(u_out, du, (size_t)N * nu * batch * e, st)) return r;
    if (iter_out) if (int r = rt_d2h(iter_out, dit, (size_t)batch * sizeof(int), st)) return r;
    if (status_out) if (int r = rt_d2h(status_out, dst, (size_t)batch * sizeof(int), st)) return r;
    return rt_sync(st);
}

