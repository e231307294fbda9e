// C-ABI of libwfcrl_b200.so (see include/wfcrl_b200.h).  Host-side only: owns device state, stages inputs and launches
// the kernels of wf_kernels.cu / wf_fast.cu.  No torch types, no exceptions across the boundary, no CPU fallback.
#include "../../include/wfcrl_b200.h"
#include "wf_device.cuh"
#include "wf_host_const.h"
#include "wf_fast_baked.inc"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

// Relative half-width of the FP32 kernel's guard band around the 0.05 m/s overlap threshold (DESIGN.md section 3).
static constexpr float kDefaultAmbEps = 2e-5f;

static thread_local std::string g_err;
static int set_err(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                              \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess)                                                                      \
            return set_err(WF_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
    } while (0)

struct WfHandle_t {
    WfConfig cfg;
    WfModel model;
    WfFastConst fast;
    WfFastConst64 fast64;
    bool fast_baked = false;  // model constants equal the compile-time baked ones -> specialised kernel
    WfState st;
    int device = 0;
    int sm_count = 0, sm_clock_khz = 0;
    size_t es = 8;  // element size of "real"
    std::vector<void*> allocs;
    // staging for wf_reset (host ids -> dense device arrays)
    uint8_t* d_mask = nullptr;
    double *d_rws = nullptr, *d_rwd = nullptr, *d_rcs = nullptr;
    uint8_t* h_mask = nullptr;
    double *h_rws = nullptr, *h_rwd = nullptr, *h_rcs = nullptr;
    // staging for wf_step_host
    float* d_action = nullptr;
    double* d_yaw_cmd = nullptr;
    WfStepOut d_out = {};
    static constexpr int kHostStreams = 6;
    cudaStream_t host_streams[kHostStreams] = {};  // one per chunk of the wf_step_host pipeline
    uint64_t launches = 0;
    // ordering of the host-buffer entry points (which run on the handle's own streams) after asynchronous calls the caller
    // queued on ITS stream: those record this event, wf_step_host / wf_update_command_host make their streams wait on it
    cudaEvent_t ev_async = nullptr;
    bool ev_pending = false;
    // staged host path of a strict FP32 handle: compact records of the re-solved envs (device + pinned host), chunk events
    float *d_fix_rec = nullptr, *h_fix_rec = nullptr;
    int* h_fix_n = nullptr;
    int fix_rec_cap = 0;
    cudaEvent_t ev_chunk[kHostStreams] = {};
    bool vtab_stale = false;  // some env's vortex-table rows do not match its geometry: launch the kernels that ignore the table
    // wf_set_kernel_timing: events around the step-kernel launch and the re-solve launch of the last step call
    bool timing = false, timing_pending = false;
    cudaEvent_t ev_t[3] = {};
    double t_step_ms = 0.0, t_fix_ms = 0.0;
    int t_calls = 0;
    uint64_t steps_since_wind_update = 1u << 30;  // wf_update_wind rebuilds the vortex table only when it is not called every step
    double* d_pool = nullptr;  // the layout pool in one allocation: [L][T] x, [L][T] y, [L][2] centres, [L] int32 turbine
                               // counts (WfModel.layout_*)
    std::vector<int> layout_n;  // host copy of the pool's turbine counts
    // wf_evaluate_yaw / wf_evaluate_actions scratch, sized for the largest B*K either has evaluated so far: the evaluation fix
    // list [eval_cap] and its 4 counters in one allocation, on a gathering FP64 handle one (v, w) scratch row per candidate
    // [eval_cap][9T], on a strict FP32 handle one transitioned-yaw row per candidate [eval_cap][T]
    int eval_cap = 0;
    int* d_eval_fix = nullptr;
    double2* d_eval_vwg = nullptr;
    double* d_eval_yaw = nullptr;
};

template <typename T> static int dev_alloc(WfHandle_t* h, T** p, size_t n) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, n * sizeof(T));
    if (e != cudaSuccess) return set_err(WF_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    e = cudaMemset(q, 0, n * sizeof(T));
    if (e != cudaSuccess) return set_err(WF_ERR_CUDA, std::string("cudaMemset: ") + cudaGetErrorString(e));
    h->allocs.push_back(q);
    *p = (T*)q;
    return WF_OK;
}
#define TRY(expr)                 \
    do {                          \
        int _r = (expr);          \
        if (_r != WF_OK) return _r; \
    } while (0)

// A row of the tables below: a pointer member of WfStepOut or WfState, named by its byte offset (the members differ in
// type), and the array it points to: element size (0 = "real") and extent, n elements per env (kB), per env and turbine
// (kBT) or in all (kAll).
enum Extent { kB, kBT, kAll };
struct Array {
    const char* name;  // of an exported state array (wf_get_state / wf_set_state), else NULL
    size_t off, elem;
    int n;
    Extent ext;
    size_t elems(size_t B, size_t T) const { return n * (ext == kBT ? B * T : ext == kB ? B : 1); }
    size_t bytes(size_t B, size_t T, size_t es) const { return elems(B, T) * (elem ? elem : es); }
};
static void* ptr_at(const void* s, const Array& a) { void* p; memcpy(&p, (const char*)s + a.off, sizeof p); return p; }
static void set_ptr_at(void* s, const Array& a, void* p) { memcpy((char*)s + a.off, &p, sizeof p); }

// The eight step outputs in WfStepOut field order.  A strict FP32 handle's compact record (wf_fixup64_kernel) holds the
// env id, then the per-env outputs, then the per-turbine outputs, each part in this order.
static constexpr Array kOut[] = {
    {nullptr, offsetof(WfStepOut, yaw), 0, 1, kBT}, {nullptr, offsetof(WfStepOut, wind_speed), 0, 1, kBT},
    {nullptr, offsetof(WfStepOut, wind_direction), 0, 1, kBT}, {nullptr, offsetof(WfStepOut, power), 0, 1, kBT},
    {nullptr, offsetof(WfStepOut, load), 0, 4, kBT}, {nullptr, offsetof(WfStepOut, reward), 0, 1, kB},
    {nullptr, offsetof(WfStepOut, freewind), 0, 2, kB}, {nullptr, offsetof(WfStepOut, truncated), 1, 1, kB}};
static constexpr int out_elems(Extent ext) { int n = 0; for (const Array& f : kOut) n += f.ext == ext ? f.n : 0; return n; }
static_assert(WF_FIX_REC_HDR == 1 + out_elems(kB), "a fix-up record starts with the env id and the per-env outputs");

// The state arrays wf_create always allocates.  Names and byte sizes are part of the ABI.
#define MEMBER(m) offsetof(WfState, m), sizeof(*WfState::m)
static constexpr Array kState[] = {
    {"yaw", MEMBER(yaw), 1, kBT}, {"acc", MEMBER(acc), 1, kBT}, {"acc_prev", MEMBER(acc_prev), 1, kBT},
    {"num_iter", MEMBER(num_iter), 1, kB}, {"num_moves", MEMBER(num_moves), 1, kB}, {"nonfinite", MEMBER(nonfinite), 1, kB},
    {"episode", MEMBER(episode), 1, kB}, {"ambiguous", MEMBER(amb), 1, kB}, {"ep_return", MEMBER(ep_return), 1, kB},
    {"ep_len", MEMBER(ep_len), 1, kB}, {"fin_sum", MEMBER(fin_sum), 1, kB}, {"fin_sumsq", MEMBER(fin_sumsq), 1, kB},
    {"fin_n", MEMBER(fin_n), 1, kB}, {"fin_len", MEMBER(fin_len), 1, kB}, {nullptr, MEMBER(reset_mask), 1, kB},
    {nullptr, MEMBER(fix_list), 1, kB}, {nullptr, MEMBER(fix_count), 4, kAll}, {"ws", MEMBER(ws), 1, kB},
    {"wd", MEMBER(wd), 1, kB}, {"ws_norm", MEMBER(ws_norm), 1, kB}, {"shaper_ref", MEMBER(shaper_ref), 1, kB},
    {"ti_ambient", MEMBER(ti_amb), 1, kB}, {"xs", MEMBER(xs), 1, kBT}, {"ys", MEMBER(ys), 1, kBT}, {"xi", MEMBER(xi), 1, kBT},
    {"yi", MEMBER(yi), 1, kBT}, {"order", MEMBER(order), 1, kBT}, {"cs", MEMBER(cs), 2, kB}, {nullptr, MEMBER(xhl), 1, kBT},
    {nullptr, MEMBER(yhl), 1, kBT}, {nullptr, MEMBER(idx), 1, kBT}, {nullptr, MEMBER(tab_lo), 1, kBT},
    {nullptr, MEMBER(tab_glo), 1, kBT}, {"layout_id", MEMBER(layout_id), 1, kB}, {"turbine_count", MEMBER(turbine_count), 1, kB}};
#undef MEMBER

// called at the end of every asynchronous entry point: later host-buffer calls must run after the work queued here
static int mark_async(WfHandle h, cudaStream_t st) {
    CUDA_TRY(cudaEventRecord(h->ev_async, st));
    h->ev_pending = true;
    return WF_OK;
}

// rotated + sorted geometry of the selected envs and, unless told otherwise, their vortex-table rows
static cudaError_t launch_geometry(WfHandle h, const uint8_t* d_mask, const double* d_cs, cudaStream_t st,
                                   bool build_table = true, bool autoreset_draw = false) {
    cudaError_t e = wf_launch_geometry(h->model, h->st, d_mask, d_cs, st, autoreset_draw);
    h->launches += 1;
    if (e == cudaSuccess && build_table && h->st.vtab_ok) {
        e = wf_launch_vortex_table(h->model, h->fast64, h->st, d_mask, st);
        h->launches += 1;
        if (!d_mask) h->vtab_stale = false;
    } else if (h->st.vtab_ok) {
        h->vtab_stale = true;
    }
    return e;
}

static int check_layouts(size_t n, const double* lx, const double* ly) {
    for (size_t k = 0; k < n; ++k)
        if (!isfinite(lx[k]) || !isfinite(ly[k])) return set_err(WF_ERR_INVALID, "layout coordinates must be finite");
    return WF_OK;
}

// Replace the layout pool by L validated host layouts [L][T] of counts[l] turbines each and store the centre of each one's
// bounding box (over its own turbines), the point the geometry kernel rotates it about.  Entries at or beyond a layout's
// count are stored as 0.  The caller makes sure that no queued kernel still reads the old pool.
static int set_pool(WfHandle h, int L, const int* counts, const double* lx, const double* ly) {
    const size_t T = h->model.T, LT = (size_t)L * T;
    std::vector<double> pool(LT * 2 + (size_t)L * 2 + ((size_t)L + 1) / 2);  // + the int32 counts
    for (int l = 0; l < L; ++l) {
        const int n = counts[l];
        const double *x = lx + l * T, *y = ly + l * T;
        memcpy(pool.data() + l * T, x, sizeof(double) * n);
        memcpy(pool.data() + LT + l * T, y, sizeof(double) * n);
        double xmin = x[0], xmax = x[0], ymin = y[0], ymax = y[0];
        for (int t = 1; t < n; ++t) {
            xmin = fmin(xmin, x[t]); xmax = fmax(xmax, x[t]);
            ymin = fmin(ymin, y[t]); ymax = fmax(ymax, y[t]);
        }
        pool[2 * LT + 2 * l] = (xmin + xmax) / 2;
        pool[2 * LT + 2 * l + 1] = (ymin + ymax) / 2;
    }
    memcpy(pool.data() + 2 * LT + 2 * L, counts, sizeof(int) * L);  // layout_counts(): behind the centres
    double* d = nullptr;
    cudaError_t e = cudaMalloc(&d, sizeof(double) * pool.size());
    if (e != cudaSuccess) return set_err(WF_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    e = cudaMemcpy(d, pool.data(), sizeof(double) * pool.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(d);
        return set_err(WF_ERR_CUDA, std::string("cudaMemcpy: ") + cudaGetErrorString(e));
    }
    if (h->d_pool) cudaFree(h->d_pool);
    h->d_pool = d;
    h->layout_n.assign(counts, counts + L);
    WfModel& m = h->model;
    m.layout_x = d; m.layout_y = d + LT; m.layout_c = d + 2 * LT; m.n_layouts = L;
    return WF_OK;
}

// Rebuild the geometry (and table rows) of the masked envs from their current layout ids, rotated by the cos/sin each env
// already uses, so that host-computed cos/sin (wf_reset with h_cos / h_sin) are kept.
static cudaError_t rebuild_geometry(WfHandle h, const uint8_t* d_mask, cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(h->d_rcs, h->st.cs, sizeof(double) * 2 * h->model.B, cudaMemcpyDeviceToDevice, st);
    return e != cudaSuccess ? e : launch_geometry(h, d_mask, h->d_rcs, st);
}

extern "C" {

const char* wf_last_error(void) { return g_err.c_str(); }
#ifndef WF_SOURCE_HASH
#define WF_SOURCE_HASH "unknown-source-hash"
#endif
// "wfcrl_b200 <version> (sm_100a) wfcrl_b200-src-sha256:<first 16 hex digits>": the hash covers csrc/*.cu|cuh|h and include/*.h
// (wfcrl_b200/build.py: source_hash) -- build() rebuilds when it differs from the tree, smoke() asserts that it matches.
const char* wf_version(void) { return "wfcrl_b200 0.2 (sm_100a) wfcrl_b200-src-sha256:" WF_SOURCE_HASH; }

int wf_default_config(WfConfig* c) {
    if (!c) return set_err(WF_ERR_INVALID, "cfg is NULL");
    wf_fill_default_config(c);
    return WF_OK;
}

int wf_destroy(WfHandle h) {
    if (!h) return WF_OK;
    cudaSetDevice(h->device);
    for (void* p : h->allocs) cudaFree(p);
    if (h->d_pool) cudaFree(h->d_pool);
    if (h->h_mask) cudaFreeHost(h->h_mask);
    if (h->h_rws) cudaFreeHost(h->h_rws);
    if (h->h_rwd) cudaFreeHost(h->h_rwd);
    if (h->h_rcs) cudaFreeHost(h->h_rcs);
    for (cudaStream_t st : h->host_streams)
        if (st) cudaStreamDestroy(st);
    if (h->ev_async) cudaEventDestroy(h->ev_async);
    for (cudaEvent_t ev : h->ev_t)
        if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : h->ev_chunk)
        if (ev) cudaEventDestroy(ev);
    if (h->h_fix_rec) cudaFreeHost(h->h_fix_rec);
    if (h->h_fix_n) cudaFreeHost(h->h_fix_n);
    if (h->d_eval_fix) cudaFree(h->d_eval_fix);
    if (h->d_eval_vwg) cudaFree(h->d_eval_vwg);
    if (h->d_eval_yaw) cudaFree(h->d_eval_yaw);
    delete h;
    return WF_OK;
}

int wf_create(const WfConfig* cfg, const double* lx, const double* ly, WfHandle* out) {
    if (!cfg || !lx || !ly || !out) return set_err(WF_ERR_INVALID, "NULL argument");
    const int T = cfg->num_turbines, B = cfg->num_envs;
    if (T < 1 || T > WF_MAX_TURBINES) return set_err(WF_ERR_INVALID, "num_turbines must be in [1, 128]");
    if (B < 1) return set_err(WF_ERR_INVALID, "num_envs must be >= 1");
    if (cfg->table_len < 2 || cfg->table_len > WF_TABLE_MAX) return set_err(WF_ERR_INVALID, "bad table_len");
    if (cfg->wind_veer != 0.0) return set_err(WF_ERR_INVALID, "wind_veer != 0 is not supported (case.yaml:39 uses 0)");
    if (!(cfg->yaw_lo < cfg->yaw_hi)) return set_err(WF_ERR_INVALID, "yaw bounds: need low < high (mdp.py:196)");
    if (cfg->precision != WF_PREC_F64 && cfg->precision != WF_PREC_F32) return set_err(WF_ERR_INVALID, "bad precision");
    if (cfg->turbine_grid_points != 0 && cfg->turbine_grid_points != 3 && cfg->turbine_grid_points != 5)
        return set_err(WF_ERR_INVALID, "turbine_grid_points must be 3 (case.yaml:16) or 5");
    if (cfg->turbine_grid_points == 5 && cfg->kernel != WF_KERNEL_BASIC)
        return set_err(WF_ERR_INVALID, "turbine_grid_points = 5 needs WF_KERNEL_BASIC (the tuned kernels are built for the 3x3 grid)");
    if (cfg->kernel != WF_KERNEL_BASIC && cfg->kernel != WF_KERNEL_FAST) return set_err(WF_ERR_INVALID, "bad kernel");
    if (!(cfg->rotor_diameter > 0.0) || !(cfg->hub_height > cfg->rotor_diameter / 2) || !(cfg->dt > 0.0) ||
        !(cfg->actuator_rate > 0.0) || !(cfg->turbulence_intensity > 0.0) || !(cfg->air_density > 0.0))
        return set_err(WF_ERR_INVALID, "rotor_diameter, dt, actuator_rate, turbulence_intensity, air_density must be "
                                       "positive and hub_height > rotor_diameter / 2");
    for (int i = 0; i < cfg->table_len; ++i)
        if (!isfinite(cfg->table_ws[i]) || !isfinite(cfg->table_cp[i]) || !isfinite(cfg->table_ct[i]) ||
            (i > 0 && !(cfg->table_ws[i] > cfg->table_ws[i - 1])))
            return set_err(WF_ERR_INVALID, "turbine table: wind speeds must be finite and strictly increasing");
    TRY(check_layouts(T, lx, ly));
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_err(WF_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return set_err(WF_ERR_INVALID, "bad device ordinal");
    CUDA_TRY(cudaSetDevice(cfg->device));
    CUDA_TRY(wf_configure_fast_kernels());
    CUDA_TRY(wf_configure_fast64_kernels());

    WfHandle_t* h = new WfHandle_t();
    h->cfg = *cfg;
    h->device = cfg->device;
    h->es = cfg->precision == WF_PREC_F64 ? 8 : 4;
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, cfg->device);
    if (e != cudaSuccess) { delete h; return set_err(WF_ERR_CUDA, cudaGetErrorString(e)); }
    h->sm_count = prop.multiProcessorCount;
    h->sm_clock_khz = prop.clockRate;

    WfModel& m = h->model;
    memset(&m, 0, sizeof(m));
    m.T = T; m.B = B;
    m.max_iter = cfg->max_iter; m.continuous = cfg->continuous_control; m.multi_agent = cfg->multi_agent;
    m.shaper = cfg->reward_shaper; m.table_len = cfg->table_len;
    m.G = cfg->turbine_grid_points ? cfg->turbine_grid_points : 3;
    m.yaw_lo_f = (float)cfg->yaw_lo; m.yaw_hi_f = (float)cfg->yaw_hi; m.yaw_step_f = (float)cfg->yaw_step;
    m.rate_f = (float)cfg->actuator_rate; m.dt_f = (float)cfg->dt;
    m.amb_eps = getenv("WFCRL_B200_AMB_EPS") ? (float)atof(getenv("WFCRL_B200_AMB_EPS")) : kDefaultAmbEps;
    if (cfg->fp32_relaxed) m.amb_eps = 0.f;  // no guard band, no FP64 re-solve: raw FP32 results
    m.load_coef = cfg->load_coef; m.shaper_reference = cfg->shaper_reference;
    m.rho = cfg->air_density; m.ref_rho = cfg->ref_density_cp_ct; m.shear = cfg->wind_shear;
    m.D = cfg->rotor_diameter; m.HH = cfg->hub_height; m.TSR = cfg->tsr; m.pP = cfg->pP;
    m.alpha = cfg->alpha; m.beta = cfg->beta; m.ka = cfg->ka; m.kb = cfg->kb; m.ad = cfg->ad; m.bd = cfg->bd;
    m.dm = cfg->dm;
    m.ch_const = cfg->ch_constant; m.ch_ai = cfg->ch_ai; m.ch_init = cfg->ch_initial; m.ch_down = cfg->ch_downstream;
    m.e3_112 = 3 * exp(1.0 / 12.0); m.e3_13 = 3 * exp(1.0 / 3.0);
    build_fast_const(*cfg, &h->fast);
    build_fast_const(*cfg, &h->fast64);
    h->fast_baked = wf_baked_matches(h->fast) && !getenv("WFCRL_B200_NO_BAKED");  // env var: force the generic kernel (tests)

    int rc = WF_OK;
    auto fail = [&](int r) { wf_destroy(h); return r; };
    double *d_ws, *d_ct, *d_pw;
    if ((rc = dev_alloc(h, &d_ws, cfg->table_len))) return fail(rc);
    if ((rc = dev_alloc(h, &d_ct, cfg->table_len))) return fail(rc);
    if ((rc = dev_alloc(h, &d_pw, cfg->table_len))) return fail(rc);
    if ((rc = set_pool(h, 1, &T, lx, ly))) return fail(rc);  // a pool of one layout; every env has layout id 0
    {
        std::vector<double> pw(cfg->table_len);
        const double area = 3.141592653589793 * pow(cfg->rotor_diameter / 2.0, 2.0);
        for (int i = 0; i < cfg->table_len; ++i)  // FLORIS Turbine.__attrs_post_init__: power / density at the nodes
            pw[i] = 0.5 * area * cfg->table_cp[i] * cfg->generator_efficiency * pow(cfg->table_ws[i], 3.0);
        cudaMemcpy(d_ws, cfg->table_ws, sizeof(double) * cfg->table_len, cudaMemcpyHostToDevice);
        cudaMemcpy(d_ct, cfg->table_ct, sizeof(double) * cfg->table_len, cudaMemcpyHostToDevice);
        cudaMemcpy(d_pw, pw.data(), sizeof(double) * cfg->table_len, cudaMemcpyHostToDevice);
    }
    m.tab_ws = d_ws; m.tab_ct = d_ct; m.tab_pw = d_pw;

    WfState& s = h->st;
    const size_t BT = (size_t)B * T;
    for (const Array& a : kState) {
        char* p;
        if ((rc = dev_alloc(h, &p, a.bytes(B, T, h->es)))) return fail(rc);
        set_ptr_at(&s, a, p);
    }
    if ((rc = dev_alloc(h, &h->d_mask, (size_t)B)) || (rc = dev_alloc(h, &h->d_rws, (size_t)B)) ||
        (rc = dev_alloc(h, &h->d_rwd, (size_t)B)) || (rc = dev_alloc(h, &h->d_rcs, (size_t)2 * B)))
        return fail(rc);
    // The vortex table trades the V sweep's arithmetic for one streamed read of 36 reals per turbine pair.  Measured on B200
    // (profiles/r2_vortex_table.md): it pays in the FP64 kernels (whose sweep is 3x more expensive), but not in the FP32 kernel,
    // where the instructions that remain are latency-bound and the direct evaluation wins by 6 % -- so the FP32 step kernel
    // never reads it.  A strict FP32 handle builds DOUBLE rows for its FP64 re-solve kernel, which reads those of the few
    // flagged envs (float rows would cost it 1e-9 of the rotor speed, too much at the foot of the power curve).
    // WFCRL_B200_NO_VTAB=1 disables every table; tables that would not fit comfortably are skipped and the kernels evaluate
    // every pair directly.
    if (cfg->kernel == WF_KERNEL_FAST && T >= 2 && !getenv("WFCRL_B200_NO_VTAB")) {
        const size_t rows_all = (size_t)B * ((size_t)T * (T - 1) / 2) * 36;
        const size_t cap = (size_t)(getenv("WFCRL_B200_VTAB_MAX_MB") ? atof(getenv("WFCRL_B200_VTAB_MAX_MB")) : 24576.0) << 20;
        auto try_alloc = [&](size_t bytes) -> void* {
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            if (bytes > cap || bytes > free_b / 2) return nullptr;
            void* p = nullptr;
            if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
            h->allocs.push_back(p);
            return p;
        };
        if (cfg->precision == WF_PREC_F64) {
            // the FP64 step kernel gathers: target-major rows + the (v, w) scratch, both or neither (then it runs the scatter
            // form with direct evaluation)
            s.vtab = (double*)try_alloc(rows_all * 8);
            if (s.vtab) s.vwg = (double2*)try_alloc(BT * 9 * sizeof(double2));
            if (s.vtab && !s.vwg) {
                cudaFree(s.vtab);
                h->allocs.pop_back();
                s.vtab = nullptr;
            }
            m.vtab_tmajor = s.vtab != nullptr;
        } else if (m.amb_eps > 0.f) {
            s.vtab = (double*)try_alloc(rows_all * 8);
        }
        if (s.vtab)
            if ((rc = dev_alloc(h, &s.vtab_ok, (size_t)B))) return fail(rc);
    }
    if (cudaMallocHost((void**)&h->h_mask, B) != cudaSuccess || cudaMallocHost((void**)&h->h_rws, sizeof(double) * B) != cudaSuccess ||
        cudaMallocHost((void**)&h->h_rwd, sizeof(double) * B) != cudaSuccess ||
        cudaMallocHost((void**)&h->h_rcs, sizeof(double) * 2 * B) != cudaSuccess)
        return fail(set_err(WF_ERR_NOMEM, "cudaMallocHost failed"));
    for (cudaStream_t& st : h->host_streams)
        if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess)
            return fail(set_err(WF_ERR_CUDA, "cudaStreamCreate failed"));
    if (cudaEventCreateWithFlags(&h->ev_async, cudaEventDisableTiming) != cudaSuccess)
        return fail(set_err(WF_ERR_CUDA, "cudaEventCreate failed"));

    // initial condition: wind (8, 270) as in FlorisCase.simul_params (data_cases.py:99-100), ambient TI from the config
    {
        std::vector<double> ws(B, 8.0), wd(B, 270.0), ti(B, cfg->turbulence_intensity);
        cudaMemcpy(h->d_rws, ws.data(), sizeof(double) * B, cudaMemcpyHostToDevice);
        cudaMemcpy(h->d_rwd, wd.data(), sizeof(double) * B, cudaMemcpyHostToDevice);
        cudaMemcpy(s.ti_amb, ti.data(), sizeof(double) * B, cudaMemcpyHostToDevice);
        cudaError_t e1 = wf_launch_reset_state(m, s, nullptr, h->d_rws, h->d_rwd, 0);
        cudaError_t e2 = launch_geometry(h, nullptr, nullptr, 0);
        h->launches += 1;
        cudaError_t e3 = cudaDeviceSynchronize();
        if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)
            return fail(set_err(WF_ERR_CUDA, std::string("init kernels failed: ") +
                                                 cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3))));
    }
    *out = h;
    return WF_OK;
}

static bool is_strict_f32(WfHandle h) {
    return h->cfg.kernel == WF_KERNEL_FAST && h->cfg.precision == WF_PREC_F32 && h->model.amb_eps > 0.f;
}

// FP64 re-solve of the envs flagged by the FP32 launches issued since the previous fix-up (all of them must precede this launch
// in stream order); d_rec / rec_cap: optional compact copies of the re-solved envs' results (host path)
static int launch_fixup(WfHandle h, int mode, const WfStepOut& out, cudaStream_t st, float* d_rec = nullptr, int rec_cap = 0) {
    cudaError_t e = wf_launch_fixup64(mode, !h->vtab_stale, h->model, h->fast64, h->st, out, h->model.B, d_rec, rec_cap, st);
    h->launches += 1;
    if (e != cudaSuccess) return set_err(WF_ERR_CUDA, std::string("fix-up kernel launch: ") + cudaGetErrorString(e));
    return WF_OK;
}

// kernel timing (wf_set_kernel_timing): fold the previous call's events into the averages
static void timing_collect(WfHandle h) {
    if (!h->timing_pending) return;
    h->timing_pending = false;
    float a = 0.f, b = 0.f;
    if (cudaEventSynchronize(h->ev_t[2]) != cudaSuccess || cudaEventElapsedTime(&a, h->ev_t[0], h->ev_t[1]) != cudaSuccess ||
        cudaEventElapsedTime(&b, h->ev_t[1], h->ev_t[2]) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    h->t_step_ms += a;
    h->t_fix_ms += b;
    h->t_calls += 1;
}

// out == NULL: no outputs are written
static int launch_step(WfHandle h, int mode, const uint8_t* d_mask, const float* d_action, const double* d_yaw,
                       const WfStepOut* outp, cudaStream_t st, int env_begin = 0, int env_count = -1,
                       bool defer_fixup = false) {
    const WfStepOut out = outp ? *outp : WfStepOut{};
    if (env_count < 0) env_count = h->model.B;
    const bool timed = h->timing && !defer_fixup && env_begin == 0 && env_count == h->model.B;
    if (timed) {
        timing_collect(h);
        cudaEventRecord(h->ev_t[0], st);
    }
    struct TimingTail {  // records the closing events on every return path
        WfHandle h; cudaStream_t st; bool on, mid = false;
        ~TimingTail() {
            if (!on) return;
            if (!mid) cudaEventRecord(h->ev_t[1], st);
            cudaEventRecord(h->ev_t[2], st);
            h->timing_pending = true;
        }
    } tail{h, st, timed};
    cudaError_t e;
    if (h->cfg.kernel == WF_KERNEL_FAST && h->cfg.precision == WF_PREC_F64)
        e = wf_launch_step_fast64(mode, !h->vtab_stale, h->model, h->fast64, h->st, d_mask, d_action, d_yaw, out, env_begin, env_count, st);
    else if (h->cfg.kernel == WF_KERNEL_FAST)
    {
        e = wf_launch_step_fast(mode, h->fast_baked, h->model, h->fast, h->st, d_mask, d_action, d_yaw, out, env_begin, env_count,
                                st);
        if (e == cudaSuccess && is_strict_f32(h) && !defer_fixup) {  // strict FP32: FP64 re-solve of whatever the launch flagged
            if (timed) { cudaEventRecord(h->ev_t[1], st); tail.mid = true; }
            h->launches += 1;
            h->steps_since_wind_update += 1;
            return launch_fixup(h, mode, out, st);
        }
    }
    else
        e = wf_launch_step_basic(h->cfg.precision, mode, h->model, h->st, d_mask, d_action, d_yaw, out, env_begin,
                                 env_count, st);
    h->launches += 1;
    h->steps_since_wind_update += 1;
    if (e != cudaSuccess) return set_err(WF_ERR_CUDA, std::string("step kernel launch: ") + cudaGetErrorString(e));
    return WF_OK;
}

int wf_reset_masked(WfHandle h, const uint8_t* d_mask, const double* d_ws, const double* d_wd, int32_t warmup,
                    const WfStepOut* out, void* stream) {
    if (!h || !d_ws || !d_wd) return set_err(WF_ERR_INVALID, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(wf_launch_reset_state(h->model, h->st, d_mask, d_ws, d_wd, st));
    CUDA_TRY(launch_geometry(h, d_mask, nullptr, st));
    h->launches += 1;
    for (int k = 0; k < warmup; ++k) TRY(launch_step(h, WF_MODE_WARMUP, d_mask, nullptr, nullptr, out, st));
    return mark_async(h, st);
}

int wf_reset_sampled(WfHandle h, const uint8_t* d_mask, uint64_t seed, int64_t env_id_offset, double ti_lo, double ti_hi,
                     int32_t warmup, const WfStepOut* out, void* stream) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    if (env_id_offset < 0) return set_err(WF_ERR_INVALID, "env_id_offset must be >= 0");
    if (ti_hi > ti_lo && !(ti_lo > 0.0)) return set_err(WF_ERR_INVALID, "turbulence-intensity range must be positive");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(wf_launch_sample_reset(h->model, h->st, d_mask, seed, env_id_offset, ti_lo, ti_hi, h->d_rws, h->d_rwd, st));
    h->launches += 1;
    return wf_reset_masked(h, d_mask, h->d_rws, h->d_rwd, warmup, out, stream);
}

int wf_reset(WfHandle h, const int32_t* ids, int32_t n, const double* ws, const double* wd, const double* hc,
             const double* hs, int32_t warmup, const WfStepOut* out, void* stream) {
    if (!h || !ws || !wd) return set_err(WF_ERR_INVALID, "NULL argument");
    if ((hc == nullptr) != (hs == nullptr)) return set_err(WF_ERR_INVALID, "h_cos and h_sin must be given together");
    const int B = h->model.B;
    if (n < 0 || n > B) return set_err(WF_ERR_INVALID, "bad n");
    if (!ids && n != B) return set_err(WF_ERR_INVALID, "h_env_ids == NULL requires n == num_envs");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    memset(h->h_mask, 0, B);
    for (int k = 0; k < n; ++k) {
        const int b = ids ? ids[k] : k;
        if (b < 0 || b >= B) return set_err(WF_ERR_INVALID, "env id out of range");
        h->h_mask[b] = 1;
        h->h_rws[b] = ws[k];
        h->h_rwd[b] = wd[k];
        if (hc) { h->h_rcs[2 * b] = hc[k]; h->h_rcs[2 * b + 1] = hs[k]; }
    }
    CUDA_TRY(cudaMemcpyAsync(h->d_mask, h->h_mask, B, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->d_rws, h->h_rws, sizeof(double) * B, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->d_rwd, h->h_rwd, sizeof(double) * B, cudaMemcpyHostToDevice, st));
    if (hc) CUDA_TRY(cudaMemcpyAsync(h->d_rcs, h->h_rcs, sizeof(double) * 2 * B, cudaMemcpyHostToDevice, st));
    CUDA_TRY(wf_launch_reset_state(h->model, h->st, h->d_mask, h->d_rws, h->d_rwd, st));
    CUDA_TRY(launch_geometry(h, h->d_mask, hc ? h->d_rcs : nullptr, st));
    h->launches += 1;
    for (int k = 0; k < warmup; ++k)
        TRY(launch_step(h, WF_MODE_WARMUP, h->d_mask, nullptr, nullptr, out, st));
    CUDA_TRY(cudaStreamSynchronize(st));  // the handle-owned pinned staging is reusable when this call returns
    return WF_OK;
}

int wf_set_layouts(WfHandle h, int32_t n_layouts, const double* lx, const double* ly) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL argument");
    if (n_layouts < 1) return set_err(WF_ERR_INVALID, "n_layouts must be >= 1");
    const std::vector<int32_t> counts(n_layouts, h->model.T);
    return wf_set_layouts_sized(h, n_layouts, counts.data(), lx, ly);
}

int wf_set_layouts_sized(WfHandle h, int32_t n_layouts, const int32_t* counts, const double* lx, const double* ly) {
    if (!h || !counts || !lx || !ly) return set_err(WF_ERR_INVALID, "NULL argument");
    if (n_layouts < 1) return set_err(WF_ERR_INVALID, "n_layouts must be >= 1");
    const int T = h->model.T;
    for (int l = 0; l < n_layouts; ++l) {
        if (counts[l] < 1 || counts[l] > T)
            return set_err(WF_ERR_INVALID, "layout " + std::to_string(l) + ": turbine count " + std::to_string(counts[l]) +
                                               " is outside [1, num_turbines = " + std::to_string(T) + "]");
        if (counts[l] < T && (h->cfg.kernel == WF_KERNEL_BASIC || h->model.multi_agent))
            return set_err(WF_ERR_INVALID, "layouts with fewer turbines than the handle (padding) are not supported on "
                                           "WF_KERNEL_BASIC or multi_agent handles: every count must equal num_turbines");
        TRY(check_layouts((size_t)counts[l], lx + (size_t)l * T, ly + (size_t)l * T));
    }
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaDeviceSynchronize());  // after every earlier asynchronous call: no queued kernel reads the old pool any more
    TRY(set_pool(h, n_layouts, counts, lx, ly));
    CUDA_TRY(cudaMemset(h->st.layout_id, 0, sizeof(int) * h->model.B));
    CUDA_TRY(rebuild_geometry(h, nullptr, 0));
    CUDA_TRY(cudaDeviceSynchronize());
    return WF_OK;
}

int wf_assign_layouts(WfHandle h, const int32_t* ids, int32_t n, const int32_t* layout_ids, void* stream) {
    if (!h || !layout_ids) return set_err(WF_ERR_INVALID, "NULL argument");
    const int B = h->model.B, L = h->model.n_layouts;
    if (n < 0 || n > B) return set_err(WF_ERR_INVALID, "bad n");
    if (!ids && n != B) return set_err(WF_ERR_INVALID, "h_env_ids == NULL requires n == num_envs");
    for (int k = 0; k < n; ++k) {
        if (ids && (ids[k] < 0 || ids[k] >= B)) return set_err(WF_ERR_INVALID, "env id out of range");
        if (layout_ids[k] < 0 || layout_ids[k] >= L)
            return set_err(WF_ERR_INVALID, "layout id out of range [0, n_layouts)");
    }
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    // read-modify-write of the id array: the envs not listed keep theirs
    std::vector<int32_t> lid(B);
    CUDA_TRY(cudaMemcpyAsync(lid.data(), h->st.layout_id, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memset(h->h_mask, 0, B);
    for (int k = 0; k < n; ++k) {
        const int b = ids ? ids[k] : k;
        lid[b] = layout_ids[k];
        h->h_mask[b] = 1;
    }
    CUDA_TRY(cudaMemcpyAsync(h->st.layout_id, lid.data(), sizeof(int32_t) * B, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->d_mask, h->h_mask, B, cudaMemcpyHostToDevice, st));
    CUDA_TRY(rebuild_geometry(h, h->d_mask, st));
    CUDA_TRY(cudaStreamSynchronize(st));  // the host staging is reusable when this call returns
    return WF_OK;
}

int wf_set_layout_sampling(WfHandle h, int32_t enabled) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    h->model.sample_layouts = enabled ? 1 : 0;
    return WF_OK;
}

int wf_set_autoreset(WfHandle h, int32_t enabled, uint64_t seed, int64_t env_id_offset, double ti_lo, double ti_hi) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    if (enabled && h->cfg.kernel != WF_KERNEL_FAST)
        return set_err(WF_ERR_INVALID, "in-kernel auto-reset needs the warp-per-env kernels (WF_KERNEL_FAST)");
    if (env_id_offset < 0) return set_err(WF_ERR_INVALID, "env_id_offset must be >= 0");
    if (ti_hi > ti_lo && !(ti_lo > 0.0)) return set_err(WF_ERR_INVALID, "turbulence-intensity range must be positive");
    WfModel& m = h->model;
    m.autoreset = enabled ? 1 : 0;
    m.ar_seed = seed; m.ar_offset = env_id_offset; m.ar_ti_lo = ti_lo; m.ar_ti_hi = ti_hi;
    return WF_OK;
}

int wf_autoreset_finish(WfHandle h, int32_t warmup, const WfStepOut* out, void* stream) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t* mask = h->st.reset_mask;
    CUDA_TRY(launch_geometry(h, mask, nullptr, st, true, /*autoreset_draw=*/true));
    for (int k = 0; k < warmup; ++k) TRY(launch_step(h, WF_MODE_WARMUP, mask, nullptr, nullptr, out, st));
    CUDA_TRY(cudaMemsetAsync(h->st.reset_mask, 0, (size_t)h->model.B, st));
    return mark_async(h, st);
}

int wf_step(WfHandle h, const float* d_action, const WfStepOut* out, void* stream) {
    if (!h || !d_action) return set_err(WF_ERR_INVALID, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    TRY(launch_step(h, WF_MODE_ENV, nullptr, d_action, nullptr, out, (cudaStream_t)stream));
    return mark_async(h, (cudaStream_t)stream);
}

int wf_update_command(WfHandle h, const double* d_yaw, const WfStepOut* out, void* stream) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    CUDA_TRY(cudaSetDevice(h->device));
    TRY(launch_step(h, WF_MODE_INTERFACE, nullptr, nullptr, d_yaw, out, (cudaStream_t)stream));
    return mark_async(h, (cudaStream_t)stream);
}

// (Re)allocate the evaluation scratch for `cap` candidates.  Synchronous on both sides: no queued evaluation may still use the
// old scratch, and the zeroing of the new one (cudaMemset runs on the legacy default stream, which a caller's non-blocking
// stream does not wait for) is complete before the first evaluation kernel reads the counters.
static int eval_reserve(WfHandle h, int cap) {
    CUDA_TRY(cudaDeviceSynchronize());
    if (h->d_eval_fix) cudaFree(h->d_eval_fix);
    if (h->d_eval_vwg) cudaFree(h->d_eval_vwg);
    if (h->d_eval_yaw) cudaFree(h->d_eval_yaw);
    h->d_eval_fix = nullptr;
    h->d_eval_vwg = nullptr;
    h->d_eval_yaw = nullptr;
    h->eval_cap = 0;
    const size_t fix_bytes = sizeof(int) * ((size_t)cap + 4);
    cudaError_t e = cudaMalloc(&h->d_eval_fix, fix_bytes);
    if (e == cudaSuccess) e = cudaMemset(h->d_eval_fix, 0, fix_bytes);
    if (e == cudaSuccess && wf_fast64_gathers(h->model, h->st)) {
        const size_t vwg_bytes = sizeof(double2) * 9 * (size_t)h->model.T * (size_t)cap;
        e = cudaMalloc(&h->d_eval_vwg, vwg_bytes);
        if (e == cudaSuccess) e = cudaMemset(h->d_eval_vwg, 0, vwg_bytes);
    }
    if (e == cudaSuccess && is_strict_f32(h))
        e = cudaMalloc(&h->d_eval_yaw, sizeof(double) * (size_t)h->model.T * (size_t)cap);  // written before it is read
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_err(e == cudaErrorMemoryAllocation ? WF_ERR_NOMEM : WF_ERR_CUDA,
                       std::string("evaluation scratch: ") + cudaGetErrorString(e));
    }
    h->eval_cap = cap;
    return WF_OK;
}

// The two evaluation entry points: yaw candidates d_yaw (interface mode, out.power only) or action candidates d_action (env
// mode, every output of out), K per env, outputs in rows of B*K
static int evaluate(WfHandle h, const char* fn, const double* d_yaw, const float* d_action, int32_t K, const WfStepOut* outp,
                    uint8_t* d_ambiguous, cudaStream_t st) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    if (h->cfg.kernel != WF_KERNEL_FAST)
        return set_err(WF_ERR_INVALID, std::string(fn) + " needs the warp-per-env kernels (WF_KERNEL_FAST)");
    // K >= 1 is also what keeps the evaluation kernels from writing state: the FP64 ones skip their commits on a run-time
    // test of K (wf_fast64.cu: solve_env64), so this refusal must stay ahead of every launch below
    if (K < 1) return set_err(WF_ERR_INVALID, "K (candidates per env) must be >= 1");
    if ((!d_yaw && !d_action) || !outp) return set_err(WF_ERR_INVALID, "NULL argument");
    const WfStepOut out = *outp;
    const int64_t BK = (int64_t)h->model.B * K;
    if (BK > (int64_t)INT32_MAX)
        return set_err(WF_ERR_INVALID, "num_envs * K = " + std::to_string(BK) + " candidates exceed the kernels' 32-bit index "
                                       "(at most 2^31 - 1 per call)");
    CUDA_TRY(cudaSetDevice(h->device));
    if (BK > h->eval_cap) TRY(eval_reserve(h, (int)BK));
    const WfEvalArgs ev = {K, h->d_eval_fix, h->d_eval_fix + h->eval_cap, d_ambiguous, h->d_eval_vwg, h->d_eval_yaw};
    // the route of a step in the handle's current state: a stale vortex table is not read
    const bool use_vtab = !h->vtab_stale;
    cudaError_t e;
    if (h->cfg.precision == WF_PREC_F64) {
        e = wf_launch_eval_fast64(use_vtab, h->model, h->fast64, h->st, ev, d_yaw, d_action, out, st);
        h->launches += 1;
    } else {
        e = wf_launch_eval_fast(h->fast_baked, h->model, h->fast, h->st, ev, d_yaw, d_action, out, st);
        h->launches += 1;
        if (e == cudaSuccess && is_strict_f32(h)) {
            e = wf_launch_eval_fixup64(use_vtab, h->model, h->fast64, h->st, ev, d_yaw, d_action != nullptr, out, st);
            h->launches += 1;
        }
    }
    if (e != cudaSuccess) return set_err(WF_ERR_CUDA, std::string("evaluation kernel launch: ") + cudaGetErrorString(e));
    return mark_async(h, st);
}

int wf_evaluate_yaw(WfHandle h, const double* d_yaw, int32_t K, void* d_power, uint8_t* d_ambiguous, void* stream) {
    WfStepOut out = {};
    out.power = d_power;
    return evaluate(h, "wf_evaluate_yaw", d_yaw, nullptr, K, d_power ? &out : nullptr, d_ambiguous, (cudaStream_t)stream);
}

int wf_evaluate_actions(WfHandle h, const float* d_action, int32_t K, const WfStepOut* out, uint8_t* d_ambiguous,
                        void* stream) {
    return evaluate(h, "wf_evaluate_actions", nullptr, d_action, K, out, d_ambiguous, (cudaStream_t)stream);
}

// Device alias of a host pointer when it is page-locked memory the GPU can address (cudaHostAlloc / cudaHostRegister
// under unified addressing, e.g. a torch pinned tensor); NULL for NULL, and for pageable memory, which clears *all.
static void* mapped_alias(const void* p, bool* all) {
    cudaPointerAttributes a;
    if (!p) return nullptr;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) cudaGetLastError();
    else if (a.type == cudaMemoryTypeHost && a.devicePointer) return a.devicePointer;
    *all = false;
    return nullptr;
}

static constexpr size_t kZeroCopyMaxElems = 163840;  // envs x turbines up to which wf_step_host maps the host buffers

// device -> host copies of env rows [b0, b0 + nb) of the outputs the caller asked for, from the staging buffers
static int copy_out_rows(WfHandle h, const WfHostOut* ho, size_t b0, size_t nb, cudaStream_t st) {
    for (const Array& f : kOut)
        if (void* dst = ptr_at(ho, f)) {
            const size_t row = f.bytes(1, h->model.T, h->es);
            CUDA_TRY(cudaMemcpyAsync((char*)dst + b0 * row, (const char*)ptr_at(&h->d_out, f) + b0 * row, nb * row,
                                     cudaMemcpyDeviceToHost, st));
        }
    return WF_OK;
}

// shared implementation of the two host-buffer entry points
static int step_host_impl(WfHandle h, int mode, const float* h_action, const double* h_yaw, const WfHostOut* ho,
                          uint64_t* h2d, uint64_t* d2h) {
    CUDA_TRY(cudaSetDevice(h->device));
    const size_t B = h->model.B, T = h->model.T, BT = B * T, es = h->es;
    const uint64_t up = (h_action ? sizeof(float) * BT : 0) + (h_yaw ? sizeof(double) * BT : 0);
    uint64_t down = 0;
    for (const Array& f : kOut)
        if (ptr_at(ho, f)) down += f.bytes(B, T, es);
    if (h2d) *h2d = up;
    if (d2h) *d2h = down;
    // run after whatever the caller queued asynchronously on its own stream (resets, wind updates, device-side steps)
    const bool wait_async = h->ev_pending;
    h->ev_pending = false;

    // ---- zero-copy path: every buffer is mapped pinned memory -> ONE launch, no copy engine.  The kernel reads the
    // commands and writes the results over PCIe itself (coalesced 128-bit / 32-bit stores from the env epilogue), so
    // result traffic overlaps the solves of the other envs instead of trailing the last one.
    // Taken for small batches, where the call is launch- and copy-latency bound; big batches go through the copy
    // engines: the kernel's result stores are scattered in the original turbine order, which PCIe handles poorly.
    // WFCRL_B200_HOST_PATH=zero_copy|staged overrides the choice.
    const char* force = getenv("WFCRL_B200_HOST_PATH");
    const bool want_zero = force ? !strcmp(force, "zero_copy") : BT <= kZeroCopyMaxElems;
    if (want_zero) {
        bool all = true;
        const float* za = (const float*)mapped_alias(h_action, &all);
        const double* zy = (const double*)mapped_alias(h_yaw, &all);
        WfStepOut z = {};
        for (const Array& f : kOut) set_ptr_at(&z, f, mapped_alias(ptr_at(ho, f), &all));
        if (all) {
            if (wait_async) CUDA_TRY(cudaStreamWaitEvent(h->host_streams[0], h->ev_async, 0));
            TRY(launch_step(h, mode, nullptr, za, zy, &z, h->host_streams[0]));
            CUDA_TRY(cudaStreamSynchronize(h->host_streams[0]));
            return WF_OK;
        }
    }

    // ---- staged path (pageable buffers): chunks of envs, one stream per chunk, so the copies of chunk c overlap the
    // kernels of the later chunks; only the last chunk's device->host copies are exposed.
    if (!h->d_action) {
        TRY(dev_alloc(h, &h->d_action, BT));
        TRY(dev_alloc(h, &h->d_yaw_cmd, BT));
        for (const Array& f : kOut) {
            char* p;
            TRY(dev_alloc(h, &p, f.bytes(B, T, es)));
            set_ptr_at(&h->d_out, f, p);
        }
    }
    WfStepOut o = {};  // the staging buffers of the outputs the caller asked for
    for (const Array& f : kOut)
        if (ptr_at(ho, f)) set_ptr_at(&o, f, ptr_at(&h->d_out, f));
    const int nchunk = (B >= 2048) ? WfHandle_t::kHostStreams : 1;
    // Strict FP32 handle: the chunks' FP32 launches share one fix-up list and ONE FP64 re-solve launch follows the last chunk,
    // so the chunks' device->host copies overlap the later chunks as before and only the re-solve of the few flagged envs
    // trails; their results come back as compact records that are scattered into the caller's arrays below.
    const bool strict = is_strict_f32(h);
    const int rec_len = WF_FIX_REC_HDR + out_elems(kBT) * (int)T;
    if (strict && !h->d_fix_rec) {
        h->fix_rec_cap = (int)(B < 1024 ? B : 1024);
        TRY(dev_alloc(h, &h->d_fix_rec, (size_t)h->fix_rec_cap * rec_len));
        if (cudaMallocHost((void**)&h->h_fix_rec, sizeof(float) * (size_t)h->fix_rec_cap * rec_len) != cudaSuccess ||
            cudaMallocHost((void**)&h->h_fix_n, sizeof(int) * 4) != cudaSuccess)
            return set_err(WF_ERR_NOMEM, "cudaMallocHost failed");
        for (int c = 0; c < WfHandle_t::kHostStreams; ++c)
            CUDA_TRY(cudaEventCreateWithFlags(&h->ev_chunk[c], cudaEventDisableTiming));
    }
    for (int c = 0; c < nchunk; ++c) {
        const size_t b0 = B * c / nchunk, b1 = B * (c + 1) / nchunk, nb = b1 - b0;
        cudaStream_t st = h->host_streams[c];
        if (wait_async) CUDA_TRY(cudaStreamWaitEvent(st, h->ev_async, 0));
        if (h_action)
            CUDA_TRY(cudaMemcpyAsync(h->d_action + b0 * T, h_action + b0 * T, sizeof(float) * nb * T, cudaMemcpyHostToDevice, st));
        if (h_yaw)
            CUDA_TRY(cudaMemcpyAsync(h->d_yaw_cmd + b0 * T, h_yaw + b0 * T, sizeof(double) * nb * T, cudaMemcpyHostToDevice, st));
        TRY(launch_step(h, mode, nullptr, h_action ? h->d_action : nullptr, h_yaw ? h->d_yaw_cmd : nullptr, &o, st,
                        (int)b0, (int)nb, /*defer_fixup=*/true));
        if (strict) CUDA_TRY(cudaEventRecord(h->ev_chunk[c], st));
        TRY(copy_out_rows(h, ho, b0, nb, st));
    }
    if (strict) {
        cudaStream_t fs = h->host_streams[0];
        for (int c = 1; c < nchunk; ++c) CUDA_TRY(cudaStreamWaitEvent(fs, h->ev_chunk[c], 0));
        TRY(launch_fixup(h, mode, o, fs, h->d_fix_rec, h->fix_rec_cap));
        CUDA_TRY(cudaMemcpyAsync(h->h_fix_n, h->st.fix_count, sizeof(int) * 4, cudaMemcpyDeviceToHost, fs));
        // the first records ride along unconditionally (a typical step re-solves ~1 % of the envs); more only if needed
        const int eager = h->fix_rec_cap < 160 ? h->fix_rec_cap : 160;
        CUDA_TRY(cudaMemcpyAsync(h->h_fix_rec, h->d_fix_rec, sizeof(float) * (size_t)eager * rec_len, cudaMemcpyDeviceToHost, fs));
        for (int c = 0; c < nchunk; ++c) CUDA_TRY(cudaStreamSynchronize(h->host_streams[c]));
        const int n = h->h_fix_n[2];
        const int have = n < h->fix_rec_cap ? n : h->fix_rec_cap;
        if (have > eager) {
            CUDA_TRY(cudaMemcpyAsync(h->h_fix_rec + (size_t)eager * rec_len, h->d_fix_rec + (size_t)eager * rec_len,
                                     sizeof(float) * (size_t)(have - eager) * rec_len, cudaMemcpyDeviceToHost, fs));
            CUDA_TRY(cudaStreamSynchronize(fs));
        }
        for (int k = 0; k < have; ++k) {
            const float* r = h->h_fix_rec + (size_t)k * rec_len;
            int b;
            memcpy(&b, r, sizeof(int));
            const float* part[2] = {r + 1, r + WF_FIX_REC_HDR};  // the per-env and the per-turbine outputs, in kOut order
            for (const Array& f : kOut) {
                const float* src = part[f.ext == kBT];
                const size_t ne = f.elems(1, T);
                part[f.ext == kBT] += ne;
                uint8_t* dst = (uint8_t*)ptr_at(ho, f);
                if (dst && f.elem == 1)  // truncated: stored as 1.f / 0.f
                    for (size_t i = 0; i < ne; ++i) dst[b * ne + i] = (uint8_t)(src[i] != 0.f);
                else if (dst)
                    memcpy(dst + sizeof(float) * b * ne, src, sizeof(float) * ne);
            }
        }
        if (n > have) {  // more re-solved envs than records (never in practice): copy their rows from the device arrays
            TRY(copy_out_rows(h, ho, 0, B, fs));
            CUDA_TRY(cudaStreamSynchronize(fs));
        }
        return WF_OK;
    }
    for (int c = 0; c < nchunk; ++c) CUDA_TRY(cudaStreamSynchronize(h->host_streams[c]));
    return WF_OK;
}

int wf_step_host(WfHandle h, const float* h_action, const WfHostOut* ho, uint64_t* h2d, uint64_t* d2h) {
    if (!h || !h_action || !ho) return set_err(WF_ERR_INVALID, "NULL argument");
    return step_host_impl(h, WF_MODE_ENV, h_action, nullptr, ho, h2d, d2h);
}

int wf_update_command_host(WfHandle h, const double* h_yaw, const WfHostOut* ho) {
    if (!h || !ho) return set_err(WF_ERR_INVALID, "NULL argument");
    return step_host_impl(h, WF_MODE_INTERFACE, nullptr, h_yaw, ho, nullptr, nullptr);
}

int wf_update_wind(WfHandle h, const uint8_t* d_mask, const double* d_ws, const double* d_wd, const double* d_cs,
                   void* stream) {
    if (!h || !d_ws || !d_wd) return set_err(WF_ERR_INVALID, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(wf_launch_set_wind(h->model, h->st, d_mask, d_ws, d_wd, st));
    // Time-series mode moves the wind before every step (interface.py:563): rebuilding the table each time would cost
    // more than it saves, so it is rebuilt only when the wind has been steady for a while (restore, occasional updates);
    // envs without valid rows take the step kernel's direct path.
    CUDA_TRY(launch_geometry(h, d_mask, d_cs, st, h->steps_since_wind_update >= 8));
    h->launches += 1;
    h->steps_since_wind_update = 0;
    return mark_async(h, st);
}

int wf_set_turbulence_intensity(WfHandle h, const double* d_ti, void* stream) {
    if (!h || !d_ti) return set_err(WF_ERR_INVALID, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMemcpyAsync(h->st.ti_amb, d_ti, sizeof(double) * h->model.B, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
    return mark_async(h, (cudaStream_t)stream);
}

// the device array of an exported state array of `bytes` bytes
static int find_state(WfHandle h, const char* name, size_t bytes, void** p) {
    for (const Array& a : kState)
        if (a.name && !strcmp(a.name, name)) {
            if (a.bytes(h->model.B, h->model.T, h->es) != bytes) return set_err(WF_ERR_INVALID, "size mismatch for state array");
            *p = ptr_at(&h->st, a);
            return WF_OK;
        }
    return set_err(WF_ERR_INVALID, std::string("unknown state array '") + name + "'");
}

int wf_get_state(WfHandle h, const char* name, void* dst, size_t bytes) {
    if (!h || !name || !dst) return set_err(WF_ERR_INVALID, "NULL argument");
    void* p;
    TRY(find_state(h, name, bytes, &p));
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(dst, p, bytes, cudaMemcpyDeviceToHost));
    return WF_OK;
}

int wf_set_state(WfHandle h, const char* name, const void* src, size_t bytes) {
    if (!h || !name || !src) return set_err(WF_ERR_INVALID, "NULL argument");
    if (!strcmp(name, "layout_id"))
        return set_err(WF_ERR_INVALID, "\"layout_id\" is read-only here: wf_assign_layouts sets it, validates the ids and "
                                       "rebuilds the geometry");
    if (!strcmp(name, "turbine_count"))
        return set_err(WF_ERR_INVALID, "\"turbine_count\" is read-only: it follows from the env's layout id");
    void* p;
    TRY(find_state(h, name, bytes, &p));
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaDeviceSynchronize());
    const bool yaw = !strcmp(name, "yaw");
    if (yaw || !strcmp(name, "acc") || !strcmp(name, "acc_prev")) {  // the padding columns of the state hold 0 at all times
        const int B = h->model.B, T = h->model.T;
        std::vector<int32_t> cnt(B);
        CUDA_TRY(cudaMemcpy(cnt.data(), h->st.turbine_count, sizeof(int32_t) * B, cudaMemcpyDeviceToHost));
        for (int e = 0; e < B; ++e)
            for (int t = cnt[e]; t < T; ++t)
                if (yaw ? ((const double*)src)[(size_t)e * T + t] != 0.0 : ((const float*)src)[(size_t)e * T + t] != 0.f)
                    return set_err(WF_ERR_INVALID, std::string("\"") + name + "\": env " + std::to_string(e) + " has " +
                                                       std::to_string(cnt[e]) + " turbines, but column " + std::to_string(t) +
                                                       " (padding) is nonzero");
    }
    CUDA_TRY(cudaMemcpy(p, src, bytes, cudaMemcpyHostToDevice));
    return WF_OK;
}

int wf_device_info(WfHandle h, int32_t* sm_count, int32_t* sm_clock_khz, int32_t* ctas_per_sm, int32_t* regs,
                   int32_t* threads, int32_t* smem) {
    if (!h) return set_err(WF_ERR_INVALID, "NULL handle");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaFuncAttributes attr;
    int ctas = 0, thr = (h->model.T + 31) / 32 * 32, sm = 0;
    if (h->cfg.kernel == WF_KERNEL_FAST && h->cfg.precision == WF_PREC_F64) {
        CUDA_TRY(wf_step_fast64_attributes(h->model, h->st, &attr, &ctas, &thr, &sm));
    } else if (h->cfg.kernel == WF_KERNEL_FAST) {
        CUDA_TRY(wf_step_fast_attributes(h->fast_baked, h->model, &attr, &ctas, &thr, &sm));
    } else {
        CUDA_TRY(wf_step_basic_attributes(h->cfg.precision, &attr, &ctas, thr));
        sm = (int)attr.sharedSizeBytes;
    }
    if (sm_count) *sm_count = h->sm_count;
    if (sm_clock_khz) *sm_clock_khz = h->sm_clock_khz;
    if (ctas_per_sm) *ctas_per_sm = ctas;
    if (regs) *regs = attr.numRegs;
    if (threads) *threads = thr;
    if (smem) *smem = sm;
    return WF_OK;
}

uint64_t wf_launch_count(WfHandle h) { return h ? h->launches : 0; }

int wf_set_kernel_timing(WfHandle h, int32_t enabled) {
    if (!h) return set_err(WF_ERR_INVALID, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    if (enabled) {
        for (cudaEvent_t& ev : h->ev_t)
            if (!ev) CUDA_TRY(cudaEventCreate(&ev));
    } else {
        timing_collect(h);
    }
    h->timing = enabled != 0;
    return WF_OK;
}

int wf_get_kernel_timing(WfHandle h, double* step_kernel_ms, double* resolve_kernel_ms, int32_t* calls) {
    if (!h) return set_err(WF_ERR_INVALID, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    timing_collect(h);
    const int n = h->t_calls;
    if (step_kernel_ms) *step_kernel_ms = n ? h->t_step_ms / n : 0.0;
    if (resolve_kernel_ms) *resolve_kernel_ms = n ? h->t_fix_ms / n : 0.0;
    if (calls) *calls = n;
    h->t_step_ms = h->t_fix_ms = 0.0;
    h->t_calls = 0;
    return WF_OK;
}

}  // extern "C"
