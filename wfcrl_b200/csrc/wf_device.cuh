// Internal device-side structures shared by the kernels and the C-ABI layer (not part of the public ABI).
#pragma once
#include "../../include/wfcrl_b200.h"  // WfStepOut: the step kernels write the caller's output pointers

#include <cuda_runtime.h>
#include <stdint.h>

#define WF_MAX_TURBINES_K 128  // == WF_MAX_TURBINES of the public header
#define WF_FIX_REC_HDR 5  // floats ahead of the per-turbine part of a fix-up record (see wf_fixup64_kernel)
#define WF_NP 9  // 3x3 rotor grid (case.yaml:16), p = 3*j + k with j lateral, k vertical

// Model constants, passed to kernels by value (kernel parameter space = constant bank, broadcast reads).
struct WfModel {
    int T, B;
    int max_iter, continuous, multi_agent, shaper, table_len;
    int G;                         // rotor grid points per side (case.yaml:16 turbine_grid_points): 3, or 5 with the basic kernels
    float yaw_lo_f, yaw_hi_f, yaw_step_f;  // float32 bounds exactly as gymnasium Box stores them (mdp.py:111-116,143-144)
    float rate_f, dt_f;
    int autoreset;                 // step kernels reset an env themselves when its step truncates (wf_set_autoreset)
    unsigned long long ar_seed;    //   key of the counter-based wind sampler
    long long ar_offset;           //   global id of env 0 (the sampler's counter word)
    double ar_ti_lo, ar_ti_hi;     //   ambient-TI range drawn at reset (ti_hi <= ti_lo: keep the current value)
    int vtab_tmajor;               // vortex-table rows are stored target-major (FP64 handle: the gather kernel), else source-major
    float amb_eps;                 // relative half-width of the guard band around the 0.05 m/s overlap threshold (FP32 kernel)
    double load_coef, shaper_reference;
    double rho, ref_rho, shear, D, HH, TSR, pP;
    double alpha, beta, ka, kb, ad, bd, dm;
    double ch_const, ch_ai, ch_init, ch_down;
    double e3_112, e3_13;          // 3*exp(1/12), 3*exp(1/3) (Gauss deflection E0)
    // The pool fields below fill the 16 bytes of the single layout's former (xc, yc), so that neither the offsets of the
    // fields after them nor the size of the struct (and with it every later kernel parameter) moved.
    const double* layout_c;        // [L][2] device: centre of each pool layout's bounding box (its rotation centre),
                                   //     followed by the [L] int32 turbine counts n <= T of the layouts (layout_counts())
    int n_layouts;                 // L: layouts in the pool (wf_set_layouts)
    int sample_layouts;            // 1 = library-sampled resets also draw the env's layout id (wf_set_layout_sampling)
    const double* tab_ws;          // [table_len] device
    const double* tab_ct;          // [table_len]
    const double* tab_pw;          // [table_len] 0.5*area*Cp*eta*ws^3 (power / density)
    const double* layout_x;        // [L][T] device: the layout pool; env b's geometry is built from row layout_id[b]
    const double* layout_y;        // [L][T]; columns at or beyond the layout's turbine count are not read
};

// The pool's per-layout turbine counts, stored behind the centres (WfModel keeps its size: no kernel parameter moves).  Read
// by the geometry kernel only, which copies the env's count to WfState.turbine_count for the other kernels.
__host__ __device__ inline const int* layout_counts(const WfModel& m) { return (const int*)(m.layout_c + 2 * m.n_layouts); }

// Per-env state, device pointers (owned by the handle).
struct WfState {
    double* yaw;        // [B][T] current yaw command / state, degrees (float32-representable in env mode)
    float* acc;         // [B][T] actuation accumulator (mdp.py:157-160, 317-318)
    float* acc_prev;    // [B][T] accumulator one joint action earlier (multi-agent staleness)
    int* num_iter;      // [B] FlorisInterface._num_iter
    int* num_moves;     // [B] WindFarmEnv.num_moves
    int* nonfinite;     // [B] number of env steps whose reward came out NaN/Inf (guard counter, SURVEY section 5)
    int* episode;       // [B] number of library-sampled resets so far (counter word of the reset sampler)
    uint8_t* amb;       // [B] FP32 kernel: 1 = a discrete decision of this solve was within the guard band of its threshold
                        //     AND could change the result (the env is re-solved by the FP64 kernel), 0 = decisions are safe
    // episode bookkeeping, advanced by the env-mode epilogue of the step kernels (no host-side mirror, no extra launches):
    double* ep_return;  // [B] sum of the (shaped) rewards of the running episode
    int* ep_len;        // [B] its number of steps
    double* fin_sum;    // [B] over the episodes this env has FINISHED (truncated): sum of returns,
    double* fin_sumsq;  // [B]   sum of squared returns,
    int* fin_n;         // [B]   their number,
    long long* fin_len; // [B]   and the sum of their lengths
    uint8_t* reset_mask;// [B] 1 = the env was reset inside a step kernel and still needs its geometry + warm-up solve
    int* fix_list;      // [B] ids of the envs flagged by the FP32 launches since the last fix-up launch (appended atomically)
    int* fix_count;     // [4] number of flagged envs, number of fix-up CTAs that have left, the number of envs the last fix-up
                        //     launch re-solved, (pad)
    double* ws;         // [B] free-stream wind speed
    double* wd;         // [B] free-stream wind direction (already % 360)
    double* ws_norm;    // [B] free-stream speed of the PREVIOUS state (reward normalisation, simple_env.py:79)
    double* shaper_ref; // [B] StepPercentage.reference
    double* ti_amb;     // [B] ambient turbulence intensity
    // geometry (rebuilt when the wind direction changes)
    double* xs;         // [B][T] rotated x, sorted ascending (stable)
    double* ys;         // [B][T] rotated y in the same order
    double* xi;         // [B][T] np.mean of the 9 identical grid x values = fl(fl(8x+x)/9)
    double* yi;         // [B][T] np.mean of the 9 grid y values (numpy reduction order)
    int* order;         // [B][T] sorted position -> original turbine index
    double* cs;         // [B][2] cosd/sind of the deviation from west actually used
    // FP32 fast-kernel geometry: positions relative to the rotation centre as float-float pairs and, per SOURCE
    // position i, the first sorted target index for which each FP64 x-mask of SURVEY A.7/A.8 becomes true
    float2* xhl;        // [B][T] (hi, lo) of xs - xc (xc, yc: the centre of the env's layout)
    float2* yhl;        // [B][T] (hi, lo) of ys - yc
    uchar4* idx;        // [B][T] .x: first t with X[t]-x_i >= 0 ; .y: first t with X[t] > x_i+0.1 ;
                        //         .z: first t with X[t] > x_i ; .w: first t with X[t] > x_i+15D   (T if none)
    // Vortex table (FP64 warp-per-env kernels): the transverse velocities one source induces on one rotor point are LINEAR in
    // the source's two circulations (tip pair Gt -- the bottom tip vortex is -vel_bot/vel_top times the top one -- and
    // wake rotation Gwr) with coefficients that depend on the geometry only.  Built once per wind direction by
    // wf_vortex_table_kernel in SORTED order, so that a kernel streams it front to back:
    //   row(i, t) for sorted source i < target t at index i*T - i*(i+1)/2 + (t - i - 1); a row is [3 columns j][3 heights k]
    //   [cVt, cVw, cWt, cWw]:  V += Gt*cVt + Gwr*cVw ;  W += max(Gt*cWt + Gwr*cWw, 0)            (SURVEY A.7)
    double* vtab;       // [B][T(T-1)/2][36] rows, read by the FP64 kernels only: on an FP64 handle target-major (m.vtab_tmajor)
                        //     for the gather step kernel, on a strict FP32 handle source-major for the re-solve of the few
                        //     flagged envs; NULL = every pair is evaluated directly
    uint8_t* vtab_ok;   // [B] 1 = the env's rows match its current geometry (cleared by the geometry kernel)
    uint8_t* tab_lo;    // [B][T] per sorted source i: first t with xs[t] - xs[i] > 1e-6 m; closer targets (x-ties) are
                        //         evaluated directly from the positions, never through the table
    uint8_t* tab_glo;   // [B][T] the same relation seen from sorted target t: number of sources j with xs[t] - xs[j] > 1e-6 m
                        //         (a prefix of the sorted order) = the table sources of t
    // FP64 gather kernel (target-major table, m.vtab_tmajor): row(j, t) of source j < target t at index t*(t-1)/2 + j, so
    // that the rows one target sums in its prologue are contiguous; the finished (v, w) of every rotor point and the direct
    // contributions between x-tied turbines live in this scratch (rewritten by every launch; L2-resident while an env runs)
    double2* vwg;       // [B][9T]; an FP64 handle has both the table and this scratch, or neither
    int* layout_id;     // [B] row of the layout pool (WfModel.layout_x / _y / _c) the env's geometry is built from
    int* turbine_count; // [B] n = turbine count of that layout (written by the geometry kernel): the env runs turbines
                        //     0..n-1 of every [B][T] row; columns n..T-1 are padding, 0 in the yaw / acc / acc_prev state
                        //     and written as 0 in every per-turbine output
};

// Constants of the tuned warp-per-env kernels, precomputed on the host in FP64 (wf_host_const.h: build_fast_const);
// R = R for the FP32 kernel, double for the FP64 bit-check instantiation.
template <typename R> struct WfFastConstT {
    R ratio[3];        // (Z_k / HH)^shear : U0[k] = ws * ratio[k]
    R mean_ratio;      // Uinf = ws * mean_ratio
    R nu4[3];          // 4 * nu_k / Uinf (independent of ws)
    R zz[6][3];        // Z_k + c_v + NUM_EPS, vortices in FLORIS order V1..V6 (see wf_kernels.cu transverse())
    R zz2[6][3];       // zz^2
    R ez[6][3];        // exp(-zz^2 / eps^2)
    R cblk[48];        // the same constants packed for the kernel's shared-memory block (see build_fast_const)
    R a_top, a_bot, a_core;   // secondary steering: mean over the own grid of z/(2 pi r) * core per unit circulation
    R inv_ss_den;             // 1 / (c_top a_top - c_bot a_bot): the steering denominator is (that) * ws * ct
    R cv[3][9], cw[3][9];     // self-induced V / W per unit (Gt, Gb, Gwr) on the own grid
    R sv[3];                  // sum over the 9 points of cv
    R D, inv_D, eps2, inv_eps2, inv_2pi;
    R c_top, c_bot, c_wr;     // G_top0 = c_top*ws*ct ; G_bot0 = c_bot*ws*ct ; Gwr = c_wr*(a-a^2)*avg
    R alpha4, beta2, ka, kb, ad, bd, dm03, e3_112, e3_13;
    R near_c;                 // 0.501 * D * sqrt(1/2)
    R d2_8;                   // D^2 / 8
    R ch_const, ch_ai, ch_init, ch_down;
    R pP3, rho_fac, ref_rho, two_D, offj[3], dz2[3];
    R load_coef, shaper_reference;
    int table_len;
    R tab_ws[64], tab_ct[64], tab_pw[64];
    unsigned char coarse[128];    // coarse[floor(x * coarse_scale)] = table interval containing that bucket's left edge
    R coarse_scale;
    int coarse_len;
};
typedef WfFastConstT<float> WfFastConst;
typedef WfFastConstT<double> WfFastConst64;

enum WfMode { WF_MODE_INTERFACE = 0, WF_MODE_ENV = 1, WF_MODE_WARMUP = 2 };

// Candidate evaluation (wf_evaluate_yaw, wf_evaluate_actions): the EVAL instantiations of the fast kernels solve K candidates
// per env, CTA c = candidate c = env c / K, candidate c % K (the K candidates of an env are adjacent, so that its geometry and
// table rows are shared in L2).  They read the candidate's yaw (or action) from the caller's [B*K][T] array, write its output
// rows c and write no WfState array.  The scratch below belongs to the handle's evaluation path alone.
struct WfEvalArgs {
    int K;             // candidates per env
    int* fix_list;     // [B*K] strict FP32: ids of the candidates the FP32 launch flagged (never the step path's fix_list)
    int* fix_count;    // [4] as WfState.fix_count, for fix_list
    uint8_t* amb;      // [B*K] or NULL: 1 = the candidate was re-solved by the FP64 kernel
    double2* vwg;      // [B*K][9T] FP64 gather form: the (v, w) scratch, one row per candidate (WfState.vwg is per env)
    double* yaw;       // [B*K][T] strict FP32, actions: the transitioned yaw of a flagged candidate, which its re-solve
                       //     reads where the step's re-solve reads the committed WfState.yaw
};

// launchers implemented in wf_kernels.cu
cudaError_t wf_launch_geometry(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_cs_override,
                               cudaStream_t stream, bool autoreset_draw = false);
cudaError_t wf_launch_step_basic(int precision, int mode, const WfModel& m, const WfState& s, const uint8_t* d_mask,
                                 const float* d_action, const double* d_yaw_cmd, const WfStepOut& out,
                                 int env_begin, int env_count, cudaStream_t stream);
cudaError_t wf_launch_vortex_table(const WfModel& m, const WfFastConst64& fc, const WfState& s, const uint8_t* d_mask,
                                   cudaStream_t stream);
cudaError_t wf_launch_set_wind(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_ws,
                               const double* d_wd, cudaStream_t stream);
cudaError_t wf_launch_sample_reset(const WfModel& m, const WfState& s, const uint8_t* d_mask, unsigned long long seed,
                                   long long env_id_offset, double ti_lo, double ti_hi, double* d_ws, double* d_wd,
                                   cudaStream_t stream);
cudaError_t wf_launch_reset_state(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_ws,
                                  const double* d_wd, cudaStream_t stream);
cudaError_t wf_step_basic_attributes(int precision, cudaFuncAttributes* attr, int* ctas_per_sm, int threads);
// Kernel attributes of the tuned kernels (dynamic shared memory above 48 KB, carveout).  They belong to the current
// device, so wf_create sets them once per handle, before the handle's first launch.
cudaError_t wf_configure_fast_kernels();    // wf_fast.cu
cudaError_t wf_configure_fast64_kernels();  // wf_fast64.cu
cudaError_t wf_launch_step_fast(int mode, bool baked, const WfModel& m, const WfFastConst& fc, const WfState& s,
                                const uint8_t* d_mask, const float* d_action, const double* d_yaw_cmd,
                                const WfStepOut& out, int env_begin, int env_count, cudaStream_t stream);
cudaError_t wf_launch_fixup64(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                              const WfStepOut& out, int env_count, float* d_rec, int rec_cap, cudaStream_t stream);
cudaError_t wf_step_fast_attributes(bool baked, const WfModel& m, cudaFuncAttributes* attr, int* ctas_per_sm, int* threads,
                                    int* smem);
cudaError_t wf_launch_step_fast64(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                  const uint8_t* d_mask, const float* d_action, const double* d_yaw_cmd,
                                  const WfStepOut& out, int env_begin, int env_count, cudaStream_t stream);
cudaError_t wf_step_fast64_attributes(const WfModel& m, const WfState& s, cudaFuncAttributes* attr, int* ctas_per_sm, int* threads,
                                      int* smem);
// candidate evaluation: one launch of B*K CTAs with out's buffers of B*K rows; on a strict FP32 handle wf_launch_eval_fixup64
// re-solves the flagged candidates (ev.fix_list) in FP64.  d_action == NULL: yaw candidates d_yaw [B*K][T] in interface mode,
// out.power only (wf_evaluate_yaw); else action candidates d_action [B*K][T] in env mode, every output (wf_evaluate_actions)
cudaError_t wf_launch_eval_fast(bool baked, const WfModel& m, const WfFastConst& fc, const WfState& s, const WfEvalArgs& ev,
                                const double* d_yaw, const float* d_action, const WfStepOut& out, cudaStream_t stream);
cudaError_t wf_launch_eval_fast64(bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                  const WfEvalArgs& ev, const double* d_yaw, const float* d_action, const WfStepOut& out,
                                  cudaStream_t stream);
cudaError_t wf_launch_eval_fixup64(bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                   const WfEvalArgs& ev, const double* d_yaw, bool actions, const WfStepOut& out,
                                   cudaStream_t stream);
bool wf_fast64_gathers(const WfModel& m, const WfState& s);  // an FP64 handle's step kernel runs the gather form
