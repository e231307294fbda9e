/*
 * wfcrl_b200 -- C-ABI of the B200-native batched Floris backend for ifpen/wfcrl-env.
 *
 * This is the drop-in boundary for ONE hot path of the reference: everything that happens behind
 * `FlorisInterface.update_command` (reference wfcrl/interface.py:557-586) for every `*_Floris` env step, i.e. the
 * FLORIS 3.5 GCH steady-state wake solve, the per-turbine measures (interface.py:622-648) and -- fused around it --
 * the WFCRL MDP transition and reward (wfcrl/mdp.py:273-319, wfcrl/simple_env.py:58-96, wfcrl/rewards.py:16-46),
 * evaluated for `num_envs` independent environments at once by hand-written sm_100a CUDA kernels.
 *
 * Conventions
 *  - plain pointers and sizes only; no C++/torch types; every function returns WF_OK (0) or an error code and
 *    never throws; `wf_last_error()` returns a thread-local human-readable message.
 *  - "real" = double when the handle was created with WF_PREC_F64 (bit-check mode, <=1e-9 relative vs the
 *    reference arithmetic) and float with WF_PREC_F32 (fast mode, <=1e-4 relative on every turbine with the tuned
 *    kernel unless WfConfig.fp32_relaxed is set).
 *  - all `d_*` pointers are DEVICE pointers on the handle's device, all `h_*` pointers are HOST pointers.
 *  - per-turbine arrays are row-major [num_envs][num_turbines] in the ORIGINAL turbine order of the layout.  An env whose
 *    layout has n < num_turbines turbines (wf_set_layouts_sized) uses columns 0..n-1; columns n.. are padding.
 *  - output buffers must be aligned to 16 bytes (`load` is written with 128-bit stores, `freewind` with 64-bit stores).
 *  - all launches are asynchronous on the `stream` argument (a cudaStream_t passed as void*; NULL = default
 *    stream); no host synchronisation happens inside unless stated.
 *  - there is NO CPU fallback: without a CUDA device `wf_create` fails with WF_ERR_CUDA.
 */
#ifndef WFCRL_B200_H
#define WFCRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WF_MAX_TURBINES 128 /* one thread per turbine inside a CTA */
#define WF_TABLE_MAX 64     /* rows of the Cp/Ct table (nrel_5MW has 51) */

typedef struct WfHandle_t* WfHandle;

enum WfStatus { WF_OK = 0, WF_ERR_INVALID = 1, WF_ERR_CUDA = 2, WF_ERR_NOMEM = 3 };
enum WfPrecision { WF_PREC_F64 = 0, WF_PREC_F32 = 1 };
/* reward shapers of wfcrl/rewards.py:16-46 */
enum WfShaper { WF_SHAPER_NONE = 0, WF_SHAPER_REFERENCE_PCT = 1, WF_SHAPER_STEP_PCT = 2 };
/* kernel variants: 0 = straightforward one-thread-per-turbine kernel (FP64 and FP32), 1 = tuned warp-per-env kernel
 * (FP32 fast mode, or its FP64 instantiation for the bit-check mode) */
enum WfKernel { WF_KERNEL_BASIC = 0, WF_KERNEL_FAST = 1 };

/*
 * Everything the reference reads from its FlorisCase / case.yaml / env kwargs for this path.
 * `wf_default_config` fills the values of wfcrl/simulators/floris/inputs/template/case.yaml:14-16,27-39,41-60,84-89,
 * FLORIS' turbine_library nrel_5MW (SURVEY.md App. B) and the env defaults of wfcrl/simple_env.py:24-25,
 * wfcrl/environments/data_cases.py:19-23 (yaw bounds), wfcrl/mdp.py:52 (actuator rate).
 */
typedef struct WfConfig {
    int32_t num_turbines;       /* T <= WF_MAX_TURBINES */
    int32_t num_envs;           /* B: environments resident on this device (the local shard) */
    int32_t device;             /* CUDA device ordinal */
    int32_t precision;          /* enum WfPrecision */
    int32_t kernel;             /* enum WfKernel */
    int32_t max_iter;           /* interface.max_iter = start_iter + max_num_steps (simple_env.py:33, interface.py:586) */
    int32_t continuous_control; /* mdp.py:300-310: 1 = Box actions clipped to +-step, 0 = {0,1,2} -> (a-1)*step */
    int32_t multi_agent;        /* 1 = actuation constraint with the per-agent staleness of multiagent_env.py:198-249 */
    int32_t reward_shaper;      /* enum WfShaper */
    int32_t fp32_relaxed;       /* WF_PREC_F32 + WF_KERNEL_FAST only.  0 (default) = strict: solves whose discrete decisions (wake
                                   overlap count, 2D window) or power-curve conditioning are beyond FP32 are detected in the
                                   step kernel and redone by the FP64 kernel in a second launch, so that every turbine meets
                                   the 1e-4 tolerance; 1 = raw FP32 results, no second launch (a few envs in 1e4 differ by up
                                   to ~1e-2, DESIGN.md section 3) */
    double yaw_lo, yaw_hi, yaw_step; /* controls["yaw"] = (low, high, step), default (-40, 40, 5) */
    double load_coef;                /* simple_env.py:25 */
    double shaper_reference;         /* ReferencePercentage.reference (StepPercentage always restarts from 0 at reset,
                                        rewards.py:45-46, whatever its constructor argument) */
    double dt;                       /* FlorisCase.dt = 60 (data_cases.py:507) */
    double actuator_rate;            /* mdp.py:52 ACTUATORS_RATE["yaw"] = 0.3 */
    /* flow field (case.yaml:30-39) */
    double air_density, turbulence_intensity, wind_shear, wind_veer;
    /* Gauss deflection / velocity parameters (case.yaml:52-60, 76-80) */
    double alpha, beta, ka, kb, ad, bd, dm;
    /* Crespo-Hernandez (case.yaml:84-89) */
    double ch_initial, ch_constant, ch_ai, ch_downstream;
    /* turbine (nrel_5MW) */
    double rotor_diameter, hub_height, tsr, pP, pT, generator_efficiency, ref_density_cp_ct;
    int32_t table_len;
    int32_t turbine_grid_points; /* rotor grid points per side (case.yaml:16): 0 or 3 = the template's 3x3 grid; 5 = 5x5, evaluated
                                    by the WF_KERNEL_BASIC kernels only (generalisation knob, SURVEY 8f row 4) */
    double table_ws[WF_TABLE_MAX], table_cp[WF_TABLE_MAX], table_ct[WF_TABLE_MAX];
} WfConfig;

/*
 * Device output buffers of one step; any pointer may be NULL (that output is skipped).
 * Replaces what the reference returns from WindFarmEnv.step (simple_env.py:86-96):
 *   yaw, wind_speed, wind_direction, freewind -> the observation dict (mdp.py:278-281)
 *   power [MW] and load -> info["power"], info["load"] (mdp.py:282-284)
 *   reward -> simple_env.py:78-85 ; truncated -> interface.py:586 ; terminated is always false (simple_env.py:87)
 */
typedef struct WfStepOut {
    void* yaw;            /* real [B][T]    yaw state after the transition, degrees */
    void* wind_speed;     /* real [B][T]    cbrt(mean(u^3)) per rotor           (interface.py:643) */
    void* wind_direction; /* real [B][T]    mean(wd - degrees(atan2(v,u)))      (interface.py:644-647) */
    void* power;          /* real [B][T]    MW in env mode (mdp.py:284), W in interface mode (interface.py:623) */
    void* load;           /* real [B][T][4] TI, std u, std v, std w (interface.py:629-637); env mode: x1e7 then /1e7,
                                            interface mode: x1e7 as stored in current_measures (interface.py:575-577) */
    void* reward;         /* real [B]       env mode only */
    void* freewind;       /* real [B][2]    free-stream wind speed, direction (interface.py:625-627) */
    uint8_t* truncated;   /* [B]            _num_iter == max_iter (interface.py:586) */
} WfStepOut;

/* Host mirror of WfStepOut for the end-to-end entry point (pinned or pageable host memory, same shapes). */
typedef WfStepOut WfHostOut;

/* Fill `cfg` with the reference defaults (see WfConfig). num_turbines / num_envs / max_iter are left 0. */
int wf_default_config(WfConfig* cfg);

/*
 * Replaces FlorisInterface.from_case / __init__ (interface.py:462-501, 526-547) and WindFarmMDP.__init__'s
 * accumulators (mdp.py:157-160) for `num_envs` envs.  layout_x/y: HOST, [T] metres: the handle's layout pool holds this
 * one layout and every env has layout id 0 (wf_set_layouts / wf_assign_layouts give envs different farms).
 * All envs start with wind (8 m/s, 270 deg) (data_cases.py:99-100), zero yaw, zero counters.
 */
int wf_create(const WfConfig* cfg, const double* h_layout_x, const double* h_layout_y, WfHandle* out);
int wf_destroy(WfHandle h);

/*
 * Layout pool: a handle holds n_layouts >= 1 farm layouts of its num_turbines turbines, and each env builds its geometry
 * from one of them, its "layout id" (state array "layout_id").  Each layout is rotated about the centre of its own bounding
 * box, (min + max) / 2 per axis, as a single-layout handle does; an env's results equal those of a handle created with
 * its layout alone.
 * wf_set_layouts replaces the pool: h_x, h_y HOST double [n_layouts][T] metres (finite).  Every env gets layout id 0 and
 * the geometry of all envs is rebuilt with their current wind; counters and yaw are kept (as in wf_update_wind).
 * Synchronous: it waits for every earlier asynchronous call on the handle.
 */
int wf_set_layouts(WfHandle h, int32_t n_layouts, const double* h_x, const double* h_y);
/*
 * The same with a turbine count per layout: layout l has h_counts[l] in [1, T] turbines, its first h_counts[l] entries of
 * h_x[l], h_y[l] ([n_layouts][T]); entries at or beyond the count are ignored and need not be finite, and the bounding-box
 * centre is taken over the layout's own turbines.  wf_set_layouts is the case of every count equal to T.
 * An env of n < T turbines runs them in columns 0..n-1 of every [B][T] array ("turbine_count" i32[B] in wf_get_state):
 *  - columns n..T-1 (padding) of yaw, wind_speed, wind_direction, power and load are written as 0 by every call;
 *  - the padding of the yaw / acc / acc_prev state holds 0 at all times (wf_set_state refuses nonzero padding; an env
 *    that moves to a smaller layout through wf_assign_layouts or a layout draw has its new padding zeroed), and actions
 *    and yaw commands in padding columns are ignored;
 *  - the reward is the mean over the env's n turbines, and every output of the env's first n columns equals, bit for bit,
 *    that of a handle created with its layout alone in the same precision and kernel mode.
 * Counts below T are rejected (WF_ERR_INVALID, before anything changes) on WF_KERNEL_BASIC and multi_agent handles, which
 * do not support padding; so are counts outside [1, T] and non-finite coordinates within a count.
 */
int wf_set_layouts_sized(WfHandle h, int32_t n_layouts, const int32_t* h_counts, const double* h_x, const double* h_y);
/*
 * Sets the layout ids of the listed envs and rebuilds their geometry.  h_env_ids: HOST int32 [n] or NULL with
 * n == num_envs meaning "all envs in order"; h_layout_ids: HOST int32 [n] in [0, n_layouts).  Out-of-range env or layout
 * ids are rejected before anything changes.  Synchronous (the stream is synchronised before returning).
 */
int wf_assign_layouts(WfHandle h, const int32_t* h_env_ids, int32_t n, const int32_t* h_layout_ids, void* stream);
/*
 * While enabled, every library-sampled reset (wf_reset_sampled and the in-kernel auto-reset) also draws the env's layout
 * id uniformly from the pool: id = floor(u53(r.x, r.y) * n_layouts) with r = Philox4x32-10 of counter (global env id lo,
 * hi, episode index, 2) under key = seed, the same key and counter as that reset's wind draw (which uses draw words 0 and 1),
 * so the winds and TI of every reset are the same with sampling on or off.  Disabled at creation.
 */
int wf_set_layout_sampling(WfHandle h, int32_t enabled);

/*
 * Replaces WindFarmMDP.reset -> FlorisInterface.init + (start_iter+1) x update_command() (mdp.py:260-270,
 * interface.py:588-613): for the selected envs set the wind, zero yaw / accumulators / iteration counters / shaper
 * state, rebuild the rotated + sorted geometry and run `warmup_solves` zero-yaw solves (each increments _num_iter,
 * which is why an env with max_num_steps=N truncates at step N-1).  `out` receives the start observation rows of
 * the selected envs (other rows untouched).
 *   h_env_ids : HOST int32 [n] or NULL with n == num_envs meaning "all envs in order"
 *   h_ws, h_wd: HOST double [n] wind speed [m/s] and direction [deg] (wd is reduced % 360 as interface.py:664)
 *   h_cos, h_sin: HOST double [n] or NULL.  When given they are used as cosd/sind of the wind deviation from west
 *                 instead of the device's own FP64 cos/sin (bit-exact geometry vs a host reference, SURVEY 7.3).
 * Synchronous: the stream is synchronised before returning (host arrays may be freed; resets are rare).
 */
int wf_reset(WfHandle h, const int32_t* h_env_ids, int32_t n, const double* h_ws, const double* h_wd,
             const double* h_cos, const double* h_sin, int32_t warmup_solves, const WfStepOut* out, void* stream);

/* Same as wf_reset but fully on device: d_mask uint8 [B] selects envs, d_ws/d_wd double [B] (read where mask!=0). */
int wf_reset_masked(WfHandle h, const uint8_t* d_mask, const double* d_ws, const double* d_wd,
                    int32_t warmup_solves, const WfStepOut* out, void* stream);

/*
 * wf_reset_masked with the winds drawn inside the library from the reference's reset distribution (mdp.py:242-258:
 * ws = clip(8 * Weibull(8), 3, 28), wd = clip(N(270, 20) % 360, 0, 360)).  numpy's Generator stream cannot be reproduced
 * on the device, so the draws come from Philox4x32-10 with key = seed and counter = (env_id_offset + b, episode index
 * of env b): an env's winds depend on its GLOBAL id and on how many sampled resets it has had ("episode" state array),
 * never on how the envs are sharded over handles / GPUs.  ws by Weibull inversion, wd by Box-Muller.  When
 * ti_hi > ti_lo the ambient turbulence intensity of the selected envs is drawn U(ti_lo, ti_hi) as well (extension; the
 * reference fixes 0.06, case.yaml:33); pass ti_lo = ti_hi = 0 to leave it alone.  With wf_set_layout_sampling on, the
 * layout id of each selected env is drawn too, and its geometry is built from that layout; otherwise each env keeps its
 * layout.  d_mask NULL = all envs.  Asynchronous.
 */
int wf_reset_sampled(WfHandle h, const uint8_t* d_mask, uint64_t seed, int64_t env_id_offset, double ti_lo, double ti_hi,
                     int32_t warmup_solves, const WfStepOut* out, void* stream);

/*
 * ENV MODE.  Replaces one WindFarmEnv.step / one full MAWindFarmEnv agent cycle for every env:
 * actuation-rate constraint (simple_env.py:65-72), action clip + yaw transition in float32 + accumulator
 * (mdp.py:291-319), FlorisInterface.update_command (interface.py:557-586), powers/1e6 and loads/1e7
 * (mdp.py:278-284), reward with the previous state's free-stream speed (simple_env.py:78-85) and the shaper.
 *   d_action: DEVICE float [B][T]; continuous: yaw increments in degrees; discrete: values in {0,1,2}.
 * A pure stream operation (one kernel launch, no host synchronisation, no allocation): it can be captured into a CUDA
 * graph together with the caller's own kernels (wf_launch_count then counts the captured launch once).
 */
int wf_step(WfHandle h, const float* d_action, const WfStepOut* out, void* stream);

/*
 * In-kernel auto-reset: the batched counterpart of "env.reset() as soon as the episode truncates" (mdp.py:260-262 behind
 * simple_env.py:49-56) without a reset launch chain of its own.  Once armed, a wf_step whose env reaches
 * _num_iter == max_iter ALSO starts that env's next episode inside the step kernel: the wind is drawn as by
 * wf_reset_sampled (key = seed, counter = (env_id_offset + b, episode index)), as is its layout id when
 * wf_set_layout_sampling is on (otherwise the env keeps its layout), yaw / accumulators / counters / shaper state
 * are zeroed, and the env is marked.  The outputs of that wf_step still hold the FINAL observation of the finished episode.
 * wf_autoreset_finish then rebuilds the geometry of the marked envs, runs their warm-up solve(s) -- overwriting their rows
 * of `out` with the start observation -- and clears the marks; with no env marked its launches exit at once, so it may be
 * called after every step or only when the caller knows an episode ended (episodes have a fixed length).
 * WF_KERNEL_FAST handles only.  enabled = 0 disarms.
 */
int wf_set_autoreset(WfHandle h, int32_t enabled, uint64_t seed, int64_t env_id_offset, double ti_lo, double ti_hi);
int wf_autoreset_finish(WfHandle h, int32_t warmup_solves, const WfStepOut* out, void* stream);

/*
 * INTERFACE MODE.  Replaces FlorisInterface.update_command(yaw=...) (interface.py:557-586) alone: no constraint, no
 * clipping, no reward.  d_yaw: DEVICE double [B][T] absolute yaw command in degrees, or NULL to keep the current
 * command (update_command() with no argument, mdp.py:262).
 */
int wf_update_command(WfHandle h, const double* d_yaw, const WfStepOut* out, void* stream);

/*
 * CANDIDATE EVALUATION.  Solve K candidate yaw settings per env in its CURRENT wind, TI, layout and geometry, without
 * changing the handle's state ("what would the farm produce with these yaws?": yaw optimisation, model-based control).
 *   d_yaw:       DEVICE double [B][K][T] absolute yaw in degrees (used as given, like wf_update_command: no clipping)
 *   d_power:     DEVICE real   [B][K][T] per-turbine power in W (interface-mode units, interface.py:623)
 *   d_ambiguous: DEVICE uint8  [B][K] or NULL: 1 = this candidate was re-solved by the FP64 kernel (strict FP32 handle;
 *                always 0 on other handles)
 * WF_KERNEL_FAST handles only.  Asynchronous on `stream`.
 *  - State: no state array changes -- none of the names wf_get_state accepts (yaw, "ambiguous", num_iter, the episode sums,
 *    nonfinite, ...), nor the re-solve list of the step path.  The next wf_step gives the same result bit for bit as if the
 *    evaluation had not happened.
 *  - Results: candidate (b, k) gives, bit for bit, the `power` row that wf_update_command with that yaw would write on this
 *    handle in its current state, including candidates that a strict FP32 handle flags and re-solves in FP64.
 *  - Layout pools of mixed counts: an env of n < T turbines ignores columns n..T-1 of its candidates (they may hold NaN)
 *    and writes 0 there.  Multi-agent handles evaluate like any other (there is no transition).
 *  - Launches: one per call, plus one FP64 re-solve launch on a strict FP32 handle (counted in wf_launch_count).
 *  - Scratch: the first call with a larger B*K than before allocates the evaluation scratch, synchronously; later calls
 *    with no larger K allocate nothing.
 *  - Envs marked by the in-kernel auto-reset must be finished (wf_autoreset_finish) first.
 * Refused with WF_ERR_INVALID before any work: WF_KERNEL_BASIC handles (and so the 5x5 grid), K < 1, NULL d_yaw or
 * d_power, and B*K > 2^31 - 1 (the kernels' index type).
 */
int wf_evaluate_yaw(WfHandle h, const double* d_yaw, int32_t K, void* d_power, uint8_t* d_ambiguous, void* stream);

/*
 * ACTION EVALUATION (one-step lookahead).  What wf_step would return for each of K candidate actions per env, from where
 * each env is now, without stepping: the batched one-step model query of model-based RL, MPC and planning baselines.
 *   d_action:    DEVICE float [B][K][T], each [T] row interpreted exactly as wf_step interprets d_action (continuous:
 *                increments clipped to +-step; discrete: values in {0, 1, 2})
 *   out:         a WfStepOut whose buffers have B*K rows, i.e. the shapes of a handle of B*K envs: real [B][K][T] yaw,
 *                wind_speed, wind_direction, power, real [B][K][T][4] load, real [B][K] reward, uint8 [B][K] truncated,
 *                real [B][K][2] freewind.  Any member may be NULL, as for wf_step.  Env-mode units (MW, loads / 1e7).
 *   d_ambiguous: DEVICE uint8 [B][K] or NULL, as for wf_evaluate_yaw
 * WF_KERNEL_FAST handles only.  Asynchronous on `stream`.
 *  - Results: row (b, k) of every output equals, bit for bit, row b of what wf_step would write on this handle in its
 *    current state with candidate k as env b's action: the actuation constraint with acc / num_moves (acc_prev on
 *    multi-agent handles), the clip, the float32 yaw transition, the loads, the reward normalised by ws_norm with its load
 *    term and shaper (StepPercentage reads shaper_ref and does not write it), truncated = (num_iter + 1 == max_iter), and
 *    candidates that a strict FP32 handle flags and re-solves in FP64.
 *  - State: as wf_evaluate_yaw, nothing changes -- yaw, acc, acc_prev, num_iter, num_moves, nonfinite, episode,
 *    "ambiguous", the episode sums, shaper_ref, ws_norm, the step path's re-solve list -- and the in-kernel auto-reset never
 *    fires or marks an env.  The next wf_step gives the same result bit for bit as if the evaluation had not happened.
 *  - Layout pools of mixed counts: actions in columns n..T-1 of an env of n < T turbines are ignored (they may hold NaN);
 *    those columns of every per-turbine output are written as 0.
 *  - Launches, scratch, auto-reset precondition: as wf_evaluate_yaw, with which it shares the scratch (calls of the two
 *    with different K may be interleaved).
 * Refused with WF_ERR_INVALID before any work: WF_KERNEL_BASIC handles, K < 1, NULL d_action or out, and
 * B*K > 2^31 - 1.
 */
int wf_evaluate_actions(WfHandle h, const float* d_action, int32_t K, const WfStepOut* out, uint8_t* d_ambiguous,
                        void* stream);

/*
 * End-to-end convenience for hosts without device buffers: `h_action` (float [B][T]) in, wf_step, every non-NULL
 * member of `h_out` out, synchronous.  Two routes, same results bit for bit:
 *   - staged: cudaMemcpyAsync into device staging owned by the handle, 6 env chunks on 6 streams so the copies of one
 *     chunk overlap the kernels of the next (any host memory; pinned is faster);
 *   - zero-copy: when EVERY buffer is page-locked memory the device can address (cudaHostAlloc / cudaHostRegister,
 *     e.g. a torch pinned tensor) and B*T <= 163840, the buffers are mapped into the step kernel, which reads the
 *     commands and writes the results over PCIe itself: one launch, no copy engine, ~25 us less latency per call.
 *     Beyond that size the copy engines win (measured, DESIGN.md section 6).
 * WFCRL_B200_HOST_PATH=staged|zero_copy in the environment forces a route.  The bytes that crossed PCIe are returned
 * through the optional counters.
 */
int wf_step_host(WfHandle h, const float* h_action, const WfHostOut* h_out, uint64_t* h2d_bytes, uint64_t* d2h_bytes);

/*
 * Host-buffer flavour of wf_update_command: the one call a reference-side binding needs to replace
 * FlorisInterface.update_command (interface.py:557-586) without managing device memory (see INTEGRATION.md).
 * h_yaw: HOST double [B][T] absolute yaw command or NULL (keep the current command).  Synchronous.
 */
int wf_update_command_host(WfHandle h, const double* h_yaw, const WfHostOut* h_out);

/* Change per-env wind without resetting counters (FlorisInterface.update_wind, interface.py:663-671; time-series
 * mode, interface.py:503-524,563).  Rebuilds the rotated/sorted geometry of the selected envs.
 *   d_mask: uint8 [B] or NULL (= all) ; d_ws, d_wd: double [B] (read where selected; wd is reduced % 360)
 *   d_cs  : double [B][2] host-computed cosd/sind of the deviation from west, or NULL to use the device's FP64 cos/sin */
int wf_update_wind(WfHandle h, const uint8_t* d_mask, const double* d_ws, const double* d_wd, const double* d_cs,
                   void* stream);

/* Per-env ambient turbulence intensity (extension; the reference keeps case.yaml's 0.06). d_ti: double [B]. */
int wf_set_turbulence_intensity(WfHandle h, const double* d_ti, void* stream);

/*
 * State access for tests / checkpoint-resume (synchronous).  `name` is one of
 *   "yaw" f64[B][T] | "acc" f32[B][T] | "acc_prev" f32[B][T] | "num_iter" i32[B] | "num_moves" i32[B] |
 *   "nonfinite" i32[B] (guard counter: env steps whose reward was NaN/Inf since creation) |
 *   "episode" i32[B] (sampled resets so far: the counter word of wf_reset_sampled) |
 *   "ambiguous" u8[B] (strict FP32 handles: 1 = the last solve of this env was redone in FP64) |
 *   episode bookkeeping kept by the env-mode step kernels: "ep_return" f64[B], "ep_len" i32[B] (running episode) and, over the
 *   episodes the env has finished, "fin_sum" f64[B], "fin_sumsq" f64[B], "fin_n" i32[B], "fin_len" i64[B] |
 *   "ws" f64[B] | "wd" f64[B] | "ws_norm" f64[B] | "shaper_ref" f64[B] | "ti_ambient" f64[B] |
 *   "order" i32[B][T] | "xs" f64[B][T] | "ys" f64[B][T] | "xi" f64[B][T] | "yi" f64[B][T] | "cs" f64[B][2] |
 *   "layout_id" i32[B] (row of the layout pool each env uses; read-only here: wf_set_state refuses it, wf_assign_layouts
 *   sets it) | "turbine_count" i32[B] (turbine count of that layout; read-only)
 * `bytes` must equal the full array size.  wf_set_state refuses "yaw", "acc" and "acc_prev" arrays that are nonzero in
 * an env's padding columns (see wf_set_layouts_sized).
 */
int wf_get_state(WfHandle h, const char* name, void* h_dst, size_t bytes);
int wf_set_state(WfHandle h, const char* name, const void* h_src, size_t bytes);

/* Introspection for bench.py: SM count of the device, and occupancy facts of the step kernel in use. */
int wf_device_info(WfHandle h, int32_t* sm_count, int32_t* sm_clock_khz, int32_t* ctas_per_sm,
                   int32_t* regs_per_thread, int32_t* threads_per_cta, int32_t* smem_per_cta);
/* Number of kernel launches issued by this handle since creation (for bench.py's gpu_launches). */
uint64_t wf_launch_count(WfHandle h);
/* Per-kernel device timing of the step calls (wf_step / wf_update_command on device buffers), for bench.py's roofline block:
 * while enabled, every step call brackets its step-kernel launch and -- on a strict FP32 handle -- its FP64 re-solve launch
 * with CUDA events on the caller's stream (and waits for the PREVIOUS call's events, so it is for measurement legs, not for
 * production loops).  wf_get_kernel_timing waits for the last call, returns the average duration of each launch over the
 * calls since the previous query (resolve_ms = 0 where there is no second launch) and their number, and restarts the
 * averages.  No reference counterpart (profiling hook). */
int wf_set_kernel_timing(WfHandle h, int32_t enabled);
int wf_get_kernel_timing(WfHandle h, double* step_kernel_ms, double* resolve_kernel_ms, int32_t* calls);

const char* wf_last_error(void);
const char* wf_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WFCRL_B200_H */
