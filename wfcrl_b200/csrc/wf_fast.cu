// Tuned FP32 step kernel for sm_100a: ONE WARP PER ENVIRONMENT (CTA = 32 threads = one env / wind condition).
//
// Design (DESIGN.md section 5):
//  * the whole per-env solver state lives in shared memory: per rotor grid point the running sum of squared velocity
//    deficits (SOSFS) and the pair (v, w); per (turbine, lateral column) the running maximum of the wake-added
//    turbulence; the rotated coordinates as float-float pairs; the precomputed FP64 mask indices; a queue of target
//    ids.  13.1 KB per env at T = 80 -> 16 envs resident per SM; no block-level barrier anywhere (only __syncwarp).
//  * sequential solver over sources i.  Per source:
//      1. prologue: rotor sums by a butterfly over the 9 lanes that own the source's grid points, then the warp-uniform
//         scalar chain (Ct, induction, secondary steering, deflection / velocity-model scalars, yaw-added recovery)
//         evaluated redundantly by every lane -- no broadcast needed;
//      2. V sweep over ALL downstream targets, 10 turbines x 3 lateral grid columns per pass (30 of 32 lanes), each lane
//         doing the 3 vertical points of its column: the three vortex pairs (real + ground mirror), evaluated directly
//         (the FP64 kernels' per-pair vortex table measured slower here: DESIGN.md section 5), and the (v, w)
//         update; the same pass ballots a compacted queue of the targets that can see the velocity deficit;
//         a source at exactly zero yaw sheds no tip vortices and runs an instantiation with the wake-rotation pair only;
//      3. D sweep over the queue only: deflection, wake widths, Gaussian deficit, sum-of-squares update, overlap count
//         and wake-added turbulence.
//  * x-direction masks are NOT evaluated in floating point here: the geometry kernel (FP64) stores, per source, the
//    first target index at which each mask turns true (SURVEY 7.3), so the kernel is FP64-free.
//  * algebra legal in FP32 mode only (each changes results by <= ~1e-6 relative): exp(-(y^2+z^2)/eps^2) =
//    exp(-y^2/eps^2) * const_z; one reciprocal per vortex pair; uR/(U0+u0) = 1/2; mirror-vortex cores = 1;
//    self-induced vortex velocities and the secondary-steering integrals as per-model constants; sum of squares instead
//    of a hypot chain; deficit contributions below exp(-5.5^2/2) dropped.
//  * BAKED instantiation: the per-model constants are compile-time literals generated at build time (wf_fast_baked.inc)
//    and used as instruction immediates; the generic instantiation reads them from kernel parameters / a shared-memory
//    float4 block.
//
// Algorithm: SURVEY.md Appendix A; reference call sites wfcrl/interface.py:557-586, 622-648; env semantics
// wfcrl/mdp.py:273-319, wfcrl/simple_env.py:58-96, wfcrl/multiagent_env.py:198-249, wfcrl/rewards.py:16-46.
#include "wf_device.cuh"
#include "wf_reset_device.cuh"
#include "wf_fast_baked.inc"

namespace {

// model constant `name`: a compile-time literal in the specialised (BAKED) instantiation, a kernel parameter otherwise
#define KC(name) (BAKED ? WfBaked::name : fc.name)


constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kDeg = 57.29577951308232f;
constexpr float kRad = 0.017453292519943295f;
constexpr float kNumEpsF = 0.001f;
constexpr int kTurbPerPass = 10;
constexpr int kMaxEvt = 8;  // ambiguous-decision records kept per env; more than that flags the env outright

__device__ __forceinline__ float frcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fsqrt(float x) { float y; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fex2(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float flg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fclamp(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

// piecewise-linear table lookup (np.interp + scipy fill values), warp-uniform or per-lane x
__device__ __forceinline__ float interp_f(const WfFastConst& fc, const float* __restrict__ fp, float x, float left,
                                          float right) {
    const int n = fc.table_len;
    const float x0 = fc.tab_ws[0], xn = fc.tab_ws[n - 1];
    if (x < x0) return left;
    if (x > xn) return right;
    int bkt = (int)((x - x0) * fc.coarse_scale);
    bkt = min(bkt, fc.coarse_len - 1);
    int idx = fc.coarse[bkt];
    while (idx + 1 < n - 1 && fc.tab_ws[idx + 1] <= x) ++idx;
    const float xa = fc.tab_ws[idx], fa = fp[idx];
    const float slope = (fp[idx + 1] - fa) * frcp(fc.tab_ws[idx + 1] - xa);
    return fmaf(slope, x - xa, fa);
}

struct SmemView {
    float* wsq;               // [9T] per rotor point, q = 9 t + 3 j + k: running sum of squared deficits
    float2* vw;               // [9T] (v, w) per rotor point (8-byte pairs: one LDS.64 / STS.64 per point)
    float2 *xhl, *yhl;        // [T]
    float *tia;               // [3T] running max of the wake-added TI per (turbine, lateral column)
    float *cyaw, *syaw, *yawr;  // [T] cos / sin / radians of the yaw (sorted order)
    float *tifin;             // [T] final rotor-mean TI
    float *ynew;              // [T] new yaw, degrees, ORIGINAL order
    uchar4* idx;              // [T]
    unsigned char* ordr;      // [T]
    unsigned char* queue;     // [T] targets whose rotor can see source i's velocity deficit (compacted per source)
    float4* cblk;             // [12] per-model vortex constants, 4 float4 per vertical index k (LDS.128 broadcast)
    float* evt_ta;            // [kMaxEvt] upper wake-added TI of an ambiguous overlap count (see the D sweep)
    uchar2* evt_tj;           // [kMaxEvt] its (target, lateral column)
};

__host__ __device__ inline size_t fast_smem_bytes(int T) {
    size_t n = 12 * 16;          // cblk
    n += (size_t)kMaxEvt * 4 + 16;  // evt_ta, evt_tj
    n += (size_t)3 * 9 * T * 4;  // wsq, v, w
    n += (size_t)2 * T * 8;      // xhl, yhl
    n += (size_t)3 * T * 4;      // tia
    n += (size_t)5 * T * 4;      // cyaw, syaw, yawr, tifin, ynew
    n += (size_t)T * 4;          // idx
    n += (size_t)((T + 15) / 16 * 16);  // ordr
    n += (size_t)((T + 15) / 16 * 16);  // queue
    return (n + 15) / 16 * 16;
}

__device__ __forceinline__ SmemView carve(unsigned char* base, int T) {
    SmemView s;
    s.cblk = (float4*)base;
    s.evt_ta = (float*)(base + 12 * 16);
    s.evt_tj = (uchar2*)(base + 12 * 16 + kMaxEvt * 4);
    float2* f2 = (float2*)(base + 12 * 16 + kMaxEvt * 4 + 16);
    s.xhl = f2;
    s.yhl = f2 + T;
    s.vw = f2 + 2 * T;  // 8-byte aligned for every T
    float* f = (float*)(f2 + 2 * T + 9 * T);
    s.wsq = f; f += 9 * T;
    s.tia = f; f += 3 * T;
    s.cyaw = f; f += T;
    s.syaw = f; f += T;
    s.yawr = f; f += T;
    s.tifin = f; f += T;
    s.ynew = f; f += T;
    s.idx = (uchar4*)f; f += T;
    s.ordr = (unsigned char*)f;
    s.queue = s.ordr + (T + 15) / 16 * 16;
    return s;
}

struct wf_true_tag { static constexpr bool value = true; };
struct wf_false_tag { static constexpr bool value = false; };

// generic instantiation: 12 is a lower bound for the register allocator; 16 envs per SM are reached
// EVAL (wf_evaluate_yaw): CTA c solves candidate c of env c / K in interface mode with the yaw row c of `yaw_cmd`, writes power
// row c of `out.power` and nothing else, and hands a flagged candidate to the evaluation fix list (wf_device.cuh: WfEvalArgs)
// EVAL + ACT (wf_evaluate_actions): CTA c runs env b = c / K's step with action row c in the run-time mode (env) of the
// step -- transition, solve, epilogue and reward -- against b's state, which it reads and never writes; every output goes
// to row c.  A flagged candidate leaves its transitioned yaw in ev.yaw row c for the re-solve.
// EVAL + ACT + ROLL (wf_evaluate_rollouts, H > 1): CTA c = row (b*K + k)*H + h runs step h of candidate k's action sequence
// on env b: the transitions of steps 0..h-1 (wf_replay, action rows c - h .. c - 1), then step h as above.  A separate
// instantiation, so that at H = 1 (h = 0 a compile-time constant) the action kernel is the one it was before rollouts.
// Unlike the FP64 kernels, this kernel keeps yaw evaluation an instantiation of its own (EVAL without ACT), with the mode a
// compile-time constant: with the env-mode epilogue (wind direction, loads, reward) compiled in, FP32 yaw evaluation ran
// 1-3 % slower (DESIGN.md section 5b)
template <bool BAKED, bool EVAL = false, bool ACT = false, bool ROLL = false>
__global__ void __launch_bounds__(32, BAKED ? 16 : 12)
wf_step_fast_kernel(const int mode_, const int env_begin, const WfModel m, const __grid_constant__ WfFastConst fc,
                    const WfState s, const uint8_t* __restrict__ mask, const float* __restrict__ action,
                    const double* __restrict__ yaw_cmd, const WfStepOut out, const WfEvalArgs ev) {
    int b, h = 0;  // h: step of the row in its candidate's sequence (0 but for rollouts)
    if constexpr (ROLL) { b = blockIdx.x / (ev.K * ev.H); h = blockIdx.x % ev.H; }
    else if constexpr (EVAL) b = blockIdx.x / ev.K;
    else b = blockIdx.x + env_begin;
    const int mode = (EVAL && !ACT) ? (int)WF_MODE_INTERFACE : mode_;
    if (mask && !mask[b]) return;
    const int T = m.T;
    const int lane = threadIdx.x;
    const size_t row = (size_t)b * T;
    const size_t orow = EVAL ? (size_t)blockIdx.x * T : row;  // row of the yaw command / action and of the outputs
    if (ROLL && h > 0) {  // a row after its candidate's truncating step (num_iter + h' + 1 == max_iter, h' < h) is not solved
        const int h_trunc = m.max_iter - s.num_iter[b] - 1;
        if (h_trunc >= 0 && h > h_trunc) { wf_zero_eval_row<float>(out, ev.amb, blockIdx.x, T, lane); return; }
    }
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SmemView sm = carve(smem_raw, T);  // sized by T: every env of the handle reserves the same shared memory
    // the env's turbine count: the one loop bound below.  Columns n..T-1 of its rows are padding (wf_device.cuh)
    const int n = s.turbine_count[b];

    // ---- env prologue on the ORIGINAL turbine order (mdp.py:291-319, simple_env.py:64-72) -------------------------
    int nm = 0;
    if (mode == WF_MODE_ENV) nm = s.num_moves[b] + 1;
    for (int tt = lane; tt < n; tt += 32) {
        float ynew;
        if (mode == WF_MODE_ENV) {
            float a = action[orow + tt];
            float acc = s.acc[row + tt];
            float acc_c = (m.multi_agent && tt != n - 1) ? s.acc_prev[row + tt] : acc;
            float y_h = 0.f;  // a rollout row: the yaw after steps 0..h-1 of its sequence (action rows c - h .. c - 1)
            if (ROLL && h > 0)
                y_h = wf_replay(m, action, orow - (size_t)h * T, T, tt, m.multi_agent && tt != n - 1, nm, h, acc, acc_c,
                                (float)s.yaw[row + tt]);
            a = wf_applied_action(m, a, acc_c, nm + h);
            ynew = wf_new_yaw(m, (ROLL && h > 0) ? y_h : (float)s.yaw[row + tt], a);
            if (!ACT) {
                s.acc_prev[row + tt] = acc;
                s.acc[row + tt] = __fadd_rn(acc, fabsf(a));
                s.yaw[row + tt] = (double)ynew;
            }
        } else if (mode == WF_MODE_INTERFACE && yaw_cmd) {
            const double y = yaw_cmd[orow + tt];
            if (!EVAL) s.yaw[row + tt] = y;
            ynew = (float)y;
        } else {
            ynew = (float)s.yaw[row + tt];
        }
        sm.ynew[tt] = ynew;
        sm.xhl[tt] = s.xhl[row + tt];
        sm.yhl[tt] = s.yhl[row + tt];
        sm.idx[tt] = s.idx[row + tt];
        sm.ordr[tt] = (unsigned char)s.order[row + tt];
    }
    if (lane < 12) sm.cblk[lane] = make_float4(fc.cblk[4 * lane], fc.cblk[4 * lane + 1], fc.cblk[4 * lane + 2], fc.cblk[4 * lane + 3]);
    for (int q = lane; q < 9 * n; q += 32) { sm.wsq[q] = 0.f; sm.vw[q] = make_float2(0.f, 0.f); }
    for (int q = lane; q < 3 * n; q += 32) sm.tia[q] = 0.f;
    __syncwarp();
    for (int tt = lane; tt < n; tt += 32) {
        const float yr = sm.ynew[sm.ordr[tt]] * kRad;
        float sy, cy;
        sincosf(yr, &sy, &cy);
        sm.yawr[tt] = yr;
        sm.cyaw[tt] = cy;
        sm.syaw[tt] = sy;
    }
    // per-env constants (warp-uniform registers)
    const double ws_d = s.ws[b], wd_d = s.wd[b];
    const float ws = (float)ws_d;
    const float I0 = (float)s.ti_amb[b];
    const float I02 = I0 * I0;
    const float I0p = __powf(I0, fc.ch_init);
    const float U0a = ws * fc.ratio[0], U0b = ws * fc.ratio[1], U0c = ws * fc.ratio[2];
    const float D = KC(D);
    __syncwarp();

    // lane -> (turbine slot g in the pass, lateral column j); each lane owns the 3 vertical points k of its column
    const int g = lane / 3, j = lane - 3 * g;
    const bool lane_ok = lane < 3 * kTurbPerPass;
    const float offj = (j == 0) ? fc.offj[0] : ((j == 1) ? fc.offj[1] : fc.offj[2]);
    // prologue mapping: lanes 0..8 (mirrored in 16..24) own rotor point pl of the SOURCE turbine
    const int pl = lane & 15;
    const bool pv = pl < 9;
    const int plc = pv ? pl : 0;
    const float U0p = (plc % 3 == 0) ? U0a : ((plc % 3 == 1) ? U0b : U0c);
    const float cvl0 = fc.cv[0][plc], cvl1 = fc.cv[1][plc], cvl2 = fc.cv[2][plc];
    const float cwl0 = fc.cw[0][plc], cwl1 = fc.cw[1][plc], cwl2 = fc.cw[2][plc];
    const float c_dec = KC(eps2) * KC(inv_2pi);
    const float c_e = -KC(inv_eps2) * kLog2e;
    const float c_ek = -(0.5f * kLog2e) * (BAKED ? WfBaked::dz2_0 : fc.dz2[0]);
    const float eps2 = KC(eps2);
    // Guard band of the ONE floating-point decision that makes the solve discontinuous: a rotor point counts towards the
    // wake overlap when deficit * U0 > 0.05 m/s.  Counts are kept for both ends of the band; where they differ the event
    // is recorded and judged when the target's turbulence intensity is final (see the source prologue).
    const bool strict = m.amb_eps > 0.f;  // flag ill-conditioned solves for the FP64 re-solve (amb_eps = 0: relaxed handle)
    const float thr_lo = 0.05f * (1.f - m.amb_eps), thr_hi = 0.05f * (1.f + m.amb_eps);
    const double two_D_d = 2.0 * m.D;
    int nevt = 0;
    bool flagged = false;

    // ---- sequential solver over sources (SURVEY A.4-A.8) -------------------------------------------------------------
    for (int i = 0; i < n; ++i) {
        // ===== source prologue =====
        // rotor sums over the source's 9 points: one point per lane, butterfly over 16-lane halves -> uniform values
        float su3, sv, sw, vq, wwq;
        {
            const float wq = sm.wsq[9 * i + plc];
            const float2 vw0 = sm.vw[9 * i + plc];
            vq = vw0.x;
            wwq = vw0.y;
            const float u = U0p - fsqrt(wq);
            su3 = pv ? u * u * u : 0.f;
            sv = pv ? vq : 0.f;
            sw = pv ? wwq : 0.f;
#pragma unroll
            for (int sft = 8; sft > 0; sft >>= 1) {
                su3 += __shfl_xor_sync(0xffffffffu, su3, sft);
                sv += __shfl_xor_sync(0xffffffffu, sv, sft);
                sw += __shfl_xor_sync(0xffffffffu, sw, sft);
            }
        }
        const float avg = cbrtf(su3 * (1.f / 9.f));
        const float ct_raw = fclamp(interp_f(fc, fc.tab_ct, avg, 0.0001f, 0.9999f), 0.0001f, 0.9999f);
        const float cy = sm.cyaw[i], sy = sm.syaw[i], yr = sm.yawr[i];
        const float ct = ct_raw * cy;
        const float s1c = fsqrt(1.f - ct * cy);
        const float a = 0.5f * frcp(cy) * (1.f - s1c);
        const float Gtop0 = KC(c_top) * ws * ct, Gbot0 = KC(c_bot) * ws * ct;
        const float Gwr = KC(c_wr) * (a - a * a) * avg;
        const float Gt = sy * cy * Gtop0, Gb = -(sy * cy * Gbot0);

        // A.5 secondary steering through the per-model grid integrals
        float val = 2.f * (sv * (1.f / 9.f) - Gwr * KC(a_core)) * frcp(Gtop0 * KC(a_top) - Gbot0 * KC(a_bot));
        val = fclamp(val, -1.f, 1.f);
        const float g_rad = -(yr + 0.5f * asinf(val));  // minus the effective yaw, radians
        const float cg = __cosf(g_rad);

        // A.6 deflection scalars
        const float sq1ct = fsqrt(1.f - ct);
        const float sqcg = fsqrt(1.f - ct * cg);
        const float sz0d = 0.5f * D * fsqrt((1.f + sqcg) * frcp(2.f * (1.f + sq1ct)));
        const float sy0d = sz0d * cg;
        const float C0 = 1.f - sq1ct;
        const float M0 = C0 * (2.f - C0);
        const float E0 = C0 * C0 - KC(e3_112) * C0 + KC(e3_13);
        const float th = KC(dm03) * g_rad * frcp(cg) * (1.f - sqcg);
        const float sM0 = fsqrt(M0);
        const float tan_th = __sinf(th) * frcp(__cosf(th));
        const float Kc = th * E0 * (1.f / 5.2f) * fsqrt(sy0d * sz0d * frcp(M0));
        const float A_ln = (1.6f + sM0) * frcp(1.6f - sM0);
        const float inv_s0d = frcp(sy0d * sz0d);

        // This turbine's wake-added TI is final now (all its sources are upstream).  An ambiguous overlap count is harmless
        // when even its upper value stays below the running maximum; otherwise the env is flagged for the FP64 re-solve.
        for (int e = 0; e < min(nevt, kMaxEvt); ++e) {
            const uchar2 tj = sm.evt_tj[e];
            if ((int)tj.x == i && sm.evt_ta[e] > sm.tia[3 * i + tj.y]) flagged = true;
        }
        // TI of the source per lateral column before the yaw-added-recovery update
        const float ta0 = sm.tia[3 * i], ta1 = sm.tia[3 * i + 1], ta2 = sm.tia[3 * i + 2];
        const float tp0 = fsqrt(fmaf(ta0, ta0, I02)), tp1 = fsqrt(fmaf(ta1, ta1, I02)), tp2 = fsqrt(fmaf(ta2, ta2, I02));
        const float tpre = (j == 0) ? tp0 : ((j == 1) ? tp1 : tp2);
        const float beta_term = KC(beta2) * (1.f - sq1ct);
        const float x0d = D * cg * (1.f + sqcg) * frcp(1.4142135623730951f * fmaf(KC(alpha4), tpre, beta_term));
        const float kyd = fmaf(KC(ka), tpre, KC(kb));
        const float inv_x0d = frcp(x0d);
        const float delta0 = tan_th * x0d;
        const float Kck = Kc * frcp(kyd);

        // own transverse velocities (A.7 on the source's own grid) + yaw-added recovery (in-place TI update)
        const uchar4 ix = sm.idx[i];
        const bool self_on = (int)ix.x <= i;  // X_i - x_i >= 0 (warp-uniform)
        float sumV = sv, sumW = sw;
        if (self_on) {
            sumV += Gt * (BAKED ? WfBaked::sv0 : fc.sv[0]) + Gb * (BAKED ? WfBaked::sv1 : fc.sv[1]) +
                    Gwr * (BAKED ? WfBaked::sv2 : fc.sv[2]);
            const float Vs = Gt * cvl0 + Gb * cvl1 + Gwr * cvl2;
            const float Ws = fmaxf(Gt * cwl0 + Gb * cwl1 + Gwr * cwl2, 0.f);
            float rw = pv ? Ws : 0.f;
#pragma unroll
            for (int sft = 8; sft > 0; sft >>= 1) rw += __shfl_xor_sync(0xffffffffu, rw, sft);
            sumW += rw;
            __syncwarp();  // the mirrored lanes 16..24 have read this turbine's (v, w) above
            if (lane < 9) sm.vw[9 * i + lane] = make_float2(vq + Vs, wwq + Ws);
        }
        const float aI = avg * tp0;
        const float kk2 = 3.f * aI * aI;  // u_term^2 = 2 k = 2 (avg I)^2 / (2/3)
        const float v_term = sumV * (1.f / 9.f), w_term = sumW * (1.f / 9.f);
        const float k_total = 0.5f * (kk2 + v_term * v_term + w_term * w_term);
        const float I_mix = fsqrt((2.f / 3.f) * k_total) * frcp(avg) - tp0;
        const float tq0 = fmaf(2.f, I_mix, tp0), tq1 = fmaf(2.f, I_mix, tp1), tq2 = fmaf(2.f, I_mix, tp2);
        if (lane == 0) sm.tifin[i] = (tq0 + tq1 + tq2) * (1.f / 3.f);
        const float tpost = (j == 0) ? tq0 : ((j == 1) ? tq1 : tq2);

        // A.8 velocity-model scalars with the updated TI (cos(-yaw) = cy ; sigma_z0 = D / (2 sqrt 2) exactly)
        const float x0v = D * cy * (1.f + sq1ct) * frcp(1.4142135623730951f * fmaf(KC(alpha4), tpost, beta_term));
        const float kyv = fmaf(KC(ka), tpost, KC(kb));
        const float inv_x0v = frcp(x0v);
        const float sz0v = KC(near_c) * (0.5f / 0.501f);  // 0.5 D sqrt(1/2)
        const float sy0v = sz0v * cy;
        const float near_s = KC(near_c) * fsqrt(ct);
        const float ctc = ct * cy * KC(d2_8);
        const float watK = KC(ch_const) * __powf(a, KC(ch_ai)) * I0p;

        const int lo = ix.x, near_i = ix.y, gt0_i = ix.z, end15 = ix.w;
        const float2 xi = sm.xhl[i], yi = sm.yhl[i];

        // Conservative lateral reach of this source's velocity deficit at column j: the Gaussian factor is below
        // exp(-kCut^2/2) (2.7e-7) when |Y - y_i| > kCut * sigma_y_bound(dx) + |deflection|_max.  sigma_y <= kyv*dx +
        // max(sigma_y0, near-wake width); |deflection| <= |delta0| + |Kc/ky| * ln(A_ln) (+ |ad + bd dx|).
        constexpr float kCut = 5.5f;
        const float reach1 = kCut * kyv;
        const float reach0 = fmaf(kCut, fmaxf(near_s, sy0v), fabsf(delta0) + fabsf(Kck) * (flg2(A_ln) * kLn2));

        // ===== V sweep: transverse velocities on ALL downstream targets, 10 turbines x 3 lateral columns per pass;
        //       builds the compacted queue of targets that can see the velocity deficit =====
        // A source at exactly zero yaw sheds no tip vortices (Gt = Gb = 0): the sweep then evaluates the wake-rotation
        // pair only -- same bits, 45 % of the work.  Warp-uniform choice, one instantiation of the loop per case.
        int qn = 0;
        auto v_pass = [&](auto yawed_tag, const int t0) {
            constexpr bool YAWED = decltype(yawed_tag)::value;
            const int tr = t0 + g;
            const bool active = lane_ok && tr < n && tr != i;
            const int t = min(tr, n - 1);  // inactive lanes compute on a valid turbine; only their stores are masked
            const float2 xt = sm.xhl[t], yt = sm.yhl[t];
            const float dx = (xt.x - xi.x) + (xt.y - xi.y);
            const float dyc = ((yt.x - yi.x) + (yt.y - yi.y)) + offj;

            const bool need = active && (t >= near_i) &&
                              (fabsf(dyc) < fmaf(reach1, dx, reach0) + fabsf(fmaf(KC(bd), dx, KC(ad))));
            const unsigned nb = __ballot_sync(0xffffffffu, need);
            const bool leader = (j == 0) && active && (((nb >> (3 * g)) & 7u) != 0u);
            const unsigned lb = __ballot_sync(0xffffffffu, leader);
            if (leader) sm.queue[qn + __popc(lb & ((1u << lane) - 1u))] = (unsigned char)t;
            qn += __popc(lb);

            // transverse velocities of the 3 vortex pairs (real + ground mirror) at the 3 vertical points
            const float yL = dyc + kNumEpsF;
            const float q = yL * yL;
            const float E = fex2(q * c_e);
            float Vk[3], Wk[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                float4 ca, cb, cc, cd;
                if (BAKED) {  // immediates
                    ca = make_float4(WfBaked::cblk(16 * k), WfBaked::cblk(16 * k + 1), WfBaked::cblk(16 * k + 2), WfBaked::cblk(16 * k + 3));
                    cb = make_float4(WfBaked::cblk(16 * k + 4), WfBaked::cblk(16 * k + 5), WfBaked::cblk(16 * k + 6), WfBaked::cblk(16 * k + 7));
                    cc = make_float4(WfBaked::cblk(16 * k + 8), WfBaked::cblk(16 * k + 9), WfBaked::cblk(16 * k + 10), WfBaked::cblk(16 * k + 11));
                    cd = make_float4(WfBaked::cblk(16 * k + 12), WfBaked::cblk(16 * k + 13), WfBaked::cblk(16 * k + 14), WfBaked::cblk(16 * k + 15));
                } else {      // LDS.128 broadcast from the shared-memory block
                    ca = sm.cblk[4 * k]; cb = sm.cblk[4 * k + 1]; cc = sm.cblk[4 * k + 2]; cd = sm.cblk[4 * k + 3];
                }
                const float r4 = q + cb.x, r5 = q + cb.y;
                const float g4 = Gwr * frcp(r4 * r5);
                const float X4 = fmaf(-E, cc.x, 1.f) * r5;
                const float NV4 = fmaf(cd.y, X4, -(cd.z * r4));
                float SV, SW;
                if (YAWED) {
                    const float r0 = q + ca.x, r2 = q + ca.y, r1 = q + ca.z, r3 = q + ca.w;
                    const float g0 = Gt * frcp(r0 * r2), g1 = Gb * frcp(r1 * r3);
                    const float X0 = fmaf(-E, cb.z, 1.f) * r2, X1 = fmaf(-E, cb.w, 1.f) * r3;
                    const float NV0 = fmaf(cc.y, X0, -(cc.z * r0)), NV1 = fmaf(cc.w, X1, -(cd.x * r1));
                    SV = fmaf(g4, NV4, fmaf(g1, NV1, g0 * NV0));
                    SW = fmaf(g4, X4 - r4, fmaf(g1, X1 - r1, g0 * (X0 - r0)));
                } else {
                    SV = g4 * NV4;
                    SW = g4 * (X4 - r4);
                }
                const float dec = c_dec * frcp(fmaf(cd.w, dx, eps2));
                Vk[k] = SV * dec;
                Wk[k] = fmaxf(SW * (-yL * dec), 0.f);
            }
            if (active) {
                const int qb = 9 * t + 3 * j;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float2 o = sm.vw[qb + k];
                    sm.vw[qb + k] = make_float2(o.x + Vk[k], o.y + Wk[k]);
                }
            }
        };
        // two passes in flight per warp (ILP): +3.5 %; unrolling the D sweep and 3-pass V unrolling measured slower
        if (sy != 0.f) {
#pragma unroll 2
            for (int t0 = lo; t0 < n; t0 += kTurbPerPass) v_pass(wf_true_tag{}, t0);
        } else {
#pragma unroll 2
            for (int t0 = lo; t0 < n; t0 += kTurbPerPass) v_pass(wf_false_tag{}, t0);
        }
        __syncwarp();

        // ===== D sweep: deflection + Gaussian deficit + wake-added TI, only on the queued targets =====
#pragma unroll 1
        for (int q0 = 0; q0 < qn; q0 += kTurbPerPass) {
            const int e = q0 + g;
            const bool active = lane_ok && e < qn;
            const int t = sm.queue[min(e, qn - 1)];
            const float2 xt = sm.xhl[t], yt = sm.yhl[t];
            const float dx = (xt.x - xi.x) + (xt.y - xi.y);
            const float dyc = ((yt.x - yi.x) + (yt.y - yi.y)) + offj;
            const float lin = fmaf(KC(bd), dx, KC(ad));

            // -- deflection of source i's wake at this column (both branches, select)
            float defl;
            {
                const float dd = dx - x0d;
                const float sgy = fmaf(kyd, dd, sy0d), sgz = fmaf(kyd, dd, sz0d);
                const float sq = fsqrt(sgy * sgz * inv_s0d);
                const float L = flg2(A_ln * fmaf(1.6f, sq, -sM0) * frcp(fmaf(1.6f, sq, sM0))) * kLn2;
                const float d_far = fmaf(Kck, L, delta0) + lin;
                const float d_near = fmaf(dx * inv_x0d, delta0, lin);
                defl = (dx <= x0d) ? d_near : d_far;
            }
            // -- Gaussian deficit: widths and the lateral factor once per column (queued targets have t >= near_i)
            float base, ek;
            {
                const bool far = dx >= x0v;
                const float dd = dx - x0v;
                const float up = dx * inv_x0v, down = 1.f - up;
                const float sgy = far ? fmaf(kyv, dd, sy0v) : fmaf(down, near_s, up * sy0v);
                const float sgz = far ? fmaf(kyv, dd, sz0v) : fmaf(down, near_s, up * sz0v);
                const float ry = frcp(sgy), rz = frcp(sgz);
                const float dy = (dyc - defl) * ry;
                const float dcl = fclamp(fmaf(-ctc * ry, rz, 1.f), 0.f, 1.f);
                const float C = 1.f - fsqrt(dcl);
                base = C * fex2((-0.5f * kLog2e) * dy * dy);
                ek = fex2(c_ek * rz * rz);
            }
            const float be = base * ek;
            const float dU0 = be * U0a, dU1 = base * U0b, dU2 = be * U0c;
            int c = 0;  // points over the threshold: low byte with the upper end of the guard band, next byte with the lower
            if (active) {
                c = ((dU0 > thr_hi) + (dU1 > thr_hi) + (dU2 > thr_hi)) |
                    (((dU0 > thr_lo) + (dU1 > thr_lo) + (dU2 > thr_lo)) << 8);
                const int qb = 9 * t + 3 * j;
                sm.wsq[qb] = fmaf(dU0, dU0, sm.wsq[qb]);
                sm.wsq[qb + 1] = fmaf(dU1, dU1, sm.wsq[qb + 1]);
                sm.wsq[qb + 2] = fmaf(dU2, dU2, sm.wsq[qb + 2]);
            }
            // -- Crespo-Hernandez wake-added TI: overlap = (#points with deficit*U0 > 0.05) / 9 over the 3 columns
            const int gb = 3 * g;
            const int c_tot = __shfl_sync(0xffffffffu, c, gb & 31) + __shfl_sync(0xffffffffu, c, (gb + 1) & 31) +
                              __shfl_sync(0xffffffffu, c, (gb + 2) & 31);
            const int c_lo = c_tot & 0xff, c_hi = c_tot >> 8;
            bool ambiguous = false;
            float ta_hi = 0.f;
            if (active && c_hi > 0 && t >= gt0_i && t < end15) {
                const float ady = fabsf(dyc);
                bool in_win = ady < KC(two_D);
                if (fabsf(ady - KC(two_D)) < 2e-3f) {  // lateral window |Y - y_i| < 2 D decided on the float-float positions
                    const double d = (((double)yt.x - (double)yi.x) + ((double)yt.y - (double)yi.y)) + (double)offj;
                    in_win = fabs(d) < two_D_d;
                    if (strict && fabs(fabs(d) - two_D_d) < 1e-7) flagged = true;
                }
                if (in_win) {
                    const float wat = watK * __powf(dx * KC(inv_D), KC(ch_down));
                    if (c_lo > 0) sm.tia[3 * t + j] = fmaxf(sm.tia[3 * t + j], (float)c_lo * (1.f / 9.f) * wat);
                    ambiguous = c_hi != c_lo;
                    ta_hi = (float)c_hi * (1.f / 9.f) * wat;
                }
            }
            const unsigned ab = __ballot_sync(0xffffffffu, ambiguous);
            if (ab) {  // rare
                const int slot = nevt + __popc(ab & ((1u << lane) - 1u));
                if (ambiguous) {
                    if (slot < kMaxEvt) { sm.evt_ta[slot] = ta_hi; sm.evt_tj[slot] = make_uchar2((unsigned char)t, (unsigned char)j); }
                    else flagged = true;
                }
                nevt += __popc(ab);
            }
        }
        __syncwarp();
    }

    // ---- epilogue: lane = sorted turbine; measures, power, loads (interface.py:565-577, 622-648) ------------------
    const bool env = (mode != WF_MODE_INTERFACE);
    const float wd = (float)wd_d;
    float rsum_p = 0.f, rsum_l = 0.f;
    for (int tt = lane; tt < n; tt += 32) {
        float u[9], vv[9], ww[9];
        float su = 0.f, su3 = 0.f, svv = 0.f, sww = 0.f, sdd = 0.f;
#pragma unroll
        for (int p = 0; p < 9; ++p) {
            const float U0k = (p % 3 == 0) ? U0a : ((p % 3 == 1) ? U0b : U0c);
            u[p] = U0k - fsqrt(sm.wsq[9 * tt + p]);
            const float2 vwp = sm.vw[9 * tt + p];
            vv[p] = vwp.x;
            ww[p] = vwp.y;
            su += u[p];
            su3 = fmaf(u[p] * u[p], u[p], su3);
            svv += vv[p];
            sww += ww[p];
            sdd += atan2f(vv[p], u[p]);
        }
        const float avg = cbrtf(su3 * (1.f / 9.f));
        const float mu = su * (1.f / 9.f), mv = svv * (1.f / 9.f), mw = sww * (1.f / 9.f);
        float qu = 0.f, qv = 0.f, qw = 0.f;
#pragma unroll
        for (int p = 0; p < 9; ++p) {
            qu = fmaf(u[p] - mu, u[p] - mu, qu);
            qv = fmaf(vv[p] - mv, vv[p] - mv, qv);
            qw = fmaf(ww[p] - mw, ww[p] - mw, qw);
        }
        const float veff = fc.rho_fac * avg * __powf(sm.cyaw[tt], fc.pP3);
        const float pw = interp_f(fc, fc.tab_pw, veff, 0.f, 0.f) * fc.ref_rho;  // [W]
        if (strict) {
            // Where the power curve is steep relative to the power itself (the foot of the table above cut-in, the cliff
            // at cut-out), a rotor speed good to ~1e-5 cannot give the power to 1e-4: hand the env to the FP64 re-solve.
            constexpr float kVelEps = 1.2e-5f;
            const float pm = interp_f(fc, fc.tab_pw, veff * (1.f - kVelEps), 0.f, 0.f) * fc.ref_rho;
            const float pp = interp_f(fc, fc.tab_pw, veff * (1.f + kVelEps), 0.f, 0.f) * fc.ref_rho;
            if (fmaxf(fabsf(pp - pw), fabsf(pw - pm)) > 1e-4f * fmaxf(pw, 1.f)) flagged = true;
        }
        float wsl = avg;
        float wdl = wd - kDeg * sdd * (1.f / 9.f);
        float loads[4] = {sm.tifin[tt], fsqrt(qu * (1.f / 9.f)), fsqrt(qv * (1.f / 9.f)), fsqrt(qw * (1.f / 9.f))};
        float p_out;
        if (env) {
            p_out = pw * 1e-6f;
            rsum_p += p_out;
            rsum_l += fabsf(loads[0]) + fabsf(loads[1]) + fabsf(loads[2]) + fabsf(loads[3]);
        } else {
            p_out = pw;
#pragma unroll
            for (int q = 0; q < 4; ++q) loads[q] *= 1e7f;
        }
        const int orig = sm.ordr[tt];
        if (EVAL && !ACT) {  // the power is written once the candidate is known not to be flagged (below)
            sm.tifin[tt] = p_out;
            continue;
        }
        float yv = sm.ynew[orig];
        if (mode == WF_MODE_WARMUP) {  // start state is clipped to the observation space (mdp.py:263-266)
            wsl = fclamp(wsl, 3.f, 28.f);
            wdl = fclamp(wdl, 0.f, 360.f);
            yv = fclamp(yv, m.yaw_lo_f, m.yaw_hi_f);
        }
        const size_t o = orow + orig;
        if (out.yaw) ((float*)out.yaw)[o] = yv;
        if (out.wind_speed) ((float*)out.wind_speed)[o] = wsl;
        if (out.wind_direction) ((float*)out.wind_direction)[o] = wdl;
        if (out.power) ((float*)out.power)[o] = p_out;
        if (out.load) ((float4*)out.load)[o] = make_float4(loads[0], loads[1], loads[2], loads[3]);
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
        rsum_p += __shfl_xor_sync(0xffffffffu, rsum_p, sft);
        rsum_l += __shfl_xor_sync(0xffffffffu, rsum_l, sft);
    }
    const bool any_flag = __any_sync(0xffffffffu, flagged);
    if constexpr (EVAL && !ACT) {  // no state is written: the flag and the power row of the candidate only
        if (lane == 0 && ev.amb) ev.amb[blockIdx.x] = (uint8_t)any_flag;
        if (any_flag && strict) {  // re-solved in interface mode by wf_fixup64_eval_kernel, from the caller's yaw_cmd row
            if (lane == 0) ev.fix_list[atomicAdd(&ev.fix_count[0], 1)] = blockIdx.x;
            return;
        }
        float* const pw_out = (float*)out.power + orow;
        for (int tt = lane; tt < n; tt += 32) pw_out[sm.ordr[tt]] = sm.tifin[tt];
        for (int tt = n + lane; tt < T; tt += 32) pw_out[tt] = 0.f;
        return;
    }
    if constexpr (ACT) {
        if (lane == 0 && ev.amb) ev.amb[blockIdx.x] = (uint8_t)any_flag;
        if (any_flag && strict) {  // re-solved in env mode by wf_fixup64_eval_kernel, from this transitioned yaw
            for (int tt = lane; tt < n; tt += 32) ev.yaw[orow + tt] = (double)sm.ynew[tt];
            if (lane == 0) ev.fix_list[atomicAdd(&ev.fix_count[0], 1)] = blockIdx.x;
            return;
        }
    } else if (lane == 0 && s.amb) {
        s.amb[b] = (uint8_t)any_flag;
    }
    if (!ACT && any_flag && strict) {
        // the FP64 re-solve (wf_fixup64_kernel, next launch on this stream) redoes this env from the committed yaw state and
        // commits the per-env epilogue state itself
        if (lane == 0) s.fix_list[atomicAdd(&s.fix_count[0], 1)] = b;
        return;
    }
    // the per-env outputs go to row ob; an evaluation commits none of the state below
    const int ob = ACT ? (int)blockIdx.x : b;
    int it = 0;
    if (lane == 0) {
        it = s.num_iter[b] + 1 + h;
        if (!ACT) s.num_iter[b] = it;
        if (out.truncated) out.truncated[ob] = (uint8_t)(it == m.max_iter);
        float fw0 = ws, fw1 = wd;
        if (mode == WF_MODE_WARMUP) { fw0 = fclamp(fw0, 3.f, 28.f); fw1 = fclamp(fw1, 0.f, 360.f); }
        if (out.freewind) ((float2*)out.freewind)[ob] = make_float2(fw0, fw1);
        if (mode == WF_MODE_ENV) {
            if (!ACT) s.num_moves[b] = nm;
            const float wn = h > 0 ? ws : (float)s.ws_norm[b];  // a step leaves ws_norm = ws for the next one
            const float invT = 1.f / (float)n;  // the mean over the env's own turbines
            float reward = rsum_p * 1e3f / (wn * wn * wn) * invT - fc.load_coef * rsum_l * (0.25f * invT);
            if (m.shaper == 1) {
                reward = (reward - fc.shaper_reference) / fc.shaper_reference;
            } else if (m.shaper == 2) {
                // a rollout keeps every row's unshaped reward, the reference of its next row; rows h >= 1 are shaped by
                // wf_launch_eval_step_pct (wf_fast64.cu: one pass for both precisions), which reads that reference
                if (ROLL && ev.rew) ev.rew[ob] = (double)reward;
                if (h == 0) {
                    const double ref = s.shaper_ref[b];
                    const float shaped = (ref == 0.0) ? 0.f : (float)(((double)reward - ref) / ref);
                    if (!ACT) s.shaper_ref[b] = (double)reward;
                    reward = shaped;
                }
            }
            if (!ACT && !isfinite(reward)) s.nonfinite[b] += 1;
            if (out.reward) ((float*)out.reward)[ob] = reward;
            if (!ACT) {
                wfreset::episode_account(s, b, (double)reward, it == m.max_iter);
                s.ws_norm[b] = ws_d;
            }
        }
    }
    // in-kernel auto-reset (wf_set_autoreset): the step that truncates also starts the env's next episode -- zero yaw /
    // accumulators / counters -- and marks the env for wf_autoreset_finish (wind draw + geometry + warm-up solve); the outputs written above remain the FINAL observation of the finished episode
    if (!ACT && mode == WF_MODE_ENV && m.autoreset && __shfl_sync(0xffffffffu, (int)(it == m.max_iter), 0)) {
        for (int tt = lane; tt < T; tt += 32) { s.yaw[row + tt] = 0.0; s.acc[row + tt] = 0.f; s.acc_prev[row + tt] = 0.f; }
        if (lane == 0) wfreset::autoreset_mark(s, b);
    }
    // padding columns n..T-1 of every per-turbine output read 0, whatever an earlier layout left there (a flagged env
    // returned above: the re-solve writes them); w = floats per turbine
    auto zero_padding = [&](void* p, const int w) {
        if (p)
#pragma unroll 1
            for (int q = n * w + lane; q < T * w; q += 32) ((float*)p)[orow * w + q] = 0.f;
    };
    zero_padding(out.yaw, 1);
    zero_padding(out.wind_speed, 1);
    zero_padding(out.wind_direction, 1);
    zero_padding(out.power, 1);
    zero_padding(out.load, 4);
}

}  // namespace

cudaError_t wf_configure_fast_kernels() {
    for (auto k : {wf_step_fast_kernel<true>, wf_step_fast_kernel<false>, wf_step_fast_kernel<true, true>,
                   wf_step_fast_kernel<false, true>, wf_step_fast_kernel<true, true, true>, wf_step_fast_kernel<false, true, true>,
                   wf_step_fast_kernel<true, true, true, true>, wf_step_fast_kernel<false, true, true, true>}) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

template <bool BAKED>
static cudaError_t launch_fast_t(int mode, const WfModel& m, const WfFastConst& fc, const WfState& s,
                                 const uint8_t* d_mask, const float* d_action, const double* d_yaw_cmd,
                                 const WfStepOut& out, int env_begin, int env_count, cudaStream_t stream) {
    wf_step_fast_kernel<BAKED><<<env_count, 32, fast_smem_bytes(m.T), stream>>>(mode, env_begin, m, fc, s, d_mask, d_action,
                                                                               d_yaw_cmd, out, WfEvalArgs{});
    return cudaGetLastError();
}

template <bool BAKED, bool ACT, bool ROLL = false>
static cudaError_t launch_eval_t(const WfModel& m, const WfFastConst& fc, const WfState& s, const WfEvalArgs& ev,
                                 const double* d_yaw, const float* d_action, const WfStepOut& out, cudaStream_t stream) {
    wf_step_fast_kernel<BAKED, true, ACT, ROLL><<<(unsigned)m.B * (unsigned)ev.K * (unsigned)ev.H, 32, fast_smem_bytes(m.T), stream>>>(
        ACT ? WF_MODE_ENV : WF_MODE_INTERFACE, 0, m, fc, s, nullptr, d_action, d_yaw, out, ev);
    return cudaGetLastError();
}

cudaError_t wf_launch_eval_fast(bool baked, const WfModel& m, const WfFastConst& fc, const WfState& s, const WfEvalArgs& ev,
                                const double* d_yaw, const float* d_action, const WfStepOut& out, cudaStream_t stream) {
    if (d_action && ev.H > 1)
        return baked ? launch_eval_t<true, true, true>(m, fc, s, ev, nullptr, d_action, out, stream)
                     : launch_eval_t<false, true, true>(m, fc, s, ev, nullptr, d_action, out, stream);
    if (d_action)
        return baked ? launch_eval_t<true, true>(m, fc, s, ev, nullptr, d_action, out, stream)
                     : launch_eval_t<false, true>(m, fc, s, ev, nullptr, d_action, out, stream);
    return baked ? launch_eval_t<true, false>(m, fc, s, ev, d_yaw, nullptr, out, stream)
                 : launch_eval_t<false, false>(m, fc, s, ev, d_yaw, nullptr, out, stream);
}

cudaError_t wf_launch_step_fast(int mode, bool baked, const WfModel& m, const WfFastConst& fc, const WfState& s,
                                const uint8_t* d_mask, const float* d_action, const double* d_yaw_cmd,
                                const WfStepOut& out, int env_begin, int env_count, cudaStream_t stream) {
    return baked ? launch_fast_t<true>(mode, m, fc, s, d_mask, d_action, d_yaw_cmd, out, env_begin, env_count, stream)
                 : launch_fast_t<false>(mode, m, fc, s, d_mask, d_action, d_yaw_cmd, out, env_begin, env_count, stream);
}

template <bool BAKED>
static cudaError_t attrs_fast_t(const WfModel& m, cudaFuncAttributes* attr, int* ctas_per_sm, int* threads, int* smem) {
    *threads = 32;
    *smem = (int)fast_smem_bytes(m.T);
    cudaError_t e = cudaFuncGetAttributes(attr, wf_step_fast_kernel<BAKED>);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, wf_step_fast_kernel<BAKED>, 32, *smem);
}

cudaError_t wf_step_fast_attributes(bool baked, const WfModel& m, cudaFuncAttributes* attr, int* ctas_per_sm, int* threads,
                                    int* smem) {
    return baked ? attrs_fast_t<true>(m, attr, ctas_per_sm, threads, smem) : attrs_fast_t<false>(m, attr, ctas_per_sm, threads, smem);
}
