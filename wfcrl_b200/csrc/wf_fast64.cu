// FP64 instantiations of the warp-per-env design: the bit-check mode at speed, and the re-solve of the envs a strict FP32
// launch flagged.  One template (solve_env64<W, OutT, FIX, GATHER>), three kernels:
//
//   wf_step_fast64_kernel<true>   one warp = one CTA = one env, GATHER form: the transverse velocities of a turbine are summed
//                                 from the target-major vortex-table rows when the turbine becomes the source (shared memory
//                                 15 KB per 80-turbine env, 128 registers -> 14-16 envs per SM);
//   wf_step_fast64_kernel<false>  the same warp-per-env solve in scatter form (V sweep over all downstream targets, compacted
//                                 deficit queue) for handles without a vortex table;
//   wf_fixup64_kernel<W>          W warps per env, built for latency: a chain warp evaluates the sources' scalar chains back to
//                                 back while W-1 worker warps apply the previous source to its targets (named barriers).
// and their candidate-evaluation forms wf_step_fast64_kernel<GATHER, true> and wf_fixup64_eval_kernel<W> (wf_evaluate_yaw in
// interface mode, wf_evaluate_actions in env mode).
//
// Everything is evaluated in double precision and every simplification of wf_fast.cu that would be visible at the 1e-9 level
// is dropped:
//   * positions are the FP64 rotated coordinates and the numpy-order means x_i, y_i of the geometry kernel;
//   * the ground-mirror vortices keep their exp(-r/eps^2) core factor;
//   * the deficit cut-off is 9.5 sigma (exp(-45) = 2.9e-20);
//   * x-direction masks come from the geometry kernel's FP64 index table (bit-exact, SURVEY 7.3).
// Algebra that only changes results at the rounding level (1e-16) is kept: exp(-(y^2+z^2)/eps^2) factorisation, paired
// reciprocals, uR/(U0+u0) = 1/2, per-model grid integrals, sum of squares instead of the hypot chain, running maximum of
// the wake-added TI, Newton-refined reciprocals / square roots / cube roots seeded in single precision.
// Parity vs the oracle: <= 1e-9 relative (tests/test_solve_parity_gpu.py, test_env_parity_gpu.py; measured max 1.1e-12).
//
// Algorithm: SURVEY.md Appendix A; reference call sites wfcrl/interface.py:557-586, 622-648; env semantics
// wfcrl/mdp.py:273-319, wfcrl/simple_env.py:58-96, wfcrl/multiagent_env.py:198-249, wfcrl/rewards.py:16-46.
#include "wf_device.cuh"
#include "wf_reset_device.cuh"

#include <math.h>

namespace {

constexpr double kPi = 3.141592653589793;
constexpr double kDeg = 180.0 / kPi;
constexpr double kRad = kPi / 180.0;
constexpr double kNumEps = 0.001;
constexpr int kTurbPerPass = 10;
constexpr int kSrcPar = 24;  // doubles per source handed from the chain warp to the worker warps (solve_env64, W > 1)

// pull the vortex-table rows of sorted source `i` into L2 ahead of their use (one bulk prefetch): the rows of its targets
// i+1 .. n-1 of an env of n turbines, in a table whose row strides are those of T
__device__ __forceinline__ void prefetch_rows64(const void* env_rows, int i, int T, int n, int lane, unsigned row_bytes) {
    if (i >= n - 1 || lane != 0) return;
    const char* p = (const char*)env_rows + ((size_t)i * T - (size_t)i * (i + 1) / 2) * row_bytes;
    const unsigned bytes = (unsigned)(n - 1 - i) * row_bytes;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// target-major table (gather kernel): the rows (j, t) of the table sources j < n_rows of sorted target `t` are contiguous
__device__ __forceinline__ void prefetch_target_rows64(const void* env_rows, int t, int n_rows, int lane) {
    if (n_rows <= 0 || lane != 0) return;
    const char* p = (const char*)env_rows + ((size_t)t * (t - 1) / 2) * 288;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"((unsigned)n_rows * 288u) : "memory");
}

// named barriers (ids 1 .. 15; 0 is __syncthreads): the producer side arrives, the consumer side waits; `count` = all threads
// taking part on either side.  Ids are immediates (a register id makes ptxas reserve all 16 barriers for the CTA).
template <int ID> __device__ __forceinline__ void bar_arrive_c(int count) { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "r"(count) : "memory"); }
template <int ID> __device__ __forceinline__ void bar_sync_c(int count) { asm volatile("bar.sync %0, %1;" ::"n"(ID), "r"(count) : "memory"); }
template <int BASE> __device__ __forceinline__ void bar_arrive(int parity, int count) { if (parity & 1) bar_arrive_c<BASE + 1>(count); else bar_arrive_c<BASE>(count); }
template <int BASE> __device__ __forceinline__ void bar_sync(int parity, int count) { if (parity & 1) bar_sync_c<BASE + 1>(count); else bar_sync_c<BASE>(count); }

// ---- lean double-precision primitives for the solver's critical path ----------------------------------------------------
// The FP64 kernels are bound by the LATENCY of one warp's chain of dependent double-precision operations, and the library
// division / sqrt / cbrt (IEEE rounding, full range, special cases) are 15-50 dependent instructions each.  The quantities
// in the chain are positive, finite and far inside the float range, and the kernels owe 1e-9, not the last bit: seed with the
// single-precision special-function unit and refine with Newton steps in double (error ~1e-15, a quarter of the instructions).
// Two Newton steps each: one was measured (profiles/r2_exp_newton.log) +2.8 % faster on the FP64 step kernels and +0.5 % on
// the strict FP32 step, but took the FP64 parity max from 1.1e-12 to 5.9e-11 (median 3e-16 -> 5e-15); the bit-check mode
// keeps the margin.
__device__ __forceinline__ double rcp64(double b) {
    float rf;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"((float)b));
    double r = (double)rf;
    r = fma(r, fma(-b, r, 1.0), r);  // 6e-8 -> 4e-15
    r = fma(r, fma(-b, r, 1.0), r);  // -> rounding
    return r;
}
__device__ __forceinline__ double sqrt64(double x) {  // x > 0
    float rf;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"((float)x));
    const double r = (double)rf, h = 0.5 * r;
    double y = x * r;
    y = fma(h, fma(-y, y, x), y);  // 1e-7 -> 1e-14
    y = fma(h, fma(-y, y, x), y);
    return y;
}
__device__ __forceinline__ double sqrt64z(double x) { return x > 1e-30 ? sqrt64(x) : sqrt(x); }  // x >= 0, possibly tiny
__device__ __forceinline__ double cbrt64(double x) {  // x > 0
    const double y0 = (double)cbrtf((float)x);
    float rf;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"((float)(3.0 * y0 * y0)));
    const double rc = (double)rf;
    double y = fma(fma(-y0 * y0, y0, x), rc, y0);  // Newton on y^3 = x with a single-precision slope: 1e-7 -> 1e-14
    y = fma(fma(-y * y, y, x), rc, y);
    return y;
}

// (Hand-rolled exp / log / asin / cos on the solver's argument ranges were tried and measured: the lean exp / log were 12-15 %
// SLOWER than libdevice's on this kernel -- FP64 rounding and integer<->double conversions are slow-pipe operations -- and the
// short asin / cos made no measurable difference; profiles/r2_vortex_table.md.)
__device__ __forceinline__ double dclamp(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

__device__ __forceinline__ double interp_d(const WfFastConst64& fc, const double* __restrict__ fp, double x, double left,
                                           double right) {
    const int n = fc.table_len;
    const double x0 = fc.tab_ws[0], xn = fc.tab_ws[n - 1];
    if (x < x0) return left;
    if (x > xn) return right;
    int bkt = (int)((x - x0) * fc.coarse_scale);
    bkt = min(bkt, fc.coarse_len - 1);
    int idx = fc.coarse[bkt];
    while (idx + 1 < n - 1 && fc.tab_ws[idx + 1] <= x) ++idx;
    const double xa = fc.tab_ws[idx], fa = fp[idx];
    if (x == xa) return fa;
    const double slope = (fp[idx + 1] - fa) * rcp64(fc.tab_ws[idx + 1] - xa);  // (table nodes are >= 0.01 m/s apart)
    return slope * (x - xa) + fa;
}

struct SmemView64 {
    double2* vw;              // [9T] (v, w) per rotor point (scatter kernels; the gather kernel keeps them in s.vwg)
    double2* gg;              // [T] (Gt, Gwr) of the sources processed so far (gather kernel)
    double2* red;             // [96] per-lane partial sums of the gather
    double* wsq;              // [9T] running sum of squared deficits
    double *xs, *ys;          // [T] sorted rotated coordinates (the sources' grid means x_i, y_i are read from global memory)
    double* tia;              // [3T]
    double *cyaw, *syaw;      // [T] cos / sin of the yaw (sorted order)
    double* tifin;            // [T]
    double* ynew;             // [T] new yaw, degrees, ORIGINAL order
    uchar4* idx;              // [T]
    unsigned char* ordr;      // [T]
    unsigned char* queue;     // [T]
    double* spar;             // [2][3][kSrcPar] scatter kernels: the source parameters, per lateral column, that the chain
                              // warp hands to the worker warps (double-buffered over the parity of the source index)
};

__host__ __device__ inline size_t fast64_smem_bytes(int T, bool gather = false) {
    size_t n = 0;
    n += gather ? (size_t)T * 16 + 96 * 16 : (size_t)9 * T * 16;  // gg + red, or vw
    n += (size_t)9 * T * 8;   // wsq
    n += (size_t)2 * T * 8;   // xs, ys
    n += (size_t)3 * T * 8;   // tia
    n += (size_t)4 * T * 8;   // cyaw, syaw, tifin, ynew
    n += (size_t)T * 4;       // idx
    n += (size_t)2 * ((T + 15) / 16 * 16);
    n = (n + 15) / 16 * 16;
    if (!gather) n += 2 * 3 * kSrcPar * 8;  // spar
    return n;
}

__device__ __forceinline__ SmemView64 carve64(unsigned char* base, int T, bool gather) {
    SmemView64 s;
    s.vw = (double2*)base;
    s.gg = (double2*)base;
    s.red = s.gg + T;
    double* f = gather ? (double*)(s.red + 96) : (double*)(s.vw + 9 * T);
    s.wsq = f; f += 9 * T;
    s.xs = f; f += T;
    s.ys = f; f += T;
    s.tia = f; f += 3 * T;
    s.cyaw = f; f += T;
    s.syaw = f; f += T;
    s.tifin = f; f += T;
    s.ynew = f; f += T;
    s.idx = (uchar4*)f;
    s.ordr = (unsigned char*)(s.idx + T);
    s.queue = s.ordr + (T + 15) / 16 * 16;
    s.spar = (double*)(base + fast64_smem_bytes(T, gather) - 2 * 3 * kSrcPar * 8);  // (not touched by the gather kernel)
    return s;
}

// Load the 12 vortex-table coefficients of one (pair, lateral column) as doubles: [k][cVt, cVw, cWt, cWw].
__device__ __forceinline__ void load_row12(const double* __restrict__ p, double* c) {
    const double2* q = (const double2*)p;
#pragma unroll
    for (int e = 0; e < 6; ++e) { const double2 v = __ldg(q + e); c[2 * e] = v.x; c[2 * e + 1] = v.y; }
}
// One env solved in FP64 by W warps (a CTA of 32 W threads).
//   W = 1: the throughput configuration of the bit-check mode (one warp = one CTA = one env, compacted deficit queue).
//   W > 1: the low-latency configuration used to re-solve the envs an FP32 launch flagged: warp 0 evaluates the sources'
//          scalar chains and applies each source to the NEXT turbine itself; warps 1 .. W-1 apply it to all other targets
//          one source behind (see the W > 1 branch of the source loop).
// GATHER (W = 1 with a target-major vortex table): the (v, w) of a turbine are not accumulated in shared memory while the
//          upstream sources are processed but summed from the table rows (j, i), j < i, in the prologue of source i, with the
//          circulations (Gt, Gwr) of the earlier sources kept in shared memory (16 bytes per turbine instead of 144); the
//          finished values -- and the contributions exchanged between x-tied turbines, evaluated directly -- live in the
//          global scratch s.vwg (L2-resident).  Shared memory per env drops from 23.5 KB to 15 KB at 80 turbines, which lets
//          12 envs share an SM instead of 9.
// OutT = type of the caller's output buffers (double for an FP64 handle, float for the re-solve on an FP32 handle).  FIX = re-solve: the FP32 kernel has already applied the action (yaw and
// accumulators are committed) but none of the per-env epilogue state, which is committed here.
// EVAL = candidate evaluation: env b's step for candidate `cand`, in the run-time mode of the step; every output goes to row
// `cand`, its flag to ev.amb[cand] (FIX: 1, else 0), and the state is read and never written.  Env mode (wf_evaluate_actions):
// the action row `cand` (FIX: the transitioned yaw row `cand` of ev.yaw).  Interface mode (wf_evaluate_yaw): the yaw row
// `cand` of `yaw_cmd`.
// ROLL = rollout row (wf_evaluate_rollouts, H > 1): step h = cand % H of its candidate's sequence (wf_replay, the step-h
// epilogue rules of wf_fast.cu).  Without it h = 0 is a compile-time constant, and the one-step evaluations compile to the
// code they had before rollouts existed.
template <int W, typename OutT, bool FIX, bool GATHER = false, bool EVAL = false, bool ROLL = false>
__device__ __forceinline__ void solve_env64(const int b, const int mode, const bool use_vtab, const WfModel& m,
                                            const WfFastConst64& fc, const WfState& s, const float* __restrict__ action,
                                            const double* __restrict__ yaw_cmd, const WfStepOut& out,
                                            float* __restrict__ rec, const WfEvalArgs& ev, const int cand) {
    const int T = m.T;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NT = 32 * W;
    auto csync = [] { if (W == 1) __syncwarp(); else __syncthreads(); };
    const size_t row = (size_t)b * T;
    const size_t orow = EVAL ? (size_t)cand * T : row;  // row of the yaw command and of the outputs
    // EVAL: no state is committed, on a test of K (always > 0) the compiler cannot fold.  The commits stay in the code, so the
    // compiler makes the same floating-point contractions as in the step and a candidate's outputs equal the step's bit for
    // bit; with the commits compiled out, multiply-adds fused differently (1 ulp off the step, DESIGN.md section 5b).  This
    // rests on the compiler's choices: the bit-equality tests of both evaluations (tests/test_evaluate_yaw_gpu.py,
    // tests/test_evaluate_actions_gpu.py) catch a compiler that makes others
    const bool commit = !EVAL || ev.K < 1;
    // EVAL: the row's step h in its candidate's action sequence (wf_evaluate_rollouts; 0 for every other evaluation)
    const int h = ROLL ? cand % ev.H : 0;
    // the env's turbine count, the bound of every loop below; columns n..T-1 of its rows are padding (wf_device.cuh).
    // Shared memory and the table's row strides stay those of T.
    const int n = s.turbine_count[b];
    extern __shared__ __align__(16) unsigned char smem_raw64[];
    static_assert(!GATHER || W == 1, "the gather form is the one-warp throughput kernel");
    const SmemView64 sm = carve64(smem_raw64, T, GATHER);
    // (v, w) per rotor point: shared memory, or the env's global scratch (cache-global accesses: lanes exchange values
    // through it between __syncwarp()s); an evaluation has a row per candidate, as the K candidates of an env run at once
    double2* const vwp = GATHER ? (EVAL ? ev.vwg + (size_t)cand * 9 * T : s.vwg + (size_t)b * 9 * T) : sm.vw;
    auto vw_ld = [&](const int q) -> double2 { return GATHER ? __ldcg(vwp + q) : vwp[q]; };
    auto vw_st = [&](const int q, const double2 v) { if (GATHER) __stcg(vwp + q, v); else vwp[q] = v; };
    // vortex table of this env (wf_device.cuh), or NULL: evaluate every pair directly
    const double* __restrict__ vrow = nullptr;
    if (use_vtab && s.vtab && s.vtab_ok[b] && (GATHER || !m.vtab_tmajor)) vrow = s.vtab + (size_t)b * ((size_t)T * (T - 1) / 2) * 36;

    // ---- env prologue on the ORIGINAL turbine order (mdp.py:291-319, simple_env.py:64-72) -------------------------
    int nm = 0;
    if (mode == WF_MODE_ENV) nm = s.num_moves[b] + 1;
    for (int tt = tid; tt < n; tt += NT) {
        double ynew;
        if (!FIX && mode == WF_MODE_ENV) {
            float a = action[orow + tt];
            float acc = s.acc[row + tt];
            float acc_c = (m.multi_agent && tt != n - 1) ? s.acc_prev[row + tt] : acc;
            float y_h = 0.f;  // a rollout row: the yaw after steps 0..h-1 of its sequence (action rows cand - h .. cand - 1)
            if (ROLL && h > 0)
                y_h = wf_replay(m, action, orow - (size_t)h * T, T, tt, m.multi_agent && tt != n - 1, nm, h, acc, acc_c,
                                (float)s.yaw[row + tt]);
            a = wf_applied_action(m, a, acc_c, nm + h);
            const float y1 = wf_new_yaw(m, (ROLL && h > 0) ? y_h : (float)s.yaw[row + tt], a);
            if (commit) {
                s.acc_prev[row + tt] = acc;
                s.acc[row + tt] = __fadd_rn(acc, fabsf(a));
            }
            ynew = (double)y1;
            if (commit) s.yaw[row + tt] = ynew;
        } else if (FIX && EVAL && mode == WF_MODE_ENV) {
            // the FP32 launch's transitioned yaw; an interface-mode candidate reads the caller's yaw_cmd below
            ynew = ev.yaw[orow + tt];
        } else if ((!FIX || EVAL) && mode == WF_MODE_INTERFACE && yaw_cmd) {
            ynew = yaw_cmd[orow + tt];
            if (!EVAL) s.yaw[row + tt] = ynew;
        } else {
            ynew = s.yaw[row + tt];
        }
        sm.ynew[tt] = ynew;
        sm.xs[tt] = s.xs[row + tt];
        sm.ys[tt] = s.ys[row + tt];
        sm.idx[tt] = s.idx[row + tt];
        sm.ordr[tt] = (unsigned char)s.order[row + tt];
    }
    for (int q = tid; q < 9 * n; q += NT) {
        sm.wsq[q] = 0.0;
        if (!GATHER) sm.vw[q] = make_double2(0.0, 0.0);
    }
    if (GATHER) {  // scratch entries of the turbines that exchange direct (x-tie) contributions start from zero
        for (int tt = tid; tt < n; tt += NT) {
            const bool tied = !vrow || (int)s.tab_glo[row + tt] < tt || (int)s.tab_lo[row + tt] > tt + 1;
            if (tied)
                for (int p = 0; p < 9; ++p) __stcg(vwp + 9 * tt + p, make_double2(0.0, 0.0));
        }
    }
    for (int q = tid; q < 3 * n; q += NT) sm.tia[q] = 0.0;
    csync();
    for (int tt = tid; tt < n; tt += NT) {
        const double yd = sm.ynew[sm.ordr[tt]];
        double sy, cy;
        sincos(yd * kRad, &sy, &cy);
        sm.cyaw[tt] = cy;
        sm.syaw[tt] = sy;
    }
    const double ws = s.ws[b], wd = s.wd[b];
    const double I0 = s.ti_amb[b];
    const double I02 = I0 * I0;
    const double I0p = exp(fc.ch_init * log(I0));
    const double rws = 1.0 / ws;
    const double U0a = ws * fc.ratio[0], U0b = ws * fc.ratio[1], U0c = ws * fc.ratio[2];
    const double D = fc.D;
    csync();

    const int g = lane / 3, j = lane - 3 * g;
    const bool lane_ok = lane < 3 * kTurbPerPass;
    const double offj = (j == 0) ? fc.offj[0] : ((j == 1) ? fc.offj[1] : fc.offj[2]);
    const int pl = lane & 15;
    const bool pv = pl < 9;
    const int plc = pv ? pl : 0;
    const double U0p = (plc % 3 == 0) ? U0a : ((plc % 3 == 1) ? U0b : U0c);
    const double cvl0 = fc.cv[0][plc], cvl1 = fc.cv[1][plc], cvl2 = fc.cv[2][plc];
    const double cwl0 = fc.cw[0][plc], cwl1 = fc.cw[1][plc], cwl2 = fc.cw[2][plc];
    const double c_dec = fc.eps2 * fc.inv_2pi;
    const double eps2 = fc.eps2;
    // scatter form: the table rows of source 0 are prefetched to L2 here, those of source i + 1 while source i is processed
    // (prefetching 2 sources ahead measured -4 %, 4 ahead -8 %)
    if (!GATHER && vrow && warp == 0) prefetch_rows64(vrow, 0, T, n, lane, 288);

    // W > 1, chain warp: the transverse velocities source i - 1 induces on turbine i are not written to shared memory but added
    // in registers at the head of source i's prologue, from table coefficients loaded one source earlier (no load latency on
    // the chain); per lane: rotor point plc of the pair (i - 1, i)
    double near_gt = 0.0, near_gwr = 0.0;
    double2 near_c0 = make_double2(0.0, 0.0), near_c1 = make_double2(0.0, 0.0);
    bool near_tab = false;
    for (int i = 0; i < n; ++i) {
        if (!GATHER && vrow && warp == 0) prefetch_rows64(vrow, i + 1, T, n, lane, 288);
        double2 next_c0 = make_double2(0.0, 0.0), next_c1 = make_double2(0.0, 0.0);
        bool next_tab = false;
        if (W > 1 && warp == 0 && vrow && i + 1 < n && i + 1 >= (int)s.tab_lo[row + i]) {
            next_tab = true;
            const double2* r = (const double2*)(vrow + ((size_t)i * T - (size_t)i * (i + 1) / 2) * 36 + 12 * (plc / 3) + 4 * (plc % 3));
            next_c0 = __ldg(r);
            next_c1 = __ldg(r + 1);
        }
        // ===== source prologue: the scalar chain of source i.  W == 1: the one warp does everything.  W > 1: warp 0 (the chain
        //       warp) evaluates it and hands the parameters of the sweeps to the worker warps through shared memory =====
        double par[kSrcPar];
        if (W == 1 || warp == 0) {
        double su3, sv, sw, vq, wwq;
        {
            const double wq = sm.wsq[9 * i + plc];
            double2 vw0;
            if (GATHER) {
                // table sources of this turbine: the sorted prefix [0, glo); the x-tied ones in [glo, i) have added
                // their part to the scratch entry directly
                const int glo = vrow ? (int)__ldg(s.tab_glo + row + i) : 0;
                vw0 = (glo < i) ? __ldcg(vwp + 9 * i + plc) : make_double2(0.0, 0.0);
                if (glo > 0) {
                    double2 acc[3] = {make_double2(0.0, 0.0), make_double2(0.0, 0.0), make_double2(0.0, 0.0)};
                    const double* __restrict__ trow = vrow + ((size_t)i * (i - 1) / 2) * 36 + 12 * j;
#pragma unroll 2
                    for (int j0 = 0; j0 < glo; j0 += kTurbPerPass) {
                        const int jj = j0 + g;
                        if (lane_ok && jj < glo) {
                            double c[12];
                            load_row12(trow + (size_t)jj * 36, c);
                            const double2 G = sm.gg[jj];
#pragma unroll
                            for (int k = 0; k < 3; ++k) {
                                acc[k].x += G.x * c[4 * k] + G.y * c[4 * k + 1];
                                acc[k].y += fmax(G.x * c[4 * k + 2] + G.y * c[4 * k + 3], 0.0);
                            }
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 3; ++k) sm.red[3 * lane + k] = acc[k];
                    __syncwarp();
                    const int rb = plc;  // lane 3 g' + column wrote [k] at 9 g' + 3 column + k = 9 g' + rotor point
                    double2 sum = make_double2(0.0, 0.0);
#pragma unroll
                    for (int gq = 0; gq < kTurbPerPass; ++gq) {
                        const double2 e = sm.red[9 * gq + rb];
                        sum.x += e.x;
                        sum.y += e.y;
                    }
                    vw0.x += sum.x;
                    vw0.y += sum.y;
                }
            } else {
                vw0 = sm.vw[9 * i + plc];
                if (W > 1 && near_tab) {
                    vw0.x += near_gt * near_c0.x + near_gwr * near_c0.y;
                    vw0.y += fmax(near_gt * near_c1.x + near_gwr * near_c1.y, 0.0);
                }
            }
            vq = vw0.x;
            wwq = vw0.y;
            const double u = U0p - sqrt64z(wq);
            su3 = pv ? u * u * u : 0.0;
            sv = pv ? vq : 0.0;
            sw = pv ? wwq : 0.0;
#pragma unroll
            for (int sft = 8; sft > 0; sft >>= 1) {
                su3 += __shfl_xor_sync(0xffffffffu, su3, sft);
                sv += __shfl_xor_sync(0xffffffffu, sv, sft);
                sw += __shfl_xor_sync(0xffffffffu, sw, sft);
            }
        }
        const double avg = cbrt64(su3 * (1.0 / 9.0));
        const double ct_raw = dclamp(interp_d(fc, fc.tab_ct, avg, 0.0001, 0.9999), 0.0001, 0.9999);
        const double cy = sm.cyaw[i], sy = sm.syaw[i], yd = sm.ynew[sm.ordr[i]];
        const double ct = ct_raw * cy;
        // The chain below is the critical path of the FP64 kernels (one warp, dependent double-precision operations): divisions
        // are shared through reciprocals and identities that hold to rounding (1e-16, the tolerance is 1e-9) are used freely.
        const double rcy = rcp64(cy), rct = rcp64(ct);
        const double a = 0.5 * rcy * (1.0 - sqrt64(1.0 - ct * cy));
        const double Gtop0 = fc.c_top * ws * ct, Gbot0 = fc.c_bot * ws * ct;
        const double Gwr = fc.c_wr * (a - a * a) * avg;
        const double Gt = sy * cy * Gtop0, Gb = -(sy * cy * Gbot0);

        // A.5 secondary steering through the per-model grid integrals (the denominator is (c_top a_top - c_bot a_bot) ws ct)
        double val = 2.0 * (sv * (1.0 / 9.0) - Gwr * fc.a_core) * (rct * fc.inv_ss_den) * rws;
        val = dclamp(val, -1.0, 1.0);
        const double g_deg = -(yd + kDeg * (0.5 * asin(val)));  // minus the effective yaw, degrees
        const double g_rad = g_deg * kRad;
        const double cg = cos(g_rad);
        const double rcg = rcp64(cg);

        // A.6 deflection scalars.  M0 = C0 (2 - C0) = 1 - (1 - C0)^2 = ct.
        const double sq1ct = sqrt64(1.0 - ct);
        const double sqcg = sqrt64(1.0 - ct * cg);
        const double sz0d = 0.5 * D * sqrt64((1.0 + sqcg) * rcp64(2.0 * (1.0 + sq1ct)));
        const double sy0d = sz0d * cg;
        const double C0 = 1.0 - sq1ct;
        const double E0 = C0 * C0 - fc.e3_112 * C0 + fc.e3_13;
        const double th = fc.dm03 * g_rad * rcg * (1.0 - sqcg);
        const double sM0 = sqrt64(ct);
        double tan_th;
        if (fabs(th) < 0.35) {
            // always taken for yaw within +-40 deg (|th| <= 0.31).  Maclaurin series of tan up to th^25 -- coefficients
            // 2^2n (2^2n - 1) |B_2n| / (2n)! -- good to 2.3e-16 relative on the interval (checked against libm); an eighth of
            // the instructions of tan() on the critical path
            const double t2 = th * th;
            double p = 0x1.0b132d39a6050p-16;
            p = p * t2 + 0x1.497d8eea25259p-15;
            p = p * t2 + 0x1.967e18afcafadp-14;
            p = p * t2 + 0x1.f57d7734d1664p-13;
            p = p * t2 + 0x1.3558248036744p-11;
            p = p * t2 + 0x1.7da36452b75e3p-10;
            p = p * t2 + 0x1.d6d3d0e157de0p-9;
            p = p * t2 + 0x1.226e355e6c23dp-7;
            p = p * t2 + 0x1.664f4882c10fap-6;
            p = p * t2 + 0x1.ba1ba1ba1ba1cp-5;
            p = p * t2 + 0x1.1111111111111p-3;
            p = p * t2 + 0x1.5555555555555p-2;
            tan_th = th + th * (t2 * p);
        } else {
            tan_th = tan(th);
        }
        const double Kc = th * E0 * (1.0 / 5.2) * sqrt64(sy0d * sz0d * rct);
        const double A_ln = (1.6 + sM0) * rcp64(1.6 - sM0);
        const double inv_s0d = rcp64(sy0d * sz0d);

        // ambient + wake-added TI per lateral column: every lane evaluates its own column, the three values travel by shuffle
        const double ta_j = sm.tia[3 * i + j];
        const double tp_j = sqrt64(ta_j * ta_j + I02);
        const double tp0 = __shfl_sync(0xffffffffu, tp_j, 0), tp1 = __shfl_sync(0xffffffffu, tp_j, 1),
                     tp2 = __shfl_sync(0xffffffffu, tp_j, 2);
        const double tpre = tp_j;
        const double beta_term = fc.beta2 * (1.0 - sq1ct);
        // x0 = N / Dn and 1 / x0 = Dn / N from one division
        const double x0d_n = D * cg * (1.0 + sqcg), x0d_d = 1.4142135623730951 * (fc.alpha4 * tpre + beta_term);
        const double x0d_r = rcp64(x0d_n * x0d_d);
        const double x0d = x0d_n * x0d_n * x0d_r, inv_x0d = x0d_d * x0d_d * x0d_r;
        const double kyd = fc.ka * tpre + fc.kb;
        const double delta0 = tan_th * x0d;
        const double Kck = Kc * rcp64(kyd);

        // own transverse velocities + yaw-added recovery (in-place TI update)
        const uchar4 ix = sm.idx[i];
        const bool self_on = (int)ix.x <= i;
        double sumV = sv, sumW = sw;
        if (self_on) {
            sumV += Gt * fc.sv[0] + Gb * fc.sv[1] + Gwr * fc.sv[2];
            const double Vs = Gt * cvl0 + Gb * cvl1 + Gwr * cvl2;
            const double Ws = fmax(Gt * cwl0 + Gb * cwl1 + Gwr * cwl2, 0.0);
            double rw = pv ? Ws : 0.0;
#pragma unroll
            for (int sft = 8; sft > 0; sft >>= 1) rw += __shfl_xor_sync(0xffffffffu, rw, sft);
            sumW += rw;
            __syncwarp();  // every reader of this turbine's (v, w) above is done
            if (tid < 9) vw_st(9 * i + tid, make_double2(vq + Vs, wwq + Ws));
        } else if (GATHER || (W > 1 && near_tab)) {
            __syncwarp();
            if (tid < 9) vw_st(9 * i + tid, make_double2(vq, wwq));
        }
        if (GATHER && tid == 0) sm.gg[i] = make_double2(Gt, Gwr);
        const double aI = avg * tp0;
        const double kk2 = 3.0 * aI * aI;
        const double v_term = sumV * (1.0 / 9.0), w_term = sumW * (1.0 / 9.0);
        const double k_total = 0.5 * (kk2 + v_term * v_term + w_term * w_term);
        const double I_mix = sqrt64((2.0 / 3.0) * k_total) * rcp64(avg) - tp0;
        const double tq0 = tp0 + 2.0 * I_mix, tq1 = tp1 + 2.0 * I_mix, tq2 = tp2 + 2.0 * I_mix;
        if (tid == 0) sm.tifin[i] = ((tq0 + tq1) + tq2) / 3.0;
        const double tpost = (j == 0) ? tq0 : ((j == 1) ? tq1 : tq2);

        // A.8 velocity-model scalars with the updated TI
        const double x0v_n = D * cy * (1.0 + sq1ct), x0v_d = 1.4142135623730951 * (fc.alpha4 * tpost + beta_term);
        const double x0v_r = rcp64(x0v_n * x0v_d);
        const double x0v = x0v_n * x0v_n * x0v_r, inv_x0v = x0v_d * x0v_d * x0v_r;
        const double kyv = fc.ka * tpost + fc.kb;
        const double sz0v = fc.near_c * (0.5 / 0.501);
        const double sy0v = sz0v * cy;
        const double near_s = fc.near_c * sM0;
        const double ctc = ct * cy * fc.d2_8;
        // Crespo-Hernandez constant ch_const a^ai I0^init.  W > 1: only the deficit sweeps need it, so the chain warp hands over
        // `a` and the power is taken where a sweep finds a target within reach (off the chain's critical path)
        const double watK = (W == 1) ? fc.ch_const * exp(fc.ch_ai * log(a)) * I0p : a;  // a^ai (pow(): 3x the instructions, same to 1e-15)

        constexpr double kCut = 9.5;
        const double reach1 = kCut * kyv;
        // (a conservative cut-off: single precision is plenty for the logarithm)
        const double reach0 = kCut * fmax(near_s, sy0v) + fabs(delta0) + fabs(Kck) * (double)(__logf((float)A_ln) * 1.0001f);
        par[0] = Gt; par[1] = Gb; par[2] = Gwr; par[3] = x0d; par[4] = inv_x0d; par[5] = delta0; par[6] = kyd; par[7] = sy0d;
        par[8] = sz0d; par[9] = inv_s0d; par[10] = A_ln; par[11] = sM0; par[12] = Kck; par[13] = x0v; par[14] = inv_x0v;
        par[15] = kyv; par[16] = sy0v; par[17] = near_s; par[18] = ctc; par[19] = watK; par[20] = reach1; par[21] = reach0;
        par[22] = 0.0; par[23] = 0.0;
        if (W > 1) {  // publish (the TI-dependent ones differ between the lateral columns: lanes 0..2 hold columns 0..2), then
                      // tell the workers that source i is ready (they wait on the same named barrier)
            if (lane < 3) {
                double2* d = (double2*)(sm.spar + ((i & 1) * 3 + lane) * kSrcPar);
#pragma unroll
                for (int q = 0; q < kSrcPar / 2; ++q) d[q] = make_double2(par[2 * q], par[2 * q + 1]);
            }
            __threadfence_block();
            __syncwarp();
            bar_arrive<1>(i, NT);
        }
        } else {
            bar_sync<1>(i, NT);
            const double2* d = (const double2*)(sm.spar + ((i & 1) * 3 + j) * kSrcPar);
#pragma unroll
            for (int q = 0; q < kSrcPar / 2; ++q) { const double2 v = d[q]; par[2 * q] = v.x; par[2 * q + 1] = v.y; }
        }
        const double Gt = par[0], Gb = par[1], Gwr = par[2], x0d = par[3], inv_x0d = par[4], delta0 = par[5], kyd = par[6],
                     sy0d = par[7], sz0d = par[8], inv_s0d = par[9], A_ln = par[10], sM0 = par[11], Kck = par[12], x0v = par[13],
                     inv_x0v = par[14], kyv = par[15], sy0v = par[16], near_s = par[17], ctc = par[18],
                     reach1 = par[20], reach0 = par[21];
        double watK = par[19];  // (W > 1: the axial induction until a sweep needs the constant)
        const double sz0v = fc.near_c * (0.5 / 0.501);
        const uchar4 ixs = sm.idx[i];
        const int lo = ixs.x, near_i = ixs.y, gt0_i = ixs.z, end15 = ixs.w;
        const double x_i = __ldg(s.xi + row + i), y_i = __ldg(s.yi + row + i);  // block-uniform, L1-resident

        // --- transverse velocities of source i on the 3 vertical points of (target t, column j), evaluated directly
        auto v_direct = [&](const int t, const double dx, const double dyc, const bool active) {
            const double yL = dyc + kNumEps;
            const double q = yL * yL;
            const double E = exp(-q * fc.inv_eps2);
            double Vk[3], Wk[3];
#pragma unroll 1
            for (int k = 0; k < 3; ++k) {  // not unrolled: keeps the FP64 kernel inside the instruction cache
                // pairs (real a, ground mirror b): (0,2) top, (1,3) bottom, (4,5) wake rotation
                const double r0 = q + fc.zz2[0][k], r2 = q + fc.zz2[2][k], r1 = q + fc.zz2[1][k], r3 = q + fc.zz2[3][k];
                const double r4 = q + fc.zz2[4][k], r5 = q + fc.zz2[5][k];
                const double p02 = r0 * r2, p13 = r1 * r3, p45 = r4 * r5, dd = fc.nu4[k] * dx + eps2;
                const double g0 = Gt * rcp64(p02), g1 = Gb * rcp64(p13), g4 = Gwr * rcp64(p45);
                const double dec = c_dec * rcp64(dd);
                const double Xa0 = (1.0 - E * fc.ez[0][k]) * r2, Xb0 = (1.0 - E * fc.ez[2][k]) * r0;
                const double Xa1 = (1.0 - E * fc.ez[1][k]) * r3, Xb1 = (1.0 - E * fc.ez[3][k]) * r1;
                const double Xa4 = (1.0 - E * fc.ez[4][k]) * r5, Xb4 = (1.0 - E * fc.ez[5][k]) * r4;
                const double SV = g0 * (fc.zz[0][k] * Xa0 - fc.zz[2][k] * Xb0) + g1 * (fc.zz[1][k] * Xa1 - fc.zz[3][k] * Xb1) +
                                  g4 * (fc.zz[4][k] * Xa4 - fc.zz[5][k] * Xb4);
                const double SW = g0 * (Xa0 - Xb0) + g1 * (Xa1 - Xb1) + g4 * (Xa4 - Xb4);
                Vk[k] = SV * dec;
                Wk[k] = fmax(SW * (-yL * dec), 0.0);
            }
            if (active) {
                const int qb = 9 * t + 3 * j;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double2 o = vw_ld(qb + k);
                    vw_st(qb + k, make_double2(o.x + Vk[k], o.y + Wk[k]));
                }
            }
        };
        // --- the same through the table row of the sorted pair (i, t): V += Gt*cVt + Gwr*cVw ; W += max(Gt*cWt + Gwr*cWw, 0)
        auto v_table = [&](const int t, const bool active) {
            if (GATHER) return;  // (the gather kernel reads the table in the target's prologue)
            double c[12];
            load_row12(vrow + ((size_t)i * T - (size_t)i * (i + 1) / 2 + (size_t)(t - i - 1)) * 36 + 12 * j, c);
            if (active) {
                const int qb = 9 * t + 3 * j;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double2 o = sm.vw[qb + k];
                    sm.vw[qb + k] = make_double2(o.x + (Gt * c[4 * k] + Gwr * c[4 * k + 1]),
                                                 o.y + fmax(Gt * c[4 * k + 2] + Gwr * c[4 * k + 3], 0.0));
                }
            }
        };
        // --- deflection, Gaussian deficit, sum of squares, overlap count and wake-added TI of source i on (target t, column j);
        //     the 3 lanes of a target must call it together (the overlap count is summed over the columns)
        auto d_apply = [&](const int t, const double dx, const double dyc, const bool active) {
            const double lin = fc.bd * dx + fc.ad;
            double defl;
            if (dx <= x0d) {
                defl = dx * inv_x0d * delta0 + lin;
            } else {
                const double dd = dx - x0d;
                const double sgy = kyd * dd + sy0d, sgz = kyd * dd + sz0d;
                const double sq = sqrt64(sgy * sgz * inv_s0d);
                const double L = log(A_ln * (1.6 * sq - sM0) * rcp64(1.6 * sq + sM0));
                defl = delta0 + Kck * L + lin;
            }
            double base, ek;
            {
                const bool far = dx >= x0v;
                const double dd = dx - x0v;
                const double up = dx * inv_x0v, down = (x0v - dx) * inv_x0v;
                const double sgy = far ? kyv * dd + sy0v : down * near_s + up * sy0v;
                const double sgz = far ? kyv * dd + sz0v : down * near_s + up * sz0v;
                const double inv = rcp64(sgy * sgz);  // one reciprocal: 1/sgy = sgz*inv, 1/sgz = sgy*inv
                const double dy = (dyc - defl) * (sgz * inv);
                const double rz = sgy * inv;
                const double dcl = dclamp(1.0 - ctc * inv, 0.0, 1.0);
                base = (1.0 - sqrt64z(dcl)) * exp(-0.5 * dy * dy);
                ek = exp(-0.5 * fc.dz2[0] * rz * rz);
            }
            const double be = base * ek;
            const double dU0 = be * U0a, dU1 = base * U0b, dU2 = be * U0c;
            int c = 0;
            if (active) {
                c = (dU0 > 0.05) + (dU1 > 0.05) + (dU2 > 0.05);
                const int qb = 9 * t + 3 * j;
                sm.wsq[qb] += dU0 * dU0;
                sm.wsq[qb + 1] += dU1 * dU1;
                sm.wsq[qb + 2] += dU2 * dU2;
            }
            const int gb = 3 * g;
            const int c_tot = __shfl_sync(0xffffffffu, c, gb & 31) + __shfl_sync(0xffffffffu, c, (gb + 1) & 31) +
                              __shfl_sync(0xffffffffu, c, (gb + 2) & 31);
            if (active && c_tot > 0 && t >= gt0_i && t < end15 && fabs(dyc) < fc.two_D) {
                const double dxp = dx + ((dx <= 0.1) ? 1.0 : 0.0);
                const double wat = watK * exp(fc.ch_down * log(dxp * fc.inv_D));
                const double ta = ((double)c_tot / 9.0) * wat;
                sm.tia[3 * t + j] = fmax(sm.tia[3 * t + j], ta);
            }
        };
        auto reach = [&](const double dx) { return reach1 * dx + reach0 + fabs(fc.bd * dx + fc.ad); };
        const int t_hi = vrow ? (int)s.tab_lo[row + i] : n;  // with the table only the x-ties take the direct path

        if (W == 1 && GATHER) {
            // ===== direct (v, w) exchange with the x-tied turbines, queue of the targets within reach of the wake (32
            //       candidates per pass), D sweep over the queue =====
#pragma unroll 1
            for (int t0 = lo; t0 < ((t_hi - lo > 1 || !vrow) ? t_hi : lo); t0 += kTurbPerPass) {  // without ties [lo, t_hi) = {i}
                const int tr = t0 + g;
                const bool active = lane_ok && tr < t_hi && tr != i;
                const int t = min(tr, n - 1);
                const double dx = sm.xs[t] - x_i;
                const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                v_direct(t, dx, dyc, active);
            }
            // The table rows of the NEXT target are pulled into L2 now, one deficit sweep ahead of their use.  Measured at
            // 8192 x 80 (profiles/r2_exp_gather_prefetch.log): no prefetch 2.25 M env-steps/s; here 2.36 M (7.6 GB read from HBM
            // per launch = the table once); at the top of the iteration 2.31 M (8.6 GB); one iteration earlier still 2.10 M
            // (12.4 GB: with 2072 resident envs the prefetched lines no longer survive in L2 until they are used).
            if (vrow && i + 1 < n) prefetch_target_rows64(vrow, i + 1, (int)s.tab_glo[row + i + 1], lane);
            int qn = 0;
#pragma unroll 1
            for (int t0 = near_i; t0 < n; t0 += 32) {
                const int tr = t0 + lane;
                const int t = min(tr, n - 1);
                const double r = reach(sm.xs[t] - x_i), yt = sm.ys[t];
                const bool need = tr < n && (fabs(__dsub_rn(__dadd_rn(yt, fc.offj[0]), y_i)) < r ||
                                             fabs(__dsub_rn(__dadd_rn(yt, fc.offj[1]), y_i)) < r ||
                                             fabs(__dsub_rn(__dadd_rn(yt, fc.offj[2]), y_i)) < r);
                const unsigned nb = __ballot_sync(0xffffffffu, need);
                if (need) sm.queue[qn + __popc(nb & ((1u << lane) - 1u))] = (unsigned char)t;
                qn += __popc(nb);
            }
            __syncwarp();
            for (int q0 = 0; q0 < qn; q0 += kTurbPerPass) {
                const int e = q0 + g;
                const bool active = lane_ok && e < qn;
                const int t = sm.queue[min(e, qn - 1)];
                const double dx = sm.xs[t] - x_i;
                const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                d_apply(t, dx, dyc, active);
            }
            __syncwarp();
        } else if (W == 1) {
            // ===== V sweep over all downstream targets (builds the compacted queue), then D sweep over the queue =====
            int qn = 0;
            auto enqueue = [&](const int t, const bool need) {
                const unsigned nb = __ballot_sync(0xffffffffu, need);
                const bool leader = (j == 0) && (((nb >> (3 * g)) & 7u) != 0u) && lane_ok;
                const unsigned lb = __ballot_sync(0xffffffffu, leader);
                if (leader) sm.queue[qn + __popc(lb & ((1u << lane) - 1u))] = (unsigned char)t;
                qn += __popc(lb);
            };
#pragma unroll 1
            for (int t0 = lo; t0 < ((t_hi - lo > 1 || !vrow) ? t_hi : lo); t0 += kTurbPerPass) {  // without ties [lo, t_hi) = {i}
                const int tr = t0 + g;
                const bool active = lane_ok && tr < t_hi && tr != i;
                const int t = min(tr, n - 1);
                const double dx = sm.xs[t] - x_i;
                const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                enqueue(t, active && (t >= near_i) && (fabs(dyc) < reach(dx)));
                v_direct(t, dx, dyc, active);
            }
            if (vrow) {
#pragma unroll 2
                for (int t0 = t_hi; t0 < n; t0 += kTurbPerPass) {
                    const int tr = t0 + g;
                    const bool active = lane_ok && tr < n;
                    const int t = min(tr, n - 1);
                    const double dx = sm.xs[t] - x_i;
                    const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                    enqueue(t, active && (t >= near_i) && (fabs(dyc) < reach(dx)));
                    v_table(t, active);
                }
            }
            __syncwarp();
            for (int q0 = 0; q0 < qn; q0 += kTurbPerPass) {
                const int e = q0 + g;
                const bool active = lane_ok && e < qn;
                const int t = sm.queue[min(e, qn - 1)];
                const double dx = sm.xs[t] - x_i;
                const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                d_apply(t, dx, dyc, active);
            }
            __syncwarp();
        } else {
            // ===== W > 1, pipelined.  Source i + 1 needs, of source i's sweeps, only what lands on turbine i + 1; so the chain
            //       warp applies source i to that one target itself and goes on to the prologue of source i + 1, while the
            //       worker warps (1 .. W-1, ten targets each per pass) apply source i to the targets from i + 2 on (and to
            //       x-tied predecessors), one source behind.  Named barriers 1, 2: "source ready" (chain arrives, workers
            //       wait); 3, 4: "sweep done" (workers arrive, chain waits), alternating with the parity of i.  The chain warp
            //       touches turbine i + 1 only after the workers' sweep of source i - 1 -- the last one that writes to it --
            //       is done. =====
            bool have_watK = false;
            auto sweep = [&](const int tr, const bool on, const bool skip_vtab) {
                const bool active = on && tr >= lo && tr < n && tr != i;
                const int t = min(max(tr, 0), n - 1);
                const double dx = sm.xs[t] - x_i;
                const double dyc = __dsub_rn(__dadd_rn(sm.ys[t], offj), y_i);
                const bool tab = vrow && t >= t_hi;
                if (__any_sync(0xffffffffu, active && !tab)) v_direct(t, dx, dyc, active && !tab);
                if (tab && !skip_vtab) v_table(t, active);
                const bool need = active && (t >= near_i) && (fabs(dyc) < reach(dx));
                const unsigned nb = __ballot_sync(0xffffffffu, need);
                if (nb) {
                    if (!have_watK) { watK = fc.ch_const * exp(fc.ch_ai * log(watK)) * I0p; have_watK = true; }
                    d_apply(t, dx, dyc, active && (((nb >> (3 * g)) & 7u) != 0u));
                }
            };
            if (warp == 0) {
                if (i > 0) bar_sync<3>(i - 1, NT);
                if (i + 1 < n) sweep(i + 1, lane < 3, next_tab);  // (its table part is deferred to the next prologue)
                __syncwarp();
                near_gt = Gt; near_gwr = Gwr; near_c0 = next_c0; near_c1 = next_c1; near_tab = next_tab;
            } else {
#pragma unroll 1
                for (int t0 = lo; t0 < i; t0 += kTurbPerPass * (W - 1))  // x-tied predecessors (none without ties: lo >= i)
                    sweep(min(t0 + kTurbPerPass * (warp - 1) + g, i), lane_ok, false);
#pragma unroll 1
                for (int t0 = i + 2; t0 < n; t0 += kTurbPerPass * (W - 1)) sweep(t0 + kTurbPerPass * (warp - 1) + g, lane_ok, false);
                __threadfence_block();
                bar_arrive<3>(i, NT);
            }
        }
    }
    if (W > 1) {
        if (warp == 0) bar_sync<3>(n - 1, NT);  // the workers' last sweep
        __syncthreads();
    }

    // ---- epilogue (first warp) ------------------------------------------------------------------------------------------
    if (warp != 0) return;
    const bool env = (mode != WF_MODE_INTERFACE);
    double rsum_p = 0.0, rsum_l = 0.0;
    for (int tt = lane; tt < n; tt += 32) {
        double u[9], vv[9], ww[9], c3[9], dd[9];
#pragma unroll
        for (int p = 0; p < 9; ++p) {
            const double U0k = (p % 3 == 0) ? U0a : ((p % 3 == 1) ? U0b : U0c);
            u[p] = U0k - sqrt(sm.wsq[9 * tt + p]);
            const double2 vwe = vw_ld(9 * tt + p);
            vv[p] = vwe.x;
            ww[p] = vwe.y;
            c3[p] = u[p] * u[p] * u[p];
            dd[p] = wd - kDeg * atan2(vv[p], u[p]);
        }
        auto sum9 = [](const double* p) {
            return (((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7]))) + p[8];
        };
        const double avg = cbrt(sum9(c3) / 9.0);
        const double veff = fc.rho_fac * avg * pow(sm.cyaw[tt], fc.pP3);
        const double pw = interp_d(fc, fc.tab_pw, veff, 0.0, 0.0) * fc.ref_rho;  // [W]
        double wsl = avg;
        double wdl = sum9(dd) / 9.0;
        double sd[3];
        {
            const double* arrs[3] = {u, vv, ww};
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const double mu = sum9(arrs[q]) / 9.0;
                double d2[9];
#pragma unroll
                for (int p = 0; p < 9; ++p) { const double e = arrs[q][p] - mu; d2[p] = e * e; }
                sd[q] = sqrt(sum9(d2) / 9.0);
            }
        }
        double loads[4] = {sm.tifin[tt], sd[0], sd[1], sd[2]};
        double p_out;
        if (env) {
            p_out = pw / 1e6;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                loads[q] = (loads[q] * 1e7) / 1e7;
                rsum_l += fabs(loads[q]);
            }
            rsum_p += p_out;
        } else {
            p_out = pw;
#pragma unroll
            for (int q = 0; q < 4; ++q) loads[q] = loads[q] * 1e7;
        }
        const int orig = sm.ordr[tt];
        double yv = sm.ynew[orig];
        if (mode == WF_MODE_WARMUP) {
            wsl = dclamp(wsl, 3.0, 28.0);
            wdl = dclamp(wdl, 0.0, 360.0);
            yv = dclamp(yv, (double)m.yaw_lo_f, (double)m.yaw_hi_f);
        }
        const size_t o = orow + orig;
        if (out.yaw) ((OutT*)out.yaw)[o] = (OutT)yv;
        if (out.wind_speed) ((OutT*)out.wind_speed)[o] = (OutT)wsl;
        if (out.wind_direction) ((OutT*)out.wind_direction)[o] = (OutT)wdl;
        if (out.power) ((OutT*)out.power)[o] = (OutT)p_out;
        if (out.load) {
            OutT* Lp = (OutT*)out.load + 4 * o;
            Lp[0] = (OutT)loads[0]; Lp[1] = (OutT)loads[1]; Lp[2] = (OutT)loads[2]; Lp[3] = (OutT)loads[3];
        }
        if (FIX && rec) {  // compact copy of the env's results for the host path (wf_step_host scatters it into the caller's arrays)
            float* r = rec + WF_FIX_REC_HDR;
            r[orig] = (float)yv; r[T + orig] = (float)wsl; r[2 * T + orig] = (float)wdl; r[3 * T + orig] = (float)p_out;
            r[4 * T + 4 * orig] = (float)loads[0]; r[4 * T + 4 * orig + 1] = (float)loads[1];
            r[4 * T + 4 * orig + 2] = (float)loads[2]; r[4 * T + 4 * orig + 3] = (float)loads[3];
        }
    }
#pragma unroll 1
    for (int tt = n + lane; tt < T; tt += 32) {  // padding columns: no stale value of an earlier layout shows
        const size_t o = orow + tt;
        if (out.yaw) ((OutT*)out.yaw)[o] = (OutT)0;
        if (out.wind_speed) ((OutT*)out.wind_speed)[o] = (OutT)0;
        if (out.wind_direction) ((OutT*)out.wind_direction)[o] = (OutT)0;
        if (out.power) ((OutT*)out.power)[o] = (OutT)0;
        if (out.load) {
            OutT* Lp = (OutT*)out.load + 4 * o;
            Lp[0] = (OutT)0; Lp[1] = (OutT)0; Lp[2] = (OutT)0; Lp[3] = (OutT)0;
        }
        if (FIX && rec) {
            float* r = rec + WF_FIX_REC_HDR;
            r[tt] = 0.f; r[T + tt] = 0.f; r[2 * T + tt] = 0.f; r[3 * T + tt] = 0.f;
            r[4 * T + 4 * tt] = 0.f; r[4 * T + 4 * tt + 1] = 0.f; r[4 * T + 4 * tt + 2] = 0.f; r[4 * T + 4 * tt + 3] = 0.f;
        }
    }
#pragma unroll
    for (int sft = 16; sft > 0; sft >>= 1) {
        rsum_p += __shfl_xor_sync(0xffffffffu, rsum_p, sft);
        rsum_l += __shfl_xor_sync(0xffffffffu, rsum_l, sft);
    }
    // the per-env outputs go to row ob; an evaluation commits none of the state below
    const int ob = EVAL ? cand : b;
    int it = 0;
    if (lane == 0) {
        it = s.num_iter[b] + 1 + h;
        if (commit) s.num_iter[b] = it;
        if (out.truncated) out.truncated[ob] = (uint8_t)(it == m.max_iter);
        double fw0 = ws, fw1 = wd;
        if (mode == WF_MODE_WARMUP) { fw0 = dclamp(fw0, 3.0, 28.0); fw1 = dclamp(fw1, 0.0, 360.0); }
        if (out.freewind) { ((OutT*)out.freewind)[2 * ob] = (OutT)fw0; ((OutT*)out.freewind)[2 * ob + 1] = (OutT)fw1; }
        if (FIX && rec) { rec[0] = __int_as_float(b); rec[1] = 0.f; rec[2] = (float)fw0; rec[3] = (float)fw1; rec[4] = (it == m.max_iter) ? 1.f : 0.f; }
        if (mode == WF_MODE_ENV) {
            if (commit) s.num_moves[b] = nm;
            const double wn = h > 0 ? ws : s.ws_norm[b];  // a step leaves ws_norm = ws for the next one
            double reward = rsum_p * 1e3 / (wn * wn * wn) / n - m.load_coef * (rsum_l / (4.0 * n));  // mean over the env's turbines
            if (m.shaper == 1) {
                reward = (reward - m.shaper_reference) / m.shaper_reference;
            } else if (m.shaper == 2) {
                // a rollout keeps every row's unshaped reward, the reference of its next row (see wf_fast.cu)
                if (ROLL && ev.rew) ev.rew[ob] = reward;
                if (h == 0) {
                    const double ref = s.shaper_ref[b];
                    const double shaped = (ref == 0.0) ? 0.0 : (reward - ref) / ref;
                    if (commit) s.shaper_ref[b] = reward;
                    reward = shaped;
                }
            }
            if (commit && !isfinite(reward)) s.nonfinite[b] += 1;
            if (out.reward) ((OutT*)out.reward)[ob] = (OutT)reward;
            if (FIX && rec) rec[1] = (float)reward;
            if (commit) {
                wfreset::episode_account(s, b, FIX ? (double)(float)reward : reward, it == m.max_iter);  // FIX: what the caller sees
                s.ws_norm[b] = ws;
            }
        }
        if (EVAL && ev.amb) ev.amb[cand] = FIX ? 1 : 0;
    }
    // in-kernel auto-reset (see wf_fast.cu): the truncating step starts the env's next episode and marks it for
    // wf_autoreset_finish; the outputs above remain the final observation
    if (commit && mode == WF_MODE_ENV && m.autoreset && __shfl_sync(0xffffffffu, (int)(it == m.max_iter), 0)) {
        for (int tt = lane; tt < T; tt += 32) { s.yaw[row + tt] = 0.0; s.acc[row + tt] = 0.f; s.acc_prev[row + tt] = 0.f; }
        if (lane == 0) wfreset::autoreset_mark(s, b);
    }
}

// The register file is split over the 4 SM sub-partitions (16 K registers each): a one-warp CTA of <= 168 registers shares a
// sub-partition with two others (12 per SM), one of 128 registers with three (16 per SM; 12-48 bytes of spills).  The kernels
// are latency-bound, throughput grows with the resident envs (measured on Turb32_Row5: 6 per SM 4.9 M env-steps/s, 9: 6.2 M,
// 12: 7.6 M, 16: 8.2 M); at 80 turbines shared memory holds 14 envs of the gather kernel per SM (9 of the scatter kernel).
// EVAL: CTA c evaluates candidate c of env c / K (wf_evaluate_yaw in interface mode, wf_evaluate_actions in env mode);
// EVAL + ROLL: row c of env c / (K H) (wf_evaluate_rollouts with H > 1)
template <bool GATHER, bool EVAL = false, bool ROLL = false>
__global__ void __launch_bounds__(32, 16)
wf_step_fast64_kernel(const int mode, const int env_begin, const bool use_vtab, const WfModel m, const __grid_constant__ WfFastConst64 fc,
                      const WfState s, const uint8_t* __restrict__ mask, const float* __restrict__ action,
                      const double* __restrict__ yaw_cmd, const WfStepOut out, const WfEvalArgs ev) {
    int b;
    if constexpr (ROLL) {
        b = blockIdx.x / (ev.K * ev.H);
        // a row after its candidate's truncating step is not solved (step 0 never is one).  Here rather than in
        // solve_env64: there the test changed the compiler's floating-point contractions of the solve (DESIGN.md 5b)
        const int h = blockIdx.x % ev.H;
        if (h > 0) {
            const int h_trunc = m.max_iter - s.num_iter[b] - 1;
            if (h_trunc >= 0 && h > h_trunc) { wf_zero_eval_row<double>(out, ev.amb, blockIdx.x, m.T, threadIdx.x); return; }
        }
    } else if constexpr (EVAL) {
        b = blockIdx.x / ev.K;
    } else {
        b = blockIdx.x + env_begin;
    }
    if (mask && !mask[b]) return;
    solve_env64<1, double, false, GATHER, EVAL, ROLL>(b, mode, use_vtab, m, fc, s, action, yaw_cmd, out, nullptr, ev, blockIdx.x);
}

// Re-solve, in FP64, of the envs an FP32 launch flagged (their ids sit in s.fix_list[0, n), n in s.fix_count[0]); launched
// right behind every FP32 step launch of a strict handle, usually with nothing or a handful of envs to do, so it is built for
// latency: W warps per env.  The last CTA to leave re-arms the counters.
template <int W>
__global__ void __launch_bounds__(32 * W, W == 1 ? 8 : 1)
wf_fixup64_kernel(const int mode, const bool use_vtab, const WfModel m, const __grid_constant__ WfFastConst64 fc,
                  const WfState s, const WfStepOut out, float* __restrict__ rec, const int rec_cap) {
    const int n = *(volatile int*)&s.fix_count[0];
    const int rec_len = WF_FIX_REC_HDR + 8 * m.T;  // header (env id, reward, freewind x2, truncated) + yaw, ws, wd, power, load x4
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        solve_env64<W, float, true>(s.fix_list[k], mode, use_vtab, m, fc, s, nullptr, nullptr, out,
                                    (rec && k < rec_cap) ? rec + (size_t)k * rec_len : nullptr, WfEvalArgs{}, 0);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&s.fix_count[1], 1) == (int)gridDim.x - 1) {
            s.fix_count[2] = n;
            s.fix_count[0] = 0;
            s.fix_count[1] = 0;
        }
    }
}

// Evaluation instantiation of the re-solve: the rows an evaluation launch flagged (ev.fix_list / ev.fix_count, row c = env
// c / (K H), step c % H), from the transitioned yaw rows in ev.yaw (env mode, wf_evaluate_actions / wf_evaluate_rollouts)
// or the yaw rows of `yaw_cmd` (interface mode, wf_evaluate_yaw); they write every output row and the flag of the row and
// commit nothing.
// A kernel of its own rather than a flag of wf_fixup64_kernel, whose parameter list (and so code) stays as it was.
template <int W>
__global__ void __launch_bounds__(32 * W, W == 1 ? 8 : 1)
wf_fixup64_eval_kernel(const int mode, const bool use_vtab, const WfModel m, const __grid_constant__ WfFastConst64 fc, const WfState s,
                       const WfStepOut out, const double* __restrict__ yaw_cmd, const WfEvalArgs ev) {
    const int n = *(volatile int*)&ev.fix_count[0];
    for (int k = blockIdx.x; k < n; k += gridDim.x) {
        const int c = ev.fix_list[k];
        solve_env64<W, float, true, false, true, true>(c / (ev.K * ev.H), mode, use_vtab, m, fc, s, nullptr, yaw_cmd, out, nullptr, ev, c);
        __syncthreads();
    }
    if (threadIdx.x == 0) {  // the last CTA to leave re-arms the evaluation counters
        __threadfence();
        if (atomicAdd(&ev.fix_count[1], 1) == (int)gridDim.x - 1) {
            ev.fix_count[2] = n;
            ev.fix_count[0] = 0;
            ev.fix_count[1] = 0;
        }
    }
}

}  // namespace

// Dynamic shared memory up to 100 KB for every FP64 kernel; the step kernels also prefer the largest shared-memory carveout.
cudaError_t wf_configure_fast64_kernels() {
    for (auto k : {wf_step_fast64_kernel<false>, wf_step_fast64_kernel<true>, wf_step_fast64_kernel<false, true>,
                   wf_step_fast64_kernel<true, true>, wf_step_fast64_kernel<false, true, true>,
                   wf_step_fast64_kernel<true, true, true>}) {
        cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
    }
    for (auto k : {wf_fixup64_kernel<1>, wf_fixup64_kernel<2>, wf_fixup64_kernel<4>, wf_fixup64_kernel<8>}) {
        const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        if (e != cudaSuccess) return e;
    }
    for (auto k : {wf_fixup64_eval_kernel<1>, wf_fixup64_eval_kernel<2>, wf_fixup64_eval_kernel<4>, wf_fixup64_eval_kernel<8>}) {
        const cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

template <int W, bool EVAL>
static cudaError_t launch_fixup_t(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                  const WfStepOut& out, int grid, float* d_rec, int rec_cap, const double* d_yaw,
                                  const WfEvalArgs& ev, cudaStream_t stream) {
    if (EVAL)
        wf_fixup64_eval_kernel<W><<<grid, 32 * W, fast64_smem_bytes(m.T), stream>>>(mode, use_vtab, m, fc, s, out, d_yaw, ev);
    else
        wf_fixup64_kernel<W><<<grid, 32 * W, fast64_smem_bytes(m.T), stream>>>(mode, use_vtab, m, fc, s, out, d_rec, rec_cap);
    return cudaGetLastError();
}

// W and the grid of a re-solve launch behind a step (or evaluation) launch of `count` CTAs
template <bool EVAL>
static cudaError_t launch_fixup_sized(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                      const WfStepOut& out, int count, float* d_rec, int rec_cap, const double* d_yaw,
                                      const WfEvalArgs& ev, cudaStream_t stream) {
    // The launch is latency-bound while the flagged envs (1-2 % of the batch) are fewer than the CTAs the GPU holds at once,
    // and each env is a sequential sweep over its turbines: W warps per env cover 10 W targets in one fused pass per source.
    // So: as many warps as the farm can use (T / 10), fewer when the batch is large enough for the flagged envs to outnumber
    // the resident CTAs (148 at W = 8, 296 at W = 4, 592 at W = 2, 1184 at W = 1 on a B200: 8 warps of ~196 registers per SM).
    int w = m.T > 40 ? 8 : (m.T > 20 ? 4 : (m.T > 10 ? 2 : 1));
    const int expected = count / 64 + 1;  // ~1.5 % of the envs
    while (w > 1 && expected > 148 * 8 / w) w >>= 1;
    const int resident = 148 * 8 / w;  // two ~196-register warps per SM sub-partition = 8 warps per SM
    const int grid = count < resident ? count : resident;
    switch (w) {
        case 8: return launch_fixup_t<8, EVAL>(mode, use_vtab, m, fc, s, out, grid, d_rec, rec_cap, d_yaw, ev, stream);
        case 4: return launch_fixup_t<4, EVAL>(mode, use_vtab, m, fc, s, out, grid, d_rec, rec_cap, d_yaw, ev, stream);
        case 2: return launch_fixup_t<2, EVAL>(mode, use_vtab, m, fc, s, out, grid, d_rec, rec_cap, d_yaw, ev, stream);
        default: return launch_fixup_t<1, EVAL>(mode, use_vtab, m, fc, s, out, grid, d_rec, rec_cap, d_yaw, ev, stream);
    }
}

cudaError_t wf_launch_fixup64(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                              const WfStepOut& out, int env_count, float* d_rec, int rec_cap, cudaStream_t stream) {
    return launch_fixup_sized<false>(mode, use_vtab, m, fc, s, out, env_count, d_rec, rec_cap, nullptr, WfEvalArgs{}, stream);
}

// W is chosen from the B*K*H CTAs of the evaluation launch by the step's rule
cudaError_t wf_launch_eval_fixup64(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                   const WfEvalArgs& ev, const double* d_yaw, const WfStepOut& out, cudaStream_t stream) {
    return launch_fixup_sized<true>(mode, use_vtab, m, fc, s, out, m.B * ev.K * ev.H, nullptr, 0, d_yaw, ev, stream);
}

// StepPercentage through a rollout: a step shapes its reward with the previous step's unshaped one as the reference.  Row
// h = 0 was shaped in the evaluation kernels with the committed shaper_ref; rows h >= 1 are shaped here, one thread per
// candidate walking its rows in order up to its truncating step, from the unshaped rewards ev.rew the kernels left (the
// float reward widened to double, or a re-solved row's double reward, as the step commits to shaper_ref).  Same expression
// as the step kernels.
template <typename OutT>
__global__ void __launch_bounds__(256)
wf_eval_step_pct_kernel(const WfModel m, const WfState s, const WfEvalArgs ev, OutT* __restrict__ reward) {
    const int bk = blockIdx.x * blockDim.x + threadIdx.x;
    if (bk >= m.B * ev.K) return;
    const int h_trunc = m.max_iter - s.num_iter[bk / ev.K] - 1;
    const int h_end = (h_trunc >= 0 && h_trunc < ev.H - 1) ? h_trunc : ev.H - 1;
    const size_t c0 = (size_t)bk * ev.H;
    for (int h = 1; h <= h_end; ++h) {
        const double ref = ev.rew[c0 + h - 1];
        reward[c0 + h] = (ref == 0.0) ? (OutT)0 : (OutT)((ev.rew[c0 + h] - ref) / ref);
    }
}

cudaError_t wf_launch_eval_step_pct(bool f64, const WfModel& m, const WfState& s, const WfEvalArgs& ev, void* d_reward,
                                    cudaStream_t stream) {
    const unsigned grid = (unsigned)(((long long)m.B * ev.K + 255) / 256);
    if (f64) wf_eval_step_pct_kernel<double><<<grid, 256, 0, stream>>>(m, s, ev, (double*)d_reward);
    else wf_eval_step_pct_kernel<float><<<grid, 256, 0, stream>>>(m, s, ev, (float*)d_reward);
    return cudaGetLastError();
}

bool wf_fast64_gathers(const WfModel& m, const WfState& s) { return m.vtab_tmajor && s.vtab && s.vwg && s.tab_glo; }

cudaError_t wf_launch_step_fast64(int mode, bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                  const uint8_t* d_mask, const float* d_action, const double* d_yaw_cmd,
                                  const WfStepOut& out, int env_begin, int env_count, cudaStream_t stream) {
    // a target-major table (and its scratch) belongs to the gather kernel; the scatter kernel evaluates every pair directly
    const bool gather = wf_fast64_gathers(m, s) && use_vtab;
    const size_t smem = fast64_smem_bytes(m.T, gather);
    if (gather)
        wf_step_fast64_kernel<true><<<env_count, 32, smem, stream>>>(mode, env_begin, true, m, fc, s, d_mask, d_action, d_yaw_cmd, out,
                                                                     WfEvalArgs{});
    else
        wf_step_fast64_kernel<false><<<env_count, 32, smem, stream>>>(mode, env_begin, use_vtab, m, fc, s, d_mask, d_action, d_yaw_cmd,
                                                                      out, WfEvalArgs{});
    return cudaGetLastError();
}

cudaError_t wf_launch_eval_fast64(bool use_vtab, const WfModel& m, const WfFastConst64& fc, const WfState& s,
                                  const WfEvalArgs& ev, const double* d_yaw, const float* d_action, const WfStepOut& out,
                                  cudaStream_t stream) {
    // the same form as the step kernel of this handle in its current state (a stale table: the scatter form, pairs direct)
    const bool gather = wf_fast64_gathers(m, s) && use_vtab;
    const size_t smem = fast64_smem_bytes(m.T, gather);
    const unsigned grid = (unsigned)m.B * (unsigned)ev.K * (unsigned)ev.H;
    const int mode = d_action ? WF_MODE_ENV : WF_MODE_INTERFACE;
    if (gather && ev.H > 1)
        wf_step_fast64_kernel<true, true, true><<<grid, 32, smem, stream>>>(mode, 0, true, m, fc, s, nullptr, d_action, d_yaw, out, ev);
    else if (gather)
        wf_step_fast64_kernel<true, true><<<grid, 32, smem, stream>>>(mode, 0, true, m, fc, s, nullptr, d_action, d_yaw, out, ev);
    else if (ev.H > 1)
        wf_step_fast64_kernel<false, true, true><<<grid, 32, smem, stream>>>(mode, 0, use_vtab, m, fc, s, nullptr, d_action, d_yaw, out,
                                                                            ev);
    else
        wf_step_fast64_kernel<false, true><<<grid, 32, smem, stream>>>(mode, 0, use_vtab, m, fc, s, nullptr, d_action, d_yaw, out, ev);
    return cudaGetLastError();
}

cudaError_t wf_step_fast64_attributes(const WfModel& m, const WfState& s, cudaFuncAttributes* attr, int* ctas_per_sm, int* threads,
                                      int* smem) {
    *threads = 32;
    const bool gather = wf_fast64_gathers(m, s);
    *smem = (int)fast64_smem_bytes(m.T, gather);
    cudaError_t e = gather ? cudaFuncGetAttributes(attr, wf_step_fast64_kernel<true>) : cudaFuncGetAttributes(attr, wf_step_fast64_kernel<false>);
    if (e != cudaSuccess) return e;
    return gather ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, wf_step_fast64_kernel<true>, 32, *smem)
                  : cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, wf_step_fast64_kernel<false>, 32, *smem);
}
