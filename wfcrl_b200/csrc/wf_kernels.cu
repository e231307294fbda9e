// Hand-written sm_100a kernels for the FLORIS GCH steady-state solve + WFCRL env step (basic variant).
//
// One CTA per environment, one thread per turbine (in downstream-sorted order).  Each thread keeps the 3x3 rotor
// grid state of ITS turbine (wake deficit, v, w, turbulence intensity) in registers; the sequential solver loop
// over sources i = 0..T-1 broadcasts the source turbine's parameters through a double-buffered shared-memory record
// with ONE __syncthreads per source.  The same template instantiates the FP64 bit-check kernel and a plain FP32
// kernel (x-direction masks always come from FP64 differences, SURVEY 7.3).
//
// Algorithm: SURVEY.md Appendix A (restatement of FLORIS 3.5 as configured by
// wfcrl/simulators/floris/inputs/template/case.yaml) -- reference call sites wfcrl/interface.py:557-586, 622-648;
// env semantics wfcrl/mdp.py:273-319, wfcrl/simple_env.py:58-96, wfcrl/multiagent_env.py:198-249, wfcrl/rewards.py.
#include "wf_device.cuh"
#include "wf_reset_device.cuh"

#include <math.h>

namespace {

constexpr double kPi = 3.141592653589793;
constexpr double kNumEps = 0.001;  // floris BaseModel.NUM_EPS

// ---------------------------------------------------------------------------------------------------------------
// math traits
// ---------------------------------------------------------------------------------------------------------------
template <typename R> struct M;
template <> struct M<double> {
    static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
    static __device__ __forceinline__ double log(double x) { return ::log(x); }
    static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
    static __device__ __forceinline__ double cbrt(double x) { return ::cbrt(x); }
    static __device__ __forceinline__ double pow(double x, double y) { return ::pow(x, y); }
    static __device__ __forceinline__ double asin(double x) { return ::asin(x); }
    static __device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
    static __device__ __forceinline__ double tan(double x) { return ::tan(x); }
    static __device__ __forceinline__ double div(double a, double b) { return a / b; }
    static __device__ __forceinline__ double hypot(double a, double b) { return ::hypot(a, b); }
    static __device__ __forceinline__ void sincos(double x, double* s, double* c) { ::sincos(x, s, c); }
    static __device__ __forceinline__ double abs(double x) { return ::fabs(x); }
    static __device__ __forceinline__ double max(double a, double b) { return ::fmax(a, b); }
    static __device__ __forceinline__ double min(double a, double b) { return ::fmin(a, b); }
};
template <> struct M<float> {
    static __device__ __forceinline__ float exp(float x) { return __expf(x); }
    static __device__ __forceinline__ float log(float x) { return __logf(x); }
    static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
    static __device__ __forceinline__ float cbrt(float x) { return cbrtf(x); }
    static __device__ __forceinline__ float pow(float x, float y) { return __powf(x, y); }
    static __device__ __forceinline__ float asin(float x) { return asinf(x); }
    static __device__ __forceinline__ float atan2(float y, float x) { return atan2f(y, x); }
    static __device__ __forceinline__ float tan(float x) { return tanf(x); }
    static __device__ __forceinline__ float div(float a, float b) { return __fdividef(a, b); }
    static __device__ __forceinline__ float hypot(float a, float b) { return sqrtf(fmaf(a, a, b * b)); }
    static __device__ __forceinline__ void sincos(float x, float* s, float* c) { sincosf(x, s, c); }
    static __device__ __forceinline__ float abs(float x) { return fabsf(x); }
    static __device__ __forceinline__ float max(float a, float b) { return fmaxf(a, b); }
    static __device__ __forceinline__ float min(float a, float b) { return fminf(a, b); }
};

// numpy's reduction order over N < 128 contiguous values (pairwise_sum: eight running sums over the blocks of 8, combined
// pairwise, then the remainder one by one); N = 9 and 25 are the 3x3 and 5x5 rotor grids
template <typename R, int N> __device__ __forceinline__ R sumN(const R* p) {
    static_assert(N >= 8 && N < 128, "grid of 3x3 .. 11x11 points");
    R r[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) r[q] = p[q];
#pragma unroll
    for (int i = 8; i < N - (N % 8); i += 8) {
#pragma unroll
        for (int q = 0; q < 8; ++q) r[q] += p[i + q];
    }
    R res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
    for (int i = N - (N % 8); i < N; ++i) res += p[i];
    return res;
}
template <typename R, int N> __device__ __forceinline__ R meanN(const R* p) { return M<R>::div(sumN<R, N>(p), R(N)); }
// the same at run time (geometry kernel)
__device__ __forceinline__ double np_mean(const double* p, int n) {
    double r[8];
    for (int q = 0; q < 8; ++q) r[q] = p[q];
    int i = 8;
    for (; i < n - (n % 8); i += 8)
        for (int q = 0; q < 8; ++q) r[q] = __dadd_rn(r[q], p[i + q]);
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, p[i]);
    return __ddiv_rn(res, (double)n);
}
// offset of grid index q on a G-point rotor grid: np.linspace(-D/4, D/4, G)[q]
__device__ __forceinline__ double grid_off(double quarter_D, int q, int G) {
    return q == G - 1 ? quarter_D : __dadd_rn(__dmul_rn((double)q, __ddiv_rn(2.0 * quarter_D, (double)(G - 1))), -quarter_D);
}

// np.interp + scipy interp1d fill values on the turbine table (table lives in global memory, L1-resident)
__device__ __forceinline__ double interp_table(double x, const double* __restrict__ xp, const double* __restrict__ fp,
                                               int n, double left, double right) {
    if (x < xp[0]) return left;
    if (x > xp[n - 1]) return right;
    if (x == xp[n - 1]) return fp[n - 1];
    int lo = 0, hi = n - 1;  // invariant xp[lo] <= x < xp[hi]
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (xp[mid] <= x) lo = mid; else hi = mid;
    }
    double x0 = xp[lo], f0 = fp[lo];
    if (x == x0) return f0;
    double slope = (fp[lo + 1] - f0) / (xp[lo + 1] - x0);
    return slope * (x - x0) + f0;
}

// ---------------------------------------------------------------------------------------------------------------
// shared-memory layouts
// ---------------------------------------------------------------------------------------------------------------
// Per-env constants computed once per step by thread 0.
template <typename R, int G> struct EnvConst {
    R U0[G], nu4[G];       // initial velocity per vertical index k; 4*nu/Uinf per k (transverse-velocity decay)
    R zq[6][G];            // Z_k + c_v + NUM_EPS for the 6 vortices (top, bottom, top-mirror, bottom-mirror, core, core-mirror)
    R Uinf, vel_top, vel_bot, eps2, inv_eps2, I0;
    double wd, ws;
};

// Per-source broadcast record (double buffered).
template <typename R, int NP> struct SrcRec {
    double x_i, y_i;       // FP64: every x-mask is decided on the FP64 difference X - x_i
    R ct, a, Gt, Gb, Gwr;  // thrust coeff (incl. cos yaw), axial induction, vortex circulations
    R cgv;                 // cosd(-yaw_i)
    R sM0, tan_th, Kc;     // deflection scalars
    R sy0d, sz0d;          // sigma_y0, sigma_z0 of the deflection model (effective yaw)
    R sy0v, sz0v;          // sigma_y0, sigma_z0 of the velocity model
    R near_s;              // 0.501 * D * sqrt(ct / 2)
    R ctc;                 // ct * cosd(-yaw_i) * D^2 / 8
    R watK;                // constant * a^ai * I0^initial
    R x0d[NP], kyd[NP];  // near-wake length (relative to x_i) and expansion rate from the PRE-update TI
    R x0v[NP], kyv[NP];  // same from the POST-update TI (velocity model)
};

// The six vortices of calculate_transverse_velocity in FLORIS' summation order V1..V6:
//   V1 top (+Gt), V2 bottom (+Gb), V3 top ground mirror (-Gt), V4 bottom ground mirror (-Gb),
//   V5 wake rotation (+Gwr), V6 wake rotation ground mirror (-Gwr).
template <typename R, int G>
__device__ __forceinline__ void transverse(const EnvConst<R, G>& ec, R Gt, R Gb, R Gwr, R yL, int k, R decay, R* V, R* W) {
    const R two_pi = R(2.0 * kPi);
    const R yy = yL * yL;
    R Vs = R(0), Ws = R(0);
    const R gam[6] = {Gt, Gb, -Gt, -Gb, Gwr, -Gwr};
#pragma unroll
    for (int q = 0; q < 6; ++q) {
        const R zz = ec.zq[q][k];
        const R r = yy + zz * zz;
        const R core = R(1) - M<R>::exp(-r * ec.inv_eps2);
        const R f = M<R>::div(core * decay, two_pi * r);
        Vs += (gam[q] * zz) * f;
        Ws += (-gam[q] * yL) * f;
    }
    *V = Vs;
    *W = Ws;
}

// lateral offset (Y - y_i) of grid column j of a target at rotated y `ys_t` from the source centre y_i
template <typename R> struct Lat {
    // returns (Y - y_i) exactly like the reference: Y = fl(ys + off_j) in FP64
    static __device__ __forceinline__ R get(double ys_t, double y_i, double offj);
};
template <> struct Lat<double> {
    static __device__ __forceinline__ double get(double ys_t, double y_i, double offj) {
        return __dsub_rn(__dadd_rn(ys_t, offj), y_i);
    }
};
template <> struct Lat<float> {
    static __device__ __forceinline__ float get(double ys_t, double y_i, double offj) {
        return (float)(ys_t - y_i) + (float)offj;
    }
};

// ---------------------------------------------------------------------------------------------------------------
// geometry kernel: rotate, stable sort, per-turbine means (SURVEY A.2).  One CTA per env, one thread per turbine.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(WF_MAX_TURBINES_K)
wf_geometry_kernel(const WfModel m, const WfState s, const uint8_t* __restrict__ mask,
                   const double* __restrict__ cs_override, const int autoreset_draw) {
    const int b = blockIdx.x;
    if (mask && !mask[b]) return;
    const int T = m.T;
    const int t = threadIdx.x;
    __shared__ double xr[WF_MAX_TURBINES_K], yr[WF_MAX_TURBINES_K], xsrt[WF_MAX_TURBINES_K];
    __shared__ double cs[2];
    if (t == 0) {
        // second half of an in-kernel auto-reset: the new episode's wind (and layout id)
        if (autoreset_draw) wfreset::autoreset_wind(m, s, b);
        double c, sn;
        if (cs_override) {
            c = cs_override[2 * b];
            sn = cs_override[2 * b + 1];
        } else {
            const double wd = s.wd[b];
            const double dev = wfreset::fmod_py(wfreset::fmod_py(wd - 270.0, 360.0) + 360.0, 360.0);
            const double rad = dev * (kPi / 180.0);
            c = cos(rad);
            sn = sin(rad);
        }
        cs[0] = c;
        cs[1] = sn;
        s.cs[2 * b] = c;
        s.cs[2 * b + 1] = sn;
    }
    __syncthreads();
    const int lay = s.layout_id[b];  // after the barrier: thread 0 may just have drawn it
    const int n = layout_counts(m)[lay];   // the env's turbines are 0..n-1; slots n..T-1 are padding
    const double cx = m.layout_c[2 * lay], cy = m.layout_c[2 * lay + 1];
    if (t < n) {
        const size_t lt = (size_t)lay * T + t;
        const double xo = __dsub_rn(m.layout_x[lt], cx), yo = __dsub_rn(m.layout_y[lt], cy);
        // every product / sum separately rounded: no FMA contraction (SURVEY 7.3)
        xr[t] = __dadd_rn(__dsub_rn(__dmul_rn(xo, cs[0]), __dmul_rn(yo, cs[1])), cx);
        yr[t] = __dadd_rn(__dadd_rn(__dmul_rn(xo, cs[1]), __dmul_rn(yo, cs[0])), cy);
    }
    __syncthreads();
    if (t < n) {
        const double x = xr[t], y = yr[t];
        int rank = 0;
        for (int q = 0; q < n; ++q) {
            const double xq = xr[q];
            rank += (xq < x) || (xq == x && q < t);  // stable ascending
        }
        const size_t o = (size_t)b * T + rank;
        s.xs[o] = x;
        s.ys[o] = y;
        s.order[o] = t;
        const double off = 0.5 * m.D / 2;  // disc_area_radius: grid offsets np.linspace(-off, off, G)
        if (m.G == 3) {
            s.xi[o] = __ddiv_rn(__dadd_rn(__dmul_rn(8.0, x), x), 9.0);
            const double ya = __dadd_rn(y, -off), yb = __dadd_rn(y, 0.0), yc = __dadd_rn(y, off);
            // flattened grid values p = 3j + k: ya ya ya yb yb yb yc yc yc ; numpy order ((p0+p1)+(p2+p3))+((p4+p5)+(p6+p7)) + p8
            const double s03 = __dadd_rn(__dadd_rn(ya, ya), __dadd_rn(ya, yb));
            const double s47 = __dadd_rn(__dadd_rn(yb, yb), __dadd_rn(yc, yc));
            s.yi[o] = __ddiv_rn(__dadd_rn(__dadd_rn(s03, s47), yc), 9.0);
        } else {  // any other grid: the same numpy reduction over the G*G flattened values p = G*j + k
            double gx[49], gy[49];
            const int G = m.G;
            for (int j = 0; j < G; ++j)
                for (int q = 0; q < G; ++q) { gx[G * j + q] = x; gy[G * j + q] = __dadd_rn(y, grid_off(off, j, G)); }
            s.xi[o] = np_mean(gx, G * G);
            s.yi[o] = np_mean(gy, G * G);
        }
        // float-float positions relative to the rotation centre for the FP32 kernel
        const double xrel = x - cx, yrel = y - cy;
        const float xh = (float)xrel, yh = (float)yrel;
        s.xhl[o] = make_float2(xh, (float)(xrel - (double)xh));
        s.yhl[o] = make_float2(yh, (float)(yrel - (double)yh));
        xsrt[rank] = x;
    } else if (t < T) {
        // padding slot: sorted position t holds "turbine" t at the origin, its masks say "none" (n), and the env's padding
        // state is zeroed (an env that moved to a smaller layout must not keep the larger layout's yaw / accumulators)
        const size_t o = (size_t)b * T + t;
        s.xs[o] = 0.0; s.ys[o] = 0.0; s.xi[o] = 0.0; s.yi[o] = 0.0;
        s.order[o] = t;
        s.xhl[o] = make_float2(0.f, 0.f);
        s.yhl[o] = make_float2(0.f, 0.f);
        s.idx[o] = make_uchar4((unsigned char)n, (unsigned char)n, (unsigned char)n, (unsigned char)n);
        s.tab_lo[o] = (unsigned char)n;
        s.tab_glo[o] = 0;
        s.yaw[o] = 0.0; s.acc[o] = 0.f; s.acc_prev[o] = 0.f;
    }
    __syncthreads();
    if (t < n) {
        // t is now a SORTED source position: first target index at which each FP64 x-mask turns true
        const size_t o = (size_t)b * T + t;
        const double x_i = s.xi[o];
        const double x01 = __dadd_rn(x_i, 0.1), x15 = __dadd_rn(15 * m.D, x_i);
        const double xtie = __dadd_rn(xsrt[t], 1e-6);
        int i0 = n, i1 = n, i2 = n, i3 = n, i4 = n, i5 = 0;
        for (int q = n - 1; q >= 0; --q) {
            const double xq = xsrt[q];
            i5 += xsrt[t] > __dadd_rn(xq, 1e-6);  // q's tab_lo <= t
            if (__dsub_rn(xq, x_i) >= 0.0) i0 = q;
            if (xq > x01) i1 = q;
            if (xq > x_i) i2 = q;
            if (xq > x15) i3 = q;
            if (xq > xtie) i4 = q;
        }
        s.idx[o] = make_uchar4((unsigned char)i0, (unsigned char)i1, (unsigned char)i2, (unsigned char)i3);
        s.tab_lo[o] = (unsigned char)i4;
        s.tab_glo[o] = (unsigned char)i5;
    }
    if (t == 0) s.turbine_count[b] = n;  // what the step kernels and the vortex-table kernel read
    if (t == 0 && s.vtab_ok) s.vtab_ok[b] = 0;  // the vortex table of this env no longer matches its geometry
}

// ---------------------------------------------------------------------------------------------------------------
// vortex table: geometry-only coefficients of the transverse velocities (SURVEY A.7), one row per sorted pair i < t.
// Evaluated in FP64 with the accurate math functions whatever the handle's precision; stored in double.
// One CTA per env; a thread owns one (row, lateral column) and writes its 12 coefficients [k][cVt, cVw, cWt, cWw].
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
wf_vortex_table_kernel(const WfModel m, const __grid_constant__ WfFastConst64 fc, const WfState s,
                       const uint8_t* __restrict__ mask) {
    const int b = blockIdx.x;
    if (mask && !mask[b]) return;
    const int T = m.T;
    __shared__ double xs[WF_MAX_TURBINES_K], ys[WF_MAX_TURBINES_K], xi[WF_MAX_TURBINES_K], yi[WF_MAX_TURBINES_K];
    __shared__ int rowoff[WF_MAX_TURBINES_K];
    const int n = s.turbine_count[b];  // rows of pairs inside the env's n turbines; row strides stay those of T
    const size_t row0 = (size_t)b * T;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        xs[t] = s.xs[row0 + t];
        ys[t] = s.ys[row0 + t];
        xi[t] = s.xi[row0 + t];
        yi[t] = s.yi[row0 + t];
        rowoff[t] = t * n - t * (t + 1) / 2;
    }
    __syncthreads();
    const int rows = n * (n - 1) / 2;
    double* __restrict__ tab = s.vtab + (size_t)b * (T * (T - 1) / 2) * 36;
    const double rho = fc.c_bot / fc.c_top;  // Gb = -rho * Gt
    const double c_dec = fc.eps2 * fc.inv_2pi;
    for (int task = threadIdx.x; task < rows * 3; task += blockDim.x) {
        const int row = task / 3, j = task - 3 * row;
        // row -> (i, t): largest i with rowoff[i] <= row
        int lo = 0, hi = n - 2;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (rowoff[mid] <= row) lo = mid; else hi = mid - 1;
        }
        const int i = lo, t = i + 1 + (row - rowoff[i]);
        const double dx = xs[t] - xi[i];
        const double dyc = __dsub_rn(__dadd_rn(ys[t], fc.offj[j]), yi[i]);
        const double yL = dyc + kNumEps;
        const double q = yL * yL;
        const double E = exp(-q * fc.inv_eps2);
        const size_t dst = (m.vtab_tmajor ? (size_t)(t * (t - 1) / 2 + i) : (size_t)(i * T - i * (i + 1) / 2 + (t - i - 1))) * 36 + j * 12;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double A[3], Bc[3];  // per unit circulation of (top pair, bottom pair, wake-rotation pair): V and W sums
#pragma unroll
            for (int pr = 0; pr < 3; ++pr) {
                const int va = (pr == 0) ? 0 : (pr == 1 ? 1 : 4), vb = (pr == 0) ? 2 : (pr == 1 ? 3 : 5);  // real, ground mirror
                const double ra = q + fc.zz2[va][k], rb = q + fc.zz2[vb][k];
                const double fa = (1.0 - E * fc.ez[va][k]) / ra, fb = (1.0 - E * fc.ez[vb][k]) / rb;
                A[pr] = fc.zz[va][k] * fa - fc.zz[vb][k] * fb;
                Bc[pr] = fa - fb;
            }
            const double dec = c_dec / (fc.nu4[k] * dx + fc.eps2);
            const double c4[4] = {dec * (A[0] - rho * A[1]), dec * A[2], -yL * dec * (Bc[0] - rho * Bc[1]), -yL * dec * Bc[2]};
#pragma unroll
            for (int e = 0; e < 4; ++e) tab[dst + 4 * k + e] = c4[e];
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) s.vtab_ok[b] = 1;  // read by later launches on the same stream only
}

// FlorisInterface.update_wind for masked envs: new free-stream wind, counters untouched (interface.py:663-671)
__global__ void wf_set_wind_kernel(const WfModel m, const WfState s, const uint8_t* __restrict__ mask,
                                   const double* __restrict__ ws, const double* __restrict__ wd) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= m.B || (mask && !mask[b])) return;
    s.ws[b] = ws[b];
    s.wd[b] = wfreset::fmod_py(wd[b], 360.0);
}

// ---------------------------------------------------------------------------------------------------------------
// reset kernels (sampler and state: wf_reset_device.cuh)
// ---------------------------------------------------------------------------------------------------------------
__global__ void wf_sample_reset_kernel(const WfModel m, const WfState s, const uint8_t* __restrict__ mask,
                                       const unsigned long long seed, const long long env_id_offset, const double ti_lo,
                                       const double ti_hi, double* __restrict__ ws, double* __restrict__ wd) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= m.B || (mask && !mask[b])) return;
    if (m.sample_layouts) wfreset::sample_layout(s, b, seed, env_id_offset, m.n_layouts);  // read by the geometry kernel next
    wfreset::sample_wind(s, b, seed, env_id_offset, ti_lo, ti_hi, &ws[b], &wd[b]);
}

// reset per-env scalars/accumulators for masked envs
__global__ void wf_reset_state_kernel(const WfModel m, const WfState s, const uint8_t* __restrict__ mask,
                                      const double* __restrict__ ws, const double* __restrict__ wd) {
    const int b = blockIdx.x;
    if (mask && !mask[b]) return;
    const int T = m.T;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
        const size_t o = (size_t)b * T + t;
        s.yaw[o] = 0.0;
        s.acc[o] = 0.f;
        s.acc_prev[o] = 0.f;
    }
    if (threadIdx.x == 0) {
        wfreset::reset_scalars(s, b, ws[b], wd[b]);
        s.reset_mask[b] = 0;  // an explicit reset supersedes a pending in-kernel auto-reset of this env
    }
}

// ---------------------------------------------------------------------------------------------------------------
// step kernel (basic variant)
// ---------------------------------------------------------------------------------------------------------------
template <typename R, int G>
__global__ void __launch_bounds__(WF_MAX_TURBINES_K)
wf_step_basic_kernel(const int mode, const int env_begin, const WfModel m, const WfState s,
                     const uint8_t* __restrict__ mask, const float* __restrict__ action,
                     const double* __restrict__ yaw_cmd, const WfStepOut out) {
    const int b = blockIdx.x + env_begin;
    if (mask && !mask[b]) return;
    const int T = m.T;
    const int t = threadIdx.x;
    const size_t row = (size_t)b * T;

    constexpr int NP = G * G;  // rotor grid points (case.yaml:16 turbine_grid_points = G), p = G*j + k, j lateral, k vertical
    __shared__ EnvConst<R, G> ec;
    __shared__ SrcRec<R, NP> rec[2];
    __shared__ double sh_yaw[WF_MAX_TURBINES_K];   // new yaw in ORIGINAL order
    __shared__ double sh_red0[WF_MAX_TURBINES_K];  // reward reduction scratch (original order)
    __shared__ double sh_red1[WF_MAX_TURBINES_K];

    const R D = (R)m.D, HH = (R)m.HH;
    const double qD = 0.5 * m.D / 2;  // grid offsets = np.linspace(-qD, qD, G)
    double offs[G];
#pragma unroll
    for (int q = 0; q < G; ++q) offs[q] = grid_off(qD, q, G);

    // ---- env prologue: thread t handles ORIGINAL turbine t (mdp.py:291-319, simple_env.py:64-72) ----------------
    int nm = 0;
    if (mode == WF_MODE_ENV) nm = s.num_moves[b] + 1;
    if (t < T) {
        double ynew;
        if (mode == WF_MODE_ENV) {
            float a = action[row + t];
            const float acc = s.acc[row + t];
            const float acc_c = (m.multi_agent && t != T - 1) ? s.acc_prev[row + t] : acc;
            // actuating_frac = acc / rate / num_moves / dt, evaluated in float32 like numpy does
            const float frac = __fdiv_rn(__fdiv_rn(__fdiv_rn(acc_c, m.rate_f), (float)nm), m.dt_f);
            if (frac >= 0.1f) a = 0.0f;
            if (m.continuous) a = fminf(fmaxf(a, -m.yaw_step_f), m.yaw_step_f);
            else a = __fmul_rn(__fsub_rn(a, 1.0f), m.yaw_step_f);
            const float y0 = fminf(fmaxf((float)s.yaw[row + t], m.yaw_lo_f), m.yaw_hi_f);
            const float y1 = fminf(fmaxf(__fadd_rn(y0, a), m.yaw_lo_f), m.yaw_hi_f);
            s.acc_prev[row + t] = acc;
            s.acc[row + t] = __fadd_rn(acc, fabsf(a));
            ynew = (double)y1;
            s.yaw[row + t] = ynew;
        } else if (mode == WF_MODE_INTERFACE && yaw_cmd) {
            ynew = yaw_cmd[row + t];
            s.yaw[row + t] = ynew;
        } else {
            ynew = s.yaw[row + t];
        }
        sh_yaw[t] = ynew;
    }
    if (t == 0) {
        const double ws = s.ws[b], wd = s.wd[b];
        ec.ws = ws;
        ec.wd = wd;
        const double I0 = s.ti_amb[b];
        ec.I0 = (R)I0;
        const double eps = 0.2 * m.D;
        ec.eps2 = (R)(eps * eps);
        ec.inv_eps2 = (R)(1.0 / (eps * eps));
        double U0[G], usum = 0.0;
        for (int k = 0; k < G; ++k) {
            const double Z = m.HH + offs[k];
            U0[k] = ws * pow(Z / m.HH, m.shear);
            usum += U0[k];
        }
        const double Uinf = usum / G;
        ec.Uinf = (R)Uinf;
        for (int k = 0; k < G; ++k) {
            const double Z = m.HH + offs[k];
            const double dU = ws * (m.shear * pow(1.0 / m.HH, m.shear) * pow(Z, m.shear - 1.0));
            const double lmda = m.D / 8, kappa = 0.41;
            const double lm = kappa * Z / (1 + kappa * Z / lmda);
            const double nu = lm * lm * fabs(dU);
            ec.U0[k] = (R)U0[k];
            ec.nu4[k] = (R)(4 * nu / Uinf);
            const double zc[6] = {-(m.HH + m.D / 2), -(m.HH - m.D / 2), (m.HH + m.D / 2), (m.HH - m.D / 2), -m.HH, m.HH};
            for (int q = 0; q < 6; ++q) ec.zq[q][k] = (R)((Z + zc[q]) + kNumEps);
        }
        ec.vel_top = (R)pow((m.HH + m.D / 2) / m.HH, m.shear);
        ec.vel_bot = (R)pow((m.HH - m.D / 2) / m.HH, m.shear);
    }
    __syncthreads();

    // ---- per-thread state: turbine at sorted position t ----------------------------------------------------------
    R wake[NP], v[NP], w[NP], ti[NP];
    double X = 0.0, Ys = 0.0, yaw_t = 0.0;
    int orig = 0;
    if (t < T) {
        X = s.xs[row + t];
        Ys = s.ys[row + t];
        orig = s.order[row + t];
        yaw_t = sh_yaw[orig];
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) { wake[p] = R(0); v[p] = R(0); w[p] = R(0); ti[p] = ec.I0; }
    const R I0 = ec.I0;
    const R inv_D = M<R>::div(R(1), D);

    // ---- sequential solver over sources ---------------------------------------------------------------------------
    for (int i = 0; i < T; ++i) {
        SrcRec<R, NP>& rc = rec[i & 1];
        if (t == i) {
            // ===== source prologue (A.4, A.5, source part of A.6-A.8) =====
            const double x_i = s.xi[row + i], y_i = s.yi[row + i];
            R u[NP], c3[NP];
#pragma unroll
            for (int p = 0; p < NP; ++p) { u[p] = ec.U0[p % G] - wake[p]; c3[p] = u[p] * u[p] * u[p]; }
            const R avg = M<R>::cbrt(meanN<R, NP>(c3));
            double ctd = interp_table((double)avg, m.tab_ws, m.tab_ct, m.table_len, 0.0001, 0.9999);
            ctd = fmin(fmax(ctd, 0.0001), 0.9999);
            R sy, cy;
            M<R>::sincos((R)(yaw_t * (kPi / 180.0)), &sy, &cy);
            const R ct = (R)ctd * cy;
            const R a = M<R>::div(R(0.5), cy) * (R(1) - M<R>::sqrt(R(1) - ct * cy));
            const R G_top0 = (R)(kPi / 8) * D * ec.vel_top * ec.Uinf * ct;
            const R G_bot0 = (R)(kPi / 8) * D * ec.vel_bot * ec.Uinf * ct;
            const R Gwr = M<R>::div((R)(0.25 * 2 * kPi) * D * (a - a * a) * avg, (R)m.TSR);
            const R Gt = sy * cy * G_top0, Gb = -(sy * cy * G_bot0);

            // A.5 secondary steering on the source's own grid: top (+G_top0), bottom (-G_bot0), wake rotation
            R vt[NP], vb[NP], vc[NP];
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                const int j = p / G, k = p % G;
                const R yL = Lat<R>::get(Ys, y_i, offs[j]) + (R)kNumEps;
                const R yy = yL * yL;
                const R two_pi = R(2.0 * kPi);
                R zz = ec.zq[0][k], r = yy + zz * zz;
                vt[p] = M<R>::div(G_top0 * zz, two_pi * r) * (R(1) - M<R>::exp(-r * ec.inv_eps2));
                zz = ec.zq[1][k]; r = yy + zz * zz;
                vb[p] = M<R>::div(-G_bot0 * zz, two_pi * r) * (R(1) - M<R>::exp(-r * ec.inv_eps2));
                zz = ec.zq[4][k]; r = yy + zz * zz;
                vc[p] = M<R>::div(Gwr * zz, two_pi * r) * (R(1) - M<R>::exp(-r * ec.inv_eps2));
            }
            R val = M<R>::div(R(2) * (meanN<R, NP>(v) - meanN<R, NP>(vc)), meanN<R, NP>(vt) + meanN<R, NP>(vb));
            val = M<R>::min(M<R>::max(val, R(-1)), R(1));
            const R eff_yaw = (R)yaw_t + (R)(180.0 / kPi) * (R(0.5) * M<R>::asin(val));

            // A.6 deflection scalars (opposite sign convention)
            const R g = -eff_yaw;
            R sg, cg;
            M<R>::sincos(g * (R)(kPi / 180.0), &sg, &cg);
            const R sq1ct = M<R>::sqrt(R(1) - ct);            // sqrt(1 - ct)
            const R sq1ctcg = M<R>::sqrt(R(1) - ct * cg);     // sqrt(1 - ct cos(g))
            {
                // uR/(U0 + u0), C0, M0, E0 do not depend on the grid point (U0 cancels)
                const R uR_over = M<R>::div(ct * cg, R(2) * (R(1) - sq1ctcg));
                const R sz0 = D * R(0.5) * M<R>::sqrt(M<R>::div(uR_over, R(1) + sq1ct));
                const R sy0 = sz0 * cg;  // cosd(veer) = 1
                const R C0 = R(1) - sq1ct;
                const R M0 = C0 * (R(2) - C0);
                const R E0 = C0 * C0 - (R)m.e3_112 * C0 + (R)m.e3_13;  // 3 e^(1/12), 3 e^(1/3)
                R th = (R)m.dm * M<R>::div(R(0.3) * (g * (R)(kPi / 180.0)), cg);
                th = th * (R(1) - sq1ctcg);
                rc.sM0 = M<R>::sqrt(M0);
                rc.tan_th = M<R>::tan(th);
                rc.Kc = M<R>::div(th * E0, R(5.2)) * M<R>::sqrt(M<R>::div(sy0 * sz0, M0));
                rc.sy0d = sy0;
                rc.sz0d = sz0;
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    rc.x0d[p] = M<R>::div(D * (cg * (R(1) + sq1ctcg)),
                                          (R)1.4142135623730951 * (R(4) * (R)m.alpha * ti[p] + R(2) * (R)m.beta * (R(1) - sq1ct)));
                    rc.kyd[p] = (R)m.ka * ti[p] + (R)m.kb;
                }
            }

            // own transverse velocities (A.7) -> yaw-added recovery TI update (in place) -> own v, w updated now
            {
                const double dxs = X - x_i;
                R Vp[NP], Wp[NP];
                if (dxs < 0.0) {
#pragma unroll
                    for (int p = 0; p < NP; ++p) { Vp[p] = R(0); Wp[p] = R(0); }
                } else {
                    const R dx = (R)dxs;
#pragma unroll
                    for (int p = 0; p < NP; ++p) {
                        const int j = p / G, k = p % G;
                        const R yL = Lat<R>::get(Ys, y_i, offs[j]) + (R)kNumEps;
                        const R decay = M<R>::div(ec.eps2, ec.nu4[k] * dx + ec.eps2);
                        transverse<R, G>(ec, Gt, Gb, Gwr, yL, k, decay, &Vp[p], &Wp[p]);
                        Wp[p] = M<R>::max(Wp[p], R(0));
                    }
                }
                const R I = ti[0];
                const R aI = avg * I;
                const R kk = M<R>::div(aI * aI, (R)(2.0 / 3.0));
                const R u_term = M<R>::sqrt(R(2) * kk);
                R tv[NP], tw[NP];
#pragma unroll
                for (int p = 0; p < NP; ++p) { tv[p] = v[p] + Vp[p]; tw[p] = w[p] + Wp[p]; }
                const R v_term = meanN<R, NP>(tv), w_term = meanN<R, NP>(tw);
                const R k_total = R(0.5) * (u_term * u_term + v_term * v_term + w_term * w_term);
                const R I_total = M<R>::div(M<R>::sqrt((R)(2.0 / 3.0) * k_total), avg);
                const R I_mix = I_total - I;
#pragma unroll
                for (int p = 0; p < NP; ++p) { ti[p] = ti[p] + R(2) * I_mix; v[p] = tv[p]; w[p] = tw[p]; }
            }

            // A.8 velocity-model scalars with the UPDATED TI (uses yaw_i, opposite sign: cos(-yaw) = cy)
            {
                const R cgv = cy;
                const R uR_over = M<R>::div(ct, R(2) * (R(1) - sq1ct));
                const R sz0 = D * R(0.5) * M<R>::sqrt(M<R>::div(uR_over, R(1) + sq1ct));
                rc.sz0v = sz0;
                rc.sy0v = sz0 * cgv;
                rc.cgv = cgv;
                rc.near_s = R(0.501) * D * M<R>::sqrt(ct * R(0.5));
                rc.ctc = ct * cgv * D * D * R(0.125);
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    rc.x0v[p] = M<R>::div(D * cgv * (R(1) + sq1ct),
                                          (R)1.4142135623730951 * (R(4) * (R)m.alpha * ti[p] + R(2) * (R)m.beta * (R(1) - sq1ct)));
                    rc.kyv[p] = (R)m.ka * ti[p] + (R)m.kb;
                }
            }
            rc.x_i = x_i;
            rc.y_i = y_i;
            rc.ct = ct;
            rc.a = a;
            rc.Gt = Gt;
            rc.Gb = Gb;
            rc.Gwr = Gwr;
            rc.watK = (R)m.ch_const * M<R>::pow(a, (R)m.ch_ai) * M<R>::pow(I0, (R)m.ch_init);
        }
        __syncthreads();
        if (t < T && t != i) {
            const double dxd = X - rc.x_i;
            if (dxd >= 0.0) {
                // ===== target update (A.6-A.8) on the 9 rotor points of turbine t =====
                const R dx = (R)dxd;
                const bool gt01 = X > __dadd_rn(rc.x_i, 0.1);   // near-wake mask bump (SURVEY A.8a)
                const bool gt0 = X > rc.x_i;
                const bool le15 = X <= __dadd_rn(15 * m.D, rc.x_i);
                const R Gt = rc.Gt, Gb = rc.Gb, Gwr = rc.Gwr;
                R dU[NP];
                int cnt = 0;
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    const int j = p / G, k = p % G;
                    const R dyc = Lat<R>::get(Ys, rc.y_i, offs[j]);  // Y - y_i
                    // -- transverse velocities
                    {
                        const R decay = M<R>::div(ec.eps2, ec.nu4[k] * dx + ec.eps2);
                        R Vq, Wq;
                        transverse<R, G>(ec, Gt, Gb, Gwr, dyc + (R)kNumEps, k, decay, &Vq, &Wq);
                        v[p] += Vq;
                        w[p] += M<R>::max(Wq, R(0));
                    }
                    // -- deflection
                    R defl;
                    {
                        const R x0 = rc.x0d[p], ky = rc.kyd[p];
                        const R delta0 = rc.tan_th * x0;
                        const R lin = (R)m.ad + (R)m.bd * dx;
                        if (dx <= x0) {
                            defl = M<R>::div(dx, x0) * delta0 + lin;
                        } else {
                            const R sgy = ky * (dx - x0) + rc.sy0d, sgz = ky * (dx - x0) + rc.sz0d;
                            const R sq = M<R>::sqrt(M<R>::div(sgy * sgz, rc.sy0d * rc.sz0d));
                            const R num = (R(1.6) + rc.sM0) * (R(1.6) * sq - rc.sM0);
                            const R den = (R(1.6) - rc.sM0) * (R(1.6) * sq + rc.sM0);
                            defl = delta0 + M<R>::div(rc.Kc, ky) * M<R>::log(M<R>::div(num, den)) + lin;
                        }
                    }
                    // -- Gauss deficit
                    R deficit = R(0);
                    {
                        const R x0 = rc.x0v[p];
                        const bool far = dx >= x0;
                        const bool near = gt01 && !far;
                        if (near || far) {
                            R sgy, sgz;
                            if (far) {
                                const R ky = rc.kyv[p];
                                sgy = ky * (dx - x0) + rc.sy0v;
                                sgz = ky * (dx - x0) + rc.sz0v;
                            } else {
                                const R up = M<R>::div(dx, x0), down = M<R>::div(x0 - dx, x0);
                                sgy = down * rc.near_s + up * rc.sy0v;
                                sgz = down * rc.near_s + up * rc.sz0v;
                            }
                            const R dy = dyc - defl;
                            const R dz = (R)(offs[k]);
                            const R r = M<R>::div(dy * dy, R(2) * sgy * sgy) + M<R>::div(dz * dz, R(2) * sgz * sgz);
                            R d = R(1) - M<R>::div(rc.ctc, sgy * sgz);
                            d = M<R>::min(M<R>::max(d, R(0)), R(1));
                            deficit = (R(1) - M<R>::sqrt(d)) * M<R>::exp(-r);
                        }
                    }
                    dU[p] = deficit * ec.U0[k];
                    cnt += dU[p] > R(0.05);
                }
                // -- Crespo-Hernandez wake-added TI (A.8e): only non-zero when the wake overlaps the rotor
                R ti_add_base = R(0);
                if (cnt > 0 && gt0 && le15) {
                    const R dxp = dx + ((dxd <= 0.1) ? R(1) : R(0));
                    const R wat = rc.watK * M<R>::pow(dxp * inv_D, (R)m.ch_down);
                    ti_add_base = ((R)cnt * (R)(1.0 / NP)) * wat;
                }
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    const int j = p / G;
                    const R dyc = Lat<R>::get(Ys, rc.y_i, offs[j]);
                    const R ta = (M<R>::abs(dyc) < R(2) * D) ? ti_add_base : R(0);
                    ti[p] = M<R>::max(M<R>::sqrt(ta * ta + I0 * I0), ti[p]);
                    wake[p] = M<R>::hypot(wake[p], dU[p]);
                }
            }
        }
    }

    // ---- epilogue: measures (interface.py:565-577, 622-648), power (A.10), reward (simple_env.py:78-85) -----------
    const bool env = (mode != WF_MODE_INTERFACE);
    R p_out = R(0), lsum = R(0);
    if (t < T) {
        R u[NP], c3[NP], dd[NP];
#pragma unroll
        for (int p = 0; p < NP; ++p) { u[p] = ec.U0[p % G] - wake[p]; c3[p] = u[p] * u[p] * u[p]; }
        const R avg = M<R>::cbrt(meanN<R, NP>(c3));
        R sy, cy;
        M<R>::sincos((R)(yaw_t * (kPi / 180.0)), &sy, &cy);
        const double veff = (double)((R)cbrt(m.rho / m.ref_rho) * avg * M<R>::pow(cy, (R)(m.pP / 3.0)));
        const double pw = interp_table(veff, m.tab_ws, m.tab_pw, m.table_len, 0.0, 0.0) * m.ref_rho;  // [W]
#pragma unroll
        for (int p = 0; p < NP; ++p) dd[p] = (R)ec.wd - (R)(180.0 / kPi) * M<R>::atan2(v[p], u[p]);
        R wdl = meanN<R, NP>(dd);
        R wsl = avg;
        const R ti_m = meanN<R, NP>(ti);
        R sd[3];
        {
            const R* arrs[3] = {u, v, w};
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                const R mu = meanN<R, NP>(arrs[q]);
                R d2[NP];
#pragma unroll
                for (int p = 0; p < NP; ++p) { const R e = arrs[q][p] - mu; d2[p] = e * e; }
                sd[q] = M<R>::sqrt(meanN<R, NP>(d2));
            }
        }
        R loads[4] = {ti_m, sd[0], sd[1], sd[2]};
        if (env) {
            p_out = (R)(pw / 1e6);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (sizeof(R) == 8) loads[q] = (R)(((double)loads[q] * 1e7) / 1e7);
                lsum += M<R>::abs(loads[q]);
            }
        } else {
            p_out = (R)pw;
#pragma unroll
            for (int q = 0; q < 4; ++q) loads[q] = (R)((double)loads[q] * 1e7);
        }
        if (mode == WF_MODE_WARMUP) {  // start state is clipped to the observation space (mdp.py:263-266)
            wsl = M<R>::min(M<R>::max(wsl, R(3)), R(28));
            wdl = M<R>::min(M<R>::max(wdl, R(0)), R(360));
        }
        const size_t o = row + orig;
        if (out.yaw) {
            R yv = (R)yaw_t;
            if (mode == WF_MODE_WARMUP) yv = M<R>::min(M<R>::max(yv, (R)m.yaw_lo_f), (R)m.yaw_hi_f);
            ((R*)out.yaw)[o] = yv;
        }
        if (out.wind_speed) ((R*)out.wind_speed)[o] = wsl;
        if (out.wind_direction) ((R*)out.wind_direction)[o] = wdl;
        if (out.power) ((R*)out.power)[o] = p_out;
        if (out.load) {
            R* L = (R*)out.load + 4 * o;
#pragma unroll
            for (int q = 0; q < 4; ++q) L[q] = loads[q];
        }
        sh_red0[orig] = (double)p_out;
        sh_red1[orig] = (double)lsum;
    }
    __syncthreads();
    if (t == 0) {
        const int it = s.num_iter[b] + 1;
        s.num_iter[b] = it;
        if (out.truncated) out.truncated[b] = (uint8_t)(it == m.max_iter);
        double fw0 = ec.ws, fw1 = ec.wd;
        if (mode == WF_MODE_WARMUP) {
            fw0 = fmin(fmax(fw0, 3.0), 28.0);
            fw1 = fmin(fmax(fw1, 0.0), 360.0);
        }
        if (out.freewind) {
            ((R*)out.freewind)[2 * b] = (R)fw0;
            ((R*)out.freewind)[2 * b + 1] = (R)fw1;
        }
        if (mode == WF_MODE_ENV) {
            s.num_moves[b] = nm;
            const double wn = s.ws_norm[b];
            const double w3 = wn * wn * wn;
            double sp = 0.0, sl = 0.0;
            for (int q = 0; q < T; ++q) {
                sp += sh_red0[q] * 1e3 / w3;
                sl += sh_red1[q];
            }
            double reward = sp / T - m.load_coef * (sl / (4.0 * T));
            if (m.shaper == 1) {
                reward = (reward - m.shaper_reference) / m.shaper_reference;
            } else if (m.shaper == 2) {
                const double ref = s.shaper_ref[b];
                const double shaped = (ref == 0.0) ? 0.0 : (reward - ref) / ref;
                s.shaper_ref[b] = reward;
                reward = shaped;
            }
            if (!isfinite(reward)) s.nonfinite[b] += 1;
            if (out.reward) ((R*)out.reward)[b] = (R)reward;
            wfreset::episode_account(s, b, (double)(R)reward, it == m.max_iter);
            s.ws_norm[b] = ec.ws;  // next state's freewind measurement (mdp.py:280)
        }
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------
static inline int round_up_warp(int n) { return (n + 31) / 32 * 32; }

cudaError_t wf_launch_geometry(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_cs_override,
                               cudaStream_t stream, bool autoreset_draw) {
    wf_geometry_kernel<<<m.B, round_up_warp(m.T), 0, stream>>>(m, s, d_mask, d_cs_override, autoreset_draw ? 1 : 0);
    return cudaGetLastError();
}

cudaError_t wf_launch_vortex_table(const WfModel& m, const WfFastConst64& fc, const WfState& s, const uint8_t* d_mask,
                                   cudaStream_t stream) {
    if (!s.vtab || m.T < 2) return cudaSuccess;
    wf_vortex_table_kernel<<<m.B, 256, 0, stream>>>(m, fc, s, d_mask);
    return cudaGetLastError();
}

cudaError_t wf_launch_set_wind(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_ws,
                               const double* d_wd, cudaStream_t stream) {
    wf_set_wind_kernel<<<(m.B + 127) / 128, 128, 0, stream>>>(m, s, d_mask, d_ws, d_wd);
    return cudaGetLastError();
}

cudaError_t wf_launch_sample_reset(const WfModel& m, const WfState& s, const uint8_t* d_mask, unsigned long long seed,
                                   long long env_id_offset, double ti_lo, double ti_hi, double* d_ws, double* d_wd,
                                   cudaStream_t stream) {
    wf_sample_reset_kernel<<<(m.B + 127) / 128, 128, 0, stream>>>(m, s, d_mask, seed, env_id_offset, ti_lo, ti_hi, d_ws, d_wd);
    return cudaGetLastError();
}

cudaError_t wf_launch_reset_state(const WfModel& m, const WfState& s, const uint8_t* d_mask, const double* d_ws,
                                  const double* d_wd, cudaStream_t stream) {
    wf_reset_state_kernel<<<m.B, 32, 0, stream>>>(m, s, d_mask, d_ws, d_wd);
    return cudaGetLastError();
}

cudaError_t wf_launch_step_basic(int precision, int mode, const WfModel& m, const WfState& s, const uint8_t* d_mask,
                                 const float* d_action, const double* d_yaw_cmd, const WfStepOut& out,
                                 int env_begin, int env_count, cudaStream_t stream) {
    const int threads = round_up_warp(m.T);
#define WF_GO(R_, G_) wf_step_basic_kernel<R_, G_><<<env_count, threads, 0, stream>>>(mode, env_begin, m, s, d_mask, d_action, d_yaw_cmd, out)
    if (m.G == 5) { if (precision == 0) WF_GO(double, 5); else WF_GO(float, 5); }
    else { if (precision == 0) WF_GO(double, 3); else WF_GO(float, 3); }
#undef WF_GO
    return cudaGetLastError();
}

cudaError_t wf_step_basic_attributes(int precision, cudaFuncAttributes* attr, int* ctas_per_sm, int threads) {
    cudaError_t e;
    if (precision == 0) {
        e = cudaFuncGetAttributes(attr, wf_step_basic_kernel<double, 3>);
        if (e != cudaSuccess) return e;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, wf_step_basic_kernel<double, 3>, threads, 0);
    }
    e = cudaFuncGetAttributes(attr, wf_step_basic_kernel<float, 3>);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, wf_step_basic_kernel<float, 3>, threads, 0);
}
