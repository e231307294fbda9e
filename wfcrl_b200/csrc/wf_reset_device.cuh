// Device-side reset of one env, shared by the reset kernels (wf_kernels.cu) and by the step kernels' in-kernel auto-reset
// (wf_fast.cu, wf_fast64.cu): the reference's reset distribution from a counter-based generator + the state zeroing of
// WindFarmMDP.reset (mdp.py:233-271).
#pragma once
#include "wf_device.cuh"

#include <math.h>

namespace wfreset {

// python float % for a positive modulus
__device__ __forceinline__ double fmod_py(double a, double m) {
    double r = fmod(a, m);
    if (r != 0.0 && r < 0.0) r += m;
    return r;
}

// reset sampler: the reference's reset distribution (mdp.py:242-258) from a counter-based generator
// Philox4x32-10 (Salmon et al., SC'11).  key = the user's 64-bit seed, counter = (global env id lo, hi, episode index
// of that env, draw index): every (env, episode) owns its words no matter how the envs are sharded over handles or
// GPUs, so 1/2/4/8-GPU runs reset to identical winds (SURVEY 8e).
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

// 53-bit uniform in [0, 1) from two words (the construction numpy's Generator.random uses on 64-bit output)
__device__ __forceinline__ double u53(unsigned a, unsigned b) {
    return (double)(((unsigned long long)(a >> 5) << 26) | (unsigned long long)(b >> 6)) * (1.0 / 9007199254740992.0);
}


// The draw of (env b, its current episode index): wind speed = clip(8 * Weibull(k = 8), 3, 28) by inversion (mdp.py:242-247),
// wind direction = clip(N(270, 20) % 360, 0, 360) (mdp.py:253-258) by Box-Muller, optionally ambient TI ~ U(ti_lo, ti_hi)
// (extension, BASELINE.json configs[2]; the reference fixes it, case.yaml:33).  Advances the env's episode counter.
__device__ __forceinline__ void sample_wind(const WfState& s, int b, unsigned long long seed, long long env_id_offset,
                                            double ti_lo, double ti_hi, double* ws, double* wd) {
    const unsigned long long gid = (unsigned long long)(env_id_offset + b);
    const unsigned ep = (unsigned)s.episode[b];
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    const uint4 r0 = philox4x32_10(make_uint4((unsigned)gid, (unsigned)(gid >> 32), ep, 0u), key);
    const uint4 r1 = philox4x32_10(make_uint4((unsigned)gid, (unsigned)(gid >> 32), ep, 1u), key);
    const double e1 = -log1p(-u53(r0.x, r0.y));  // Weibull(k) = Exp(1)^(1/k)
    *ws = fmin(fmax(8.0 * pow(e1, 0.125), 3.0), 28.0);
    const double rad = sqrt(-2.0 * log1p(-u53(r0.z, r0.w)));
    const double z = rad * cospi(2.0 * u53(r1.x, r1.y));
    *wd = fmin(fmax(fmod_py(270.0 + 20.0 * z, 360.0), 0.0), 360.0);
    if (ti_hi > ti_lo) s.ti_amb[b] = ti_lo + (ti_hi - ti_lo) * u53(r1.z, r1.w);
    s.episode[b] = (int)(ep + 1u);
}

// Layout draw of the same (env b, episode index): id = floor(u53 * L) from draw word 2 of sample_wind's key and counter, so
// the winds and TI of a reset are the same whether layouts are drawn or not.  Call BEFORE sample_wind advances the episode
// counter.  u53 < 1 rounds below L after the product, so the id is in [0, L).
__device__ __forceinline__ void sample_layout(const WfState& s, int b, unsigned long long seed, long long env_id_offset,
                                              int n_layouts) {
    const unsigned long long gid = (unsigned long long)(env_id_offset + b);
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32));
    const uint4 r2 = philox4x32_10(make_uint4((unsigned)gid, (unsigned)(gid >> 32), (unsigned)s.episode[b], 2u), key);
    s.layout_id[b] = (int)floor(u53(r2.x, r2.y) * n_layouts);
}

// per-env scalars of a reset (one thread); the per-turbine arrays (yaw, acc, acc_prev) are zeroed by the caller's threads
__device__ __forceinline__ void reset_scalars(const WfState& s, int b, double ws, double wd) {
    s.ws[b] = ws;
    s.wd[b] = fmod_py(wd, 360.0);                // interface.py:664
    s.ws_norm[b] = fmin(fmax(ws, 3.0), 28.0);    // start_state is clipped to the observation space (mdp.py:266)
    s.num_iter[b] = 0;
    s.num_moves[b] = 0;
    // WindFarmEnv.reset calls reward_shaper.reset(), and StepPercentage.reset() puts its reference back to 0.0 whatever
    // the constructor argument was (rewards.py:45-46): the first shaped reward of every episode is 0
    s.shaper_ref[b] = 0.0;
    s.ep_return[b] = 0.0;                        // an explicit reset abandons the running episode
    s.ep_len[b] = 0;
}

// Episode bookkeeping of one env step (one thread): accumulate the reward; a truncating step closes the episode into the env's
// finished-episode sums (what VecWindFarmEnv.episode_statistics reduces and all-gathers) and starts the next one at zero.
__device__ __forceinline__ void episode_account(const WfState& s, int b, double reward, bool truncated) {
    double er = s.ep_return[b] + reward;
    int el = s.ep_len[b] + 1;
    if (truncated) {
        s.fin_sum[b] += er;
        s.fin_sumsq[b] += er * er;
        s.fin_n[b] += 1;
        s.fin_len[b] += el;
        er = 0.0;
        el = 0;
    }
    s.ep_return[b] = er;
    s.ep_len[b] = el;
}

// In-kernel auto-reset of a step kernel (one thread): zero the per-env counters and mark the env; the wind of its next episode
// is drawn by the geometry kernel of wf_autoreset_finish (autoreset_wind), which keeps double-precision math out of the step
// kernels.  The per-turbine arrays (yaw, acc, acc_prev) are zeroed by the caller's threads.
__device__ __forceinline__ void autoreset_mark(const WfState& s, int b) {
    s.num_iter[b] = 0;
    s.num_moves[b] = 0;
    s.shaper_ref[b] = 0.0;
    s.reset_mask[b] = 1;
}

// second half, first thing in the geometry kernel of a marked env: draw the layout id (when sampling is on) and the wind,
// finish the scalar reset
__device__ __forceinline__ void autoreset_wind(const WfModel& m, const WfState& s, int b) {
    if (m.sample_layouts) sample_layout(s, b, m.ar_seed, m.ar_offset, m.n_layouts);
    double ws, wd;
    sample_wind(s, b, m.ar_seed, m.ar_offset, m.ar_ti_lo, m.ar_ti_hi, &ws, &wd);
    s.ws[b] = ws;
    s.wd[b] = fmod_py(wd, 360.0);
    s.ws_norm[b] = fmin(fmax(ws, 3.0), 28.0);
}

}  // namespace wfreset
