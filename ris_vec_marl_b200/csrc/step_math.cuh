// The per-step arithmetic of the rollout kernels, written once.
// Reference: Simulation-SARL/Environment.py:318-359 (localProcRev, step) and
//            Simulation-MARL-BCD/Environment.py:555-731.
//
// Every helper is the exact operation sequence its callers used to spell out: the same intrinsics, the same
// operand order, no other rounding or contraction.  The kernels keep what differs between them (thread mapping,
// which lane writes what, how inputs arrive); what one step computes from its inputs lives here.
#pragma once
#include "common.cuh"

namespace risvec {

__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }

// ln(1 + x) for x >= 0 through the SFU: MUFU.LG2 of the rounded sum.  Absolute error <= 6e-8 near
// zero (the rounding of 1 + x) and ~2^-22 relative elsewhere -- inside the SARL rate tolerance
// (tests/parity.py), and SARL has no threshold on the rate itself.
__device__ __forceinline__ float log1p_sfu(float x) { return __fmul_rn(__log2f(__fadd_rn(1.0f, x)), 0.693147180559945309f); }

// cbrt(x) for x >= 0: SFU seed exp2(log2(x) / 3) (rel. error ~5e-7) + one Newton step
// y <- y - (y^3 - x) / (3 y^2), which brings it to ~1 ulp; cbrt(0) = 0.
__device__ __forceinline__ float cbrt_sfu(float x) {
    const float y = exp2f(__fmul_rn(__log2f(x), 0.333333343f));
    const float y2 = __fmul_rn(y, y);
    const float r = __fdividef(__fmaf_rn(-y2, y, x), __fmul_rn(3.0f, y2));
    return (x > 0.f) ? __fadd_rn(y, r) : 0.f;
}

// ln(1 + x) for x >= 0 with relative error < 1e-6 everywhere: far-user NOMA SINRs are << 1, where
// 1 + x would lose x, so below 1/4 a degree-11 series in x is used (truncation < 2e-8 relative) and
// above it MUFU.LG2 of (1 + x) (there |log2| >= 0.32 and the unit's absolute error 2^-22 is < 6e-7
// relative).  Both branches are evaluated, one select; about a third of the library's log1pf.
__device__ __forceinline__ float log1p_pos(float x) {
    const float big = __fmul_rn(__log2f(__fadd_rn(1.0f, x)), 0.693147180559945309f);
    float p = 0.0909090909f;                       // 1/11
    p = __fmaf_rn(p, x, -0.1f);
    p = __fmaf_rn(p, x, 0.111111111f);
    p = __fmaf_rn(p, x, -0.125f);
    p = __fmaf_rn(p, x, 0.142857143f);
    p = __fmaf_rn(p, x, -0.166666667f);
    p = __fmaf_rn(p, x, 0.2f);
    p = __fmaf_rn(p, x, -0.25f);
    p = __fmaf_rn(p, x, 0.333333333f);
    p = __fmaf_rn(p, x, -0.5f);
    p = __fmaf_rn(p, x, 1.0f);
    return x < 0.25f ? __fmul_rn(p, x) : big;
}

// ---------------------------------------------------------------------------------------
// Queue recursions as max-plus maps (time-parallel kernels)
// ---------------------------------------------------------------------------------------
// max-plus affine map x -> max(x + a, b): the DataBuf step x -> max(x - d, 0) + inc is (inc - d, inc)
struct MaxPlus {
    double a, b;
};
__device__ __forceinline__ MaxPlus mp_then(const MaxPlus& f, const MaxPlus& g) {  // g after f
    MaxPlus r;
    r.a = f.a + g.a;
    const double fb = f.b + g.a;
    r.b = fb > g.b ? fb : g.b;
    return r;
}
__device__ __forceinline__ double mp_apply(const MaxPlus& f, double x) {
    const double y = x + f.a;
    return y > f.b ? y : f.b;
}

// Inclusive scan of the composed maps f of a group of W consecutive lanes (idx = position in the group, the
// lanes hold consecutive runs of steps): ex = the maps of the lanes before mine, all = the whole group's map.
// (The rounds are unrolled by recursion, not by a loop: the compiler then sees the literal offsets, and the
// code is the same as the written-out scan's.)
template <int W, int O = 1>
__device__ __forceinline__ void mp_scan(MaxPlus f, int idx, MaxPlus& ex, MaxPlus& all) {
    if constexpr (O < W) {
        const MaxPlus q{__shfl_up_sync(kFull, f.a, O, W), __shfl_up_sync(kFull, f.b, O, W)};
        const MaxPlus fo = mp_then(q, f);
        if (idx >= O) f = fo;
        mp_scan<W, 2 * O>(f, idx, ex, all);
    } else {
        ex = MaxPlus{__shfl_up_sync(kFull, f.a, 1, W), __shfl_up_sync(kFull, f.b, 1, W)};
        all = MaxPlus{__shfl_sync(kFull, f.a, W - 1, W), __shfl_sync(kFull, f.b, W - 1, W)};
    }
}

// Geometry phasors w(v, m0 + i) = z^(m0 + i), i < MPL, of the lane's vehicle (SARL:134-145) as float32 element
// pairs: float64 from one sincospi per lane, rounded once; elements from m1 on and inactive lanes are 0.
template <int MPL>
__device__ __forceinline__ void phasor_pairs(const Dims& d, const State& s, size_t ev, bool act, int m0, int m1,
                                             float2 (&WX)[MPL / 2], float2 (&WY)[MPL / 2]) {
    const double2 z = unit_phasor64(act ? d.angle_BR - s.angle[ev] : 0.0);
    double2 wv = cpow64(z, (unsigned)m0);
#pragma unroll
    for (int i = 0; i < MPL; ++i) {
        const bool on = act && (m0 + i < m1);
        const float re = on ? (float)wv.x : 0.f, im = on ? (float)wv.y : 0.f;
        if (i & 1) { WX[i >> 1].y = re; WY[i >> 1].y = im; }
        else       { WX[i >> 1].x = re; WY[i >> 1].x = im; }
        wv = cmul64(wv, z);
    }
}

// ---------------------------------------------------------------------------------------
// MARL step (MARL:555-731)
// ---------------------------------------------------------------------------------------
// a / den correctly rounded, without the library's special-case branches (Markstein: q0 = RN(a*r),
// rem = a - q0*b exactly by FMA, q = RN(q0 + rem*r) with r = RN(1/den))
__device__ __forceinline__ double div_rn_fma(double a, double den, double rden) {
    const double q0 = __dmul_rn(a, rden);
    return __fma_rn(__fma_rn(-q0, den, a), rden, q0);
}

// ---------------------------------------------------------------------------------------
// SARL step (SARL:318-359)
// ---------------------------------------------------------------------------------------
// scalar constants of the step in float64, rounded once: the TMA and tcgen05 kernels take them from the host as
// kernel parameters (constant-bank operands, no registers), the FP32-pipe kernels form them on the device (device
// and host cbrt need not round alike)
struct SarlConsts {
    float c_dt;    // time_fast * bandwidth * 1000        (SARL:160, data_t = rate * c_dt)
    float c_dp;    // cbrt(1 / k) * time_fast / L / 1000  (SARL:331)
    float c_rev;   // 1000 * L / time_fast * cbrt(k)      (SARL:318-319)
    float nt1, nt2;  // -t_factor1, -t_factor2            (SARL:341-352)
    float pen1, pen2;
    float lam;     // Poisson arrival rate (on-device draws)
    double tf;     // time_fast
};
__host__ __device__ inline SarlConsts sarl_consts(const risvec_params_t& p) {
    SarlConsts c;
    c.c_dt = (float)(p.time_fast * p.bandwidth * 1000.0);
    c.c_dp = (float)(cbrt(1.0 / p.k) * p.time_fast / p.L / 1000.0);
    c.c_rev = (float)(1000.0 * p.L / p.time_fast * cbrt(p.k));
    c.nt1 = -(float)p.t_factor1;
    c.nt2 = -(float)p.t_factor2;
    c.pen1 = (float)p.penalty1;
    c.pen2 = (float)p.penalty2;
    c.lam = (float)p.rate;
    c.tf = p.time_fast;
    return c;
}

// rate = ln(1 + a0 * coef * |S|^2) (SARL:159), data_t = rate * c_dt, data_p = cbrt(a1) * c_dp (SARL:331) of two
// steps in packed fp32x2, from Re S and Im S
__device__ __forceinline__ void sarl_rate2(float2 re, float2 im, float2 a0, float2 a1, float coef, const SarlConsts& c,
                                           float2& rate, float2& dt, float2& dp) {
    const float2 g2 = __ffma2_rn(re, re, __fmul2_rn(im, im));
    const float2 y = __fadd2_rn(f2(1.0f), __fmul2_rn(a0, __fmul2_rn(f2(coef), g2)));
    rate = __fmul2_rn(make_float2(__log2f(y.x), __log2f(y.y)), f2(0.693147180559945309f));
    dt = __fmul2_rn(rate, f2(c.c_dt));
    dp = __fmul2_rn(make_float2(cbrt_sfu(a1.x), cbrt_sfu(a1.y)), f2(c.c_dp));
}

// One step of the DataBuf recursion from its true start value `cur` (dd = data_t + data_p, inc = the arrivals):
// the terms the reward needs, and DataBuf after the step (SARL:333-356).  A step with !ok leaves `cur` alone.
__device__ __forceinline__ void sarl_settle(double& cur, double dd, float dp, double inc, bool ok, float& overd,
                                            float& nbf, float& barg, bool& pos, float& curf) {
    const double raw = __dsub_rn(cur, dd);  // SARL:334
    const bool neg = raw < 0.0;
    pos = raw > 0.0;
    barg = fmaxf(0.f, (float)(raw + (double)dp));  // argument of localProcRev (SARL:337)
    const float rawf = (float)raw;
    overd = fmaxf(0.f, -rawf);                      // over_data = -DataBuf where it went negative
    nbf = fmaxf(0.f, rawf);
    if (ok) cur = __dadd_rn(neg ? 0.0 : raw, inc);  // SARL:354-356
    curf = (float)cur;
}

// localProcRev of the settled steps (SARL:336-339; over_power where the buffer went negative) and the base reward
// -t_factor1 (a0 + a1) - t_factor2 DataBuf (SARL:341) of two steps in packed fp32x2
__device__ __forceinline__ void sarl_reward2(float2 barg, float2 nbf, float2 a0, float2 a1, const SarlConsts& c,
                                             float2& op, float2& base2) {
    const float2 b = __fmul2_rn(barg, f2(c.c_rev));
    const float2 b3 = __fmul2_rn(__fmul2_rn(b, b), b);
    op = __fadd2_rn(a1, make_float2(-b3.x, -b3.y));
    base2 = __ffma2_rn(nbf, f2(c.nt2), __fmul2_rn(__fadd2_rn(a0, a1), f2(c.nt1)));
}

// What one step leaves in the per-vehicle state (SarlLast of the last step is written back after the rollout)
struct SarlLast {
    float rate, data_t, data_p, overp, overd;
    int arr;
};

// The sequential part of one scalar SARL step (SARL:333-358) from rate and data_p: updates DataBuf in `buf`.
// ru = the vehicle's reward term before the mean over the vehicles.
struct SarlStep {
    float data_t, overp, overd, ru;
};
__device__ __forceinline__ SarlStep sarl_step(double& buf, float rate, float data_p, float a0, float a1, int arr,
                                              float c_dt, float c_rev, float t1, float t2, float pen1, float pen2,
                                              double tf) {
    SarlStep o;
    o.data_t = __fmul_rn(rate, c_dt);
    const double raw = __dsub_rn(buf, __dadd_rn((double)o.data_t, (double)data_p));  // SARL:334
    const bool neg = raw < 0.0;
    const float b = __fmul_rn((float)fmax(0.0, raw + (double)data_p), c_rev);
    o.overp = neg ? __fsub_rn(a1, __fmul_rn(__fmul_rn(b, b), b)) : 0.f;  // SARL:336-339
    o.overd = neg ? (float)(-raw) : 0.f;
    const double nb = neg ? 0.0 : raw;
    const float base = __fsub_rn(-__fmul_rn(t1, __fadd_rn(a0, a1)), __fmul_rn(t2, (float)nb));
    const float pen = (nb > 0.0) ? pen1 : ((o.overd > 2.0f) ? pen2 : 0.f);  // SARL:343-352
    o.ru = __fsub_rn(base, pen);
    buf = __dadd_rn(nb, __dmul_rn(__dmul_rn((double)arr, tf), 1000.0));  // SARL:354-356
    return o;
}

// the six optional per-step traces of one vehicle (DataBuf after the step, then the step's values)
__device__ __forceinline__ void sarl_store_traces(const risvec_sarl_out_t& out, size_t tev, float buf, const SarlLast& l) {
    if (out.DataBuf != nullptr) out.DataBuf[tev] = buf;
    if (out.data_t != nullptr) out.data_t[tev] = l.data_t;
    if (out.data_p != nullptr) out.data_p[tev] = l.data_p;
    if (out.over_power != nullptr) out.over_power[tev] = l.overp;
    if (out.over_data != nullptr) out.over_data[tev] = l.overd;
    if (out.rate != nullptr) out.rate[tev] = l.rate;
}

// the reference object's per-vehicle attributes after the last step
__device__ __forceinline__ void sarl_store_last(const State& s, size_t ev, const SarlLast& l) {
    s.rate[ev] = l.rate;
    s.data_t[ev] = l.data_t;
    s.data_p[ev] = l.data_p;
    s.over_power[ev] = l.overp;
    s.over_data[ev] = l.overd;
    s.data_r[ev] = l.arr;
}

}  // namespace risvec
