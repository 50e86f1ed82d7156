// Fused T-step rollouts of Environ.step for E env instances (T = 1 is a plain step).
// Reference: Simulation-MARL-BCD/Environment.py:331-372,547-731 and
//            Simulation-SARL/Environment.py:149-171,318-359.
//
// Thread mapping: an env owns VP = pow2ceil(V) adjacent lanes of one warp (lane v = vehicle v),
// so a warp carries 32 / VP envs and every cross-vehicle term (NOMA partner lookup, sum of edge
// cycles, means) is a segmented warp shuffle.  State (DataBuf, MEC queue, gains, phasor table)
// lives in registers for the whole rollout; per step only actions / phases / arrivals stream
// in from HBM and the requested traces stream out.
#pragma once
#include <type_traits>

#include "common.cuh"
#include "step_math.cuh"

namespace risvec {

constexpr int kRisvecStatSlots = 64;  // == RISVEC_STAT_SLOTS: one 256-byte line pair per slot
struct MarlArgs {
    int T;
    const float* action;   // [T,E,2,V]
    const int* partner;    // [E,V]
    const int* ngroups;    // [E]
    const int* arrivals;   // [T,E,V] or null
    risvec_marl_out_t out;
    const float* in_rec;   // packed layout: [T,E,RISVEC_MARL_IN_WORDS]  (see include/risvec.h)
    float* out_rec;        // packed layout: [T,E,RISVEC_MARL_OUT_WORDS]
    // fused driver step (risvec_step_marl_fused, SURVEY.md 8f row 1; k_marl_v8 only): `raw` = the actors' tanh
    // outputs [T,E,V,2] mapped in the prologue instead of reading `action`; `obs` [E,V,5] = marl_get_state of the
    // state after the last step, written in the epilogue
    const float* raw;
    float* obs;
    // statistics accumulator attached to the handle (risvec_attach_stats_accumulator): kRisvecStatSlots slots of 32
    // doubles; kernels that fold the statistics pass add the sums of their last step into slot blockIdx.x % slots
    double* stats_slots;
};

struct SarlArgs {
    int T;
    const float* action;  // [T,E,2,V]
    const float* phase;   // [T,E,M]
    const int* arrivals;  // [T,E,V] or null
    risvec_sarl_out_t out;
    const float* in_rec;  // packed layout: [T,E,24 + M]  (see include/risvec.h)
    float* out_rec;       // packed layout: [T,E,RISVEC_SARL_OUT_WORDS]
    float* g2;            // [T,E,V] scratch |S_v|^2 between the cascade and scan kernels (large M)
    int t_chunk;          // steps per block of the cascade kernel (even)
    // fused driver step (risvec_step_sarl_fused, SURVEY.md 8f row 1; k_sarl_mma only): `raw` = the actor's tanh
    // outputs [T,E,2V+M] mapped in the prologue instead of reading `action` / `phase`; `obs` [E,V,M/V+5] =
    // get_state of the state after the last step, written in the epilogue
    const float* raw;
    float* obs;
    double* stats_slots;  // as in MarlArgs
};

__device__ inline int draw_arrival(const Dims& d, int e, int v, long long step, float lam) {
    const uint4 r = rng_draw(d, e, (unsigned long long)step, (unsigned)v, kRngArrival);
    return poisson_inv(lam, u01f(r.x));
}

// ---------------------------------------------------------------------------------------
// MARL step (row a11 + a10 of SURVEY.md 8a)
// ---------------------------------------------------------------------------------------
// PE: per-env step parameters from the attached table `envp` (risvec_attach_env_params); unused without PE
template <int VP, bool PE = false>
__global__ void __launch_bounds__(128) k_marl_rollout(Dims d, State s, risvec_params_t p, MarlArgs a,
                                                      const double* __restrict__ envp) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int e = gtid / VP, v = gtid % VP;
    const int E = d.E, V = d.V;
    if constexpr (PE) env_params_marl(p, env_param_row(envp, min(e, E - 1)));
    const bool env_ok = e < E;
    const bool act = env_ok && v < V;
    const size_t ev = (size_t)e * V + v;

    // ---- per-rollout state -> registers
    double buf = act ? s.databuf[ev] : 0.0;
    const double g = act ? s.gains[ev] : 0.0;
    const int code = act ? a.partner[ev] : RISVEC_PARTNER_NONE;
    const int ng = env_ok ? a.ngroups[e] : 1;
    double Q = env_ok ? s.mecq[e] : 0.0;
    const long long step0 = env_ok ? s.step_ctr[e] : 0;

    const bool paired = code >= 0;
    const bool second = paired && (code & RISVEC_PARTNER_SECOND);
    int other = paired ? (code & (RISVEC_PARTNER_SECOND - 1)) : v;
    other = min(max(other, 0), VP - 1);
    const int src = (lane & ~(VP - 1)) + other;
    const double g_o = __shfl_sync(kFull, g, src);
    // MARL:355: the first listed user is "near" only if its gain is strictly larger
    const bool first_near = second ? (g_o > g) : (g > g_o);
    const bool near = paired ? (second ? !first_near : first_near) : true;
    const float gn = (float)(g / p.noise_power);
    const float frac = (float)(1.0 / (double)max(1, ng));  // MARL:341-342
    const bool scheduled = code != RISVEC_PARTNER_NONE;

    // ---- constants
    const float ps = (float)p.power_scale, Pmax = (float)p.P_max;
    const float c_dt = (float)(p.time_fast * p.bandwidth * 1000.0);
    const float c_thr = (float)(p.bandwidth * 1000.0);
    double floor_d = p.cpu_share_floor;
    if (!isfinite(floor_d)) floor_d = 0.10;
    floor_d = fmax(0.0, fmin(floor_d, 0.95));
    const float floor_f = (float)floor_d;
    const double Cpb = p.cycles_per_bit;
    const double kbit2cyc_den = Cpb * 1000.0;
    const double edge_cap = p.f_edge_max * p.time_fast;
    const float inv_fedge = (float)(1.0 / (p.f_edge_max + 1e-12));
    const float inv_tf = (float)(1.0 / p.time_fast);
    const float wd = (float)p.w_d, we = (float)p.w_e, pen = (float)p.qos_penalty, clipv = (float)p.reward_clip;
    const float Rmin = (float)p.R_min_bpsHz, Dmax = (float)p.D_max_s;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;

    float o_rate = 0.f, o_dt = 0.f, o_dp = 0.f, o_rew = 0.f, o_glob = 0.f, o_overp = 0.f;
    int o_arr = 0;

    for (int t = 0; t < a.T; ++t) {
        const size_t tev = ((size_t)t * E + e) * V + v;
        const size_t ta = ((size_t)t * E + e) * 2 * V + v;
        const float a0 = act ? a.action[ta] : 0.f;
        const float a1 = act ? a.action[ta + V] : 0.f;
        int arr = 0;
        if (act) arr = a.arrivals != nullptr ? a.arrivals[tev] : draw_arrival(d, e, v, step0 + t, lam);

        // power projection (MARL:555-561)
        float p0 = fmaxf(a0, 0.f) * ps, p1 = fmaxf(a1, 0.f) * ps;
        const float sm = p0 + p1;
        if (sm > 1.0f) {
            const float den = sm + 1e-12f;
            p0 = p0 / den;
            p1 = p1 / den;
        }
        const float P0 = p0 * Pmax, P1 = p1 * Pmax;
        const float P0_o = __shfl_sync(kFull, P0, src);

        // NOMA / OMA rate (MARL:339-370); log2(1+x) as log1p(x)/ln2 keeps tiny far-user SINRs
        const float sig = P0 * gn;
        const float sinr = near ? sig : sig / (P0_o * gn + 1.0f);
        const float rate = scheduled ? frac * (log1pf(sinr) * 1.44269504088896341f) : 0.f;
        const float data_t = rate * c_dt;

        // local CPU (MARL:572-592) -- float64 with the reference's operation order so that the
        // rounding residues of DataBuf - data_p (which min/max select) are reproduced
        const float share = fmaxf(fminf(fmaxf(a1, 0.f), 1.f), floor_f);
        const double f_local = __dmul_rn((double)share, p.f_local_max);
        const double backlog_kbit = buf;
        const double backlog_cyc = __dmul_rn(__dmul_rn(backlog_kbit, 1000.0), Cpb);
        const double cap = __dmul_rn(f_local, p.time_fast);
        const double used = fmin(cap, backlog_cyc);
        const double local_done = __ddiv_rn(used, kbit2cyc_den);
        const double remaining = fmax(0.0, __dsub_rn(backlog_kbit, local_done));
        const double off = fmin((double)data_t, remaining);  // MARL:595-596
        const float thr = rate * c_thr;
        const float off_f = (float)off;
        const float t_tx = off_f / (thr + 1e-12f);  // MARL:599-601

        // MEC FCFS queue, one per env (MARL:604-610)
        const double edge_in = __dmul_rn(__dmul_rn(off, 1000.0), Cpb);
        const double edge_sum = seg_sum<VP>(edge_in);
        const double q_before = Q;
        Q = Q + edge_sum;
        const double served = fmin(edge_cap, Q);
        Q = Q - served;

        buf = fmax(0.0, __dsub_rn(buf, __dadd_rn(local_done, off)));  // MARL:617-618

        // delays (MARL:622-633), energy (MARL:659-661)
        const float f_local_f = (float)f_local;
        const float d_local = (float)fmax(0.0, backlog_cyc - edge_in) / (f_local_f + 1e-12f);
        const float edge_in_f = (float)edge_in;
        const float sh = edge_in_f / (float)(edge_sum + 1e-12);
        const float d_eq = sh * ((float)q_before * inv_fedge);
        const float d_ec = edge_in_f * inv_fedge;
        const float delay = ((d_local + t_tx) + d_eq) + d_ec;
        const float E_tx = P0 * t_tx;
        const float E_loc = (float)(p.k * f_local * f_local) * (float)used;
        const float energy = E_tx + E_loc;

        // QoS penalty and reward (MARL:669-703)
        const bool viol = p.qos_enable && ((rate < Rmin) || (delay > Dmax));
        float rew = -(wd * delay + we * energy) - (viol ? pen : 0.f);
        rew = fminf(fmaxf(rew, -clipv), clipv);
        const float glob = seg_sum<VP>(act ? rew : 0.f) * invV;  // MARL:721
        const float overp = fmaxf(0.f, (P0 + P1) - Pmax);        // MARL:727-729

        // arrivals (MARL:717-719): DataBuf += (data_r * time_fast) * 1000
        buf = __dadd_rn(buf, __dmul_rn(__dmul_rn((double)arr, p.time_fast), 1000.0));

        const bool last = (t == a.T - 1);
        if (a.out.stats != nullptr || a.out.last_power != nullptr || last) {
            // last_* scalars (MARL:612-614,636-656,677,706-711)
            const float m_delay = seg_sum<VP>(act ? delay : 0.f) * invV;
            const float m_energy = seg_sum<VP>(act ? energy : 0.f) * invV;
            const float m_dl = seg_sum<VP>(act ? d_local : 0.f) * invV;
            const float m_dq = seg_sum<VP>(act ? d_eq : 0.f) * invV;
            const float m_dc = seg_sum<VP>(act ? d_ec : 0.f) * invV;
            const float m_ttx = seg_sum<VP>(act ? t_tx : 0.f) * invV;
            const float m_back = seg_sum<VP>(act ? (float)backlog_kbit : 0.f) * invV;
            const float util = (float)(used / (cap + 1e-12));
            const float m_util = seg_sum<VP>(act ? util : 0.f) * invV;
            const float m_viol = seg_sum<VP>((act && viol) ? 1.f : 0.f) * invV;
            const float s_off = seg_sum<VP>(act ? off_f : 0.f);
            const float s_loc = seg_sum<VP>(act ? (float)local_done : 0.f);
            const float mec_util = (float)(served / (edge_cap + 1e-12));
            const float q_f = (float)Q;
            auto stat_of = [&](int col) -> float {
                switch (col) {
                    case RISVEC_S_DELAY_MEAN: return m_delay;
                    case RISVEC_S_ENERGY_MEAN: return m_energy;
                    case RISVEC_S_DELAY_LOCAL_MEAN: return m_dl;
                    case RISVEC_S_DELAY_EDGE_Q_MEAN: return m_dq;
                    case RISVEC_S_DELAY_EDGE_C_MEAN: return m_dc;
                    case RISVEC_S_T_TX_MEAN: return m_ttx;
                    case RISVEC_S_BACKLOG_KBIT_MEAN: return m_back;
                    case RISVEC_S_MEC_UTILIZATION: return mec_util;
                    case RISVEC_S_LOCAL_UTIL_MEAN: return m_util;
                    case RISVEC_S_QOS_VIOLATION: return m_viol;
                    case RISVEC_S_OFF_KBIT_SUM: return s_off;
                    case RISVEC_S_LOCAL_KBIT_SUM: return s_loc;
                    case RISVEC_S_MEC_QUEUE_CYCLES: return q_f;
                    default: return 0.f;
                }
            };
            // lane v of the env writes stat columns v, v + VP, ... (coalesced rows of NSTAT floats)
            if (env_ok) {
                for (int col = v; col < RISVEC_NSTAT; col += VP) {
                    const float val = stat_of(col);
                    if (a.out.stats != nullptr) a.out.stats[((size_t)t * E + e) * RISVEC_NSTAT + col] = val;
                    if (last) s.stats[(size_t)e * RISVEC_NSTAT + col] = val;
                }
            }
            if (act) {  // last_power_W = [E_tx, E_loc] / time_fast (MARL:664-666)
                const float ptx = E_tx * inv_tf, ploc = E_loc * inv_tf;
                if (a.out.last_power != nullptr) {
                    a.out.last_power[ta] = ptx;
                    a.out.last_power[ta + V] = ploc;
                }
                if (last) {
                    s.last_power[(size_t)e * 2 * V + v] = ptx;
                    s.last_power[(size_t)e * 2 * V + V + v] = ploc;
                }
            }
        }
        if (act) {
            if (a.out.reward_user != nullptr) a.out.reward_user[tev] = rew;
            if (a.out.DataBuf != nullptr) a.out.DataBuf[tev] = (float)buf;
            if (a.out.data_t != nullptr) a.out.data_t[tev] = data_t;
            if (a.out.data_p != nullptr) a.out.data_p[tev] = (float)local_done;
            if (a.out.rate != nullptr) a.out.rate[tev] = rate;
            if (a.out.over_power != nullptr) a.out.over_power[tev] = overp;
            if (v == 0 && a.out.reward != nullptr) a.out.reward[(size_t)t * E + e] = glob;
        }
        o_rate = rate; o_dt = data_t; o_dp = (float)local_done; o_rew = rew; o_glob = glob; o_overp = overp;
        o_arr = arr;
    }

    // ---- registers -> state
    if (act && a.T > 0) {
        s.databuf[ev] = buf;
        s.rate[ev] = o_rate;
        s.data_t[ev] = o_dt;
        s.data_p[ev] = o_dp;
        s.reward_user[ev] = o_rew;
        s.over_power[ev] = o_overp;
        s.data_r[ev] = o_arr;
        if (v == 0) {
            s.mecq[e] = Q;
            s.reward[e] = o_glob;
            s.step_ctr[e] = step0 + a.T;
        }
    }
}

// sin/cos of two float32 angles (radians, |x| < ~1e4; RIS phases live in [0, 2*pi]) in packed
// fp32x2 arithmetic: Cody-Waite reduction to [-pi/4, pi/4] by quadrants, Cephes minimax
// polynomials (<= 1 ulp there), quadrant fix-up with integer sign flips.
__device__ __forceinline__ void sincos_fast2(float2 x, float2* sn, float2* cs) {
    const float2 t = __ffma2_rn(x, f2(0.63661977236758134f), f2(12582912.f));  // 1.5 * 2^23: rint
    const float2 kf = __fadd2_rn(t, f2(-12582912.f));
    float2 r = __ffma2_rn(kf, f2(-1.5707963705062866f), x);
    r = __ffma2_rn(kf, f2(4.3711390001862426e-8f), r);
    const float2 r2 = __fmul2_rn(r, r);
    float2 ps = __ffma2_rn(r2, f2(-1.9515295891e-4f), f2(8.3321608736e-3f));
    ps = __ffma2_rn(ps, r2, f2(-1.6666654611e-1f));
    const float2 s0 = __ffma2_rn(__fmul2_rn(ps, r2), r, r);
    float2 pc = __ffma2_rn(r2, f2(2.443315711809948e-5f), f2(-1.388731625493765e-3f));
    pc = __ffma2_rn(pc, r2, f2(4.166664568298827e-2f));
    const float2 c0 = __ffma2_rn(__fmul2_rn(pc, r2), r2, __ffma2_rn(r2, f2(-0.5f), f2(1.0f)));
    // the low mantissa bits of t hold the quadrant k mod 4
    const int qa = __float_as_int(t.x), qb = __float_as_int(t.y);
    const float sa = (qa & 1) ? c0.x : s0.x, ca = (qa & 1) ? s0.x : c0.x;
    const float sb = (qb & 1) ? c0.y : s0.y, cb = (qb & 1) ? s0.y : c0.y;
    sn->x = __int_as_float(__float_as_int(sa) ^ ((qa << 30) & 0x80000000));
    cs->x = __int_as_float(__float_as_int(ca) ^ (((qa + 1) << 30) & 0x80000000));
    sn->y = __int_as_float(__float_as_int(sb) ^ ((qb << 30) & 0x80000000));
    cs->y = __int_as_float(__float_as_int(cb) ^ (((qb + 1) << 30) & 0x80000000));
}

__device__ __forceinline__ float2 shfl_xor2(float2 x, int o) {
    return make_float2(__shfl_xor_sync(kFull, x.x, o), __shfl_xor_sync(kFull, x.y, o));
}

// ---------------------------------------------------------------------------------------
// SARL step (row a12): per step the V x M cascaded RIS reduction
//   S_v = sum_m exp(j*phase_m) * phasor(v, m),  rate_v = ln(1 + P0_v * amp_v * |S_v|^2 / sigma^2)
// The geometry phasor table (depends only on positions) is built once per launch in float64
// and kept in registers: lane (env, v) of warp w holds elements [w*slice, (w+1)*slice).
// WPE warps share one env group and combine their partial sums through shared memory.
// ---------------------------------------------------------------------------------------
__device__ __noinline__ void phasor_f32(double x, float* re, float* im) {
    double s64, c64;
    sincospi(x, &s64, &c64);
    *re = (float)c64;
    *im = (float)s64;
}

// float64 complex helpers for building phasor tables: exp(j*pi*m*delta) = z^m with
// Used when ONE warp serves an env group (M <= 40); larger M goes through k_sarl_cascade2 +
// k_sarl_scan below (several warps per env: the per-vehicle phase would be a serial section of
// one warp per block and step).

// PE: per-env step parameters from the attached table `envp` (risvec_attach_env_params); unused without PE
// NE: per-env RIS size `n_elem` (risvec_attach_ris_elements): the phasor pairs of the elements m >= n are zero, so the
// step loop is unchanged; unused without NE
template <int VP, int MPL, int WPE, bool PE = false, bool NE = false>
__global__ void __launch_bounds__(32 * WPE) k_sarl_rollout(Dims d, State s, risvec_params_t p, SarlArgs a,
                                                           const double* __restrict__ envp,
                                                           const int* __restrict__ n_elem) {
    static_assert(MPL % 4 == 0, "elements are processed four at a time (LDS.128 + FFMA2 pairs)");
    constexpr int EPW = 32 / VP;  // envs per warp (= per block)
    constexpr int NT = 32 * WPE;
    extern __shared__ __align__(16) float sarl_smem[];
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    // theta = exp(j*phase) of the block's envs as three planes (cos, sin, -sin) so that two
    // consecutive elements load as one float2 FFMA2 operand; double-buffered over steps.
    // MS = padded plane stride (covers the pad elements of the last slice, 16 B aligned quads).
    const int MS = ((M + 4 * WPE + 7) / 4) * 4;
    const int plane = EPW * MS;
    float* th = sarl_smem;                                              // [2][3][EPW][MS]
    float2* part = reinterpret_cast<float2*>(sarl_smem + 6 * plane);    // [2][WPE][32] (WPE > 1)
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int el = lane / VP, v = lane % VP;
    const int e0 = blockIdx.x * EPW;
    const int e = e0 + el;
    const bool env_ok = e < E;
    const bool act = env_ok && v < V;
    const size_t ev = (size_t)e * V + v;
    const int slice = (((M + WPE - 1) / WPE) + 3) & ~3;  // multiples of 4 keep the float4 quads aligned
    const int m0 = w * slice;
    const int m1 = min(M, m0 + slice);
    if constexpr (PE) env_params_sarl(p, env_param_row(envp, min(e, E - 1)));

    // ---- geometry phasor table -> registers (float64 argument reduction), as element pairs
    float2 WX[MPL / 2], WY[MPL / 2];
    phasor_pairs<MPL>(d, s, ev, act, m0, NE ? min(m1, ris_count<NE>(n_elem, min(e, E - 1), M)) : m1, WX, WY);
    for (int i = threadIdx.x; i < 6 * plane; i += NT) th[i] = 0.f;  // pad elements must stay finite
    const bool cphase = (w == 0);
    const int t_begin = 0, t_end = T;
    double buf = (act && cphase) ? s.databuf[ev] : 0.0;
    const float coef = act ? (float)(s.amp[ev] / (kSigma * kSigma)) : 0.f;  // SARL:157-159
    const long long step0 = env_ok ? s.step_ctr[e] : 0;

    const SarlConsts sc = sarl_consts(p);  // SARL:160, 318-319, 331
    const float t1 = (float)p.t_factor1, t2 = (float)p.t_factor2, pen1 = (float)p.penalty1, pen2 = (float)p.penalty2;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;
    const int n_env_here = min(EPW, E - e0);
    const int n_ph = n_env_here * M;  // the EPW rows of phase[t] are contiguous in HBM

    SarlLast last{};
    float o_rew = 0.f;

    // theta(t) -> smem buffer t & 1: thread k handles elements k, k + NT, ... in packed pairs.
    // The first pair of every step is prefetched one step ahead into (pf0, pf1).  All stream
    // addresses are running pointers bumped by one step stride (no per-step 64-bit index math).
    const size_t stepM = (size_t)E * M;
    const bool hasA = (int)threadIdx.x < n_ph, hasB = (int)threadIdx.x + NT < n_ph;
    const float* fetch_ptr = a.phase + ((size_t)t_begin * E + e0) * M + threadIdx.x;  // step the next fetch reads
    int fetch_t = t_begin;
    float pf0 = 0.f, pf1 = 0.f;
    auto fetch_phase = [&]() {  // loads step `fetch_t`, then moves on
        if (fetch_t < T) {
            pf0 = hasA ? __ldg(fetch_ptr) : 0.f;
            pf1 = hasB ? __ldg(fetch_ptr + NT) : 0.f;
        }
        fetch_ptr += stepM;
        ++fetch_t;
    };
    const int idxA = threadIdx.x, idxB = threadIdx.x + NT;  // my two elements of the first pass
    const int offA = (idxA / M) * MS + idxA % M, offB = (idxB / M) * MS + idxB % M;
    const bool l2_lane = (threadIdx.x & 7) == 0 && hasA;  // one 32 B sector per 8 threads
    auto produce_theta = [&](int t, const float* ph_t) {  // ph_t = phase row of step t for this block
        float* c_pl = th + (t & 1) * 3 * plane;
        float* s_pl = c_pl + plane;
        float* n_pl = s_pl + plane;
        if (l2_lane && t + 8 < T) asm volatile("prefetch.global.L2 [%0];" ::"l"(ph_t + 8 * stepM + threadIdx.x));
        if (hasA) {
            float2 sn, cs;
            sincos_fast2(make_float2(pf0, pf1), &sn, &cs);  // SARL:125-131
            c_pl[offA] = cs.x; s_pl[offA] = sn.x; n_pl[offA] = -sn.x;
            if (hasB) { c_pl[offB] = cs.y; s_pl[offB] = sn.y; n_pl[offB] = -sn.y; }
            if (t == T - 1) {
                s.phase_real[(size_t)e0 * M + idxA] = pf0;
                if (hasB) s.phase_real[(size_t)e0 * M + idxB] = pf1;
            }
        }
        for (int idx = threadIdx.x + 2 * NT; idx < n_ph; idx += 2 * NT) {  // only when n_ph > 2 * NT
            const int idx2 = idx + NT;
            const float ph0 = __ldg(ph_t + idx), ph1 = idx2 < n_ph ? __ldg(ph_t + idx2) : 0.f;
            float2 sn, cs;
            sincos_fast2(make_float2(ph0, ph1), &sn, &cs);
            const int ea = idx / M, ma = idx - ea * M;
            c_pl[ea * MS + ma] = cs.x; s_pl[ea * MS + ma] = sn.x; n_pl[ea * MS + ma] = -sn.x;
            if (idx2 < n_ph) {
                const int eb = idx2 / M, mb = idx2 - eb * M;
                c_pl[eb * MS + mb] = cs.y; s_pl[eb * MS + mb] = sn.y; n_pl[eb * MS + mb] = -sn.y;
            }
            if (t == T - 1) {
                s.phase_real[(size_t)e0 * M + idx] = ph0;
                if (idx2 < n_ph) s.phase_real[(size_t)e0 * M + idx2] = ph1;
            }
        }
    };
    // scalar inputs of the C-phase warp, prefetched one step ahead
    float na0 = 0.f, na1 = 0.f;
    int narr = 0;
    auto fetch_scalars = [&](int t) {
        if (cphase && act && t < T) {
            const size_t ta = ((size_t)t * E + e) * 2 * V + v;
            na0 = __ldg(a.action + ta);
            na1 = __ldg(a.action + ta + V);
            narr = a.arrivals != nullptr ? __ldg(a.arrivals + ((size_t)t * E + e) * V + v) : 0;
        }
    };

    __syncthreads();  // zero fill done
    const float* row = a.phase + ((size_t)t_begin * E + e0) * M;  // phase row of the step being produced
    fetch_phase();
    fetch_scalars(t_begin);
    if (t_begin < t_end) produce_theta(t_begin, row);
    row += stepM;
    fetch_phase();
    __syncthreads();
    for (int t = t_begin; t < t_end; ++t) {
        if (t + 1 < t_end) produce_theta(t + 1, row);  // overlaps with this step's MACs (other buffer)
        row += stepM;
        fetch_phase();
        const float a0 = na0, a1 = na1;
        const int arr_in = narr;
        fetch_scalars(t + 1);

        // (2) cascaded reduction over this warp's element slice: four elements per LDS.128 of each
        // theta plane, two elements per FFMA2
        const float* c_pl = th + (t & 1) * 3 * plane + el * MS + m0;
        const float4* c4 = reinterpret_cast<const float4*>(c_pl);
        const float4* s4 = reinterpret_cast<const float4*>(c_pl + plane);
        const float4* n4 = reinterpret_cast<const float4*>(c_pl + 2 * plane);
        float2 REa = make_float2(0.f, 0.f), IMa = REa, REb = REa, IMb = REa;
        auto quad = [&](int gq) {
            const float4 tx = c4[gq], ty = s4[gq], nty = n4[gq];
            const float2 txa = make_float2(tx.x, tx.y), txb = make_float2(tx.z, tx.w);
            const float2 tya = make_float2(ty.x, ty.y), tyb = make_float2(ty.z, ty.w);
            const float2 nya = make_float2(nty.x, nty.y), nyb = make_float2(nty.z, nty.w);
            REa = __ffma2_rn(txa, WX[2 * gq], REa); REa = __ffma2_rn(nya, WY[2 * gq], REa);
            IMa = __ffma2_rn(txa, WY[2 * gq], IMa); IMa = __ffma2_rn(tya, WX[2 * gq], IMa);
            REb = __ffma2_rn(txb, WX[2 * gq + 1], REb); REb = __ffma2_rn(nyb, WY[2 * gq + 1], REb);
            IMb = __ffma2_rn(txb, WY[2 * gq + 1], IMb); IMb = __ffma2_rn(tyb, WX[2 * gq + 1], IMb);
        };
        if (m1 - m0 == MPL) {  // full slice (warp-uniform): no per-quad guards
#pragma unroll
            for (int gq = 0; gq < MPL / 4; ++gq) quad(gq);
        } else {
#pragma unroll
            for (int gq = 0; gq < MPL / 4; ++gq)
                if (m0 + 4 * gq < m1) quad(gq);
        }
        float sr = (REa.x + REa.y) + (REb.x + REb.y);
        float si = (IMa.x + IMa.y) + (IMb.x + IMb.y);
        if (WPE > 1) {
            float2* pt = part + (t & 1) * WPE * 32;
            pt[w * 32 + lane] = make_float2(sr, si);
            __syncthreads();  // also publishes theta(t + 1)
            if (cphase) {
                sr = 0.f; si = 0.f;
#pragma unroll
                for (int k = 0; k < WPE; ++k) {
                    const float2 q = pt[k * 32 + lane];
                    sr += q.x; si += q.y;
                }
            }
        } else {
            __syncwarp();
        }

        // (3) per-vehicle queue update and reward (SARL:327-358), first warp of the block
        if (cphase) {
            const size_t tev = ((size_t)t * E + e) * V + v;
            int arr = arr_in;
            if (act && a.arrivals == nullptr) arr = draw_arrival(d, e, v, step0 + t, lam);

            const float g2 = __fmaf_rn(sr, sr, __fmul_rn(si, si));
            const float rate = log1p_sfu(__fmul_rn(a0, __fmul_rn(coef, g2)));  // natural log, SARL:159
            const float data_p = __fmul_rn(cbrt_sfu(a1), sc.c_dp);
            const SarlStep st = sarl_step(buf, rate, data_p, a0, a1, arr, sc.c_dt, sc.c_rev, t1, t2, pen1, pen2, p.time_fast);
            const float rew = __fmul_rn(seg_sum<VP>(act ? st.ru : 0.f), invV);
            last = SarlLast{rate, st.data_t, data_p, st.overp, st.overd, arr};
            if (act) {
                sarl_store_traces(a.out, tev, (float)buf, last);
                if (v == 0 && a.out.reward != nullptr) a.out.reward[(size_t)t * E + e] = rew;
            }
            o_rew = rew;
        }
        if (WPE == 1) __syncwarp();  // theta(t + 1) of this warp is complete before the next MACs
    }

    if (cphase && act && T > 0) {
        s.databuf[ev] = buf;
        sarl_store_last(s, ev, last);
        if (v == 0) {
            s.reward[e] = o_rew;
            s.step_ctr[e] = step0 + T;
        }
    }
}

// Cascade kernel for several warps per env (large M), two steps per barrier: a block serves one
// env group for a chunk of steps and only produces |S_v|^2 (a.g2).  Per pair of steps every
// thread evaluates theta = exp(j*phase) of its element(s) for BOTH steps in one packed sin/cos,
// every warp runs its element slice against both steps' theta planes (the phasor table in
// registers is read once per pair), and one __syncthreads per pair publishes the partial sums
// that the first warp folds over the WPE warps.  theta planes and partial sums are
// double-buffered over pairs.  NE: as k_sarl_rollout
template <int VP, int MPL, int WPE, bool NE = false>
__global__ void __launch_bounds__(32 * WPE, (WPE <= 8 && MPL <= 32) ? 16 / WPE : 1)
    k_sarl_cascade2(Dims d, State s, SarlArgs a, const int* __restrict__ n_elem) {
    static_assert(MPL % 4 == 0 && WPE > 1, "");
    constexpr int EPW = 32 / VP;
    constexpr int NT = 32 * WPE;
    extern __shared__ __align__(16) float sarl_smem[];
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const int MS = ((M + 4 * WPE + 7) / 4) * 4;
    const int plane = EPW * MS;
    float* th = sarl_smem;                                               // [2 bufs][2 steps][2 planes][EPW][MS]
    float2* part = reinterpret_cast<float2*>(sarl_smem + 8 * plane);     // [2 bufs][2 steps][WPE][32]
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int el = lane / VP, v = lane % VP;
    const int e0 = blockIdx.x * EPW, e = e0 + el;
    const bool act = e < E && v < V;
    const size_t ev = (size_t)e * V + v;
    const int slice = (((M + WPE - 1) / WPE) + 3) & ~3;
    const int m0 = w * slice, m1 = min(M, m0 + slice);

    float2 WX[MPL / 2], WY[MPL / 2];
    phasor_pairs<MPL>(d, s, ev, act, m0, NE ? min(m1, ris_count<NE>(n_elem, min(e, E - 1), M)) : m1, WX, WY);
    for (int i = threadIdx.x; i < 8 * plane; i += NT) th[i] = 0.f;  // pad elements must stay finite
    const int t_begin = (int)blockIdx.y * a.t_chunk, t_end = min(T, t_begin + a.t_chunk);
    const int n_ph = min(EPW, E - e0) * M;
    const size_t stepM = (size_t)E * M;

    // element(s) of this thread: idx = tid, tid + NT, ...; the first one is register-prefetched
    const bool has0 = (int)threadIdx.x < n_ph;
    const int off0 = ((int)threadIdx.x / M) * MS + (int)threadIdx.x % M;
    const float* row = a.phase + ((size_t)t_begin * E + e0) * M;  // phase row of the pair being produced
    float pfa = 0.f, pfb = 0.f;                                   // phases of (step, step + 1) for element tid
    auto fetch_pair = [&](const float* r, int t) {
        pfa = (has0 && t < T) ? __ldg(r + threadIdx.x) : 0.f;
        pfb = (has0 && t + 1 < T) ? __ldg(r + stepM + threadIdx.x) : 0.f;
    };
    auto produce_pair = [&](int t, const float* r, int bufi) {  // theta of steps (t, t + 1) -> buffer bufi
        float* b0 = th + bufi * 4 * plane;
        float* b1 = b0 + 2 * plane;
        if (has0) {
            float2 sn, cs;
            sincos_fast2(make_float2(pfa, pfb), &sn, &cs);  // SARL:125-131
            b0[off0] = cs.x; b0[plane + off0] = sn.x;
            b1[off0] = cs.y; b1[plane + off0] = sn.y;
            if (t == T - 1) s.phase_real[(size_t)e0 * M + threadIdx.x] = pfa;
            if (t + 1 == T - 1) s.phase_real[(size_t)e0 * M + threadIdx.x] = pfb;
        }
        for (int idx = threadIdx.x + NT; idx < n_ph; idx += NT) {  // only when n_ph > NT
            const float pa = __ldg(r + idx), pb = (t + 1 < T) ? __ldg(r + stepM + idx) : 0.f;
            float2 sn, cs;
            sincos_fast2(make_float2(pa, pb), &sn, &cs);
            const int o = (idx / M) * MS + idx % M;
            b0[o] = cs.x; b0[plane + o] = sn.x;
            b1[o] = cs.y; b1[plane + o] = sn.y;
            if (t == T - 1) s.phase_real[(size_t)e0 * M + idx] = pa;
            if (t + 1 == T - 1) s.phase_real[(size_t)e0 * M + idx] = pb;
        }
    };

    __syncthreads();
    fetch_pair(row, t_begin);
    if (t_begin < t_end) produce_pair(t_begin, row, 0);
    row += 2 * stepM;
    fetch_pair(row, t_begin + 2);
    __syncthreads();
    float* g2_ptr = a.g2 + ((size_t)t_begin * E + e) * V + v;
    const size_t sEV = (size_t)E * V;
    int bufi = 0;
    for (int t = t_begin; t < t_end; t += 2, bufi ^= 1) {
        if (t + 2 < t_end) produce_pair(t + 2, row, bufi ^ 1);
        row += 2 * stepM;
        fetch_pair(row, t + 4);

        const float* base = th + bufi * 4 * plane + el * MS + m0;
        float2 RE[2][2], IM[2][2];
#pragma unroll
        for (int u = 0; u < 2; ++u) RE[u][0] = RE[u][1] = IM[u][0] = IM[u][1] = make_float2(0.f, 0.f);
        auto quad = [&](int gq) {
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const float4* c4 = reinterpret_cast<const float4*>(base + u * 2 * plane);
                const float4 tx = c4[gq];
                const float4 ty = reinterpret_cast<const float4*>(base + u * 2 * plane + plane)[gq];
                const float2 txa = make_float2(tx.x, tx.y), txb = make_float2(tx.z, tx.w);
                const float2 tya = make_float2(ty.x, ty.y), tyb = make_float2(ty.z, ty.w);
                const float2 nya = make_float2(-ty.x, -ty.y), nyb = make_float2(-ty.z, -ty.w);  // operand negation, no extra plane
                RE[u][0] = __ffma2_rn(txa, WX[2 * gq], RE[u][0]); RE[u][0] = __ffma2_rn(nya, WY[2 * gq], RE[u][0]);
                IM[u][0] = __ffma2_rn(txa, WY[2 * gq], IM[u][0]); IM[u][0] = __ffma2_rn(tya, WX[2 * gq], IM[u][0]);
                RE[u][1] = __ffma2_rn(txb, WX[2 * gq + 1], RE[u][1]); RE[u][1] = __ffma2_rn(nyb, WY[2 * gq + 1], RE[u][1]);
                IM[u][1] = __ffma2_rn(txb, WY[2 * gq + 1], IM[u][1]); IM[u][1] = __ffma2_rn(tyb, WX[2 * gq + 1], IM[u][1]);
            }
        };
        if (m1 - m0 == MPL) {
#pragma unroll
            for (int gq = 0; gq < MPL / 4; ++gq) quad(gq);
        } else {
#pragma unroll
            for (int gq = 0; gq < MPL / 4; ++gq)
                if (m0 + 4 * gq < m1) quad(gq);
        }
        float2* pt = part + bufi * 2 * WPE * 32;
#pragma unroll
        for (int u = 0; u < 2; ++u)
            pt[(u * WPE + w) * 32 + lane] = make_float2((RE[u][0].x + RE[u][0].y) + (RE[u][1].x + RE[u][1].y),
                                                        (IM[u][0].x + IM[u][0].y) + (IM[u][1].x + IM[u][1].y));
        __syncthreads();  // partial sums of this pair + theta of the next pair are complete
        if (w == 0) {
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                float sr = 0.f, si = 0.f;
#pragma unroll
                for (int k = 0; k < WPE; ++k) {
                    const float2 q = pt[(u * WPE + k) * 32 + lane];
                    sr += q.x; si += q.y;
                }
                if (act && t + u < t_end) g2_ptr[u * sEV] = __fmaf_rn(sr, sr, __fmul_rn(si, si));
            }
            g2_ptr += 2 * sEV;
        }
    }
}

// Second half of the split SARL step for large M: per-vehicle queue update and reward
// (SARL:327-358) from the |S_v|^2 the cascade kernel left in a.g2.  An env owns VP lanes of a
// warp (lane = vehicle); inputs of step t + 1 are prefetched while step t computes.
// PE: as k_sarl_rollout
template <int VP, bool PE = false>
__global__ void __launch_bounds__(128) k_sarl_scan(Dims d, State s, risvec_params_t p, SarlArgs a,
                                                   const double* __restrict__ envp) {
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
    const int e = gtid / VP, v = gtid % VP;
    const int E = d.E, V = d.V, T = a.T;
    if constexpr (PE) env_params_sarl(p, env_param_row(envp, min(e, E - 1)));
    const bool env_ok = e < E;
    const bool act = env_ok && v < V;
    const size_t ev = (size_t)min(e, E - 1) * V + min(v, V - 1);
    double buf = s.databuf[ev];
    const float coef = (float)(s.amp[ev] / (kSigma * kSigma));  // SARL:157-159
    const long long step0 = s.step_ctr[min(e, E - 1)];
    const SarlConsts sc = sarl_consts(p);  // SARL:160, 318-319, 331
    const float t1 = (float)p.t_factor1, t2 = (float)p.t_factor2, pen1 = (float)p.penalty1, pen2 = (float)p.penalty2;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;
    const size_t sV = (size_t)E * V, s2V = 2 * sV;
    const float* ac = a.action + (size_t)min(e, E - 1) * 2 * V + min(v, V - 1);
    // inputs are fetched four steps ahead through a small register ring (the loads of steps
    // t+4..t+7 are in flight while steps t..t+3 compute), plus an L2 prefetch 32 steps ahead
    constexpr int D = 4;
    float ra0[D], ra1[D], rg2[D];
    int rarr[D];
    auto fetch = [&](int slot, int t) {
        const int tc = min(t, T - 1);
        ra0[slot] = __ldg(ac + (size_t)tc * s2V);
        ra1[slot] = __ldg(ac + (size_t)tc * s2V + V);
        rg2[slot] = __ldg(a.g2 + (size_t)tc * sV + ev);
        rarr[slot] = a.arrivals != nullptr ? __ldg(a.arrivals + (size_t)tc * sV + ev) : 0;
    };
#pragma unroll
    for (int k = 0; k < D; ++k) fetch(k, k);
    SarlLast last{};
    float o_rew = 0.f;
    for (int tb = 0; tb < T; tb += D) {
        float ca0[D], ca1[D], cg2[D];
        int carr[D];
#pragma unroll
        for (int k = 0; k < D; ++k) { ca0[k] = ra0[k]; ca1[k] = ra1[k]; cg2[k] = rg2[k]; carr[k] = rarr[k]; }
#pragma unroll
        for (int k = 0; k < D; ++k) fetch(k, tb + D + k);
        if (tb + 32 < T && (threadIdx.x & 7) == 0) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(a.g2 + (size_t)(tb + 32) * sV + ev));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(ac + (size_t)(tb + 32) * s2V));
        }
#pragma unroll
        for (int k = 0; k < D; ++k) {
        const int t = tb + k;
        if (t >= T) break;
        const float a0 = ca0[k], a1 = ca1[k], g2 = cg2[k];
        int arr = carr[k];
        if (act && a.arrivals == nullptr) arr = draw_arrival(d, e, v, step0 + t, lam);
        const float rate = log1p_sfu(__fmul_rn(a0, __fmul_rn(coef, g2)));  // natural log, SARL:159
        const float data_p = __fmul_rn(cbrt_sfu(a1), sc.c_dp);
        const SarlStep st = sarl_step(buf, rate, data_p, a0, a1, arr, sc.c_dt, sc.c_rev, t1, t2, pen1, pen2, p.time_fast);
        const float rew = __fmul_rn(seg_sum<VP>(act ? st.ru : 0.f), invV);
        last = SarlLast{rate, st.data_t, data_p, st.overp, st.overd, arr};
        if (act) {
            sarl_store_traces(a.out, (size_t)t * sV + ev, (float)buf, last);
            if (v == 0 && a.out.reward != nullptr) a.out.reward[(size_t)t * E + e] = rew;
        }
        o_rew = rew;
        }
    }
    if (act && T > 0) {
        s.databuf[ev] = buf;
        sarl_store_last(s, ev, last);
        if (v == 0) {
            s.reward[e] = o_rew;
            s.step_ctr[e] = step0 + T;
        }
    }
}

// =========================================================================================
// SARL fast path for V <= 8, M <= 8 * MPI (BASELINE configs 1-2: V = 8, M = 40, MPI = 5)
// =========================================================================================
// One warp = 4 envs; lane = (env el, part).  For the cascaded reduction the 8 lanes of an env
// split the ELEMENT axis: lane `part` owns elements m = part + 8 i (i < MPI), evaluates
// exp(j*phase_m) for them once, and multiplies them into the partial sums of ALL 8 vehicles.
// The geometry phasors of its elements x 8 vehicles sit in registers as packed float2 pairs
// (FFMA2 on Blackwell), stored in the lane-dependent vehicle order slot = v ^ part so that the
// 3-stage reduce-scatter over lanes xor 4, 2, 1 needs no selects: a lane always keeps the low
// half of its slots and sends the high half, and ends with the total S_v of vehicle v = part,
// for which it then runs the per-vehicle queue update.
// No shared memory, no block barrier.  Two consecutive steps are processed together: their
// state-independent parts (phasors, reduction, rate, data_t, data_p) are independent
// instruction streams -- the sin/cos evaluation is packed across the two steps (fp32x2) --
// and only the DataBuf recursion is sequential.  Inputs of the next two steps are prefetched
// into registers while the current ones compute.

// theta_m * w[slot] accumulated for the 4 slot pairs of one element
__device__ __forceinline__ void sarl_mac(float cs, float sn, const float2 (&WX)[4], const float2 (&WY)[4],
                                         float2 (&RE)[4], float2 (&IM)[4]) {
    const float2 TX = f2(cs), TY = f2(sn), NTY = f2(__int_as_float(__float_as_int(sn) ^ 0x80000000));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        RE[k] = __ffma2_rn(TX, WX[k], RE[k]);
        RE[k] = __ffma2_rn(NTY, WY[k], RE[k]);
        IM[k] = __ffma2_rn(TX, WY[k], IM[k]);
        IM[k] = __ffma2_rn(TY, WX[k], IM[k]);
    }
}

// reduce-scatter of the 8 slot sums over the env's 8 lanes (slot = v ^ part): returns |S_v|^2
__device__ __forceinline__ float sarl_reduce_abs2(float2 (&RE)[4], float2 (&IM)[4]) {
    float2 r0 = __fadd2_rn(RE[0], shfl_xor2(RE[2], 4)), r1 = __fadd2_rn(RE[1], shfl_xor2(RE[3], 4));
    float2 i0 = __fadd2_rn(IM[0], shfl_xor2(IM[2], 4)), i1 = __fadd2_rn(IM[1], shfl_xor2(IM[3], 4));
    r0 = __fadd2_rn(r0, shfl_xor2(r1, 2));
    i0 = __fadd2_rn(i0, shfl_xor2(i1, 2));
    const float sr = r0.x + __shfl_xor_sync(kFull, r0.y, 1);
    const float si = i0.x + __shfl_xor_sync(kFull, i0.y, 1);
    return __fmaf_rn(sr, sr, __fmul_rn(si, si));
}

struct SarlScalarIn {  // what the sequential part of a step needs from its inputs
    float a0, a1;
    int arr;
};
struct SarlHeavyOut {  // state-independent results of a step
    float rate, data_p;
};

// PACKED records have V == 8 and E % 4 == 0, i.e. every lane of every warp owns a vehicle.  `act` is then a
// compile-time constant: no predicated store regions, which otherwise cut the loop body into separately scheduled
// blocks (packed SARL: 0.156 -> 0.148 ms, packed MARL: 0.133 -> 0.118 ms).  The per-array MARL kernel measured
// slower without its predicates (0.116 -> 0.131 ms), so only the packed instantiations drop them.
template <int MPI, bool MFULL, bool FULL, bool PACKED>
__global__ void __launch_bounds__(32) k_sarl_v8(Dims d, State s, risvec_params_t p, SarlArgs a) {
    static_assert(!PACKED || (MFULL && FULL), "the packed record layout carries every stream");
    constexpr int RIN = 24 + 8 * MPI;            // packed input record (words): a0[8] a1[8] arr[8] phase[M]
    constexpr int ROUT = RISVEC_SARL_OUT_WORDS;  // packed output record: six traces x 8 vehicles
    const int lane = threadIdx.x & 31, el = lane >> 3, part = lane & 7;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const int e_raw = blockIdx.x * 4 + el;
    const bool env_ok = e_raw < E;
    const int e = min(e_raw, E - 1), v = part, vc = min(v, V - 1);  // clamped copies are load-only
    const bool act = PACKED || (env_ok && v < V);
    const size_t ev = (size_t)e * V + vc;

    // ---- geometry phasors of my elements for the 8 vehicles (slot = v ^ part) -> registers
    float2 WX[MPI][4], WY[MPI][4];
    {
        // one sincospi per lane: z of my own vehicle; the other vehicles' z arrive by shuffle and
        // w(v2, part + 8 i) = z^part * (z^8)^i is formed in float64, rounded to float32 once
        const double2 my_z = unit_phasor64(d.angle_BR - s.angle[ev]);
#pragma unroll
        for (int sl = 0; sl < 8; ++sl) {
            const int v2 = sl ^ part;
            const int src = (lane & ~7) + v2;
            const double2 z = make_double2(__shfl_sync(kFull, my_z.x, src), __shfl_sync(kFull, my_z.y, src));
            const bool ok2 = env_ok && v2 < V;
            double2 w = cpow64(z, (unsigned)part);
            const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
#pragma unroll
            for (int i = 0; i < MPI; ++i) {
                const bool on = ok2 && (part + 8 * i < M);
                const float re = on ? (float)w.x : 0.f, im = on ? (float)w.y : 0.f;
                if (sl & 1) { WX[i][sl >> 1].y = re; WY[i][sl >> 1].y = im; }
                else        { WX[i][sl >> 1].x = re; WY[i][sl >> 1].x = im; }
                w = cmul64(w, z8);
            }
        }
    }
    double buf = s.databuf[ev];
    const float coef = (float)(s.amp[ev] / (kSigma * kSigma));  // SARL:157-159
    const long long step0 = s.step_ctr[e];
    const SarlConsts sc = sarl_consts(p);  // SARL:160, 318-319, 331
    const float t1 = (float)p.t_factor1, t2 = (float)p.t_factor2, pen1 = (float)p.penalty1, pen2 = (float)p.penalty2;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;
    const double tf = p.time_fast;

    // ---- per-lane stream bases; step t of a stream sits t * (warp-uniform 32-bit stride) further
    // (the host checks that every stride fits 32 bits; the product is formed in 64 bits)
    // PACKED: one input and one output record per (step, env); every field of a lane sits at a
    // compile-time offset from ONE base pointer per direction, so a step costs two pointer bumps
    // instead of ten 64-bit address computations.
    const unsigned sM = (unsigned)E * M, s2V = (unsigned)E * 2 * V, sV = (unsigned)E * V, sE = (unsigned)E;
    const unsigned sIn = (unsigned)E * RIN, sOut = (unsigned)E * ROUT;
    // (records are tiled per warp: for each field the 4 envs x 8 vehicles of a warp are one
    //  contiguous 128 B line, so every load/store instruction still covers whole lines)
    const size_t grp = blockIdx.x;
    const float* const in_b = PACKED ? a.in_rec + grp * (4 * RIN) + el * 8 + part : nullptr;
    float* const out_b = PACKED ? a.out_rec + grp * (4 * ROUT) + el * 8 + part : nullptr;
    const float* const ph_b = PACKED ? a.in_rec + grp * (4 * RIN) + 96 + el * (8 * MPI) + part
                                     : a.phase + (size_t)e * M + part;
    const float* const ac_b = PACKED ? in_b : a.action + (size_t)e * 2 * V + vc;
    const int* const ar_b = PACKED ? nullptr : ((FULL || a.arrivals != nullptr) ? a.arrivals + ev : nullptr);
    float* const o_buf = (!PACKED && a.out.DataBuf) ? a.out.DataBuf + ev : nullptr;
    float* const o_dt = (!PACKED && a.out.data_t) ? a.out.data_t + ev : nullptr;
    float* const o_dp = (!PACKED && a.out.data_p) ? a.out.data_p + ev : nullptr;
    float* const o_op = (!PACKED && a.out.over_power) ? a.out.over_power + ev : nullptr;
    float* const o_od = (!PACKED && a.out.over_data) ? a.out.over_data + ev : nullptr;
    float* const o_rt = (!PACKED && a.out.rate) ? a.out.rate + ev : nullptr;
    float* const o_rw = a.out.reward ? a.out.reward + e : nullptr;
    const unsigned Tm1 = (unsigned)(T - 1);

    auto load_ph = [&](float (&ph)[MPI], unsigned t) {
        const float* q = ph_b + (size_t)min(t, Tm1) * (PACKED ? sIn : sM);
#pragma unroll
        for (int i = 0; i < MPI; ++i) ph[i] = (MFULL || part + 8 * i < M) ? __ldg(q + 8 * i) : 0.f;
    };
    auto load_sc = [&](SarlScalarIn& in, unsigned t) {
        const unsigned tc = min(t, Tm1);
        if constexpr (PACKED) {
            const float* q = in_b + (size_t)tc * sIn;
            in.a0 = __ldg(q);
            in.a1 = __ldg(q + 32);
            in.arr = __ldg(reinterpret_cast<const int*>(q) + 64);
        } else {
            const float* q = ac_b + (size_t)tc * s2V;
            in.a0 = __ldg(q);
            in.a1 = __ldg(q + V);
            in.arr = (FULL || ar_b != nullptr) ? __ldg(ar_b + (size_t)tc * sV) : 0;
        }
    };

    // L2 prefetch of everything the warp reads in step t: its 4 envs' rows are contiguous in each
    // stream (PACKED: one 4*RIN*4 B slab; else 4*M*4 B of phases, 4*2V*4 B of actions, 4*V*4 B of
    // arrivals); one 32 B sector per lane
    const int e0 = blockIdx.x * 4;
    const char* pf_base;
    size_t pf_stride;
    bool pf_on = true;
    if constexpr (PACKED) {
        pf_base = (const char*)(a.in_rec + grp * (4 * RIN)) + 32 * lane;
        pf_stride = (size_t)sIn * 4;
        pf_on = lane < (4 * RIN * 4) / 32;  // whole sectors of the slab only: never past the buffer
    } else {
        // whole sectors of each slab only, so a prefetch never points past the end of a buffer
        const int n_ph = (4 * M * 4) / 32, n_ac = (4 * 2 * V * 4) / 32, n_ar = (4 * V * 4) / 32;
        if (lane < n_ph) {
            pf_base = (const char*)(a.phase + (size_t)e0 * M) + 32 * lane;
            pf_stride = (size_t)sM * 4;
        } else if (lane < n_ph + n_ac) {
            pf_base = (const char*)(a.action + (size_t)e0 * 2 * V) + 32 * (lane - n_ph);
            pf_stride = (size_t)s2V * 4;
        } else if (lane < n_ph + n_ac + n_ar && (FULL || a.arrivals != nullptr)) {
            pf_base = (const char*)(a.arrivals + (size_t)e0 * V) + 32 * (lane - n_ph - n_ac);
            pf_stride = (size_t)sV * 4;
        } else {
            pf_base = (const char*)a.phase;
            pf_stride = 0;
            pf_on = false;
        }
    }
    pf_on = pf_on && (e0 + 4 <= E);  // the last, partial warp simply does not prefetch
    auto prefetch_l2 = [&](unsigned t) {
        if (pf_on) asm volatile("prefetch.global.L2 [%0];" ::"l"(pf_base + (size_t)min(t, Tm1) * pf_stride));
    };

    // state-independent part of two steps: theta = exp(j*phase) (packed over the two steps),
    // cascaded reduction, rate = ln(1 + a0 * coef * |S|^2) (SARL:159), data_p (SARL:331)
    auto heavy = [&](const float (&ph0)[MPI], const float (&ph1)[MPI], const SarlScalarIn& i0, const SarlScalarIn& i1,
                     SarlHeavyOut& h0, SarlHeavyOut& h1) {
        float2 RE0[4], IM0[4], RE1[4], IM1[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) RE0[k] = IM0[k] = RE1[k] = IM1[k] = make_float2(0.f, 0.f);
#pragma unroll
        for (int i = 0; i < MPI; ++i) {
            float2 sn, cs;
            sincos_fast2(make_float2(ph0[i], ph1[i]), &sn, &cs);
            sarl_mac(cs.x, sn.x, WX[i], WY[i], RE0, IM0);
            sarl_mac(cs.y, sn.y, WX[i], WY[i], RE1, IM1);
        }
        const float g0 = sarl_reduce_abs2(RE0, IM0), g1 = sarl_reduce_abs2(RE1, IM1);
        h0.rate = log1p_sfu(__fmul_rn(i0.a0, __fmul_rn(coef, g0)));
        h1.rate = log1p_sfu(__fmul_rn(i1.a0, __fmul_rn(coef, g1)));
        h0.data_p = __fmul_rn(cbrt_sfu(i0.a1), sc.c_dp);
        h1.data_p = __fmul_rn(cbrt_sfu(i1.a1), sc.c_dp);
    };

    float l_rate = 0.f, l_dt = 0.f, l_dp = 0.f, l_overp = 0.f, l_overd = 0.f, l_rew = 0.f;
    int l_arr = 0;

    // sequential part of one step (SARL:333-358), branch-free so that it can be interleaved
    // with the next pair's heavy part (written out, not sarl_step: the helper compiles to different code here)
    auto scan_step = [&](const SarlScalarIn& in, const SarlHeavyOut& h, unsigned t) {
        int arr = in.arr;
        if (!FULL && ar_b == nullptr) arr = act ? draw_arrival(d, e, v, step0 + t, lam) : 0;
        const float data_t = __fmul_rn(h.rate, sc.c_dt);
        const double raw = __dsub_rn(buf, __dadd_rn((double)data_t, (double)h.data_p));  // SARL:334
        const bool neg = raw < 0.0;
        // (explicit _rn intrinsics: no FMA contraction, so the loop copy and the tail copy of this
        //  code -- and therefore T = 1 launches and fused rollouts -- round identically)
        const float b = __fmul_rn((float)fmax(0.0, raw + (double)h.data_p), sc.c_rev);
        const float overp = neg ? __fsub_rn(in.a1, __fmul_rn(__fmul_rn(b, b), b)) : 0.f;  // SARL:337
        const float overd = neg ? (float)(-raw) : 0.f;
        const double nb = neg ? 0.0 : raw;
        const float base = __fsub_rn(-__fmul_rn(t1, __fadd_rn(in.a0, in.a1)), __fmul_rn(t2, (float)nb));
        const float pen = (nb > 0.0) ? pen1 : ((overd > 2.0f) ? pen2 : 0.f);  // SARL:343-352
        const float ru = __fsub_rn(base, pen);
        const float rew = __fmul_rn(seg_sum<8>(act ? ru : 0.f), invV);
        buf = __dadd_rn(nb, __dmul_rn(__dmul_rn((double)arr, tf), 1000.0));  // SARL:354-356
        if (act) {
            if constexpr (PACKED) {
                float* q = out_b + (size_t)t * sOut;
                q[0] = (float)buf; q[32] = data_t; q[64] = h.data_p; q[96] = overp; q[128] = overd; q[160] = h.rate;
            } else {
                const size_t o = (size_t)t * sV;
                if (FULL || o_buf) o_buf[o] = (float)buf;
                if (FULL || o_dt) o_dt[o] = data_t;
                if (FULL || o_dp) o_dp[o] = h.data_p;
                if (FULL || o_op) o_op[o] = overp;
                if (FULL || o_od) o_od[o] = overd;
                if (FULL || o_rt) o_rt[o] = h.rate;
            }
            if (v == 0 && (FULL || o_rw)) o_rw[(size_t)t * sE] = rew;
        }
        l_rate = h.rate; l_dt = data_t; l_dp = h.data_p; l_overp = overp; l_overd = overd; l_rew = rew; l_arr = arr;
    };

    // ---- software pipeline over pairs of steps: in one iteration the inputs of pair p + 2 are
    // requested, pair p + 1 runs its heavy part and pair p is scanned.  Two input buffers (X, Y)
    // alternate roles, so the loop is written for two pairs per trip.
    float phX0[MPI], phX1[MPI], phY0[MPI], phY1[MPI];
    SarlScalarIn c0, c1, x0, x1, y0, y1;
    SarlHeavyOut h0, h1, g0, g1;
    load_ph(phX0, 0); load_ph(phX1, 1);
    load_sc(c0, 0); load_sc(c1, 1);
    load_ph(phY0, 2); load_ph(phY1, 3);
    load_sc(y0, 2); load_sc(y1, 3);
    heavy(phX0, phX1, c0, c1, h0, h1);
    const unsigned P = (unsigned)T >> 1;
    // invariant at the top of a trip for pair pr: (c, h) = scalars + heavy results of pair pr,
    // buffer Y = inputs of pair pr + 1 (requested earlier), buffer X = free
    auto trip = [&](float (&phL0)[MPI], float (&phL1)[MPI], SarlScalarIn& l0, SarlScalarIn& l1,
                    float (&phU0)[MPI], float (&phU1)[MPI], SarlScalarIn& u0, SarlScalarIn& u1, unsigned pr) {
        const unsigned t = 2 * pr;
        prefetch_l2(t + 8); prefetch_l2(t + 9);      // pair pr + 4 -> L2 (no register cost)
        load_ph(phL0, t + 4); load_ph(phL1, t + 5);  // pair pr + 2 -> the free buffer
        load_sc(l0, t + 4); load_sc(l1, t + 5);
        heavy(phU0, phU1, u0, u1, g0, g1);            // pair pr + 1 (clamped past the end: unused)
        scan_step(c0, h0, t);
        scan_step(c1, h1, t + 1);
        c0 = u0; c1 = u1; h0 = g0; h1 = g1;
    };
    unsigned pr = 0;
    for (; pr + 2 <= P; pr += 2) {
        trip(phX0, phX1, x0, x1, phY0, phY1, y0, y1, pr);
        trip(phY0, phY1, y0, y1, phX0, phX1, x0, x1, pr + 1);
    }
    if (pr < P) trip(phX0, phX1, x0, x1, phY0, phY1, y0, y1, pr);
    if (T & 1) scan_step(c0, h0, Tm1);

    if (env_ok && T > 0) {  // elements_phase_shift_real = the last action_phase (SARL:128)
        const float* q = ph_b + (size_t)Tm1 * (PACKED ? sIn : sM);
#pragma unroll
        for (int i = 0; i < MPI; ++i)
            if (MFULL || part + 8 * i < M) s.phase_real[(size_t)e * M + part + 8 * i] = __ldg(q + 8 * i);
    }
    if (act && T > 0) {
        s.databuf[ev] = buf;
        s.rate[ev] = l_rate;
        s.data_t[ev] = l_dt;
        s.data_p[ev] = l_dp;
        s.over_power[ev] = l_overp;
        s.over_data[ev] = l_overd;
        s.data_r[ev] = l_arr;
        if (v == 0) {
            s.reward[e] = l_rew;
            s.step_ctr[e] = step0 + T;
        }
    }
}

// =========================================================================================
// MARL fast path for V <= 8 (BASELINE config 3: V = 8): one warp = 4 envs, lane = (env, vehicle)
// =========================================================================================
// Same pipeline shape as k_sarl_v8: two steps per trip, inputs of the next pair prefetched into
// registers, the state-independent part of a step (power projection, NOMA/OMA rate, data_t,
// CPU share -> f_local, cap) separated from the sequential float64 queue recursion
// (DataBuf, MEC queue).  The `last_*` statistics are produced only for the final step of the
// launch (they are state, not a per-step trace, in this kernel); launches that ask for the
// `stats` / `last_power` traces use the shape-generic k_marl_rollout.
#ifndef RISVEC_MARL_U
#define RISVEC_MARL_U 4  // steps per software-pipeline group of k_marl_v8 (2: 0.145 ms, 3-6: 0.115 ms, 8: 0.118 ms)
#endif
struct MarlIn {
    float a0, a1;
    int arr;
};
struct MarlHeavy {
    float P0, P1, rate, data_t, f_local_f;
    double f_local, cap;
};

// FUSED = the one-launch driver step (risvec_step_marl_fused): actions from the actors' raw outputs, observation out
// PE: per-env step parameters from the attached table `envp` (risvec_attach_env_params); unused without PE
template <bool FULL, bool PACKED, bool FUSED = false, bool PE = false>
__global__ void __launch_bounds__(32) k_marl_v8(Dims d, State s, risvec_params_t p, MarlArgs a,
                                                const double* __restrict__ envp) {
    static_assert(!FUSED || (!FULL && !PACKED), "the fused driver step is a variant of the generic form");
    static_assert(!PACKED || FULL, "the packed record layout carries every stream");
    static_assert(!PE || !PACKED, "packed records take no per-env parameter table");
    constexpr int RIN = RISVEC_MARL_IN_WORDS, ROUT = RISVEC_MARL_OUT_WORDS;
    const int lane = threadIdx.x & 31, el = lane >> 3, v = lane & 7;
    const int E = d.E, V = d.V, T = a.T;
    const int e_raw = blockIdx.x * 4 + el;
    const bool env_ok = e_raw < E;
    const int e = min(e_raw, E - 1), vc = min(v, V - 1);
    const bool act = PACKED || (env_ok && v < V);
    const size_t ev = (size_t)e * V + vc;
    if constexpr (PE) env_params_marl(p, env_param_row(envp, e));

    double buf = act ? s.databuf[ev] : 0.0;
    const double g = act ? s.gains[ev] : 0.0;
    const int code = act ? a.partner[ev] : RISVEC_PARTNER_NONE;
    const int ng = a.ngroups[e];
    double Q = s.mecq[e];
    const long long step0 = s.step_ctr[e];

    const bool paired = code >= 0;
    const bool second = paired && (code & RISVEC_PARTNER_SECOND);
    int other = paired ? (code & (RISVEC_PARTNER_SECOND - 1)) : v;
    other = min(max(other, 0), 7);
    const int src = (lane & ~7) + other;
    const double g_o = __shfl_sync(kFull, g, src);
    const bool first_near = second ? (g_o > g) : (g > g_o);  // MARL:355
    const bool near = paired ? (second ? !first_near : first_near) : true;
    const float gn = (float)(g / p.noise_power);
    // rate = (1/G) * log2(1 + sinr) = (log2(e)/G) * log1p(sinr); 0 when unscheduled (MARL:341-349).
    // log1p, not log2(1 + x): with destructive-interference gains the SINR falls below 2^-24 and
    // the reference still derives a non-zero rate (and a full-slot t_tx) from it.
    const float frac = (code != RISVEC_PARTNER_NONE)
                           ? (float)(1.0 / (double)max(1, ng)) * 1.44269504088896341f : 0.f;

    const float ps = (float)p.power_scale, Pmax = (float)p.P_max;
    const float c_dt = (float)(p.time_fast * p.bandwidth * 1000.0);
    const float c_thr = (float)(p.bandwidth * 1000.0);
    double floor_d = p.cpu_share_floor;
    if (!isfinite(floor_d)) floor_d = 0.10;
    floor_d = fmax(0.0, fmin(floor_d, 0.95));
    const float floor_f = (float)floor_d;
    const double Cpb = p.cycles_per_bit, den = Cpb * 1000.0, tf = p.time_fast, flm = p.f_local_max;
    const double rden = 1.0 / den;  // correctly rounded reciprocal for div_rn_fma
    const double edge_cap = p.f_edge_max * p.time_fast;
    const float inv_fedge = (float)(1.0 / (p.f_edge_max + 1e-12));
    const float kf = (float)p.k;
    const float wd = (float)p.w_d, we = (float)p.w_e, pen = p.qos_enable ? (float)p.qos_penalty : 0.f;
    const float clipv = (float)p.reward_clip;
    const float Rmin = p.qos_enable ? (float)p.R_min_bpsHz : -1.f, Dmax = p.qos_enable ? (float)p.D_max_s : 3.0e38f;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;

    const unsigned s2V = (unsigned)E * 2 * V, sV = (unsigned)E * V, sE = (unsigned)E;
    const unsigned sIn = (unsigned)E * RIN, sOut = (unsigned)E * ROUT;
    const size_t grp = blockIdx.x;  // records are tiled per warp (4 envs): each field is one 128 B line
    const float* const in_b = PACKED ? a.in_rec + grp * (4 * RIN) + el * 8 + v : nullptr;
    float* const out_b = PACKED ? a.out_rec + grp * (4 * ROUT) + el * 8 + v : nullptr;
    const float* const ac_b = PACKED ? in_b : a.action + (size_t)e * 2 * V + vc;
    const int* const ar_b = PACKED ? nullptr : ((FULL || a.arrivals != nullptr) ? a.arrivals + ev : nullptr);
    float* const o_ru = (!PACKED && a.out.reward_user) ? a.out.reward_user + ev : nullptr;
    float* const o_buf = (!PACKED && a.out.DataBuf) ? a.out.DataBuf + ev : nullptr;
    float* const o_dt = (!PACKED && a.out.data_t) ? a.out.data_t + ev : nullptr;
    float* const o_dp = (!PACKED && a.out.data_p) ? a.out.data_p + ev : nullptr;
    float* const o_rt = (!PACKED && a.out.rate) ? a.out.rate + ev : nullptr;
    float* const o_op = (!PACKED && a.out.over_power) ? a.out.over_power + ev : nullptr;
    float* const o_rw = a.out.reward ? a.out.reward + e : nullptr;
    const unsigned Tm1 = (unsigned)(T - 1);

    auto load_in = [&](MarlIn& in, unsigned t) {
        const unsigned tc = min(t, Tm1);
        if constexpr (PACKED) {  // tile: a0[4][8] a1[4][8] arr[4][8]
            const float* q = in_b + (size_t)tc * sIn;
            in.a0 = __ldg(q);
            in.a1 = __ldg(q + 32);
            in.arr = __ldg(reinterpret_cast<const int*>(q) + 64);
        } else {
            if (FUSED) {  // action mapping of the driver (marl_train_bcd.py:1601-1608), as k_map_actions_marl
                const float2 r = act ? __ldg(reinterpret_cast<const float2*>(a.raw) + (size_t)tc * sV + ev) : make_float2(-1.f, -1.f);
                in.a0 = (fminf(fmaxf(r.x, -0.999f), 0.999f) + 1.f) / 2.f;
                in.a1 = fmaxf((fminf(fmaxf(r.y, -0.999f), 0.999f) + 1.f) / 2.f, floor_f);
                if (!act) in.a0 = in.a1 = 0.f;
            } else {
                const float* q = ac_b + (size_t)tc * s2V;
                in.a0 = act ? __ldg(q) : 0.f;
                in.a1 = act ? __ldg(q + V) : 0.f;
            }
            in.arr = (act && (FULL || ar_b != nullptr)) ? __ldg(ar_b + (size_t)tc * sV) : 0;
        }
    };

    // state-independent part of a step
    auto heavy = [&](const MarlIn& in, MarlHeavy& h) {
        float p0 = __fmul_rn(fmaxf(in.a0, 0.f), ps), p1 = __fmul_rn(fmaxf(in.a1, 0.f), ps);  // MARL:555-561
        const float sm = __fadd_rn(p0, p1);
        const float sc = (sm > 1.0f) ? __fdividef(1.0f, __fadd_rn(sm, 1e-12f)) : 1.0f;
        p0 = __fmul_rn(p0, sc); p1 = __fmul_rn(p1, sc);
        h.P0 = __fmul_rn(p0, Pmax); h.P1 = __fmul_rn(p1, Pmax);
        const float P0_o = __shfl_sync(kFull, h.P0, src);
        const float sig = __fmul_rn(h.P0, gn);
        const float sinr = near ? sig : __fdividef(sig, __fmaf_rn(P0_o, gn, 1.0f));  // MARL:362-369
        h.rate = __fmul_rn(frac, log1p_pos(sinr));
        h.data_t = __fmul_rn(h.rate, c_dt);                                             // MARL:570
        const float share = fmaxf(fminf(fmaxf(in.a1, 0.f), 1.f), floor_f);             // MARL:572-578
        h.f_local = __dmul_rn((double)share, flm);
        h.cap = __dmul_rn(h.f_local, tf);
        h.f_local_f = (float)h.f_local;
    };

    float l_rate = 0.f, l_dt = 0.f, l_dp = 0.f, l_rew = 0.f, l_glob = 0.f, l_overp = 0.f;
    int l_arr = 0;
    using No = std::false_type;   // steps before the last: no `last_*` statistics
    using Yes = std::true_type;   // the final step also produces the `last_*` state

    // sequential part of a step: local CPU, offload, MEC queue, delays, energy, reward (written out, as k_marl_tma's
    // copy: shared helpers for the power / rate, delay / reward and last_* parts changed this kernel's code)
    auto scan_step = [&](const MarlIn& in, const MarlHeavy& h, unsigned t, auto with_stats) {
        int arr = in.arr;
        if (!FULL && ar_b == nullptr) arr = act ? draw_arrival(d, e, v, step0 + t, lam) : 0;
        const double backlog_kbit = buf;
        const double backlog_cyc = __dmul_rn(__dmul_rn(backlog_kbit, 1000.0), Cpb);  // MARL:585-592
        const double used = fmin(h.cap, backlog_cyc);
        const double local_done = div_rn_fma(used, den, rden);
        const double remaining = fmax(0.0, __dsub_rn(backlog_kbit, local_done));
        const double off = fmin((double)h.data_t, remaining);                       // MARL:595-596
        const double edge_in = __dmul_rn(__dmul_rn(off, 1000.0), Cpb);               // MARL:604
        const double edge_sum = seg_sum<8>(edge_in);
        const double q_before = Q;
        Q = __dadd_rn(Q, edge_sum);
        const double served = fmin(edge_cap, Q);
        Q = __dsub_rn(Q, served);                                                    // MARL:606-610
        buf = fmax(0.0, __dsub_rn(buf, __dadd_rn(local_done, off)));                 // MARL:617-618
        buf = __dadd_rn(buf, __dmul_rn(__dmul_rn((double)arr, tf), 1000.0));         // MARL:717-719

        const float off_f = (float)off, edge_in_f = (float)edge_in;
        const float t_tx = __fdividef(off_f, __fmaf_rn(h.rate, c_thr, 1e-12f));      // MARL:599-601
        const float d_local = __fdividef((float)fmax(0.0, __dsub_rn(backlog_cyc, edge_in)),
                                         __fadd_rn(h.f_local_f, 1e-12f));             // MARL:623-626
        const float sh = __fdividef(edge_in_f, (float)(edge_sum + 1e-12));           // MARL:629
        const float d_eq = __fmul_rn(sh, __fmul_rn((float)q_before, inv_fedge));
        const float d_ec = __fmul_rn(edge_in_f, inv_fedge);
        const float delay = __fadd_rn(__fadd_rn(__fadd_rn(d_local, t_tx), d_eq), d_ec);  // MARL:633
        const float E_tx = __fmul_rn(h.P0, t_tx);                                      // MARL:659-661
        const float E_loc = __fmul_rn(__fmul_rn(__fmul_rn(kf, h.f_local_f), h.f_local_f), (float)used);
        const float energy = __fadd_rn(E_tx, E_loc);
        const bool viol = (h.rate < Rmin) || (delay > Dmax);                           // MARL:669-677
        float rew = __fsub_rn(-__fmaf_rn(wd, delay, __fmul_rn(we, energy)), viol ? pen : 0.f);
        rew = fminf(fmaxf(rew, -clipv), clipv);                                        // MARL:696-703
        const float glob = __fmul_rn(seg_sum<8>(act ? rew : 0.f), invV);               // MARL:721
        const float overp = fmaxf(0.f, __fsub_rn(__fadd_rn(h.P0, h.P1), Pmax));        // MARL:727-729
        if (act) {
            if constexpr (PACKED) {  // tile: reward_user | DataBuf | data_t | data_p | rate, each [4][8]
                float* q = out_b + (size_t)t * sOut;
                q[0] = rew; q[32] = (float)buf; q[64] = h.data_t; q[96] = (float)local_done; q[128] = h.rate;
            } else {
                const size_t o = (size_t)t * sV;
                if (FULL || o_ru) o_ru[o] = rew;
                if (FULL || o_buf) o_buf[o] = (float)buf;
                if (FULL || o_dt) o_dt[o] = h.data_t;
                if (FULL || o_dp) o_dp[o] = (float)local_done;
                if (FULL || o_rt) o_rt[o] = h.rate;
                if (!FULL && o_op) o_op[o] = overp;
            }
            if (v == 0 && (FULL || o_rw)) o_rw[(size_t)t * sE] = glob;
        }
        l_rate = h.rate; l_dt = h.data_t; l_dp = (float)local_done; l_rew = rew; l_glob = glob; l_overp = overp;
        l_arr = arr;
        if constexpr (decltype(with_stats)::value) {  // last_* scalars (MARL:612-614,636-656,677,706-711)
            const float m_delay = seg_sum<8>(act ? delay : 0.f) * invV;
            const float m_energy = seg_sum<8>(act ? energy : 0.f) * invV;
            const float m_dl = seg_sum<8>(act ? d_local : 0.f) * invV;
            const float m_dq = seg_sum<8>(act ? d_eq : 0.f) * invV;
            const float m_dc = seg_sum<8>(act ? d_ec : 0.f) * invV;
            const float m_ttx = seg_sum<8>(act ? t_tx : 0.f) * invV;
            const float m_back = seg_sum<8>(act ? (float)backlog_kbit : 0.f) * invV;
            const float m_util = seg_sum<8>(act ? (float)(used / (h.cap + 1e-12)) : 0.f) * invV;
            const float m_viol = seg_sum<8>((act && viol && p.qos_enable) ? 1.f : 0.f) * invV;
            const float s_off = seg_sum<8>(act ? off_f : 0.f);
            const float s_loc = seg_sum<8>(act ? (float)local_done : 0.f);
            const float vals[RISVEC_NSTAT] = {m_delay, m_energy, m_dl, m_dq, m_dc, m_ttx, m_back,
                                              (float)(served / (edge_cap + 1e-12)), m_util, m_viol, s_off, s_loc,
                                              (float)Q, 0.f, 0.f, 0.f};
            if (env_ok) {
#pragma unroll
                for (int c = 0; c < RISVEC_NSTAT; ++c)
                    if ((c & 7) == v) s.stats[(size_t)e * RISVEC_NSTAT + c] = vals[c];
            }
            if (act) {
                const float inv_tf = (float)(1.0 / p.time_fast);
                s.last_power[(size_t)e * 2 * V + v] = E_tx * inv_tf;  // MARL:664-666
                s.last_power[(size_t)e * 2 * V + V + v] = E_loc * inv_tf;
            }
        }
    };

    // software pipeline over groups of U steps: inputs of group q+2 are requested, group q+1 runs
    // its state-independent part, group q runs the queue recursion.  The last step of the
    // launch is always scanned outside the loop (it also produces the `last_*` state).
    constexpr int U = RISVEC_MARL_U;
    MarlIn c[U], n[U], m[U];
    MarlHeavy h[U], hn[U];
    const unsigned NQ = (T > 0) ? (unsigned)(T - 1) / U : 0;  // full groups strictly before the last step
#pragma unroll
    for (int u = 0; u < U; ++u) { load_in(c[u], u); load_in(n[u], U + u); }
#pragma unroll
    for (int u = 0; u < U; ++u) heavy(c[u], h[u]);
    unsigned t = 0;
    for (unsigned q = 0; q < NQ; ++q, t += U) {
#pragma unroll
        for (int u = 0; u < U; ++u) load_in(m[u], t + 2 * U + u);
#pragma unroll
        for (int u = 0; u < U; ++u) heavy(n[u], hn[u]);
#pragma unroll
        for (int u = 0; u < U; ++u) scan_step(c[u], h[u], t + u, No{});
#pragma unroll
        for (int u = 0; u < U; ++u) { c[u] = n[u]; n[u] = m[u]; h[u] = hn[u]; }
    }
    if (T > 0) {  // 1..U steps left; (c, h) hold them
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (t + u + 1 < (unsigned)T) scan_step(c[u], h[u], t + u, No{});
            else if (t + u + 1 == (unsigned)T) scan_step(c[u], h[u], t + u, Yes{});
        }
    }

    if (act && T > 0) {
        s.databuf[ev] = buf;
        s.rate[ev] = l_rate;
        s.data_t[ev] = l_dt;
        s.data_p[ev] = l_dp;
        s.reward_user[ev] = l_rew;
        s.over_power[ev] = l_overp;
        s.data_r[ev] = l_arr;
        if (v == 0) {
            s.mecq[e] = Q;
            s.reward[e] = l_glob;
            s.step_ctr[e] = step0 + T;
        }
        if (FUSED && a.obs != nullptr) {  // marl_get_state of the new state (marl_train_bcd.py:819-827), as k_observe
            float* o = a.obs + ev * 5;
            o[0] = (float)(buf / 10.0);
            o[1] = l_dt / 10.f;
            o[2] = l_dp / 10.f;
            o[3] = s.over_data[ev] / 10.f;
            o[4] = l_rate / 20.f;
        }
    }
}

// =========================================================================================
// Driver-side glue on device (SURVEY.md 8f row 1): observation assembly and action mapping
// =========================================================================================
// marl_get_state (marl_train_bcd.py:819-827): per agent [DataBuf/10, data_t/10, data_p/10,
// over_data/10, vehicle_rate/20]; get_state (ddpg_train.py:47-73) prepends the agent's slice of
// `elements_phase_shift_real` (theta_number = int(M / n_veh) raw radians).  obs is [E, V, W].
__global__ void k_observe(Dims d, State s, float* __restrict__ obs, int n_theta) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.V) return;
    const int e = (int)(ix / d.V), v = (int)(ix % d.V);
    const int W = n_theta + 5;
    float* o = obs + ix * W;
    for (int k = 0; k < n_theta; ++k) o[k] = s.phase_real[(size_t)e * d.M + v * n_theta + k];
    o[n_theta + 0] = (float)(s.databuf[ix] / 10.0);
    o[n_theta + 1] = s.data_t[ix] / 10.f;
    o[n_theta + 2] = s.data_p[ix] / 10.f;
    o[n_theta + 3] = s.over_data[ix] / 10.f;
    o[n_theta + 4] = s.rate[ix] / 20.f;
}

// MARL action mapping (marl_train_bcd.py:1601-1608): raw [E,V,2] in [-1,1] (per-agent tanh power
// heads) -> action_for_env [E,2,V]: clip to +-0.999, (a + 1) / 2, CPU share floored.
__global__ void k_map_actions_marl(Dims d, risvec_params_t p, const float* __restrict__ raw, float* __restrict__ act) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.V) return;
    const int e = (int)(ix / d.V), v = (int)(ix % d.V);
    const float floor_f = (float)fmax(0.0, fmin(p.cpu_share_floor, 0.95));
    const float a0 = (fminf(fmaxf(raw[ix * 2 + 0], -0.999f), 0.999f) + 1.f) / 2.f;
    const float a1 = (fminf(fmaxf(raw[ix * 2 + 1], -0.999f), 0.999f) + 1.f) / 2.f;
    act[((size_t)e * 2 + 0) * d.V + v] = a0;
    act[((size_t)e * 2 + 1) * d.V + v] = fmaxf(a1, floor_f);
}

// SARL action mapping (ddpg_train.py:151-160): raw [E, 2V + M] in [-1,1] -> power [E,2,V] =
// (a + 1) / 2 and phase [E,M] = (a + 1) / 2 * 2 pi.
__global__ void k_map_actions_sarl(Dims d, const float* __restrict__ raw, float* __restrict__ act,
                                   float* __restrict__ phase) {
    const int W = 2 * d.V + d.M;
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * W) return;
    const int e = (int)(ix / W), k = (int)(ix % W);
    const float a = (fminf(fmaxf(raw[ix], -0.999f), 0.999f) + 1.f) / 2.f;
    if (k < 2 * d.V) act[(size_t)e * 2 * d.V + k] = a;
    else phase[(size_t)e * d.M + (k - 2 * d.V)] = a * 3.14159265358979323846f * 2.f;
}

}  // namespace risvec
