// SARL rollout with the cascaded RIS reduction on the tensor cores (row a12 of SURVEY.md 8a).
// Reference: Simulation-SARL/Environment.py:125-131 (get_next_phase), :149-171 (compute_data_rate),
//            :318-359 (localProcRev, step).
//
// With T steps fused, the per-step reduction  S_v(t) = sum_m exp(j*phase_m(t)) * w(v, m)  of one env is
// a real GEMM  [2V x 2M] . [2M x T]:  rows = (Re S_v, Im S_v), K = (cos, sin) of every element,
// columns = time steps.  One WARP owns one env and walks the rollout in tiles of 8 steps:
//
//   A (16 x 16 per k-tile, row major) = geometry phasors of the env, constant over the rollout, kept in
//       registers as mma fragments:  A[v][(m, cos)] = Re w, A[v][(m, sin)] = -Im w,
//                                    A[8 + v][(m, cos)] = Im w, A[8 + v][(m, sin)] = Re w;
//   B (16 x 8 per k-tile, column major) = theta = (cos, sin)(phase[t0 + n][m]) -- lane (g, tig) evaluates
//       exactly the two elements its B fragment holds for step t0 + g (one packed sin/cos), so theta
//       goes from the sin/cos polynomial straight into the mma operand registers (no shared memory);
//   D (16 x 8, float32) -> lane (g, tig) ends with Re/Im S_g of steps t0 + 2 tig and t0 + 2 tig + 1.
//
// Precision: every operand is split into two binary16 pieces x = hi + lo (22 significant bits) and
// the product is formed as hi*hi + hi*lo + lo*hi with float32 accumulation (hi*hi in its own
// accumulator); the dropped lo*lo term is below 2^-24.  Measured against the float64 oracle this is
// as accurate as the float32 FFMA chain of k_sarl_v8 (tests/parity.py, sarl_rate_atol).
//
// The per-vehicle queue recursion (SARL:333-358) stays the reference's sequential float64 chain:
// the four lanes that hold one vehicle's eight steps pass DataBuf along by shuffles, so results do
// not depend on where a rollout is cut into launches or tiles.
#pragma once
#include <cuda.h>  // CUtensorMap (types only; cuTensorMapEncodeTiled is resolved at run time)
#include <cuda_fp16.h>

#include "step.cuh"

namespace risvec {

// D += A * B, m16n8k16, binary16 operands, float32 accumulate (legacy tensor path: HMMA in SASS)
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// (x0, x1) -> packed binary16 pairs hi and lo with x = hi + lo up to 2^-22 |x| (and 2^-25 absolute
// in the binary16 subnormal range); x0 goes to the low half (= the lower k / column index)
__device__ __forceinline__ void split_h2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(x0, x1);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn(__fsub_rn(x0, back.x), __fsub_rn(x1, back.y));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__device__ __forceinline__ void split_h2(double x0, double x1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn((float)x0, (float)x1);
    const float2 back = __half22float2(h);
    const __half2 l = __floats2half2_rn((float)(x0 - (double)back.x), (float)(x1 - (double)back.y));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ double shfl_f64(double x, int src) { return __shfl_sync(kFull, x, src); }

struct SarlMmaIn {     // inputs of one 8-step tile, as one lane needs them
    float a0[2], a1[2];  // action rows of vehicle g at steps t0 + 2 tig + {0, 1}
    int arr[2];
};

// KT = k-tiles of 8 RIS elements (M <= 8 KT, M even).  Block = 4 warps = 4 adjacent envs.
// FUSED = the one-launch driver step (risvec_step_sarl_fused): inputs from the actor's raw row, observation out
// PE: per-env step parameters from the attached table `envp` (risvec_attach_env_params); unused without PE
// NE: per-env RIS size `n_elem` (risvec_attach_ris_elements): the A operand is zero at the elements m >= n; unused
// without NE
template <int KT, bool FUSED = false, bool PE = false, bool NE = false>
__global__ void __launch_bounds__(128, 4) k_sarl_mma(Dims d, State s, risvec_params_t p, SarlArgs a,
                                                     const double* __restrict__ envp, const int* __restrict__ n_elem) {
    const int lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const int e = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (e >= E) return;  // warps are independent: no block-level synchronisation below
    const bool vact = g < V;
    const int vc = min(g, V - 1);
    const size_t ev = (size_t)e * V + vc;

    // ---- A operand: phasors of vehicle g at the elements m = 8 j + 2 tig + {0, 1} of every k-tile (written out, as in
    // k_sarl_mma_tma: a shared builder with the mask as an argument changed this kernel's code)
    // (fragment columns 2 tig, 2 tig + 1 hold element 8 j + 2 tig, columns 2 tig + 8, + 9 element
    //  8 j + 2 tig + 1: the same element order the B fragments below use)
    uint32_t Ah[KT][4], Al[KT][4];
    {
        const int n = ris_count<NE>(n_elem, e, M);
        const double2 z = unit_phasor64(d.angle_BR - s.angle[ev]);  // w(v, m) = z^m, float64 (SARL:134-145)
        const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
        double2 w = cpow64(z, 2u * (unsigned)tig);
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const int ma = 8 * j + 2 * tig;
            double2 wa = w, wb = cmul64(w, z);
            if (!(vact && ma < n)) wa = make_double2(0.0, 0.0);
            if (!(vact && ma + 1 < n)) wb = make_double2(0.0, 0.0);
            split_h2(wa.x, -wa.y, Ah[j][0], Al[j][0]);  // row g     (Re S_g): ( Re w, -Im w)
            split_h2(wa.y, wa.x, Ah[j][1], Al[j][1]);   // row g + 8 (Im S_g): ( Im w,  Re w)
            split_h2(wb.x, -wb.y, Ah[j][2], Al[j][2]);
            split_h2(wb.y, wb.x, Ah[j][3], Al[j][3]);
            w = cmul64(w, z8);
        }
    }
    double buf = s.databuf[ev];  // replicated over the 4 lanes of vehicle g
    const float coef = (float)(s.amp[ev] / (kSigma * kSigma));  // SARL:157-159
    const long long step0 = s.step_ctr[e];
    const SarlConsts sc = sarl_consts(p);  // SARL:160, 318-319, 331
    const float t1 = (float)p.t_factor1, t2 = (float)p.t_factor2, pen1 = (float)p.penalty1, pen2 = (float)p.penalty2;
    const float invV = 1.0f / (float)V;
    const float lam = (float)p.rate;
    const double tf = p.time_fast;
    // PE: the env's step parameters are read at each use from its row (env_param_at_use), in the expressions above
    const double* const prow = PE ? env_param_row(envp, e) : nullptr;
    auto at = [&](float handle_value, int col) -> float {
        if constexpr (PE) return (float)env_param_at_use(prow, col);
        else return handle_value;
    };
    auto c_dt_e = [&]() -> float {
        if constexpr (PE) return (float)(p.time_fast * env_param_at_use(prow, RISVEC_ENVP_BANDWIDTH) * 1000.0);
        else return sc.c_dt;
    };

    const size_t sM = (size_t)E * M, s2V = (size_t)E * 2 * V, sV = (size_t)E * V;
    const float* const ph_b = a.phase + (size_t)e * M + 2 * tig;
    const float* const ac_b = a.action + (size_t)e * 2 * V + vc;
    const int* const ar_b = a.arrivals != nullptr ? a.arrivals + ev : nullptr;
    const int Tm1 = T - 1;

    // fused driver step: the action mapping of ddpg_train.py:151-160 (k_map_actions_sarl) applied to the raw row
    constexpr bool fused = FUSED;
    const size_t sW = (size_t)E * (2 * V + M);
    const float* const raw_e = fused ? a.raw + (size_t)e * (2 * V + M) : nullptr;  // + t sW: [power 2V | phase M]
    auto map01 = [](float r) { return (fminf(fmaxf(r, -0.999f), 0.999f) + 1.f) / 2.f; };
    auto map_phase = [&](float r) { return map01(r) * 3.14159265358979323846f * 2.f; };
    auto load_phases = [&](float2 (&ph)[KT], int t0) {
        if (fused) {
            const float* q = raw_e + (size_t)min(t0 + g, Tm1) * sW + 2 * V + 2 * tig;
#pragma unroll
            for (int j = 0; j < KT; ++j) {
                const float2 r = (8 * j + 2 * tig < M) ? __ldg(reinterpret_cast<const float2*>(q + 8 * j)) : make_float2(-1.f, -1.f);
                ph[j] = make_float2(map_phase(r.x), map_phase(r.y));
            }
            return;
        }
        const float* q = ph_b + (size_t)min(t0 + g, Tm1) * sM;  // B fragment column g = step t0 + g
#pragma unroll
        for (int j = 0; j < KT; ++j)
            ph[j] = 8 * j + 2 * tig < M ? __ldg(reinterpret_cast<const float2*>(q + 8 * j))
                                                  : make_float2(0.f, 0.f);
    };
    auto load_scalars = [&](SarlMmaIn& in, int t0) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const size_t t = (size_t)min(t0 + 2 * tig + i, Tm1);
            if (fused) {
                in.a0[i] = map01(__ldg(raw_e + t * sW + vc));
                in.a1[i] = map01(__ldg(raw_e + t * sW + V + vc));
            } else {
                in.a0[i] = __ldg(ac_b + t * s2V);
                in.a1[i] = __ldg(ac_b + t * s2V + V);
            }
            in.arr[i] = ar_b != nullptr ? __ldg(ar_b + t * sV) : 0;
        }
    };
    // L2 prefetch of the env's rows of a later tile: lane (g, tig) covers sectors of row t0 + g
    auto prefetch_tile = [&](int t0) {
        if (fused) return;  // one step: nothing to pull ahead
        const size_t t = (size_t)min(t0 + g, Tm1);
        const float* q = a.phase + t * sM + (size_t)e * M + tig * 8;  // M <= 64: at most two sectors per lane
        if (tig * 8 < M) asm volatile("prefetch.global.L2 [%0];" ::"l"(q));
        if (tig * 8 + 32 < M) asm volatile("prefetch.global.L2 [%0];" ::"l"(q + 32));
        if (tig * 8 < 2 * V) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.action + t * s2V + (size_t)e * 2 * V + tig * 8));
        if (tig == 3 && ar_b != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.arrivals + t * sV + (size_t)e * V));
    };

    // values of the two steps of the latest tile (the owner of step T - 1 writes them to the state)
    float o_rate[2] = {0.f, 0.f}, o_dt[2] = {0.f, 0.f}, o_dp[2] = {0.f, 0.f}, o_overp[2] = {0.f, 0.f};
    float o_overd[2] = {0.f, 0.f}, o_rew[2] = {0.f, 0.f};
    int o_arr[2] = {0, 0};

    auto tile = [&](const float2 (&ph)[KT], const SarlMmaIn& in, int t0) {
        // ---- cascaded reduction of 8 steps on the tensor cores
        float accM[4] = {0.f, 0.f, 0.f, 0.f}, accX[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            float2 sn, cs;
            sincos_fast2(ph[j], &sn, &cs);  // theta = exp(j*phase) of elements 8 j + 2 tig + {0, 1} (SARL:125-131)
            uint32_t b0h, b0l, b1h, b1l;
            split_h2(cs.x, sn.x, b0h, b0l);
            split_h2(cs.y, sn.y, b1h, b1l);
            mma_16816(accM, Ah[j], b0h, b1h);
            mma_16816(accX, Ah[j], b0l, b1l);
            mma_16816(accX, Al[j], b0h, b1h);
        }
        // lane (g, tig): S_g of steps t0 + 2 tig (acc[0] + j acc[2]) and t0 + 2 tig + 1 (acc[1] + j acc[3])
        double dd[2], inc[2];
        float dp[2], rate[2], dt[2];
        int arr[2];
        bool ok[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int t = t0 + 2 * tig + i;
            ok[i] = t < T;
            const float re = __fadd_rn(accM[i], accX[i]), im = __fadd_rn(accM[2 + i], accX[2 + i]);
            const float g2 = __fmaf_rn(re, re, __fmul_rn(im, im));
            rate[i] = log1p_sfu(__fmul_rn(in.a0[i], __fmul_rn(coef, g2)));  // natural log, SARL:159
            dt[i] = __fmul_rn(rate[i], c_dt_e());
            dp[i] = __fmul_rn(cbrt_sfu(in.a1[i]), sc.c_dp);                    // SARL:331
            arr[i] = in.arr[i];
            if (ar_b == nullptr) arr[i] = (vact && ok[i]) ? draw_arrival(d, e, vc, step0 + t, at(lam, RISVEC_ENVP_RATE)) : 0;
            // steps past the end of the rollout are the identity of the recursion (DataBuf >= 0)
            dd[i] = ok[i] ? __dadd_rn((double)dt[i], (double)dp[i]) : 0.0;
            inc[i] = ok[i] ? __dmul_rn(__dmul_rn((double)arr[i], tf), 1000.0) : 0.0;
        }
        // ---- DataBuf recursion (SARL:333-356), sequential float64 in the reference's order: the lanes
        // tig = 0..3 of vehicle g hold steps (0,1), (2,3), (4,5), (6,7); the value is passed along.
        double x = buf, xin = buf;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double r0 = __dsub_rn(x, dd[0]);
            const double y = __dadd_rn(r0 < 0.0 ? 0.0 : r0, inc[0]);
            const double r1 = __dsub_rn(y, dd[1]);
            const double x2 = __dadd_rn(r1 < 0.0 ? 0.0 : r1, inc[1]);
            x = shfl_f64(x2, (lane & ~3) | q);  // the lane that really holds steps (2q, 2q + 1)
            if (q < 3 && tig == q + 1) xin = x;
        }
        buf = x;
        // ---- my two steps again from their true start value: overflow terms, reward, traces.  (Not sarl_step: the
        // step starts from the tile's dd / inc and reads the per-env values at use, under the 128-register cap.)
        double cur = xin;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int t = t0 + 2 * tig + i;
            const double raw = __dsub_rn(cur, dd[i]);  // SARL:334
            const bool neg = raw < 0.0;
            const float b = __fmul_rn((float)fmax(0.0, raw + (double)dp[i]), sc.c_rev);
            const float overp = neg ? __fsub_rn(in.a1[i], __fmul_rn(__fmul_rn(b, b), b)) : 0.f;  // SARL:336-339
            const float overd = neg ? (float)(-raw) : 0.f;
            const double nb = neg ? 0.0 : raw;
            const float base = __fsub_rn(-__fmul_rn(at(t1, RISVEC_ENVP_T_FACTOR1), __fadd_rn(in.a0[i], in.a1[i])),
                                         __fmul_rn(at(t2, RISVEC_ENVP_T_FACTOR2), (float)nb));
            const float pen = (nb > 0.0) ? at(pen1, RISVEC_ENVP_PENALTY1)
                                         : ((overd > 2.0f) ? at(pen2, RISVEC_ENVP_PENALTY2) : 0.f);  // SARL:343-352
            float ru = vact ? __fsub_rn(base, pen) : 0.f;
            ru += __shfl_xor_sync(kFull, ru, 4);   // mean over the vehicles: same tree as seg_sum<8>
            ru += __shfl_xor_sync(kFull, ru, 8);
            ru += __shfl_xor_sync(kFull, ru, 16);
            const float rew = __fmul_rn(ru, invV);
            cur = __dadd_rn(nb, inc[i]);  // SARL:354-356
            if (vact && ok[i]) {
                const size_t o = (size_t)t * sV + ev;
                if (a.out.DataBuf) a.out.DataBuf[o] = (float)cur;
                if (a.out.data_t) a.out.data_t[o] = dt[i];
                if (a.out.data_p) a.out.data_p[o] = dp[i];
                if (a.out.over_power) a.out.over_power[o] = overp;
                if (a.out.over_data) a.out.over_data[o] = overd;
                if (a.out.rate) a.out.rate[o] = rate[i];
                if (g == 0 && a.out.reward) a.out.reward[(size_t)t * E + e] = rew;
            }
            o_rate[i] = rate[i]; o_dt[i] = dt[i]; o_dp[i] = dp[i]; o_overp[i] = overp; o_overd[i] = overd;
            o_rew[i] = rew; o_arr[i] = arr[i];
        }
    };

    // ---- software pipeline over tiles: the inputs of tile k + 1 are in flight (registers) and tile
    // k + 3 is being pulled into L2 while tile k computes; two register sets alternate roles
    const int NT = (T + 7) >> 3;
    float2 phX[KT], phY[KT];
    SarlMmaIn inX, inY;
    load_phases(phX, 0);
    load_scalars(inX, 0);
    prefetch_tile(8);
    prefetch_tile(16);
    int k = 0;
    for (; k + 2 <= NT; k += 2) {
        prefetch_tile(8 * (k + 3));
        load_phases(phY, 8 * (k + 1));
        load_scalars(inY, 8 * (k + 1));
        tile(phX, inX, 8 * k);
        prefetch_tile(8 * (k + 4));
        load_phases(phX, 8 * (k + 2));  // clamped past the end: unused
        load_scalars(inX, 8 * (k + 2));
        tile(phY, inY, 8 * (k + 1));
    }
    if (k < NT) tile(phX, inX, 8 * k);

    // ---- registers -> state (what the reference object holds after the last step)
    for (int m = lane; m < M; m += 32)  // elements_phase_shift_real = the last action_phase (SARL:128)
        s.phase_real[(size_t)e * M + m] = fused ? map_phase(__ldg(raw_e + (size_t)Tm1 * sW + 2 * V + m))
                                                : __ldg(a.phase + (size_t)Tm1 * sM + (size_t)e * M + m);
    const int last = Tm1 & 7;  // position of step T - 1 in its tile: lane tig = last / 2, slot last % 2
    if (fused && a.obs != nullptr && vact) {  // get_state of the new state (ddpg_train.py:47-73), as k_observe
        const int n_theta = M / V, W = n_theta + 5;
        float* o = a.obs + ev * W;
        for (int k = tig; k < n_theta; k += 4) o[k] = map_phase(__ldg(raw_e + (size_t)Tm1 * sW + 2 * V + g * n_theta + k));
        if (tig == (last >> 1)) {
            const int i = last & 1;
            o[n_theta + 0] = (float)(buf / 10.0);
            o[n_theta + 1] = (i ? o_dt[1] : o_dt[0]) / 10.f;
            o[n_theta + 2] = (i ? o_dp[1] : o_dp[0]) / 10.f;
            o[n_theta + 3] = (i ? o_overd[1] : o_overd[0]) / 10.f;
            o[n_theta + 4] = (i ? o_rate[1] : o_rate[0]) / 20.f;
        }
    }
    if (tig == (last >> 1) && vact) {
        const int i = last & 1;
        s.databuf[ev] = buf;
        s.rate[ev] = i ? o_rate[1] : o_rate[0];
        s.data_t[ev] = i ? o_dt[1] : o_dt[0];
        s.data_p[ev] = i ? o_dp[1] : o_dp[0];
        s.over_power[ev] = i ? o_overp[1] : o_overp[0];
        s.over_data[ev] = i ? o_overd[1] : o_overd[0];
        s.data_r[ev] = i ? o_arr[1] : o_arr[0];
        if (g == 0) {
            s.reward[e] = i ? o_rew[1] : o_rew[0];
            s.step_ctr[e] = step0 + T;
        }
    }
}

// =========================================================================================
// The same rollout with TMA-staged inputs: the BASELINE shape (V = 8, M = 8 KT, every trace written)
// =========================================================================================
// What k_sarl_mma above still pays for is addressing and exposed load latency: its prefetched LDGs share
// the warp's six scoreboard slots with the MUFU / shuffle / float64 traffic of the step, so the loads are
// waited for long before their data is needed.  Here every warp owns a ring of shared-memory stages and
// one lane per warp issues, per 16 steps, three cp.async.bulk.tensor copies (the env's rows of phase
// [T, E*M], action [T, E*16] and arrivals [T, E*8], as 2-D tensor maps with boxes {M,16}, {16,16}, {8,16})
// that complete on the stage's mbarrier: loads cost no issue slots, no registers and no scoreboard, and
// run two stages ahead.  A stage is processed as two independent 8-step mma tiles (shared A fragments,
// interleaved instruction streams).  The DataBuf recursion x -> max(x - d, 0) + inc is a max-plus affine
// map, so the four lanes of a vehicle combine their two-step maps with a 2-round shuffle scan (float64)
// and then redo their own two steps sequentially from the resulting start value; across launches the
// results are reproducible for the same tiling (tiles start at the launch's first step).
// Index arithmetic is 32-bit (the host checks T*E*M < 2^32).  Rows past T (last, partial stage) are
// zero-filled by TMA and act as identity steps.

// sin/cos of two float32 angles, packed fp32x2: k = rint(x / pi), r = x - k*pi in [-pi/2, pi/2]
// (Cody-Waite, two terms), minimax polynomials of degree 9 / 10 on that interval (fitted for this file:
// |error| <= 1.5e-7 absolute, 2-3e-8 rms on [0, 2 pi] in float32 arithmetic), sign (-1)^k on both --
// no quadrant swap, so the fix-up is one shift and two XORs per angle.
__device__ __forceinline__ void sincos_pi2(float2 x, float2* sn, float2* cs) {
    const float2 t = __ffma2_rn(x, f2(0.318309886183790672f), f2(12582912.f));  // 1.5 * 2^23: rint
    const float2 kf = __fadd2_rn(t, f2(-12582912.f));
    float2 r = __ffma2_rn(kf, f2(-3.1415927410125732f), x);
    r = __ffma2_rn(kf, f2(8.742277657347586e-8f), r);
    const float2 r2 = __fmul2_rn(r, r);
    float2 ps = __ffma2_rn(r2, f2(2.599751496745739e-06f), f2(-0.00019806479394901544f));
    ps = __ffma2_rn(ps, r2, f2(0.008333015255630016f));
    ps = __ffma2_rn(ps, r2, f2(-0.16666656732559204f));
    const float2 s0 = __ffma2_rn(__fmul2_rn(ps, r2), r, r);
    float2 pc = __ffma2_rn(r2, f2(-2.607421833999979e-07f), f2(2.4761729946476407e-05f));
    pc = __ffma2_rn(pc, r2, f2(-0.0013888400280848145f));
    pc = __ffma2_rn(pc, r2, f2(0.04166664183139801f));
    pc = __ffma2_rn(pc, r2, f2(-0.5f));
    const float2 c0 = __ffma2_rn(pc, r2, f2(1.0f));
    const int sa = __float_as_int(t.x) << 31, sb = __float_as_int(t.y) << 31;  // parity of k
    sn->x = __int_as_float(__float_as_int(s0.x) ^ sa);
    cs->x = __int_as_float(__float_as_int(c0.x) ^ sa);
    sn->y = __int_as_float(__float_as_int(s0.y) ^ sb);
    cs->y = __int_as_float(__float_as_int(c0.y) ^ sb);
}

// ---- mbarrier / TMA primitives (PTX; SASS: SYNCS.*, UTMALDG)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tmap), "r"(c0), "r"(c1), "r"(bar) : "memory");
}

__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(tmap), "r"(src), "r"(c0), "r"(c1) : "memory");
}

constexpr int kSarlTmaRows = 16;    // steps per stage (two 8-step mma tiles)
constexpr int kSarlTmaStages = 2;   // input stages per warp (one in use, one in flight)
__host__ __device__ constexpr int sarl_tma_stage_bytes(int KT) { return kSarlTmaRows * (8 * KT + 16 + 8) * 4; }
constexpr int kSarlOutTileBytes = 6 * kSarlTmaRows * 32 * 4 + kSarlTmaRows * 4 * 4;  // six traces [16][4 envs][8] + reward [16][4]
__host__ __device__ constexpr int sarl_tma_smem_bytes(int KT) {
    return 4 * kSarlTmaStages * sarl_tma_stage_bytes(KT) + kSarlOutTileBytes + 4 * kSarlTmaStages * 8 + 128;
}

// output tensor maps of one rollout (order of the out tile in shared memory)
struct SarlOutMaps {
    CUtensorMap trace[6];  // DataBuf, data_t, data_p, over_power, over_data, rate: [T, E*8] f32, box {32, 16}
    CUtensorMap reward;    // [T, E] f32, box {4, 16}
};

#ifndef RISVEC_TMA_MINB
#define RISVEC_TMA_MINB 4  // resident blocks (of four warps) per SM the register allocation aims at
#endif
template <int KT>
__global__ void __launch_bounds__(128, RISVEC_TMA_MINB)
    k_sarl_mma_tma(Dims d, State s, const SarlConsts c, SarlArgs a, const __grid_constant__ CUtensorMap tm_ph,
                   const __grid_constant__ CUtensorMap tm_ac, const __grid_constant__ CUtensorMap tm_ar,
                   const __grid_constant__ SarlOutMaps tm_out) {
    constexpr int M = 8 * KT, V = 8, R = kSarlTmaRows, STAGES = kSarlTmaStages;
    constexpr int PH_BYTES = R * M * 4, AC_BYTES = R * 2 * V * 4, AR_BYTES = R * V * 4;
    constexpr int STAGE_BYTES = PH_BYTES + AC_BYTES + AR_BYTES;
    constexpr int TRACE_WORDS = R * 32;  // one trace of the out tile: [16 steps][4 envs][8 vehicles]
    static_assert(STAGE_BYTES == sarl_tma_stage_bytes(KT) && STAGE_BYTES % 128 == 0, "");
    extern __shared__ unsigned char sarl_tma_smem_raw[];
    // block = four warps = four ADJACENT envs (E % 4 == 0).  The warps only meet at the out tile.
    const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);  // warp-uniform for the compiler
    const int lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int E = d.E, T = a.T;
    const int e0 = blockIdx.x * 4, e = e0 + warp;

    // ---- shared memory: [4 warps][STAGES] input stages | out tile | mbarriers   (128 B aligned)
    const uint32_t base = (smem_u32(sarl_tma_smem_raw) + 127u) & ~127u;
    unsigned char* base_g = sarl_tma_smem_raw + (base - smem_u32(sarl_tma_smem_raw));
    const uint32_t ring = base + (uint32_t)warp * (STAGES * STAGE_BYTES);
    const unsigned char* ring_g = base_g + warp * (STAGES * STAGE_BYTES);
    const uint32_t out_s = base + 4u * STAGES * STAGE_BYTES;
    float* out_g = reinterpret_cast<float*>(base_g + 4 * STAGES * STAGE_BYTES);
    const uint32_t bars = out_s + kSarlOutTileBytes + (uint32_t)warp * (STAGES * 8);
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < STAGES; ++st) mbar_init(bars + 8 * st, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();
    const int NS = (T + R - 1) / R;  // stages of 16 steps in this rollout
    auto issue = [&](int k) {       // lane 0: my env's rows of steps [16 k, 16 k + 16) -> stage k % STAGES
        const uint32_t dst = ring + (uint32_t)(k % STAGES) * STAGE_BYTES, bar = bars + 8 * (k % STAGES);
        mbar_expect_tx(bar, STAGE_BYTES);
        tma_load_2d(dst, &tm_ph, e * M, k * R, bar);
        tma_load_2d(dst + PH_BYTES, &tm_ac, e * 2 * V, k * R, bar);
        tma_load_2d(dst + PH_BYTES + AC_BYTES, &tm_ar, e * V, k * R, bar);
    };
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < STAGES; ++k)
            if (k < NS) issue(k);
    }

    // ---- A operand (see k_sarl_mma): phasors of vehicle g at elements 8 j + 2 tig + {0, 1}
    const size_t ev = (size_t)e * V + g;
    uint32_t Ah[KT][4], Al[KT][4];
    {
        const double2 z = unit_phasor64(d.angle_BR - s.angle[ev]);
        const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
        double2 w = cpow64(z, 2u * (unsigned)tig);
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const double2 wb = cmul64(w, z);
            split_h2(w.x, -w.y, Ah[j][0], Al[j][0]);
            split_h2(w.y, w.x, Ah[j][1], Al[j][1]);
            split_h2(wb.x, -wb.y, Ah[j][2], Al[j][2]);
            split_h2(wb.y, wb.x, Ah[j][3], Al[j][3]);
            w = cmul64(w, z8);
        }
    }
    double buf = s.databuf[ev];  // replicated over the 4 lanes of vehicle g
    const float coef = (float)(s.amp[ev] / (kSigma * kSigma));  // SARL:157-159
    // my slots of the out tile: trace n at out_w[n * TRACE_WORDS + 32 i] for my step i = 0..3
    float* const out_w = out_g + (4 * tig) * 32 + warp * 8 + g;
    float* const out_r = out_g + 6 * TRACE_WORDS + (4 * tig) * 4 + warp;  // + 4 g': mean reward of step 4 tig + g'

    // values of the lane's latest step; those of step T - 1 become the env's state after the loop
    struct LastStep {
        float rate, dt, dp, overp, overd, rew;
        int arr;
        bool mine;  // this lane holds step T - 1
    };
    // One stage = 16 steps, spread over the two mma tiles so that lane (g, tig) ends up with FOUR
    // CONSECUTIVE steps 4 tig .. 4 tig + 3 of vehicle g: column c of tile A is step 4 (c >> 1) + (c & 1),
    // column c of tile B the step two later (the accumulator columns of a lane are 2 tig and 2 tig + 1).
    // TAIL = the stage reaches past step T - 1 (only the last stage of a rollout whose length is not a
    // multiple of 16): the missing steps are identity steps, TMA zero-fills their inputs and clips their
    // output rows.
    auto stage = [&](auto tail_tag, int k, LastStep& fin) {
        constexpr bool TAIL = decltype(tail_tag)::value;
        mbar_wait(bars + 8 * (k % STAGES), (uint32_t)(k / STAGES) & 1u);
        const unsigned char* st = ring_g + (k % STAGES) * STAGE_BYTES;
        // ---- cascaded reduction: B column g of tile A = row 4 (g >> 1) + (g & 1), of tile B two rows later
        const float* ph = reinterpret_cast<const float*>(st) + (4 * (g >> 1) + (g & 1)) * M + 2 * tig;
        float mA[4] = {0.f, 0.f, 0.f, 0.f}, xA[4] = {0.f, 0.f, 0.f, 0.f};
        float mB[4] = {0.f, 0.f, 0.f, 0.f}, xB[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < KT; ++j) {
            const float2 pa = *reinterpret_cast<const float2*>(ph + 8 * j);
            const float2 pb = *reinterpret_cast<const float2*>(ph + 2 * M + 8 * j);
            float2 sn, cs;
            uint32_t b0h, b0l, b1h, b1l;
            sincos_pi2(pa, &sn, &cs);  // theta = exp(j*phase) of elements 8 j + 2 tig + {0, 1} (SARL:125-131)
            split_h2(cs.x, sn.x, b0h, b0l);
            split_h2(cs.y, sn.y, b1h, b1l);
            mma_16816(mA, Ah[j], b0h, b1h);
            mma_16816(xA, Ah[j], b0l, b1l);
            mma_16816(xA, Al[j], b0h, b1h);
            sincos_pi2(pb, &sn, &cs);
            split_h2(cs.x, sn.x, b0h, b0l);
            split_h2(cs.y, sn.y, b1h, b1l);
            mma_16816(mB, Ah[j], b0h, b1h);
            mma_16816(xB, Ah[j], b0l, b1l);
            mma_16816(xB, Al[j], b0h, b1h);
        }
        // ---- per-step part for my steps tb + {0,1,2,3}, as packed pairs (0,1) from tile A, (2,3) from tile B
        const int tb = k * R + 4 * tig;
        const float* ac = reinterpret_cast<const float*>(st + PH_BYTES) + (4 * tig) * (2 * V) + g;
        const int* ar = reinterpret_cast<const int*>(st + PH_BYTES + AC_BYTES) + (4 * tig) * V + g;
        float2 a0[2], a1[2], rate[2], dt[2], dp[2];
        int arr[4];
        double dd[4], inc[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float(&accM)[4] = h ? mB : mA;
            const float(&accX)[4] = h ? xB : xA;
            a0[h] = make_float2(ac[(2 * h) * 2 * V], ac[(2 * h + 1) * 2 * V]);
            a1[h] = make_float2(ac[(2 * h) * 2 * V + V], ac[(2 * h + 1) * 2 * V + V]);
            arr[2 * h] = ar[(2 * h) * V];
            arr[2 * h + 1] = ar[(2 * h + 1) * V];
            const float2 re = __fadd2_rn(make_float2(accM[0], accM[1]), make_float2(accX[0], accX[1]));
            const float2 im = __fadd2_rn(make_float2(accM[2], accM[3]), make_float2(accX[2], accX[3]));
            sarl_rate2(re, im, a0[h], a1[h], coef, c, rate[h], dt[h], dp[h]);
        }
        // the inputs of this stage are in registers: its buffer can take the stage after next
        __syncwarp();
        if (lane == 0 && k + STAGES < NS) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(k + STAGES);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const bool ok = !TAIL || tb + i < T;  // steps past the end of the rollout are identity steps (DataBuf >= 0)
            const float dti = (i & 1) ? dt[i >> 1].y : dt[i >> 1].x, dpi = (i & 1) ? dp[i >> 1].y : dp[i >> 1].x;
            dd[i] = ok ? __dadd_rn((double)dti, (double)dpi) : 0.0;
            inc[i] = ok ? __dmul_rn(__dmul_rn((double)arr[i], c.tf), 1000.0) : 0.0;
        }
        // ---- DataBuf at my first step: inclusive scan of the lanes' four-step maps over tig = 0..3
        MaxPlus ex, all;  // the maps before mine, the whole stage
        mp_scan<4>(mp_then(mp_then(MaxPlus{inc[0] - dd[0], inc[0]}, MaxPlus{inc[1] - dd[1], inc[1]}),
                           mp_then(MaxPlus{inc[2] - dd[2], inc[2]}, MaxPlus{inc[3] - dd[3], inc[3]})),
                   tig, ex, all);
        const double xin = mp_apply(ex, buf);
        double cur = tig == 0 ? buf : xin;
        buf = mp_apply(all, buf);
        // ---- my four steps in the reference's order (SARL:333-358); past-the-end steps are identity steps
        float overd[4], nbf[4], barg[4], curf[4];
        bool pos[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            sarl_settle(cur, dd[i], (i & 1) ? dp[i >> 1].y : dp[i >> 1].x, inc[i], true, overd[i], nbf[i], barg[i],
                        pos[i], curf[i]);
        // ---- the out tile is free again once the TMA stores of the previous stage have read it
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();
        float rew[4];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float2 op, base2;
            sarl_reward2(make_float2(barg[2 * h], barg[2 * h + 1]), make_float2(nbf[2 * h], nbf[2 * h + 1]), a0[h],
                         a1[h], c, op, base2);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int i = 2 * h + u;
                const float od = overd[i];
                const float overp = od > 0.f ? (u ? op.y : op.x) : 0.f;  // only where the buffer went negative
                const float pen = pos[i] ? c.pen1 : ((od > 2.0f) ? c.pen2 : 0.f);  // SARL:343-352 (a helper changed the code)
                rew[i] = __fsub_rn(u ? base2.y : base2.x, pen);
                float* o = out_w + 32 * i;
                o[0 * TRACE_WORDS] = curf[i];
                o[1 * TRACE_WORDS] = u ? dt[h].y : dt[h].x;
                o[2 * TRACE_WORDS] = u ? dp[h].y : dp[h].x;
                o[3 * TRACE_WORDS] = overp;
                o[4 * TRACE_WORDS] = od;
                o[5 * TRACE_WORDS] = u ? rate[h].y : rate[h].x;
                if (TAIL ? (tb + i == T - 1) : (i == 3)) {  // dead code except in the rollout's last stage
                    fin.rate = u ? rate[h].y : rate[h].x;
                    fin.dt = u ? dt[h].y : dt[h].x;
                    fin.dp = u ? dp[h].y : dp[h].x;
                    fin.overp = overp;
                    fin.overd = od;
                    fin.arr = arr[i];
                    fin.mine = TAIL ? true : (tig == 3);
                }
            }
        }
        // mean over the vehicles (lanes g = 0..7 of the same tig): same tree as seg_sum<8>
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            rew[i] += __shfl_xor_sync(kFull, rew[i], 4);
            rew[i] += __shfl_xor_sync(kFull, rew[i], 8);
            rew[i] += __shfl_xor_sync(kFull, rew[i], 16);
            rew[i] = __fmul_rn(rew[i], 0.125f);
        }
        {  // every lane of a tig group holds the four means: lane g < 4 files the one of step tb + g
            const float r01 = (g & 1) ? rew[1] : rew[0], r23 = (g & 1) ? rew[3] : rew[2];
            const float mine = (g & 2) ? r23 : r01;
            if (g < 4) out_r[4 * g] = mine;
            if (TAIL ? (g < 4 && tb + g == T - 1) : (g == 3)) fin.rew = mine;
        }
        // ---- out tile -> HBM: full 128-byte lines per (trace, step) for the block's four envs
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
#pragma unroll
            for (int n = 0; n < 6; ++n) tma_store_2d(&tm_out.trace[n], out_s + n * (TRACE_WORDS * 4), e0 * V, k * R);
            tma_store_2d(&tm_out.reward, out_s + 6 * (TRACE_WORDS * 4), e0, k * R);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    };
    LastStep fin{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0, false}, scratch = fin;
    for (int k = 0; k < NS - 1; ++k) stage(std::false_type{}, k, scratch);
    if (T % R == 0)
        stage(std::false_type{}, NS - 1, fin);
    else
        stage(std::true_type{}, NS - 1, fin);

    // ---- registers -> state
    for (int m = lane; m < M; m += 32)  // elements_phase_shift_real = the last action_phase (SARL:128)
        s.phase_real[(size_t)e * M + m] = __ldg(a.phase + ((size_t)(T - 1) * E + e) * M + m);
    if (fin.mine) {  // the reference object's attributes after the last step
        s.rate[ev] = fin.rate;
        s.data_t[ev] = fin.dt;
        s.data_p[ev] = fin.dp;
        s.over_power[ev] = fin.overp;
        s.over_data[ev] = fin.overd;
        s.data_r[ev] = fin.arr;
    }
    // the mean reward of step T - 1 sits in the lane (g = (T - 1) & 3, tig = ((T - 1) & 15) >> 2) that filed it
    if (g == ((T - 1) & 3) && tig == (((T - 1) & 15) >> 2)) s.reward[e] = fin.rew;
    if (tig == 0) s.databuf[ev] = buf;
    if (lane == 0) s.step_ctr[e] += T;
    if (a.stats_slots != nullptr) {  // the statistics pass folded in: what k_shard_stats would sum after this launch
        __shared__ float blk_rew[4];  // (SARL kernels write no `last_*` columns: the sum is the reward's)
        if (g == ((T - 1) & 3) && tig == (((T - 1) & 15) >> 2)) blk_rew[warp] = fin.rew;
        __syncthreads();
        if (threadIdx.x == 0)
            atomicAdd(a.stats_slots + (blockIdx.x % kRisvecStatSlots) * 32 + RISVEC_NSTAT,
                      ((double)blk_rew[0] + (double)blk_rew[1]) + ((double)blk_rew[2] + (double)blk_rew[3]));
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
}

}  // namespace risvec
