// MARL rollout (row a11 + a10 of SURVEY.md 8a), time-parallel form for the BASELINE shape (V = 8, E % 4 == 0,
// the six bench traces + injected arrivals).  Reference: Simulation-MARL-BCD/Environment.py:331-372, 547-731.
//
// k_marl_v8 (step.cuh) walks the T steps of 4 envs with one warp: 1024 warps for 4096 envs, every step a
// chain of dependent float64 operations -- it is bound by instruction latency at 0.33 of the HBM roofline.
// Here, as in k_sarl_mma_tma, ONE WARP owns ONE env and a stage of 16 steps is spread over its lanes:
// lane (g, tig) = vehicle g, steps 4 tig .. 4 tig + 3.  What makes that possible is that both recursions of
// the step are max-plus affine maps:
//     DataBuf' = max(DataBuf - (c + data_t), 0) + arrivals      c = local CPU capacity of the step in kbit
//     Q'       = max(Q + (S - cap_edge), 0)                     S = sum of the vehicles' offloaded cycles
// (MARL:585-618 and :604-610 collapse to these in exact arithmetic), so the start value of every lane's four
// steps comes from a 2-round shuffle scan of composed maps, after which the lane redoes its own four steps
// in the reference's float64 operation order (the rounding residues that `min`/`max` select are formed by
// the same operations as in k_marl_v8; only the start values can differ by an ulp of float64).
// Inputs arrive through per-warp TMA stage rings, the traces leave through a shared out tile and TMA tensor
// stores as full 128-byte lines (same machinery as sarl_mma.cuh).
#pragma once
#include "sarl_mma.cuh"

namespace risvec {

struct MarlConsts {  // formed on the host in float64, rounded once (constant-bank operands)
    float ps, Pmax, c_dt, c_thr, floor_f, inv_fedge, kf, wd, we, pen, clipv, Rmin, Dmax, inv_tf;
    int qos_enable, _pad;
    double flm, tf, Cpb, den, rden, edge_cap, noise_power;
};
inline MarlConsts marl_consts(const risvec_params_t& p) {
    MarlConsts c;
    c.ps = (float)p.power_scale; c.Pmax = (float)p.P_max;
    c.c_dt = (float)(p.time_fast * p.bandwidth * 1000.0);
    c.c_thr = (float)(p.bandwidth * 1000.0);
    double floor_d = p.cpu_share_floor;
    if (!std::isfinite(floor_d)) floor_d = 0.10;
    floor_d = fmax(0.0, fmin(floor_d, 0.95));
    c.floor_f = (float)floor_d;
    c.inv_fedge = (float)(1.0 / (p.f_edge_max + 1e-12));
    c.kf = (float)p.k;
    c.wd = (float)p.w_d; c.we = (float)p.w_e;
    c.pen = p.qos_enable ? (float)p.qos_penalty : 0.f;
    c.clipv = (float)p.reward_clip;
    c.Rmin = p.qos_enable ? (float)p.R_min_bpsHz : -1.f;
    c.Dmax = p.qos_enable ? (float)p.D_max_s : 3.0e38f;
    c.inv_tf = (float)(1.0 / p.time_fast);
    c.qos_enable = p.qos_enable; c._pad = 0;
    c.flm = p.f_local_max; c.tf = p.time_fast; c.Cpb = p.cycles_per_bit;
    c.den = p.cycles_per_bit * 1000.0; c.rden = 1.0 / c.den;
    c.edge_cap = p.f_edge_max * p.time_fast;
    c.noise_power = p.noise_power;
    return c;
}

struct MarlOutMaps {
    CUtensorMap trace[5];  // reward_user, DataBuf, data_t, data_p, rate: [T, E*8] f32, box {32, 16}
    CUtensorMap reward;    // [T, E] f32, box {4, 16}
};
constexpr int kMarlStageBytes = 16 * (16 + 8) * 4;                       // actions [16][2][8] + arrivals [16][8]
constexpr int kMarlOutTileBytes = 5 * 16 * 32 * 4 + 16 * 4 * 4;
constexpr int kMarlStages = 2;
constexpr int kMarlSmemBytes = 4 * kMarlStages * kMarlStageBytes + kMarlOutTileBytes + 4 * kMarlStages * 8 + 128;

__global__ void __launch_bounds__(128, 4)
    k_marl_tma(Dims d, State s, const MarlConsts c, MarlArgs a, const __grid_constant__ CUtensorMap tm_ac,
               const __grid_constant__ CUtensorMap tm_ar, const __grid_constant__ MarlOutMaps tm_out) {
    constexpr int V = 8, R = 16, STAGES = kMarlStages, STAGE_BYTES = kMarlStageBytes, AC_BYTES = 16 * 16 * 4;
    constexpr int TRACE_WORDS = R * 32;
    extern __shared__ unsigned char marl_tma_smem_raw[];
    const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int E = d.E, T = a.T;
    const int e0 = blockIdx.x * 4, e = e0 + warp;

    const uint32_t base = (smem_u32(marl_tma_smem_raw) + 127u) & ~127u;
    unsigned char* base_g = marl_tma_smem_raw + (base - smem_u32(marl_tma_smem_raw));
    const uint32_t ring = base + (uint32_t)warp * (STAGES * STAGE_BYTES);
    const unsigned char* ring_g = base_g + warp * (STAGES * STAGE_BYTES);
    const uint32_t out_s = base + 4u * STAGES * STAGE_BYTES;
    float* out_g = reinterpret_cast<float*>(base_g + 4 * STAGES * STAGE_BYTES);
    const uint32_t bars = out_s + kMarlOutTileBytes + (uint32_t)warp * (STAGES * 8);
    if (lane == 0) {
#pragma unroll
        for (int st = 0; st < STAGES; ++st) mbar_init(bars + 8 * st, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncwarp();
    const int NS = (T + R - 1) / R;
    auto issue = [&](int k) {
        const uint32_t dst = ring + (uint32_t)(k % STAGES) * STAGE_BYTES, bar = bars + 8 * (k % STAGES);
        mbar_expect_tx(bar, STAGE_BYTES);
        tma_load_2d(dst, &tm_ac, e * 2 * V, k * R, bar);
        tma_load_2d(dst + AC_BYTES, &tm_ar, e * V, k * R, bar);
    };
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < STAGES; ++k)
            if (k < NS) issue(k);
    }

    // ---- per-rollout state of vehicle g (replicated over its 4 lanes) and of the env
    const size_t ev = (size_t)e * V + g;
    double buf = s.databuf[ev];
    double Q = s.mecq[e];
    const double gain = s.gains[ev];
    const int code = a.partner[ev];
    const int ng = a.ngroups[e];
    const bool paired = code >= 0;
    const bool second = paired && (code & RISVEC_PARTNER_SECOND);
    int other = paired ? (code & (RISVEC_PARTNER_SECOND - 1)) : g;
    other = min(max(other, 0), 7);
    const int src = (other << 2) | tig;  // the partner's lane that holds the same steps
    const double g_o = __shfl_sync(kFull, gain, src);
    const bool first_near = second ? (g_o > gain) : (gain > g_o);  // MARL:355
    const bool near = paired ? (second ? !first_near : first_near) : true;
    const float gn = (float)(gain / c.noise_power);
    const float frac = (code != RISVEC_PARTNER_NONE) ? (float)(1.0 / (double)max(1, ng)) * 1.44269504088896341f : 0.f;
    float* const out_w = out_g + (4 * tig) * 32 + warp * 8 + g;
    float* const out_r = out_g + 5 * TRACE_WORDS + (4 * tig) * 4 + warp;

    struct Fin {  // per-lane values of the step that may be step T - 1 (state + last_* statistics)
        float rate, dt, dp, rew, overp, delay, energy, d_local, d_eq, d_ec, t_tx, backlog, util, viol, off, E_tx, E_loc;
        float glob, served_frac;
        int arr;
    };

    auto stage = [&](auto tail_tag, int k, Fin& fin) {
        constexpr bool TAIL = decltype(tail_tag)::value;
        mbar_wait(bars + 8 * (k % STAGES), (uint32_t)(k / STAGES) & 1u);
        const unsigned char* st = ring_g + (k % STAGES) * STAGE_BYTES;
        const float* ac = reinterpret_cast<const float*>(st) + (4 * tig) * (2 * V) + g;
        const int* ar = reinterpret_cast<const int*>(st + AC_BYTES) + (4 * tig) * V + g;
        const int tb = k * R + 4 * tig;
        float a0[4], a1[4];
        int arr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            a0[i] = ac[i * 2 * V];
            a1[i] = ac[i * 2 * V + V];
            arr[i] = ar[i * V];
        }
        __syncwarp();
        if (lane == 0 && k + STAGES < NS) {  // the stage's inputs are in registers: refill its buffer
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            issue(k + STAGES);
        }
        // ---- state-independent part of my four steps (MARL:555-578); this step and the delays / reward below are also
        // written out in k_marl_v8: shared helpers changed that kernel's code
        float P0[4], P1[4], rate[4], dt[4], flf[4];
        double cap[4], cl[4], inc[4], dd[4];
        bool ok[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            ok[i] = !TAIL || tb + i < T;
            float p0 = __fmul_rn(fmaxf(a0[i], 0.f), c.ps), p1 = __fmul_rn(fmaxf(a1[i], 0.f), c.ps);  // MARL:555-561
            const float sm = __fadd_rn(p0, p1);
            const float sc = (sm > 1.0f) ? __fdividef(1.0f, __fadd_rn(sm, 1e-12f)) : 1.0f;
            p0 = __fmul_rn(p0, sc); p1 = __fmul_rn(p1, sc);
            P0[i] = __fmul_rn(p0, c.Pmax); P1[i] = __fmul_rn(p1, c.Pmax);
            const float P0_o = __shfl_sync(kFull, P0[i], src);
            const float sig = __fmul_rn(P0[i], gn);
            const float sinr = near ? sig : __fdividef(sig, __fmaf_rn(P0_o, gn, 1.0f));  // MARL:362-369
            rate[i] = __fmul_rn(frac, log1p_pos(sinr));
            dt[i] = __fmul_rn(rate[i], c.c_dt);                                          // MARL:570
            const float share = fmaxf(fminf(fmaxf(a1[i], 0.f), 1.f), c.floor_f);        // MARL:572-578
            const double f_local = __dmul_rn((double)share, c.flm);
            cap[i] = __dmul_rn(f_local, c.tf);
            flf[i] = (float)f_local;
            // local capacity in kbit = cap / den, correctly rounded (same FMA division as the step itself)
            cl[i] = div_rn_fma(cap[i], c.den, c.rden);
            inc[i] = ok[i] ? __dmul_rn(__dmul_rn((double)arr[i], c.tf), 1000.0) : 0.0;
            dd[i] = ok[i] ? cl[i] + (double)dt[i] : 0.0;  // a step removes min(DataBuf, cl + data_t)
        }
        // ---- DataBuf at my first step: scan of the four-step maps over tig (identity steps past T)
        double xin;
        {
            MaxPlus ex, all;
            mp_scan<4>(mp_then(mp_then(MaxPlus{inc[0] - dd[0], inc[0]}, MaxPlus{inc[1] - dd[1], inc[1]}),
                               mp_then(MaxPlus{inc[2] - dd[2], inc[2]}, MaxPlus{inc[3] - dd[3], inc[3]})),
                       tig, ex, all);
            const double xi = mp_apply(ex, buf);
            xin = tig == 0 ? buf : xi;
            buf = mp_apply(all, buf);
        }
        // ---- my four steps in the reference's float64 order (MARL:585-618): offload, edge cycles, DataBuf
        double backlog[4], bcyc[4], used[4], ldone[4], off[4], edge_in[4], S[4];
        float bufn[4];
        {
            double cur = xin;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                backlog[i] = cur;
                bcyc[i] = __dmul_rn(__dmul_rn(cur, 1000.0), c.Cpb);
                used[i] = fmin(cap[i], bcyc[i]);
                ldone[i] = div_rn_fma(used[i], c.den, c.rden);
                const double remaining = fmax(0.0, __dsub_rn(cur, ldone[i]));
                off[i] = fmin((double)dt[i], remaining);                                   // MARL:595-596
                edge_in[i] = __dmul_rn(__dmul_rn(off[i], 1000.0), c.Cpb);                  // MARL:604
                const double nxt = __dadd_rn(fmax(0.0, __dsub_rn(cur, __dadd_rn(ldone[i], off[i]))), inc[i]);
                if (ok[i]) cur = nxt;                                                      // MARL:617-618, 717-719
                else { off[i] = 0.0; edge_in[i] = 0.0; }
                bufn[i] = (float)cur;
                double sum = edge_in[i];  // S = sum over the env's vehicles (lanes g of the same tig)
                sum += __shfl_xor_sync(kFull, sum, 4);
                sum += __shfl_xor_sync(kFull, sum, 8);
                sum += __shfl_xor_sync(kFull, sum, 16);
                S[i] = sum;
            }
        }
        // ---- MEC queue at my first step (MARL:604-610): Q' = max(Q + S - cap_edge, 0), same scan
        double qin;
        {
            // (a step past T is the identity: its map is {0, 0} because Q >= 0)
            double sa[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) sa[i] = ok[i] ? S[i] - c.edge_cap : 0.0;
            MaxPlus ex, all;
            mp_scan<4>(mp_then(mp_then(MaxPlus{sa[0], 0.0}, MaxPlus{sa[1], 0.0}),
                               mp_then(MaxPlus{sa[2], 0.0}, MaxPlus{sa[3], 0.0})),
                       tig, ex, all);
            const double qi = mp_apply(ex, Q);
            qin = tig == 0 ? Q : qi;
            Q = mp_apply(all, Q);
        }
        // ---- delays, energy, reward of my four steps (MARL:599-601, 622-703, 721)
        if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        __syncthreads();  // the out tile is free again (TMA stores of the previous stage have read it)
        float rew[4], glob[4];
        {
            double qc = qin;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const double q_before = qc;
                double qq = __dadd_rn(qc, S[i]);
                const double served = fmin(c.edge_cap, qq);
                qq = __dsub_rn(qq, served);                                                // MARL:606-610
                if (ok[i]) qc = qq;
                const float off_f = (float)off[i], edge_in_f = (float)edge_in[i];
                const float t_tx = __fdividef(off_f, __fmaf_rn(rate[i], c.c_thr, 1e-12f));  // MARL:599-601
                const float d_local = __fdividef((float)fmax(0.0, __dsub_rn(bcyc[i], edge_in[i])),
                                                 __fadd_rn(flf[i], 1e-12f));                // MARL:623-626
                const float sh = __fdividef(edge_in_f, (float)(S[i] + 1e-12));              // MARL:629
                const float d_eq = __fmul_rn(sh, __fmul_rn((float)q_before, c.inv_fedge));
                const float d_ec = __fmul_rn(edge_in_f, c.inv_fedge);
                const float delay = __fadd_rn(__fadd_rn(__fadd_rn(d_local, t_tx), d_eq), d_ec);  // MARL:633
                const float E_tx = __fmul_rn(P0[i], t_tx);                                  // MARL:659-661
                const float E_loc = __fmul_rn(__fmul_rn(__fmul_rn(c.kf, flf[i]), flf[i]), (float)used[i]);
                const float energy = __fadd_rn(E_tx, E_loc);
                const bool viol = (rate[i] < c.Rmin) || (delay > c.Dmax);                   // MARL:669-677
                float rw = __fsub_rn(-__fmaf_rn(c.wd, delay, __fmul_rn(c.we, energy)), viol ? c.pen : 0.f);
                rw = fminf(fmaxf(rw, -c.clipv), c.clipv);                                   // MARL:696-703
                rew[i] = rw;
                float gl = rw;  // mean over the vehicles: same tree as seg_sum<8> (MARL:721)
                gl += __shfl_xor_sync(kFull, gl, 4);
                gl += __shfl_xor_sync(kFull, gl, 8);
                gl += __shfl_xor_sync(kFull, gl, 16);
                glob[i] = __fmul_rn(gl, 0.125f);
                float* o = out_w + 32 * i;  // out tile: reward_user | DataBuf | data_t | data_p | rate
                o[0 * TRACE_WORDS] = rw;
                o[1 * TRACE_WORDS] = bufn[i];
                o[2 * TRACE_WORDS] = dt[i];
                o[3 * TRACE_WORDS] = (float)ldone[i];
                o[4 * TRACE_WORDS] = rate[i];
                if (TAIL ? (tb + i == T - 1) : (i == 3)) {  // dead code except in the rollout's last stage
                    fin.rate = rate[i]; fin.dt = dt[i]; fin.dp = (float)ldone[i]; fin.rew = rw;
                    fin.overp = fmaxf(0.f, __fsub_rn(__fadd_rn(P0[i], P1[i]), c.Pmax));     // MARL:727-729
                    fin.delay = delay; fin.energy = energy; fin.d_local = d_local; fin.d_eq = d_eq; fin.d_ec = d_ec;
                    fin.t_tx = t_tx; fin.backlog = (float)backlog[i];
                    fin.util = (float)(used[i] / (cap[i] + 1e-12));
                    fin.viol = (viol && c.qos_enable) ? 1.f : 0.f;
                    fin.off = off_f; fin.E_tx = E_tx; fin.E_loc = E_loc; fin.arr = arr[i];
                    fin.glob = glob[i];
                    fin.served_frac = (float)(served / (c.edge_cap + 1e-12));
                }
            }
        }
        {  // every lane of a tig group holds the four global rewards: lane g < 4 files the one of step tb + g
            const float r01 = (g & 1) ? glob[1] : glob[0], r23 = (g & 1) ? glob[3] : glob[2];
            if (g < 4) out_r[4 * g] = (g & 2) ? r23 : r01;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
#pragma unroll
            for (int n = 0; n < 5; ++n) tma_store_2d(&tm_out.trace[n], out_s + n * (TRACE_WORDS * 4), e0 * V, k * R);
            tma_store_2d(&tm_out.reward, out_s + 5 * (TRACE_WORDS * 4), e0, k * R);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    };
    Fin fin{}, scratch{};
    for (int k = 0; k < NS - 1; ++k) stage(std::false_type{}, k, scratch);
    if (T % R == 0)
        stage(std::false_type{}, NS - 1, fin);
    else
        stage(std::true_type{}, NS - 1, fin);

    // ---- state after the last step: the lanes that hold step T - 1 (tig = ((T - 1) & 15) >> 2) write it,
    // including the `last_*` statistics (MARL:612-614, 636-656, 677, 706-711): means over the 8 vehicles
    const bool mine = tig == (((T - 1) & 15) >> 2);
    auto mean8 = [&](float x) {
        x += __shfl_xor_sync(kFull, x, 4);
        x += __shfl_xor_sync(kFull, x, 8);
        x += __shfl_xor_sync(kFull, x, 16);
        return x;
    };
    const float m_delay = mean8(fin.delay) * 0.125f, m_energy = mean8(fin.energy) * 0.125f;
    const float m_dl = mean8(fin.d_local) * 0.125f, m_dq = mean8(fin.d_eq) * 0.125f, m_dc = mean8(fin.d_ec) * 0.125f;
    const float m_ttx = mean8(fin.t_tx) * 0.125f, m_back = mean8(fin.backlog) * 0.125f;
    const float m_util = mean8(fin.util) * 0.125f, m_viol = mean8(fin.viol) * 0.125f;
    const float s_off = mean8(fin.off), s_loc = mean8(fin.dp);
    if (mine) {
        s.databuf[ev] = buf;
        s.rate[ev] = fin.rate;
        s.data_t[ev] = fin.dt;
        s.data_p[ev] = fin.dp;
        s.reward_user[ev] = fin.rew;
        s.over_power[ev] = fin.overp;
        s.data_r[ev] = fin.arr;
        s.last_power[(size_t)e * 2 * V + g] = fin.E_tx * c.inv_tf;  // MARL:664-666
        s.last_power[(size_t)e * 2 * V + V + g] = fin.E_loc * c.inv_tf;
        const float vals[RISVEC_NSTAT] = {m_delay, m_energy, m_dl, m_dq, m_dc, m_ttx, m_back, fin.served_frac, m_util, m_viol,
                                          s_off, s_loc, (float)Q, 0.f, 0.f, 0.f};
#pragma unroll
        for (int col = 0; col < RISVEC_NSTAT; ++col)
            if ((col & 7) == g) s.stats[(size_t)e * RISVEC_NSTAT + col] = vals[col];
        if (g == 0) {
            s.mecq[e] = Q;
            s.reward[e] = fin.glob;
            s.step_ctr[e] += T;
        }
    }
    if (a.stats_slots != nullptr) {  // the statistics pass folded in: what k_shard_stats would sum after this launch
        __shared__ float blk_stat[4][RISVEC_NSTAT + 1];
        if (mine) {
            const float vals[RISVEC_NSTAT] = {m_delay, m_energy, m_dl, m_dq, m_dc, m_ttx, m_back, fin.served_frac, m_util, m_viol,
                                              s_off, s_loc, (float)Q, 0.f, 0.f, 0.f};
#pragma unroll
            for (int col = 0; col < RISVEC_NSTAT; ++col)
                if ((col & 7) == g) blk_stat[warp][col] = vals[col];
            if (g == 0) blk_stat[warp][RISVEC_NSTAT] = fin.glob;
        }
        __syncthreads();
        if (threadIdx.x <= RISVEC_NSTAT) {
            const int c2 = threadIdx.x;
            atomicAdd(a.stats_slots + (blockIdx.x % kRisvecStatSlots) * 32 + c2,
                      ((double)blk_stat[0][c2] + (double)blk_stat[1][c2]) + ((double)blk_stat[2][c2] + (double)blk_stat[3][c2]));
        }
    }
    if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
}

}  // namespace risvec
