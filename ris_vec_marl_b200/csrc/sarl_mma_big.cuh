// SARL rollout for MANY vehicles / RIS elements (BASELINE config 4: V = 32, M = 256): the cascaded
// reduction of one env is the real GEMM  [2V x 2M] . [2M x T]  (= [64 x 512] per step column) on the
// tensor cores, one thread BLOCK per env.  Reference: Simulation-SARL/Environment.py:125-131, 149-171,
// 318-359.  Same operand split (two binary16 pieces, 3 mma per product) and the same max-plus treatment
// of the DataBuf recursion as k_sarl_mma_tma (sarl_mma.cuh); what differs is the decomposition into
// WARP ROLES that only meet at mbarriers (no block-wide barrier in the loop):
//
//   16 mma warps = 4 row tiles r (8 vehicles: rows Re S_v, Im S_v) x 4 K-quarters q (M / 4 elements each).
//   Warp (r, q) keeps ITS slice of the geometry phasors in registers as mma A fragments (8 k-tiles x
//   8 registers) for the whole rollout.  theta = exp(j*phase) of a 16-step stage is evaluated ONCE per
//   block (every mma warp produces 4 of the 64 B-fragment sets: one packed sin/cos per lane and set),
//   split, and parked in shared memory in fragment order (double buffered: stage k + 2 is produced while
//   stage k + 1 multiplies); the warps stream the fragments of their K-quarter with LDS.128 and leave
//   their partial sums in a double-buffered area.  The mma warps synchronise among themselves with one
//   named barrier per stage and run up to two stages ahead of
//   8 step warps (two per row tile, 4 vehicles each): lane = (vehicle, steps 2 t8, 2 t8 + 1) -- the per-step part of
//   k_sarl_mma_tma with the max-plus shuffle scan over the vehicle's 8 lanes, then the lane's two steps in
//   the reference's float64 order.  A step warp waits for "partials of stage k full" (mbarrier, 4 arrivals),
//   folds the four K-quarter sums, hands the buffer back ("empty", 2 arrivals), and files its results in the
//   out tile [6][16][V]; the step warps meet at a named barrier and one thread issues the TMA tensor stores
//   (full rows of V floats per trace and step).  (One step warp per row tile with four steps per lane was
//   the critical path: ~1100 dependent instructions per stage; the mma warps need 390.)
#pragma once
#include "sarl_mma.cuh"

namespace risvec {

struct SarlBigOutMaps {
    CUtensorMap trace[6];  // DataBuf, data_t, data_p, over_power, over_data, rate: [T, E*V] f32, box {V, 16}
};

constexpr int kBigMmaWarps = 16, kBigStepWarps = 8;
constexpr int kBigThreads = 32 * (kBigMmaWarps + kBigStepWarps);
constexpr int kBigPartStride = 40;  // floats per (warp, g) row of the partial-sum area (32 used; pad breaks bank conflicts)
constexpr int kBigPartFloats = 16 * 8 * kBigPartStride;  // one stage of partial sums (double buffered)
__host__ __device__ constexpr int sarl_big_smem_bytes(int KQ, int V) {
    return 2 * (4 * KQ) * 2 * 32 * 16            // B fragments, two stages
           + 2 * kBigPartFloats * 4              // K-quarter partial sums, two stages
           + 2 * (4 * KQ) * 2 * 32 * 8           // staged phases (cp.async), two stages
           + 8 * 16 * 4                          // reward partial sums [step warp][step]
           + 6 * 16 * V * 4                      // out tile
           + 16 * 8                              // mbarriers full[4][2], empty[4][2]
           + 256;                                // alignment slack
}

__device__ __noinline__ int draw_arrival_cold(const Dims& d, int e, int v, long long step, float lam) {
    return draw_arrival(d, e, v, step, lam);  // on-device Philox arrivals: kept out of the step warps' hot loop
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

template <int KQ>
__global__ void __launch_bounds__(kBigThreads, 1)
    k_sarl_mma_big(Dims d, State s, const SarlConsts c, SarlArgs a, const __grid_constant__ SarlBigOutMaps tm_out) {
    constexpr int KT = 4 * KQ, R = 16;
    extern __shared__ unsigned char big_smem_raw[];
    const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const int e = blockIdx.x;
    const int NS = (T + R - 1) / R;

    // ---- shared memory carve-up (128 B aligned: the out tile is a TMA source)
    const uint32_t base_s = (smem_u32(big_smem_raw) + 127u) & ~127u;
    unsigned char* base_g = big_smem_raw + (base_s - smem_u32(big_smem_raw));
    constexpr int BF_STAGE = KT * 2 * 32 * 16;
    uint4* const bf = reinterpret_cast<uint4*>(base_g);                                  // [2][KT][2][32]
    float* const part = reinterpret_cast<float*>(base_g + 2 * BF_STAGE);                 // [2][16][8][kBigPartStride]
    float2* const phs = reinterpret_cast<float2*>(part + 2 * kBigPartFloats);            // [2][16 warps][NSETS][32] staged phases
    float* const rsum = reinterpret_cast<float*>(phs + 2 * 16 * ((KT * 2) / 16) * 32);   // [8][16]
    float* const out_g = rsum + 8 * 16;                                                  // [6][16][V]
    const uint32_t out_s = base_s + (uint32_t)((unsigned char*)out_g - base_g);
    const int TRACE_WORDS = R * V;
    const uint32_t bars = (out_s + 6 * TRACE_WORDS * 4 + 7u) & ~7u;  // full[r][b] at 8 (2 r + b), empty at + 64
    if (threadIdx.x == 0) {
        for (int i = 0; i < 8; ++i) {
            mbar_init(bars + 8 * i, 4);        // full: the four K-quarter warps of the row tile
            mbar_init(bars + 64 + 8 * i, 2);   // empty: the row tile's two step warps
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp < kBigMmaWarps) {
        // ================================ mma warps ================================
        const int r = warp >> 2, q = warp & 3;
        const int v = 8 * r + g;
        const bool vact = v < V;
        const size_t ev = (size_t)e * V + min(v, V - 1);
        // A operand: vehicle v, elements 8 j + 2 tig + {0, 1} of the k-tiles j = KQ q .. KQ q + KQ - 1
        // Only the fragments of row g + 8 (Im S_v): packed (Im w, Re w), are kept -- 4 registers per k-tile.  The
        // fragment of row g (Re S_v) is (Re w, -Im w) = the same register with its halves swapped and the sign of
        // the high half flipped (binary16 rounding is symmetric, so this holds for the hi and the lo piece): two
        // ALU instructions at the point of use instead of 32 more registers per lane.
        uint32_t Aih[KQ][2], Ail[KQ][2];
        {
            const double2 z = unit_phasor64(d.angle_BR - s.angle[ev]);  // w(v, m) = z^m, float64 (SARL:134-145)
            const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
            double2 w = cpow64(z, 2u * (unsigned)tig + 8u * (unsigned)(KQ * q));
#pragma unroll
            for (int jj = 0; jj < KQ; ++jj) {
                const int ma = 8 * (KQ * q + jj) + 2 * tig;
                double2 wa = w, wb = cmul64(w, z);
                if (!(vact && ma < M)) wa = make_double2(0.0, 0.0);
                if (!(vact && ma + 1 < M)) wb = make_double2(0.0, 0.0);
                split_h2(wa.y, wa.x, Aih[jj][0], Ail[jj][0]);   // row g + 8 (Im S_v): ( Im w,  Re w), element 8 j + 2 tig
                split_h2(wb.y, wb.x, Aih[jj][1], Ail[jj][1]);   // ... element 8 j + 2 tig + 1
                w = cmul64(w, z8);
            }
        }
        auto re_row = [](uint32_t im_row) {  // (Im w, Re w) -> (Re w, -Im w)
            return __funnelshift_l(im_row, im_row, 16) ^ 0x80000000u;
        };
        // producer side: this warp makes the B fragments of sets warp + 16 u (k-tile (warp >> 1) + 8 u, n-tile
        // warp & 1).  B column n = g of tile A is step 4 (g >> 1) + (g & 1) of the stage, of tile B the step two
        // later, so that an accumulator lane (g, tig') ends up with the four consecutive steps 4 tig' .. 4 tig' + 3.
        constexpr int NSETS = (KT * 2) / 16;
        static_assert(KT * 2 == NSETS * 16, "the 2 KT fragment sets divide evenly over the 16 mma warps");
        const int row_w = 4 * (g >> 1) + (g & 1) + 2 * (warp & 1);
        const unsigned sM = (unsigned)E * M;  // 32-bit indices (host-checked)
        const int m_w = 8 * (warp >> 1) + 2 * tig;                       // element of set u: m_w + 64 u
        const float* const ph_w = a.phase + (unsigned)e * M + m_w;       // + t * sM + 64 u
        uint4* const bf_w = bf + warp * 32 + lane;                       // + buffer * (KT * 64) + u * 512
        // The phases of the next stage to produce travel global -> shared by cp.async into a lane-private slot
        // (no registers, no scoreboard: a register prefetch was spilled by the 80-register budget and the
        // spill store then waited for the load every stage).  Slots of sets beyond M stay zero.
        float2* const ph_slot = phs + (warp * NSETS) * 32 + lane;        // + buffer * (16 NSETS 32) + u * 32
#pragma unroll
        for (int u = 0; u < NSETS; ++u) ph_slot[u * 32] = ph_slot[16 * NSETS * 32 + u * 32] = make_float2(0.f, 0.f);
        auto load_phases = [&](int k) {
            const float* q0 = ph_w + (unsigned)min(k * R + row_w, T - 1) * sM;
            const uint32_t dst = smem_u32(ph_slot + (k & 1) * (16 * NSETS * 32));
#pragma unroll
            for (int u = 0; u < NSETS; ++u)
                if (m_w + 64 * u < M)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + u * 256), "l"(q0 + 64 * u) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        auto produce = [&](int k) {  // phases of stage k (my slots) -> bf[k & 1]
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            uint4* dst = bf_w + (k & 1) * (KT * 64);
            const float2* src = ph_slot + (k & 1) * (16 * NSETS * 32);
#pragma unroll
            for (int u = 0; u < NSETS; ++u) {
                float2 sn, cs;
                sincos_pi2(src[u * 32], &sn, &cs);  // theta = exp(j*phase) (SARL:125-131)
                uint4 f;  // (b0 hi, b1 hi, b0 lo, b1 lo): every mma B operand is an adjacent register pair
                split_h2(cs.x, sn.x, f.x, f.z);  // b0: element 8 j + 2 tig
                split_h2(cs.y, sn.y, f.y, f.w);  // b1: element 8 j + 2 tig + 1
                dst[u * 512] = f;
            }
        };
        float4* const part_w = reinterpret_cast<float4*>(part + (warp * 8 + g) * kBigPartStride + tig * 8);
        auto mma_stage = [&](int k) {  // fragments bf[k & 1] -> my K-quarter's partial sums in part[k & 1]
            float mA[4] = {0.f, 0.f, 0.f, 0.f}, xA[4] = {0.f, 0.f, 0.f, 0.f};
            float mB[4] = {0.f, 0.f, 0.f, 0.f}, xB[4] = {0.f, 0.f, 0.f, 0.f};
            const uint4* bk = bf + ((k & 1) * KT * 2 + 2 * (KQ * q)) * 32 + lane;  // sets 2 j, 2 j + 1 of my k-tiles
#pragma unroll
            for (int jj = 0; jj < KQ; ++jj) {
                const uint4 fa = bk[(2 * jj) * 32], fb = bk[(2 * jj + 1) * 32];
                const uint32_t Ah[4] = {re_row(Aih[jj][0]), Aih[jj][0], re_row(Aih[jj][1]), Aih[jj][1]};
                const uint32_t Al[4] = {re_row(Ail[jj][0]), Ail[jj][0], re_row(Ail[jj][1]), Ail[jj][1]};
                mma_16816(mA, Ah, fa.x, fa.y);
                mma_16816(xA, Ah, fa.z, fa.w);
                mma_16816(xA, Al, fa.x, fa.y);
                mma_16816(mB, Ah, fb.x, fb.y);
                mma_16816(xB, Ah, fb.z, fb.w);
                mma_16816(xB, Al, fb.x, fb.y);
            }
            // the step warp must have handed this buffer back (its previous tenant was stage k - 2)
            mbar_wait(bars + 64 + 8 * (2 * r + (k & 1)), (((uint32_t)k >> 1) & 1u) ^ 1u);
            // partial S of my lane's four steps 4 tig + i: (Re, Im) pairs, i = 0, 1 from tile A, 2, 3 from tile B
            float4* pw = part_w + (k & 1) * (kBigPartFloats / 4);
            pw[0] = make_float4(mA[0] + xA[0], mA[2] + xA[2], mA[1] + xA[1], mA[3] + xA[3]);
            pw[1] = make_float4(mB[0] + xB[0], mB[2] + xB[2], mB[1] + xB[1], mB[3] + xB[3]);
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 8 * (2 * r + (k & 1)));  // full[r][k & 1]
        };
        constexpr int MMA_THREADS = 32 * kBigMmaWarps;
        load_phases(0);
        produce(0);
        load_phases(1 < NS ? 1 : 0);
        named_bar_sync(1, MMA_THREADS);
        for (int k = 0; k < NS; ++k) {
            if (k + 1 < NS) {  // theta of stage k + 1 -> the other fragment buffer (free since the barrier of stage k - 1)
                produce(k + 1);
                load_phases(k + 2 < NS ? k + 2 : k + 1);
            }
            mma_stage(k);
            named_bar_sync(1, MMA_THREADS);  // fragments of stage k + 1 complete, those of stage k consumed
        }
    } else {
        // ================================ step warps ================================
        // step warp (r, h) serves vehicles 8 r + 4 h + {0..3}: lane = (g4, t8) = vehicle, steps 2 t8 and 2 t8 + 1
        const int sw = warp - kBigMmaWarps, r = sw >> 1, h = sw & 1;
        const int g4 = lane >> 3, t8 = lane & 7;
        const int gv = 4 * h + g4;          // vehicle within the row tile
        const int v = 8 * r + gv;
        const bool vact = v < V;
        const int vc = min(v, V - 1);
        const size_t ev = (size_t)e * V + vc;
        constexpr int STEP_THREADS = 32 * kBigStepWarps;
        const bool leader = sw == 0 && lane == 0;
        double buf = s.databuf[ev];  // replicated over the 8 lanes of the vehicle
        const float coef = vact ? (float)(s.amp[ev] / (kSigma * kSigma)) : 0.f;  // SARL:157-159
        const long long step0 = s.step_ctr[e];
        const unsigned s2V = (unsigned)E * 2 * V, sVv = (unsigned)E * V;
        const float* const ac_w = a.action + (unsigned)e * 2 * V + vc;
        const int* const ar_w = a.arrivals != nullptr ? a.arrivals + (unsigned)e * V + vc : nullptr;
        float2 na0, na1;
        int narr0 = 0, narr1 = 0;
        auto load_scalars = [&](int k) {
            const unsigned t0 = (unsigned)min(k * R + 2 * t8, T - 1), t1 = (unsigned)min(k * R + 2 * t8 + 1, T - 1);
            na0 = make_float2(__ldg(ac_w + t0 * s2V), __ldg(ac_w + t1 * s2V));
            na1 = make_float2(__ldg(ac_w + t0 * s2V + V), __ldg(ac_w + t1 * s2V + V));
            if (ar_w != nullptr) {
                narr0 = __ldg(ar_w + t0 * sVv);
                narr1 = __ldg(ar_w + t1 * sVv);
            }
        };
        // steps 2 t8, 2 t8 + 1 of vehicle gv sit in accumulator lane (gv, tig' = t8 >> 1), slots 2 (t8 & 1) + {0, 1},
        // of the mma warps (r, 0..3): one 16-byte (Re, Im, Re, Im) read per K-quarter
        const float* const part_r = part + (r * 32 + gv) * kBigPartStride + (t8 >> 1) * 8 + (t8 & 1) * 4;
        float* const out_w = out_g + (2 * t8) * V + v;
        float f_rate = 0.f, f_dt = 0.f, f_dp = 0.f, f_overp = 0.f, f_overd = 0.f;
        int f_arr = 0;
        bool f_mine = false;
        load_scalars(0);
        for (int k = 0; k < NS; ++k) {
            const float2 a0 = na0, a1 = na1;
            int arr0 = narr0, arr1 = narr1;
            if (k + 1 < NS) load_scalars(k + 1);
            // ---- the four K-quarter sums of stage k
            mbar_wait(bars + 8 * (2 * r + (k & 1)), ((uint32_t)k >> 1) & 1u);
            float2 re = make_float2(0.f, 0.f), im = re;
            const float* pr = part_r + (k & 1) * kBigPartFloats;
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
                const float4 p0 = *reinterpret_cast<const float4*>(pr + qq * 8 * kBigPartStride);
                re.x += p0.x; im.x += p0.y; re.y += p0.z; im.y += p0.w;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 64 + 8 * (2 * r + (k & 1)));  // empty[r][k & 1]: my half handed back
            // ---- per-step part (SARL:327-358) of my steps tb, tb + 1 (packed fp32x2 where both steps do the same)
            const int tb = k * R + 2 * t8;
            const bool ok0 = vact && tb < T, ok1 = vact && tb + 1 < T;
            if (a.arrivals == nullptr) {
                arr0 = ok0 ? draw_arrival_cold(d, e, vc, step0 + tb, c.lam) : 0;
                arr1 = ok1 ? draw_arrival_cold(d, e, vc, step0 + tb + 1, c.lam) : 0;
            }
            float2 rate, dt, dp;
            sarl_rate2(re, im, a0, a1, coef, c, rate, dt, dp);
            const double d0 = ok0 ? __dadd_rn((double)dt.x, (double)dp.x) : 0.0;  // identity step when not ok
            const double d1 = ok1 ? __dadd_rn((double)dt.y, (double)dp.y) : 0.0;
            const double i0 = ok0 ? __dmul_rn(__dmul_rn((double)arr0, c.tf), 1000.0) : 0.0;
            const double i1 = ok1 ? __dmul_rn(__dmul_rn((double)arr1, c.tf), 1000.0) : 0.0;
            // DataBuf at my first step: inclusive scan of the lanes' two-step maps over the vehicle's 8 lanes
            // (the loop, not mp_scan<8>: the unrolled helper compiles to different code for this kernel)
            MaxPlus f = mp_then(MaxPlus{i0 - d0, i0}, MaxPlus{i1 - d1, i1});
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const MaxPlus pq{__shfl_up_sync(kFull, f.a, o, 8), __shfl_up_sync(kFull, f.b, o, 8)};
                const MaxPlus fo = mp_then(pq, f);
                if (t8 >= o) f = fo;
            }
            const MaxPlus ex{__shfl_up_sync(kFull, f.a, 1, 8), __shfl_up_sync(kFull, f.b, 1, 8)};  // maps before mine
            const MaxPlus all{__shfl_sync(kFull, f.a, 7, 8), __shfl_sync(kFull, f.b, 7, 8)};       // the whole stage
            const double xin = mp_apply(ex, buf);
            double cur = t8 == 0 ? buf : xin;
            buf = mp_apply(all, buf);
            // my two steps in the reference's order (SARL:333-358)
            float overd[2], nbf[2], barg[2], curf[2];
            bool pos[2];
#pragma unroll
            for (int i = 0; i < 2; ++i)
                sarl_settle(cur, i ? d1 : d0, i ? dp.y : dp.x, i ? i1 : i0, i ? ok1 : ok0, overd[i], nbf[i], barg[i],
                            pos[i], curf[i]);
            float2 op, base2;
            sarl_reward2(make_float2(barg[0], barg[1]), make_float2(nbf[0], nbf[1]), a0, a1, c, op, base2);
            // the out tile is free again once the TMA stores of the previous stage have read it
            if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            named_bar_sync(2, STEP_THREADS);
            float rew[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float od = overd[i];
                const float overp = od > 0.f ? (i ? op.y : op.x) : 0.f;  // only where the buffer went negative
                const float pen = pos[i] ? c.pen1 : ((od > 2.0f) ? c.pen2 : 0.f);  // SARL:343-352 (a helper changed the code)
                rew[i] = (i ? ok1 : ok0) ? __fsub_rn(i ? base2.y : base2.x, pen) : 0.f;
                if (vact) {
                    float* o = out_w + i * V;
                    o[0 * TRACE_WORDS] = curf[i];
                    o[1 * TRACE_WORDS] = i ? dt.y : dt.x;
                    o[2 * TRACE_WORDS] = i ? dp.y : dp.x;
                    o[3 * TRACE_WORDS] = overp;
                    o[4 * TRACE_WORDS] = od;
                    o[5 * TRACE_WORDS] = i ? rate.y : rate.x;
                }
                if ((i ? ok1 : ok0) && tb + i == T - 1) {
                    f_rate = i ? rate.y : rate.x; f_dt = i ? dt.y : dt.x; f_dp = i ? dp.y : dp.x;
                    f_overp = overp; f_overd = od; f_arr = i ? arr1 : arr0; f_mine = true;
                }
                rew[i] += __shfl_xor_sync(kFull, rew[i], 8);   // sum over the warp's 4 vehicles (8 warps meet in smem)
                rew[i] += __shfl_xor_sync(kFull, rew[i], 16);
            }
            if (g4 == 0) {
                rsum[sw * 16 + 2 * t8] = rew[0];
                rsum[sw * 16 + 2 * t8 + 1] = rew[1];
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            named_bar_sync(2, STEP_THREADS);  // out tile and reward sums of the stage complete
            if (leader) {
#pragma unroll
                for (int n = 0; n < 6; ++n) tma_store_2d(&tm_out.trace[n], out_s + n * (TRACE_WORDS * 4), e * V, k * R);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            if (sw == 0 && lane < 16 && k * R + lane < T) {
                float acc = 0.f;
#pragma unroll
                for (int w2 = 0; w2 < kBigStepWarps; ++w2) acc += rsum[w2 * 16 + lane];
                const float rw = __fmul_rn(acc, 1.0f / (float)V);
                if (a.out.reward != nullptr) a.out.reward[(size_t)(k * R + lane) * E + e] = rw;
                if (k * R + lane == T - 1) s.reward[e] = rw;
            }
        }
        // ---- registers -> state
        if (f_mine) {
            s.rate[ev] = f_rate;
            s.data_t[ev] = f_dt;
            s.data_p[ev] = f_dp;
            s.over_power[ev] = f_overp;
            s.over_data[ev] = f_overd;
            s.data_r[ev] = f_arr;
        }
        if (t8 == 0 && vact) s.databuf[ev] = buf;
        if (leader) {
            s.step_ctr[e] = step0 + T;
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
        }
    }
    // elements_phase_shift_real = the last action_phase (SARL:128)
    for (int m = threadIdx.x; m < M; m += kBigThreads)
        s.phase_real[(size_t)e * M + m] = __ldg(a.phase + ((size_t)(T - 1) * E + e) * M + m);
}

}  // namespace risvec
