// SARL rollout for MANY vehicles / RIS elements (BASELINE config 4: V = 32, M = 256) on the 5th-generation
// tensor cores: the cascaded reduction of one env, the real GEMM  [2V x 2M] . [2M x T]  (SARL:149-171), is
// issued as tcgen05.mma (M = 128, N = 32, K = 16) by ONE thread: the constant operand A and the accumulators
// live in tensor memory, the per-stage operand B in shared memory.  One thread block per env.  Reference: Simulation-SARL/Environment.py:125-131, 149-171,
// 318-359.  Same operand split as sarl_mma.cuh (x = hi + lo in binary16, float32 accumulation, the hi*hi
// product in its own accumulator) and the same max-plus treatment of the DataBuf recursion.  Both pieces of
// both operands ride in ONE instruction per k-step: the rows of A are (hi rows | lo rows), the columns of B
// (hi steps | lo steps), so D holds the four partial products side by side and the step warps add them.
//
//   A  [128 x 16 KT] binary16 in TENSOR MEMORY (lane = row, one 32-bit column per RIS element = its two K
//      values; 8 KT columns): the geometry phasors w(v, m) = z_v^m of the env, written ONCE per rollout with
//      tcgen05.st by the 16 non-MMA warps.  Lane quarter q (rows 32 q .. 32 q + 31) belongs to vehicles
//      8 q .. 8 q + 7: rows 32 q + g / + 8 + g = hi piece of the Re S / Im S row of vehicle 8 q + g, rows
//      32 q + 16 + g / + 24 + g = the lo piece of the same rows.
//   B  [32 x 16 KT] binary16 in shared memory, K-major core matrices (8 rows x 16 bytes), no swizzle, double buffered: theta = exp(j*phase) of a 16-step stage, rows
//      0-15 the hi piece, rows 16-31 the lo piece, produced by 8 warps (packed sin/cos polynomial, split, one
//      8-byte store per piece and element pair).  Tile row c (mod 16) holds step 4 ((c & 7) >> 1) + 2 (c >> 3)
//      + (c & 1) of the stage, so that the accumulator fragment of a lane (tcgen05.ld 16x256b) is FOUR
//      CONSECUTIVE steps of one vehicle.
//   D  [128 x 32] float32, columns 0-15 = . x hi theta, 16-31 = . x lo theta; kUmmaChains accumulators per stage
//      (k-step j adds into chain j % kUmmaChains), double buffered, in the tensor-memory columns after A.
//
// Warp roles (they only meet at mbarriers):
//   warps 0-3 / 4-7  step warps of the even / odd stages: warp q reads rows 32 q .. 32 q + 31 of D (its
//                    tensor-memory lane quarter), lane (g, tig) = vehicle 8 q + g, steps 4 tig .. 4 tig + 3: the
//                    per-step part of k_sarl_mma_tma.  The two sets overlap in time: everything of a stage
//                    except "apply the stage's composed max-plus map to DataBuf" is independent of the stage
//                    before, so the only serial link is a hand-off of 8 doubles per warp (hbuf + mbarrier).
//   warps 8-15       producers of B (stage k + 1 while stage k multiplies)
//   warp 16          one lane: waits "B full" + "D empty", issues KT tcgen05.mma, commits to "B empty" + "D full"
// Measured (B200, globaltimer stamps per block, T = 256): tensor-memory allocation 0.26 us, A 4.0 us, first B
// stage 1.7 us later, then one stage per 1.5 us, 1.7 us from the last "D full" to the end of the block: 33 us per
// env.  The steady state is bound by the tensor core's DISPATCH of these small instructions: 32 per stage take
// 1.44 us (~83 clocks each, where the datapath needs 16) -- the same with N = 64 per instruction (timing
// experiment) and the same with two alternating accumulator chains: the instruction time follows the bytes of
// operand A (shared memory, unswizzled: ~32 B per clock; tensor memory: ~50-64 B per clock), not N.  A variant
// with 32-step stages (N = 64: half the instructions per step, both step-warp sets on one accumulator) was
// correct but slower (0.249 ms): the two sets then run in lock-step, and a set needs ~2.8 us per 16-step
// stage -- the step warps, two sets of four, are the other limit of the steady state.  (History: with A in shared memory an instruction took ~128 clocks, three M = 64,
// N = 16 instructions per k-step ~62 clocks each.)
#pragma once
#include "sarl_mma.cuh"
#include "sarl_mma_big.cuh"

namespace risvec {

constexpr int kUmmaStepWarps = 8, kUmmaProdWarps = 8;
constexpr int kUmmaThreads = 32 * (kUmmaStepWarps + kUmmaProdWarps + 1);
#ifndef RISVEC_UMMA_CHAINS
#define RISVEC_UMMA_CHAINS 2
#endif
// accumulators per stage: k-step j adds into chain j % kUmmaChains and the step warps add the chains.  Not for
// speed (the instruction rate does not depend on it) but for accuracy: the tensor core adds every k-step into a
// float32 D of magnitude ~sqrt(2 M); shorter chains keep that rounding inside the rate tolerance at M = 256.
constexpr int kUmmaChains = RISVEC_UMMA_CHAINS;
__host__ __device__ constexpr int umma_tmem_cols(int KQ) {  // A (8 KT columns) + 2 stages x chains x 32 columns, power of two
    return 32 * KQ + 64 * kUmmaChains <= 128 ? 128 : (32 * KQ + 64 * kUmmaChains <= 256 ? 256 : 512);
}
static_assert(32 * 8 + 64 * kUmmaChains <= 512, "tensor memory: A of the largest shape + the accumulators");
// instruction descriptor of tcgen05.mma kind::f16: D = F32 (bits 4-5 = 1), A = B = F16 (0), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28
constexpr uint32_t kUmmaIdesc = (1u << 4) | ((32u >> 3) << 17) | ((128u >> 4) << 24);

__host__ __device__ constexpr int sarl_umma_smem_bytes(int KQ, int V) {
    return 2 * (4 * KQ) * 1024           // B [buffer] (hi and lo rows)
           + 2 * 6 * 16 * V * 4          // out tiles of the two step-warp sets
           + 2 * 2 * 16 * 3 * V * 4      // input tiles [set][buffer]: actions [16][2 V] + arrivals [16][V] (TMA)
           + 2 * 4 * 16 * 4              // reward partial sums [set][warp][step]
           + 4 * 2 * 8 * 8               // DataBuf hand-off [warp][writer set][vehicle]
           + 20 * 8 + 16                 // mbarriers, tensor-memory base address
           + 256;                        // alignment slack
}
// one block per SM (a block owns up to all 512 tensor-memory columns): the launch asks for more than half of the
// SM's shared memory whatever the block needs
__host__ __device__ constexpr int sarl_umma_smem_request(int KQ, int V) {
    return sarl_umma_smem_bytes(KQ, V) > 120 * 1024 ? sarl_umma_smem_bytes(KQ, V) : 120 * 1024;
}

// shared-memory matrix descriptor: K-major, no swizzle; core matrices of one 8-row group are 128 B apart
// along K (leading byte offset), 8-row groups 256 B apart (stride byte offset); version 1 (Blackwell)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]), "r"(r[1]),
                 "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, float (&r)[8]) {
    uint32_t u[8];
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                 : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = __uint_as_float(u[i]);
}

template <int KQ>
// (17 warps are allotted registers as 20: at most 96 per thread)
__global__ void __launch_bounds__(kUmmaThreads, 1)
    k_sarl_umma(Dims d, State s, const SarlConsts c, SarlArgs a, const __grid_constant__ SarlBigOutMaps tm_out,
                const __grid_constant__ CUtensorMap tm_ac, const __grid_constant__ CUtensorMap tm_ar) {
    constexpr int KT = 4 * KQ, R = 16;
    constexpr int B_BYTES = KT * 1024, A_COLS = 8 * KT, TMEM_COLS = umma_tmem_cols(KQ);
    extern __shared__ unsigned char umma_smem_raw[];
    const int warp = __shfl_sync(kFull, (int)(threadIdx.x >> 5), 0);
    int lane_id = threadIdx.x & 31;
    asm volatile("" : "+r"(lane_id));  // opaque: keeps ptxas from re-deriving lane-dependent addresses from %tid in the loops
    const int lane = lane_id, g = lane >> 2, tig = lane & 3;
    const int E = d.E, V = d.V, M = d.M, T = a.T;
    const int e = blockIdx.x;
    const int NS = (T + R - 1) / R;
    const int kt_run = min(KT, (2 * M + 15) >> 4);  // k-steps that hold elements (the rest of A is zero)

    // ---- shared memory carve-up (128 B aligned)
    const uint32_t base_s = (smem_u32(umma_smem_raw) + 127u) & ~127u;
    unsigned char* const base_g = umma_smem_raw + (base_s - smem_u32(umma_smem_raw));
    const uint32_t b_s = base_s;                                       // + buffer * B_BYTES
    const int TRACE_WORDS = R * V;
    const uint32_t out_s = b_s + 2 * B_BYTES;                          // + set * 6 TRACE_WORDS 4
    float* const out_g = reinterpret_cast<float*>(base_g + 2 * B_BYTES);
    const int IN_BYTES = R * 3 * V * 4;                                // one input tile: actions [16][2 V] | arrivals [16][V]
    const uint32_t in_s = out_s + 2 * 6 * TRACE_WORDS * 4;             // + (set * 2 + buffer) * IN_BYTES
    unsigned char* const in_g = reinterpret_cast<unsigned char*>(out_g + 2 * 6 * TRACE_WORDS);
    float* const rsum = reinterpret_cast<float*>(in_g + 4 * IN_BYTES);  // [set][4][16]
    double* const hbuf = reinterpret_cast<double*>(rsum + 2 * 4 * 16);  // [warp][writer set][8]
    const uint32_t bars = in_s + 4 * IN_BYTES + 2 * 4 * 16 * 4 + 4 * 2 * 8 * 8;
    // mbarriers: B full [2] (8 producer warps), B empty [2] (commit), D full [2] (commit), D empty [2] (4 step warps),
    //            hand-off [4 warps][2 writer sets] (1), inputs full [2 sets][2 buffers] (TMA transaction bytes)
    const uint32_t bar_bfull = bars, bar_bempty = bars + 16, bar_dfull = bars + 32, bar_dempty = bars + 48, bar_h = bars + 64;
    const uint32_t bar_in = bars + 128;
    uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(base_g + (bars + 160 - base_s));
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(bar_bfull + 8 * i, kUmmaProdWarps);
            mbar_init(bar_bempty + 8 * i, 1);
            mbar_init(bar_dfull + 8 * i, 1);
            mbar_init(bar_dempty + 8 * i, 4);
        }
        for (int i = 0; i < 8; ++i) mbar_init(bar_h + 8 * i, 1);
        for (int i = 0; i < 4; ++i) mbar_init(bar_in + 8 * i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == kUmmaStepWarps + kUmmaProdWarps) {  // tensor memory: A + two stages of accumulators
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    constexpr int D_COLS = 32 * kUmmaChains;  // one stage of accumulators
    const uint32_t tmem_d = tmem + A_COLS;    // + D_COLS * buffer + 32 * chain
    const int n_chains = min(kUmmaChains, kt_run);
    if (warp < kUmmaStepWarps + kUmmaProdWarps) {
        // ---- A operand, once per rollout: warp -> lane quarter q = warp & 3 and the elements [2 KT kp, 2 KT (kp + 1)),
        // kp = warp >> 2; lane i -> row 32 q + i: vehicle 8 q + (i & 7), Re / Im row (bit 3), hi / lo piece (bit 4)
        const int q = warp & 3, kp = warp >> 2;
        const int v = 8 * q + (lane & 7);
        const bool im_row = (lane >> 3) & 1, lo_piece = (lane >> 4) & 1;
        const bool vact = v < V;
        // The four lanes of a vehicle (Re / Im row x hi / lo piece) share the work: lane c = lane >> 3 walks the
        // elements m = c (mod 4) of the warp's range (w <- w z^4, float64), rounds to float32 and splits ONCE:
        // P = (hi Re w, hi Im w), Q = (lo Re w, lo Im w) as packed binary16 pairs.  Every row of the vehicle is a
        // permutation of those: the Re S row holds (Re w, -Im w) = the pair with the sign of its high half
        // flipped, the Im S row (Im w, Re w) = the pair with its halves swapped (rounding is symmetric).
        const int c4 = lane >> 3;
        const double2 z = unit_phasor64(d.angle_BR - s.angle[(size_t)e * V + min(v, V - 1)]);  // w(v, m) = z^m (SARL:134-145)
        const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2);
        double2 w = cpow64(z, (unsigned)(2 * KT * kp + c4));
        const uint32_t t_a = tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)(2 * KT * kp);
        { // L2 prefetch of the first two stages' phase rows (the producers' first loads then come from L2)
            const int t = threadIdx.x;  // 512 threads: 32 rows x 16 segments of 64 B ... of up to 1 KB per row
            const int row = min(t >> 4, T - 1), seg = (t & 15) * 16;
            if (seg < M) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.phase + ((size_t)row * E + e) * M + seg));
        }
#pragma unroll 1
        for (int cch = 0; cch < KT / 4; ++cch) {  // 8 elements = 8 columns per store
            uint32_t col[8];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const bool on = vact && 2 * KT * kp + 8 * cch + 4 * h + c4 < M;  // my element of this group of four
                uint32_t P, Q;
                split_h2(on ? (float)w.x : 0.f, on ? (float)w.y : 0.f, P, Q);
                w = cmul64(w, z4);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t p = __shfl_sync(kFull, P, (lane & 7) + 8 * i), qq = __shfl_sync(kFull, Q, (lane & 7) + 8 * i);
                    const uint32_t x = lo_piece ? qq : p;
                    col[4 * h + i] = im_row ? __byte_perm(x, x, 0x1032) : (x ^ 0x80000000u);
                }
            }
            tmem_st_32x32b_x8(t_a + 8 * cch, col);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    if (warp < kUmmaStepWarps) {
        // ================================ step warps ================================
        const int set = warp >> 2, wq = warp & 3;
        const int v = 8 * wq + g;
        const bool vact = v < V;
        const int vc = min(v, V - 1);
        const size_t ev = (size_t)e * V + vc;
        const bool leader = wq == 0 && lane == 0;
        const float coef = vact ? (float)(s.amp[ev] / (kSigma * kSigma)) : 0.f;  // SARL:157-159
        const long long step0 = s.step_ctr[e];
        // my lane quarter: lanes 0-15 the hi rows, 16-31 the lo rows; columns 0-15 x hi theta, 16-31 x lo theta
        const uint32_t t_hh = tmem_d + ((uint32_t)(32 * wq) << 16) + (uint32_t)(D_COLS * set), t_hl = t_hh + 16;
        const uint32_t t_lh = t_hh + (16u << 16), t_ll = t_lh + 16;
        float* const tile = out_g + set * 6 * TRACE_WORDS;
        const uint32_t tile_s = out_s + (uint32_t)set * 6 * TRACE_WORDS * 4;
        float* const out_w = tile + (4 * tig) * V + v;
        float* const rs = rsum + (set * 4) * 16;
        double* const h_mine = hbuf + (wq * 2 + set) * 8;         // what I hand to the other set
        const double* const h_other = hbuf + (wq * 2 + (set ^ 1)) * 8;
        const uint32_t bar_h_mine = bar_h + 8 * (wq * 2 + set), bar_h_other = bar_h + 8 * (wq * 2 + (set ^ 1));
        const int bar_id = 1 + set;
        // action rows and arrivals of a stage arrive by TMA in the set's input tiles (two in flight per set); the
        // leader issues the tile of stage k + 4 once the set has read the one of stage k
        const bool has_ar = a.arrivals != nullptr;
        auto issue_inputs = [&](int kk) {  // leader only
            const int nb = (kk >> 1) & 1;
            const uint32_t dst = in_s + (uint32_t)(set * 2 + nb) * IN_BYTES, bar = bar_in + 8 * (set * 2 + nb);
            mbar_expect_tx(bar, (uint32_t)(R * 2 * V * 4 + (has_ar ? R * V * 4 : 0)));
            tma_load_2d(dst, &tm_ac, e * 2 * V, kk * R, bar);
            if (has_ar) tma_load_2d(dst + R * 2 * V * 4, &tm_ar, e * V, kk * R, bar);
        };
        if (leader) {
            if (set < NS) issue_inputs(set);
            if (set + 2 < NS) issue_inputs(set + 2);
        }
        float f_rate = 0.f, f_dt = 0.f, f_dp = 0.f, f_overp = 0.f, f_overd = 0.f;
        int f_arr = 0;
        bool f_mine = false;
        double buf = s.databuf[ev];  // DataBuf before stage 0 (set 0 starts from the state)
        for (int k = set; k < NS; k += 2) {
            const int n = k >> 1;
            float2 a0[2], a1[2];
            int arr[4] = {0, 0, 0, 0};
            {
                mbar_wait(bar_in + 8 * (set * 2 + (n & 1)), (uint32_t)(n >> 1) & 1u);
                const float* ac = reinterpret_cast<const float*>(in_g + (set * 2 + (n & 1)) * IN_BYTES) + (4 * tig) * 2 * V + vc;
                const int* ar = reinterpret_cast<const int*>(in_g + (set * 2 + (n & 1)) * IN_BYTES + R * 2 * V * 4) + (4 * tig) * V + vc;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    a0[h] = make_float2(ac[(2 * h) * 2 * V], ac[(2 * h + 1) * 2 * V]);
                    a1[h] = make_float2(ac[(2 * h) * 2 * V + V], ac[(2 * h + 1) * 2 * V + V]);
                    if (has_ar) {
                        arr[2 * h] = ar[(2 * h) * V];
                        arr[2 * h + 1] = ar[(2 * h + 1) * V];
                    }
                }
            }
            // ---- the accumulators of stage k: rows g (Re) and g + 8 (Im) of my lane quarter, my four steps
            mbar_wait(bar_dfull + 8 * set, (uint32_t)n & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            float dm[8], dx[8];
            {
                float hl[8], lh[8], ll[8];
                tmem_ld_16x256b_x2(t_hh, dm);
                tmem_ld_16x256b_x2(t_hl, hl);
                tmem_ld_16x256b_x2(t_lh, lh);
                tmem_ld_16x256b_x2(t_ll, ll);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int i = 0; i < 8; ++i) dx[i] = (hl[i] + lh[i]) + ll[i];
#pragma unroll
                for (int ch = 1; ch < kUmmaChains; ++ch) {
                    if (ch < n_chains) {  // block-uniform
                        float hh[8];
                        tmem_ld_16x256b_x2(t_hh + 32 * ch, hh);
                        tmem_ld_16x256b_x2(t_hl + 32 * ch, hl);
                        tmem_ld_16x256b_x2(t_lh + 32 * ch, lh);
                        tmem_ld_16x256b_x2(t_ll + 32 * ch, ll);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            dm[i] += hh[i];
                            dx[i] += (hl[i] + lh[i]) + ll[i];
                        }
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_dempty + 8 * set);
            const int tb = k * R + 4 * tig;
            bool ok[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                ok[i] = vact && tb + i < T;
                if (a.arrivals == nullptr) arr[i] = ok[i] ? draw_arrival_cold(d, e, vc, step0 + tb + i, c.lam) : 0;
            }
            float2 rate[2], dt[2], dp[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float2 re = __fadd2_rn(make_float2(dm[4 * h], dm[4 * h + 1]), make_float2(dx[4 * h], dx[4 * h + 1]));
                const float2 im = __fadd2_rn(make_float2(dm[4 * h + 2], dm[4 * h + 3]), make_float2(dx[4 * h + 2], dx[4 * h + 3]));
                sarl_rate2(re, im, a0[h], a1[h], coef, c, rate[h], dt[h], dp[h]);
            }
            double dd[4], inc[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {  // steps past the end of the rollout (and unused vehicles) are identity steps
                const float dti = (i & 1) ? dt[i >> 1].y : dt[i >> 1].x, dpi = (i & 1) ? dp[i >> 1].y : dp[i >> 1].x;
                dd[i] = ok[i] ? __dadd_rn((double)dti, (double)dpi) : 0.0;
                inc[i] = ok[i] ? __dmul_rn(__dmul_rn((double)arr[i], c.tf), 1000.0) : 0.0;
            }
            // ---- composed map of my four steps, inclusive scan over tig (state independent)
            MaxPlus ex, all;  // the maps before mine, the whole stage
            mp_scan<4>(mp_then(mp_then(MaxPlus{inc[0] - dd[0], inc[0]}, MaxPlus{inc[1] - dd[1], inc[1]}),
                               mp_then(MaxPlus{inc[2] - dd[2], inc[2]}, MaxPlus{inc[3] - dd[3], inc[3]})),
                       tig, ex, all);
            // ---- the serial link: DataBuf after stage k - 1 from the other set, DataBuf after stage k to it
            if (k > 0) {
                mbar_wait(bar_h_other, (uint32_t)((k - 1) >> 1) & 1u);
                buf = h_other[g];
            }
            const double xin = mp_apply(ex, buf);
            double cur = tig == 0 ? buf : xin;
            buf = mp_apply(all, buf);
            if (k + 1 < NS) {
                if (tig == 0) h_mine[g] = buf;
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_h_mine);
            }
            // ---- my four steps in the reference's order (SARL:333-358)
            float overd[4], nbf[4], barg[4], curf[4];
            bool pos[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                sarl_settle(cur, dd[i], (i & 1) ? dp[i >> 1].y : dp[i >> 1].x, inc[i], ok[i], overd[i], nbf[i], barg[i],
                            pos[i], curf[i]);
            // ---- my set's out tile is free again once the TMA stores of its previous stage have read it
            if (leader) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            named_bar_sync(bar_id, 128);
            if (leader && k + 4 < NS) {  // every warp of the set has read the stage's input tile: refill it
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                issue_inputs(k + 4);
            }
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
                    rew[i] = ok[i] ? __fsub_rn(u ? base2.y : base2.x, pen) : 0.f;
                    if (vact) {
                        float* o = out_w + i * V;
                        o[0 * TRACE_WORDS] = curf[i];
                        o[1 * TRACE_WORDS] = u ? dt[h].y : dt[h].x;
                        o[2 * TRACE_WORDS] = u ? dp[h].y : dp[h].x;
                        o[3 * TRACE_WORDS] = overp;
                        o[4 * TRACE_WORDS] = od;
                        o[5 * TRACE_WORDS] = u ? rate[h].y : rate[h].x;
                    }
                    if (ok[i] && tb + i == T - 1) {
                        f_rate = u ? rate[h].y : rate[h].x; f_dt = u ? dt[h].y : dt[h].x; f_dp = u ? dp[h].y : dp[h].x;
                        f_overp = overp; f_overd = od; f_arr = arr[i]; f_mine = true;
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {  // sum over the warp's 8 vehicles; the set's 4 warps meet in shared memory
                rew[i] += __shfl_xor_sync(kFull, rew[i], 4);
                rew[i] += __shfl_xor_sync(kFull, rew[i], 8);
                rew[i] += __shfl_xor_sync(kFull, rew[i], 16);
            }
            {  // every lane of a tig group holds the four sums: lane g < 4 files the one of step tb + g
                const float r01 = (g & 1) ? rew[1] : rew[0], r23 = (g & 1) ? rew[3] : rew[2];
                if (g < 4) rs[wq * 16 + 4 * tig + g] = (g & 2) ? r23 : r01;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            named_bar_sync(bar_id, 128);  // out tile and reward sums of the stage complete
            if (leader) {
#pragma unroll
                for (int nn = 0; nn < 6; ++nn) tma_store_2d(&tm_out.trace[nn], tile_s + nn * (TRACE_WORDS * 4), e * V, k * R);
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            if (wq == 0 && lane < 16 && k * R + lane < T) {
                const float acc = (rs[lane] + rs[16 + lane]) + (rs[32 + lane] + rs[48 + lane]);
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
        if (set == ((NS - 1) & 1)) {  // my set ran the last stage
            if (tig == 0 && vact) s.databuf[ev] = buf;
            if (leader) s.step_ctr[e] = step0 + T;
        }
        if (leader) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before exit
    } else if (warp < kUmmaStepWarps + kUmmaProdWarps) {
        // ================================ producers of B ================================
        // warp pw makes the element blocks j = (pw >> 1) + 4 u (8 elements = one k-step) of the tile rows 8 rh + g,
        // rh = pw & 1: lane (g, tig) = row, elements 8 j + 2 tig + {0, 1}.  Row c of the tile is step sigma(c).
        const int pw = warp - kUmmaStepWarps, rh = pw & 1, j0 = pw >> 1;
        constexpr int NT = KT / 4;
        const int row_step = 4 * (g >> 1) + 2 * rh + (g & 1);
        const size_t sM = (size_t)E * M;
        const bool full = M == 8 * KT;  // every element block of every lane exists (block-uniform fast path)
        const int nu = min(NT, max(0, (M - 8 * j0 - 2 * tig + 31) >> 5));  // my element blocks j0 + 4 u that hold elements
        const float* const ph_w = a.phase + (size_t)e * M + 8 * j0 + 2 * tig;
        const float* q_last = ph_w + (size_t)(T - 1) * sM;
        const float* q = ph_w + (size_t)row_step * sM;  // my row of the stage to load next (clamped to step T - 1)
        size_t q_stride = (size_t)R * sM;
        asm volatile("" : "+l"(q_last), "+l"(q), "+l"(q_stride));  // opaque: held in registers, not re-derived per load
        // my 8 bytes of every element block: + buffer B_BYTES + piece 512 + u 4096
        const uint32_t b_w = b_s + (uint32_t)(j0 * 1024 + rh * 256 + (tig >> 1) * 128 + g * 16 + (tig & 1) * 8);
        float2 ph[NT];
        auto load_phases = [&](int k) {
            const float* qq = (k * R + row_step < T) ? q : q_last;
            q += q_stride;
            asm volatile("" : "+l"(qq));  // one address register pair for the loads below
            if (full) {
#pragma unroll
                for (int u = 0; u < NT; ++u) ph[u] = __ldg(reinterpret_cast<const float2*>(qq + 32 * u));
            } else {
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    ph[u] = u < nu ? __ldg(reinterpret_cast<const float2*>(qq + 32 * u)) : make_float2(0.f, 0.f);
            }
        };
        auto make_block = [&](float2 phase2, uint32_t dst) {
            float2 sn, cs;
            sincos_pi2(phase2, &sn, &cs);  // theta = exp(j*phase) (SARL:125-131)
            uint2 hi, lo;
            split_h2(cs.x, sn.x, hi.x, lo.x);  // element 8 j + 2 tig:     K = (cos, sin)
            split_h2(cs.y, sn.y, hi.y, lo.y);  // element 8 j + 2 tig + 1
            asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(dst), "r"(hi.x), "r"(hi.y) : "memory");
            asm volatile("st.shared.v2.b32 [%0+512], {%1, %2};" ::"r"(dst), "r"(lo.x), "r"(lo.y) : "memory");
        };
        load_phases(0);
        for (int k = 0; k < NS; ++k) {
            const int b = k & 1;
            float2 cur[NT];
#pragma unroll
            for (int u = 0; u < NT; ++u) cur[u] = ph[u];
            if (k + 1 < NS) load_phases(k + 1);
            mbar_wait(bar_bempty + 8 * b, (((uint32_t)k >> 1) & 1u) ^ 1u);  // the MMAs of stage k - 2 have read this buffer
            const uint32_t dst = b_w + (uint32_t)b * B_BYTES;
            if (full) {
#pragma unroll
                for (int u = 0; u < NT; ++u) make_block(cur[u], dst + u * 4096);
            } else {
#pragma unroll
                for (int u = 0; u < NT; ++u)
                    if (j0 + 4 * u < kt_run) make_block(cur[u], dst + u * 4096);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_bfull + 8 * b);
        }
    } else {
        // ================================ MMA issue ================================
        if (lane == 0) {
            for (int k = 0; k < NS; ++k) {
                const int b = k & 1;
                const uint32_t par = ((uint32_t)k >> 1) & 1u;
                mbar_wait(bar_bfull + 8 * b, par);
                mbar_wait(bar_dempty + 8 * b, par ^ 1u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_acc = tmem_d + (uint32_t)(D_COLS * b);
                uint64_t bd = umma_desc(b_s + b * B_BYTES, 128u, 256u);  // core matrices 128 B apart along K, 8-row groups 256 B apart
                for (int j = 0; j < kt_run; ++j) {
                    // A: 8 columns (16 K values) per k-step; D: chain j % kUmmaChains
                    umma_f16_ts(d_acc + 32 * (j % kUmmaChains), tmem + 8 * j, bd, kUmmaIdesc, j >= kUmmaChains);
                    bd += 1024 >> 4;  // B: next k-step; the start address field counts 16-byte units
                }
                umma_commit(bar_bempty + 8 * b);  // B buffer reusable once these MMAs have read it
                umma_commit(bar_dfull + 8 * b);   // ... and the accumulators complete
            }
        }
        __syncwarp();
    }
    // elements_phase_shift_real = the last action_phase (SARL:128)
    for (int m = threadIdx.x; m < M; m += kUmmaThreads)
        s.phase_real[(size_t)e * M + m] = __ldg(a.phase + ((size_t)(T - 1) * E + e) * M + m);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == kUmmaStepWarps + kUmmaProdWarps)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
}

}  // namespace risvec
