// Batched NOMA pairing: the stage the MARL driver runs before every Environ.step to build
// `noma_groups` (Simulation-MARL-BCD/marl_train_bcd.py:1315-1561 and the helpers at :128-398,
// :842-881).  One warp per env; every decision is warp-uniform, the N x N matrices and the 2^N
// matching table live in that warp's slice of shared memory.  All score arithmetic is float64
// with explicit round-to-nearest intrinsics in the reference's operation order (thresholds are
// order statistics of the very values they are compared with, so exact ties are structural and
// must survive); pair_affinity_hist is float32 as in the reference (:1288).
#pragma once
#include <math_constants.h>

#include "common.cuh"

namespace risvec {

struct PairArgs {
    const float* p01;        // [E, *] offload power in [0,1] (row 0 of the env action), env stride below
    long long p01_stride;
    const int* reuse;        // [E] or NULL: != 0 -> frozen groups (:1542-1547), solve skipped
    int topk;                // K_now (:1324)
    double tau_q;            // q_now (:1329)
    int recalc, decay, fresh;   // fresh: first step of an episode (:1282-1297) -- history / streak start from zero
    int min_pairs, backoff_rounds;
    double accept_q, accept_q_step, completion_q;
    int relax_topk_step;
    double relax_tau_factor, tau_floor;
    double w_delta, abs_min_db, qos_pen;
    float w_hist, decay_f;
    int qos_enable;
    double noise, P_max, sinr_min;   // sinr_min: see build_qos
    // state (arena fields RISVEC_F_PAIR_* / RISVEC_F_NOMA_*)
    float* hist;
    int* streak;
    double* tau;
    int* lastk;
    int* partner;
    int* ngroups;
    int* pairs;
    int* npairs;
    int* rounds;
    unsigned char* mask;
    // per-env episode state (risvec_pair_noma_episodes); null = the scalar recalc / fresh / topk / tau_q above
    const unsigned char* start;  // [E] != 0: first step of the env's episode (recalc_mask = new_episode = 1)
    const int* ep_index;         // [E] i_episode: K_now / q_now of the mask curriculum, computed per env
    int sched_topk_start, sched_topk_end, sched_warmup;
    double sched_tau_q_start, sched_tau_q_end;
};

// batched.mask_schedule (`_anneal_topk` marl_train_bcd.py:128-132 and :1323-1332) for one env: python's round is
// half-to-even (rint), and the explicit round-to-nearest intrinsics keep every operation as python evaluates it
__device__ __forceinline__ void mask_schedule_dev(const PairArgs& a, int N, int ep, int* K, double* q) {
    const int k_start = a.sched_topk_start < 0 ? N - 1 : a.sched_topk_start;
    const int k_end = a.sched_topk_end < 0 ? max(4, N / 2) : a.sched_topk_end;
    const int warm = a.sched_warmup;
    const double w = (double)max(1, warm);
    const int i = max(0, min(ep, warm));
    const double kf = __dadd_rn((double)k_end, __dmul_rn((double)(k_start - k_end), __dsub_rn(1.0, __ddiv_rn((double)i, w))));
    const int k = (int)rint(kf);
    const double prog = fmin(1.0, __ddiv_rn((double)ep, w));
    *K = min(max(k, 1), N - 1);
    *q = __dadd_rn(a.sched_tau_q_start, __dmul_rn(__dsub_rn(a.sched_tau_q_end, a.sched_tau_q_start), prog));
}

__host__ __device__ inline size_t pair_smem_bytes(int N) {
    const size_t NN = (size_t)N * N, NS = (size_t)1 << N;
    size_t b = 8 * (4 * (size_t)N + 2 * NN + NS + 2);   // gl, pw, g15, g12 | S, W | dp | slot
    b += 4 * (NN + (size_t)N + 2);                      // Hs (f32) | pr (int)
    b += NS + 4 * NN + (size_t)N;                       // ch | feas, qos, tmp, valid | wk
    return (b + 15) / 16 * 16;
}

template <int N>
struct PairCtx {
    static constexpr int NN = N * N, NS = 1 << N;
    int lane;
    double *gl, *pw, *g15, *g12, *S, *W, *dp, *slot;
    float* Hs;
    int* pr;
    signed char* ch;
    unsigned char *feas, *qos, *tmp, *valid, *wk;

    __device__ void carve(unsigned char* base, int ln) {
        lane = ln;
        s_ranked = false;
        rn = 0;
        gl = (double*)base; pw = gl + N; g15 = pw + N; g12 = g15 + N;
        S = g12 + N; W = S + NN; dp = W + NN; slot = dp + NS;
        Hs = (float*)(slot + 2);
        pr = (int*)(Hs + NN);
        ch = (signed char*)(pr + N + 2);
        feas = (unsigned char*)(ch + NS); qos = feas + NN; tmp = qos + NN; valid = tmp + NN; wk = valid + NN;
    }

    static __device__ __forceinline__ int wsum(int v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
        return v;
    }

    // Order statistics by counting.  rank_pass: every lane keeps its ceil(N^2 / 32) entries of `vals`
    // in registers and counts, over one broadcast pass of the array, how many values are smaller
    // (rl) and how many are equal (re): an entry is the k-th order statistic iff rl <= k < rl + re.
    // `vals` must hold +inf wherever `valid` is 0.  The counts stay valid until the array changes,
    // so several quantiles of the same values (the matching's accept threshold and the
    // completion's threshold, :346 and :300) cost one pass.
    static constexpr int EPL = (NN + 31) / 32;
    double rv[EPL];
    int rl[EPL], re[EPL], rn;

    // `flag[e]` marks the valid entries (zero for e >= len, where vals holds +inf); `mul` is the
    // multiplicity of every stored value (2 when only the upper triangle of a symmetric matrix is stored)
    const unsigned char* rflag;
    int rmul;
    __device__ void rank_pass(const double* vals, int len, const unsigned char* flag, int mul) {
        rflag = flag;
        rmul = mul;
        int c = 0;
        for (int e = lane; e < NN; e += 32) c += flag[e] ? 1 : 0;
        rn = wsum(c) * mul;
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
            const int e = lane + 32 * k;
            rv[k] = e < NN ? vals[e] : CUDART_INF;
            rl[k] = 0;
            re[k] = 0;
        }
        if (rn == 0) return;
#pragma unroll 8
        for (int o = 0; o < len; ++o) {
            const double u = vals[o];
#pragma unroll
            for (int k = 0; k < EPL; ++k) {
                rl[k] += u < rv[k];
                re[k] += u == rv[k];
            }
        }
#pragma unroll
        for (int k = 0; k < EPL; ++k) { rl[k] *= mul; re[k] *= mul; }
    }

    // numpy.quantile(values of the last rank_pass, q, method="linear") incl. numpy's two-sided _lerp
    __device__ double select(double q) {
        const int n = rn;
        if (n == 0) return 0.0;
        const double vi = __dmul_rn((double)(n - 1), q);
        int lo, hi;
        double t = 0.0;
        if (vi >= (double)(n - 1)) lo = hi = n - 1;
        else if (vi < 0.0) lo = hi = 0;
        else { const double f = floor(vi); lo = (int)f; hi = lo + 1; t = __dsub_rn(vi, f); }
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
            const int e = lane + 32 * k;
            if (e < NN && rflag[e]) {   // equal values may be published by several lanes: same bits
                if (rl[k] <= lo && lo < rl[k] + re[k]) slot[0] = rv[k];
                if (rl[k] <= hi && hi < rl[k] + re[k]) slot[1] = rv[k];
            }
        }
        __syncwarp();
        const double a = slot[0], b = slot[1];
        __syncwarp();
        const double dlt = __dsub_rn(b, a);
        double res = __dadd_rn(a, __dmul_rn(dlt, t));
        if (t >= 0.5) res = __dsub_rn(b, __dmul_rn(dlt, __dsub_rn(1.0, t)));
        return res;
    }

    // _adaptive_threshold_from_delta_g (:842-855): quantile of |g_s - g_w| over strong x weak (the
    // halves of the stable gain order); the nS * nW differences are stored compactly so that the
    // counting pass runs over them only
    __device__ double adaptive_tau(double q) {
        if constexpr (N < 2) {
            return 0.0;
        } else {
        if (lane < N) {
            int r = 0;
            const double v = g15[lane];
            for (int o = 0; o < N; ++o) r += (g15[o] < v || (g15[o] == v && o < lane)) ? 1 : 0;
            pr[r] = lane;       // pr is free here: vehicle at each rank
        }
        __syncwarp();
        constexpr int nW = N / 2, nS = N - nW, n = nS * nW;
        for (int e = lane; e < NN; e += 32) {
            const bool ok = e < n;
            valid[e] = ok;
            W[e] = ok ? fabs(__dsub_rn(g15[pr[nW + e / nW]], g15[pr[e % nW]])) : CUDART_INF;
        }
        __syncwarp();
        rank_pass(W, n, valid, 1);
        s_ranked = false;
        const double tau = rn ? select(q) : 0.0;
        __syncwarp();
        return tau;
        }
    }

    // _build_feasible_mask_from_delta_g (:134-156) -> feas
    __device__ void build_mask(double tau, int K) {
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            tmp[e] = (i != j) && !(fabs(__dsub_rn(g15[i], g15[j])) < tau);
        }
        __syncwarp();
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            unsigned char keep = tmp[e];
            if (keep) {
                const double dme = fabs(__dsub_rn(g15[i], g15[j]));
                int cnt = 0, r = 0;
                for (int o = 0; o < N; ++o) {
                    if (!tmp[i * N + o]) continue;
                    ++cnt;
                    const double du = fabs(__dsub_rn(g15[i], g15[o]));
                    r += (du > dme || (du == dme && o < j)) ? 1 : 0;
                }
                if (cnt > K && r >= K) keep = 0;
            }
            qos[e] = keep;      // scratch (the QoS mask is built later)
        }
        __syncwarp();
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            feas[e] = qos[e] & qos[j * N + i];
        }
        __syncwarp();
    }

    // call-site loop :1428-1440 over _qos_pair_feasible (:858-881) -> qos
    __device__ void build_qos(const PairArgs& a) {
        const double nz = __dadd_rn(a.noise, 1e-12);
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            unsigned char ok = 0;
            if (i != j) {
                const double pi = __dmul_rn(pw[i], a.P_max), pj = __dmul_rn(pw[j], a.P_max);
                const double gi = gl[i], gj = gl[j];
                double g_near, g_far, p_near, p_far;
                if (gi >= gj) { g_near = gi; g_far = gj; p_near = pi; p_far = pj; }
                else { g_near = gj; g_far = gi; p_near = pj; p_far = pi; }
                const double den = __dadd_rn(__dadd_rn(__dmul_rn(p_near, g_far), a.noise), 1e-12);
                const double sf = __ddiv_rn(__dmul_rn(p_far, g_far), den);
                const double sn = __ddiv_rn(__dmul_rn(p_near, g_near), nz);
                // log2(1 + max(0, sinr)) >= R_min  <=>  max(0, sinr) >= a.sinr_min, the smallest double
                // for which the host libm evaluates the left side true (log2(1 + x) is monotone)
                ok = (fmax(0.0, sf) >= a.sinr_min) && (fmax(0.0, sn) >= a.sinr_min);
            }
            qos[e] = ok;
        }
        __syncwarp();
    }

    // _score_matrix_from_gain_and_history (:164-194) -> S
    __device__ void score(const PairArgs& a) {
        const double ninf = -CUDART_INF;
        s_ranked = false;
        bool any = false;
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            const double d12 = fabs(__dsub_rn(g12[i], g12[j]));
            const bool ok = (g12[i] >= a.abs_min_db) || (g12[j] >= a.abs_min_db);
            S[e] = __dadd_rn(__dmul_rn(a.w_delta, d12), (double)__fmul_rn(a.w_hist, Hs[e]));
            tmp[e] = ok;
            any |= (feas[e] > 0) && ok;
        }
        any = __any_sync(kFull, any);
        __syncwarp();
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            const bool keep = (feas[e] > 0) && (any ? (tmp[e] != 0) : true);
            double v = keep ? S[e] : ninf;
            if (a.qos_enable && qos[e] == 0 && isfinite(v)) v = __dsub_rn(v, a.qos_pen);
            if (i == j) v = ninf;
            S[e] = v;
        }
        __syncwarp();
    }

    // _relax_mask_once (:260-275): feas |= (delta >= tau_db, off-diagonal) | row top-k by delta
    __device__ void relax(double tau_db, int topk) {
        const int k = min(topk, N - 1);
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            const double dme = fabs(__dsub_rn(g12[i], g12[j]));
            bool on = feas[e] > 0 || ((dme >= tau_db) && i != j);
            if (!on && topk >= 1) {
                int r = 0;
                for (int o = 0; o < N; ++o) {
                    const double du = fabs(__dsub_rn(g12[i], g12[o]));
                    r += (du > dme || (du == dme && o < j)) ? 1 : 0;
                }
                on = r < k;
            }
            tmp[e] = on;
        }
        __syncwarp();
        for (int e = lane; e < NN; e += 32) feas[e] = tmp[e];
        __syncwarp();
    }

    // ranks of the finite entries of S (edges); cached until `score` rewrites S
    bool s_ranked;
    __device__ void rank_edges() {
        if (s_ranked) return;
        bool sym = true;
        for (int e = lane; e < NN; e += 32) {
            const int i = e / N, j = e - i * N;
            const bool ok = isfinite(S[e]);
            valid[e] = ok;
            sym = sym && (S[e] == S[j * N + i]);          // -inf == -inf; S holds no NaN
        }
        sym = __all_sync(kFull, sym);
        __syncwarp();
        if (sym && N >= 2) {
            // symmetric scores (always, unless a back-off round or an exact gain tie broke it): every
            // value occurs twice, so the counting pass runs over the N (N - 1) / 2 upper-triangle values
            constexpr int NT = N * (N - 1) / 2;
            for (int e = lane; e < NN; e += 32) { tmp[e] = 0; W[e] = CUDART_INF; }
            __syncwarp();
            for (int e = lane; e < NN; e += 32) {
                const int i = e / N, j = e - i * N;
                if (i < j) {
                    const int t = i * N - (i * (i + 1)) / 2 + (j - i - 1);
                    tmp[t] = valid[e];
                    W[t] = valid[e] ? S[e] : CUDART_INF;
                }
            }
            __syncwarp();
            rank_pass(W, NT, tmp, 2);
        } else {
            for (int e = lane; e < NN; e += 32) W[e] = valid[e] ? S[e] : CUDART_INF;   // the layout rank_pass wants
            __syncwarp();
            rank_pass(W, NN, valid, 1);
        }
        __syncwarp();
        s_ranked = true;
    }

    // _mwm_primary (:326-398), allow_singles = True.  Returns the number of pairs written to pr.
    // dp(mask) always expands the lowest unused vehicle i, so the table is filled by "lowest unset
    // bit" levels i = N-1 .. 0: level i holds the 2^(N-1-i) masks (ones below i, zero at i, any bits
    // above) and depends only on levels > i.  Values and option order (single first, then j
    // ascending, strict >) are those of the reference's memoised recursion.  A non-edge carries
    // W = -inf, and -inf + dp never beats the single option, which is the reference's `continue`.
    __device__ int mwm_primary(double accept_q) {
        const double ninf = -CUDART_INF;
        rank_edges();
        if (rn == 0) return 0;
        const double q = fmin(fmax(accept_q, 0.0), 1.0);
        const double thr = select(__dsub_rn(1.0, q));
        for (int e = lane; e < NN; e += 32) W[e] = (valid[e] && S[e] >= thr) ? S[e] : ninf;
        constexpr int full = NS - 1;
        if (lane == 0) { dp[full] = 0.0; ch[full] = -1; }
#pragma unroll
        for (int i = N - 1; i >= 0; --i) {
            __syncwarp();
            const int low = (1 << i) - 1, cnt = 1 << (N - 1 - i);
            for (int k = lane; k < cnt; k += 32) {
                const int m = low | (k << (i + 1));
                const int mi = m | (1 << i);
                double bw = dp[mi];             // option 1: i stays single (always finite)
                int c = -1;
#pragma unroll
                for (int j = i + 1; j < N; ++j) {
                    const double sum = __dadd_rn(W[i * N + j], dp[mi | (1 << j)]);
                    if (!(m >> j & 1) && sum > bw) { bw = sum; c = j; }
                }
                dp[m] = bw;
                ch[m] = (signed char)c;
            }
        }
        __syncwarp();
        int np = 0;
        if (lane == 0) {
            int m = 0;
            while (m != full) {
                const int i = __ffs(~m) - 1;
                const int c = ch[m];
                if (c >= 0) { pr[2 * np] = i; pr[2 * np + 1] = c; ++np; m |= (1 << i) | (1 << c); }
                else m |= 1 << i;
            }
        }
        np = __shfl_sync(kFull, np, 0);
        __syncwarp();
        return np;
    }

    // _mwm_completion (:276-324): greedy top-up, candidates ordered by (S, i, j) descending
    __device__ int completion(int np, int min_pairs, double cq) {
        rank_edges();
        if (rn == 0) return np;
        const double thr = select(cq);
        unsigned occ = 0;
        for (int k = 0; k < 2 * np; ++k) occ |= 1u << pr[k];
        while (np < min_pairs) {
            double bv = -CUDART_INF;
            int be = -1;
            for (int e = lane; e < NN; e += 32) {
                const int i = e / N, j = e - i * N;
                if (i >= j || !valid[e] || !(S[e] >= thr)) continue;
                if ((occ >> i & 1u) || (occ >> j & 1u)) continue;
                if (be < 0 || S[e] > bv || (S[e] == bv && e > be)) { bv = S[e]; be = e; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(kFull, bv, o);
                const int oe = __shfl_xor_sync(kFull, be, o);
                if (oe >= 0 && (be < 0 || ov > bv || (ov == bv && oe > be))) { bv = ov; be = oe; }
            }
            if (be < 0) break;
            const int i = be / N, j = be - i * N;
            if (lane == 0) { pr[2 * np] = i; pr[2 * np + 1] = j; }
            occ |= (1u << i) | (1u << j);
            ++np;
        }
        __syncwarp();
        return np;
    }
};

template <int N>
__global__ void k_pair_noma(Dims d, State s, PairArgs a) {
    extern __shared__ __align__(16) unsigned char pair_smem[];
    constexpr int NN = N * N;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const long long e = (long long)blockIdx.x * wpc + wib;
    if (e >= d.E) return;    // whole warps leave together; only __syncwarp is used below
    PairCtx<N> c;
    c.carve(pair_smem + pair_smem_bytes(N) * wib, lane);
    int recalc = a.recalc, fresh = a.fresh, topk = a.topk;
    double tau_q = a.tau_q;
    if (a.start != nullptr) {                                 // per-env episode state
        recalc = fresh = a.start[e] != 0;
        if (recalc) mask_schedule_dev(a, N, a.ep_index[e], &topk, &tau_q);
    }

    float* H = a.hist + e * NN;
    for (int x = lane; x < NN; x += 32) {
        const float h = fresh ? 0.f : H[x];
        c.Hs[x] = a.decay ? __fmul_rn(h, a.decay_f) : h;     // :1406 (float32 array *= python float)
    }
    if (lane < N) {
        const double g = s.gains[e * N + lane];
        c.gl[lane] = g;
        c.pw[lane] = (double)a.p01[e * a.p01_stride + lane];
        c.g15[lane] = __dmul_rn(10.0, log10(fmax(g, 1e-15)));
        c.g12[lane] = __dmul_rn(10.0, log10(fmax(g, 1e-12)));
    }
    __syncwarp();

    double tau;
    int K;
    if (recalc) {                                             // :1319-1343
        tau = c.adaptive_tau(tau_q);
        K = topk;
        c.build_mask(tau, K);
        for (int x = lane; x < NN; x += 32) a.mask[e * NN + x] = c.feas[x];
        if (lane == 0) { a.tau[e] = tau; a.lastk[e] = K; }
    } else {                                                  // :1421-1424 (mask_mat is None on these steps)
        tau = a.tau[e];
        K = a.lastk[e];
        for (int x = lane; x < NN; x += 32) { const int i = x / N; c.feas[x] = (x - i * N) != i; }
        __syncwarp();
    }

    int np = 0, rounds = 0;
    const bool frozen = !fresh && a.reuse != nullptr && a.reuse[e] != 0 && a.ngroups[e] > 0;
    if (frozen) {                                             // :1542-1547
        np = a.npairs[e];
        if (lane < 2 * np) c.pr[lane] = a.pairs[e * N + lane];
        __syncwarp();
    } else {
        if (a.qos_enable) c.build_qos(a);
        c.score(a);                                           // :1441-1450
        double accept_q = a.accept_q;
        np = c.mwm_primary(accept_q);                         // :1456-1461
        if (np < a.min_pairs) np = c.completion(np, a.min_pairs, a.completion_q);   // :1464-1465
        int K_back = K;
        double tau_back = tau;
        while (np < a.min_pairs && rounds < a.backoff_rounds) {     // :1493-1524
            ++rounds;
            K_back = min(N - 1, K_back + a.relax_topk_step);
            tau_back = fmax(a.tau_floor, __dmul_rn(tau_back, a.relax_tau_factor));
            c.relax(tau_back, K_back);
            c.score(a);
            accept_q = fmax(0.05, __dsub_rn(accept_q, a.accept_q_step));
            np = c.mwm_primary(accept_q);
            if (np < a.min_pairs) np = c.completion(np, a.min_pairs, a.completion_q);
        }
        __syncwarp();
        // groups = pairs + singles (:1550-1553) in the partner / ngroups encoding of the rollout
        unsigned used = 0;
        for (int k = 0; k < 2 * np; ++k) used |= 1u << c.pr[k];
        if (lane < N) {
            int p = RISVEC_PARTNER_SINGLE;
            for (int k = 0; k < np; ++k) {
                if (c.pr[2 * k] == lane) p = c.pr[2 * k + 1];
                if (c.pr[2 * k + 1] == lane) p = c.pr[2 * k] | RISVEC_PARTNER_SECOND;
            }
            a.partner[e * N + lane] = p;
        }
        if (lane < N) a.pairs[e * N + lane] = lane < 2 * np ? c.pr[lane] : -1;
        if (lane == 0) {
            a.npairs[e] = np;
            a.ngroups[e] = np + (N - __popc(used));
        }
    }
    if (lane == 0) a.rounds[e] = rounds;

    // history / streak updates (:1556-1561)
    unsigned used = 0;
    for (int k = 0; k < 2 * np; ++k) used |= 1u << c.pr[k];
    if (lane < np) {
        const int i = c.pr[2 * lane], j = c.pr[2 * lane + 1];
        c.Hs[i * N + j] = __fadd_rn(c.Hs[i * N + j], 1.0f);
        c.Hs[j * N + i] = __fadd_rn(c.Hs[j * N + i], 1.0f);
    }
    __syncwarp();
    for (int x = lane; x < NN; x += 32) H[x] = c.Hs[x];
    if (lane < N) {
        int* sk = a.streak + e * N + lane;
        *sk = (used >> lane & 1u) ? 0 : (fresh ? 0 : *sk) + 1;
    }
}

// new episode (:1282-1297) of env e by the threads x0, x0 + step, ... (x0 < step): history, streak, thresholds and
// frozen groups cleared.  The fused episode start (episode.cuh) runs it with the env's 8 lanes.
__device__ __forceinline__ void pair_reset_env(const PairArgs& a, int N, long long e, int x0, int step) {
    const int NN = N * N;
    for (int x = x0; x < NN; x += step) {
        a.hist[e * NN + x] = 0.f;
        a.mask[e * NN + x] = 0;
    }
    for (int x = x0; x < N; x += step) {
        a.streak[e * N + x] = 0;
        a.partner[e * N + x] = RISVEC_PARTNER_NONE;
        a.pairs[e * N + x] = -1;
    }
    if (x0 == 0) { a.tau[e] = 0.0; a.lastk[e] = 0; a.ngroups[e] = 0; a.npairs[e] = 0; a.rounds[e] = 0; }
}

__global__ void k_pair_reset(Dims d, PairArgs a, const unsigned char* __restrict__ env_mask, EnvGate g) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int N = d.V, NN = N * N;
    if (t >= (long long)d.E * NN) return;
    auto on = [&](long long e) { return (env_mask == nullptr || env_mask[e] != 0) && g.on(e); };  // per-env reset
    if (on(t / NN)) {
        a.hist[t] = 0.f;
        a.mask[t] = 0;
    }
    if (t < (long long)d.E * N && on(t / N)) { a.streak[t] = 0; a.partner[t] = RISVEC_PARTNER_NONE; a.pairs[t] = -1; }
    if (t < d.E && on(t)) { a.tau[t] = 0.0; a.lastk[t] = 0; a.ngroups[t] = 0; a.npairs[t] = 0; a.rounds[t] = 0; }
}

}  // namespace risvec
