// Per-env episode sums and the log of completed episodes (risvec_episode_accumulate): one launch per driver step,
// no host decision, so it can sit in a captured CUDA graph next to the episode clock and the fused step.
#pragma once
#include "common.cuh"

namespace risvec {

struct EpisodeLogArgs {
    double* running;            // [E, RISVEC_EPLOG_RUN_COLS(n_user)]
    const unsigned char* done;  // [E], or null: done_all for every env
    int done_all;
    int n_user;                 // V (MARL) or 0 (SARL)
    double* records;            // [capacity, RISVEC_EPLOG_REC_COLS(n_user)]
    long long capacity;
    unsigned long long* count;
};

// One (env, column) element per thread: a block takes kEpLogThreads / C envs (39 at V = 8, at most 56), so every
// thread issues its loads at once instead of walking several elements one memory round trip after another.
constexpr int kEpLogThreads = 1024;
constexpr int kEpLogClaim = 64;  // warps 0 and 1 claim the record slots of the block's done envs
static_assert(kEpLogThreads / RISVEC_EPLOG_RUN_COLS(0) <= kEpLogClaim, "a block's envs fit the claiming warps");

__host__ __device__ inline int episode_log_envs_per_block(int n_user) {
    return kEpLogThreads / RISVEC_EPLOG_RUN_COLS(n_user);
}

// The stats / reward_user reads and the read-modify-write of `running` walk contiguous rows.  Every element of
// `running` gets exactly one addition per call, so the sums do not depend on the mapping.  Slots are claimed with one
// atomicAdd per warp, in lane order; a slot past `capacity` is counted but not written.
__global__ void __launch_bounds__(kEpLogThreads) k_episode_accumulate(Dims d, State s, EpisodeLogArgs a) {
    __shared__ long long slot[kEpLogClaim];  // the env's record slot, or -1 when its episode goes on
    const int C = RISVEC_EPLOG_RUN_COLS(a.n_user), per = episode_log_envs_per_block(a.n_user);
    const long long e0 = (long long)blockIdx.x * per;
    const int ne = (int)min((long long)per, (long long)d.E - e0);
    if (threadIdx.x < kEpLogClaim) {
        const int t = threadIdx.x, lane = t & 31;
        const bool done = t < ne && (a.done != nullptr ? a.done[e0 + t] != 0 : a.done_all != 0);
        const unsigned m = __ballot_sync(kFull, done);
        unsigned long long base = 0;
        if (m != 0) {
            const int leader = __ffs(m) - 1;
            if (lane == leader) base = atomicAdd(a.count, (unsigned long long)__popc(m));
            base = __shfl_sync(kFull, base, leader);
        }
        slot[t] = done ? (long long)(base + __popc(m & ((1u << lane) - 1u))) : -1;
    }
    __syncthreads();
    const int i = threadIdx.x;
    if (i >= ne * C) return;
    const int el = i / C, c = i - el * C;
    const long long e = e0 + el;
    double x;
    if (c == 0) x = 1.0;
    else if (c <= RISVEC_NSTAT) x = (double)s.stats[e * RISVEC_NSTAT + (c - 1)];
    else if (c == RISVEC_NSTAT + 1) x = (double)s.reward[e];
    else x = (double)s.reward_user[e * d.V + (c - (RISVEC_NSTAT + 2))];
    double* r = a.running + e * C + c;
    const double v = *r + x;
    const long long k = slot[el];
    if (k < 0) {
        *r = v;
        return;
    }
    *r = 0.0;
    if (k < a.capacity) {
        double* rec = a.records + k * (C + 2);
        rec[2 + c] = v;
        if (c == 0) {
            rec[0] = (double)(d.env_base + e);
            rec[1] = (double)s.step_ctr[e];
        }
    }
}

}  // namespace risvec
