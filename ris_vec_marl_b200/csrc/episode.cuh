// Episode start for any subset of the envs in one launch, and the per-env episode clock that decides it on the
// device (risvec_begin_episode, risvec_episode_tick).  The stage bodies are the device functions of geom.cuh,
// ris.cuh and pairing.cuh, so every env ends bit-identical to running its stages as the separate kernels.
#pragma once
#include "common.cuh"
#include "geom.cuh"
#include "pairing.cuh"
#include "ris.cuh"

namespace risvec {

struct EpisodeArgs {
    unsigned stages;                  // begin: the call's stage set; tick: the schedule's stages
    const unsigned char* stages_env;  // begin: [E] per-env bits (AND-ed with `stages`), or null = `stages` for all
    const double* uniforms;           // begin: [E, n_uni] injected renew_positions uniforms, or null (Philox)
    int n_uni;
    int* used_out;                    // begin: [E] uniforms consumed (0 for envs that do not renew), or null
    unsigned long long reset_call, mob_call;  // begin: host call counters that key the draws
    // clock (tick)
    int* ep_step;
    int* ep_index;
    int steps_per_episode, positions_every;
    unsigned char* start_out;  // [E] or null
    unsigned char* done_out;   // [E] or null
    unsigned char* bits_out;   // k_episode_clock: [E] stage bits for the per-stage kernels
    int* key_out;              // k_episode_clock: [E] episode index before the advance (the draws' call key)
};

// One tick of env e's clock: start / done outputs, the advance, and the stages this env runs now.
// *key = the episode index the tick's draws are keyed by (the value before the advance).
__device__ __forceinline__ unsigned episode_clock(const EpisodeArgs& a, long long e, int* key) {
    const int st = a.ep_step[e], ix = a.ep_index[e];
    unsigned bits = 0;
    if (st == 0) {
        bits = a.stages;
        if (ix % a.positions_every != 0) bits &= ~(unsigned)RISVEC_EP_POSITIONS;
    }
    if (a.start_out != nullptr) a.start_out[e] = st == 0;
    if (a.done_out != nullptr) a.done_out[e] = st == a.steps_per_episode - 1;
    if (st + 1 >= a.steps_per_episode) {
        a.ep_step[e] = 0;
        a.ep_index[e] = ix + 1;
    } else {
        a.ep_step[e] = st + 1;
    }
    *key = ix;
    return bits;
}

// the clock alone, for the shapes the fused kernel does not take: one thread per env
__global__ void k_episode_clock(Dims d, EpisodeArgs a) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    int key;
    a.bits_out[e] = (unsigned char)episode_clock(a, e, &key);
    a.key_out[e] = key;
}

// Fused episode start, the mapping of k_bcd_v8 (V <= 8, ncand <= 8, M <= 256, free channel): one warp = 4 envs,
// lane = (env el, k).  Lane k = 0 runs make_new_game and renew_positions (sequential draw cursors); lanes (env, v)
// run compute_parms and keep the angle / amplitude in registers; the BCD runs on the whole warp with theta left in
// shared memory, where lanes (env, vehicle) read it for the channel gains; the pairing reset comes last.  Envs
// without CHANNEL in a warp that runs the BCD take part in its shuffles and write nothing.  CLOCK: the bits come
// from the episode clock (advanced here) and the draws are keyed by the episode index (RNG kinds 5-7).
template <bool CLOCK>
__global__ void __launch_bounds__(128) k_begin_episode(Dims d, State s, risvec_params_t p, PairArgs pa, EpisodeArgs a) {
    extern __shared__ double2 bcd_smem[];
    const int wpb = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, el = lane >> 3, k = lane & 7;
    const int e_raw = (blockIdx.x * wpb + warp) * 4 + el;
    const bool env_ok = e_raw < d.E;
    const int e = min(e_raw, d.E - 1);
    const int V = d.V, M = d.M, base = lane & ~7;
    unsigned bits = 0;
    int key = 0;
    if (k == 0 && env_ok) {
        if constexpr (CLOCK) bits = episode_clock(a, e, &key);
        else bits = (a.stages_env != nullptr ? (unsigned)a.stages_env[e] : 0xffu) & a.stages;
    }
    bits = __shfl_sync(kFull, bits, base);
    if (__all_sync(kFull, bits == 0)) {  // nothing starts in this warp
        if (!CLOCK && k == 0 && env_ok && a.used_out != nullptr) a.used_out[e] = 0;
        return;
    }
    if (k == 0 && env_ok) {
        const unsigned long long rkey = CLOCK ? (unsigned long long)(unsigned)key : a.reset_call;
        const unsigned long long mkey = CLOCK ? (unsigned long long)(unsigned)key : a.mob_call;
        if (bits & RISVEC_EP_RESET)
            make_new_game_env(d, s, p, e, nullptr, 0, nullptr, 0, rkey, CLOCK ? kRngEpReset : kRngReset);
        int used = 0;
        if (bits & RISVEC_EP_POSITIONS)
            used = renew_positions_env(d, s, p, e, CLOCK ? nullptr : a.uniforms, a.n_uni, mkey,
                                       CLOCK ? kRngEpMobility : kRngMobility);
        if (!CLOCK && a.used_out != nullptr) a.used_out[e] = used;
    }
    __syncwarp();
    // compute_parms: lane (env, v); lanes k >= V hold vehicle V - 1 (the angle k_bcd_v8 gives them) and write nothing
    const size_t ev = (size_t)e * V + min(k, V - 1);
    double angle, amp;
    if (bits & RISVEC_EP_POSITIONS) {
        const Parms r = compute_parms_of(d, s.pos_x[ev], s.pos_y[ev]);
        if (env_ok && k < V) {
            s.dist[ev] = r.dist;
            s.angle[ev] = r.angle;
            s.amp[ev] = r.amp;
        }
        angle = r.angle;
        amp = r.amp;
    } else {
        angle = s.angle[ev];
        amp = s.amp[ev];
    }
    if (__any_sync(kFull, (bits & RISVEC_EP_CHANNEL) != 0)) {
        const bool ch = env_ok && (bits & RISVEC_EP_CHANNEL) != 0;
        double2* c = bcd_smem + (size_t)(warp * 4 + el) * 2 * M;
        double2* th = c + M;
        bcd_v8_warp(d, s, e, ch, angle, c, th);
        __syncwarp();
        if (ch && k < V) s.gains[ev] = gains_free_lane(d, angle, amp, &th[0].x, &th[0].y, 2);
    }
    if (env_ok && (bits & RISVEC_EP_PAIRING)) pair_reset_env(pa, V, e, k, 8);
}

}  // namespace risvec
