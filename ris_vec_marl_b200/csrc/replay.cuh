// Device-resident replay memory of the MARL driver (Simulation-MARL-BCD/buffer.py:3-39) and the
// transition assembly the driver does before `store_transition` (marl_train_bcd.py:1776-1799),
// batched: E envs store E transitions per step into consecutive ring slots.  Pure copies, one block
// per transition row, every segment written coalesced.
#pragma once
#include "common.cuh"

namespace risvec {

struct ReplayMem {
    long long mem_size;
    int S, A, N;     // input_shape * n_agents, n_actions * n_agents, n_agents
    float *state, *action, *reward_g, *reward_l, *state_, *mask;
    unsigned char* terminal;
};

// Sources of one store call.  MARL = 0: `action` / `mask_f` are the assembled rows of buffer.py:16;
// MARL = 1: the driver's pieces (marl_train_bcd.py:1776-1790): action row = per agent [intent probs
// (N, diagonal zeroed at :1390) | raw power (2)], mask row = float32 of the u8 feasibility mask.
// A NULL mask stores all ones (the driver's choice when the step built no mask, :1786-1789).
struct ReplaySrc {
    const float *state, *state_, *action, *probs, *power, *reward_g, *reward_l, *mask_f;
    const unsigned char *mask_u8, *done;
    int done_all;
};

// Ring counter of a handle in device-counter mode (risvec_replay_use_device_counter): `count` is mem_cntr, `ticket`
// counts the blocks of the running store that are done reading it.  Both live in the replay arena.
struct ReplayCtr {
    long long* count;
    unsigned* ticket;
};

// DEVCNT stores: thread 0 of each block reads the count, then takes a ticket (__threadfence, then atomicAdd) before
// the block writes anything.  The block that draws the last ticket knows every block of the launch has read the count,
// so it advances the count by E and resets the ticket for the next store.  One launch, nothing for the host to reset
// between replays.  Claiming at the start keeps the fence away from the block's stores: a fence after them would wait
// for them to drain and hold the block's slot on the SM.
__device__ __forceinline__ long long devcnt_claim(const ReplayCtr& c, int E) {
    __shared__ long long s_count;
    if (threadIdx.x == 0) {
        const long long count = max(*(volatile long long*)c.count, 0LL);   // a negative count is taken as 0
        s_count = count;
        __threadfence();
        if (atomicAdd(c.ticket, 1u) == gridDim.x * gridDim.y - 1) {
            *(volatile long long*)c.count = count + E;
            *(volatile unsigned*)c.ticket = 0;
        }
    }
    __syncthreads();
    return s_count;
}

template <int VEC>
struct RVec;
template <>
struct RVec<1> { using T = float; };
template <>
struct RVec<4> { using T = float4; };

// Flat copy: the E rows of a call land in consecutive ring slots, so every field is one (at most
// once wrapped) contiguous destination range.  A thread moves VEC consecutive floats of one field
// of one row; VEC = 4 needs every row width to be a multiple of 4 (true at V = 8: 40, 80, 8, 64).
// DEVCNT = 1: `first` is ignored, the block reads it from `ctr` (see devcnt_claim).
template <int VEC, int MARL, int DEVCNT>
__global__ void k_replay_store(ReplayMem m, long long first, int E, ReplaySrc src, ReplayCtr ctr) {
    using V4 = typename RVec<VEC>::T;
    if constexpr (DEVCNT) first = devcnt_claim(ctr, E);
    const int N = m.N, NN = N * N, AW = N + 2;
    const long long uS = (long long)E * (m.S / VEC), uA = (long long)E * (m.A / VEC), uN = (long long)E * (N / VEC),
                    uM = (long long)E * (NN / VEC);
    const long long total = 2 * uS + uA + uN + uM + E;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        long long u = t;
        if (u < 2 * uS) {                                   // state, new_state
            const bool second = u >= uS;
            if (second) u -= uS;
            const int w = m.S / VEC;
            const long long e = u / w;
            const int c = (int)(u - e * w);
            const long long slot = (first + e) % m.mem_size;
            const V4 v = ((const V4*)((second ? src.state_ : src.state) + e * m.S))[c];
            ((V4*)((second ? m.state_ : m.state) + slot * m.S))[c] = v;
            continue;
        }
        u -= 2 * uS;
        if (u < uA) {                                       // action
            const int w = m.A / VEC;
            const long long e = u / w;
            const int c = (int)(u - e * w);
            const long long slot = (first + e) % m.mem_size;
            float o[VEC];
            if (MARL) {
#pragma unroll
                for (int x = 0; x < VEC; ++x) {
                    const int col = c * VEC + x, i = col / AW, k = col - i * AW;
                    o[x] = k < N ? (k == i ? 0.f : src.probs[(e * N + i) * N + k]) : src.power[(e * N + i) * 2 + (k - N)];
                }
            } else {
                const V4 v = ((const V4*)(src.action + e * m.A))[c];
                memcpy(o, &v, sizeof(v));
            }
            V4 v;
            memcpy(&v, o, sizeof(v));
            ((V4*)(m.action + slot * m.A))[c] = v;
            continue;
        }
        u -= uA;
        if (u < uN) {                                       // reward_local
            const int w = N / VEC;
            const long long e = u / w;
            const int c = (int)(u - e * w);
            const long long slot = (first + e) % m.mem_size;
            ((V4*)(m.reward_l + slot * N))[c] = ((const V4*)(src.reward_l + e * N))[c];
            continue;
        }
        u -= uN;
        if (u < uM) {                                       // mask
            const int w = NN / VEC;
            const long long e = u / w;
            const int c = (int)(u - e * w);
            const long long slot = (first + e) % m.mem_size;
            float o[VEC];
#pragma unroll
            for (int x = 0; x < VEC; ++x) {
                const long long at = e * NN + c * VEC + x;
                o[x] = MARL ? (src.mask_u8 ? (float)src.mask_u8[at] : 1.f) : (src.mask_f ? src.mask_f[at] : 1.f);
            }
            V4 v;
            memcpy(&v, o, sizeof(v));
            ((V4*)(m.mask + slot * NN))[c] = v;
            continue;
        }
        u -= uM;                                            // reward_global, terminal
        const long long slot = (first + u) % m.mem_size;
        m.reward_g[slot] = src.reward_g[u];
        m.terminal[slot] = src.done ? (src.done[u] != 0) : (src.done_all != 0);
    }
}

// float4 form of the same store without per-element row arithmetic: blockIdx.y selects the field; because
// the E rows land in consecutive ring slots, every field is a FLAT copy of E * width floats whose
// destination is contiguous up to one wrap of the ring (n_wrap = rows before the wrap).  Only the assembled
// MARL action rows need a row index (one 32-bit division per 16 bytes).  DEVCNT = 1: `slot0` / `n_wrap` are ignored,
// the block computes them from the count it reads from `ctr`.
template <int MARL, int DEVCNT>
__global__ void __launch_bounds__(256) k_replay_store_flat(ReplayMem m, long long slot0, int n_wrap, int E, ReplaySrc src,
                                                           ReplayCtr ctr) {
    if constexpr (DEVCNT) {
        slot0 = devcnt_claim(ctr, E) % m.mem_size;
        n_wrap = (int)(m.mem_size - slot0 < E ? m.mem_size - slot0 : E);
    }
    const int N = m.N, NN = N * N, AW = N + 2;
    const unsigned tid = blockIdx.x * blockDim.x + threadIdx.x, nthr = gridDim.x * blockDim.x;
    auto flat_copy = [&](float* dst_field, const float* src_field, int W) {  // W floats per row, W % 4 == 0
        const unsigned n4 = (unsigned)E * (W / 4), w4 = (unsigned)n_wrap * (W / 4);
        float4* d0 = reinterpret_cast<float4*>(dst_field + slot0 * W);
        float4* d1 = reinterpret_cast<float4*>(dst_field);
        const float4* sp = reinterpret_cast<const float4*>(src_field);
        for (unsigned i = tid; i < n4; i += nthr) {
            const float4 v = __ldg(sp + i);
            if (i < w4) d0[i] = v;
            else d1[i - w4] = v;
        }
    };
    switch (blockIdx.y) {
        case 0: flat_copy(m.state, src.state, m.S); break;
        case 1: flat_copy(m.state_, src.state_, m.S); break;
        case 2: flat_copy(m.reward_l, src.reward_l, N); break;
        case 3: {
            if (!MARL) { flat_copy(m.action, src.action, m.A); break; }
            const unsigned rw = m.A / 4, n4 = (unsigned)E * rw, w4 = (unsigned)n_wrap * rw;
            float4* d0 = reinterpret_cast<float4*>(m.action + slot0 * m.A);
            float4* d1 = reinterpret_cast<float4*>(m.action);
            for (unsigned i = tid; i < n4; i += nthr) {
                const unsigned e = i / rw, c = i - e * rw;
                float o[4];
#pragma unroll
                for (int x = 0; x < 4; ++x) {  // row = per agent [intent probs (N, diagonal zeroed) | raw power (2)]
                    const int col = (int)c * 4 + x, a = col / AW, k = col - a * AW;
                    o[x] = k < N ? (k == a ? 0.f : __ldg(src.probs + ((size_t)e * N + a) * N + k))
                                 : __ldg(src.power + ((size_t)e * N + a) * 2 + (k - N));
                }
                const float4 v = make_float4(o[0], o[1], o[2], o[3]);
                if (i < w4) d0[i] = v;
                else d1[i - w4] = v;
            }
            break;
        }
        case 4: {
            const unsigned n4 = (unsigned)E * (NN / 4), w4 = (unsigned)n_wrap * (NN / 4);
            float4* d0 = reinterpret_cast<float4*>(m.mask + slot0 * NN);
            float4* d1 = reinterpret_cast<float4*>(m.mask);
            const float4* sf = reinterpret_cast<const float4*>(src.mask_f);
            const uchar4* su = reinterpret_cast<const uchar4*>(src.mask_u8);
            for (unsigned i = tid; i < n4; i += nthr) {
                float4 v = make_float4(1.f, 1.f, 1.f, 1.f);  // no mask supplied: all ones (marl_train_bcd.py:1786-1789)
                if (MARL) {
                    if (su) { const uchar4 b = __ldg(su + i); v = make_float4(b.x, b.y, b.z, b.w); }
                } else if (sf) {
                    v = __ldg(sf + i);
                }
                if (i < w4) d0[i] = v;
                else d1[i - w4] = v;
            }
            break;
        }
        default:
            for (unsigned u = tid; u < (unsigned)E; u += nthr) {  // reward_global, terminal
                const long long slot = (int)u < n_wrap ? slot0 + u : (long long)u - n_wrap;
                m.reward_g[slot] = src.reward_g[u];
                m.terminal[slot] = src.done ? (src.done[u] != 0) : (src.done_all != 0);
            }
    }
}

// sample_buffer (buffer.py:27-39) for caller-drawn indices: one block per sampled row.  DEVCNT = 1: `idx` holds
// draws, row b is slot draws[b] % min(count, mem_size) (slot 0 while count == 0), read as unsigned: never outside.
template <int DEVCNT>
__global__ void k_replay_sample(ReplayMem m, int B, const long long* __restrict__ idx, float* __restrict__ states,
                                float* __restrict__ actions, float* __restrict__ rewards_g,
                                float* __restrict__ rewards_l, float* __restrict__ states_,
                                unsigned char* __restrict__ dones, float* __restrict__ masks,
                                const long long* __restrict__ count) {
    const int b = blockIdx.x;
    if (b >= B) return;
    long long slot;
    if constexpr (DEVCNT) {
        const unsigned long long n = (unsigned long long)min(max(*count, 0LL), m.mem_size);
        slot = n ? (long long)((unsigned long long)idx[b] % n) : 0;
    } else {
        slot = min(max(idx[b], 0LL), m.mem_size - 1);   // out-of-range indices are clamped, never read outside
    }
    const int NN = m.N * m.N;
    for (int c = threadIdx.x; c < m.S; c += blockDim.x) {
        states[(size_t)b * m.S + c] = m.state[slot * m.S + c];
        states_[(size_t)b * m.S + c] = m.state_[slot * m.S + c];
    }
    for (int c = threadIdx.x; c < m.A; c += blockDim.x) actions[(size_t)b * m.A + c] = m.action[slot * m.A + c];
    for (int c = threadIdx.x; c < m.N; c += blockDim.x) rewards_l[(size_t)b * m.N + c] = m.reward_l[slot * m.N + c];
    for (int c = threadIdx.x; c < NN; c += blockDim.x) masks[(size_t)b * NN + c] = m.mask[slot * NN + c];
    if (threadIdx.x == 0) {
        rewards_g[b] = m.reward_g[slot];
        dones[b] = m.terminal[slot];
    }
}

}  // namespace risvec
