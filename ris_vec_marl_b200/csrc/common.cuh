// Shared device-side definitions for the risvec kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/risvec.h"

namespace risvec {

// Module constants of the reference (Simulation-MARL-BCD/Environment.py:29-42).
constexpr double kRisX = 220.0, kRisY = 220.0, kRisZ = 25.0;
constexpr double kBsX = 0.0, kBsY = 0.0, kBsZ = 25.0;
constexpr double kVehZ = 1.5;
constexpr double kRo = 1e-2;
constexpr double kSigma = 1e-7;
constexpr double kAlpha1 = 2.2, kAlpha2 = 2.5;

constexpr unsigned kFull = 0xffffffffu;

// Problem dimensions + RNG keys, passed by value to every kernel.
struct Dims {
    int E, V, M, ncand, variant;
    unsigned long long seed;
    long long env_base;
    double dist_BR, angle_BR;
};

// Pointers into the state arena (layout: include/risvec.h, enum risvec_field).
struct State {
    double *pos_x, *pos_y, *dist, *angle, *amp, *theta_re, *theta_im, *gains, *databuf, *mecq;
    int *dir, *vel, *data_r;
    float *phase_real, *data_t, *data_p, *over_data, *over_power, *rate, *reward_user, *reward, *stats, *last_power;
    long long* step_ctr;
};

// ---------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator (Salmon et al., SC'11), keyed by (seed) and indexed
// by (global env index, per-call counter, slot, stream kind): draws do not depend on how
// envs are sharded over GPUs or on launch geometry.
// ---------------------------------------------------------------------------------------
// kinds 5-7: the draws of risvec_episode_tick, keyed by the env's episode index instead of a host call counter
enum RngKind : unsigned {
    kRngReset = 1, kRngMobility = 2, kRngArrival = 3, kRngChannel = 4,
    kRngEpReset = 5, kRngEpMobility = 6, kRngEpChannel = 7
};

// Per-env selection of the episode-start kernels (risvec_begin_episode / risvec_episode_tick on the shapes the
// fused kernel does not take).  Zero-initialised = every env, host-keyed draws: exactly the plain entry points.
struct EnvGate {
    const unsigned char* bits;  // [E] per-env RISVEC_EP_* bits, or null (every env runs this launch)
    unsigned bit;               // the stage this launch runs
    const int* call;            // [E] per-env RNG call = episode index (device-keyed draws), or null (host counter)
    __device__ bool on(long long e) const { return bits == nullptr || (bits[e] & bit) != 0; }
    __device__ unsigned long long key(long long e, unsigned long long host_call) const {
        return call != nullptr ? (unsigned long long)(unsigned)call[e] : host_call;
    }
    __device__ unsigned kind(unsigned host_kind, unsigned device_kind) const {
        return call != nullptr ? device_kind : host_kind;
    }
};

__host__ __device__ inline uint4 philox4x32_10(uint4 c, uint2 k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c.x, p1 = (uint64_t)M1 * c.z;
        uint4 n;
        n.x = (uint32_t)(p1 >> 32) ^ c.y ^ k.x;
        n.y = (uint32_t)p1;
        n.z = (uint32_t)(p0 >> 32) ^ c.w ^ k.y;
        n.w = (uint32_t)p0;
        c = n;
        k.x += W0;
        k.y += W1;
    }
    return c;
}

__device__ inline uint4 rng_draw(const Dims& d, long long env_local, unsigned long long call, unsigned slot,
                                 unsigned kind) {
    unsigned long long ge = (unsigned long long)(d.env_base + env_local);
    uint4 c;
    c.x = (uint32_t)ge;
    c.y = (uint32_t)(ge >> 32) ^ (kind << 28);
    c.z = (uint32_t)call;
    c.w = (uint32_t)(call >> 32) ^ (slot << 4);
    uint2 k = make_uint2((uint32_t)d.seed, (uint32_t)(d.seed >> 32));
    return philox4x32_10(c, k);
}

__device__ inline float u01f(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-8f; }  // [0,1)
__device__ inline double u01d(uint32_t hi, uint32_t lo) {
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);
}

// Poisson(lam) by sequential inversion; lam is small in every reference configuration
// (rate = 1 or 3, MARL/config.yaml:140, Environment.py:156).
__device__ inline int poisson_inv(float lam, float u) {
    if (!(lam > 0.f)) return 0;
    float p = __expf(-lam), s = p;
    int k = 0;
    const int kmax = (int)(lam + 12.f * sqrtf(lam) + 16.f);
    while (u > s && k < kmax) {
        ++k;
        p *= lam / (float)k;
        s += p;
    }
    return k;
}

// segmented (width = W lanes) butterfly sum; every lane of the segment gets the total
template <int W, typename T>
__device__ inline T seg_sum(T x) {
#pragma unroll
    for (int o = 1; o < W; o <<= 1) x += __shfl_xor_sync(kFull, x, o);
    return x;
}

// z = exp(j*pi*delta) evaluated ONCE per vehicle (sincospi) and raised by float64 complex
// multiplications (each ~1e-16 relative), instead of one sincospi per table entry.
__device__ __noinline__ double2 unit_phasor64(double delta) {
    double s64, c64;
    sincospi(delta, &s64, &c64);
    return make_double2(c64, s64);
}
__device__ __forceinline__ double2 cmul64(double2 a, double2 b) {
    return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ double2 cpow64(double2 z, unsigned n) {  // z^n by squaring
    double2 r = make_double2(1.0, 0.0);
    while (n) {
        if (n & 1u) r = cmul64(r, z);
        z = cmul64(z, z);
        n >>= 1;
    }
    return r;
}

}  // namespace risvec
