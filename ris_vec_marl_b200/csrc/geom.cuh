// Reset, Manhattan-grid mobility and vehicle<->RIS geometry for E env instances.
// Reference: Simulation-MARL-BCD/Environment.py:381-410,412-542,241-253,733-737
// (Simulation-SARL/Environment.py:176-205,207-316,134-145,361-365).
#pragma once
#include "common.cuh"

namespace risvec {

// make_new_game of env e by one thread (the draws of one env are consumed sequentially); `kind` / `call` key the
// Philox draws.  Shared by k_make_new_game and the fused episode start (episode.cuh).
__device__ __forceinline__ void make_new_game_env(const Dims& d, const State& s, const risvec_params_t& p, int e,
                                                  const int* __restrict__ ints, int n_ints, const int* __restrict__ dirs,
                                                  int n_dirs, unsigned long long call, unsigned kind) {
    const int V = d.V;
    int cur = 0, curd = 0;
    auto randint = [&](int lo, int hi) -> int {
        int v;
        if (ints != nullptr) {
            v = cur < n_ints ? ints[(size_t)e * n_ints + cur] : lo;
        } else {
            uint4 r = rng_draw(d, e, call, (unsigned)cur, kind);
            v = lo + (int)__umulhi(r.x, (unsigned)(hi - lo));
        }
        ++cur;
        return v;
    };
    auto place = [&](int slot, double x, double y, int heading, int vel) {
        s.pos_x[(size_t)e * V + slot] = x;
        s.pos_y[(size_t)e * V + slot] = y;
        s.dir[(size_t)e * V + slot] = heading;
        s.vel[(size_t)e * V + slot] = vel;
    };
    int slot = 0;
    for (int r = 0; r < V / 4; ++r) {
        int ind = randint(0, p.n_down);
        // MARL:386 starts the 'd' vehicle on down_lanes[ind]; SARL:181 always on down_lanes[0]
        double xd = (d.variant == RISVEC_VARIANT_MARL) ? p.down_lanes[ind] : p.down_lanes[0];
        int y = randint(220, 230);
        place(slot++, xd, (double)y, RISVEC_DIR_DOWN, randint(10, 15));
        y = randint(170, 180);
        place(slot++, p.up_lanes[0], (double)y, RISVEC_DIR_UP, randint(10, 15));
        int x = randint(220, 230);
        place(slot++, (double)x, p.left_lanes[0], RISVEC_DIR_LEFT, randint(10, 15));
        x = randint(170, 180);
        place(slot++, (double)x, p.right_lanes[0], RISVEC_DIR_RIGHT, randint(10, 15));
    }
    for (int r = 0; r < V % 4; ++r) {  // MARL:402-407
        int ind = randint(0, p.n_down);
        int heading;
        if (dirs != nullptr) {
            heading = curd < n_dirs ? dirs[(size_t)e * n_dirs + curd] : RISVEC_DIR_DOWN;
        } else {
            uint4 q = rng_draw(d, e, call, 1024u + (unsigned)curd, kind);
            heading = (int)(q.x & 3u);
        }
        ++curd;
        int y = randint(0, (int)p.height);
        place(slot++, p.down_lanes[ind], (double)y, heading, randint(15, 20));
    }
    const int half = randint(5, p.data_buf_size - 1);  // MARL:737
    const double buf = (double)half / 2.0;
    for (int v = 0; v < V; ++v) s.databuf[(size_t)e * V + v] = buf;
}

// make_new_game: one thread per env.  env_mask (risvec_make_new_game_masked) and the gate select envs.
__global__ void k_make_new_game(Dims d, State s, risvec_params_t p, const int* __restrict__ ints, int n_ints,
                                const int* __restrict__ dirs, int n_dirs, unsigned long long call,
                                const unsigned char* __restrict__ env_mask, EnvGate g) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    if (env_mask != nullptr && env_mask[e] == 0) return;  // per-env reset: this env keeps its state
    if (!g.on(e)) return;
    make_new_game_env(d, s, p, e, ints, n_ints, dirs, n_dirs, g.key(e, call), g.kind(kRngReset, kRngEpReset));
}

// renew_positions of env e by one thread, vehicles in index order; arithmetic uses the
// round-to-nearest intrinsics so no FMA contraction can change a bit w.r.t. the reference.
// Returns the number of uniforms consumed.
__device__ __forceinline__ int renew_positions_env(const Dims& d, const State& s, const risvec_params_t& p, int e,
                                                   const double* __restrict__ uniforms, int n_uni,
                                                   unsigned long long call, unsigned kind) {
    const int V = d.V;
    int cur = 0;
    for (int i = 0; i < V; ++i) {
        const size_t ix = (size_t)e * V + i;
        const double delta = __dmul_rn((double)s.vel[ix], p.time_slow);
        int heading = s.dir[ix];
        const bool vertical = (heading == RISVEC_DIR_UP) || (heading == RISVEC_DIR_DOWN);
        const bool forward = (heading == RISVEC_DIR_UP) || (heading == RISVEC_DIR_RIGHT);
        double c = vertical ? s.pos_y[ix] : s.pos_x[ix];  // coordinate along the heading
        double o = vertical ? s.pos_x[ix] : s.pos_y[ix];  // lateral coordinate
        bool turned = false;
        for (int which = 0; which < 2 && !turned; ++which) {
            // u/d test left lanes then right lanes; r/l test up lanes then down lanes
            const double* fam = vertical ? (which == 0 ? p.left_lanes : p.right_lanes)
                                         : (which == 0 ? p.up_lanes : p.down_lanes);
            const int nf = vertical ? (which == 0 ? p.n_left : p.n_right) : (which == 0 ? p.n_up : p.n_down);
            for (int j = 0; j < nf; ++j) {
                const double lane = fam[j];
                bool hit;
                double gap;
                if (forward) {
                    hit = (c <= lane) && (__dadd_rn(c, delta) >= lane);
                    gap = __dsub_rn(lane, c);
                } else {
                    hit = (c >= lane) && (__dsub_rn(c, delta) <= lane);
                    gap = __dsub_rn(c, lane);
                }
                if (!hit) continue;
                double u;
                if (uniforms != nullptr) {
                    u = cur < n_uni ? uniforms[(size_t)e * n_uni + cur] : 1.0;
                } else {
                    uint4 r = rng_draw(d, e, call, (unsigned)(i * 16 + which * 8 + j), kind);
                    u = u01d(r.x, r.y);
                }
                ++cur;
                if (u < 0.4) {
                    if (vertical) {  // MARL:428-441,453-467 (note `delta + gap` for the right turn)
                        o = (which == 0) ? __dsub_rn(o, __dsub_rn(delta, gap)) : __dadd_rn(o, __dadd_rn(delta, gap));
                        heading = (which == 0) ? RISVEC_DIR_LEFT : RISVEC_DIR_RIGHT;
                    } else {  // MARL:480-491,503-514
                        o = (which == 0) ? __dadd_rn(o, __dsub_rn(delta, gap)) : __dsub_rn(o, __dsub_rn(delta, gap));
                        heading = (which == 0) ? RISVEC_DIR_UP : RISVEC_DIR_DOWN;
                    }
                    c = lane;
                    turned = true;
                    break;
                }
            }
        }
        if (!turned) c = forward ? __dadd_rn(c, delta) : __dsub_rn(c, delta);
        double x = vertical ? o : c, y = vertical ? c : o;
        if (x < 0 || y < 0 || x > p.width || y > p.height) {  // MARL:522-540
            if (heading == RISVEC_DIR_UP) {
                heading = RISVEC_DIR_RIGHT;
                y = p.right_lanes[p.n_right - 1];
            } else if (heading == RISVEC_DIR_DOWN) {
                heading = RISVEC_DIR_LEFT;
                y = p.left_lanes[0];
            } else if (heading == RISVEC_DIR_LEFT) {
                heading = RISVEC_DIR_UP;
                x = p.up_lanes[0];
            } else {
                heading = RISVEC_DIR_DOWN;
                x = p.down_lanes[p.n_down - 1];
            }
        }
        s.pos_x[ix] = x;
        s.pos_y[ix] = y;
        s.dir[ix] = heading;
    }
    return cur;
}

// renew_positions: one thread per env.  Envs the gate leaves out keep their state and report 0 draws used.
__global__ void k_renew_positions(Dims d, State s, risvec_params_t p, const double* __restrict__ uniforms, int n_uni,
                                  int* __restrict__ used_out, unsigned long long call, EnvGate g) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.E) return;
    int cur = 0;
    if (g.on(e))
        cur = renew_positions_env(d, s, p, e, uniforms, n_uni, g.key(e, call), g.kind(kRngMobility, kRngEpMobility));
    if (used_out != nullptr) used_out[e] = cur;
}

// compute_parms: one thread per (env, vehicle).  Distances and angles follow the reference's
// operation order exactly; the V x M phasor table `phases_R_i` is NOT materialised in HBM --
// the channel kernels regenerate exp(j*pi*m*(angle_BR - angle_v)) from `angle` in float64.
struct Parms {
    double dist, angle, amp;
};
__device__ __forceinline__ Parms compute_parms_of(const Dims& d, double x, double y) {
    const double dx = __dsub_rn(x, kRisX);
    const double dy = __dsub_rn(y, kRisY);
    const double dz = kVehZ - kRisZ;
    const double dist = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), dz * dz));
    Parms r;
    r.dist = dist;
    r.angle = __ddiv_rn(dx, dist);
    r.amp = (kRo * kRo) / (pow(dist, kAlpha1) * pow(d.dist_BR, kAlpha2));
    return r;
}

__global__ void k_compute_parms(Dims d, State s, EnvGate g) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.V) return;
    if (!g.on((long long)(ix / d.V))) return;
    const Parms r = compute_parms_of(d, s.pos_x[ix], s.pos_y[ix]);
    s.dist[ix] = r.dist;
    s.angle[ix] = r.angle;
    s.amp[ix] = r.amp;
}

}  // namespace risvec
