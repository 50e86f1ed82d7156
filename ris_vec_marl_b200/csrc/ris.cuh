// RIS phase state, BCD phase optimiser and per-episode channel gains (float64).
// Reference: Simulation-MARL-BCD/Environment.py:208-239,255-327.
#pragma once
#include "common.cuh"

namespace risvec {

// get_next_phase (MARL:233-239): theta_m = exp(j * phase_m), one thread per (env, element).
__global__ void k_set_phase(Dims d, State s, const float* __restrict__ phase) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.M) return;
    const float ph = phase[ix];
    double sn, cs;
    sincos((double)ph, &sn, &cs);
    s.phase_real[ix] = ph;
    s.theta_re[ix] = cs;
    s.theta_im[ix] = sn;
}

// Random_phase (MARL:203-206): theta_real[m] = possible_angles[k], k uniform in [0, 2^control_bit)
// (injected `idx`, or Philox when NULL); possible_angles = linspace(0, 2 pi, n, endpoint=False)
// (:169) = k * (2 pi / n).  theta_c = exp(j * theta_real) in float64.
__global__ void k_random_phase(Dims d, State s, const int* __restrict__ idx, unsigned long long call) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.M) return;
    const int e = (int)(ix / d.M), m = (int)(ix - (size_t)e * d.M);
    int k;
    if (idx != nullptr) k = idx[ix];
    else k = (int)(rng_draw(d, e, call, (unsigned)m, kRngChannel).x % (unsigned)d.ncand);
    k = min(max(k, 0), d.ncand - 1);
    const double step = __ddiv_rn(2.0 * 3.14159265358979323846, (double)d.ncand);
    const double ang = __dmul_rn((double)k, step);
    double sn, cs;
    sincos(ang, &sn, &cs);
    s.phase_real[ix] = (float)ang;
    s.theta_re[ix] = cs;
    s.theta_im[ix] = sn;
}

// The direct V2I link the reference defines but never calls: get_path_loss (MARL:192-196) and
// get_shadowing (MARL:198-201, AR(1) over delta_distance = velocity * time_slow (:410) with the
// V2I_Shadowing drawn at reset (:409) and one N(0, 8) draw), for every vehicle.
__global__ void k_direct_link(Dims d, State s, risvec_params_t p, const double* __restrict__ shadow_state,
                              const double* __restrict__ normals, double* __restrict__ path_loss,
                              double* __restrict__ shadowing, unsigned long long call) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.V) return;
    const int e = (int)(ix / d.V), v = (int)(ix - (size_t)e * d.V);
    if (path_loss != nullptr) {
        const double dist = hypot(fabs(s.pos_x[ix] - kBsX), fabs(s.pos_y[ix] - kBsY));
        const double hz = kBsZ - 1.5;
        const double d3 = sqrt(__dadd_rn(__dmul_rn(dist, dist), __dmul_rn(hz, hz)));
        path_loss[ix] = __dadd_rn(128.1, __dmul_rn(37.6, log10(__ddiv_rn(d3, 1000.0))));
    }
    if (shadowing != nullptr) {
        double n8;
        if (normals != nullptr) n8 = normals[ix];
        else {  // Box-Muller from two Philox uniforms, sigma = 8 dB
            const uint4 r = rng_draw(d, e, call, (unsigned)v, kRngChannel);
            const double u1 = fmax(u01d(r.x, r.y), 1e-300), u2 = u01d(r.z, r.w);
            n8 = 8.0 * sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
        }
        const double dd = __dmul_rn((double)s.vel[ix], p.time_slow);
        const double r = __ddiv_rn(dd, 10.0);  // Decorrelation_distance = 10 (MARL:86)
        const double a = exp(__dmul_rn(-1.0, r));
        const double b = sqrt(__dsub_rn(1.0, exp(__dmul_rn(-2.0, r))));
        shadowing[ix] = __dadd_rn(__dmul_rn(a, shadow_state[ix]), __dmul_rn(b, n8));
    }
}

// Geometry phasor of vehicle v and element m:
//   phases_R_i[v][m] * phase_R[m] = exp(-j*pi*angle_v*m) * exp(+j*pi*angle_BR*m)   (MARL:179,253)
// evaluated as sincospi(m * (angle_BR - angle_v)) -- sincospi reduces its argument exactly.
__device__ inline void geom_phasor(double delta, int m, double* re, double* im) {
    sincospi((double)m * delta, im, re);
}

// optimize_phase_shift (MARL:208-231): one warp per env.
// The reference objective sums `img` over ALL vehicles and elements (the same S for every
// vehicle), so x(theta) = K * |S|^2 with S = sum_m theta_m c_m, c_m = sum_v phasor(v, m) and
// K > 0 independent of theta.  The coordinate search therefore keeps S incrementally:
// for each m the candidate maximising |S - theta_m c_m + e_k c_m|^2 wins, first maximum on
// ties, accepted only if strictly positive (best starts at 0, MARL:210-218).
// NE: per-env RIS size `n_elem` (risvec_attach_ris_elements): the env's elements m < n only; unused without NE
template <bool NE = false>
__global__ void k_bcd(Dims d, State s, EnvGate g, const int* __restrict__ n_elem) {
    extern __shared__ double2 bcd_smem[];
    const int wpb = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * wpb + warp;
    if (e >= d.E || !g.on(e)) return;  // whole warp leaves together
    const int V = d.V, M = d.M, n = ris_count<NE>(n_elem, e, M);
    double2* c = bcd_smem + (size_t)warp * 2 * M;
    double2* th = c + M;
    double sr = 0.0, si = 0.0;
    for (int m = lane; m < n; m += 32) {
        double cr = 0.0, ci = 0.0;
        for (int v = 0; v < V; ++v) {
            double re, im;
            geom_phasor(d.angle_BR - s.angle[(size_t)e * V + v], m, &re, &im);
            cr += re;
            ci += im;
        }
        const double tr = s.theta_re[(size_t)e * M + m], ti = s.theta_im[(size_t)e * M + m];
        c[m] = make_double2(cr, ci);
        th[m] = make_double2(tr, ti);
        sr += tr * cr - ti * ci;
        si += tr * ci + ti * cr;
    }
    sr = seg_sum<32>(sr);
    si = seg_sum<32>(si);
    __syncwarp();
    // candidates: up to 32 -> lane k owns candidate k and its e_k = exp(j 2 pi k / ncand) is formed
    // once; more -> lanes stride over them.  The arg-max (first maximum wins) is reduced on
    // (value, k) only, over the 2^ceil(log2 ncand) lanes that hold candidates; the winner's partial
    // sums are then fetched from its lane.
    const bool one = d.ncand <= 32;
    double er0 = 0.0, ei0 = 0.0;
    if (one && lane < d.ncand) sincospi(2.0 * (double)lane / (double)d.ncand, &ei0, &er0);
    int width = 32;
    if (one) { width = 1; while (width < d.ncand) width <<= 1; }
    for (int m = 0; m < n; ++m) {
        const double2 cm = c[m], tm = th[m];
        const double rr = sr - (tm.x * cm.x - tm.y * cm.y);
        const double ri = si - (tm.x * cm.y + tm.y * cm.x);
        double best = -1.0, bsr = rr, bsi = ri, ber = 0.0, bei = 0.0;
        int bk = 0x7fffffff;
        if (one) {
            if (lane < d.ncand) {
                const double cr = rr + (er0 * cm.x - ei0 * cm.y);
                const double ci = ri + (er0 * cm.y + ei0 * cm.x);
                const double val = cr * cr + ci * ci;
                if (val > best) { best = val; bk = lane; bsr = cr; bsi = ci; ber = er0; bei = ei0; }
            }
        } else {
            for (int k = lane; k < d.ncand; k += 32) {
                double er, ei;
                sincospi(2.0 * (double)k / (double)d.ncand, &ei, &er);
                const double cr = rr + (er * cm.x - ei * cm.y);
                const double ci = ri + (er * cm.y + ei * cm.x);
                const double val = cr * cr + ci * ci;
                if (val > best) { best = val; bk = k; bsr = cr; bsi = ci; ber = er; bei = ei; }
            }
        }
        double wv = best;
        int wk = bk;
        for (int o = width >> 1; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(kFull, wv, o);
            const int ok = __shfl_xor_sync(kFull, wk, o);
            if (ov > wv || (ov == wv && ok < wk)) { wv = ov; wk = ok; }
        }
        wv = __shfl_sync(kFull, wv, 0);
        wk = __shfl_sync(kFull, wk, 0);
        if (wv > 0.0) {
            const int src = wk & 31;   // the lane whose own best candidate is the winner
            sr = __shfl_sync(kFull, bsr, src);
            si = __shfl_sync(kFull, bsi, src);
            if (lane == src) th[m] = make_double2(ber, bei);
        } else {  // never improved on best = 0: the reference stores the integer 0
            sr = rr; si = ri;
            if (lane == 0) th[m] = make_double2(0.0, 0.0);
        }
        __syncwarp();
    }
    for (int m = lane; m < n; m += 32) {
        s.theta_re[(size_t)e * M + m] = th[m].x;
        s.theta_im[(size_t)e * M + m] = th[m].y;
    }
}

// optimize_phase_shift for ncand <= 8, V <= 8 (every shipped configuration: control_bit = 3,
// V = 8): one warp = 4 envs, lane = (env el, candidate k), so all 32 lanes score candidates in the
// sequential element loop.  c_m = sum_v z_v^m is accumulated from ONE sincospi per lane
// (z_v = exp(j pi (angle_BR - angle_v)) of vehicle v = k, shuffled to the env's lanes) and float64
// complex powers: lane k owns the elements m = k + 8 i, w = z^k * (z^8)^i.  Same search, same
// tie rule (first maximum), same acceptance test as k_bcd.
// bcd_v8_warp is the body for the env e of this lane's group: `angle` = angle of vehicle min(k, V - 1) of env e,
// c / th = the env's 2 M double2 of shared memory (th holds the result afterwards).  All 32 lanes must call it
// (full-warp shuffles); only `write` envs store theta.  Shared by k_bcd_v8 and the fused episode start.
__device__ __forceinline__ void bcd_v8_warp(const Dims& d, const State& s, int e, bool write, double angle,
                                            double2* c, double2* th) {
    const int lane = threadIdx.x & 31, k = lane & 7;
    const int V = d.V, M = d.M, base = lane & ~7;
    const double2 my_z = unit_phasor64(d.angle_BR - angle);
    for (int m = k; m < M; m += 8) c[m] = make_double2(0.0, 0.0);
    for (int v = 0; v < V; ++v) {
        const double2 z = make_double2(__shfl_sync(kFull, my_z.x, base + v), __shfl_sync(kFull, my_z.y, base + v));
        double2 w = cpow64(z, (unsigned)k);
        const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
        for (int m = k; m < M; m += 8) {
            c[m].x += w.x;
            c[m].y += w.y;
            w = cmul64(w, z8);
        }
    }
    double sr = 0.0, si = 0.0;
    for (int m = k; m < M; m += 8) {
        const double tr = s.theta_re[(size_t)e * M + m], ti = s.theta_im[(size_t)e * M + m];
        const double2 cm = c[m];
        th[m] = make_double2(tr, ti);
        sr += tr * cm.x - ti * cm.y;
        si += tr * cm.y + ti * cm.x;
    }
    sr = seg_sum<8>(sr);
    si = seg_sum<8>(si);
    __syncwarp();
    double er0 = 0.0, ei0 = 0.0;
    if (k < d.ncand) sincospi(2.0 * (double)k / (double)d.ncand, &ei0, &er0);
    for (int m = 0; m < M; ++m) {
        const double2 cm = c[m], tm = th[m];
        const double rr = sr - (tm.x * cm.x - tm.y * cm.y);
        const double ri = si - (tm.x * cm.y + tm.y * cm.x);
        double best = -1.0, bsr = rr, bsi = ri;
        int bk = 0x7fffffff;
        if (k < d.ncand) {
            const double cr = rr + (er0 * cm.x - ei0 * cm.y);
            const double ci = ri + (er0 * cm.y + ei0 * cm.x);
            const double val = cr * cr + ci * ci;
            if (val > best) { best = val; bk = k; bsr = cr; bsi = ci; }
        }
        double wv = best;
        int wk = bk;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(kFull, wv, o);
            const int ok = __shfl_xor_sync(kFull, wk, o);
            if (ov > wv || (ov == wv && ok < wk)) { wv = ov; wk = ok; }
        }
        // (wv, wk) is uniform over the env's 8 lanes after the butterfly; the 4 envs of the warp may
        // decide differently, so the shuffles stay unconditional
        const bool acc = wv > 0.0;
        const int src = base + (acc ? (wk & 7) : 0);
        const double nsr = __shfl_sync(kFull, bsr, src), nsi = __shfl_sync(kFull, bsi, src);
        sr = acc ? nsr : rr;
        si = acc ? nsi : ri;
        if (acc) {
            if (lane == src) th[m] = make_double2(er0, ei0);
        } else if (k == 0) {  // never improved on best = 0: the reference stores the integer 0
            th[m] = make_double2(0.0, 0.0);
        }
        __syncwarp();
    }
    if (write)
        for (int m = k; m < M; m += 8) {
            s.theta_re[(size_t)e * M + m] = th[m].x;
            s.theta_im[(size_t)e * M + m] = th[m].y;
        }
}

// bcd_v8_warp for a per-env RIS size: env e's lanes score and write the elements m < n only (n = its own count).  The
// element loop runs to the largest count of the warp's four envs, because its shuffles need every lane; an env past
// its count takes part in them and keeps its state.  For m < n the operations are those of bcd_v8_warp on a handle
// with M = n.  A separate copy: a count argument in bcd_v8_warp changed the machine code of k_begin_episode.
__device__ __forceinline__ void bcd_v8_warp_n(const Dims& d, const State& s, int e, bool write, double angle,
                                              double2* c, double2* th, int n) {
    const int lane = threadIdx.x & 31, k = lane & 7;
    const int V = d.V, M = d.M, base = lane & ~7;
    const int nw = max(max(__shfl_sync(kFull, n, 0), __shfl_sync(kFull, n, 8)),
                       max(__shfl_sync(kFull, n, 16), __shfl_sync(kFull, n, 24)));
    const double2 my_z = unit_phasor64(d.angle_BR - angle);
    for (int m = k; m < n; m += 8) c[m] = make_double2(0.0, 0.0);
    for (int v = 0; v < V; ++v) {
        const double2 z = make_double2(__shfl_sync(kFull, my_z.x, base + v), __shfl_sync(kFull, my_z.y, base + v));
        double2 w = cpow64(z, (unsigned)k);
        const double2 z2 = cmul64(z, z), z4 = cmul64(z2, z2), z8 = cmul64(z4, z4);
        for (int m = k; m < n; m += 8) {
            c[m].x += w.x;
            c[m].y += w.y;
            w = cmul64(w, z8);
        }
    }
    double sr = 0.0, si = 0.0;
    for (int m = k; m < n; m += 8) {
        const double tr = s.theta_re[(size_t)e * M + m], ti = s.theta_im[(size_t)e * M + m];
        const double2 cm = c[m];
        th[m] = make_double2(tr, ti);
        sr += tr * cm.x - ti * cm.y;
        si += tr * cm.y + ti * cm.x;
    }
    sr = seg_sum<8>(sr);
    si = seg_sum<8>(si);
    __syncwarp();
    double er0 = 0.0, ei0 = 0.0;
    if (k < d.ncand) sincospi(2.0 * (double)k / (double)d.ncand, &ei0, &er0);
    for (int m = 0; m < nw; ++m) {
        const bool own = m < n;  // uniform over the env's 8 lanes
        const double2 cm = own ? c[m] : make_double2(0.0, 0.0), tm = own ? th[m] : make_double2(0.0, 0.0);
        const double rr = sr - (tm.x * cm.x - tm.y * cm.y);
        const double ri = si - (tm.x * cm.y + tm.y * cm.x);
        double best = -1.0, bsr = rr, bsi = ri;
        int bk = 0x7fffffff;
        if (k < d.ncand) {
            const double cr = rr + (er0 * cm.x - ei0 * cm.y);
            const double ci = ri + (er0 * cm.y + ei0 * cm.x);
            const double val = cr * cr + ci * ci;
            if (val > best) { best = val; bk = k; bsr = cr; bsi = ci; }
        }
        double wv = best;
        int wk = bk;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(kFull, wv, o);
            const int ok = __shfl_xor_sync(kFull, wk, o);
            if (ov > wv || (ov == wv && ok < wk)) { wv = ov; wk = ok; }
        }
        const bool acc = wv > 0.0;
        const int src = base + (acc ? (wk & 7) : 0);
        const double nsr = __shfl_sync(kFull, bsr, src), nsi = __shfl_sync(kFull, bsi, src);
        if (own) {
            sr = acc ? nsr : rr;
            si = acc ? nsi : ri;
            if (acc) {
                if (lane == src) th[m] = make_double2(er0, ei0);
            } else if (k == 0) {  // never improved on best = 0: the reference stores the integer 0
                th[m] = make_double2(0.0, 0.0);
            }
        }
        __syncwarp();
    }
    if (write)
        for (int m = k; m < n; m += 8) {
            s.theta_re[(size_t)e * M + m] = th[m].x;
            s.theta_im[(size_t)e * M + m] = th[m].y;
        }
}

// NE: as k_bcd; the four envs of a warp may have different counts (the element loop is per env's lane group)
template <bool NE = false>
__global__ void k_bcd_v8(Dims d, State s, EnvGate g, const int* __restrict__ n_elem) {
    extern __shared__ double2 bcd_smem[];
    const int wpb = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, el = lane >> 3, k = lane & 7;
    const int e_raw = (blockIdx.x * wpb + warp) * 4 + el;
    const int e = min(e_raw, d.E - 1);
    const bool env_ok = e_raw < d.E && g.on(e);
    double2* c = bcd_smem + (size_t)(warp * 4 + el) * 2 * d.M;
    const double angle = s.angle[(size_t)e * d.V + min(k, d.V - 1)];
    if constexpr (NE) bcd_v8_warp_n(d, s, e, env_ok, angle, c, c + d.M, ris_count<NE>(n_elem, e, d.M));
    else bcd_v8_warp(d, s, e, env_ok, angle, c, c + d.M);
}

// update_channel_gains, "free" model, lane = (env, vehicle): the vehicle's phasor z_v^m is stepped
// by one float64 complex multiplication per element (re-anchored by an exact sincospi every 32
// elements), the M products theta_m z_v^m are summed in order -- no shuffles at all.
// gains_free_lane is the per-vehicle body: theta_m = (tr[m * ts], ti[m * ts]) (ts = 1: the state arrays; ts = 2: an
// interleaved double2 copy in shared memory), summed over the elements m < n (d.M, or the env's per-env RIS size).
// Shared by k_gains_free_v and the fused episode start.
__device__ __forceinline__ double gains_free_lane(const Dims& d, double angle, double amp, const double* tr,
                                                  const double* ti, int ts, int n) {
    const double delta = d.angle_BR - angle;
    const double2 z = unit_phasor64(delta);
    double sr = 0.0, si = 0.0;
    double2 w = make_double2(1.0, 0.0);
    for (int m = 0; m < n; ++m) {
        if ((m & 31) == 0 && m) w = unit_phasor64((double)m * delta);
        const double a = tr[(size_t)m * ts], b = ti[(size_t)m * ts];
        sr += a * w.x - b * w.y;
        si += a * w.y + b * w.x;
        w = cmul64(w, z);
    }
    return amp * (sr * sr + si * si);
}

// NE: as k_bcd
template <int VP, bool NE = false>
__global__ void k_gains_free_v(Dims d, State s, EnvGate g, const int* __restrict__ n_elem) {
    const long long gtid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int e_raw = (int)(gtid / VP), v = (int)(gtid % VP);
    const int e = min(e_raw, d.E - 1), M = d.M;
    const bool act = e_raw < d.E && v < d.V && g.on(e);
    const size_t ev = (size_t)e * d.V + min(v, d.V - 1);
    const double gain = gains_free_lane(d, s.angle[ev], s.amp[ev], s.theta_re + (size_t)e * M,
                                        s.theta_im + (size_t)e * M, 1, ris_count<NE>(n_elem, e, M));
    if (act) s.gains[ev] = gain;
}

// update_channel_gains, "free" model (MARL:263-273): the cascaded RIS reduction
//   gain_v = amp_v * | sum_m theta_m * phasor(v, m) |^2
// one warp per env, lanes stride over the M elements, complex warp-shuffle reduction.  NE: as k_bcd
template <bool NE = false>
__global__ void k_gains_free(Dims d, State s, EnvGate g, const int* __restrict__ n_elem) {
    const int wpb = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int e = blockIdx.x * wpb + warp;
    if (e >= d.E || !g.on(e)) return;
    const int V = d.V, M = d.M, n = ris_count<NE>(n_elem, e, M);
    for (int v = 0; v < V; ++v) {
        const double delta = d.angle_BR - s.angle[(size_t)e * V + v];
        double sr = 0.0, si = 0.0;
        for (int m = lane; m < n; m += 32) {
            double re, im;
            geom_phasor(delta, m, &re, &im);
            const double tr = s.theta_re[(size_t)e * M + m], ti = s.theta_im[(size_t)e * M + m];
            sr += tr * re - ti * im;
            si += tr * im + ti * re;
        }
        sr = seg_sum<32>(sr);
        si = seg_sum<32>(si);
        if (lane == 0) s.gains[(size_t)e * V + v] = s.amp[(size_t)e * V + v] * (sr * sr + si * si);
    }
}

// update_channel_gains, simplified 3GPP TR 38.901 UMi / UMa branch (MARL:275-327): direct
// vehicle<->BS link with LOS draw, log-normal shadowing and Rayleigh / Rice small-scale power.  No RIS term, so it
// takes no per-env RIS size.
// One thread per (env, vehicle).  Draw order per vehicle in the reference: rand, normal,
// then exponential (K = 0) or two normals.
__global__ void k_gains_3gpp(Dims d, State s, risvec_params_t p, const double* __restrict__ c_rand,
                             const double* __restrict__ c_normal, const double* __restrict__ c_exp,
                             unsigned long long call_host, EnvGate g) {
    const size_t ix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (ix >= (size_t)d.E * d.V) return;
    const int e = (int)(ix / d.V), v = (int)(ix % d.V);
    if (!g.on(e)) return;
    const unsigned long long call = g.key(e, call_host);
    const unsigned kind = g.kind(kRngChannel, kRngEpChannel);
    double u, z0, z1, z2, ex;
    if (c_rand != nullptr) {
        u = c_rand[ix];
        z0 = c_normal[ix * 3 + 0]; z1 = c_normal[ix * 3 + 1]; z2 = c_normal[ix * 3 + 2];
        ex = c_exp[ix];
    } else {
        const uint4 a = rng_draw(d, e, call, (unsigned)(v * 4 + 0), kind);
        const uint4 b = rng_draw(d, e, call, (unsigned)(v * 4 + 1), kind);
        const uint4 c = rng_draw(d, e, call, (unsigned)(v * 4 + 2), kind);
        u = u01d(a.x, a.y);
        ex = -log1p(-u01d(a.z, a.w));
        // Box-Muller pairs
        const double r0 = sqrt(-2.0 * log1p(-u01d(b.x, b.y))), t0 = 2.0 * u01d(b.z, b.w);
        const double r1 = sqrt(-2.0 * log1p(-u01d(c.x, c.y))), t1 = 2.0 * u01d(c.z, c.w);
        z0 = r0 * cospi(t0); z1 = r0 * sinpi(t0); z2 = r1 * cospi(t1);
        (void)t1;
    }
    const double dx = fabs(s.pos_x[ix] - kBsX), dy = fabs(s.pos_y[ix] - kBsY), dz = fabs(kBsZ - kVehZ);
    const double d2d = hypot(dx, dy);
    const double d3d = sqrt(d2d * d2d + dz * dz);
    const bool los = u < 0.7 * exp(-d2d / 200.0);
    const double dd = fmax(d3d, 1.0), fc = p.fc_GHz;
    double pl = 0.0;
    if (p.channel_model == RISVEC_CHANNEL_3GPP_UMI) {
        pl = los ? 32.4 + 21.0 * log10(fc) + 20.0 * log10(dd) : 36.7 + 22.7 * log10(fc) + 26.0 * log10(dd);
    } else if (p.channel_model == RISVEC_CHANNEL_3GPP_UMA) {
        pl = los ? 28.0 + 22.0 * log10(fc) + 20.0 * log10(dd)
                 : 13.54 + 39.08 * log10(dd) + 20.0 * log10(fc) - 0.6 * p.veh_ant_gain;
    }
    const double large = pow(10.0, -pl / 10.0);
    const double shadow = pow(10.0, (z0 * (los ? p.shadow_std_los : p.shadow_std_nlos)) / 10.0);
    double small;
    if (p.rician_K_dB <= 1e-6) {
        small = ex;
    } else {
        const double K = pow(10.0, p.rician_K_dB / 10.0);
        const double sm = sqrt(K / (K + 1.0)), sg = 1.0 / sqrt(2.0 * (K + 1.0));
        const double hr = sm + sg * z1, hi = sg * z2;
        small = hr * hr + hi * hi;
    }
    s.gains[ix] = large * shadow * small;
}

}  // namespace risvec
