/*
 * risvec.h -- C ABI of the B200-native batched RIS-VEC environment library.
 *
 * One handle = E independent env instances (V vehicles, M RIS elements each) resident in
 * the HBM of ONE GPU.  Each entry point replaces, for all E instances at once, one method of
 * the reference python class `Environ`; the reference has no FFI of its own (SURVEY.md 8b),
 * so the binding a reference maintainer would add is the ctypes stub in INTEGRATION.md.
 * Citations: MARL = Simulation-MARL-BCD/Environment.py, SARL = Simulation-SARL/Environment.py.
 *
 * Conventions
 *   - every function returns 0 on success or a negative RISVEC_ERR_* code; the message of the
 *     last failure on the calling thread is available from risvec_last_error();
 *   - all pointer arguments of the non-`_host` functions are DEVICE pointers on the handle's GPU,
 *     caller-owned, dense row-major with the shapes given below; NULL = "not supplied";
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are
 *     asynchronous on it; calls on one handle must be externally serialised;
 *   - there is no CPU fallback: creation fails when no sm_100 device is usable.
 */
#ifndef RISVEC_H
#define RISVEC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RISVEC_ABI_VERSION 1

enum {
    RISVEC_OK = 0,
    RISVEC_ERR_INVALID = -1,     /* bad argument (shape, NULL handle, ...) */
    RISVEC_ERR_UNSUPPORTED = -2, /* size outside what the kernels cover (V > 32, M > 1024, ...) */
    RISVEC_ERR_CUDA = -3,        /* CUDA runtime / launch failure */
    RISVEC_ERR_NODEVICE = -4     /* no usable sm_100 device */
};

enum { RISVEC_VARIANT_MARL = 0, RISVEC_VARIANT_SARL = 1 };
enum { RISVEC_CHANNEL_FREE = 0, RISVEC_CHANNEL_3GPP_UMI = 1, RISVEC_CHANNEL_3GPP_UMA = 2,
       RISVEC_CHANNEL_UNKNOWN = 3 };

/* vehicle heading codes (the reference stores the characters 'u','d','l','r') */
enum { RISVEC_DIR_UP = 0, RISVEC_DIR_DOWN = 1, RISVEC_DIR_LEFT = 2, RISVEC_DIR_RIGHT = 3 };

/* batched form of the ragged `noma_groups` list of MARL:331-372: one int32 per user */
#define RISVEC_PARTNER_SINGLE (-1)       /* group of one (OMA)                                  */
#define RISVEC_PARTNER_NONE (-2)         /* in no group, or in a group of size != 1,2 -> rate 0 */
#define RISVEC_PARTNER_SECOND (1 << 16)  /* OR-ed onto the partner index of the user that is
                                            listed SECOND in its pair (tie rule of MARL:355)   */

#define RISVEC_MAX_LANES 8

/* Scalar parameters.  Mirrors the attributes the reference drivers set on the env object
 * (SURVEY.md 8b "attributes WRITTEN"); defaults are filled by risvec_default_params(). */
typedef struct risvec_params {
    /* map (MARL:57-64) */
    int32_t n_up, n_down, n_left, n_right;
    double up_lanes[RISVEC_MAX_LANES], down_lanes[RISVEC_MAX_LANES];
    double left_lanes[RISVEC_MAX_LANES], right_lanes[RISVEC_MAX_LANES];
    double width, height;
    /* shared (MARL:101-105,156-158; SARL:64-78) */
    double time_slow, time_fast, bandwidth, k, L, rate;
    int32_t data_buf_size;
    int32_t channel_model; /* RISVEC_CHANNEL_* (MARL:185) */
    /* MARL (MARL:70-143,555) */
    double noise_power, P_max, power_scale, f_local_max, f_edge_max, cycles_per_bit, cpu_share_floor;
    double w_d, w_e, R_min_bpsHz, D_max_s, qos_penalty, reward_clip;
    int32_t qos_enable;
    int32_t _pad0;
    double fc_GHz, shadow_std_los, shadow_std_nlos, rician_K_dB, veh_ant_gain;
    /* SARL (SARL:80-83) */
    double t_factor1, t_factor2, penalty1, penalty2;
} risvec_params_t;

/* State fields owned by the library, exposed as device pointers for zero-copy views. */
enum risvec_field {
    RISVEC_F_POS_X = 0,      /* f64 [E,V]  vehicles[i].position[0]                       */
    RISVEC_F_POS_Y,          /* f64 [E,V]  vehicles[i].position[1]                       */
    RISVEC_F_DIR,            /* i32 [E,V]  RISVEC_DIR_*                                  */
    RISVEC_F_VEL,            /* i32 [E,V]  velocity (m/s)                                */
    RISVEC_F_DIST,           /* f64 [E,V]  distances_R_i                                 */
    RISVEC_F_ANGLE,          /* f64 [E,V]  angles_R_i                                    */
    RISVEC_F_AMP,            /* f64 [E,V]  ro^2 / (d^alpha1 * dBR^alpha2)                */
    RISVEC_F_THETA_RE,       /* f64 [E,M]  Re elements_phase_shift_complex               */
    RISVEC_F_THETA_IM,       /* f64 [E,M]  Im elements_phase_shift_complex               */
    RISVEC_F_PHASE_REAL,     /* f32 [E,M]  elements_phase_shift_real (radians)           */
    RISVEC_F_GAINS,          /* f64 [E,V]  channel_gains                                 */
    RISVEC_F_DATABUF,        /* f64 [E,V]  DataBuf (kbit)                                */
    RISVEC_F_DATA_T,         /* f32 [E,V]  data_t                                        */
    RISVEC_F_DATA_P,         /* f32 [E,V]  data_p                                        */
    RISVEC_F_OVER_DATA,      /* f32 [E,V]  over_data                                     */
    RISVEC_F_OVER_POWER,     /* f32 [E,V]  over_power of the last step                   */
    RISVEC_F_RATE,           /* f32 [E,V]  vehicle_rate                                  */
    RISVEC_F_DATA_R,         /* i32 [E,V]  data_r (last arrivals)                        */
    RISVEC_F_REWARD_USER,    /* f32 [E,V]  per-user reward of the last step              */
    RISVEC_F_REWARD,         /* f32 [E]    global reward of the last step                */
    RISVEC_F_MECQ,           /* f64 [E]    mec_queue_cycles                              */
    RISVEC_F_STATS,          /* f32 [E,RISVEC_NSTAT] last_* scalars of the last step     */
    RISVEC_F_LAST_POWER,     /* f32 [E,2,V] last_power_W                                 */
    RISVEC_F_STEP_CTR,       /* i64 [E]    steps taken (keys the on-device RNG)          */
    RISVEC_F_V2I_SHADOWING,  /* f64 [E,V]  V2I_Shadowing drawn at reset (MARL:409); read only by risvec_direct_link */
    /* NOMA pairing stage of the MARL driver (risvec_pair_noma) */
    RISVEC_F_PAIR_HIST,      /* f32 [E,V*V] pair_affinity_hist (marl_train_bcd.py:1288)  */
    RISVEC_F_PAIR_STREAK,    /* i32 [E,V]  unpaired_streak (:1290)                       */
    RISVEC_F_PAIR_TAU,       /* f64 [E]    last_tau_now (:1341)                          */
    RISVEC_F_PAIR_K,         /* i32 [E]    last_K_now (:1342)                            */
    RISVEC_F_PAIR_MASK,      /* u8  [E,V*V] last_mask_mat, 1 = selectable (:1337-1340)   */
    RISVEC_F_PAIR_ROUNDS,    /* i32 [E]    back-off rounds used by the last solve (:1493)*/
    RISVEC_F_NOMA_PARTNER,   /* i32 [E,V]  noma_groups, partner encoding (rollout input) */
    RISVEC_F_NOMA_NGROUPS,   /* i32 [E]    len(noma_groups); 0 = no groups yet           */
    RISVEC_F_NOMA_PAIRS,     /* i32 [E,V]  pairs (i0,j0,i1,j1,...) in list order, -1 pad */
    RISVEC_F_NOMA_NPAIRS,    /* i32 [E]    len(pairs)                                    */
    /* per-env episode clock (risvec_episode_tick); both zero at creation */
    RISVEC_F_EP_STEP,        /* i32 [E]    step of its episode the env's next driver step takes; 0 = starts */
    RISVEC_F_EP_INDEX,       /* i32 [E]    the env's i_episode                           */
    RISVEC_F_COUNT
};

/* columns of RISVEC_F_STATS / of the per-step `stats` trace (MARL:612-614,636-656,677,706-711) */
enum risvec_stat {
    RISVEC_S_DELAY_MEAN = 0, RISVEC_S_ENERGY_MEAN, RISVEC_S_DELAY_LOCAL_MEAN, RISVEC_S_DELAY_EDGE_Q_MEAN,
    RISVEC_S_DELAY_EDGE_C_MEAN, RISVEC_S_T_TX_MEAN, RISVEC_S_BACKLOG_KBIT_MEAN, RISVEC_S_MEC_UTILIZATION,
    RISVEC_S_LOCAL_UTIL_MEAN, RISVEC_S_QOS_VIOLATION, RISVEC_S_OFF_KBIT_SUM, RISVEC_S_LOCAL_KBIT_SUM,
    RISVEC_S_MEC_QUEUE_CYCLES, RISVEC_NSTAT_USED, RISVEC_NSTAT = 16
};

typedef struct risvec_env risvec_env_t;

/* Per-step output traces of a MARL rollout; every member may be NULL (not written).
 * What MARL:731 returns plus the attributes the driver reads after each step. */
typedef struct risvec_marl_out {
    float* reward_user; /* [T,E,V]   */
    float* reward;      /* [T,E]     global_reward                       */
    float* DataBuf;     /* [T,E,V]   after arrivals                      */
    float* data_t;      /* [T,E,V]   */
    float* data_p;      /* [T,E,V]   */
    float* rate;        /* [T,E,V]   vehicle_rate                        */
    float* over_power;  /* [T,E,V]   */
    float* stats;       /* [T,E,RISVEC_NSTAT]                            */
    float* last_power;  /* [T,E,2,V] last_power_W                        */
} risvec_marl_out_t;

/* Per-step output traces of a SARL rollout (SARL:359); every member may be NULL. */
typedef struct risvec_sarl_out {
    float* reward;     /* [T,E]   */
    float* DataBuf;    /* [T,E,V] after arrivals */
    float* data_t;     /* [T,E,V] */
    float* data_p;     /* [T,E,V] */
    float* over_power; /* [T,E,V] */
    float* over_data;  /* [T,E,V] */
    float* rate;       /* [T,E,V] */
} risvec_sarl_out_t;

int risvec_abi_version(void);
const char* risvec_last_error(void);

/* Reference class defaults (MARL:70-143 or SARL:64-83) and the drivers' lane constants
 * (marl_train_bcd.py:446-449). */
int risvec_default_params(int variant, risvec_params_t* out);

/* Environ.__init__ (MARL:57-190, SARL:37-106) for E instances.  `env_index_base` is the global
 * index of this shard's first env (keys the on-device RNG so results do not depend on how envs
 * are sharded over GPUs); `seed` keys all on-device randomness. */
int risvec_create(const risvec_params_t* params, int variant, int E, int V, int M, int control_bit, int device,
                  uint64_t seed, int64_t env_index_base, risvec_env_t** out);
int risvec_destroy(risvec_env_t* env);

/* attribute writes of the drivers (marl_train_bcd.py:563-594,750-779) */
int risvec_set_params(risvec_env_t* env, const risvec_params_t* params);
int risvec_get_params(const risvec_env_t* env, risvec_params_t* out);

/* zero-copy access to library-owned state; *rows x *cols elements of `*elem_bytes` bytes */
int risvec_field(risvec_env_t* env, int field, void** dev_ptr, int64_t* rows, int64_t* cols, int* elem_bytes,
                 int* is_float);

/* make_new_game (MARL:733-737 + 381-410; SARL:361-365 + 176-205).
 * reset_ints [E,n_ints] i32: the randint draws in the reference's call order
 * (9 per round of four vehicles, 3 per extra vehicle, 1 for DataBuf); reset_dirs [E,V%4] i32
 * heading codes of the extra vehicles.  Both NULL -> on-device Philox draws. */
int risvec_make_new_game(risvec_env_t* env, const int32_t* reset_ints, int n_ints, const int32_t* reset_dirs,
                         int n_dirs, void* stream);
/* ... for a SUBSET of the envs: env_mask [E] u8 (device), != 0 = reset this env, 0 = leave every field of it
 * untouched (a batched driver restarts the envs whose episode ended while the others run on; the reference
 * object is one env, so its make_new_game is the all-ones mask).  NULL = all envs.  reset_ints / reset_dirs
 * keep their [E, n] shape; rows of unmasked envs are ignored. */
int risvec_make_new_game_masked(risvec_env_t* env, const uint8_t* env_mask, const int32_t* reset_ints, int n_ints,
                                const int32_t* reset_dirs, int n_dirs, void* stream);

/* renew_positions (MARL:412-542).  uniforms [E,n] f64 consumed per env by a cursor in the
 * reference's draw order (NULL -> Philox); used_out [E] i32 receives the draws consumed. */
int risvec_renew_positions(risvec_env_t* env, const double* uniforms, int n, int32_t* used_out, void* stream);

/* compute_parms (MARL:241-253) */
int risvec_compute_parms(risvec_env_t* env, void* stream);

/* get_next_phase (MARL:233-239): phase [E,M] f32 radians */
int risvec_set_phase(risvec_env_t* env, const float* phase, void* stream);

/* optimize_phase_shift (MARL:208-231), float64 */
int risvec_optimize_phase_shift(risvec_env_t* env, void* stream);

/* update_channel_gains (MARL:255-327).  For the 3GPP models: chan_rand [E,V] f64 U(0,1),
 * chan_normal [E,V,3] f64 N(0,1) (shadowing, Rice re, Rice im), chan_exp [E,V] f64 Exp(1);
 * all NULL -> Philox.  Ignored for RISVEC_CHANNEL_FREE. */
int risvec_update_channel_gains(risvec_env_t* env, const double* chan_rand, const double* chan_normal,
                                const double* chan_exp, void* stream);

/* T consecutive Environ.step calls (MARL:547-731) fused in one launch; T = 1 is a plain step.
 * action [T,E,2,V] f32; partner [E,V] i32 and ngroups [E] i32 (fixed over the T steps, see
 * RISVEC_PARTNER_*); arrivals [T,E,V] i32 Poisson draws (NULL -> Philox). */
int risvec_rollout_marl(risvec_env_t* env, int T, const float* action, const int32_t* partner,
                        const int32_t* ngroups, const int32_t* arrivals, const risvec_marl_out_t* out, void* stream);

/* T consecutive SARL Environ.step calls (SARL:321-359).  action [T,E,2,V] f32,
 * phase [T,E,M] f32 radians, arrivals [T,E,V] i32 (NULL -> Philox). */
int risvec_rollout_sarl(risvec_env_t* env, int T, const float* action, const float* phase, const int32_t* arrivals,
                        const risvec_sarl_out_t* out, void* stream);

/* Packed (tiled) record layout -- the library's native streaming format for the BASELINE shapes
 * (V == 8 vehicles, E a multiple of 4; SARL additionally M in {16, 40}).  Envs are taken in
 * groups of 4 (= one warp); per step and group there is ONE input tile and ONE output tile whose
 * fields are each [4 envs][8 vehicles] = one 128-byte line, so a rollout reads one stream and
 * writes one stream (+ the per-env reward), every access is a full line, and all fields of a
 * lane sit at compile-time offsets from one base pointer:
 *   SARL in  [T, E/4, 4*(24+M)] words: action_power[0] [4][8] f32 | action_power[1] [4][8] f32 |
 *                                      arrivals [4][8] i32 | action_phase [4][M] f32 (radians)
 *   SARL out [T, E/4, 4*48] f32: DataBuf | data_t | data_p | over_power | over_data | rate, each [4][8]
 *   MARL in  [T, E/4, 4*24] words: action_power[0] [4][8] | action_power[1] [4][8] | arrivals [4][8] i32
 *   MARL out [T, E/4, 4*40] f32: reward_user | DataBuf | data_t | data_p | rate, each [4][8]
 *   reward   [T, E] f32 (mean / global reward), a separate array in both variants.
 * Same arithmetic, bit-identical results to the per-array entry points.  Other shapes return
 * RISVEC_ERR_UNSUPPORTED (use the per-array entry points). */
#define RISVEC_SARL_IN_WORDS(M) (24 + (M))
#define RISVEC_SARL_OUT_WORDS 48
#define RISVEC_MARL_IN_WORDS 24
#define RISVEC_MARL_OUT_WORDS 40
int risvec_rollout_sarl_packed(risvec_env_t* env, int T, const void* in_rec, float* out_rec, float* reward,
                               void* stream);
int risvec_rollout_marl_packed(risvec_env_t* env, int T, const void* in_rec, const int32_t* partner,
                               const int32_t* ngroups, float* out_rec, float* reward, void* stream);
/* ... and with (pinned) HOST records: chunked H2D -> rollout -> D2H pipeline on three streams */
int risvec_rollout_sarl_packed_host(risvec_env_t* env, int T, const void* in_rec, float* out_rec, float* reward,
                                    void* stream);
int risvec_rollout_marl_packed_host(risvec_env_t* env, int T, const void* in_rec, const int32_t* partner,
                                    const int32_t* ngroups, float* out_rec, float* reward, void* stream);

/* Same two calls with HOST buffers (pinned for full PCIe speed): inputs are copied to device
 * staging owned by the handle, the rollout runs, the non-NULL traces are copied back.  All on
 * `stream`; the caller synchronises the stream before reading the outputs. */
int risvec_rollout_marl_host(risvec_env_t* env, int T, const float* action, const int32_t* partner,
                             const int32_t* ngroups, const int32_t* arrivals, const risvec_marl_out_t* out,
                             void* stream);
int risvec_rollout_sarl_host(risvec_env_t* env, int T, const float* action, const float* phase,
                             const int32_t* arrivals, const risvec_sarl_out_t* out, void* stream);

/* Driver-side glue on device (SURVEY.md 8f row 1).
 * risvec_observe: marl_get_state (marl_train_bcd.py:819-827) / get_state (ddpg_train.py:47-73) for
 * every agent of every env: obs [E, V, n_theta + 5] f32 where n_theta = 0 (MARL) or M / V (SARL).
 * risvec_map_actions: raw policy outputs in [-1,1] -> env actions.  MARL (marl_train_bcd.py:1601-1608):
 * raw [E,V,2] -> action [E,2,V] (phase ignored).  SARL (ddpg_train.py:151-160): raw [E, 2V+M] ->
 * action [E,2,V] and phase [E,M] radians. */
int risvec_observe(risvec_env_t* env, float* obs, void* stream);
int risvec_map_actions(risvec_env_t* env, const float* raw, float* action, float* phase, void* stream);

/* One MARL driver step in ONE launch (SURVEY.md 8f row 1): `raw` = the actors' tanh outputs [E, V, 2]; the action
 * mapping of marl_train_bcd.py:1601-1608 (risvec_map_actions) runs in the step kernel's prologue, then Environ.step
 * (MARL/Environment.py:547-731, no traces: the results are the state views), and marl_get_state of the NEW state
 * (marl_train_bcd.py:819-827, risvec_observe) is written to `obs` [E, V, 5] in its epilogue.  `arrivals` [E, V] or
 * NULL (on-device draws).  Bit-identical to the three separate calls.  V <= 8 runs fused (k_marl_v8); other shapes
 * run the three kernels back to back from this one call. */
int risvec_step_marl_fused(risvec_env_t* env, const float* raw, const int32_t* partner, const int32_t* ngroups,
                           const int32_t* arrivals, float* obs, void* stream);
/* The SARL driver step in one launch: `raw` = the actor's tanh outputs [E, 2V + M] (power rows, then the RIS phases);
 * the mapping of ddpg_train.py:151-160, Environ.step (SARL/Environment.py:321-359) and get_state of the new state
 * (ddpg_train.py:47-73) -> `obs` [E, V, M / V + 5].  Fused for V <= 8, M even <= 64 (k_sarl_mma); other shapes run
 * the three kernels back to back from this one call.  Bit-identical to the three separate calls. */
int risvec_step_sarl_fused(risvec_env_t* env, const float* raw, const int32_t* arrivals, float* obs, void* stream);

/* Random_phase (MARL:203-206; not called by the shipped drivers): every element gets one of the
 * 2^control_bit quantised angles linspace(0, 2 pi, n, endpoint=False)[k] (:169).  idx [E,M] i32
 * (device) injects the choices k (python `random.choice` in the reference); NULL draws them on the
 * device (Philox). */
int risvec_random_phase(risvec_env_t* env, const int32_t* idx, void* stream);
/* The direct V2I link that the reference defines but never calls (SURVEY 8a row a9):
 * path_loss [E,V] f64 = get_path_loss(position) in dB (MARL:192-196); shadowing [E,V] f64 =
 * get_shadowing(delta_distance = velocity * time_slow, vehicle) (MARL:198-201) from the
 * RISVEC_F_V2I_SHADOWING state and one N(0, 8) draw per vehicle (normals [E,V] f64 injected, or
 * NULL: Philox).  Either output may be NULL.  Nothing on the step path reads these (as in the
 * reference); RISVEC_F_V2I_SHADOWING is written by the caller (compat: the numpy draw of :409). */
int risvec_direct_link(risvec_env_t* env, const double* normals, double* path_loss, double* shadowing, void* stream);

/* ---- NOMA pairing (SURVEY 8f row 2): the stage that builds `noma_groups` for Environ.step ----
 * Knobs of the pairing pipeline; defaults = Config.__init__ and the getattr fall-backs at the call
 * site (marl_train_bcd.py:435-441,489-503,1404-1418,1481-1498); yaml != 0 applies the overlay of
 * the shipped config.yaml (:639-660,716-732). */
typedef struct risvec_pairing {
    int32_t min_pair_target;     /* :489,1413  (max(1, .) is applied by the library) */
    int32_t mwm_backoff_rounds;  /* :440,1493 */
    int32_t relax_topk_step;     /* :1482 */
    int32_t qos_enable;          /* :1427 */
    double mwm_accept_quantile, mwm_accept_q_step;      /* :439,441 */
    double completion_min_quantile;                     /* :282,300 */
    double relax_tau_factor_per_round, tau_back_floor_db; /* :1483,1498 */
    double score_w_delta_db, score_w_history;           /* :1416-1417 */
    double abs_gain_min_db;                             /* :1418 (-inf = off) */
    double qos_soft_penalty_dbscore;                    /* :1449 */
    double pair_hist_decay;                             /* :1404 */
} risvec_pairing_t;

#define RISVEC_PAIR_MAX_V 12 /* the matching is an exact DP over 2^V vehicle subsets (:360-393) */

int risvec_default_pairing(int n_veh, int yaml, risvec_pairing_t* out);

/* One driver step of the pairing stage for every env (marl_train_bcd.py:1315-1344,1404-1406,
 * 1413-1524,1542-1561): [decay != 0: pair_affinity_hist *= pair_hist_decay]; [recalc_mask != 0:
 * tau = quantile_{tau_q}(|dg_dB| strong x weak), mask from tau and row top-`topk` -> PAIR_TAU,
 * PAIR_K, PAIR_MASK; else the solve runs on the all-ones mask as the reference does]; QoS soft mask
 * from `p01` (offload power in [0,1], row 0 of the env action: pass `action` with
 * p01_env_stride = 2V) and the env's noise_power / P_max / R_min_bpsHz; score matrix; exact
 * max-weight matching on the edges above the (1 - accept_q) quantile; greedy completion; back-off
 * rounds; then noma_groups -> NOMA_PARTNER / NOMA_NGROUPS (feed them to risvec_rollout_marl),
 * NOMA_PAIRS / NOMA_NPAIRS, and the history / streak updates.  reuse [E] i32 (device, may be
 * NULL): != 0 keeps that env's frozen groups (:1542-1547) and only updates history / streak.
 * new_episode != 0: the call is the first step of an episode -- history, streak and frozen groups are
 * taken as cleared (what risvec_pair_reset does, without the extra launch); needs recalc_mask != 0.
 * V <= RISVEC_PAIR_MAX_V.  Results are exact (same pairs as the reference) up to float64 ulp
 * differences of log10 / log2 at non-structural near-ties; at exact ties numpy's argsort order is
 * taken as stable (lower index first). */
int risvec_pair_noma(risvec_env_t* env, const risvec_pairing_t* cfg, const float* p01, int64_t p01_env_stride,
                     int topk, double tau_q, int recalc_mask, const int32_t* reuse, int decay, int new_episode,
                     void* stream);
/* start of an episode (:1282-1297): history, streak, thresholds, mask and frozen groups cleared */
int risvec_pair_reset(risvec_env_t* env, void* stream);
/* ... for the envs with env_mask [E] u8 (device) != 0 only (NULL = all) */
int risvec_pair_reset_masked(risvec_env_t* env, const uint8_t* env_mask, void* stream);

/* ---- episode starts per env (marl_train_bcd.py:1268-1332): the device-side work at the start of an episode ----
 * Stage bits; stages always run in this order.  The MARL driver runs all four (POSITIONS every
 * env_refresh_every-th episode), the SARL driver POSITIONS only. */
enum {
    RISVEC_EP_RESET = 1,     /* make_new_game                                              */
    RISVEC_EP_POSITIONS = 2, /* renew_positions + compute_parms                            */
    RISVEC_EP_CHANNEL = 4,   /* optimize_phase_shift + update_channel_gains                */
    RISVEC_EP_PAIRING = 8    /* pair_reset                                                 */
};
/* Every stage in `stages` for the envs whose stages_env [E] u8 (device) entry has its bit, in one call.
 * stages_env NULL = every env runs `stages`.  The host cannot read stages_env without a synchronisation, so the
 * kernel ANDs each entry with `stages` (bits outside `stages` are ignored); an env whose resulting bits are 0 keeps
 * every field bit for bit.  uniforms [E, n_uni] f64 / used_out [E] i32 as in risvec_renew_positions (rows of envs
 * that do not renew are ignored; their used_out is 0).  The draws are keyed like the separate calls and the host
 * call counter of every stage in `stages` advances as the separate calls would, so each env ends bit-identical to
 * running its stages as separate calls.  V <= 8, ncand <= 8, M <= 256 with the free channel runs as ONE launch
 * (k_begin_episode); other shapes run the separate kernels back to back, restricted to the selected envs.
 * RISVEC_ERR_INVALID for bits outside RISVEC_EP_*. */
int risvec_begin_episode(risvec_env_t* env, const uint8_t* stages_env, int stages, const double* uniforms, int n_uni,
                         int32_t* used_out, void* stream);

/* Fixed-length episodes of the reference driver; positions_every = env_refresh_every (marl_train_bcd.py:1268). */
typedef struct risvec_episode_schedule {
    int32_t steps_per_episode, positions_every, stages, _pad;
} risvec_episode_schedule_t;
/* The episode clock: call once per driver step, before the step.  For every env:
 *   start = (ep_step == 0); on start run `stages` (without POSITIONS unless ep_index % positions_every == 0);
 *   done = (ep_step == steps_per_episode - 1), the terminal flag of the transition this step stores;
 *   then ep_step += 1, and on wrap ep_step = 0, ep_index += 1.
 * start_out / done_out [E] u8 (device) may be NULL.  Nothing is decided on the host, so the call can be captured in
 * a CUDA graph.  Its draws are therefore keyed from device state, not from the host call counters (a graph freezes
 * kernel arguments): RNG kinds reset / mobility / channel of the tick, call = the env's ep_index.  They stay seeded
 * and independent of the sharding (global env index), differ per episode, and deliberately differ from the draws
 * of risvec_begin_episode; the host call counters do not move.  Injected uniforms do not apply.  Staggered
 * episodes: after make_new_game and one risvec_begin_episode for all envs, write per-env offsets into
 * RISVEC_F_EP_STEP (for example e % steps_per_episode). */
int risvec_episode_tick(risvec_env_t* env, const risvec_episode_schedule_t* schedule, uint8_t* start_out,
                        uint8_t* done_out, void* stream);

/* The driver's mask curriculum (batched.mask_schedule, marl_train_bcd.py:128-132,1323-1332); -1 selects the
 * driver defaults topk_start = V - 1, topk_end = max(4, V / 2). */
typedef struct risvec_pair_schedule {
    int32_t topk_start, topk_end, warmup_episodes, _pad;
    double tau_q_start, tau_q_end;
} risvec_pair_schedule_t;
/* risvec_pair_noma with per-env episode state: recalc_mask = new_episode = start[e] (start [E] u8, device), K_now /
 * q_now from the env's RISVEC_F_EP_INDEX and `schedule`; envs with start[e] == 0 run as the call with
 * recalc_mask = 0 and `reuse`.  Feed it the start_out of risvec_episode_tick. */
int risvec_pair_noma_episodes(risvec_env_t* env, const risvec_pairing_t* cfg, const float* p01, int64_t p01_env_stride,
                              const risvec_pair_schedule_t* schedule, const uint8_t* start, const int32_t* reuse,
                              int decay, void* stream);

/* ---- replay memory (SURVEY 8f row 4): Simulation-MARL-BCD/buffer.py, device resident ----
 * Same seven arrays as ReplayBuffer.__init__ (buffer.py:4-14): state / new_state [mem_size,
 * input_shape * n_agents] f32, action [mem_size, n_actions * n_agents] f32, reward_global [mem_size]
 * f32, reward_local [mem_size, n_agents] f32, terminal [mem_size] u8 (bool), mask [mem_size,
 * n_agents^2] f32; zero-filled at creation. */
typedef struct risvec_replay risvec_replay_t;
enum risvec_replay_field {
    RISVEC_RB_STATE = 0, RISVEC_RB_ACTION, RISVEC_RB_REWARD_G, RISVEC_RB_REWARD_L, RISVEC_RB_NEW_STATE,
    RISVEC_RB_TERMINAL, RISVEC_RB_MASK, RISVEC_RB_COUNT
};
int risvec_replay_create(int device, int64_t mem_size, int input_shape, int n_actions, int n_agents,
                         risvec_replay_t** out);
int risvec_replay_destroy(risvec_replay_t* rb);
int risvec_replay_field(risvec_replay_t* rb, int field, void** dev_ptr, int64_t* rows, int64_t* cols, int* elem_bytes);
int64_t risvec_replay_count(const risvec_replay_t* rb); /* mem_cntr */
int risvec_replay_set_count(risvec_replay_t* rb, int64_t mem_cntr); /* restore mem_cntr (checkpoint resume) */
/* store_transition (buffer.py:16-25) for E transitions at once: transition e goes to slot
 * (mem_cntr + e) % mem_size, then mem_cntr += E.  All pointers device; done [E] u8 may be NULL
 * (then done_all applies to every row); mask_flat [E, n_agents^2] f32 may be NULL (all ones, the
 * driver's choice when a step built no mask, marl_train_bcd.py:1786-1787). */
int risvec_replay_store(risvec_replay_t* rb, int E, const float* state, const float* action, const float* reward_g,
                        const float* reward_l, const float* state_, const uint8_t* done, int done_all,
                        const float* mask_flat, void* stream);
/* the same with the driver's assembly fused in (marl_train_bcd.py:1776-1790): action row = per agent
 * [intent_probs[i, :] with the diagonal zeroed (:1390) | power_raw[i, 0:2]] (n_actions must be
 * n_agents + 2); mask from the u8 RISVEC_F_PAIR_MASK layout [E, n_agents^2] (NULL: all ones). */
int risvec_replay_store_marl(risvec_replay_t* rb, int E, const float* state, const float* intent_probs,
                             const float* power_raw, const float* reward_g, const float* reward_l,
                             const float* state_, const uint8_t* done, int done_all, const uint8_t* mask_u8,
                             void* stream);
/* sample_buffer (buffer.py:27-39) for B caller-drawn slot indices idx [B] i64 (device), each in
 * [0, min(mem_cntr, mem_size)) (indices outside [0, mem_size) are clamped); outputs are [B, ...]
 * device arrays shaped like the fields. */
int risvec_replay_sample(risvec_replay_t* rb, int B, const int64_t* idx, float* states, float* actions,
                         float* rewards_g, float* rewards_l, float* states_, uint8_t* dones, float* masks,
                         void* stream);
/* Device-counter mode (opt-in): the ring counter lives on the device, in the handle's memory, and every store reads
 * and advances it there, so stores and draws can be captured in a CUDA graph and each replay lands in fresh slots.
 * risvec_replay_use_device_counter seeds the device counter from the host mem_cntr (a 1-thread launch on `stream`)
 * and returns its address (*dev_count, one int64; writing it moves the ring, a negative value counts as 0).  Call it
 * once, outside capture; a second call is refused.  From then on risvec_replay_store, risvec_replay_store_marl and
 * risvec_replay_set_count return RISVEC_ERR_INVALID and risvec_replay_count returns -1, so the two counters can
 * never silently diverge.  risvec_replay_sample (caller indices) keeps working: it does not read the counter. */
int risvec_replay_use_device_counter(risvec_replay_t* rb, int64_t** dev_count, void* stream);
/* risvec_replay_store / risvec_replay_store_marl with the count on the device: same arguments and checks, transition
 * e goes to slot (count + e) % mem_size, then count += E, all in one launch with no host decision (the last block to
 * finish advances the count).  RISVEC_ERR_INVALID on a handle not in device-counter mode. */
int risvec_replay_store_devcnt(risvec_replay_t* rb, int E, const float* state, const float* action,
                               const float* reward_g, const float* reward_l, const float* state_, const uint8_t* done,
                               int done_all, const float* mask_flat, void* stream);
int risvec_replay_store_marl_devcnt(risvec_replay_t* rb, int E, const float* state, const float* intent_probs,
                                    const float* power_raw, const float* reward_g, const float* reward_l,
                                    const float* state_, const uint8_t* done, int done_all, const uint8_t* mask_u8,
                                    void* stream);
/* sample_buffer with the count on the device: draws [B] i64 (device, uniform over [0, 2^62) for a uniform draw, read
 * as unsigned); row b is slot draws[b] % min(count, mem_size), so the modulo bias is below mem_size / 2^62.  With
 * count == 0 every row is slot 0 (all zeros until the first store), where buffer.py's np.random.choice(0, B) raises.
 * The randomness is the caller's: the library draws nothing.  Outputs as risvec_replay_sample. */
int risvec_replay_sample_devcnt(risvec_replay_t* rb, int B, const int64_t* draws, float* states, float* actions,
                                float* rewards_g, float* rewards_l, float* states_, uint8_t* dones, float* masks,
                                void* stream);

/* Episode statistics for the multi-GPU reduction: sums over this shard's E envs of the
 * RISVEC_F_STATS columns and of RISVEC_F_REWARD, written (accumulate = 0) or added (accumulate != 0)
 * to out [RISVEC_NSTAT + 1] f64 (device). */
int risvec_shard_stats(risvec_env_t* env, double* out, int accumulate, void* stream);

/* Statistics WITHOUT a separate pass per rollout.  `slots` = RISVEC_STAT_SLOTS (64) x 32 float64 (256-byte aligned,
 * zeroed by the caller), 17 used per slot.  Once attached, every risvec_rollout_sarl / _marl (their _host forms:
 * the last chunk; the fused driver steps too; not the packed-record entry points) adds the per-env statistics of its LAST step -- exactly what risvec_shard_stats would sum right
 * after it -- into the slots: the tensor-core rollouts (k_sarl_mma_tma, k_marl_tma) do it in their last instructions
 * (one float64 atomic per block and statistic, slot = block index % 64, so concurrent blocks hit different L2
 * lines); every other kernel is followed by one k_shard_stats launch into slot 0.  NULL detaches.
 * risvec_collect_stats: out[17] (+)= the sum over the slots, which are cleared (once per statistics interval). */
#define RISVEC_STAT_SLOTS 64
int risvec_attach_stats_accumulator(risvec_env_t* env, double* slots);
int risvec_collect_stats(risvec_env_t* env, double* slots, double* out, int accumulate, void* stream);

/* Per-episode statistics of staggered episodes: per-env running sums on the device and a log of completed episodes.
 * n_user = V for MARL, 0 for SARL.  All memory is owned by the caller.
 * running [E, RISVEC_EPLOG_RUN_COLS(n_user)] f64, zero-filled by the caller, one row per env:
 *   col 0 = steps accumulated, cols 1..16 = sums of the RISVEC_F_STATS columns, col 17 = sum of RISVEC_F_REWARD,
 *   cols 18.. = sums of RISVEC_F_REWARD_USER (MARL only).
 * records [capacity, RISVEC_EPLOG_REC_COLS(n_user)] f64: col 0 = global env index (env_index_base + e),
 *   col 1 = the env's RISVEC_F_STEP_CTR after the step, then the env's running row as it stood at its done step.
 * count: one u64 (device) = records claimed since the caller last zeroed it.
 * Call once after each driver step (T = 1).  For every env: the step's stats, reward and reward_user are converted to
 * float64 and added to its running row, and col 0 gains 1.  If done[e] != 0 (done NULL: done_all != 0; done is the
 * done_out of risvec_episode_tick for this step), the env claims slot k = count++, writes its record when
 * k < capacity, and its running row is zeroed.  A record with k >= capacity is dropped but still counted, so
 * count - capacity episodes were lost.  One launch, nothing decided on the host: the call can be captured in a CUDA
 * graph.  Slots are claimed in no fixed order across warps; sort the records by (step, env). */
#define RISVEC_EPLOG_RUN_COLS(n_user) (RISVEC_NSTAT + 2 + (n_user))
#define RISVEC_EPLOG_REC_COLS(n_user) (RISVEC_NSTAT + 4 + (n_user))
int risvec_episode_accumulate(risvec_env_t* env, double* running, const uint8_t* done, int done_all,
                              double* records, int64_t capacity, unsigned long long* count, void* stream);

/* Statistics reduction WITHOUT a collective (one node, NVLink / NVSwitch): one rank creates a small device buffer
 * and publishes its 64-byte CUDA IPC handle; every other rank (= process) maps it and passes the mapped pointer as
 * `out` of risvec_shard_stats(accumulate != 0).  k_shard_stats then adds the shard's sums into the owner's HBM with
 * float64 atomics over peer memory (or sums locally and pushes once per interval with risvec_shared_buffer_add):
 * no rank waits for another, nothing but 17 atomics per block / interval crosses NVLink;
 * the owner reads the totals after the job's own barrier.  (The portable alternative is an all-reduce of the
 * vector: ris_vec_marl_b200/dist.py.)  owner != 0 frees the buffer, owner == 0 unmaps it. */
int risvec_shared_buffer_create(int device, uint64_t bytes, void** dev_ptr, unsigned char ipc_handle[64]);
int risvec_shared_buffer_open(int device, const unsigned char ipc_handle[64], void** dev_ptr);
int risvec_shared_buffer_close(int device, void* dev_ptr, int owner);
/* dst[i] += src[i] (float64 atomics, i < n) on `stream`: a rank that sums its statistics locally over an interval
 * pushes them into the (peer-mapped) accumulator with ONE launch per interval. */
int risvec_shared_buffer_add(int device, double* dst, const double* src, int n, void* stream);

/* Host-side call counters that key the on-device Philox draws of make_new_game, renew_positions and the channel /
 * Random_phase draws (out / in = {reset, mobility, channel}).  Together with the RISVEC_F_* fields (which
 * include step_ctr, the key of the arrival draws) and the params they are the whole state of a handle:
 * a checkpoint that restores them continues the original random streams. */
int risvec_get_rng_counters(const risvec_env_t* env, uint64_t out[3]);
int risvec_set_rng_counters(risvec_env_t* env, const uint64_t in[3]);

/* number of kernels this handle has launched so far (bench.py reports it as gpu_launches) */
int64_t risvec_launch_count(const risvec_env_t* env);
/* name of the kernel(s) the latest risvec_rollout_* call on this handle launched ("k_sarl_mma_tma", "k_sarl_mma",
 * "k_sarl_umma", "k_sarl_mma_big", "k_sarl_v8", "k_sarl_rollout", "k_sarl_cascade2+k_sarl_scan", "k_marl_tma",
 * "k_marl_v8", "k_marl_rollout"; "" before the first rollout).  The choice follows the shape; RISVEC_SARL_PATH =
 * auto | mma | mma-ldg | mma-sync | v8 | generic (read at risvec_create) pins the SARL one for tests and A/B
 * measurements (mma-sync: the mma.sync kernel instead of the tcgen05 one for V > 8 or M > 64).  bench.py reports it
 * as roofline.kernel. */
const char* risvec_last_step_kernel(const risvec_env_t* env);

#ifdef __cplusplus
}
#endif
#endif /* RISVEC_H */
