"""ctypes binding of `librisvec.so` (C ABI declared in include/risvec.h).

There is deliberately no fallback: if the shared library is missing or cannot be loaded
the import of the product path fails loudly (`RisvecLibraryError`).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.environ.get("RISVEC_LIB") or os.path.join(PKG_DIR, "librisvec.so")  # override: A/B builds
SOURCES = ["risvec.cu"]
HEADERS = sorted(f for f in os.listdir(CSRC) if f.endswith(".cuh"))  # every one is a rebuild dependency
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "-shared", "-split-compile", "0"]

MAX_LANES = 8
NSTAT = 16
PARTNER_SINGLE, PARTNER_NONE, PARTNER_SECOND = -1, -2, 1 << 16
VARIANT = {"marl": 0, "sarl": 1}
CHANNEL = {"free": 0, "3gpp_umi": 1, "3gpp_uma": 2}

# packed record layout (include/risvec.h): words per (step, env) record, field order of the outputs
SARL_OUT_WORDS, MARL_IN_WORDS, MARL_OUT_WORDS = 48, 24, 40
SARL_OUT_FIELDS = ("DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
MARL_OUT_FIELDS = ("reward_user", "DataBuf", "data_t", "data_p", "rate")


def sarl_in_words(M):
    return 24 + M


# episode log (risvec_episode_accumulate): width of the per-env running row and of a completed-episode record
def eplog_run_cols(n_user):
    return NSTAT + 2 + n_user


def eplog_rec_cols(n_user):
    return NSTAT + 4 + n_user


STAT_COLUMNS = ("delay_mean", "energy_mean", "delay_local_mean", "delay_edge_q_mean", "delay_edge_c_mean",
                "t_tx_mean", "backlog_kbit_mean", "mec_utilization", "local_util_mean", "qos_violation",
                "off_kbit_sum", "local_kbit_sum", "mec_queue_cycles")

FIELDS = ("pos_x", "pos_y", "dir", "vel", "dist", "angle", "amp", "theta_re", "theta_im", "phase_real", "gains",
          "DataBuf", "data_t", "data_p", "over_data", "over_power", "vehicle_rate", "data_r", "reward_user",
          "reward", "mec_queue_cycles", "stats", "last_power_W", "step_ctr",
          "V2I_Shadowing", "pair_hist", "unpaired_streak", "pair_tau", "pair_k", "pair_mask", "pair_rounds",
          "noma_partner", "noma_ngroups", "noma_pairs", "noma_npairs", "ep_step", "ep_index")
PAIR_MAX_V = 12
# stage bits of risvec_begin_episode / risvec_episode_tick (RISVEC_EP_*), in the order the stages run
EP_STAGES = {"reset": 1, "positions": 2, "channel": 4, "pairing": 8}
REPLAY_FIELDS = ("state_memory", "action_memory", "reward_global_memory", "reward_local_memory", "new_state_memory",
                 "terminal_memory", "mask_memory")


class RisvecLibraryError(RuntimeError):
    pass


class RisvecError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"risvec error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    """Mirror of `risvec_params_t`."""

    _fields_ = [
        ("n_up", C.c_int32), ("n_down", C.c_int32), ("n_left", C.c_int32), ("n_right", C.c_int32),
        ("up_lanes", C.c_double * MAX_LANES), ("down_lanes", C.c_double * MAX_LANES),
        ("left_lanes", C.c_double * MAX_LANES), ("right_lanes", C.c_double * MAX_LANES),
        ("width", C.c_double), ("height", C.c_double),
        ("time_slow", C.c_double), ("time_fast", C.c_double), ("bandwidth", C.c_double), ("k", C.c_double),
        ("L", C.c_double), ("rate", C.c_double),
        ("data_buf_size", C.c_int32), ("channel_model", C.c_int32),
        ("noise_power", C.c_double), ("P_max", C.c_double), ("power_scale", C.c_double),
        ("f_local_max", C.c_double), ("f_edge_max", C.c_double), ("cycles_per_bit", C.c_double),
        ("cpu_share_floor", C.c_double),
        ("w_d", C.c_double), ("w_e", C.c_double), ("R_min_bpsHz", C.c_double), ("D_max_s", C.c_double),
        ("qos_penalty", C.c_double), ("reward_clip", C.c_double),
        ("qos_enable", C.c_int32), ("_pad0", C.c_int32),
        ("fc_GHz", C.c_double), ("shadow_std_los", C.c_double), ("shadow_std_nlos", C.c_double),
        ("rician_K_dB", C.c_double), ("veh_ant_gain", C.c_double),
        ("t_factor1", C.c_double), ("t_factor2", C.c_double), ("penalty1", C.c_double), ("penalty2", C.c_double),
    ]


class Pairing(C.Structure):
    """Mirror of `risvec_pairing_t` (knobs of the NOMA pairing stage, marl_train_bcd.py:435-441,1404-1498)."""

    _fields_ = [
        ("min_pair_target", C.c_int32), ("mwm_backoff_rounds", C.c_int32), ("relax_topk_step", C.c_int32),
        ("qos_enable", C.c_int32),
        ("mwm_accept_quantile", C.c_double), ("mwm_accept_q_step", C.c_double),
        ("completion_min_quantile", C.c_double),
        ("relax_tau_factor_per_round", C.c_double), ("tau_back_floor_db", C.c_double),
        ("score_w_delta_db", C.c_double), ("score_w_history", C.c_double), ("abs_gain_min_db", C.c_double),
        ("qos_soft_penalty_dbscore", C.c_double), ("pair_hist_decay", C.c_double),
    ]


class EpisodeSchedule(C.Structure):
    """Mirror of `risvec_episode_schedule_t`."""

    _fields_ = [("steps_per_episode", C.c_int32), ("positions_every", C.c_int32), ("stages", C.c_int32),
                ("_pad", C.c_int32)]


class PairSchedule(C.Structure):
    """Mirror of `risvec_pair_schedule_t` (the mask curriculum of `batched.mask_schedule`; -1 = driver default)."""

    _fields_ = [("topk_start", C.c_int32), ("topk_end", C.c_int32), ("warmup_episodes", C.c_int32), ("_pad", C.c_int32),
                ("tau_q_start", C.c_double), ("tau_q_end", C.c_double)]


class MarlOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate",
                                          "over_power", "stats", "last_power")]


class SarlOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")]


EXPORTS = {
    "risvec_abi_version": (C.c_int, []),
    "risvec_last_error": (C.c_char_p, []),
    "risvec_default_params": (C.c_int, [C.c_int, C.POINTER(Params)]),
    "risvec_create": (C.c_int, [C.POINTER(Params), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64,
                                C.c_int64, C.POINTER(C.c_void_p)]),
    "risvec_destroy": (C.c_int, [C.c_void_p]),
    "risvec_set_params": (C.c_int, [C.c_void_p, C.POINTER(Params)]),
    "risvec_get_params": (C.c_int, [C.c_void_p, C.POINTER(Params)]),
    "risvec_field": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                               C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "risvec_make_new_game": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "risvec_make_new_game_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                              C.c_void_p]),
    "risvec_pair_reset_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_renew_positions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "risvec_compute_parms": (C.c_int, [C.c_void_p, C.c_void_p]),
    "risvec_set_phase": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_optimize_phase_shift": (C.c_int, [C.c_void_p, C.c_void_p]),
    "risvec_update_channel_gains": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_rollout_marl": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.POINTER(MarlOut), C.c_void_p]),
    "risvec_rollout_sarl": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SarlOut),
                                      C.c_void_p]),
    "risvec_rollout_marl_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.POINTER(MarlOut), C.c_void_p]),
    "risvec_rollout_sarl_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.POINTER(SarlOut), C.c_void_p]),
    "risvec_rollout_sarl_packed": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_rollout_marl_packed": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "risvec_rollout_sarl_packed_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_void_p]),
    "risvec_rollout_marl_packed_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_observe": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_map_actions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_random_phase": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_direct_link": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_default_pairing": (C.c_int, [C.c_int, C.c_int, C.POINTER(Pairing)]),
    "risvec_pair_noma": (C.c_int, [C.c_void_p, C.POINTER(Pairing), C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_int,
                                   C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "risvec_pair_reset": (C.c_int, [C.c_void_p, C.c_void_p]),
    "risvec_begin_episode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "risvec_episode_tick": (C.c_int, [C.c_void_p, C.POINTER(EpisodeSchedule), C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_pair_noma_episodes": (C.c_int, [C.c_void_p, C.POINTER(Pairing), C.c_void_p, C.c_int64,
                                            C.POINTER(PairSchedule), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "risvec_replay_create": (C.c_int, [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "risvec_replay_destroy": (C.c_int, [C.c_void_p]),
    "risvec_replay_field": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "risvec_replay_count": (C.c_int64, [C.c_void_p]),
    "risvec_replay_store": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_void_p, C.c_void_p]),
    "risvec_replay_store_marl": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p, C.c_void_p]),
    "risvec_replay_sample": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_void_p]),
    "risvec_replay_use_device_counter": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]),
    "risvec_replay_store_devcnt": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_void_p,
                                                                                         C.c_void_p]),
    "risvec_replay_store_marl_devcnt": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 7 + [C.c_int, C.c_void_p,
                                                                                              C.c_void_p]),
    "risvec_replay_sample_devcnt": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_void_p]),
    "risvec_shard_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "risvec_step_marl_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_step_sarl_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "risvec_episode_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64,
                                            C.c_void_p, C.c_void_p]),
    "risvec_attach_stats_accumulator": (C.c_int, [C.c_void_p, C.c_void_p]),
    "risvec_collect_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "risvec_shared_buffer_create": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]),
    "risvec_shared_buffer_open": (C.c_int, [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    "risvec_shared_buffer_close": (C.c_int, [C.c_int, C.c_void_p, C.c_int]),
    "risvec_shared_buffer_add": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "risvec_get_rng_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "risvec_set_rng_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "risvec_replay_set_count": (C.c_int, [C.c_void_p, C.c_int64]),
    "risvec_launch_count": (C.c_int64, [C.c_void_p]),
    "risvec_last_step_kernel": (C.c_char_p, [C.c_void_p]),
}


def _stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(REPO_ROOT, "include", "risvec.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.isfile(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a with nvcc into `librisvec.so` (in-tree)."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC") or "nvcc"
    if not any(os.access(os.path.join(p, nvcc), os.X_OK) for p in os.environ.get("PATH", "").split(os.pathsep)) \
            and os.path.isfile("/usr/local/cuda/bin/nvcc"):
        nvcc = "/usr/local/cuda/bin/nvcc"
    cmd = [nvcc] + NVCC_FLAGS + ["-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RisvecLibraryError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return LIB_PATH


_LIB = None


def load_library():
    """dlopen `librisvec.so` and type every export.  No CUDA call is made here."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.isfile(LIB_PATH):
        raise RisvecLibraryError(
            f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as exc:
        raise RisvecLibraryError(f"cannot load {LIB_PATH}: {exc}") from exc
    for name, (res, args) in EXPORTS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise RisvecLibraryError(f"{LIB_PATH} does not export {name}") from exc
        fn.restype, fn.argtypes = res, args
    _LIB = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RisvecError(rc, load_library().risvec_last_error().decode("utf-8", "replace"))
