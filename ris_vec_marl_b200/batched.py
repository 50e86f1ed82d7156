"""`BatchedEnviron`: E independent reference `Environ` instances stepped on one B200.

Host-side mirror of the reference class (Simulation-MARL-BCD/Environment.py:56 and
Simulation-SARL/Environment.py:36) with the same method names; every method is one call
into the C ABI (include/risvec.h) and therefore one or a few sm_100a kernel launches.
PyTorch is used only for device memory, streams and (in `dist.py`) NCCL.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (CHANNEL, EP_STAGES, FIELDS, NSTAT, STAT_COLUMNS, VARIANT, EpisodeSchedule, MarlOut, Pairing,
                   PairSchedule, Params, SarlOut, check)

_PARAM_NAMES = {n for n, _ in Params._fields_} - {"_pad0"}
_PAIRING_NAMES = {n for n, _ in Pairing._fields_}
_LANE_FIELDS = ("up_lanes", "down_lanes", "left_lanes", "right_lanes")
MARL_TRACES = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate", "over_power", "stats", "last_power")
SARL_TRACES = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")


class _DevView:
    """Minimal `__cuda_array_interface__` holder so torch can alias library-owned memory."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


def default_params(variant: str) -> Params:
    p = Params()
    check(_lib.load_library().risvec_default_params(VARIANT[variant], C.byref(p)))
    return p


def default_pairing(n_veh: int, yaml: bool = False) -> Pairing:
    p = Pairing()
    check(_lib.load_library().risvec_default_pairing(int(n_veh), int(bool(yaml)), C.byref(p)))
    return p


def mask_schedule(i_episode: int, n_veh: int, topk_start=None, topk_end=None, tau_q_start=0.2, tau_q_end=0.4,
                  warmup_episodes=200):
    """(K_now, q_now) of the driver's mask curriculum (`_anneal_topk` marl_train_bcd.py:128-132 and
    :1323-1332).  Defaults are `Config.__init__` (:499-503); config.yaml uses 7, 7, 0.10, 0.25."""
    k_start = n_veh - 1 if topk_start is None else topk_start
    k_end = max(4, n_veh // 2) if topk_end is None else topk_end
    i = max(0, min(i_episode, warmup_episodes))
    k = round(k_end + (k_start - k_end) * (1.0 - i / max(1, warmup_episodes)))
    prog = min(1.0, i_episode / max(1, warmup_episodes))
    return int(min(max(k, 1), n_veh - 1)), float(tau_q_start + (tau_q_end - tau_q_start) * prog)


def marl_yaml_overrides() -> dict:
    """Values in force after marl_train_bcd.py:547-779 overlays config.yaml (SURVEY.md 8a)."""
    n0 = 10 ** ((-174 - 30) / 10)
    return dict(rate=1.0, f_local_max=3e9, f_edge_max=2e9, cycles_per_bit=300.0, k=1e-28, cpu_share_floor=0.10,
                P_max=2.0, bandwidth=5.0, noise_power=n0 * (5.0 * 1e6), power_scale=0.7, w_d=1.0, w_e=1.0,
                qos_enable=1, R_min_bpsHz=0.15, D_max_s=0.12, qos_penalty=1.5, reward_clip=50.0)


def encode_groups(noma_groups, V):
    """Ragged `noma_groups` of one env (Environment.py:339-370) -> (partner[V] int32, ngroups)."""
    partner = np.full(V, _lib.PARTNER_NONE, dtype=np.int32)
    for g in noma_groups:
        if len(g) == 1:
            partner[int(g[0])] = _lib.PARTNER_SINGLE
        elif len(g) == 2:
            partner[int(g[0])] = int(g[1])
            partner[int(g[1])] = int(g[0]) | _lib.PARTNER_SECOND
    return partner, len(noma_groups)


class BatchedEnviron:
    def __init__(self, variant, n_envs, n_veh=8, M=40, control_bit=3, device=0, seed=1234, env_index_base=0,
                 lanes=None, width=None, height=None, **param_overrides):
        if variant not in VARIANT:
            raise ValueError("variant must be 'marl' or 'sarl'")
        self._lib = _lib.load_library()  # raises if the CUDA library is absent: no fallback
        if not torch.cuda.is_available():
            raise _lib.RisvecLibraryError("no CUDA device: the batched env has no CPU path")
        self.variant, self.E, self.V, self.M = variant, int(n_envs), int(n_veh), int(M)
        self.control_bit = int(control_bit)
        self.device = torch.device("cuda", int(device))
        self.params = default_params(variant)
        if lanes is not None:
            for name, vals in zip(("down", "up", "left", "right"), lanes):
                self._set_lanes(name, vals)
        if width is not None:
            self.params.width = float(width)
        if height is not None:
            self.params.height = float(height)
        self._apply(param_overrides)
        h = C.c_void_p()
        check(self._lib.risvec_create(C.byref(self.params), VARIANT[variant], self.E, self.V, self.M, self.control_bit,
                                      self.device.index, int(seed), int(env_index_base), C.byref(h)))
        self._h = h
        self._views = {}
        for i, name in enumerate(FIELDS):
            ptr, rows, cols, eb, fl = C.c_void_p(), C.c_int64(), C.c_int64(), C.c_int(), C.c_int()
            check(self._lib.risvec_field(self._h, i, C.byref(ptr), C.byref(rows), C.byref(cols), C.byref(eb),
                                         C.byref(fl)))
            typestr = "|u1" if eb.value == 1 else ("<f" if fl.value else "<i") + str(eb.value)
            per_env_scalar = name in ("reward", "mec_queue_cycles", "step_ctr", "pair_tau", "pair_k", "pair_rounds",
                                      "noma_ngroups", "noma_npairs", "ep_step", "ep_index")
            shape = (rows.value,) if per_env_scalar else (rows.value, cols.value)
            self._views[name] = torch.as_tensor(_DevView(ptr.value, shape, typestr), device=self.device)
        self._views["last_power_W"] = self._views["last_power_W"].view(self.E, 2, self.V)
        for name in ("pair_hist", "pair_mask"):
            self._views[name] = self._views[name].view(self.E, self.V, self.V)
        self.pairing = default_pairing(self.V)

    # ------------------------------------------------------------------ params
    def _set_lanes(self, name, vals):
        vals = [float(v) for v in vals]
        if not 1 <= len(vals) <= _lib.MAX_LANES:
            raise ValueError("1..8 lanes per family")
        arr = getattr(self.params, name + "_lanes")
        for i, v in enumerate(vals):
            arr[i] = v
        setattr(self.params, "n_" + name, len(vals))

    def _apply(self, kw):
        for k, v in kw.items():
            if k == "channel_model" and isinstance(v, str):
                v = CHANNEL.get(v, 3)  # unknown keyword -> RISVEC_CHANNEL_UNKNOWN (Environment.py:315-317)
            if k not in _PARAM_NAMES or k in _LANE_FIELDS:
                raise AttributeError(f"unknown env parameter {k!r}")
            setattr(self.params, k, type(getattr(self.params, k))(v))

    def set_params(self, **kw):
        """Attribute writes of the reference drivers (marl_train_bcd.py:563-594,750-779)."""
        self._apply(kw)
        check(self._lib.risvec_set_params(self._h, C.byref(self.params)))

    def get_param(self, name):
        return getattr(self.params, name)

    # ------------------------------------------------------------------ helpers
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._views.clear()
            self._lib.risvec_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _dev(self, x, dtype, shape=None):
        if x is None:
            return None
        t = torch.as_tensor(x)
        if t.dtype != dtype or t.device != self.device or not t.is_contiguous():
            t = t.to(device=self.device, dtype=dtype).contiguous()
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        return t

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)

    def state(self, name):
        """Zero-copy torch view of a library-owned state field (see `_lib.FIELDS`)."""
        return self._views[name]

    def __getattr__(self, name):
        views = self.__dict__.get("_views")
        if views is not None and name in views:
            return views[name]
        raise AttributeError(name)

    @property
    def launch_count(self):
        return int(self._lib.risvec_launch_count(self._h))

    def last_kernel(self):
        """Name of the kernel(s) the latest rollout / step call launched (`risvec_last_step_kernel`)."""
        return self._lib.risvec_last_step_kernel(self._h).decode()

    # ------------------------------------------------------------------ reference methods
    def make_new_game(self, reset_ints=None, reset_dirs=None, mask=None):
        """`make_new_game` of every env, or -- `mask` [E] bool / u8 -- of the envs with mask != 0 only (the
        others keep every field: per-env episode restarts of a batched driver)."""
        ri = self._dev(reset_ints, torch.int32)
        rd = self._dev(reset_dirs, torch.int32)
        n_i = 0 if ri is None else ri.shape[1]
        n_d = 0 if rd is None or rd.numel() == 0 else rd.shape[1]
        if rd is not None and rd.numel() == 0:
            rd = None
        mk = None if mask is None else self._dev(torch.as_tensor(mask).to(torch.uint8), torch.uint8, (self.E,))
        check(self._lib.risvec_make_new_game_masked(self._h, self._p(mk), self._p(ri), n_i, self._p(rd), n_d, self.stream))

    def renew_positions(self, uniforms=None):
        u = self._dev(uniforms, torch.float64)
        used = torch.empty(self.E, dtype=torch.int32, device=self.device)
        n = 0 if u is None else u.shape[1]
        check(self._lib.risvec_renew_positions(self._h, self._p(u), n, self._p(used), self.stream))
        return used

    def compute_parms(self):
        check(self._lib.risvec_compute_parms(self._h, self.stream))

    def get_next_phase(self, action_phase):
        ph = self._dev(action_phase, torch.float32, (self.E, self.M))
        check(self._lib.risvec_set_phase(self._h, self._p(ph), self.stream))

    def Random_phase(self, indices=None):
        """`Random_phase` (MARL/Environment.py:203-206): quantised random RIS phases; `indices` [E,M]
        int32 injects the choices, None draws them on the device."""
        ix = self._dev(indices, torch.int32, (self.E, self.M))
        check(self._lib.risvec_random_phase(self._h, self._p(ix), self.stream))

    def get_path_loss(self):
        """`get_path_loss` (MARL/Environment.py:192-196) of every vehicle -> [E,V] float64 dB."""
        out = torch.empty(self.E, self.V, dtype=torch.float64, device=self.device)
        check(self._lib.risvec_direct_link(self._h, None, self._p(out), None, self.stream))
        return out

    def get_shadowing(self, normals=None):
        """`get_shadowing(delta_distance, vehicle)` (MARL/Environment.py:198-201) of every vehicle with
        `delta_distance = velocity * time_slow` (:410) -> [E,V] float64; `normals` [E,V] are the
        N(0, 8) draws (None: on-device Philox).  Reads the `V2I_Shadowing` state field."""
        nz = self._dev(normals, torch.float64, (self.E, self.V))
        out = torch.empty(self.E, self.V, dtype=torch.float64, device=self.device)
        check(self._lib.risvec_direct_link(self._h, self._p(nz), None, self._p(out), self.stream))
        return out

    def optimize_phase_shift(self):
        check(self._lib.risvec_optimize_phase_shift(self._h, self.stream))

    def update_channel_gains(self, chan_rand=None, chan_normal=None, chan_exp=None):
        r = self._dev(chan_rand, torch.float64)
        n = self._dev(chan_normal, torch.float64)
        x = self._dev(chan_exp, torch.float64)
        check(self._lib.risvec_update_channel_gains(self._h, self._p(r), self._p(n), self._p(x), self.stream))

    def get_channel_gains(self):
        return self._views["gains"]

    # ------------------------------------------------------------------ steps / rollouts
    def _trace_shape(self, name, T):
        E, V = self.E, self.V
        return {"reward": (T, E), "stats": (T, E, NSTAT), "last_power": (T, E, 2, V)}.get(name, (T, E, V))

    def _alloc_traces(self, names, T, all_names):
        out = {}
        for n in names:
            if n not in all_names:
                raise ValueError(f"unknown trace {n!r}")
            out[n] = torch.empty(self._trace_shape(n, T), dtype=torch.float32, device=self.device)
        return out

    @staticmethod
    def _check(name, t, dtype, shape, device):
        """A caller's tensor goes to the library as a raw pointer, and the library derives every extent it reads or
        writes from the handle's shape: refuse anything but a contiguous `dtype` tensor of exactly `shape` on
        `device`.  Never convert: a converted copy is not the buffer the caller reads the results from."""
        if (not isinstance(t, torch.Tensor) or tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != device
                or not t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {tuple(shape)} on {device}")

    def _check_out(self, out, T, all_names, device):
        """Preallocated traces: the names in `all_names`, each exactly the buffer `_alloc_traces` would make, but on
        `device`."""
        for k, v in out.items():
            if k not in all_names:
                raise ValueError(f"unknown trace {k!r}")
            self._check(f"out[{k!r}]", v, torch.float32, self._trace_shape(k, T), device)

    def rollout_marl(self, actions, partner, ngroups, arrivals=None, traces=MARL_TRACES, out=None):
        """T fused Environ.step calls; actions [T,E,2,V]; returns {trace: tensor [T,...]}.
        `out` may hold preallocated trace tensors (as made by `_alloc_traces`)."""
        a = self._dev(actions, torch.float32)
        T = a.shape[0]
        if tuple(a.shape) != (T, self.E, 2, self.V):
            raise ValueError(f"actions must be [T,{self.E},2,{self.V}]")
        pt = self._dev(partner, torch.int32, (self.E, self.V))
        ng = self._dev(ngroups, torch.int32, (self.E,))
        ar = self._dev(arrivals, torch.int32, (T, self.E, self.V)) if arrivals is not None else None
        if out is None:
            out = self._alloc_traces(traces, T, MARL_TRACES)
        else:
            self._check_out(out, T, MARL_TRACES, self.device)
        o = MarlOut(**{k: v.data_ptr() for k, v in out.items()})
        check(self._lib.risvec_rollout_marl(self._h, T, self._p(a), self._p(pt), self._p(ng), self._p(ar), C.byref(o),
                                            self.stream))
        return out

    def rollout_sarl(self, actions, phases, arrivals=None, traces=SARL_TRACES, out=None):
        a = self._dev(actions, torch.float32)
        T = a.shape[0]
        if tuple(a.shape) != (T, self.E, 2, self.V):
            raise ValueError(f"actions must be [T,{self.E},2,{self.V}]")
        ph = self._dev(phases, torch.float32, (T, self.E, self.M))
        ar = self._dev(arrivals, torch.int32, (T, self.E, self.V)) if arrivals is not None else None
        if out is None:
            out = self._alloc_traces(traces, T, SARL_TRACES)
        else:
            self._check_out(out, T, SARL_TRACES, self.device)
        o = SarlOut(**{k: v.data_ptr() for k, v in out.items()})
        check(self._lib.risvec_rollout_sarl(self._h, T, self._p(a), self._p(ph), self._p(ar), C.byref(o), self.stream))
        return out

    def step_marl(self, action, partner, ngroups, arrivals=None, traces=()):
        a = self._dev(action, torch.float32, (self.E, 2, self.V))
        ar = self._dev(arrivals, torch.int32, (self.E, self.V))[None] if arrivals is not None else None
        return {k: v[0] for k, v in self.rollout_marl(a[None], partner, ngroups, ar, traces).items()}

    def step_marl_fused(self, raw, partner, ngroups, arrivals=None, obs_out=None):
        """One driver step in one launch (SURVEY.md 8f row 1): `raw` = the actors' tanh outputs [E,V,2]; the action
        mapping (marl_train_bcd.py:1601-1608), Environ.step and marl_get_state (:819-827) of the new state.
        Returns the observation [E,V,5]; the step's results are the state views (`reward`, `reward_user`, ...)."""
        if self.variant != "marl":
            raise ValueError("step_marl_fused is the MARL driver step")
        r = self._dev(raw, torch.float32, (self.E, self.V, 2))
        pt = self._dev(partner, torch.int32, (self.E, self.V))
        ng = self._dev(ngroups, torch.int32, (self.E,))
        ar = self._dev(arrivals, torch.int32, (self.E, self.V)) if arrivals is not None else None
        if obs_out is None:
            obs_out = torch.empty(self.E, self.V, 5, dtype=torch.float32, device=self.device)
        elif obs_out.dtype != torch.float32 or tuple(obs_out.shape) != (self.E, self.V, 5) or not obs_out.is_contiguous() \
                or obs_out.device != self.device:
            raise ValueError(f"obs_out must be a contiguous float32 [{self.E},{self.V},5] tensor on {self.device}")
        check(self._lib.risvec_step_marl_fused(self._h, self._p(r), self._p(pt), self._p(ng), self._p(ar), self._p(obs_out),
                                               self.stream))
        return obs_out

    def step_sarl_fused(self, raw, arrivals=None, obs_out=None):
        """The SARL driver step in one launch: `raw` = the actor's tanh outputs [E, 2V+M]; the mapping of
        ddpg_train.py:151-160, Environ.step and get_state (:47-73) of the new state.  Returns the observation
        [E, V, M//V + 5]; the step's results are the state views."""
        if self.variant != "sarl":
            raise ValueError("step_sarl_fused is the SARL driver step")
        r = self._dev(raw, torch.float32, (self.E, 2 * self.V + self.M))
        ar = self._dev(arrivals, torch.int32, (self.E, self.V)) if arrivals is not None else None
        W = self.M // self.V + 5
        if obs_out is None:
            obs_out = torch.empty(self.E, self.V, W, dtype=torch.float32, device=self.device)
        elif obs_out.dtype != torch.float32 or tuple(obs_out.shape) != (self.E, self.V, W) or not obs_out.is_contiguous() \
                or obs_out.device != self.device:
            raise ValueError(f"obs_out must be a contiguous float32 [{self.E},{self.V},{W}] tensor on {self.device}")
        check(self._lib.risvec_step_sarl_fused(self._h, self._p(r), self._p(ar), self._p(obs_out), self.stream))
        return obs_out

    def step_sarl(self, action, phase, arrivals=None, traces=()):
        a = self._dev(action, torch.float32, (self.E, 2, self.V))
        ph = self._dev(phase, torch.float32, (self.E, self.M))
        ar = self._dev(arrivals, torch.int32, (self.E, self.V))[None] if arrivals is not None else None
        return {k: v[0] for k, v in self.rollout_sarl(a[None], ph[None], ar, traces).items()}

    # ---- host-buffer entry points (the end-to-end path: H2D + rollout + D2H on one stream)
    @staticmethod
    def _steps(t):
        """T of a [T, ...] host argument (None when `t` is no tensor: `_check` then refuses it)."""
        return t.shape[0] if isinstance(t, torch.Tensor) and t.dim() > 0 else None

    def rollout_sarl_host(self, actions, phases, arrivals, out):
        """`rollout_sarl` with CPU tensors (pinned for full copy speed): `actions` [T,E,2,V] f32, `phases` [T,E,M]
        f32, `arrivals` [T,E,V] i32 or None, and the `out` traces, all contiguous.  Other input is refused."""
        cpu, T = torch.device("cpu"), self._steps(actions)
        self._check("actions", actions, torch.float32, (T, self.E, 2, self.V), cpu)
        self._check("phases", phases, torch.float32, (T, self.E, self.M), cpu)
        if arrivals is not None:
            self._check("arrivals", arrivals, torch.int32, (T, self.E, self.V), cpu)
        self._check_out(out, T, SARL_TRACES, cpu)
        o = SarlOut(**{k: v.data_ptr() for k, v in out.items()})
        check(self._lib.risvec_rollout_sarl_host(self._h, T, self._p(actions), self._p(phases), self._p(arrivals),
                                                 C.byref(o), self.stream))

    def rollout_marl_host(self, actions, partner, ngroups, arrivals, out):
        """`rollout_marl` with CPU tensors (pinned for full copy speed): `actions` [T,E,2,V] f32, `partner` [E,V] i32,
        `ngroups` [E] i32, `arrivals` [T,E,V] i32 or None, and the `out` traces, all contiguous.  Other input is
        refused."""
        cpu, T = torch.device("cpu"), self._steps(actions)
        self._check("actions", actions, torch.float32, (T, self.E, 2, self.V), cpu)
        self._check("partner", partner, torch.int32, (self.E, self.V), cpu)
        self._check("ngroups", ngroups, torch.int32, (self.E,), cpu)
        if arrivals is not None:
            self._check("arrivals", arrivals, torch.int32, (T, self.E, self.V), cpu)
        self._check_out(out, T, MARL_TRACES, cpu)
        o = MarlOut(**{k: v.data_ptr() for k, v in out.items()})
        check(self._lib.risvec_rollout_marl_host(self._h, T, self._p(actions), self._p(partner), self._p(ngroups),
                                                 self._p(arrivals), C.byref(o), self.stream))

    # ---- packed record layout: the native streaming format for V == 8 (include/risvec.h)
    def pack_inputs(self, actions, arrivals, phases=None):
        """[T,E,2,8] f32 actions, [T,E,8] i32 arrivals (+ [T,E,M] f32 phases for SARL) -> the tiled
        record tensor [T, E/4, 4*W] f32 (arrivals bit-cast into their words).  Any device."""
        a = torch.as_tensor(actions, dtype=torch.float32)
        T, E = a.shape[0], a.shape[1]
        if E % 4 or a.shape[3] != 8:
            raise ValueError("packed records need E % 4 == 0 and V == 8")
        G = E // 4
        arr = torch.as_tensor(arrivals, dtype=torch.int32).to(a.device).view(torch.float32)
        parts = [a[:, :, 0, :].reshape(T, G, 32), a[:, :, 1, :].reshape(T, G, 32), arr.reshape(T, G, 32)]
        if self.variant == "sarl":
            parts.append(torch.as_tensor(phases, dtype=torch.float32).to(a.device).reshape(T, G, 4 * self.M))
        return torch.cat(parts, dim=2).contiguous()

    def unpack_outputs(self, out_rec, reward):
        """[T, E/4, 4*W] output tiles -> {trace: [T,E,8]} (+ reward), names as the per-array API."""
        names = _lib.SARL_OUT_FIELDS if self.variant == "sarl" else _lib.MARL_OUT_FIELDS
        T, G = out_rec.shape[0], out_rec.shape[1]
        d = {n: out_rec[:, :, 32 * i:32 * i + 32].reshape(T, G * 4, 8) for i, n in enumerate(names)}
        d["reward"] = reward
        return d

    def packed_out_words(self):
        return _lib.SARL_OUT_WORDS if self.variant == "sarl" else _lib.MARL_OUT_WORDS

    def rollout_packed(self, in_rec, partner=None, ngroups=None, out_rec=None, reward=None):
        """One fused rollout on device-resident packed records; returns (out_rec, reward)."""
        rec = self._dev(in_rec, torch.float32)
        T = rec.shape[0]
        if out_rec is None:
            out_rec = torch.empty(T, self.E // 4, 4 * self.packed_out_words(), dtype=torch.float32, device=self.device)
        if reward is None:
            reward = torch.empty(T, self.E, dtype=torch.float32, device=self.device)
        if self.variant == "sarl":
            if rec.numel() != T * self.E * _lib.sarl_in_words(self.M):
                raise ValueError("SARL input tiles must be [T,E/4,4*(24+M)]")
            check(self._lib.risvec_rollout_sarl_packed(self._h, T, self._p(rec), self._p(out_rec), self._p(reward),
                                                       self.stream))
        else:
            if rec.numel() != T * self.E * _lib.MARL_IN_WORDS:
                raise ValueError("MARL input tiles must be [T,E/4,4*24]")
            pt = self._dev(partner, torch.int32, (self.E, self.V))
            ng = self._dev(ngroups, torch.int32, (self.E,))
            check(self._lib.risvec_rollout_marl_packed(self._h, T, self._p(rec), self._p(pt), self._p(ng),
                                                       self._p(out_rec), self._p(reward), self.stream))
        return out_rec, reward

    def rollout_packed_host(self, in_rec, out_rec, reward, partner=None, ngroups=None):
        """Same with CPU tensors (pinned for full copy speed), all contiguous f32 unless noted: `in_rec`
        [T, E/4, 4*W_in], `out_rec` [T, E/4, 4*W_out], `reward` [T, E]; MARL also `partner` [E,V] i32 and `ngroups`
        [E] i32.  Other input is refused.  Chunked H2D -> rollout -> D2H pipeline."""
        cpu, T, G = torch.device("cpu"), self._steps(in_rec), self.E // 4
        w_in = _lib.sarl_in_words(self.M) if self.variant == "sarl" else _lib.MARL_IN_WORDS
        self._check("in_rec", in_rec, torch.float32, (T, G, 4 * w_in), cpu)
        self._check("out_rec", out_rec, torch.float32, (T, G, 4 * self.packed_out_words()), cpu)
        self._check("reward", reward, torch.float32, (T, self.E), cpu)
        if self.variant == "sarl":
            check(self._lib.risvec_rollout_sarl_packed_host(self._h, T, self._p(in_rec), self._p(out_rec),
                                                            self._p(reward), self.stream))
        else:
            self._check("partner", partner, torch.int32, (self.E, self.V), cpu)
            self._check("ngroups", ngroups, torch.int32, (self.E,), cpu)
            check(self._lib.risvec_rollout_marl_packed_host(self._h, T, self._p(in_rec), self._p(partner),
                                                            self._p(ngroups), self._p(out_rec), self._p(reward),
                                                            self.stream))

    # ---- driver-side glue on device (SURVEY.md 8f row 1)
    def observe(self, out=None):
        """Per-agent observations [E, V, W]: MARL W = 5 (marl_train_bcd.py:819-827), SARL
        W = M // V + 5 with the agent's RIS phase slice first (ddpg_train.py:47-73)."""
        W = (self.M // self.V if self.variant == "sarl" else 0) + 5
        if out is None:
            out = torch.empty(self.E, self.V, W, dtype=torch.float32, device=self.device)
        check(self._lib.risvec_observe(self._h, self._p(out), self.stream))
        return out

    def map_actions(self, raw):
        """Raw policy outputs in [-1, 1] -> env actions.  MARL: raw [E,V,2] -> action [E,2,V]
        (marl_train_bcd.py:1601-1608); SARL: raw [E,2V+M] -> (action [E,2,V], phase [E,M])
        (ddpg_train.py:151-160)."""
        r = self._dev(raw, torch.float32)
        act = torch.empty(self.E, 2, self.V, dtype=torch.float32, device=self.device)
        if self.variant == "marl":
            check(self._lib.risvec_map_actions(self._h, self._p(r), self._p(act), self._p(None), self.stream))
            return act
        ph = torch.empty(self.E, self.M, dtype=torch.float32, device=self.device)
        check(self._lib.risvec_map_actions(self._h, self._p(r), self._p(act), self._p(ph), self.stream))
        return act, ph

    # ------------------------------------------------------------------ stats / checkpoint
    def last_stats(self):
        """{name: tensor [E]} of the reference's `last_*` attributes after the latest step."""
        st = self._views["stats"]
        return {n: st[:, i] for i, n in enumerate(STAT_COLUMNS)}

    # ------------------------------------------------------------------ NOMA pairing (driver stage)
    def set_pairing(self, yaml=False, **kw):
        """Pairing knobs (`risvec_pairing_t`); `yaml=True` starts from the shipped config.yaml overlay."""
        if yaml:
            self.pairing = default_pairing(self.V, yaml=True)
        for k, v in kw.items():
            if k not in _PAIRING_NAMES:
                raise AttributeError(f"unknown pairing parameter {k!r}")
            setattr(self.pairing, k, type(getattr(self.pairing, k))(v))

    def pair_reset(self, mask=None):
        """Start of an episode (marl_train_bcd.py:1282-1297); `mask` [E]: only the envs with mask != 0."""
        mk = None if mask is None else self._dev(torch.as_tensor(mask).to(torch.uint8), torch.uint8, (self.E,))
        check(self._lib.risvec_pair_reset_masked(self._h, self._p(mk), self.stream))

    def pair_noma(self, p01, topk, tau_q, recalc_mask=True, reuse=None, decay=True, new_episode=False):
        """One driver step of the pairing stage (marl_train_bcd.py:1315-1561) for every env.

        `p01`: offload power in [0,1], either [E,V] or the env action [E,2,V] (row 0 is used).
        `topk`, `tau_q`: K_now / q_now of the mask curriculum (`mask_schedule`).  `new_episode=True`
        makes the call the first step of an episode (`pair_reset` folded into the same launch).  Returns the
        zero-copy views `(noma_partner [E,V], noma_ngroups [E])` to hand to `rollout_marl`."""
        t = self._dev(p01, torch.float32)
        if tuple(t.shape) == (self.E, 2, self.V):
            stride = 2 * self.V
        elif tuple(t.shape) == (self.E, self.V):
            stride = self.V
        else:
            raise ValueError(f"p01 must be [E,V] or [E,2,V], got {tuple(t.shape)}")
        ru = self._dev(reuse, torch.int32, (self.E,))
        check(self._lib.risvec_pair_noma(self._h, C.byref(self.pairing), self._p(t), stride, int(topk), float(tau_q),
                                         int(bool(recalc_mask)), self._p(ru), int(bool(decay)), int(bool(new_episode)),
                                         self.stream))
        return self._views["noma_partner"], self._views["noma_ngroups"]

    # ------------------------------------------------------------------ episodes per env
    @staticmethod
    def _stage_bits(stages):
        if isinstance(stages, int):
            return stages
        bits = 0
        for st in stages:
            if st not in EP_STAGES:
                raise ValueError(f"unknown episode stage {st!r} (one of {tuple(EP_STAGES)})")
            bits |= EP_STAGES[st]
        return bits

    def begin_episode(self, stages=("positions", "channel", "pairing"), per_env=None, uniforms=None):
        """The device-side work at the start of an episode (marl_train_bcd.py:1268-1309), for every env or -- `per_env`
        [E] u8 of `EP_STAGES` bits -- for each env the stages its entry selects (AND-ed with `stages`).  Stages run in
        the order reset, positions, channel, pairing; each env ends bit-identical to running its stages as the separate
        calls (`make_new_game`, `renew_positions` + `compute_parms`, `optimize_phase_shift` + `update_channel_gains`,
        `pair_reset`).  One launch for V <= 8 with the free channel.  `uniforms` [E, n] as in `renew_positions`.
        Returns `used` [E] int32 when positions are renewed, else None.

        Staggered episodes: `make_new_game()`, then one `begin_episode()` for all envs, then write per-env offsets into
        `env.ep_step` (for example `torch.arange(E) % 100`); from then on `episode_tick` runs the starts."""
        bits = self._stage_bits(stages)
        pe = None if per_env is None else self._dev(torch.as_tensor(per_env).to(torch.uint8), torch.uint8, (self.E,))
        u = self._dev(uniforms, torch.float64)
        n = 0 if u is None else u.shape[1]
        used = torch.empty(self.E, dtype=torch.int32, device=self.device) if bits & EP_STAGES["positions"] else None
        check(self._lib.risvec_begin_episode(self._h, self._p(pe), bits, self._p(u), n, self._p(used), self.stream))
        return used

    def episode_tick(self, steps_per_episode=100, positions_every=5, stages=("positions", "channel", "pairing"),
                     out=None):
        """The per-env episode clock; call once per driver step, before the step.  Envs with `ep_step == 0` start an
        episode and run `stages` (positions only when `ep_index % positions_every == 0`, the driver's
        env_refresh_every); `done` flags the last step of an episode (the terminal of the transition stored this
        step); then the clock advances.  Returns `(start, done)` u8 [E]; pass the previous result as `out` to reuse its
        buffers (a CUDA graph capture needs fixed buffers).  The draws are keyed by the env's episode index, not by
        host counters, so a captured graph draws fresh numbers every episode (they differ from `begin_episode`'s)."""
        sch = EpisodeSchedule(int(steps_per_episode), int(positions_every), self._stage_bits(stages), 0)
        if out is None:
            out = (torch.empty(self.E, dtype=torch.uint8, device=self.device),
                   torch.empty(self.E, dtype=torch.uint8, device=self.device))
        start, done = out
        for t in (start, done):
            if t.dtype != torch.uint8 or tuple(t.shape) != (self.E,) or t.device != self.device or not t.is_contiguous():
                raise ValueError(f"out must hold two contiguous uint8 [{self.E}] tensors on {self.device}")
        check(self._lib.risvec_episode_tick(self._h, C.byref(sch), self._p(start), self._p(done), self.stream))
        return start, done

    def pair_noma_episodes(self, p01, start, schedule=(None, None, 0.2, 0.4, 200), reuse=None, decay=True):
        """`pair_noma` with per-env episode state: envs with `start` [E] != 0 build the mask and solve as the first step
        of an episode, with K_now / q_now of `mask_schedule(env.ep_index[e], ...)`; the others run the non-recalc step
        with `reuse`.  `schedule` = (topk_start, topk_end, tau_q_start, tau_q_end, warmup_episodes), None = driver
        default (config.yaml: 7, 7, 0.10, 0.25, 200).  Returns the views `(noma_partner, noma_ngroups)`."""
        t = self._dev(p01, torch.float32)
        if tuple(t.shape) == (self.E, 2, self.V):
            stride = 2 * self.V
        elif tuple(t.shape) == (self.E, self.V):
            stride = self.V
        else:
            raise ValueError(f"p01 must be [E,V] or [E,2,V], got {tuple(t.shape)}")
        st = self._dev(start, torch.uint8, (self.E,))
        ru = self._dev(reuse, torch.int32, (self.E,))
        k0, k1, q0, q1, warm = schedule
        sch = PairSchedule(-1 if k0 is None else int(k0), -1 if k1 is None else int(k1), int(warm), 0, float(q0), float(q1))
        check(self._lib.risvec_pair_noma_episodes(self._h, C.byref(self.pairing), self._p(t), stride, C.byref(sch),
                                                  self._p(st), self._p(ru), int(bool(decay)), self.stream))
        return self._views["noma_partner"], self._views["noma_ngroups"]

    def shard_stats(self, out=None, accumulate=False):
        """f64 [NSTAT + 1] sums over this shard's envs (stats columns, then global reward);
        with `out` given the sums are written into it (or added, `accumulate=True`)."""
        if out is None:
            out = torch.empty(NSTAT + 1, dtype=torch.float64, device=self.device)
            accumulate = False
        check(self._lib.risvec_shard_stats(self._h, self._p(out), 1 if accumulate else 0, self.stream))
        return out

    def attach_stats_accumulator(self, attach=True):
        """From now on every `rollout_sarl` / `rollout_marl` (and `_host`) call adds the statistics of its last step --
        what `shard_stats` would sum right after it -- into a device accumulator: no separate pass per rollout
        (the tensor-core rollouts do it in their last instructions).  `collect_stats()` returns and clears the sums."""
        if attach:
            self._stat_slots = torch.zeros(64, 32, dtype=torch.float64, device=self.device)
            check(self._lib.risvec_attach_stats_accumulator(self._h, self._p(self._stat_slots)))
        else:
            check(self._lib.risvec_attach_stats_accumulator(self._h, self._p(None)))
            self._stat_slots = None

    def collect_stats(self, out=None, accumulate=False):
        """f64 [NSTAT + 1] sums accumulated since the last collect (written or, `accumulate=True`, added to `out`)."""
        if getattr(self, "_stat_slots", None) is None:
            raise RuntimeError("attach_stats_accumulator() first")
        if out is None:
            out = torch.empty(NSTAT + 1, dtype=torch.float64, device=self.device)
            accumulate = False
        check(self._lib.risvec_collect_stats(self._h, self._p(self._stat_slots), self._p(out), 1 if accumulate else 0, self.stream))
        return out

    def state_dict(self):
        """Everything a resumed run needs to CONTINUE this one: the state arena, the host-side call counters
        that key the on-device Philox draws, the scalar parameters and the pairing knobs."""
        ctr = (C.c_uint64 * 3)()
        check(self._lib.risvec_get_rng_counters(self._h, ctr))
        sd = {k: v.clone() for k, v in self._views.items()}
        sd["_rng_counters"] = [int(x) for x in ctr]
        sd["_params"] = bytes(self.params)
        sd["_pairing"] = bytes(self.pairing)
        return sd

    def load_state_dict(self, sd):
        for k, v in sd.items():
            if not k.startswith("_"):
                self._views[k].copy_(v.to(self.device))
        if "_rng_counters" in sd:
            check(self._lib.risvec_set_rng_counters(self._h, (C.c_uint64 * 3)(*sd["_rng_counters"])))
        if "_params" in sd:
            C.memmove(C.byref(self.params), sd["_params"], C.sizeof(Params))
            check(self._lib.risvec_set_params(self._h, C.byref(self.params)))
        if "_pairing" in sd:
            C.memmove(C.byref(self.pairing), sd["_pairing"], C.sizeof(Pairing))
