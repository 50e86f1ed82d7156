"""Adapter: golden scenario inputs -> `BatchedEnviron` (the CUDA library through the C ABI).
Same interface as `tests.replay.OracleBackend`, so `tests.replay.replay` drives both."""
import contextlib
import os

import numpy as np
import torch

from ris_vec_marl_b200 import STAT_COLUMNS, BatchedEnviron, marl_yaml_overrides


def np64(t):
    return t.detach().to("cpu").numpy().astype(np.float64)


FAST_MARL_TRACES = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")


@contextlib.contextmanager
def kernel_paths(sarl=None, marl=None):
    """`with kernel_paths(sarl="v8"): env = BatchedEnviron("sarl", ...)` pins the rollout kernels of the handles
    created inside: risvec_create reads RISVEC_SARL_PATH = auto | mma | mma-ldg | mma-sync | v8 | generic and
    RISVEC_MARL_PATH (v8 keeps the MARL fast path on k_marl_v8).  A None path leaves its variable as it is."""
    paths = {k: v for k, v in (("RISVEC_SARL_PATH", sarl), ("RISVEC_MARL_PATH", marl)) if v is not None}
    old = {k: os.environ.get(k) for k in paths}
    os.environ.update(paths)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


class GpuBackend:
    """mode="fast": the shape-specialised kernels where they apply (k_sarl_v8 / k_marl_v8; the MARL
    one takes `last_*`, `last_power_W`, `over_power` from the state views, as the compat layer
    does).  mode="generic": RISVEC_FORCE_GENERIC=1, the shape-generic kernels with every trace."""

    def __init__(self, g, device=0, mode="fast"):
        over = marl_yaml_overrides() if (g["variant"] == "marl" and g["params"] == "yaml") else {}
        self.g, self.mode = g, mode
        old = os.environ.get("RISVEC_FORCE_GENERIC")
        os.environ["RISVEC_FORCE_GENERIC"] = "1" if mode == "generic" else "0"
        try:
            self.env = BatchedEnviron(g["variant"], g["E"], g["V"], g["M"], 3, device=device, **over)
        finally:
            if old is None:
                os.environ.pop("RISVEC_FORCE_GENERIC", None)
            else:
                os.environ["RISVEC_FORCE_GENERIC"] = old

    def make_new_game(self):
        g = self.g
        self.env.make_new_game(g["reset_ints"].astype(np.int32), g["reset_dirs"].astype(np.int32))

    def vehicles(self):
        e = self.env
        pos = np.stack([np64(e.pos_x), np64(e.pos_y)], axis=-1)
        return pos, e.dir.cpu().numpy().astype(np.int64), e.vel.cpu().numpy().astype(np.int64)

    def renew_positions(self, uniforms):
        return self.env.renew_positions(np.ascontiguousarray(uniforms)).cpu().numpy().astype(np.int64)

    def compute_parms(self):
        self.env.compute_parms()

    def geometry(self):
        return np64(self.env.dist), np64(self.env.angle)

    def optimize_phase_shift(self):
        self.env.optimize_phase_shift()

    def update_channel_gains(self):
        self.env.update_channel_gains()

    def gains(self):
        return np64(self.env.gains)

    def theta(self):
        return np64(self.env.theta_re) + 1j * np64(self.env.theta_im)

    def DataBuf(self):
        return np64(self.env.DataBuf)

    def mec_queue_cycles(self):
        return np64(self.env.mec_queue_cycles)

    def step_marl(self, actions, partner, ngroups, arrivals):
        e = self.env
        part, ng, arr = partner.astype(np.int32), np.asarray(ngroups, dtype=np.int32), arrivals.astype(np.int32)
        if self.mode == "fast" and e.V <= 8:
            r = e.step_marl(actions, part, ng, arr, traces=FAST_MARL_TRACES)
            out = {k: np64(r[k]) for k in FAST_MARL_TRACES}
            out["over_power"] = np64(e.over_power)
            out["last_power_W"] = np64(e.last_power_W)
            st = np64(e.stats)
            assert torch.equal(e.reward_user, r["reward_user"]) and torch.equal(e.reward, r["reward"])
        else:
            r = e.step_marl(actions, part, ng, arr, traces=FAST_MARL_TRACES + ("over_power", "stats", "last_power"))
            out = {k: np64(r[k]) for k in FAST_MARL_TRACES + ("over_power",)}
            out["last_power_W"] = np64(r["last_power"])
            st = np64(r["stats"])
            assert torch.equal(e.stats, r["stats"])
        for i, n in enumerate(STAT_COLUMNS):
            out["last_" + n] = st[:, i]
        # the state views must agree with the traces of the same step
        assert torch.equal(e.vehicle_rate, r["rate"]) and torch.equal(e.data_t, r["data_t"])
        return out

    def step_sarl(self, actions, phases, arrivals):
        r = self.env.step_sarl(actions, phases, arrivals.astype(np.int32),
                               traces=("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate"))
        assert torch.equal(self.env.over_data, r["over_data"])
        return {k: np64(v) for k, v in r.items()}
