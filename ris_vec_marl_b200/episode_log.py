"""`EpisodeLog`: per-episode statistics of a batched driver whose envs run staggered episodes.

Each env keeps running float64 sums of its per-step `stats`, `reward` and (MARL) `reward_user` on the device; when its
episode ends, the sums go into a device-side log as one record (`risvec_episode_accumulate`).  The host reads the log
once per logging interval with `drain()`.  The buffers are fixed at construction, so `accumulate` can be captured in a
CUDA graph next to `episode_tick` and the fused step."""
from __future__ import annotations

import numpy as np
import torch

from ._lib import NSTAT, STAT_COLUMNS, check, eplog_rec_cols, eplog_run_cols


class EpisodeLog:
    """Running sums `running` [E, C] f64 (one row per env), completed-episode records `records` [capacity, C + 2] f64
    and the record counter `count` (one u64, held as int64), all on `env.device`.  C = `eplog_run_cols(n_user)`,
    n_user = V for MARL and 0 for SARL (include/risvec.h documents the columns)."""

    def __init__(self, env, capacity=65536):
        if int(capacity) < 1:
            raise ValueError("capacity must be >= 1")
        self.env, self.capacity = env, int(capacity)
        self.n_user = env.V if env.variant == "marl" else 0
        dev = env.device
        self.running = torch.zeros(env.E, eplog_run_cols(self.n_user), dtype=torch.float64, device=dev)
        self.records = torch.zeros(self.capacity, eplog_rec_cols(self.n_user), dtype=torch.float64, device=dev)
        self.count = torch.zeros(1, dtype=torch.int64, device=dev)

    def accumulate(self, done):
        """Add this step's statistics to every env's sums and log the envs whose episode ended: `done` is the [E]
        uint8 / bool device tensor of `episode_tick` for this step, or a python bool for every env (lock-step
        episodes).  One launch.  Any other `done` is refused, never converted: a converted copy would be a new buffer
        at every call, which a captured graph cannot follow."""
        env = self.env
        if isinstance(done, bool):
            d, d_all = None, int(done)
        else:
            if (not isinstance(done, torch.Tensor) or done.dtype not in (torch.uint8, torch.bool)
                    or tuple(done.shape) != (env.E,) or done.device != env.device or not done.is_contiguous()):
                raise ValueError(f"done must be a python bool or a contiguous uint8 / bool tensor of shape ({env.E},) "
                                 f"on {env.device}")
            d, d_all = done, 0
        check(env._lib.risvec_episode_accumulate(env._h, env._p(self.running), env._p(d), d_all, env._p(self.records),
                                                 self.capacity, env._p(self.count), env.stream))

    def drain(self):
        """Synchronise and return the episodes completed since the last drain, sorted by (step, env), then clear the
        log.  Keys: `env`, `step`, `length` int64 [n]; `stats` {STAT_COLUMNS name: float64 [n]} (episode sums);
        `reward` float64 [n]; `reward_user` float64 [n, V] (MARL); `dropped`: episodes that found the log full."""
        n = int(self.count.item())
        kept = min(n, self.capacity)
        rec = self.records[:kept].cpu().numpy()
        self.count.zero_()
        rec = rec[np.lexsort((rec[:, 0], rec[:, 1]))]
        out = {"env": rec[:, 0].astype(np.int64), "step": rec[:, 1].astype(np.int64),
               "length": rec[:, 2].astype(np.int64),
               "stats": {name: rec[:, 3 + i].copy() for i, name in enumerate(STAT_COLUMNS)},
               "reward": rec[:, 3 + NSTAT].copy(), "dropped": n - kept}
        if self.n_user:
            out["reward_user"] = rec[:, 4 + NSTAT:].copy()
        return out

    def state_dict(self):
        """The running sums, the records not yet drained and the counter: a resumed run continues the log."""
        n = int(self.count.item())
        return {"running": self.running.clone(), "records": self.records[:min(n, self.capacity)].clone(), "count": n}

    def load_state_dict(self, sd):
        rec = sd["records"]
        if (tuple(sd["running"].shape) != tuple(self.running.shape) or rec.dim() != 2
                or rec.shape[1] != self.records.shape[1] or rec.shape[0] > self.capacity):
            raise ValueError("state dict of an episode log of another shape or a larger capacity")
        self.running.copy_(sd["running"].to(self.env.device))
        self.records[:sd["records"].shape[0]].copy_(sd["records"].to(self.env.device))
        self.count.fill_(int(sd["count"]))
