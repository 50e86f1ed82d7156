"""Device-resident `ReplayBuffer` with the reference's interface (Simulation-MARL-BCD/buffer.py),
batched over envs: `store_transitions` writes E transitions per call through `librisvec.so`."""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib
from ._lib import REPLAY_FIELDS, check
from .batched import _DevView


class ReplayBuffer:
    """`ReplayBuffer(max_size, input_shape, n_actions, n_agents)` (buffer.py:4).  The seven
    `*_memory` arrays are zero-copy torch views of library-owned device memory; `mem_cntr` counts
    stored transitions as in the reference.

    `device_counter=True` keeps that count on the device instead of the host: `count` is a zero-copy int64 [1] view
    of it, every store reads and advances it in its one kernel, and a draw without `idx` reads it there too.  Stores
    and draws then decide nothing on the host, so a CUDA graph can capture them (each replay writes the next slots
    and samples the current fill level).  In that mode the stores refuse, never convert, tensors that are not ready
    for the kernel (see `store_transitions`)."""

    def __init__(self, max_size, input_shape, n_actions, n_agents, device=0, device_counter=False):
        self._lib = _lib.load_library()
        if not torch.cuda.is_available():
            raise _lib.RisvecLibraryError("no CUDA device: the replay memory has no CPU path")
        self.mem_size, self.n_agents = int(max_size), int(n_agents)
        self.input_shape, self.n_actions = int(input_shape), int(n_actions)
        self.device = torch.device("cuda", int(device))
        h = C.c_void_p()
        check(self._lib.risvec_replay_create(self.device.index, self.mem_size, self.input_shape, self.n_actions,
                                             self.n_agents, C.byref(h)))
        self._h = h
        for i, name in enumerate(REPLAY_FIELDS):
            ptr, rows, cols, eb = C.c_void_p(), C.c_int64(), C.c_int64(), C.c_int()
            check(self._lib.risvec_replay_field(self._h, i, C.byref(ptr), C.byref(rows), C.byref(cols), C.byref(eb)))
            shape = (rows.value,) if cols.value == 1 else (rows.value, cols.value)
            t = torch.as_tensor(_DevView(ptr.value, shape, "|u1" if eb.value == 1 else "<f4"), device=self.device)
            setattr(self, name, t.view(torch.bool) if eb.value == 1 else t)
        self.device_counter, self.count = bool(device_counter), None
        if self.device_counter:
            ptr = C.c_void_p()
            check(self._lib.risvec_replay_use_device_counter(self._h, C.byref(ptr), self._stream))
            self.count = torch.as_tensor(_DevView(ptr.value, (1,), "<i8"), device=self.device)

    @property
    def mem_cntr(self):
        """Transitions stored so far.  With `device_counter=True` this reads `count` back, which waits for the work
        queued on the current stream: keep it out of a loop that should not synchronise."""
        if self.device_counter:
            return int(self.count.item())
        return int(self._lib.risvec_replay_count(self._h))

    def state_dict(self):
        return {**{n: getattr(self, n).clone() for n in REPLAY_FIELDS}, "_mem_cntr": self.mem_cntr}

    def load_state_dict(self, sd):
        """Restore the seven arrays and the count.  The count is a plain number, so a state dict saved with either
        counter mode loads into either; one of another shape is refused."""
        for n in REPLAY_FIELDS:
            if tuple(sd[n].shape) != tuple(getattr(self, n).shape):
                raise ValueError(f"state dict of a replay memory of another shape: {n} is {tuple(sd[n].shape)}, "
                                 f"this buffer's is {tuple(getattr(self, n).shape)}")
        if self.device_counter and int(sd["_mem_cntr"]) < 0:
            raise ValueError("negative _mem_cntr")
        for n in REPLAY_FIELDS:
            getattr(self, n).copy_(sd[n].to(self.device))
        if self.device_counter:
            self.count.fill_(int(sd["_mem_cntr"]))
        else:
            check(self._lib.risvec_replay_set_count(self._h, int(sd["_mem_cntr"])))

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _f(self, x, shape, dtype=torch.float32):
        if x is None:
            return None
        t = torch.as_tensor(x)
        if t.dtype != dtype or t.device != self.device or not t.is_contiguous():
            t = t.to(device=self.device, dtype=dtype).contiguous()
        if t.numel() != int(torch.Size(shape).numel()):
            raise ValueError(f"expected {tuple(shape)} elements, got {tuple(t.shape)}")
        return t

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)

    def _done(self, done, E):
        if isinstance(done, (bool, int)):
            return None, int(bool(done))
        return self._f(done, (E,), torch.uint8 if torch.as_tensor(done).dtype != torch.bool else torch.bool), 0

    def _exact(self, x, name, E, row, dtype=torch.float32):
        """Device-counter mode: `x` itself if it is a contiguous `dtype` tensor on the buffer's device of shape
        (E, *row) or (E, prod(row)), else ValueError.  Never a converted copy: that would be a new buffer at every
        call, which a captured graph cannot follow."""
        if x is None:
            return None
        shapes = {(E, *row), (E, math.prod(row))} if row else {(E,)}
        if (not isinstance(x, torch.Tensor) or x.dtype != dtype or x.device != self.device or not x.is_contiguous()
                or tuple(x.shape) not in shapes):
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape "
                             f"{' or '.join(str(s) for s in sorted(shapes))} on {self.device} "
                             "(a buffer with device_counter=True converts nothing)")
        return x

    def _done_exact(self, done, E):
        if isinstance(done, bool):
            return None, int(done)
        if not isinstance(done, torch.Tensor) or done.dtype not in (torch.uint8, torch.bool):
            raise ValueError(f"done must be a python bool or a contiguous uint8 / bool tensor of shape ({E},) on "
                             f"{self.device}")
        return self._exact(done, "done", E, (), done.dtype).view(torch.uint8), 0

    def _rows(self, reward_g):
        """E of a device-counter store, from `reward_g` [E] (anything else is refused by `_exact`)"""
        return reward_g.shape[0] if isinstance(reward_g, torch.Tensor) and reward_g.dim() == 1 else -1

    def store_transitions(self, state, action, reward_g, reward_l, state_, done, mask_flat=None):
        """`store_transition` (buffer.py:16-25) for E transitions: row e -> slot (mem_cntr + e) % mem_size.

        With `device_counter=True` every tensor must already be contiguous, on the buffer's device, float32, of shape
        (E, width) or (E, n_agents, width / n_agents) -- `reward_g` (E,) -- and `done` a python bool or an (E,)
        uint8 / bool device tensor such as the `done` of `BatchedEnviron.episode_tick`; anything else raises
        ValueError and launches nothing."""
        N, S, A = self.n_agents, self.input_shape * self.n_agents, self.n_actions * self.n_agents
        if self.device_counter:
            E = self._rows(reward_g)
            args = [self._exact(state, "state", E, (N, self.input_shape)),
                    self._exact(action, "action", E, (N, self.n_actions)), self._exact(reward_g, "reward_g", E, ()),
                    self._exact(reward_l, "reward_l", E, (N,)), self._exact(state_, "state_", E, (N, self.input_shape))]
            m = self._exact(mask_flat, "mask_flat", E, (N, N))
            d, d_all = self._done_exact(done, E)
            fn = self._lib.risvec_replay_store_devcnt
        else:
            E = int(torch.as_tensor(reward_g).numel())
            d, d_all = self._done(done, E)
            if d is not None and d.dtype == torch.bool:
                d = d.view(torch.uint8)
            args = [self._f(state, (E, S)), self._f(action, (E, A)), self._f(reward_g, (E,)),
                    self._f(reward_l, (E, N)), self._f(state_, (E, S))]
            m = self._f(mask_flat, (E, N * N))
            fn = self._lib.risvec_replay_store
        check(fn(self._h, E, *[self._p(t) for t in args], self._p(d), d_all, self._p(m), self._stream))

    def store_transition(self, state, action, reward_g, reward_l, state_, done, mask_flat):
        """Single transition, reference signature."""
        f = lambda x: torch.as_tensor(x, dtype=torch.float32, device=self.device).reshape(1, -1)  # noqa: E731
        self.store_transitions(f(state), f(action), f([float(reward_g)]).reshape(1), f(reward_l), f(state_),
                               bool(done), f(mask_flat))

    def store_marl(self, state, intent_probs, power_raw, reward_g, reward_l, state_, done, mask_u8=None):
        """The driver's assembly (marl_train_bcd.py:1776-1799) fused with the store: `intent_probs`
        [E,N,N] (diagonal ignored), `power_raw` [E,N,2], `mask_u8` = `env.pair_mask` or None (ones).
        With `device_counter=True` the tensors are checked as in `store_transitions` (`mask_u8` uint8)."""
        N, S = self.n_agents, self.input_shape * self.n_agents
        if self.device_counter:
            E = self._rows(reward_g)
            args = [self._exact(state, "state", E, (N, self.input_shape)),
                    self._exact(intent_probs, "intent_probs", E, (N, N)),
                    self._exact(power_raw, "power_raw", E, (N, 2)), self._exact(reward_g, "reward_g", E, ()),
                    self._exact(reward_l, "reward_l", E, (N,)), self._exact(state_, "state_", E, (N, self.input_shape))]
            m = self._exact(mask_u8, "mask_u8", E, (N, N), torch.uint8)
            d, d_all = self._done_exact(done, E)
            fn = self._lib.risvec_replay_store_marl_devcnt
        else:
            E = int(torch.as_tensor(reward_g).numel())
            d, d_all = self._done(done, E)
            if d is not None and d.dtype == torch.bool:
                d = d.view(torch.uint8)
            args = [self._f(state, (E, S)), self._f(intent_probs, (E, N, N)), self._f(power_raw, (E, N, 2)),
                    self._f(reward_g, (E,)), self._f(reward_l, (E, N)), self._f(state_, (E, S))]
            m = self._f(mask_u8, (E, N * N), torch.uint8)
            fn = self._lib.risvec_replay_store_marl
        check(fn(self._h, E, *[self._p(t) for t in args], self._p(d), d_all, self._p(m), self._stream))

    def sample_buffer(self, batch_size, idx=None, generator=None, draws=None, out=None):
        """`sample_buffer` (buffer.py:27-39); indices uniform with replacement over the filled part
        (`np.random.choice(max_mem, batch_size)`), drawn on the device unless `idx` is given.

        With `device_counter=True` and no `idx`, row b is slot draws[b] % min(count, mem_size), computed on the device
        with no synchronisation, so a CUDA graph can capture the draw.  `draws` is an int64 (B,) device tensor,
        by default `torch.randint(0, 2**62, (B,), generator=generator)` (modulo bias below mem_size / 2**62).  A
        `generator` used inside a capture must be registered with the graph (`CUDAGraph.register_generator_state`).
        While count == 0 every row is slot 0 (zeros until the first store), where the reference's
        `np.random.choice(0, batch_size)` raises.

        `out`: seven preallocated device tensors (states, actions, rewards_g, rewards_l, states_, dones (bool or
        uint8), masks), written in place and returned, so that a captured graph keeps its outputs."""
        B = int(batch_size)
        N, S, A = self.n_agents, self.input_shape * self.n_agents, self.n_actions * self.n_agents
        if out is None:
            mk = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=self.device)  # noqa: E731
            out = [mk(B, S), mk(B, A), mk(B), mk(B, N), mk(B, S), mk(B, dt=torch.bool), mk(B, N * N)]
        else:
            if len(out) != 7:
                raise ValueError("out must hold seven tensors")
            rows = ((S,), (A,), (), (N,), (S,), (), (N * N,))
            dones_dt = torch.bool if getattr(out[5], "dtype", None) == torch.bool else torch.uint8
            out = [self._exact(t, f"out[{i}]", B, r, dones_dt if i == 5 else torch.float32)
                   for i, (t, r) in enumerate(zip(out, rows))]
        ptrs = [self._p(t) for t in out]
        if self.device_counter and idx is None:
            if draws is None:
                draws = torch.randint(0, 2 ** 62, (B,), device=self.device, generator=generator)
            draws = self._exact(draws, "draws", B, (), torch.int64)
            check(self._lib.risvec_replay_sample_devcnt(self._h, B, self._p(draws), *ptrs, self._stream))
        else:
            if draws is not None:
                raise ValueError("draws need device_counter=True and no idx")
            if idx is None:
                max_mem = min(self.mem_cntr, self.mem_size)
                idx = torch.randint(0, max_mem, (B,), device=self.device, generator=generator)
            idx = self._f(idx, (B,), torch.int64)
            check(self._lib.risvec_replay_sample(self._h, B, self._p(idx), *ptrs, self._stream))
        return tuple(out)

    def close(self):
        if getattr(self, "_h", None):
            for name in REPLAY_FIELDS:
                if hasattr(self, name):
                    delattr(self, name)
            self.count = None
            self._lib.risvec_replay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
