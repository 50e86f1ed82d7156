"""Device-counter replay memory (`ReplayBuffer(..., device_counter=True)`, `risvec_replay_*_devcnt`).

Every comparison is exact: the stores are pure float32 copies.  Each device-counter buffer is checked against the
oracle (oracle/replay_oracle.py) and against a host-counter twin fed the same tensors, eagerly and as CUDA-graph
replays whose captured stores must land in fresh slots on every replay."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.replay_oracle import ReplayOracle, assemble_marl_action, assemble_marl_mask
from ris_vec_marl_b200 import BatchedEnviron, EpisodeLog, ReplayBuffer, _lib, marl_yaml_overrides

pytestmark = pytest.mark.gpu

FIELDS = _lib.REPLAY_FIELDS
ALL = ("reset", "positions", "channel", "pairing")
YAML_SCHED = (7, 7, 0.10, 0.25, 200)
DEV = torch.device("cuda", 0)


# ------------------------------------------------------------------ fixtures
def assert_same_memory(a, b, what):
    """two ReplayBuffers, or a ReplayBuffer and the oracle: every array and the count"""
    assert a.mem_cntr == b.mem_cntr, f"{what}: count {a.mem_cntr} != {b.mem_cntr}"
    for name in FIELDS:
        x, y = getattr(a, name), getattr(b, name)
        x = x.cpu().numpy() if isinstance(x, torch.Tensor) else x
        y = y.cpu().numpy() if isinstance(y, torch.Tensor) else y
        assert np.array_equal(x, y), f"{what}: {name} differs"


def flat_batch(rng, E, N, S1, A1, done_kind, with_mask):
    """device tensors of one `store_transitions` call and the numpy arrays the oracle takes"""
    t = dict(state=rng.normal(size=(E, S1 * N)), action=rng.normal(size=(E, A1 * N)), reward_g=rng.normal(size=E),
             reward_l=rng.normal(size=(E, N)), state_=rng.normal(size=(E, S1 * N)))
    t = {k: v.astype(np.float32) for k, v in t.items()}
    mask = (rng.random((E, N * N)) < 0.5).astype(np.float32) if with_mask else None
    done = {"per_env": rng.random(E) < 0.3, "per_env_bool": rng.random(E) < 0.5, "all": True, "none": False}[done_kind]
    dev = {k: torch.as_tensor(v).to(DEV) for k, v in t.items()}
    if isinstance(done, bool):
        d = done
    else:
        d = torch.as_tensor(done).to(DEV) if done_kind == "per_env_bool" else torch.as_tensor(done.astype(np.uint8)).to(DEV)
    dev.update(done=d, mask_flat=None if mask is None else torch.as_tensor(mask).to(DEV))
    return dev, dict(t, done=done, mask_flat=mask)


def marl_batch(rng, E, N, S1, done_kind, with_mask):
    """device tensors of one `store_marl` call (driver layout) and the oracle's assembled rows"""
    state = rng.normal(size=(E, N, S1)).astype(np.float32)
    state_ = rng.normal(size=(E, N, S1)).astype(np.float32)
    probs = rng.random((E, N, N)).astype(np.float32)
    power = rng.uniform(-1, 1, (E, N, 2)).astype(np.float32)
    rg, rl = rng.normal(size=E).astype(np.float32), rng.normal(size=(E, N)).astype(np.float32)
    mask = (rng.random((E, N, N)) < 0.6).astype(np.uint8) if with_mask else None
    done = {"per_env": rng.random(E) < 0.3, "all": True, "none": False}[done_kind]
    dev = [torch.as_tensor(x).to(DEV) for x in (state, probs, power, rg, rl, state_)]
    d = done if isinstance(done, bool) else torch.as_tensor(done.astype(np.uint8)).to(DEV)
    m = None if mask is None else torch.as_tensor(mask).to(DEV)
    action = np.stack([assemble_marl_action(probs[e], power[e]) for e in range(E)])
    mflat = np.stack([assemble_marl_mask(None if mask is None else mask[e], N) for e in range(E)])
    orc = (state.reshape(E, -1), action, rg, rl, state_.reshape(E, -1), done, mflat)
    return dev, d, m, orc


CALLS = ((1, "per_env", True), (257, "all", True), (600, "none", False), (333, "per_env_bool", True))  # 1191 rows


def capture(fn):
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            out = fn()
    torch.cuda.current_stream().wait_stream(s)
    return g, out


# ------------------------------------------------------------------ eager stores
@pytest.mark.parametrize("N", [8, 5])  # 8: k_replay_store_flat; 5: rows not a multiple of 4, k_replay_store<1, .>
def test_store_transitions_against_oracle_and_host_twin(N):
    rng = np.random.default_rng(N)
    S1, A1, cap = 5, 10, 1000
    dc, hc, orc = ReplayBuffer(cap, S1, A1, N, device_counter=True), ReplayBuffer(cap, S1, A1, N), \
        ReplayOracle(cap, S1, A1, N)
    assert dc.count.dtype == torch.int64 and tuple(dc.count.shape) == (1,) and dc.mem_cntr == 0
    for E, done_kind, with_mask in CALLS:
        dev, ref = flat_batch(rng, E, N, S1, A1, done_kind, with_mask)
        dc.store_transitions(**dev)
        hc.store_transitions(**dev)
        orc.store_transitions(**ref)
        assert_same_memory(dc, orc, f"E = {E}: device counter vs oracle")
        assert_same_memory(dc, hc, f"E = {E}: device counter vs host counter")
    assert int(dc.count.item()) == 1191
    dc.close(); hc.close()


@pytest.mark.parametrize("N", [8, 5])
def test_store_marl_against_oracle_and_host_twin(N):
    rng = np.random.default_rng(10 + N)
    S1, cap = 5, 1000
    dc, hc, orc = ReplayBuffer(cap, S1, N + 2, N, device_counter=True), ReplayBuffer(cap, S1, N + 2, N), \
        ReplayOracle(cap, S1, N + 2, N)
    for E, done_kind, with_mask in CALLS:
        dev, d, m, ref = marl_batch(rng, E, N, S1, "per_env" if done_kind == "per_env_bool" else done_kind, with_mask)
        dc.store_marl(*dev, done=d, mask_u8=m)
        hc.store_marl(*dev, done=d, mask_u8=m)
        orc.store_transitions(*ref)
        assert_same_memory(dc, orc, f"E = {E}: device counter vs oracle")
        assert_same_memory(dc, hc, f"E = {E}: device counter vs host counter")
    dc.close(); hc.close()


# ------------------------------------------------------------------ graph replays of a store
@pytest.mark.parametrize("E,cap", [(1003, 5000), (1024, 4096)])  # 5000 % 1003 != 0; 4096 = 4 E: wraps on a boundary
def test_captured_store_replayed_250_times(E, cap):
    N, S1, reps = 8, 5, 250
    dc, hc = ReplayBuffer(cap, S1, N + 2, N, device_counter=True), ReplayBuffer(cap, S1, N + 2, N)
    g = torch.Generator(device=DEV).manual_seed(E)
    ins = [torch.empty(E, N, S1, device=DEV), torch.empty(E, N, N, device=DEV), torch.empty(E, N, 2, device=DEV),
           torch.empty(E, device=DEV), torch.empty(E, N, device=DEV), torch.empty(E, N, S1, device=DEV)]
    done = torch.empty(E, dtype=torch.uint8, device=DEV)
    mask = torch.empty(E, N, N, dtype=torch.uint8, device=DEV)
    graph, _ = capture(lambda: dc.store_marl(*ins, done=done, mask_u8=mask))
    torch.cuda.synchronize()
    assert dc.mem_cntr == 0, "capturing a store runs nothing"
    for r in range(reps):
        for t in ins:
            t.copy_(torch.rand(t.shape, device=DEV, generator=g) * 2 - 1)
        done.copy_(torch.rand(E, device=DEV, generator=g) < 0.2)
        mask.copy_(torch.rand(E, N, N, device=DEV, generator=g) < 0.6)
        graph.replay()
        hc.store_marl(*ins, done=done, mask_u8=mask)
        for name in FIELDS:
            assert torch.equal(getattr(dc, name), getattr(hc, name)), f"replay {r}: {name} differs"
    assert dc.mem_cntr == reps * E == hc.mem_cntr
    dc.close(); hc.close()


# ------------------------------------------------------------------ the whole staggered driver step as one graph
def make_env(E, seed=11):
    env = BatchedEnviron("marl", E, 8, 40, device=0, seed=seed, **marl_yaml_overrides())
    env.set_pairing(yaml=True)
    return env


class DriverStep:
    """episode_tick, map_actions, pair_noma_episodes, step_marl_fused, EpisodeLog.accumulate and store_marl with the
    tick's per-env done; the actions are a fixed function of the observation so eager and graph forms agree."""

    def __init__(self, env, log, rb, spe):
        self.env, self.log, self.rb, self.spe = env, log, rb, spe
        E, V = env.E, env.V
        self.obs = [torch.empty(E, V, 5, device=env.device), torch.empty(E, V, 5, device=env.device)]
        env.observe(out=self.obs[0])
        self.reuse = torch.ones(E, dtype=torch.int32, device=env.device)
        self.tick = (torch.empty(E, dtype=torch.uint8, device=env.device),
                     torch.empty(E, dtype=torch.uint8, device=env.device))

    def one(self, parity):
        env, cur, nxt = self.env, self.obs[parity], self.obs[parity ^ 1]
        start, done = env.episode_tick(steps_per_episode=self.spe, positions_every=1, stages=ALL, out=self.tick)
        raw = torch.tanh(cur[:, :, 1:3] * 3.0).contiguous()
        part, ng = env.pair_noma_episodes(env.map_actions(raw), start, schedule=YAML_SCHED, reuse=self.reuse)
        logits = cur[:, :, 3:4] - cur[:, None, :, 4]
        probs = torch.softmax(logits.masked_fill(env.pair_mask == 0, -1e9), dim=-1)
        env.step_marl_fused(raw, part, ng, obs_out=nxt)
        self.log.accumulate(done)
        self.rb.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=done, mask_u8=env.pair_mask)


def test_staggered_driver_step_as_one_graph():
    E, spe, steps, cap = 1003, 7, 24, 20_000  # the ring wraps once
    a, b = make_env(E), make_env(E)
    a.make_new_game()
    a.begin_episode(stages=ALL)
    a.ep_step.copy_((torch.arange(E, dtype=torch.int32) % spe).to(a.device))
    b.load_state_dict(a.state_dict())
    la, lb = EpisodeLog(a), EpisodeLog(b)
    ra, rb = ReplayBuffer(cap, 5, 10, 8), ReplayBuffer(cap, 5, 10, 8, device_counter=True)
    eager, graphed = DriverStep(a, la, ra, spe), DriverStep(b, lb, rb, spe)
    graphs = [capture(lambda p=p: graphed.one(p))[0] for p in (0, 1)]  # one graph per observation-buffer parity
    for t in range(steps):
        eager.one(t % 2)
        graphs[t % 2].replay()
    torch.cuda.synchronize()
    assert ra.mem_cntr == steps * E and rb.mem_cntr == steps * E
    assert_same_memory(rb, ra, "graph vs eager")
    assert int(rb.terminal_memory.sum()) > 2 * E, "the tick's per-env done flags reached the memory"
    for k in _lib.FIELDS:
        assert torch.equal(a.state(k).contiguous().view(torch.uint8), b.state(k).contiguous().view(torch.uint8)), k
    assert torch.equal(eager.obs[0], graphed.obs[0]) and torch.equal(eager.obs[1], graphed.obs[1])
    ea, eb = la.drain(), lb.drain()
    assert len(ea["env"]) > 2 * E and len(ea["env"]) == len(eb["env"])
    for k in ("env", "step", "length", "reward", "reward_user"):
        assert np.array_equal(ea[k], eb[k]), k
    for n in ea["stats"]:
        assert np.array_equal(ea["stats"][n], eb["stats"][n]), n
    a.close(); b.close(); ra.close(); rb.close()


# ------------------------------------------------------------------ sampling
def test_sample_devcnt_eager_graph_and_empty():
    N, S1, cap, E, B = 8, 5, 700, 300, 512
    rng = np.random.default_rng(3)
    dc, orc = ReplayBuffer(cap, S1, N + 2, N, device_counter=True), ReplayOracle(cap, S1, N + 2, N)

    def check_rows(got, draws, count, what):
        n = min(count, cap)
        idx = draws.cpu().numpy() % n if n else np.zeros(len(draws), np.int64)
        for i, (x, y) in enumerate(zip(got, orc.sample(idx))):
            assert np.array_equal(x.cpu().numpy(), y), f"{what}: output {i}"

    # count == 0: every row is slot 0, zeros at creation
    draws = torch.randint(0, 2 ** 62, (B,), device=DEV)
    got = dc.sample_buffer(B, draws=draws)
    check_rows(got, draws, 0, "empty")
    assert all(float(t.float().abs().sum()) == 0.0 for t in got) and got[5].dtype == torch.bool
    # eager, after stores
    for k in range(2):
        dev, d, m, ref = marl_batch(rng, E, N, S1, "per_env", True)
        dc.store_marl(*dev, done=d, mask_u8=m)
        orc.store_transitions(*ref)
        draws = torch.as_tensor(rng.integers(0, 2 ** 62, B)).to(DEV)
        check_rows(dc.sample_buffer(B, draws=draws), draws, orc.mem_cntr, f"eager {k}")
    # the default draws: torch.randint(0, 2**62) from the generator, on the device
    g1, g2 = torch.Generator(device=DEV).manual_seed(5), torch.Generator(device=DEV).manual_seed(5)
    got = dc.sample_buffer(B, generator=g1)
    check_rows(got, torch.randint(0, 2 ** 62, (B,), device=DEV, generator=g2), orc.mem_cntr, "default draws")
    # explicit idx in device-counter mode: the caller-index gather
    idx = torch.as_tensor(rng.integers(0, cap, B))
    for x, y in zip(dc.sample_buffer(B, idx=idx), orc.sample(idx.numpy())):
        assert np.array_equal(x.cpu().numpy(), y)
    # inside a graph: sample, store, sample; fresh draws and sources copied in before every replay; out= reused
    ins = [torch.empty_like(t) for t in dev]
    done = torch.empty(E, dtype=torch.uint8, device=DEV)
    mask = torch.empty(E, N, N, dtype=torch.uint8, device=DEV)
    d0, d1 = torch.empty(B, dtype=torch.int64, device=DEV), torch.empty(B, dtype=torch.int64, device=DEV)
    mk = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=DEV)  # noqa: E731
    S, A = S1 * N, (N + 2) * N
    out0 = (mk(B, S), mk(B, A), mk(B), mk(B, N), mk(B, S), mk(B, dt=torch.bool), mk(B, N * N))
    out1 = (mk(B, S), mk(B, A), mk(B), mk(B, N), mk(B, S), mk(B, dt=torch.uint8), mk(B, N * N))

    def step():
        r0 = dc.sample_buffer(B, draws=d0, out=out0)
        dc.store_marl(*ins, done=done, mask_u8=mask)
        r1 = dc.sample_buffer(B, draws=d1, out=out1)
        return r0, r1

    graph, (r0, r1) = capture(step)
    assert all(x is y for x, y in zip(r0, out0)) and all(x is y for x, y in zip(r1, out1)), "out= is returned as given"
    for k in range(5):
        before = orc.mem_cntr
        dev, d, m, ref = marl_batch(rng, E, N, S1, "per_env", True)
        for t, s in zip(ins, dev):
            t.copy_(s)
        done.copy_(d)
        mask.copy_(m)
        d0.copy_(torch.as_tensor(rng.integers(0, 2 ** 62, B)))
        d1.copy_(torch.as_tensor(rng.integers(0, 2 ** 62, B)))
        graph.replay()
        torch.cuda.synchronize()
        check_rows(out0, d0, before, f"graph replay {k}, before the store")
        orc.store_transitions(*ref)
        check_rows(out1, d1, orc.mem_cntr, f"graph replay {k}, after the store")
        assert_same_memory(dc, orc, f"graph replay {k}")
    assert dc.mem_cntr == 7 * E
    dc.close()


# ------------------------------------------------------------------ refusals
def _raw_store_args(rb, E, dev, d, m):
    return [rb._h, E] + [rb._p(t) for t in dev] + [rb._p(d), 0, rb._p(m), rb._stream]


def test_refusals():
    N, S1, cap, E = 8, 5, 64, 16
    rng = np.random.default_rng(7)
    dc, hc = ReplayBuffer(cap, S1, N + 2, N, device_counter=True), ReplayBuffer(cap, S1, N + 2, N)
    lib = dc._lib
    dev, d, m, _ = marl_batch(rng, E, N, S1, "per_env", True)
    fdev, _ = flat_batch(rng, E, N, S1, N + 2, "per_env", True)
    flat = [fdev[k] for k in ("state", "action", "reward_g", "reward_l", "state_")]
    dc.store_marl(*dev, done=d, mask_u8=m)
    torch.cuda.synchronize()
    snap = {n: getattr(dc, n).clone() for n in FIELDS}

    # host-counter calls on a device-counter handle, and the other way round
    assert lib.risvec_replay_store_marl(*_raw_store_args(dc, E, dev, d, m)) == -1
    assert b"risvec_replay_store_marl_devcnt" in lib.risvec_last_error()
    assert lib.risvec_replay_store(*_raw_store_args(dc, E, flat, d, fdev["mask_flat"])) == -1
    assert lib.risvec_replay_set_count(dc._h, 5) == -1
    assert lib.risvec_replay_count(dc._h) == -1
    ptr = C.c_void_p()
    assert lib.risvec_replay_use_device_counter(dc._h, C.byref(ptr), None) == -1, "a second switch is refused"
    assert lib.risvec_replay_store_marl_devcnt(*_raw_store_args(hc, E, dev, d, m)) == -1
    assert b"risvec_replay_use_device_counter" in lib.risvec_last_error()
    assert lib.risvec_replay_store_devcnt(*_raw_store_args(hc, E, flat, d, fdev["mask_flat"])) == -1
    outs = hc.sample_buffer(4, idx=torch.zeros(4, dtype=torch.int64))
    draws = torch.zeros(4, dtype=torch.int64, device=DEV)
    assert lib.risvec_replay_sample_devcnt(hc._h, 4, hc._p(draws), *[hc._p(t) for t in outs], hc._stream) == -1
    assert lib.risvec_replay_count(hc._h) == 0
    # E out of [1, mem_size] and NULL arguments
    for bad_E in (0, cap + 1):
        assert lib.risvec_replay_store_marl_devcnt(*_raw_store_args(dc, bad_E, dev, d, m)) == -1
        assert lib.risvec_replay_store_devcnt(*_raw_store_args(dc, bad_E, flat, d, fdev["mask_flat"])) == -1
    for i in range(2, 8):
        args = _raw_store_args(dc, E, dev, d, m)
        args[i] = C.c_void_p(None)
        assert lib.risvec_replay_store_marl_devcnt(*args) == -1, f"NULL argument {i}"
    for i in range(2, 7):
        args = _raw_store_args(dc, E, flat, d, None)
        args[i] = C.c_void_p(None)
        assert lib.risvec_replay_store_devcnt(*args) == -1, f"NULL argument {i}"
    sample_args = [dc._h, 4, dc._p(draws)] + [dc._p(t) for t in outs] + [dc._stream]
    for i in [2] + list(range(3, 10)):
        args = list(sample_args)
        args[i] = C.c_void_p(None)
        assert lib.risvec_replay_sample_devcnt(*args) == -1, f"NULL argument {i}"
    assert lib.risvec_replay_sample_devcnt(dc._h, 0, *sample_args[2:]) == -1
    ptr = C.c_void_p()
    assert lib.risvec_replay_use_device_counter(hc._h, None, None) == -1

    # tensors that would need a conversion, or of the wrong shape, are refused before any launch
    state, probs, power, rg, rl, state_ = dev
    bad_calls = [
        dict(state=state.cpu()), dict(state=state.double()), dict(state=state.transpose(1, 2).contiguous()),
        dict(state=state[:, :, :4]), dict(probs=probs.transpose(1, 2)), dict(power=power.reshape(E, 2, N)),
        dict(rg=rg.reshape(E, 1)), dict(rg=rg.cpu().numpy()), dict(rl=rl[:, :N - 1]), dict(state_=state_.half()),
        dict(mask=m.float()), dict(mask=m.bool()), dict(d=d.int()), dict(d=d.cpu()), dict(d=1),
        dict(d=torch.zeros(2 * E, dtype=torch.uint8, device=DEV)[::2]),
    ]
    base = dict(state=state, probs=probs, power=power, rg=rg, rl=rl, state_=state_, d=d, mask=m)
    for bad in bad_calls:
        a = dict(base, **bad)
        with pytest.raises(ValueError):
            dc.store_marl(a["state"], a["probs"], a["power"], a["rg"], a["rl"], a["state_"], done=a["d"],
                          mask_u8=a["mask"])
    for bad in (dict(action=flat[1].reshape(E, N + 2, N).transpose(1, 2)), dict(mask_flat=fdev["mask_flat"].cpu()),
                dict(reward_g=fdev["reward_g"].double())):
        with pytest.raises(ValueError):
            dc.store_transitions(**dict(fdev, **bad))
    for bad in (torch.zeros(4, dtype=torch.int32, device=DEV), torch.zeros(4, dtype=torch.int64),
                torch.zeros(5, dtype=torch.int64, device=DEV)):
        with pytest.raises(ValueError):
            dc.sample_buffer(4, draws=bad)
    with pytest.raises(ValueError):
        hc.sample_buffer(4, draws=draws)
    with pytest.raises(ValueError):
        dc.sample_buffer(4, out=outs[:6])
    with pytest.raises(ValueError):
        dc.sample_buffer(4, out=outs[:5] + (outs[5].float(), outs[6]))
    torch.cuda.synchronize()
    assert dc.mem_cntr == E
    for n in FIELDS:
        assert torch.equal(getattr(dc, n), snap[n]), f"a refused call changed {n}"
    dc.close(); hc.close()


# ------------------------------------------------------------------ checkpoints
def test_state_dict_round_trip_across_modes():
    N, S1, cap, E = 8, 5, 500, 180
    rng = np.random.default_rng(9)
    batches = [marl_batch(rng, E, N, S1, "per_env", True)[:3] for _ in range(6)]
    src = ReplayBuffer(cap, S1, N + 2, N, device_counter=True)
    for dev, d, m in batches[:3]:
        src.store_marl(*dev, done=d, mask_u8=m)
    sd = src.state_dict()
    assert sd["_mem_cntr"] == 3 * E
    resumed = [ReplayBuffer(cap, S1, N + 2, N, device_counter=True), ReplayBuffer(cap, S1, N + 2, N)]
    for rb in resumed:
        rb.load_state_dict(sd)
        assert_same_memory(rb, src, "loaded")
    back = ReplayBuffer(cap, S1, N + 2, N, device_counter=True)
    back.load_state_dict(resumed[1].state_dict())  # a host-counter state dict into a device-counter buffer
    for dev, d, m in batches[3:]:
        for rb in [src, back] + resumed:
            rb.store_marl(*dev, done=d, mask_u8=m)
    for rb in [back] + resumed:
        assert_same_memory(rb, src, "resumed")
    assert src.mem_cntr == 6 * E
    other = ReplayBuffer(cap + 1, S1, N + 2, N, device_counter=True)
    with pytest.raises(ValueError):
        other.load_state_dict(sd)
    with pytest.raises(ValueError):
        resumed[0].load_state_dict(dict(sd, mask_memory=sd["mask_memory"][:, :N]))
    for rb in [src, back, other] + resumed:
        rb.close()


# ------------------------------------------------------------------ one kernel per store
@pytest.mark.parametrize("N", [8, 5])
def test_one_kernel_per_store(N):
    from torch.profiler import ProfilerActivity, profile

    rng = np.random.default_rng(20 + N)
    S1, cap, E = 5, 1000, 333
    dc = ReplayBuffer(cap, S1, N + 2, N, device_counter=True)
    dev, d, m, _ = marl_batch(rng, E, N, S1, "per_env", True)
    fdev, _ = flat_batch(rng, E, N, S1, N + 2, "per_env", True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            dc.store_marl(*dev, done=d, mask_u8=m)
            dc.store_transitions(**fdev)
            with pytest.raises(ValueError):
                dc.store_marl(*dev, done=d.cpu(), mask_u8=m)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "k_replay" in e.name]
    assert len(names) == 6, names
    assert all(("k_replay_store_flat" in n) == (N == 8) for n in names), names
    assert dc.mem_cntr == 6 * E
    dc.close()
