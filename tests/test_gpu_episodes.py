"""Per-env episode starts on the device (`risvec_begin_episode`, `risvec_episode_tick`, `risvec_pair_noma_episodes`).

Every comparison is bit for bit: the fused kernel calls the same device functions as the separate kernels, the
fallback shapes run the separate kernels restricted to the selected envs, and the clock's draws are keyed from
device state so eager runs, CUDA graph replays and shardings agree exactly."""
import ctypes as C

import numpy as np
import pytest
import torch

from ris_vec_marl_b200 import EP_STAGES, BatchedEnviron, RisvecError, _lib, marl_yaml_overrides, mask_schedule

pytestmark = pytest.mark.gpu

ALL = ("reset", "positions", "channel", "pairing")
YAML_SCHED = (7, 7, 0.10, 0.25, 200)
DEFAULT_SCHED = (None, None, 0.2, 0.4, 200)


def _raw(t):
    return t.contiguous().view(torch.uint8)


def _same(a, b):
    return torch.equal(_raw(a), _raw(b))


def assert_fields_equal(a, b, rows=None, names=_lib.FIELDS, what=""):
    """Every state field of handles / state dicts `a` and `b` bit-identical (on the env rows `rows` if given)."""
    for k in names:
        x, y = a[k], b[k]
        if rows is not None:
            x, y = x[rows], y[rows]
        assert _same(x, y), f"{what}: field {k} differs"


def views(env):
    return {k: env.state(k) for k in _lib.FIELDS}


def counters(env):
    ctr = (C.c_uint64 * 3)()
    _lib.check(env._lib.risvec_get_rng_counters(env._h, ctr))
    return list(ctr)


def make_env(E, V, M, seed=11, yaml=True, pairing=True, **kw):
    over = marl_yaml_overrides() if yaml else {}
    over.update(kw)
    env = BatchedEnviron("marl", E, V, M, device=0, seed=seed, **over)
    if yaml:
        env.set_pairing(yaml=True)
    # a mid-run state: theta, gains and the pairing state are all non-trivial before an episode starts
    env.make_new_game(); env.renew_positions(); env.compute_parms(); env.optimize_phase_shift()
    env.update_channel_gains()
    env.renew_positions(); env.compute_parms()
    if pairing and V <= _lib.PAIR_MAX_V:
        g = torch.Generator(device="cpu").manual_seed(seed)
        p01 = torch.rand(E, V, generator=g).to(env.device)
        env.pair_noma(p01, V - 1, 0.2, recalc_mask=True, new_episode=True)
        env.pair_noma(p01, V - 1, 0.2, recalc_mask=False)
    torch.cuda.synchronize()
    return env


def separate(env, stages, uniforms=None):
    """The existing calls for `stages`, in the order the episode start runs them."""
    used = None
    if "reset" in stages:
        env.make_new_game()
    if "positions" in stages:
        used = env.renew_positions(uniforms)
        env.compute_parms()
    if "channel" in stages:
        env.optimize_phase_shift()
        env.update_channel_gains()
    if "pairing" in stages:
        env.pair_reset()
    return used


def stage_names(bits):
    return tuple(n for n, b in EP_STAGES.items() if bits & b)


# ------------------------------------------------------------------ fused == separate
@pytest.mark.parametrize("inject", [False, True], ids=["philox", "uniforms"])
@pytest.mark.parametrize("V,M,yaml", [(8, 40, True), (8, 40, False), (6, 7, False)])
def test_fused_equals_separate_calls(V, M, yaml, inject):
    E = 301  # not a multiple of 4: the last warp has tail lanes
    a, b = make_env(E, V, M, yaml=yaml), make_env(E, V, M, yaml=yaml)
    assert_fields_equal(views(a), views(b), what="twins")
    u = None
    if inject:
        u = torch.as_tensor(np.random.default_rng(3).random((E, 4 * V))).to(a.device)
    n0 = a.launch_count
    used_a = a.begin_episode(stages=ALL, uniforms=u)
    assert a.launch_count == n0 + 1, "the fused episode start is one launch"
    used_b = separate(b, ALL, u)
    torch.cuda.synchronize()
    assert torch.equal(used_a, used_b)
    assert_fields_equal(views(a), views(b), what=f"V={V} M={M}")
    assert counters(a) == counters(b)
    a.close(); b.close()


# ------------------------------------------------------------------ per-env bits
def check_per_env(make, E, stages_all=ALL, uniforms=False):
    """Random per-env bits: each env equals a twin that ran only its own stages (counters aligned by loading the
    twin's pre-call state); envs with bits 0 are bit-identical to before the call."""
    rng = np.random.default_rng(7)
    a, b = make(), make()
    full = sum(EP_STAGES[s] for s in stages_all)
    bits = rng.integers(0, 16, E).astype(np.uint8)
    bits[:5] = 0
    bits[5:10] = 15
    u = torch.as_tensor(rng.random((E, 64))).to(a.device) if uniforms else None
    before = b.state_dict()
    used = a.begin_episode(stages=stages_all, per_env=torch.as_tensor(bits), uniforms=u)
    after = views(a)
    for s in range(16):
        rows = torch.as_tensor(np.nonzero((bits & full) == s)[0], device=a.device)
        if rows.numel() == 0:
            continue
        b.load_state_dict(before)
        names = stage_names(s)
        used_b = separate(b, names, u)
        torch.cuda.synchronize()
        assert_fields_equal(after, views(b), rows=rows, what=f"stages {names}")
        if used is not None and used_b is not None:
            assert torch.equal(used[rows], used_b[rows])
        if s == 0:
            assert_fields_equal(after, before, rows=rows, what="envs without bits")
    b.load_state_dict(before)
    separate(b, stages_all)
    assert counters(a) == counters(b), "the counters of the stages in `stages` advance once"
    a.close(); b.close()


def test_per_env_bits():
    check_per_env(lambda: make_env(512, 8, 40), 512)
    check_per_env(lambda: make_env(512, 8, 40), 512, uniforms=True)


def test_bits_outside_stages_are_ignored():
    a, b = make_env(200, 8, 40), make_env(200, 8, 40)
    a.begin_episode(stages=("positions", "pairing"), per_env=torch.full((200,), 15, dtype=torch.uint8))
    separate(b, ("positions", "pairing"))
    torch.cuda.synchronize()
    assert_fields_equal(views(a), views(b), what="stages AND per_env")
    a.close(); b.close()


@pytest.mark.parametrize("case", ["v32_m256", "3gpp", "generic"])
def test_fallback_shapes(case, monkeypatch):
    if case == "v32_m256":
        make = lambda: make_env(64, 32, 256, yaml=False)
        E = 64
    elif case == "3gpp":
        make = lambda: make_env(256, 8, 40, channel_model="3gpp_umi")
        E = 256
    else:
        monkeypatch.setenv("RISVEC_FORCE_GENERIC", "1")
        make = lambda: make_env(256, 8, 40)
        E = 256
    a, b = make(), make()
    a.begin_episode(stages=ALL)
    separate(b, ALL)
    torch.cuda.synchronize()
    assert_fields_equal(views(a), views(b), what=case)
    assert counters(a) == counters(b)
    a.close(); b.close()
    check_per_env(make, E)


# ------------------------------------------------------------------ the clock
def test_clock_schedule():
    E, V, M, T, P = 200, 8, 40, 250, 5
    env = make_env(E, V, M)
    twin = make_env(E, V, M)
    env.make_new_game()
    env.begin_episode(stages=ALL)
    # staggered steps and episode indices, so that renewals (ep_index % 5 == 0) fall on many ticks
    st = np.arange(E) % 100
    ix = (np.arange(E) * 3) % 7
    env.ep_step.copy_(torch.as_tensor(st, dtype=torch.int32))
    env.ep_index.copy_(torch.as_tensor(ix, dtype=torch.int32))
    out = None
    n_pos_checks = 0
    for t in range(T):
        env.pair_hist.fill_(1.0)  # the pairing reset of the starting envs must clear it
        pre = env.state_dict()
        n0 = env.launch_count
        out = env.episode_tick(steps_per_episode=100, positions_every=P, stages=("positions", "channel", "pairing"),
                               out=out)
        assert env.launch_count == n0 + 1
        start, done = out[0].cpu().numpy(), out[1].cpu().numpy()
        want_start = st == 0
        want_pos = want_start & (ix % P == 0)
        assert np.array_equal(start, want_start), t
        assert np.array_equal(done, st == 99), t
        st = st + 1
        wrap = st >= 100
        ix = ix + wrap
        st[wrap] = 0
        assert np.array_equal(env.ep_step.cpu().numpy(), st), t
        assert np.array_equal(env.ep_index.cpu().numpy(), ix), t
        moved = (env.pos_x != pre["pos_x"]).any(1) | (env.pos_y != pre["pos_y"]).any(1)
        assert np.array_equal(moved.cpu().numpy(), want_pos), t
        cleared = (env.pair_hist == 0).flatten(1).all(1).cpu().numpy()
        ones = (env.pair_hist == 1).flatten(1).all(1).cpu().numpy()
        assert np.array_equal(cleared, want_start) and np.array_equal(ones, ~want_start), t
        idle = torch.as_tensor(np.nonzero(~want_start)[0], device=env.device)
        assert_fields_equal(views(env), pre, rows=idle, names=[f for f in _lib.FIELDS if not f.startswith("ep_")],
                            what=f"idle envs at tick {t}")
        if want_pos.any() and n_pos_checks < 4:
            # the separate calls on the tick's positions: compute_parms, BCD from the pre-tick theta, gains
            n_pos_checks += 1
            twin.load_state_dict(pre)
            for f in ("pos_x", "pos_y", "dir"):
                twin.state(f).copy_(env.state(f))
            twin.compute_parms(); twin.optimize_phase_shift(); twin.update_channel_gains()
            torch.cuda.synchronize()
            rows = torch.as_tensor(np.nonzero(want_pos)[0], device=env.device)
            assert_fields_equal(views(env), views(twin), rows=rows,
                                names=("dist", "angle", "amp", "theta_re", "theta_im", "gains"), what=f"tick {t}")
    assert n_pos_checks >= 2
    env.close(); twin.close()


# ------------------------------------------------------------------ device keys
def staggered(env, steps, graph=False, positions_every=1, base=0, total=None):
    """The staggered driver loop: tick, pair_noma_episodes, step_marl_fused (arrivals: on-device draws).  The
    actions of global envs [base, base + E) of a `total`-env job."""
    E, V = env.E, env.V
    g = torch.Generator(device="cpu").manual_seed(99)
    raw = (torch.rand(total or E, V, 2, generator=g) * 2 - 1)[base:base + E].contiguous().to(env.device)
    act = env.map_actions(raw)
    reuse = torch.ones(E, dtype=torch.int32, device=env.device)
    obs = torch.empty(E, V, 5, device=env.device)
    out = (torch.empty(E, dtype=torch.uint8, device=env.device), torch.empty(E, dtype=torch.uint8, device=env.device))

    def one():
        start, _ = env.episode_tick(steps_per_episode=100, positions_every=positions_every, stages=ALL, out=out)
        part, ng = env.pair_noma_episodes(act, start, schedule=YAML_SCHED, reuse=reuse)
        env.step_marl_fused(raw, part, ng, obs_out=obs)

    if not graph:
        for _ in range(steps):
            one()
    else:
        cg = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(cg, stream=s):
                one()
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(steps):
            cg.replay()
    torch.cuda.synchronize()


def start_staggered(env, offsets=None):
    env.make_new_game()
    env.begin_episode(stages=ALL)
    E = env.E
    off = torch.arange(E, dtype=torch.int32) % 100 if offsets is None else offsets
    env.ep_step.copy_(off.to(env.device))


def test_graph_replay_equals_eager():
    a, b = make_env(64, 8, 40), make_env(64, 8, 40)
    start_staggered(a)
    start_staggered(b)
    staggered(a, 250)
    staggered(b, 250, graph=True)
    assert_fields_equal(views(a), views(b), what="eager vs graph")
    assert int(a.ep_index.sum()) > 64, "episodes wrapped during the loop"
    a.close(); b.close()


def test_sharding_invariant():
    def fresh(E, base):
        env = BatchedEnviron("marl", E, 8, 40, device=0, seed=21, env_index_base=base, **marl_yaml_overrides())
        env.set_pairing(yaml=True)
        return env

    one = fresh(64, 0)
    halves = [fresh(32, 0), fresh(32, 32)]
    start_staggered(one)
    offs = torch.arange(64, dtype=torch.int32) % 100
    for i, env in enumerate(halves):
        start_staggered(env, offs[32 * i:32 * (i + 1)])
    staggered(one, 250)
    for i, env in enumerate(halves):
        staggered(env, 250, base=32 * i, total=64)
    for k in _lib.FIELDS:
        cat = torch.cat([h.state(k) for h in halves])
        assert _same(one.state(k), cat), f"field {k}: one handle of 64 != two handles of 32"
    one.close()
    for h in halves:
        h.close()


def test_renewals_draw_per_episode():
    E = 512
    env = make_env(E, 8, 40)
    # every vehicle heads up 0.875 m below the first horizontal lane: its renewal draws a turn decision
    env.pos_y.fill_(200.0)
    env.dir.fill_(0)
    env.vel.fill_(10)
    pre = env.state_dict()
    got = []
    for ep in (0, 1, 0):
        env.load_state_dict(pre)
        env.ep_step.zero_()
        env.ep_index.fill_(ep)
        env.episode_tick(steps_per_episode=100, positions_every=1, stages=("positions",))
        got.append((env.pos_x.clone(), env.pos_y.clone(), env.dir.clone()))
    same = lambda i, j: all(torch.equal(x, y) for x, y in zip(got[i], got[j]))
    assert same(0, 2), "the tick's draws are a function of (seed, env, episode)"
    differs = ((got[0][0] != got[1][0]) | (got[0][1] != got[1][1]) | (got[0][2] != got[1][2])).any(1)
    assert int(differs.sum()) > 0, "two renewals of the same env drew the same uniforms"
    # the reset draws too
    env.load_state_dict(pre)
    env.ep_step.zero_(); env.ep_index.fill_(3)
    env.episode_tick(stages=("reset",))
    r3 = env.pos_y.clone()
    env.load_state_dict(pre)
    env.ep_step.zero_(); env.ep_index.fill_(4)
    env.episode_tick(stages=("reset",))
    assert float((env.pos_y != r3).any(1).float().mean()) > 0.9
    env.close()


# ------------------------------------------------------------------ pairing with per-env episode state
@pytest.mark.parametrize("sched,yaml", [(YAML_SCHED, True), (DEFAULT_SCHED, False)])
def test_pair_noma_episodes_equals_scalar_calls(sched, yaml):
    E, V = 256, 8
    a, b = make_env(E, V, 40, yaml=yaml), make_env(E, V, 40, yaml=yaml)
    rng = np.random.default_rng(5)
    eps = rng.choice([0, 7, 150, 250], E).astype(np.int32)
    start = (rng.random(E) < 0.4).astype(np.uint8)
    reuse = (rng.random(E) < 0.5).astype(np.int32)
    p01 = torch.as_tensor(rng.random((E, V)).astype(np.float32)).to(a.device)
    for env in (a, b):
        env.ep_index.copy_(torch.as_tensor(eps))
    pre = b.state_dict()
    a.pair_noma_episodes(p01, torch.as_tensor(start), schedule=sched, reuse=torch.as_tensor(reuse))
    after = views(a)
    k0, k1, q0, q1, warm = sched
    for ep in (0, 7, 150, 250):
        rows = np.nonzero((start == 1) & (eps == ep))[0]
        if rows.size == 0:
            continue
        K, q = mask_schedule(ep, V, k0, k1, q0, q1, warm)
        b.load_state_dict(pre)
        b.pair_noma(p01, K, q, recalc_mask=True, reuse=torch.as_tensor(reuse), new_episode=True)
        torch.cuda.synchronize()
        assert_fields_equal(after, views(b), rows=torch.as_tensor(rows, device=a.device), what=f"start, episode {ep}")
    rows = np.nonzero(start == 0)[0]
    b.load_state_dict(pre)
    b.pair_noma(p01, V - 1, 0.3, recalc_mask=False, reuse=torch.as_tensor(reuse))
    torch.cuda.synchronize()
    assert_fields_equal(after, views(b), rows=torch.as_tensor(rows, device=a.device), what="no start")
    a.close(); b.close()


# ------------------------------------------------------------------ arguments, persistence
def test_arguments_and_state_dict():
    env = make_env(64, 8, 40)
    lib, h, s = env._lib, env._h, env.stream
    assert lib.risvec_begin_episode(h, None, 16, None, 0, None, s) == -1
    assert lib.risvec_begin_episode(h, None, 2, C.c_void_p(env.pos_x.data_ptr()), 0, None, s) == -1
    assert lib.risvec_begin_episode(None, None, 2, None, 0, None, s) == -1
    bad = [(0, 5, 6), (100, 0, 6), (100, 5, 32)]
    for spe, pe, stg in bad:
        sch = _lib.EpisodeSchedule(spe, pe, stg, 0)
        assert lib.risvec_episode_tick(h, C.byref(sch), None, None, s) == -1
    assert lib.risvec_episode_tick(h, None, None, None, s) == -1
    with pytest.raises(RisvecError) as ei:
        env.begin_episode(stages=32)
    assert ei.value.code == -1
    start = torch.ones(64, dtype=torch.uint8, device=env.device)
    p01 = torch.rand(64, 8, device=env.device)
    for sched in ((7, 7, 1.5, 0.25, 200), (7, 7, 0.1, -0.1, 200)):
        with pytest.raises(RisvecError) as ei:
            env.pair_noma_episodes(p01, start, schedule=sched)
        assert ei.value.code == -1
    sch = _lib.PairSchedule(-1, -1, 200, 0, 0.2, 0.4)
    assert lib.risvec_pair_noma_episodes(h, C.byref(env.pairing), C.c_void_p(p01.data_ptr()), 8, C.byref(sch), None,
                                         None, 1, s) == -1
    big = BatchedEnviron("marl", 4, 16, 8, device=0, seed=1)
    with pytest.raises(RisvecError) as ei:
        big.pair_noma_episodes(torch.zeros(4, 16, device=big.device), torch.ones(4, dtype=torch.uint8), schedule=DEFAULT_SCHED)
    assert ei.value.code == -2
    big.close()
    # the clock is state: a state_dict round trip restores it
    fresh = BatchedEnviron("marl", 64, 8, 40, device=0, seed=2)
    assert int(fresh.ep_step.abs().sum()) == 0 and int(fresh.ep_index.abs().sum()) == 0, "zero at creation"
    fresh.close()
    env.ep_step.copy_(torch.arange(64, dtype=torch.int32) % 100)
    env.ep_index.copy_(torch.arange(64, dtype=torch.int32) // 3)
    sd = env.state_dict()
    for _ in range(7):
        env.episode_tick()
    assert not torch.equal(env.ep_step, sd["ep_step"])
    env.load_state_dict(sd)
    assert torch.equal(env.ep_step, sd["ep_step"]) and torch.equal(env.ep_index, sd["ep_index"])
    env.close()
