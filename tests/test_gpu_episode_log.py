"""Per-episode statistics of staggered episodes (`risvec_episode_accumulate`, `EpisodeLog`).

Every comparison is bit for bit.  The host restatement reads `stats`, `reward`, `reward_user`, `step_ctr` and `done`
after each step and adds them in float64, in the column order of include/risvec.h: each element of an env's running
row gets one float64 addition per step, exactly what the kernel does, so the sums agree in every bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from ris_vec_marl_b200 import STAT_COLUMNS, BatchedEnviron, EpisodeLog, _lib, marl_yaml_overrides

pytestmark = pytest.mark.gpu

ALL = ("reset", "positions", "channel", "pairing")
YAML_SCHED = (7, 7, 0.10, 0.25, 200)
NSTAT = _lib.NSTAT


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def assert_same(a, b, what):
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert np.array_equal(bits(a), bits(b)), f"{what} differs"


def sort_rows(rec):
    """records [n, C + 2] sorted by (step, env), as `drain` sorts them"""
    rec = np.asarray(rec, dtype=np.float64)
    return rec[np.lexsort((rec[:, 0], rec[:, 1]))]


def raw_records(log):
    """the log's records as they stand (before a drain), sorted"""
    torch.cuda.synchronize()
    n = min(int(log.count.item()), log.capacity)
    return sort_rows(log.records[:n].cpu().numpy())


def assert_fields_equal(a, b, what=""):
    for k in _lib.FIELDS:
        assert torch.equal(a.state(k).contiguous().view(torch.uint8), b.state(k).contiguous().view(torch.uint8)), \
            f"{what}: field {k} differs"


def make_env(E, variant="marl", seed=11, base=0):
    if variant == "marl":
        env = BatchedEnviron("marl", E, 8, 40, device=0, seed=seed, env_index_base=base, **marl_yaml_overrides())
        env.set_pairing(yaml=True)
    else:
        env = BatchedEnviron("sarl", E, 8, 40, device=0, seed=seed, env_index_base=base)
    return env


def stages_of(env):
    return ALL if env.variant == "marl" else ("positions",)


def start_staggered(env, spe, offsets=None):
    """make_new_game, one episode start for all envs, then per-env clock offsets (e % spe unless given)"""
    env.make_new_game()
    env.begin_episode(stages=stages_of(env))
    off = torch.arange(env.E, dtype=torch.int32) % spe if offsets is None else offsets
    env.ep_step.copy_(off.to(env.device))


class Restatement:
    """float64 numpy restatement of the running sums and the records"""

    def __init__(self, env, base=0):
        self.E, self.base = env.E, base
        self.n_user = env.V if env.variant == "marl" else 0
        self.run = np.zeros((env.E, _lib.eplog_run_cols(self.n_user)))
        self.recs = []

    def step(self, env, done):
        torch.cuda.synchronize()
        E = self.E
        cols = [np.ones((E, 1)), env.stats.cpu().numpy().astype(np.float64),
                env.reward.cpu().numpy().astype(np.float64)[:, None]]
        if self.n_user:
            cols.append(env.reward_user.cpu().numpy().astype(np.float64))
        self.run = self.run + np.concatenate(cols, axis=1)
        d = done.cpu().numpy() != 0 if isinstance(done, torch.Tensor) else np.full(E, bool(done))
        ctr = env.step_ctr.cpu().numpy()
        for e in np.nonzero(d)[0]:
            self.recs.append(np.concatenate([[self.base + e, ctr[e]], self.run[e]]))
        self.run[d] = 0.0

    def records(self, start=0):
        return sort_rows(np.array(self.recs[start:]).reshape(-1, _lib.eplog_rec_cols(self.n_user)))


def assert_drained(eps, want, n_user, what):
    """a drain's dict against sorted record rows [n, C + 2]"""
    assert len(eps["env"]) == len(want), f"{what}: {len(eps['env'])} records, want {len(want)}"
    for k, col in (("env", 0), ("step", 1), ("length", 2)):
        assert eps[k].dtype == np.int64 and np.array_equal(eps[k], want[:, col].astype(np.int64)), f"{what}: {k}"
    assert list(eps["stats"]) == list(STAT_COLUMNS)
    for i, name in enumerate(STAT_COLUMNS):
        assert_same(eps["stats"][name], want[:, 3 + i], f"{what}: stats {name}")
    assert_same(eps["reward"], want[:, 3 + NSTAT], f"{what}: reward")
    if n_user:
        assert_same(eps["reward_user"], want[:, 4 + NSTAT:], f"{what}: reward_user")
    else:
        assert "reward_user" not in eps


def cat_sorted(parts):
    """drains of several intervals / shards as one dict sorted by (step, env)"""
    env = np.concatenate([p["env"] for p in parts])
    step = np.concatenate([p["step"] for p in parts])
    o = np.lexsort((env, step))
    out = {"env": env[o], "step": step[o], "length": np.concatenate([p["length"] for p in parts])[o],
           "stats": {n: np.concatenate([p["stats"][n] for p in parts])[o] for n in STAT_COLUMNS},
           "reward": np.concatenate([p["reward"] for p in parts])[o], "dropped": sum(p["dropped"] for p in parts)}
    if "reward_user" in parts[0]:
        out["reward_user"] = np.concatenate([p["reward_user"] for p in parts])[o]
    return out


def assert_eps_equal(a, b, what):
    assert a["dropped"] == b["dropped"] == 0, what
    for k in ("env", "step", "length"):
        assert np.array_equal(a[k], b[k]), f"{what}: {k}"
    for n in STAT_COLUMNS:
        assert_same(a["stats"][n], b["stats"][n], f"{what}: stats {n}")
    assert_same(a["reward"], b["reward"], f"{what}: reward")
    if "reward_user" in a:
        assert_same(a["reward_user"], b["reward_user"], f"{what}: reward_user")


class Loop:
    """The staggered driver loop: episode_tick, pair_noma_episodes, fused step (arrivals: on-device draws), then
    `log.accumulate(done)`.  The actions of global envs [base, base + E) of a `total`-env job."""

    def __init__(self, env, log, spe, base=0, total=None):
        self.env, self.log, self.spe = env, log, spe
        E, V, M, dev = env.E, env.V, env.M, env.device
        g = torch.Generator(device="cpu").manual_seed(99)
        width = (V, 2) if env.variant == "marl" else (2 * V + M,)
        self.raw = (torch.rand(total or E, *width, generator=g) * 2 - 1)[base:base + E].contiguous().to(dev)
        if env.variant == "marl":
            self.act = env.map_actions(self.raw)
            self.obs = torch.empty(E, V, 5, device=dev)
        else:
            self.obs = torch.empty(E, V, M // V + 5, device=dev)
        self.reuse = torch.ones(E, dtype=torch.int32, device=dev)
        self.out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))

    def one(self):
        env = self.env
        start, done = env.episode_tick(steps_per_episode=self.spe, positions_every=1, stages=stages_of(env),
                                       out=self.out)
        if env.variant == "marl":
            part, ng = env.pair_noma_episodes(self.act, start, schedule=YAML_SCHED, reuse=self.reuse)
            env.step_marl_fused(self.raw, part, ng, obs_out=self.obs)
        else:
            env.step_sarl_fused(self.raw, obs_out=self.obs)
        self.log.accumulate(done)

    def run(self, steps, restate=None):
        for _ in range(steps):
            self.one()
            if restate is not None:
                restate.step(self.env, self.out[1])
        torch.cuda.synchronize()

    def run_graph(self, steps):
        cg = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(cg, stream=s):
                self.one()
        torch.cuda.current_stream().wait_stream(s)
        for _ in range(steps):
            cg.replay()
        torch.cuda.synchronize()


# ------------------------------------------------------------------ staggered MARL loop against the restatement
def test_marl_staggered_against_restatement():
    E, spe = 1003, 7  # not a multiple of 4 or 32: the last block and warp have tail envs
    env = make_env(E)
    log = EpisodeLog(env, capacity=4096)
    start_staggered(env, spe)
    loop, ref = Loop(env, log, spe), Restatement(env)
    drains, seen = [], 0
    for _ in range(3):
        loop.run(20, ref)
        want = ref.records(seen)
        assert_same(raw_records(log), want, "records before the drain")
        eps = log.drain()
        assert_drained(eps, want, env.V, "drain")
        assert eps["dropped"] == 0 and int(log.count.item()) == 0
        drains.append(eps)
        seen = len(ref.recs)
    assert_same(log.running.cpu().numpy(), ref.run, "running sums of the open episodes")
    eps = cat_sorted(drains)
    assert len(eps["env"]) > 5 * E
    for e in range(E):
        lens = eps["length"][eps["env"] == e]
        assert lens[0] == spe - e % spe and np.all(lens[1:] == spe), f"env {e}: episode lengths {lens}"
    env.close()


# ------------------------------------------------------------------ SARL
def test_sarl_against_restatement():
    E, spe = 300, 5
    env = make_env(E, "sarl")
    log = EpisodeLog(env, capacity=2048)
    assert tuple(log.running.shape) == (E, NSTAT + 2) and tuple(log.records.shape) == (2048, NSTAT + 4)
    start_staggered(env, spe)
    loop, ref = Loop(env, log, spe), Restatement(env)
    loop.run(23, ref)
    want = ref.records()
    assert_same(raw_records(log), want, "records")
    eps = log.drain()
    assert_drained(eps, want, 0, "SARL drain")
    assert len(eps["env"]) > 3 * E
    for n in STAT_COLUMNS:
        assert np.all(eps["stats"][n] == 0.0), "the SARL step writes no stats"
    assert np.any(eps["reward"] != 0.0)
    assert_same(log.running.cpu().numpy(), ref.run, "running sums")
    env.close()


# ------------------------------------------------------------------ lock-step: done_all
def test_lockstep_done_all_equals_done_tensor():
    E = 257
    env = make_env(E)
    a, b = EpisodeLog(env, capacity=2048), EpisodeLog(env, capacity=2048)
    start_staggered(env, 100, offsets=torch.zeros(E, dtype=torch.int32))
    loop = Loop(env, EpisodeLog(env), 100)  # the loop's own log; `a` and `b` take one accumulate per step
    ones = torch.ones(E, dtype=torch.uint8, device=env.device)
    zeros = torch.zeros(E, dtype=torch.bool, device=env.device)
    ref = Restatement(env)
    for t in range(40):
        loop.run(1)
        flag = t % 10 == 9
        b.accumulate(flag)
        ref.step(env, flag)
        a.accumulate(ones if flag else zeros)
    eb = raw_records(b)
    assert len(eb) == 4 * E
    assert_same(eb, ref.records(), "done_all against the restatement")
    assert_same(raw_records(a), eb, "done tensor vs done_all")
    assert_same(a.running.cpu().numpy(), b.running.cpu().numpy(), "running")
    assert_same(b.running.cpu().numpy(), ref.run, "running against the restatement")
    env.close()


# ------------------------------------------------------------------ graph
def test_graph_replay_equals_eager():
    E, spe = 64, 7
    a = make_env(E)
    start_staggered(a, spe)
    b = make_env(E)
    b.load_state_dict(a.state_dict())
    la, lb = EpisodeLog(a), EpisodeLog(b)
    lb.load_state_dict(la.state_dict())
    Loop(a, la, spe).run(250)
    Loop(b, lb, spe).run_graph(250)
    assert_same(lb.running.cpu().numpy(), la.running.cpu().numpy(), "running sums")
    ea, eb = la.drain(), lb.drain()
    assert len(ea["env"]) > 30 * E
    assert_eps_equal(ea, eb, "eager vs graph")
    assert_fields_equal(a, b, "eager vs graph")
    a.close(); b.close()


# ------------------------------------------------------------------ overflow
def test_overflow_drops_and_counts():
    E, cap, canary = 256, 100, -7.25e300
    env = make_env(E)
    start_staggered(env, 100, offsets=torch.zeros(E, dtype=torch.int32))
    log = EpisodeLog(env, capacity=cap)
    big = torch.full((cap + 40, log.records.shape[1]), canary, dtype=torch.float64, device=env.device)
    log.records = big[:cap]
    loop, ref = Loop(env, log, 100), Restatement(env)
    loop.run(2, ref)
    rng = np.random.default_rng(4)
    done_np = rng.random(E) < 0.7
    done = torch.as_tensor(done_np.astype(np.uint8)).to(env.device)
    loop.one()
    log.accumulate(done)  # a second accumulate of the same step: the restatement adds the step twice too
    ref.step(env, loop.out[1])
    ref.step(env, done)
    n_done = int(done_np.sum())
    assert n_done > cap
    torch.cuda.synchronize()
    assert int(log.count.item()) == n_done
    want = {bits(r).tobytes() for r in ref.records()}
    kept = raw_records(log)
    eps_env = kept[:, 0].astype(np.int64)
    assert len(kept) == cap and len(set(eps_env)) == cap
    assert all(bits(r).tobytes() in want for r in kept), "a kept record is not one of the expected records"
    assert torch.all(big[cap:] == canary), "rows past capacity were written"
    run = log.running.cpu().numpy()
    assert np.all(run[done_np] == 0.0), "running rows of done envs (kept and dropped) are zeroed"
    assert_same(run, ref.run, "running sums")
    eps = log.drain()
    assert eps["dropped"] == n_done - cap and len(eps["env"]) == cap
    assert int(log.count.item()) == 0
    env.close()


# ------------------------------------------------------------------ sharding
def test_sharding_global_env_indices():
    spe = 7
    one = make_env(64, seed=21)
    halves = [make_env(32, seed=21, base=0), make_env(32, seed=21, base=32)]
    offs = torch.arange(64, dtype=torch.int32) % spe
    start_staggered(one, spe, offs)
    l1 = EpisodeLog(one)
    Loop(one, l1, spe).run(60)
    parts = []
    for i, env in enumerate(halves):
        start_staggered(env, spe, offs[32 * i:32 * (i + 1)])
        lg = EpisodeLog(env)
        Loop(env, lg, spe, base=32 * i, total=64).run(60)
        parts.append(lg.drain())
    assert set(parts[1]["env"]) == set(range(32, 64))
    e1 = l1.drain()
    assert len(e1["env"]) > 8 * 64
    assert_eps_equal(e1, cat_sorted(parts), "one handle of 64 vs two of 32")
    one.close()
    for h in halves:
        h.close()


# ------------------------------------------------------------------ resume
def test_resume_from_state_dicts():
    E, spe = 128, 7
    a = make_env(E)
    start_staggered(a, spe)
    la = EpisodeLog(a)
    Loop(a, la, spe).run(11)  # mid-episode for every env, with records not yet drained
    sd_env, sd_log = a.state_dict(), la.state_dict()
    assert sd_log["count"] > 0 and float((sd_log["running"][:, 0] > 0).float().mean()) > 0.8
    Loop(a, la, spe).run(20)
    b = make_env(E)
    b.load_state_dict(sd_env)
    lb = EpisodeLog(b)
    for bad in (dict(sd_log, records=torch.zeros(1, _lib.eplog_rec_cols(0), dtype=torch.float64)),  # a SARL log's
                dict(sd_log, running=sd_log["running"][:, :-1])):
        with pytest.raises(ValueError):
            lb.load_state_dict(bad)
    lb.load_state_dict(sd_log)
    Loop(b, lb, spe).run(20)
    assert_same(lb.running.cpu().numpy(), la.running.cpu().numpy(), "running sums")
    assert_eps_equal(la.drain(), lb.drain(), "original vs resumed")
    a.close(); b.close()


# ------------------------------------------------------------------ launches and arguments
def test_one_launch_and_refused_arguments():
    E = 64
    env = make_env(E)
    log = EpisodeLog(env)
    done = torch.zeros(E, dtype=torch.uint8, device=env.device)
    for d in (done, done.bool(), True, False):
        n0 = env.launch_count
        log.accumulate(d)
        assert env.launch_count == n0 + 1
    bad = [torch.zeros(E, dtype=torch.int32, device=env.device), torch.zeros(E, dtype=torch.float32, device=env.device),
           torch.zeros(E + 1, dtype=torch.uint8, device=env.device), torch.zeros(E, 1, dtype=torch.uint8, device=env.device),
           torch.zeros(E, dtype=torch.uint8), torch.zeros(2 * E, dtype=torch.uint8, device=env.device)[::2],
           np.zeros(E, dtype=np.uint8), 1, None]
    n0 = env.launch_count
    for d in bad:
        with pytest.raises(ValueError):
            log.accumulate(d)
    assert env.launch_count == n0, "a refused done launches nothing"
    lib, h, p = env._lib, env._h, env._p
    call = [h, p(log.running), None, 1, p(log.records), log.capacity, p(log.count), env.stream]
    # NULL handle, running, records or count, and capacity < 1
    for i, v in ((0, None), (1, None), (4, None), (6, None), (5, 0), (5, -1)):
        c = list(call)
        c[i] = v
        assert lib.risvec_episode_accumulate(*c) == -1, f"argument {i} = {v}"
    assert lib.risvec_episode_accumulate(*call) == 0
    with pytest.raises(ValueError):
        EpisodeLog(env, capacity=0)
    env.close()
