"""Per-env RIS size (`risvec_attach_ris_elements`, `BatchedEnviron.attach_ris_elements` / `set_ris_elements`).

An env whose RIS is the first n elements of an M-element array is an env of a handle with M = n: the geometry
phasors depend on m only and every quantity that depends on M is a sum over the elements.  The MARL episode kernels
are therefore compared bit for bit against one handle per size (the on-device draws are keyed by global env index and
seed, not by M), the SARL step against the float64 oracle run with M = n.  Kernels are pinned with RISVEC_*_PATH,
which `risvec_create` reads."""
import dataclasses
import os

import numpy as np
import pytest
import torch

from oracle.env_oracle import EnvOracle, InjectedDraws, OracleParams
from ris_vec_marl_b200 import BatchedEnviron, EpisodeLog, _lib, encode_groups, marl_yaml_overrides
from ris_vec_marl_b200._lib import RisvecError
from tests.gpu_backend import kernel_paths
from tests.parity import RTOL, sarl_rate_atol, sarl_reward_band

pytestmark = pytest.mark.gpu

SIZES = (20, 40, 60, 80, 100, 120)
SARL_TRACES = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
MARL_TRACES = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate", "over_power")


def clear_paths(monkeypatch):
    for var in ("RISVEC_SARL_PATH", "RISVEC_MARL_PATH", "RISVEC_FORCE_GENERIC"):
        monkeypatch.delenv(var, raising=False)


def make(variant, E, V, M, sarl=None, marl=None, generic=False, seed=5, base=0, **over):
    kw = dict(marl_yaml_overrides()) if variant == "marl" else {}
    kw.update(over)
    old = os.environ.get("RISVEC_FORCE_GENERIC")
    os.environ["RISVEC_FORCE_GENERIC"] = "1" if generic else "0"
    try:
        with kernel_paths(sarl=sarl, marl=marl):
            env = BatchedEnviron(variant, E, V, M, seed=seed, env_index_base=base, **kw)
    finally:
        if old is None:
            os.environ.pop("RISVEC_FORCE_GENERIC")
        else:
            os.environ["RISVEC_FORCE_GENERIC"] = old
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    if variant == "marl":
        env.set_pairing(yaml=True)
    return env


def same(a, b):
    a, b = a.detach().contiguous().cpu(), b.detach().contiguous().cpu()
    return a.shape == b.shape and torch.equal(a.view(torch.uint8), b.view(torch.uint8))


def assert_state_equal(a, b, what, rows=None):
    for k in _lib.FIELDS:
        x, y = a.state(k), b.state(k)
        if rows is not None:
            x, y = x[rows], y[rows]
        assert same(x, y), f"{what}: field {k} differs"


def cycling(E, sizes=SIZES, device="cuda"):
    """counts[e] = sizes[e % len(sizes)]: the four envs of a k_bcd_v8 warp get four different counts"""
    return torch.tensor([sizes[e % len(sizes)] for e in range(E)], dtype=torch.int32, device=device)


class SarlInputs:
    def __init__(self, E, V, M, T=12, seed=7):
        g = torch.Generator().manual_seed(seed)
        self.act = torch.rand(T, E, 2, V, generator=g).cuda()
        self.ph = (torch.rand(T, E, M, generator=g) * 6.2831853).cuda()
        self.arr = torch.poisson(torch.full((T, E, V), 2.0), generator=g).to(torch.int32).cuda()
        self.raw = (torch.rand(E, 2 * V + M, generator=g) * 2 - 1).cuda()


def sarl_calls(env, inp):
    """yields (what, {name: tensor}) after each SARL call"""
    yield "rollout_sarl", env.rollout_sarl(inp.act, inp.ph, None)
    yield "rollout_sarl arrivals", env.rollout_sarl(inp.act, inp.ph, inp.arr)
    yield "step_sarl_fused", {"obs": env.step_sarl_fused(inp.raw, inp.arr[0]).clone()}
    T = inp.act.shape[0]
    out = {k: torch.empty(env._trace_shape(k, T), dtype=torch.float32).pin_memory() for k in SARL_TRACES}
    env.rollout_sarl_host(inp.act.cpu().pin_memory(), inp.ph.cpu().pin_memory(), inp.arr.cpu().pin_memory(), out)
    torch.cuda.synchronize()
    yield "rollout_sarl_host", out


def compare_runs(a, b, calls):
    for (wa, ra), (wb, rb) in zip(calls(a), calls(b)):
        assert wa == wb and a.last_kernel() == b.last_kernel(), (wa, a.last_kernel(), b.last_kernel())
        assert set(ra) == set(rb)
        for k in ra:
            assert same(ra[k], rb[k]), f"{wa}: {k} differs"
        assert_state_equal(a, b, wa)


# ------------------------------------------------------------------ 1. full counts = no array, on the same kernel
SARL_FULL = [(8, 40, "mma-ldg", "k_sarl_mma"), (8, 15, "generic", "k_sarl_rollout"),
             (32, 256, "generic", "k_sarl_cascade2+k_sarl_scan")]


@pytest.mark.parametrize("V,M,path,kernel", SARL_FULL)
def test_sarl_full_counts_are_bit_identical(V, M, path, kernel, monkeypatch):
    clear_paths(monkeypatch)
    E = 24
    a, b = make("sarl", E, V, M, sarl=path), make("sarl", E, V, M, sarl=path)
    counts = a.attach_ris_elements()
    assert counts.dtype == torch.int32 and torch.equal(counts.cpu(), torch.full((E,), M, dtype=torch.int32))
    inp = SarlInputs(E, V, M)
    compare_runs(a, b, lambda env: sarl_calls(env, inp))
    a.rollout_sarl(inp.act, inp.ph, inp.arr)
    assert a.last_kernel() == kernel
    a.close(); b.close()


def marl_channel(env):
    env.optimize_phase_shift()
    yield "optimize_phase_shift", {}
    env.update_channel_gains()
    yield "update_channel_gains", {}


def marl_episodes(env, spe=3):
    env.begin_episode(stages=("reset", "positions", "channel", "pairing"))
    yield "begin_episode", {}
    env.ep_step.copy_(torch.arange(env.E, dtype=torch.int32, device=env.device) % spe)
    out = None
    for t in range(2 * spe):
        out = env.episode_tick(steps_per_episode=spe, positions_every=2, out=out)
        yield f"episode_tick {t}", {"start": out[0].clone(), "done": out[1].clone()}


@pytest.mark.parametrize("V,M,generic", [(8, 40, False), (8, 40, True), (32, 256, False)])
def test_marl_full_counts_are_bit_identical(V, M, generic, monkeypatch):
    """k_bcd_v8 + k_gains_free_v and the fused k_begin_episode (V = 8), the per-stage fallback k_bcd + k_gains_free
    (RISVEC_FORCE_GENERIC) and k_bcd + k_gains_free_v with per-stage episode starts (V = 32)"""
    clear_paths(monkeypatch)
    E = 24
    a, b = make("marl", E, V, M, generic=generic), make("marl", E, V, M, generic=generic)
    a.attach_ris_elements()
    for calls in (marl_channel, marl_episodes):
        for (wa, ra), (wb, rb) in zip(calls(a), calls(b)):
            for k in ra:
                assert same(ra[k], rb[k]), f"{wa}: {k} differs"
            assert_state_equal(a, b, wa)
    a.close(); b.close()


# ------------------------------------------------------------------ 2. MARL = one handle of that size
@pytest.mark.parametrize("generic", [False, True])
def test_marl_equals_a_handle_of_that_size(generic, monkeypatch):
    clear_paths(monkeypatch)
    E, V, spe, T = 48, 8, 3, 6
    a = make("marl", E, V, 120, marl="v8", generic=generic)
    counts = a.attach_ris_elements(counts=cycling(E))
    assert len(set(counts[:4].tolist())) == 4
    handles = {n: make("marl", E, V, n, marl="v8", generic=generic) for n in SIZES}
    g = torch.Generator().manual_seed(3)
    acts = torch.rand(T, E, 2, V, generator=g).cuda()
    part = torch.as_tensor(np.tile(encode_groups([[v, v + 1] for v in range(0, V, 2)], V)[0], (E, 1))).cuda()
    ng = torch.full((E,), V // 2, dtype=torch.int32, device="cuda")

    def check(what):
        for n, b in handles.items():
            rows = (counts == n).nonzero().flatten()
            assert same(a.theta_re[rows, :n], b.theta_re[rows]), f"{what}: theta_re, n = {n}"
            assert same(a.theta_im[rows, :n], b.theta_im[rows]), f"{what}: theta_im, n = {n}"
            assert same(a.gains[rows], b.gains[rows]), f"{what}: gains, n = {n}"

    for env in [a, *handles.values()]:
        env.begin_episode(stages=("positions", "channel", "pairing"))
    check("begin_episode")
    for env in [a, *handles.values()]:
        env.ep_step.copy_(torch.arange(E, dtype=torch.int32, device=env.device) % spe)
    outs = {id(env): None for env in [a, *handles.values()]}
    for t in range(2 * spe):
        for env in [a, *handles.values()]:
            outs[id(env)] = env.episode_tick(steps_per_episode=spe, positions_every=2, out=outs[id(env)])
        check(f"tick {t}")
    got = a.rollout_marl(acts, part, ng, None, traces=MARL_TRACES)
    for n, b in handles.items():
        rows = (counts == n).nonzero().flatten()
        want = b.rollout_marl(acts, part, ng, None, traces=MARL_TRACES)
        assert a.last_kernel() == b.last_kernel()
        for k in MARL_TRACES:
            assert same(got[k][:, rows], want[k][:, rows]), f"rollout_marl {k}, n = {n}"
        b.close()
    a.close()


# ------------------------------------------------------------------ 3. SARL against the float64 oracle
def reset_draws(rng, E, V):
    pattern = [(0, 4), (220, 230), (10, 15), (170, 180), (10, 15), (220, 230), (10, 15), (170, 180), (10, 15)] * (V // 4)
    pattern += [(5, 9)]
    return np.stack([rng.integers(lo, hi, E) for lo, hi in pattern], axis=1).astype(np.int32)


def close(got, want, atol, what, mask=None):
    got, want = np.asarray(got, float), np.asarray(want, float)
    bad = np.abs(got - want) > atol + RTOL * np.abs(want)
    if mask is not None:
        bad &= ~mask
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} out of tolerance, max abs err {np.abs(got - want)[bad].max():.3g}"


SARL_ORACLE = [("auto", 8, 40, "rollout", "k_sarl_mma"), ("auto", 8, 40, "fused", "k_sarl_mma"),
               ("generic", 8, 40, "rollout", "k_sarl_rollout"),
               ("generic", 8, 64, "rollout", "k_sarl_cascade2+k_sarl_scan")]
PARAM_FACTORS = (1.0, 0.75, 1.5, 1.25)
SARL_COLS = ("bandwidth", "rate", "t_factor1", "t_factor2", "penalty1", "penalty2")


@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("path,V,M,entry,kernel", SARL_ORACLE)
def test_sarl_heterogeneous_against_oracle(path, V, M, entry, kernel, table, monkeypatch):
    """4096 envs, counts spread over 1 .. M; with `table`, a per-env parameter table as well (group e % 4).  The
    oracle runs each group of equal (count, parameters) with M = n and phase[..., :n]."""
    clear_paths(monkeypatch)
    E, T = 4096, 16
    sizes = sorted({1, 2, 7, M // 4, M // 2 + 1, M - 2, M - 1, M})
    rng = np.random.default_rng(11)
    ri, mob = reset_draws(rng, E, V), rng.random((E, 8 * V))
    acts = rng.random((T, E, 2, V)).astype(np.float32)
    phs = (rng.random((T, E, M)) * 2 * np.pi).astype(np.float32)
    arr = rng.poisson(3.0, (T, E, V)).astype(np.int32)
    raw = (rng.random((T, E, 2 * V + M)) * 2 - 1).astype(np.float32)
    with kernel_paths(sarl=None if path == "auto" else path):
        env = BatchedEnviron("sarl", E, V, M)
    env.make_new_game(ri); env.renew_positions(mob); env.compute_parms()
    counts = cycling(E, sizes)
    env.attach_ris_elements(counts=counts)
    group = np.arange(E) % 4 if table else np.zeros(E, dtype=int)
    base = OracleParams()
    prm = [{c: getattr(base, c) * PARAM_FACTORS[(g + i) % 4] for i, c in enumerate(SARL_COLS)} for g in range(4)]
    if table:
        env.attach_env_params()
        for c in SARL_COLS:
            env.set_env_params(**{c: torch.tensor([prm[g][c] for g in group], dtype=torch.float64, device="cuda")})
    if entry == "rollout":
        got = {k: v.cpu().numpy() for k, v in env.rollout_sarl(acts, phs, arr).items()}
    else:  # the fused driver step, one step per call; the oracle gets the mapped actions
        got = {k: [] for k in ("rate", "DataBuf", "reward")}
        for t in range(T):
            r = torch.as_tensor(raw[t]).cuda()
            a_t, p_t = env.map_actions(r)
            acts[t], phs[t] = a_t.cpu().numpy(), p_t.cpu().numpy()
            env.step_sarl_fused(r, torch.as_tensor(arr[t]).cuda())
            for k, f in (("rate", "vehicle_rate"), ("DataBuf", "DataBuf"), ("reward", "reward")):
                got[k].append(env.state(f).cpu().numpy().copy())
        got = {k: np.stack(v) for k, v in got.items()}
    assert env.last_kernel() == kernel, (env.last_kernel(), kernel)
    n_e = counts.cpu().numpy()
    checked = 0
    for n in sizes:
        for g in sorted(set(group.tolist())):
            idx = np.nonzero((n_e == n) & (group == g))[0]
            p = dataclasses.replace(base, **prm[g]) if table else base
            d = InjectedDraws(reset_ints=ri[idx], arrivals=arr[:, idx])
            o = EnvOracle("sarl", V, n, 3, E=len(idx), params=p, draws=d)
            o.make_new_game()
            d.set_mobility_uniforms(mob[idx])
            o.renew_positions(); o.compute_parms()
            ra = sarl_rate_atol(n)
            n_band = 0
            for t in range(T):
                rew, over_p = o.step_sarl(acts[t][idx], phs[t][idx, :n])
                band = sarl_reward_band(o.last["buf_signed"], o.over_data, n).any(axis=1)
                n_band += int(band.sum())
                what = f"n = {n}, group {g}, t = {t}"
                close(got["rate"][t][idx], o.vehicle_rate, ra, f"rate {what}")
                close(got["DataBuf"][t][idx], o.DataBuf, 4 * ra, f"DataBuf {what}")
                close(got["reward"][t][idx], rew, 4e-6, f"reward {what}", mask=band)
                if entry == "rollout":
                    close(got["data_p"][t][idx], o.data_p, 1e-5, f"data_p {what}")
                    close(got["over_data"][t][idx], o.over_data, 4 * ra, f"over_data {what}")
                    close(got["over_power"][t][idx], over_p, 4e-6 + 0.7 * ra, f"over_power {what}")
            assert n_band <= 0.05 * len(idx) * T
            checked += len(idx)
    assert checked == E
    env.close()


# ------------------------------------------------------------------ 4. absent elements do nothing; 5. clamping
@pytest.mark.parametrize("V,M,path", [(8, 40, "mma-ldg"), (8, 15, "generic"), (32, 256, "generic")])
def test_sarl_absent_columns_and_clamping(V, M, path, monkeypatch):
    clear_paths(monkeypatch)
    E = 24
    counts = cycling(E, (1, 3, M // 2, M - 1, M))
    a, b = make("sarl", E, V, M, sarl=path), make("sarl", E, V, M, sarl=path)
    a.attach_ris_elements(counts=counts.clone())
    b.attach_ris_elements(counts=counts.clone())
    inp = SarlInputs(E, V, M)
    other = SarlInputs(E, V, M, seed=99)
    absent = torch.arange(M, device="cuda")[None, :] >= counts[:, None]        # [E, M]
    inp_b = SarlInputs(E, V, M)
    inp_b.ph = torch.where(absent[None], other.ph, inp.ph)
    inp_b.raw[:, 2 * V:] = torch.where(absent, other.raw[:, 2 * V:], inp.raw[:, 2 * V:])
    for (wa, ra), (wb, rb) in zip(sarl_calls(a, inp), sarl_calls(b, inp_b)):
        for k in ra:
            # the observation's first M / V columns per vehicle echo the phases the caller gave, absent ones included
            x, y = (ra[k][..., M // V:], rb[k][..., M // V:]) if k == "obs" else (ra[k], rb[k])
            assert same(x, y), f"absent columns changed {wa}: {k}"
    # out-of-range counts: 0 and negative act as 1, above M as M
    c, d = make("sarl", E, V, M, sarl=path), make("sarl", E, V, M, sarl=path)
    wild = counts.clone()
    wild[counts == 1] = torch.tensor([0, -7], dtype=torch.int32, device="cuda").repeat(E)[: int((counts == 1).sum())]
    wild[counts == M] = M + 1000
    c.attach_ris_elements(counts=wild)
    d.attach_ris_elements(counts=counts.clone())
    compare_runs(c, d, lambda env: sarl_calls(env, inp))
    for env in (a, b, c, d):
        env.close()


@pytest.mark.parametrize("generic", [False, True])
def test_marl_absent_elements_and_clamping(generic, monkeypatch):
    clear_paths(monkeypatch)
    E, V, M = 24, 8, 40
    counts = cycling(E, (1, 5, 20, 39, 40, 17))
    a, b = make("marl", E, V, M, generic=generic), make("marl", E, V, M, generic=generic)
    for env in (a, b):
        env.attach_ris_elements(counts=counts.clone())
    g = torch.Generator().manual_seed(5)
    ph = (torch.rand(E, M, generator=g) * 6.28).cuda()
    ph2 = torch.where(torch.arange(M, device="cuda")[None, :] >= counts[:, None], ph.flip(1) + 1.0, ph)
    ix = torch.randint(0, 8, (E, M), generator=g, dtype=torch.int32).cuda()
    ix2 = torch.where(torch.arange(M, device="cuda")[None, :] >= counts[:, None], (ix + 3) % 8, ix)
    for set_a, set_b in ((lambda: a.get_next_phase(ph), lambda: b.get_next_phase(ph2)),
                         (lambda: a.Random_phase(ix), lambda: b.Random_phase(ix2))):
        set_a(); set_b()
        a.update_channel_gains(); b.update_channel_gains()
        assert same(a.gains, b.gains), "theta of absent elements changed the gains"
        th_b = b.theta_re.clone()
        a.optimize_phase_shift(); b.optimize_phase_shift()
        present = torch.arange(M, device="cuda")[None, :] < counts[:, None]
        assert same(a.theta_re[present], b.theta_re[present]) and same(a.theta_im[present], b.theta_im[present])
        assert same(b.theta_re[~present], th_b[~present]), "the BCD wrote theta of absent elements"
    # clamping: 0 / negative -> 1, above M -> M
    c, d = make("marl", E, V, M, generic=generic), make("marl", E, V, M, generic=generic)
    wild = counts.clone()
    wild[counts == 1] = 0
    wild[counts == 17] = -3
    wild[counts == M] = 4 * M
    c.attach_ris_elements(counts=wild)
    tame = counts.clone()
    tame[counts == 17] = 1
    d.attach_ris_elements(counts=tame)
    for calls in (marl_channel, marl_episodes):
        for (wc, _), (wd, _) in zip(calls(c), calls(d)):
            assert_state_equal(c, d, f"clamped {wc}")
    for env in (a, b, c, d):
        env.close()


# ------------------------------------------------------------------ 6. graphs
class MarlLoop:
    """The staggered MARL loop of INTEGRATION.md section 3; every env that starts an episode at this tick draws a new
    RIS size, on the device, from its episode index"""

    def __init__(self, env, spe):
        E, V, dev = env.E, env.V, env.device
        g = torch.Generator().manual_seed(99)
        self.env, self.spe = env, spe
        self.raw = (torch.rand(E, V, 2, generator=g) * 2 - 1).to(dev)
        self.act = env.map_actions(self.raw)
        self.obs = torch.empty(E, V, 5, device=dev)
        self.reuse = torch.ones(E, dtype=torch.int32, device=dev)
        self.out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))
        self.idx = torch.arange(E, dtype=torch.int32, device=dev)
        self.log = EpisodeLog(env, capacity=4096)

    def redraw(self):
        env = self.env
        draw = 20 + 20 * torch.remainder(env.ep_index * 7 + self.idx * 3, 6).to(torch.int32)
        env.set_ris_elements(torch.where(env.ep_step == 0, draw, env.ris_elements))

    def one(self):
        env = self.env
        self.redraw()
        start, done = env.episode_tick(steps_per_episode=self.spe, positions_every=2, out=self.out)
        part, ng = env.pair_noma_episodes(self.act, start, schedule=(7, 7, 0.10, 0.25, 200), reuse=self.reuse)
        env.step_marl_fused(self.raw, part, ng, obs_out=self.obs)
        self.log.accumulate(done)


class SarlLoop:
    def __init__(self, env, spe):
        E, V, M, dev = env.E, env.V, env.M, env.device
        g = torch.Generator().manual_seed(98)
        self.env, self.spe = env, spe
        self.raw = (torch.rand(E, 2 * V + M, generator=g) * 2 - 1).to(dev)
        self.obs = torch.empty(E, V, M // V + 5, device=dev)
        self.out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))
        self.idx = torch.arange(E, dtype=torch.int32, device=dev)

    def one(self):
        env = self.env
        draw = 8 + torch.remainder(env.ep_index * 5 + self.idx, env.M - 7).to(torch.int32)
        env.set_ris_elements(torch.where(env.ep_step == 0, draw, env.ris_elements))
        env.episode_tick(steps_per_episode=self.spe, positions_every=2, stages=("positions",), out=self.out)
        env.step_sarl_fused(self.raw, obs_out=self.obs)


@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_graph_replay_equals_eager(variant, monkeypatch):
    clear_paths(monkeypatch)
    E, spe, steps = 64, 7, 200
    M = 120 if variant == "marl" else 40
    envs, loops = [], []
    for _ in range(2):
        env = make(variant, E, 8, M, seed=11)
        env.attach_ris_elements(counts=cycling(E, (20, 40, 60, 80, 100, 120) if variant == "marl" else (8, 16, 40)))
        env.begin_episode(stages=("reset", "positions", "channel", "pairing") if variant == "marl" else
                          ("reset", "positions"))
        env.ep_step.copy_((torch.arange(E, dtype=torch.int32) % spe).to(env.device))
        loop = MarlLoop(env, spe) if variant == "marl" else SarlLoop(env, spe)
        envs.append(env); loops.append(loop)
    for _ in range(steps):
        loops[0].one()
    cg, s = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(cg, stream=s):
            loops[1].one()
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(steps):
        cg.replay()
    torch.cuda.synchronize()
    a, b = envs
    assert torch.equal(a.ris_elements.cpu(), b.ris_elements.cpu())
    assert len(torch.unique(a.ris_elements)) >= 4, "the count was redrawn per env"
    assert_state_equal(a, b, "eager vs graph")
    if variant == "marl":
        ea, eb = loops[0].log.drain(), loops[1].log.drain()
        assert len(ea["env"]) > 20 * E and ea["dropped"] == eb["dropped"] == 0
        for k in ("env", "step", "length", "reward", "reward_user"):
            assert np.array_equal(ea[k], eb[k]), k
        for k in ea["stats"]:
            assert np.array_equal(ea["stats"][k], eb["stats"][k]), k
    a.close(); b.close()


# ------------------------------------------------------------------ 7. with a per-env parameter table: MARL
def test_marl_with_table_equals_one_handle_per_value(monkeypatch):
    """counts cycle over SIZES and each size has its own parameter group: env e of the M = 120 handle matches the
    handle with M = n and that group's params, bit for bit"""
    clear_paths(monkeypatch)
    E, V, T = 48, 8, 6
    a = make("marl", E, V, 120, marl="v8")
    counts = a.attach_ris_elements(counts=cycling(E))
    cols = _lib.ENV_PARAM_COLUMNS[:10]
    groups = {n: {c: float(getattr(a.params, c)) * PARAM_FACTORS[(i + j) % 4] for j, c in enumerate(cols)}
              for i, n in enumerate(SIZES)}
    a.attach_env_params()
    for c in cols:
        a.set_env_params(**{c: torch.tensor([groups[int(n)][c] for n in counts.tolist()], dtype=torch.float64,
                                            device="cuda")})
    handles = {n: make("marl", E, V, n, marl="v8", **groups[n]) for n in SIZES}
    g = torch.Generator().manual_seed(4)
    acts = torch.rand(T, E, 2, V, generator=g).cuda()
    p01 = torch.rand(E, V, generator=g).cuda()
    for env in [a, *handles.values()]:
        env.begin_episode(stages=("positions", "channel", "pairing"))
        env.pair_noma(p01, 7, 0.10, recalc_mask=True, new_episode=True)
    got = a.rollout_marl(acts, a.noma_partner.clone(), a.noma_ngroups.clone(), None, traces=MARL_TRACES)
    assert a.last_kernel() == "k_marl_v8"
    for n, b in handles.items():
        rows = (counts == n).nonzero().flatten()
        want = b.rollout_marl(acts, b.noma_partner.clone(), b.noma_ngroups.clone(), None, traces=MARL_TRACES)
        assert same(a.gains[rows], b.gains[rows]), f"gains, n = {n}"
        for k in MARL_TRACES:
            assert same(got[k][:, rows], want[k][:, rows]), f"{k}, n = {n}"
        b.close()
    a.close()


# ------------------------------------------------------------------ 8. API
CHOICE = [  # (variant, V, M, E, entry, kernel with an array, launches)
    ("sarl", 8, 40, 8, "rollout", "k_sarl_mma", 1),
    ("sarl", 8, 16, 8, "host", "k_sarl_mma", None),
    ("sarl", 8, 40, 8, "fused", "k_sarl_mma", 1),
    ("sarl", 8, 15, 8, "rollout", "k_sarl_rollout", 1),
    ("sarl", 8, 15, 8, "fused", "k_sarl_rollout", 3),   # odd M: map_actions, rollout, observe
    ("sarl", 12, 128, 4, "rollout", "k_sarl_cascade2+k_sarl_scan", 2),
    ("sarl", 32, 256, 4, "rollout", "k_sarl_cascade2+k_sarl_scan", 2),
    ("marl", 8, 40, 8, "rollout", "k_marl_tma", None),   # MARL never reads M: the choice without an array
    ("marl", 8, 40, 8, "fused", "k_marl_v8", 1),
]


def one_call(env, entry, T=4):
    E, V, M, dev = env.E, env.V, env.M, env.device
    g = torch.Generator().manual_seed(3)
    acts = torch.rand(T, E, 2, V, generator=g)
    arr = torch.poisson(torch.full((T, E, V), 2.0), generator=g).to(torch.int32)
    phs = torch.rand(T, E, M, generator=g) * 6.2831853
    part = torch.as_tensor(np.tile(encode_groups([[v] for v in range(V)], V)[0], (E, 1)))
    ng = torch.full((E,), V, dtype=torch.int32)
    torch.cuda.synchronize()
    n0 = env.launch_count
    if entry == "fused":
        if env.variant == "sarl":
            env.step_sarl_fused((torch.rand(E, 2 * V + M, generator=g) * 2 - 1).to(dev))
        else:
            env.step_marl_fused((torch.rand(E, V, 2, generator=g) * 2 - 1).to(dev), part, ng)
    elif entry == "host":
        out = {k: torch.empty(env._trace_shape(k, T), dtype=torch.float32) for k in SARL_TRACES}
        env.rollout_sarl_host(acts, phs, arr, out)
    elif env.variant == "sarl":
        env.rollout_sarl(acts.to(dev), phs.to(dev), arr.to(dev))
    else:
        env.rollout_marl(acts.to(dev), part.to(dev), ng.to(dev), arr.to(dev), traces=MARL_TRACES[:-1])
    torch.cuda.synchronize()
    return env.last_kernel(), env.launch_count - n0


@pytest.mark.parametrize("variant,V,M,E,entry,kernel,launches", CHOICE)
def test_kernel_choice_with_and_after_array(variant, V, M, E, entry, kernel, launches, monkeypatch):
    clear_paths(monkeypatch)
    env, fresh = make(variant, E, V, M), make(variant, E, V, M)
    env.attach_ris_elements()
    got, n = one_call(env, entry)
    assert got == kernel
    if launches is not None:
        assert n == launches
    env.attach_ris_elements(False)
    assert env.ris_elements is None
    assert one_call(env, entry) == one_call(fresh, entry)
    env.close(); fresh.close()


@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_packed_records(variant, monkeypatch):
    """the packed SARL records are refused while an array is attached; MARL's step never reads M, so its packed form
    runs and matches the handle without an array"""
    clear_paths(monkeypatch)
    E, V, M, T = 8, 8, 40, 4
    env, fresh = make(variant, E, V, M), make(variant, E, V, M)
    env.attach_ris_elements()
    acts, arr = torch.rand(T, E, 2, V), torch.zeros(T, E, V, dtype=torch.int32)
    rec = env.pack_inputs(acts, arr, torch.rand(T, E, M) if variant == "sarl" else None)
    part = torch.as_tensor(np.tile(encode_groups([[v] for v in range(V)], V)[0], (E, 1)))
    ng = torch.full((E,), V, dtype=torch.int32)
    if variant == "marl":
        ra = env.rollout_packed(rec.to(env.device), part, ng)
        rb = fresh.rollout_packed(rec.to(fresh.device), part, ng)
        assert env.last_kernel() == fresh.last_kernel()
        assert all(same(x, y) for x, y in zip(ra, rb))
    else:
        with pytest.raises(RisvecError) as ex:
            env.rollout_packed(rec.to(env.device), part, ng)
        assert ex.value.code == -2 and "RIS size" in str(ex.value)
        out_rec = torch.empty(T, E // 4, 4 * env.packed_out_words())
        with pytest.raises(RisvecError) as ex:
            env.rollout_packed_host(rec, out_rec, torch.empty(T, E), part, ng)
        assert ex.value.code == -2 and "RIS size" in str(ex.value)
        env.attach_ris_elements(False)
        env.rollout_packed(rec.to(env.device), part, ng)
    torch.cuda.synchronize()
    env.close(); fresh.close()


def test_python_refusals():
    E = 8
    env = make("sarl", E, 8, 40)
    with pytest.raises(RuntimeError):
        env.set_ris_elements(3)
    for bad in (torch.zeros(E + 1, dtype=torch.int32, device="cuda"),
                torch.zeros(E, dtype=torch.int64, device="cuda"),
                torch.zeros(E, dtype=torch.float32, device="cuda"),
                torch.zeros(E, dtype=torch.int32),
                torch.zeros(2 * E, dtype=torch.int32, device="cuda")[::2]):
        with pytest.raises(ValueError):
            env.attach_ris_elements(counts=bad)
        assert env.ris_elements is None
    mine = torch.full((E,), 7, dtype=torch.int32, device="cuda")
    assert env.attach_ris_elements(counts=mine) is mine and env.ris_elements is mine
    with pytest.raises(RuntimeError):
        env.attach_ris_elements()   # a second array would leave a captured graph on the first one
    for bad in (torch.ones(E, dtype=torch.int64, device="cuda"), torch.ones(E, dtype=torch.int32),
                torch.ones(E + 1, dtype=torch.int32, device="cuda")):
        with pytest.raises(ValueError):
            env.set_ris_elements(bad)
    env.set_ris_elements(12)
    assert torch.all(mine == 12)
    env.set_ris_elements(torch.arange(E, dtype=torch.int32, device="cuda"))
    assert torch.equal(mine.cpu(), torch.arange(E, dtype=torch.int32))
    env.close()


@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_state_dict_round_trip(variant, monkeypatch):
    clear_paths(monkeypatch)
    E, V, M = 16, 8, 40
    a = make(variant, E, V, M)
    a.attach_ris_elements(counts=cycling(E, (5, 16, 33, 40)))
    inp = SarlInputs(E, V, M)
    if variant == "marl":
        calls = lambda env: marl_channel(env)
    else:
        calls = lambda env: sarl_calls(env, inp)
    list(calls(a))
    sd = a.state_dict()
    assert "_ris_elements" in sd and torch.equal(sd["_ris_elements"], a.ris_elements)
    b = make(variant, E, V, M)
    b.load_state_dict(sd)
    assert b.ris_elements is not None and torch.equal(b.ris_elements, a.ris_elements)
    assert_state_equal(a, b, "after load")
    compare_runs(a, b, calls)
    sd.pop("_ris_elements")
    b.load_state_dict(sd)   # a state without an array detaches one
    assert b.ris_elements is None
    a.close(); b.close()
