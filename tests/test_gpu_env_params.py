"""Per-env step parameters (`risvec_attach_env_params`, `BatchedEnviron.attach_env_params` / `set_env_params`).

Where the same kernel runs on both sides the comparison is bit for bit: the on-device draws are keyed by global env
index and seed, so a handle of 16 envs at `env_index_base = 16 g` draws what envs 16 g .. 16 g + 15 of a 64-env handle
draw.  The kernels are pinned with RISVEC_MARL_PATH / RISVEC_SARL_PATH, which `risvec_create` reads."""
import dataclasses

import numpy as np
import pytest
import torch

from ris_vec_marl_b200 import BatchedEnviron, _lib, encode_groups, marl_yaml_overrides
from ris_vec_marl_b200._lib import ENV_PARAM_COLUMNS, RisvecError
from tests.gpu_backend import GpuBackend
from tests.parity import compare_replays
from tests.replay import OracleBackend, load_golden, oracle_params, replay
from oracle.env_oracle import EnvOracle

pytestmark = pytest.mark.gpu

MARL_COLS = ENV_PARAM_COLUMNS[:10]
SARL_COLS = ("bandwidth", "rate", "t_factor1", "t_factor2", "penalty1", "penalty2")
FACTORS = (1.0, 0.75, 1.5, 1.25)
MARL_V8_TRACES = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate", "over_power")
SARL_TRACES = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
TMA_OR_TCGEN05 = ("k_marl_tma", "k_sarl_mma_tma", "k_sarl_umma", "k_sarl_mma_big")
SHAPES = [(8, 40), (32, 256)]


def cols_of(variant):
    return MARL_COLS if variant == "marl" else SARL_COLS


def group_params(variant, base, g):
    """group g's value of every column the variant reads: each column scaled by its own factor per group, so any two
    groups differ in every column"""
    return {n: float(getattr(base, n)) * FACTORS[(g + i) % 4] for i, n in enumerate(cols_of(variant))}


def pin(monkeypatch):
    for var in ("RISVEC_SARL_PATH", "RISVEC_MARL_PATH", "RISVEC_FORCE_GENERIC"):
        monkeypatch.delenv(var, raising=False)
    monkeypatch.setenv("RISVEC_MARL_PATH", "v8")
    monkeypatch.setenv("RISVEC_SARL_PATH", "mma-ldg")


def make(variant, E, V, M, base=0, seed=5, **over):
    kw = dict(marl_yaml_overrides()) if variant == "marl" else {}
    kw.update(over)
    env = BatchedEnviron(variant, E, V, M, seed=seed, env_index_base=base, **kw)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    if variant == "marl":
        env.optimize_phase_shift(); env.update_channel_gains()
        env.set_pairing(yaml=True)
    return env


class Inputs:
    """the inputs of a `total`-env job: actions, phases, raw actor outputs, arrivals, pairing powers, groups"""

    def __init__(self, variant, total, V, M, T=12, seed=7):
        g = torch.Generator().manual_seed(seed)
        self.variant = variant
        self.act = torch.rand(T, total, 2, V, generator=g)
        self.ph = torch.rand(T, total, M, generator=g) * 6.2831853
        width = (V, 2) if variant == "marl" else (2 * V + M,)
        self.raw = torch.rand(total, *width, generator=g) * 2 - 1
        self.p01 = torch.rand(total, V, generator=g)
        self.start = (torch.arange(total) % 3 == 0).to(torch.uint8)
        self.arr = torch.poisson(torch.full((T, total, V), 2.0), generator=g).to(torch.int32)
        self.partner = torch.as_tensor(np.tile(encode_groups([[v, v + 1] if v + 1 < V else [v]
                                                              for v in range(0, V, 2)], V)[0], (total, 1)))
        self.ngroups = torch.full((total,), (V + 1) // 2, dtype=torch.int32)


def run_calls(env, inp, sl, pairing):
    """The driver calls of one handle on the rows `sl` of `inp`; yields (what, {name: tensor}) after each call"""
    dev = env.device
    r = lambda t: t[sl].contiguous().to(dev)
    rt = lambda t: t[:, sl].contiguous().to(dev)
    if env.variant == "marl":
        traces = MARL_V8_TRACES if env.V <= 8 else MARL_V8_TRACES + ("stats", "last_power")
        if pairing:
            part, ng = env.pair_noma(r(inp.p01), 7, 0.10, recalc_mask=True, new_episode=True)
            yield "pair_noma", {}
            env.ep_index.copy_((torch.arange(sl.start, sl.stop, dtype=torch.int32, device=dev) * 37) % 300)
            env.pair_noma_episodes(r(inp.p01), r(inp.start), schedule=(7, 7, 0.10, 0.25, 200))
            yield "pair_noma_episodes", {}
            part, ng = part.clone(), ng.clone()
        else:
            part, ng = r(inp.partner), r(inp.ngroups)
        yield "rollout_marl", env.rollout_marl(rt(inp.act), part, ng, None, traces=traces)
        yield "rollout_marl arrivals", env.rollout_marl(rt(inp.act), part, ng, rt(inp.arr), traces=traces)
        yield "step_marl_fused", {"obs": env.step_marl_fused(r(inp.raw), part, ng).clone()}
        out = {k: torch.empty(env._trace_shape(k, inp.act.shape[0]), dtype=torch.float32).pin_memory()
               for k in traces}
        env.rollout_marl_host(inp.act[:, sl].contiguous().pin_memory(), part.cpu(), ng.cpu(), None, out)
        torch.cuda.synchronize()
        yield "rollout_marl_host", out
    else:
        yield "rollout_sarl", env.rollout_sarl(rt(inp.act), rt(inp.ph), None)
        yield "rollout_sarl arrivals", env.rollout_sarl(rt(inp.act), rt(inp.ph), rt(inp.arr))
        yield "step_sarl_fused", {"obs": env.step_sarl_fused(r(inp.raw)).clone()}


def same(a, b):
    a, b = a.detach().contiguous(), b.detach().contiguous()
    return a.shape == b.shape and torch.equal(a.view(torch.uint8), b.view(torch.uint8))


def assert_state_equal(a, b, sl, what):
    for k in _lib.FIELDS:
        assert same(a.state(k)[sl].cpu(), b.state(k).cpu()), f"{what}: field {k} differs"


def assert_results_equal(ra, rb, sl, what):
    """rows `sl` of `ra` against `rb`: the observation is [E, ...], every trace [T, E, ...]"""
    assert set(ra) == set(rb)
    for k in ra:
        x = ra[k][sl] if k == "obs" else ra[k][:, sl]
        assert same(x.cpu(), rb[k].cpu()), f"{what}: {k} differs"


# ------------------------------------------------------------------ 1. a uniform table changes nothing
@pytest.mark.parametrize("variant", ["marl", "sarl"])
@pytest.mark.parametrize("V,M", SHAPES)
def test_uniform_table_is_bit_identical(variant, V, M, monkeypatch):
    pin(monkeypatch)
    E = 24
    a, b = make(variant, E, V, M), make(variant, E, V, M)
    table = a.attach_env_params()
    assert tuple(table.shape) == (E, len(ENV_PARAM_COLUMNS)) and table.dtype == torch.float64
    want = torch.tensor([float(getattr(a.params, n)) for n in ENV_PARAM_COLUMNS], dtype=torch.float64)
    assert torch.equal(table.cpu(), want.repeat(E, 1))
    inp = Inputs(variant, E, V, M)
    allrows = slice(0, E)
    for (wa, ra), (wb, rb) in zip(run_calls(a, inp, allrows, V <= 8 and variant == "marl"),
                                  run_calls(b, inp, allrows, V <= 8 and variant == "marl")):
        assert wa == wb and a.last_kernel() == b.last_kernel(), (wa, a.last_kernel(), b.last_kernel())
        assert_results_equal(ra, rb, allrows, wa)
        assert_state_equal(a, b, allrows, wa)
    want_kernel = {("marl", 8): "k_marl_v8", ("marl", 32): "k_marl_rollout", ("sarl", 8): "k_sarl_mma",
                   ("sarl", 32): "k_sarl_cascade2+k_sarl_scan"}[(variant, V)]
    if variant == "sarl":
        b.rollout_sarl(inp.act.to(b.device)[:, :E], inp.ph.to(b.device)[:, :E])
    else:
        b.rollout_marl(inp.act.to(b.device)[:, :E], inp.partner.to(b.device), inp.ngroups.to(b.device),
                       traces=MARL_V8_TRACES if V <= 8 else MARL_V8_TRACES + ("stats", "last_power"))
    assert b.last_kernel() == want_kernel
    a.close(); b.close()


# ------------------------------------------------------------------ 2. each env follows its own row
def group_of(e):
    """neighbouring envs (the 4 envs of a k_marl_v8 warp, the 4 warps of a k_pair_noma block) get different groups,
    and the pattern shifts every 16 envs"""
    return (e % 4 + e // 16) % 4


@pytest.mark.parametrize("variant", ["marl", "sarl"])
@pytest.mark.parametrize("V,M", SHAPES)
def test_each_env_follows_its_row(variant, V, M, monkeypatch):
    """handle A: E envs, env e with group_of(e)'s row; handle B_g: the same E envs with group g's values as its
    params.  A's envs of group g match B_g's bit for bit: every lane reads its own env's row."""
    pin(monkeypatch)
    E = 64
    a = make(variant, E, V, M)
    a.attach_env_params()
    groups = [group_params(variant, a.params, g) for g in range(4)]
    for name in cols_of(variant):
        a.set_env_params(**{name: torch.tensor([groups[group_of(e)][name] for e in range(E)], dtype=torch.float64,
                                               device=a.device)})
    inp = Inputs(variant, E, V, M)
    pairing = variant == "marl" and V <= 8
    allrows = slice(0, E)
    runs_a = list((w, {k: v.clone() for k, v in r.items()}) for w, r in run_calls(a, inp, allrows, pairing))
    state_a = {k: a.state(k).clone() for k in _lib.FIELDS}
    for g in range(4):
        rows = torch.tensor([e for e in range(E) if group_of(e) == g])
        b = make(variant, E, V, M, **groups[g])
        for (wa, ra), (wb, rb) in zip(runs_a, run_calls(b, inp, allrows, pairing)):
            assert wa == wb
            for k in ra:
                x, y = (ra[k][rows], rb[k][rows]) if k == "obs" else (ra[k][:, rows], rb[k][:, rows])
                assert same(x.cpu(), y.cpu()), f"group {g}: {wb}: {k} differs"
        for k in _lib.FIELDS:
            assert same(state_a[k][rows.to(a.device)].cpu(), b.state(k)[rows.to(b.device)].cpu()), \
                f"group {g}: field {k} differs"
        b.close()
    a.close()


# ------------------------------------------------------------------ 3. against the float64 oracle
def split_env(g, e):
    """a golden scenario (inputs and results) restricted to env e: [E, ...] arrays for reset_* and the final queue,
    [episodes or steps, E, ...] for the others"""
    out = {}
    for k, v in g.items():
        if not isinstance(v, np.ndarray) or v.ndim == 0:
            out[k] = v
        elif k.startswith("reset_") or k == "final_mec_queue_cycles":
            out[k] = v[e:e + 1]
        else:
            out[k] = v[:, e:e + 1]
    out["E"] = 1
    return out


@pytest.mark.parametrize("name", ["marl_v8_m40_yaml", "sarl_v8_m40"])
def test_heterogeneous_against_oracle(name):
    """every env of the scenario gets its own row; the oracle runs each env with that env's parameters"""
    g = load_golden(name)
    gpu = GpuBackend(g)
    gpu.env.attach_env_params()
    rows = [group_params(g["variant"], gpu.env.params, e) for e in range(g["E"])]
    for col in cols_of(g["variant"]):
        gpu.env.set_env_params(**{col: torch.tensor([r[col] for r in rows], dtype=torch.float64,
                                                    device=gpu.env.device)})
    got = replay(g, gpu)
    assert gpu.env.last_kernel() == ("k_marl_v8" if g["variant"] == "marl" else "k_sarl_mma")
    for e in range(g["E"]):
        ge = split_env(g, e)
        p = dataclasses.replace(oracle_params(g), **rows[e])
        ob = OracleBackend(ge)
        ob.env = EnvOracle(ge["variant"], ge["V"], ge["M"], 3, E=1, params=p, draws=ob.draws)
        want = replay(ge, ob)
        # the fixture holds results for the default parameters: the expected values are the oracle's
        ref = dict(ge, **{k: v for k, v in want.items() if not k.startswith("step_x_")})
        report = compare_replays(ref, split_env(got, e), want, params=p)
        assert report["checked"] > 10
    gpu.env.close()


# ------------------------------------------------------------------ 4. graph
class Loop:
    """The staggered MARL loop of INTEGRATION.md section 3; every env that starts an episode gets a new P_max, drawn on
    the device from its episode index"""

    def __init__(self, env, spe):
        E, V, dev = env.E, env.V, env.device
        g = torch.Generator().manual_seed(99)
        self.env, self.spe = env, spe
        self.raw = (torch.rand(E, V, 2, generator=g) * 2 - 1).to(dev)
        self.act = env.map_actions(self.raw)
        self.obs = torch.empty(E, V, 5, device=dev)
        self.reuse = torch.ones(E, dtype=torch.int32, device=dev)
        self.out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))
        self.idx = torch.arange(E, dtype=torch.float64, device=dev)

    def one(self):
        env = self.env
        start, done = env.episode_tick(steps_per_episode=self.spe, positions_every=2, out=self.out)
        draw = 1.0 + torch.remainder(env.ep_index.to(torch.float64) * 0.618 + self.idx * 0.37, 1.5)
        env.set_env_params(P_max=torch.where(start.bool(), draw, env.env_params[:, 0]))
        part, ng = env.pair_noma_episodes(self.act, start, schedule=(7, 7, 0.10, 0.25, 200), reuse=self.reuse)
        env.step_marl_fused(self.raw, part, ng, obs_out=self.obs)
        self.log.accumulate(done)


def test_graph_replay_equals_eager():
    from ris_vec_marl_b200 import EpisodeLog
    E, spe, steps = 64, 7, 200
    envs, loops = [], []
    for _ in range(2):
        env = make("marl", E, 8, 40, seed=11)
        env.begin_episode(stages=("reset", "positions", "channel", "pairing"))
        env.ep_step.copy_((torch.arange(E, dtype=torch.int32) % spe).to(env.device))
        env.attach_env_params()
        loop = Loop(env, spe)
        loop.log = EpisodeLog(env, capacity=4096)
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
    assert torch.equal(a.env_params.cpu(), b.env_params.cpu())
    assert len(torch.unique(a.env_params[:, 0])) > 4, "P_max was redrawn per env"
    assert_state_equal(a, b, slice(0, E), "eager vs graph")
    ea, eb = loops[0].log.drain(), loops[1].log.drain()
    assert len(ea["env"]) > 20 * E and ea["dropped"] == eb["dropped"] == 0
    for k in ("env", "step", "length", "reward", "reward_user"):
        assert np.array_equal(ea[k], eb[k]), k
    for k in ea["stats"]:
        assert np.array_equal(ea["stats"][k], eb["stats"][k]), k
    a.close(); b.close()


# ------------------------------------------------------------------ 5. kernel choice and refusals
CHOICE = [  # (variant, V, M, E, entry, kernel with a table)
    ("marl", 8, 40, 8, "rollout", "k_marl_v8"),
    ("marl", 8, 40, 8, "host", "k_marl_v8"),
    ("marl", 8, 40, 8, "fused", "k_marl_v8"),
    ("marl", 12, 40, 4, "fused", "k_marl_rollout"),
    ("sarl", 8, 40, 8, "rollout", "k_sarl_mma"),
    ("sarl", 8, 16, 8, "host", "k_sarl_mma"),
    ("sarl", 8, 40, 8, "fused", "k_sarl_mma"),
    ("sarl", 8, 15, 8, "rollout", "k_sarl_rollout"),
    ("sarl", 8, 15, 8, "fused", "k_sarl_rollout"),
    ("sarl", 12, 128, 4, "rollout", "k_sarl_cascade2+k_sarl_scan"),
    ("sarl", 12, 40, 4, "rollout", "k_sarl_rollout"),
]


def one_call(env, entry, T=4):
    E, V, M, dev = env.E, env.V, env.M, env.device
    g = torch.Generator().manual_seed(3)
    acts = torch.rand(T, E, 2, V, generator=g)
    arr = torch.poisson(torch.full((T, E, V), 2.0), generator=g).to(torch.int32)
    phs = torch.rand(T, E, M, generator=g) * 6.2831853
    part = torch.as_tensor(np.tile(encode_groups([[v] for v in range(V)], V)[0], (E, 1)))
    ng = torch.full((E,), V, dtype=torch.int32)
    if entry == "fused":
        if env.variant == "sarl":
            env.step_sarl_fused((torch.rand(E, 2 * V + M, generator=g) * 2 - 1).to(dev))
        else:
            env.step_marl_fused((torch.rand(E, V, 2, generator=g) * 2 - 1).to(dev), part, ng)
    elif entry == "host":
        names = SARL_TRACES if env.variant == "sarl" else MARL_V8_TRACES[:-1]
        out = {k: torch.empty(env._trace_shape(k, T), dtype=torch.float32) for k in names}
        if env.variant == "sarl":
            env.rollout_sarl_host(acts, phs, arr, out)
        else:
            env.rollout_marl_host(acts, part, ng, arr, out)
    elif env.variant == "sarl":
        env.rollout_sarl(acts.to(dev), phs.to(dev), arr.to(dev))
    else:
        env.rollout_marl(acts.to(dev), part.to(dev), ng.to(dev), arr.to(dev), traces=MARL_V8_TRACES[:-1])
    torch.cuda.synchronize()
    return env.last_kernel()


@pytest.mark.parametrize("variant,V,M,E,entry,kernel", CHOICE)
def test_kernel_choice_with_and_after_table(variant, V, M, E, entry, kernel, monkeypatch):
    for var in ("RISVEC_SARL_PATH", "RISVEC_MARL_PATH", "RISVEC_FORCE_GENERIC"):
        monkeypatch.delenv(var, raising=False)
    env, fresh = make(variant, E, V, M), make(variant, E, V, M)
    env.attach_env_params()
    got = one_call(env, entry)
    assert got == kernel and got not in TMA_OR_TCGEN05
    env.attach_env_params(False)
    assert env.env_params is None
    assert one_call(env, entry) == one_call(fresh, entry)
    env.close(); fresh.close()


@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_packed_records_refuse_a_table(variant):
    E, V, M, T = 8, 8, 40, 4
    env = make(variant, E, V, M)
    env.attach_env_params()
    acts, arr = torch.rand(T, E, 2, V), torch.zeros(T, E, V, dtype=torch.int32)
    rec = env.pack_inputs(acts, arr, torch.rand(T, E, M) if variant == "sarl" else None)
    part = torch.as_tensor(np.tile(encode_groups([[v] for v in range(V)], V)[0], (E, 1)))
    ng = torch.full((E,), V, dtype=torch.int32)
    with pytest.raises(RisvecError) as ex:
        env.rollout_packed(rec.to(env.device), part, ng)
    assert ex.value.code == -2 and "table" in str(ex.value)
    out_rec = torch.empty(T, E // 4, 4 * env.packed_out_words())
    with pytest.raises(RisvecError) as ex:
        env.rollout_packed_host(rec, out_rec, torch.empty(T, E), part, ng)
    assert ex.value.code == -2 and "table" in str(ex.value)
    env.attach_env_params(False)
    env.rollout_packed(rec.to(env.device), part, ng)
    torch.cuda.synchronize()
    env.close()


def test_python_refusals():
    E = 8
    env = make("marl", E, 8, 40)
    with pytest.raises(RuntimeError):
        env.set_env_params(P_max=1.0)
    cols = len(ENV_PARAM_COLUMNS)
    for bad in (torch.zeros(E, cols + 1, dtype=torch.float64, device=env.device),
                torch.zeros(E, cols, dtype=torch.float32, device=env.device),
                torch.zeros(E, cols, dtype=torch.float64),
                torch.zeros(cols, E, dtype=torch.float64, device=env.device).t()):
        with pytest.raises(ValueError):
            env.attach_env_params(table=bad)
        assert env.env_params is None
    mine = torch.zeros(E, cols, dtype=torch.float64, device=env.device)
    assert env.attach_env_params(table=mine) is mine
    with pytest.raises(RuntimeError):
        env.attach_env_params()   # a second table would leave a captured graph on the first one
    assert env.env_params is mine
    with pytest.raises(ValueError):
        env.set_env_params(bogus=1.0)
    with pytest.raises(ValueError):
        env.set_env_params(time_fast=0.002)   # per handle
    with pytest.raises(ValueError):
        env.set_env_params(P_max=torch.ones(E + 1, device=env.device))
    with pytest.raises(ValueError):
        env.set_env_params(P_max=torch.ones(E, dtype=torch.float64))   # host tensor
    with pytest.raises(ValueError):
        env.set_env_params(P_max=torch.ones(E, device=env.device))   # float32 would round the values
    env.set_env_params(P_max=2.5, rate=torch.arange(E, dtype=torch.float64, device=env.device))
    assert torch.all(mine[:, 0] == 2.5) and torch.equal(mine[:, 3].cpu(), torch.arange(E, dtype=torch.float64))
    env.close()


@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_state_dict_round_trip(variant, monkeypatch):
    pin(monkeypatch)
    E, V, M = 16, 8, 40
    a = make(variant, E, V, M)
    a.attach_env_params()
    for name in cols_of(variant):
        a.set_env_params(**{name: torch.tensor([group_params(variant, a.params, e % 4)[name] for e in range(E)],
                                               dtype=torch.float64, device=a.device)})
    inp = Inputs(variant, E, V, M)
    list(run_calls(a, inp, slice(0, E), False))
    sd = a.state_dict()
    assert "_env_params" in sd and torch.equal(sd["_env_params"], a.env_params)
    b = make(variant, E, V, M, seed=5)
    b.load_state_dict(sd)
    assert b.env_params is not None and torch.equal(b.env_params, a.env_params)
    assert_state_equal(a, b, slice(0, E), "after load")
    for (wa, ra), (wb, rb) in zip(run_calls(a, inp, slice(0, E), False), run_calls(b, inp, slice(0, E), False)):
        assert_results_equal(ra, rb, slice(0, E), f"resumed {wa}")
        assert_state_equal(a, b, slice(0, E), f"resumed {wa}")
    sd.pop("_env_params")
    c = make(variant, E, V, M)
    c.load_state_dict(sd)   # a state dict without a table loads as before: no table is attached
    assert c.env_params is None
    b.load_state_dict(sd)   # ... and a handle that has one detaches it: it follows the saved params again
    assert b.env_params is None
    a.close(); b.close(); c.close()
