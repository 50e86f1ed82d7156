"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference
fixtures.  Run on the B200 box: pytest -m gpu."""
import numpy as np
import pytest
import torch

from tests.parity import compare_replays
from tests.replay import OracleBackend, golden_names, load_golden, replay

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "GPU tests selected but no CUDA device"
    from ris_vec_marl_b200 import load_library

    load_library()  # fails loudly when the extension is missing


@pytest.mark.parametrize("mode", ["fast", "generic"])
@pytest.mark.parametrize("name", golden_names())
def test_fixture_parity_single_steps(name, mode):
    from tests.gpu_backend import GpuBackend

    g = load_golden(name)
    got = replay(g, GpuBackend(g, mode=mode))
    want = replay(g, OracleBackend(g))
    rep = compare_replays(g, got, want)
    assert rep["checked"] >= 12


@pytest.mark.parametrize("mode", ["fast", "generic"])
@pytest.mark.parametrize("name", ["marl_v8_m40_yaml", "sarl_v8_m40", "sarl_v32_m256", "marl_v6_m7_ragged",
                                  "sarl_v5_m33_ragged"])
def test_fused_rollout_equals_single_steps(name, mode):
    """One launch over T steps must give bit-identical traces and final state to T launches
    (odd and even T, so both the paired loop and the tail of the fast kernels are hit)."""
    from tests.gpu_backend import FAST_MARL_TRACES, GpuBackend

    g = load_golden(name)
    T = g["T"] - (1 if name == "marl_v8_m40_yaml" else 0)
    a, b = GpuBackend(g, mode=mode), GpuBackend(g, mode=mode)
    for be in (a, b):
        be.make_new_game()
        be.renew_positions(g["ep_mob_uniforms"][0])
        be.compute_parms()
        if g["variant"] == "marl":
            be.optimize_phase_shift()
            be.update_channel_gains()
    acts = torch.as_tensor(g["actions"][:T]).cuda()
    arr = torch.as_tensor(g["arrivals"][:T].astype(np.int32)).cuda()
    if g["variant"] == "marl":
        part = g["ep_partner"][0].astype(np.int32)
        ng = np.asarray(g["ep_ngroups"][0], dtype=np.int32)
        tr = FAST_MARL_TRACES if mode == "fast" else FAST_MARL_TRACES + ("over_power", "stats", "last_power")
        fused = a.env.rollout_marl(acts, part, ng, arr, traces=tr)
        single = [b.env.step_marl(acts[t], part, ng, arr[t], traces=tr) for t in range(T)]
    else:
        ph = torch.as_tensor(g["phases"][:T]).cuda()
        fused = a.env.rollout_sarl(acts, ph, arr)
        single = [b.env.step_sarl(acts[t], ph[t], arr[t], traces=tuple(fused)) for t in range(T)]
    for k, v in fused.items():
        assert torch.equal(v, torch.stack([s[k] for s in single])), k
    for f in ("DataBuf", "data_t", "data_p", "vehicle_rate", "reward", "reward_user", "mec_queue_cycles", "step_ctr",
              "stats", "last_power_W", "over_power", "over_data", "data_r", "phase_real"):
        assert torch.equal(a.env.state(f), b.env.state(f)), f


def test_fast_and_generic_kernels_agree():
    """The shape-specialised kernels against the shape-generic ones on the same inputs:
    identical integer/float64 state, float32 traces within a few ulp (different summation
    trees in the cascaded reduction, MUFU log2 vs log1pf in the MARL rate)."""
    from tests.gpu_backend import FAST_MARL_TRACES, GpuBackend

    for name in ("marl_v8_m40_yaml", "sarl_v8_m40"):
        g = load_golden(name)
        T = g["T"]
        envs = [GpuBackend(g, mode=m) for m in ("fast", "generic")]
        outs = []
        for be in envs:
            be.make_new_game(); be.renew_positions(g["ep_mob_uniforms"][0]); be.compute_parms()
            acts = torch.as_tensor(g["actions"][:T]).cuda()
            arr = torch.as_tensor(g["arrivals"][:T].astype(np.int32)).cuda()
            if g["variant"] == "marl":
                be.optimize_phase_shift(); be.update_channel_gains()
                outs.append(be.env.rollout_marl(acts, g["ep_partner"][0].astype(np.int32),
                                                np.asarray(g["ep_ngroups"][0], dtype=np.int32), arr,
                                                traces=FAST_MARL_TRACES))
            else:
                outs.append(be.env.rollout_sarl(acts, torch.as_tensor(g["phases"][:T]).cuda(), arr))
        for k in outs[0]:
            np.testing.assert_allclose(outs[0][k].cpu().numpy(), outs[1][k].cpu().numpy(), rtol=2e-5, atol=2e-5,
                                       err_msg=f"{name}:{k}")
        assert torch.equal(envs[0].env.data_r, envs[1].env.data_r)


def test_host_buffer_entry_point_matches_device_path():
    from ris_vec_marl_b200 import BatchedEnviron

    E, V, M, T = 64, 8, 40, 16
    gen = torch.Generator().manual_seed(3)
    acts = torch.rand(T, E, 2, V, generator=gen).pin_memory()
    ph = (torch.rand(T, E, M, generator=gen) * 6.2831853).pin_memory()
    arr = torch.poisson(torch.full((T, E, V), 3.0), generator=gen).to(torch.int32).pin_memory()
    envs = [BatchedEnviron("sarl", E, V, M, seed=5) for _ in range(2)]
    for e in envs:
        e.make_new_game()
        e.renew_positions()
        e.compute_parms()
    dev = envs[0].rollout_sarl(acts.cuda(), ph.cuda(), arr.cuda())
    host = {k: torch.empty(v.shape, dtype=torch.float32).pin_memory() for k, v in dev.items()}
    envs[1].rollout_sarl_host(acts, ph, arr, host)
    torch.cuda.synchronize()
    for k in dev:
        assert torch.equal(dev[k].cpu(), host[k]), k
    assert torch.equal(envs[0].DataBuf, envs[1].DataBuf)


def test_device_rng_is_deterministic_and_shard_invariant():
    """Philox draws are keyed by the GLOBAL env index: 1 x 64 envs == 2 shards x 32 envs."""
    from ris_vec_marl_b200 import BatchedEnviron

    V, M, T = 8, 40, 50
    full = BatchedEnviron("sarl", 64, V, M, seed=99)
    lo = BatchedEnviron("sarl", 32, V, M, seed=99, env_index_base=0)
    hi = BatchedEnviron("sarl", 32, V, M, seed=99, env_index_base=32)
    gen = torch.Generator().manual_seed(1)
    acts = torch.rand(T, 64, 2, V, generator=gen).cuda()
    ph = (torch.rand(T, 64, M, generator=gen) * 6.28).cuda()
    for e in (full, lo, hi):
        e.make_new_game()
        e.renew_positions()
        e.compute_parms()
    a = full.rollout_sarl(acts, ph)
    b = lo.rollout_sarl(acts[:, :32].contiguous(), ph[:, :32].contiguous())
    c = hi.rollout_sarl(acts[:, 32:].contiguous(), ph[:, 32:].contiguous())
    for k in a:
        assert torch.equal(a[k], torch.cat([b[k], c[k]], dim=1)), k
    assert torch.equal(full.pos_x, torch.cat([lo.pos_x, hi.pos_x]))
    # arrivals ~ Poisson(rate = 3): mean and variance over 64*8*50 draws
    d = full.data_r.double()
    assert d.min() >= 0
    tr = a["DataBuf"]
    assert torch.isfinite(tr).all()


def test_device_poisson_moments():
    from ris_vec_marl_b200 import BatchedEnviron

    E, V, M = 2048, 8, 40
    env = BatchedEnviron("sarl", E, V, M, seed=7, rate=3.0)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    draws = []
    z = torch.zeros(E, 2, V, device="cuda")
    ph = torch.zeros(E, M, device="cuda")
    for _ in range(8):
        env.step_sarl(z, ph)
        draws.append(env.data_r.clone())
    d = torch.stack(draws).double()
    n = d.numel()
    assert abs(d.mean().item() - 3.0) < 5 * (3.0 / n) ** 0.5
    assert abs(d.var().item() - 3.0) < 0.1
    assert not torch.equal(draws[0], draws[1])


def test_host_pipeline_multi_chunk_and_shard_stats():
    """4096 envs x 64 steps = several pipeline chunks: the chunked host entry must be bit-identical
    to one device launch (SARL and MARL), and shard_stats must equal the column sums."""
    from ris_vec_marl_b200 import BatchedEnviron, encode_groups, marl_yaml_overrides

    E, V, M, T = 4096, 8, 40, 64
    gen = torch.Generator().manual_seed(11)
    acts = torch.rand(T, E, 2, V, generator=gen).pin_memory()
    ph = (torch.rand(T, E, M, generator=gen) * 6.2831853).pin_memory()
    arr = torch.poisson(torch.full((T, E, V), 2.0), generator=gen).to(torch.int32).pin_memory()
    # SARL
    envs = [BatchedEnviron("sarl", E, V, M, seed=5) for _ in range(2)]
    for e in envs:
        e.make_new_game(); e.renew_positions(); e.compute_parms()
    dev = envs[0].rollout_sarl(acts.cuda(), ph.cuda(), arr.cuda())
    host = {k: torch.empty(v.shape, dtype=torch.float32).pin_memory() for k, v in dev.items()}
    envs[1].rollout_sarl_host(acts, ph, arr, host)
    torch.cuda.synchronize()
    for k in dev:
        assert torch.equal(dev[k].cpu(), host[k]), k
    assert torch.equal(envs[0].DataBuf, envs[1].DataBuf)
    st = envs[0].shard_stats().cpu()
    assert abs(st[16].item() - envs[0].reward.double().sum().item()) < 1e-6
    # MARL
    part, ng = encode_groups([[0, 1], [2, 3], [4, 5], [6], [7]], V)
    partner = torch.as_tensor(np.tile(part, (E, 1))).pin_memory()
    ngroups = torch.full((E,), ng, dtype=torch.int32).pin_memory()
    envs = [BatchedEnviron("marl", E, V, M, seed=6, **marl_yaml_overrides()) for _ in range(2)]
    for e in envs:
        e.make_new_game(); e.renew_positions(); e.compute_parms(); e.optimize_phase_shift(); e.update_channel_gains()
    names = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")
    dev = envs[0].rollout_marl(acts.cuda(), partner.cuda(), ngroups.cuda(), arr.cuda(), traces=names)
    host = {k: torch.empty(v.shape, dtype=torch.float32).pin_memory() for k, v in dev.items()}
    envs[1].rollout_marl_host(acts, partner, ngroups, arr, host)
    torch.cuda.synchronize()
    for k in dev:
        assert torch.equal(dev[k].cpu(), host[k]), k
    assert torch.equal(envs[0].mec_queue_cycles, envs[1].mec_queue_cycles)
    st = envs[0].shard_stats().cpu().numpy()
    want = envs[0].stats.double().sum(dim=0).cpu().numpy()
    np.testing.assert_allclose(st[:16], want, rtol=1e-12, atol=1e-9)
    assert abs(st[16] - envs[0].reward.double().sum().item()) < 1e-6


def test_packed_records_are_bit_identical_to_per_array_api():
    """The packed record entry points (device and pinned-host pipelines) against the per-array
    ones: same kernels' arithmetic, so every trace and the final state must match bit for bit."""
    from ris_vec_marl_b200 import BatchedEnviron, RisvecError, encode_groups, marl_yaml_overrides
    from tests.gpu_backend import kernel_paths

    E, V, M, T = 1028, 8, 40, 37  # odd T; E % 4 == 0 as the tiled layout requires
    gen = torch.Generator().manual_seed(21)
    acts = torch.rand(T, E, 2, V, generator=gen)
    ph = torch.rand(T, E, M, generator=gen) * 6.2831853
    arr = torch.poisson(torch.full((T, E, V), 2.0), generator=gen).to(torch.int32)
    for variant in ("sarl", "marl"):
        over = marl_yaml_overrides() if variant == "marl" else {}
        with kernel_paths(sarl="v8"):  # the packed SARL records run k_sarl_v8: compare with the same kernel's per-array form
            envs = [BatchedEnviron(variant, E, V, M, seed=5, **over) for _ in range(3)]
        for e in envs:
            e.make_new_game(); e.renew_positions(); e.compute_parms()
            if variant == "marl":
                e.optimize_phase_shift(); e.update_channel_gains()
        if variant == "sarl":
            ref = envs[0].rollout_sarl(acts.cuda(), ph.cuda(), arr.cuda())
            rec = envs[1].pack_inputs(acts, arr, ph)
            extra = {}
        else:
            part, ng = encode_groups([[0, 1], [3, 2], [4, 5], [6], [7]], V)
            extra = dict(partner=torch.as_tensor(np.tile(part, (E, 1))), ngroups=torch.full((E,), ng, dtype=torch.int32))
            names = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")
            ref = envs[0].rollout_marl(acts.cuda(), extra["partner"], extra["ngroups"], arr.cuda(), traces=names)
            rec = envs[1].pack_inputs(acts, arr)
        out_rec, rew = envs[1].rollout_packed(rec.cuda(), **extra)
        got = envs[1].unpack_outputs(out_rec, rew)
        h_out = torch.empty(out_rec.shape).pin_memory()
        h_rew = torch.empty(rew.shape).pin_memory()
        pinned = {k: v.pin_memory() for k, v in extra.items()}
        envs[2].rollout_packed_host(rec.pin_memory(), h_out, h_rew, **pinned)
        torch.cuda.synchronize()
        got_h = envs[2].unpack_outputs(h_out, h_rew)
        for k, v in ref.items():
            assert torch.equal(v, got[k]), (variant, k)
            assert torch.equal(v.cpu(), got_h[k]), (variant, "host", k)
        for f in ("DataBuf", "vehicle_rate", "reward", "mec_queue_cycles", "step_ctr", "stats", "phase_real"):
            assert torch.equal(envs[0].state(f), envs[1].state(f)) and torch.equal(envs[0].state(f), envs[2].state(f)), f
    odd = BatchedEnviron("sarl", 6, 8, 40)  # E % 4 != 0: the tiled layout does not apply
    with pytest.raises(RisvecError):
        odd.rollout_packed(torch.zeros(2, 6 * (24 + 40)))


def test_observation_and_action_mapping_match_the_driver_formulas():
    """Device glue vs a numpy restatement of the drivers' own functions
    (marl_train_bcd.py:819-827,1601-1608; ddpg_train.py:47-73,151-160)."""
    from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides

    E, V, M = 33, 8, 40
    rng = np.random.default_rng(5)
    # MARL
    env = BatchedEnviron("marl", E, V, M, **marl_yaml_overrides())
    env.make_new_game(); env.renew_positions(); env.compute_parms(); env.optimize_phase_shift(); env.update_channel_gains()
    raw = (rng.random((E, V, 2)) * 2.2 - 1.1).astype(np.float32)
    act = env.map_actions(raw).cpu().numpy()
    c = np.clip(raw, -0.999, 0.999)
    want = np.stack([(c[..., 0] + 1) / 2, np.maximum((c[..., 1] + 1) / 2, 0.10)], axis=1)
    np.testing.assert_allclose(act, want, rtol=1e-6, atol=1e-7)
    part = np.full((E, V), -1, dtype=np.int32)
    env.step_marl(act, part, np.full(E, V, dtype=np.int32))
    obs = env.observe().cpu().numpy()
    f = lambda n: env.state(n).cpu().numpy().astype(np.float64)
    want = np.stack([f("DataBuf") / 10, f("data_t") / 10, f("data_p") / 10, f("over_data") / 10, f("vehicle_rate") / 20], -1)
    np.testing.assert_allclose(obs, want, rtol=1e-6, atol=1e-7)
    # SARL
    env = BatchedEnviron("sarl", E, V, M)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    raw = (rng.random((E, 2 * V + M)) * 2.2 - 1.1).astype(np.float32)
    act, ph = (t.cpu().numpy() for t in env.map_actions(raw))
    c = (np.clip(raw, -0.999, 0.999) + 1) / 2
    np.testing.assert_allclose(act, c[:, :2 * V].reshape(E, 2, V), rtol=1e-6)
    np.testing.assert_allclose(ph, c[:, 2 * V:] * np.pi * 2, rtol=1e-6)
    env.step_sarl(act, ph)
    obs = env.observe().cpu().numpy()
    f = lambda n: env.state(n).cpu().numpy().astype(np.float64)
    th = f("phase_real").reshape(E, V, M // V)
    want = np.concatenate([th, np.stack([f("DataBuf") / 10, f("data_t") / 10, f("data_p") / 10, f("over_data") / 10,
                                         f("vehicle_rate") / 20], -1)], axis=-1)
    np.testing.assert_allclose(obs, want, rtol=1e-6, atol=1e-7)
    assert obs.reshape(E, -1).shape[1] == 80  # the DDPG input size of ddpg_train.py:75


@pytest.mark.parametrize("model,K_dB", [("3gpp_umi", 0.0), ("3gpp_uma", 0.0), ("3gpp_umi", 6.0), ("bogus", 0.0)])
def test_3gpp_channel_branch_matches_oracle(model, K_dB):
    """update_channel_gains for channel_model != "free" (MARL/Environment.py:275-327) with injected
    LOS / shadowing / small-scale draws; an unknown keyword falls back to path loss 0 dB (:315-317)."""
    from oracle.env_oracle import EnvOracle, InjectedDraws, OracleParams
    from ris_vec_marl_b200 import BatchedEnviron

    E, V, M = 37, 8, 40
    rng = np.random.default_rng(9)
    pat = [(0, 4), (220, 230), (10, 15), (170, 180), (10, 15), (220, 230), (10, 15), (170, 180), (10, 15)] * 2 + [(5, 9)]
    ints = np.stack([rng.integers(lo, hi, E) for lo, hi in pat], axis=1).astype(np.int32)
    c_rand, c_norm, c_exp = rng.random((E, V)), rng.standard_normal((E, V, 3)), rng.exponential(1.0, (E, V))
    env = BatchedEnviron("marl", E, V, M, channel_model=model, rician_K_dB=K_dB)
    env.make_new_game(ints)
    env.update_channel_gains(c_rand, c_norm, c_exp)
    p = OracleParams()
    p.channel_model, p.rician_K_dB = model, K_dB
    d = InjectedDraws(reset_ints=ints)
    o = EnvOracle("marl", V, M, 3, E=E, params=p, draws=d)
    o.make_new_game()
    # the oracle pops per vehicle: rand, normal, then exponential or two more normals
    n_norm = 1 if K_dB <= 1e-6 else 3
    d.set_channel_draws(c_rand, c_norm[:, :, :n_norm].reshape(E, -1), c_exp)
    o.update_channel_gains()
    np.testing.assert_allclose(env.gains.cpu().numpy(), o.channel_gains, rtol=1e-11)
    # on-device Philox draws: finite, positive, reproducible per (seed, env index)
    env.update_channel_gains()
    g1 = env.gains.clone()
    assert torch.isfinite(g1).all() and (g1 > 0).all()


def test_checkpoint_roundtrip_and_attribute_writes():
    """state_dict / load_state_dict resume bit-exactly; parameter writes between episodes
    (marl_train_bcd.py:563-594) take effect on the next launch."""
    from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides

    E, V, M, T = 64, 8, 40, 10
    gen = torch.Generator(device="cuda").manual_seed(4)
    acts = torch.rand(2 * T, E, 2, V, device="cuda", generator=gen)
    part = torch.full((E, V), -1, dtype=torch.int32, device="cuda")
    ng = torch.full((E,), V, dtype=torch.int32, device="cuda")
    a = BatchedEnviron("marl", E, V, M, seed=3, **marl_yaml_overrides())
    a.make_new_game(); a.renew_positions(); a.compute_parms(); a.optimize_phase_shift(); a.update_channel_gains()
    a.rollout_marl(acts[:T], part, ng)
    sd = a.state_dict()
    ref = a.rollout_marl(acts[T:], part, ng)
    b = BatchedEnviron("marl", E, V, M, seed=3, **marl_yaml_overrides())
    b.load_state_dict(sd)
    got = b.rollout_marl(acts[T:], part, ng)  # on-device arrivals continue from the restored step counters
    for k in ref:
        assert torch.equal(ref[k], got[k]), k
    b.load_state_dict(sd)
    b.set_params(w_d=2.0, w_e=0.0, qos_penalty=0.0)
    got2 = b.rollout_marl(acts[T:], part, ng)
    assert torch.equal(got2["rate"], ref["rate"]) and not torch.equal(got2["reward_user"], ref["reward_user"])
    want = -(2.0 * b.stats[:, 0])  # reward = -(w_d * delay) when w_e = 0 and no QoS penalty
    np.testing.assert_allclose(b.reward.cpu().numpy(), want.cpu().numpy(), rtol=1e-5, atol=1e-7)


def test_resumed_run_continues_the_random_streams():
    """A run that is checkpointed, loaded into a FRESH handle (default parameters, counters at zero) and
    resumed must equal the uninterrupted run: the on-device Philox draws of renew_positions and make_new_game
    are keyed by host-side call counters, which `state_dict` carries along with the params and the arena."""
    from ris_vec_marl_b200 import BatchedEnviron, ReplayBuffer, marl_yaml_overrides

    E, V, M, T = 32, 8, 40, 6
    gen = torch.Generator(device="cuda").manual_seed(9)
    acts = torch.rand(3 * T, E, 2, V, device="cuda", generator=gen)
    part = torch.full((E, V), -1, dtype=torch.int32, device="cuda")
    ng = torch.full((E,), V, dtype=torch.int32, device="cuda")

    def episode(env, k):
        env.renew_positions(); env.compute_parms(); env.optimize_phase_shift(); env.update_channel_gains()
        return env.rollout_marl(acts[k * T:(k + 1) * T], part, ng)

    whole = BatchedEnviron("marl", E, V, M, seed=11, **marl_yaml_overrides())
    whole.make_new_game()
    ref = [episode(whole, k) for k in range(3)]
    first = BatchedEnviron("marl", E, V, M, seed=11, **marl_yaml_overrides())
    first.make_new_game()
    episode(first, 0)
    sd = first.state_dict()
    resumed = BatchedEnviron("marl", E, V, M, seed=11)  # NOT given the yaml overrides: they come from the checkpoint
    resumed.load_state_dict(sd)
    for k in (1, 2):
        got = episode(resumed, k)
        for name in ref[k]:
            assert torch.equal(ref[k][name], got[name]), (k, name)
    assert torch.equal(whole.pos_x, resumed.pos_x) and torch.equal(whole.DataBuf, resumed.DataBuf)
    # replay memory: mem_cntr travels with the arrays
    rb = ReplayBuffer(64, 5, V + 2, V)
    st = torch.rand(8, V * 5, device="cuda")
    rb.store_transitions(st, torch.rand(8, V * (V + 2), device="cuda"), torch.rand(8, device="cuda"),
                         torch.rand(8, V, device="cuda"), st, False)
    rb2 = ReplayBuffer(64, 5, V + 2, V)
    rb2.load_state_dict(rb.state_dict())
    assert rb2.mem_cntr == rb.mem_cntr == 8 and torch.equal(rb2.state_memory, rb.state_memory)


def test_masked_reset_touches_only_the_selected_envs():
    """risvec_make_new_game_masked / risvec_pair_reset_masked: envs outside the mask keep every field."""
    from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides

    E, V, M = 64, 8, 40
    rng = np.random.default_rng(5)
    pat = [(0, 4), (220, 230), (10, 15), (170, 180), (10, 15), (220, 230), (10, 15), (170, 180), (10, 15)] * (V // 4) + [(5, 9)]
    ri = np.stack([rng.integers(lo, hi, E) for lo, hi in pat], axis=1).astype(np.int32)
    env = BatchedEnviron("marl", E, V, M, seed=2, **marl_yaml_overrides())
    env.make_new_game(); env.renew_positions(); env.compute_parms(); env.optimize_phase_shift(); env.update_channel_gains()
    env.rollout_marl(torch.rand(5, E, 2, V, device="cuda"), torch.full((E, V), -1, dtype=torch.int32, device="cuda"),
                     torch.full((E,), V, dtype=torch.int32, device="cuda"))
    env.pair_hist.fill_(0.25)
    before = {k: env.state(k).clone() for k in ("pos_x", "pos_y", "dir", "vel", "DataBuf", "pair_hist", "noma_ngroups")}
    mask = torch.zeros(E, dtype=torch.bool, device="cuda")
    mask[::3] = True
    env.make_new_game(ri, mask=mask)
    env.pair_reset(mask=mask)
    full = BatchedEnviron("marl", E, V, M, seed=2, **marl_yaml_overrides())
    full.make_new_game(ri)
    for k in ("pos_x", "pos_y", "dir", "vel", "DataBuf"):
        assert torch.equal(env.state(k)[~mask], before[k][~mask]), k          # untouched
        assert torch.equal(env.state(k)[mask], full.state(k)[mask]), k        # exactly a reset with the same draws
    assert torch.equal(env.pair_hist[~mask], before["pair_hist"][~mask]) and (env.pair_hist[mask] == 0).all()
    with pytest.raises(ValueError):  # preallocated traces are validated before their pointers reach a kernel
        env.rollout_marl(torch.rand(5, E, 2, V, device="cuda"), torch.full((E, V), -1, dtype=torch.int32, device="cuda"),
                         torch.full((E,), V, dtype=torch.int32, device="cuda"),
                         out={"rate": torch.empty(4, E, V, device="cuda")})


def test_shared_statistics_accumulator_single_process():
    """`dist.SharedStats` (risvec_shared_buffer_*): the owner's side of the peer-memory statistics reduction.
    (The mapping by a second process and the equality with an NCCL all-reduce: tools/check_shared_stats.py
    under torchrun.)"""
    from ris_vec_marl_b200 import BatchedEnviron
    from ris_vec_marl_b200._lib import NSTAT
    from ris_vec_marl_b200.dist import SharedStats

    E, V, M = 256, 8, 40
    env = BatchedEnviron("sarl", E, V, M, seed=5)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    shared = SharedStats(0, 0, 1)
    shared.zero_()
    local = torch.zeros(NSTAT + 1, dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    for _ in range(3):
        env.step_sarl(torch.rand(E, 2, V, device="cuda", generator=g), torch.rand(E, M, device="cuda", generator=g) * 6.28)
        env.shard_stats(out=local, accumulate=True)              # per-rollout sums stay local ...
        env.shard_stats(out=shared.tensor, accumulate=True)      # ... or go straight into the accumulator
    shared.add_(local)                                           # the per-interval push
    total = shared.read()
    assert torch.equal(total, 2.0 * local.cpu()) and float(total[NSTAT]) != 0.0
    shared.close()


@pytest.mark.parametrize("V,inject", [(8, True), (8, False), (5, True), (12, True)])
def test_fused_driver_step_is_bit_identical_to_the_three_calls(V, inject):
    """risvec_step_marl_fused (SURVEY.md 8f row 1: action mapping in the step kernel's prologue, observation in
    its epilogue) against map_actions -> step_marl -> observe on a twin env: every state view and the observation
    are bit-identical over several steps (V = 12: the shapes the fused kernel does not take run the three kernels
    from the one call)."""
    from ris_vec_marl_b200 import BatchedEnviron, encode_groups, marl_yaml_overrides

    E, M = 130, 40
    envs = [BatchedEnviron("marl", E, V, M, seed=11, **marl_yaml_overrides()) for _ in range(2)]
    for env in envs:
        env.make_new_game(); env.renew_positions(); env.compute_parms(); env.optimize_phase_shift(); env.update_channel_gains()
    groups = [[i, i + 1] for i in range(0, V - 2, 2)] + [[V - 1]]
    part, ng = encode_groups(groups, V)
    partner = torch.as_tensor(np.tile(part, (E, 1))).cuda()
    ngroups = torch.full((E,), ng, dtype=torch.int32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(3)
    for step in range(5):
        raw = torch.rand(E, V, 2, device="cuda", generator=g) * 2.2 - 1.1   # beyond [-1, 1]: the clip is exercised
        arr = torch.poisson(torch.full((E, V), 1.0, device="cuda"), generator=g).to(torch.int32) if inject else None
        a, b = envs
        obs_a = a.step_marl_fused(raw, partner, ngroups, arr)
        b.step_marl(b.map_actions(raw), partner, ngroups, arr)
        obs_b = b.observe()
        assert torch.equal(obs_a, obs_b), f"observation differs at step {step}"
        for name in ("DataBuf", "data_t", "data_p", "vehicle_rate", "reward", "reward_user", "over_power", "mec_queue_cycles", "stats", "last_power_W", "data_r"):
            va, vb = getattr(a, name), getattr(b, name)
            assert torch.equal(va, vb), f"{name} differs at step {step}"
    assert envs[0].last_kernel() == ("k_marl_v8" if V <= 8 else "k_marl_rollout")


@pytest.mark.parametrize("V,M,inject", [(8, 40, True), (8, 40, False), (5, 30, True), (8, 64, True), (12, 48, True)])
def test_fused_sarl_driver_step_is_bit_identical_to_the_three_calls(V, M, inject):
    """risvec_step_sarl_fused against map_actions -> step_sarl -> observe on a twin env ((12, 48): a shape the
    fused kernel does not take runs the three kernels from the one call)."""
    from ris_vec_marl_b200 import BatchedEnviron
    from tests.gpu_backend import kernel_paths

    E = 70
    with kernel_paths(sarl="mma"):   # both twins on the tensor-core kernel (the fused form lives in k_sarl_mma)
        envs = [BatchedEnviron("sarl", E, V, M, seed=21) for _ in range(2)]
    for env in envs:
        env.make_new_game(); env.renew_positions(); env.compute_parms()
    g = torch.Generator(device="cuda").manual_seed(4)
    for step in range(5):
        raw = torch.rand(E, 2 * V + M, device="cuda", generator=g) * 2.2 - 1.1
        arr = torch.poisson(torch.full((E, V), 3.0, device="cuda"), generator=g).to(torch.int32) if inject else None
        a, b = envs
        obs_a = a.step_sarl_fused(raw, arr)
        act, ph = b.map_actions(raw)
        b.step_sarl(act, ph, arr)
        obs_b = b.observe()
        assert torch.equal(obs_a, obs_b), f"observation differs at step {step}: {(obs_a - obs_b).abs().max()}"
        for name in ("DataBuf", "data_t", "data_p", "vehicle_rate", "reward", "over_power", "over_data", "phase_real", "data_r"):
            assert torch.equal(getattr(a, name), getattr(b, name)), f"{name} differs at step {step}"


@pytest.mark.parametrize("variant,path,kernel,E", [("sarl", "mma", "k_sarl_mma_tma", 4096), ("sarl", "v8", "k_sarl_v8", 4096),
                                                    ("marl", "tma", "k_marl_tma", 4096), ("marl", "v8", "k_marl_v8", 516)])
def test_attached_statistics_accumulator_equals_shard_stats(variant, path, kernel, E):
    """risvec_attach_stats_accumulator: the statistics pass folded into the rollout (k_sarl_mma_tma / k_marl_tma add
    their last step's sums in the kernel tail; other kernels are followed by k_shard_stats) gives what a
    shard_stats() call after every rollout gives (float64 sums of the same float32 values: order only)."""
    from ris_vec_marl_b200 import BatchedEnviron, encode_groups, marl_yaml_overrides
    from tests.gpu_backend import kernel_paths

    V, M, T = 8, 40, 40
    with kernel_paths(sarl=path if variant == "sarl" else "auto", marl=path if variant == "marl" else "tma"):
        over = marl_yaml_overrides() if variant == "marl" else {}
        envs = [BatchedEnviron(variant, E, V, M, seed=9, **over) for _ in range(2)]
    rng = np.random.default_rng(5)
    for env in envs:
        env.make_new_game(); env.renew_positions(); env.compute_parms()
        if variant == "marl":
            env.optimize_phase_shift(); env.update_channel_gains()
    a, b = envs
    a.attach_stats_accumulator()
    want = torch.zeros(17, dtype=torch.float64, device="cuda")
    part, ng = encode_groups([[0, 1], [2, 3], [4], [5, 6], [7]], V)
    partner = np.tile(part, (E, 1)); ngroups = np.full(E, ng, np.int32)
    for r in range(3):
        acts = rng.random((T, E, 2, V)).astype(np.float32)
        arr = rng.poisson(2.0, (T, E, V)).astype(np.int32)
        for env in envs:
            if variant == "sarl":
                phs = (np.random.default_rng(r).random((T, E, M)) * 6.28).astype(np.float32)
                env.rollout_sarl(acts, phs, arr)
            else:
                env.rollout_marl(acts, partner, ngroups, arr, traces=("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate"))
        assert a.last_kernel() == kernel, a.last_kernel()
        b.shard_stats(out=want, accumulate=True)
    got = a.collect_stats()
    assert torch.equal(a.collect_stats(), torch.zeros_like(got)), "collect clears the accumulator"
    w = want.cpu().numpy(); g_ = got.cpu().numpy()
    assert np.abs(w).max() > 0
    np.testing.assert_allclose(g_, w, rtol=1e-12, atol=1e-9 * np.abs(w).max())
    # the host-buffer form counts the last chunk only
    if variant == "sarl" and path == "mma":
        h = lambda x: torch.as_tensor(x).pin_memory()  # noqa: E731
        out = {k: torch.empty((T, E) if k == "reward" else (T, E, V), dtype=torch.float32).pin_memory()
               for k in ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")}
        a.rollout_sarl_host(h(acts), h(phs), h(arr), out)   # 2 chunks at this size (32 + 8 steps)
        b.rollout_sarl(acts, phs, arr)
        torch.cuda.synchronize()
        np.testing.assert_allclose(a.collect_stats().cpu().numpy(), b.shard_stats().cpu().numpy(), rtol=1e-12, atol=1e-9)
