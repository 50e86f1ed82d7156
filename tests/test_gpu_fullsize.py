"""BASELINE.json sizes (4096 envs per GPU): the CUDA path against the batched float64 oracle
on identical seeded inputs, plus size-independent invariants of the queue dynamics."""
import numpy as np
import pytest
import torch

from oracle.env_oracle import EnvOracle, InjectedDraws, OracleParams, encode_groups
from tests.parity import RTOL, sarl_rate_atol, sarl_reward_band

pytestmark = pytest.mark.gpu


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


def _sarl_env(path, E, V, M):
    """SARL env whose rollouts go through one named kernel path (ris_vec_marl_b200/csrc/risvec.cu
    `launch_sarl`): RISVEC_SARL_PATH is read once, when the handle is created."""
    from ris_vec_marl_b200 import BatchedEnviron
    from tests.gpu_backend import kernel_paths

    with kernel_paths(sarl={"packed": "v8"}.get(path, path)):
        return BatchedEnviron("sarl", E, V, M)


# every SARL step kernel at BASELINE size: (path, V, M, E, kernel it must run)
SARL_PATHS = [("mma", 8, 40, 4096, "k_sarl_mma_tma"), ("mma-ldg", 8, 40, 4096, "k_sarl_mma"),
              ("mma", 8, 16, 4096, "k_sarl_mma_tma"), ("mma", 8, 24, 4096, "k_sarl_mma"), ("v8", 8, 40, 4096, "k_sarl_v8"),
              ("packed", 8, 40, 4096, "k_sarl_v8"), ("generic", 8, 40, 4096, "k_sarl_rollout"),
              ("generic", 8, 64, 4096, "k_sarl_cascade2+k_sarl_scan"),
              ("mma", 32, 256, 1024, "k_sarl_umma"),                         # BASELINE config 4 (tcgen05)
              ("mma-sync", 32, 256, 1024, "k_sarl_mma_big"), ("mma", 16, 128, 1024, "k_sarl_umma"),
              ("generic", 32, 256, 1024, "k_sarl_cascade2+k_sarl_scan")]


@pytest.mark.parametrize("path,V,M,E,kernel", SARL_PATHS, ids=[f"{p}-V{v}-M{m}" for p, v, m, _, _ in SARL_PATHS])
def test_sarl_4096_envs_rollout_matches_oracle(path, V, M, E, kernel):
    T = 32 if V == 8 else 24
    rng = np.random.default_rng(2024)
    ri = reset_draws(rng, E, V)
    mob = rng.random((E, 8 * V))
    acts = rng.random((T, E, 2, V)).astype(np.float32)
    phs = (rng.random((T, E, M)) * 2 * np.pi).astype(np.float32)
    arr = rng.poisson(3.0, (T, E, V)).astype(np.int32)

    env = _sarl_env(path, E, V, M)
    env.make_new_game(ri)
    used = env.renew_positions(mob)
    env.compute_parms()
    if path == "packed":
        out_rec, reward = env.rollout_packed(env.pack_inputs(torch.as_tensor(acts), torch.as_tensor(arr), torch.as_tensor(phs)))
        got = {k: v.cpu().numpy() for k, v in env.unpack_outputs(out_rec, reward).items()}
    else:
        got = {k: v.cpu().numpy() for k, v in env.rollout_sarl(acts, phs, arr).items()}
    assert env.last_kernel() == kernel, (env.last_kernel(), kernel)

    d = InjectedDraws(reset_ints=ri, arrivals=arr)
    o = EnvOracle("sarl", V, M, 3, E=E, draws=d)
    o.make_new_game()
    d.set_mobility_uniforms(mob)
    o.renew_positions(); o.compute_parms()
    assert np.array_equal(used.cpu().numpy(), d.mob_draws_used)
    assert np.array_equal(env.pos_x.cpu().numpy(), o.pos[..., 0]) and np.array_equal(env.pos_y.cpu().numpy(), o.pos[..., 1])
    ra = sarl_rate_atol(M)
    n_band = 0
    worst = 0.0
    for t in range(T):
        rew, over_p = o.step_sarl(acts[t], phs[t])
        band = sarl_reward_band(o.last["buf_signed"], o.over_data, M).any(axis=1)  # reward penalties jump here
        n_band += int(band.sum())
        worst = max(worst, float((np.abs(got["rate"][t] - o.vehicle_rate) / (ra + RTOL * np.abs(o.vehicle_rate))).max()))
        close(got["data_p"][t], o.data_p, 1e-5, f"data_p t={t}")
        close(got["DataBuf"][t], o.DataBuf, 4 * ra, f"DataBuf t={t}")
        close(got["over_data"][t], o.over_data, 4 * ra, f"over_data t={t}")
        # over_power = P1 - localProcRev(DataBuf + data_p): |d over_power / d DataBuf| <= 3 c_rev^3 x^2 <= 0.7 (x <= 4.31 kbit),
        # so the rate's absolute floor (sqrt(M) growth, tests/parity.py) reaches it scaled by 0.7
        close(got["over_power"][t], over_p, 4e-6 + 0.7 * ra, f"over_power t={t}")
        close(got["reward"][t], rew, 4e-6, f"reward t={t}", mask=band)
    assert worst <= 1.0, f"rate: worst error {worst:.2f} of its tolerance ({ra:.2e} + {RTOL:g} |rate|)"
    # the reward is the RL signal: it must be compared on (nearly) every env-step
    assert n_band <= 0.05 * E * T, f"{n_band} of {E * T} env-steps band-excluded from the reward check"
    print(f"[{kernel}] reward compared on {E * T - n_band} of {E * T} env-steps ({n_band} on a penalty threshold); "
          f"worst rate error = {worst:.2f} of its tolerance")
    # the state after the rollout is the last step's
    np.testing.assert_allclose(env.DataBuf.cpu().numpy(), o.DataBuf, rtol=RTOL, atol=4 * ra)
    close(env.reward.cpu().numpy(), rew, 4e-6, "state reward", mask=band)
    # invariants at full size
    assert (got["DataBuf"] >= 0).all() and (got["over_data"] >= 0).all() and (got["rate"] >= 0).all()
    assert np.all((got["over_data"] > 0) <= (got["DataBuf"] - arr <= 1e-6))  # overflow only when the buffer drained


@pytest.mark.parametrize("path,kernel,T", [("tma", "k_marl_tma", 40), ("tma", "k_marl_tma", 32), ("v8", "k_marl_v8", 12)])
def test_marl_4096_envs_rollout_matches_oracle(path, kernel, T):
    from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides
    from tests.gpu_backend import kernel_paths

    E, V, M = 4096, 8, 40
    rng = np.random.default_rng(77)
    ri = reset_draws(rng, E, V)
    mob = rng.random((E, 8 * V))
    acts = rng.random((T, E, 2, V)).astype(np.float32)
    acts[:, :, 1, :] = np.maximum(acts[:, :, 1, :], np.float32(0.1))
    arr = rng.poisson(1.0, (T, E, V)).astype(np.int32)
    part, ng = encode_groups([[0, 1], [3, 2], [4, 5], [6], [7]], V)
    partner, ngroups = np.tile(part, (E, 1)), np.full(E, ng, dtype=np.int32)

    with kernel_paths(marl=path):
        env = BatchedEnviron("marl", E, V, M, **marl_yaml_overrides())
    env.make_new_game(ri); env.renew_positions(mob); env.compute_parms()
    phase0 = np.zeros((E, M), dtype=np.float32)
    env.get_next_phase(phase0)  # theta = 1: includes destructive-interference gains
    env.update_channel_gains()
    got = {k: v.cpu().numpy() for k, v in env.rollout_marl(
        acts, partner, ngroups, arr, traces=("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")).items()}
    assert env.last_kernel() == kernel, (env.last_kernel(), kernel)

    d = InjectedDraws(reset_ints=ri, arrivals=arr)
    o = EnvOracle("marl", V, M, 3, E=E, params=OracleParams.marl_yaml(), draws=d)
    o.make_new_game()
    d.set_mobility_uniforms(mob)
    o.renew_positions(); o.compute_parms(); o.get_next_phase(phase0.astype(np.float64)); o.update_channel_gains()
    np.testing.assert_allclose(env.gains.cpu().numpy(), o.channel_gains, rtol=1e-7, atol=1e-26)
    p = o.p
    for t in range(T):
        r_user, r_glob, over_p = o.step_marl(acts[t], partner, ngroups)
        L = o.last
        band = (np.abs(o.vehicle_rate - p.R_min_bpsHz) < 1e-5 * p.R_min_bpsHz) | (np.abs(L["delay"] - p.D_max_s) < 1e-5 * p.D_max_s)
        amp = (L["edge_in_sum"] < 1e-3) & (L["q_before"] > 0) & (L["edge_in_sum"] > 0)
        band |= amp[:, None]
        close(got["rate"][t], o.vehicle_rate, 1e-6, f"rate t={t}")
        close(got["data_t"][t], o.data_t, 1e-5, f"data_t t={t}")
        close(got["data_p"][t], o.data_p, 1e-5, f"data_p t={t}")
        close(got["DataBuf"][t], o.DataBuf, 1e-5, f"DataBuf t={t}")
        close(got["reward_user"][t], r_user, 2e-6, f"reward_user t={t}", mask=band)
        close(got["reward"][t], r_glob, 2e-6, f"reward t={t}", mask=band.any(axis=1))
    np.testing.assert_allclose(env.mec_queue_cycles.cpu().numpy(), o.mec_queue_cycles, rtol=1e-6, atol=1.0)
    # the state after the rollout is the last step's (`last_*` statistics included)
    np.testing.assert_allclose(env.DataBuf.cpu().numpy(), o.DataBuf, rtol=RTOL, atol=1e-5)
    st = env.stats.cpu().numpy()
    amp_env = amp | band.any(axis=1)
    close(st[:, 0], L["delay_mean"], 1e-9, "last_delay_mean", mask=amp_env)
    close(st[:, 1], L["energy_mean"], 1e-9, "last_energy_mean")
    close(st[:, 6], L["backlog_kbit_mean"], 1e-5, "last_backlog_kbit_mean")
    close(st[:, 10], L["off_kbit_sum"], 1e-5, "last_off_kbit_sum")
    close(st[:, 11], L["local_kbit_sum"], 1e-5, "last_local_kbit_sum")
    close(env.reward.cpu().numpy(), r_glob, 2e-6, "state reward", mask=band.any(axis=1))
    assert (got["DataBuf"] >= 0).all() and (got["rate"] >= 0).all() and (np.abs(got["reward_user"]) <= 50).all()
