"""SURVEY 8a rows a5 (`Random_phase`) and a9 (`get_path_loss`, `get_shadowing`): functions the
reference defines but its drivers never call.  CPU: oracle vs the live reference; GPU: kernels vs oracle."""
import numpy as np
import pytest

from oracle import ref_harness as rh
from oracle.env_oracle import EnvOracle

POS = [[197.375, 225], [200.875, 173], [223, 200.875], [173, 197.375], [199.125, 300], [202.625, 50],
       [350, 202.625], [20, 199.125]]          # KAT-1 positions (SURVEY 8c)


def _oracle(E=1, V=8, M=40):
    o = EnvOracle("marl", V, M, 3, E=E)
    o.set_vehicles(np.asarray(POS, float)[None, :V], np.zeros((E, V), int), np.arange(10, 10 + V)[None])
    return o


@pytest.mark.skipif(not rh.reference_available(), reason="reference tree not mounted")
@pytest.mark.parametrize("variant", ["marl", "sarl"])
def test_oracle_vs_reference_dead_rows(variant):
    import random

    log = rh.DrawLog()
    mod, env = rh.make_reference_env(variant, 8, 40, 3, log, "record", np.random.RandomState(5))
    for i, p in enumerate(POS):
        env.add_new_vehicles(list(p), "u", 10 + i)
    env.V2I_Shadowing = np.random.RandomState(1).normal(0, 8, 8)
    o = _oracle()
    # a9: path loss and shadowing
    want_pl = np.array([env.get_path_loss(v.position) for v in env.vehicles])
    assert np.array_equal(o.path_loss()[0], want_pl)
    got_sh = []
    for i, v in enumerate(env.vehicles):
        got_sh.append(env.get_shadowing(v.velocity * env.time_slow, i)[0])
    twin = np.random.RandomState(5)     # same stream as the env's: nothing else has drawn from it
    normals = np.array([twin.normal(0, 8, 1)[0] for _ in range(8)]).reshape(1, 8)
    assert np.array_equal(o.shadowing(env.V2I_Shadowing[None], normals)[0], np.array(got_sh))
    # a5: Random_phase
    random.seed(11)
    env.Random_phase()
    picks = np.array(log.q["choice"][-40:])
    idx = np.array([int(np.argmin(np.abs(env.possible_angles - a))) for a in picks])
    o.random_phase(idx[None])
    assert np.array_equal(o.elements_phase_shift_real[0], np.asarray(env.elements_phase_shift_real))
    assert np.array_equal(o.elements_phase_shift_complex[0], env.elements_phase_shift_complex)


@pytest.mark.gpu
def test_gpu_dead_rows_vs_oracle():
    import torch

    from ris_vec_marl_b200 import BatchedEnviron

    E, V, M = 64, 8, 40
    rng = np.random.default_rng(2)
    env = BatchedEnviron("marl", n_envs=E, n_veh=V, M=M, device=0, seed=3)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    o = EnvOracle("marl", V, M, 3, E=E)
    pos = np.stack([env.pos_x.cpu().numpy(), env.pos_y.cpu().numpy()], axis=-1)
    o.set_vehicles(pos, env.state("dir").cpu().numpy(), env.vel.cpu().numpy())
    o.compute_parms()
    np.testing.assert_allclose(env.get_path_loss().cpu().numpy(), o.path_loss(), rtol=1e-14, atol=0)
    shadow = rng.normal(0, 8, (E, V)); normals = rng.normal(0, 8, (E, V))
    env.V2I_Shadowing.copy_(torch.as_tensor(shadow, device=env.device))
    np.testing.assert_allclose(env.get_shadowing(normals).cpu().numpy(), o.shadowing(shadow, normals), rtol=1e-14, atol=1e-15)
    sh = env.get_shadowing().cpu().numpy()          # on-device N(0, 8): moments only
    resid = (sh - np.exp(-o.vel * 0.1 / 10) * shadow) / np.sqrt(1 - np.exp(-2 * o.vel * 0.1 / 10))
    assert abs(resid.mean()) < 1.5 and 6.0 < resid.std() < 10.0
    idx = rng.integers(0, 8, (E, M)).astype(np.int32)
    env.Random_phase(idx)
    o.random_phase(idx)
    th = env.theta_re.cpu().numpy() + 1j * env.theta_im.cpu().numpy()
    np.testing.assert_allclose(th, o.elements_phase_shift_complex, rtol=0, atol=2e-16)
    np.testing.assert_allclose(env.phase_real.cpu().numpy(), o.elements_phase_shift_real, rtol=1e-7)
    env.update_channel_gains(); o.update_channel_gains()
    np.testing.assert_allclose(env.gains.cpu().numpy(), o.channel_gains, rtol=1e-9)
    env.Random_phase()                               # on-device draws: every angle a multiple of pi/4
    k = env.phase_real.cpu().numpy().astype(np.float64) / (np.pi / 4)
    assert np.allclose(k, np.round(k), atol=1e-6) and k.min() >= 0 and k.max() <= 7 and len(np.unique(np.round(k))) == 8
    env.close()


@pytest.mark.gpu
@pytest.mark.parametrize("control_bit", [0, 1, 4, 10])
def test_gpu_random_phase_every_resolution(control_bit):
    """`Random_phase` at the other phase resolutions (1 ... 1024 candidates; control_bit 3 is the test above):
    injected choices give the oracle's theta, and the gains on it; on-device draws land on the grid of 2 pi / ncand
    and, with ncand <= 8, take every value."""
    from ris_vec_marl_b200 import BatchedEnviron

    E, V, M = 64, 8, 40
    ncand = 2 ** control_bit
    rng = np.random.default_rng(2)
    env = BatchedEnviron("marl", n_envs=E, n_veh=V, M=M, control_bit=control_bit, device=0, seed=3)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    o = EnvOracle("marl", V, M, control_bit, E=E)
    pos = np.stack([env.pos_x.cpu().numpy(), env.pos_y.cpu().numpy()], axis=-1)
    o.set_vehicles(pos, env.state("dir").cpu().numpy(), env.vel.cpu().numpy())
    o.compute_parms()
    idx = rng.integers(0, ncand, (E, M)).astype(np.int32)
    idx[0, :min(M, ncand)] = np.arange(min(M, ncand))  # the first candidates, 0 included, at least once
    idx[1, :] = ncand - 1                              # and the last one
    env.Random_phase(idx)
    o.random_phase(idx)
    th = env.theta_re.cpu().numpy() + 1j * env.theta_im.cpu().numpy()
    # the same angle k * (2 pi / ncand) on both sides; CUDA sincos and numpy exp are each within an ulp of its phasor
    np.testing.assert_allclose(th, o.elements_phase_shift_complex, rtol=0, atol=2.5e-16)
    np.testing.assert_allclose(env.phase_real.cpu().numpy(), o.elements_phase_shift_real, rtol=1e-7)
    env.update_channel_gains(); o.update_channel_gains()
    np.testing.assert_allclose(env.gains.cpu().numpy(), o.channel_gains, rtol=1e-9)
    env.Random_phase()                               # on-device draws: every angle a multiple of 2 pi / ncand
    th = env.theta_re.cpu().numpy() + 1j * env.theta_im.cpu().numpy()
    k = np.mod(np.angle(th), 2 * np.pi) / (2 * np.pi / ncand)
    k = np.where(np.abs(k - ncand) < 1e-9, 0.0, k)   # angle 0 may read as 2 pi - ulp
    kr = np.round(k).astype(int)
    assert np.allclose(k, kr, rtol=0, atol=1e-9) and kr.min() >= 0 and kr.max() <= ncand - 1
    np.testing.assert_allclose(th, np.exp(1j * o.possible_angles[kr]), rtol=0, atol=2.5e-16)
    np.testing.assert_allclose(env.phase_real.cpu().numpy(), o.possible_angles[kr], rtol=1e-7)
    if ncand <= 8:
        assert len(np.unique(kr)) == ncand
    env.close()


@pytest.mark.gpu
def test_gpu_compat_random_phase_follows_python_random():
    import random

    from ris_vec_marl_b200.compat_env import MarlEnviron
    from oracle.ref_harness import DOWN_LANES, HEIGHT, LEFT_LANES, RIGHT_LANES, UP_LANES, WIDTH

    env = MarlEnviron(DOWN_LANES, UP_LANES, LEFT_LANES, RIGHT_LANES, WIDTH, HEIGHT, 8, 40, 3)
    np.random.seed(0); random.seed(0)
    env.make_new_game()
    random.seed(11)
    env.Random_phase()
    random.seed(11)
    want = np.array([random.choice(np.linspace(0, 2 * np.pi, 8, endpoint=False)) for _ in range(40)])
    np.testing.assert_allclose(np.asarray(env.elements_phase_shift_real, float), want, rtol=1e-7)
    assert np.asarray(env.V2I_Shadowing).shape == (8,)
    pl = env.get_path_loss(env.vehicles[2].position)
    assert 80 < float(pl) < 140
