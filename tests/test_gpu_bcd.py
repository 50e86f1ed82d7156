"""The channel stage of an episode start -- the BCD phase search (`optimize_phase_shift`) and the free-space RIS gains
(`update_channel_gains`) -- against the float64 reference at every phase resolution, every kernel form and RIS sizes
up to the 1024-element cap.

Geometry comes from the kernels (`make_new_game` with injected draws, `renew_positions`, `compute_parms`); the same
positions go to `EnvOracle.set_vehicles` + `compute_parms`.  The reference search is `oracle.bcd_oracle.bcd_search`
(itself pinned to `EnvOracle.optimize_phase_shift` by tests/test_bcd_oracle.py), run from the theta the kernel
started from, read back from the device.

Kernel forms (`launch_bcd`, `launch_begin_episode`): `k_bcd_v8` for ncand <= 8, V <= 8, M <= 256 (4 warps per block
up to M = 64, 1 above), else `k_bcd` (lane k owns candidate k up to 32 candidates, lanes stride over them above; more
than 48 KB of dynamic shared memory above M = 384); RISVEC_FORCE_GENERIC=1 (read at handle creation) takes `k_bcd` and
`k_gains_free` everywhere.  E = 301 is neither a multiple of 4 nor of 16, so warps and blocks have tail lanes."""

import numpy as np
import pytest
import torch

from oracle.bcd_oracle import bcd_search, choice_index, coefficients, compare_choices
from oracle.env_oracle import EnvOracle

pytestmark = pytest.mark.gpu

E = 301
# An env with a decision whose reference margin (best - runner_up) / best is below MARGIN is not compared.  The
# kernel and the reference score the same |S|^2 from coefficients c_m that differ by rounding only: the reference's
# phasors exp(j x) take an argument x of size up to pi * M rounded to an ulp (|dc_m| up to ~1e-11 at M = 1024), the
# kernel's are sincospi (exact argument reduction) or float64 powers within a few ulps, and both update S
# incrementally.  Running bcd_search on both kinds of coefficients (exp of the rounded argument, and exp(j pi x) with
# x = m * delta reduced exactly mod 2) moves the margins by at most 2.6e-13 at M = 1024, V = 32 from off-grid starts
# and by < 1e-15 at M = 33; a margin above 1e-12 is therefore decided by the geometry, not by rounding.  (1e-10
# would exclude 1 to 3 of the 301 envs at 1024 candidates and at M = 1024, where margins of 1e-11 are common.)
MARGIN = 1e-12
MAX_EXCLUDED = 0.001  # at most 0.1 % of the envs may be excluded from the exact check
THETA_TOL = 1e-15  # |theta * conj(theta_ref) - 1|: sincospi(2k / n) against exp(j linspace(0, 2 pi, n)[k])
GAIN_RTOL = 1e-9
EPS = np.finfo(np.float64).eps


def gain_atol(amp, n):
    """Absolute floor of the gain check, `amp * |S_v|^2` with S_v = sum_{m < n} theta_m w_vm and |theta_m| <= 1.

    Each term carries a phase error of at most about (pi m + 64) ulp: the reference rounds its exp argument at a
    magnitude of up to pi m, and the kernel's phasor takes up to 31 complex products since its last exact anchor
    (k_gains_free_v) or one sincospi (k_gains_free).  So |dS| <= sum_m (pi m + 64) eps <= (pi n^2 / 2 + 64 n) eps,
    and the gain moves by at most amp (2 |S| dS + dS^2).  rtol 1e-9 covers that wherever |S| >= 2e9 dS (0.8 at
    n = 1024); below that |S| is far under sqrt(n), the size of a sum of n unit phasors of random phase, which the
    floor takes for |S|.  Where the phasors interfere destructively (|S| << sqrt(n)) the check rests on this floor,
    of order amp * n^2.5 * ulp."""
    dS = (np.pi * n * n / 2 + 64 * n) * EPS
    return amp * (2 * np.sqrt(n) * dS + dS * dS)


def reset_inputs(rng, E, V):
    pat = [(0, 4), (220, 230), (10, 15), (170, 180), (10, 15), (220, 230), (10, 15), (170, 180), (10, 15)] * (V // 4)
    pat += [(0, 4), (0, 400), (15, 20)] * (V % 4) + [(5, 9)]
    ints = np.stack([rng.integers(lo, hi, E) for lo, hi in pat], axis=1).astype(np.int32)
    dirs = rng.integers(0, 4, (E, V % 4)).astype(np.int32)
    return ints, dirs


def make(E, V, M, control_bit, generic, monkeypatch, seed=11):
    """A MARL handle with injected reset draws and one move, and the oracle on the same positions."""
    monkeypatch.setenv("RISVEC_FORCE_GENERIC", "1" if generic else "0")
    from ris_vec_marl_b200 import BatchedEnviron

    env = BatchedEnviron("marl", E, V, M, control_bit=control_bit, seed=seed)
    rng = np.random.default_rng(1000 * V + M + 17 * control_bit + seed)
    ints, dirs = reset_inputs(rng, E, V)
    env.make_new_game(ints, dirs if V % 4 else None)
    env.renew_positions(rng.random((E, 8 * V)))
    env.compute_parms()
    o = EnvOracle("marl", V, M, control_bit, E=E)
    return env, sync_oracle(env, o), rng


def sync_oracle(env, o):
    """Give the oracle the kernels' positions and check its geometry against theirs."""
    pos = np.stack([env.pos_x.cpu().numpy(), env.pos_y.cpu().numpy()], axis=-1)
    o.set_vehicles(pos, env.state("dir").cpu().numpy(), env.vel.cpu().numpy())
    o.compute_parms()
    np.testing.assert_allclose(env.angle.cpu().numpy(), o.angles_R_i, rtol=1e-14, atol=0)
    return o


def theta_of(env):
    return env.theta_re.cpu().numpy() + 1j * env.theta_im.cpu().numpy()


def set_start(env, kind, rng):
    """The theta a search starts from: the zero arena, off-grid phases (`get_next_phase`) or grid phases
    (`Random_phase`); returns it as the device holds it."""
    if kind == "offgrid":
        env.get_next_phase(rng.uniform(0, 2 * np.pi, (env.E, env.M)).astype(np.float32))
    elif kind == "grid":
        env.Random_phase(rng.integers(0, 2 ** env.control_bit, (env.E, env.M)).astype(np.int32))
    else:
        assert kind in ("zero", "carried")
    th = theta_of(env)
    if kind == "zero":
        assert not th.any()
    return th


def check_theta(got, theta0, o, control_bit, n=None, free0=False, label=""):
    """The kernel's theta against the reference search from theta0 (see `compare_choices`); elements m >= n keep
    theta0 bit for bit.  Returns the number of excluded envs."""
    En, M = got.shape
    n = np.full(En, M) if n is None else np.asarray(n)
    _, want, margin = bcd_search(coefficients(o), theta0, control_bit, n)
    searched = want != -2
    assert np.array_equal(got[~searched], theta0[~searched]), f"{label}: theta of an element m >= n changed"
    got_idx = np.where(searched, choice_index(np.where(searched, got, 0), control_bit, THETA_TOL), -2)
    free0 = np.asarray(free0) | (n == 1)
    excluded, wrong = compare_choices(got_idx, want, margin, control_bit, free0, MARGIN)
    nx = int(excluded.sum())
    print(f"\n{label}: {nx} of {En} envs excluded (reference margin < {MARGIN:g})", end="")
    assert not wrong.any(), (f"{label}: {wrong.sum()} envs chose differently from the reference, first env "
                             f"{np.flatnonzero(wrong)[0]}")
    assert nx <= MAX_EXCLUDED * En, f"{label}: {nx} of {En} envs excluded"
    return nx


def check_gains(env, o, n=None, label=""):
    """The kernel's gains against `EnvOracle.update_channel_gains` evaluated on the kernel's own theta (restricted
    to the env's first n elements)."""
    th = theta_of(env)
    En, M = th.shape
    n = np.full(En, M) if n is None else np.asarray(n)
    o.elements_phase_shift_complex = np.where(np.arange(M)[None, :] < n[:, None], th, 0)
    o.update_channel_gains()
    got, want = env.gains.cpu().numpy(), o.channel_gains
    amp = env.amp.cpu().numpy()
    tol = gain_atol(amp, n[:, None]) + GAIN_RTOL * np.abs(want)
    bad = np.abs(got - want) > tol
    assert not bad.any(), (f"{label}: {bad.sum()} gains out of tolerance; worst relative "
                           f"{np.max(np.abs(got - want) / np.maximum(want, 1e-300)):.3g}")


def run_case(V, M, control_bit, generic, monkeypatch, En=E, starts=("zero", "carried", "offgrid", "grid")):
    env, o, rng = make(En, V, M, control_bit, generic, monkeypatch)
    for kind in starts:
        label = f"V={V} M={M} cb={control_bit} generic={generic} E={En} {kind}"
        theta0 = set_start(env, kind, rng)
        env.optimize_phase_shift()
        check_theta(theta_of(env), theta0, o, control_bit, free0=kind == "zero", label=label)
        env.update_channel_gains()
        check_gains(env, o, label=label)
    env.close()


# (V, M, control_bit, generic)
V8_FOUR_WARPS = [(8, 40, 0, False), (8, 40, 1, False), (8, 40, 2, False), (8, 40, 3, False), (5, 7, 1, False),
                 (1, 1, 3, False), (3, 64, 2, False)]
V8_ONE_WARP = [(8, 65, 3, False), (8, 120, 0, False), (8, 120, 3, False), (6, 256, 2, False)]
GENERIC_LANE = [(8, 40, 4, False), (8, 40, 5, False), (12, 40, 3, False), (32, 100, 5, False), (8, 40, 0, True),
                (8, 40, 3, True)]
GENERIC_STRIDED = [(8, 40, 6, False), (4, 33, 10, False), (32, 64, 7, False)]
GENERIC_LARGE_M = [(8, 257, 3, False), (9, 385, 3, False), (32, 1024, 3, False), (8, 1024, 4, False)]


@pytest.mark.parametrize("V,M,control_bit,generic",
                         V8_FOUR_WARPS + V8_ONE_WARP + GENERIC_LANE + GENERIC_STRIDED + GENERIC_LARGE_M)
def test_bcd_and_gains_vs_reference(V, M, control_bit, generic, monkeypatch):
    run_case(V, M, control_bit, generic, monkeypatch)


def test_bcd_single_env(monkeypatch):
    """E = 1: one env in a warp of four; the other three lane groups are idle."""
    run_case(8, 40, 3, False, monkeypatch, En=1)


SIZES = (20, 40, 60, 80, 100, 120)


@pytest.mark.parametrize("M", SIZES)
def test_ris_size_sweep_one_handle_per_size(M, monkeypatch):
    run_case(8, M, 3, False, monkeypatch, starts=("zero", "grid"))


@pytest.mark.parametrize("generic", [False, True])
def test_ris_size_sweep_per_env_counts(generic, monkeypatch):
    """One M = 120 handle with per-env sizes cycling over 20 ... 120: each env against the reference restricted to
    its first n[e] elements; the elements m >= n[e] keep their theta."""
    M = 120
    env, o, rng = make(E, 8, M, 3, generic, monkeypatch)
    n = np.array([SIZES[e % len(SIZES)] for e in range(E)])
    env.attach_ris_elements(counts=torch.as_tensor(n, dtype=torch.int32, device=env.device))
    for kind in ("zero", "carried", "offgrid", "grid"):
        label = f"per-env sizes generic={generic} {kind}"
        theta0 = set_start(env, kind, rng)
        env.optimize_phase_shift()
        check_theta(theta_of(env), theta0, o, 3, n=n, free0=kind == "zero", label=label)
        env.update_channel_gains()
        check_gains(env, o, n=n, label=label)
    env.close()


@pytest.mark.parametrize("V,M,control_bit", [(8, 40, 0), (8, 40, 3), (8, 120, 3), (8, 256, 2), (5, 80, 1)])
def test_fused_episode_start_vs_reference(V, M, control_bit, monkeypatch):
    """`begin_episode(stages=("channel",))` takes the fused k_begin_episode (V <= 8, ncand <= 8, M <= 256): the
    search and the gains from theta held in shared memory."""
    env, o, rng = make(E, V, M, control_bit, False, monkeypatch)
    for kind in ("zero", "carried", "offgrid", "grid"):
        label = f"begin_episode V={V} M={M} cb={control_bit} {kind}"
        theta0 = set_start(env, kind, rng)
        env.begin_episode(stages=("channel",))
        check_theta(theta_of(env), theta0, o, control_bit, free0=kind == "zero", label=label)
        check_gains(env, o, label=label)
    env.close()


@pytest.mark.parametrize("fused", [False, True])
def test_full_size_chained_episodes(fused, monkeypatch):
    """E = 4096, V = 8, M = 40, control_bit 3, as the driver runs it: a search from the zero arena, then three
    episodes of new positions, search and gains with theta carried over; compared after every call."""
    En, V, M, cb = 4096, 8, 40, 3
    env, o, rng = make(En, V, M, cb, False, monkeypatch)
    theta0 = set_start(env, "zero", rng)
    env.optimize_phase_shift()
    check_theta(theta_of(env), theta0, o, cb, free0=True, label="E=4096 zero start")
    env.update_channel_gains()
    check_gains(env, o, label="E=4096 zero start")
    for ep in range(3):
        label = f"E=4096 fused={fused} episode {ep}"
        theta0 = theta_of(env)
        mob = rng.random((En, 8 * V))
        if fused:
            env.begin_episode(stages=("positions", "channel"), uniforms=mob)
        else:
            env.renew_positions(mob)
            env.compute_parms()
        o = sync_oracle(env, o)
        if not fused:
            env.optimize_phase_shift()
        check_theta(theta_of(env), theta0, o, cb, label=label)
        if not fused:
            env.update_channel_gains()
        check_gains(env, o, label=label)
    env.close()


@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("V", [1, 8, 32])
@pytest.mark.parametrize("M", [40, 256, 1024])
def test_gains_on_non_coherent_theta(M, V, generic, monkeypatch):
    """k_gains_free_v (phasor recurrence re-anchored every 32 elements) and k_gains_free (one sincospi per term) on
    theta = 1 and on off-grid random theta, where the sum interferes destructively and its absolute error counts."""
    env, o, rng = make(E, V, M, 3, generic, monkeypatch)
    for kind in ("ones", "offgrid"):
        ph = np.zeros((E, M)) if kind == "ones" else rng.uniform(0, 2 * np.pi, (E, M))
        env.get_next_phase(ph.astype(np.float32))
        env.update_channel_gains()
        check_gains(env, o, label=f"gains V={V} M={M} generic={generic} {kind}")
    env.close()


@pytest.mark.parametrize("generic", [False, True])
def test_exact_ties_go_to_the_smallest_index(generic, monkeypatch):
    """V = 2 with angle_BR - angle = +0.5 and -0.5 exactly: c_m = i^m + (-i)^m is 0 exactly for odd m in both
    kernels (sincospi of a half-integer, powers of +-i), so every candidate scores |S - theta_m c_m|^2 there and the
    reference rule (first maximum, strict `best < x`) picks candidate 0: theta_m = 1."""
    V, M, cb = 2, 40, 3
    env, o, rng = make(E, V, M, cb, generic, monkeypatch)
    a_br = o.angle_B_R
    angle = np.empty((E, V))
    angle[:, 0], angle[:, 1] = a_br - 0.5, a_br + 0.5
    assert (a_br - angle[:, 0] == 0.5).all() and (a_br - angle[:, 1] == -0.5).all()
    env.angle.copy_(torch.as_tensor(angle, device=env.device))
    m = np.arange(M)
    c = np.tile(np.where(m % 2 == 1, 0.0, np.where(m % 4 == 0, 2.0, -2.0)), (E, 1)).astype(complex)
    theta0 = set_start(env, "offgrid", rng)
    env.optimize_phase_shift()
    got = theta_of(env)
    _, want, margin = bcd_search(c, theta0, cb)
    odd = (m % 2 == 1)[None, :].repeat(E, axis=0)
    assert (want[odd] == 0).all() and (margin[odd] == 0).all()
    assert (got.real[odd] == 1.0).all() and (got.imag[odd] == 0.0).all(), "an exact tie did not go to candidate 0"
    got_idx = choice_index(got, cb, THETA_TOL)
    excluded, wrong = compare_choices(got_idx, want, np.where(odd, 1.0, margin), cb, False, MARGIN)
    assert not wrong.any() and excluded.sum() <= MAX_EXCLUDED * E
    env.close()
