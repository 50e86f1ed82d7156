"""The host-buffer rollouts (`risvec_rollout_*_host`): the chunked H2D -> rollout -> D2H pipeline over several chunks,
the statistics of its last chunk, and the argument checks that must refuse a bad buffer before anything is enqueued."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from ris_vec_marl_b200 import BatchedEnviron, _lib, encode_groups, marl_yaml_overrides

pytestmark = pytest.mark.gpu

V, M = 8, 40
GROUPS = [[0, 1], [2, 3], [4], [5, 6], [7]]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    assert torch.cuda.is_available(), "GPU tests selected but no CUDA device"
    _lib.load_library()  # fails loudly when the extension is missing


def chunk_steps(T, in_bytes_per_step):
    """The chunk length of the host pipeline (`chunk_steps` in risvec.cu)."""
    mb = max(1, int(os.environ.get("RISVEC_HOST_CHUNK_MB", "24")))
    tc = max(1, (mb << 20) // in_bytes_per_step)
    n = min(-(-T // tc), 64)
    steps = -(-T // n)
    return steps if steps <= 16 else -(-steps // 16) * 16


def assert_several_chunks(T, in_bytes_per_step):
    tc = chunk_steps(T, in_bytes_per_step)
    assert -(-T // tc) >= 3 and T % tc != 0, (T, tc)  # three chunks or more, the last one shorter


def same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


def make_envs(variant, E, n=2):
    over = marl_yaml_overrides() if variant == "marl" else {}
    envs = [BatchedEnviron(variant, E, V, M, seed=17, **over) for _ in range(n)]
    for e in envs:
        e.make_new_game(); e.renew_positions(); e.compute_parms()
        if variant == "marl":
            e.optimize_phase_shift(); e.update_channel_gains()
    return envs


def groups(E):
    part, ng = encode_groups(GROUPS, V)
    return torch.as_tensor(np.tile(part, (E, 1))), torch.full((E,), ng, dtype=torch.int32)


def inputs(T, E, seed):
    gen = torch.Generator().manual_seed(seed)
    acts = torch.rand(T, E, 2, V, generator=gen)
    ph = torch.rand(T, E, M, generator=gen) * 6.2831853
    arr = torch.poisson(torch.full((T, E, V), 2.0), generator=gen).to(torch.int32)
    return acts, ph, arr


@pytest.mark.parametrize("variant, T", [("sarl", 80), ("marl", 160)])
def test_packed_host_over_several_chunks_is_bit_identical_to_the_device_form(variant, T):
    E = 4096
    in_words = _lib.sarl_in_words(M) if variant == "sarl" else _lib.MARL_IN_WORDS
    assert_several_chunks(T, E * in_words * 4)  # SARL: 1 MiB per step, 32 + 32 + 16 steps at the default 24 MB
    dev_env, host_env = make_envs(variant, E)
    acts, ph, arr = inputs(T, E, seed=3)
    rec = dev_env.pack_inputs(acts, arr, ph if variant == "sarl" else None)
    extra = {}
    if variant == "marl":
        extra = dict(zip(("partner", "ngroups"), groups(E)))
    out_rec, rew = dev_env.rollout_packed(rec.cuda(), **{k: v.cuda() for k, v in extra.items()})
    h_out = torch.empty(out_rec.shape).pin_memory()
    h_rew = torch.empty(rew.shape).pin_memory()
    host_env.rollout_packed_host(rec.pin_memory(), h_out, h_rew, **{k: v.pin_memory() for k, v in extra.items()})
    torch.cuda.synchronize()
    assert same_bits(out_rec.cpu(), h_out)
    assert same_bits(rew.cpu(), h_rew)
    for f in _lib.FIELDS:
        assert same_bits(dev_env.state(f), host_env.state(f)), f


def test_marl_host_over_several_chunks_feeds_the_accumulator_its_last_step_only():
    E, T = 4096, 160
    assert_several_chunks(T, E * 3 * V * 4)  # the MARL chunk length counts action and arrivals
    dev_env, host_env = make_envs("marl", E)
    host_env.attach_stats_accumulator()
    acts, _, arr = inputs(T, E, seed=4)
    partner, ngroups = groups(E)
    names = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")
    ref = dev_env.rollout_marl(acts.cuda(), partner.cuda(), ngroups.cuda(), arr.cuda(), traces=names)
    out = {k: torch.empty(v.shape).pin_memory() for k, v in ref.items()}
    host_env.rollout_marl_host(acts.pin_memory(), partner.pin_memory(), ngroups.pin_memory(), arr.pin_memory(), out)
    got = host_env.collect_stats()
    want = dev_env.shard_stats()
    torch.cuda.synchronize()
    for k in ref:
        assert same_bits(ref[k].cpu(), out[k]), k
    w = want.cpu().numpy()
    assert np.abs(w).max() > 0
    np.testing.assert_allclose(got.cpu().numpy(), w, rtol=1e-12, atol=1e-9 * np.abs(w).max())


# ---- argument checks of the Python host wrappers: every bad buffer is at least as large as the good one, so a
# wrapper that let one through would still copy inside the caller's memory
E_SMALL, T_SMALL = 64, 4


def good_args(form, env):
    T, E = T_SMALL, E_SMALL
    acts, ph, arr = inputs(T, E, seed=5)
    partner, ngroups = groups(E)
    if form == "sarl":
        out = {k: torch.empty(env._trace_shape(k, T)) for k in ("reward", "DataBuf", "rate")}
        return dict(actions=acts, phases=ph, arrivals=arr, out=out)
    if form == "marl":
        out = {k: torch.empty(env._trace_shape(k, T)) for k in ("reward", "DataBuf", "stats", "last_power")}
        return dict(actions=acts, partner=partner, ngroups=ngroups, arrivals=arr, out=out)
    rec = env.pack_inputs(acts, arr, ph if env.variant == "sarl" else None)
    args = dict(in_rec=rec, out_rec=torch.empty(T, E // 4, 4 * env.packed_out_words()), reward=torch.empty(T, E))
    if env.variant == "marl":
        args.update(partner=partner, ngroups=ngroups)
    return args


def run(form, env, args):
    {"sarl": env.rollout_sarl_host, "marl": env.rollout_marl_host}.get(form, env.rollout_packed_host)(**args)


FAULTS = {
    "cuda": lambda t: t.cuda(),
    "shape": lambda t: torch.zeros(t.shape[:-1] + (t.shape[-1] + 1,), dtype=t.dtype),  # one more entry per row
    "dtype": lambda t: torch.zeros(t.shape, dtype=torch.float64 if t.is_floating_point() else torch.int64),
    "noncontiguous": lambda t: torch.zeros(t.shape[:-1] + (2 * t.shape[-1],), dtype=t.dtype)[..., ::2],
}


@pytest.mark.parametrize("form, variant", [("sarl", "sarl"), ("marl", "marl"), ("packed", "sarl"), ("packed", "marl")])
def test_host_wrappers_refuse_bad_buffers_before_anything_is_enqueued(form, variant):
    env = make_envs(variant, E_SMALL, n=1)[0]
    n0 = env.launch_count
    good = good_args(form, env)
    for fault, make in FAULTS.items():
        for name, t in good.items():
            targets = [(name, k) for k in t] if name == "out" else [(name, None)]
            for arg, key in targets:
                bad = dict(good)
                if key is None:
                    bad[arg] = make(t)
                else:
                    bad[arg] = {**t, key: make(t[key])}
                with pytest.raises(ValueError):
                    run(form, env, bad)
                assert env.launch_count == n0, (fault, arg, key)
    if form != "packed":
        with pytest.raises(ValueError, match="unknown trace"):
            run(form, env, {**good, "out": {**good["out"], "bogus": good["out"]["DataBuf"]}})
        assert env.launch_count == n0
    run(form, env, good)  # the same arguments unspoilt are accepted
    torch.cuda.synchronize()
    assert env.launch_count > n0


def test_per_array_host_exports_refuse_a_handle_of_the_other_variant():
    """At the C ABI, before any copy: the buffers are sized for the call, so even a late refusal stays inside them."""
    lib = _lib.load_library()
    sarl, marl = make_envs("sarl", E_SMALL, n=1)[0], make_envs("marl", E_SMALL, n=1)[0]
    acts, ph, _ = (x.pin_memory() for x in inputs(T_SMALL, E_SMALL, seed=6))
    partner, ngroups = (x.pin_memory() for x in groups(E_SMALL))
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    n_sarl, n_marl = sarl.launch_count, marl.launch_count
    rc = lib.risvec_rollout_marl_host(sarl._h, T_SMALL, p(acts), p(partner), p(ngroups), None, None, sarl.stream)
    assert rc == -1 and b"not a MARL env" in lib.risvec_last_error()
    rc = lib.risvec_rollout_sarl_host(marl._h, T_SMALL, p(acts), p(ph), None, None, marl.stream)
    assert rc == -1 and b"not a SARL env" in lib.risvec_last_error()
    torch.cuda.synchronize()
    assert (sarl.launch_count, marl.launch_count) == (n_sarl, n_marl)
