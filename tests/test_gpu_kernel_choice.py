"""Which rollout kernel each call launches: shape, given traces and arrivals, pointer alignment, packed records and
the A/B overrides (RISVEC_SARL_PATH, RISVEC_MARL_PATH, RISVEC_FORCE_GENERIC, read at handle creation) against
`last_kernel()` and the number of launches the call adds (k_shard_stats for an attached accumulator included)."""
import numpy as np
import pytest
import torch

from ris_vec_marl_b200 import BatchedEnviron, encode_groups

pytestmark = pytest.mark.gpu

T = 4
SARL_ALL = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
MARL_FAST = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")
CASCADE = "k_sarl_cascade2+k_sarl_scan"


def case(variant, kernel, launches, V=8, M=40, E=8, over=None, traces=None, arrivals=True, misaligned=None,
         entry="rollout", stats=False):
    """misaligned: the name of a trace, or "raw" for a fused step, placed 4 bytes off a 16-byte boundary"""
    if traces is None:
        traces = SARL_ALL if variant == "sarl" else MARL_FAST
    return dict(variant=variant, kernel=kernel, launches=launches, V=V, M=M, E=E, over=over or {}, traces=traces,
                arrivals=arrivals, misaligned=misaligned, entry=entry, stats=stats)


SARL = "RISVEC_SARL_PATH"
CASES = {
    # SARL rollouts
    "sarl-tma-m16": case("sarl", "k_sarl_mma_tma", 1, M=16),
    "sarl-tma-m40": case("sarl", "k_sarl_mma_tma", 1),
    "sarl-tma-spelled-mma": case("sarl", "k_sarl_mma_tma", 1, over={SARL: "mma"}),
    "sarl-tma-unknown-spelling": case("sarl", "k_sarl_mma_tma", 1, over={SARL: "bogus"}),
    "sarl-tma-stats": case("sarl", "k_sarl_mma_tma", 1, stats=True),
    "sarl-mma-m24": case("sarl", "k_sarl_mma", 1, M=24),
    "sarl-mma-no-arrivals": case("sarl", "k_sarl_mma", 1, arrivals=False),
    "sarl-mma-e6": case("sarl", "k_sarl_mma", 1, E=6),
    "sarl-mma-misaligned": case("sarl", "k_sarl_mma", 1, misaligned="data_t"),
    "sarl-mma-ldg": case("sarl", "k_sarl_mma", 1, over={SARL: "mma-ldg"}),
    "sarl-mma-stats": case("sarl", "k_sarl_mma", 2, M=24, stats=True),
    "sarl-v8-odd-m": case("sarl", "k_sarl_v8", 1, M=15),
    "sarl-umma": case("sarl", "k_sarl_umma", 1, V=12, M=128, E=4),
    "sarl-umma-m40": case("sarl", "k_sarl_umma", 1, V=12, M=40, E=4),
    "sarl-mma-sync": case("sarl", "k_sarl_mma_big", 1, V=12, M=128, E=4, over={SARL: "mma-sync"}),
    "sarl-mma-sync-small": case("sarl", "k_sarl_mma_tma", 1, over={SARL: "mma-sync"}),
    "sarl-mma-ldg-big": case("sarl", CASCADE, 2, V=12, M=128, E=4, over={SARL: "mma-ldg"}),
    "sarl-cascade-v6": case("sarl", CASCADE, 2, V=6, M=100, E=4),
    "sarl-cascade-v2": case("sarl", CASCADE, 2, V=2, M=100, E=4),
    "sarl-rollout-missing-trace": case("sarl", "k_sarl_rollout", 1, V=12, E=4, traces=SARL_ALL[:-1]),
    "sarl-rollout-stats": case("sarl", "k_sarl_rollout", 2, V=12, E=4, traces=SARL_ALL[:-1], stats=True),
    "sarl-v8": case("sarl", "k_sarl_v8", 1, over={SARL: "v8"}),
    "sarl-v8-m16": case("sarl", "k_sarl_v8", 1, M=16, over={SARL: "v8"}),
    "sarl-v8-m64": case("sarl", CASCADE, 2, M=64, over={SARL: "v8"}),
    "sarl-generic": case("sarl", "k_sarl_rollout", 1, over={SARL: "generic"}),
    "sarl-generic-m64": case("sarl", CASCADE, 2, M=64, over={SARL: "generic"}),
    "sarl-force-generic": case("sarl", "k_sarl_rollout", 1, over={"RISVEC_FORCE_GENERIC": "1"}),
    "sarl-force-generic-m64": case("sarl", CASCADE, 2, M=64, over={"RISVEC_FORCE_GENERIC": "1"}),
    "sarl-packed-m16": case("sarl", "k_sarl_v8", 1, M=16, entry="packed"),
    "sarl-packed-m40": case("sarl", "k_sarl_v8", 1, entry="packed"),
    # SARL driver steps and host-buffer calls
    "sarl-fused": case("sarl", "k_sarl_mma", 1, entry="fused"),
    "sarl-fused-stats": case("sarl", "k_sarl_mma", 2, entry="fused", stats=True),
    "sarl-fused-odd-m": case("sarl", "k_sarl_v8", 3, M=15, entry="fused"),
    "sarl-fused-misaligned-raw": case("sarl", "k_sarl_mma", 3, entry="fused", misaligned="raw"),
    "sarl-fused-v8": case("sarl", "k_sarl_v8", 3, entry="fused", over={SARL: "v8"}),
    "sarl-fused-mma-ldg": case("sarl", "k_sarl_mma", 1, entry="fused", over={SARL: "mma-ldg"}),
    "sarl-fused-force-generic": case("sarl", "k_sarl_rollout", 3, entry="fused", over={"RISVEC_FORCE_GENERIC": "1"}),
    "sarl-host": case("sarl", "k_sarl_mma_tma", 1, entry="host"),
    "sarl-packed-host": case("sarl", "k_sarl_v8", 1, entry="packed_host"),
    # MARL rollouts
    "marl-tma": case("marl", "k_marl_tma", 1),
    "marl-tma-stats": case("marl", "k_marl_tma", 1, stats=True),
    "marl-v8-override": case("marl", "k_marl_v8", 1, over={"RISVEC_MARL_PATH": "v8"}),
    "marl-v8-stats": case("marl", "k_marl_v8", 2, over={"RISVEC_MARL_PATH": "v8"}, stats=True),
    "marl-v8-no-arrivals": case("marl", "k_marl_v8", 1, arrivals=False),
    "marl-v8-over-power": case("marl", "k_marl_v8", 1, traces=MARL_FAST + ("over_power",)),
    "marl-v8-misaligned": case("marl", "k_marl_v8", 1, misaligned="data_p"),
    "marl-v8-e6": case("marl", "k_marl_v8", 1, E=6),
    "marl-v8-v5": case("marl", "k_marl_v8", 1, V=5),
    "marl-rollout-stats-trace": case("marl", "k_marl_rollout", 1, traces=MARL_FAST + ("stats",)),
    "marl-rollout-last-power": case("marl", "k_marl_rollout", 1, traces=MARL_FAST + ("last_power",)),
    "marl-rollout-v12": case("marl", "k_marl_rollout", 1, V=12),
    "marl-force-generic": case("marl", "k_marl_rollout", 1, over={"RISVEC_FORCE_GENERIC": "1"}),
    "marl-packed": case("marl", "k_marl_v8", 1, entry="packed"),
    # MARL driver steps and host-buffer calls
    "marl-fused": case("marl", "k_marl_v8", 1, entry="fused"),
    "marl-fused-stats": case("marl", "k_marl_v8", 2, entry="fused", stats=True),
    "marl-fused-v12": case("marl", "k_marl_rollout", 3, V=12, entry="fused"),
    "marl-fused-misaligned-raw": case("marl", "k_marl_v8", 3, entry="fused", misaligned="raw"),
    "marl-fused-force-generic": case("marl", "k_marl_rollout", 3, entry="fused", over={"RISVEC_FORCE_GENERIC": "1"}),
    "marl-host": case("marl", "k_marl_tma", 1, entry="host"),
    "marl-packed-host": case("marl", "k_marl_v8", 1, entry="packed_host"),
}


def tensor(shape, dtype, device, fill, offset=False):
    """a contiguous tensor; `offset`: its data starts 4 bytes past a 16-byte boundary"""
    n = int(np.prod(shape))
    base = torch.empty(n + 4, dtype=dtype, device=device)
    t = base[1:n + 1].view(shape) if offset else base[:n].view(shape)
    t.copy_(torch.as_tensor(fill).to(dtype))
    return t


@pytest.mark.parametrize("name", list(CASES))
def test_rollout_kernel_choice(name, monkeypatch):
    c = CASES[name]
    for var in ("RISVEC_SARL_PATH", "RISVEC_MARL_PATH", "RISVEC_FORCE_GENERIC"):
        monkeypatch.delenv(var, raising=False)
    for var, val in c["over"].items():
        monkeypatch.setenv(var, val)
    variant, E, V, M, entry = c["variant"], c["E"], c["V"], c["M"], c["entry"]
    env = BatchedEnviron(variant, E, V, M, seed=3)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    if variant == "marl":
        env.optimize_phase_shift(); env.update_channel_gains()
    if c["stats"]:
        env.attach_stats_accumulator()
    rng = np.random.default_rng(11)
    cuda, cpu = env.device, torch.device("cpu")
    acts = rng.random((T, E, 2, V)).astype(np.float32)
    arr = rng.poisson(2.0, (T, E, V)).astype(np.int32)
    phs = (rng.random((T, E, M)) * 2 * np.pi).astype(np.float32)
    partner = np.tile(encode_groups([[v] for v in range(V)], V)[0], (E, 1))
    ngroups = np.full(E, V, np.int32)
    torch.cuda.synchronize()
    n0 = env.launch_count

    if entry in ("rollout", "host"):
        dev = cuda if entry == "rollout" else cpu
        out = {k: tensor(env._trace_shape(k, T), torch.float32, dev, 0.0, offset=k == c["misaligned"])
               for k in c["traces"]}
        a = tensor(acts.shape, torch.float32, dev, acts)
        ar = tensor(arr.shape, torch.int32, dev, arr) if c["arrivals"] else None
        if variant == "sarl":
            ph = tensor(phs.shape, torch.float32, dev, phs)
            if entry == "rollout":
                env.rollout_sarl(a, ph, ar, out=out)
            else:
                env.rollout_sarl_host(a, ph, ar, out)
        else:
            pt, ng = torch.as_tensor(partner).to(dev), torch.as_tensor(ngroups).to(dev)
            if entry == "rollout":
                env.rollout_marl(a, pt, ng, ar, out=out)
            else:
                env.rollout_marl_host(a, pt, ng, ar, out)
    elif entry in ("packed", "packed_host"):
        rec = env.pack_inputs(torch.as_tensor(acts), torch.as_tensor(arr),
                              torch.as_tensor(phs) if variant == "sarl" else None)
        if entry == "packed":
            env.rollout_packed(rec.to(cuda), partner, ngroups)
        else:
            out_rec = torch.empty(T, E // 4, 4 * env.packed_out_words(), dtype=torch.float32)
            env.rollout_packed_host(rec, out_rec, torch.empty(T, E, dtype=torch.float32),
                                    torch.as_tensor(partner), torch.as_tensor(ngroups))
    else:  # fused driver step
        shape = (E, 2 * V + M) if variant == "sarl" else (E, V, 2)
        raw = tensor(shape, torch.float32, cuda, rng.random(shape) * 2 - 1, offset=c["misaligned"] == "raw")
        a1 = torch.as_tensor(arr[0]).to(cuda)
        if variant == "sarl":
            env.step_sarl_fused(raw, a1)
        else:
            env.step_marl_fused(raw, partner, ngroups, a1)
    torch.cuda.synchronize()
    assert (env.last_kernel(), env.launch_count - n0) == (c["kernel"], c["launches"])
