#!/usr/bin/env python
"""What a per-env RIS size (`attach_ris_elements`) costs, and what it saves, on one GPU, in one run.

1. SARL rollout at E = 4096, T = 256, V = 8, M = 40, every trace, injected arrivals; three handles:
     array    - an array attached, every env at 40 elements (k_sarl_mma, the NE instantiation),
     pinned   - no array, the same kernel pinned (RISVEC_SARL_PATH=mma-ldg),
     default  - no array, the default choice (k_sarl_mma_tma).
2. The RIS sweep of plt/plt-ris.py (20, 40, ... 120 elements) done both ways, V = 8:
     one_handle - one handle of M = 120 and E envs, counts 20 ... 120 spread over its envs,
     six_handles - six handles of M = 20 ... 120 with E / 6 envs each, launched one after the other.
   Timed: the MARL channel stage (`begin_episode(stages=("channel",))`: BCD + channel gains) and the SARL rollout
   (T = --sweep-T).
The configurations of one comparison run in alternating rounds (CUDA events around --reps calls per round); the JSON
reports the median over rounds of the per-call time, with the GPU's name, power limit and max SM clock.  --out FILE also
writes the JSON there."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides  # noqa: E402

V = 8
SIZES = (20, 40, 60, 80, 100, 120)


def make_env(variant, E, M, sarl_path=None):
    """a handle created with RISVEC_SARL_PATH set or not (risvec_create reads the variable)"""
    old = os.environ.pop("RISVEC_SARL_PATH", None)
    if sarl_path:
        os.environ["RISVEC_SARL_PATH"] = sarl_path
    try:
        kw = marl_yaml_overrides() if variant == "marl" else {}
        env = BatchedEnviron(variant, E, V, M, seed=1234, **kw)
    finally:
        os.environ.pop("RISVEC_SARL_PATH", None)
        if old is not None:
            os.environ["RISVEC_SARL_PATH"] = old
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    return env


def sarl_rollout_fn(env, T):
    dev, E, M = env.device, env.E, env.M
    g = torch.Generator(device=dev).manual_seed(0)
    act = torch.rand(T, E, 2, V, device=dev, generator=g)
    arr = torch.poisson(torch.full((T, E, V), 2.0, device=dev), generator=g).to(torch.int32)
    ph = torch.rand(T, E, M, device=dev, generator=g) * 6.283185307179586
    names = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
    out = env._alloc_traces(names, T, names)
    return lambda: env.rollout_sarl(act, ph, arr, out=out)


def channel_fn(env):
    return lambda: env.begin_episode(stages=("channel",))


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def compare(configs, rounds, reps):
    """configs: {name: (kernel name getter, fn)}; alternating rounds; median ms per call and the kernel it ran"""
    for _, fn in configs.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(rounds):
        for k, (_, fn) in configs.items():
            times[k].append(timed(fn, reps))
    out = {}
    for k, (kernel, _) in configs.items():
        t = sorted(times[k])
        out[k] = {"kernel": kernel(), "ms_median": t[len(t) // 2], "ms_min": t[0], "ms_max": t[-1]}
    return out


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["nvidia_smi"] = q[0] if q else ""
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def sweep(variant, E, T, rounds, reps):
    per = E // len(SIZES)
    one = make_env(variant, per * len(SIZES), max(SIZES))
    one.attach_ris_elements(counts=torch.tensor(SIZES, dtype=torch.int32, device=one.device).repeat_interleave(per))
    six = [make_env(variant, per, n) for n in SIZES]
    if variant == "marl":
        fns = [channel_fn(one)] + [channel_fn(env) for env in six]
    else:
        fns = [sarl_rollout_fn(one, T)] + [sarl_rollout_fn(env, T) for env in six]

    def all_six():
        for f in fns[1:]:
            f()

    cfg = {"one_handle": (lambda: one.last_kernel() if variant == "sarl" else "k_begin_episode", fns[0]),
           "six_handles": (lambda: [e.last_kernel() for e in six] if variant == "sarl" else "k_begin_episode",
                           all_six)}
    r = compare(cfg, rounds, reps)
    r["one_over_six"] = r["one_handle"]["ms_median"] / r["six_handles"]["ms_median"]
    r["envs"] = per * len(SIZES)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--T", type=int, default=256)
    ap.add_argument("--sweep-T", type=int, default=64)
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_ris_elements needs a CUDA device")
    res = {"gpu": gpu_info(), "E": args.envs, "T": args.T, "sweep_T": args.sweep_T, "V": V, "rounds": args.rounds,
           "reps": args.reps}
    cfg = {}
    for name, path, attach in (("array", "mma-ldg", True), ("pinned", "mma-ldg", False), ("default", None, False)):
        env = make_env("sarl", args.envs, 40, path)
        if attach:
            env.attach_ris_elements()
        cfg[name] = (env.last_kernel, sarl_rollout_fn(env, args.T))
    r = compare(cfg, args.rounds, args.reps)
    for k in ("array", "pinned", "default"):
        r[k]["env_steps_per_s"] = args.envs * args.T / (r[k]["ms_median"] * 1e-3)
    r["array_over_pinned"] = r["array"]["ms_median"] / r["pinned"]["ms_median"]
    r["array_over_default"] = r["array"]["ms_median"] / r["default"]["ms_median"]
    res["rollout_sarl_m40"] = r
    res["sweep_marl_channel"] = sweep("marl", args.envs, args.sweep_T, args.rounds, args.reps)
    res["sweep_sarl_rollout"] = sweep("sarl", args.envs, args.sweep_T, args.rounds, args.reps)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
