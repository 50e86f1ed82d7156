#!/usr/bin/env python
"""What a per-env parameter table (`attach_env_params`) costs, on one GPU, in one run.

Rollouts at E = 4096, T = 256 (V = 8, M = 40, every trace, injected arrivals), per variant three handles:
  table     - a table attached (k_marl_v8 / k_sarl_mma, the PE instantiations),
  pinned    - no table, the same kernel pinned (RISVEC_MARL_PATH=v8 / RISVEC_SARL_PATH=mma-ldg),
  default   - no table, the default choice (k_marl_tma / k_sarl_mma_tma).
The fused driver step (`step_*_fused`) at E = 8192, with and without a table, and the SARL one also at M = 64,
where `k_sarl_mma` runs with KT = 8 k-tiles and spills (with a table somewhat more, DESIGN.md).  The configurations
of one comparison run in alternating rounds (CUDA events around --reps launches per round); the JSON reports the median
over rounds of the per-launch time, with the GPU's name and power limit.  --out FILE also writes the JSON there."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides  # noqa: E402

V, M = 8, 40
PIN = {"marl": ("RISVEC_MARL_PATH", "v8"), "sarl": ("RISVEC_SARL_PATH", "mma-ldg")}


def make_env(variant, E, pinned, M=M):
    """a handle created with the variant's kernel pinned or not (risvec_create reads the variable)"""
    var, val = PIN[variant]
    old = os.environ.pop(var, None)
    if pinned:
        os.environ[var] = val
    try:
        kw = marl_yaml_overrides() if variant == "marl" else {}
        env = BatchedEnviron(variant, E, V, M, seed=1234, **kw)
    finally:
        os.environ.pop(var, None)
        if old is not None:
            os.environ[var] = old
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    if variant == "marl":
        env.optimize_phase_shift(); env.update_channel_gains()
    return env


def heterogeneous(env):
    """a table whose rows differ: P_max / rate (MARL) or rate / t_factor1 (SARL) spread over the envs"""
    env.attach_env_params()
    x = torch.linspace(0.5, 1.5, env.E, dtype=torch.float64, device=env.device)
    if env.variant == "marl":
        env.set_env_params(P_max=env.params.P_max * x, rate=env.params.rate * x)
    else:
        env.set_env_params(rate=env.params.rate * x, t_factor1=env.params.t_factor1 * x)


def rollout_fn(env, T):
    dev, E = env.device, env.E
    g = torch.Generator(device=dev).manual_seed(0)
    act = torch.rand(T, E, 2, V, device=dev, generator=g)
    arr = torch.poisson(torch.full((T, E, V), 2.0, device=dev), generator=g).to(torch.int32)
    if env.variant == "marl":
        names = ("reward_user", "reward", "DataBuf", "data_t", "data_p", "rate")
        out = env._alloc_traces(names, T, names)
        part = torch.full((E, V), -1, dtype=torch.int32, device=dev)   # every vehicle its own OMA group
        ng = torch.full((E,), V, dtype=torch.int32, device=dev)
        return lambda: env.rollout_marl(act, part, ng, arr, out=out)
    ph = torch.rand(T, E, M, device=dev, generator=g) * 6.283185307179586
    names = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
    out = env._alloc_traces(names, T, names)
    return lambda: env.rollout_sarl(act, ph, arr, out=out)


def fused_fn(env):
    dev, E, M = env.device, env.E, env.M
    g = torch.Generator(device=dev).manual_seed(1)
    if env.variant == "marl":
        raw = torch.rand(E, V, 2, device=dev, generator=g) * 2 - 1
        obs = torch.empty(E, V, 5, device=dev)
        part = torch.full((E, V), -1, dtype=torch.int32, device=dev)
        ng = torch.full((E,), V, dtype=torch.int32, device=dev)
        return lambda: env.step_marl_fused(raw, part, ng, obs_out=obs)
    raw = torch.rand(E, 2 * V + M, device=dev, generator=g) * 2 - 1
    obs = torch.empty(E, V, M // V + 5, device=dev)
    return lambda: env.step_sarl_fused(raw, obs_out=obs)


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def compare(configs, rounds, reps):
    """configs: {name: (env, fn)}; alternating rounds; median ms per launch and the kernel each one ran"""
    for _, fn in configs.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in configs}
    for _ in range(rounds):
        for k, (_, fn) in configs.items():
            times[k].append(timed(fn, reps))
    out = {}
    for k, (env, _) in configs.items():
        t = sorted(times[k])
        out[k] = {"kernel": env.last_kernel(), "ms_median": t[len(t) // 2], "ms_min": t[0], "ms_max": t[-1]}
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--T", type=int, default=256)
    ap.add_argument("--fused-envs", type=int, default=8192)
    ap.add_argument("--rounds", type=int, default=11)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_env_params needs a CUDA device")
    res = {"gpu": gpu_info(), "E": args.envs, "T": args.T, "V": V, "M": M, "fused_E": args.fused_envs,
           "rounds": args.rounds, "reps": args.reps}
    for variant in ("marl", "sarl"):
        cfg = {}
        for name, pinned, table in (("table", True, True), ("pinned", True, False), ("default", False, False)):
            env = make_env(variant, args.envs, pinned)
            if table:
                heterogeneous(env)
            cfg[name] = (env, rollout_fn(env, args.T))
        r = compare(cfg, args.rounds, args.reps)
        for v in r.values():
            v["env_steps_per_s"] = args.envs * args.T / (v["ms_median"] * 1e-3)
        r["table_over_pinned"] = r["table"]["ms_median"] / r["pinned"]["ms_median"]
        r["table_over_default"] = r["table"]["ms_median"] / r["default"]["ms_median"]
        res[f"rollout_{variant}"] = r
        cfg = {}
        for name, table in (("table", True), ("no_table", False)):
            env = make_env(variant, args.fused_envs, False)
            if table:
                heterogeneous(env)
            cfg[name] = (env, fused_fn(env))
        r = compare(cfg, args.rounds, 5 * args.reps)
        r["table_over_no_table"] = r["table"]["ms_median"] / r["no_table"]["ms_median"]
        res[f"step_{variant}_fused"] = r
    cfg = {}
    for name, table in (("table", True), ("no_table", False)):
        env = make_env("sarl", args.fused_envs, False, M=64)
        if table:
            heterogeneous(env)
        cfg[name] = (env, fused_fn(env))
    r = compare(cfg, args.rounds, 5 * args.reps)
    r["table_over_no_table"] = r["table"]["ms_median"] / r["no_table"]["ms_median"]
    res["step_sarl_fused_m64"] = r
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
