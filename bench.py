#!/usr/bin/env python
"""Benchmark of the batched Environ.step hot path (contract: task prompt, section 4).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--workload sarl|marl]

One bench "step" = one fused T-step rollout launch over E envs per GPU (T*E env-steps) with
pre-staged synthetic actions in the reference's own array layout; the metric is env-steps/s
(BASELINE.json).  For N > 1 launch with torchrun (one rank per GPU); envs are sharded, the only
collective is ONE NCCL all-reduce of the episode-statistics vector per timed region.  The JSON line
also carries a `secondary` block with short measurements of the other BASELINE configs.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"


def algorithmic_bytes(workload, V, M, T, E):
    """Bytes one rollout launch must move (DESIGN.md, 'Algorithmic bytes'; SURVEY.md 8d).
    MARL: per step 28V + 4, per env per rollout 2(4V + 8) + 4V + 4V + 4.
    SARL: per step 36V + 4M + 4 (actions 8V, phases 4M, arrivals 4V, six traces 24V, reward 4),
          per env per rollout 2 * 4V (DataBuf in/out) + 8V (angle f64) + 4V (amplitude)."""
    if workload == "marl":
        return E * (T * (28 * V + 4) + 2 * (4 * V + 8) + 4 * V + 4 * V + 4)
    return E * (T * (36 * V + 4 * M + 4) + 2 * 4 * V + 8 * V + 4 * V)


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(kernel):
    """{dram_bytes_per_launch, source} of the named kernel from the committed `ncu --set full` capture
    (profiles/traffic.json; a bench run cannot measure DRAM traffic itself), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's own per-env step loop (unmodified `Environ` objects from the reference
# tree when it is reachable: /root/reference or the staged baseline/_ref), else the oracle port of it;
# one env object per process on every host core
# ------------------------------------------------------------------------------------------
def reference_root():
    from oracle import ref_harness as rh

    return rh.REFERENCE_ROOT if rh.reference_available() else None


def _cpu_worker(args):
    workload, V, M, seconds, seed, use_ref = args
    import numpy as np

    np.random.seed(seed)
    groups = [[i, i + 1] for i in range(0, 3 * V // 4, 2)] + [[i] for i in range(3 * V // 4, V)]
    if use_ref:
        from oracle import ref_harness as rh

        _, env = rh.make_reference_env(workload, V, M, 3)   # the unmodified reference class
        np.random.seed(seed)                                   # (the SARL module reseeds numpy at import)
        if workload == "marl":
            rh.apply_marl_yaml_params(env)
        step_marl = lambda a: env.step(a[0], groups)
        step_sarl = lambda a, ph: env.step(a[0], ph[0])
    else:
        from oracle.env_oracle import EnvOracle, GlobalNumpyDraws, OracleParams, encode_groups

        p = OracleParams.marl_yaml() if workload == "marl" else OracleParams()
        env = EnvOracle(workload, V, M, 3, E=1, params=p, draws=GlobalNumpyDraws())
        partner, ng = encode_groups(groups, V)
        step_marl = lambda a: env.step_marl(a, partner[None], np.array([ng]))
        step_sarl = lambda a, ph: env.step_sarl(a, ph)
    env.make_new_game()
    rng = np.random.default_rng(seed)
    steps, t0 = 0, time.perf_counter()
    episode = 0
    while time.perf_counter() - t0 < seconds:
        # loop shape of the reference drivers (marl_train_bcd.py:1268-1309, ddpg_train.py:120-162)
        if workload == "marl":
            if episode % 5 == 0:
                env.renew_positions(); env.compute_parms()
            env.optimize_phase_shift(); env.update_channel_gains()
        elif episode % 100 == 0:
            env.renew_positions(); env.compute_parms()
        for _ in range(100):
            a = rng.random((1, 2, V))
            if workload == "marl":
                step_marl(a)
            else:
                step_sarl(a, rng.random((1, M)) * 2 * np.pi)
            steps += 1
        episode += 1
    return steps, time.perf_counter() - t0


def cpu_throughput(workload, V, M, seconds, cores):
    """(env-steps/s over all cores, env-steps run, kind) of the CPU step loop."""
    use_ref = reference_root() is not None
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(workload, V, M, seconds, 100 + i, use_ref) for i in range(cores)])
    total = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return total / wall, total, ("reference" if use_ref else "port")


def cpu_sample_text(kind, cores, seconds, n=None):
    what = ("the unmodified reference Environ.step loop (" + os.path.basename(os.path.dirname(reference_root() + "/")) + ")"
            if kind == "reference" else "oracle/env_oracle.py port of the reference step loop")
    tail = f" = {n} env-steps" if n is not None else ""
    return f"{what}, one env object per process in the drivers' loop shape, {cores} processes x {seconds:.1f} s{tail}"


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cores = host_cores()
    V, M = args.V, args.M
    # every "step" of this arm is a bounded sample of the same workload: `sample_s` seconds of
    # the per-env python loop on every host core
    per_step_s = max(1.0, min(10.0, 40.0 / max(1, args.steps + args.warmup)))
    # at most 40 samples are actually run (~1 min), whatever K the caller asks for: the per-sample
    # throughput of the CPU loop does not depend on how many samples are averaged
    warm = min(args.warmup, 3)
    n_run = warm + min(args.steps, 40 - warm)
    vals = []
    for i in range(n_run):
        v, n, kind = cpu_throughput(args.workload, V, M, per_step_s, cores)
        if i >= warm:
            vals.append(v)
    value = sum(vals) / len(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": cpu_sample_text(kind, cores, per_step_s) + f" per bench step, {len(vals)} timed samples"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world=1):
    name = {"sarl": "Simulation-SARL Environment (DDPG single-agent variant)",
            "marl": "Simulation-MARL-BCD Environment (config.yaml parameters)"}[args.workload]
    return {"workload": f"{name}, V={args.V} vehicles, M={args.M} RIS elements, {args.envs} batched envs per GPU, "
                        f"fused T={args.T}-step rollout per launch with pre-staged actions",
            "envs_per_gpu": args.envs, "V": args.V, "M": args.M, "T": args.T,
            "layout": "the reference's own array layout: action [T,E,2,V] f32, phase [T,E,M] f32, arrivals [T,E,V] i32 "
                      "in; one [T,E,V] f32 array per trace + reward [T,E] out (no packing / conversion pass anywhere)",
            "stats_interval": f"statistics interval = the timed region ({args.steps} rollouts x {args.T} steps); every "
                              "rollout adds its last step's statistics to the attached accumulator in the kernel's "
                              "tail, one collect per interval, all inside the timed region",
            "l2_policy": "inputs+outputs of one launch exceed the 126 MB L2; nothing is re-read between launches"}


def event_time_launches(torch, fn, n, warm=3):
    """(avg ms, min ms) of `fn` over n launches, CUDA events on the current stream."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return sum(ms) / len(ms), ms[0]


class Ranks:
    """max / gather over the ranks (identity on one GPU)."""

    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def max(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, vals):
        t = self.torch.tensor([float(v) for v in vals], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [t.tolist()]
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [o.tolist() for o in out]

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()


def make_inputs(torch, wl, E, V, M, T, dev, seed, lam, floor=None):
    gen = torch.Generator(device=dev).manual_seed(seed)
    actions = torch.rand(T, E, 2, V, device=dev, generator=gen)
    arrivals = torch.poisson(torch.full((T, E, V), lam, device=dev), generator=gen).to(torch.int32)
    phases = None
    if wl == "marl":
        actions[:, :, 1, :].clamp_(min=floor)
    else:
        phases = torch.rand(T, E, M, device=dev, generator=gen) * 6.283185307179586
    return actions, arrivals, phases


def marl_groups(torch, E, V, dev):
    """3V/8 pairs + V/4 singletons (SURVEY.md 8d synthetic inputs)."""
    import numpy as np

    from ris_vec_marl_b200 import encode_groups

    groups = [[i, i + 1] for i in range(0, 3 * V // 4, 2)] + [[i] for i in range(3 * V // 4, V)]
    part, ng = encode_groups(groups, V)
    return torch.as_tensor(np.tile(part, (E, 1))).to(dev), torch.full((E,), ng, dtype=torch.int32, device=dev)


SARL_TRACE_NAMES = ("reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate")
MARL_TRACE_NAMES = ("reward_user", "reward", "data_t", "data_p", "rate", "DataBuf")
DUMP_BYTES = 60_000_000   # --dump-outputs budget for all traces together (the .npy headers add < 1 KB)


def sample_traces(torch, out, E):
    """{name: float32 ndarray} of the rollout traces `out` ([T, E, ...] each), restricted to a fixed, seeded sample of
    env indices (the same sample for every trace; all E envs when they fit DUMP_BYTES)."""
    import numpy as np

    per_env = sum(v[:, 0].numel() * v.element_size() for v in out.values())
    n = min(E, DUMP_BYTES // per_env)
    if n < 1:
        raise SystemExit(f"--dump-outputs: the traces of one env alone exceed {DUMP_BYTES} bytes")
    idx = np.arange(E) if n == E else np.sort(np.random.default_rng(0).choice(E, n, replace=False))
    sel = torch.as_tensor(idx, device=next(iter(out.values())).device)
    return {k: v.index_select(1, sel).cpu().numpy() for k, v in out.items()}


def make_rollout(torch, wl, E, V, M, T, local, rank, dev, sarl_path=None):
    """(env, one_step callable, buffers dict) for one workload in the reference layout."""
    from ris_vec_marl_b200 import BatchedEnviron, marl_yaml_overrides

    over = marl_yaml_overrides() if wl == "marl" else {}
    old = os.environ.get("RISVEC_SARL_PATH")
    if sarl_path:
        os.environ["RISVEC_SARL_PATH"] = sarl_path
    try:
        env = BatchedEnviron(wl, E, V, M, 3, device=local, seed=1234, env_index_base=rank * E, **over)
    finally:
        if sarl_path:
            os.environ.pop("RISVEC_SARL_PATH", None) if old is None else os.environ.__setitem__("RISVEC_SARL_PATH", old)
    env.make_new_game(); env.renew_positions(); env.compute_parms()
    lam = float(env.get_param("rate"))
    floor = float(env.get_param("cpu_share_floor")) if wl == "marl" else None
    actions, arrivals, phases = make_inputs(torch, wl, E, V, M, T, dev, rank, lam, floor)
    buf = dict(actions=actions, arrivals=arrivals, phases=phases)
    if wl == "marl":
        env.optimize_phase_shift(); env.update_channel_gains()
        partner, ngroups = marl_groups(torch, E, V, dev)
        out = env._alloc_traces(MARL_TRACE_NAMES, T, MARL_TRACE_NAMES)
        buf.update(partner=partner, ngroups=ngroups, out=out)
        one = lambda: env.rollout_marl(actions, partner, ngroups, arrivals, out=out)
    else:
        out = env._alloc_traces(SARL_TRACE_NAMES, T, SARL_TRACE_NAMES)
        buf.update(out=out)
        one = lambda: env.rollout_sarl(actions, phases, arrivals, out=out)
    return env, one, buf


def kernel_line(torch, ranks, wl, E, V, M, T, one, env, peak, n=10):
    avg, mn = event_time_launches(torch, one, n)
    avg = ranks.max(avg)
    alg = algorithmic_bytes(wl, V, M, T, E)
    return {"kernel": env.last_kernel(), "ms_per_launch": avg, "ms_min": mn, "env_steps_per_launch": E * T,
            "value": ranks.world * E * T / (avg * 1e-3), "unit": UNIT,
            "hbm_frac": alg / (avg * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": alg}


def secondary_block(torch, ranks, args, rank, local, dev, peak):
    """The other BASELINE.json configs and A/B variants, measured in the same run (short: a few launches
    each, CUDA events, max over ranks; whole-job values).  Every entry names the kernel that ran."""
    sec = {}
    world = ranks.world
    E, V, M, T = 4096, 8, 40, 256
    try:  # config 3: MARL-BCD, 8 vehicles, 4096 envs per GPU
        env, one, buf = make_rollout(torch, "marl", E, V, M, T, local, rank, dev)
        sec["config3_marl_v8_m40"] = kernel_line(torch, ranks, "marl", E, V, M, T, one, env, peak)
        del env, one, buf
    except Exception as exc:
        sec["config3_marl_v8_m40"] = {"error": repr(exc)[:200]}
    try:  # config 2 A/B: the FP32-pipe kernel on the same arrays, and on its private packed records
        env, one, buf = make_rollout(torch, "sarl", E, V, M, T, local, rank, dev, sarl_path="v8")
        sec["config2_sarl_fp32_pipe_kernel"] = kernel_line(torch, ranks, "sarl", E, V, M, T, one, env, peak)
        rec = env.pack_inputs(buf["actions"], buf["arrivals"], buf["phases"])
        out_rec = torch.empty(T, E // 4, 4 * env.packed_out_words(), dtype=torch.float32, device=dev)
        rew = torch.empty(T, E, dtype=torch.float32, device=dev)
        line = kernel_line(torch, ranks, "sarl", E, V, M, T, lambda: env.rollout_packed(rec, out_rec=out_rec, reward=rew),
                           env, peak)
        line["note"] = "round-1 headline path: tiled records; the pack / unpack conversion passes are NOT in this time"
        sec["config2_sarl_packed_records"] = line
        del env, one, buf, rec, out_rec, rew
    except Exception as exc:
        sec["config2_sarl_ab"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()
    try:  # config 4: 32 vehicles, 256 RIS elements, 1024 envs per GPU
        E4, V4, M4, T4 = 1024, 32, 256, 256
        c4 = {"envs_per_gpu": E4, "V": V4, "M": M4, "T": T4}
        env, one, buf = make_rollout(torch, "sarl", E4, V4, M4, T4, local, rank, dev)
        c4["sarl_step"] = kernel_line(torch, ranks, "sarl", E4, V4, M4, T4, one, env, peak, n=5)
        flops = 8.0 * V4 * M4 * E4 * T4
        c4["sarl_step"]["cascade_tflops"] = flops / (c4["sarl_step"]["ms_per_launch"] * 1e-3) / 1e12
        del env, one, buf
        for key, path in (("sarl_step_mma_sync_kernel", "mma-sync"), ("sarl_step_round1_kernels", "generic")):  # A/B arms
            env, one, buf = make_rollout(torch, "sarl", E4, V4, M4, T4, local, rank, dev, sarl_path=path)
            c4[key] = kernel_line(torch, ranks, "sarl", E4, V4, M4, T4, one, env, peak, n=5)
            del env, one, buf
        c4["sarl_speedup_vs_round1_kernels"] = c4["sarl_step_round1_kernels"]["ms_per_launch"] / c4["sarl_step"]["ms_per_launch"]
        env, one, buf = make_rollout(torch, "marl", E4, V4, M4, T4, local, rank, dev)
        c4["marl_step"] = kernel_line(torch, ranks, "marl", E4, V4, M4, T4, one, env, peak, n=5)
        c4["bcd_us_per_launch"] = ranks.max(event_time_launches(torch, env.optimize_phase_shift, 5)[0]) * 1e3
        c4["gains_us_per_launch"] = ranks.max(event_time_launches(torch, env.update_channel_gains, 5)[0]) * 1e3
        del env, one, buf
        sec["config4_v32_m256"] = c4
    except Exception as exc:
        sec["config4_v32_m256"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()
    try:  # config 5: the driver's per-step loop with the actors in torch, 8192 envs per GPU
        from tools.bench_actor_loop import driver_loop

        sec["config5_driver_loop_actor_in_torch"] = driver_loop(8192, 50, True, "bf16", rank, world, local, ranks)
    except Exception as exc:
        sec["config5_driver_loop_actor_in_torch"] = {"error": repr(exc)[:200]}
    torch.cuda.empty_cache()
    return sec


# ------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="sarl", choices=["sarl", "marl"])
    ap.add_argument("--envs", type=int, default=4096, help="env instances per GPU")
    ap.add_argument("--T", type=int, default=256, help="env steps fused per launch")
    ap.add_argument("--V", type=int, default=8)
    ap.add_argument("--M", type=int, default=40)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other configs' short measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the traces the last timed rollout returned (rank 0's shard) as DIR/<name>.npy, float32 "
                         f"[T, n, ...] over a fixed, seeded sample of n env indices (all envs when they fit {DUMP_BYTES} "
                         "bytes); the same arguments give the same inputs on every run, so two builds compare output "
                         "for output (bench_outputs/ in the repository is git-ignored for this)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA rollout's traces: it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist

    from ris_vec_marl_b200 import load_library

    load_library()  # no CUDA extension => hard failure, never a fallback
    assert torch.cuda.is_available(), "bench.py needs a GPU for --impl ours"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ranks = Ranks(torch, dist, world, dev)

    E, V, M, T = args.envs, args.V, args.M, args.T
    wl = args.workload
    env, one_step, buf = make_rollout(torch, wl, E, V, M, T, local, rank, dev)
    stats_sum = torch.zeros(17, dtype=torch.float64, device=dev)
    shared, stats_mode = None, "one device (no reduction)"
    if world > 1:
        # statistics reduction: rank 0's accumulator mapped into every rank (CUDA IPC over NVLink peer access);
        # k_shard_stats adds each shard's sums into it with float64 atomics -- no collective, no rank waits.
        # RISVEC_BENCH_STATS=nccl (or a failed mapping) selects ONE NCCL all-reduce per timed region instead.
        ok = torch.ones(1, device=dev)
        if os.environ.get("RISVEC_BENCH_STATS", "peer") == "peer":
            try:
                from ris_vec_marl_b200.dist import SharedStats

                shared = SharedStats(local, rank, world)
            except Exception as exc:  # all ranks must take the same path
                sys.stderr.write(f"[bench] rank {rank}: peer mapping unavailable ({exc!r})\n")
                ok.zero_()
        else:
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok.item()) < 1.0 and shared is not None:
            shared.close()
            shared = None
        stats_mode = ("every rank sums its per-rollout statistics in its own HBM and, once per interval, adds the 17 sums "
                      "into rank 0's accumulator with float64 atomics over NVLink peer memory (CUDA IPC mapping, one "
                      "launch): no collective, no rank waits for another; totals read after the end barrier"
                      if shared is not None else "one NCCL all-reduce of the 17-entry vector per timed region")

    # per-rollout statistics: folded into the rollout kernel's tail (risvec_attach_stats_accumulator), no separate pass
    # (RISVEC_BENCH_FOLD=0: the separate k_shard_stats launch after every rollout, for A/B runs)
    fold = os.environ.get("RISVEC_BENCH_FOLD", "1") != "0"
    env.attach_stats_accumulator(fold)

    def episode_stats():
        if not fold:
            env.shard_stats(out=stats_sum, accumulate=True)

    def reduce_stats():   # the only exchange on the path (SURVEY.md 8e): once per statistics interval
        if fold:
            env.collect_stats(out=stats_sum, accumulate=True)
        if shared is not None:
            shared.add_(stats_sum)
        elif world > 1:
            dist.all_reduce(stats_sum)

    for _ in range(args.warmup):
        one_step(); episode_stats()
    reduce_stats()
    torch.cuda.synchronize()

    # ---- timed region: K steps, device-timed, max over ranks
    sampler = ClockSampler(local)
    if rank == 0:
        # the spin below runs for a wall-clock time, not a step count: restore the env afterwards so that the timed
        # steps start from the state the warm-up left, the same on every run with the same arguments
        warm_state = env.state_dict()
        sampler.start()
        t_spin = time.time()
        while True:  # keep the GPU under load until nvidia-smi delivers its first sample (<= 3 s)
            for _ in range(max(args.warmup, 20)):
                one_step()
            torch.cuda.synchronize()
            if sampler.lines or sampler.proc is None or time.time() - t_spin > 3.0:
                break
        sampler.lines.clear()
        env.load_state_dict(warm_state)
        del warm_state
    if fold:
        env.collect_stats()  # discard what the warm-up rollouts accumulated
    stats_sum.zero_()
    if shared is not None:
        shared.zero_()
    ranks.barrier()
    torch.cuda.synchronize()
    if world > 1:
        # the host-side barrier releases the ranks tens of microseconds apart; a tiny all-reduce on the stream
        # makes the timed region START at the same device instant on every rank (its completion is
        # simultaneous), so that max-over-ranks measures the slowest rank's work and not the barrier skew
        dist.all_reduce(torch.zeros(1, device=dev))
        # ... followed by a ~0.25 ms device-side spin: the rank whose host joined that all-reduce last would
        # otherwise start its timed region with an EMPTY queue (its first rollout is still being enqueued by
        # python) and time its own launch latency; every rank's queue is full when the spin ends
        torch.cuda._sleep(500_000)
    l0 = env.launch_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    h0 = time.perf_counter()
    ev[0].record()
    kev_every = int(os.environ.get("RISVEC_BENCH_KEV_EVERY", "1"))  # diagnostic: time every n-th launch only
    for i in range(args.steps):
        if i % kev_every == 0:
            kev[i][0].record()
        one_step()
        if i % kev_every == 0:
            kev[i][1].record()
        episode_stats()
    ev[1].record()
    h1 = time.perf_counter()
    reduce_stats()
    ev[2].record()
    torch.cuda.synchronize()
    ranks.barrier()
    launches = env.launch_count - l0 + (1 if shared is not None else 0)   # + the interval's k_atomic_add_f64
    stats_total = shared.read() if shared is not None else stats_sum.cpu()
    mean_reward = float(stats_total[16]) / (world * E * args.steps)
    ms_local = ev[0].elapsed_time(ev[2])
    kern_ms = sorted(a.elapsed_time(b) for i, (a, b) in enumerate(kev) if i % kev_every == 0)
    kern_ms_avg = sum(kern_ms) / len(kern_ms)
    per_rank = ranks.gather([ms_local, kern_ms_avg, ev[1].elapsed_time(ev[2]), (h1 - h0) / args.steps * 1e6])
    ms_total = ranks.max(ms_local)
    clocks = sampler.stop() if rank == 0 else None
    value = world * E * T * args.steps / (ms_total * 1e-3)
    kernel_name = env.last_kernel()
    dumped = sample_traces(torch, buf["out"], E) if args.dump_outputs and rank == 0 else None

    # ---- end to end through the public host-buffer API (pinned host in, pinned host out), same layout
    actions, arrivals, phases, out = buf["actions"], buf["arrivals"], buf["phases"], buf["out"]
    h_act, h_arr = actions.cpu().pin_memory(), arrivals.cpu().pin_memory()
    h_o = {k: torch.empty(v.shape, dtype=torch.float32).pin_memory() for k, v in out.items()}
    h_rew = h_o["reward"]
    if wl == "marl":
        h_part, h_ng = buf["partner"].cpu().pin_memory(), buf["ngroups"].cpu().pin_memory()
        run_host = lambda: env.rollout_marl_host(h_act, h_part, h_ng, h_arr, h_o)
        h2d = (h_act.numel() + h_arr.numel() + h_part.numel() + h_ng.numel()) * 4
    else:
        h_ph = phases.cpu().pin_memory()
        run_host = lambda: env.rollout_sarl_host(h_act, h_ph, h_arr, h_o)
        h2d = (h_act.numel() + h_arr.numel() + h_ph.numel()) * 4
    d2h = sum(v.numel() * 4 for v in h_o.values())
    run_host(); torch.cuda.synchronize()
    ranks.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.e2e_steps):
        run_host()
        torch.cuda.current_stream().synchronize()  # the caller reads the step's result on the host
        _ = float(h_rew[-1, 0])
    e1.record()
    torch.cuda.synchronize()
    e2e_ms_local = e0.elapsed_time(e1)
    e2e_ranks = ranks.gather([e2e_ms_local])
    e2e_value = world * E * T * args.e2e_steps / (ranks.max(e2e_ms_local) * 1e-3)
    # lean variant of the same public call: arrivals drawn on the device (Philox), only the traces a
    # learner consumes (reward, DataBuf, data_t, data_p, rate) copied back
    e2e_lean = None
    if wl == "sarl":
        lean = {k: h_o[k] for k in ("reward", "DataBuf", "data_t", "data_p", "rate")}
        run_lean = lambda: env.rollout_sarl_host(h_act, h_ph, None, lean)
        run_lean(); torch.cuda.synchronize()
        ranks.barrier()
        e0.record()
        for _ in range(args.e2e_steps):
            run_lean()
            torch.cuda.current_stream().synchronize()
            _ = float(h_rew[-1, 0])
        e1.record()
        torch.cuda.synchronize()
        lean_ms = ranks.max(e0.elapsed_time(e1))
        e2e_lean = {"value": world * E * T * args.e2e_steps / (lean_ms * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": (h_act.numel() + h_ph.numel()) * 4,
                    "d2h_bytes_per_step": sum(v.numel() * 4 for v in lean.values()), "kernel": env.last_kernel(),
                    "what": "arrivals drawn on the device (Philox), 5 of the 7 traces copied back"}
    # the copy roofline of the e2e step, measured here: this rank's host<->device link with plain pinned copies of
    # the step's byte counts, one direction alone and both directions at once (two streams)
    pcie = None
    try:
        hb_in = torch.empty(h2d, dtype=torch.uint8).pin_memory()
        hb_out = torch.empty(d2h, dtype=torch.uint8).pin_memory()
        db_in = torch.empty(h2d, dtype=torch.uint8, device=dev)
        db_out = torch.empty(d2h, dtype=torch.uint8, device=dev)
        s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

        def copy_ms(do_in, do_out, reps=3):
            torch.cuda.synchronize()
            ranks.barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            s_in.wait_event(a0); s_out.wait_event(a0)
            for _ in range(reps):
                if do_in:
                    with torch.cuda.stream(s_in):
                        db_in.copy_(hb_in, non_blocking=True)
                if do_out:
                    with torch.cuda.stream(s_out):
                        hb_out.copy_(db_out, non_blocking=True)
            torch.cuda.current_stream().wait_stream(s_in); torch.cuda.current_stream().wait_stream(s_out)
            a1.record()
            torch.cuda.synchronize()
            return a0.elapsed_time(a1) / reps

        copy_ms(True, True, 1)
        t_in, t_out, t_both = copy_ms(True, False), copy_ms(False, True), copy_ms(True, True)
        pcie = {"h2d_alone_gbs": h2d / t_in / 1e6, "d2h_alone_gbs": d2h / t_out / 1e6,
                "both_directions_ms_per_step": ranks.max(t_both),
                "copy_bound_value": world * E * T / (ranks.max(t_both) * 1e-3),
                "what": "plain pinned cudaMemcpyAsync of one step's H2D and D2H byte counts on two streams, all ranks at "
                        "once: the env-steps/s a zero-cost kernel would reach through this host link"}
        del hb_in, hb_out, db_in, db_out
    except Exception as exc:  # a measurement aid, never fatal
        pcie = {"error": repr(exc)[:200]}
    del h_act, h_arr, h_o
    peak, peak_src = measured_peak_gbs()
    secondary = None
    if not args.no_secondary:
        del env, one_step, buf, actions, arrivals, phases, out
        torch.cuda.empty_cache()
        secondary = secondary_block(torch, ranks, args, rank, local, dev, peak)

    if rank == 0:
        alg = algorithmic_bytes(wl, V, M, T, E)
        achieved = alg / (kern_ms_avg * 1e-3) / 1e9
        traffic = recorded_traffic(kernel_name) if (E, V, M, T) == (4096, 8, 40, 256) else None
        step_s = [r[0] / 1e3 / args.e2e_steps for r in e2e_ranks]
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, world), stats_reduction=stats_mode),
            "clocks": clocks, "mean_reward_last_steps": mean_reward,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps,
                    "per_rank": [{"rank": r, "ms_per_step": s * 1e3, "h2d_gbs": h2d / s / 1e9, "d2h_gbs": d2h / s / 1e9}
                                 for r, s in enumerate(step_s)],
                    "copy_roofline": pcie,
                    "limiter": "host<->device copies: PCIe Gen5 x16 per GPU at N=1; at N>1 the ranks share the host's "
                               "memory / root-complex bandwidth (per-rank GB/s above), the kernel is <1 % of the step",
                    "lean": e2e_lean},
            "gpu_launches": launches,
            "ranks": [{"rank": r, "ms_total": v[0], "kernel_ms_avg": v[1], "stats_reduce_ms": v[2],
                       "host_enqueue_us_per_step": v[3]} for r, v in enumerate(per_rank)],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                         "traffic_source": (traffic or {}).get("source"),
                         "kernel": kernel_name, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "kernel_ms_avg": kern_ms_avg,
                         "kernel_ms_min": kern_ms[0], "env_steps_per_launch": E * T},
        }
        if secondary is not None:
            line["secondary"] = secondary
        if world == 1 and not args.no_cpu_baseline:
            cores = host_cores()
            v, n, kind = cpu_throughput(wl, V, M, args.cpu_seconds, cores)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": cpu_sample_text(kind, cores, args.cpu_seconds, n)}
        if dumped is not None:
            import numpy as np

            os.makedirs(args.dump_outputs, exist_ok=True)
            for k, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, f"{k}.npy"), a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
