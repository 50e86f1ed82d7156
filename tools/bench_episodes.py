#!/usr/bin/env python
"""Per-env episode starts (risvec_begin_episode / risvec_episode_tick), CUDA-event timed after warm-up.

(a) `begin_episode` (the driver's refresh: positions + channel + pairing reset) fused in one launch against the
    separate chain it replaces (renew_positions, compute_parms, optimize_phase_shift, update_channel_gains,
    pair_reset), alternated in the same run: all envs and 1 % of the envs (the separate chain has no per-env form, so
    it always runs on all envs), at E = 4096, V = 8, M = 40 with the config.yaml parameters; and the config-4 shape
    (E = 1024, V = 32, M = 256), where begin_episode takes the per-stage fallback.
(b) The `--driver` loop of bench_actor_loop.py in four forms: lock-step episodes as there (host branch on the step
    counter); staggered episodes (episode_tick + pair_noma_episodes + fused step + replay store with the per-env done
    flags); the staggered loop with the env part (tick, actors, pairing, intent head, step) replayed as a CUDA graph
    and the store of a host-counter replay buffer issued eagerly after each replay (`staggered_graph`); and the whole
    staggered step, store included, as one graph on a device-counter replay buffer (`staggered_graph_full`).

Writes one JSON object (stdout and --out)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_actor_loop import Actors  # noqa: E402
from ris_vec_marl_b200 import BatchedEnviron, ReplayBuffer, marl_yaml_overrides, mask_schedule  # noqa: E402

DRIVER = ("positions", "channel", "pairing")
YAML_SCHED = (7, 7, 0.10, 0.25, 200)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"nvidia-smi failed: {q.stderr.strip()[:200]}"


def event_time(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / n  # us per call


def ab(fns, n, rounds):
    """Median us per call of each named fn, the fns alternated round by round."""
    for f in fns.values():
        for _ in range(3):
            f()
    got = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            got[k].append(event_time(f, n))
    return {k: {"median_us": float(np.median(v)), "min_us": float(np.min(v)), "max_us": float(np.max(v))}
            for k, v in got.items()}


def part_a(E, V, M, n, rounds):
    env = BatchedEnviron("marl", E, V, M, device=0, seed=1234, **marl_yaml_overrides())
    env.set_pairing(yaml=True)
    env.make_new_game()
    env.begin_episode(stages=("reset",) + DRIVER)
    rng = np.random.default_rng(0)
    one_pct = torch.as_tensor((rng.random(E) < 0.01).astype(np.uint8)).to(env.device)
    full = torch.full((E,), 15, dtype=torch.uint8, device=env.device)

    def chain():
        env.renew_positions(); env.compute_parms(); env.optimize_phase_shift(); env.update_channel_gains(); env.pair_reset()

    n0 = env.launch_count
    env.begin_episode(stages=DRIVER)
    fused_launches = env.launch_count - n0
    n0 = env.launch_count
    chain()
    chain_launches = env.launch_count - n0
    fns = {"fused_all": lambda: env.begin_episode(stages=DRIVER),
           "fused_all_per_env_mask": lambda: env.begin_episode(stages=DRIVER, per_env=full),
           "fused_1pct": lambda: env.begin_episode(stages=DRIVER, per_env=one_pct),
           "separate_chain_all": chain}
    res = ab(fns, n, rounds)
    res["config"] = {"envs": E, "V": V, "M": M, "params": "config.yaml", "stages": list(DRIVER),
                     "envs_1pct": int(one_pct.sum()), "launches_begin_episode": fused_launches,
                     "launches_separate_chain": chain_launches, "calls_per_timing": n, "rounds": rounds}
    env.close()
    return res


def part_b(E, steps, rounds):
    V, M = 8, 40
    dev = torch.device("cuda", 0)
    env = BatchedEnviron("marl", E, V, M, device=0, seed=1234, **marl_yaml_overrides())
    env.set_pairing(yaml=True)
    env.make_new_game()
    env.begin_episode(stages=("reset",) + DRIVER)
    actors = Actors(V, dev)
    rb = ReplayBuffer(min(1_000_000, max(4 * E, 65536)), 5, V + 2, V, device=0)
    rb_dev = ReplayBuffer(min(1_000_000, max(4 * E, 65536)), 5, V + 2, V, device=0, device_counter=True)
    obs, obs2 = torch.empty(E, V, 5, device=dev), torch.empty(E, V, 5, device=dev)
    bufs = [obs, obs2]
    env.observe(out=obs)
    K, q = mask_schedule(10, V, 7, 7, 0.10, 0.25, 200)
    frozen = torch.ones(E, dtype=torch.int32, device=dev)
    ctr = [0]

    def lockstep():  # bench_actor_loop.py --driver
        first = ctr[0] % 100 == 0
        ctr[0] += 1
        cur, nxt = bufs[0], bufs[1]
        raw = actors(cur).float()
        act = env.map_actions(raw)
        part, ng = env.pair_noma(act, K, q, recalc_mask=first, reuse=None if first else frozen, new_episode=first)
        probs = actors.intent(env.pair_mask)
        env.step_marl_fused(raw, part, ng, obs_out=nxt)
        rb.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=(ctr[0] % 100 == 0), mask_u8=env.pair_mask)
        bufs[0], bufs[1] = nxt, cur

    tick_out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))

    def env_part(cur, nxt):  # everything but the store: graph-capturable
        start, done = env.episode_tick(steps_per_episode=100, positions_every=5, stages=DRIVER, out=tick_out)
        raw = actors(cur).float()
        act = env.map_actions(raw)
        part, ng = env.pair_noma_episodes(act, start, schedule=YAML_SCHED, reuse=frozen)
        probs = actors.intent(env.pair_mask)
        env.step_marl_fused(raw, part, ng, obs_out=nxt)
        return raw, probs, done

    def staggered():
        cur, nxt = bufs[0], bufs[1]
        raw, probs, done = env_part(cur, nxt)
        rb.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=done, mask_u8=env.pair_mask)
        bufs[0], bufs[1] = nxt, cur

    # staggered start: envs e start their episodes at offsets e % 100
    env.ep_step.copy_(torch.arange(E, dtype=torch.int32, device=dev) % 100)
    def full_step(cur, nxt):  # the whole staggered step, store on the device-counter buffer included
        raw, probs, done = env_part(cur, nxt)
        rb_dev.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=done, mask_u8=env.pair_mask)

    # two graphs per form, one per observation-buffer parity: env part (then the eager store), and the full step
    graphs, full_graphs = [], []
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            env_part(obs, obs2)
            env_part(obs2, obs)
        torch.cuda.synchronize()
        for cur, nxt in ((obs, obs2), (obs2, obs)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                outs = env_part(cur, nxt)
            graphs.append((g, cur, nxt, outs))
        for cur, nxt in ((obs, obs2), (obs2, obs)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                full_step(cur, nxt)
            full_graphs.append(g)
    torch.cuda.current_stream().wait_stream(s)
    gi = [0]

    def staggered_graph():
        g, cur, nxt, (raw, probs, done) = graphs[gi[0]]
        gi[0] ^= 1
        g.replay()
        rb.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=done, mask_u8=env.pair_mask)

    fi = [0]

    def staggered_graph_full():
        full_graphs[fi[0]].replay()
        fi[0] ^= 1

    def loop(fn):
        return lambda: [fn() for _ in range(steps)]

    # the graph form always starts from buffer parity 0; keep the eager forms on an even number of steps too
    assert steps % 2 == 0
    arms = {"lockstep": loop(lockstep), "staggered": loop(staggered), "staggered_graph": loop(staggered_graph),
            "staggered_graph_full": loop(staggered_graph_full)}
    res = ab(arms, 1, rounds)
    for k in arms:
        r = res[k]
        r["us_per_step"] = r["median_us"] / steps
        r["env_steps_per_s"] = E * steps / (r["median_us"] * 1e-6)
    res["config"] = {"envs": E, "V": V, "M": M, "steps_per_timing": steps, "rounds": rounds,
                     "actor": "8 x MLP 5-512-256-{2, V} (bmm), fp32",
                     "graph_part": "episode_tick, actors, map_actions, pair_noma_episodes, intent head, step_marl_fused",
                     "staggered_graph": "graph_part as a graph, then the store of a host-counter buffer, eager",
                     "staggered_graph_full": "graph_part and the store of a device-counter buffer, one graph"}
    res["replay_rows"] = int(rb.mem_cntr)
    res["replay_rows_device_counter"] = int(rb_dev.mem_cntr)
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--driver-envs", type=int, default=8192)
    ap.add_argument("--driver-steps", type=int, default=200)
    ap.add_argument("--driver-rounds", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_episodes.py measures on the GPU"
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0),
           "unit": "us per call (CUDA events after warm-up, median over alternated rounds)"}
    res["begin_episode_v8_m40"] = part_a(4096, 8, 40, a.calls, a.rounds)
    res["begin_episode_config4_v32_m256"] = part_a(1024, 32, 256, max(5, a.calls // 5), a.rounds)
    res["driver_loop"] = part_b(a.driver_envs, a.driver_steps, a.driver_rounds)
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
