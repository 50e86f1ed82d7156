#!/usr/bin/env python
"""Per-episode statistics (risvec_episode_accumulate / EpisodeLog), CUDA-event timed after warm-up.

(a) One `accumulate` call at E = 8192 and 65536 (MARL, V = 8, M = 40), with 1 % and with 100 % of the envs done, the
    cases alternated round by round.  Each case is timed as eager python calls and as the same calls captured in one
    CUDA graph: the graph form is the device time, the eager form adds the host's enqueue of each call.  The log's
    counter is cleared before every timed window and the capacity holds every record of the window, so each done env
    really writes its record.  The algorithmic bytes per call (stats,
    reward, reward_user and done read, the running rows read and written, the records written) are computed from the
    shapes and divided by the median time.
(b) The staggered driver loop of bench_episodes.py part (b) at 8192 envs with its env part replayed as a CUDA graph,
    once as there and once with `log.accumulate(done)` captured in the same graph, the two forms alternated.  The
    replay store stays an eager launch after each replay in both forms (its slot counter lives on the host).

Writes one JSON object (stdout and --out)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_actor_loop import Actors  # noqa: E402
from bench_episodes import DRIVER, YAML_SCHED, ab, gpu_info  # noqa: E402
from ris_vec_marl_b200 import BatchedEnviron, EpisodeLog, ReplayBuffer, _lib, marl_yaml_overrides  # noqa: E402


def marl_env(E):
    env = BatchedEnviron("marl", E, 8, 40, device=0, seed=1234, **marl_yaml_overrides())
    env.set_pairing(yaml=True)
    env.make_new_game()
    env.begin_episode(stages=("reset",) + DRIVER)
    return env


def part_a(E, n, rounds):
    V = 8
    env = marl_env(E)
    # one step, so stats / reward / reward_user hold a step's values
    raw = torch.rand(E, V, 2, device=env.device) * 2 - 1
    part, ng = env.pair_noma(env.map_actions(raw), V - 1, 0.2, recalc_mask=True, new_episode=True)
    env.step_marl_fused(raw, part, ng)
    log = EpisodeLog(env, capacity=E * n)
    rng = np.random.default_rng(0)
    done = {"1pct": torch.as_tensor((rng.random(E) < 0.01).astype(np.uint8)).to(env.device),
            "100pct": torch.ones(E, dtype=torch.uint8, device=env.device)}
    n0 = env.launch_count
    log.accumulate(done["1pct"])
    launches = env.launch_count - n0

    # the n calls once more as a captured graph: device time without the host's per-call enqueue
    graphs = {}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for k, d in done.items():
            graphs[k] = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graphs[k], stream=s):
                for _ in range(n):
                    log.accumulate(d)
    torch.cuda.current_stream().wait_stream(s)

    def window(d, g=None):
        def f():
            log.count.zero_()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if g is not None:
                g.replay()
            else:
                for _ in range(n):
                    log.accumulate(d)
            b.record()
            torch.cuda.synchronize()
            assert int(log.count.item()) == n * int(d.sum()) <= log.capacity
            return a.elapsed_time(b) * 1e3 / n
        return f

    fns = {}
    for k, d in done.items():
        fns[k] = window(d)
        fns[k + "_graph"] = window(d, graphs[k])
    for f in fns.values():
        f()
    got = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            got[k].append(f())
    C = _lib.eplog_run_cols(V)
    res = {}
    for k in fns:
        nd = int(done[k.replace("_graph", "")].sum())
        byts = E * (4 * _lib.NSTAT + 4 + 4 * V + 1 + 2 * 8 * C) + nd * 8 * (C + 2)
        med = float(np.median(got[k]))
        res[k] = {"median_us": med, "min_us": float(np.min(got[k])), "max_us": float(np.max(got[k])),
                  "envs_done": nd, "algorithmic_bytes": byts, "achieved_GBps": byts / (med * 1e-6) / 1e9}
    res["config"] = {"envs": E, "V": V, "M": 40, "running_cols": C, "launches_per_call": launches,
                     "calls_per_timing": n, "rounds": rounds}
    env.close()
    return res


def part_b(E, steps, rounds):
    V = 8
    dev = torch.device("cuda", 0)
    env = marl_env(E)
    actors = Actors(V, dev)
    rb = ReplayBuffer(min(1_000_000, max(4 * E, 65536)), 5, V + 2, V, device=0)
    log = EpisodeLog(env, capacity=1 << 20)
    obs, obs2 = torch.empty(E, V, 5, device=dev), torch.empty(E, V, 5, device=dev)
    env.observe(out=obs)
    frozen = torch.ones(E, dtype=torch.int32, device=dev)
    tick_out = (torch.empty(E, dtype=torch.uint8, device=dev), torch.empty(E, dtype=torch.uint8, device=dev))

    def env_part(cur, nxt, with_log):  # bench_episodes.py part (b), + the episode log
        start, done = env.episode_tick(steps_per_episode=100, positions_every=5, stages=DRIVER, out=tick_out)
        raw = actors(cur).float()
        act = env.map_actions(raw)
        part, ng = env.pair_noma_episodes(act, start, schedule=YAML_SCHED, reuse=frozen)
        probs = actors.intent(env.pair_mask)
        env.step_marl_fused(raw, part, ng, obs_out=nxt)
        if with_log:
            log.accumulate(done)
        return raw, probs, done

    env.ep_step.copy_(torch.arange(E, dtype=torch.int32, device=dev) % 100)
    graphs = {False: [], True: []}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            env_part(obs, obs2, False)
            env_part(obs2, obs, False)
        torch.cuda.synchronize()
        for with_log in (False, True):
            for cur, nxt in ((obs, obs2), (obs2, obs)):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=s):
                    outs = env_part(cur, nxt, with_log)
                graphs[with_log].append((g, cur, nxt, outs))
    torch.cuda.current_stream().wait_stream(s)

    def loop(with_log):
        def f():
            for i in range(steps):
                g, cur, nxt, (raw, probs, done) = graphs[with_log][i & 1]
                g.replay()
                rb.store_marl(cur, probs, raw, env.reward, env.reward_user, nxt, done=done, mask_u8=env.pair_mask)
        return f

    assert steps % 2 == 0  # each loop ends on buffer parity 0, where the next one starts
    res = ab({"staggered_graph": loop(False), "staggered_graph_with_log": loop(True)}, 1, rounds)
    for k in ("staggered_graph", "staggered_graph_with_log"):
        r = res[k]
        r["us_per_step"] = r["median_us"] / steps
        r["env_steps_per_s"] = E * steps / (r["median_us"] * 1e-6)
    res["log_cost_us_per_step"] = (res["staggered_graph_with_log"]["us_per_step"]
                                   - res["staggered_graph"]["us_per_step"])
    eps = log.drain()
    res["episodes_logged"] = int(len(eps["env"]))
    res["episodes_dropped"] = int(eps["dropped"])
    res["config"] = {"envs": E, "V": V, "M": 40, "steps_per_episode": 100, "steps_per_timing": steps,
                     "rounds": rounds, "actor": "8 x MLP 5-512-256-{2, V} (bmm), fp32",
                     "graph_part": "episode_tick, actors, map_actions, pair_noma_episodes, intent head, step_marl_fused"
                                   " [, EpisodeLog.accumulate]",
                     "eager_after_each_replay": "replay store"}
    env.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--driver-envs", type=int, default=8192)
    ap.add_argument("--driver-steps", type=int, default=200)
    ap.add_argument("--driver-rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_episode_log.py measures on the GPU"
    res = {"gpu": gpu_info(), "device": torch.cuda.get_device_name(0),
           "unit": "us per call (CUDA events after warm-up, median over alternated rounds)"}
    for E in (8192, 65536):
        res[f"accumulate_E{E}"] = part_a(E, a.calls, a.rounds)
    res["driver_loop"] = part_b(a.driver_envs, a.driver_steps, a.driver_rounds)
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
