#!/usr/bin/env python
"""Replay-memory write path (SURVEY.md 8f row 4): fused `store_marl` of E transitions per call, CUDA-event timed,
against the achieved-bytes roofline (pure copy: reads + writes of one 936 B row per env at V = 8).  Also the same
store on a device-counter buffer (`device_counter=True`), eager and as a graph of 20 stores: there every captured
store lands in fresh slots on every replay, which the run checks from the count."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from ris_vec_marl_b200 import ReplayBuffer  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--V", type=int, default=8)
    ap.add_argument("--size", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    E, V = a.envs, a.V
    dev = torch.device("cuda", 0)
    rb = ReplayBuffer(a.size, 5, V + 2, V)
    g = torch.Generator(device=dev).manual_seed(0)
    r = lambda *s: torch.rand(*s, device=dev, generator=g)  # noqa: E731
    state, state_, probs, power = r(E, 5 * V), r(E, 5 * V), r(E, V, V), r(E, V, 2)
    rg, rl = r(E), r(E, V)
    mask = (r(E, V, V) < 0.7).to(torch.uint8)

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(a.reps):
            fn()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / a.reps * 1e3

    us = timed(lambda: rb.store_marl(state, probs, power, rg, rl, state_, False, mask))
    # the python call (eight argument conversions) costs more than the kernel: replay 20 stores as ONE CUDA
    # graph to see the device time of a store
    us_graph = None
    try:
        gph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            rb.store_marl(state, probs, power, rg, rl, state_, False, mask)
            torch.cuda.synchronize()
            with torch.cuda.graph(gph, stream=side):
                for _ in range(20):
                    rb.store_marl(state, probs, power, rg, rl, state_, False, mask)
        us_graph = timed(gph.replay) / 20
    except Exception as exc:  # capture is best-effort
        us_graph = None
        print("graph capture failed:", repr(exc)[:200], file=sys.stderr)
    # device-counter buffer: the count is read and advanced on the device, so the 20 captured stores write 20 * E
    # fresh rows per replay (a host-counter capture rewrites the same slots every replay)
    rbd = ReplayBuffer(a.size, 5, V + 2, V, device_counter=True)
    state3, state3_ = state.view(E, V, 5), state_.view(E, V, 5)
    store_d = lambda: rbd.store_marl(state3, probs, power, rg, rl, state3_, False, mask)  # noqa: E731
    us_d = timed(store_d)
    gd = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(gd, stream=side):
            for _ in range(20):
                store_d()
    torch.cuda.current_stream().wait_stream(side)
    n0 = rbd.mem_cntr
    us_d_graph = timed(gd.replay) / 20
    rows_per_replay = (rbd.mem_cntr - n0) / (a.reps + 3)
    assert rows_per_replay == 20 * E, rows_per_replay
    row_w = 4 * (2 * 5 * V + V * (V + 2) + 1 + V + V * V) + 1
    row_r = 4 * (2 * 5 * V + V * V + 2 * V + 1 + V) + V * V
    B = 4096
    idx = torch.randint(0, min(rb.mem_cntr, a.size), (B,), device=dev)
    us_s = timed(lambda: rb.sample_buffer(B, idx=idx))
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6549.4)
    except Exception:
        peak = 6549.4
    gbs = (row_w + row_r) * E / ((us_graph or us) * 1e-6) / 1e9
    print(json.dumps({"config": {"envs": E, "V": V, "mem_size": a.size}, "store_marl_us": us,
                      "store_marl_us_device_graph": us_graph,
                      "transitions_per_s": E / (us * 1e-6), "bytes_per_row": {"read": row_r, "written": row_w},
                      "achieved_GBps": gbs, "frac_of_hbm_peak": gbs / peak, "sample_4096_us": us_s,
                      "device_counter": {"store_marl_us": us_d, "store_marl_us_device_graph": us_d_graph,
                                         "rows_per_replay_of_20_stores": rows_per_replay}}))


if __name__ == "__main__":
    main()
