"""bench.py: the reference arm prints ONE JSON line with the contract's keys (no GPU needed); the CUDA arm's
--dump-outputs files (GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-500:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    # "reference" = the unmodified Environ classes (mounted tree or the staged baseline/_ref), "port" = the oracle
    assert d["cpu_baseline"]["kind"] in ("port", "reference")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_our_arm_refuses_to_run_without_gpu():
    import torch

    if torch.cuda.is_available():
        return
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode != 0          # no CPU fallback: the product arm fails loudly
    assert "{\"metric\"" not in res.stdout


def test_dump_sample_is_one_seeded_env_subset_for_every_trace():
    """Traces over the --dump-outputs budget: every trace keeps the same fixed, seeded, sorted subset of env indices,
    as many envs as fit the budget."""
    import numpy as np
    import torch

    import bench

    T, E, V = 64, 8192, 8
    env_id = torch.arange(E, dtype=torch.float32)
    out = {k: (env_id.expand(T, E) if k == "reward" else env_id[:, None].expand(E, V).expand(T, E, V)).contiguous()
           for k in bench.SARL_TRACE_NAMES}
    got = bench.sample_traces(torch, out, E)
    n = bench.DUMP_BYTES // (T * (6 * V + 1) * 4)
    assert n < E
    idx = got["reward"][0]
    assert idx.shape == (n,) and np.all(np.diff(idx) > 0)
    for k, a in got.items():
        assert a.dtype == np.float32 and a.shape[:2] == (T, n), k
        assert np.array_equal(a, idx[None, :, None].repeat(T, 0).repeat(V, 2) if a.ndim == 3 else idx[None].repeat(T, 0)), k
    assert sum(a.nbytes for a in got.values()) <= bench.DUMP_BYTES
    assert np.array_equal(bench.sample_traces(torch, out, E)["rate"], got["rate"])


@pytest.mark.gpu
@pytest.mark.parametrize("workload,envs", [("sarl", 4096), ("marl", 300)])
def test_dump_outputs_are_reproducible(workload, envs, tmp_path):
    """Two runs with the same arguments dump the same traces of the last timed rollout (float32, within the size
    budget), however long the clock sampler's spin before the timed region lasted; the dumped reward is the one the
    run's statistics summed (one timed rollout: mean_reward_last_steps = the mean reward of its last step)."""
    import numpy as np

    def run(name):
        d = tmp_path / name
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--envs", str(envs),
                              "--T", "64", "--steps", "1", "--warmup", "3", "--e2e-steps", "1", "--no-secondary",
                              "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 1
        return {p.stem: np.load(p) for p in sorted(d.glob("*.npy"))}, line["mean_reward_last_steps"]

    (a, mean_reward), (b, _) = run("a"), run("b")
    names = {"sarl": {"reward", "DataBuf", "data_t", "data_p", "over_power", "over_data", "rate"},
             "marl": {"reward_user", "reward", "data_t", "data_p", "rate", "DataBuf"}}[workload]
    assert set(a) == set(b) == names
    assert sum(v.nbytes for v in a.values()) <= 64_000_000
    for k in names:
        assert a[k].dtype == np.float32 and a[k].shape[:2] == (64, envs) and np.isfinite(a[k]).all(), k
        assert np.array_equal(a[k], b[k]), k
    last = a["reward"][-1].astype(np.float64).mean()
    assert abs(last - mean_reward) <= 1e-6 * abs(mean_reward) + 1e-9, (last, mean_reward)
    assert np.ptp(a["DataBuf"][-1]) > 0
