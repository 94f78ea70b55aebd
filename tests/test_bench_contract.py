"""bench.py prints ONE JSON line with the contract's keys (CPU arm here; CUDA arm under -m gpu)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def _run(args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                       env={**os.environ, **(env or {})}, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    return lines


def test_reference_arm_line():
    lines = _run(["--impl", "reference", "--steps", "30", "--warmup", "1", "--workload", "cleanup3_b4096", "--envs", "64", "--no-train"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "agent-steps/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["cpu_baseline_port"]["kind"] == "port" and d["cpu_baseline_port"]["value"] > 0
    from baseline import refloop
    assert d["cpu_baseline"]["kind"] == ("reference" if refloop.available() else "port")
    assert set(d["config"]) == {"workload", "env", "map", "num_agents", "view_size", "envs_per_gpu", "global_envs", "episode_limit",
                                "actions", "extra_args", "obs_color", "obs_format"}
    assert d["e2e"] == {"value": d["value"], "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["dtype"] == "u8" and d["data"] == "synthetic"


def test_reference_arm_other_ranks_exit_quietly():
    assert _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--envs", "64"], env={"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_reference_arm_times_the_reference_training_loop():
    from baseline import refloop
    if not refloop.available():
        pytest.skip("reference sources absent")
    d = json.loads(_run(["--impl", "reference", "--steps", "10", "--warmup", "1", "--workload", "cleanup3_b4096", "--train-t-max", "150"])[0])
    t = d["train_e2e"]
    assert t["unit"] == "env-steps/s" and t["reference"]["env_steps"] == 200 and t["reference"]["value"] > 0


@pytest.mark.gpu
def test_cuda_arm_line():
    lines = _run(["--steps", "5000", "--warmup", "20", "--envs", "512", "--e2e-steps", "5", "--no-extra", "--no-train"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS | {"clocks", "gpu_launches", "roofline"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 5000 and d["scaling"] == "weak" and d["dtype"] == "u8"
    assert d["gpu_launches"] >= 5000
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 512 * 5 and e["d2h_bytes_per_step"] > 512 * 5 * 3 * 31 * 31 and 0 < e["value"] < d["value"]
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] > 0
    assert d["replays"] >= 5 and d["replay_ms"]["min"] <= d["replay_ms"]["median"] <= d["replay_ms"]["max"]
    assert "l2" not in d["config"] and "parallelism" not in d["config"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs: what the last timed step returned, float32, identical in two runs with the same arguments and with
    graphs + 8 env ranges or a Python loop + one launch per step, and equal to an oracle rollout of sampled envs with the
    same seed and actions for the same number of steps.  The launch counter of the Python-loop run pins the timed steps."""
    import numpy as np
    import torch
    from homophily_marl_b200 import mapspec
    from oracle import oracle as O
    B, K, W = 512, 250, 7
    args = ["--steps", str(K), "--replays", "2", "--warmup", str(W), "--envs", str(B), "--e2e-steps", "1", "--no-extra",
            "--no-train", "--no-cpu-baseline"]
    lines, dumps = [], []
    for k, more in enumerate(([], [], ["--no-graph", "--groups", "1"])):
        out = tmp_path / str(k)
        d = json.loads(_run(args + more + ["--dump-outputs", str(out)])[0])
        assert d["steps"] == K and d["timed_steps"] == K and d["replays"] == 2
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 * 10 ** 6
        lines.append(d)
        dumps.append({f.stem: np.load(f) for f in out.iterdir()})
    a = dumps[0]
    assert set(a) == {"reward", "clean", "apple_cnt", "done", "obs", "envs", "obs_envs"}
    for b in dumps[1:]:
        for k in a:
            assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    T = lines[0]["env_steps"]
    assert T == lines[2]["env_steps"] and T >= W + K
    assert lines[2]["gpu_launches"] == K + sum(t % 100 == 0 for t in range(T - K, T))       # one step launch + resets
    assert a["reward"].shape == (B, 5) and a["done"].shape == (B,) and np.array_equal(a["envs"], np.arange(B))
    assert a["obs"].shape == (256, 5, 3, 31, 31) and len(np.unique(a["obs_envs"])) == 256

    spec = mapspec.compile_map("harvest", "default5", 5, 15, 100, obs_color="simplified")
    g = torch.Generator(device="cuda").manual_seed(0)                                         # bench.py DeviceRollout, seed 0
    acts = torch.randint(0, spec.n_actions, (100, B, 5), generator=g, device="cuda", dtype=torch.int32).to(torch.uint8).cpu().numpy()
    for j in (0, 101, 255):
        e = int(a["obs_envs"][j])
        ob = O.OracleBatch.from_spec(spec, n_envs=1, seed=0, env_gid0=e, random_spawn_point=False, spawn_rotation=0)
        for t in range(T):
            if t % 100 == 0:
                ob.reset()
            o = ob.step(acts[t % 100, e:e + 1])
        assert np.array_equal(a["obs"][j], o["obs"][0]), e
        assert np.array_equal(a["reward"][e], o["reward"][0]) and np.array_equal(a["clean"][e], o["clean"][0]), e
        assert a["apple_cnt"][e] == o["apple_cnt"][0] and a["done"][e] == o["done"][0], e


def test_timed_steps_are_the_steps_argument():
    """--steps K times exactly K steps, split into replays of near-equal length."""
    bench = _bench_module()
    for K in (1, 7, 99, 100, 250, 20000, 20001):
        for R in (1, 3, 20, 200):
            lens = bench.replay_lengths(K, R)
            assert sum(lens) == K and len(lens) == min(R, K) and max(lens) - min(lens) <= 1
    auto = lambda K: bench.auto_replays(type("A", (), {"replays": 0}), K)  # noqa: E731
    assert [auto(K) for K in (1, 999, 2000, 5500, 20000, 50000)] == [1, 1, 2, 5, 20, 20]


def test_env_range_rule():
    """Small batches are stepped as env ranges (profiles/r2_notes.md sections 2-3); every range size must divide the batch."""
    bench = _bench_module()
    assert [bench.auto_groups(b) for b in (512, 2048, 4096, 8192, 16384, 65536, 4095, 10000)] == [8, 8, 8, 4, 8, 1, 1, 1]
    for b in (512, 2048, 4096, 8192, 16384):
        assert b % bench.auto_groups(b) == 0
