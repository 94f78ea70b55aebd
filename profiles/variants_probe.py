"""Per-env variants: what they cost and what a sweep gains (profiles/r8_notes.md).

  python profiles/variants_probe.py --parent-lib PATH/libssd_b200.so [--out FILE.jsonl]

Three measurements, all in one process on one GPU, CUDA graphs of `--steps` steps replayed and timed with CUDA events:
  * no regression: this build without variants against the parent commit's library (--parent-lib), alternating, on the bench
    workloads (Harvest / Cleanup default5 at 4 096 envs in 8 ranges and at 65 536 envs, Cleanup default10 at 16 384 envs in
    ranges of 2 048);
  * the cost of a mixed batch: the same workloads with 8 round-robin variants set;
  * what a sweep gains: one 4 096-env launch running 8 variants against 8 handles of 512 envs stepped one after another.
Every configuration is timed `--rounds` times, interleaved; the JSON lines carry every sample, so the spread of each
configuration is the run-to-run spread.  Observations are written (RGB), state images are not, as in bench.py.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = [  # name, env, map, agents, view, B, ranges
    ("harvest5_b4096", "harvest", "default5", 5, 15, 4096, 8),
    ("harvest5_b65536", "harvest", "default5", 5, 15, 65536, 1),
    ("cleanup5_b4096", "cleanup", "default5", 5, 7, 4096, 8),
    ("cleanup5_b65536", "cleanup", "default5", 5, 7, 65536, 1),
    ("cleanup10_b16384", "cleanup", "default10", 10, 7, 16384, 8),
]


def sweep(env_name):
    """8 variants of the dynamics the SSD papers sweep: Harvest regrowth, Cleanup depletion / restoration."""
    if env_name == "harvest":
        return [{"spawn_prob": [0.0, 0.005 * k, 0.02 * k, 0.05 * k]} for k in range(1, 9)]
    return [{"threshold_depletion": 0.4 + 0.07 * k, "apple_respawn_prob": 0.05 * k} for k in range(1, 9)]


class _Tolerant:
    """The parent's library lacks the variant entry points; the binding may configure them, nothing calls them."""

    def __init__(self, lib):
        self.__dict__["_lib"] = lib

    def __getattr__(self, k):
        try:
            return getattr(self._lib, k)
        except AttributeError:
            return types.SimpleNamespace()

    def __setattr__(self, k, v):
        setattr(self._lib, k, v)


def load_lib(path, tolerant):
    from homophily_marl_b200 import _capi
    _capi._lib, _capi.LIB_PATH = None, path
    if tolerant:
        real = C.CDLL
        C.CDLL = lambda p: _Tolerant(real(p))
        try:
            return _capi.load()
        finally:
            C.CDLL = real
    return _capi.load()


def make_env(lib, w, variants=None, B=None, gid_base=0, spec=None):
    """A handle of workload w: with `variants`, or created with the single config `spec` (a compiled variant), or plain."""
    from homophily_marl_b200 import _capi
    from homophily_marl_b200.batch_env import SSDBatchEnv
    _capi._lib = lib
    _, env, mp, n, view, B0, _ = w
    kw = {} if spec is None else dict(rows=spec.rows, params=spec.params, fire_cost=spec.fire_cost,
                                      hit_penalty=spec.hit_penalty)
    return SSDBatchEnv(env, B or B0, n, map=mp, view_size=view, episode_limit=100, seed=1, env_gid_base=gid_base,
                       extra_args=dict(random_spawn_point=True, random_spawn_rotation=None), variants=variants, **kw)


class Graph:
    """`steps` steps of `envs` (each as `ranges` step_range launches, one after another on one stream) in one CUDA graph."""

    def __init__(self, envs, ranges, steps):
        import torch
        self.torch, self.envs = torch, envs
        rs = np.random.RandomState(0)
        self.acts = [torch.as_tensor(rs.randint(0, e.n_actions, size=(steps, e.B, e.n)).astype(np.uint8), device=e.device)
                     for e in envs]
        self.stream = torch.cuda.Stream(device=envs[0].device)

        def body():
            for t in range(steps):
                for e, a in zip(envs, self.acts):
                    per = e.B // ranges
                    for r in range(ranges):
                        e.step_range(a[t], r * per, per)

        for e in envs:
            e.reset()
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            body()                                              # warm-up
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=self.stream):
                body()
        self.stream.synchronize()
        self.steps = steps

    def time_ms_per_step(self, replays):
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(self.stream):
            self.graph.replay()
            e0.record(self.stream)
            for _ in range(replays):
                self.graph.replay()
            e1.record(self.stream)
        e1.synchronize()
        return e0.elapsed_time(e1) / (replays * self.steps)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return out.strip().splitlines()[0] if out.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--replays", type=int, default=10)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    from homophily_marl_b200 import _capi
    this_lib = os.path.join(ROOT, "homophily_marl_b200", "libssd_b200.so")
    parent, this = load_lib(a.parent_lib, True), load_lib(this_lib, False)
    card = gpu_info()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        rec["gpu"] = card
        if out is not None:
            out.write(json.dumps(rec) + "\n")
            out.flush()
        print(json.dumps(rec), flush=True)

    for w in WORKLOADS:
        name, env_name, B, ranges = w[0], w[1], w[5], w[6]
        graphs = {"parent": Graph([make_env(parent, w)], ranges, a.steps),
                  "this": Graph([make_env(this, w)], ranges, a.steps),
                  "this_8_variants": Graph([make_env(this, w, sweep(env_name))], ranges, a.steps)}
        samples = {k: [] for k in graphs}
        for r in range(a.rounds):
            order = list(graphs) if r % 2 == 0 else list(graphs)[::-1]
            for k in order:
                samples[k].append(graphs[k].time_ms_per_step(a.replays) * 1e3)
        for k, v in samples.items():
            emit(dict(what="step", workload=name, B=B, ranges=ranges, config=k, us_per_step_median=float(np.median(v)),
                      us_min=float(np.min(v)), us_max=float(np.max(v)), samples=[round(x, 3) for x in v]))
        for g in graphs.values():
            for e in g.envs:
                e.close()
        torch.cuda.synchronize()

    for w in (WORKLOADS[0], WORKLOADS[2]):                       # a sweep of 8 settings: one mixed launch vs 8 handles
        name, env_name = w[0], w[1]
        one = Graph([make_env(this, w, sweep(env_name), B=4096)], 1, a.steps)
        specs = one.envs[0].variant_specs                       # each of the 8 handles is created with one setting, no variants
        eight = Graph([make_env(this, w, B=512, gid_base=512 * k, spec=s) for k, s in enumerate(specs)], 1, a.steps)
        samples = {"one_launch_8_variants": [], "eight_handles_512": []}
        for r in range(a.rounds):
            samples["one_launch_8_variants"].append(one.time_ms_per_step(a.replays) * 1e3)
            samples["eight_handles_512"].append(eight.time_ms_per_step(a.replays) * 1e3)
        for k, v in samples.items():
            emit(dict(what="sweep", workload=name.replace("_b4096", ""), B=4096, config=k,
                      us_per_step_median=float(np.median(v)), us_min=float(np.min(v)), us_max=float(np.max(v)),
                      samples=[round(x, 3) for x in v]))
        for g in (one, eight):
            for e in g.envs:
                e.close()
    _capi._lib = this
    if out is not None:
        out.close()


if __name__ == "__main__":
    main()
