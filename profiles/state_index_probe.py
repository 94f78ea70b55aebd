"""Cost of a step that also writes the state image (``want_state``), with an RGB state image and with a packed colour-index
state image (state_format "index4"), under both observation formats, same process, alternating.

Workloads: Cleanup default3 / default5 / default10 (view 7) and Harvest default5 (view 15), each at 4 096 envs as 8 env ranges
on 8 streams (programmatic launch) and at 65 536 envs (one launch per step).  Actions are uniform over the movement actions.
Each of the four (obs_format, state_format) variants is a CUDA graph of K steps writing into rings of observation buffers and
of state buffers, each ring larger than the 126 MB L2; replays are timed with CUDA events and the variants alternate replay by
replay (the order reverses every round).  One JSON line per (workload, obs_format, state_format) with us/step, the bytes the
step writes per env for observations and for the state image, the card name and its power limit.

    python profiles/state_index_probe.py [--out FILE.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [(f"{env}{n}_b{B}" + (f"_g{g}" if g > 1 else ""), env, f"default{n}", n, view, B, g)
             for env, n, view in (("cleanup", 3, 7), ("cleanup", 5, 7), ("cleanup", 10, 7), ("harvest", 5, 15))
             for B, g in ((4096, 8), (65536, 1))]                    # name, env, map, agents, view, envs, ranges
VARIANTS = [(o, s) for o in ("rgb", "index4") for s in ("rgb", "index4")]
RING_BYTES = 256 << 20                                                # > 126 MB of L2


class Variant:
    def __init__(self, env_name, mp, n, view, B, groups, obs, state, K, seed=1):
        dev = torch.device("cuda:0")
        self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=10 ** 9, seed=seed, device=dev,
                               extra_args=dict(obs_format=obs, state_format=state), want_state=True)
        self.obs, self.state, self.K, self.groups = obs, state, K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, 5, (K, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        e = self.env
        self.obs_ring = [e.new_obs_buffer() for _ in range(max(2, math.ceil(RING_BYTES / (B * e.obs_layout.env_stride))))]
        self.state_ring = [torch.zeros_like(e.state_buf)
                           for _ in range(max(2, math.ceil(RING_BYTES / (B * e.state_layout.env_stride))))]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
        e.reset()
        torch.cuda.synchronize()

    def _step(self, t, lo=None, cnt=None):
        e = self.env
        e.state_buf = self.state_ring[t % len(self.state_ring)]     # the step writes the state image into state_buf
        if lo is None:
            e.step(self.actions[t], obs_out=self.obs_ring[t % len(self.obs_ring)], want_state=True)
        else:
            e.step_range(self.actions[t], lo, cnt, obs_out=self.obs_ring[t % len(self.obs_ring)], want_state=True)

    def run(self):
        """Enqueues K steps on the current stream (forked into the env ranges)."""
        main = torch.cuda.current_stream()
        Bg = self.env.B // self.groups
        if self.groups == 1:
            for t in range(self.K):
                self._step(t)
            return
        for gi, gs in enumerate(self.gstreams):
            gs.wait_stream(main)
            with torch.cuda.stream(gs):
                for t in range(self.K):
                    self._step(t, gi * Bg, Bg)
        for gs in self.gstreams:
            main.wait_stream(gs)

    def capture(self):
        with torch.cuda.stream(self.stream):
            self.run()                                         # warm-up, eager
        self.stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            self.run()


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                     # noqa: BLE001
        pl = f"unknown ({e})"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=300, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=10, help="timed replays per variant")
    ap.add_argument("--only", default=None, help="comma-separated workload names (default: all)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("state_index_probe needs a CUDA device")
    name, power = card()
    lines = []
    only = set(a.only.split(",")) if a.only else None
    for wname, env_name, mp, n, view, B, groups in WORKLOADS:
        if only and wname not in only:
            continue
        vs = [Variant(env_name, mp, n, view, B, groups, o, s, a.steps) for o, s in VARIANTS]
        for v in vs:
            v.capture()
        times = {id(v): [] for v in vs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (vs if r % 2 == 0 else vs[::-1]):
                with torch.cuda.stream(v.stream):
                    ev[0].record()
                    v.graph.replay()
                    ev[1].record()
                v.stream.synchronize()
                if r >= 2:
                    times[id(v)].append(ev[0].elapsed_time(ev[1]) * 1e3 / a.steps)
        for v in vs:
            ts = sorted(times[id(v)])
            rec = dict(probe="state_index_probe", workload=wname, envs=B, env_ranges=groups, obs_format=v.obs,
                       state_format=v.state, replays=len(ts), steps_per_replay=a.steps, us_per_step_median=ts[len(ts) // 2],
                       us_per_step_min=ts[0], us_per_step_max=ts[-1], obs_bytes_per_env=v.env.obs_layout.env_stride,
                       state_bytes_per_env=v.env.state_layout.env_stride, obs_ring=len(v.obs_ring),
                       state_ring=len(v.state_ring), timing="cuda_graph_events", gpu=name, power_limit=power)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        for v in vs:
            v.graph = None
            v.env.close()
        del vs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
