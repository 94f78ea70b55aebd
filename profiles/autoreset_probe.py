"""Cost of auto-reset: a step without any reset (the lower bound), the three-launch path ``step`` + masked ``ssd_reset`` +
``ssd_render`` of the state image (whole batch only: env ranges have no reset of their own), and ``ssd_step_autoreset``
(auto-reset in the step launch), same process, alternating.

Workloads: Harvest default5 (view 15), Cleanup default5 and default10 (view 7), each at 4 096 envs as 8 env ranges on 8 streams
(programmatic launch; the three-launch variant steps the 4 096 envs as one batch) and at 65 536 envs (one launch per step), with
RGB and index4 observations, with and without the state image (in the observation's format).  Episode clocks are staggered
(t0 = env % 100, episode_limit 100), so about 1 % of the envs end their episode in each step.  Actions are uniform over the
movement actions.  Each variant is a CUDA graph of K steps writing into rings of observation and state buffers larger than
the 126 MB L2; replays are timed with CUDA events and the variants alternate replay by replay (the order reverses every
round).  One JSON line per (workload, variant) with us/step (median, min, max), the card name and its power limit.

    python profiles/autoreset_probe.py [--out FILE.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [(f"{env}{n}_b{B}" + (f"_g{g}" if g > 1 else "") + f"_{obs}" + ("_state" if st else ""), env, f"default{n}", n, view,
              B, g, obs, st)
             for env, n, view in (("harvest", 5, 15), ("cleanup", 5, 7), ("cleanup", 10, 7))
             for B, g in ((4096, 8), (65536, 1)) for obs in ("rgb", "index4") for st in (False, True)]
VARIANTS = ("step", "sequence", "fused")
RING_BYTES = 256 << 20                                                # > 126 MB of L2
LIMIT = 100


class Variant:
    def __init__(self, env_name, mp, n, view, B, groups, obs, want_state, mode, K, seed=1):
        dev = torch.device("cuda:0")
        self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=LIMIT, seed=seed, device=dev,
                               extra_args=dict(obs_format=obs, state_format=obs), want_state=True)
        self.mode, self.want_state, self.K = mode, want_state, K
        self.groups = 1 if mode == "sequence" else groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, 5, (K, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        e = self.env
        self.obs_ring = [e.new_obs_buffer() for _ in range(max(2, math.ceil(RING_BYTES / (B * e.obs_layout.env_stride))))]
        self.state_ring = [torch.zeros_like(e.state_buf)
                           for _ in range(max(2, math.ceil(RING_BYTES / (B * e.state_layout.env_stride))))]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
        e.reset()
        e.load_state(t=np.arange(B, dtype=np.int32) % LIMIT)
        torch.cuda.synchronize()

    def _step(self, t, lo=None, cnt=None):
        e = self.env
        e.state_buf = self.state_ring[t % len(self.state_ring)]     # the step writes the state image into state_buf
        obs, ws = self.obs_ring[t % len(self.obs_ring)], self.want_state
        if self.mode == "sequence":                                # the three-launch path
            e.step(self.actions[t], obs_out=obs, want_state=ws)
            e.reset(mask=e.done, obs_out=obs)
            if ws:
                e.render(want_obs=False, want_state=True)
        elif lo is None:
            e.step(self.actions[t], obs_out=obs, want_state=ws, auto_reset=self.mode == "fused")
        else:
            e.step_range(self.actions[t], lo, cnt, obs_out=obs, want_state=ws, auto_reset=self.mode == "fused")

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
        before = self.env.launch_count
        with torch.cuda.stream(self.stream):
            self.run()                                         # warm-up, eager
        self.stream.synchronize()
        self.launches = (self.env.launch_count - before) / self.K
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
    ap.add_argument("--steps", type=int, default=200, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=8, help="timed replays per variant")
    ap.add_argument("--only", default=None, help="comma-separated workload names (default: all)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autoreset_probe needs a CUDA device")
    name, power = card()
    lines = []
    only = set(a.only.split(",")) if a.only else None
    for wname, env_name, mp, n, view, B, groups, obs, st in WORKLOADS:
        if only and wname not in only:
            continue
        vs = [Variant(env_name, mp, n, view, B, groups, obs, st, m, a.steps) for m in VARIANTS]
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
            rec = dict(probe="autoreset_probe", workload=wname, variant=v.mode, envs=B, env_ranges=v.groups, obs_format=obs,
                       want_state=st, replays=len(ts), steps_per_replay=a.steps, us_per_step_median=ts[len(ts) // 2],
                       us_per_step_min=ts[0], us_per_step_max=ts[-1], episode_limit=LIMIT,
                       launches_per_step=v.launches, obs_ring=len(v.obs_ring), state_ring=len(v.state_ring),
                       timing="cuda_graph_events", gpu=name, power_limit=power)
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
