"""Cost of the shaped rewards (extra_args reward_shaping): time per step with shaping off and on, same process, alternating.

Workloads: Harvest default5 at 4 096 envs in 8 env ranges of 512 on 8 streams (programmatic dependent launch, where one more
launch per step costs the most) and at 65 536 envs, and Cleanup default5 at 65 536 envs (one launch per step); RGB observations,
tag_timeout 0, uniform random actions over every action.  Shaping on uses Hughes' Cleanup weights with some prosocial mixing
(alpha 5, beta 0.05, decay 0.99 * 0.975, prosocial 0.25).  Each variant is a CUDA graph of K steps writing into a ring of
observation buffers (no state image, as in bench.py); replays are timed with CUDA events and off / on alternate replay by replay
after two warm-up rounds.  The 4 096-env workload is also timed eagerly (every step launched from Python, host-synchronised per
replay), where the extra launch adds host launch overhead too.  One JSON line per (workload, mode, shaping), with the card name and
power limit read in the same run.

    python profiles/shaping_probe.py [--out FILE.jsonl] [--steps K] [--replays R]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 5, 15, 4096, 8, 4),      # name, env, map, n, view, envs, ranges, ring
             ("harvest5_b65536", "harvest", "default5", 5, 15, 65536, 1, 2),
             ("cleanup5_b65536", "cleanup", "default5", 5, 7, 65536, 1, 2)]
SHAPING = {"alpha": 5.0, "beta": 0.05, "prosocial": 0.25}


class Variant:
    def __init__(self, wl, shaping, K, seed=1):
        _, env_name, mp, n, view, B, groups, ring = wl
        dev = torch.device("cuda:0")
        self.shaping = shaping
        self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=10 ** 4, seed=seed, device=dev,
                               extra_args=dict(disable_fire_action=False, disable_rotation_action=False,
                                               reward_shaping=SHAPING if shaping else None))
        self.K, self.groups = K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, self.env.n_actions, (K, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        self.ring = [self.env.new_obs_buffer() for _ in range(ring)]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
        self.env.reset()
        torch.cuda.synchronize()

    def run(self):
        """Enqueues K steps on the current stream (forked into the env ranges)."""
        env, main = self.env, torch.cuda.current_stream()
        Bg = env.B // self.groups
        for gi, gs in enumerate(self.gstreams):
            gs.wait_stream(main)
            with torch.cuda.stream(gs):
                for t in range(self.K):
                    env.step_range(self.actions[t], gi * Bg, Bg, obs_out=self.ring[t % len(self.ring)])
        for gs in self.gstreams:
            main.wait_stream(gs)

    def capture(self):
        with torch.cuda.stream(self.stream):
            self.run()                                         # warm-up, eager
        self.stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            self.run()

    def time_graph(self, ev):
        with torch.cuda.stream(self.stream):
            ev[0].record()
            self.graph.replay()
            ev[1].record()
        self.stream.synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e3 / self.K

    def time_eager(self, ev):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.cuda.stream(self.stream):
            self.run()
        self.stream.synchronize()
        return (time.perf_counter() - t0) * 1e6 / self.K


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                     # noqa: BLE001
        q = f"unknown ({e})"
    return torch.cuda.get_device_name(0), q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=200, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=10, help="timed replays per variant")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shaping_probe needs a CUDA device")
    name, smi = card()
    cases = [(wl, "graph") for wl in WORKLOADS] + [(WORKLOADS[0], "eager")]
    lines = []
    for wl, mode in cases:
        vs = [Variant(wl, shaping, a.steps) for shaping in (False, True)]
        for v in vs:
            v.capture()
        times = {v.shaping: [] for v in vs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (vs if r % 2 == 0 else vs[::-1]):
                dt = v.time_graph(ev) if mode == "graph" else v.time_eager(ev)
                if r >= 2:
                    times[v.shaping].append(dt)
        med = {}
        for v in vs:
            ts = sorted(times[v.shaping])
            med[v.shaping] = ts[len(ts) // 2]
            rec = dict(probe="shaping_probe", workload=wl[0], envs=wl[5], env_ranges=wl[6], mode=mode, reward_shaping=v.shaping,
                       steps_per_replay=a.steps, replays=len(ts), us_per_step_median=ts[len(ts) // 2], us_per_step_min=ts[0],
                       us_per_step_max=ts[-1], launches_per_step_per_range=2 if v.shaping else 1, gpu=name,
                       nvidia_smi_name_power_limit_max_sm_clock=smi)
            if v.shaping:
                rec["on_over_off"] = med[True] / med[False]
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        for v in vs:
            v.graph = None
            v.env.close()
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
