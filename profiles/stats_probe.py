"""Cost of the per-agent episode counters (extra_args episode_stats): time per step with counters off and on, same process,
alternating.

Workloads: Harvest default5 at 4 096 envs (8 env ranges on 8 streams, programmatic launch) and at 65 536 envs, Cleanup default5
at 65 536 envs and Cleanup default10 at 16 384 envs (one launch per step); each with RGB and index4 observations, tag_timeout 0
and 25, and uniform random actions over every action (FIRE and CLEAN included).  Two extra rows per Harvest / Cleanup default5
workload use FIRE-heavy actions (half of all actions FIRE, tag_timeout 0, RGB), where the counting kernels walk every FIRE ray
that the reference-default kernels skip while hit_penalty is 0.  Each variant is a CUDA graph of K steps writing into a ring of
observation buffers (no state image, as in bench.py); replays are timed with CUDA events and off / on alternate replay by replay
after two warm-up rounds.  One JSON line per (workload, obs format, tag_timeout, actions), with the card name and power limit
read in the same run.

    python profiles/stats_probe.py [--out FILE.jsonl] [--steps K] [--replays R]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 5, 15, 4096, 8, 4),      # name, env, map, n, view, envs, ranges, ring
             ("harvest5_b65536", "harvest", "default5", 5, 15, 65536, 1, 2),
             ("cleanup5_b65536", "cleanup", "default5", 5, 7, 65536, 1, 2),
             ("cleanup10_b16384", "cleanup", "default10", 10, 7, 16384, 1, 2)]
FIRE = 7


class Variant:
    def __init__(self, wl, obs, T, fire_share, stats, K, seed=1):
        _, env_name, mp, n, view, B, groups, ring = wl
        dev = torch.device("cuda:0")
        self.stats = stats
        self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=10 ** 4, seed=seed, device=dev,
                               extra_args=dict(tag_timeout=T, disable_fire_action=False, disable_rotation_action=False,
                                               obs_format=obs, episode_stats=stats))
        self.K, self.groups = K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        a = torch.randint(0, self.env.n_actions, (K, B, n), generator=g, device=dev, dtype=torch.int32)
        if fire_share:
            a = torch.where(torch.rand((K, B, n), generator=g, device=dev) < fire_share, FIRE, a)
        self.actions = a.to(torch.uint8)
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
        raise SystemExit("stats_probe needs a CUDA device")
    name, smi = card()
    cases = [(wl, obs, T, 0.0) for wl in WORKLOADS for obs in ("rgb", "index4") for T in (0, 25)]
    cases += [(wl, "rgb", 0, 0.5) for wl in WORKLOADS[:3]]
    lines = []
    for wl, obs, T, fire in cases:
        vs = [Variant(wl, obs, T, fire, stats, a.steps) for stats in (False, True)]
        for v in vs:
            v.capture()
        times = {v.stats: [] for v in vs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (vs if r % 2 == 0 else vs[::-1]):
                with torch.cuda.stream(v.stream):
                    ev[0].record()
                    v.graph.replay()
                    ev[1].record()
                v.stream.synchronize()
                if r >= 2:
                    times[v.stats].append(ev[0].elapsed_time(ev[1]) * 1e3 / a.steps)
        med = {}
        for v in vs:
            ts = sorted(times[v.stats])
            med[v.stats] = ts[len(ts) // 2]
            rec = dict(probe="stats_probe", workload=wl[0], envs=wl[5], env_ranges=wl[6], obs_format=obs, tag_timeout=T,
                       fire_share=fire or "uniform", episode_stats=v.stats, steps_per_replay=a.steps, replays=len(ts),
                       us_per_step_median=ts[len(ts) // 2], us_per_step_min=ts[0], us_per_step_max=ts[-1], gpu=name,
                       nvidia_smi_name_power_limit_max_sm_clock=smi)
            if v.stats:
                rec["on_over_off"] = med[True] / med[False]
                rec["apples_fires_hits_per_env_step"] = [
                    round(float(x), 4) for x in v.env.stats().to(torch.float64).sum((0, 2))[[0, 2, 3]] / (v.env.B * int(v.env.t_buf[0]))]
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
