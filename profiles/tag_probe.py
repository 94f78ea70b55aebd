"""Cost of tagging-out timers: time per step with tag_timeout 0 (the reference) and 25, same process, alternating.

Workloads: the headline (Harvest default5, 4 096 envs as 8 env ranges on 8 streams, programmatic launch) and Cleanup default5 at
65 536 envs (one launch per step).  Actions are uniform over every action, FIRE included, so agents do get tagged.  Each
variant is a CUDA graph of K steps writing into a ring of observation buffers; replays are timed with CUDA events and the
variants alternate replay by replay.  The fraction of agent-steps spent out of play is counted in an untimed eager run of the
same schedule.  One JSON line per (workload, tag_timeout), with the card name and power limit.

    python profiles/tag_probe.py [--out FILE.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 15, 4096, 8, 4),
             ("cleanup5_b65536", "cleanup", "default5", 7, 65536, 1, 2)]      # name, env, map, view, envs, ranges, ring


class Variant:
    def __init__(self, env_name, mp, view, B, groups, ring, T, K, seed=1):
        dev = torch.device("cuda:0")
        self.env = SSDBatchEnv(env_name, B, 5, map=mp, view_size=view, episode_limit=10 ** 9, seed=seed, device=dev,
                               extra_args=dict(tag_timeout=T, disable_fire_action=False, disable_rotation_action=False))
        self.T, self.K, self.groups = T, K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, self.env.n_actions, (K, B, 5), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
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

    def out_fraction(self, steps):
        env, n = self.env, self.env.n
        out = torch.zeros((), dtype=torch.int64, device=env.device)
        for t in range(steps):
            env.step(self.actions[t % self.K], obs_out=self.ring[0])
            out += ((env.agent_buf[:, :n] >> 24) != 0).sum()
        return int(out) / (steps * env.B * n)


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
    ap.add_argument("--steps", type=int, default=500, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=12, help="timed replays per variant")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tag_probe needs a CUDA device")
    name, power = card()
    lines = []
    for wname, env_name, mp, view, B, groups, ring in WORKLOADS:
        vs = [Variant(env_name, mp, view, B, groups, ring, T, a.steps) for T in (0, 25)]
        for v in vs:
            v.capture()
        times = {v.T: [] for v in vs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (vs if r % 2 == 0 else vs[::-1]):
                with torch.cuda.stream(v.stream):
                    ev[0].record()
                    v.graph.replay()
                    ev[1].record()
                v.stream.synchronize()
                if r >= 2:
                    times[v.T].append(ev[0].elapsed_time(ev[1]) * 1e3 / a.steps)
        for v in vs:
            ts = sorted(times[v.T])
            rec = dict(probe="tag_probe", workload=wname, envs=B, env_ranges=groups, tag_timeout=v.T, steps_per_replay=a.steps,
                       replays=len(ts), us_per_step_median=ts[len(ts) // 2], us_per_step_min=ts[0], us_per_step_max=ts[-1],
                       out_fraction=v.out_fraction(300), gpu=name, power_limit=power)
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
