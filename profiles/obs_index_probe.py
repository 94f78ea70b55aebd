"""Cost of a step with RGB observations and with packed colour-index observations (obs_format "index4"), same process,
alternating.

Workloads: Harvest default5 and Cleanup default5, each at 4 096 envs as 8 env ranges on 8 streams (programmatic launch) and at
65 536 envs (one launch per step); plus ``step_host`` (actions up, step, every output and the observations down, stream sync)
for Harvest default5 at 4 096 envs.  Actions are uniform over the movement actions.  Each graph variant is a CUDA graph of K
steps writing into a ring of observation buffers larger than the 126 MB L2; replays are timed with CUDA events and the
variants alternate replay by replay.  ``step_host`` cannot be captured: it is timed with the host clock over calls that each
end in a stream synchronise.  One JSON line per (workload, format) with us/step, algorithmic bytes per env-step, achieved
GB/s, the card name and its power limit.

    python profiles/obs_index_probe.py [--out FILE.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402

WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 15, 4096, 8),
             ("harvest5_b65536", "harvest", "default5", 15, 65536, 1),
             ("cleanup5_b4096_g8", "cleanup", "default5", 7, 4096, 8),
             ("cleanup5_b65536", "cleanup", "default5", 7, 65536, 1)]      # name, env, map, view, envs, ranges
RING_BYTES = 256 << 20                                                      # > 126 MB of L2


class Variant:
    def __init__(self, env_name, mp, view, B, groups, fmt, K, seed=1):
        dev = torch.device("cuda:0")
        self.env = SSDBatchEnv(env_name, B, 5, map=mp, view_size=view, episode_limit=10 ** 9, seed=seed, device=dev,
                               extra_args=dict(obs_format=fmt))
        self.fmt, self.K, self.groups = fmt, K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, 5, (K, B, 5), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        buf_bytes = B * self.env.obs_layout.env_stride
        self.ring = [self.env.new_obs_buffer() for _ in range(max(2, math.ceil(RING_BYTES / buf_bytes)))]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
        self.env.reset()
        torch.cuda.synchronize()

    def run(self):
        """Enqueues K steps on the current stream (forked into the env ranges)."""
        env, main = self.env, torch.cuda.current_stream()
        Bg = env.B // self.groups
        if self.groups == 1:
            for t in range(self.K):
                env.step(self.actions[t], obs_out=self.ring[t % len(self.ring)])
            return
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
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                     # noqa: BLE001
        pl = f"unknown ({e})"
    return name, pl


def record(wname, v, B, groups, ts, **extra):
    ts = sorted(ts)
    med = ts[len(ts) // 2]
    nbytes = v.env.bytes_per_env_step()
    return dict(probe="obs_index_probe", workload=wname, envs=B, env_ranges=groups, obs_format=v.fmt, replays=len(ts),
                us_per_step_median=med, us_per_step_min=ts[0], us_per_step_max=ts[-1], bytes_per_env_step=nbytes,
                achieved_GBps=nbytes * B / (med * 1e-6) / 1e9, **extra)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=500, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=12, help="timed replays per variant")
    ap.add_argument("--host-steps", type=int, default=300, help="timed step_host calls per round")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("obs_index_probe needs a CUDA device")
    name, power = card()
    lines = []

    def emit(rec):
        rec.update(gpu=name, power_limit=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    for wname, env_name, mp, view, B, groups in WORKLOADS:
        vs = [Variant(env_name, mp, view, B, groups, fmt, a.steps) for fmt in ("rgb", "index4")]
        for v in vs:
            v.capture()
        times = {v.fmt: [] for v in vs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (vs if r % 2 == 0 else vs[::-1]):
                with torch.cuda.stream(v.stream):
                    ev[0].record()
                    v.graph.replay()
                    ev[1].record()
                v.stream.synchronize()
                if r >= 2:
                    times[v.fmt].append(ev[0].elapsed_time(ev[1]) * 1e3 / a.steps)
        for v in vs:
            emit(record(wname, v, B, groups, times[v.fmt], steps_per_replay=a.steps, ring=len(v.ring), timing="cuda_graph_events"))
        for v in vs:
            v.graph = None
            v.env.close()
        torch.cuda.empty_cache()

    # step_host: host buffers in and out, one stream synchronise per call
    B = 4096
    vs = [Variant("harvest", "default5", 15, B, 1, fmt, 1) for fmt in ("rgb", "index4")]
    ios = {v.fmt: v.env.make_host_io(with_obs=True) for v in vs}
    times = {v.fmt: [] for v in vs}
    for r in range(a.replays + 2):
        for v in (vs if r % 2 == 0 else vs[::-1]):
            io = ios[v.fmt]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.host_steps):
                v.env.step_host(io)
            dt = time.perf_counter() - t0
            if r >= 2:
                times[v.fmt].append(dt * 1e6 / a.host_steps)
    for v in vs:
        emit(record("harvest5_b4096_step_host", v, B, 1, times[v.fmt], steps_per_round=a.host_steps, timing="host_clock",
                    host_obs_bytes_per_step=B * v.env.obs_layout.env_stride))
        v.env.close()

    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
