"""Tracked against untracked observation rings on the benchmark's schedule (row masks, DESIGN.md §3 item 19).

Harvest default5 (5 agents, V = 15) with bench.py's DeviceRollout: 4 096 envs in 8 PDL-chained ranges, or 65 536 envs in one
launch, observations written round-robin into the benchmark's ring.  Three arms in one process, alternated replay by replay:
  tracked  the ring from new_obs_buffer(), with row masks: zero rows that were zero are not stored
  plain    the same ring as plain torch.zeros tensors: every row stored (the parent's stores)
  no_obs   the same steps and resets writing no observations: the floor of logic, state traffic and launch chaining
The rows actually stored come from the masks, on a separate eager pass over one episode period of the tracked arm: a launch into
a slot stores the rows whose bit is set before or after it.  Prints one JSON line per workload.

    python profiles/obs_skip_probe.py [--envs 4096 65536] [--replays 20] [--steps 1000]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

LIMIT = bench.LIMIT


class NoObs(bench.DeviceRollout):
    def _one_step(self, t, group=None):
        env = self.env
        if group is None:
            if t % LIMIT == 0:
                env.reset(obs=False)
            env.step(self.actions[t % LIMIT], want_obs=False)
        else:
            Bg = env.B // self.groups
            if t % LIMIT == 0:
                env.reset(mask=self.gmask[group], obs=False)
            env.step_range(self.actions[t % LIMIT], group * Bg, Bg, want_obs=False)


def rollout(arm, a, B):
    cfg = bench.workload_config(a, 1, "harvest5_b4096", envs=B)
    ro = (NoObs if arm == "no_obs" else bench.DeviceRollout)(cfg, a, "cuda:0", gid_base=0, groups=bench.auto_groups(B))
    if arm == "plain":
        ro.ring = [torch.zeros_like(x) for x in ro.ring]
        assert all(ro.env.obs_mask(x) is None for x in ro.ring)
    elif arm == "tracked":
        assert all(ro.env.obs_mask(x) is not None for x in ro.ring)
    return ro


def popcount(t):
    return int(np.unpackbits(t.cpu().numpy().view(np.uint8)).sum())


def rows_stored(ro):
    """Rows stored per step over one episode period (its reset included), whole-batch launches, from the masks."""
    env, ring, R = ro.env, ro.ring, ro.ring_n
    total = 0
    s = ro.s
    for t in range(s, s + LIMIT):
        if t % LIMIT == 0:
            before = env.obs_mask(ring[t % R]).clone()
            env.reset(obs_out=ring[t % R])
            total += popcount(before | env.obs_mask(ring[t % R]))
        slot = ring[(t + 1) % R]
        before = env.obs_mask(slot).clone()
        env.step(ro.actions[t % LIMIT], obs_out=slot)
        total += popcount(before | env.obs_mask(slot))
    torch.cuda.synchronize()
    ro.s += LIMIT
    return total / LIMIT


def gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except Exception as e:                                    # noqa: BLE001
        return f"unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 65536])
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--steps", type=int, default=1000, help="steps per replay")
    ap.add_argument("--warmup", type=int, default=300)
    p = ap.parse_args()
    saved, sys.argv = sys.argv, [sys.argv[0]]
    a = bench.parse()                                         # the benchmark's defaults
    sys.argv = saved
    for B in p.envs:
        arms = {k: rollout(k, a, B) for k in ("tracked", "plain", "no_obs")}
        k = min(p.steps, 1000)
        for ro in arms.values():
            ro.eager(p.warmup)
            ro.eager((-ro.s) % LIMIT)
            ro.enqueue(k)                                     # captures the graph of this phase
            ro.eager((-ro.s) % LIMIT)
            ro.stream.synchronize()
        per = {name: [] for name in arms}
        for _ in range(p.replays):
            for name, ro in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(ro.stream)
                ro.enqueue(k)
                e1.record(ro.stream)
                ro.stream.synchronize()
                per[name].append(e0.elapsed_time(e1) / k * 1e3)   # us per step
                ro.eager((-ro.s) % LIMIT)
        env = arms["tracked"].env
        lay = env.layout
        rows = rows_stored(arms["tracked"])
        all_rows = env.B * env.n * 3 * env.N
        state_bytes = env.B * (env.bytes_per_env_step() - env.n * 3 * env.N * env.N)   # algorithmic non-observation bytes
        obs_full = env.B * lay.obs_env_stride
        med = {n: float(np.median(v)) for n, v in per.items()}
        out = dict(workload=f"harvest5 default5 V=15, {B} envs, {arms['tracked'].groups} range(s)", gpu=gpu_info(),
                   ring_n=arms["tracked"].ring_n, replays=p.replays, steps_per_replay=k,
                   us_per_step={n: dict(median=med[n], min=float(np.min(v)), max=float(np.max(v))) for n, v in per.items()},
                   speedup_tracked_vs_plain=med["plain"] / med["tracked"],
                   rows_stored_per_step=rows, rows_per_step=all_rows, rows_stored_frac=rows / all_rows,
                   obs_bytes_stored_per_step=rows * 32, obs_bytes_full_per_step=obs_full,
                   store_rate_TBps=dict(plain=(obs_full + state_bytes) / (med["plain"] * 1e-6) / 1e12,
                                        tracked=(rows * 32 + state_bytes) / (med["tracked"] * 1e-6) / 1e12))
        print(json.dumps(out), flush=True)
        for ro in arms.values():
            ro.close()
        del arms
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
