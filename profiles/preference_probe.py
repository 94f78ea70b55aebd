"""Cost of per-agent preference sets (extra_args reward_shaping as a list of one dict per agent, with social value orientation;
DESIGN.md §3 item 20), against the parent tree, in one run.

Four arms per workload, built with the same seed and action schedule:
  off         no shaping (what bench.py runs);
  item17      one dict (Hughes' Cleanup weights with some prosocial mixing), set through ssd_set_reward_shaping;
  roster      a mixed population without SVO: one dict per agent, set through ssd_set_reward_preferences with a roster;
  roster_svo  the same population with social value orientation on three of the five agents.
Workloads: Harvest default5 at 4 096 envs in 8 env ranges of 512 on 8 streams (programmatic dependent launch), and Harvest and
Cleanup default5 at 65 536 envs; RGB observations into a ring of buffers, no state image, tag_timeout 0, uniform random actions
over every action.  Each arm is a CUDA graph of K steps; replays are timed with CUDA events, the arms alternating replay by replay
after two warm-up rounds.  A tree whose reward_shaping takes no list (the parent) runs the first two arms only.

With --parent DIR the probe alternates worker processes on the parent's tree and on this tree, round by round, and then runs
bench.py (--no-extra --no-train --no-cpu-baseline) in each tree, alternated too.  One JSON line per measurement, with the card
name and power limit read in the same run.

    python profiles/preference_probe.py --parent DIR [--rounds R] [--out FILE.jsonl] [--steps K] [--replays N]
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 5, 15, 4096, 8, 4),      # name, env, map, n, view, envs, ranges, ring
             ("harvest5_b65536", "harvest", "default5", 5, 15, 65536, 1, 2),
             ("cleanup5_b65536", "cleanup", "default5", 5, 7, 65536, 1, 2)]
HUGHES = {"alpha": 5.0, "beta": 0.05, "prosocial": 0.25}
ROSTER = [HUGHES, {"prosocial": 0.5}, {}, {"beta": 1.0, "decay": 0.9}, {"alpha": 1.0}]
SVO = [{}, {"svo_angle": 45, "svo_weight": 0.5}, {}, {"svo_angle": 90, "svo_weight": 2.0}, {"svo_angle": -30, "svo_weight": 0.1}]
ARMS = {"off": None, "item17": HUGHES, "roster": ROSTER, "roster_svo": [dict(r, **s) for r, s in zip(ROSTER, SVO)]}


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                     # noqa: BLE001
        q = f"unknown ({e})"
    return torch.cuda.get_device_name(0), q


class Arm:
    def __init__(self, SSDBatchEnv, wl, arm, K, seed=1):
        import torch
        _, env_name, mp, n, view, B, groups, ring = wl
        dev = torch.device("cuda:0")
        self.arm = arm
        self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=10 ** 4, seed=seed, device=dev,
                               extra_args=dict(disable_fire_action=False, disable_rotation_action=False,
                                               reward_shaping=ARMS[arm]))
        self.K, self.groups = K, groups
        g = torch.Generator(device=dev).manual_seed(seed)
        self.actions = torch.randint(0, self.env.n_actions, (K, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        self.ring = [self.env.new_obs_buffer() for _ in range(ring)]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
        self.env.reset()
        torch.cuda.synchronize()

    def run(self):
        import torch
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
        import torch
        with torch.cuda.stream(self.stream):
            self.run()                                         # warm-up, eager
        self.stream.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            self.run()

    def time_graph(self, ev):
        import torch
        with torch.cuda.stream(self.stream):
            ev[0].record()
            self.graph.replay()
            ev[1].record()
        self.stream.synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e3 / self.K


def worker(a):
    """Times every arm this tree supports on every workload; one JSON line per (workload, arm)."""
    sys.path.insert(0, a.tree)
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    if not torch.cuda.is_available():
        raise SystemExit("preference_probe needs a CUDA device")
    name, smi = card()
    for wl in WORKLOADS:
        arms = []
        for arm in ARMS:
            try:
                arms.append(Arm(SSDBatchEnv, wl, arm, a.steps))
            except (TypeError, ValueError):                    # the parent's reward_shaping takes one dict only
                continue
        for v in arms:
            v.capture()
        times = {v.arm: [] for v in arms}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for v in (arms if r % 2 == 0 else arms[::-1]):
                dt = v.time_graph(ev)
                if r >= 2:
                    times[v.arm].append(dt)
        off = sorted(times["off"])[len(times["off"]) // 2]
        for v in arms:
            ts = sorted(times[v.arm])
            rec = dict(probe="preference_probe", tree=a.label, workload=wl[0], envs=wl[5], env_ranges=wl[6], arm=v.arm,
                       steps_per_replay=a.steps, replays=len(ts), us_per_step_median=ts[len(ts) // 2], us_per_step_min=ts[0],
                       us_per_step_max=ts[-1], over_off=ts[len(ts) // 2] / off, gpu=name,
                       nvidia_smi_name_power_limit_max_sm_clock=smi)
            print(json.dumps(rec), flush=True)
        for v in arms:
            v.graph = None
            v.env.close()
        torch.cuda.empty_cache()


def driver(a):
    lines = []

    def run(cmd, cwd, label):
        r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=3600)
        if r.returncode != 0:
            raise SystemExit(f"{label} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
        out = [json.loads(line) for line in r.stdout.splitlines() if line.startswith("{")]
        for rec in out:
            rec.setdefault("tree", label)
            print(json.dumps(rec), flush=True)
        lines.extend(out)

    trees = (("parent", os.path.abspath(a.parent)), ("this", HERE))
    for _ in range(a.rounds):
        for label, tree in trees:
            run([sys.executable, os.path.abspath(__file__), "--worker", "--tree", tree, "--label", label, "--steps",
                 str(a.steps), "--replays", str(a.replays)], tree, label)
    for _ in range(a.rounds):
        for label, tree in trees:
            run([sys.executable, "bench.py", "--gpus", "1", "--steps", "5000", "--warmup", "500", "--no-extra", "--no-train",
                 "--no-cpu-baseline"], tree, label)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", default=None, help="the parent commit's tree, its library built: alternate it with this tree")
    ap.add_argument("--rounds", type=int, default=2, help="parent / this alternations")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=200, help="steps per graph replay")
    ap.add_argument("--replays", type=int, default=10, help="timed replays per arm")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--tree", default=HERE, help=argparse.SUPPRESS)
    ap.add_argument("--label", default="this", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker or a.parent is None:
        worker(a)
    else:
        driver(a)


if __name__ == "__main__":
    main()
