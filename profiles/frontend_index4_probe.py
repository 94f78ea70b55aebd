"""Cost of the fused observation front end on RGB planes (``ObsFrontEnd.forward``) and on packed colour-index observations
(``forward_index4``), and of a batched-runner rollout with each, same process, alternating replay by replay.

(a) Front end alone, on the same env states: an RGB env and an index4 env stepped from one seed write each step into a ring of
    observation buffers larger than the 126 MB L2; one CUDA graph per format runs one forward per ring slot, replays are timed
    with CUDA events.  The outputs of the two formats are compared bit for bit on every slot.  Harvest default5 (V=15) and
    Cleanup default5 (V=7), 5 agents, 4 096 envs (20 480 views) and 65 536 envs (327 680 views).
(b) ``BatchedEpisodeRunner.run()`` at B = 4 096 in 8 env ranges, one whole episode per run, host clock around a device
    synchronise.  Variants: RGB + fused front end, index4 + torch module on ``batch["obs"]`` (what index4 had before), index4 +
    fused front end.  The MAC is a stand-in with the reference agent's shape: ``rgb_preprocess`` (Conv2d(3, 6, 3) + LeakyReLU
    + Linear(6 P^2, 32) + LeakyReLU), a GRUCell(32, 64) per agent and a Linear(64, n_actions) + argmax; the incentive actions
    are constant.

One JSON line per (workload, variant) with the median, min and max time, the card name and its power limit.

    python profiles/frontend_index4_probe.py [--out FILE.jsonl]
"""
import argparse
import json
import math
import os
import sys
import time
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from homophily_marl_b200.batch_env import SSDBatchEnv  # noqa: E402
from homophily_marl_b200.frontend import ObsFrontEnd  # noqa: E402
from obs_index_probe import card  # noqa: E402

RING_BYTES = 256 << 20                                         # > 126 MB of L2
FRONT = [("harvest5", "harvest", "default5", 15), ("cleanup5", "cleanup", "default5", 7)]
RUNNER = [("cleanup3", "cleanup", "default3", 3, 7), ("harvest5", "harvest", "default5", 5, 15)]


def module(view, seed=0):
    torch.manual_seed(seed)
    P = 2 * view - 1
    return torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                               torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU()).cuda()


def front_end_alone(wname, env_name, mp, view, B, a, emit):
    dev = torch.device("cuda:0")
    envs = {fmt: SSDBatchEnv(env_name, B, 5, map=mp, view_size=view, episode_limit=10 ** 9, seed=1, device=dev,
                             extra_args=dict(obs_format=fmt, random_spawn_point=True, random_spawn_rotation=None))
            for fmt in ("rgb", "index4")}
    g = torch.Generator(device=dev).manual_seed(1)
    rings = {}
    for fmt, env in envs.items():
        rings[fmt] = [env.new_obs_buffer() for _ in range(max(2, math.ceil(RING_BYTES / (B * env.obs_layout.env_stride))))]
    K = max(len(r) for r in rings.values())
    for env in envs.values():
        env.reset()
    for t in range(K):                                         # the same states in both formats
        act = torch.randint(0, 5, (B, 5), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        for fmt, env in envs.items():
            env.step(act, obs_out=rings[fmt][t % len(rings[fmt])])
    fe = ObsFrontEnd.from_module(module(view), view, device=dev)
    rows, lay, ilay, lut = B * 5, envs["rgb"].layout, envs["index4"].obs_layout, envs["index4"].spec.lut
    outs = {fmt: [torch.empty((rows, 32), device=dev) for _ in rings[fmt]] for fmt in rings}

    def run(fmt):
        for buf, out in zip(rings[fmt], outs[fmt]):
            if fmt == "rgb":
                fe.forward(buf, rows, lay.obs_agent_stride, lay.obs_plane_stride, lay.obs_row_stride, out=out)
            else:
                fe.forward_index4(buf, rows, ilay.agent_stride, ilay.row_stride, lut, out=out)

    stream = torch.cuda.Stream(device=dev)
    graphs = {}
    for fmt in rings:
        with torch.cuda.stream(stream):
            run(fmt)                                           # warm-up, eager (allocates the handle's scratch)
        stream.synchronize()
        graphs[fmt] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[fmt], stream=stream):
            run(fmt)
    graphs["rgb"].replay()
    graphs["index4"].replay()
    torch.cuda.synchronize()
    # slot i of a ring holds the last of the K steps with step % len(ring) == i: compare the slots that hold the same step
    last = {fmt: {max(s for s in range(K) if s % len(r) == i): i for i in range(len(r))} for fmt, r in rings.items()}
    same = [(last["rgb"][s], last["index4"][s]) for s in last["rgb"] if s in last["index4"]]
    identical = all(torch.equal(outs["rgb"][i], outs["index4"][j]) for i, j in same)
    times = {fmt: [] for fmt in rings}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(a.replays + 2):                             # the first two rounds are warm-up
        for fmt in (("rgb", "index4") if r % 2 == 0 else ("index4", "rgb")):
            with torch.cuda.stream(stream):
                ev[0].record()
                graphs[fmt].replay()
                ev[1].record()
            stream.synchronize()
            if r >= 2:
                times[fmt].append(ev[0].elapsed_time(ev[1]) * 1e3 / len(rings[fmt]))
    for fmt in rings:
        ts = sorted(times[fmt])
        obs_bytes = rows * (lay.obs_agent_stride if fmt == "rgb" else ilay.agent_stride)
        emit(dict(probe="frontend_index4_probe", part="a_front_end", workload=f"{wname}_b{B}", view=view, views=rows,
                  obs_format=fmt, us_per_forward_median=ts[len(ts) // 2], us_per_forward_min=ts[0], us_per_forward_max=ts[-1],
                  forwards_per_replay=len(rings[fmt]), replays=len(ts), obs_bytes_per_forward=obs_bytes,
                  bit_identical_to_rgb=identical, slots_compared=len(same), timing="cuda_graph_events"))
    graphs.clear()
    fe.close()
    for env in envs.values():
        env.close()
    torch.cuda.empty_cache()


class StandInMAC:
    """The reference MAC's calls as the runner makes them, with its agent's feature path (``agent.rgb_preprocess``)."""

    def __init__(self, view, n, n_actions):
        self.N, self.n = 2 * view + 1, n
        mod = module(view)
        self.gru, self.q = torch.nn.GRUCell(32, 64).cuda(), torch.nn.Linear(64, n_actions).cuda()
        self.agent = types.SimpleNamespace(conv_to_fc=mod, rgb_preprocess=mod)
        self.h_env = self.h_inc = None

    def init_hidden(self, batch_size):
        self.h_env = torch.zeros((batch_size * self.n, 64), device="cuda")

    def select_actions_env(self, batch, t_ep, t_env, test_mode=False):
        x = self.agent.rgb_preprocess(batch["obs"][:, t_ep].reshape(-1, 3, self.N, self.N))
        self.h_env = self.gru(x, self.h_env)
        return self.q(self.h_env).argmax(-1).view(batch.batch_size, self.n, 1)

    def select_actions_inc(self, actions, batch, t_ep, t_env, test_mode=False, agent_pos_replay=None):
        return torch.zeros((batch.batch_size, self.n, self.n, 1), dtype=torch.long, device="cuda")


def runner_rollouts(wname, env_name, mp, n, view, a, emit):
    from test_batched_runner import FakeBatch, _scheme
    from homophily_marl_b200.batched_runner import BatchedEpisodeRunner
    B, G, T = 4096, 8, a.episode_limit
    variants = [("rgb", True), ("index4", False), ("index4", "index4")]
    runners = []
    for fmt, fused in variants:
        extra = dict(random_spawn_point=True, random_spawn_rotation=None, obs_format=fmt)
        env_args = dict(num_agents=n, episode_limit=T, view_size=view, map=mp, extra_args=extra, seed=3)
        args = types.SimpleNamespace(batch_size_run=B, env=env_name, env_args=env_args, device="cuda:0", name="homophily",
                                     mac="homophily_mac", n_actions=None, ind_reward=True, runner_log_interval=10 ** 12,
                                     test_nepisode=B, env_groups=G, fused_frontend=fused, rgb_input=True)
        r = BatchedEpisodeRunner(args, types.SimpleNamespace(log_stat=lambda *x: None))
        info = r.get_env_info()
        args.n_actions = info["n_actions"]
        mac = StandInMAC(view, n, info["n_actions"])
        r.setup(None, None, None, mac, batch_cls=lambda *x, **k: None)
        assert (r.front is not None) == bool(fused)
        scheme = _scheme(n, info["n_actions"], *info["state_dims"], info["obs_dims"][0])
        r.use_batch_factory(lambda s=scheme: FakeBatch(s, B, T + 1, "cuda:0"))
        runners.append((fmt, fused, r))
    times = {i: [] for i in range(len(runners))}
    for rep in range(a.runs + 1):                              # the first round is warm-up
        order = range(len(runners)) if rep % 2 == 0 else reversed(range(len(runners)))
        for i in order:
            r = runners[i][2]
            r.batch = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r.run(test_mode=True)
            torch.cuda.synchronize()
            if rep >= 1:
                times[i].append((time.perf_counter() - t0) * 1e6 / (T + 1))
            r.batch = None                                     # Harvest: 24 GB of f32 observations per episode batch
    for i, (fmt, fused, r) in enumerate(runners):
        ts = sorted(times[i])
        emit(dict(probe="frontend_index4_probe", part="b_runner", workload=f"{wname}_b{B}_g{G}", envs=B, env_ranges=G, view=view,
                  obs_format=fmt, fused_frontend=fused, episode_steps=T + 1, us_per_step_median=ts[len(ts) // 2],
                  us_per_step_min=ts[0], us_per_step_max=ts[-1], runs=len(ts), timing="host_clock_device_sync",
                  mac="stand-in (rgb_preprocess + GRUCell(32, 64) + Linear + argmax)"))
        r.batch = None
        if r.front is not None:
            r.front.detach()
        r.close_env()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--replays", type=int, default=12, help="timed graph replays per format (a)")
    ap.add_argument("--runs", type=int, default=4, help="timed episodes per variant (b)")
    ap.add_argument("--episode-limit", type=int, default=100)
    ap.add_argument("--part", choices=("a", "b", "ab"), default="ab")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("frontend_index4_probe needs a CUDA device")
    name, power = card()
    lines = []

    def emit(rec):
        rec.update(gpu=name, power_limit=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    if "a" in a.part:
        for wname, env_name, mp, view in FRONT:
            for B in (4096, 65536):
                front_end_alone(wname, env_name, mp, view, B, a, emit)
    if "b" in a.part:
        with torch.no_grad():
            for wname, env_name, mp, n, view in RUNNER:
                runner_rollouts(wname, env_name, mp, n, view, a, emit)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
