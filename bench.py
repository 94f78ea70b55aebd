#!/usr/bin/env python
"""Benchmark of the SSD env hot path (fused step + observation render).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU env on the box's host cores

Metric (BASELINE.json): agent-steps/s, device-timed, + fraction of the HBM roofline.
A "step" is one fused step+obs pass over the whole resident batch (the synchronous episode reset every
`episode_limit` steps is inside the timed region).  Default workload = BASELINE configs[1]: Harvest map=default5,
5 agents, 4096 envs per GPU, uniform random actions, yaml-default extra_args.  Weak scaling: every rank owns 4096
envs keyed by global env id; no collective on the step path.

Timing: exactly K = --steps steps are timed.  They are split into R replays of near-equal length (one per 1000 steps, at
most 20; --replays overrides), each captured as CUDA graphs (launch-bound inner loop).  The same schedule is
first run once untimed (graph upload, TLB warm-up over the observation ring), then the R replays are timed one by one with
CUDA events on the launch stream, bracketed by a barrier + synchronize; `ms_per_step` is the MEDIAN over replays of replay
time / replay steps, MAX over ranks (min / median / max replay times are all in the line).  Observations go round-robin
into a ring of buffers larger than L2.  Prints ONE JSON line on rank 0.

    python bench.py --steps 2000 --warmup 100 --dump-outputs DIR

writes what the last timed step returned as DIR/<name>.npy (see dump_outputs); the inputs depend on the arguments only, so
two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                                # the benchmark leaves the tree as it found it

WORKLOADS = {
    # name: (env, map, num_agents, view_size, envs_per_gpu, BASELINE.json config it is)
    "harvest5_b4096": ("harvest", "default5", 5, 15, 4096, "configs[1] Harvest default5, 5 agents, 4096 envs"),
    "cleanup5_b4096": ("cleanup", "default5", 5, 7, 4096, "configs[0] map/agents at B=4096"),
    "cleanup10_b2048": ("cleanup", "default10", 10, 7, 2048, "configs[2] Cleanup default10, 16384 envs over 8 GPUs"),
    "cleanup3_b4096": ("cleanup", "default3", 3, 7, 4096, "configs[3] map/agents at B=4096"),
    "harvest5_b65536": ("harvest", "default5", 5, 15, 65536, "configs[4] Harvest default5, 65536 envs obs stress"),
    "cleanup5_b65536": ("cleanup", "default5", 5, 7, 65536, "configs[0] map/agents at B=65536 (large-batch regime)"),
    "cleanup10_b16384": ("cleanup", "default10", 10, 7, 16384, "configs[2] whole 16384-env job on ONE GPU"),
}
# extra workloads measured into the same JSON line (<= ~1 s each): name -> scaling under --gpus N
EXTRA_N1 = ("harvest5_b65536", "cleanup10_b2048", "cleanup5_b4096", "cleanup3_b4096", "cleanup5_b65536", "cleanup10_b16384")
L2_BYTES = 126 * 2 ** 20
LIMIT = 100                                                   # episode_limit of both yaml files
METRIC = "agent-steps/sec (step+obs, device-timed)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20000, help="number of timed steps K of the headline workload")
    ap.add_argument("--warmup", type=int, default=500)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="harvest5_b4096", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="override envs per GPU")
    ap.add_argument("--replays", type=int, default=0,
                    help="the K timed steps are split into this many individually timed replays (0 = auto: one per 1000 steps, <= 20)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (obs, reward, clean, apple_cnt, done) as "
                         "DIR/<name>.npy (float32; obs of a fixed sample of envs); rank 0's envs only")
    ap.add_argument("--groups", type=int, default=0,
                    help="step the batch as G independent env ranges on G streams (SSDBatchEnv.step_range, the asynchronous-sampler "
                         "API BatchedEpisodeRunner uses with args.env_groups); 0 = auto: 8 ranges for <= 4096 envs, 4 for <= 8192, else 1")
    ap.add_argument("--no-graph", action="store_true", help="launch every step from Python instead of CUDA graphs")
    ap.add_argument("--e2e-steps", type=int, default=60)
    ap.add_argument("--random-spawn", action="store_true")
    ap.add_argument("--obs-color", default="simplified", choices=["simplified", "full"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the other BASELINE configs (`workloads` key)")
    ap.add_argument("--no-train", action="store_true", help="skip the end-to-end training-loop timing (`train_e2e` key)")
    ap.add_argument("--train-t-max", type=int, default=2500)
    ap.add_argument("--ring", type=int, default=0,
                    help="DIAGNOSTIC: force the number of observation ring buffers (1 = L2-resident stores; not a valid bench number)")
    ap.add_argument("--masked-actions", action="store_true",
                    help="draw actions from the yaml-masked set ({0-4,8} cleanup / {0-4} harvest) instead of all n_actions")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def extra_args(a):
    e = dict(obs_color=a.obs_color)
    if a.random_spawn:
        e.update(random_spawn_point=True, random_spawn_rotation=None)
    return e


def workload_config(a, world, name=None, envs=None):
    """`config` of the JSON line: identical for both arms (nothing implementation-specific in here)."""
    name = name or a.workload
    env, mp, n, view, B, what = WORKLOADS[name]
    B = envs or (a.envs if name == a.workload and a.envs else B)
    return dict(workload=f"{name}: {what}", env=env, map=mp, num_agents=n, view_size=view, envs_per_gpu=B,
                global_envs=B * world, episode_limit=LIMIT,
                actions="uniform over the yaml-masked set" if a.masked_actions else "uniform over all n_actions",
                extra_args="yaml defaults" if not a.random_spawn else "random spawn point+rotation",
                obs_color=a.obs_color, obs_format="u8 RGB planes, pixel rows padded to a multiple of 4 bytes")


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML, 2 ms)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        self.samples, self.mask, self.max_mhz, self._stop, self._thr, self.h = [], 0, None, threading.Event(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def bind_cpu_affinity(self):
        """Pins this rank's host threads to the CPUs NVML calls ideal for its GPU (NUMA-local pinned buffers for the e2e copies)."""
        try:
            if self.h is not None:
                self.nv.nvmlDeviceSetCpuAffinity(self.h)
                return sorted(os.sched_getaffinity(0))
        except Exception:
            pass
        return None

    def sample(self):
        if self.h is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            self.mask |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self.sample()
            self._stop.wait(0.002)

    def __enter__(self):
        if self.h is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in self.REASONS.items() if self.mask & k), "samples": len(self.samples)}


# --------------------------------------------------------------------------- CPU arms
def oracle_batch(cfg, B, seed, gid0, a):
    from homophily_marl_b200 import mapspec
    from oracle import oracle as O
    spec = mapspec.compile_map(cfg["env"], cfg["map"], cfg["num_agents"], cfg["view_size"], cfg["episode_limit"], obs_color=a.obs_color)
    return spec, O.OracleBatch.from_spec(spec, n_envs=B, seed=seed, env_gid0=gid0, random_spawn_point=a.random_spawn,
                                         spawn_rotation=None if a.random_spawn else 0)


def time_oracle(cfg, a, steps, warmup, budget_s, threads):
    """Times the C port of the reference env (step + get_obs) on a bounded sample of the workload."""
    B_full = cfg["envs_per_gpu"]
    spec, probe = oracle_batch(cfg, min(256, B_full), a.seed, 0, a)
    rs = np.random.RandomState(a.seed)
    probe.reset(threads=threads)
    acts = rs.randint(0, spec.n_actions, size=(probe.B, spec.n_agents)).astype(np.uint8)
    out = probe.step(acts, threads=threads)
    t0 = time.perf_counter()
    for _ in range(4):
        probe.step(acts, threads=threads, out=out)
    per_env = (time.perf_counter() - t0) / (4 * probe.B)
    B = int(max(64, min(B_full, budget_s / max(steps + warmup, 1) / per_env)))
    spec, ob = oracle_batch(cfg, B, a.seed, 0, a)
    ob.reset(threads=threads)
    actions = rs.randint(0, spec.n_actions, size=(min(steps + warmup, 64), B, spec.n_agents)).astype(np.uint8)
    out, t = None, 0
    for s in range(warmup):
        out = ob.step(actions[s % len(actions)], threads=threads, out=out)
        t += 1
        if t % cfg["episode_limit"] == 0:
            ob.reset(threads=threads)
    t0 = time.perf_counter()
    for s in range(steps):
        out = ob.step(actions[(s + warmup) % len(actions)], threads=threads, out=out)
        t += 1
        if t % cfg["episode_limit"] == 0:
            ob.reset(threads=threads)
    dt = time.perf_counter() - t0
    return dict(value=B * spec.n_agents * steps / dt, seconds=dt, envs=B, steps=steps, ms_per_step=dt / steps * 1e3)


def time_python_reference(cfg, a, steps, warmup, procs, budget_s):
    """The reference's OWN env (unmodified MapEnv.step + get_obs from baseline/_ref or /root/reference), `procs` independent
    single-env processes.  None when no reference sources travelled to this box."""
    from baseline import refloop
    if not refloop.available() or a.random_spawn or a.obs_color != "simplified" or a.masked_actions:
        return None
    r = refloop.time_reference_env(cfg["env"], cfg["map"], cfg["num_agents"], cfg["view_size"], steps=steps, warmup=warmup,
                                   procs=procs, seed=a.seed, budget_s=budget_s)
    r["sample"] = (f"{procs} of {cfg['envs_per_gpu']} envs x {r['env_steps'] // procs} steps, unmodified reference MapEnv.step()+get_obs() "
                   f"(map_env.py:874-945), {procs} single-env processes")
    return r


def run_reference(a):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    cfg = workload_config(a, a.gpus)
    threads = os.cpu_count() or 1
    port = time_oracle(cfg, a, min(a.steps, 200), min(a.warmup, 20), budget_s=20.0, threads=threads)
    port_line = {"value": port["value"], "unit": "agent-steps/s", "cores": threads, "kind": "port",
                 "sample": f"{port['envs']} of {cfg['envs_per_gpu']} envs x {port['steps']} steps (step+get_obs), {threads} OpenMP threads"}
    ref = time_python_reference(cfg, a, steps=a.steps, warmup=min(a.warmup, 100), procs=threads, budget_s=45.0)
    if ref is not None:
        value, ms = ref["value"], ref["ms_per_env_step_per_proc"]
        cpu = {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "reference", "sample": ref["sample"]}
        note = ("the reference is pure Python: this arm runs its unmodified env from baseline/_ref on all host cores (one "
                "single-env process per core; the reference itself has no parallel runner, episode_runner.py:13); "
                "`cpu_baseline_port` is the C restatement (oracle/ssd_oracle.c, OpenMP) on the same cores")
    else:
        value, ms = port["value"], port["ms_per_step"]
        cpu = dict(port_line)
        note = "no reference sources on this box (baseline/_ref absent): this arm times oracle/ssd_oracle.c, the C port pinned bit-exact against the reference"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "agent-steps/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
            "cpu_baseline": cpu, "cpu_baseline_port": port_line,
            "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": note}
    if not a.no_train:
        line["train_e2e"] = train_e2e(a, which=("reference",))
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------- end-to-end training loop (BASELINE configs[3])
def train_e2e(a, which=("b200", "b200_batched", "b200_batched_4096", "reference")):
    """`run.run_sequential` of the UNCHANGED reference (rollouts + replay + HomophilyLearner updates + test episodes),
    Cleanup default3 / 3 agents / yaml hyper-parameters, t_max env steps: on the CUDA env through the reference's own
    single-env EpisodeRunner ('b200'), through BatchedEpisodeRunner at B=256 with the fused u8 front end, the device epsilon-greedy
    selector and DeviceHomophilyLearner ('b200_batched', 100 x t_max env steps; MAC and replay buffer are the reference's), and on
    the reference's own CPU env ('reference').  env-steps/s = train env steps / wall seconds (test episodes are extra work)."""
    from baseline import refloop
    out = {"what": "run_sequential, Cleanup default3, 3 agents, homophily IQL, yaml defaults; env-steps/s incl. learner updates + tests",
           "t_max": a.train_t_max, "unit": "env-steps/s"}
    if not refloop.available():
        out["unavailable"] = "reference sources absent (baseline/_ref)"
        return out
    import torch
    cuda = torch.cuda.is_available()
    common = dict(seed=a.seed, use_cuda=cuda, save_model=False, test_nepisode=4, test_interval=1000, log_interval=1000,
                  runner_log_interval=1000, learner_log_interval=1000, env_args=dict(num_agents=3, map="default3"))
    # untimed warm-up with the SAME shapes as the timed single-env runs (CUDA context, cuDNN / cuBLAS heuristics for batch 1
    # rollouts and batch 16 learner steps, autograd kernels): 18 episodes, two learner updates
    try:
        warm = refloop.load_config("cleanup", t_max=min(1700, a.train_t_max), **common)
        refloop.run_training(warm, backend="reference" if (which == ("reference",) or not cuda) else "b200")
    except Exception as e:
        out["warmup_error"] = f"{type(e).__name__}: {e}"[:200]
    for key in which:
        try:
            if key.startswith("b200_batched"):
                B = 4096 if key.endswith("4096") else 256
                t_max = (3 * B * LIMIT) if B == 4096 else 100 * a.train_t_max   # 4 / 10 rollouts of B episodes, one learner step each
                if cuda:                                                   # untimed: the batched stack's own kernels / cuDNN shapes
                    wcfg = refloop.load_config("cleanup", t_max=1, runner="batched", batch_size_run=B, buffer_size=2 * B,
                                               buffer_cpu_only=False, fused_frontend=True, action_selector="epsilon_greedy_b200",
                                               learner="homophily_learner_b200",
                                               **{**common, "test_nepisode": B, "test_interval": 10 ** 9})
                    refloop.run_training(wcfg, backend="b200")
                cfg = refloop.load_config("cleanup", t_max=t_max, runner="batched", batch_size_run=B, buffer_size=(4 if B == 256 else 1) * B,
                                          buffer_cpu_only=False, fused_frontend=True, action_selector="epsilon_greedy_b200",
                                          learner="homophily_learner_b200",
                                          **{**common, "test_nepisode": B, "test_interval": t_max})
                per_run = B * LIMIT
            else:
                t_max = a.train_t_max
                cfg = refloop.load_config("cleanup", t_max=t_max, **common)
                per_run = LIMIT
            if key != "reference" and not cuda:
                continue
            r = refloop.run_training(cfg, backend="reference" if key == "reference" else "b200")
            steps = (t_max // per_run + 1) * per_run                       # run_sequential loops while t_env <= t_max
            out[key] = {"value": steps / r["seconds"], "env_steps": steps, "seconds": r["seconds"],
                        "return_mean": float(r["stats"].get("return_mean", float("nan"))),
                        "loss_value_env": float(r["stats"].get("loss_value_env", float("nan")))}
        except Exception as e:                                             # the bench line must still be printed
            out[key] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


# --------------------------------------------------------------------------- policy-side kernel (SURVEY 8f f2)
def frontend_probe(cfg, a, dev):
    """Fused u8-obs front end (conv3x3 + LeakyReLU on CUDA cores -> Linear on tcgen05) on the observations of the headline
    workload, next to the torch module it replaces (u8 -> fp32 /256 -> Conv2d -> Linear).  Bound: the conv's fp32 FMAs."""
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    from homophily_marl_b200.frontend import ObsFrontEnd
    B, n, view = cfg["envs_per_gpu"], cfg["num_agents"], cfg["view_size"]
    env = SSDBatchEnv(cfg["env"], B, n, map=cfg["map"], view_size=view, episode_limit=LIMIT, extra_args=extra_args(a), seed=a.seed, device=dev)
    env.reset()
    P = 2 * view - 1
    torch.manual_seed(a.seed)
    mod = torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                              torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU()).to(dev)
    fe = ObsFrontEnd.from_module(mod, view, device=dev)
    x8 = env.obs_view().reshape(B * n, 3, env.N, env.N)

    def timed(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3
    with torch.no_grad():
        t_fused = timed(lambda: fe.forward_env(env))
        t_torch = timed(lambda: mod(x8.float() / 256))
        err = float((fe.forward_env(env) - mod(x8.float() / 256)).abs().max())
    rows = B * n
    conv_flop = rows * 6 * P * P * 27 * 2
    fc_flop = rows * 6 * P * P * 32 * 2
    sm_mhz = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"] if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1965.0
    fp32_peak = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 2 * sm_mhz * 1e6 / 1e12
    fe.close()
    env.close()
    return {"what": "ssd_frontend_forward on the workload's u8 observations: conv3x3(3->6)+LeakyReLU -> Linear(->32)+LeakyReLU",
            "agent_views": rows, "us": t_fused * 1e6, "views_per_s": rows / t_fused,
            "torch_module_us": t_torch * 1e6, "speedup_vs_torch": t_torch / t_fused, "max_abs_diff_vs_torch_default": err,
            "roofline": {"bound": "fp32 FMA on the CUDA cores (conv); the tcgen05 Linear and HBM are far from their limits",
                         "conv_tflops": conv_flop / t_fused / 1e12, "fp32_peak_tflops": fp32_peak,
                         "frac": conv_flop / t_fused / 1e12 / fp32_peak, "fc_tensor_tflops_3x_tf32": 3 * fc_flop / t_fused / 1e12,
                         "hbm_gbs": rows * env_bytes_per_view(view) / t_fused / 1e9}}


def env_bytes_per_view(view):
    N = 2 * view + 1
    return 3 * N * ((N + 3) // 4 * 4) + 32 * 4


# --------------------------------------------------------------------------- CUDA arm
def ring_len(obs_bytes, forced=0):
    """Observation ring > 2.2 x L2, rounded up to a divisor of the episode length so the launch schedule has period LIMIT."""
    if forced > 0:
        return forced
    need = max(2, int(math.ceil(2.2 * L2_BYTES / obs_bytes)))
    for d in (2, 4, 5, 10, 20, 25, 50, 100):
        if d >= need:
            return d
    return 100


class DeviceRollout:
    """K-step schedules of the fused step+obs launch (plus the reset every LIMIT steps) as cached CUDA graphs."""

    def __init__(self, cfg, a, dev, gid_base, groups=1):
        import torch
        from homophily_marl_b200.batch_env import SSDBatchEnv
        self.torch, self.dev, self.groups = torch, dev, max(1, groups)
        B, n = cfg["envs_per_gpu"], cfg["num_agents"]
        self.env = env = SSDBatchEnv(cfg["env"], B, n, map=cfg["map"], view_size=cfg["view_size"], episode_limit=LIMIT,
                                     extra_args=extra_args(a), seed=a.seed, device=dev, env_gid_base=gid_base)
        self.obs_bytes = B * env.layout.obs_env_stride
        self.ring_n = ring_len(self.obs_bytes, a.ring)
        self.ring = [env.new_obs_buffer() for _ in range(self.ring_n)]
        g = torch.Generator(device=dev).manual_seed(a.seed * 1000 + gid_base)
        self.actions = torch.randint(0, env.n_actions, (LIMIT, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        if a.masked_actions:                                   # disable_rotation_action / disable_fire_action (yaml defaults)
            allowed = torch.tensor([0, 1, 2, 3, 4] + ([8] if env.n_actions == 9 else []), device=dev, dtype=torch.uint8)
            self.actions = allowed[torch.randint(0, len(allowed), (LIMIT, B, n), generator=g, device=dev)]
        self.stream = torch.cuda.Stream(device=dev)
        self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(self.groups)] if self.groups > 1 else []
        if self.groups > 1:
            if B % self.groups:
                raise SystemExit("--groups must divide the number of envs")
            self.gmask = []
            for k in range(self.groups):
                m = torch.zeros(B, dtype=torch.uint8, device=dev)
                m[k * (B // self.groups):(k + 1) * (B // self.groups)] = 1
                self.gmask.append(m)
        self.s = 0                                             # global step index of the NEXT step
        self.cache = {}                                        # (phase, k) -> (graph, launches captured)
        self.use_graph = not a.no_graph

    def _one_step(self, t, group=None):
        env = self.env
        if group is None:
            if t % LIMIT == 0:
                env.reset(obs_out=self.ring[t % self.ring_n])
            env.step(self.actions[t % LIMIT], obs_out=self.ring[(t + 1) % self.ring_n])
        else:
            Bg = env.B // self.groups
            if t % LIMIT == 0:
                env.reset(mask=self.gmask[group], obs_out=self.ring[t % self.ring_n])
            env.step_range(self.actions[t % LIMIT], group * Bg, Bg, obs_out=self.ring[(t + 1) % self.ring_n])

    def _run_steps(self, t0, k):
        """Enqueues steps [t0, t0+k) on the current (capturing or live) stream(s)."""
        torch = self.torch
        if self.groups == 1:
            for i in range(k):
                self._one_step(t0 + i)
            return
        main = torch.cuda.current_stream(self.dev)
        for gidx, gs in enumerate(self.gstreams):              # fork: every group advances k steps on its own stream
            gs.wait_stream(main)
            with torch.cuda.stream(gs):
                for i in range(k):
                    self._one_step(t0 + i, gidx)
        for gs in self.gstreams:                               # join
            main.wait_stream(gs)

    def eager(self, k):
        with self.torch.cuda.stream(self.stream):
            self._run_steps(self.s, k)
        self.s += k

    def enqueue(self, K):
        """Steps [s, s+K) as graph replays (chunks <= 1000 steps; graphs keyed by the schedule phase).  Returns launches."""
        torch, launched = self.torch, 0
        with torch.cuda.stream(self.stream):
            if not self.use_graph:
                n0 = self.env.launch_count
                self._run_steps(self.s, K)
                self.s += K
                return self.env.launch_count - n0
            todo = K
            while todo > 0:
                k = min(1000, todo)
                key = (self.s % LIMIT, k)
                if key not in self.cache:
                    self.stream.synchronize()
                    n0 = self.env.launch_count
                    gr = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr, stream=self.stream):
                        self._run_steps(self.s, k)               # capture does not execute
                    self.cache[key] = (gr, self.env.launch_count - n0)
                gr, n = self.cache[key]
                gr.replay()
                launched += n
                self.s += k
                todo -= k
        return launched

    def close(self):
        self.cache.clear()
        self.env.close()


def auto_groups(B):
    """Env ranges per step (SSDBatchEnv.step_range, one stream each): up to 4 096 envs as 8 ranges, up to 16 384 as ranges of 2 048
    (the largest launch that is chained by programmatic dependent launch); larger batches as one launch -- measured optimum in
    each regime (profiles/r2_notes.md sections 2-3)."""
    if B <= 4096 and B % 8 == 0:
        return 8
    if B <= 16384 and B % 2048 == 0:
        return B // 2048
    return 1


def replay_lengths(K, replays):
    """K timed steps as `replays` replays of near-equal length (they sum to K)."""
    R = max(1, min(replays, K))
    q, r = divmod(K, R)
    return [q + (i < r) for i in range(R)]


def measure(cfg, a, dev, rank, world, K, warmup, replays, groups=1, clock=None, dist=None):
    """Warm-up, one untimed pass over the schedule of the timed part, then exactly K timed steps as `replays` individually
    timed replays."""
    import torch
    ro = DeviceRollout(cfg, a, dev, gid_base=rank * cfg["envs_per_gpu"] if "gid_base" not in cfg else cfg["gid_base"], groups=groups)
    ro.eager(max(warmup, 3))
    lens = replay_lengths(K, replays)
    s0 = ro.s
    for k in lens:
        ro.enqueue(k)                                          # untimed: captures + uploads every graph the timed part uses
    ro.eager((s0 - ro.s) % LIMIT)                              # back to the same schedule phase, so the timed part reuses them
    ro.stream.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(lens) + 1)]
    launches = 0
    barrier()
    ctx = clock if clock is not None else _Null()
    with ctx:
        with torch.cuda.stream(ro.stream):
            torch.cuda._sleep(2 * 10 ** 6)                    # ~1 ms spin: the first replay is queued before the clock starts
        evs[0].record(ro.stream)
        s_start = ro.s
        for r, k in enumerate(lens):
            launches += ro.enqueue(k)
            evs[r + 1].record(ro.stream)
        timed_steps = ro.s - s_start
        if clock is not None:
            clock.sample()                                    # the GPU is still executing the enqueued replays here
        barrier()
    per = np.array([evs[r].elapsed_time(evs[r + 1]) for r in range(len(lens))])  # ms per replay
    per_step = per / np.array(lens)
    stats = torch.tensor([np.median(per_step), np.median(per), per.min(), per.max(), per.sum()], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_step, med, mn, mx, tot = (float(x) for x in stats)
    env = ro.env
    B, n = env.B, env.n
    alg = env.bytes_per_env_step() * B
    res = dict(ms_per_step=ms_step, value=B * n * world / (ms_step * 1e-3), replay_ms={"min": mn, "median": med, "max": mx},
               steps=K, timed_steps=timed_steps, env_steps=ro.s, replays=len(lens), launches=launches, alg_bytes=alg,
               bytes_per_env_step=env.bytes_per_env_step(), obs_bytes=ro.obs_bytes, ring_n=ro.ring_n, total_ms=tot)
    return res, ro


def dump_outputs(ro, out_dir, obs_envs=256, envs=65536):
    """Writes what the last timed step returned as float32 ``out_dir/<name>.npy``: ``reward`` / ``clean`` [E, n] and
    ``apple_cnt`` / ``done`` [E] of the envs listed in ``envs`` (all of them up to 65 536), and ``obs`` [S, n, 3, N, N] (u8
    pixel values) of the envs listed in ``obs_envs`` (a fixed sample of 256).  The samples depend on the batch size only;
    at most ~60 MB in all."""
    env = ro.env
    B = env.B

    def pick(cap):
        return np.arange(B) if B <= cap else np.sort(np.random.RandomState(0).choice(B, cap, replace=False))
    e_idx, o_idx = pick(envs), pick(obs_envs)
    ei, oi = (ro.torch.as_tensor(i, device=env.device) for i in (e_idx, o_idx))
    obs = env.obs_view(ro.ring[ro.s % ro.ring_n])             # step t wrote its observations to ring[(t + 1) % ring_n]
    out = {"reward": env.reward[ei], "clean": env.clean[ei], "apple_cnt": env.apple_cnt[ei], "done": env.done[ei],
           "obs": obs[oi], "envs": e_idx, "obs_envs": o_idx}
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        v = v.cpu().numpy() if hasattr(v, "cpu") else v
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(v, dtype=np.float32))


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def auto_replays(a, K):
    """Replays the K timed steps are split into: one per 1000 steps, 1 to 20 (--replays overrides).  A replay ends when
    its slowest env range does, so shorter replays cost time per step: 100-step replays +0.7-0.9% over 1000-step ones at
    4096 envs in 8 ranges (profiles/r3_replay_length.jsonl, B200 at a 1000 W power limit).  Below 2000 steps that leaves one
    replay, which the line's `timing` says."""
    return a.replays if a.replays > 0 else max(1, min(20, K // 1000))


def run_b200(a):
    import torch
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    clk = ClockSampler(local_rank)
    affinity = clk.bind_cpu_affinity() if world > 1 else None

    cfg = workload_config(a, world)
    B, n = cfg["envs_per_gpu"], cfg["num_agents"]
    K, R = a.steps, auto_replays(a, a.steps)
    if a.groups <= 0:                                         # one wave of warps cannot overlap its own logic and store phases
        a.groups = auto_groups(B)
    single = None
    if a.groups > 1:                                          # the same K steps as ONE launch per step, for the record
        r1, ro1 = measure(cfg, a, dev, rank, world, K, a.warmup, max(1, R // 4), groups=1, dist=dist)
        single = {"us_per_step": r1["ms_per_step"] * 1e3, "value": r1["value"],
                  "frac": r1["alg_bytes"] / (r1["ms_per_step"] * 1e-3) / 1e9 / hbm_peak()[0],
                  "what": "same workload, one ssd_step launch per step over the whole batch (--groups 1)"}
        ro1.close()
        del ro1
        torch.cuda.empty_cache()
    res, ro = measure(cfg, a, dev, rank, world, K, a.warmup, R, groups=a.groups, clock=clk, dist=dist)
    if a.dump_outputs and rank == 0:
        dump_outputs(ro, a.dump_outputs)
    env = ro.env
    peak, peak_src = hbm_peak()

    # ---- e2e: the reference-facing call with HOST buffers (H2D actions, D2H results+obs every step)
    io = env.make_host_io(with_obs=True)
    h_actions = ro.actions[:64].cpu()
    e2e_steps = max(1, min(a.e2e_steps, a.steps))
    with torch.cuda.stream(ro.stream):
        for s in range(3):
            io["actions"].copy_(h_actions[s % len(h_actions)])
            env.step_host(io)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(e2e_steps):
            io["actions"].copy_(h_actions[s % len(h_actions)])
            env.step_host(io)
            if bool(io["done"][0]):
                env.reset(obs=False)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t[0])
    obs_bytes = res["obs_bytes"]
    ro.close()
    del ro, io

    # ---- the other BASELINE configs, same method (100-step schedule, 7 timed replays each)
    extra = {}
    if not a.no_extra:
        todo = [(name, None, "weak") for name in EXTRA_N1 if name != a.workload] if world == 1 else \
               [("harvest5_b65536", None, "weak"), ("cleanup10_b16384", "strong", "strong")]
        for name, split, scaling in todo:
            c2 = workload_config(a, world, name=name)
            if split == "strong":                              # configs[2]: 16384 envs in total, contiguous shards by global env id
                from homophily_marl_b200.sharding import shard_range
                lo, hi = shard_range(WORKLOADS[name][4], rank, world)
                c2["envs_per_gpu"], c2["global_envs"], c2["gid_base"] = hi - lo, WORKLOADS[name][4], lo
            try:
                g2 = auto_groups(c2["envs_per_gpu"])
                r2, ro2 = measure(c2, a, dev, rank, world, 7 * LIMIT, 5, 7, groups=g2, dist=dist)
                ro2.close()
                del ro2
                torch.cuda.empty_cache()
                if split == "strong":                          # value was computed as envs_per_gpu * world; shards may differ by one env
                    r2["value"] = c2["global_envs"] * c2["num_agents"] * LIMIT / (r2["replay_ms"]["median"] * 1e-3)
                ach = r2["alg_bytes"] / (r2["ms_per_step"] * 1e-3) / 1e9
                extra[name] = {"value": r2["value"], "us_per_step": r2["ms_per_step"] * 1e3, "frac": ach / peak, "achieved_gbs_per_gpu": ach,
                               "envs_per_gpu": c2["envs_per_gpu"], "global_envs": c2["global_envs"], "scaling": scaling,
                               "env_ranges": g2, "what": WORKLOADS[name][5], "replay_ms": r2["replay_ms"]}
            except Exception as e:
                extra[name] = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        achieved = res["alg_bytes"] / (res["ms_per_step"] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(a.workload, {}).get("dram_bytes_per_launch")
        d2h = B * (2 * n + 2 + 1) + obs_bytes
        line = {"metric": METRIC, "value": res["value"], "unit": "agent-steps/s", "n_gpus": world, "steps": K,
                "timed_steps": res["timed_steps"], "env_steps": res["env_steps"],
                "warmup": max(a.warmup, 3), "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
                "replays": res["replays"], "replay_ms": res["replay_ms"],
                "timing": "the K timed steps as `replays` individually event-timed CUDA-graph replays, after one untimed pass over "
                          "the same schedule; median over replays of time per step, MAX over ranks"
                          + ("; ONE replay: a single sample, min = median = max, no spread" if res["replays"] == 1 else ""),
                "l2": f"obs written round-robin into {res['ring_n']} buffers x {obs_bytes / 2**20:.1f} MiB (> {L2_BYTES >> 20} MiB L2), like an episode buffer",
                "parallelism": f"env-sharded x{world} (no collective on the step path)" + (f", {a.groups} env ranges on {a.groups} streams" if a.groups > 1 else ""),
                "clocks": clk.summary(), "gpu_launches": res["launches"],
                "gpu_launches_how": "ssd_launch_count deltas recorded while each graph was captured, summed over the graphs of the K timed steps",
                "launch_mode": "cuda-graph" if not a.no_graph else "python-loop",
                "e2e": {"value": B * n * world * e2e_steps / (e2e_ms * 1e-3), "unit": "agent-steps/s",
                        "h2d_bytes_per_step": B * n, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                        "what": "ssd_step_host: pinned actions H2D, kernel, reward/clean/apple_cnt/done/obs D2H, stream sync"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "kernel": "ssd_kernel<MODE_STEP>", "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": res["alg_bytes"] // max(a.groups, 1),
                             "launches_per_step": max(a.groups, 1),
                             "achieved_how": "algorithmic bytes of one step over the whole batch / median step time (a step = "
                                             f"{max(a.groups, 1)} concurrent range launch(es))",
                             "bytes_per_env_step": res["bytes_per_env_step"],
                             "avg_launch_us": res["ms_per_step"] * 1e3}}
        if single is not None:
            line["single_launch"] = single
        if affinity:
            line["cpu_affinity"] = f"{len(affinity)} cpus (nvmlDeviceSetCpuAffinity)"
        if extra:
            line["workloads"] = extra
        if world == 1 and not a.no_cpu_baseline:
            threads = os.cpu_count() or 1
            r = time_oracle(cfg, a, steps=20, warmup=3, budget_s=10.0, threads=threads)
            port = {"value": r["value"], "unit": "agent-steps/s", "cores": threads, "kind": "port",
                    "sample": f"{r['envs']} envs x 20 steps of the same workload (C port of the reference env, step+get_obs, OpenMP)"}
            ref = time_python_reference(cfg, a, steps=2000, warmup=50, procs=threads, budget_s=12.0)
            if ref is not None:
                line["cpu_baseline"] = {"value": ref["value"], "unit": "agent-steps/s", "cores": threads, "kind": "reference", "sample": ref["sample"]}
                line["cpu_baseline_port"] = port
                r1 = time_python_reference(cfg, a, steps=1000, warmup=50, procs=1, budget_s=8.0)
                line["cpu_baseline_reference_1core"] = {"value": r1["value"], "unit": "agent-steps/s", "cores": 1, "kind": "reference",
                                                        "sample": r1["sample"] + " -- the reference's only execution mode"}
            else:
                line["cpu_baseline"] = port
        if world == 1 and not a.no_extra:
            try:
                line["frontend"] = frontend_probe(cfg, a, dev)
            except Exception as e:
                line["frontend"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world == 1 and not a.no_train:
            line["train_e2e"] = train_e2e(a)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("bench.py: --dump-outputs writes the outputs of the CUDA arm; it has no meaning with --impl reference")
    sys.exit(run_reference(args) if args.impl == "reference" else run_b200(args))
