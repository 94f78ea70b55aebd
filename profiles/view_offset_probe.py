"""Cost of forward-offset observation windows (extra_args view_offset): time per step at offsets 0, V // 2 and V, same process,
alternating.

Workloads: Harvest default5 (V = 15, nibble-map gather) and Cleanup default5 (V = 7, direct gather), each at 4 096 envs in 8 env
ranges of 512 on 8 streams (programmatic dependent launch) and at 65 536 envs (one launch per step); RGB observations,
tag_timeout 0, uniform random actions over every action.  Four handles per workload:
  - offset 0 on the shipped (compile-time geometry) kernels, what every user without the option runs;
  - offset 0 with SSD_B200_GENERIC=1, the runtime-geometry kernels: the like-for-like baseline of the offset kernels, which
    also run on runtime geometry values;
  - offset V // 2 and offset V (the offset kernels).
Each handle is a CUDA graph of K steps writing into a ring of observation buffers larger than twice the 126 MB L2 (no state
image, as in bench.py); replays are timed with CUDA events, the four handles in rotating order replay by replay after two
warm-up rounds.  One JSON line per (workload, handle), with the card name and power limit read in the same run and the handle's
dynamic shared memory per CTA (tile_bytes, restating make_geo in ssd_b200.cu).

    python profiles/view_offset_probe.py [--out FILE.jsonl] [--steps K] [--replays R]
    python profiles/view_offset_probe.py --tiles     # no GPU: the largest staging tile over every geometry ssd_create accepts
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

WORKLOADS = [("harvest5_b4096_g8", "harvest", "default5", 5, 15, 4096, 8),      # name, env, map, n, view, envs, ranges
             ("harvest5_b65536", "harvest", "default5", 5, 15, 65536, 1),
             ("cleanup5_b4096_g8", "cleanup", "default5", 5, 7, 4096, 8),
             ("cleanup5_b65536", "cleanup", "default5", 5, 7, 65536, 1)]
L2_BYTES = 126 * 2 ** 20
KWARPS = 4                                                     # env instances (warps) per CTA
OPTIN = 227 * 1024                                             # opt-in shared memory per block on sm_100


def ru(v, m):
    return (v + m - 1) // m * m


def tile_bytes(H, W, V, f):
    """(PMS, dynamic shared memory per CTA) of make_geo(kind, H, W, V, f): four staging tiles."""
    N = 2 * V + 1
    LPn, nw8M, nw8T = ru(V + f, 8), (W + 7) // 8, (H + 7) // 8
    wm = max((LPn + W + V + f + 7) // 8, LPn // 8 + nw8M)
    wm += wm % 2 == 0
    wt = max((LPn + H + V + f + 7) // 8, LPn // 8 + nw8T)
    wt += wt % 2 == 0
    pms = ru((W + 2 * V) * 4 * wt, 16) + 16 + ru((H + 2 * V) * 4 * wm, 16) + 16 + 32
    direct = ru(N, 4) <= 16
    padF = ru((V + f) * W + 48, 16) if direct else 16
    padB = ru((V + f) * W + 32, 16) if direct else 32
    if direct:
        pms = 0
    return pms, KWARPS * (padF + ru(H * W, 16) + padB + pms)


def tiles():
    """The largest tile over H, W in 3..255 with H * W <= 2048, V in 1..31, f in 0..V, per gather path."""
    best = {}
    for V in range(1, 32):
        path = "direct" if ru(2 * V + 1, 4) <= 16 else "map"
        for H in range(3, 256):
            for W in range(3, min(255, 2048 // H) + 1):
                for f in range(V + 1):
                    pms, t = tile_bytes(H, W, V, f)
                    key = (path, f > 0)
                    if t > best.get(key, (0,))[0]:
                        best[key] = (t, pms, H, W, V, f)
    for (path, off), (t, pms, H, W, V, f) in sorted(best.items()):
        print(json.dumps(dict(path=path, offset_gt_0=off, tile_bytes_per_cta=t, with_colour_luts=t + 256, PMS=pms, H=H, W=W, V=V,
                              f=f, optin=OPTIN, fits=t + 256 <= OPTIN and pms < 60000)))


def card(torch):
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
    ap.add_argument("--replays", type=int, default=10, help="timed replays per handle")
    ap.add_argument("--tiles", action="store_true", help="print the largest staging tiles (no GPU) and exit")
    a = ap.parse_args()
    if a.tiles:
        return tiles()
    import torch
    from homophily_marl_b200.batch_env import SSDBatchEnv
    if not torch.cuda.is_available():
        raise SystemExit("view_offset_probe needs a CUDA device")
    name, smi = card(torch)
    dev = torch.device("cuda:0")

    class Handle:
        def __init__(self, wl, label, f, generic, K, seed=1):
            _, env_name, mp, n, view, B, groups = wl
            self.label, self.f, self.K, self.groups = label, f, K, groups
            old = os.environ.get("SSD_B200_GENERIC")
            os.environ["SSD_B200_GENERIC"] = "1" if generic else "0"          # read by ssd_create
            try:
                self.env = SSDBatchEnv(env_name, B, n, map=mp, view_size=view, episode_limit=10 ** 4, seed=seed, device=dev,
                                       extra_args=dict(disable_fire_action=False, disable_rotation_action=False, view_offset=f))
            finally:
                if old is None:
                    del os.environ["SSD_B200_GENERIC"]
                else:
                    os.environ["SSD_B200_GENERIC"] = old
            e = self.env
            self.smem = tile_bytes(e.H, e.W, view, f)[1]
            g = torch.Generator(device=dev).manual_seed(seed)
            self.actions = torch.randint(0, e.n_actions, (K, B, n), generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
            ring = max(2, -(-2 * L2_BYTES // (B * e.obs_layout.env_stride)))
            self.ring = [e.new_obs_buffer() for _ in range(ring)]
            self.stream = torch.cuda.Stream(device=dev)
            self.gstreams = [torch.cuda.Stream(device=dev) for _ in range(groups)]
            e.reset()
            torch.cuda.synchronize()

        def run(self):
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
                self.run()
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

    lines = []
    for wl in WORKLOADS:
        V = wl[4]
        hs = [Handle(wl, "shipped_f0", 0, False, a.steps), Handle(wl, "generic_f0", 0, True, a.steps),
              Handle(wl, f"offset_f{V // 2}", V // 2, False, a.steps), Handle(wl, f"offset_f{V}", V, False, a.steps)]
        for h in hs:
            h.capture()
        times = {h.label: [] for h in hs}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for r in range(a.replays + 2):                         # the first two rounds are warm-up
            for h in hs[r % 4:] + hs[:r % 4]:
                dt = h.time_graph(ev)
                if r >= 2:
                    times[h.label].append(dt)
        med = {}
        for h in hs:
            ts = sorted(times[h.label])
            med[h.label] = ts[len(ts) // 2]
            rec = dict(probe="view_offset_probe", workload=wl[0], envs=wl[5], env_ranges=wl[6], view=V, handle=h.label,
                       view_offset=h.f, dynamic_smem_bytes_per_cta=h.smem, obs_ring_buffers=len(h.ring), steps_per_replay=a.steps,
                       replays=len(ts), us_per_step_median=ts[len(ts) // 2], us_per_step_min=ts[0], us_per_step_max=ts[-1],
                       gpu=name, nvidia_smi_name_power_limit_max_sm_clock=smi)
            if h.label != "shipped_f0":
                rec["over_shipped_f0"] = med[h.label] / med["shipped_f0"]
                rec["over_generic_f0"] = med[h.label] / med["generic_f0"]
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        for h in hs:
            h.graph = None
            h.env.close()
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
