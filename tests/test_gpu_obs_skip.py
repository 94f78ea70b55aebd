"""GPU suite: tracked observation buffers (row masks, ssd_set_obs_mask; DESIGN.md §3 item 19) hold exactly the bytes of untracked ones.

Every test runs two envs with the same seed and actions: one writes into buffers from ``new_obs_buffer()`` (tracked: rows that are
zero now and were zero at the buffer's last write are not stored), its twin into plain ``torch.zeros`` buffers.  Every slot is
compared byte for byte after every launch, and every mask is checked against its buffer: a clear bit must cover an all-zero row."""
import gc
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import lockstep
from harness import env_var, make_env, random_actions

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def plain(env):
    return torch.zeros((env.B, env.obs_layout.env_stride), dtype=torch.uint8, device=env.device)


def check_mask(env, buf, what):
    """Every row whose bit is clear is all zero in ``buf``."""
    mask = env.obs_mask(buf)
    assert mask is not None, what
    B, n, N = env.B, env.n, env.N
    rows = env.obs_view(buf).reshape(B, n, 3, N, N).permute(0, 2, 1, 3, 4).reshape(B, 3, n * N, N)
    nz = (rows != 0).any(-1).cpu().numpy()                                    # [B, plane, u]
    m = mask.cpu().numpy().view(np.uint32).reshape(B, -1, 3)                  # [B, trip, plane]
    u = np.arange(n * N)
    bits = (m[:, u >> 5, :] >> (u & 31)[None, :, None]) & 1                  # [B, u, plane]
    assert not (nz & (bits.transpose(0, 2, 1) == 0)).any(), what


class Twins:
    """A tracked env / ring and its untracked twin, stepped alike."""

    def __init__(self, key, B, ring, mk=None, **kw):
        mk = mk or (lambda: make_env(key, B, **kw))
        self.a, self.b = mk(), mk()
        assert self.a.obs_mask_words > 0
        self.ra = [self.a.new_obs_buffer() for _ in range(ring)]
        self.rb = [plain(self.b) for _ in range(ring)]
        assert all(self.a.obs_mask(x) is not None for x in self.ra) and all(self.b.obs_mask(x) is None for x in self.rb)

    def both(self, fn):
        fn(self.a, self.ra)
        fn(self.b, self.rb)

    def compare(self, what):
        for i, (x, y) in enumerate(zip(self.ra, self.rb)):
            assert torch.equal(x, y), (what, i)
            check_mask(self.a, x, (what, i))
        for k in ("reward", "done", "grid_buf", "agent_buf", "t_buf", "tick_buf"):
            assert torch.equal(getattr(self.a, k), getattr(self.b, k)), (what, k)


@pytest.mark.parametrize("ring", [1, 2, 5])
def test_ring_with_whole_and_masked_resets(ring):
    tw = Twins("harvest5", 256, ring, T=3, seed=5)
    rs = np.random.RandomState(ring)
    tw.both(lambda e, r: e.reset(obs_out=r[0]))
    tw.compare("reset")
    for t in range(40):
        act = torch.as_tensor(random_actions(rs, tw.a, fire=0.3), device=tw.a.device)
        slot = (t + 1) % ring
        tw.both(lambda e, r: e.step(act, obs_out=r[slot]))
        tw.compare(("step", t))
        if t % 13 == 12:
            mask = torch.as_tensor(rs.rand(256) < 0.5, device=tw.a.device)
            tw.both(lambda e, r: e.reset(mask=mask, obs_out=r[slot]))
            tw.compare(("masked reset", t))
        if t == 25:
            tw.both(lambda e, r: e.reset(obs_out=r[slot]))
            tw.compare(("reset", t))
        if t % 10 == 4:
            tw.both(lambda e, r: e.render(obs_out=r[(slot + 1) % ring]))
            tw.compare(("render", t))


@pytest.mark.parametrize("generic", [False, True])
def test_bench_schedule_in_a_cuda_graph(generic):
    """The benchmark's schedule: per-range masked resets and 8 step_range chains on 8 streams, captured in one CUDA graph."""
    B, G, R, K, LIMIT = 1024, 8, 5, 12, 10
    Bg = B // G
    with env_var("SSD_B200_GENERIC", "1" if generic else "0"):
        tw = Twins("harvest5", B, R, limit=LIMIT, seed=7, random_spawn=False)
    rs = np.random.RandomState(2)
    acts = [torch.as_tensor(random_actions(rs, tw.a), device=tw.a.device) for _ in range(LIMIT)]
    gmask = [(torch.arange(B, device=tw.a.device) // Bg == g).to(torch.uint8) for g in range(G)]
    streams = [torch.cuda.Stream(device=tw.a.device) for _ in range(G)]

    def schedule(e, ring, t0):
        cur = torch.cuda.current_stream(e.device)
        for g, s in enumerate(streams):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                for t in range(t0, t0 + K):
                    if t % LIMIT == 0:
                        e.reset(mask=gmask[g], obs_out=ring[t % R])
                    e.step_range(acts[t % LIMIT], g * Bg, Bg, obs_out=ring[(t + 1) % R])
        for s in streams:
            cur.wait_stream(s)

    graphs = {}
    for e, ring in ((tw.a, tw.ra), (tw.b, tw.rb)):
        torch.cuda.synchronize()
        side = torch.cuda.Stream(device=e.device)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=side):
            schedule(e, ring, 0)
        graphs[id(e)] = gr
    for rep in range(3):
        graphs[id(tw.a)].replay()
        graphs[id(tw.b)].replay()
        torch.cuda.synchronize()
        tw.compare(("replay", rep))
    for rep in range(2):                                   # the same schedule launched live
        tw.both(lambda e, r: schedule(e, r, rep * K))
        torch.cuda.synchronize()
        tw.compare(("live", rep))


@pytest.mark.parametrize("color", ["simplified", "full"])
def test_autoreset_with_episode_end_buffers(color):
    tw = Twins("harvest5", 256, 3, T=3, seed=11, limit=7, color=color, keep_episode_end=True)
    tw.a.end_obs_buf = tw.a.new_obs_buffer()              # track the episode-end buffer too
    assert tw.a.obs_mask(tw.a.end_obs_buf) is not None and tw.b.obs_mask(tw.b.end_obs_buf) is None
    rs = np.random.RandomState(4)
    tw.both(lambda e, r: e.reset(obs_out=r[0]))
    ended = 0
    for t in range(30):
        act = torch.as_tensor(random_actions(rs, tw.a, fire=0.3), device=tw.a.device)
        tw.both(lambda e, r: e.step_range(act, 0, 128, obs_out=r[(t + 1) % 3], auto_reset=True))
        tw.both(lambda e, r: e.step_range(act, 128, 128, obs_out=r[(t + 1) % 3], auto_reset=True))
        tw.compare(("autoreset", t))
        assert torch.equal(tw.a.end_obs_buf, tw.b.end_obs_buf), t
        check_mask(tw.a, tw.a.end_obs_buf, ("end", t))
        ended += int(tw.a.done.sum())
    assert ended > 0


@pytest.mark.parametrize("case", ["offset", "variants", "full_colour_tagging"])
def test_view_offset_variants_and_full_colour(case):
    """Offset windows (their own kernels), per-env variants, and the full-colour repaint with tagging and random spawn."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B = 256
    if case == "offset":
        name, mp, n, view, c = lockstep.CONFIGS["harvest5"]
        extra = dict(obs_color=c, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=3, view_offset=6)
        tw = Twins(None, B, 3, mk=lambda: SSDBatchEnv(name, B, n, map=mp, view_size=view, seed=13, extra_args=extra))
    elif case == "variants":
        tw = Twins("harvest5", B, 3, T=3, seed=13,
                   variants=[{}, {"tag_timeout": 0, "fire_cost": 2}, {"spawn_prob": [0.0, 0.005, 0.02, 0.05]}])
    else:
        tw = Twins("harvest5", B, 3, T=3, seed=13, color="full")
    rs = np.random.RandomState(6)
    tw.both(lambda e, r: e.reset(obs_out=r[0]))
    for t in range(30):
        act = torch.as_tensor(random_actions(rs, tw.a, fire=0.3), device=tw.a.device)
        tw.both(lambda e, r: e.step(act, obs_out=r[(t + 1) % 3]))
        tw.compare((case, t))


def test_caller_writes_then_marks_dirty():
    tw = Twins("harvest5", 128, 2, seed=3)
    rs = np.random.RandomState(1)
    tw.both(lambda e, r: e.reset(obs_out=r[0]))
    for t in range(6):
        act = torch.as_tensor(random_actions(rs, tw.a), device=tw.a.device)
        if t == 3:                                         # the caller scribbles over both slots of the tracked ring
            for x in tw.ra:
                x.fill_(0x5A)
                tw.a.mark_obs_dirty(x)
            for x in tw.rb:
                x.fill_(0x5A)
            assert all(bool((tw.a.obs_mask(x) == -1).all()) for x in tw.ra)
        tw.both(lambda e, r: e.step(act, obs_out=r[t % 2]))
        tw.both(lambda e, r: e.step(act, obs_out=r[(t + 1) % 2]))
        tw.compare(("dirty", t))
    # a launch into a view of a tracked buffer (same address, fewer bytes) stores every row and marks the buffer dirty
    half = tw.a.B // 2
    tw.a.render(obs_out=tw.ra[0][:half])
    tw.b.render(obs_out=tw.rb[0][:half])
    assert bool((tw.a.obs_mask(tw.ra[0]) == -1).all())
    tw.compare("view")


def test_freed_buffer_address_reused_by_a_plain_tensor():
    tw = Twins("harvest5", 128, 1, seed=8)
    rs = np.random.RandomState(9)
    env = tw.a
    buf = env.new_obs_buffer()
    env.reset(obs_out=buf)
    tw.b.reset(obs_out=tw.rb[0])
    ptr = buf.data_ptr()
    assert ptr in env._obs_masks
    del buf
    gc.collect()
    assert ptr not in env._obs_masks
    held = []                                              # allocate until the caching allocator hands the block out again
    for _ in range(16):
        held.append(torch.full((env.B, env.obs_layout.env_stride), 0x77, dtype=torch.uint8, device=env.device))
        if held[-1].data_ptr() == ptr:
            break
    other = held[-1]
    if other.data_ptr() != ptr:
        pytest.skip("the caching allocator did not hand the freed block out again")
    assert env.obs_mask(other) is None
    act = torch.as_tensor(random_actions(rs, env), device=env.device)
    env.step(act, obs_out=other)
    tw.b.step(act, obs_out=tw.rb[0])
    assert torch.equal(other, tw.rb[0])


def test_untracked_geometries_keep_full_stores():
    """Cleanup (direct gather), Harvest view 7 and index4 have no row masks."""
    for key, obs in (("cleanup5", "rgb"), ("harvest10_full", "rgb"), ("harvest5", "index4")):
        e = make_env(key, 8, obs=obs)
        assert e.obs_mask_words == 0, key
        assert e.obs_mask(e.new_obs_buffer()) is None, key
    e = make_env("harvest5", 8)
    assert e.obs_mask_words == 3 * ((5 * 31 + 31) // 32)
    e.set_obs_format("index4")
    assert e.obs_mask_words == 0 and e.obs_mask(e.new_obs_buffer()) is None


def test_checked_build_finds_no_non_zero_skipped_row():
    """On the checked build every skipped row is read back; a non-zero one would be counted by ssd_debug_oob_count."""
    if os.environ.get("SSD_B200_CHECKED") == "1":
        pytest.skip("already running on the checked build")
    from homophily_marl_b200 import _build
    _build.build_checked()
    nodes = [f"tests/test_gpu_obs_skip.py::{n}" for n in (
        "test_ring_with_whole_and_masked_resets", "test_bench_schedule_in_a_cuda_graph",
        "test_autoreset_with_episode_end_buffers", "test_view_offset_variants_and_full_colour",
        "test_caller_writes_then_marks_dirty")]
    r = subprocess.run([sys.executable, "-m", "pytest", "-p", "no:cacheprovider", "-q", "-rA", "-m", "gpu"] + nodes, cwd=ROOT,
                       env={**os.environ, "SSD_B200_CHECKED": "1"}, capture_output=True, text=True, timeout=3600)
    print(r.stdout[-8000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert " passed" in r.stdout and " failed" not in r.stdout
