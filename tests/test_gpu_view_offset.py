"""GPU suite: forward-offset observation windows (extra_args view_offset, ``ssd_set_view_offset``; DESIGN.md §3 item 18).

After every step the observation buffer, pads included, equals the NumPy restatement (tests/view_offset_ref.py) built from the
handle's own state, and every other buffer equals that of a twin handle with offset 0: on every shipped config in both
observation formats, with and without tagging, at offsets 1, V // 2 and V, under Philox draws and under injected draws with
teleports that put agents on every border facing every way; on the runtime geometry (odd views, V = 31 at f = 31, 16 agents, a
2 048-cell map); through auto-reset, masked reset, ssd_render and ssd_step_host; with variants, episode counters and shaping on;
on 8 env ranges on 8 streams; in a CUDA graph; at 65 536 envs; when the offset is switched between steps; in the batched runner
and the PyMARL facade; and through the fused observation front end."""
import numpy as np
import pytest

import lockstep
from harness import (CUSTOM, STATE, ScriptedMAC, action_tables, assert_same_buffers, custom_params, env_var, make_runner,
                     random_actions, random_draws, random_map)
from obs_index_ref import pack
from view_offset_ref import offset_views, rgb_buffer

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
OTHER = STATE + ("state_buf",)                                  # every buffer the offset must leave alone


def offsets(V):
    return sorted({1, V // 2, V} - {0})


def make(key, B, f, *, obs="rgb", T=0, seed=9, limit=1000, **kw):
    """An SSDBatchEnv of config ``key`` (random spawn point and rotation, want_state) with view_offset f."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    name, mp, n, view, c = lockstep.CONFIGS[key]
    extra = dict(obs_color=c, random_spawn_point=True, random_spawn_rotation=None, tag_timeout=T, obs_format=obs,
                 view_offset=f)
    extra.update(kw.pop("extra", {}))
    return SSDBatchEnv(name, B, n, map=mp, view_size=view, episode_limit=limit, extra_args=extra, seed=seed, want_state=True, **kw)


def make_custom(case, B, f, *, obs="rgb", T=3, seed=9):
    from homophily_marl_b200.batch_env import SSDBatchEnv
    kind, H, W, n, view, color = case
    rows = random_map(np.random.RandomState(H * W + n), kind, H, W, n_spawn=min(32, n + 3))
    extra = dict(random_spawn_point=True, random_spawn_rotation=None, obs_color=color, tag_timeout=T, obs_format=obs,
                 view_offset=f)
    return SSDBatchEnv(kind, B, n, view_size=view, episode_limit=1000, rows=rows, params=custom_params(kind), seed=seed,
                       extra_args=extra, want_state=True)


def set_offset(env, f):
    from homophily_marl_b200 import _capi
    _capi.check(env.lib.ssd_set_view_offset(env._h, f))
    env.view_offset = f


def expected(env, f, envs):
    """The observation bytes of ``envs`` the restatement gives from the env's current state, in the env's format."""
    grid, pos = env.grid.cpu().numpy(), env.agent_pos.cpu().numpy()
    ori, tag = env.agent_orient.cpu().numpy(), env.tag_out.cpu().numpy()
    full = env.extra_args["obs_color"] == "full"
    out = []
    for b in envs:
        idx = offset_views(grid[b], pos[b], ori[b], env.spec.view, f, full, tag[b])
        if env.obs_format == "index4":
            out.append(pack(idx))
        else:
            out.append(rgb_buffer(env.spec.lut, idx, env.layout.obs_row_stride, env.layout.obs_agent_stride))
    return np.stack(out)


def assert_obs(env, what, f=None, buf=None, envs=None):
    f = env.view_offset if f is None else f
    envs = range(env.B) if envs is None else envs
    got = (env.obs_buf if buf is None else buf).cpu().numpy()[list(envs)]
    want = expected(env, f, envs)
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError((what, "obs", "first mismatch", bad[0].tolist(), len(bad), "bytes"))


def teleport(rs, envs):
    """The same teleport on every env of ``envs``: agents onto distinct free cells of the playable area's border ring (row 1,
    row H-2, column 1, column W-2), orientations cycling over all four, so that every border is seen facing every way."""
    e0 = envs[0]
    grid = e0.grid.cpu().numpy()
    H, W, n = e0.H, e0.W, e0.n
    pos = np.zeros((e0.B, n, 2), np.int64)
    for b in range(e0.B):
        free = np.argwhere(grid[b] != 1)
        ring = free[(free[:, 0] == 1) | (free[:, 0] == H - 2) | (free[:, 1] == 1) | (free[:, 1] == W - 2)]
        pick = ring[rs.permutation(len(ring))][:n]
        if len(pick) < n:
            rest = free[rs.permutation(len(free))]
            rest = np.array([p for p in rest if not any((p == q).all() for q in pick)])[:n - len(pick)]
            pick = np.concatenate([pick, rest])
        pos[b] = pick
    orient = (np.arange(e0.B)[:, None] + np.arange(n)[None, :] + rs.randint(4)) % 4
    for e in envs:
        e.load_state(pos_rc=pos, orient=orient)


def run_twins(envs, rs, steps, check, philox=18):
    """Steps the handles of ``envs`` ({f: env}, f = 0 among them) with the same actions: Philox draws first, then injected
    draws with a teleport (and an ssd_render) every third step.  After every step and render every env's observations equal the
    restatement and its other buffers equal the f = 0 twin's."""
    base = envs[0]
    for e in envs.values():
        e.reset()
    check(envs, "reset")
    for t in range(steps):
        at = torch.as_tensor(random_actions(rs, base, fire=0.3, clean=0.2), device=base.device)
        draws = None
        if t >= philox:
            draws = random_draws(rs, base)
            if t % 3 == 0:
                teleport(rs, list(envs.values()))
                for e in envs.values():
                    e.render(want_obs=True, want_state=True)
                check(envs, ("render", t))
        for e in envs.values():
            e.step(at, draws=draws, want_state=True)
        check(envs, t)


def check_all(envs, what):
    for f, e in envs.items():
        assert_obs(e, (f, what))
        if f:
            assert_same_buffers(e, envs[0], OTHER, (f, what))


@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("obs", ["rgb", "index4"])
@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_shipped_configs_match_the_restatement(key, obs, T):
    V = lockstep.CONFIGS[key][3]
    envs = {f: make(key, 16, f, obs=obs, T=T) for f in [0] + offsets(V)}
    rs = np.random.RandomState(10 * sorted(lockstep.CONFIGS).index(key) + T + (obs == "index4"))
    run_twins(envs, rs, 30, check_all)
    for e in envs.values():
        e.close()


@pytest.mark.parametrize("case", CUSTOM)
def test_runtime_geometry(case):
    """Odd views, both gather paths, V = 31 at f = 31, 16 agents and a 2 048-cell map, in both formats; the f = 0 twin runs the
    runtime geometry's own kernels."""
    V = case[4]
    for obs in ("rgb", "index4"):
        envs = {f: make_custom(case, 8, f, obs=obs) for f in [0] + offsets(V)}
        run_twins(envs, np.random.RandomState(case[1] * case[2]), 12, check_all, philox=6)
        for e in envs.values():
            e.close()


def test_largest_tiles_fit_and_bad_offsets_change_nothing():
    """Over every geometry ssd_create accepts, the staging tile is largest on an 8 x 255 map: 149 824 bytes for V = 31 at f >= 27
    (map path) and 37 184 bytes for V = 7 at f = 7 (direct path), both under the 227 KB opt-in limit (profiles/r11_notes.md),
    so every offset 0..V of those geometries is accepted and renders right.  Offsets outside 0..V are refused with the handle
    unchanged."""
    from homophily_marl_b200 import _capi
    for case, fs in ((("harvest", 8, 255, 2, 31, "full"), range(32)), (("cleanup", 8, 255, 2, 7, "full"), range(8)),
                     (("cleanup", 255, 8, 2, 7, "simplified"), (3, 7)), (("harvest", 32, 64, 16, 31, "full"), (16, 31))):
        env = make_custom(case, 4, 0)
        env.reset()
        before = env.obs_buf.clone()
        for f in (-1, case[4] + 1, 1000):
            assert env.lib.ssd_set_view_offset(env._h, f) == _capi.SSD_ERR_INVALID
        env.render()
        assert torch.equal(env.obs_buf, before)
        for f in fs:
            set_offset(env, f)
            env.render()
            assert_obs(env, (case, f))
        env.close()


def test_autoreset_masked_reset_render_and_host_step():
    """ssd_step_autoreset writes the finished step's offset views to end_obs and the new episode's first offset views to obs
    (equal to a step, then a masked reset); a masked reset with obs, ssd_render and ssd_step_host honour the offset too."""
    for key, obs in (("cleanup5_full", "rgb"), ("harvest5", "index4"), ("harvest10_full", "rgb")):
        V = lockstep.CONFIGS[key][3]
        f = V
        fused = make(key, 64, f, obs=obs, T=3, limit=8, keep_episode_end=True)
        seq = make(key, 64, f, obs=obs, T=3, limit=8)
        twin = make(key, 64, 0, obs=obs, T=3, limit=8, keep_episode_end=True)
        rs = np.random.RandomState(6)
        t0 = rs.randint(0, 8, size=64)
        for e in (fused, seq, twin):
            e.reset()
            e.load_state(t=t0)
        ended = 0
        for t in range(20):
            at = torch.as_tensor(random_actions(rs, fused, fire=0.4, clean=0.3), device=fused.device)
            fused.step(at, auto_reset=True, want_state=True)
            twin.step(at, auto_reset=True, want_state=True)
            seq.step(at, want_state=True)
            assert_obs(seq, (key, t, "step"))
            d = seq.done.bool()
            assert torch.equal(fused.end_obs_buf[d], seq.obs_buf[d]), (key, t)
            seq.reset(mask=d)
            assert_obs(seq, (key, t, "masked reset"))
            assert torch.equal(fused.obs_buf, seq.obs_buf), (key, t)
            assert_obs(fused, (key, t, "autoreset"))
            assert_same_buffers(fused, twin, OTHER + ("end_state_buf", "end_ep_ret_buf"), (key, t))
            ended += int(d.sum())
        assert ended > 0
        fused.render(want_obs=True, want_state=True)
        assert_obs(fused, (key, "render"))
        io = fused.make_host_io()
        a = random_actions(rs, fused)
        io["actions"].copy_(torch.as_tensor(a))
        fused.step_host(io)
        assert np.array_equal(io["obs"].numpy(), expected(fused, f, range(64))), key
        assert_obs(fused, (key, "step_host"))
        for e in (fused, seq, twin):
            e.close()


@pytest.mark.parametrize("key", ["cleanup5_full", "harvest5"])
def test_twins_with_variants_counters_and_shaping(key):
    V = lockstep.CONFIGS[key][3]
    var = [{}, {"tag_timeout": 4}, {"fire_cost": 0, "hit_penalty": 1, "reward_shaping": {"beta": 2.0}}]
    kw = dict(T=0, limit=10, keep_episode_end=True, variants=var,
              extra=dict(episode_stats=True, reward_shaping={"alpha": 5.0, "beta": 0.05}))
    envs = {f: make(key, 48, f, **kw) for f in (0, V)}
    rs = np.random.RandomState(12)
    for e in envs.values():
        e.reset()
        e.load_state(t=np.random.RandomState(1).randint(0, 10, size=48))
    keys = OTHER + ("end_state_buf", "end_ep_ret_buf", "stats_buf", "end_stats_buf", "shaped_buf", "shape_trace_buf")
    for t in range(25):
        at = torch.as_tensor(random_actions(rs, envs[0], fire=0.4, clean=0.3), device=envs[0].device)
        for e in envs.values():
            e.step(at, auto_reset=True, want_state=True)
        assert_obs(envs[V], (key, t))
        assert_same_buffers(envs[V], envs[0], keys, (key, t))
    assert envs[V].stats_buf.any() and envs[V].end_obs_buf.any()


@pytest.mark.parametrize("pdl", ["1", "0"])
def test_ranges_on_eight_streams(pdl):
    with env_var("SSD_B200_PDL", pdl):
        whole, parts = make("harvest5", 4096, 7, T=3, limit=10), make("harvest5", 4096, 7, T=3, limit=10)
    streams = [torch.cuda.Stream(device=parts.device) for _ in range(8)]
    rs = np.random.RandomState(3)
    for e in (whole, parts):
        e.reset()
        e.load_state(t=np.random.RandomState(1).randint(0, 10, size=4096))
    torch.cuda.synchronize()
    sample = np.random.RandomState(4).choice(4096, 64, replace=False)
    for t in range(16):
        at = torch.as_tensor(random_actions(rs, whole, fire=0.4), device=whole.device)
        ar = t % 3 == 2
        whole.step(at, auto_reset=ar)
        main = torch.cuda.current_stream(parts.device)
        for k, s in enumerate(streams):
            s.wait_stream(main)
            with torch.cuda.stream(s):
                parts.step_range(at, 512 * k, 512, auto_reset=ar)
        for s in streams:
            main.wait_stream(s)
        assert_same_buffers(whole, parts, OTHER + ("obs_buf",), (pdl, t))
        assert_obs(parts, (pdl, t), envs=sample)


def test_cuda_graph_keeps_its_captured_offset():
    """A graph captured at offset 2 replays offset-2 views after ssd_set_view_offset(5); eager steps then use 5."""
    eager, graphed = make("harvest5", 256, 2, T=3, limit=7), make("harvest5", 256, 2, T=3, limit=7)
    rs = np.random.RandomState(9)
    acts = [torch.as_tensor(random_actions(rs, eager, fire=0.4), device=eager.device) for _ in range(4)]
    for e in (eager, graphed):
        e.reset()
    torch.cuda.synchronize()
    s = torch.cuda.Stream(device=graphed.device)
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        graphed.step(acts[0], auto_reset=True)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            for a in acts:
                graphed.step(a, auto_reset=True)
    eager.step(acts[0], auto_reset=True)
    set_offset(graphed, 5)
    for _ in range(3):
        g.replay()
        for a in acts:
            eager.step(a, auto_reset=True)
    torch.cuda.synchronize()
    assert_same_buffers(eager, graphed, OTHER + ("obs_buf",), "graph")
    assert_obs(graphed, "graph", f=2)
    graphed.step(acts[1])
    eager.step(acts[1])
    assert_obs(graphed, "eager after the graph", f=5)
    assert_same_buffers(eager, graphed, OTHER, "eager after the graph")
    assert not torch.equal(eager.obs_buf, graphed.obs_buf)


def test_65536_envs():
    big, twin = make("cleanup5", 65536, 7, limit=8), make("cleanup5", 65536, 0, limit=8)
    rs = np.random.RandomState(2)
    sample = rs.choice(65536, 128, replace=False)
    for e in (big, twin):
        e.reset()
    for t in range(6):
        at = torch.as_tensor(random_actions(rs, big, fire=0.3, clean=0.3), device=big.device)
        for e in (big, twin):
            e.step(at, auto_reset=True, want_state=True)
        assert_same_buffers(big, twin, OTHER, t)
        assert_obs(big, t, envs=sample)


def test_setting_0_and_switching_offsets():
    """A handle set to 3 and back to 0 is bit-identical to one never set; switching offsets between steps renders each step
    at the offset set before it."""
    never, back = make("harvest5", 64, 0, T=3), make("harvest5", 64, 0, T=3)
    set_offset(back, 3)
    set_offset(back, 0)
    sw = make("harvest5", 64, 0, T=3)
    rs = np.random.RandomState(1)
    for e in (never, back, sw):
        e.reset()
    for t, f in enumerate((1, 0, 15, 7, 0, 2, 15, 1)):
        at = torch.as_tensor(random_actions(rs, never, fire=0.3), device=never.device)
        set_offset(sw, f)
        for e in (never, back, sw):
            e.step(at, want_state=True)
        assert_same_buffers(never, back, OTHER + ("obs_buf",), t)
        assert_same_buffers(never, sw, OTHER, t)
        assert_obs(sw, (t, f))


def test_facade_and_batched_runner():
    """The batched runner with extra_args view_offset fills batch["obs"] with the facade's get_obs() episode for episode, and
    the facade's get_obs() is the restatement of its own state."""
    from homophily_marl_b200 import REGISTRY
    B, T, n, f = 4, 9, 3, 5
    runner = make_runner("cleanup", "default3", n, 7, B=B, T=T, extra=dict(obs_color="full", view_offset=f))
    assert runner.env.view_offset == f
    table, table_inc = action_tables(runner, 2)
    runner.mac = ScriptedMAC(table, table_inc)
    batch = runner.run(test_mode=True)
    A = runner.env.n_actions
    for b in range(B):
        env = REGISTRY["cleanup"](**runner.args.env_args, quiet=True, env_gid_base=b)
        assert env.sim.view_offset == f
        env.reset()
        terminated, t = False, 0
        while True:
            obs = np.stack(env.get_obs())
            want = expected(env.sim, f, [0])[0]
            lay = env.sim.layout
            want = want.reshape(n, lay.obs_agent_stride)[:, :3 * lay.obs_plane_stride].reshape(n, 3, env.sim.N, lay.obs_row_stride)
            assert np.array_equal(obs, want[..., :env.sim.N] / 256), (b, t)
            assert np.array_equal(batch["obs"][b, t].cpu().numpy(), obs.astype(np.float32)), (b, t)
            if terminated:
                break
            _, terminated, _ = env.step((table[b:b + 1, t] % A)[0])
            t += 1
        env.close()


def _module(view, seed):
    torch.manual_seed(seed)
    P = 2 * view - 1
    return torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                               torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU())


@pytest.mark.parametrize("key", ["cleanup5_full", "harvest5"])
def test_fused_front_end_on_offset_views(key):
    """forward_env on offset views is within test_gpu_frontend.py's tolerance of the torch module (1e-6 (1 + |y|) of fp64,
    3e-6 (1 + |y|) of fp32), and forward_env_index4 on the index4 twin gives the same bits."""
    from homophily_marl_b200.frontend import ObsFrontEnd
    V = lockstep.CONFIGS[key][3]
    a, b = make(key, 64, V, T=3), make(key, 64, V, obs="index4", T=3)
    mod = _module(V, seed=21)
    fe = ObsFrontEnd.from_module(mod, V, device=a.device)
    rs = np.random.RandomState(5)
    for e in (a, b):
        e.reset()
    for t in range(6):
        at = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(at)
        b.step(at)
    got = fe.forward_env(a)
    assert torch.equal(fe.forward_env_index4(b), got)
    x = a.obs_view().reshape(-1, 3, a.N, a.N)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            w32 = mod.to(a.device)(x.float() / 256).cpu().double()
            w64 = mod.to("cpu").double()(x.cpu().double() / 256)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    g = got.cpu().double()
    err64 = ((g - w64).abs() / (1 + w64.abs())).max().item()
    err32 = ((g - w32).abs() / (1 + w32.abs())).max().item()
    assert err64 < 1e-6 and err32 < 3e-6, (err64, err32)
    fe.close()


NODES = [f"tests/test_gpu_view_offset.py::{t}" for t in (
    "test_shipped_configs_match_the_restatement[cleanup10_full-rgb-3]",
    "test_shipped_configs_match_the_restatement[cleanup5-index4-0]",
    "test_shipped_configs_match_the_restatement[harvest5-rgb-3]",
    "test_shipped_configs_match_the_restatement[harvest5-index4-0]",
    "test_shipped_configs_match_the_restatement[harvest10_full-index4-3]",
    "test_runtime_geometry", "test_largest_tiles_fit_and_bad_offsets_change_nothing",
    "test_autoreset_masked_reset_render_and_host_step", "test_twins_with_variants_counters_and_shaping",
    "test_ranges_on_eight_streams")]


def test_checked_build_sees_no_shared_memory_violation():
    """The checked library (-DSSD_BOUNDS_CHECK) runs the offset workloads of every mode, gather path, format, tagging and
    variant setting above with no shared-memory index violation (the conftest session fixture asserts the count is 0)."""
    import os
    import subprocess
    import sys
    from homophily_marl_b200 import _build
    _build.build_checked()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "pytest", "-p", "no:cacheprovider", "-q", "-rA", "-m", "gpu"] + NODES, cwd=root,
                       env={**os.environ, "SSD_B200_CHECKED": "1"}, capture_output=True, text=True, timeout=3600)
    print(r.stdout[-20000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    passed = [line.split()[1] for line in r.stdout.splitlines() if line.startswith("PASSED ")]
    for node in NODES:
        assert any(p == node or p.startswith(node + "[") for p in passed), node
