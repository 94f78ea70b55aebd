"""GPU suite: packed colour-index observations (obs_format "index4", SSD_OBS_INDEX4), bit-exact throughout.

The unpacked index equals the NumPy restatement (tests/obs_index_ref.py) applied to the oracle's (or tagging reference's) state
in every shipped configuration, both colour schemes, with and without tagging-out timers, with injected draws and teleports; an
RGB handle and an index4 handle stepped from one seed keep equal state; ``obs_float`` equals the RGB ``obs_view() / 256``; pad
nibbles and bytes are written as 0; and reset, render, env ranges, 65 536 envs, the runtime geometry, ``step_host``,
switching formats, the batched runner and the PyMARL facade all carry the format."""
import numpy as np
import pytest

import lockstep
from harness import (CUSTOM, FIRE, STATE, ScriptedMAC, action_tables, assert_same_buffers, env_var, make_custom_env, make_env,
                     make_ref, make_runner, random_actions)
from obs_index_ref import index_views, obs_layout, ora_index, pack

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def ref_index(env, ora, envs=None):
    full = env.spec.obs_color == "full"
    envs = range(env.B) if envs is None else envs
    return np.stack([ora_index(ora, b, full, ora.tag_out[b] if env.spec.tag_timeout else None) for b in envs])


def state_index(env, envs):
    """The restatement applied to the env's own device state (timers included)."""
    grid, pos, ori, out = (x.cpu().numpy() for x in (env.grid, env.agent_pos, env.agent_orient, env.tag_out))
    full = env.spec.obs_color == "full"
    return np.stack([index_views(grid[b], pos[b], ori[b], env.spec.view, full, out[b]) for b in envs])


def assert_index(env, ora, what, buf=None):
    """Every byte of the buffer (pads included) equals the packed restatement of the reference's state."""
    buf = env.obs_buf if buf is None else buf
    want = ref_index(env, ora)
    assert np.array_equal(env.obs_index(buf).cpu().numpy(), want), (what, "index")
    assert np.array_equal(buf.cpu().numpy(), pack(want)), (what, "packed bytes")


def assert_twins(a, b, what):
    """a: RGB env, b: index4 env stepped with the same inputs."""
    assert_same_buffers(a, b, STATE, what)
    if a.state_rgb is not None:
        assert torch.equal(a.state_rgb, b.state_rgb), (what, "state_rgb")
    assert torch.equal(b.obs_float(), a.obs_view().float() / 256), (what, "obs_float")


def run_lockstep(make, B=32, steps=40):
    """An RGB env, an index4 env and the reference, all from one seed, Philox draws; obs buffers prefilled with 0xFF."""
    a, b = make("rgb"), make("index4")
    ora = make_ref(b)
    a.reset()
    b.obs_buf.fill_(0xFF)
    b.reset()
    ora.reset()
    assert_index(b, ora, "reset")
    assert_twins(a, b, "reset")
    rs = np.random.RandomState(B + steps)
    tagged = 0
    for t in range(steps):
        act = random_actions(rs, b, fire=0.35 if b.spec.tag_timeout else 0)
        at = torch.as_tensor(act, device=b.device)
        b.obs_buf.fill_(0xFF)
        a.step(at, want_state=True)
        b.step(at, want_state=True)
        ora.step(act, want_obs=False, threads=8)
        if b.spec.tag_timeout:
            tagged += int((ora.tag_out > 0).sum())
        assert_index(b, ora, t)
        assert_twins(a, b, t)
        if t % 10 == 9:                                           # ssd_render writes the same bytes
            buf = torch.full_like(b.obs_buf, 0xFF)
            b.render(obs_out=buf, want_obs=True)
            assert_index(b, ora, (t, "render"), buf=buf)
    assert int(ora.envs["error"].sum()) == 0
    a.close()
    b.close()
    return tagged


@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("color", ["simplified", "full"])
@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_every_config_matches_reference(key, color, T):
    tagged = run_lockstep(lambda fmt: make_env(key, 32, obs=fmt, color=color, T=T))
    assert T == 0 or tagged > 0


@pytest.mark.parametrize("key,T", [("cleanup5", 0), ("cleanup10_full", 3), ("harvest5", 0), ("harvest10_full", 3),
                                   ("harvest10_n5", 2), ("cleanup3", 0)])
def test_injected_draws_and_teleports(key, T):
    """One env, every draw injected, teleports (duplicate occupancy included) every 7 steps."""
    a, b = make_env(key, 1, T=T), make_env(key, 1, obs="index4", T=T)
    ora = make_ref(b, seed=0)
    n = b.n
    sched = lockstep.schedule_for(key, seed=200 + T, teleport_every=7)
    rs = np.random.RandomState(T)
    d0 = sched.reset_draws()
    for e in (a, b):
        e.reset(draws=dict(spawn_key=d0["spawn_key"].reshape(1, n, -1), rot=d0["rot"].reshape(1, n)))
    ora.reset_one(0, dict(spawn_key=d0["spawn_key"].reshape(n, -1), rot=d0["rot"]))
    assert_index(b, ora, "reset")
    for t in range(120):
        act, draws, tele = sched.step_inputs(t)
        if T:
            act = np.where(rs.rand(n) < 0.4, FIRE, act).astype(np.uint8)
        rd = sched.reset_draws()
        draws.update(spawn_key=rd["spawn_key"], rot=rd["rot"])
        if tele is not None:
            for e in (a, b):
                e.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
            ora.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
        b.obs_buf.fill_(0xFF)
        for e in (a, b):
            e.step(torch.as_tensor(act.reshape(1, n), device=e.device), draws={k: v.reshape(1, -1) for k, v in draws.items()},
                   want_state=True)
        ora.step_one(act, 0, {k: v.reshape(-1) for k, v in draws.items()})
        assert_index(b, ora, (key, t))
        assert_twins(a, b, (key, t))


def test_layout_strides_every_shipped_geometry():
    import ctypes as C
    from homophily_marl_b200 import _capi
    seen = set()
    for key in sorted(lockstep.CONFIGS):
        e = make_env(key, 2)
        rs_, agent, env_stride = obs_layout(e.N, e.n)
        lay = e.get_obs_layout("index4")
        assert (lay.format, lay.row_stride, lay.plane_stride, lay.agent_stride, lay.env_stride) == (
            _capi.SSD_OBS_INDEX4, rs_, 0, agent, env_stride)
        lay, L = e.get_obs_layout("rgb"), e.layout
        assert (lay.format, lay.row_stride, lay.plane_stride, lay.agent_stride, lay.env_stride) == (
            _capi.SSD_OBS_RGB, L.obs_row_stride, L.obs_plane_stride, L.obs_agent_stride, L.obs_env_stride)
        assert e.obs_layout.env_stride == e.layout.obs_env_stride            # RGB at creation
        lay = _capi.SsdObsLayout()
        assert e.lib.ssd_get_obs_layout(e._h, 2, C.byref(lay)) == _capi.SSD_ERR_INVALID
        assert e.lib.ssd_set_obs_format(e._h, 2) == _capi.SSD_ERR_INVALID
        assert e.lib.ssd_set_obs_format(e._h, -1) == _capi.SSD_ERR_INVALID
        seen.add((e.H, e.W, e.spec.view))
        e.close()
    assert obs_layout(31, 5) == (16, 496, 2480) and obs_layout(15, 5) == (8, 128, 640)
    assert len(seen) == 5
    # algorithmic bytes per env-step (DESIGN.md Roofline)
    want = {("harvest", "default5", 5, 15): (15157, 3222), ("cleanup", "default5", 5, 7): (4333, 1558),
            ("cleanup", "default10", 10, 7): (8591, 3041), ("cleanup", "default3", 3, 7): (2261, 596)}
    from homophily_marl_b200.batch_env import SSDBatchEnv
    for (name, mp, n, view), (rgb, idx) in want.items():
        e = SSDBatchEnv(name, 2, n, map=mp, view_size=view)
        assert e.bytes_per_env_step() == rgb
        e.set_obs_format("index4")
        assert e.bytes_per_env_step() == idx
        e.close()


def test_masked_reset_and_auto_reset_at_scale():
    """4 096 envs, tagging on, over two episodes: auto_reset at the episode end plus masked resets mid-episode."""
    B, T, L = 4096, 4, 30
    b = make_env("cleanup5", B, obs="index4", T=T, seed=21, limit=L)
    ora = make_ref(b)
    b.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(5)
    resets = 0
    for t in range(70):
        act = random_actions(rs, b, fire=0.35)
        b.obs_buf.fill_(0xFF)
        b.step(torch.as_tensor(act, device=b.device), auto_reset=True)
        out = ora.step(act, want_obs=False, threads=8)
        for k in out["done"].nonzero()[0]:
            ora.reset_one(int(k))
        if t % 5 == 0 or out["done"].any():                     # the step's views; first views of the envs just reset
            assert_index(b, ora, t)
        if t % 13 == 6:
            mask = rs.rand(B) < 0.3
            buf = torch.full_like(b.obs_buf, 0xFF)
            b.reset(mask=torch.as_tensor(mask.astype(np.uint8)), obs_out=buf)
            for k in np.flatnonzero(mask):
                ora.reset_one(int(k))
            sel = np.flatnonzero(mask)
            got = buf.cpu().numpy()[sel]
            assert np.array_equal(got, pack(ref_index(b, ora, sel))), (t, "masked reset")
            assert (buf.cpu().numpy()[~mask] == 0xFF).all()               # envs not reset are not written
            resets += len(sel)
    assert resets > 0


def test_env_ranges_on_streams_equal_one_launch():
    B, G = 4096, 8
    a = make_env("harvest5", B, obs="index4", T=3, seed=4)
    b = make_env("harvest5", B, obs="index4", T=3, seed=4)
    a.reset()
    b.reset()
    rs = np.random.RandomState(8)
    streams = [torch.cuda.Stream(device=b.device) for _ in range(G)]
    obs_b = b.new_obs_buffer()
    fl = torch.empty((B, b.n, 3, b.N, b.N), dtype=torch.float32, device=b.device)
    for t in range(30):
        act = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(act)
        cur = torch.cuda.current_stream(b.device)
        for g, s in enumerate(streams):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                b.step_range(act, g * (B // G), B // G, obs_out=obs_b)
                b.obs_float(g * (B // G), B // G, buf=obs_b, out=fl[g * (B // G):(g + 1) * (B // G)])
        for s in streams:
            cur.wait_stream(s)
        torch.cuda.synchronize()
        assert_same_buffers(a, b, STATE, t)
        assert torch.equal(a.obs_buf, obs_b), t
        assert torch.equal(a.obs_float(), fl), t


def test_harvest_65536_envs_sampled():
    B = 65536
    a = make_env("harvest5", B, seed=13)
    b = make_env("harvest5", B, obs="index4", seed=13)
    a.reset()
    b.reset()
    rs = np.random.RandomState(2)
    sample = np.sort(rs.choice(B, 64, replace=False))
    st = torch.as_tensor(sample, device=b.device)
    before = b.launch_count
    for t in range(6):
        act = torch.as_tensor(random_actions(rs, a), device=a.device)
        a.step(act)
        b.obs_buf.fill_(0xFF)
        b.step(act)
        assert_same_buffers(a, b, STATE, t)
        got = b.obs_buf[st].cpu().numpy()
        assert np.array_equal(got, pack(state_index(b, sample))), t
        for lo in (0, int(sample[10]), B - 7):
            cnt = min(7, B - lo)
            assert torch.equal(b.obs_float(lo, cnt), a.obs_view()[lo:lo + cnt].float() / 256), (t, lo)
    assert b.launch_count - before == 6 + 6 * 3                       # one step and three expansions per iteration


def test_step_host_copies_the_index4_buffer():
    b = make_env("harvest5", 64, obs="index4", seed=3)
    io = b.make_host_io(with_obs=True, with_state=True)
    assert io["obs"].shape == (64, b.obs_layout.env_stride)
    b.reset()
    rs = np.random.RandomState(1)
    for t in range(5):
        io["actions"].copy_(torch.as_tensor(random_actions(rs, b)))
        io["obs"].fill_(0xEE)
        b.step_host(io)
        assert torch.equal(io["obs"], b.obs_buf.cpu()), t
        assert np.array_equal(io["obs"].numpy(), pack(state_index(b, range(64)))), t


def test_switching_format_mid_episode():
    a = make_env("cleanup10_full", 16, T=2, seed=6)
    b = make_env("cleanup10_full", 16, obs="index4", T=2, seed=6)
    a.reset()
    b.reset()
    rs = np.random.RandomState(4)
    for t in range(24):
        if t == 8:
            a.set_obs_format("index4")
            b.set_obs_format("rgb")
        if t == 16:
            a.set_obs_format("rgb")
            b.set_obs_format("index4")
        act = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(act)
        b.step(act)
        rgb, idx = (b, a) if 8 <= t < 16 else (a, b)
        assert_twins(rgb, idx, t)
        assert np.array_equal(idx.obs_index().cpu().numpy(), state_index(idx, range(16))), t
    with pytest.raises(ValueError):
        b.obs_view()
    with pytest.raises(ValueError):
        a.obs_float()
    with pytest.raises(ValueError):
        a.set_obs_format("rgb8")


@pytest.mark.parametrize("case", CUSTOM, ids=lambda c: "%s_%dx%d_n%d_v%d" % c[:5])
def test_runtime_geometry_custom_maps(case):
    assert run_lockstep(lambda fmt: make_custom_env(case, 16, obs=fmt, T=2), B=16, steps=25) > 0


def test_runtime_geometry_on_shipped_maps():
    """SSD_B200_GENERIC=1: the GeoD index4 instantiations on the shipped maps."""
    for key in ("cleanup5", "harvest5", "harvest10_full"):
        for T in (0, 3):
            with env_var("SSD_B200_GENERIC", "1"):
                run_lockstep(lambda fmt, key=key, T=T: make_env(key, 16, obs=fmt, T=T), B=16, steps=20)


@pytest.mark.parametrize("groups", [1, 3])
def test_batched_runner_fills_the_same_batch(groups):
    batches = {}
    for fmt in ("rgb", "index4"):
        runner = make_runner(groups=groups, extra=dict(obs_color="full", tag_timeout=2, obs_format=fmt))
        runner.mac = ScriptedMAC(*action_tables(runner, 0, high=2 * runner.env.n_actions))
        batches[fmt] = runner.run(test_mode=True)
        runner.close_env()
    a, b = batches["rgb"], batches["index4"]
    for k in a.data:
        assert torch.equal(a.data[k], b.data[k]), k
    assert a.data["obs"].abs().sum() > 0


def test_batched_runner_refuses_fused_frontend_with_index4():
    runner = make_runner(extra=dict(obs_color="full", tag_timeout=2, obs_format="index4"), fused_frontend=True, rgb_input=True)
    mac = ScriptedMAC(*action_tables(runner, 0, high=2 * runner.env.n_actions))
    with pytest.raises(ValueError, match="index4"):
        runner.setup(None, None, None, mac, batch_cls=lambda *a, **k: None)
    runner.close_env()


def test_pymarl_facade_get_obs_stays_rgb():
    from homophily_marl_b200 import REGISTRY
    kw = dict(num_agents=5, map="default5", view_size=15, episode_limit=30, seed=3, quiet=True)
    plain = REGISTRY["harvest"](extra_args=dict(disable_fire_action=False), **kw)
    keyed = REGISTRY["harvest"](extra_args=dict(disable_fire_action=False, obs_format="index4"), **kw)
    assert keyed.sim.obs_format == "rgb"
    plain.reset()
    keyed.reset()
    rs = np.random.RandomState(0)
    for t in range(30):
        acts = rs.randint(0, 8, size=5)
        r1, d1, _ = plain.step(acts)
        r2, d2, _ = keyed.step(acts)
        assert np.array_equal(r1, r2) and d1 == d2
        for x, y in zip(plain.get_obs(), keyed.get_obs()):
            assert np.array_equal(x, y), t
    plain.close()
    keyed.close()
