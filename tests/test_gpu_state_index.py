"""GPU suite: packed colour-index state images (state_format "index4", ssd_set_state_format(h, SSD_OBS_INDEX4)), bit-exact.

Four envs -- RGB and index4 observations, each with an RGB and an index4 state image -- are stepped in lockstep from one seed.
In every shipped configuration, both colour schemes, with and without tagging-out timers, with injected draws and teleports:
``lut[unpack(state)]`` is the RGB state image byte for byte, the packed bytes (pads included, buffers pre-filled with 0xFF)
equal the NumPy restatement (tests/state_index_ref.py) of the reference's state, and ``state_float`` equals
``state_rgb.float() / 256``.  Also covered: ssd_render, env ranges on streams, 65 536 envs, the runtime geometry, ``step_host``,
switching formats, ``auto_reset`` and the batched runner's ``batch["state"]``."""
import numpy as np
import pytest

import harness
import lockstep
from harness import (COMBOS, FIRE, STATE, ScriptedMAC, action_tables, assert_same_buffers, env_var, make_custom_env, make_env,
                     make_ref, make_runner, random_actions)
from state_index_ref import index_state, ora_state, pack, rgb_of, state_layout, unpack

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def ref_state(env, ora, envs=None):
    full = env.spec.obs_color == "full"
    envs = range(env.B) if envs is None else envs
    return np.stack([ora_state(ora, b, full, ora.tag_out[b] if env.spec.tag_timeout else None) for b in envs])


def device_state(env, envs):
    """The restatement applied to the env's own device state (timers included)."""
    grid, pos, out = (x.cpu().numpy() for x in (env.grid, env.agent_pos, env.tag_out))
    full = env.spec.obs_color == "full"
    return np.stack([index_state(grid[b], pos[b], full, out[b]) for b in envs])


def check_quad(envs, what, ora=None, with_float=True):
    """envs: {(obs, state): env} stepped with the same inputs; index4 state buffers were pre-filled with 0xFF."""
    base = envs[("rgb", "rgb")]
    for e in envs.values():
        assert_same_buffers(base, e, STATE, what)
    for obs in ("rgb", "index4"):
        a, b = envs[(obs, "rgb")], envs[(obs, "index4")]
        assert b.state_rgb is None and b.state_buf.shape == (b.B, b.state_layout.env_stride)
        got = b.state_buf.cpu().numpy()
        want = ref_state(b, ora) if ora is not None else device_state(b, range(b.B))
        assert np.array_equal(got, pack(want)), (what, obs, "packed bytes")               # pads are 0 too
        assert np.array_equal(rgb_of(b.spec.lut, unpack(got, b.H, b.W)), a.state_rgb.cpu().numpy()), (what, obs, "lut")
        assert torch.equal(b.state_index().cpu(), torch.as_tensor(want)), (what, obs, "state_index")
        assert torch.equal(a.state_rgb, base.state_rgb), (what, obs, "rgb state")
        if with_float:
            assert torch.equal(b.state_float(), a.state_rgb.float() / 256), (what, obs, "state_float")


def fill_state(envs):
    for (_, s), e in envs.items():
        if s == "index4":
            e.state_buf.fill_(0xFF)


def run_lockstep(make, B=32, steps=40):
    """Four envs and the reference, all from one seed, Philox draws."""
    envs = {c: make(*c) for c in COMBOS}
    any_env = envs[("rgb", "index4")]
    ora = make_ref(any_env)
    for e in envs.values():
        e.reset()
    ora.reset()
    fill_state(envs)
    for e in envs.values():                                    # the state image of the fresh episodes
        e.render(want_obs=False, want_state=True)
    check_quad(envs, "reset", ora)
    rs = np.random.RandomState(B + steps)
    tagged = 0
    for t in range(steps):
        act = random_actions(rs, any_env, fire=0.35 if any_env.spec.tag_timeout else 0)
        at = torch.as_tensor(act, device=any_env.device)
        fill_state(envs)
        for e in envs.values():
            e.step(at, want_state=True)
        ora.step(act, want_obs=False, threads=8)
        if any_env.spec.tag_timeout:
            tagged += int((ora.tag_out > 0).sum())
        check_quad(envs, t, ora, with_float=t % 4 == 0)
        if t % 10 == 9:                                           # ssd_render writes the same bytes, obs or not
            fill_state(envs)
            for (o, s), e in envs.items():
                e.render(want_obs=o == "index4", want_state=True)
            check_quad(envs, (t, "render"), ora, with_float=False)
    assert int(ora.envs["error"].sum()) == 0
    for e in envs.values():
        e.close()
    return tagged


@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("color", ["simplified", "full"])
@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_every_config_matches_reference(key, color, T):
    tagged = run_lockstep(lambda o, s: make_env(key, 32, obs=o, state=s, color=color, T=T))
    assert T == 0 or tagged > 0


@pytest.mark.parametrize("key,T", [("cleanup5", 0), ("cleanup10_full", 3), ("harvest5", 0), ("harvest10_full", 3),
                                   ("harvest10_n5", 2), ("cleanup3", 0)])
def test_injected_draws_and_teleports(key, T):
    """One env, every draw injected, teleports (duplicate occupancy included) every 7 steps."""
    envs = {(o, s): make_env(key, 1, obs=o, state=s, T=T) for o, s in COMBOS}
    b = envs[("rgb", "index4")]
    ora = make_ref(b, seed=0)
    n = b.n
    sched = lockstep.schedule_for(key, seed=300 + T, teleport_every=7)
    rs = np.random.RandomState(T + 1)
    d0 = sched.reset_draws()
    for e in envs.values():
        e.reset(draws=dict(spawn_key=d0["spawn_key"].reshape(1, n, -1), rot=d0["rot"].reshape(1, n)))
    ora.reset_one(0, dict(spawn_key=d0["spawn_key"].reshape(n, -1), rot=d0["rot"]))
    teleports = 0
    for t in range(120):
        act, draws, tele = sched.step_inputs(t)
        if T:
            act = np.where(rs.rand(n) < 0.4, FIRE, act).astype(np.uint8)
        rd = sched.reset_draws()
        draws.update(spawn_key=rd["spawn_key"], rot=rd["rot"])
        if tele is not None:
            teleports += 1
            for e in envs.values():
                e.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
            ora.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
        fill_state(envs)
        for e in envs.values():
            e.step(torch.as_tensor(act.reshape(1, n), device=e.device), draws={k: v.reshape(1, -1) for k, v in draws.items()},
                   want_state=True)
        ora.step_one(act, 0, {k: v.reshape(-1) for k, v in draws.items()})
        check_quad(envs, (key, t), ora)
        assert np.array_equal(envs[("rgb", "rgb")].state_rgb[0].cpu().numpy(), ora.state_one(0)), (key, t)
    assert teleports > 0


def test_layout_strides_every_shipped_geometry():
    import ctypes as C
    from homophily_marl_b200 import _capi
    seen = {}
    for key in sorted(lockstep.CONFIGS):
        e = make_env(key, 2)
        rs_, env_stride = state_layout(e.H, e.W)
        lay = e.get_state_layout("index4")
        assert (lay.format, lay.row_stride, lay.plane_stride, lay.env_stride) == (_capi.SSD_OBS_INDEX4, rs_, 0, env_stride)
        lay = e.get_state_layout("rgb")
        assert (lay.format, lay.row_stride, lay.plane_stride, lay.env_stride) == (_capi.SSD_OBS_RGB, e.W, e.G, 3 * e.G)
        assert e.state_layout.env_stride == 3 * e.G and e.state_rgb.shape == (2, 3, e.H, e.W)      # RGB at creation
        lay = _capi.SsdStateLayout()
        assert e.lib.ssd_get_state_layout(e._h, 2, C.byref(lay)) == _capi.SSD_ERR_INVALID
        assert e.lib.ssd_get_state_layout(e._h, _capi.SSD_OBS_RGB, None) == _capi.SSD_ERR_INVALID
        assert e.lib.ssd_set_state_format(e._h, 2) == _capi.SSD_ERR_INVALID
        assert e.lib.ssd_set_state_format(e._h, -1) == _capi.SSD_ERR_INVALID
        buf = torch.zeros(16, dtype=torch.uint8, device=e.device)
        out = torch.zeros(16, dtype=torch.float32, device=e.device)
        for lo, cnt in ((-1, 1), (0, 3), (2, 1), (0, -1)):
            assert e.lib.ssd_expand_state(e._h, C.c_void_p(buf.data_ptr()), lo, cnt, C.c_void_p(out.data_ptr()),
                                          None) == _capi.SSD_ERR_INVALID
        seen[(e.H, e.W)] = env_stride
        e.close()
    assert seen == {(10, 10): 80, (25, 18): 304, (48, 18): 576, (9, 38): 192}


def test_env_ranges_on_streams_equal_one_launch():
    B, G = 4096, 8
    a = make_env("harvest5", B, T=3, seed=4)
    b = make_env("harvest5", B, obs="index4", state="index4", T=3, seed=4)
    a.reset()
    b.reset()
    rs = np.random.RandomState(8)
    streams = [torch.cuda.Stream(device=b.device) for _ in range(G)]
    fl = torch.empty((B, 3, b.H, b.W), dtype=torch.float32, device=b.device)
    for t in range(30):
        act = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(act, want_state=True)
        b.state_buf.fill_(0xFF)
        cur = torch.cuda.current_stream(b.device)
        for g, s in enumerate(streams):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                b.step_range(act, g * (B // G), B // G, want_state=True)
                b.state_float(g * (B // G), B // G, out=fl[g * (B // G):(g + 1) * (B // G)])
        for s in streams:
            cur.wait_stream(s)
        torch.cuda.synchronize()
        assert_same_buffers(a, b, STATE, t)
        assert torch.equal(fl, a.state_rgb.float() / 256), t
        assert np.array_equal(b.state_buf.cpu().numpy(), pack(device_state(b, range(B)))), t


@pytest.mark.parametrize("key", ["harvest5", "cleanup10"])
def test_65536_envs_sampled(key):
    B = 65536
    a = make_env(key, B, seed=13)
    b = make_env(key, B, obs="index4", state="index4", seed=13)
    a.reset()
    b.reset()
    rs = np.random.RandomState(2)
    sample = np.sort(rs.choice(B, 64, replace=False))
    st = torch.as_tensor(sample, device=b.device)
    before = b.launch_count
    for t in range(6):
        act = torch.as_tensor(random_actions(rs, a), device=a.device)
        a.step(act, want_state=True)
        b.state_buf.fill_(0xFF)
        b.step(act, want_state=True)
        assert_same_buffers(a, b, STATE, t)
        got = b.state_buf[st].cpu().numpy()
        assert np.array_equal(got, pack(device_state(b, sample))), t
        assert np.array_equal(rgb_of(b.spec.lut, unpack(got, b.H, b.W)), a.state_rgb[st].cpu().numpy()), t
        for lo in (0, int(sample[10]), B - 7):
            cnt = min(7, B - lo)
            assert torch.equal(b.state_float(lo, cnt), a.state_rgb[lo:lo + cnt].float() / 256), (t, lo)
    assert b.launch_count - before == 6 + 6 * 3                       # one step and three expansions per iteration


def test_step_host_copies_the_state_format():
    B = 64
    b = make_env("harvest5", B, state="index4", seed=3)
    a = make_env("harvest5", B, seed=3)
    ES = b.state_layout.env_stride
    io, ioa = b.make_host_io(with_obs=True, with_state=True), a.make_host_io(with_obs=True, with_state=True)
    assert io["state"].shape == (B, ES) and ioa["state"].shape == (B, 3, a.H, a.W)
    big = torch.full((B * ES + 64,), 0xEE, dtype=torch.uint8).pin_memory()
    io["state"] = big[:B * ES]                                # the bytes past B * env_stride must stay untouched
    a.reset()
    b.reset()
    rs = np.random.RandomState(1)
    for t in range(5):
        act = torch.as_tensor(random_actions(rs, b))
        io["actions"].copy_(act)
        ioa["actions"].copy_(act)
        io["state"].fill_(0xEE)
        b.step_host(io)
        a.step_host(ioa)
        assert torch.equal(io["state"], b.state_buf.cpu().reshape(-1)), t
        assert (big[B * ES:] == 0xEE).all(), t
        assert np.array_equal(io["state"].numpy(), pack(device_state(b, range(B))).reshape(-1)), t
        assert np.array_equal(rgb_of(b.spec.lut, unpack(io["state"].numpy().reshape(B, ES), b.H, b.W)), ioa["state"].numpy())
    io = b.make_host_io(with_obs=False, with_state=True)
    b.pull_host(io, obs=False, agent=False)                   # renders the state image into state_buf, then copies it
    assert torch.equal(io["state"], b.state_buf.cpu())
    b.set_state_format("rgb")
    with pytest.raises(ValueError, match="state format"):
        b.step_host(dict(io, actions=ioa["actions"], d_actions=ioa["d_actions"], reward=ioa["reward"], clean=ioa["clean"],
                         apple_cnt=ioa["apple_cnt"], done=ioa["done"], obs=None))


def test_switching_format_between_steps_and_auto_reset():
    B, L = 16, 12
    a = make_env("cleanup10_full", B, obs="index4", T=2, seed=6, limit=L)
    b = make_env("cleanup10_full", B, obs="index4", state="index4", T=2, seed=6, limit=L)
    a.reset()
    b.reset()
    rs = np.random.RandomState(4)
    for t in range(3 * L):
        if t == 8:
            a.set_state_format("index4")
            b.set_state_format("rgb")
        if t == 20:
            a.set_state_format("rgb")
            b.set_state_format("index4")
        rgb, idx = (b, a) if 8 <= t < 20 else (a, b)
        assert rgb.state_rgb is not None and idx.state_rgb is None
        idx.state_buf.fill_(0xFF)
        act = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(act, want_state=True, auto_reset=True)
        b.step(act, want_state=True, auto_reset=True)
        assert_same_buffers(a, b, STATE, t)
        got = idx.state_buf.cpu().numpy()
        assert np.array_equal(got, pack(device_state(idx, range(B)))), t
        assert np.array_equal(rgb_of(idx.spec.lut, unpack(got, idx.H, idx.W)), rgb.state_rgb.cpu().numpy()), t
        assert torch.equal(idx.state_float(), rgb.state_rgb.float() / 256), t
    assert int(a.t_buf.max()) < L                              # episodes were reset on the device
    with pytest.raises(ValueError):
        a.state_float()
    with pytest.raises(ValueError):
        a.state_packed()
    with pytest.raises(ValueError):
        a.set_state_format("rgb8")


def test_state_float_validates_out():
    b = make_env("cleanup5", 8, state="index4")
    b.reset()
    b.render(want_obs=False, want_state=True)
    with pytest.raises(ValueError):
        b.state_float(0, 8, out=torch.empty((8, 3, b.H, b.W), dtype=torch.float64, device=b.device))
    with pytest.raises(ValueError):
        b.state_float(0, 4, out=torch.empty((8, 3, b.H, b.W), dtype=torch.float32, device=b.device))
    out = torch.full((3, 3, b.H, b.W), -1.0, device=b.device)
    b.state_float(2, 3, out=out)
    assert torch.equal(out, b.state_float()[2:5])


# the shared custom maps plus three more, so that both stride cases occur: ceil(W/2) is a multiple of 4 for W = 15, 16, 64 and
# not for 11, 13, 33, 38, 50; H * row_stride is a multiple of 16 for (12, 11), (20, 33), (16, 16), (40, 50), (32, 64) and not
# for the others.
CUSTOM = harness.CUSTOM + [("cleanup", 7, 16, 4, 5, "full"), ("harvest", 13, 15, 6, 7, "full"),
                           ("harvest", 11, 13, 6, 7, "simplified")]


@pytest.mark.parametrize("case", CUSTOM, ids=lambda c: "%s_%dx%d_n%d_v%d" % c[:5])
def test_runtime_geometry_custom_maps(case):
    assert run_lockstep(lambda o, s: make_custom_env(case, 16, obs=o, state=s, T=2), B=16, steps=25) > 0


def test_custom_maps_cover_both_stride_cases():
    strides = [state_layout(H, W) for _, H, W, *_ in CUSTOM]
    half = [(W + 1) // 2 for _, H, W, *_ in CUSTOM]
    assert {h % 4 == 0 for h in half} == {True, False}
    assert {(H * rs_) % 16 == 0 for (_, H, *_), (rs_, _) in zip(CUSTOM, strides)} == {True, False}


def test_runtime_geometry_on_shipped_maps():
    """SSD_B200_GENERIC=1: the GeoD instantiations on the shipped maps."""
    for key in ("cleanup5", "cleanup10_full", "harvest5", "harvest10_full"):
        for T in (0, 3):
            with env_var("SSD_B200_GENERIC", "1"):
                run_lockstep(lambda o, s, key=key, T=T: make_env(key, 16, obs=o, state=s, T=T), B=16, steps=20)


@pytest.mark.parametrize("groups", [1, 3])
def test_batched_runner_fills_the_same_batch(groups):
    batches = {}
    for obs, state in COMBOS:
        runner = make_runner(groups=groups, extra=dict(obs_color="full", tag_timeout=2, obs_format=obs, state_format=state))
        runner.mac = ScriptedMAC(*action_tables(runner, 0, high=2 * runner.env.n_actions))
        assert runner.env.state_format == state
        batches[(obs, state)] = runner.run(test_mode=True)
        runner.close_env()
    a = batches[("rgb", "rgb")]
    for key, b in batches.items():
        for k in a.data:
            assert torch.equal(a.data[k], b.data[k]), (key, k)
    assert a.data["state"].dtype == torch.float32 and a.data["state"].abs().sum() > 0


def test_pymarl_facade_get_state_stays_rgb():
    from homophily_marl_b200 import REGISTRY
    kw = dict(num_agents=5, map="default5", view_size=7, episode_limit=30, seed=3, quiet=True)
    plain = REGISTRY["cleanup"](extra_args=dict(disable_fire_action=False), **kw)
    keyed = REGISTRY["cleanup"](extra_args=dict(disable_fire_action=False, state_format="index4"), **kw)
    assert keyed.sim.state_format == "rgb" and keyed.sim.state_rgb is not None
    plain.reset()
    keyed.reset()
    rs = np.random.RandomState(0)
    for t in range(20):
        acts = rs.randint(0, 9, size=5)
        plain.step(acts)
        keyed.step(acts)
        assert np.array_equal(plain.get_state(), keyed.get_state()), t
    plain.close()
    keyed.close()
