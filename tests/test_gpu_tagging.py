"""GPU suite: tagging-out timers (tag_timeout > 0) are bit-exact against the tagging reference (tests/tag_oracle.c) -- grid, positions, orientations, timers,
rewards, clean counts, apple counts, done flags, u8 observations and state images -- in every shipped configuration, with
injected draws and teleports, with Philox draws at scale across episodes, split into env ranges and on the runtime geometry; and
the PyMARL facade and the batched runner carry the feature through ``extra_args``."""
import numpy as np
import pytest

import lockstep
from harness import (FIRE, STATE, ScriptedMAC, assert_outputs_match_oracle, assert_same_buffers, assert_state_matches_oracle,
                     env_var, make_env, make_ref, make_runner, random_actions, step_one_outputs)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def run_philox_case(key, B=48, T=3, steps=60):
    """B envs, Philox draws, FIRE-heavy random play; step outputs and ssd_render both checked.  Returns (tags, respawns)."""
    env = make_env(key, B, T=T, limit=steps + 5)
    ora = make_ref(env)
    assert ora.tag_timeout == T
    env.reset()
    ora.reset()
    rs = np.random.RandomState(len(key) * 7 + T)
    tags = respawns = 0
    for t in range(steps):
        act = random_actions(rs, env, fire=0.35)
        before = ora.tag_out.copy()
        env.step(torch.as_tensor(act, device=env.device), want_state=True)
        out = ora.step(act, threads=8)
        tags += int(((ora.tag_out == T) & (before == 0)).sum())
        respawns += int(((before == 1) & (ora.tag_out == 0)).sum())
        assert_outputs_match_oracle(env, out, (key, t))
        assert_state_matches_oracle(env, ora, (key, t))
        state = np.stack([ora.state_one(b) for b in range(B)])
        assert np.array_equal(env.state_rgb.cpu().numpy(), state), (key, t, "state")
        if t % 10 == 9:                                            # ssd_render honours the timers too
            obs2 = env.new_obs_buffer()
            env.render(obs_out=obs2, want_obs=True, want_state=True)
            assert np.array_equal(env.obs_view(obs2).cpu().numpy(), out["obs"]), (key, t, "render obs")
            assert np.array_equal(env.state_rgb.cpu().numpy(), state), (key, t, "render state")
    assert int(ora.envs["error"].sum()) == 0
    env.close()
    return tags, respawns


@pytest.mark.parametrize("key", sorted(lockstep.CONFIGS))
def test_every_config_matches_oracle_with_tagging(key):
    tags, respawns = run_philox_case(key)
    assert tags > 0 and respawns > 0, (tags, respawns)


@pytest.mark.parametrize("key,T", [("cleanup5", 1), ("harvest5", 3), ("cleanup10_full", 25), ("harvest10_full", 3)])
def test_injected_draws_and_teleports(key, T):
    """One env, every draw injected (spawn_key / rot included, so respawns read them), FIRE-heavy, teleports every 7 steps."""
    env = make_env(key, 1, T=T, seed=0)
    ora = make_ref(env)
    n = env.n
    sched = lockstep.schedule_for(key, seed=100 + T, teleport_every=7)
    rs = np.random.RandomState(T)
    d0 = sched.reset_draws()
    env.reset(draws=dict(spawn_key=d0["spawn_key"].reshape(1, n, -1), rot=d0["rot"].reshape(1, n)))
    ora.reset_one(0, dict(spawn_key=d0["spawn_key"].reshape(n, -1), rot=d0["rot"]))
    tags = respawns = 0
    for t in range(150):
        actions, draws, tele = sched.step_inputs(t)
        actions = np.where(rs.rand(n) < 0.4, FIRE, actions).astype(np.uint8)
        rd = sched.reset_draws()
        draws.update(spawn_key=rd["spawn_key"], rot=rd["rot"])
        if tele is not None:
            env.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
            ora.set_state(0, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
        before = ora.tag_out.copy()
        env.step(torch.as_tensor(actions.reshape(1, n), device=env.device),
                 draws={k: v.reshape(1, -1) for k, v in draws.items()}, want_state=True)
        out = step_one_outputs(ora, actions, draws)
        tags += int(((ora.tag_out == T) & (before == 0)).sum())
        respawns += int(((before == 1) & (ora.tag_out == 0)).sum())
        assert_outputs_match_oracle(env, out, (key, t))
        assert_state_matches_oracle(env, ora, (key, t))
        assert np.array_equal(env.state_rgb[0].cpu().numpy(), ora.state_one(0)), (key, t, "state")
    assert tags > 0 and respawns > 0, (tags, respawns)


def test_philox_at_scale_with_masked_reset_and_auto_reset():
    """4 096 envs over more than two episodes: auto_reset at the episode end, plus masked resets of some envs mid-episode."""
    B, T, L = 4096, 4, 30
    env = make_env("cleanup5", B, T=T, seed=21, limit=L)
    ora = make_ref(env)
    env.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(5)
    tags = respawns = cleared = 0
    for t in range(75):
        act = random_actions(rs, env, fire=0.35)
        before = ora.tag_out.copy()
        env.step(torch.as_tensor(act, device=env.device), auto_reset=True)
        out = ora.step(act, threads=8)
        tags += int(((ora.tag_out == T) & (before == 0)).sum())
        respawns += int(((before == 1) & (ora.tag_out == 0)).sum())
        assert_outputs_match_oracle(env, dict(out, obs=None), t)
        done = np.flatnonzero(out["done"])
        for b in done:
            ora.reset_one(int(b))
        if t % 13 == 6:                                            # masked reset of envs with agents out right now
            mask = (ora.tag_out > 0).any(1) & (rs.rand(B) < 0.5)
            cleared += int((ora.tag_out[mask] > 0).sum())
            env.reset(mask=torch.as_tensor(mask.astype(np.uint8)))
            for b in np.flatnonzero(mask):
                ora.reset_one(int(b))
        assert_state_matches_oracle(env, ora, t)
        if t % 5 == 0 or len(done):                                # the step's views; first views of the envs just reset
            want = np.stack([ora.obs_one(b) for b in range(B)])
            assert np.array_equal(env.obs_view().cpu().numpy(), want), (t, "obs")
    assert tags > 0 and respawns > 0 and cleared > 0, (tags, respawns, cleared)
    assert not ora.tag_out[ora.envs["t"] == 0].any()


def test_env_ranges_equal_one_launch():
    B, T = 4096, 3
    a = make_env("harvest5", B, T=T, seed=4)
    b = make_env("harvest5", B, T=T, seed=4)
    a.reset()
    b.reset()
    rs = np.random.RandomState(8)
    streams = [torch.cuda.Stream(device=b.device) for _ in range(8)]
    obs_b = b.new_obs_buffer()
    for t in range(40):
        act = torch.as_tensor(random_actions(rs, a, fire=0.35), device=a.device)
        a.step(act)
        cur = torch.cuda.current_stream(b.device)
        for g, s in enumerate(streams):
            s.wait_stream(cur)
            with torch.cuda.stream(s):
                b.step_range(act, g * (B // 8), B // 8, obs_out=obs_b)
        for s in streams:
            cur.wait_stream(s)
        torch.cuda.synchronize()
        assert_same_buffers(a, b, STATE, t)
        assert torch.equal(a.obs_buf, obs_b), t
    assert int((a.tag_out > 0).sum()) > 0


def test_runtime_geometry_kernels():
    """SSD_B200_GENERIC=1: the GeoD instantiations (tagging variant) on the shipped maps."""
    for key in ("cleanup5", "harvest5", "harvest10_full"):
        with env_var("SSD_B200_GENERIC", "1"):
            tags, respawns = run_philox_case(key, B=24, steps=30)
        assert tags > 0 and respawns > 0, (key, tags, respawns)


def test_pymarl_facade_with_tagging():
    from homophily_marl_b200 import REGISTRY
    env = REGISTRY["harvest"](num_agents=5, map="default5", view_size=15, episode_limit=200, seed=3, quiet=True,
                              extra_args=dict(tag_timeout=25, disable_fire_action=False, disable_rotation_action=False))
    env.reset()
    rs = np.random.RandomState(0)
    seen = 0
    for t in range(200):
        actions = np.where(rs.rand(5) < 0.5, FIRE, rs.randint(0, 7, size=5))
        reward, terminated, info = env.step(actions)
        assert type(terminated) is bool
        out = env.sim.tag_out[0].cpu().numpy()
        obs = env.get_obs()
        for i in range(5):
            assert (not np.any(obs[i])) == bool(out[i]), (t, i)
        seen += int((out > 0).sum())
        if terminated:
            break
    assert seen > 0
    env.close()


def test_batched_runner_with_tagging():
    """One runner episode with tagging on: the stored observation rows of agents out of play are zero, all others are not."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, T, n = 8, 40, 5
    runner = make_runner(mp="default5", n=n, B=B, T=T, extra=dict(tag_timeout=6))
    A, dev = runner.env.n_actions, runner.env.device
    g = torch.Generator().manual_seed(1)
    table = torch.randint(0, A, (B, T + 1, n, 1), generator=g)
    table = torch.where(torch.rand(table.shape, generator=g) < 0.4, torch.full_like(table, FIRE), table).to(dev)
    table_inc = torch.zeros((B, T + 1, n, n, 1), dtype=torch.long, device=dev)
    runner.mac = ScriptedMAC(table, table_inc)
    batch = runner.run(test_mode=True)
    # the same episode on a twin env gives the timers at every stored step
    twin = SSDBatchEnv("cleanup", B, n, map="default5", view_size=7, episode_limit=T, extra_args=runner.args.env_args["extra_args"],
                       seed=3)
    twin.reset()
    out_steps = 0
    for t in range(T + 1):
        out = twin.tag_out > 0
        rows = batch["obs"][:, t].reshape(B, n, -1)
        assert torch.equal(rows.abs().sum(-1) == 0, out), t
        out_steps += int(out.sum())
        if t < T:
            twin.step((table[:, t, :, 0] % A).to(torch.uint8).contiguous())
    assert out_steps > 0
