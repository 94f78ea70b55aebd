"""GPU suite: auto-reset inside the step launch (ssd_step_autoreset), bit for bit.

A fused env and a twin that runs the three-launch sequence the contract names -- ssd_step_range, a masked ssd_reset of the
envs the step finished with the same draws, ssd_render -- are stepped from one seed on staggered episode clocks and compared in
every buffer, pads included; the twin's observation, state image and ep_ret just before its reset must equal the fused env's
episode-end buffers.  Also: the C oracle (and the tagging reference) with per-env resets on every shipped config and a
runtime-geometry map, sentinel bytes in the slots of envs that did not finish or lie outside the range, 8 ranges on 8 streams
with and without programmatic dependent launch, 65 536 envs and CUDA-graph capture."""
import numpy as np
import pytest

import lockstep
from harness import (BUFS, COMBOS, END_BUFS, assert_same_buffers, custom_params, env_var, make_env, make_ref, random_actions,
                     random_draws, random_map)

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
SENTINEL = 0xEE


def stagger(env, limit):
    t0 = np.arange(env.B, dtype=np.int32) % limit
    env.load_state(t=t0)
    return t0


def fill_end(env):
    env.end_obs_buf.fill_(SENTINEL)
    env.end_state_buf.fill_(SENTINEL)
    env.end_ep_ret_buf.fill_(-7)


def sequence_step(env, act, draws=None):
    """The three launches the fused step must equal; returns the pre-reset obs / state / ep_ret and the done mask."""
    env.step(act, draws=draws, want_state=True)
    pre = (env.obs_buf.clone(), env.state_buf.clone(), env.ep_ret_buf.clone())
    done = env.done.clone()
    env.reset(mask=done, draws=draws)
    env.render(want_obs=True, want_state=True)
    return pre, done.bool()


def assert_twins(fused, seq, pre, done, what):
    assert_same_buffers(fused, seq, BUFS, what)
    obs, state, ep_ret = pre
    d = done.cpu().numpy().astype(bool)
    assert np.array_equal(fused.end_obs_buf.cpu().numpy()[d], obs.cpu().numpy()[d]), (what, "end obs")
    assert np.array_equal(fused.end_state_buf.cpu().numpy()[d], state.cpu().numpy()[d]), (what, "end state")
    assert np.array_equal(fused.end_ep_ret.cpu().numpy()[d], ep_ret[:, :fused.n].cpu().numpy()[d]), (what, "end ep_ret")
    assert (fused.end_ep_ret_buf[:, fused.n:].cpu().numpy() == -7).all(), (what, "end ep_ret pads are not written")
    assert (fused.end_obs_buf.cpu().numpy()[~d] == SENTINEL).all(), (what, "end obs of envs that did not finish")
    assert (fused.end_state_buf.cpu().numpy()[~d] == SENTINEL).all(), (what, "end state of envs that did not finish")
    assert (fused.end_ep_ret_buf.cpu().numpy()[~d] == -7).all(), (what, "end ep_ret of envs that did not finish")


@pytest.mark.parametrize("T", [0, 3])
@pytest.mark.parametrize("color", ["simplified", "full"])
@pytest.mark.parametrize("key", ["cleanup5", "harvest5", "harvest10_full", "cleanup3"])
def test_fused_equals_the_three_launch_sequence(key, color, T):
    """Twin envs on staggered clocks, all four format combinations, random spawn point and rotation, FIRE with tagging."""
    B, L = 24, 7
    resets = back_at_end = 0
    for obs, state in COMBOS:
        fused = make_env(key, B, obs=obs, state=state, color=color, T=T, limit=L, keep_episode_end=True)
        seq = make_env(key, B, obs=obs, state=state, color=color, T=T, limit=L)
        for e in (fused, seq):
            e.reset()
            stagger(e, L)
        rs = np.random.RandomState(B + T)
        for t in range(2 * L + 3):
            act = torch.as_tensor(random_actions(rs, fused, fire=0.35 if T else 0), device=fused.device)
            timers = seq.tag_out.clone()
            fill_end(fused)
            fused.obs_buf.fill_(SENTINEL)
            seq.obs_buf.fill_(SENTINEL)
            fused.step(act, want_state=True, auto_reset=True)
            pre, done = sequence_step(seq, act)
            assert_twins(fused, seq, pre, done, (key, color, T, obs, state, t))
            resets += int(done.sum())
            back_at_end += int(((timers == 1).any(1) & done).sum())      # a tagged agent returned in the episode's last step
        fused.close()
        seq.close()
    assert resets >= 4 * B
    assert T == 0 or back_at_end > 0


@pytest.mark.parametrize("key,T", [("cleanup5", 0), ("cleanup10_full", 3), ("harvest5", 0), ("harvest10_full", 2)])
def test_injected_draws_and_teleports(key, T):
    B, L = 6, 5
    for obs, state in COMBOS:
        fused = make_env(key, B, obs=obs, state=state, T=T, limit=L, keep_episode_end=True)
        seq = make_env(key, B, obs=obs, state=state, T=T, limit=L)
        sched = lockstep.schedule_for(key, seed=40 + T, teleport_every=3)
        rs = np.random.RandomState(T)
        d0 = random_draws(rs, fused)
        for e in (fused, seq):
            e.reset(draws=dict(spawn_key=d0["spawn_key"], rot=d0["rot"]))
            stagger(e, L)
        for t in range(3 * L):
            draws = random_draws(rs, fused)
            act = random_actions(rs, fused, fire=0.35 if T else 0)
            _, _, tele = sched.step_inputs(t)
            if tele is not None:                                # clustered agents, duplicate occupancy: collisions
                for e in (fused, seq):
                    e.set_state(t % B, grid=tele["grid"], pos_rc=tele["pos"], orient=tele["orient"])
            at = torch.as_tensor(act, device=fused.device)
            fill_end(fused)
            fused.step(at, draws=draws, want_state=True, auto_reset=True)
            pre, done = sequence_step(seq, at, draws)
            assert_twins(fused, seq, pre, done, (key, obs, state, t))
        fused.close()
        seq.close()


def oracle_run(env, ora, L, steps, envs=None):
    """Fused auto-reset steps against the reference stepped as a batch and reset env by env."""
    t0 = stagger(env, L)
    ora.envs["t"][:] = t0
    rs = np.random.RandomState(11)
    envs = np.arange(env.B) if envs is None else envs
    resets = 0
    for t in range(steps):
        act = random_actions(rs, env, fire=0.35 if env.spec.tag_timeout else 0)
        env.end_obs_buf.fill_(SENTINEL)
        env.step(torch.as_tensor(act, device=env.device), want_state=True, auto_reset=True)
        out = ora.step(act, want_obs=True, threads=8)
        done = out["done"].astype(bool)
        assert np.array_equal(env.done.cpu().numpy(), out["done"]) and np.array_equal(env.reward.cpu().numpy(), out["reward"]), t
        end_obs = env.obs_view(env.end_obs_buf).cpu().numpy()
        sel = envs[done[envs]]
        assert np.array_equal(end_obs[sel], out["obs"][sel]), (t, "end obs")
        assert np.array_equal(env.end_ep_ret.cpu().numpy()[sel], ora.ep_ret[sel]), (t, "end ep_ret")
        assert (end_obs[~done] == SENTINEL).all(), t
        for b in np.flatnonzero(done):
            ora.reset_one(int(b))
            resets += 1
        obs = env.obs_view().cpu().numpy()
        assert np.array_equal(obs[envs], np.stack([ora.obs_one(int(b)) for b in envs])), t
        assert np.array_equal(env.state_rgb.cpu().numpy()[envs], np.stack([ora.state_one(int(b)) for b in envs])), t
        assert np.array_equal(env.grid.cpu().numpy(), ora.grid) and np.array_equal(env.t_buf.cpu().numpy(), ora.envs["t"]), t
        assert np.array_equal(env.ep_ret.cpu().numpy(), ora.ep_ret), t
    return resets


@pytest.mark.parametrize("key", ["cleanup3", "cleanup5", "cleanup10", "harvest5", "harvest10_full"])
def test_every_shipped_config_matches_the_oracle(key):
    B, L = 32, 6
    env = make_env(key, B, limit=L, keep_episode_end=True)
    ora = make_ref(env)
    env.reset()
    ora.reset()
    assert oracle_run(env, ora, L, 3 * L) >= 2 * B


def test_runtime_geometry_matches_the_oracle():
    """SSD_B200_GENERIC=1 (the GeoD kernels) on a shipped map, and a custom map that only the runtime geometry serves."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    with env_var("SSD_B200_GENERIC", "1"):
        env = make_env("cleanup10_full", 16, limit=5, keep_episode_end=True)
    rows = random_map(np.random.RandomState(5), "harvest", 13, 15, n_spawn=9)
    custom = SSDBatchEnv("harvest", 16, 6, view_size=9, episode_limit=5, rows=rows, params=custom_params("harvest"), seed=3,
                         want_state=True, extra_args=dict(random_spawn_point=True, random_spawn_rotation=None, obs_color="full"),
                         keep_episode_end=True)
    for e in (env, custom):
        ora = make_ref(e)
        e.reset()
        ora.reset()
        assert oracle_run(e, ora, 5, 12) > 0


def ranges_case():
    """8 disjoint ranges on 8 streams, no host sync between steps, == one whole-batch launch.  Ranges of 23 and 40 envs start
    inside cache lines of the state arrays."""
    sizes = [23, 40, 64, 23, 40, 96, 33, 65]
    B, L = sum(sizes), 6
    starts = np.concatenate([[0], np.cumsum(sizes)[:-1]])
    one = make_env("harvest5", B, obs="index4", state="index4", T=2, limit=L, keep_episode_end=True)
    grp = make_env("harvest5", B, obs="index4", state="index4", T=2, limit=L, keep_episode_end=True)
    for e in (one, grp):
        e.reset()
        stagger(e, L)
        fill_end(e)
    rs = np.random.RandomState(3)
    acts = torch.as_tensor(np.stack([random_actions(rs, one, fire=0.35) for _ in range(3 * L)]), device=one.device)
    streams = [torch.cuda.Stream() for _ in sizes]
    main = torch.cuda.current_stream()
    for g, s in enumerate(streams):
        s.wait_stream(main)
        with torch.cuda.stream(s):
            for t in range(len(acts)):
                grp.step_range(acts[t], int(starts[g]), sizes[g], want_state=True, auto_reset=True)
    for s in streams:
        main.wait_stream(s)
    for t in range(len(acts)):
        one.step(acts[t], want_state=True, auto_reset=True)
    torch.cuda.synchronize()
    assert_same_buffers(one, grp, BUFS + END_BUFS, "ranges")
    # a range never writes outside itself
    e = make_env("cleanup5", 64, limit=1, keep_episode_end=True)
    e.reset()
    fill_end(e)
    e.obs_buf.fill_(SENTINEL)
    e.step_range(torch.zeros((64, e.n), dtype=torch.uint8, device=e.device), 10, 23, want_state=True, auto_reset=True)
    done = e.done.cpu().numpy()
    assert done[10:33].all() and not done[:10].any() and not done[33:].any()
    for buf in (e.end_obs_buf, e.end_state_buf, e.obs_buf):
        b = buf.cpu().numpy()
        assert (b[:10] == SENTINEL).all() and (b[33:] == SENTINEL).all() and not (b[10:33] == SENTINEL).all()
    assert (e.t_buf.cpu().numpy()[10:33] == 0).all()


def test_ranges_on_streams_equal_one_launch_with_pdl():
    ranges_case()


def test_ranges_on_streams_equal_one_launch_without_pdl():
    with env_var("SSD_B200_PDL", "0"):
        ranges_case()


def test_65536_envs():
    B, L = 65536, 50
    env = make_env("cleanup5", B, obs="index4", state="index4", limit=L, keep_episode_end=True)
    ora = make_ref(env)
    env.reset()
    ora.reset(threads=8)
    t0 = stagger(env, L)
    ora.envs["t"][:] = t0
    rs = np.random.RandomState(2)
    sample = np.sort(rs.choice(B, 48, replace=False))
    for t in range(3):
        act = random_actions(rs, env)
        env.step(torch.as_tensor(act, device=env.device), want_state=True, auto_reset=True)
        out = ora.step(act, want_obs=False, threads=8)
        done = out["done"].astype(bool)
        assert 0.01 * B < done.sum() < 0.03 * B
        assert np.array_equal(env.done.cpu().numpy(), out["done"]), t
        for b in np.flatnonzero(done):
            ora.reset_one(int(b))
        grid, tt = env.grid.cpu().numpy(), env.t_buf.cpu().numpy()
        assert np.array_equal(grid[sample], ora.grid[sample]) and np.array_equal(tt, ora.envs["t"]), t
        assert np.array_equal(env.agent_pos.cpu().numpy()[sample], ora.pos_rc[sample]), t
        assert (tt[done] == 0).all()
        g = env.grid_buf[:, :env.G]
        counts = ((g == 2).sum(1) | ((g == 3).sum(1) << 16)).to(torch.int32)
        assert torch.equal(counts, env.counts_buf), t


def test_cuda_graph_capture_equals_eager():
    B, L, K = 64, 4, 9
    a = make_env("cleanup10_full", B, obs="index4", T=2, limit=L, keep_episode_end=True)
    b = make_env("cleanup10_full", B, obs="index4", T=2, limit=L, keep_episode_end=True)
    for e in (a, b):
        e.reset()
        stagger(e, L)
    rs = np.random.RandomState(0)
    acts = torch.as_tensor(np.stack([random_actions(rs, a, fire=0.35) for _ in range(K)]), device=a.device)
    before = a.launch_count
    for t in range(K):
        a.step(acts[t], want_state=True, auto_reset=True)
    assert a.launch_count - before == K                        # one launch per fused step
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(graph, stream=s):
        for t in range(K):
            b.step(acts[t], want_state=True, auto_reset=True)
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    assert_same_buffers(a, b, BUFS + END_BUFS, "graph")


def test_format_switch_reallocates_the_episode_end_buffers():
    e = make_env("harvest5", 8, limit=7, keep_episode_end=True)
    assert e.end_obs_buf.shape == e.obs_buf.shape and e.end_state_buf.shape == e.state_buf.shape
    assert e.end_ep_ret.shape == (8, e.n) and e.end_ep_ret.dtype == torch.int32
    e.set_obs_format("index4")
    e.set_state_format("index4")
    assert e.end_obs_buf.shape == e.obs_buf.shape == (8, e.obs_layout.env_stride)
    assert e.end_state_buf.shape == e.state_buf.shape == (8, e.state_layout.env_stride)
    e.reset()
    e.load_state(t=np.full(8, 6, dtype=np.int32))
    e.step(torch.zeros((8, e.n), dtype=torch.uint8, device=e.device), want_state=True, auto_reset=True)
    assert e.done.all()
    end = e.state_float(buf=e.end_state_buf)
    assert end.shape == (8, 3, e.H, e.W) and not torch.equal(end, e.state_float())   # the last state, not the new episode's
    f = make_env("harvest5", 8, limit=7, keep_episode_end=False)
    assert f.end_obs_buf is None and f.end_state_buf is None and f.end_ep_ret is None
