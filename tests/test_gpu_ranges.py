"""GPU suite: ssd_step_range (groups of env instances stepped on separate streams), interleaved runtime-geometry handles
(per-function shared-memory attribute), and the optional action-range check of the batched API."""
import numpy as np
import pytest

from harness import custom_params, random_map
from oracle import oracle as O

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.mark.parametrize("name,mp,n,view,groups,per", [("harvest", "default5", 5, 15, 4, 96), ("cleanup", "default10", 10, 7, 3, 96),
                                                         ("cleanup", "default5", 5, 7, 3, 40), ("harvest", "default5", 5, 15, 5, 23)])
def test_groups_on_streams_equal_one_batch(name, mp, n, view, groups, per):
    """G disjoint env ranges stepped concurrently on G streams (each at its own pace) == the same envs stepped as one batch:
    draws are keyed by the global env id, so the split is invisible.  The launches of a range are chained by programmatic
    dependent launch and overlap those of the other ranges; ranges of 40 / 23 envs share cache lines of the state arrays at
    their boundaries."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, T = per * groups, 23
    extra = dict(random_spawn_point=True, random_spawn_rotation=None)
    kw = dict(map=mp, view_size=view, episode_limit=1000, extra_args=extra, seed=9, env_gid_base=100)
    one = SSDBatchEnv(name, B, n, **kw)
    grp = SSDBatchEnv(name, B, n, **kw)
    ora = O.OracleBatch.from_spec(one.spec, n_envs=B, seed=9, env_gid0=100, random_spawn_point=True, spawn_rotation=None)
    one.reset()
    grp.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(0)
    acts = torch.as_tensor(rs.randint(0, one.n_actions, size=(T, B, n)).astype(np.uint8), device=one.device)
    streams = [torch.cuda.Stream() for _ in range(groups)]
    Bg = B // groups
    main = torch.cuda.current_stream()
    for g, s in enumerate(streams):                            # every group runs ALL its T steps back to back on its own stream
        s.wait_stream(main)
        with torch.cuda.stream(s):
            for t in range(T):
                grp.step_range(acts[t], g * Bg, Bg)
    for s in streams:
        main.wait_stream(s)
    for t in range(T):
        one.step(acts[t])
        out = ora.step(acts[t].cpu().numpy(), threads=8)
    torch.cuda.synchronize()
    for k in ("reward", "clean", "done", "apple_cnt", "grid_buf", "agent_buf", "ep_ret_buf", "t_buf", "tick_buf", "obs_buf"):
        assert torch.equal(getattr(one, k), getattr(grp, k)), k
    assert np.array_equal(one.obs_view().cpu().numpy(), out["obs"]) and np.array_equal(one.grid.cpu().numpy(), ora.grid)
    with pytest.raises(Exception):
        grp.step_range(acts[0], B - 1, 2)                      # range outside the batch -> SSD_ERR_INVALID


def test_interleaved_generic_handles_of_different_sizes():
    """Two runtime-geometry handles share ONE kernel instantiation; the larger one must keep working after the smaller one
    made its first launch (cudaFuncAttributeMaxDynamicSharedMemorySize is per function, only ever raised)."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    rs = np.random.RandomState(3)
    params = custom_params("harvest")
    big = SSDBatchEnv("harvest", 8, 4, view_size=31, episode_limit=50, rows=random_map(rs, "harvest", 32, 64, 6), params=params, seed=1)
    small = SSDBatchEnv("harvest", 8, 2, view_size=3, episode_limit=50, rows=random_map(rs, "harvest", 6, 7, 4), params=params, seed=2)
    ob = O.OracleBatch.from_spec(big.spec, n_envs=8, seed=1)
    osm = O.OracleBatch.from_spec(small.spec, n_envs=8, seed=2)
    big.reset()
    ob.reset()
    small.reset()                                              # first launch of the small handle happens after the big one's
    osm.reset()
    for t in range(6):
        ab = rs.randint(0, 8, size=(8, 4)).astype(np.uint8)
        asm = rs.randint(0, 8, size=(8, 2)).astype(np.uint8)
        big.step(torch.as_tensor(ab, device=big.device))
        small.step(torch.as_tensor(asm, device=small.device))
        assert np.array_equal(big.obs_view().cpu().numpy(), ob.step(ab)["obs"]), t
        assert np.array_equal(small.obs_view().cpu().numpy(), osm.step(asm)["obs"]), t


def test_check_actions_raises_keyerror_like_the_reference():
    from homophily_marl_b200.batch_env import SSDBatchEnv
    env = SSDBatchEnv("harvest", 4, 2, map="default10", view_size=7, check_actions=True)
    env.reset()
    ok = torch.zeros((4, 2), dtype=torch.uint8, device=env.device)
    env.step(ok)
    bad = ok.clone()
    bad[3, 1] = 8                                              # CLEAN does not exist in Harvest (agent.py:176)
    with pytest.raises(KeyError):
        env.step(bad)
    with pytest.raises(KeyError):
        env.step_range(bad, 0, 4)


def test_masked_auto_reset_with_envs_on_different_episode_clocks():
    """step(auto_reset=True): envs whose episode ends this step are reset in place (masked ssd_reset on the same stream) and
    continue with a fresh episode while the others carry on -- checked against per-env oracle resets."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, n, limit = 48, 5, 9
    extra = dict(random_spawn_point=True, random_spawn_rotation=None)
    env = SSDBatchEnv("cleanup", B, n, map="default5", view_size=7, episode_limit=limit, extra_args=extra, seed=21, want_state=True)
    ora = O.OracleBatch.from_spec(env.spec, n_envs=B, seed=21, random_spawn_point=True, spawn_rotation=None)
    env.reset()
    ora.reset()
    t0 = np.arange(B, dtype=np.int32) % limit                   # staggered episode clocks
    env.load_state(t=t0)
    ora.envs["t"][:] = t0
    rs = np.random.RandomState(4)
    n_resets = 0
    for t in range(3 * limit):
        act = rs.randint(0, env.n_actions, size=(B, n)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device), auto_reset=True, want_state=True)
        out = ora.step(act)
        assert np.array_equal(env.done.cpu().numpy(), out["done"]) and np.array_equal(env.reward.cpu().numpy(), out["reward"]), t
        for b in np.nonzero(out["done"])[0]:
            ora.reset_one(int(b))
            n_resets += 1
        want_obs = np.stack([ora.obs_one(b) for b in range(B)])
        assert np.array_equal(env.obs_view().cpu().numpy(), want_obs), t
        assert np.array_equal(env.state_rgb.cpu().numpy(), np.stack([ora.state_one(b) for b in range(B)])), t
        assert np.array_equal(env.grid.cpu().numpy(), ora.grid) and np.array_equal(env.t_buf.cpu().numpy(), ora.envs["t"]), t
    assert n_resets >= 2 * B
