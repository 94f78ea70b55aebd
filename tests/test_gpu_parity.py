"""GPU parity suite (-m gpu): the CUDA path, called through the C ABI, against
(a) the golden traces of the unmodified reference and (b) the C oracle on the same seeded
inputs -- bit-exact for grid, positions, orientations, rewards, clean counts, apple counts,
dones, u8 observations and u8 global state."""
import os

import numpy as np
import pytest

import lockstep as ls
from harness import assert_outputs_match_oracle, assert_state_matches_oracle, make_env, make_ref
from oracle import oracle as O

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KEYS = sorted(ls.CONFIGS)


@pytest.mark.parametrize("key", KEYS)
def test_cuda_matches_reference_golden(key):
    g = np.load(os.path.join(GOLDEN_DIR, key + ".npz"))
    g = {k: g[k] for k in g.files}
    tr = ls.run_trace(ls.CudaBackend(key, random_spawn=bool(g["random_spawn"])),
                      ls.schedule_for(key, int(g["seed"])), int(g["steps"]))
    ls.assert_traces_equal(g, tr, key)


@pytest.mark.parametrize("key", KEYS)
def test_cuda_matches_oracle_lockstep_injected(key):
    """Fresh seeds (not the golden ones), dense teleports: collisions, swaps, chains, duplicates."""
    for seed, rnd in ((201, False), (202, True)):
        sched = dict(teleport_every=5)
        a = ls.run_trace(ls.OracleBackend(key, random_spawn=rnd), ls.schedule_for(key, seed, **sched), 150)
        b = ls.run_trace(ls.CudaBackend(key, random_spawn=rnd), ls.schedule_for(key, seed, **sched), 150)
        ls.assert_traces_equal(a, b, f"{key}/seed{seed}")


@pytest.mark.parametrize("key", KEYS)
def test_cuda_matches_oracle_philox_batched(key):
    """B envs, on-device Philox draws, episode resets, clustered restarts every 8 steps."""
    B, limit, T = 192, 25, 70
    env = make_env(key, B, limit=limit, seed=1234, env_gid_base=1000)
    ora = make_ref(env)
    rs = np.random.RandomState(99)
    env.reset()
    ora.reset(threads=4)
    assert_state_matches_oracle(env, ora, "reset")
    assert np.array_equal(env.obs_view().cpu().numpy(), np.stack([ora.obs_one(b) for b in range(B)]))
    for t in range(T):
        if t % 8 == 3:
            pos, orient = ls.cluster_states(rs, env.spec, B)
            env.load_state(pos_rc=pos, orient=orient)
            for b in range(B):
                ora.set_state(b, pos_rc=pos[b], orient=orient[b])
        act = rs.randint(0, env.n_actions, size=(B, env.n)).astype(np.uint8)
        if t % 2:
            act[:, : env.n // 2 + 1] = rs.randint(0, 4, size=(B, env.n // 2 + 1))
        env.step(torch.as_tensor(act, device=env.device), want_state=True)
        out = ora.step(act, threads=4)
        assert_outputs_match_oracle(env, out, f"{key} t={t}")
        assert_state_matches_oracle(env, ora, f"{key} t={t}")
        assert np.array_equal(env.state_rgb.cpu().numpy(), np.stack([ora.state_one(b) for b in range(B)]))
        if out["done"].any():
            assert out["done"].all()
            env.reset()
            ora.reset(threads=4)
            assert_state_matches_oracle(env, ora, f"{key} reset@{t}")
    assert int(ora.envs["error"].sum()) == 0


def test_full_size_harvest_4096_vs_oracle_and_invariants():
    """BASELINE configs[1]: Harvest default5, 5 agents, 4096 envs (yaml-default extra_args)."""
    B, T = 4096, 30
    env = make_env("harvest5", B, limit=100, seed=3, random_spawn=False)
    ora = make_ref(env)
    env.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(1)
    for t in range(T):
        act = rs.randint(0, env.n_actions, size=(B, env.n)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device))
        out = ora.step(act, threads=8)
        assert_outputs_match_oracle(env, out, f"t={t}")
    assert_state_matches_oracle(env, ora, "final")
    grid = env.grid.cpu().numpy()
    assert np.array_equal((grid == 2).reshape(B, -1).sum(1), env.apple_cnt.cpu().numpy().view(np.uint16))
    pos = env.agent_pos.cpu().numpy()
    assert (grid[np.arange(B)[:, None], pos[..., 0], pos[..., 1]] != 1).all()        # nobody inside a wall
    obs = env.obs_view().cpu().numpy()
    V = env.spec.view
    assert (obs[:, :, 2, V, V] == 255).all()                                         # own cell is agent-blue


def test_cleanup10_16384_sharded_matches_single():
    """BASELINE configs[2] shape at reduced B: shards keyed by global env id give identical trajectories."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, T = 512, 20
    mk = lambda nb, g0: SSDBatchEnv("cleanup", nb, 10, map="default10", view_size=7, episode_limit=100,  # noqa: E731
                                    extra_args=dict(random_spawn_point=True, random_spawn_rotation=None), seed=9, env_gid_base=g0)
    whole, lo, hi = mk(B, 0), mk(B // 2, 0), mk(B // 2, B // 2)
    for e in (whole, lo, hi):
        e.reset()
    rs = np.random.RandomState(5)
    for t in range(T):
        act = torch.as_tensor(rs.randint(0, 9, size=(B, 10)).astype(np.uint8), device=whole.device)
        whole.step(act)
        lo.step(act[: B // 2].contiguous())
        hi.step(act[B // 2:].contiguous())
        assert torch.equal(whole.obs_view(), torch.cat([lo.obs_view(), hi.obs_view()]))
        assert torch.equal(whole.reward, torch.cat([lo.reward, hi.reward]))
    assert torch.equal(whole.grid, torch.cat([lo.grid, hi.grid]))


def test_step_host_equals_device_step():
    env = make_env("cleanup5", 64, limit=100, seed=21)
    ora = make_ref(env)
    env.reset()
    ora.reset()
    io = env.make_host_io(with_obs=True)
    rs = np.random.RandomState(2)
    for t in range(10):
        act = rs.randint(0, 9, size=(64, 5)).astype(np.uint8)
        io["actions"].copy_(torch.from_numpy(act))
        env.step_host(io)
        out = ora.step(act)
        assert np.array_equal(io["reward"].numpy(), out["reward"])
        assert np.array_equal(io["done"].numpy(), out["done"])
        assert np.array_equal(io["apple_cnt"].numpy().view(np.uint16), out["apple_cnt"])
        lay = env.layout
        host_obs = io["obs"].as_strided((64, 5, 3, env.N, env.N),
                                        (lay.obs_env_stride, lay.obs_agent_stride, lay.obs_plane_stride, lay.obs_row_stride, 1))
        assert np.array_equal(host_obs.numpy(), out["obs"])


def test_reset_mask_only_touches_selected_envs():
    env = make_env("cleanup3", 32, limit=100, seed=4)
    env.reset()
    rs = np.random.RandomState(8)
    for t in range(12):
        env.step(torch.as_tensor(rs.randint(0, 9, size=(32, 3)).astype(np.uint8), device=env.device))
    before = env.grid.clone(), env.t_buf.clone(), env.obs_view().clone()
    mask = torch.zeros(32, dtype=torch.uint8)
    mask[::3] = 1
    env.reset(mask=mask)
    keep = (mask == 0).to(env.device)
    assert torch.equal(env.grid[keep], before[0][keep])
    assert torch.equal(env.t_buf[keep], before[1][keep])
    assert torch.equal(env.obs_view()[keep], before[2][keep])
    assert (env.t_buf[~keep] == 0).all()
    assert (env.ep_ret[~keep] == 0).all()


def test_obs_padding_bytes_stay_zero_and_ring_buffers_work():
    env = make_env("harvest10_n5", 16, limit=100, seed=6)
    ora = make_ref(env)
    ring = [env.new_obs_buffer() for _ in range(3)]
    env.reset(obs_out=ring[0])
    ora.reset()
    rs = np.random.RandomState(3)
    for t in range(6):
        act = rs.randint(0, 8, size=(16, 5)).astype(np.uint8)
        buf = ring[(t + 1) % 3]
        env.step(torch.as_tensor(act, device=env.device), obs_out=buf)
        out = ora.step(act)
        assert np.array_equal(env.obs_view(buf).cpu().numpy(), out["obs"])
        lay = env.layout
        flat = buf.view(16, env.n, lay.obs_agent_stride).cpu().numpy()
        planes = flat[:, :, : 3 * lay.obs_plane_stride].reshape(16, env.n, 3, env.N, lay.obs_row_stride)
        assert (planes[..., env.N:] == 0).all() and (flat[:, :, 3 * lay.obs_plane_stride:] == 0).all()


def test_hit_penalty_and_fire_cost_parameters():
    """north_star 'penalties': non-default fire_cost / hit_penalty (the reference fixes 1 / 0, SURVEY D4)."""
    from homophily_marl_b200 import mapspec
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B = 128
    env = SSDBatchEnv("harvest", B, 10, map="default10", view_size=7, episode_limit=50, seed=11,
                      extra_args=dict(random_spawn_point=True, random_spawn_rotation=None), fire_cost=2, hit_penalty=5)
    ora = O.OracleBatch.from_spec(env.spec, n_envs=B, seed=11, random_spawn_point=True, spawn_rotation=None)
    env.reset()
    ora.reset()
    rs = np.random.RandomState(12)
    hits = 0
    for t in range(40):
        if t % 4 == 0:
            pos, orient = ls.cluster_states(rs, env.spec, B)
            env.load_state(pos_rc=pos, orient=orient)
            for b in range(B):
                ora.set_state(b, pos_rc=pos[b], orient=orient[b])
        act = rs.choice([0, 1, 2, 3, 4, 7, 7, 7], size=(B, 10)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device))
        out = ora.step(act)
        assert_outputs_match_oracle(env, out, f"t={t}")
        hits += int((out["reward"] <= -5).sum())
    assert hits > 0


def test_incentive_bookkeeping_matches_torch():
    """homophily_learner.py:98-115 restated with the same op order in torch on the same device."""
    import ctypes as C
    from homophily_marl_b200 import _capi
    lib = _capi.load()
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cpu").manual_seed(0)
    bs, T, n = 6, 11, 5
    actions_inc = torch.randint(0, 3, (bs, T, n, n, 1), generator=g).to(dev)
    rewards = torch.randint(-1, 2, (bs, T, n), generator=g).float().to(dev)
    incentive, cost, ratio, max_seq = 0.7, 0.3, 1.5, 101
    mask = (1 - torch.eye(n, device=dev)).view(1, 1, n, n, 1).long()
    am = actions_inc * mask
    give = (am != 0).sum(dim=(3, 4))
    rv = (am == 1).sum(dim=(2, 4)) - (am == 2).sum(dim=(2, 4))
    want_env = (rewards + rv * ratio * incentive) / max_seq
    want_inc = (rewards - give * cost * incentive) / max_seq
    outs = [torch.empty(bs, T, n, device=dev) for _ in range(3)]
    a = actions_inc.contiguous()
    ok = False
    for T_arg in (max_seq, -max_seq):          # true division (CPU torch) / reciprocal multiply (CUDA torch)
        rc = lib.ssd_incentive(a.data_ptr(), rewards.data_ptr(), bs * T, n, incentive, cost, ratio, T_arg,
                               outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(),
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        torch.cuda.synchronize()
        assert torch.equal(outs[2], torch.sign(rv.float()))
        ok = ok or (torch.equal(outs[0], want_env) and torch.equal(outs[1], want_inc))
        assert torch.allclose(outs[0], want_env, rtol=0, atol=1e-7) and torch.allclose(outs[1], want_inc, rtol=0, atol=1e-7)
    assert ok, "neither division mode is bit-identical to torch on this device"


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_env_on_second_device_leaves_current_device_alone():
    """The C ABI makes the handle's device current only for the duration of a call (one process may hold several)."""
    assert torch.cuda.current_device() == 0
    env1 = make_env("cleanup5", 32, limit=50, seed=8)
    ora = make_ref(env1)
    from homophily_marl_b200.batch_env import SSDBatchEnv
    env2 = SSDBatchEnv("cleanup", 32, 5, map="default5", view_size=7, episode_limit=50, seed=8, device="cuda:1",
                       extra_args=dict(random_spawn_point=True, random_spawn_rotation=None))
    assert torch.cuda.current_device() == 0
    env1.reset()
    env2.reset()
    ora.reset()
    rs = np.random.RandomState(4)
    for t in range(10):
        act = rs.randint(0, 9, size=(32, 5)).astype(np.uint8)
        env1.step(torch.as_tensor(act, device="cuda:0"))
        env2.step(torch.as_tensor(act, device="cuda:1"))
        out = ora.step(act)
        assert torch.cuda.current_device() == 0
        assert np.array_equal(env1.obs_view().cpu().numpy(), out["obs"])
        assert np.array_equal(env2.obs_view().cpu().numpy(), out["obs"])
    env2.close()


def test_full_size_harvest_65536_properties_and_sampled_oracle():
    """BASELINE configs[4]: Harvest default5, 65536 envs x 5 agents.  Size-independent properties on the whole batch
    (determinism, apple-count checksum, walls never entered, own pixel, padding zero) + the oracle on sampled envs."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B, T = 65536, 12
    mk = lambda: SSDBatchEnv("harvest", B, 5, map="default5", view_size=15, episode_limit=100, seed=17,  # noqa: E731
                             extra_args=dict(random_spawn_point=True, random_spawn_rotation=None))
    env, twin = mk(), mk()
    sample = list(range(0, B, 4099)) + [B - 1]
    oras = {b: O.OracleBatch.from_spec(env.spec, n_envs=1, seed=17, env_gid0=b, random_spawn_point=True, spawn_rotation=None)
            for b in sample}
    env.reset()
    twin.reset()
    for o in oras.values():
        o.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    for t in range(T):
        act = torch.randint(0, 8, (B, 5), generator=g, device="cuda", dtype=torch.int32).to(torch.uint8)
        env.step(act)
        twin.step(act)
        a_host = act[sample].cpu().numpy()
        obs_s = env.obs_view()[sample].cpu().numpy()
        rew_s = env.reward[sample].cpu().numpy()
        for k, b in enumerate(sample):
            out = oras[b].step(a_host[k:k + 1])
            assert np.array_equal(obs_s[k], out["obs"][0]) and np.array_equal(rew_s[k], out["reward"][0]), (t, b)
    assert torch.equal(env.obs_buf, twin.obs_buf) and torch.equal(env.grid_buf, twin.grid_buf)          # deterministic
    assert torch.equal((env.grid == 2).flatten(1).sum(1).to(torch.int32), env.apple_cnt.to(torch.int32) & 0xFFFF)
    pos = env.agent_pos.long()
    cell = env.grid[torch.arange(B, device="cuda")[:, None], pos[..., 0], pos[..., 1]]
    assert bool((cell != 1).all())
    assert bool((env.obs_view()[:, :, 2, 15, 15] == 255).all())
    lay = env.layout
    rows = env.obs_buf.view(B, 5, 3, 31, lay.obs_row_stride)
    assert bool((rows[..., 31:] == 0).all())
    assert len(torch.unique(env.agent_buf[:4096], dim=0)) > 4000                                          # envs really differ


def test_full_size_cleanup10_16384_vs_oracle():
    """BASELINE configs[2] on one GPU: Cleanup default10, 10 agents, 16384 envs, a few steps against the oracle."""
    B = 16384
    env = make_env("cleanup10", B, limit=100, seed=23)
    ora = make_ref(env)
    env.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(6)
    for t in range(6):
        act = rs.randint(0, 9, size=(B, 10)).astype(np.uint8)
        act[:, :4] = 8 if t % 2 else act[:, :4]                    # plenty of CLEAN beams so that spawning switches on
        env.step(torch.as_tensor(act, device=env.device))
        out = ora.step(act, threads=8)
        assert_outputs_match_oracle(env, out, f"t={t}")
    assert_state_matches_oracle(env, ora, "final")


def test_single_env_1000_steps_like_baseline_config0():
    """BASELINE configs[0] shape: Cleanup default5, 5 agents, ONE env, 1000 random-action steps in a single episode."""
    env = make_env("cleanup5", 1, limit=1000, seed=0, random_spawn=False)
    ora = make_ref(env)
    env.reset()
    ora.reset()
    rs = np.random.RandomState(123)
    acts = rs.randint(0, 9, size=(1000, 1, 5)).astype(np.uint8)
    dev_acts = torch.as_tensor(acts, device=env.device)
    obs_sum = 0
    for t in range(1000):
        env.step(dev_acts[t])
        out = ora.step(acts[t])
        if t % 50 == 49 or t == 999:
            assert_outputs_match_oracle(env, out, f"t={t}")
            assert_state_matches_oracle(env, ora, f"t={t}")
        obs_sum += int(out["obs"].sum())
    assert bool(env.done[0].item()) and obs_sum > 0
    assert np.array_equal(env.ep_ret.cpu().numpy(), ora.ep_ret)


def test_incentive_python_wrapper():
    from homophily_marl_b200.incentive import incentive_rewards
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(1)
    a = torch.randint(0, 3, (4, 7, 3, 3, 1), generator=g).to(dev)
    r = torch.randint(-1, 2, (4, 7, 3), generator=g).float().to(dev)
    mask = (1 - torch.eye(3, device=dev)).view(1, 1, 3, 3, 1).long()
    am = a * mask
    give = (am != 0).sum(dim=(3, 4))
    rv = (am == 1).sum(dim=(2, 4)) - (am == 2).sum(dim=(2, 4))
    env_r, inc_r, sgn = incentive_rewards(a, r, 1.0, 0.5, 2.0, 101, recip=True)
    assert env_r.shape == r.shape and torch.equal(sgn, torch.sign(rv.float()))
    assert torch.allclose(env_r, (r + rv * 2.0 * 1.0) / 101, rtol=0, atol=1e-7)
    assert torch.allclose(inc_r, (r - give * 0.5 * 1.0) / 101, rtol=0, atol=1e-7)
    with pytest.raises(RuntimeError):
        incentive_rewards(a.cpu(), r.cpu(), 1.0, 0.5, 2.0, 101)
