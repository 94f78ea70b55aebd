"""GPU suite (VERDICT r1 item 1 / BASELINE configs[3]): the reference's UNCHANGED rollout + learning code runs end to end
on the CUDA env.

  (i)   ``runners.episode_runner.EpisodeRunner.run()`` (episode_runner.py:48-141) with the reference's ``EpisodeBatch`` and
        ``HomophilyMAC`` over ``pymarl_env.REGISTRY['cleanup']``; what it stored is re-derived by the C oracle from the stored
        actions and compared bit-exactly;
  (ii)  ``run.run_sequential`` (run.py:81-244), Cleanup default3, >= 2500 env steps, learner updates and test episodes included;
  (iii) ``BatchedEpisodeRunner`` with the reference's ``EpisodeBatch`` / ``ReplayBuffer`` / MAC / learner at B = 256.

The reference sources come from ``baseline/_ref`` (git-ignored copy made by ``baseline/fetch_ref.py``; ``/root/reference``
does not exist on the GPU box) through ``baseline/refloop.py``; matplotlib / pyclustering are stubbed (SURVEY 8c).
"""
import numpy as np
import pytest

from baseline import refloop
from harness import _cfg

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not refloop.available(), reason="reference sources absent (baseline/_ref)")]
torch = pytest.importorskip("torch")


def _oracle_replay(batch, spec, seed, b0=0, ticks_before=0):
    """Re-derives every env-produced field of an EpisodeBatch from its stored actions with the C oracle (Philox mode)."""
    from oracle import oracle as O
    B, T1 = batch.batch_size, batch.max_seq_length
    n = spec.n_agents
    ora = O.OracleBatch.from_spec(spec, n_envs=B, seed=seed, env_gid0=b0)
    ora.envs["tick"][:] = ticks_before
    ora.reset()
    A = spec.n_actions
    acts = (batch["actions"].cpu().numpy()[..., 0] % A).astype(np.uint8)          # [B, T+1, n]
    orient_vec = np.array([[-1, 0], [1, 0], [0, -1], [0, 1]], dtype=np.float32)    # map_env.py:28-31
    for t in range(T1):
        obs = np.stack([ora.obs_one(b) for b in range(B)]).astype(np.float32) / 256
        state = np.stack([ora.state_one(b) for b in range(B)]).astype(np.float32) / 256
        assert np.array_equal(batch["obs"][:, t].cpu().numpy(), obs), ("obs", t)
        assert np.array_equal(batch["state"][:, t].cpu().numpy(), state), ("state", t)
        assert np.array_equal(batch["agent_pos"][:, t].cpu().numpy(), ora.pos_rc.astype(np.float32)), ("pos", t)
        assert np.array_equal(batch["agent_orientation"][:, t].cpu().numpy(), orient_vec[ora.orient]), ("orient", t)
        if t == T1 - 1:
            break
        out = ora.step(acts[:, t], want_obs=False)
        assert np.array_equal(batch["reward"][:, t].cpu().numpy(), out["reward"].astype(np.float32)), ("reward", t)
        assert np.array_equal(batch["clean_num"][:, t].cpu().numpy(), out["clean"].astype(np.float32)), ("clean", t)
        den = (out["apple_cnt"].astype(np.float64) / spec.G).astype(np.float32)
        assert np.array_equal(batch["apple_den"][:, t].cpu().numpy(), np.repeat(den[:, None], n, 1)), ("apple_den", t)
        assert np.array_equal(batch["terminated"][:, t, 0].cpu().numpy(), out["done"]), ("terminated", t)
    return ora


def test_unmodified_episode_runner_fills_the_batch_from_the_cuda_env():
    cfg = _cfg(env_args=dict(num_agents=3, map="default3", episode_limit=30))
    c = refloop.build_components(cfg, backend="b200")
    import runners.episode_runner as er
    from homophily_marl_b200 import pymarl_env
    assert type(c.runner) is er.EpisodeRunner and isinstance(c.runner.env, pymarl_env.CleanupEnv)
    spec = c.runner.env.sim.spec
    for ep in range(3):
        batch = c.runner.run(test_mode=False)
        assert bool(batch["filled"].all()) and batch.max_seq_length == 31
        # the facade replays tick 0 at its first reset(); every later reset() continues the env's tick counter
        _oracle_replay(batch, spec, seed=cfg["seed"], ticks_before=ep * 31)
        c.buffer.insert_episode_batch(batch)
    assert c.runner.t_env == 90
    sample = c.buffer.sample(3)
    sample.to(c.args.device)
    c.learner.train(sample, c.runner.t_env, 3)                 # HomophilyLearner.cal_loss_and_step on CUDA
    for k in ("loss_value_env", "loss_value_inc", "loss_sim"):
        assert np.isfinite(c.logger.stats[k][-1][1]), k
    c.runner.close_env()


def test_run_sequential_cleanup3_end_to_end_on_the_cuda_env():
    """BASELINE configs[3]: Cleanup default3, 3 agents, full homophily IQL rollout + Q-learning update loop."""
    cfg = _cfg(t_max=2500, batch_size=16, buffer_size=64, test_nepisode=2, test_interval=1000, log_interval=1000,
               runner_log_interval=1000, learner_log_interval=1000)
    r = refloop.run_training(cfg, backend="b200")
    st = r["stats"]
    for k in ("return_mean", "test_return_mean", "loss_value_env", "loss_value_inc", "loss_sim", "epsilon",
              "collective_return_mean", "equality_metric_mean", "ep_length_mean", "clean_num_mean", "apple_den_mean"):
        assert k in st and np.isfinite(st[k]), k
    assert st["ep_length_mean"] == 100.0
    t_logged, episodes = r["logger"].stats["episode"][-1]      # logged every 1000 env steps (run.py:236-240)
    assert t_logged >= 2000 and episodes >= 20
    print("run_sequential on the CUDA env: %.1f env-steps/s" % (2600 / r["seconds"]))


def test_batched_runner_with_the_reference_episodebatch_mac_and_learner():
    B = 256
    cfg = _cfg(runner="batched", batch_size_run=B, buffer_size=2 * B, batch_size=16, buffer_cpu_only=False,
               test_nepisode=B, env_args=dict(num_agents=3, map="default3", episode_limit=25))
    c = refloop.build_components(cfg, backend="b200")
    from components.episode_buffer import EpisodeBatch
    from homophily_marl_b200.batched_runner import BatchedEpisodeRunner
    assert type(c.runner) is BatchedEpisodeRunner
    spec = c.runner.env.spec
    ticks = 0
    for ep in range(2):
        batch = c.runner.run(test_mode=False)
        assert type(batch) is EpisodeBatch and batch.batch_size == B and bool(batch["filled"].all())
        assert batch["obs"].is_cuda and batch["obs"].dtype == torch.float32
        _oracle_replay(batch, spec, seed=cfg["seed"], ticks_before=ticks)
        ticks += 26
        c.buffer.insert_episode_batch(batch)
    assert c.runner.t_env == 2 * B * 25
    sample = c.buffer.sample(16)
    c.learner.train(sample[:, :sample.max_t_filled()], c.runner.t_env, 2 * B)
    for k in ("loss_value_env", "loss_value_inc", "loss_sim"):
        assert np.isfinite(c.logger.stats[k][-1][1]), k
    c.runner.run(test_mode=True)
    assert "test_return_mean" in c.logger.stats
    c.runner.close_env()


def test_run_sequential_with_the_batched_runner():
    B = 64
    # the whole B200 stack behind run_sequential: batched runner with 4 pipelined env ranges, fused u8 front end,
    # device epsilon-greedy, DeviceHomophilyLearner; MAC, agent network and replay buffer are the reference's
    cfg = _cfg(runner="batched", batch_size_run=B, buffer_size=4 * B, batch_size=16, buffer_cpu_only=False,
               env_groups=4, fused_frontend=True, action_selector="epsilon_greedy_b200", learner="homophily_learner_b200",
               t_max=3 * B * 100, test_nepisode=B, test_interval=2 * B * 100, log_interval=B * 100,
               runner_log_interval=B * 100, learner_log_interval=B * 100)
    r = refloop.run_training(cfg, backend="b200")
    st = r["stats"]
    for k in ("return_mean", "test_return_mean", "loss_value_env", "loss_value_inc", "loss_sim", "ep_length_mean"):
        assert k in st and np.isfinite(st[k]), k
    assert st["ep_length_mean"] == 100.0


def test_batched_runner_with_fused_front_end_and_device_selector():
    """f2 + f3 wired into the rollout: the MAC's rgb_preprocess is served by the tcgen05 front-end kernel from the env's u8
    buffer and epsilon-greedy runs as one kernel; the module path stays in place for the learner (autograd)."""
    B = 128
    cfg = _cfg(runner="batched", batch_size_run=B, buffer_size=2 * B, batch_size=8, buffer_cpu_only=False, fused_frontend=True,
               action_selector="epsilon_greedy_b200", test_nepisode=B, env_args=dict(num_agents=3, map="default3", episode_limit=20))
    c = refloop.build_components(cfg, backend="b200")
    from homophily_marl_b200.frontend import MacFrontEnd
    from homophily_marl_b200.selectors import DeviceEpsilonGreedySelector
    assert isinstance(c.runner.front, MacFrontEnd) and isinstance(c.mac.action_selector, DeviceEpsilonGreedySelector)
    calls = {"fused": 0}
    fwd = c.runner.front._front_end().forward

    def counting(*a, **k):
        calls["fused"] += 1
        return fwd(*a, **k)
    c.runner.front._front_end().forward = counting
    batch = c.runner.run(test_mode=False)
    assert calls["fused"] == 21 and bool(batch["filled"].all())               # one per select_actions_env call (T + 1)
    # the fused features equal the module's on the stored fp32 observations (tolerance: tests/test_gpu_frontend.py)
    t = 7
    x = batch["obs"][:, t].reshape(B * 3, 3, 15, 15)
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False      # the reference module in true fp32
    try:
        with torch.no_grad():
            want = c.runner.front.original(x)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    c.runner.env.obs_buf.zero_()
    lay = c.runner.env.layout
    u8 = (batch["obs"][:, t] * 256).to(torch.uint8)
    c.runner.env.obs_view().copy_(u8)
    got = c.runner.front._front_end().forward_env(c.runner.env)
    assert torch.allclose(got, want, rtol=0, atol=1e-5 * (1 + want.abs().max().item()))
    _oracle_replay(batch, c.runner.env.spec, seed=cfg["seed"])
    c.buffer.insert_episode_batch(batch)
    sample = c.buffer.sample(8)
    c.learner.train(sample[:, :sample.max_t_filled()], c.runner.t_env, B)      # optimiser step -> parameter versions change
    stamp = c.runner.front._stamp
    c.runner.run(test_mode=True)
    assert c.runner.front._stamp != stamp                                      # the weights were re-packed after the update
    assert np.isfinite(c.logger.stats["loss_value_env"][-1][1])
    c.runner.close_env()
