"""GPU suite (SURVEY 8f f1): the batched runner fills an EpisodeBatch exactly as B runs of the reference's single-env
runner loop would (src/runners/episode_runner.py:48-141), while keeping every tensor on the device."""
import numpy as np
import pytest

from harness import FakeBatch, ScriptedMAC, _scheme, action_tables, make_runner

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.mark.parametrize("name,mp,n,view,groups", [("cleanup", "default3", 3, 7, 1), ("harvest", "default10", 5, 15, 1),
                                                    ("cleanup", "default3", 3, 7, 3)])
def test_batched_runner_equals_sequential_facade_runs(name, mp, n, view, groups):
    from homophily_marl_b200 import REGISTRY
    B, T = 6, 9
    logged = {}
    runner = make_runner(name, mp, n, view, B=B, T=T, groups=groups, extra=dict(obs_color="full"),
                         log_stat=lambda k, v, t: logged.__setitem__(k, v))
    env_args, A, dev = runner.args.env_args, runner.env.n_actions, runner.env.device
    table, table_inc = action_tables(runner, 0, high=2 * A)                          # exercises `actions % n_actions`
    runner.mac = ScriptedMAC(table, table_inc)
    info = runner.get_env_info()
    scheme = _scheme(n, A, *info["state_dims"], info["obs_dims"][0])
    batch = runner.run(test_mode=True)
    assert runner.t == T and runner.t_env == 0 and bool(batch["filled"].all())
    assert set(logged) >= {"test_return_mean", "test_collective_return_mean", "test_equality_metric_mean", "test_ep_length_mean"}
    assert logged["test_ep_length_mean"] == T

    # the same episodes, one env at a time, through the PyMARL facade and the reference runner's call order
    coll = []
    for b in range(B):
        env = REGISTRY[name](**env_args, quiet=True, env_gid_base=b)
        ref = FakeBatch(scheme, 1, T + 1, dev)
        env.reset()
        terminated, t = False, 0
        while not terminated:
            ref.update({"state": [env.get_state()], "avail_actions": [env.get_avail_actions()], "obs": [np.stack(env.get_obs())],
                        "agent_pos": [env.get_agent_pos()], "agent_orientation": [env.get_agent_orientation()]}, ts=t)
            actions = table[b:b + 1, t]
            reward, terminated, env_info = env.step((actions % A)[0])
            ref.update({"actions": actions, "reward": [(reward,)], "terminated": [(terminated,)],
                        "clean_num": [(env_info["clean_num"],)], "apple_den": [(env_info["apple_den"],)]}, ts=t)
            ref.update({"actions_inc": table_inc[b:b + 1, t]}, ts=t)
            t += 1
        ref.update({"state": [env.get_state()], "avail_actions": [env.get_avail_actions()], "obs": [np.stack(env.get_obs())],
                    "agent_pos": [env.get_agent_pos()], "agent_orientation": [env.get_agent_orientation()]}, ts=t)
        ref.update({"actions_inc": table_inc[b:b + 1, t]}, ts=t)
        ref.update({"actions": table[b:b + 1, t]}, ts=t)
        for k in scheme:
            if not torch.equal(batch[k][b:b + 1], ref[k]):
                bad = (batch[k][b:b + 1] != ref[k]).nonzero()
                raise AssertionError((name, b, k, bad[:5].tolist(), batch[k][b:b + 1][tuple(bad[0])].item(), ref[k][tuple(bad[0])].item()))
        coll.append(env_info["collective_return"])
        assert env_info["equality_metric"] == runner.last_env_info["equality_metric"][b]
        env.close()
    assert np.array_equal(np.array(coll), runner.last_env_info["collective_return"])
    assert logged["test_collective_return_mean"] == pytest.approx(np.mean(coll))
