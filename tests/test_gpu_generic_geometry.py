"""GPU suite: geometries outside the compile-time specialisations -- custom ASCII maps, odd view sizes (generic row
pitch, non-zero agent-block tail), up to 16 agents, tiny and near-maximum maps -- against the oracle, Philox mode."""
import os
import runpy

import numpy as np
import pytest

from harness import custom_params, random_map
from oracle import oracle as O

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


CASES = [  # kind, H, W, n_agents, view
    ("cleanup", 5, 5, 2, 1), ("cleanup", 7, 9, 3, 2), ("cleanup", 12, 11, 16, 3), ("cleanup", 20, 33, 7, 5),
    ("cleanup", 40, 50, 10, 9), ("harvest", 6, 6, 4, 4), ("harvest", 9, 38, 5, 6), ("harvest", 16, 16, 16, 11),
    ("harvest", 31, 66, 8, 20), ("cleanup", 45, 45, 12, 31),
]


@pytest.mark.parametrize("kind,H,W,n,view", CASES)
def test_generic_geometry_matches_oracle(kind, H, W, n, view):
    from homophily_marl_b200.batch_env import SSDBatchEnv
    rs = np.random.RandomState(H * 1000 + W * 10 + n)
    rows = random_map(rs, kind, H, W, n_spawn=min(32, n + 3))
    params = custom_params(kind)
    B, T = 24, 30
    color = "full" if (H + W) % 2 else "simplified"
    env = SSDBatchEnv(kind, B, n, view_size=view, episode_limit=11, rows=rows, params=params, seed=42, env_gid_base=7,
                      extra_args=dict(random_spawn_point=True, random_spawn_rotation=None, obs_color=color), want_state=True)
    lay = env.layout
    assert lay.obs_row_stride == (2 * view + 4) // 4 * 4 and lay.obs_agent_stride % 16 == 0
    ora = O.OracleBatch.from_spec(env.spec, n_envs=B, seed=42, env_gid0=7, random_spawn_point=True, spawn_rotation=None)
    env.reset()
    ora.reset()
    assert np.array_equal(env.obs_view().cpu().numpy(), np.stack([ora.obs_one(b) for b in range(B)]))
    for t in range(T):
        act = rs.randint(0, env.n_actions, size=(B, n)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device), want_state=True)
        out = ora.step(act)
        for k in ("reward", "clean", "done"):
            assert np.array_equal(getattr(env, k).cpu().numpy(), out[k]), (t, k)
        assert np.array_equal(env.apple_cnt.cpu().numpy().view(np.uint16), out["apple_cnt"]), t
        assert np.array_equal(env.grid.cpu().numpy(), ora.grid), t
        assert np.array_equal(env.agent_pos.cpu().numpy(), ora.pos_rc), t
        assert np.array_equal(env.obs_view().cpu().numpy(), out["obs"]), t
        assert np.array_equal(env.state_rgb.cpu().numpy(), np.stack([ora.state_one(b) for b in range(B)])), t
        if out["done"].all():
            env.reset()
            ora.reset()
    # pad bytes (row padding and agent-block tail) are zero
    flat = env.obs_buf.view(B, n, lay.obs_agent_stride).cpu().numpy()
    planes = flat[:, :, : 3 * lay.obs_plane_stride].reshape(B, n, 3, env.N, lay.obs_row_stride)
    assert (planes[..., env.N:] == 0).all() and (flat[:, :, 3 * lay.obs_plane_stride:] == 0).all()
    assert int(ora.envs["error"].sum()) == 0


def test_maximum_map_size_and_rejects():
    from homophily_marl_b200 import _capi
    from homophily_marl_b200.batch_env import SSDBatchEnv
    rs = np.random.RandomState(1)
    rows = random_map(rs, "harvest", 32, 64, 8)                      # 2048 cells = SSD_MAX_CELLS
    env = SSDBatchEnv("harvest", 4, 8, view_size=7, episode_limit=5, rows=rows, seed=1,
                      params=__import__("homophily_marl_b200").mapspec.EnvParams(1, "custom", spawn_prob=(0, .1, .2, .3)))
    ora = O.OracleBatch.from_spec(env.spec, n_envs=4, seed=1)
    env.reset()
    ora.reset()
    for t in range(5):
        act = rs.randint(0, 8, size=(4, 8)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device))
        assert np.array_equal(env.obs_view().cpu().numpy(), ora.step(act)["obs"])
    with pytest.raises(ValueError):
        SSDBatchEnv("harvest", 4, 2, view_size=7, rows=random_map(rs, "harvest", 33, 64, 4))     # > SSD_MAX_CELLS
    with pytest.raises(_capi.SsdError) as ei:
        SSDBatchEnv("harvest", 4, 2, view_size=7, rows=["@@@@", "@PP ", "@@@@"])                  # open border
    assert ei.value.code == _capi.SSD_ERR_MAP


def test_all_paths_workload():
    """profiles/sanitizer_case.py: both envs, both colour schemes, every kernel mode, the specialised and the runtime geometry,
    injected draws.  tests/test_gpu_checked_build.py runs it on the checked build."""
    runpy.run_path(os.path.join(ROOT, "profiles", "sanitizer_case.py"), run_name="__main__")


@pytest.mark.parametrize("B,n", [(1, 1), (3, 1), (5, 2), (4097, 5)])
def test_ragged_batch_sizes_and_single_agent(B, n):
    """Batch sizes that do not fill the last CTA, and a single agent (no conflicts, every lane but one idle)."""
    from homophily_marl_b200.batch_env import SSDBatchEnv
    extra = dict(random_spawn_point=True, random_spawn_rotation=None)
    env = SSDBatchEnv("harvest", B, n, map="default10", view_size=15, episode_limit=9, seed=31, extra_args=extra)
    ora = O.OracleBatch.from_spec(env.spec, n_envs=B, seed=31, random_spawn_point=True, spawn_rotation=None)
    env.reset()
    ora.reset(threads=8)
    rs = np.random.RandomState(B)
    for t in range(12):
        act = rs.randint(0, 8, size=(B, n)).astype(np.uint8)
        env.step(torch.as_tensor(act, device=env.device))
        out = ora.step(act, threads=8)
        assert np.array_equal(env.reward.cpu().numpy(), out["reward"]) and np.array_equal(env.done.cpu().numpy(), out["done"])
        assert np.array_equal(env.obs_view().cpu().numpy(), out["obs"]), t
        if out["done"].all():
            env.reset()
            ora.reset(threads=8)
    assert np.array_equal(env.grid.cpu().numpy(), ora.grid)
