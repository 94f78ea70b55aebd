"""PyMARL ``MultiAgentEnv`` facade over the CUDA simulator (one env instance).

Drop-in for ``envs.REGISTRY['cleanup' | 'harvest']`` of the reference
(src/envs/__init__.py:6-11): same constructor kwargs (config/envs/*.yaml
``env_args``), same method names, argument meaning, return types and error
behaviour as ``MapEnv`` (src/envs/ssd/map_env.py:874-1022), so the unchanged
``EpisodeRunner`` (src/runners/episode_runner.py) and ``run_sequential`` drive it.

Every transition / observation comes from the sm_100a kernels; this file only
converts device buffers to the exact Python / NumPy types the callers expect.
"""
from __future__ import annotations

import os
from functools import partial

import numpy as np
import torch

from . import mapspec
from .batch_env import SSDBatchEnv
from .batched_runner import EVENT_FIELDS, SOCIAL_KEYS


class MultiAgentEnv(object):
    """Abstract surface (mirrors src/envs/multiagentenv.py:6-75)."""

    def step(self, actions):
        raise NotImplementedError

    def get_obs(self):
        raise NotImplementedError

    def get_own_feature_size(self):
        return None

    def get_obs_agent(self, agent_id):
        raise NotImplementedError

    def get_obs_size(self):
        raise NotImplementedError

    def get_state(self):
        raise NotImplementedError

    def get_state_size(self):
        raise NotImplementedError

    def get_avail_actions(self):
        raise NotImplementedError

    def get_avail_agent_actions(self, agent_id):
        raise NotImplementedError

    def get_total_actions(self):
        raise NotImplementedError

    def reset(self):
        raise NotImplementedError

    def render(self):
        raise NotImplementedError

    def close(self):
        raise NotImplementedError

    def seed(self):
        raise NotImplementedError

    def save_replay(self):
        raise NotImplementedError

    def get_units_type_id(self):
        return None

    def get_env_info(self):
        return {"state_shape": self.get_state_size(), "obs_shape": self.get_obs_size(),
                "n_actions": self.get_total_actions(), "n_agents": self.n_agents,
                "episode_limit": self.episode_limit, "units_type_id": self.get_units_type_id(),
                "own_feature_size": self.get_own_feature_size()}


class _SSDEnv(MultiAgentEnv):
    ENV_NAME = None

    def __init__(self, ascii_map=None, num_agents=1, render=False, seed=None, episode_limit=100,
                 is_replay=False, view_size=7, map="default", extra_args=None, device=None, quiet=False,
                 env_gid_base=0):
        extra = dict(random_spawn_point=False, random_spawn_rotation=0, disable_rotation_action=True,
                     disable_fire_action=True, obs_color="simplified")
        extra.update(extra_args or {})
        # get_obs / get_state are the reference's RGB arrays whatever extra_args says: the facade always runs the env in the
        # "rgb" formats
        extra["obs_format"] = extra["state_format"] = "rgb"
        # `ascii_map` is accepted and IGNORED, as in the reference: CleanupEnv / HarvestEnv replace it with the map that
        # `map=` selects (cleanup.py:31-54, harvest.py:18-22).  Custom maps: SSDBatchEnv(rows=...).
        device = device or os.environ.get("SSD_B200_DEVICE", "cuda:0")
        self.sim = SSDBatchEnv(self.ENV_NAME, 1, num_agents, map=map, view_size=view_size,
                               episode_limit=episode_limit, extra_args=extra, seed=0 if seed is None else int(seed),
                               device=device, want_state=True, env_gid_base=env_gid_base)
        if not quiet:                                   # cleanup.py:56-58 / harvest.py:24-26
            print("map difficulty: {}".format(map))
            for row in self.sim.spec.rows:
                print(row)
        self.extra_args = extra
        self.num_agents = self.n_agents = num_agents
        self.n_actions = self.sim.n_actions
        self.episode_limit = episode_limit
        self.view_size = view_size
        self.is_replay = is_replay
        self.env_name = self.ENV_NAME
        self._episode_steps = 0
        self.rewards = None
        self.clean_num = np.zeros(num_agents)
        self.apple_den = np.zeros(num_agents)
        self._io = self.sim.make_host_io(with_obs=True, with_state=True)   # pinned host mirrors: one sync per call
        lay = self.sim.layout
        self._obs_host = self._io["obs"].numpy().reshape(-1)[: lay.obs_env_stride]
        self._obs_strides = (lay.obs_agent_stride, lay.obs_plane_stride, lay.obs_row_stride, 1)
        self._act_host = self._io["actions"].numpy()[0]   # NumPy view of the pinned action row
        # reward_shaping: step() returns the shaped rewards (pinned mirror) and the episode's shaped return goes into info
        self._shaped_host = None if self.sim.shaped_buf is None else torch.zeros(self.sim.shaped_buf.shape).pin_memory()
        self._shaped_ret = np.zeros(num_agents, dtype=np.float32)
        self.sim.reset()                                # valid state before the first reset() ...
        self.sim.tick_buf.zero_()                       # ... which then replays the same draws (tick 0)
        self.sim.pull_host(self._io)

    # ------------------------------------------------------------------ step / reset
    def step(self, actions):
        """Returns reward, terminated, info (map_env.py:874-915)."""
        if isinstance(actions, torch.Tensor):            # the runner passes a device LongTensor [n, 1]: one D2H, not n
            acts = [int(a) for a in actions.reshape(-1).tolist()]
        else:
            acts = [int(a) for a in actions]
        for a in acts[:self.num_agents]:
            if not 0 <= a < self.n_actions:
                raise KeyError(a)                        # agent.py:176,237 action_map lookup
        io, sim = self._io, self.sim
        self._act_host[:] = acts[:self.num_agents]
        if sim.stats_buf is None and sim.shaped_buf is None:
            sim.step_host(io)                            # H2D actions, fused step+obs+state kernel, D2H results, sync
        else:                                            # episode_stats: ssd_step_host leaves the counters alone, so the same
            io["d_actions"].copy_(io["actions"], non_blocking=True)      # copies go around ssd_step (reward_shaping: and
            sim.step(io["d_actions"], want_state=True)                   # one more for the shaped rewards)
            for k in ("reward", "clean", "apple_cnt", "done"):
                io[k].copy_(getattr(sim, k), non_blocking=True)
            io["obs"].copy_(sim.obs_buf, non_blocking=True)
            io["state"].copy_(sim.state_buf, non_blocking=True)
            if self._shaped_host is not None:
                self._shaped_host.copy_(sim.shaped_buf, non_blocking=True)
        sim.pull_host(io, obs=False, state=False, agent=True)
        reward = io["reward"][0].numpy().astype(float)
        if self.rewards is None:
            self.rewards = reward
        else:
            self.rewards += reward
        if self._shaped_host is not None:                # what the learner sees; the termination metrics stay extrinsic
            shaped = self._shaped_host[0, :self.num_agents].numpy()
            self._shaped_ret += shaped
            reward = shaped.astype(float)
        self._episode_steps += 1
        terminated = bool(io["done"][0])                 # python bool: SURVEY 8b pitfall
        info = {}
        if terminated:
            collective_return = self.rewards.sum()
            equality_metric = 1.0
            if self.rewards.sum() != 0:
                equality_metric = 1 - (np.abs(self.rewards.reshape(1, -1) - self.rewards.reshape(-1, 1)).sum()) / (
                    2 * len(self.rewards) * np.abs(self.rewards).sum())
            info = {"collective_return": collective_return, "equality_metric": equality_metric}
            if sim.stats_buf is not None:                # episode_stats: one more D2H copy, at episode end only
                m, tot = sim.social_metrics(), sim.stats()[0].double().sum(1)
                vals = torch.cat([m[k] for k in SOCIAL_KEYS] + [tot[list(EVENT_FIELDS.values())]]).cpu().tolist()
                info.update(zip(SOCIAL_KEYS + tuple(EVENT_FIELDS), vals))
            if self._shaped_host is not None:            # mean over agents of the episode's shaped return, as the batched runner
                info["shaped_return"] = float(self._shaped_ret.astype(np.float64).mean())
        self.clean_num = io["clean"][0].numpy().astype(float)
        density = (int(io["apple_cnt"][0]) & 0xFFFF) / sim.G
        self.apple_den = np.full(self.n_agents, density, dtype=float)
        info["clean_num"] = self.clean_num
        info["apple_den"] = self.apple_den
        return reward, terminated, info

    def reset(self):
        """Reset the environment (map_env.py:986-993); returns None like the reference."""
        self.sim.reset()
        self.sim.pull_host(self._io)
        self._episode_steps = 0
        self.rewards = None
        self._shaped_ret[:] = 0
        return

    # ------------------------------------------------------------------ queries (served from the pinned mirrors)
    def _agent_records(self):
        return self._io["agent"][0, :self.num_agents].numpy().astype(np.int64)

    def get_agent_pos(self):
        a = self._agent_records()
        return np.stack([a & 0xFF, (a >> 8) & 0xFF], axis=-1).astype(float)

    def get_agent_orientation(self):
        return mapspec.ORIENT_VEC[(self._agent_records() >> 16) & 3].astype(float)

    def _obs_u8(self):
        n, N = self.num_agents, self.sim.N
        return np.lib.stride_tricks.as_strided(self._obs_host, shape=(n, 3, N, N), strides=self._obs_strides)

    def get_obs(self):
        """List of n arrays (3, N, N) float = u8 / 256 (map_env.py:923-945).  Always RGB: the facade ignores
        ``extra_args["obs_format"]``."""
        return list(self._obs_u8() / 256)

    def get_obs_agent(self, agent_id):
        return self._obs_u8()[int(agent_id)] / 256

    def get_obs_size(self):
        return (3, self.sim.N, self.sim.N)

    def get_state(self):
        """(3, H, W) float = u8 / 256 (map_env.py:950-957)."""
        return self._io["state"][0].numpy() / 256

    def get_state_size(self):
        return (3, self.sim.H, self.sim.W)

    def get_own_feature_size(self):
        return None

    def get_avail_actions(self):
        return [self.get_avail_agent_actions(i) for i in range(self.num_agents)]

    def get_avail_agent_actions(self, agent_id):
        available_actions = [1] * self.n_actions            # map_env.py:972-980 (advisory, SURVEY D10)
        if self.extra_args["disable_rotation_action"]:
            available_actions[5] = 0
            available_actions[6] = 0
        if self.extra_args["disable_fire_action"]:
            available_actions[7] = 0
        return available_actions

    def get_total_actions(self):
        return self.n_actions

    def get_env_info(self):
        info = super().get_env_info()
        info["state_dims"] = (self.sim.H, self.sim.W)
        info["obs_dims"] = (self.sim.N, self.sim.N)
        return info

    def get_stats(self):
        return {}

    def render(self):
        return None

    def close(self):
        self.sim.close()

    def seed(self):
        return None

    def save_replay(self):
        return None


class CleanupEnv(_SSDEnv):
    ENV_NAME = "cleanup"


class HarvestEnv(_SSDEnv):
    ENV_NAME = "harvest"


def env_fn(env, **kwargs) -> MultiAgentEnv:
    return env(**kwargs)


REGISTRY = {"harvest": partial(env_fn, env=HarvestEnv), "cleanup": partial(env_fn, env=CleanupEnv)}
