"""Batched episode runner (SURVEY 8f row f1): B env instances in lockstep, device-resident episode data.

Mirrors ``EpisodeRunner`` of the reference (src/runners/episode_runner.py:8-152) -- same ``setup`` / ``run`` /
``reset`` / ``get_env_info`` / ``close_env`` / ``save_replay`` surface, same order of ``batch.update`` calls, same
keys -- but drives ``SSDBatchEnv`` with ``batch_size_run = B`` and hands **device tensors** to
``EpisodeBatch.update`` (its tensor fast path, src/components/episode_buffer.py:103-104), so no observation ever
visits the host.  ``new_batch`` is the reference's own ``partial(EpisodeBatch, scheme, groups, B, T+1, ...)``;
``mac`` is the reference's ``HomophilyMAC`` (or anything with the same three methods).

Differences that follow from B > 1 (all envs share ``episode_limit`` and terminate together, ``get_done`` is
constantly False in the reference, agent.py:192,243):
  * ``t_env`` advances by ``B * t`` per call (total env steps), ``n_episodes`` by B;
  * ``collective_return`` / ``equality_metric`` are summed over the B envs into the stats dict exactly as B
    successive single-env episodes would;
  * the step loop never synchronises with the host: ``terminated`` is the host-side step count (all envs share
    ``episode_limit``), and the state image comes out of the same launch as the step (``ssd_step_out.state_rgb``);
  * ``args.env_groups = G`` rolls the batch out as G env ranges on G streams (asynchronous sampler, ``ssd_step_range``).
"""
from __future__ import annotations

from functools import partial

import numpy as np
import torch

from . import _capi, mapspec
from .batch_env import SSDBatchEnv

# extra_args episode_stats: the social metrics and per-env event totals (summed over agents) added to env_info at episode end
SOCIAL_KEYS = ("efficiency", "sustainability", "peace")
EVENT_FIELDS = {"apples": _capi.SSD_STAT_APPLES, "fires": _capi.SSD_STAT_FIRES, "hits": _capi.SSD_STAT_HITS_DEALT,
                "cleaned": _capi.SSD_STAT_CLEANED}


class BatchedEpisodeRunner:
    def __init__(self, args, logger):
        self.args = args
        self.logger = logger
        self.batch_size = self.args.batch_size_run
        env_args = dict(self.args.env_args)
        env_args.pop("render", None)
        env_args.pop("is_replay", None)
        device = getattr(self.args, "device", "cuda:0")
        self.env = SSDBatchEnv(self.args.env, self.batch_size, env_args.pop("num_agents"),
                               map=env_args.pop("map", "default"), view_size=env_args.pop("view_size", 7),
                               episode_limit=env_args.pop("episode_limit", 100), extra_args=env_args.pop("extra_args", None),
                               seed=env_args.pop("seed", 0) or 0, device=device if str(device).startswith("cuda") else "cuda:0",
                               env_gid_base=getattr(self.args, "env_gid_base", 0), want_state=True)
        self.episode_limit = self.env.episode_limit
        self.t = 0
        self.t_env = 0
        self.train_returns, self.test_returns = [], []
        self.train_stats, self.test_stats = {}, {}
        self.log_train_stats_t = -1000000
        e = self.env
        avail = [1] * e.n_actions                             # map_env.py:972-980
        if e.extra_args["disable_rotation_action"]:
            avail[5] = avail[6] = 0
        if e.extra_args["disable_fire_action"]:
            avail[7] = 0
        self._avail = torch.tensor(avail, dtype=torch.int32, device=e.device).expand(e.B, e.n, e.n_actions).contiguous()
        self._orient_vec = torch.as_tensor(mapspec.ORIENT_VEC, dtype=torch.float32, device=e.device)
        self.groups = max(1, int(getattr(self.args, "env_groups", 1) or 1))
        if self.batch_size % self.groups:
            raise ValueError("env_groups must divide batch_size_run")
        self._streams = [torch.cuda.Stream(device=e.device) for _ in range(self.groups)] if self.groups > 1 else []
        self._actions_u8 = torch.zeros((e.B, e.n), dtype=torch.uint8, device=e.device)
        self.front = None
        self._vstats = {}                                     # per-variant sums since the last flush, by test_mode

    # ---- reference surface ------------------------------------------------------------------------------
    def setup(self, scheme, groups, preprocess, mac, batch_cls=None):
        """As episode_runner.py:28-31.  ``batch_cls`` defaults to the reference's EpisodeBatch when it is importable."""
        if batch_cls is None:
            from components.episode_buffer import EpisodeBatch as batch_cls   # the reference package (src/ on sys.path)
        self.new_batch = partial(batch_cls, scheme, groups, self.batch_size, self.episode_limit + 1,
                                 preprocess=preprocess, device=self.args.device)
        self.mac = mac
        # args.fused_frontend: during rollouts the MAC's rgb_preprocess (conv3x3 + FC on fp32 obs, homophily_controller.py:132-136)
        # is served by the fused u8 front-end kernel reading the env's observation buffer (frontend.MacFrontEnd).  True reads RGB
        # planes, "index4" packed colour indices; each needs the env to write that format.
        self.front = None
        fused = getattr(self.args, "fused_frontend", False)
        if fused is True and self.env.obs_format != "rgb":
            raise ValueError("fused_frontend: True reads RGB observation planes; with obs_format 'index4' use fused_frontend: index4")
        if fused == "index4" and self.env.obs_format != "index4":
            raise ValueError(f"fused_frontend: index4 needs obs_format 'index4', the env writes {self.env.obs_format!r}")
        if fused and fused is not True and fused != "index4":
            raise ValueError(f"fused_frontend must be False, True or 'index4', got {fused!r}")
        if fused and getattr(self.args, "rgb_input", False):
            from .frontend import MacFrontEnd
            self.front = MacFrontEnd(mac, self.env, obs_format="index4" if fused == "index4" else "rgb")

    def use_batch_factory(self, new_batch):
        """``new_batch()`` must return a fresh reference ``EpisodeBatch`` for B episodes of T+1 steps."""
        self.new_batch = new_batch

    def get_env_info(self):
        e = self.env
        return {"state_shape": (3, e.H, e.W), "obs_shape": (3, e.N, e.N), "n_actions": e.n_actions, "n_agents": e.n,
                "episode_limit": self.episode_limit, "units_type_id": None, "own_feature_size": None,
                "state_dims": (e.H, e.W), "obs_dims": (e.N, e.N)}

    def save_replay(self):
        return None

    def close_env(self):
        self.env.close()

    def reset(self):
        self.batch = self.new_batch()
        self.env.reset()
        self.env.render(want_obs=False, want_state=True)      # get_state() of the fresh episode; later states come from step
        self.t = 0

    # ---- device-side views of what the reference env returns per step -------------------------------------
    def _pre_transition(self, sl=slice(None)):
        e = self.env                                          # obs AND state image were written by the last step / reset launch
        lo, hi, _ = sl.indices(e.B)
        if e.obs_format == "rgb":
            obs = e.obs_view()[sl].float() / 256
        else:                                                 # index4: expanded on the current (the range's) stream
            obs = e.obs_float(lo, hi - lo)
        if e.state_format == "rgb":
            state = e.state_rgb[sl].float() / 256
        else:                                                 # index4 state image: expanded the same way
            state = e.state_float(lo, hi - lo)
        return {"state": state, "avail_actions": self._avail[sl],
                "obs": obs, "agent_pos": e.agent_pos[sl].float(),
                "agent_orientation": self._orient_vec[e.agent_orient[sl].long()]}

    def _range_step(self, r, t, last, homophily, test_mode, Bg):
        """One time step of one env range, in the call order of episode_runner.py:56-118."""
        e, mac, sl, batch = self.env, self.mac, r["sl"], r["batch"]
        self._give_hidden(r["hidden"])
        if self.front is not None:
            self.front.rows = (r["lo"] * e.n, Bg * e.n)
        batch.update(self._pre_transition(sl), ts=t)
        if homophily:
            actions = mac.select_actions_env(batch, t_ep=t, t_env=self.t_env, test_mode=test_mode)
        else:
            actions = mac.select_actions(batch, t_ep=t, t_env=self.t_env, test_mode=test_mode)
        if not last:
            self._actions_u8[sl] = (actions % self.args.n_actions).reshape(Bg, e.n).to(device=e.device, dtype=torch.uint8)
            if self.groups == 1:
                e.step(self._actions_u8, want_state=True)
            else:
                e.step_range(self._actions_u8, r["lo"], Bg, want_state=True)
            reward = e.reward[sl].float()
            r["ret"] += reward
            if e.shaped_buf is not None:                      # reward_shaping: the learner gets the shaped reward; the statistics
                reward = e.shaped_reward()[sl]                # stay extrinsic, plus shaped_return
                r["sret"] += reward
            post = {"actions": actions, "reward": reward if getattr(self.args, "ind_reward", True) else reward.sum(1, keepdim=True),
                    "terminated": e.done[sl].view(Bg, 1), "clean_num": e.clean[sl].float(),
                    "apple_den": (e.apple_cnt[sl].to(torch.int32) & 0xFFFF).double().view(Bg, 1).expand(Bg, e.n) / e.G}
            batch.update(post, ts=t)
        if homophily:
            actions_inc = mac.select_actions_inc(actions, batch, t_ep=t, t_env=self.t_env, test_mode=test_mode,
                                                 agent_pos_replay=e.agent_pos[sl].float())
            batch.update({"actions_inc": actions_inc}, ts=t)
        if last:
            batch.update({"actions": actions}, ts=t)
        r["hidden"] = self._take_hidden()

    def run(self, test_mode=False):
        if getattr(self, "front", None) is not None:
            self.front.active = True
        try:
            # rollouts never back-propagate; the reference's one-env runner simply lets autograd record them, which at
            # B envs x 100 steps keeps the whole episode's activations alive (176 GB at B = 4096)
            with torch.no_grad():
                return self._run(test_mode)
        finally:
            if getattr(self, "front", None) is not None:
                self.front.active = False

    def _take_hidden(self):
        return tuple(getattr(self.mac, k, None) for k in ("h_env", "h_inc"))

    def _give_hidden(self, hidden):
        for k, v in zip(("h_env", "h_inc"), hidden):
            if v is not None:
                setattr(self.mac, k, v)

    def _run(self, test_mode=False):
        """One episode of all B envs.  With ``args.env_groups = G > 1`` the batch is rolled out as G independent env ranges,
        each with its own MAC hidden state and CUDA stream (``SSDBatchEnv.step_range``): while the GPU steps and renders one
        range, the host is already launching the policy of the next, and the logic phase of one range overlaps the
        observation stores of another.  Trajectories do not depend on G (draws are keyed by the global env id)."""
        self.reset()
        e, B, G = self.env, self.batch_size, self.groups
        Bg = B // G
        homophily = "homophily" in getattr(self.args, "name", "homophily")
        if getattr(self.args, "mac", None) == "separate_mac":
            self.mac.init_latent(batch_size=Bg)
        main = torch.cuda.current_stream(e.device)
        ranges = []
        for k in range(G):
            sl = slice(k * Bg, (k + 1) * Bg)
            self.mac.init_hidden(batch_size=Bg)
            ranges.append({"sl": sl, "lo": k * Bg, "batch": self.batch if G == 1 else self.batch[sl],
                           "stream": main if G == 1 else self._streams[k], "hidden": self._take_hidden(),
                           "ret": torch.zeros(Bg, e.n, device=e.device),
                           "sret": None if e.shaped_buf is None else torch.zeros(Bg, e.n, device=e.device)})
            if G > 1:
                self._streams[k].wait_stream(main)
        # no host sync in the step loop: every env shares episode_limit and get_done() is constantly False in the reference
        # (agent.py:192,243; map_env.py:890-894), so termination is a host-side step count; the device-side `done` flags (what
        # goes into the batch) are checked against it once per episode below
        for t in range(self.episode_limit + 1):
            self.t = t
            for r in ranges:
                with torch.cuda.stream(r["stream"]):
                    self._range_step(r, t, t == self.episode_limit, homophily, test_mode, Bg)
        if G > 1:
            for k in range(G):
                main.wait_stream(self._streams[k])
        self.t = self.episode_limit
        episode_return = torch.cat([r["ret"] for r in ranges], dim=0)

        # termination info of every env (map_env.py:897-912), accumulated like B single-env episodes
        if not bool(e.done.all().item()):                     # first host sync of the episode
            raise RuntimeError("device-side done flags disagree with the host step count")
        R = e.ep_ret.double()
        if e.stats_buf is not None:                           # episode_stats: metrics and event totals ride on the same copy
            m, tot = e.social_metrics(), e.stats().double().sum(2)
            R = torch.cat([R] + [m[k][:, None] for k in SOCIAL_KEYS] + [tot[:, k, None] for k in EVENT_FIELDS.values()], 1)
        if e.shaped_buf is not None:                          # reward_shaping: the shaped returns ride on the same copy
            R = torch.cat([R, torch.cat([r["sret"] for r in ranges]).double()], 1)
        R = R.cpu().numpy()
        shaped = None
        if e.shaped_buf is not None:
            R, shaped = R[:, :-e.n], R[:, -e.n:].mean(axis=1)
        R, X = R[:, :e.n], R[:, e.n:]
        coll = R.sum(axis=1)
        denom = 2 * e.n * np.abs(R).sum(axis=1)
        pair = np.abs(R[:, None, :] - R[:, :, None]).sum(axis=(1, 2))
        eq = np.where(coll != 0, 1 - pair / np.where(denom == 0, 1, denom), 1.0)
        env_info = {"collective_return": float(coll.sum()), "equality_metric": float(eq.sum())}
        self.last_env_info = {"collective_return": coll, "equality_metric": eq}
        for j, k in enumerate(SOCIAL_KEYS + tuple(EVENT_FIELDS) if X.shape[1] else ()):
            env_info[k] = float(X[:, j].sum())
            self.last_env_info[k] = X[:, j]
        if shaped is not None:
            env_info["shaped_return"] = float(shaped.sum())
            self.last_env_info["shaped_return"] = shaped
        returns = episode_return.cpu().numpy()
        if len(e.variant_specs) > 1:                          # a sweep: the pooled means alone average the variants away
            vid = np.minimum(e.variant.cpu().numpy().astype(np.int64), len(e.variant_specs) - 1)
            self.last_env_info["variant"] = vid
            acc = self._vstats.setdefault(bool(test_mode), {})
            for k in np.unique(vid):
                m = vid == k
                a = acc.setdefault(int(k), {"n": 0, "return": 0.0, "collective_return": 0.0, "equality_metric": 0.0})
                a["n"] += int(m.sum())
                a["return"] += float(returns[m].mean(axis=1).sum())
                a["collective_return"] += float(coll[m].sum())
                a["equality_metric"] += float(eq[m].sum())
                for j, key in enumerate(SOCIAL_KEYS if X.shape[1] else ()):
                    a[key] = a.get(key, 0.0) + float(X[m, j].sum())
                if shaped is not None:
                    a["shaped_return"] = a.get("shaped_return", 0.0) + float(shaped[m].sum())

        self._account(env_info, returns, test_mode)
        return self.batch

    # ---- statistics: same keys and denominators as episode_runner.py:121-152, accumulated over B episodes at once ----
    def _account(self, env_info, returns, test_mode):
        B = self.batch_size
        stats, rets, prefix = ((self.test_stats, self.test_returns, "test_") if test_mode
                               else (self.train_stats, self.train_returns, ""))
        for key in set(stats) | set(env_info):
            stats[key] = stats.get(key, 0) + env_info.get(key, 0)
        stats["n_episodes"] = stats.get("n_episodes", 0) + B
        stats["ep_length"] = stats.get("ep_length", 0) + self.t * B
        if not test_mode:
            self.t_env += self.t * B
        rets.extend(returns)
        due_test = test_mode and len(self.test_returns) >= getattr(self.args, "test_nepisode", 1)
        due_train = self.t_env - self.log_train_stats_t >= getattr(self.args, "runner_log_interval", 10000)
        if due_test or due_train:
            self._flush(rets, stats, prefix)
            if not due_test:
                eps = getattr(getattr(self.mac, "action_selector", None), "epsilon", None)
                if eps is not None:
                    self.logger.log_stat("epsilon", eps, self.t_env)
                self.log_train_stats_t = self.t_env

    def _flush(self, rets, stats, prefix):
        log = self.logger.log_stat
        log(prefix + "return_mean", np.mean(rets), self.t_env)
        log(prefix + "return_std", np.std(rets), self.t_env)
        episodes = stats["n_episodes"]
        skip = {"n_episodes", "clean_num", "apple_den", "agent_pos", "agent_orientation"}
        for key in [k for k in stats if k not in skip]:
            log(prefix + key + "_mean", stats[key] / episodes, self.t_env)
        for k, a in sorted(self._vstats.pop(prefix == "test_", {}).items()):
            extra = tuple(q for q in SOCIAL_KEYS + ("shaped_return",) if q in a)
            for key in ("return", "collective_return", "equality_metric") + extra:
                log(f"{prefix}v{k}_{key}_mean", a[key] / a["n"], self.t_env)
        rets.clear()
        stats.clear()
